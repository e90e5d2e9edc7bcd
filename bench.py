#!/usr/bin/env python
"""bench.py — Mrays/s (primary+secondary) of the render hot path on N B200s, with roofline and CPU baseline.

    python bench.py --gpus N --steps K --warmup W            # our arm (one rank per GPU under torchrun for N > 1)
    python bench.py --impl reference --gpus N --steps K ...  # the CPU arm: the oracle port on the box's host cores
    python bench.py ... --dump-outputs DIR                   # also write the film and counters of the timed steps (dump_outputs)

Workload (BASELINE.json configs[3], SURVEY §8d C4): synthetic 1M-triangle random mesh inside the Cornell walls,
1920x1080, one 4096-spp frame rendered in additive passes. One STEP = one pass of `--spp-per-step` samples per pixel
per GPU over the frame, tile-sharded across ranks exactly like the reference's master/worker mode
(tray_rust_b200.dist.shard_blocks == master.rs:88-120): at N GPUs a step renders N*spp_per_step samples per pixel,
each rank its own interleaved share of the Morton block list; the per-rank films stay on the GPUs over the passes of
the frame and are SUM-reduced ONCE (ncclReduce called by libtrb itself, trb_comm_reduce_film) — the timed region of K
steps ends with that one reduce. Per-GPU work is therefore constant in N: "scaling": "weak".

`value`  : rays/s of the whole job with the scene resident in HBM and the film left on the device.
`e2e`    : the same metric through the reference-facing call trb_render (== Exec::render): per step it runs
           Scene::update_frame (TLAS rebuild + upload), the kernels, and copies the film back to host memory.
`roofline`: dominant kernel's algorithmic bytes (48 B/ray + 32 B/node test + 48 B/triangle test + 64 B/instance test,
           SURVEY §8d; counted by the kernel's own test counters in an untimed replay of the same passes) over its
           measured duration, against the measured HBM peak in MEASURED_PEAKS.json — AND, because the BVH is L2-resident,
           what ncu measured for the same launches (profiles/traffic.json): real DRAM bytes (`traffic`, `dram_gbs`,
           `dram_frac`), L2 sector traffic (`l2_gbs`), the L1TEX data-pipe and issue-slot utilisation, and what limits the kernel (`limiter`).
"""
import argparse
import json
import math
import os
import subprocess
import sys
import threading
import time

import numpy as np

REPO = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, REPO)

WORKLOAD = "C4 synthetic 1M-triangle random mesh in Cornell walls, 1920x1080, 4096 spp frame in passes (BASELINE configs[3])"
METRIC = "Mrays/s (primary+secondary)"


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=6)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--tris", type=int, default=1_000_000)
    ap.add_argument("--width", type=int, default=1920)
    ap.add_argument("--height", type=int, default=1080)
    ap.add_argument("--spp", type=int, default=4096)
    ap.add_argument("--spp-per-step", type=int, default=8)
    ap.add_argument("--seed", type=int, default=1)
    ap.add_argument("--cpu-seconds", type=float, default=15.0, help="target CPU time of the bounded cpu_baseline sample")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write what the timed path returned after its last step as DIR/<name>.npy")
    return ap.parse_args()


DUMP_PIXELS = 1 << 21   # 32 MiB of RGBW float32 (+ 16 MiB of float64 indices when sampled): the default 1920x1080 film goes whole


def dump_outputs(path, film, stats):
    """film.npy: the RGBW film the timed passes accumulated from zero (H x W x 4 float32; above DUMP_PIXELS pixels a fixed, seeded
    sample of them, N x 4, with their flat indices in film_pixel_index.npy); counters.npy: the trb_stats ray and test
    counters of the timed steps (float64; the two timing fields of trb_stats are left out). The film is summed with float
    atomics, so two runs agree to float32 rounding of those sums; the counters agree exactly."""
    os.makedirs(path, exist_ok=True)
    px = film.reshape(-1, 4)
    if len(px) > DUMP_PIXELS:
        idx = np.sort(np.random.default_rng(0).choice(len(px), DUMP_PIXELS, replace=False))
        np.save(os.path.join(path, "film_pixel_index.npy"), idx.astype(np.float64))
        film = px[idx]
    np.save(os.path.join(path, "film.npy"), film.astype(np.float32))
    np.save(os.path.join(path, "counters.npy"), stats[:8].astype(np.float64))


def alg_bytes(rays, node, tri, inst):
    """SURVEY §8d: 32 B ray in + 16 B hit out, 32 B per node box tested, 48 B per triangle tested, 64 B per instance tested."""
    return 48 * rays + 32 * node + 48 * tri + 64 * inst


class ClockSampler:
    """nvidia-smi clocks / throttle reasons DURING the timed region (B200_PROFILING.md)."""
    Q = "index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, index):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "--query-gpu=" + self.Q, "--format=csv,noheader,nounits", "-lms", "200", "-i", str(self.index)],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([x.strip() for x in line.split(",")])

    def stop(self):
        if self.proc:
            self.proc.terminate()
        sm = [float(r[1]) for r in self.rows if len(r) >= 8 and r[1].replace(".", "").isdigit()]
        mx = [float(r[2]) for r in self.rows if len(r) >= 8 and r[2].replace(".", "").isdigit()]
        reasons = set()
        for r in self.rows:
            if len(r) >= 8:
                for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[4:8]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None, "reasons": sorted(reasons), "samples": len(sm)}


def host_threads():
    """All host cores this process may use (torchrun exports OMP_NUM_THREADS=1, so the count is passed explicitly)."""
    try:
        return len(os.sched_getaffinity(0))
    except Exception:
        return os.cpu_count() or 1


def host_info():
    """What the CPU arm ran on: logical CPUs, affinity mask size, physical cores and the model name (from /proc/cpuinfo)."""
    info = {"nproc": os.cpu_count(), "affinity": host_threads(), "physical_cores": None, "model": None, "cgroup_cpu_quota_cores": None}
    try:   # a container CPU quota caps the all-core rate whatever nproc says
        q, per = open("/sys/fs/cgroup/cpu.max").read().split()
        info["cgroup_cpu_quota_cores"] = None if q == "max" else float(q) / float(per)
    except Exception:
        pass
    try:
        cores, phys, core = set(), None, None
        for line in open("/proc/cpuinfo"):
            if line.startswith("model name") and info["model"] is None:
                info["model"] = line.split(":", 1)[1].strip()
            elif line.startswith("physical id"):
                phys = line.split(":")[1].strip()
            elif line.startswith("core id"):
                core = line.split(":")[1].strip()
            elif not line.strip():
                if phys is not None and core is not None:
                    cores.add((phys, core))
                phys = core = None
        info["physical_cores"] = len(cores) or None
    except Exception:
        pass
    return info


def build_scene_desc(a):
    from tray_rust_b200 import scenebuild as SB
    return SB.scene_c4(a.tris, a.width, a.height, a.spp).finish()


def pin_openmp():
    """Pin the CPU arm's OpenMP threads (must happen before libgomp starts): one thread per core, neighbours close."""
    os.environ.setdefault("OMP_PROC_BIND", "close")
    os.environ.setdefault("OMP_PLACES", "cores")


def cpu_arm(a, desc, seconds, reps):
    """The timed CPU implementation of the path: the oracle port (the Rust reference cannot be built here: no cargo/rustc),
    baseline mode (per-ray transform recomposition like the reference), built -O3 -march=x86-64-v3 against glibc's libm
    (oracle/_build/liboracle_fast.so; the detmath build is the parity checker, not the timed arm). Single-thread rate on a
    small sample, then `reps` all-core repetitions of a bounded sample of the same workload; min / median / max reported so
    that a noisy or oversubscribed box is visible in the line."""
    from tray_rust_b200 import _ffi as F
    host = host_info()                 # before OpenMP pins this thread
    pin_openmp()
    from oracle import pyoracle as O   # the CPU arm: the one place besides tests/smoke that may execute oracle/
    threads = host_threads()
    if host.get("cgroup_cpu_quota_cores"):   # a container quota below the visible CPUs: more threads than that only adds throttling
        threads = max(1, min(threads, int(math.ceil(host["cgroup_cpu_quota_cores"]))))
    o = O.OracleScene(desc, "fast", baseline=True)
    o.update_frame(0, 0.0, 0.0)
    nb = o.n_blocks()
    mid = nb // 2
    kw = dict(flags=F.RENDER_NO_UPDATE, sample_first=0, sample_count=1, seed=a.seed)
    t0 = time.time()
    _, st = o.render(threads=1, block_start=mid, block_count=16, **kw)          # probe: single thread, 16 blocks
    dt = max(time.time() - t0, 1e-4)
    n1 = int(min(nb // 4, max(16, 16 * 2.5 / dt)))                               # ~2.5 s single-thread sample
    t0 = time.time()
    _, st1 = o.render(threads=1, block_start=mid - n1 // 2, block_count=n1, **kw)
    dt1 = time.time() - t0
    single = st1.rays_total() / dt1 / 1e6
    per_block = st1.rays_total() / n1
    count = int(min(nb, max(64 * threads, single * 1e6 * threads * 0.5 * seconds / reps / per_block)))   # assume ~50 % parallel efficiency for sizing
    start = max(0, mid - count // 2)
    vals, rays, samples, wall = [], 0, 0, 0.0
    for r in range(reps):
        t0 = time.time()
        _, stn = o.render(threads=threads, block_start=start, block_count=count, flags=F.RENDER_NO_UPDATE, sample_first=r, sample_count=1, seed=a.seed)
        dt = time.time() - t0
        vals.append(stn.rays_total() / dt / 1e6); rays += stn.rays_total(); samples += stn.camera_samples; wall += dt
    o.close()
    vals_sorted = sorted(vals)
    return {"value": float(np.median(vals)), "unit": "Mrays/s", "cores": threads, "kind": "port",
            "sample": "%d repetitions of %d of %d Morton blocks (8x8 px) x 1 spp of the same C4 scene, %.1f s wall in total; oracle port, baseline mode, "
                      "-O3 -march=x86-64-v3 + glibc libm, %d OpenMP threads pinned (OMP_PROC_BIND=%s)" % (reps, count, nb, wall, threads, os.environ.get("OMP_PROC_BIND")),
            "all_core": {"min": vals_sorted[0], "median": float(np.median(vals)), "max": vals_sorted[-1], "reps": vals},
            "single_thread": {"value": single, "sample": "%d blocks x 1 spp, %.1f s" % (n1, dt1)},
            "parallel_speedup": float(np.median(vals)) / single if single > 0 else None,
            "host": host, "samples_per_s": samples / wall, "rays": rays, "wall_s": wall}


def run_reference(a):
    """--impl reference: the CPU implementation of the path (oracle port, see cpu_arm) with all host threads; each step is one
    repetition of a bounded sample of the workload."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    desc = build_scene_desc(a)
    reps = a.warmup + a.steps
    c = cpu_arm(a, desc, seconds=4.0 * reps, reps=reps)
    vals = c["all_core"]["reps"][a.warmup:]
    v = float(np.mean(vals))
    c = dict(c, value=v)
    line = {"impl": "reference", "metric": METRIC, "value": v, "unit": "Mrays/s", "n_gpus": a.gpus, "steps": a.steps, "warmup": a.warmup,
            "ms_per_step": 1e3 * c["wall_s"] / reps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": WORKLOAD, "tris": a.tris, "width": a.width, "height": a.height, "spp": a.spp},
            "samples_per_s": c["samples_per_s"], "cpu_baseline": c,
            "e2e": {"value": v, "unit": "Mrays/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line, default=float))


def run_ours(a):
    import torch
    import torch.distributed as dist
    from tray_rust_b200 import api, _ffi as F
    from tray_rust_b200.dist import shard_interleaved, max_over_ranks, sum_over_ranks

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise RuntimeError("bench.py needs a CUDA device: tray_rust_b200 has no CPU fallback")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    # stdout carries exactly one JSON line: anything a library prints to fd 1 (e.g. NCCL's version banner) goes to stderr
    sys.stdout.flush()
    json_out = os.fdopen(os.dup(1), "w")
    os.dup2(2, 1)
    comm = None
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)   # plumbing only: barriers, max-over-ranks, shipping the NCCL unique id
    lib = F.load_trb()
    if world > 1:   # the data-path collective is the library's own: ncclReduce of the film from libtrb (trb_comm_*)
        uid = torch.tensor(list(api.Comm.unique_id()) if rank == 0 else [0] * 128, dtype=torch.uint8, device=dev)
        dist.broadcast(uid, 0)
        comm = api.Comm(bytes(uid.cpu().tolist()), world, rank, local)

    desc = build_scene_desc(a)
    t0 = time.time()
    g = api.Scene(desc, local)
    create_s = time.time() - t0
    g.update_frame(0, 0.0, 0.0)
    nb = g.n_blocks()
    shard = shard_interleaved(rank, world, chunk=32)   # contiguous ranges (master.rs) leave the ranks unevenly loaded
    bstart, bcount = 0, 0
    spp_step = a.spp_per_step * world            # weak scaling: N x the samples per pixel per step, tile-sharded
    n_total = a.warmup + a.steps
    assert spp_step * n_total <= g.spp, "not enough spp in the frame for the requested steps"

    film = torch.zeros((a.height, a.width, 4), dtype=torch.float32, device=dev)
    stats = torch.zeros(10, dtype=torch.int64, device=dev)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)   # > 126 MB L2
    stream = torch.cuda.current_stream().cuda_stream

    def step(i, flags=0, st=stats):
        flush.fill_(i & 0xFF)                                         # L2 flush between timed iterations
        g.render_device(film.data_ptr(), st.data_ptr(), stream, spp=a.spp, sample_first=i * spp_step, sample_count=spp_step,
                        block_start=bstart, block_count=bcount, seed=a.seed, **shard, flags=flags)

    for i in range(a.warmup):
        step(i)
    if comm:
        comm.reduce_film(film.data_ptr(), film.numel(), 0, stream)     # warm the communicator
    film.zero_()                                                        # the timed passes accumulate one frame's film from zero on every rank
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    stats.zero_()
    clocks = ClockSampler(local)
    if rank == 0:
        clocks.start()
    launches0 = lib.trb_launch_count()
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(a.steps)]
    kev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(a.steps)]
    e_begin, e_end = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    e_begin.record()
    for k in range(a.steps):
        i = a.warmup + k
        flush.fill_(i & 0xFF)
        kev[k][0].record()
        g.render_device(film.data_ptr(), stats.data_ptr(), stream, spp=a.spp, sample_first=i * spp_step, sample_count=spp_step,
                        block_start=bstart, block_count=bcount, seed=a.seed, **shard)
        kev[k][1].record()
    if comm:
        comm.reduce_film(film.data_ptr(), film.numel(), 0, stream)     # ONE film reduce for the passes of the frame (design: once per frame)
    e_end.record()
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    launches = lib.trb_launch_count() - launches0
    clk = clocks.stop() if rank == 0 else None
    total_ms = max_over_ranks(e_begin.elapsed_time(e_end), dev)
    kernel_ms = [kev[k][0].elapsed_time(kev[k][1]) for k in range(a.steps)]
    st = stats.cpu().numpy()
    if rank == 0 and a.dump_outputs:   # before the film buffer is reused below; rank 0 holds the reduced film
        dump_outputs(a.dump_outputs, film.cpu().numpy(), st)
    tot = sum_over_ranks([st[0], st[1], st[2], st[3], st[4]], dev)     # samples, primary, shadow, mis, continuation (all ranks)
    rays_all = sum(tot[1:5])

    # --- roofline of the dominant kernel (k_wf_trace), from two untimed replays of this rank's timed passes:
    #     (1) CUDA events around every trace launch -> its duration; (2) the test counters on -> its algorithmic bytes
    cstats = torch.zeros(10, dtype=torch.int64, device=dev)
    scratch = torch.zeros_like(film)
    for k in range(a.steps):
        i = a.warmup + k
        flush.fill_(i & 0xFF)
        g.render_device(scratch.data_ptr(), cstats.data_ptr(), stream, spp=a.spp, sample_first=i * spp_step, sample_count=spp_step,
                        block_start=bstart, block_count=bcount, seed=a.seed, **shard, flags=F.RENDER_TIME_TRACE)
    torch.cuda.synchronize()
    trace_ms, trace_launches = g.trace_time()
    cstats.zero_()
    for k in range(a.steps):
        i = a.warmup + k
        g.render_device(scratch.data_ptr(), cstats.data_ptr(), stream, spp=a.spp, sample_first=i * spp_step, sample_count=spp_step,
                        block_start=bstart, block_count=bcount, seed=a.seed, **shard, flags=F.RENDER_STATS)
    torch.cuda.synchronize()
    cs = cstats.cpu().numpy()
    rank_rays = int(cs[1:5].sum())
    bytes_total = alg_bytes(rank_rays, int(cs[5]), int(cs[6]), int(cs[7]))
    del scratch

    # --- primary + shadow rays only (the north-star target is quoted on them): the same scene with max_depth 0,
    #     i.e. one primary and one shadow ray per camera sample; secondary measurement, device-resident like `value`
    direct = None
    if world == 1:
        from tray_rust_b200 import scenebuild as SB
        b0 = SB.scene_c4(a.tris, a.width, a.height, a.spp)
        b0.integrator = (0, 0, 0)
        g0 = api.Scene(b0.finish(), local)
        g0.update_frame(0, 0.0, 0.0)
        dstats = torch.zeros(10, dtype=torch.int64, device=dev)
        for i in range(2):
            g0.render_device(film.data_ptr(), dstats.data_ptr(), stream, spp=a.spp, sample_first=i * spp_step, sample_count=spp_step, seed=a.seed)
        torch.cuda.synchronize(); dstats.zero_()
        d0, d1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        d0.record()
        for i in range(2, 2 + a.steps):
            g0.render_device(film.data_ptr(), dstats.data_ptr(), stream, spp=a.spp, sample_first=i * spp_step, sample_count=spp_step, seed=a.seed)
        d1.record(); torch.cuda.synchronize()
        ds = dstats.cpu().numpy()
        dms = d0.elapsed_time(d1)
        direct = {"mrays_s": float(ds[1:5].sum()) / dms / 1e3, "msamples_s": float(ds[0]) / dms / 1e3, "primary": int(ds[1]), "shadow": int(ds[2]),
                  "ms_per_step": dms / a.steps, "note": "same C4 scene, pathtracer max_depth 0: one primary + one (any-hit) shadow ray per camera sample"}
        g0.close()

    # --- e2e: through the public API with host buffers; per step: Scene::update_frame (TLAS rebuild + H2D upload),
    #     the kernels, the film reduce (N > 1) and the film D2H copy, all inside the timed region
    n_inst = desc.n_instances
    h2d = 2 * 1536 + 64   # update_frame runs on the device: per step only the two kernels' parameter blocks (scene header with the camera, build pointers) + the render config
    e2e_steps = max(2, min(a.steps, 4))
    if world == 1:
        hfilm = np.zeros((a.height, a.width, 4), np.float32)
        g.render(hfilm, spp=a.spp, sample_first=0, sample_count=spp_step, seed=a.seed)   # warm
        rays_e, t_e = 0, 0.0
        for k in range(e2e_steps):
            t0 = time.perf_counter()
            _, s_e = g.render(hfilm, spp=a.spp, sample_first=(a.warmup + k) * spp_step, sample_count=spp_step, seed=a.seed)
            t_e += time.perf_counter() - t0
            rays_e += s_e.rays_total()
        api_name = "trb_render (Exec::render): update_frame + kernels + film D2H"
    else:   # one trb_render_sharded per step on every rank: update_frame, this rank's shard, ONE ncclReduce, root's film D2H + host add
        hfilm = np.zeros((a.height, a.width, 4), np.float32) if rank == 0 else None
        comm.render_sharded(g, hfilm, 0, spp=a.spp, sample_first=0, sample_count=spp_step, seed=a.seed, shard_chunk=32)   # warm
        dist.barrier(); torch.cuda.synchronize()
        rays_rank, t0 = 0, time.perf_counter()
        for k in range(e2e_steps):
            _, s_e = comm.render_sharded(g, hfilm, 0, spp=a.spp, sample_first=(a.warmup + k) * spp_step, sample_count=spp_step, seed=a.seed, shard_chunk=32)
            rays_rank += s_e.rays_total()
        dist.barrier()
        t_e = max_over_ranks(time.perf_counter() - t0, dev)
        rays_e = sum(sum_over_ranks([rays_rank], dev))
        api_name = "trb_render_sharded on every rank (Exec::render of the distributed mode): update_frame + its tile shard + one ncclReduce of the film + root film D2H"
    e2e = {"value": rays_e / t_e / 1e6, "unit": "Mrays/s", "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": int(a.width * a.height * 16 + 80),
           "ms_per_step": 1e3 * t_e / e2e_steps, "steps": e2e_steps, "api": api_name}

    cpu = None
    if rank == 0 and world == 1 and not a.no_cpu_baseline:
        cpu = cpu_arm(a, desc, seconds=a.cpu_seconds, reps=3)

    if rank == 0:
        peaks = {}
        try:
            peaks = json.load(open(os.path.join(REPO, "MEASURED_PEAKS.json")))
        except Exception:
            pass
        peak = float(peaks.get("hbm_gbs", 6650.0))
        avg_kernel_ms = float(np.mean(kernel_ms))
        trace_launches = max(1, trace_launches)
        bytes_per_launch = bytes_total / trace_launches
        achieved = bytes_total / (trace_ms * 1e-3) / 1e9        # == bytes per launch / average launch duration
        # what ncu measured for the trace launches of one step of this same command (tools/traffic_from_ncu.py -> profiles/traffic.json)
        prof = {}
        try:
            prof = json.load(open(os.path.join(REPO, "profiles", "traffic.json")))
        except Exception:
            pass
        traffic = prof.get("dram_bytes_per_launch")
        launch_s = trace_ms / trace_launches * 1e-3
        dram_gbs = traffic / launch_s / 1e9 if traffic else None
        l2_gbs = prof["l2_bytes_per_launch"] / launch_s / 1e9 if prof.get("l2_bytes_per_launch") else None
        line = {
            "metric": METRIC, "value": rays_all / (total_ms * 1e-3) / 1e6, "unit": "Mrays/s", "n_gpus": world, "steps": a.steps, "warmup": a.warmup,
            "ms_per_step": total_ms / a.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": WORKLOAD, "tris": a.tris, "width": a.width, "height": a.height, "spp": a.spp, "spp_per_step": spp_step,
                       "blocks_per_rank": nb // world, "parallelism": "tile-sharded x%d (interleaved 32-block chunks of the Morton block list) + ONE film SUM-reduce (ncclReduce from libtrb) at the end of the timed passes" % world,
                       "l2": "256 MiB buffer written between timed steps (L2 flush)", "scene_create_s": round(create_s, 2)},
            "samples_per_s": tot[0] / (total_ms * 1e-3),
            "rays": {"primary": tot[1], "shadow": tot[2], "mis": tot[3], "continuation": tot[4],
                     "primary_plus_shadow_mrays_s": (tot[1] + tot[2]) / (total_ms * 1e-3) / 1e6},
            "roofline": {"bound": "hbm", "kernel": "k_wf_trace", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                         "peak_source": "MEASURED_PEAKS.json hbm_gbs (measured)" if peaks else "fallback 6650 GB/s",
                         "traffic": traffic, "dram_gbs": dram_gbs, "dram_frac": dram_gbs / peak if dram_gbs else None,
                         "l2_gbs": l2_gbs, "l1tex_data_pipe_pct": prof.get("l1tex_data_pipe_pct"), "issue_active_pct": prof.get("issue_active_pct"),
                         "limiter": "latency of dependent node fetches + SIMT divergence",
                         "note": "frac = ALGORITHMIC bytes (SURVEY 8d definition, reference data structure) over time vs the HBM peak; the ~90 MB BVH is L2-resident, so the "
                                 "HBM bandwidth ncu measures for the same launches is dram_gbs (dram_frac of peak). The busiest unit ncu shows is the L1TEX data pipe "
                                 "(l1tex_data_pipe_pct), but it is not the limiter: one more L1-hitting 256-bit load per node visit costs 2 % "
                                 "(profiles/r02_c16_diag_extra_l1_load.log); 38 % of warp time waits on the fetch of the next node record, 15.7 of 32 lanes are active",
                         "algorithmic_bytes_per_launch": bytes_per_launch, "launches": trace_launches,
                         "avg_launch_ms": trace_ms / trace_launches, "trace_ms_per_step": trace_ms / a.steps,
                         "step_kernels_ms": avg_kernel_ms,
                         "per_ray": {"node_tests": cs[5] / max(1, rank_rays), "tri_tests": cs[6] / max(1, rank_rays), "inst_tests": cs[7] / max(1, rank_rays)}},
            "primary_shadow_only": direct,
            "gpu_launches": int(launches), "clocks": clk, "e2e": e2e, "cpu_baseline": cpu,
        }
        json_out.write(json.dumps(line, default=float) + "\n")
        json_out.flush()
    g.close()
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    args = parse()
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)
