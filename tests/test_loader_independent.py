"""Independent check of the loader half of the drop-in (VERDICT r01 "parity is self-referential above the ABI"): every scene
file the reference ships is flattened twice — by the product's C++ loader (trb_desc_load_json) and by tests/loader_ref.py
(numpy restatement of tray_rust's src/scene.rs + keyframe.rs with LAPACK's SVD) — and compared field by field:
instance order / kinds / shapes / parameters, transform stacks (group levels, B-spline degree and knots), every TRS keyframe
of the f64-SVD polar decomposition, colour keys, materials, cameras, film, OBJ vertex unification and the MERL import.

The scene JSONs are the committed fixtures under tests/golden/scenes: re-serialised copies of the six files in tray_rust's
scenes/ directory (tests/golden/make_tr15.py). Assets that the reference repository does not contain (every OBJ but
cube.obj, every MERL file) are generated stand-ins (tests/golden/make_tr15.py)."""
import ctypes as C
import json
import os
import shutil
import sys

import numpy as np
import pytest

from tray_rust_b200 import _ffi as F

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, HERE)
sys.path.insert(0, os.path.join(HERE, "golden"))
import loader_ref as LR  # noqa: E402
import make_tr15  # noqa: E402

FIXTURES = {"cornell_box": "c1_cornell_box.json", "smallpt": "c2_smallpt.json", "logo_shadow": "logo_shadow.json",
            "logo_with_friends": "logo_with_friends.json", "suzanne_scene": "suzanne_scene.json", "tr15": "c5_tr15.json"}
SCENES = list(FIXTURES)


def stage(name, tmp):
    """Copy the scene JSON into tmp and put stand-in assets where its relative paths point."""
    src = os.path.join(HERE, "golden", "scenes", FIXTURES[name])
    dst = os.path.join(tmp, name + ".json")
    shutil.copy(src, dst)
    d = json.load(open(dst))
    wanted = {}

    def walk(objs):
        for o in objs:
            g = o.get("geometry")
            if g and g["type"] == "mesh":
                wanted.setdefault(g["file"], []).append(g["model"])
            if o["type"] == "group":
                walk(o["objects"])
    walk(d["objects"])
    for rel, models in wanted.items():
        p = os.path.join(tmp, rel)
        os.makedirs(os.path.dirname(p), exist_ok=True)
        if os.path.basename(rel) in ("cube.obj", "unit_cube.obj"):
            shutil.copy(os.path.join(HERE, "golden", "scenes", "models", "unit_cube.obj"), p)   # quads, distinct v/vt/vn indices
        elif rel in make_tr15.MODELS and set(models) <= {s[0] for s in make_tr15.MODELS[rel]}:
            make_tr15.write_obj(p, [s for s in make_tr15.MODELS[rel]])
        else:
            make_tr15.write_obj(p, [(m, "ico", 2, (1.0, 1.2, 0.8), 0.05, 100 + i) for i, m in enumerate(sorted(set(models)))])
    for i, m in enumerate(d["materials"]):
        if m["type"] == "merl":
            make_tr15.write_merl(os.path.join(tmp, m["file"]), (0.2 + 0.1 * i, 0.5, 0.9 - 0.1 * i, 0.03 + 0.01 * i))
    return dst


def close(a, b, tol=2e-5):
    a, b = np.asarray(a, np.float64), np.asarray(b, np.float64)
    return bool(np.all(np.abs(a - b) <= tol * np.maximum(1.0, np.maximum(np.abs(a), np.abs(b)))))


def check_levels(desc, first, count, levels, what):
    assert count == len(levels), what
    for k, lv in enumerate(levels):
        sp = desc.splines[first + k]
        assert sp.n_ctrl == len(lv["keys"]), what
        if sp.n_ctrl > 1:
            assert sp.degree == lv["degree"] and sp.n_knots == len(lv["knots"]), what
            assert [desc.knots[sp.knot_first + i] for i in range(sp.n_knots)] == [float(x) for x in lv["knots"]], what
        for i, key in enumerate(lv["keys"]):
            kf = desc.keyframes[sp.ctrl_first + i]
            assert close(list(kf.translation), key["t"]), (what, "translation", k, i)
            assert close(list(kf.scaling), key["s"]), (what, "scaling", k, i, list(kf.scaling), key["s"])
            q = np.array(list(kf.rotation), np.float64)
            if i == 0:   # q and -q are the same rotation; later keys are tied to the first by the shortest-path rule
                sign = 1.0 if np.linalg.norm(q - key["q"]) <= np.linalg.norm(q + key["q"]) else -1.0
            assert close(q, sign * key["q"].astype(np.float64)), (what, "rotation", k, i, q, key["q"])


@pytest.mark.parametrize("name", SCENES)
def test_loader_matches_the_independent_restatement(name, tmp_path, trb):
    path = stage(name, str(tmp_path))
    ref = LR.flatten(path)
    d = C.POINTER(F.SceneDesc)()
    assert trb.trb_desc_load_json(path.encode(), 0, 0, 0, C.byref(d)) == F.TRB_OK, trb.trb_last_error()
    try:
        desc = d.contents
        # film / integrator
        fj = ref["film"]
        assert (desc.film.width, desc.film.height, desc.film.samples, desc.film.frames, desc.film.start_frame, desc.film.end_frame) == \
               (fj["width"], fj["height"], fj["samples"], fj["frames"], fj["start_frame"], fj["end_frame"])
        assert desc.film.scene_time == np.float32(fj["scene_time"])
        flt = fj["filter"]
        assert desc.film.filter_type == {"mitchell_netravali": 0, "gaussian": 1}[flt["type"]]
        assert (desc.film.filter_w, desc.film.filter_h) == (np.float32(flt["width"]), np.float32(flt["height"]))
        if flt["type"] == "mitchell_netravali":
            assert (desc.film.filter_b, desc.film.filter_c) == (np.float32(flt["b"]), np.float32(flt["c"]))
        assert (desc.integrator.type, desc.integrator.min_depth, desc.integrator.max_depth) == (0, ref["integrator"]["min_depth"], ref["integrator"]["max_depth"])
        # cameras
        assert desc.n_cameras == len(ref["cameras"])
        for i, c in enumerate(ref["cameras"]):
            dc = desc.cameras[i]
            assert dc.shutter_size == c["shutter_size"] and dc.active_at == c["active_at"]
            check_levels(desc, dc.spline_first, dc.n_splines, c["levels"], "camera %d" % i)
            if isinstance(c["fov"], list):
                assert dc.n_fov_ctrl == len(c["fov"]) and dc.fov_degree == c["fov_degree"] and dc.n_fov_knots == len(c["fov_knots"])
                assert [desc.fov_floats[dc.fov_ctrl_first + k] for k in range(dc.n_fov_ctrl)] == [float(x) for x in c["fov"]]
            else:
                assert dc.n_fov_ctrl == 0 and dc.fov == c["fov"]
        # materials
        assert desc.n_materials == len(ref["materials"])
        for i, m in enumerate(ref["materials"]):
            dm = desc.materials[i]
            assert dm.type == m["type"], i
            if m["type"] != 6:
                assert list(dm.c0) == [float(x) for x in m["c0"]] and list(dm.c1) == [float(x) for x in m["c1"]], i
                assert dm.roughness == np.float32(m["roughness"]), i
                if m["eta"] is not None:
                    assert dm.eta == m["eta"], i
            else:
                assert dm.merl == m["merl"], i
        assert desc.n_merl == len(ref["merl"])
        for i, t in enumerate(ref["merl"]):
            got = np.ctypeslib.as_array(desc.merl_tables[i], shape=(F.MERL_TABLE_FLOATS,))
            assert got.tobytes() == t.tobytes(), "MERL table %d" % i
        # instances in JSON object order (Q20), transform stacks, emission, geometry
        assert desc.n_instances == len(ref["instances"])
        seen_mesh = {}
        for i, r in enumerate(ref["instances"]):
            di = desc.instances[i]
            what = "instance %d" % i
            assert (di.kind, di.shape) == (r["kind"], r["shape"]), what
            if r["shape"] != 4:
                assert (di.p0, di.p1) == (float(r["p0"]), float(r["p1"])), what
            if r["material"] is not None:
                assert di.material == r["material"], what
            check_levels(desc, di.spline_first, di.n_splines, r["levels"], what)
            if r["emission"] is not None:
                assert di.n_emission == len(r["emission"]), what
                for k, (col, time) in enumerate(r["emission"]):
                    ck = desc.color_keys[di.emission_first + k]
                    assert list(ck.rgba) == [float(x) for x in col] and ck.time == float(time), (what, k)
            if r["mesh"] is not None:
                seen_mesh.setdefault(r["mesh"], di.mesh)
                assert seen_mesh[r["mesh"]] == di.mesh, what          # the same (file, model) is loaded once and shared
                pos, nrm, uv, idx = ref["meshes"][r["mesh"]]
                dm = desc.meshes[di.mesh]
                assert (dm.n_verts, dm.n_tris) == (len(pos), len(idx)), what
                assert np.array_equal(np.ctypeslib.as_array(dm.indices, shape=(dm.n_tris * 3,)), idx.reshape(-1)), what
                assert close(np.ctypeslib.as_array(dm.positions, shape=(dm.n_verts * 3,)), pos.reshape(-1), 1e-7), what
                assert close(np.ctypeslib.as_array(dm.normals, shape=(dm.n_verts * 3,)), nrm.reshape(-1), 1e-7), what
                assert close(np.ctypeslib.as_array(dm.texcoords, shape=(dm.n_verts * 2,)), uv.reshape(-1), 1e-7), what
        assert len(seen_mesh) == desc.n_meshes
    finally:
        trb.trb_desc_free(d)
