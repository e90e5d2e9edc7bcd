"""BASELINE configs[4]: the reference's scenes/tr15.json with synthetic stand-ins for its assets.

tr15.json references 13 OBJ files (cone, teapot, teapot2, u_logo, buddha, dragon, rust_logo, lucy, ajax, cow and three
kenny_nl trees) and 5 MERL BRDF files that are NOT in the reference repository (SURVEY §8d). This script

  * fixture(scenes): re-serialises tr15.json from a tray_rust checkout's scenes/ directory into tests/golden/scenes/c5_tr15.json
                (and logo_shadow / logo_with_friends / suzanne_scene.json, which only the loader test reads) —
                the scene DESCRIPTION (camera / group / object keyframes, materials, lights) is the reference's, unchanged;
  * write_assets(root): generates, next to that JSON, procedural OBJ files carrying the model names tr15.json asks for
                (closed noisy icospheres / cones with normals and uvs, sized like the originals' roles: ~80 k triangles for the
                scanned statues, a few thousand for props) and MERL-format binaries from analytic lobes (one tint per file).
                ~190 MB, generated where needed (GPU box, CPU tests), never committed.

    python tests/golden/make_tr15.py [--force] [SCENES]   # write the assets; with SCENES, refresh the fixtures from it first
"""
import json
import math
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
REPO = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, REPO)
SCENES = os.path.join(HERE, "scenes")
FIXTURES = {"tr15.json": "c5_tr15.json", "logo_shadow.json": "logo_shadow.json", "logo_with_friends.json": "logo_with_friends.json",
            "suzanne_scene.json": "suzanne_scene.json"}

# file -> [(model name, kind, subdivisions, anisotropic scale, noise, seed)]
MODELS = {
    "models/cone.obj": [("Cone", "cone", 48, (1.0, 1.0, 1.0), 0.0, 1)],
    "models/teapot.obj": [("Teapot", "ico", 4, (1.3, 0.8, 1.0), 0.08, 2)],
    "models/teapot2.obj": [("Base", "ico", 4, (1.3, 0.7, 1.0), 0.06, 3), ("Top", "ico", 3, (0.5, 0.25, 0.5), 0.04, 4, (0.0, 0.9, 0.0))],
    "models/u_logo.obj": [("U_Logo", "ico", 4, (1.0, 1.4, 0.3), 0.03, 5)],
    "models/buddha.obj": [("buddha", "ico", 6, (0.5, 1.2, 0.5), 0.07, 6)],
    "models/dragon.obj": [("dragon", "ico", 6, (1.4, 0.7, 0.6), 0.09, 7)],
    "models/rust_logo.obj": [("rust_logo", "ico", 5, (1.0, 1.0, 0.15), 0.05, 8)],
    "models/lucy.obj": [("lucy", "ico", 6, (0.45, 1.5, 0.4), 0.06, 9)],
    "models/ajax.obj": [("Ajax", "ico", 5, (0.7, 1.0, 0.7), 0.05, 10)],
    "models/cow.obj": [("Cow", "ico", 4, (1.3, 0.8, 0.6), 0.08, 11)],
    "models/kenny_nl/Tree_01.obj": [("Leaves", "cone", 24, (1.0, 1.6, 1.0), 0.0, 12, (0.0, 1.0, 0.0)), ("Trunk", "ico", 2, (0.2, 0.6, 0.2), 0.0, 13)],
    "models/kenny_nl/Tree_02.obj": [("Leaves", "cone", 32, (1.2, 1.3, 1.2), 0.0, 14, (0.0, 0.9, 0.0)), ("Trunk", "ico", 2, (0.25, 0.5, 0.25), 0.0, 15)],
    "models/kenny_nl/tree_1_ornamented.obj": [
        ("Leaves", "cone", 32, (1.1, 1.7, 1.1), 0.0, 16, (0.0, 1.0, 0.0)), ("Trunk", "ico", 2, (0.2, 0.6, 0.2), 0.0, 17),
        ("Tinsel", "ico", 3, (1.15, 0.08, 1.15), 0.02, 18, (0.0, 1.4, 0.0)), ("Sphere1", "ico", 3, (0.15, 0.15, 0.15), 0.0, 19, (0.7, 1.2, 0.2)),
        ("Sphere2", "ico", 3, (0.15, 0.15, 0.15), 0.0, 20, (-0.6, 1.5, 0.3)), ("Sphere3", "ico", 3, (0.15, 0.15, 0.15), 0.0, 21, (0.2, 1.9, -0.6)),
        ("Sphere4", "ico", 3, (0.15, 0.15, 0.15), 0.0, 22, (-0.3, 2.2, -0.4)), ("Sphere5", "ico", 3, (0.15, 0.15, 0.15), 0.0, 23, (0.4, 2.5, 0.3)),
        ("Bunny", "ico", 4, (0.25, 0.3, 0.2), 0.08, 24, (0.9, 0.3, 0.0)), ("Suzanne", "ico", 4, (0.3, 0.25, 0.25), 0.07, 25, (-0.9, 0.3, 0.2))],
}
MERL = {"brdfs/black-oxidized-steel.binary": (0.25, 0.25, 0.27, 0.03), "brdfs/silver-paint.binary": (0.8, 0.8, 0.82, 0.06),
        "brdfs/gold-metallic-paint.binary": (0.9, 0.7, 0.3, 0.05), "brdfs/blue-acrylic.binary": (0.15, 0.3, 0.8, 0.02),
        "brdfs/brass.binary": (0.85, 0.65, 0.35, 0.04)}


def fixture(scenes):
    """Refresh the scene fixtures under tests/golden/scenes from `scenes`, the scenes/ directory of a tray_rust checkout."""
    for src, dst in FIXTURES.items():
        d = json.load(open(os.path.join(scenes, src)))
        json.dump(d, open(os.path.join(SCENES, dst), "w"), separators=(",", ":"))


def cone_mesh(segments):
    """Closed cone, apex up: side fan + base fan, smooth side normals, planar-ish uvs."""
    ang = np.arange(segments) * (2 * math.pi / segments)
    ring = np.stack([np.cos(ang), np.zeros(segments), np.sin(ang)], axis=1)
    v = np.concatenate([ring, [[0, 1, 0]], [[0, 0, 0]]])
    apex, centre = segments, segments + 1
    f = [(i, apex, (i + 1) % segments) for i in range(segments)] + [((i + 1) % segments, centre, i) for i in range(segments)]
    n = v.copy()
    n[:segments, 1] = 1.0
    n[apex] = (0, 1, 0); n[centre] = (0, -1, 0)
    n /= np.linalg.norm(n, axis=1, keepdims=True)
    uv = np.stack([0.5 + 0.5 * v[:, 0], 0.5 + 0.5 * v[:, 2]], axis=1)
    return v, n, uv, np.array(f, np.int64)


def model_mesh(spec):
    from tray_rust_b200 import scenebuild as SB
    name, kind, level, scale, noise, seed = spec[:6]
    offset = spec[6] if len(spec) > 6 else (0.0, 0.0, 0.0)
    if kind == "cone":
        v, n, uv, f = cone_mesh(level)
    else:
        v, n, uv, f = SB.icosphere_mesh(level, 1.0, noise, seed)
        v, n, uv, f = v.astype(np.float64), n.astype(np.float64), uv.astype(np.float64), f.astype(np.int64)
    s = np.array(scale)
    v = v * s + np.array(offset)
    n = n / s
    n /= np.linalg.norm(n, axis=1, keepdims=True)
    return name, v, n, uv, f


def write_obj(path, specs):
    os.makedirs(os.path.dirname(path), exist_ok=True)
    base = 0
    with open(path, "w") as out:
        out.write("# procedural stand-in written by tests/golden/make_tr15.py (the original model is not redistributable)\n")
        for spec in specs:
            name, v, n, uv, f = model_mesh(spec)
            out.write("o %s\n" % name)
            out.write("".join("v %.6f %.6f %.6f\n" % tuple(p) for p in v))
            out.write("".join("vt %.6f %.6f\n" % tuple(t) for t in uv))
            out.write("".join("vn %.6f %.6f %.6f\n" % tuple(x) for x in n))
            g = f + base + 1
            out.write("".join("f %d/%d/%d %d/%d/%d %d/%d/%d\n" % (a, a, a, b, b, b, c, c, c) for a, b, c in g))
            base += len(v)


def write_merl(path, tint):
    """MERL file format (material/merl.rs:51-84): int32 dims (90, 90, 180), then the r, g, b planes as float64."""
    os.makedirs(os.path.dirname(path), exist_ok=True)
    r, g, b, width = tint
    th = (np.arange(90) / 90.0) ** 2 * (np.pi / 2)
    td = np.arange(90) / 90.0 * (np.pi / 2)
    base = (np.exp(-(th[:, None] ** 2) / width) * 3.0 + 0.15) * (0.3 + 0.04 + 0.96 * (1 - np.cos(td[None, :])) ** 5)
    t = np.repeat(base[:, :, None], 180, axis=2).reshape(-1)
    with open(path, "wb") as f:
        f.write(np.array([90, 90, 180], np.int32).tobytes())
        for scale, k in ((1500.0, r), (1500.0, g), (1500.0 / 1.66, b)):
            f.write((t * k * scale).astype(np.float64).tobytes())


def write_assets(root=SCENES, force=False):
    for rel, specs in MODELS.items():
        p = os.path.join(root, rel)
        if force or not os.path.exists(p):
            write_obj(p, specs)
    for rel, tint in MERL.items():
        p = os.path.join(root, rel)
        if force or not os.path.exists(p):
            write_merl(p, tint)
    return root


if __name__ == "__main__":
    ref = [a for a in sys.argv[1:] if a != "--force"]
    if ref:
        fixture(ref[0])
        print("fixtures refreshed from", ref[0])
    print("assets under", write_assets(force="--force" in sys.argv))
