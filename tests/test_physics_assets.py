"""Physics asset pipeline (mb2_process_rigid_body_assets) against the reference's own
RigidBodyAssets::processRigidBodyAssets (src/physics/physics_assets.cpp:1268, run by
oracle/assets_probe.cpp; its output is stored under tests/golden): half-edge numbering, face planes, AABBs and the mass
properties (centre of mass, diagonalised inertia, inertia frame) must be bit-identical."""
import hashlib
import os
import struct
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))

from sims.objects import orient_faces  # noqa: E402

GOLDEN = os.path.join(ROOT, "tests", "golden", "assets_probe_ref.npz")


def _prism(n, sx=1.0, sy=1.0, sz=1.0, offset=(0, 0, 0)):
    ang = 2.0 * np.pi * np.arange(n) / n
    ring = [(0.5 * np.cos(a), 0.5 * np.sin(a)) for a in ang]
    v = np.array([[x * sx + offset[0], y * sy + offset[1], z * sz + offset[2]]
                  for z in (-0.5, 0.5) for (x, y) in ring], dtype=np.float32)
    faces = [list(range(n)), list(range(n, 2 * n))] + [[i, (i + 1) % n, (i + 1) % n + n, i + n] for i in range(n)]
    return v, orient_faces(v, faces)


def _box(sx, sy, sz, offset=(0, 0, 0)):
    v = np.array([[x * sx + offset[0], y * sy + offset[1], z * sz + offset[2]]
                  for z in (-0.5, 0.5) for y in (-0.5, 0.5) for x in (-0.5, 0.5)], dtype=np.float32)
    faces = [[0, 2, 3, 1], [4, 5, 7, 6], [0, 1, 5, 4], [2, 6, 7, 3], [0, 4, 6, 2], [1, 3, 7, 5]]
    return v, faces


def _wedge():
    t = 1.0 / 3.0
    tri = [(-t, -t), (2 * t, -t), (-t, 2 * t)]
    v = np.array([[x * 2.0, y * 3.0, z] for y in (-0.5, 0.5) for (x, z) in tri], dtype=np.float32)
    faces = [[0, 1, 2], [3, 4, 5], [0, 1, 4, 3], [0, 2, 5, 3], [1, 2, 5, 4]]
    return v, orient_faces(v, faces)


def _tetra():
    v = np.array([[0.1, 0.2, 0.3], [1.3, 0.1, 0.2], [0.2, 1.1, 0.4], [0.3, 0.4, 1.7]], dtype=np.float32)
    return v, orient_faces(v, [[0, 1, 2], [0, 1, 3], [1, 2, 3], [0, 2, 3]])


def _random_hull(seed):
    """Convex polyhedron with merged coplanar faces: a box cut by random planes is awkward to
    mesh here, so use an irregular bipyramid (all faces triangles, no coplanarity)."""
    rng = np.random.default_rng(seed)
    n = int(rng.integers(5, 9))
    ang = np.sort(rng.uniform(0, 2 * np.pi, n))
    ang = ang + np.arange(n) * 1e-3
    r = rng.uniform(0.8, 1.2)
    ring = [[r * np.cos(a), r * np.sin(a), 0.0] for a in ang]
    v = np.array(ring + [[0.05, -0.03, rng.uniform(0.5, 1.5)], [0.02, 0.04, -rng.uniform(0.5, 1.5)]],
                 dtype=np.float32)
    v += rng.uniform(-0.3, 0.3, 3).astype(np.float32)
    faces = []
    for i in range(n):
        faces.append([i, (i + 1) % n, n])
        faces.append([i, (i + 1) % n, n + 1])
    return v, orient_faces(v, faces)


def _case():
    hulls = [_box(1, 1, 1), _box(1.5, 0.5, 2.5, (0.25, -1.0, 0.5)), _wedge(), _prism(6), _prism(24, 2.0, 1.0, 0.5),
             _tetra()] + [_random_hull(s) for s in range(6)]
    objects = [
        dict(prims=[("hull", 0)], inv_mass=0.1, mu_s=0.5, mu_d=0.75),
        dict(prims=[("hull", 1)], inv_mass=0.02, mu_s=0.4, mu_d=0.6),
        dict(prims=[("hull", 2)], inv_mass=0.5),
        dict(prims=[("hull", 3)], inv_mass=0.25),
        dict(prims=[("hull", 4)], inv_mass=0.05),
        dict(prims=[("hull", 5)], inv_mass=1.5),
        dict(prims=[("sphere", 0.75)], inv_mass=2.0),
        dict(prims=[("plane",)], inv_mass=0.0),
        dict(prims=[("hull", 0)], inv_mass=0.0),                       # static box: inverse inertia 0
        dict(prims=[("hull", 1), ("hull", 3)], inv_mass=0.125),         # compound
        dict(prims=[("hull", 2), ("sphere", 0.5), ("hull", 5)], inv_mass=0.2),
    ] + [dict(prims=[("hull", 6 + s)], inv_mass=0.3 + 0.1 * s) for s in range(6)]
    return hulls, objects


def _write_probe_input(path, hulls, objects):
    types = {"sphere": 1, "hull": 2, "plane": 4}
    with open(path, "wb") as f:
        f.write(struct.pack("<I", len(hulls)))
        for pos, faces in hulls:
            idx = [v for loop in faces for v in loop]
            f.write(struct.pack("<III", len(pos), len(faces), len(idx)))
            f.write(np.ascontiguousarray(pos, dtype=np.float32).tobytes())
            f.write(np.asarray([len(loop) for loop in faces], dtype=np.uint32).tobytes())
            f.write(np.asarray(idx, dtype=np.uint32).tobytes())
        f.write(struct.pack("<I", len(objects)))
        for obj in objects:
            f.write(struct.pack("<Ifff", len(obj["prims"]), obj["inv_mass"], obj.get("mu_s", 0.5),
                                obj.get("mu_d", 0.5)))
            for p in obj["prims"]:
                f.write(struct.pack("<IfI", types[p[0]], float(p[1]) if p[0] == "sphere" else 0.0,
                                    int(p[1]) if p[0] == "hull" else 0))


def _read_probe_output(path):
    raw = open(path, "rb").read()
    at = 0

    def take(n):
        nonlocal at
        out = raw[at:at + n]
        at += n
        return out
    n_he, n_f, n_v, n_p, n_o = struct.unpack("<5I", take(20))
    out = {
        "half_edges": np.frombuffer(take(12 * n_he), dtype=np.uint32).reshape(-1, 3),
        "face_base": np.frombuffer(take(4 * n_f), dtype=np.uint32),
        "planes": np.frombuffer(take(16 * n_f), dtype=np.float32).reshape(-1, 4),
        "vertices": np.frombuffer(take(12 * n_v), dtype=np.float32).reshape(-1, 3),
    }
    prims = []
    for _ in range(n_p):
        (type_,) = struct.unpack("<I", take(4))
        if type_ == 1:
            prims.append((type_, struct.unpack("<f", take(4))[0]))
        elif type_ == 2:
            prims.append((type_,) + struct.unpack("<6I", take(24)))
        else:
            prims.append((type_,))
    out["prims"] = prims
    out["prim_aabbs"] = np.frombuffer(take(24 * n_p), dtype=np.float32).reshape(-1, 6)
    out["metadatas"] = np.frombuffer(take(52 * n_o), dtype=np.float32).reshape(-1, 13)
    out["obj_aabbs"] = np.frombuffer(take(24 * n_o), dtype=np.float32).reshape(-1, 6)
    out["prim_offsets"] = np.frombuffer(take(4 * n_o), dtype=np.uint32)
    out["prim_counts"] = np.frombuffer(take(4 * n_o), dtype=np.uint32)
    assert at == len(raw)
    return out


def _compare(mine, ref):
    for key in ("half_edges", "face_base", "planes", "vertices", "prim_aabbs", "metadatas", "obj_aabbs",
                "prim_offsets", "prim_counts"):
        a = np.ascontiguousarray(mine[key]).view(np.uint8).reshape(-1)
        b = np.ascontiguousarray(ref[key]).view(np.uint8).reshape(-1)
        assert a.shape == b.shape, key
        assert np.array_equal(a, b), f"{key} differs from the reference"
    assert len(mine["prims"]) == len(ref["prims"])
    for a, b in zip(mine["prims"], ref["prims"]):
        if a[0] == 1:
            assert a[0] == b[0] and np.float32(a[1]) == np.float32(b[1])
        elif a[0] == 2:
            assert a[:7] == b[:7]
            assert a[7] == a[2]      # planes start where the face array does
        else:
            assert a == b


def test_matches_reference_pipeline(tmp_path):
    # the reference pipeline's output for _case() is stored in tests/golden/assets_probe_ref.npz
    # (tests/golden/make_golden.py runs the probe)
    import madrona_b200 as mb
    hulls, objects = _case()
    inp, outp = str(tmp_path / "in.bin"), str(tmp_path / "out.bin")
    _write_probe_input(inp, hulls, objects)
    golden = np.load(GOLDEN)
    assert hashlib.sha256(open(inp, "rb").read()).hexdigest() == str(golden["input_sha256"]), \
        "the probe input differs from the one the golden output was made from"
    golden["output"].tofile(outp)
    ref = _read_probe_output(outp)
    assets = mb.RigidBodyAssets(hulls, objects, gpu_id=-1)
    _compare(assets.host_arrays(), ref)
    assets.close()


def test_known_answers():
    """Unit cube: inertia of unit mass 1/6 on every axis, centre of mass at the origin, Newell
    planes at distance 0.5; sphere: 2/5 r^2; plane and static objects: inverse inertia 0."""
    import madrona_b200 as mb
    hulls = [_box(1, 1, 1), _box(2, 1, 1, (3.0, 0.0, 0.0))]
    objects = [dict(prims=[("hull", 0)], inv_mass=1.0), dict(prims=[("sphere", 2.0)], inv_mass=1.0),
               dict(prims=[("plane",)], inv_mass=0.0), dict(prims=[("hull", 1)], inv_mass=0.5)]
    arrs = mb.RigidBodyAssets(hulls, objects).host_arrays()
    meta = arrs["metadatas"]
    np.testing.assert_allclose(meta[0, 1:4], 6.0, rtol=1e-5)
    np.testing.assert_allclose(meta[0, 4:7], 0.0, atol=1e-6)
    np.testing.assert_allclose(meta[1, 1:4], 1.0 / (0.4 * 4.0), rtol=1e-5)
    assert np.all(meta[2, 0:4] == 0.0)
    np.testing.assert_allclose(meta[3, 4:7], [3.0, 0.0, 0.0], atol=1e-5)
    inv_i = np.sort(meta[3, 1:4])
    np.testing.assert_allclose(inv_i, np.sort(0.5 / np.array([2 / 12, 5 / 12, 5 / 12])), rtol=1e-4)
    np.testing.assert_allclose(np.abs(arrs["planes"][:6, 3]), 0.5, rtol=1e-6)
    np.testing.assert_allclose(arrs["obj_aabbs"][0], [-0.5] * 3 + [0.5] * 3)
    assert arrs["half_edges"].shape == (48, 3)
    # twins are (2k, 2k+1): opposite directions of the same edge
    he = arrs["half_edges"][:24]
    for k in range(12):
        a, b = he[2 * k], he[2 * k + 1]
        assert he[a[0]][1] == b[1] and he[b[0]][1] == a[1]


def test_rejects_open_mesh():
    import madrona_b200 as mb
    v, faces = _box(1, 1, 1)
    with pytest.raises(mb.MadronaB200Error):
        mb.RigidBodyAssets([(v, faces[:5])], [dict(prims=[("hull", 0)], inv_mass=1.0)])


@pytest.mark.gpu
def test_pipeline_objects_drive_the_room_fixture():
    """sims/room stepped with the ObjectManager the pipeline built on the GPU: same trace, bit
    for bit, as with a hand-assembled blob carrying the same numbers (checks the upload and the
    pointer rebasing), and the pipeline's mass properties are the unit cube's."""
    import madrona_b200 as mb
    from sims.objects import box_half_edge_mesh, build_objects
    from trace_utils import make_inputs, rollout_gpu

    hulls = [_box(1, 1, 1)]
    objects = [dict(prims=[("hull", 0)], inv_mass=0.1, mu_s=0.5, mu_d=0.75),
               dict(prims=[("hull", 0)], inv_mass=0.0),
               dict(prims=[("hull", 0)], inv_mass=1.0 / 50.0),
               dict(prims=[("plane",)], inv_mass=0.0)]
    assets = mb.RigidBodyAssets(hulls, objects, gpu_id=0)
    arrs = assets.host_arrays()
    mesh = box_half_edge_mesh()
    assert np.array_equal(arrs["half_edges"], mesh["half_edges"])
    specs = [dict(mesh=(mesh if o < 3 else "plane"), meta=arrs["metadatas"][o].tobytes()) for o in range(4)]
    inputs = make_inputs("room", 4, 60)
    piped, _ = rollout_gpu("room", 4, 60, inputs, cfg=dict(objects_fn=lambda: assets))
    hand, _ = rollout_gpu("room", 4, 60, inputs,
                          cfg=dict(objects_fn=lambda: build_objects(specs, plane_extent=3.4028234663852886e38)))
    for key in hand:
        assert np.array_equal(np.asarray(hand[key]).view(np.uint8), np.asarray(piped[key]).view(np.uint8)), key
        assert np.isfinite(np.asarray(piped[key], dtype=np.float64)).all(), key
    assets.close()
