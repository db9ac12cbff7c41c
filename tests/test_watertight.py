"""The `--mc` watertight remesh: marching-cubes table (CPU), distance oracle (CPU), the training data's double-shell
convention (CPU, tests/golden/config1_mouse.npz), and the CUDA distance field / marching cubes / mesh_to_pc path (GPU).

Conventions: grid of size^3 nodes, h = 2/size, node (i, j, k) at -1 + (i, j, k) h; field min(d, 2h); marching cubes at
level h, inside = field < level, triangles oriented towards increasing field (csrc/watertight.cu).
"""
import os
import sys
from collections import Counter

import numpy as np
import pytest

from oracle import watertight as ow

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "tools"))
import make_mc_table as mct  # noqa: E402

gpu = pytest.mark.gpu
GOLDEN = os.path.join(ROOT, "tests", "golden")


# ------------------------------------------------------------------------------------------------ helpers

def icosphere(subdiv=3, radius=1.0):
    t = (1.0 + 5 ** 0.5) / 2
    v = [(-1, t, 0), (1, t, 0), (-1, -t, 0), (1, -t, 0), (0, -1, t), (0, 1, t), (0, -1, -t), (0, 1, -t),
         (t, 0, -1), (t, 0, 1), (-t, 0, -1), (-t, 0, 1)]
    f = [(0, 11, 5), (0, 5, 1), (0, 1, 7), (0, 7, 10), (0, 10, 11), (1, 5, 9), (5, 11, 4), (11, 10, 2), (10, 7, 6),
         (7, 1, 8), (3, 9, 4), (3, 4, 2), (3, 2, 6), (3, 6, 8), (3, 8, 9), (4, 9, 5), (2, 4, 11), (6, 2, 10), (8, 6, 7),
         (9, 8, 1)]
    v = [np.array(p, dtype=np.float64) / np.linalg.norm(p) for p in v]
    for _ in range(subdiv):
        mid, nf = {}, []

        def m(a, b):
            k = (min(a, b), max(a, b))
            if k not in mid:
                p = v[a] + v[b]
                v.append(p / np.linalg.norm(p))
                mid[k] = len(v) - 1
            return mid[k]
        for a, b, c in f:
            ab, bc, ca = m(a, b), m(b, c), m(c, a)
            nf += [(a, ab, ca), (b, bc, ab), (c, ca, bc), (ab, bc, ca)]
        f = nf
    return np.asarray(v) * radius, np.asarray(f, dtype=np.int64)


def disc(rings=4, seg=24, radius=0.7):
    v = [(0.0, 0.0, 0.0)]
    for r in range(1, rings + 1):
        for s in range(seg):
            a = 2 * np.pi * s / seg
            v.append((radius * r / rings * np.cos(a), radius * r / rings * np.sin(a), 0.0))
    f = []
    for s in range(seg):
        f.append((0, 1 + s, 1 + (s + 1) % seg))
    for r in range(1, rings):
        b0, b1 = 1 + (r - 1) * seg, 1 + r * seg
        for s in range(seg):
            s1 = (s + 1) % seg
            f += [(b0 + s, b1 + s, b1 + s1), (b0 + s, b1 + s1, b0 + s1)]
    return np.asarray(v), np.asarray(f, dtype=np.int64)


def soup(n=300, seed=0):
    rng = np.random.RandomState(seed)
    c = rng.uniform(-0.8, 0.8, (n, 1, 3))
    v = (c + rng.normal(0, 0.08, (n, 3, 3))).reshape(-1, 3)
    v = np.clip(v, -0.9, 0.9)
    f = np.arange(3 * n).reshape(n, 3)
    f[5] = [7, 7, 7]                      # repeated indices: a point
    f[6] = [9, 9, 10]                     # a segment
    v[3 * 8 + 2] = 0.5 * (v[3 * 8] + v[3 * 8 + 1])     # collinear: zero area
    return v, f


def example_mesh(name):
    d = np.load(os.path.join(GOLDEN, "example_meshes.npz"))
    return d[name + "_vertices"].astype(np.float64), d[name + "_faces"].astype(np.int64)


def unit(vertices):
    import mesh_to_pc
    return mesh_to_pc.normalize_vertices(np.asarray(vertices, dtype=np.float64))[0].astype(np.float32)


def rotation(seed):
    q, _ = np.linalg.qr(np.random.RandomState(seed).randn(3, 3))
    return q * np.sign(np.linalg.det(q))


def topology(faces):
    """(closed: every directed edge once and its reverse once, Euler characteristic, connected components)."""
    f = np.asarray(faces)
    e = np.concatenate([f[:, [0, 1]], f[:, [1, 2]], f[:, [2, 0]]])
    cnt = Counter(map(tuple, e.tolist()))
    closed = all(n == 1 and cnt.get((b, a), 0) == 1 for (a, b), n in cnt.items())
    used = np.unique(f)
    chi = len(used) - len(cnt) // 2 + len(f)
    parent = {int(u): int(u) for u in used}

    def find(x):
        while parent[x] != x:
            parent[x] = parent[parent[x]]
            x = parent[x]
        return x
    for a, b in e.tolist():
        ra, rb = find(a), find(b)
        if ra != rb:
            parent[ra] = rb
    return closed, chi, len({find(int(u)) for u in used})


def signed_volume(v, f):
    v = np.asarray(v, dtype=np.float64)
    return float(np.einsum("ij,ij->i", v[f[:, 0]], np.cross(v[f[:, 1]], v[f[:, 2]])).sum() / 6.0)


def mouse_signature():
    """Double-shell signature of the reference's own example cloud (the output of its --mc pipeline) and the gap that
    pipeline implies: 2 * level in the cloud's units, level = 2/128 on the grid of the +-0.9 normalisation."""
    raw = np.load(os.path.join(GOLDEN, "config1_mouse.npz"))["raw"].astype(np.float64)
    extent = (raw[:, :3].max(0) - raw[:, :3].min(0)).max()
    return ow.double_shell_signature(raw[:, :3], raw[:, 3:]), 2 * (2 / 128) * extent / 1.8


# ------------------------------------------------------------------------------------------------ CPU

TABLE = mct.load_table()


def test_table_is_generated_from_the_rule():
    assert TABLE == mct.build_table()
    assert TABLE[0] == [] and TABLE[255] == []


def test_table_is_watertight_by_construction():
    """All 256 cases: triangle vertices lie on crossing edges; the triangles of a case form closed, consistently wound
    loops whose boundary segments lie on the cube faces; the segments on a face depend on that face's 4 corner bits
    only, and the cell across the face sees the same segments reversed."""
    face_segs = {}
    for case in range(256):
        tris = TABLE[case]
        crossing = {e for e, (a, b) in enumerate(mct.EDGES) if ((case >> a) & 1) != ((case >> b) & 1)}
        assert {e for t in tris for e in t} == crossing, case
        directed = Counter((t[i], t[(i + 1) % 3]) for t in tris for i in range(3))
        assert all(n == 1 for n in directed.values()), case
        boundary = {d for d in directed if (d[1], d[0]) not in directed}
        for e0, e1 in boundary:
            assert mct.face_of_edges(e0, e1), (case, e0, e1)
        # every crossing edge starts exactly one boundary segment and ends exactly one: closed loops
        assert Counter(a for a, _ in boundary) == Counter(b for _, b in boundary) == Counter(crossing), case
        for fi, (_, ring) in enumerate(mct.FACES):
            bits = tuple((case >> c) & 1 for c in ring)
            segs = frozenset((a, b) for a, b in boundary if set(mct.EDGES[a]) | set(mct.EDGES[b]) <= set(ring))
            assert face_segs.setdefault((fi, bits), segs) == segs, (case, fi)
    # shared faces: face 2*axis+1 of a cell is face 2*axis of its neighbour along axis
    for axis in range(3):
        shift = {mct.edge_id(a | (1 << axis), b | (1 << axis)): mct.edge_id(a, b)
                 for a, b in mct.EDGES if not (a >> axis) & 1 and not (b >> axis) & 1}
        for (fi, bits), segs in face_segs.items():
            if fi != 2 * axis + 1:
                continue
            seen = face_segs[(2 * axis, bits)]
            assert {(shift[b], shift[a]) for a, b in segs} == set(seen), (axis, bits)


def test_table_orients_outwards_on_a_numpy_sphere():
    S = 32
    g = -1 + np.arange(S) * (2 / S)
    r = np.sqrt((g[:, None, None] ** 2) + (g[None, :, None] ** 2) + (g[None, None, :] ** 2)).astype(np.float32)
    v, f = ow.marching_cubes(r, 0.5, TABLE)
    closed, chi, comps = topology(f)
    assert closed and chi == 2 and comps == 1
    assert abs(signed_volume(v, f) - 4 / 3 * np.pi * 0.125) < 0.02


def test_oracle_point_triangle_distance_hand_cases():
    a, b, c = np.array([0.0, 0, 0]), np.array([1.0, 0, 0]), np.array([0.0, 1, 0])
    d = lambda p, *t: float(ow.point_triangle_distance(np.array(p, dtype=np.float64), *(t or (a, b, c))))  # noqa: E731
    assert d([0.25, 0.25, 0.3]) == pytest.approx(0.3, abs=1e-15)          # interior: plane distance
    assert d([0.25, 0.25, -0.3]) == pytest.approx(0.3, abs=1e-15)
    assert d([-1.0, -1.0, 0.0]) == pytest.approx(2 ** 0.5, abs=1e-15)      # vertex region
    assert d([2.0, 0.0, 1.0]) == pytest.approx(2 ** 0.5, abs=1e-15)
    assert d([0.5, -2.0, 0.0]) == pytest.approx(2.0, abs=1e-15)            # edge regions
    assert d([1.0, 1.0, 0.0]) == pytest.approx(0.5 ** 0.5, abs=1e-15)
    assert d([0.5, 0.5, 0.0]) == 0.0
    # degenerate triangles: a point, a segment, three collinear points
    assert d([1.0, 2.0, 2.0], a, a, a) == pytest.approx(3.0, abs=1e-15)
    assert d([0.5, 1.0, 0.0], a, b, b) == pytest.approx(1.0, abs=1e-15)
    assert d([3.0, 0.0, 4.0], a, b, 0.5 * b) == pytest.approx(np.hypot(2, 4), abs=1e-15)
    assert not np.isnan(ow.point_triangle_distance(np.zeros((4, 3)), a, a, a)).any()


def test_mouse_fixture_is_a_double_shell_at_twice_the_level():
    """The reference's example cloud pc_examples/mouse.npy is the output of the --mc pipeline: each point has an
    opposite-normal partner 2 * level behind it (in the cloud's units) and its normal points away from it."""
    (gap, away, pairs), expected = mouse_signature()
    assert pairs > 3500
    assert abs(gap - expected) < 0.03 * expected, (gap, expected)
    assert away >= 0.95, away


def test_watertight_rejects_bad_meshes_before_the_kernel():
    import mesh_to_pc
    v, f = icosphere(1)
    stub = (None, None)                # validation runs before anything touches the library or the device
    for bad_v, bad_f in ((v, f + 100), (v, f - 1), (np.where(np.arange(len(v))[:, None] == 3, np.nan, v), f)):
        with pytest.raises(ValueError):
            mesh_to_pc._watertight_gpu(stub, mesh_to_pc.SimpleMesh(bad_v, bad_f), 7)
    with pytest.raises(ValueError):
        mesh_to_pc._watertight_gpu(stub, mesh_to_pc.SimpleMesh(v, f), 9)


# ------------------------------------------------------------------------------------------------ GPU

def _dev():
    import torch
    return torch.device("cuda:0")


def _udf(v32, f, size):
    import torch
    from meshanything_b200 import capi
    field = capi.mesh_udf(torch.from_numpy(np.ascontiguousarray(v32)).to(_dev()),
                          torch.from_numpy(np.ascontiguousarray(f.astype(np.int32))).to(_dev()), size)
    return field.cpu().numpy()


def _udf_mesh(name):
    if name == "icosphere":
        v, f = icosphere(3, 0.85)
    elif name == "disc":
        v, f = disc()
        v = v @ rotation(3).T
    elif name == "soup":
        v, f = soup()
    else:
        v, f = example_mesh(name)
    return unit(v) if name == "wand" else v.astype(np.float32), f


def _check_nodes(v32, f, size, rng):
    S = size
    nodes = rng.randint(0, S, (20000, 3))
    h = 2 / S
    tri = v32.astype(np.float64)[f[rng.choice(len(f), min(len(f), 200), replace=False)]]
    near = []
    for t in tri:
        lo = np.maximum(np.floor((t.min(0) + 1 - 2 * h) / h).astype(int), 0)
        hi = np.minimum(np.ceil((t.max(0) + 1 + 2 * h) / h).astype(int), S - 1)
        g = np.stack(np.meshgrid(*[np.arange(lo[a], hi[a] + 1) for a in range(3)], indexing="ij"), -1).reshape(-1, 3)
        near.append(g)
    return np.unique(np.concatenate([nodes] + near), axis=0)


@gpu
@pytest.mark.parametrize("size", [64, 128])
@pytest.mark.parametrize("name", ["icosphere", "disc", "soup", "wand"])
def test_udf_matches_the_oracle_and_is_order_independent(name, size):
    v32, f = _udf_mesh(name)
    field = _udf(v32, f, size)
    assert field.shape == (size, size, size) and np.isfinite(field).all()
    assert field.max() <= np.float32(4 / size) and field.min() >= 0
    nodes = _check_nodes(v32, f, size, np.random.RandomState(size))
    want = ow.mesh_udf(v32, f, nodes, size)
    got = field[nodes[:, 0], nodes[:, 1], nodes[:, 2]]
    err = np.abs(got - want)
    assert err.max() <= 2e-6, (err.max(), nodes[np.argmax(err)])
    assert (want < 4 / size).sum() > 1000                    # the band was actually exercised
    assert np.array_equal(_udf(v32, f, size).view(np.uint32), field.view(np.uint32))
    perm = np.random.RandomState(1).permutation(len(f))
    assert np.array_equal(_udf(v32, f[perm], size).view(np.uint32), field.view(np.uint32))


def _analytic(kind, S):
    g = -1 + np.arange(S) * (2 / S)
    X, Y, Z = np.meshgrid(g, g, g, indexing="ij")
    if kind == "sphere":
        return np.sqrt(X ** 2 + Y ** 2 + Z ** 2).astype(np.float32), 0.55, 2
    return np.sqrt((np.sqrt(X ** 2 + Y ** 2) - 0.5) ** 2 + Z ** 2).astype(np.float32), 0.2, 0


def _gpu_mc(field, level, inv_scale=1.0, centre=(0.0, 0.0, 0.0)):
    import torch
    from meshanything_b200 import capi
    v, f = capi.marching_cubes(torch.from_numpy(field).to(_dev()), level, inv_scale, centre)
    return v.cpu().numpy().astype(np.float64), f.cpu().numpy().astype(np.int64)


@gpu
@pytest.mark.parametrize("kind", ["sphere", "torus"])
def test_marching_cubes_on_analytic_fields(kind):
    S = 64
    field, level, chi_want = _analytic(kind, S)
    v, f = _gpu_mc(field, level)
    closed, chi, comps = topology(f)
    assert closed and chi == chi_want and comps == 1
    assert len(np.unique(f)) == len(v)                       # every vertex is used: one per crossing edge
    # every vertex on a grid edge at t = (level - f0) / (f1 - f0)
    rv, rf = ow.marching_cubes(field, level, TABLE)
    assert np.abs(v - rv).max() < 1e-6 and np.array_equal(f, rf)
    h = 2 / S
    idx = (v + 1) / h
    off = np.abs(idx - np.round(idx))
    assert ((off < 1e-4).sum(1) >= 2).all()                  # two coordinates on the grid
    if kind == "sphere":
        assert signed_volume(v, f) > 0
        assert abs(signed_volume(v, f) - 4 / 3 * np.pi * level ** 3) < 0.01
    # the frame mapping of the emit pass
    v2, f2 = _gpu_mc(field, level, 2.0, (1.0, -2.0, 0.5))
    assert np.array_equal(f2, f) and np.abs(v2 - (v * 2.0 + np.array([1.0, -2.0, 0.5]))).max() < 1e-5


@gpu
def test_marching_cubes_equals_the_numpy_restatement_at_32():
    rng = np.random.RandomState(0)
    field = rng.rand(32, 32, 32).astype(np.float32)          # every ambiguous configuration occurs
    v, f = _gpu_mc(field, 0.5)
    rv, rf = ow.marching_cubes(field, 0.5, TABLE)
    assert np.array_equal(f, rf) and np.abs(v - rv).max() < 1e-6
    for kind in ("sphere", "torus"):
        fld, level, _ = _analytic(kind, 32)
        v, f = _gpu_mc(fld, level)
        rv, rf = ow.marching_cubes(fld, level, TABLE)
        assert np.array_equal(f, rf) and np.abs(v - rv).max() < 1e-6


# Linear interpolation along a grid edge of length h puts a vertex where the interpolated distance is h.  Where the
# nearest feature is a plane the distance is linear and the vertex is exact; near an edge or a point of the surface the
# distance is convex, the vertex lies closer, by at most (1 - sqrt(3)/2) h (a point at distance h/2 from the edge's
# line, the edge ending on the h sphere); where the distances to two sheets meet (concave creases, sheets about 2 level
# apart) it lies farther.
CONVEX_DIP = 1 - 3 ** 0.5 / 2


def _level_error(mesh_v, mesh_f, out_v, depth):
    """(exact distance from the remeshed vertices to the input mesh - level) / h, in the grid's units."""
    import mesh_to_pc
    _, _, factor = mesh_to_pc.normalize_vertices(np.asarray(mesh_v, dtype=np.float64))
    h = 2 / 2 ** depth
    d = ow.distance_to_mesh(out_v, mesh_v, mesh_f, 3 * h / factor) * factor
    return (d - h) / h


@gpu
@pytest.mark.parametrize("depth", [6, 7])
def test_export_to_watertight_end_to_end(depth):
    import mesh_to_pc
    v, f = icosphere(3)
    out = mesh_to_pc.export_to_watertight(mesh_to_pc.SimpleMesh(v * 3.0 + 1.0, f), depth)
    assert isinstance(out, mesh_to_pc.SimpleMesh)
    closed, chi, comps = topology(out.faces)
    assert closed and chi == 4 and comps == 2                # two closed shells
    assert np.abs(_level_error(v * 3.0 + 1.0, f, out.vertices, depth)).max() < 0.1
    dv, df = disc()
    for seed in range(3):
        rv = dv @ rotation(seed).T * 2.0
        out = mesh_to_pc.export_to_watertight(mesh_to_pc.SimpleMesh(rv, df), depth)
        closed, chi, comps = topology(out.faces)
        assert closed and chi == 2 and comps == 1, (seed, chi, comps)
        err = _level_error(rv, df, out.vertices, depth)      # a flat disc: planar and convex (rim) distances only
        assert err.max() < 1e-3 and err.min() > -CONVEX_DIP - 1e-3, (err.min(), err.max())
        assert np.median(np.abs(err)) < 0.01
    wv, wf = example_mesh("wand")
    out = mesh_to_pc.export_to_watertight(mesh_to_pc.SimpleMesh(wv, wf), depth)
    closed, _, _ = topology(out.faces)
    assert closed and len(out.faces) > 1000
    err = _level_error(wv, wf, out.vertices, depth)
    print("wand depth %d: %d vertices, (d - level) / h min %.4f max %.4f median |.| %.4f" % (
        depth, len(err), err.min(), err.max(), np.median(np.abs(err))))
    assert err.min() > -CONVEX_DIP - 1e-3 and np.median(np.abs(err)) < 0.02 and err.max() < 1.0


@gpu
def test_process_mesh_to_pc_with_marching_cubes():
    """The CUDA --mc path end to end, and the training data's convention on a closed sphere: the cloud is a double
    shell 2 * level apart with normals pointing away from the other shell, as in the reference's mouse example.  (The
    wand is thinner than 2 * level along most of its length: its shells merge there, so it has no such signature.)"""
    import mesh_to_pc
    wv, wf = example_mesh("wand")
    sv, sf = icosphere(4)
    for name, v, f in (("wand", wv, wf), ("sphere", sv, sf)):
        mesh = mesh_to_pc.SimpleMesh(v, f)
        np.random.seed(7)
        clouds, used = mesh_to_pc.process_mesh_to_pc([mesh], marching_cubes=True)
        pc = clouds[0]
        assert pc.shape == (4096, 6) and pc.dtype == np.float16
        assert np.abs(np.linalg.norm(pc[:, 3:].astype(np.float32), axis=1) - 1).max() < 2e-3
        assert isinstance(used[0], mesh_to_pc.SimpleMesh) and used[0] is not mesh
        assert topology(used[0].faces)[0]
        np.random.seed(7)
        again, _ = mesh_to_pc.process_mesh_to_pc([mesh], marching_cubes=True)
        assert np.array_equal(again[0], pc)
        _, _, factor = mesh_to_pc.normalize_vertices(np.asarray(v, dtype=np.float64))
        expected = 2 * (2 / 128) / factor
        gap, away, pairs = ow.double_shell_signature(pc[:, :3].astype(np.float64), pc[:, 3:].astype(np.float64))
        print("%s double shell: gap %.5f expected %.5f away %.3f pairs %d" % (name, gap, expected, away, pairs))
        if name == "sphere":
            assert pairs > 3500 and abs(gap - expected) < 0.05 * expected and away >= 0.95


@gpu
def test_main_cli_mc_writes_obj(tmp_path):
    """`python main.py --input_type mesh --input_path x.obj --mc ...` (the reference's third way to run) writes
    x_gen.obj."""
    import subprocess
    wv, wf = example_mesh("wand")
    obj = tmp_path / "wand.obj"
    with open(obj, "w") as fh:
        fh.writelines("v %.6f %.6f %.6f\n" % tuple(p) for p in wv)
        fh.writelines("f %d %d %d\n" % tuple(t + 1) for t in wf)
    out_dir = tmp_path / "out"
    r = subprocess.run([sys.executable, os.path.join(ROOT, "main.py"), "--input_type", "mesh", "--input_path", str(obj),
                        "--mc", "--out_dir", str(out_dir), "--pretrained_weights", "synthetic", "--n_max_triangles", "6",
                        "--seed", "0"], cwd=ROOT, capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr[-2000:]
    assert "MC over!" in r.stdout
    objs = [os.path.join(dp, f) for dp, _, fs in os.walk(out_dir) for f in fs if f.endswith("_gen.obj")]
    assert [os.path.basename(o) for o in objs] == ["wand_gen.obj"]


@gpu
def test_bad_arguments_return_errors():
    import ctypes as C
    import torch
    from meshanything_b200 import capi
    L = capi.lib()
    field = torch.zeros((32, 32, 32), dtype=torch.float32, device=_dev())
    ws = torch.empty(L.ma_marching_cubes_workspace_bytes(32), dtype=torch.uint8, device=_dev())
    cnt = torch.empty(2, dtype=torch.int32, device=_dev())
    v = torch.zeros((3, 3), dtype=torch.float32, device=_dev())
    f = torch.zeros((1, 3), dtype=torch.int32, device=_dev())
    s = capi.stream_ptr()
    assert L.ma_mesh_udf(capi.ptr(v), capi.ptr(f), 0, 32, capi.ptr(field), s) == 1
    assert b"ma_mesh_udf" in L.ma_last_error()
    assert L.ma_mesh_udf(capi.ptr(v), capi.ptr(f), 1, 16, capi.ptr(field), s) == 1
    assert L.ma_mesh_udf(None, capi.ptr(f), 1, 32, capi.ptr(field), s) == 1
    assert L.ma_marching_cubes_workspace_bytes(512) == 0
    assert L.ma_marching_cubes_count(capi.ptr(field), 300, C.c_float(0.1), capi.ptr(cnt), capi.ptr(ws), s) == 1
    assert L.ma_marching_cubes_count(capi.ptr(field), 32, C.c_float(0.1), None, capi.ptr(ws), s) == 1
    assert L.ma_marching_cubes_emit(capi.ptr(field), 32, C.c_float(0.1), C.c_float(1), C.c_float(0), C.c_float(0),
                                    C.c_float(0), None, None, capi.ptr(ws), s) == 1
    assert L.ma_mesh_udf(capi.ptr(v), capi.ptr(f), 1, 32, capi.ptr(field), s) == 0
    torch.cuda.synchronize()
