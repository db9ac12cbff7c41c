"""Device time of the `--mc` watertight remesh stages (csrc/watertight.cu) and of the surface sampler that follows them.

Stages per mesh: udf (ma_mesh_udf), count (ma_marching_cubes_count), emit (ma_marching_cubes_emit), sample
(ma_sample_surface, 4096 points), each timed with CUDA events over --reps launches after --warmup; `total` is their sum,
`e2e_ms` the host clock around mesh_to_pc's whole GPU path (upload, two-count readback, remesh) ending in a synchronise.
Cases: the reference's wand and screwdriver (tests/golden/example_meshes.npz) at depth 7, a 327 680-face icosphere, and
2000 large random triangles (a bounding-box splat would touch most of the grid for each).  The device name and power
limit are read in the same run.

usage: python tools/bench_watertight.py [--depth 7] [--reps 20] [--warmup 3] [--out FILE]
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import mesh_to_pc  # noqa: E402
from meshanything_b200 import capi  # noqa: E402


def icosphere(subdiv):
    t = (1.0 + 5 ** 0.5) / 2
    v = np.array([(-1, t, 0), (1, t, 0), (-1, -t, 0), (1, -t, 0), (0, -1, t), (0, 1, t), (0, -1, -t), (0, 1, -t),
                  (t, 0, -1), (t, 0, 1), (-t, 0, -1), (-t, 0, 1)], dtype=np.float64)
    f = np.array([(0, 11, 5), (0, 5, 1), (0, 1, 7), (0, 7, 10), (0, 10, 11), (1, 5, 9), (5, 11, 4), (11, 10, 2),
                  (10, 7, 6), (7, 1, 8), (3, 9, 4), (3, 4, 2), (3, 2, 6), (3, 6, 8), (3, 8, 9), (4, 9, 5), (2, 4, 11),
                  (6, 2, 10), (8, 6, 7), (9, 8, 1)], dtype=np.int64)
    for _ in range(subdiv):
        e = np.sort(np.concatenate([f[:, [0, 1]], f[:, [1, 2]], f[:, [2, 0]]]), axis=1)
        uniq, inv = np.unique(e, axis=0, return_inverse=True)
        mid = len(v) + inv.reshape(3, -1)              # midpoint index of edges ab, bc, ca of every face
        v = np.concatenate([v, 0.5 * (v[uniq[:, 0]] + v[uniq[:, 1]])])
        ab, bc, ca = mid
        f = np.concatenate([np.stack([f[:, 0], ab, ca], 1), np.stack([f[:, 1], bc, ab], 1),
                            np.stack([f[:, 2], ca, bc], 1), np.stack([ab, bc, ca], 1)])
    return v / np.linalg.norm(v, axis=1, keepdims=True), f


def cases():
    d = np.load(os.path.join(ROOT, "tests", "golden", "example_meshes.npz"))
    out = [(n, d[n + "_vertices"].astype(np.float64), d[n + "_faces"].astype(np.int64)) for n in ("wand", "screwdriver")]
    v, f = icosphere(7)
    out.append(("icosphere_%d" % len(f), v, f))
    rng = np.random.RandomState(0)
    out.append(("random_large_2000", rng.uniform(-1, 1, (6000, 3)), np.arange(6000).reshape(2000, 3)))
    return out


def device_info():
    info = {"device": torch.cuda.get_device_name(0)}
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
        info["power_limit_and_max_sm_clock"] = q
    except Exception as e:  # noqa: BLE001
        info["power_limit_and_max_sm_clock"] = f"unavailable ({e})"
    return info


def timed(fn, reps, warmup):
    for _ in range(warmup):
        fn()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    a.record()
    for _ in range(reps):
        fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / reps


def bench_case(name, v, f, depth, reps, warmup):
    L, dev = capi.lib(), torch.device("cuda:0")
    size, level = 2 ** depth, 2.0 / 2 ** depth
    unit, centre, factor = mesh_to_pc.normalize_vertices(v)
    vt = torch.as_tensor(unit.astype(np.float32), device=dev)
    ft = torch.as_tensor(f.astype(np.int32), device=dev)
    field = torch.empty((size, size, size), dtype=torch.float32, device=dev)
    ws = torch.empty(L.ma_marching_cubes_workspace_bytes(size), dtype=torch.uint8, device=dev)
    counts = torch.empty(2, dtype=torch.int32, device=dev)
    s = capi.stream_ptr()
    udf = lambda: capi.check(L.ma_mesh_udf(capi.ptr(vt), capi.ptr(ft), len(f), size, capi.ptr(field), s), "udf")  # noqa
    count = lambda: capi.check(L.ma_marching_cubes_count(capi.ptr(field), size, C.c_float(level), capi.ptr(counts),  # noqa
                                                         capi.ptr(ws), s), "count")
    t_udf = timed(udf, reps, warmup)
    t_count = timed(count, reps, warmup)
    nv, nf = counts.tolist()
    ov = torch.empty((nv, 3), dtype=torch.float32, device=dev)
    of = torch.empty((nf, 3), dtype=torch.int32, device=dev)
    cx, cy, cz = (float(c) for c in centre)
    emit = lambda: capi.check(L.ma_marching_cubes_emit(  # noqa: E731
        capi.ptr(field), size, C.c_float(level), C.c_float(1 / factor), C.c_float(cx), C.c_float(cy), C.c_float(cz),
        capi.ptr(ov), capi.ptr(of), capi.ptr(ws), s), "emit")
    t_emit = timed(emit, reps, warmup)
    t_sample = timed(lambda: capi.sample_surface(ov, of, 4096, seed=1), reps, warmup)
    mesh = mesh_to_pc.SimpleMesh(v, f)
    gpu = mesh_to_pc._gpu_sampler()
    for _ in range(warmup):
        mesh_to_pc._watertight_gpu(gpu, mesh, depth)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for _ in range(reps):
        rv, rf = mesh_to_pc._watertight_gpu(gpu, mesh, depth)
        capi.sample_surface(rv, rf, 4096, seed=1)
    torch.cuda.synchronize()
    e2e = (time.perf_counter() - t0) * 1e3 / reps
    return {"case": name, "faces_in": int(len(f)), "depth": depth, "vertices_out": nv, "faces_out": nf,
            "udf_ms": round(t_udf, 4), "count_ms": round(t_count, 4), "emit_ms": round(t_emit, 4),
            "sample_ms": round(t_sample, 4), "total_ms": round(t_udf + t_count + t_emit + t_sample, 4),
            "e2e_ms": round(e2e, 3)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--depth", type=int, default=7)
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("bench_watertight needs a CUDA device")
    res = {"info": device_info(), "results": []}
    print(json.dumps(res["info"]))
    for name, v, f in cases():
        r = bench_case(name, v, f, a.depth, a.reps, a.warmup)
        res["results"].append(r)
        print(json.dumps(r), flush=True)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as fh:
            json.dump(res, fh, indent=1)


if __name__ == "__main__":
    main()
