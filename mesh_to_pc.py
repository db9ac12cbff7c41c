"""Drop-in for /root/reference/mesh_to_pc.py: mesh -> (4096, 6) fp16 point cloud with normals.

With a CUDA device the whole path runs in CUDA: `marching_cubes=True` (`--mc`) rebuilds the mesh as a watertight double shell
(distance field + marching cubes, csrc/watertight.cu) and the points are drawn by the CUDA surface sampler.  Without a
GPU, or with MA_PC_SAMPLER=host, it uses trimesh / mesh2sdf / skimage when they are installed (same calls as the
reference); otherwise a small numpy implementation of area-weighted surface sampling (what `trimesh.Trimesh.sample`
does) is used (OBJ and ASCII/binary PLY readers included) and `marching_cubes=True` raises (mesh2sdf is required for the
host watertight conversion).
"""
import numpy as np

try:  # optional host-side dependencies of the reference
    import trimesh
except Exception:  # pragma: no cover
    trimesh = None


class SimpleMesh:
    """Minimal triangle mesh (vertices [V,3], faces [F,3]) with the two members the pipeline needs."""

    def __init__(self, vertices, faces):
        self.vertices = np.asarray(vertices, dtype=np.float64)
        self.faces = np.asarray(faces, dtype=np.int64)

    @property
    def face_normals(self):
        t = self.vertices[self.faces]
        n = np.cross(t[:, 1] - t[:, 0], t[:, 2] - t[:, 0])
        ln = np.linalg.norm(n, axis=1, keepdims=True)
        return n / np.where(ln > 0, ln, 1.0)

    def sample(self, count, return_index=False):
        t = self.vertices[self.faces]
        area = 0.5 * np.linalg.norm(np.cross(t[:, 1] - t[:, 0], t[:, 2] - t[:, 0]), axis=1)
        idx = np.searchsorted(np.cumsum(area), np.random.random(count) * area.sum())
        idx = np.minimum(idx, len(area) - 1)
        r = np.random.random((count, 2))
        flip = r.sum(axis=1) > 1.0
        r[flip] = 1.0 - r[flip]
        tri = t[idx]
        pts = tri[:, 0] + r[:, :1] * (tri[:, 1] - tri[:, 0]) + r[:, 1:] * (tri[:, 2] - tri[:, 0])
        return (pts, idx) if return_index else pts

    @staticmethod
    def load_obj(path):
        vs, fs = [], []
        with open(path) as f:
            for line in f:
                p = line.split()
                if not p:
                    continue
                if p[0] == "v":
                    vs.append([float(x) for x in p[1:4]])
                elif p[0] == "f":
                    ids = [int(x.split("/")[0]) for x in p[1:]]
                    ids = [i - 1 if i > 0 else len(vs) + i for i in ids]
                    for k in range(1, len(ids) - 1):          # fan triangulation
                        fs.append([ids[0], ids[k], ids[k + 1]])
        return SimpleMesh(vs, fs)


    _PLY_TYPES = {"char": "i1", "int8": "i1", "uchar": "u1", "uint8": "u1", "short": "i2", "int16": "i2",
                  "ushort": "u2", "uint16": "u2", "int": "i4", "int32": "i4", "uint": "u4", "uint32": "u4",
                  "float": "f4", "float32": "f4", "double": "f8", "float64": "f8"}

    @staticmethod
    def load_ply(path):
        """ASCII and binary (little/big endian) PLY: `vertex` (x, y, z among any other scalar properties) and `face`
        (one list property of vertex indices, polygons fan-triangulated).  Other elements are skipped."""
        T = SimpleMesh._PLY_TYPES
        with open(path, "rb") as f:
            if f.readline().strip() != b"ply":
                raise ValueError(f"{path}: not a PLY file")
            fmt, elements = None, []
            while True:
                line = f.readline()
                if not line:
                    raise ValueError(f"{path}: truncated PLY header")
                p = line.decode("ascii", "replace").split()
                if not p or p[0] in ("comment", "obj_info"):
                    continue
                if p[0] == "format":
                    fmt = p[1]
                elif p[0] == "element":
                    elements.append({"name": p[1], "count": int(p[2]), "props": []})
                elif p[0] == "property":
                    if p[1] == "list":
                        elements[-1]["props"].append(("list", p[4], T[p[2]], T[p[3]]))
                    else:
                        elements[-1]["props"].append(("scalar", p[2], T[p[1]]))
                elif p[0] == "end_header":
                    break
            if fmt not in ("ascii", "binary_little_endian", "binary_big_endian"):
                raise ValueError(f"{path}: unsupported PLY format {fmt!r}")
            end = ">" if fmt == "binary_big_endian" else "<"
            verts, faces = None, []
            for el in elements:
                n, props = el["count"], el["props"]
                has_list = any(pr[0] == "list" for pr in props)
                if fmt == "ascii":
                    rows = [f.readline().split() for _ in range(n)]
                    if el["name"] == "vertex":
                        names = [pr[1] for pr in props]
                        ix = [names.index(c) for c in "xyz"]
                        verts = np.array([[float(r[i]) for i in ix] for r in rows], dtype=np.float64).reshape(-1, 3)
                    elif el["name"] == "face":
                        for r in rows:   # list property first (the usual layout); scalar face properties follow it
                            k = int(r[0])
                            ids = [int(x) for x in r[1:1 + k]]
                            faces.extend([ids[0], ids[j], ids[j + 1]] for j in range(1, k - 1))
                    continue
                if not has_list:
                    dt = np.dtype([(pr[1], end + pr[2]) for pr in props])
                    block = np.frombuffer(f.read(dt.itemsize * n), dtype=dt, count=n)
                    if el["name"] == "vertex":
                        verts = np.stack([block[c].astype(np.float64) for c in "xyz"], axis=1)
                    continue
                for _ in range(n):       # element with a list property: variable-length records
                    for pr in props:
                        if pr[0] == "scalar":
                            f.read(np.dtype(pr[2]).itemsize)
                            continue
                        k = int(np.frombuffer(f.read(np.dtype(pr[2]).itemsize), dtype=end + pr[2])[0])
                        ids = np.frombuffer(f.read(np.dtype(pr[3]).itemsize * k), dtype=end + pr[3]).astype(np.int64)
                        if el["name"] == "face":
                            faces.extend([ids[0], ids[j], ids[j + 1]] for j in range(1, k - 1))
        if verts is None or not faces:
            raise ValueError(f"{path}: PLY without vertex/face elements (point clouds go through --input_type pc_normal)")
        return SimpleMesh(verts, np.asarray(faces, dtype=np.int64))


def load_mesh(path):
    if trimesh is not None:
        return trimesh.load(path)
    low = path.lower()
    if low.endswith(".obj"):
        return SimpleMesh.load_obj(path)
    if low.endswith(".ply"):
        return SimpleMesh.load_ply(path)
    raise ImportError(f"{path}: trimesh is needed to load meshes other than .obj / .ply")


def normalize_vertices(vertices, scale=0.9):
    """Centre on the bounding box and scale its longest side to 2*scale; returns (vertices, centre, factor)."""
    lo, hi = vertices.min(0), vertices.max(0)
    centre = 0.5 * (lo + hi)
    factor = 2.0 * scale / (hi - lo).max()
    return (vertices - centre) * factor, centre, factor


def _watertight_gpu(gpu, mesh, octree_depth):
    """(vertices fp32 [V, 3], faces int32 [F, 3]) of the watertight remesh, on the device: the mesh normalised to +-0.9
    on the host in float64, min(distance, 2h) on the 2^depth grid (ma_mesh_udf), marching cubes at level h = 2/size
    mapped back to the input frame (ma_marching_cubes_*)."""
    capi, torch = gpu
    if not 5 <= octree_depth <= 8:
        raise ValueError(f"octree_depth must be in 5..8, got {octree_depth}")
    vertices = np.asarray(mesh.vertices, dtype=np.float64)
    faces = np.asarray(mesh.faces, dtype=np.int64)
    if vertices.ndim != 2 or vertices.shape[1] != 3 or faces.ndim != 2 or faces.shape[1] != 3 or len(faces) == 0:
        raise ValueError(f"watertight remesh needs vertices [V, 3] and at least one face [F, 3], got "
                         f"{vertices.shape} / {faces.shape}")
    if not np.isfinite(vertices).all():
        raise ValueError("watertight remesh: the mesh has non-finite vertices")
    if faces.min() < 0 or faces.max() >= len(vertices):
        raise ValueError(f"watertight remesh: face indices outside [0, {len(vertices)})")
    size = 2 ** octree_depth
    unit_vertices, centre, factor = normalize_vertices(vertices)
    dev = torch.device("cuda", torch.cuda.current_device())
    v = torch.as_tensor(unit_vertices.astype(np.float32), device=dev)
    f = torch.as_tensor(faces.astype(np.int32), device=dev)
    field = capi.mesh_udf(v, f, size)
    return capi.marching_cubes(field, 2 / size, inv_scale=1.0 / factor, centre=centre)


def export_to_watertight(normalized_mesh, octree_depth: int = 7):
    """Watertight remesh used by `--mc` (reference mesh_to_pc.py:13-40): unsigned distance field on a 2^depth grid,
    marching cubes at iso level 2/size, mapped back to the input frame.  With a CUDA device it runs in CUDA and returns a
    SimpleMesh; otherwise it needs mesh2sdf / skimage / trimesh, as the reference does."""
    gpu = _gpu_sampler()
    if gpu is not None:
        v, f = _watertight_gpu(gpu, normalized_mesh, octree_depth)
        return SimpleMesh(v.cpu().numpy(), f.cpu().numpy())
    try:
        import mesh2sdf.core
        import skimage.measure
    except Exception as e:  # pragma: no cover
        raise ImportError("--mc needs mesh2sdf, scikit-image and trimesh") from e
    size = 2 ** octree_depth
    unit_vertices, centre, factor = normalize_vertices(normalized_mesh.vertices)
    field = np.abs(mesh2sdf.core.compute(unit_vertices, normalized_mesh.faces, size=size))
    verts, faces, normals, _ = skimage.measure.marching_cubes(field, 2 / size)
    verts = (verts / size * 2 - 1) / factor + centre
    return trimesh.Trimesh(verts, faces, normals=normals)


def _gpu_sampler():
    """The CUDA surface sampler (ma_sample_surface) when a GPU and the library are there; MA_PC_SAMPLER=host keeps the
    trimesh / numpy sampler (same distribution, numpy's random stream: what the reference draws)."""
    import os
    if os.environ.get("MA_PC_SAMPLER", "gpu") != "gpu":
        return None
    try:
        import torch
        if not torch.cuda.is_available():
            return None
        from meshanything_b200 import capi
        capi.lib()
        return capi, torch
    except Exception:
        return None


def process_mesh_to_pc(mesh_list, marching_cubes=False, sample_num=4096):
    """[mesh] -> ([fp16 (sample_num, 6) points + face normals], [mesh actually sampled]).  On a GPU box the points are
    drawn by the CUDA sampler (seeded from numpy's generator, so `set_seed` still decides them), and with
    `marching_cubes=True` the watertight remesh (a SimpleMesh in `used`) is built in CUDA too."""
    clouds, used = [], []
    gpu = _gpu_sampler()
    for mesh in mesh_list:
        if marching_cubes and gpu is not None:        # the rebuilt mesh stays on the device for the sampler
            v, f = _watertight_gpu(gpu, mesh, 7)
            mesh = SimpleMesh(v.cpu().numpy(), f.cpu().numpy())
            print("MC over!")
        elif marching_cubes:
            mesh = export_to_watertight(mesh)
            print("MC over!")
        if gpu is not None:
            capi, torch = gpu
            dev = torch.device("cuda", torch.cuda.current_device())
            if not marching_cubes:
                v = torch.as_tensor(np.asarray(mesh.vertices, dtype=np.float32), device=dev)
                f = torch.as_tensor(np.asarray(mesh.faces, dtype=np.int32), device=dev)
            seed = int(np.random.randint(0, 2 ** 31 - 1))
            clouds.append(capi.sample_surface(v, f, sample_num, seed=seed).cpu().numpy())
            used.append(mesh)
            print("process mesh success")
            continue
        pts, tri = mesh.sample(sample_num, return_index=True)
        clouds.append(np.concatenate([pts, mesh.face_normals[tri]], axis=-1, dtype=np.float16))
        used.append(mesh)
        print("process mesh success")
    return clouds, used
