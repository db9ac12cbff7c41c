"""float64 numpy statements of the watertight remesh (meshanything_b200/csrc/watertight.cu), for the tests.

  point_triangle_distance   exact Euclidean distance from points to triangles (zero-area triangles: their edges/points)
  mesh_udf                  min(d, 2h) at chosen grid nodes, d the distance to the nearest triangle of a mesh
  marching_cubes            the same table, vertex order and triangle order as the kernels, in numpy
  double_shell_signature    what a cloud sampled from a double shell looks like: the gap to the opposite shell along
                            the normal, and how often the normal points away from it
"""
import numpy as np


def _seg_d2(p, a, b):
    ab, ap = b - a, p - a
    l2 = (ab * ab).sum(-1)
    t = np.where(l2 > 0, (ap * ab).sum(-1) / np.where(l2 > 0, l2, 1.0), 0.0)
    t = np.clip(t, 0.0, 1.0)
    d = ap - t[..., None] * ab
    return (d * d).sum(-1)


def point_triangle_distance(p, a, b, c):
    """Distance from points p [..., 3] to triangles (a, b, c) [..., 3] (broadcast), in float64."""
    p, a, b, c = (np.asarray(x, dtype=np.float64) for x in (p, a, b, c))
    n = np.cross(b - a, c - a)
    nn = (n * n).sum(-1)
    s0 = (np.cross(b - a, p - a) * n).sum(-1)
    s1 = (np.cross(c - b, p - b) * n).sum(-1)
    s2 = (np.cross(a - c, p - c) * n).sum(-1)
    inside = (nn > 0) & (s0 >= 0) & (s1 >= 0) & (s2 >= 0)
    plane = np.abs(((p - a) * n).sum(-1)) / np.sqrt(np.where(nn > 0, nn, 1.0))
    edges = np.sqrt(np.minimum(_seg_d2(p, a, b), np.minimum(_seg_d2(p, b, c), _seg_d2(p, c, a))))
    return np.where(inside, plane, edges)


def node_positions(nodes, size):
    """Grid nodes (i, j, k) [n, 3] -> positions (-1 + i h, ...), h = 2 / size."""
    return -1.0 + np.asarray(nodes, dtype=np.float64) * (2.0 / size)


def distance_to_mesh(points, vertices, faces, reach, chunk=128):
    """Exact distance from points [n, 3] to the nearest triangle wherever it is below `reach` (inf or a value >= reach
    elsewhere): each chunk of nearby points is measured against the triangles whose bounding box comes within reach."""
    tri = np.asarray(vertices, dtype=np.float64)[np.asarray(faces)]
    lo, hi = tri.min(1) - reach, tri.max(1) + reach
    p = np.asarray(points, dtype=np.float64)
    cell = np.floor((p - p.min(0)) / (4.0 * reach)).astype(np.int64)
    order = np.lexsort((cell[:, 2], cell[:, 1], cell[:, 0]))
    out = np.full(len(p), np.inf)
    for s in range(0, len(p), chunk):
        idx = order[s:s + chunk]
        q = p[idx]
        cand = np.nonzero(((hi >= q.min(0)) & (lo <= q.max(0))).all(1))[0]
        if len(cand):
            t = tri[cand]
            out[idx] = point_triangle_distance(q[:, None], t[None, :, 0], t[None, :, 1], t[None, :, 2]).min(1)
    return out


def mesh_udf(vertices, faces, nodes, size):
    """min(d, 2h) at the given grid nodes [n, 3] for the mesh (vertices [V, 3], faces [F, 3])."""
    band = 2.0 * (2.0 / size)
    return np.minimum(distance_to_mesh(node_positions(nodes, size), vertices, faces, band), band)


# cube edge e = 4 * axis + o, o = offsets of the two other axes (lower axis in bit 0); see tools/make_mc_table.py
def _edge_offset(e):
    axis, o = divmod(e, 4)
    others = [x for x in range(3) if x != axis]
    d = [0, 0, 0]
    d[others[0]], d[others[1]] = o & 1, (o >> 1) & 1
    return axis, d


def marching_cubes(field, level, table):
    """(vertices [V, 3] float64 in the grid's [-1, 1) frame, faces [F, 3]) with the kernels' table and orders."""
    f = np.asarray(field, dtype=np.float64)
    S = f.shape[0]
    h = 2.0 / S
    ins = f < np.float32(level)
    cross = np.zeros((S, S, S, 3), dtype=bool)
    cross[:-1, :, :, 0] = ins[:-1] != ins[1:]
    cross[:, :-1, :, 1] = ins[:, :-1] != ins[:, 1:]
    cross[:, :, :-1, 2] = ins[:, :, :-1] != ins[:, :, 1:]
    node, axis = np.nonzero(cross.reshape(-1, 3))              # node-major, then axis: the kernel's vertex order
    ijk = np.stack(np.unravel_index(node, (S, S, S)), axis=1).astype(np.float64)
    step = np.eye(3, dtype=np.int64)[axis]
    i0 = tuple(np.stack(np.unravel_index(node, (S, S, S)), axis=1).T)
    i1 = tuple((np.stack(np.unravel_index(node, (S, S, S)), axis=1) + step).T)
    f0, f1 = f[i0].astype(np.float32), f[i1].astype(np.float32)
    t = ((np.float32(level) - f0) / (f1 - f0)).astype(np.float64)
    pos = ijk.copy()
    pos[np.arange(len(pos)), axis] += t
    verts = pos * h - 1.0
    vid = -np.ones((S, S, S, 3), dtype=np.int64)
    vid.reshape(-1, 3)[node, axis] = np.arange(len(node))
    case = np.zeros((S - 1, S - 1, S - 1), dtype=np.int64)
    for c in range(8):
        dx, dy, dz = c & 1, (c >> 1) & 1, (c >> 2) & 1
        case |= ins[dx:S - 1 + dx, dy:S - 1 + dy, dz:S - 1 + dz].astype(np.int64) << c
    faces = []
    for cell in np.argwhere(case > 0):                          # C order = the kernel's cell order
        for tri in table[case[tuple(cell)]]:
            ids = []
            for e in tri:
                ax, d = _edge_offset(e)
                ids.append(vid[cell[0] + d[0], cell[1] + d[1], cell[2] + d[2], ax])
            faces.append(ids)
    return verts, np.asarray(faces, dtype=np.int64).reshape(-1, 3)


def double_shell_signature(points, normals, k=32, opposite=-0.8):
    """For every point, the nearest point whose normal is opposite (dot < `opposite`) among its k nearest: returns
    (median gap along the point's normal to it, share of pairs whose normal points away from it, pairs found)."""
    from scipy.spatial import cKDTree
    p = np.asarray(points, dtype=np.float64)
    n = np.asarray(normals, dtype=np.float64)
    n = n / np.linalg.norm(n, axis=1, keepdims=True)
    _, nb = cKDTree(p).query(p, k=k)
    dots = np.einsum("pc,pkc->pk", n, n[nb])
    ok = dots < opposite
    has = ok.any(1)
    first = nb[np.arange(len(p)), np.argmax(ok, axis=1)][has]
    gap = ((p[has] - p[first]) * n[has]).sum(1)                # > 0: the other shell lies behind the normal
    return float(np.median(np.abs(gap))), float((gap > 0).mean()), int(has.sum())
