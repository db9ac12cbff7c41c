"""Generates meshanything_b200/csrc/mc_table.cuh, the 256-case marching-cubes table of csrc/watertight.cu.

Conventions (shared with watertight.cu and tests/test_watertight.py):
  corner c of a cell = bits (x, y, z) = (c & 1, c >> 1 & 1, c >> 2 & 1); bit c of the case index is set when the field
  at that corner is below the level ("inside");
  edge e = 4 * axis + o, where o packs the offsets of the two other axes in increasing axis order (lower axis in bit 0);
  the edge runs from its lower corner (offset 0 along `axis`) to the upper one.

The table is derived, not typed: on each of the 6 faces the crossing edges are paired into segments by a rule that reads
only that face's 4 corner bits (two crossings: one segment; four crossings, the ambiguous face: two segments, each cutting
off one outside corner, so the inside corners stay connected).  Each segment is directed so that, seen from outside the
cube, the outside corner of its start edge lies to its left: the two cells that share a face then get the same segments
with opposite directions.  The directed segments of a case chain into closed loops, and every loop is fan-triangulated
from an apex chosen so that no fan diagonal joins two vertices of one cube face (such a chord could be repeated by the
neighbouring cell).  A triangle's normal (v1 - v0) x (v2 - v0) then points out of the inside region.

usage: python tools/make_mc_table.py   (rewrites meshanything_b200/csrc/mc_table.cuh)
"""
import os

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
OUT = os.path.join(ROOT, "meshanything_b200", "csrc", "mc_table.cuh")


def corner_pos(c):
    return np.array([c & 1, (c >> 1) & 1, (c >> 2) & 1], dtype=np.float64)


def edge_corners(e):
    """(lower corner, upper corner) of cube edge e."""
    axis, o = divmod(e, 4)
    others = [a for a in range(3) if a != axis]
    c = ((o & 1) << others[0]) | (((o >> 1) & 1) << others[1])
    return c, c | (1 << axis)


def edge_mid(e):
    a, b = edge_corners(e)
    return 0.5 * (corner_pos(a) + corner_pos(b))


EDGES = [edge_corners(e) for e in range(12)]


def faces():
    """The 6 cube faces: (outward normal, 4 corners in cyclic order)."""
    out = []
    for axis in range(3):
        u, v = [a for a in range(3) if a != axis]
        for side in (0, 1):
            base = side << axis
            ring = [base, base | (1 << u), base | (1 << u) | (1 << v), base | (1 << v)]
            n = np.zeros(3)
            n[axis] = 1.0 if side else -1.0
            out.append((n, ring))
    return out


FACES = faces()


def edge_id(c0, c1):
    for e, (a, b) in enumerate(EDGES):
        if {a, b} == {c0, c1}:
            return e
    raise KeyError((c0, c1))


def face_segments(case, normal, ring):
    """Directed segments (start edge, end edge) of one face; a function of the face's four corner bits only."""
    inside = [(case >> c) & 1 for c in ring]
    cross = [k for k in range(4) if inside[k] != inside[(k + 1) % 4]]      # ring side k joins ring[k] and ring[k+1]
    if not cross:
        return []
    if len(cross) == 2:
        pairs = [tuple(cross)]
    else:  # ambiguous face: cut off each outside corner by the two sides that meet at it
        pairs = [((k - 1) % 4, k) for k in range(4) if not inside[k]]
    segs = []
    for s0, s1 in pairs:
        e0 = edge_id(ring[s0], ring[(s0 + 1) % 4])
        e1 = edge_id(ring[s1], ring[(s1 + 1) % 4])
        p, q = edge_mid(e0), edge_mid(e1)
        a, b = EDGES[e0]
        out_corner = corner_pos(a if not (case >> a) & 1 else b)
        # direction: the outside corner of the start edge lies to the left of p -> q seen from outside the face
        if np.dot(np.cross(normal, q - p), out_corner - p) < 0:
            e0, e1 = e1, e0
        segs.append((e0, e1))
    return segs


def face_of_edges(e0, e1):
    """True when cube edges e0 and e1 lie on a common cube face."""
    c = set(EDGES[e0]) | set(EDGES[e1])
    return any(c <= set(ring) for _, ring in FACES)


def case_loops(case):
    nxt = {}
    for normal, ring in FACES:
        for e0, e1 in face_segments(case, normal, ring):
            assert e0 not in nxt, (case, e0)
            nxt[e0] = e1
    loops, seen = [], set()
    for start in sorted(nxt):
        if start in seen:
            continue
        loop, e = [], start
        while e not in seen:
            seen.add(e)
            loop.append(e)
            e = nxt[e]
        assert e == start, (case, loop)
        loops.append(loop)
    return loops, nxt


def fan(loop, nxt):
    """Fan triangles of one loop from the first apex (in loop order) none of whose diagonals is a face chord."""
    n = len(loop)
    for r in range(n):
        lp = loop[r:] + loop[:r]
        diag = [(lp[0], lp[i]) for i in range(2, n - 1)]
        if all(not face_of_edges(a, b) for a, b in diag):
            return [(lp[0], lp[i], lp[i + 1]) for i in range(1, n - 1)]
    raise AssertionError(f"no chord-free fan apex for loop {loop}")


def build_table():
    table = []
    for case in range(256):
        loops, nxt = case_loops(case)
        tris = []
        for lp in loops:
            tris.extend(fan(lp, nxt))
        table.append(tris)
    return table


def render(table):
    width = max(len(t) for t in table)
    lines = [
        "// mc_table.cuh -- GENERATED by tools/make_mc_table.py; do not edit.  Conventions are stated there.",
        "#pragma once",
        "#include <stdint.h>",
        "",
        "namespace ma {",
        "",
        f"constexpr int MC_MAX_TRIS = {width};",
        "// triangles of each case",
        "__device__ __constant__ uint8_t mc_ntri[256] = {",
    ]
    for r in range(0, 256, 32):
        lines.append("    " + ", ".join(str(len(table[c])) for c in range(r, r + 32)) + ",")
    lines.append("};")
    lines.append(f"// cube edges of each triangle, 3 x 4 bits packed per uint16 (v0 | v1 << 4 | v2 << 8)")
    lines.append(f"__device__ __constant__ uint16_t mc_tris[256][{width}] = {{")
    for c in range(256):
        ent = [str(a | (b << 4) | (d << 8)) for a, b, d in table[c]] + ["0"] * (width - len(table[c]))
        lines.append("    {" + ", ".join(ent) + "},")
    lines.append("};")
    lines += ["", "}  // namespace ma", ""]
    return "\n".join(lines)


def load_table(path=OUT):
    """Parses the generated header back into [case] -> [(e0, e1, e2), ...] (used by the tests)."""
    txt = open(path).read()
    ntri = [int(x) for x in txt.split("mc_ntri[256] = {")[1].split("};")[0].replace("\n", " ").split(",") if x.strip()]
    body = txt.split("mc_tris[256]")[1].split("= {", 1)[1].split("};")[0]
    rows = [r.strip().strip(",").strip("{}") for r in body.strip().splitlines()]
    out = []
    for c, r in enumerate(rows):
        vals = [int(x) for x in r.split(",")]
        out.append([(v & 15, (v >> 4) & 15, (v >> 8) & 15) for v in vals[:ntri[c]]])
    return out


if __name__ == "__main__":
    t = build_table()
    with open(OUT, "w") as f:
        f.write(render(t))
    print("wrote", OUT, "max triangles per case", max(len(x) for x in t), "total", sum(len(x) for x in t))
