"""Generate csrc/mc_tables.cuh, the marching-cubes case table of csrc/mesh.cu, from one construction rule.

    python joint-tensorf_b200/csrc/gen_mc_tables.py          # rewrites mc_tables.cuh next to this file

Numbering. Corner i of a cell is the lattice point (x, y, z) = (i & 1, i >> 1 & 1, i >> 2 & 1) from the cell's
origin; bit i of the case is set when corner i is inside (value > level). Edge e joins EDGE_CORNER[e] (its lower
end) to EDGE_CORNER[e] + unit vector of EDGE_AXIS[e]: edges 0-3 run along x, 4-7 along y, 8-11 along z. The
vertex of an edge belongs to the lattice point at its lower end.

Construction, per case:
- Face segments. A cube face with two sign-change edges gets one segment joining them. A face with four (an
  ambiguous face) gets one segment per inside corner, joining that corner's two edges: each inside corner is cut
  off on its own. The rule reads only the face's four corners, so the two cells sharing a face draw the same
  segments and the mesh has no cracks.
- Direction. Every segment runs with the inside corners on its left, seen from outside the cube. The neighbouring
  cell sees the face from the other side and runs the segment the other way, and within a cell the segments chain
  head to tail into closed loops.
- Triangulation. Each loop becomes a fan. Its root is the first loop vertex (in loop order) from which no fan
  diagonal joins two vertices on the same cube face; otherwise both cells next to an ambiguous face could draw the
  same diagonal and that mesh edge would be shared by four triangles.
- Winding. Triangles wind so that their normals point out of the inside region, toward decreasing value.

This is not the classic Lorensen-Cline table: intersection points are the same as any marching cubes (linear
interpolation along lattice edges); the triangulation inside a cell may differ.
"""
import os

EDGE_CORNER, EDGE_AXIS = [], []
for _ax in range(3):
    for _c in range(8):
        if not (_c >> _ax) & 1:
            EDGE_CORNER.append(_c)
            EDGE_AXIS.append(_ax)
MAX_TRI = 5


def _corner_pos(c):
    return (c & 1, (c >> 1) & 1, (c >> 2) & 1)


def _edge_mid(e):
    p = list(_corner_pos(EDGE_CORNER[e]))
    p[EDGE_AXIS[e]] += 0.5
    return p


def _edge_faces(e):
    """Faces (axis, side) the edge lies on."""
    c = EDGE_CORNER[e]
    return {(b, (c >> b) & 1) for b in range(3) if b != EDGE_AXIS[e]}


def _edge_ends(e):
    return EDGE_CORNER[e], EDGE_CORNER[e] | (1 << EDGE_AXIS[e])


def _sub(a, b):
    return [a[i] - b[i] for i in range(3)]


def _cross(a, b):
    return [a[1] * b[2] - a[2] * b[1], a[2] * b[0] - a[0] * b[2], a[0] * b[1] - a[1] * b[0]]


def _dot(a, b):
    return sum(a[i] * b[i] for i in range(3))


def _face_segments(case, axis, side):
    """Directed segments (from edge, to edge) on one face."""
    inside = [(case >> c) & 1 for c in range(8)]
    edges = [e for e in range(12) if (axis, side) in _edge_faces(e)]
    cross = [e for e in edges if inside[_edge_ends(e)[0]] != inside[_edge_ends(e)[1]]]
    corners = [c for c in range(8) if ((c >> axis) & 1) == side and inside[c]]
    if len(cross) == 2:
        pairs = [(cross[0], cross[1], corners[0])]
    elif len(cross) == 4:
        pairs = []
        for c in corners:
            a, b = [e for e in cross if c in _edge_ends(e)]
            pairs.append((a, b, c))
    else:
        assert not cross
        pairs = []
    normal = [0, 0, 0]
    normal[axis] = 1 if side else -1
    out = []
    for a, b, c in pairs:
        p, q, w = _edge_mid(a), _edge_mid(b), _corner_pos(c)
        left = _dot(_cross(normal, _sub(q, p)), _sub(w, p))
        assert left != 0
        out.append((a, b) if left > 0 else (b, a))
    return out


def _loops(case):
    succ = {}
    for axis in range(3):
        for side in range(2):
            for a, b in _face_segments(case, axis, side):
                assert a not in succ
                succ[a] = b
    assert sorted(succ) == sorted(succ.values())          # every vertex: one segment in, one out
    loops, seen = [], set()
    for e in sorted(succ):
        if e in seen:
            continue
        loop = [e]
        seen.add(e)
        while succ[loop[-1]] != e:
            loop.append(succ[loop[-1]])
            seen.add(loop[-1])
        loops.append(loop)
    return loops


def _fan(loop):
    n = len(loop)
    for r in range(n):
        ring = loop[r:] + loop[:r]
        if all(not (_edge_faces(ring[0]) & _edge_faces(v)) for v in ring[2:n - 1]):
            # (root, next, previous) winding: the loop runs with the inside on its left, so this reverses it and
            # the normal points away from the inside corners
            return [(ring[0], ring[i + 1], ring[i]) for i in range(1, n - 1)]
    raise AssertionError(f"no fan root without a same-face diagonal for loop {loop}")


def tables():
    """(ntri [256], tris [256] lists of (e0, e1, e2))."""
    tris = []
    for case in range(256):
        t = []
        for loop in _loops(case):
            t += _fan(loop)
        assert len(t) <= MAX_TRI
        tris.append(t)
    # winding check on case 1 (corner 0 inside): the normal points away from corner 0
    (a, b, c), = tris[1]
    pa, pb, pc = _edge_mid(a), _edge_mid(b), _edge_mid(c)
    assert _dot(_cross(_sub(pb, pa), _sub(pc, pa)), pa) > 0
    return [len(t) for t in tris], tris


def header_text():
    ntri, tris = tables()
    lines = [
        "// Generated by gen_mc_tables.py from its construction rule; do not edit, regenerate.",
        "// Marching-cubes case table of mesh.cu. Corner i of a cell is (x, y, z) = (i & 1, i >> 1 & 1, i >> 2 & 1); bit i",
        "// of the case is set when corner i is inside (value > level). Edge e joins corner kMcEdgeCorner[e] to the next",
        "// corner along axis kMcEdgeAxis[e]. Triangle k of case c has vertices on edges kMcTri[c][3k .. 3k+2] and its",
        f"// normal points toward decreasing value. {sum(ntri)} triangles in all, at most {MAX_TRI} per case.",
        "#pragma once",
        "",
        "namespace jt {",
        "",
        "__device__ const unsigned char kMcEdgeCorner[12] = {" + ", ".join(map(str, EDGE_CORNER)) + "};",
        "__device__ const unsigned char kMcEdgeAxis[12] = {" + ", ".join(map(str, EDGE_AXIS)) + "};",
        "",
        "__device__ const unsigned char kMcNumTri[256] = {",
    ]
    for r in range(0, 256, 32):
        lines.append("    " + ", ".join(map(str, ntri[r:r + 32])) + ",")
    lines += ["};", "", f"__device__ const unsigned char kMcTri[256][{3 * MAX_TRI}] = {{"]
    for c in range(256):
        flat = [e for t in tris[c] for e in t]
        flat += [255] * (3 * MAX_TRI - len(flat))
        lines.append("    {" + ", ".join(map(str, flat)) + f"}},  // {c}")
    lines += ["};", "", "}  // namespace jt", ""]
    return "\n".join(lines)


HEADER = os.path.join(os.path.dirname(os.path.abspath(__file__)), "mc_tables.cuh")

if __name__ == "__main__":
    with open(HEADER, "w") as f:
        f.write(header_text())
    print(f"wrote {HEADER}")
