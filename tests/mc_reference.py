"""Vectorised numpy marching cubes with the table of csrc/gen_mc_tables.py and the vertex / triangle order of
csrc/mesh.cu, plus the mesh properties the tests check (closure, Euler characteristic, signed volume).

Order: one vertex per lattice edge whose ends straddle the level (inside = value > level), ids ordered by the
linear index (z*gy + y)*gx + x of the edge's lower end, then by axis x < y < z; triangles ordered by the linear
index of the cell's corner 0, then by table order. Lattice point (i, j, k) is aabb0*(1-s) + aabb1*s with s from
the per-axis tables `lin`; vertices interpolate linearly along their edge in `dtype`."""
import importlib.util
import os

import numpy as np

_GEN = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "joint-tensorf_b200", "csrc",
                    "gen_mc_tables.py")


def load_generator():
    spec = importlib.util.spec_from_file_location("gen_mc_tables", _GEN)
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


GEN = load_generator()
_NT, _TRIS = GEN.tables()
NUM_TRI = np.array(_NT, dtype=np.int64)
TRI = np.full((256, 3 * GEN.MAX_TRI), -1, dtype=np.int64)
for _c, _t in enumerate(_TRIS):
    TRI[_c, :3 * len(_t)] = [e for t in _t for e in t]
EDGE_CORNER = np.array(GEN.EDGE_CORNER)
EDGE_AXIS = np.array(GEN.EDGE_AXIS)


def lattice(lin, aabb, dtype=np.float64):
    """Per-axis world coordinates of the lattice: [x table, y table, z table]."""
    aabb = np.asarray(aabb, dtype=dtype).reshape(2, 3)
    return [aabb[0, a] * (1 - np.asarray(lin[a], dtype=dtype)) + aabb[1, a] * np.asarray(lin[a], dtype=dtype)
            for a in range(3)]


def cell_cases(vol, level):
    """uint8 case of every cell [gz-1, gy-1, gx-1]."""
    ins = np.asarray(vol) > np.float32(level)
    case = np.zeros(tuple(s - 1 for s in ins.shape), dtype=np.int64)
    for c in range(8):
        x, y, z = c & 1, (c >> 1) & 1, (c >> 2) & 1
        case |= ins[z:z + ins.shape[0] - 1, y:y + ins.shape[1] - 1, x:x + ins.shape[2] - 1].astype(np.int64) << c
    return case


def marching_cubes(vol, level, lin, aabb, dtype=np.float64):
    """vol [gz, gy, gx] (fp32 values), level (compared in fp32) -> (verts [V,3] dtype, faces [F,3] int64)."""
    vol = np.asarray(vol, dtype=np.float32)
    level = np.float32(level)
    gz, gy, gx = vol.shape
    ins = vol > level
    coord = lattice(lin, aabb, dtype)
    # crossing mask per (point, axis), points in linear order -> vertex ids
    cross = np.zeros((gz, gy, gx, 3), dtype=bool)
    cross[:, :, :-1, 0] = ins[:, :, :-1] != ins[:, :, 1:]
    cross[:, :-1, :, 1] = ins[:, :-1, :] != ins[:, 1:, :]
    cross[:-1, :, :, 2] = ins[:-1] != ins[1:]
    flat = cross.reshape(-1)
    vid = np.full(flat.shape, -1, dtype=np.int64)
    vid[flat] = np.arange(int(flat.sum()))
    z, y, x, a = np.nonzero(cross)
    va = vol[z, y, x].astype(dtype)
    step = np.stack([(a == 0), (a == 1), (a == 2)], 1).astype(np.int64)
    z1, y1, x1 = z + step[:, 2], y + step[:, 1], x + step[:, 0]
    vb = vol[z1, y1, x1].astype(dtype)
    t = (dtype(level) - va) / (vb - va)
    pa = np.stack([coord[0][x], coord[1][y], coord[2][z]], 1)
    pb = np.stack([coord[0][x1], coord[1][y1], coord[2][z1]], 1)
    verts = pa + t[:, None] * (pb - pa)
    # triangles: cells in linear order of corner 0, table order within a cell
    case = cell_cases(vol, level)
    cz, cy, cx = np.nonzero(NUM_TRI[case] > 0)
    cc = case[cz, cy, cx]
    nt = NUM_TRI[cc]
    rep = np.repeat(np.arange(cc.size), nt)
    k = np.arange(rep.size) - np.repeat(np.cumsum(nt) - nt, nt)
    faces = np.empty((rep.size, 3), dtype=np.int64)
    for j in range(3):
        e = TRI[cc[rep], 3 * k + j]
        c0 = EDGE_CORNER[e]
        ox, oy, oz = cx[rep] + (c0 & 1), cy[rep] + ((c0 >> 1) & 1), cz[rep] + ((c0 >> 2) & 1)
        faces[:, j] = vid[(((oz * gy + oy) * gx + ox) * 3) + EDGE_AXIS[e]]
    assert (faces >= 0).all()
    return verts, faces


# ------------------------------------------------------------------ mesh properties
def directed_edges_closed(faces, n_verts):
    """Every directed edge appears exactly once and its reverse exactly once."""
    f = np.asarray(faces, dtype=np.int64)
    a = np.concatenate([f[:, 0], f[:, 1], f[:, 2]])
    b = np.concatenate([f[:, 1], f[:, 2], f[:, 0]])
    key = np.sort(a * n_verts + b)
    rev = np.sort(b * n_verts + a)
    return bool(key.size == 0 or (np.all(np.diff(key) != 0) and np.array_equal(key, rev)))


def euler_characteristic(faces, n_verts):
    """V - E + F of a closed mesh (E = 3F / 2); counts only vertices used by a face."""
    f = np.asarray(faces)
    return int(np.unique(f).size) - 3 * f.shape[0] // 2 + f.shape[0]


def signed_volume(verts, faces):
    v = np.asarray(verts, dtype=np.float64)
    f = np.asarray(faces, dtype=np.int64)
    p0, p1, p2 = v[f[:, 0]], v[f[:, 1]], v[f[:, 2]]
    return float(np.einsum("ij,ij->i", p0, np.cross(p1, p2)).sum() / 6.0)


# ------------------------------------------------------------------ test fields
def padded_random(shape, seed, pad_value=-1.0):
    """Uniform [0, 1) values with a border of pad_value: any level in [0, 1) gives a closed mesh."""
    v = np.random.default_rng(seed).random(shape).astype(np.float32)
    v[0], v[-1], v[:, 0], v[:, -1], v[:, :, 0], v[:, :, -1] = (pad_value,) * 6
    return v


def unit_lin(shape_zyx):
    """Lattice tables s = torch.linspace(0, 1, g) for [x, y, z] (fp32), the tables getDenseAlpha uses."""
    import torch
    gz, gy, gx = shape_zyx
    return [torch.linspace(0, 1, g).numpy() for g in (gx, gy, gz)]


def voxel_aabb(shape_zyx):
    """aabb that makes the lattice spacing one unit per voxel."""
    gz, gy, gx = shape_zyx
    return np.array([[0.0, 0.0, 0.0], [gx - 1.0, gy - 1.0, gz - 1.0]])


def sphere_field(n, radius):
    """radius - distance from the grid centre (positive inside), on an n^3 grid, in voxel units."""
    c = (n - 1) / 2.0
    z, y, x = np.meshgrid(*[np.arange(n, dtype=np.float64)] * 3, indexing="ij")
    return (radius - np.sqrt((x - c) ** 2 + (y - c) ** 2 + (z - c) ** 2)).astype(np.float32)


def torus_field(n, big, small):
    """small - distance from the circle of radius big around the z axis (positive inside)."""
    c = (n - 1) / 2.0
    z, y, x = np.meshgrid(*[np.arange(n, dtype=np.float64)] * 3, indexing="ij")
    q = np.sqrt((x - c) ** 2 + (y - c) ** 2) - big
    return (small - np.sqrt(q ** 2 + (z - c) ** 2)).astype(np.float32)
