"""Float64 restatement of the vertex normals of jt_mc_normals (csrc/mesh.cu), in the vertex order of
tests/mc_reference.py.

Lattice coordinate c_a(i) = aabb0*(1-s) + aabb1*s rounded to fp32 after each operation, as mc_coord computes it.
Gradient at lattice point i along axis a: (v[i+1] - v[i-1]) / (c_a(i+1) - c_a(i-1)), one-sided at the border
((v[1] - v[0]) / (c(1) - c(0)), the same at the top end). The vertex on edge p0 -> p1 has
t = (level - v0) / (v1 - v0) in fp32 (the t of its position) and normal -normalize((1-t) g(p0) + t g(p1)),
(0, 0, 0) where that vector is zero. Everything after the fp32 t and the fp32 lattice coordinates is float64."""
import numpy as np


def lattice_f32(lin, aabb):
    """Per-axis fp32 lattice coordinates [x, y, z], rounded as mc_coord rounds them."""
    aabb = np.asarray(aabb, dtype=np.float32).reshape(2, 3)
    out = []
    for a in range(3):
        s = np.asarray(lin[a], dtype=np.float32)
        out.append(aabb[0, a] * (np.float32(1.0) - s) + aabb[1, a] * s)
    return out


def volume_gradient(vol, coord):
    """g [gz, gy, gx, 3] float64 in world units; component a is the derivative along lattice axis a (x, y, z)."""
    v = np.asarray(vol, dtype=np.float64)
    g = np.empty(v.shape + (3,))
    for a, ax in ((0, 2), (1, 1), (2, 0)):
        n = v.shape[ax]
        i = np.arange(n)
        lo, hi = np.maximum(i - 1, 0), np.minimum(i + 1, n - 1)
        c = np.asarray(coord[a], dtype=np.float64)
        shape = [1, 1, 1]
        shape[ax] = n
        g[..., a] = (np.take(v, hi, axis=ax) - np.take(v, lo, axis=ax)) / (c[hi] - c[lo]).reshape(shape)
    return g


def vertex_normals(vol, level, lin, aabb):
    """-> (normals [V, 3], blended gradient (1-t) g(p0) + t g(p1) [V, 3]), float64, in mc_reference's vertex order
    (linear index of the edge's lower end, then axis x < y < z)."""
    vol = np.asarray(vol, dtype=np.float32)
    level = np.float32(level)
    ins = vol > level
    cross = np.zeros(vol.shape + (3,), dtype=bool)
    cross[:, :, :-1, 0] = ins[:, :, :-1] != ins[:, :, 1:]
    cross[:, :-1, :, 1] = ins[:, :-1, :] != ins[:, 1:, :]
    cross[:-1, :, :, 2] = ins[:-1] != ins[1:]
    z, y, x, a = np.nonzero(cross)
    z1, y1, x1 = z + (a == 2), y + (a == 1), x + (a == 0)
    va, vb = vol[z, y, x], vol[z1, y1, x1]
    t = ((level - va) / (vb - va)).astype(np.float64)            # fp32 operations, as the kernel's t
    g = volume_gradient(vol, lattice_f32(lin, aabb))
    q = (1.0 - t)[:, None] * g[z, y, x] + t[:, None] * g[z1, y1, x1]
    length = np.linalg.norm(q, axis=1, keepdims=True)
    normals = np.where(length > 0, -q / np.where(length > 0, length, 1.0), 0.0)
    return normals, q


def face_normals(verts, faces):
    """Unnormalised right-hand normals (p1 - p0) x (p2 - p0) of the triangles, float64."""
    v = np.asarray(verts, dtype=np.float64)
    f = np.asarray(faces, dtype=np.int64)
    return np.cross(v[f[:, 1]] - v[f[:, 0]], v[f[:, 2]] - v[f[:, 0]])


def winding_agreement(verts, faces, normals):
    """Share of faces whose normal has a positive dot product with the mean of its three vertex normals."""
    f = np.asarray(faces, dtype=np.int64)
    n = np.asarray(normals, dtype=np.float64)
    mean = n[f[:, 0]] + n[f[:, 1]] + n[f[:, 2]]
    return float(np.mean(np.einsum("ij,ij->i", face_normals(verts, faces), mean) > 0)) if f.shape[0] else 1.0


def blob_field(shape_zyx, seed, k=12):
    """Smooth random field: a sum of k Gaussian blobs centred in the middle 40 % of the grid, small at the border."""
    rng = np.random.default_rng(seed)
    gz, gy, gx = shape_zyx
    z, y, x = np.meshgrid(np.arange(gz), np.arange(gy), np.arange(gx), indexing="ij")
    v = np.zeros(shape_zyx)
    for _ in range(k):
        c = rng.uniform(0.3, 0.7, 3) * np.array([gx - 1, gy - 1, gz - 1])
        r = rng.uniform(0.06, 0.14) * min(shape_zyx)
        v += rng.uniform(0.5, 1.0) * np.exp(-((x - c[0]) ** 2 + (y - c[1]) ** 2 + (z - c[2]) ** 2) / (2 * r * r))
    return v.astype(np.float32)
