"""Mesh export (csrc/mesh.cu, ops.marching_cubes, B200_VMSplit.extract_mesh / export_mesh) against the numpy oracle
of tests/mc_reference.py and against mesh properties, from single cells up to the benchmark's field sizes."""
import math

import numpy as np
import pytest
import torch

import joint_tensorf_b200 as jt
import mc_reference as mr
from joint_tensorf_b200 import ops

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
AABB = np.array([[-1.5, -1.67, -2.0], [1.5, 1.67, 1.0]])


def _lin(shape_zyx):
    gz, gy, gx = shape_zyx
    return [torch.linspace(0, 1, g).to(DEV) for g in (gx, gy, gz)]


def _gpu_mc(vol, level, aabb=AABB):
    v = torch.from_numpy(np.ascontiguousarray(vol, dtype=np.float32)).to(DEV)
    return ops.marching_cubes(v, level, _lin(vol.shape), torch.as_tensor(aabb))


def _oracle(vol, level, aabb=AABB):
    return mr.marching_cubes(vol, level, [t.cpu().numpy() for t in _lin(vol.shape)], aabb)


def _assert_matches_oracle(vol, level, aabb=AABB):
    verts, faces = _gpu_mc(vol, level, aabb)
    rv, rf = _oracle(vol, level, aabb)
    assert verts.dtype == torch.float32 and faces.dtype == torch.int32
    assert tuple(verts.shape) == rv.shape and tuple(faces.shape) == rf.shape
    assert torch.equal(faces.long().cpu(), torch.from_numpy(rf))
    extent = float(np.max(np.asarray(aabb)[1] - np.asarray(aabb)[0]))
    if rv.shape[0]:
        assert float(np.abs(verts.double().cpu().numpy() - rv).max()) <= 1e-6 * extent
    return verts, faces


def test_random_padded_fields_match_oracle_exactly_and_close():
    seen = set()
    for shape, seed in (((23, 29, 37), 0), ((16, 21, 11), 1), ((40, 9, 17), 2), ((31, 33, 35), 3)):
        vol = mr.padded_random(shape, seed)
        for level in (0.15, 0.5, 0.85):
            verts, faces = _assert_matches_oracle(vol, level)
            assert faces.shape[0] > 0
            assert mr.directed_edges_closed(faces.cpu().numpy(), verts.shape[0])
            assert mr.signed_volume(verts.cpu().numpy(), faces.cpu().numpy()) > 0
            seen |= set(np.unique(mr.cell_cases(vol, level)).tolist())
    assert seen >= set(range(1, 255)), sorted(set(range(1, 255)) - seen)


def test_unpadded_field_with_surface_on_the_border_matches_oracle():
    vol = np.random.default_rng(5).standard_normal((13, 7, 45)).astype(np.float32)
    _assert_matches_oracle(vol, 0.1)


def test_all_256_cases_on_single_cells():
    for c in range(256):
        vol = np.array([[[1.0 if (c >> (4 * z + 2 * y + x)) & 1 else -1.0 for x in range(2)] for y in range(2)]
                        for z in range(2)], dtype=np.float32)
        verts, faces = _assert_matches_oracle(vol, 0.0)
        assert faces.shape[0] == mr.NUM_TRI[c], c
        assert torch.isfinite(verts).all()


def test_values_equal_to_the_level():
    # corner 0 sits exactly on the level (outside), corner 1 above: the x edge's vertex is corner 0 itself
    vol = np.full((2, 2, 2), 0.25, dtype=np.float32)
    vol[0, 0, 1] = 1.0
    verts, faces = _assert_matches_oracle(vol, 0.25, aabb=mr.voxel_aabb(vol.shape))
    assert torch.isfinite(verts).all() and faces.shape[0] == 1
    assert verts.shape[0] == 3
    assert torch.equal(verts[0].cpu(), torch.zeros(3))
    vol = mr.padded_random((12, 11, 10), 7)
    vol[vol > 0.6] = 0.5                              # many values exactly at the level
    verts, _ = _assert_matches_oracle(vol, 0.5)
    assert torch.isfinite(verts).all()
    for level in (2.0, -2.0, 0.5):                    # above the max, below the min; a flat volume
        v = vol if level != 0.5 else np.full((5, 6, 7), 0.5, dtype=np.float32)
        verts, faces = _gpu_mc(v, level)
        assert tuple(verts.shape) == (0, 3) and tuple(faces.shape) == (0, 3)
        assert verts.device.type == "cuda" and faces.dtype == torch.int32


def test_rejects_bad_input():
    vol = torch.rand((5, 6, 7), device=DEV)
    lin = _lin(vol.shape)
    with pytest.raises(jt._lib.JtError):
        ops.marching_cubes(vol.cpu(), 0.5, lin, AABB)
    with pytest.raises(jt._lib.JtError):
        ops.marching_cubes(vol.double(), 0.5, lin, AABB)
    with pytest.raises(jt._lib.JtError):
        ops.marching_cubes(vol.transpose(0, 2), 0.5, lin, AABB)
    with pytest.raises(jt._lib.JtError):
        ops.marching_cubes(torch.rand((1, 6, 7), device=DEV), 0.5, _lin((1, 6, 7)), AABB)
    for level in (float("nan"), float("inf"), -float("inf")):
        with pytest.raises(jt._lib.JtError):
            ops.marching_cubes(vol, level, lin, AABB)


def test_sphere_and_torus_on_the_gpu():
    vol = mr.sphere_field(24, 8.0)
    aabb = mr.voxel_aabb(vol.shape)
    verts, faces = _assert_matches_oracle(vol, 0.0, aabb)
    v, f = verts.cpu().numpy(), faces.cpu().numpy()
    assert mr.directed_edges_closed(f, v.shape[0])
    assert mr.euler_characteristic(f, v.shape[0]) == 2
    vol_ref = 4.0 / 3.0 * math.pi * 8.0 ** 3
    sv = mr.signed_volume(v, f)
    assert sv > 0 and abs(sv - vol_ref) <= 0.02 * vol_ref
    again = _gpu_mc(vol, 0.0, aabb)
    assert torch.equal(again[0], verts) and torch.equal(again[1], faces)
    vol = mr.torus_field(32, 9.0, 4.0)
    verts, faces = _assert_matches_oracle(vol, 0.0, mr.voxel_aabb(vol.shape))
    assert mr.directed_edges_closed(faces.cpu().numpy(), verts.shape[0])
    assert mr.euler_characteristic(faces.cpu().numpy(), verts.shape[0]) == 0


def _small_module(grid):
    torch.manual_seed(0)
    kw, _ = jt.synth.config("cfg4")
    kw = dict(kw, gridSize=grid)
    return jt.B200_VMSplit(torch.tensor(kw.pop("aabb")), kw.pop("gridSize"), DEV, **kw)


def _quantile(t, q):
    flat = t.reshape(-1).sort().values
    return float(flat[int(q * (flat.numel() - 1))])


def _assert_module_mesh(m, level, grid=None):
    g = m._grid if grid is None else grid
    verts, faces = m.extract_mesh(level, grid)
    rv, rf = ops.marching_cubes(m._dense_alpha_zyx(g), level, m._dense_tables(g), m._h_aabb)
    assert torch.equal(verts, rv) and torch.equal(faces, rf) and faces.shape[0] > 0
    extent = float((m.aabb[1] - m.aabb[0]).max())
    assert bool((verts >= m.aabb[0] - 1e-6 * extent).all()) and bool((verts <= m.aabb[1] + 1e-6 * extent).all())
    return verts, faces


def test_extract_mesh_equals_op_on_dense_alpha_with_mask_grid_and_shrink(tmp_path):
    m = _small_module([48, 44, 40])
    alpha = m._dense_alpha_zyx(m._grid)
    level = _quantile(alpha, 0.5)
    _assert_module_mesh(m, level)
    _assert_module_mesh(m, level, [37, 29, 23])
    m.alphaMask_thres = _quantile(alpha, 0.99)      # the 5^3 max-pool keeps most voxels; this drops some
    m.updateAlphaMask([48, 44, 40])
    masked = m._dense_alpha_zyx(m._grid)
    assert bool((masked == 0).any())                  # the mask removes part of the field
    _assert_module_mesh(m, level)
    _assert_module_mesh(m, level, [37, 29, 23])
    m.shrink(m.aabb * 0.6)
    assert m._grid != [48, 44, 40]
    _assert_module_mesh(m, level)
    # PLY round trip
    path = str(tmp_path / "mesh.ply")
    verts, faces = m.extract_mesh(level)
    nv, nf = m.export_mesh(path, level)
    assert (nv, nf) == (verts.shape[0], faces.shape[0])
    raw = open(path, "rb").read()
    head, body = raw.split(b"end_header\n", 1)
    assert head.decode().splitlines()[:3] == ["ply", "format binary_little_endian 1.0", f"element vertex {nv}"]
    assert f"element face {nf}" in head.decode() and "property list uchar int vertex_indices" in head.decode()
    v = np.frombuffer(body[:12 * nv], dtype="<f4").reshape(nv, 3)
    f = np.frombuffer(body[12 * nv:], dtype=[("n", "u1"), ("i", "<i4", (3,))])
    assert f.shape[0] == nf and (f["n"] == 3).all()
    assert np.array_equal(v, verts.cpu().numpy()) and np.array_equal(f["i"], faces.cpu().numpy())


def _closed_on_gpu(faces, nv):
    f = faces.long()
    a = torch.cat([f[:, 0], f[:, 1], f[:, 2]])
    b = torch.cat([f[:, 1], f[:, 2], f[:, 0]])
    key = (a * nv + b).sort().values
    del a, b
    rev = ((key % nv) * nv + key // nv).sort().values
    return bool((key[1:] != key[:-1]).all()) and torch.equal(key, rev)


@pytest.mark.parametrize("wl", ["cfg2", "cfg4"])
def test_full_size_field_at_the_median_level(wl):
    kw, _ = jt.synth.config(wl)
    kw = dict(kw)
    torch.manual_seed(0)
    m = jt.B200_VMSplit(torch.tensor(kw.pop("aabb")), kw.pop("gridSize"), DEV, **kw)
    alpha = m._dense_alpha_zyx(m._grid)
    level = _quantile(alpha, 0.5)
    verts, faces = m.extract_mesh(level)
    lv = torch.tensor(level, dtype=torch.float32)
    ins = alpha > lv.item()
    gz, gy, gx = ins.shape
    nv = sum(int((ins.narrow(d, 0, s - 1) != ins.narrow(d, 1, s - 1)).sum()) for d, s in enumerate(ins.shape))
    assert verts.shape[0] == nv
    case = torch.zeros((gz - 1, gy - 1, gx - 1), dtype=torch.uint8, device=DEV)
    for c in range(8):
        x, y, z = c & 1, (c >> 1) & 1, (c >> 2) & 1
        case |= ins[z:z + gz - 1, y:y + gy - 1, x:x + gx - 1].to(torch.uint8) << c
    ntri = torch.from_numpy(mr.NUM_TRI).to(DEV)
    assert faces.shape[0] == int(ntri[case.long()].sum())
    del case
    # every vertex on its edge at the interpolated position, slab by slab of owner z
    lin = [t.double() for t in m._dense_tables(m._grid)]
    a0, a1 = m._h_aabb.double().tolist()
    coord = [a0[i] * (1 - lin[i]) + a1[i] * lin[i] for i in range(3)]
    extent = max(a1[i] - a0[i] for i in range(3))
    off, slab = 0, 16
    for z0 in range(0, gz, slab):
        z1 = min(gz, z0 + slab)
        m3 = torch.zeros((z1 - z0, gy, gx, 3), dtype=torch.bool, device=DEV)
        m3[:, :, :-1, 0] = ins[z0:z1, :, :-1] != ins[z0:z1, :, 1:]
        m3[:, :-1, :, 1] = ins[z0:z1, :-1, :] != ins[z0:z1, 1:, :]
        ze = min(z1, gz - 1)
        m3[:ze - z0, :, :, 2] = ins[z0:ze] != ins[z0 + 1:ze + 1]
        z, y, x, a = m3.nonzero().unbind(1)
        z = z + z0
        va = alpha[z, y, x].double()
        vb = alpha[z + (a == 2), y + (a == 1), x + (a == 0)].double()
        t = (lv.double().to(DEV) - va) / (vb - va)
        pa = torch.stack([coord[0][x], coord[1][y], coord[2][z]], 1)
        pb = torch.stack([coord[0][x + (a == 0)], coord[1][y + (a == 1)], coord[2][z + (a == 2)]], 1)
        exp = pa + t[:, None] * (pb - pa)
        got = verts[off:off + exp.shape[0]].double()
        assert float((got - exp).abs().max()) <= 1e-6 * extent, z0
        off += exp.shape[0]
        del m3, z, y, x, a, va, vb, t, pa, pb, exp, got
    assert off == verts.shape[0]
    del verts, faces
    if wl == "cfg2":                                  # closure needs a surface that stays off the border
        alpha[0], alpha[-1], alpha[:, 0], alpha[:, -1], alpha[:, :, 0], alpha[:, :, -1] = (level - 1.0,) * 6
        verts, faces = ops.marching_cubes(alpha, level, m._dense_tables(m._grid), m._h_aabb)
        assert faces.shape[0] > 0 and _closed_on_gpu(faces, verts.shape[0])
