"""Vertex normals of the mesh export (jt_mc_normals, ops.marching_cubes(normals=True)) against the float64 reference
of tests/mc_normals_reference.py, on the volumes test_gpu_mesh.py uses and on smooth and analytic fields."""
import numpy as np
import pytest
import torch

import mc_normals_reference as nr
import mc_reference as mr
from gpu_common import record_err
from joint_tensorf_b200 import ops

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
AABB = np.array([[-1.5, -1.67, -2.0], [1.5, 1.67, 1.0]])


def _lin(shape_zyx):
    gz, gy, gx = shape_zyx
    return [torch.linspace(0, 1, g).to(DEV) for g in (gx, gy, gz)]


def _check(vol, level, aabb=AABB):
    """normals=True against normals=False (bitwise) and against the reference; returns (verts, faces, normals)."""
    v = torch.from_numpy(np.ascontiguousarray(vol, dtype=np.float32)).to(DEV)
    lin = _lin(vol.shape)
    verts0, faces0 = ops.marching_cubes(v, level, lin, torch.as_tensor(aabb))
    verts, faces, normals = ops.marching_cubes(v, level, lin, torch.as_tensor(aabb), normals=True)
    assert torch.equal(verts, verts0) and torch.equal(faces, faces0)
    assert normals.dtype == torch.float32 and tuple(normals.shape) == tuple(verts.shape)
    ref, q = nr.vertex_normals(vol, level, [t.cpu().numpy() for t in lin], aabb)
    got = normals.double().cpu().numpy()
    qn = np.linalg.norm(q, axis=1)
    if qn.size:
        sel = qn >= 1e-3 * qn.max()
        err = float(np.abs(got[sel] - ref[sel]).max())
        assert err <= 1e-5, err
        assert np.array_equal(np.all(got == 0, axis=1), qn == 0)
    again = ops.marching_cubes(v, level, lin, torch.as_tensor(aabb), normals=True)[2]
    assert torch.equal(again, normals)
    return verts, faces, normals, ref


def test_random_padded_and_unpadded_fields_match_the_reference():
    shares = []
    for shape, seed in (((23, 29, 37), 0), ((16, 21, 11), 1), ((40, 9, 17), 2), ((31, 33, 35), 3)):
        vol = mr.padded_random(shape, seed)
        for level in (0.15, 0.5, 0.85):
            verts, faces, normals, ref = _check(vol, level)
            # white noise: the central difference over three lattice points says little about one facet, so the
            # winding agreement is a property of the definition (about 0.73 to 0.90); ours equals the reference's
            v, f = verts.double().cpu().numpy(), faces.cpu().numpy()
            share, share_ref = nr.winding_agreement(v, f, normals.cpu().numpy()), nr.winding_agreement(v, f, ref)
            assert abs(share - share_ref) * f.shape[0] <= 2, (share, share_ref)
            shares.append(share)
    record_err("mc_normals_winding_white_noise", min=min(shares), max=max(shares))
    _check(np.random.default_rng(5).standard_normal((13, 7, 45)).astype(np.float32), 0.1)


def test_all_256_single_cell_cases():
    for c in range(256):
        vol = np.array([[[1.0 if (c >> (4 * z + 2 * y + x)) & 1 else -1.0 for x in range(2)] for y in range(2)]
                        for z in range(2)], dtype=np.float32)
        _, _, normals, _ = _check(vol, 0.0)
        assert torch.isfinite(normals).all()


def test_normals_agree_with_the_winding_on_smooth_random_fields():
    bad = total = 0
    for shape, seed in (((40, 44, 48), 0), ((33, 31, 29), 1), ((48, 24, 40), 2)):
        vol = nr.blob_field(shape, seed)
        for level in (0.2, 0.4, 0.6):
            verts, faces, normals, _ = _check(vol, level)
            share = nr.winding_agreement(verts.double().cpu().numpy(), faces.cpu().numpy(), normals.cpu().numpy())
            bad += round((1.0 - share) * faces.shape[0])
            total += faces.shape[0]
    record_err("mc_normals_winding_smooth", share=1.0 - bad / total, faces=total)
    assert total > 10000 and bad <= 1e-3 * total, (bad, total)


def test_sphere_normals_are_radial_and_unit():
    vol = mr.sphere_field(24, 8.0)
    verts, faces, normals, _ = _check(vol, 0.0, mr.voxel_aabb(vol.shape))
    r = verts.double() - 11.5
    r = r / r.norm(dim=1, keepdim=True)
    ang = torch.rad2deg(torch.arccos((r * normals.double()).sum(1).clamp(-1, 1)))
    assert float(ang.max()) < 1.0
    assert float((normals.double().norm(dim=1) - 1).abs().max()) <= 1e-6
    assert nr.winding_agreement(verts.double().cpu().numpy(), faces.cpu().numpy(), normals.cpu().numpy()) == 1.0


def test_empty_mesh_returns_empty_normals():
    v = torch.full((5, 6, 7), 0.5, device=DEV)
    verts, faces, normals = ops.marching_cubes(v, 0.5, _lin(v.shape), AABB, normals=True)
    assert tuple(normals.shape) == (0, 3) and normals.device.type == "cuda"
