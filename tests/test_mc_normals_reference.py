"""The float64 vertex-normal reference (tests/mc_normals_reference.py) on fields whose normals are known."""
import numpy as np

import mc_normals_reference as nr
import mc_reference as mr


def _angles_to_radial(verts, normals, centre):
    r = verts - centre
    r /= np.linalg.norm(r, axis=1, keepdims=True)
    return np.degrees(np.arccos(np.clip(np.einsum("ij,ij->i", r, normals), -1.0, 1.0)))


def test_sphere_normals_are_radial():
    vol = mr.sphere_field(24, 8.0)
    aabb = mr.voxel_aabb(vol.shape)
    lin = mr.unit_lin(vol.shape)
    verts, faces = mr.marching_cubes(vol, 0.0, lin, aabb)
    normals, _ = nr.vertex_normals(vol, 0.0, lin, aabb)
    assert normals.shape == verts.shape
    assert np.allclose(np.linalg.norm(normals, axis=1), 1.0)
    assert _angles_to_radial(verts, normals, 11.5).max() < 1.0
    assert nr.winding_agreement(verts, faces, normals) == 1.0


def test_sphere_on_an_anisotropic_world_lattice_is_radial_in_world_units():
    aabb = np.array([[-1.0, -2.0, -0.5], [1.0, 2.0, 0.5]])
    shape = (21, 61, 31)                                            # spacing 0.05, 0.0667, 0.05
    lin = mr.unit_lin(shape)
    cz, cy, cx = np.meshgrid(*[aabb[0, a] * (1 - lin[a].astype(np.float64)) + aabb[1, a] * lin[a] for a in (2, 1, 0)],
                             indexing="ij")
    vol = (0.4 - np.sqrt(cx ** 2 + cy ** 2 + cz ** 2)).astype(np.float32)
    verts, _ = mr.marching_cubes(vol, 0.0, lin, aabb)
    normals, _ = nr.vertex_normals(vol, 0.0, lin, aabb)
    assert _angles_to_radial(verts, normals, np.zeros(3)).max() < 2.0


def test_linear_field_has_its_gradient_everywhere_including_the_border():
    shape = (6, 9, 7)
    aabb = np.array([[-1.0, -1.5, 0.0], [2.0, 1.5, 1.0]])
    lin = mr.unit_lin(shape)
    coord = nr.lattice_f32(lin, aabb)
    a = np.array([0.7, -1.3, 2.1])
    z, y, x = np.meshgrid(*[coord[i].astype(np.float64) for i in (2, 1, 0)], indexing="ij")
    vol = (a[0] * x + a[1] * y + a[2] * z).astype(np.float32)
    g = nr.volume_gradient(vol, coord)
    assert np.abs(g - a).max() <= 1e-5 * np.abs(a).max()           # fp32 volume values
    normals, _ = nr.vertex_normals(vol, 0.3, lin, aabb)
    assert normals.shape[0] > 0
    assert np.abs(normals + a / np.linalg.norm(a)).max() <= 1e-5


def test_winding_agreement_on_smooth_random_fields():
    bad = total = 0
    for shape, seed in (((40, 44, 48), 0), ((33, 31, 29), 1), ((48, 24, 40), 2)):
        vol = nr.blob_field(shape, seed)
        lin = mr.unit_lin(shape)
        for level in (0.2, 0.4, 0.6):
            verts, faces = mr.marching_cubes(vol, level, lin, [[-1.5, -1.67, -2.0], [1.5, 1.67, 1.0]])
            normals, _ = nr.vertex_normals(vol, level, lin, [[-1.5, -1.67, -2.0], [1.5, 1.67, 1.0]])
            share = nr.winding_agreement(verts, faces, normals)
            bad += round((1.0 - share) * faces.shape[0])
            total += faces.shape[0]
    assert total > 10000 and bad <= 1e-3 * total, (bad, total)
