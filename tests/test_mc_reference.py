"""The marching-cubes case table (csrc/mc_tables.cuh) is what its generator builds, and the numpy oracle built on
it (tests/mc_reference.py) yields closed, consistently oriented meshes of the right topology and volume."""
import math

import numpy as np
import pytest
import torch

import mc_reference as mr
from joint_tensorf_b200 import _lib, ops


def test_committed_table_equals_generator_output():
    with open(mr.GEN.HEADER) as f:
        committed = f.read()
    assert committed == mr.GEN.header_text(), "mc_tables.cuh is stale: run csrc/gen_mc_tables.py"


def test_table_shape():
    assert mr.NUM_TRI[0] == 0 and mr.NUM_TRI[255] == 0
    assert (mr.NUM_TRI[1:255] > 0).all()
    assert int(mr.NUM_TRI.sum()) == 820 and int(mr.NUM_TRI.max()) == 5
    # a case and its complement cut the same edges
    for c in range(256):
        used = set(mr.TRI[c][mr.TRI[c] >= 0].tolist())
        assert used == set(mr.TRI[255 - c][mr.TRI[255 - c] >= 0].tolist())
        ins = [(c >> k) & 1 for k in range(8)]
        crossing = {e for e in range(12)
                    if ins[mr.EDGE_CORNER[e]] != ins[mr.EDGE_CORNER[e] | (1 << mr.EDGE_AXIS[e])]}
        assert used == crossing, c


@pytest.mark.parametrize("shape,seed", [((9, 8, 7), 0), ((12, 10, 11), 1), ((23, 29, 37), 2)])
@pytest.mark.parametrize("level", [0.2, 0.5, 0.8])
def test_random_padded_fields_close_with_positive_volume(shape, seed, level):
    vol = mr.padded_random(shape, seed)
    verts, faces = mr.marching_cubes(vol, level, mr.unit_lin(shape), mr.voxel_aabb(shape))
    assert faces.shape[0] > 0
    assert mr.directed_edges_closed(faces, verts.shape[0])
    assert np.unique(faces).size == verts.shape[0]           # every vertex is used
    assert mr.signed_volume(verts, faces) > 0


def test_sphere_and_torus_topology_and_volume():
    n = 24
    vol = mr.sphere_field(n, 8.0)
    verts, faces = mr.marching_cubes(vol, 0.0, mr.unit_lin(vol.shape), mr.voxel_aabb(vol.shape))
    assert mr.directed_edges_closed(faces, verts.shape[0])
    assert mr.euler_characteristic(faces, verts.shape[0]) == 2
    ref = 4.0 / 3.0 * math.pi * 8.0 ** 3
    assert abs(mr.signed_volume(verts, faces) - ref) <= 0.02 * ref
    vol = mr.torus_field(32, 9.0, 4.0)
    verts, faces = mr.marching_cubes(vol, 0.0, mr.unit_lin(vol.shape), mr.voxel_aabb(vol.shape))
    assert mr.directed_edges_closed(faces, verts.shape[0])
    assert mr.euler_characteristic(faces, verts.shape[0]) == 0
    assert mr.signed_volume(verts, faces) > 0


def test_every_case_in_a_single_cell_is_closed_in_its_padded_neighbourhood():
    """Each case on a 2x2x2 block inside a 4x4x4 low border: a closed mesh of positive volume."""
    for c in range(1, 255):
        vol = np.full((4, 4, 4), -1.0, dtype=np.float32)
        for k in range(8):
            vol[1 + ((k >> 2) & 1), 1 + ((k >> 1) & 1), 1 + (k & 1)] = 1.0 if (c >> k) & 1 else -1.0
        verts, faces = mr.marching_cubes(vol, 0.0, mr.unit_lin(vol.shape), mr.voxel_aabb(vol.shape))
        assert mr.directed_edges_closed(faces, verts.shape[0]), c
        assert mr.signed_volume(verts, faces) > 0, c


def test_entry_points_reject_bad_arguments_without_gpu():
    lib = _lib.lib()
    assert lib.jt_mc_scratch_bytes(617, 687, 617) == -(-617 * 687 * 617 // 2048) * 1304
    assert lib.jt_mc_scratch_bytes(1, 5, 5) == -1
    assert lib.jt_mc_scratch_bytes(2048, 2048, 1024) == -1          # 2^32 lattice points
    assert lib.jt_mc_count(0, 4, 4, 4, 0.0, 0, 0, 0) == -1
    assert lib.jt_mc_emit(0, 4, 4, 4, 0.0, 0, 0, 0, 0, 0, 0, 0, 0, 0) == -1
    with pytest.raises(_lib.JtError):
        ops.marching_cubes(torch.rand((4, 4, 4)), 0.5, [torch.linspace(0, 1, 4)] * 3, mr.voxel_aabb((4, 4, 4)))
