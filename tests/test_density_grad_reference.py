"""CPU checks of the float64 density-gradient reference (tests/density_grad_reference.py)."""
import torch

from density_grad_reference import density_and_grad, lattice_coords, outward_normals, safe_points


def _field(grid, comps, seed):
    g = torch.Generator().manual_seed(seed)
    mat = ((0, 1), (0, 2), (1, 2))
    vec = (2, 1, 0)
    planes = [torch.randn((1, comps, grid[mat[i][1]], grid[mat[i][0]]), generator=g, dtype=torch.float64)
              for i in range(3)]
    lines = [torch.randn((1, comps, grid[vec[i]], 1), generator=g, dtype=torch.float64) for i in range(3)]
    return planes, lines


def test_gradient_matches_central_differences():
    grid = (7, 5, 9)
    planes, lines = _field(grid, 4, 0)
    aabb = torch.tensor([[-1.0, -0.5, -2.0], [1.5, 0.5, 1.0]])
    gen = torch.Generator().manual_seed(1)
    xyz = safe_points(aabb, grid, 300, gen, margin=1e-2).double()
    for act, shift in (("softplus", -1.0), ("relu", 0.5)):
        sigma, grad = density_and_grad(planes, lines, aabb, xyz, shift, act)
        h = 1e-7
        for a in range(3):
            d = torch.zeros(3, dtype=torch.float64)
            d[a] = h
            sp, _ = density_and_grad(planes, lines, aabb, xyz + d, shift, act)
            sm, _ = density_and_grad(planes, lines, aabb, xyz - d, shift, act)
            fd = (sp - sm) / (2 * h)
            # relu: skip points whose pre-activation is within the step of the kink
            ok = (sigma > 1e-5) | (act == "softplus")
            assert torch.allclose(grad[ok, a], fd[ok], rtol=1e-5, atol=1e-6 * float(grad.abs().max()))


def test_points_keep_their_margin_and_reach_the_border_band():
    grid = (11, 6, 20)
    aabb = torch.tensor([[-1.0, -1.0, -0.3], [1.0, 2.0, 0.3]])
    xyz = safe_points(aabb, grid, 4000, torch.Generator().manual_seed(2), margin=1e-3)
    c = lattice_coords(aabb, grid, xyz)
    frac = c - torch.floor(c)
    assert float(torch.minimum(frac, 1 - frac).min()) > 0.9e-3
    for a in range(3):
        assert float(c[:, a].min()) < 0 and float(c[:, a].max()) > grid[a] - 1     # both zero-padded bands


def test_outside_points_and_mask_give_zero():
    grid = (6, 6, 6)
    planes, lines = _field(grid, 4, 3)
    aabb = torch.tensor([[-1.0, -1.0, -1.0], [1.0, 1.0, 1.0]])
    xyz = torch.tensor([[3.0, 0.0, 0.0], [0.1, 0.2, 0.3], [0.0, -5.0, 0.0]])
    keep = torch.tensor([True, False, True])
    sigma, grad = density_and_grad(planes, lines, aabb, xyz, 0.0, "relu", keep=keep)
    assert float(sigma.abs().sum()) == 0.0 and float(grad.abs().sum()) == 0.0
    n = outward_normals(torch.tensor([[0.0, 0.0, 0.0], [0.0, 3.0, -4.0]]))
    assert torch.equal(n[0], torch.zeros(3, dtype=torch.float64))
    assert torch.allclose(n[1], torch.tensor([0.0, -0.6, 0.8], dtype=torch.float64))


def test_grid_option_evaluates_inside_the_fp32_cell():
    """A point on a lattice face: with `grid`, the derivative is the one-sided one of the cell fp32 selects, and
    sigma is evaluated at the fp32 lattice coordinate."""
    grid = (5, 5, 5)
    planes, lines = _field(grid, 4, 4)
    aabb = torch.tensor([[-1.0, -1.0, -1.0], [1.0, 1.0, 1.0]])
    xyz = torch.tensor([[-1.0, 0.1, 0.2], [0.0, 0.3, -0.4]])          # x on the first texel, x on texel 2
    _, g_face = density_and_grad(planes, lines, aabb, xyz, 0.5, "softplus", grid=grid)
    _, g_in = density_and_grad(planes, lines, aabb, xyz + torch.tensor([1e-6, 0.0, 0.0]), 0.5, "softplus")
    assert torch.allclose(g_face, g_in, rtol=1e-4, atol=1e-9)
