"""Float64 reference for the density field's gradient at points (jt_field_density_grad, compute_density_grad,
compute_normals, render_normals): the density feature through torch.nn.functional.grid_sample (bilinear,
align_corners=True, zero padding) in float64 on the CPU, feature2density, and torch.autograd.grad with respect to the
points. Also draws points that keep a margin from the cells' boundaries, where the derivative is one-sided."""
import torch
import torch.nn.functional as F

MAT_MODE = ((0, 1), (0, 2), (1, 2))
VEC_MODE = (2, 1, 0)


def fp32_lattice(aabb, inv, grid, xyz):
    """The lattice coordinate of fp32 points on each axis as the kernels compute it: u = ((p - aabb0) * inv) - 1 and
    x = (u + 1) * ((g - 1) / 2), every operation rounded to fp32 (normalize_coord, make_tap). Float64 result."""
    a0 = aabb[0].detach().float().cpu()
    inv32 = torch.as_tensor(inv).float().cpu()
    u = ((xyz.detach().float().cpu() - a0) * inv32) - 1.0
    scale = torch.tensor([0.5 * (int(g) - 1) for g in grid], dtype=torch.float32)
    return ((u + 1.0) * scale).double()


def density_and_grad(planes, lines, aabb, xyz, shift, act, inv=None, keep=None, grid=None):
    """planes: three [1,C,H,W] tensors, lines: three [1,C,L,1] (the module's logical layout); aabb [2,3]; xyz [n,3]
    points in the field's input coordinates; act "softplus" or "relu"; inv: per-axis 2 / aabb size (default: from
    aabb); keep [n] bool: points the occupancy mask keeps (the others give sigma 0, grad 0).
    grid (gx, gy, gz): evaluate the field at the lattice coordinate the fp32 kernels compute (fp32_lattice), moved
    at most 1e-9 texel into the cell its floor selects. The comparison then measures the gather's arithmetic, not the
    fp32 rounding of the coordinate normalisation that every path shares (2e-5 texel at 300^3); and on a cell face,
    where the derivative is one-sided, it takes the side the kernels take (the marcher's first sample of every ray
    lies on an aabb face). Returns float64 (sigma [n], grad [n,3]), grad = d sigma / d xyz."""
    aabb = aabb.detach().double().cpu()
    inv = (2.0 / (aabb[1] - aabb[0])) if inv is None else torch.as_tensor(inv).double().cpu()
    x = xyz.detach().double().cpu().clone()
    if grid is not None:
        g1 = torch.tensor([float(v) - 1.0 for v in grid], dtype=torch.float64)
        lat = fp32_lattice(aabb, inv, grid, xyz)
        k = torch.floor(lat)
        lat = torch.minimum(torch.maximum(lat, k + 1e-9), k + 1.0 - 1e-9)
        x = aabb[0] + (2.0 * lat / g1) / inv
    x.requires_grad_(True)
    u = (x - aabb[0]) * inv - 1.0
    n = x.shape[0]
    feat = torch.zeros((n,), dtype=torch.float64)
    for i in range(3):
        p = planes[i].detach().double().cpu()
        l = lines[i].detach().double().cpu()
        cp = u[:, list(MAT_MODE[i])].view(1, -1, 1, 2)
        cl = torch.stack((torch.zeros_like(u[:, 0]), u[:, VEC_MODE[i]]), dim=-1).view(1, -1, 1, 2)
        pc = F.grid_sample(p, cp, mode="bilinear", align_corners=True).view(-1, n)
        lc = F.grid_sample(l, cl, mode="bilinear", align_corners=True).view(-1, n)
        feat = feat + torch.sum(pc * lc, dim=0)
    sigma = F.softplus(feat + shift) if act == "softplus" else F.relu(feat + shift)
    (grad,) = torch.autograd.grad(sigma.sum(), x) if n else (torch.zeros((0, 3), dtype=torch.float64),)
    sigma, grad = sigma.detach(), grad.detach()
    if keep is not None:
        keep = keep.cpu()
        sigma = torch.where(keep, sigma, torch.zeros_like(sigma))
        grad = torch.where(keep[:, None], grad, torch.zeros_like(grad))
    return sigma, grad


def outward_normals(grad):
    """-grad / |grad| (float64), 0 where grad is 0."""
    g = grad.double()
    nrm = g.norm(dim=-1, keepdim=True)
    return torch.where(nrm > 0, -g / torch.where(nrm > 0, nrm, torch.ones_like(nrm)), torch.zeros_like(g))


def safe_points(aabb, grid, n, generator, margin=1e-3, border=True):
    """n fp32 points whose lattice coordinate on every axis is at least `margin` texels from an integer. Axis a has
    grid[a] texels (the planes and the line that sample it); with `border`, the cells -1 and grid[a] - 1 (the
    zero-padded bands just outside the first and last texel, one tap in range) are drawn too."""
    aabb = aabb.detach().double().cpu()
    inv = 2.0 / (aabb[1] - aabb[0])
    cols = []
    for a in range(3):
        g = int(grid[a])
        lo = -1 if border else 0
        hi = g if border else g - 1                          # cells lo .. hi-1
        k = torch.randint(lo, hi, (n,), generator=generator).double()
        f = margin + (1.0 - 2.0 * margin) * torch.rand((n,), generator=generator, dtype=torch.float64)
        u = 2.0 * (k + f) / (g - 1) - 1.0
        cols.append(aabb[0, a] + (u + 1.0) / inv[a])
    return torch.stack(cols, dim=-1).float()


def lattice_coords(aabb, grid, xyz, inv=None):
    """The lattice coordinate (u + 1) / 2 * (g - 1) of points on each axis (float64)."""
    aabb = aabb.detach().double().cpu()
    inv = (2.0 / (aabb[1] - aabb[0])) if inv is None else torch.as_tensor(inv).double().cpu()
    u = (xyz.detach().double().cpu() - aabb[0]) * inv - 1.0
    g = torch.tensor([float(v) for v in grid], dtype=torch.float64)
    return (u + 1.0) / 2.0 * (g - 1.0)
