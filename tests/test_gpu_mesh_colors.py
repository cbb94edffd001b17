"""Colour of the field at arbitrary points (B200_VMSplit.compute_rgb) against the oracle's app_feature + shading
head, and the coloured mesh export (extract_mesh / export_mesh with colors=True)."""
import numpy as np
import pytest
import torch

import joint_tensorf_b200 as jt
from common import field_from_golden, golden_names, load_golden, rel_err
from gpu_common import default_opt, forward_kwargs, module_from_golden, record_err
from joint_tensorf_b200 import ops
from oracle import vm_oracle as vo

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
TOL = 1e-4               # strict fp32 head and the tensor-core heads with the hi/lo bf16 split
TOL_FP16 = 1e-3          # MLP_Fea tensor-core head, no-grad fp16 operand tiles (tc_infer_fp16)
TOL_BF16 = 2e-2          # bf16 factor storage, relative


def _points(m, n, seed, n_out=64):
    """n world points inside the aabb, n_out outside it, and non-unit view directions."""
    g = torch.Generator().manual_seed(seed)
    lo, hi = m.aabb[0].cpu(), m.aabb[1].cpu()
    xyz = lo + (hi - lo) * torch.rand(n, 3, generator=g)
    out = lo + (hi - lo) * (torch.rand(n_out, 3, generator=g) * 1.6 - 0.3)
    out[:, 0] = torch.where(torch.rand(n_out, generator=g) < 0.5, lo[0] - 0.2, hi[0] + 0.2)
    d = torch.randn(n + n_out, 3, generator=g)
    d = d / d.norm(dim=1, keepdim=True) * (0.5 + torch.rand(n + n_out, 1, generator=g))
    return torch.cat([xyz, out]).to(DEV), d.to(DEV)


def _oracle_rgb(field, m, xyz, dirs, taps=None):
    fc = vo.grid_constants(field.aabb, field.grid, field.step_ratio)
    u = m.normalize_coord(xyz).cpu()
    with torch.no_grad():
        return vo._SHADERS[field.shading](field, dirs.cpu(), vo.app_feature(field, fc, u, taps))


def _module_field(m):
    """Oracle field holding the module's current parameters."""
    params = {k: v.detach().cpu() for k, v in m.state_dict().items() if not k.startswith("alphaMask")}
    return vo.Field(aabb=m.aabb.cpu(), grid=list(m._grid), params=params, shading=m.shadingMode, view_pe=m.view_pe,
                    fea_pe=m.fea_pe)


def _variants(m):
    """(name, head_precision, tc_fwd_split, tc_infer_fp16, factor_storage, tolerance, relative)"""
    out = [("fp32", "fp32", 2, True, "fp32", TOL, False), ("bf16", "auto", 2, True, "bf16", TOL_BF16, True)]
    if m.tc_available():
        out.append(("tc_split2", "tc", 2, False, "fp32", TOL, False))
        if m.shadingMode == "MLP_Fea":
            out.append(("tc_fp16", "tc", 2, True, "fp32", TOL_FP16, False))
    return out


def _set(m, head, split, fp16, storage):
    m.head_precision, m.tc_fwd_split, m.tc_infer_fp16, m.factor_storage = head, split, fp16, storage


@pytest.mark.parametrize("name", golden_names())
def test_compute_rgb_matches_the_oracle(name):
    g = load_golden(name)
    m = module_from_golden(g, DEV)
    field = field_from_golden(g, requires_grad=False)
    xyz, dirs = _points(m, 3000, 1)
    taps = None
    if g["case"]["blur"] is not None:           # a forward caches the colour kernel; compute_rgb blurs with it
        with torch.no_grad():
            m.forward(default_opt(g["case"]["shading"], g["case"].get("ndc", False)), g["rays_o"].to(DEV),
                      g["rays_d"].to(DEV), **forward_kwargs(g, DEV))
        fc = vo.grid_constants(field.aabb, field.grid, field.step_ratio)
        taps = vo.blur_taps(fc, "uniform-gaussian", g["case"]["blur"][1], 64)
    ref = _oracle_rgb(field, m, xyz, dirs, taps)
    for tag, head, split, fp16, storage, tol, relative in _variants(m):
        _set(m, head, split, fp16, storage)
        rgb = m.compute_rgb(xyz, dirs)
        assert rgb.shape == (xyz.shape[0], 3) and rgb.dtype == torch.float32
        err = rel_err(rgb.cpu(), ref) if relative else float((rgb.cpu().double() - ref.double()).abs().max())
        record_err(f"compute_rgb[{name},{tag}]", err=err, tol=tol)
        assert err <= tol, (tag, err)


@pytest.mark.parametrize("name", ["cubic_mlp", "sh_vm48", "ndc_weakview"])
def test_compute_rgb_rows_do_not_depend_on_chunking_or_order(name):
    g = load_golden(name)
    m = module_from_golden(g, DEV)
    xyz, dirs = _points(m, 5000, 2)
    perm = torch.randperm(xyz.shape[0], generator=torch.Generator().manual_seed(3)).to(DEV)
    for _, head, split, fp16, storage, _, _ in _variants(m):
        _set(m, head, split, fp16, storage)
        m._RGB_CHUNK = 1 << 20
        whole = m.compute_rgb(xyz, dirs)
        assert torch.equal(m.compute_rgb(xyz[perm], dirs[perm]), whole[perm])
        m._RGB_CHUNK = 1000                      # chunk boundaries inside the tensor-core heads' 128-row tiles
        assert torch.equal(m.compute_rgb(xyz, dirs), whole)
        assert torch.equal(m.compute_rgb(xyz[:1], dirs[:1]), whole[:1])
    m._RGB_CHUNK = 1 << 20
    # shapes: [..., 3] points, one [3] direction for all of them
    d1 = dirs[0]
    assert torch.equal(m.compute_rgb(xyz.view(8, -1, 3), d1),
                       m.compute_rgb(xyz, d1.expand(xyz.shape[0], 3)).view(8, -1, 3))
    assert m.compute_rgb(xyz[:0], dirs[:0]).shape == (0, 3)


def test_compute_rgb_rejects_what_forward_rejects():
    m = module_from_golden(load_golden("sh"), DEV)           # 3 x 12 components: no tensor-core head
    xyz, dirs = _points(m, 10, 0)
    m.head_precision = "tc"
    with pytest.raises(jt._lib.JtError, match="head='tc' needs"):
        m.compute_rgb(xyz, dirs)
    m.head_precision, m.factor_storage = "auto", "fp16"
    with pytest.raises(jt._lib.JtError, match="factor_storage"):
        m.compute_rgb(xyz, dirs)
    m.factor_storage = "fp32"
    with pytest.raises(jt._lib.JtError):
        m.compute_rgb(xyz, dirs[:5])
    with pytest.raises(jt._lib.JtError):
        m.compute_rgb(xyz.cpu(), dirs)


# ------------------------------------------------------------------ coloured export
def _median_level(m):
    flat = m._dense_alpha_zyx(m._grid).reshape(-1).sort().values
    return float(flat[int(0.5 * (flat.numel() - 1))])


def _assert_coloured_mesh(m, level, grid=None):
    verts0, faces0 = m.extract_mesh(level, grid)
    verts, faces, normals, rgb = m.extract_mesh(level, grid, colors=True)
    g = m._grid if grid is None else grid
    _, _, n_op = ops.marching_cubes(m._dense_alpha_zyx(g), level, m._dense_tables(g), m._h_aabb, normals=True)
    assert torch.equal(verts, verts0) and torch.equal(faces, faces0) and faces.shape[0] > 0
    assert torch.equal(normals, n_op)
    assert torch.equal(rgb, m.compute_rgb(verts, -normals))
    return verts, faces, normals, rgb


def _today_ply(verts, faces):
    """The colors=False PLY as written before colours existed."""
    v = verts.cpu().numpy().astype("<f4")
    f = np.empty((faces.shape[0],), dtype=[("n", "u1"), ("i", "<i4", (3,))])
    f["n"] = 3
    f["i"] = faces.cpu().numpy()
    header = ("ply\nformat binary_little_endian 1.0\n"
              f"element vertex {v.shape[0]}\nproperty float x\nproperty float y\nproperty float z\n"
              f"element face {f.shape[0]}\nproperty list uchar int vertex_indices\nend_header\n")
    return header.encode("ascii") + v.tobytes() + f.tobytes()


def _read_coloured_ply(path):
    raw = open(path, "rb").read()
    head, body = raw.split(b"end_header\n", 1)
    lines = head.decode("ascii").splitlines()
    assert lines[:2] == ["ply", "format binary_little_endian 1.0"]
    nv = int(lines[2].split()[2])
    props = [tuple(l.split()[1:]) for l in lines[3:] if l.startswith("property") and "list" not in l]
    assert props == [("float", "x"), ("float", "y"), ("float", "z"), ("float", "nx"), ("float", "ny"),
                     ("float", "nz"), ("uchar", "red"), ("uchar", "green"), ("uchar", "blue")]
    nf = int([l for l in lines if l.startswith("element face")][0].split()[2])
    assert lines[-1] == "property list uchar int vertex_indices"
    vt = np.dtype([("x", "<f4"), ("y", "<f4"), ("z", "<f4"), ("nx", "<f4"), ("ny", "<f4"), ("nz", "<f4"),
                   ("red", "u1"), ("green", "u1"), ("blue", "u1")])
    v = np.frombuffer(body[:vt.itemsize * nv], dtype=vt)
    f = np.frombuffer(body[vt.itemsize * nv:], dtype=[("n", "u1"), ("i", "<i4", (3,))])
    assert f.shape[0] == nf and (f["n"] == 3).all()
    return v, f["i"]


@pytest.mark.parametrize("name", ["cubic_mlp", "sh_vm48", "ndc_weakview_blur", "alpha_mask"])
def test_coloured_export_on_golden_fields_with_mask_and_shrink(name, tmp_path):
    g = load_golden(name)
    m = module_from_golden(g, DEV)
    if g["case"]["blur"] is not None:
        with torch.no_grad():
            m.forward(default_opt(g["case"]["shading"], g["case"].get("ndc", False)), g["rays_o"].to(DEV),
                      g["rays_d"].to(DEV), **forward_kwargs(g, DEV))
    level = _median_level(m)
    _assert_coloured_mesh(m, level)
    _assert_coloured_mesh(m, level, [19, 23, 17])
    if name == "cubic_mlp":
        flat = m._dense_alpha_zyx(m._grid).reshape(-1).sort().values
        m.alphaMask_thres = float(flat[int(0.99 * (flat.numel() - 1))])
        m.updateAlphaMask(m._grid)
        _assert_coloured_mesh(m, level)
        m.shrink(m.aabb * 0.6)
        _assert_coloured_mesh(m, level)
    # PLY round trip
    verts, faces, normals, rgb = m.extract_mesh(level, colors=True)
    path = str(tmp_path / "c.ply")
    assert m.export_mesh(path, level, colors=True) == (verts.shape[0], faces.shape[0])
    v, f = _read_coloured_ply(path)
    assert np.array_equal(np.stack([v["x"], v["y"], v["z"]], 1), verts.cpu().numpy())
    assert np.array_equal(np.stack([v["nx"], v["ny"], v["nz"]], 1), normals.cpu().numpy())
    q = np.floor(np.clip(rgb.cpu().numpy(), 0, 1).astype(np.float32) * np.float32(255) + np.float32(0.5))
    assert np.array_equal(np.stack([v["red"], v["green"], v["blue"]], 1), q.astype(np.uint8))
    assert np.array_equal(f, faces.cpu().numpy())
    plain = str(tmp_path / "p.ply")
    assert m.export_mesh(plain, level) == (verts.shape[0], faces.shape[0])
    assert open(plain, "rb").read() == _today_ply(verts, faces)


@pytest.mark.parametrize("wl", ["cfg2_sh", "cfg2", "cfg4"])
def test_full_size_coloured_mesh_against_the_oracle(wl):
    kw, _ = jt.synth.config(wl)
    kw = dict(kw)
    torch.manual_seed(0)
    m = jt.B200_VMSplit(torch.tensor(kw.pop("aabb")), kw.pop("gridSize"), DEV, **kw)
    flat = m._dense_alpha_zyx(m._grid).reshape(-1).sort().values
    level = float(flat[int(0.99 * (flat.numel() - 1))])
    del flat
    verts, faces, normals, rgb = m.extract_mesh(level, colors=True)
    again = m.extract_mesh(level, colors=True)
    assert all(torch.equal(a, b) for a, b in zip((verts, faces, normals, rgb), again))
    del again
    sel = torch.randperm(verts.shape[0], generator=torch.Generator().manual_seed(0))[:4096].to(DEV)
    ref = _oracle_rgb(_module_field(m), m, verts[sel], -normals[sel])
    err = float((rgb[sel].cpu().double() - ref.double()).abs().max())
    tol = TOL_FP16 if (m.shadingMode == "MLP_Fea" and m.tc_available() and m.tc_infer_fp16) else TOL
    record_err(f"mesh_rgb_full_size[{wl}]", err=err, tol=tol, V=verts.shape[0], F=faces.shape[0])
    assert err <= tol, err
    length = normals.norm(dim=1)
    assert float((length[length > 0] - 1).abs().max()) <= 1e-6
