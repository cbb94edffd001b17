"""The render op's C-ABI call sequence, recorded on the CPU against tests/golden/render_calls.json.

The CUDA library is replaced by a recorder: every call keeps its name and its arguments, classified with
`_lib.SIGNATURES` -- a pointer as NULL or non-NULL, an int or float by value, a ctypes array by value (a pointer
array as the NULL-ness of each entry). Device tensors are CPU tensors, so nothing is computed; what the test pins is
which kernels the forward and backward launch, in which order, with which scalar arguments and which buffers
present, plus the regions a gradient synchroniser is handed and which inputs receive a gradient. It covers every
head implementation, every backward scatter schedule and the frozen-parameter cases.

Regenerate the golden file (only when a change of the launch sequence is intended):
    python tests/test_render_call_sequence.py --regenerate
"""
import ctypes
import json
import math
import os
import sys

import pytest
import torch

from common import GOLDEN_DIR, golden_names, load_golden

from joint_tensorf_b200 import _lib, ops, render  # noqa: E402
from joint_tensorf_b200.options import default_opt  # noqa: E402
from gpu_common import forward_kwargs, module_from_golden  # noqa: E402

GOLDEN = os.path.join(GOLDEN_DIR, "render_calls.json")
STAGE_BYTES = 1 << 10


def _arg(kind, v):
    if isinstance(v, ctypes.Array):
        if v._type_ is ctypes.c_void_p:
            return [int(bool(x)) for x in v]
        return [x for x in v]
    if kind is ctypes.c_void_p:
        return "p" if v else "0"
    return float(v) if kind is ctypes.c_float else int(v)


class _Recorder:
    def __init__(self):
        self.calls = []

    def __getattr__(self, name):
        if name in ("jt_head_tc_stage_bytes", "jt_wv_stage_bytes"):
            return lambda n: STAGE_BYTES
        sig = _lib.SIGNATURES[name]

        def call(*args):
            assert len(args) == len(sig), (name, len(args), len(sig))
            self.calls.append([name] + [_arg(k, v) for k, v in zip(sig, args)])
            return 0
        return call


class _Sync:
    """Gradient synchroniser with the interface of tests/test_gpu_vm_adjoint.py::_StubSync that records its regions."""

    def __init__(self, log, per_plane=False, split21=False, reserve_sms=0):
        self.per_plane, self.split21, self.reserve_sms = per_plane, split21, reserve_sms
        self.log = log

    def _active(self):
        return True

    def use_split21(self, n_app, n_total):
        return self.split21

    def on_app_grads(self, region):
        self.log.append(["on_app_grads", region.storage_offset(), region.numel()])

    def on_rest(self, region):
        self.log.append(["on_rest", region.storage_offset(), region.numel()])


def _freeze(m, group):
    params = {"density": [*m.density_plane, *m.density_line], "app": [*m.app_plane, *m.app_line],
              "basis": [m.basis_mat.weight],
              "mlp": list(m.renderModule.parameters()) if m.renderModule is not None else []}[group]
    for p in params:
        p.requires_grad_(False)


def cases():
    """name -> (fixture, settings)."""
    out = {}
    for name in golden_names():
        heads = ["fp32"] + (["tc"] if module_from_golden(load_golden(name), "cpu").tc_available() else [])
        for head in heads:
            for mode in ("train", "no_grad", "frozen_scene"):
                out[f"{name}/{head}/{mode}"] = (name, dict(head=head, mode=mode))
    for name in ("sh_vm48", "cubic_mlp", "ndc_weakview"):
        for head in ("fp32", "tc"):
            for group in ("density", "app", "basis", "mlp"):
                if not (group == "mlp" and name == "sh_vm48"):
                    out[f"{name}/{head}/freeze_{group}"] = (name, dict(head=head, mode="train", freeze=group))
    for name, head in (("sh_vm48", "tc"), ("cubic_mlp", "tc"), ("ndc_weakview", "tc"), ("cubic_mlp", "fp32")):
        for taps in (False, True):
            out[f"{name}/{head}/bf16_taps{int(taps)}"] = (name, dict(head=head, mode="train", storage="bf16",
                                                                    bf16_backward_taps=taps))
    for name in ("sh_vm48", "cubic_mlp"):
        out[f"{name}/tc/split1"] = (name, dict(head="tc", mode="train", tc_fwd_split=1))
        out[f"{name}/tc/split1_no_grad"] = (name, dict(head="tc", mode="no_grad", tc_fwd_split=1))
    out["cubic_mlp/tc/no_fp16_no_grad"] = ("cubic_mlp", dict(head="tc", mode="no_grad", tc_infer_fp16=False))
    for name, head in (("sh_vm48", "tc"), ("cubic_mlp", "fp32"), ("ndc_weakview", "tc")):
        out[f"{name}/{head}/app_capacity"] = (name, dict(head=head, mode="train", app_capacity=2000))
    for name, head in (("sh_vm48", "tc"), ("sh", "fp32")):
        for sname, kw in (("per_plane", dict(per_plane=True)), ("split21", dict(split21=True)),
                          ("two_rank", dict()), ("reserve8", dict(reserve_sms=8))):
            out[f"{name}/{head}/sync_{sname}"] = (name, dict(head=head, mode="train", sync=kw))
        out[f"{name}/{head}/sync_frozen_scene"] = (name, dict(head=head, mode="frozen_scene", sync=dict()))
    return out


def trace(name, s):
    """The recorded calls of one forward (+ backward) on fixture `name`; the library must be patched."""
    rec = _lib._lib
    rec.calls.clear()
    g = load_golden(name)
    torch.manual_seed(0)
    m = module_from_golden(g, "cpu")
    m.head_precision = s["head"]
    m.factor_storage = s.get("storage", "fp32")
    m.bf16_backward_taps = s.get("bf16_backward_taps", False)
    m.tc_fwd_split = s.get("tc_fwd_split", 2)
    m.tc_infer_fp16 = s.get("tc_infer_fp16", True)
    m.app_capacity = s.get("app_capacity", None)
    sync_log = []
    if "sync" in s:
        m.grad_sync = _Sync(sync_log, **s["sync"])
    if s["mode"] == "frozen_scene":
        m.freeze_scene()
    if "freeze" in s:
        _freeze(m, s["freeze"])
    o = g["rays_o"].clone().requires_grad_(s["mode"] != "no_grad")
    d = g["rays_d"].clone().requires_grad_(s["mode"] != "no_grad")
    opt = default_opt(g["case"]["shading"], g["case"].get("ndc", False))
    with torch.set_grad_enabled(s["mode"] != "no_grad"):
        rgb, depth, acc = m.forward(opt, o, d, **forward_kwargs(g, "cpu"))
    n_fwd = len(rec.calls)
    grads = []
    if s["mode"] != "no_grad":
        (rgb.sum() + acc.sum()).backward()
        grads = sorted(k for k, p in m.named_parameters() if p.grad is not None)
        grads += [k for k, t in (("rays_o", o), ("rays_d", d)) if t.grad is not None]
    return dict(forward=rec.calls[:n_fwd], backward=rec.calls[n_fwd:], sync=sync_log, grads=grads)


@pytest.fixture
def recorder(monkeypatch):
    monkeypatch.setattr(_lib, "_lib", _Recorder())
    monkeypatch.setattr(ops, "_need_cuda", lambda t, name: None)
    monkeypatch.setattr(ops, "_stream", lambda: 0)
    monkeypatch.setattr(render, "_stream", lambda: 0)
    yield


def _golden():
    with open(GOLDEN) as f:
        return json.load(f)


def _mismatch(got, want, where):
    """The first place where `got` differs from `want`, or None. Floats compare to 1e-3 relative (denormals to 1e-30
    absolute): the blur taps are computed on the host by torch CPU kernels (the blur width is a mean over the grid,
    the taps an exp), whose last bits differ between machines, and the far tail of the Gaussian turns one ulp of the
    width into ~1e-5 relative. Call names, ints, pointer NULL-ness and array lengths compare exactly."""
    if isinstance(want, list) and isinstance(got, list) and len(got) == len(want):
        return next((m for i, (g, w) in enumerate(zip(got, want)) if (m := _mismatch(g, w, f"{where}[{i}]"))), None)
    if isinstance(want, float) and isinstance(got, float):
        return None if math.isclose(got, want, rel_tol=1e-3, abs_tol=1e-30) else f"{where}: {got!r} != {want!r}"
    return None if type(got) is type(want) and got == want else f"{where}: {got!r} != {want!r}"


@pytest.mark.parametrize("case", sorted(cases()))
def test_render_call_sequence(recorder, case):
    want = _golden()[case]
    got = json.loads(json.dumps(trace(*cases()[case])))
    for part in ("forward", "backward", "sync", "grads"):
        m = _mismatch(got[part], want[part], part)
        assert m is None, m[:2000]


def test_golden_covers_every_case():
    assert sorted(_golden()) == sorted(cases())


if __name__ == "__main__":
    if "--regenerate" not in sys.argv:
        sys.exit(pytest.main([__file__, "-q"]))
    mp = pytest.MonkeyPatch()
    with mp.context() as ctx:
        ctx.setattr(_lib, "_lib", _Recorder())
        ctx.setattr(ops, "_need_cuda", lambda t, name: None)
        ctx.setattr(ops, "_stream", lambda: 0)
        ctx.setattr(render, "_stream", lambda: 0)
        out = {c: trace(*s) for c, s in sorted(cases().items())}
    with open(GOLDEN, "w") as f:
        json.dump(out, f, indent=0, separators=(",", ":"), sort_keys=True)
        f.write("\n")
    print(f"wrote {len(out)} traces to {GOLDEN}")
