"""Argument checks of the frozen-scene (no weight gradient) entry points; they run before any device work."""
from joint_tensorf_b200 import _lib

FAKE = 1 << 20               # a non-NULL, 128-byte aligned address that is never dereferenced


def _head_bwd(lib, name, wgrads, n_max=1):
    if name == "jt_head_bwd_tc":
        return lib.jt_head_bwd_tc(FAKE, FAKE, 32, FAKE, FAKE, FAKE, FAKE, 0, n_max, 1.0, FAKE, 1, FAKE, *wgrads, 0)
    return lib.jt_wv_head_bwd_tc(FAKE, FAKE, FAKE, FAKE, FAKE, FAKE, 0, n_max, 1.0, FAKE, FAKE, *wgrads, 0)


def test_head_bwd_rejects_a_mix_of_null_and_non_null_weight_gradients():
    lib = _lib.lib()
    for name in ("jt_head_bwd_tc", "jt_wv_head_bwd_tc"):
        for i in range(7):
            mixed = [FAKE] * 7
            mixed[i] = 0
            assert _head_bwd(lib, name, mixed) == -1, (name, i)
            only = [0] * 7
            only[i] = FAKE
            assert _head_bwd(lib, name, only) == -1, (name, i)
        # all NULL (frozen head and basis_mat) or all set: accepted (n_max = 0 returns before any launch)
        assert _head_bwd(lib, name, [0] * 7, n_max=0) == 0
        assert _head_bwd(lib, name, [FAKE] * 7, n_max=0) == 0


def test_sh_bwd_needs_a_stage_only_for_the_weight_gradient():
    lib = _lib.lib()
    assert lib.jt_sh_bwd_tc(FAKE, FAKE, 32, FAKE, 0, 0, FAKE, 1, 0, FAKE, 0) == -1      # gWb without a stage
    assert lib.jt_sh_bwd_tc(FAKE, FAKE, 32, FAKE, 0, 0, FAKE, 1, 0, 0, 0) == 0          # frozen basis_mat, no stage
    assert lib.jt_sh_bwd_tc(FAKE, FAKE, 32, FAKE, 0, 0, FAKE, 1, FAKE, FAKE, 0) == 0


def test_scatter_accepts_null_factor_gradients():
    lib = _lib.lib()
    # NULL gradients select the coordinate-only walk; the other arguments are still checked
    assert lib.jt_vm_scatter_rays(1, 0, 0, FAKE, FAKE, 0, FAKE, 0, 16, FAKE, 0, 8, FAKE, FAKE, FAKE, 0, 7, 0) == -1
    assert lib.jt_vm_scatter_rays(1, FAKE, 0, FAKE, FAKE, 0, FAKE, 0, 16, FAKE, 0, 8, FAKE, FAKE, FAKE, 0, 9, 0) == -1
    assert lib.jt_vm_scatter_rays(1, FAKE, 0, FAKE, FAKE, 0, FAKE, 0, 0, FAKE, 0, 8, FAKE, FAKE, FAKE, 0, 7, 0) == 0


def test_abi_version_marks_the_null_gradient_semantics():
    assert _lib.lib().jt_version() >= 3
