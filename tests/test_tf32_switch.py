"""CPU: when the 1x1-convolution GEMMs run one TF32 pass, the C ABI of PM_F32_TF32, and the one-pass precision bound
(emulated on the host) against the error it has to tell apart."""
import contextlib
import ctypes
import subprocess
import sys

import pytest
import torch

from test_gpu_tf32_gemm import bias_tol, tf32_bound
from test_gpu_gemm_kernels import tf32_rn, tf32_trunc

PM_F32, PM_BF16, PM_F32_TF32 = 0, 1, 2
PM_ERR_DTYPE, PM_ERR_ALIGN = -2, -6


@contextlib.contextmanager
def tf32_flags(matmul, cudnn):
    old = (torch.backends.cuda.matmul.allow_tf32, torch.backends.cudnn.allow_tf32)
    torch.backends.cuda.matmul.allow_tf32, torch.backends.cudnn.allow_tf32 = matmul, cudnn
    try:
        yield
    finally:
        torch.backends.cuda.matmul.allow_tf32, torch.backends.cudnn.allow_tf32 = old


# ------------------------------------------------------------------------------------------------ the switch
@pytest.mark.parametrize("matmul,cudnn", [(False, False), (True, False), (False, True), (True, True)])
def test_tf32_needs_both_switches(matmul, cudnn):
    from pinthememory_b200 import capi

    with tf32_flags(matmul, cudnn):
        assert capi.tf32() is (matmul and cudnn)


@pytest.mark.parametrize("precision,want", [("highest", False), ("high", True), ("medium", True)])
def test_float32_matmul_precision_sets_the_matmul_switch(precision, want):
    from pinthememory_b200 import capi

    old = torch.get_float32_matmul_precision()
    try:
        with tf32_flags(False, True):
            torch.set_float32_matmul_precision(precision)
            assert capi.tf32() is want
    finally:
        torch.set_float32_matmul_precision(old)


def test_default_is_off():
    """torch's defaults (matmul off, cuDNN on) keep the 3xTF32 products: checked in a fresh interpreter."""
    code = ("import torch; from pinthememory_b200 import capi; "
            "assert torch.backends.cudnn.allow_tf32 and not torch.backends.cuda.matmul.allow_tf32; "
            "assert capi.tf32() is False; print('ok')")
    import os

    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    r = subprocess.run([sys.executable, "-c", code], cwd=root, capture_output=True, text=True, timeout=300)
    assert r.returncode == 0 and r.stdout.strip() == "ok", r.stderr


def test_operands_carry_their_mode():
    """The operands of a one-pass GEMM have no lo part; the dtype code of a GEMM follows its operands."""
    from pinthememory_b200 import capi

    f, b = torch.empty(4, 8), torch.empty(4, 8, dtype=torch.bfloat16)
    assert capi.operands_tf32((f, None)) and not capi.operands_tf32((f, f)) and not capi.operands_tf32((b, None))
    assert capi._gemm_code(f, None) == PM_F32_TF32 and capi._gemm_code(f, f) == PM_F32 and capi._gemm_code(b, None) == PM_BF16


# ------------------------------------------------------------------------------------------------ the C ABI
def test_tf32_code_only_on_the_conv1x1_entries():
    """PM_F32_TF32 reaches the alignment check of every pm_conv1x1_* entry (misaligned pointers, so nothing runs) and
    its size queries answer as for PM_F32; other entries reject it."""
    from pinthememory_b200 import capi

    lib = capi.load()
    a16, bad = ctypes.c_void_p(16), ctypes.c_void_p(8)
    B, K, M, hw = 2, 64, 96, 4
    assert lib.pm_conv1x1_fwd(bad, a16, None, a16, None, B, K, M, hw, 0, PM_F32_TF32, None) == PM_ERR_ALIGN
    assert lib.pm_conv1x1_fwd_affine(bad, a16, None, a16, a16, a16, 1, B, K, M, hw, PM_F32_TF32, None) == PM_ERR_ALIGN
    assert lib.pm_conv1x1_wgrad(bad, a16, a16, a16, B, M, K, hw, 0, PM_F32_TF32, None) == PM_ERR_ALIGN
    assert lib.pm_conv1x1_dgrad_bnbwd(bad, a16, a16, None, a16, a16, a16, a16, a16, a16, a16, a16, 1, 1, B, K, M, hw,
                                      PM_F32_TF32, None) == PM_ERR_ALIGN
    assert lib.pm_conv1x1_fwd_ordered(bad, a16, None, a16, a16, a16, B, K, M, hw, PM_F32_TF32, None) == PM_ERR_ALIGN
    for b_, m_, hw_ in ((2, 96, 4), (8, 256, 9216), (5, 160, 4864)):
        assert lib.pm_conv1x1_stats_scratch_bytes(b_, m_, hw_, PM_F32_TF32) == lib.pm_conv1x1_stats_scratch_bytes(b_, m_, hw_, PM_F32)
        assert (lib.pm_conv1x1_wgrad_workspace_floats(b_, m_, 288, hw_, PM_F32_TF32)
                == lib.pm_conv1x1_wgrad_workspace_floats(b_, m_, 288, hw_, PM_F32))
    assert lib.pm_conv1x1_stats_scratch_bytes(2, 96, 4, 3) == PM_ERR_DTYPE
    # the prep entries need no lo buffer in this mode (a zero-sized weight stops them before any launch)
    assert lib.pm_conv1x1_prep(a16, 0, 8, 0, PM_F32_TF32, a16, None, None) == -5
    assert lib.pm_conv1x1_prep(a16, 0, 8, 0, PM_F32, a16, None, None) == -1
    assert lib.pm_conv1x1_prep_both(a16, 0, 8, PM_F32_TF32, a16, None, a16, None, None, 0, None) == -5
    # every other entry keeps rejecting it
    assert lib.pm_read_fwd(a16, a16, None, None, a16, a16, a16, None, 1, 256, 4, 4, 19, PM_F32_TF32, None) == PM_ERR_DTYPE
    assert lib.pm_bn_apply(a16, a16, a16, a16, a16, None, a16, None, 0, 2, 64, 16, PM_F32_TF32, None) == PM_ERR_DTYPE
    assert b"PM_F32_TF32" in lib.pm_status_string(PM_ERR_DTYPE)


# ------------------------------------------------------------------------ the precision bound, emulated on the host
def _one_pass(A, x, trunc_x):
    """float64 emulation of a one-pass product with A rounded to nearest TF32 and x rounded or truncated."""
    xr = tf32_trunc(x) if trunc_x else tf32_rn(x)
    return tf32_rn(A).double() @ xr.double()


@pytest.mark.parametrize("K", [8, 40, 288, 1024])
def test_bound_accepts_round_to_nearest(K):
    """Gaussian data with 2^-8..2^8 row / column scales: rounded operands stay inside the element-wise bound."""
    gen = torch.Generator().manual_seed(K)
    A = torch.randn(64, K, generator=gen) * torch.exp2(torch.randint(-8, 9, (64, 1), generator=gen).float())
    x = torch.randn(K, 512, generator=gen) * torch.exp2(torch.randint(-8, 9, (K, 1), generator=gen).float())
    y64 = A.double() @ x.double()
    err = (_one_pass(A, x, False) - y64).abs()
    assert float((err / tf32_bound(K, A.double().abs() @ x.double().abs())).max()) <= 1.0


@pytest.mark.parametrize("K", [96, 288])
def test_bias_check_rejects_truncated_activations(K):
    """All-positive operands: rounded activations have a mean signed relative error inside bias_tol(K) (a few percent of
    it in float64), activations truncated as the tensor core truncates an fp32 container are shifted far outside it."""
    gen = torch.Generator().manual_seed(100 + K)
    A = 0.5 + 1.5 * torch.rand(256, K, generator=gen)
    x = 0.5 + 1.5 * torch.rand(K, 2048, generator=gen)
    y64 = A.double() @ x.double()
    rn = float(((_one_pass(A, x, False) - y64) / y64).mean())
    tr = float(((_one_pass(A, x, True) - y64) / y64).mean())
    assert abs(rn) <= bias_tol(K), rn
    assert tr < -3 * bias_tol(K), (tr, bias_tol(K))
