"""The one-pass TF32 GEMMs of csrc/pm_gemm.cu (dtype PM_F32_TF32) kernel by kernel, against float64 torch on the device.

Same layout as test_gpu_gemm_kernels.py, whose case tables, guard bands and helpers this file reuses. Three tiers:
  * exact: integer operands below 2^11 in magnitude (exact in TF32, so rounding to nearest must leave them alone) with
    partial sums below 2^24 -- outputs, statistics and weight gradients equal float64 bit for bit;
  * precision: element-wise, half a TF32 ulp on each operand plus the fp32 accumulation of the 3-pass bound (tf32_bound);
  * bias: all-positive operands, where the mean signed relative error shows whether activations were rounded to nearest
    (zero mean) or left to the tensor core, which truncates an fp32 container (a shift of a few 1e-4 per operand).
`test_tf32_routing` pins the instantiations every case launches and that all new ones are reached."""
import contextlib
import re

import pytest
import torch

from golden_util import rel_l2
from test_gpu_gemm_kernels import (DGRAD_CASES, ELEM_C, ELEM_K0, FP32_CASES, MODES, WGRAD_ACCUMULATE, WGRAD_FP32, Guarded,
                                   _bn_coefficients, _gemm_exact_inputs, _ints, _lib, _ok, _sparse_signs, _stream,
                                   deterministic_flag, scaled_gaussian, wgrad_chunks)

gpu = pytest.mark.gpu

PM_F32, PM_F32_TF32 = 0, 2

# one TF32 pass: each operand rounded to nearest TF32 is off by at most half an ulp, 2^-11 relative, so a product by
# 2^-10 + 2^-22; the K fp32 additions are those of the 3-pass bound (ELEM_C, ELEM_K0 of test_gpu_gemm_kernels.py)
TF32_PRODUCT = 2.0 ** -10 + 2.0 ** -22


def tf32_bound(K, mag):
    """Element-wise bound on |y - y64| of a one-pass TF32 product with K-long dot products; mag = |A|.|x| in float64."""
    return (TF32_PRODUCT + ELEM_C * (K + ELEM_K0) * 2.0 ** -24) * mag


def bias_tol(K):
    """|mean signed relative error| allowed on all-positive operands: every fp32 addition of the accumulation rounding
    down by a full ulp (its expectation is half that). Truncated activations shift the mean by ~3e-4 per operand."""
    return K * 2.0 ** -23


# input gradient with the BatchNorm backward: the module's shapes plus the wide tiles with a single row tile
TF32_DGRAD_CASES = dict(DGRAD_CASES, wide_mt1=(8, 64, 96, 9216))


def _prep1(A, transpose=False):
    """A rounded to nearest TF32 through capi (the one-pass operand: no lo part)."""
    from pinthememory_b200 import capi

    hi, lo = capi.conv1x1_prep(A.contiguous(), transpose, torch.float32, tf32=True)
    assert lo is None
    return hi


def _run_fwd1(mode, x, hi, B, K, M, hw, y0=None, scale=None, shift=None):
    """One PM_F32_TF32 call of the entry `mode` exercises, on guarded buffers (A_lo = NULL). Returns (y, stats or None)."""
    lib = _lib()
    y = Guarded(B * M * hw, torch.float32, fill=None if mode == "accumulate" else float("nan"))
    if mode == "accumulate":
        y.t.copy_(y0.flatten())
        y.ref = y.buf.clone()
    stats = scratch = None
    if mode in ("plain", "accumulate", "stats"):
        if mode == "stats":
            stats = Guarded(2 * M, torch.float64, fill=0.0)
        rc = lib.pm_conv1x1_fwd(x.data_ptr(), hi.data_ptr(), None, y.t.data_ptr(),
                                None if stats is None else stats.t.data_ptr(), B, K, M, hw, int(mode == "accumulate"),
                                PM_F32_TF32, _stream())
        _ok(rc, "pm_conv1x1_fwd")
    elif mode == "stats_ordered":
        stats = Guarded(2 * M, torch.float64, fill=0.0)
        nbytes = lib.pm_conv1x1_stats_scratch_bytes(B, M, hw, PM_F32_TF32)
        assert nbytes == lib.pm_conv1x1_stats_scratch_bytes(B, M, hw, PM_F32)   # same tiles, same CTAs
        scratch = Guarded(nbytes // 8, torch.float64)
        rc = lib.pm_conv1x1_fwd_ordered(x.data_ptr(), hi.data_ptr(), None, y.t.data_ptr(), stats.t.data_ptr(),
                                        scratch.t.data_ptr(), B, K, M, hw, PM_F32_TF32, _stream())
        _ok(rc, "pm_conv1x1_fwd_ordered")
    else:
        rc = lib.pm_conv1x1_fwd_affine(x.data_ptr(), hi.data_ptr(), None, y.t.data_ptr(), scale.data_ptr(), shift.data_ptr(),
                                       int(mode == "affine_relu"), B, K, M, hw, PM_F32_TF32, _stream())
        _ok(rc, "pm_conv1x1_fwd_affine")
    torch.cuda.synchronize()
    y.check("y")
    if stats is not None:
        stats.check("stats")
    if scratch is not None:
        scratch.check("ordered-statistics scratch")
    return y.t.view(B, M, hw), (None if stats is None else stats.t.clone())


# ================================================================================== forward / input gradient
@gpu
@pytest.mark.parametrize("mode", MODES)
@pytest.mark.parametrize("name,case", list(FP32_CASES.items()), ids=lambda v: v if isinstance(v, str) else "")
def test_tf32_fwd_exact(name, case, mode):
    """Exact tier: every entry equals the float64 product bit for bit. The plain mode uses activations of 11 significant
    bits (|x| <= 2047): the in-place rounding must keep all of them, as it must keep every TF32 value."""
    B, K, M, hw = case
    gen = torch.Generator(device="cuda").manual_seed(7000 + 7 * K + M + hw)
    if mode == "plain":
        A, x = _sparse_signs(M, K, gen), _ints((B, K, hw), -2047, 2047, gen)      # |y| <= 16 * 2047
        A[0] = 0
    else:
        A, x = _gemm_exact_inputs(torch.float32, B, K, M, hw, mode, gen)
    hi = _prep1(A)
    y64 = torch.matmul(A.double(), x.double())
    y0 = scale = shift = None
    if mode == "accumulate":
        y0 = _ints((B, M, hw), -1000, 1000, gen)
        y64 = y64 + y0.double()
    if mode.startswith("affine"):
        scale = torch.exp2(torch.randint(-3, 4, (M,), generator=gen, device="cuda").float())
        shift = _ints((M,), -8, 8, gen)
        y64 = y64 * scale.double().view(M, 1) + shift.double().view(M, 1)
        if mode == "affine_relu":
            y64 = y64.clamp_min(0.0)
    y, stats = _run_fwd1(mode, x, hi, B, K, M, hw, y0, scale, shift)
    bad = y != y64.float()
    assert not bool(bad.any()), "%d of %d elements differ; first at (b, row, px) = %s" % (
        int(bad.sum()), bad.numel(), tuple(bad.nonzero()[0].tolist()))
    if stats is not None:
        ref = torch.cat([y64.sum((0, 2)), (y64 * y64).sum((0, 2))])
        assert torch.equal(stats, ref), "statistics differ at %s" % (stats != ref).nonzero().flatten()[:8].tolist()
    if mode == "stats_ordered":
        y2, stats2 = _run_fwd1(mode, x, hi, B, K, M, hw)
        assert torch.equal(y2.view(torch.int32), y.view(torch.int32)), "output not reproducible"
        assert torch.equal(stats2.view(torch.int64), stats.view(torch.int64)), "statistics not reproducible"


@gpu
@pytest.mark.parametrize("name,case", list(FP32_CASES.items()), ids=lambda v: v if isinstance(v, str) else "")
def test_tf32_fwd_precision(name, case):
    """Precision tier: Gaussian data with 2^-8..2^8 scales on rows of A and channels of x, element-wise bound."""
    B, K, M, hw = case
    gen = torch.Generator(device="cuda").manual_seed(8000 + 7 * K + M + hw)
    A = scaled_gaussian((M, K), 0, gen, "cuda")
    x = scaled_gaussian((B, K, hw), 1, gen, "cuda")
    y, _ = _run_fwd1("plain", x, _prep1(A), B, K, M, hw)
    y64 = torch.matmul(A.double(), x.double())
    ratio = float(((y.double() - y64).abs() / tf32_bound(K, torch.matmul(A.double().abs(), x.double().abs()))
                   .clamp_min(1e-300)).max())
    print("tf32 fwd %s K=%d rel_l2=%.3e elem/bound=%.3f" % (name, K, rel_l2(y, y64), ratio))
    assert ratio <= 1.0, "element-wise bound exceeded by %.2fx" % ratio


def _positive(shape, gen):
    """Uniform in [0.5, 2): mantissas spread over the whole binade, so truncation would shift every operand."""
    return (0.5 + 1.5 * torch.rand(*shape, generator=gen, device="cuda")).contiguous()


@gpu
def test_tf32_fwd_unbiased():
    """Bias test at K = 288 (the folded output convolution): all-positive operands, mean signed relative error ~ 0."""
    B, K, M, hw = 8, 288, 256, 9216
    gen = torch.Generator(device="cuda").manual_seed(8800)
    A, x = _positive((M, K), gen), _positive((B, K, hw), gen)
    y, _ = _run_fwd1("plain", x, _prep1(A), B, K, M, hw)
    y64 = torch.matmul(A.double(), x.double())
    bias = float(((y.double() - y64) / y64).mean())
    print("tf32 fwd K=%d mean signed relative error %.3e (tol %.1e)" % (K, bias, bias_tol(K)))
    assert abs(bias) <= bias_tol(K), bias


# ============================================================================================ weight gradient
def _run_wgrad1(dY, X, B, M, N, hw, dW0=None):
    lib = _lib()
    nws = lib.pm_conv1x1_wgrad_workspace_floats(B, M, N, hw, PM_F32_TF32)
    assert nws == lib.pm_conv1x1_wgrad_workspace_floats(B, M, N, hw, PM_F32)
    ws = Guarded(nws, torch.float32)
    dW = Guarded(M * N, torch.float32, fill=None if dW0 is not None else float("nan"))
    if dW0 is not None:
        dW.t.copy_(dW0.flatten())
        dW.ref = dW.buf.clone()
    rc = lib.pm_conv1x1_wgrad(dY.data_ptr(), X.data_ptr(), ws.t.data_ptr(), dW.t.data_ptr(), B, M, N, hw,
                              int(dW0 is not None), PM_F32_TF32, _stream())
    _ok(rc, "pm_conv1x1_wgrad")
    torch.cuda.synchronize()
    ws.check("workspace", scratch=True)
    dW.check("dW")
    return dW.t.view(M, N).clone()


def _wgrad_ref(dY, X):
    return torch.einsum("bmp,bnp->mn", dY.double(), X.double())


@gpu
@pytest.mark.parametrize("name,case", list(WGRAD_FP32.items()), ids=lambda v: v if isinstance(v, str) else "")
def test_tf32_wgrad_exact(name, case):
    """Exact tier: integer operands, |dW| <= 49 B hw < 2^24; bitwise equal to float64, and to itself on a second run."""
    B, M, N, hw = case
    gen = torch.Generator(device="cuda").manual_seed(9000 + M + N + hw)
    dY, X = _ints((B, M, hw), -7, 7, gen), _ints((B, N, hw), -7, 7, gen)
    dY[:, 0] = 0
    ref = _wgrad_ref(dY, X)
    dW = _run_wgrad1(dY, X, B, M, N, hw)
    bad = dW.double() != ref
    assert not bool(bad.any()), "%d elements differ, first at %s" % (int(bad.sum()), bad.nonzero()[0].tolist())
    assert torch.equal(_run_wgrad1(dY, X, B, M, N, hw).view(torch.int32), dW.view(torch.int32)), "not reproducible"
    if (torch.float32, name) in WGRAD_ACCUMULATE:
        dW0 = _ints((M, N), -1000, 1000, gen)
        assert torch.equal(_run_wgrad1(dY, X, B, M, N, hw, dW0=dW0).double(), ref + dW0.double()), "accumulate"


@gpu
@pytest.mark.parametrize("name,case", list(WGRAD_FP32.items()), ids=lambda v: v if isinstance(v, str) else "")
def test_tf32_wgrad_precision(name, case):
    """Precision tier; the accumulation term follows the split-K chunk length and the number of chunks."""
    B, M, N, hw = case
    gen = torch.Generator(device="cuda").manual_seed(9500 + M + N + hw)
    dY, X = scaled_gaussian((B, M, hw), 1, gen, "cuda"), scaled_gaussian((B, N, hw), 1, gen, "cuda")
    dW = _run_wgrad1(dY, X, B, M, N, hw)
    ref = _wgrad_ref(dY, X)
    mag = torch.einsum("bmp,bnp->mn", dY.double().abs(), X.double().abs())
    kc, nch = wgrad_chunks(torch.float32, B, M, hw)
    ratio = float(((dW.double() - ref).abs() / tf32_bound(kc + nch, mag).clamp_min(1e-300)).max())
    print("tf32 wgrad %s chunk=%d x %d rel_l2=%.3e elem/bound=%.3f" % (name, kc, nch, rel_l2(dW, ref), ratio))
    assert ratio <= 1.0, "element-wise bound exceeded by %.2fx" % ratio


@gpu
def test_tf32_wgrad_unbiased():
    """Bias test on the cfg-2 weight gradient (73 728 pixels): both operands are activations, so truncation would scale
    dW down by ~6e-4; rounded to nearest the mean signed relative error stays at the accumulation's level."""
    B, M, N, hw = 8, 256, 288, 9216
    gen = torch.Generator(device="cuda").manual_seed(9900)
    dY, X = _positive((B, M, hw), gen), _positive((B, N, hw), gen)
    dW = _run_wgrad1(dY, X, B, M, N, hw)
    ref = _wgrad_ref(dY, X)
    kc, nch = wgrad_chunks(torch.float32, B, M, hw)
    bias = float(((dW.double() - ref) / ref).mean())
    print("tf32 wgrad chunk=%d mean signed relative error %.3e (tol %.1e)" % (kc, bias, bias_tol(kc + nch)))
    assert abs(bias) <= bias_tol(kc + nch), bias


# ==================================================================== input gradient with the BatchNorm backward
@gpu
@pytest.mark.parametrize("relu", [True, False], ids=["relu", "norelu"])
@pytest.mark.parametrize("training", [True, False], ids=["train", "eval"])
@pytest.mark.parametrize("name,case", list(TF32_DGRAD_CASES.items()), ids=lambda v: v if isinstance(v, str) else "")
def test_tf32_dgrad_bnbwd(name, case, training, relu):
    """The stored dz is the fp32 value, bit for bit what the 3xTF32 kernel stores (the same expression; only the GEMM
    operand is rounded); dx = W^T.dz passes the one-pass bound against float64 W^T . dz."""
    from pinthememory_b200 import capi

    B, Kc, Mc, hw = case
    gen = torch.Generator(device="cuda").manual_seed(9700 + Kc + Mc + hw)
    mean, invstd, gamma, beta, dgamma, dbeta = _bn_coefficients(Kc, gen)
    z = (mean.view(1, Kc, 1) + torch.randn(B, Kc, hw, generator=gen, device="cuda") / invstd.view(1, Kc, 1)).contiguous()
    dy = torch.randn(B, Kc, hw, generator=gen, device="cuda")
    W = scaled_gaussian((Kc, Mc), 1, gen, "cuda")
    outs = {}
    for code in (PM_F32, PM_F32_TF32):
        hiT, loT = capi.conv1x1_prep(W, True, torch.float32, tf32=code == PM_F32_TF32)
        dx = Guarded(B * Mc * hw, torch.float32)
        dz = Guarded(B * Kc * hw, torch.float32)
        rc = _lib().pm_conv1x1_dgrad_bnbwd(dy.data_ptr(), z.data_ptr(), hiT.data_ptr(), None if loT is None else loT.data_ptr(),
                                           dx.t.data_ptr(), dz.t.data_ptr(), mean.data_ptr(), invstd.data_ptr(),
                                           gamma.data_ptr(), beta.data_ptr(), dgamma.data_ptr(), dbeta.data_ptr(), int(relu),
                                           int(training), B, Kc, Mc, hw, code, _stream())
        _ok(rc, "pm_conv1x1_dgrad_bnbwd")
        torch.cuda.synchronize()
        dx.check("dx")
        dz.check("dz")
        outs[code] = (dx.t.view(B, Mc, hw).clone(), dz.t.view(B, Kc, hw).clone())
    dx1, dz1 = outs[PM_F32_TF32]
    assert torch.equal(dz1.view(torch.int32), outs[PM_F32][1].view(torch.int32)), "stored dz is not the fp32 dz"
    A64, dz64 = W.double().t(), dz1.double()
    dx64 = torch.matmul(A64, dz64)
    ratio = float(((dx1.double() - dx64).abs() / tf32_bound(Kc, torch.matmul(A64.abs(), dz64.abs())).clamp_min(1e-300)).max())
    print("tf32 dgrad_bnbwd %s train=%d relu=%d dx rel_l2=%.3e elem/bound=%.3f" % (
        name, training, relu, rel_l2(dx1, dx64), ratio))
    assert ratio <= 1.0, ratio


@gpu
def test_tf32_dgrad_bnbwd_unbiased():
    """Bias test of the dz operand, which the transform warps form and then round: eval-mode BatchNorm without ReLU
    (dz = gamma*invstd*dy) and all-positive dy, gamma and W, at the cfg-2 shape (K = 256 output channels). Left to the
    tensor core's truncation, dz would shift dx by ~3e-4; rounded, the mean signed relative error stays near zero."""
    from pinthememory_b200 import capi

    B, Kc, Mc, hw = 8, 256, 288, 9216
    gen = torch.Generator(device="cuda").manual_seed(9750)
    ones, zeros = torch.ones(Kc, device="cuda"), torch.zeros(Kc, device="cuda")
    gamma = _positive((Kc,), gen)                            # invstd = 1: sc = gamma, full mantissas
    dy, z = _positive((B, Kc, hw), gen), _positive((B, Kc, hw), gen)
    W = _positive((Kc, Mc), gen)
    hiT, loT = capi.conv1x1_prep(W, True, torch.float32, tf32=True)
    dx, dz = capi.conv1x1_dgrad_bnbwd(dy.view(B, Kc, 1, hw), z.view(B, Kc, 1, hw), hiT, loT, Mc, zeros, ones, gamma, zeros,
                                      zeros, zeros, False, False)
    torch.cuda.synchronize()
    assert torch.equal(dz.view(B, Kc, hw), gamma.view(1, Kc, 1) * dy), "dz = gamma * dy in eval mode"
    dx64 = torch.matmul(W.double().t(), dz.view(B, Kc, hw).double())
    bias = float(((dx.view(B, Mc, hw).double() - dx64) / dx64).mean())
    print("tf32 dgrad_bnbwd K=%d mean signed relative error %.3e (tol %.1e)" % (Kc, bias, bias_tol(Kc)))
    assert abs(bias) <= bias_tol(Kc), bias


# =================================================================================================== routing
def _launched1():
    """Context collecting (BN, MT, NT, KB, ORD) of every one-pass conv1x1_nn_kernel and the T of every conv1x1_wgrad_kernel."""
    from torch.profiler import ProfilerActivity, profile

    @contextlib.contextmanager
    def ctx():
        out = {"nn": set(), "wg": set(), "nn3": set()}
        torch.cuda.synchronize()
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            yield out
            torch.cuda.synchronize()
        for e in prof.events():
            if e.device_type != torch.autograd.DeviceType.CUDA:
                continue
            m = re.search(r"conv1x1_nn_kernel<pm::Tf32OnePass<(true|false)>, (\d+), (\d+), (\d+), (true|false)>", e.name)
            if m:
                out["nn"].add((m.group(1) == "true", int(m.group(2)), int(m.group(3)), int(m.group(4)), m.group(5) == "true"))
            elif "conv1x1_nn_kernel<float" in e.name:
                out["nn3"].add(e.name)
            m = re.search(r"conv1x1_wgrad_kernel<([\w:<> ]+?)>\(", e.name)
            if m:
                out["wg"].add(m.group(1).strip())
    return ctx()


def tf32_nn_instantiations(B, K, M, hw, ordered, bnbwd=False):
    """(BN, MT, NT, KB, ORD) of every launch conv1x1_fwd_impl makes in PM_F32_TF32: the 3-pass tile shapes; with the
    BatchNorm backward only the first launch forms dz."""
    mtiles = (M + 127) // 128
    mts = [2] * (mtiles // 2) + [1] * (mtiles % 2)
    NT, KB = (256, 16) if B * ((hw + 255) // 256) >= 96 else (128, 32)
    return {(bnbwd and i == 0, mt, NT, KB, ordered) for i, mt in enumerate(mts)}


@gpu
def test_tf32_routing():
    """Every case launches the one-pass instantiations it was written for and never a 3-pass one; together they reach
    all 12 one-pass conv1x1_nn_kernel instantiations and the one-pass conv1x1_wgrad_kernel."""
    from pinthememory_b200 import capi

    wrong, reached = [], set()
    for name, (B, K, M, hw) in FP32_CASES.items():
        x = torch.zeros(B, K, 1, hw, device="cuda")
        hi = _prep1(torch.zeros(M, K, device="cuda"))
        for ordered in (False, True):
            stats = torch.zeros(2 * M, dtype=torch.float64, device="cuda") if ordered else None
            with deterministic_flag() if ordered else contextlib.nullcontext(), _launched1() as got:
                capi.conv1x1_fwd(x, hi, None, M, stats=stats)
            want = tf32_nn_instantiations(B, K, M, hw, ordered)
            if got["nn"] != want or got["nn3"]:
                wrong.append((name, ordered, sorted(got["nn"]), sorted(want), sorted(got["nn3"])))
            reached |= got["nn"]
    for name, (B, Kc, Mc, hw) in TF32_DGRAD_CASES.items():
        z = torch.zeros(B, Kc, 1, hw, device="cuda")
        hiT = _prep1(torch.zeros(Kc, Mc, device="cuda"), transpose=True)
        v = torch.ones(Kc, device="cuda")
        with _launched1() as got:
            capi.conv1x1_dgrad_bnbwd(z, z, hiT, None, Mc, v, v, v, v, v, v, True, True)
        want = tf32_nn_instantiations(B, Mc, Mc, hw, False, bnbwd=True)
        if got["nn"] != want or got["nn3"]:
            wrong.append(("dgrad " + name, sorted(got["nn"]), sorted(want), sorted(got["nn3"])))
        reached |= got["nn"]
    for name, (B, M, N, hw) in WGRAD_FP32.items():
        dy, x = torch.zeros(B, M, 1, hw, device="cuda"), torch.zeros(B, N, 1, hw, device="cuda")
        with _launched1() as got:
            capi.conv1x1_wgrad(dy, x, tf32=True)
        if got["wg"] != {"pm::Tf32OnePass<false>"}:
            wrong.append(("wgrad " + name, sorted(got["wg"])))
    assert not wrong, wrong
    every = {(False, mt, nt, kb, o) for (nt, kb) in ((256, 16), (128, 32)) for mt in (1, 2) for o in (False, True)}
    every |= {(True, mt, nt, kb, False) for (nt, kb) in ((256, 16), (128, 32)) for mt in (1, 2)}
    print("reached one-pass conv1x1_nn_kernel:", sorted(reached))
    assert reached == every, sorted(every - reached)


def test_tf32_case_tables_reach_every_instantiation():
    """Host side of the routing pin: the tables above cover all 12 one-pass forward instantiations by construction."""
    got = set()
    for B, K, M, hw in FP32_CASES.values():
        for o in (False, True):
            got |= tf32_nn_instantiations(B, K, M, hw, o)
    for B, Kc, Mc, hw in TF32_DGRAD_CASES.values():
        got |= tf32_nn_instantiations(B, Mc, Mc, hw, False, bnbwd=True)
    assert len(got) == 12, sorted(got)
