"""The 1x1-convolution GEMMs of csrc/pm_gemm.cu kernel by kernel, against float64 torch on the device.

Two tiers. The exact tier uses integer-valued operands whose every partial sum stays below 2^24: the TF32 split is then
hi = value, lo = 0, every fp32 accumulation is exact, and each kernel must equal the float64 product bit for bit (bf16
outputs equal the float64 result rounded to bf16). That tier finds indexing, tiling, tail, pipeline-phase and
stale-accumulator errors with zero tolerance. The precision tier uses Gaussian data with power-of-two scales spread over
the rows of A and the channels of x, so a row or channel mix-up shows element by element, and bounds the 3xTF32 error
norm-wise (TAU) and element-wise (ELEM_C). CPU tests show that both bounds reject the two plausible wrong products
(1-pass TF32, and 3xTF32 without the A_lo.x_hi term) at every shape used here.

The case tables name the code path each shape reaches (see DESIGN 4b); `test_gemm_routing` pins the instantiation every
case launches, and that all 12 conv1x1_nn_kernel and both conv1x1_wgrad_kernel instantiations are reached.

Every non-accumulating output is pre-filled with NaN, and every output, statistics vector and workspace sits between
two guard bands that must be left untouched."""
import contextlib
import ctypes
import re
import types

import pytest
import torch

from golden_util import assert_close, rel_l2

gpu = pytest.mark.gpu

PM_F32, PM_BF16 = 0, 1
PM_ERR_SHAPE, PM_ERR_ALIGN = -5, -6
GUARD_BYTES = 256


# ------------------------------------------------------------------------------------------------- tolerances
def TAU(K):
    """Norm-wise rel-L2 bound of a 3xTF32 product with K-long dot products: the tensor core adds in fp32 with truncation,
    so the error grows linearly with K. Measured on the B200 with the row/channel-scaled data below: 8.0e-9 K at
    K = 256..1024 (forward and weight-gradient chunks alike), 3-8e-7 below K = 100."""
    return max(1e-6, 1e-8 * K)


# element-wise: |y - y64| <= ELEM_C * (K + ELEM_K0) * 2^-24 * (|A|.|x|): K truncating fp32 adds plus the split's own
# per-product residuals (dropped lo.lo terms, lo parts truncated to TF32), which do not grow with K
# (measured on the B200: at most 0.3 of the bound with ELEM_C = 1, at K = 24)
ELEM_C, ELEM_K0 = 1.0, 16
# bf16 outputs: the fp32 accumulator (exact products, fp32 adds) rounded once to bf16 -- at most half an ulp, 2^-8 |y|
BF16_HALF_ULP = 2.0 ** -8
# BatchNorm backward formed in the operand path: sc*(g - k1 - xhat*k2) with its fp32 roundings (measured: 0.87 of the
# bound in training mode; eval mode is one rounding of sc*g, 0.25)
DZ_C = 4.0


# ---------------------------------------------------------------------------------------------- case tables
# fp32 forward / input-gradient GEMM (B, K, M, hw): what each reaches in conv1x1_fwd_impl
FP32_CASES = {
    "one_kstep_row32": (1, 8, 32, 4),            # one UMMA K step, a quarter-filled row tile, the smallest legal row
    "ktail_mtail_pxtail": (2, 40, 96, 100),      # K tail inside a 32-channel block, M < 128, pixel tail in a 32-px chunk
    "mt2_then_mt1": (3, 288, 288, 1296),         # MT = 2, then MT = 1 at m_tile0 = 2 (the 32 score-plane rows)
    "px128_190_tiles": (5, 256, 160, 4864),      # B*ceil(hw/256) = 95 -> 128-pixel tiles, 190 tiles on 148 CTAs
    "px256_one_acc": (3, 256, 160, 8192),        # = 96 -> 256-pixel tiles, one accumulator stage
    "persistent_wrap": (16, 96, 416, 9216),      # ~4 tiles per CTA (accumulator and ring phases wrap), rows 416..511 padded
    "k1024_m512": (12, 1024, 512, 2308),         # 64 weight blocks, two MT = 2 launches, a 4-pixel tail tile
    "wide_ktail": (8, 24, 256, 9216),            # K tail inside a 16-channel block of the wide path
    "wide_mt1": (4, 32, 288, 6144),              # 256-pixel tiles with MT = 2 then MT = 1
}
# bf16 (always 128-pixel tiles, 64-channel blocks): hw % 8 == 0, K tails against KB = 64
BF16_CASES = {
    "one_kstep_row32": (1, 16, 32, 8),
    "ktail_mtail_pxtail": (2, 80, 96, 104),
    "mt2_then_mt1": (3, 288, 288, 1296),
    "persistent_wrap": (16, 96, 416, 9216),      # ~8 tiles per CTA
    "k1024_m512": (12, 1024, 512, 2312),
}
GEMM_CASES = [(torch.float32, n, c) for n, c in FP32_CASES.items()] + [(torch.bfloat16, n, c) for n, c in BF16_CASES.items()]
MODES = ["plain", "accumulate", "stats", "stats_ordered", "affine", "affine_relu"]

# weight gradient (B, M, N, hw)
WGRAD_FP32 = {
    "smallest": (1, 32, 32, 4),
    "pxtail_mtail": (2, 160, 96, 100),           # pixel tail of the 32-pixel chunk, M tail
    "ni2": (3, 256, 288, 1296),                  # NI = 2, NW = 144
    "cols_256_64": (2, 128, 320, 2304),          # column blocks of 256 + 64
    "cols_256_288": (2, 256, 544, 2304),         # column blocks of 256 + 288, the second with NI = 2
    "cols_4x256": (1, 512, 1024, 9216),          # 4 x 256 columns, 4 row tiles
    "chunk_per_image": (80, 256, 64, 36),        # B * mtiles > 148 -> one chunk per image
    "cfg2": (8, 256, 288, 9216),
}
WGRAD_BF16 = {                                   # pixel tails against the 64-pixel chunks
    "smallest": (1, 32, 32, 8),
    "pxtail_mtail": (2, 160, 96, 104),
    "ni2_pxtail": (3, 256, 288, 1304),
    "cols_256_288": (2, 256, 544, 2312),
    "chunk_per_image": (80, 256, 64, 40),
}
WGRAD_CASES = [(torch.float32, n, c) for n, c in WGRAD_FP32.items()] + [(torch.bfloat16, n, c) for n, c in WGRAD_BF16.items()]
WGRAD_ACCUMULATE = {(torch.float32, "pxtail_mtail"), (torch.float32, "cols_256_288"), (torch.float32, "chunk_per_image"),
                    (torch.bfloat16, "pxtail_mtail")}

# input gradient with the BatchNorm backward in its operand path (B, Kc = conv output channels, Mc = conv input, hw)
DGRAD_CASES = {
    "narrow": (2, 64, 96, 100),                  # KB = 32: coefficients loaded per element
    "three_row_tiles": (3, 256, 288, 1296),      # launches after the first read the stored dz
    "wide_cfg2": (8, 256, 288, 9216),            # KB = 16: coefficients loaded once per thread
    "wide_tails": (12, 32, 416, 2308),           # wide tiles with M and pixel tails
}


# ----------------------------------------------------------------------------------------------- host logic
def nn_instantiations(dtype, B, K, M, hw, ordered):
    """(T, MT, NT, KB, ORD) of every launch conv1x1_fwd_impl makes for this shape."""
    mtiles = (M + 127) // 128
    mts = [2] * (mtiles // 2) + [1] * (mtiles % 2)
    if dtype == torch.bfloat16:
        return {("bf16", mt, 128, 64, ordered) for mt in mts}
    wide = B * ((hw + 255) // 256) >= 96
    return {("f32", mt, 256, 16, ordered) if wide else ("f32", mt, 128, 32, ordered) for mt in mts}


def wgrad_chunks(dtype, B, M, hw):
    """(pixels per split-K chunk, number of chunks) of pm_conv1x1_wgrad (wgrad_split)."""
    pxc = 32 if dtype == torch.float32 else 64
    mtiles, nblk = (M + 127) // 128, (hw + pxc - 1) // pxc
    want = min(max(148 // (mtiles * B), 1), nblk)
    bpc = (nblk + want - 1) // want
    return bpc * pxc, B * ((nblk + bpc - 1) // bpc)


def tf32_rn(t):
    """fp32 -> TF32 rounded to nearest (ties away from zero), as conv1x1_prep_kernel does."""
    return ((t.view(torch.int32) + 0x1000) & ~0x1FFF).view(torch.float32)


def tf32_trunc(t):
    """fp32 -> TF32 by truncation, as the tensor core reads an fp32 container."""
    return (t.view(torch.int32) & ~0x1FFF).view(torch.float32)


def scaled_gaussian(shape, axis, gen, device):
    """Gaussian values times 2^e, e uniform in -8..8 along `axis` (rows of A, channels of x)."""
    t = torch.randn(*shape, generator=gen, device=device)
    e = torch.randint(-8, 9, (shape[axis],), generator=gen, device=device).double()
    view = [1] * len(shape)
    view[axis] = shape[axis]
    return (t * torch.exp2(e).float().view(view)).contiguous()


# ------------------------------------------------------------------------------------------------- plumbing
def _lib():
    from pinthememory_b200 import capi

    return capi.load()


def _stream():
    return torch.cuda.current_stream().cuda_stream


def _ok(rc, what):
    assert rc == 0, "%s failed with status %d: %s" % (what, rc, _lib().pm_status_string(rc).decode())


class Guarded:
    """`n` elements inside one allocation, with GUARD_BYTES of random bits before and after them (and `offset_bytes`
    extra in front, to move the base off 16-byte alignment). `t` is the inner tensor."""

    def __init__(self, n, dtype, fill=float("nan"), offset_bytes=0):
        esz = torch.empty(0, dtype=dtype).element_size()
        self.lo = (GUARD_BYTES + offset_bytes) // esz
        self.hi = self.lo + n
        self.buf = torch.empty(self.hi + GUARD_BYTES // esz, dtype=dtype, device="cuda")
        self.buf.view(torch.uint8).random_(0, 256)
        self.t = self.buf[self.lo:self.hi]
        if fill is not None:
            self.t.fill_(fill)
        self.ref = self.buf.clone()

    def check(self, what, scratch=False):
        """Guards unchanged; unless `scratch`, every element written (no NaN left)."""
        b, r = self.buf.view(torch.uint8), self.ref.view(torch.uint8)
        esz = self.buf.element_size()
        assert torch.equal(b[: self.lo * esz], r[: self.lo * esz]), what + ": guard band before the buffer overwritten"
        assert torch.equal(b[self.hi * esz:], r[self.hi * esz:]), what + ": guard band after the buffer overwritten"
        if self.t.is_floating_point() and not scratch:
            assert not bool(torch.isnan(self.t).any()), what + ": elements left unwritten (NaN)"


@contextlib.contextmanager
def deterministic_flag():
    prev = torch.are_deterministic_algorithms_enabled()
    torch.use_deterministic_algorithms(True)
    try:
        yield
    finally:
        torch.use_deterministic_algorithms(prev)


def _prep(A, dtype):
    """(hi, lo) operands of A [M, K] through capi (the prep kernels are tested on their own below)."""
    from pinthememory_b200 import capi

    return capi.conv1x1_prep(A.contiguous(), False, dtype)


def _code(dtype):
    return PM_F32 if dtype == torch.float32 else PM_BF16


def _ints(shape, lo, hi, gen):
    return torch.randint(lo, hi + 1, shape, generator=gen, device="cuda").float()


def _sparse_signs(M, K, gen, nnz=16):
    """A in {-1, 0, 1} with at most `nnz` nonzeros per row: |A.x| <= nnz for x in {-1, 0, 1}."""
    A = _ints((M, K), -1, 1, gen)
    keep = torch.rand(M, K, generator=gen, device="cuda").argsort(dim=1) < nnz
    return A * keep


# ================================================================================== forward / input gradient
def _gemm_exact_inputs(dtype, B, K, M, hw, mode, gen):
    small = mode.startswith("stats") or (mode == "accumulate" and dtype == torch.bfloat16)
    if small:
        # statistics: |y| <= 16, so a 256-pixel tile's sum of y^2 stays below 2^24; bf16 accumulate: |y0 + y| <= 256
        A, x = _sparse_signs(M, K, gen), _ints((B, K, hw), -1, 1, gen)
    else:
        A, x = _ints((M, K), -7, 7, gen), _ints((B, K, hw), -7, 7, gen)     # |partial sums| <= 49 K < 2^24
    A[0] = 0                                                                 # rows whose weights are all zero
    A[M // 2] = 0
    return A, x.to(dtype)


def _run_fwd(mode, dtype, x, hi, lo, B, K, M, hw, y0=None, scale=None, shift=None):
    """One call of the entry `mode` exercises, on guarded buffers. Returns (y, stats or None)."""
    lib = _lib()
    n = B * M * hw
    y = Guarded(n, dtype, fill=None if mode == "accumulate" else float("nan"))
    if mode == "accumulate":
        y.t.copy_(y0.flatten())
        y.ref = y.buf.clone()
    stats = scratch = None
    p = lambda t: None if t is None else t.data_ptr()
    if mode in ("plain", "accumulate", "stats"):
        if mode == "stats":
            stats = Guarded(2 * M, torch.float64, fill=0.0)
        rc = lib.pm_conv1x1_fwd(p(x), p(hi), p(lo), y.t.data_ptr(), None if stats is None else stats.t.data_ptr(), B, K, M,
                                hw, int(mode == "accumulate"), _code(dtype), _stream())
        _ok(rc, "pm_conv1x1_fwd")
    elif mode == "stats_ordered":
        stats = Guarded(2 * M, torch.float64, fill=0.0)
        nbytes = lib.pm_conv1x1_stats_scratch_bytes(B, M, hw, _code(dtype))
        assert nbytes > 0 and nbytes % 8 == 0
        scratch = Guarded(nbytes // 8, torch.float64)
        rc = lib.pm_conv1x1_fwd_ordered(p(x), p(hi), p(lo), y.t.data_ptr(), stats.t.data_ptr(), scratch.t.data_ptr(), B, K,
                                        M, hw, _code(dtype), _stream())
        _ok(rc, "pm_conv1x1_fwd_ordered")
    else:
        rc = lib.pm_conv1x1_fwd_affine(p(x), p(hi), p(lo), y.t.data_ptr(), scale.data_ptr(), shift.data_ptr(),
                                       int(mode == "affine_relu"), B, K, M, hw, _code(dtype), _stream())
        _ok(rc, "pm_conv1x1_fwd_affine")
    torch.cuda.synchronize()
    y.check("y")
    if stats is not None:
        stats.check("stats")
    if scratch is not None:
        scratch.check("ordered-statistics scratch")
    return y.t.view(B, M, hw), (None if stats is None else stats.t.clone())


@gpu
@pytest.mark.parametrize("mode", MODES)
@pytest.mark.parametrize("dtype,name,case", GEMM_CASES, ids=lambda v: v if isinstance(v, str) else "")
def test_conv1x1_fwd_exact(dtype, name, case, mode):
    """Exact tier: every entry of the forward GEMM equals the float64 product bit for bit."""
    B, K, M, hw = case
    gen = torch.Generator(device="cuda").manual_seed(1000 + 7 * K + M + hw)
    A, x = _gemm_exact_inputs(dtype, B, K, M, hw, mode, gen)
    hi, lo = _prep(A, dtype)
    y64 = torch.matmul(A.double(), x.double())                               # [B, M, hw]
    y0 = scale = shift = None
    if mode == "accumulate":
        y0 = _ints((B, M, hw), -200, 200, gen) if dtype == torch.bfloat16 else _ints((B, M, hw), -1000, 1000, gen)
        y64 = y64 + y0.double()
        y0 = y0.to(dtype)
    if mode.startswith("affine"):
        scale = torch.exp2(torch.randint(-3, 4, (M,), generator=gen, device="cuda").float())   # powers of two
        shift = _ints((M,), -8, 8, gen)                                                        # integers
        y64 = y64 * scale.double().view(M, 1) + shift.double().view(M, 1)
        if mode == "affine_relu":
            y64 = y64.clamp_min(0.0)
    y, stats = _run_fwd(mode, dtype, x, hi, lo, B, K, M, hw, y0, scale, shift)
    want = y64.to(dtype)
    bad = y != want
    assert not bool(bad.any()), "%d of %d elements differ; first at (b, row, px) = %s: %r vs %r" % (
        int(bad.sum()), bad.numel(), tuple(bad.nonzero()[0].tolist()), float(y[bad][0]), float(want[bad][0]))
    if not mode.startswith("affine"):
        zero_rows = y[:, [0, M // 2]] if mode != "accumulate" else None
        if zero_rows is not None:
            assert bool((zero_rows == 0).all()), "rows with all-zero weights are not exactly 0"
    if stats is not None:
        ref = torch.cat([y64.sum((0, 2)), (y64 * y64).sum((0, 2))])
        bad = stats != ref
        assert not bool(bad.any()), "statistics differ at %s" % bad.nonzero().flatten()[:8].tolist()
    if mode == "stats_ordered":                                              # bitwise reproducible across runs
        y2, stats2 = _run_fwd(mode, dtype, x, hi, lo, B, K, M, hw)
        ib = torch.int32 if dtype == torch.float32 else torch.int16
        assert torch.equal(y2.view(ib), y.view(ib)), "output not reproducible"
        assert torch.equal(stats2.view(torch.int64), stats.view(torch.int64)), "statistics not reproducible"


@gpu
@pytest.mark.parametrize("dtype,name,case", GEMM_CASES, ids=lambda v: v if isinstance(v, str) else "")
def test_conv1x1_fwd_precision(dtype, name, case):
    """Precision tier: Gaussian data with 2^-8..2^8 scales on rows of A and channels of x."""
    B, K, M, hw = case
    gen = torch.Generator(device="cuda").manual_seed(2000 + 7 * K + M + hw)
    A = scaled_gaussian((M, K), 0, gen, "cuda")
    x = scaled_gaussian((B, K, hw), 1, gen, "cuda").to(dtype)
    hi, lo = _prep(A, dtype)
    y, _ = _run_fwd("plain", dtype, x, hi, lo, B, K, M, hw)
    Ad = A.double() if dtype == torch.float32 else A.to(dtype).double()     # bf16: the operand is bf16(A)
    y64 = torch.matmul(Ad, x.double())
    mag = torch.matmul(Ad.abs(), x.double().abs())
    err = (y.double() - y64).abs()
    bound = ELEM_C * (K + ELEM_K0) * 2.0 ** -24 * mag
    if dtype == torch.bfloat16:
        bound = bound + BF16_HALF_ULP * y64.abs()
    ratio = float((err / bound.clamp_min(1e-300)).max())
    r = rel_l2(y, y64)
    print("fwd %s %s K=%d rel_l2=%.3e (tau %.1e) elem/bound=%.3f" % (dtype, name, K, r, TAU(K), ratio))
    assert ratio <= 1.0, "element-wise bound exceeded by %.2fx" % ratio
    if dtype == torch.float32:
        assert r <= TAU(K), "rel_l2 %.3e > tau(K=%d) = %.1e" % (r, K, TAU(K))
    else:
        assert r <= 2.0 ** -8, r


# ============================================================================================ weight gradient
def _run_wgrad(dtype, dY, X, B, M, N, hw, dW0=None):
    lib = _lib()
    nws = lib.pm_conv1x1_wgrad_workspace_floats(B, M, N, hw, _code(dtype))
    assert nws > 0
    ws = Guarded(nws, torch.float32)
    dW = Guarded(M * N, torch.float32, fill=None if dW0 is not None else float("nan"))
    if dW0 is not None:
        dW.t.copy_(dW0.flatten())
        dW.ref = dW.buf.clone()
    rc = lib.pm_conv1x1_wgrad(dY.data_ptr(), X.data_ptr(), ws.t.data_ptr(), dW.t.data_ptr(), B, M, N, hw,
                              int(dW0 is not None), _code(dtype), _stream())
    _ok(rc, "pm_conv1x1_wgrad")
    torch.cuda.synchronize()
    ws.check("workspace", scratch=True)       # (sized for the widest column block; a narrower one uses less)
    dW.check("dW")
    return dW.t.view(M, N).clone()


def _wgrad_ref(dY, X):
    return torch.einsum("bmp,bnp->mn", dY.double(), X.double())


@gpu
@pytest.mark.parametrize("dtype,name,case", WGRAD_CASES, ids=lambda v: v if isinstance(v, str) else "")
def test_conv1x1_wgrad_exact(dtype, name, case):
    """Exact tier: integer operands, |dW| <= 49 B hw < 2^24; bitwise equal to float64, and to itself on a second run."""
    B, M, N, hw = case
    gen = torch.Generator(device="cuda").manual_seed(3000 + M + N + hw)
    dY, X = _ints((B, M, hw), -7, 7, gen).to(dtype), _ints((B, N, hw), -7, 7, gen).to(dtype)
    dY[:, 0] = 0
    ref = _wgrad_ref(dY, X)
    dW = _run_wgrad(dtype, dY, X, B, M, N, hw)
    bad = dW.double() != ref
    assert not bool(bad.any()), "%d elements differ, first at %s" % (int(bad.sum()), bad.nonzero()[0].tolist())
    assert torch.equal(_run_wgrad(dtype, dY, X, B, M, N, hw).view(torch.int32), dW.view(torch.int32)), "not reproducible"
    if (dtype, name) in WGRAD_ACCUMULATE:
        dW0 = _ints((M, N), -1000, 1000, gen)
        acc = _run_wgrad(dtype, dY, X, B, M, N, hw, dW0=dW0)
        assert torch.equal(acc.double(), ref + dW0.double()), "accumulate"


@gpu
@pytest.mark.parametrize("dtype,name,case", WGRAD_CASES, ids=lambda v: v if isinstance(v, str) else "")
def test_conv1x1_wgrad_precision(dtype, name, case):
    """Precision tier; the dot products are the split-K chunks, so the bound follows the chunk length."""
    B, M, N, hw = case
    gen = torch.Generator(device="cuda").manual_seed(4000 + M + N + hw)
    dY = scaled_gaussian((B, M, hw), 1, gen, "cuda").to(dtype)
    X = scaled_gaussian((B, N, hw), 1, gen, "cuda").to(dtype)
    dW = _run_wgrad(dtype, dY, X, B, M, N, hw)
    ref = _wgrad_ref(dY, X)
    mag = torch.einsum("bmp,bnp->mn", dY.double().abs(), X.double().abs())
    kc, nch = wgrad_chunks(dtype, B, M, hw)
    bound = ELEM_C * (kc + nch + ELEM_K0) * 2.0 ** -24 * mag
    ratio = float(((dW.double() - ref).abs() / bound.clamp_min(1e-300)).max())
    r = rel_l2(dW, ref)
    print("wgrad %s %s chunk=%d x %d rel_l2=%.3e (tau %.1e) elem/bound=%.3f" % (dtype, name, kc, nch, r, TAU(kc), ratio))
    assert ratio <= 1.0, "element-wise bound exceeded by %.2fx" % ratio
    assert r <= TAU(kc), "rel_l2 %.3e > tau(%d) = %.1e" % (r, kc, TAU(kc))


# ==================================================================== input gradient with the BatchNorm backward
def _bn_coefficients(K, gen):
    """Per-channel BatchNorm state with few mantissa bits, so that the kernel's fp32 sc = invstd*gamma and
    sh = beta - mean*sc are exact however they are evaluated (fused or not): the ReLU gate has no rounding ties."""
    mean = _ints((K,), -16, 16, gen) / 16
    invstd = torch.exp2(_ints((K,), -2, 2, gen))
    gamma = _ints((K,), 1, 24, gen) / 8 * torch.where(torch.rand(K, generator=gen, device="cuda") < 0.2, -1.0, 1.0)
    beta = _ints((K,), -16, 16, gen) / 16
    dgamma = torch.randn(K, generator=gen, device="cuda") * 100
    dbeta = torch.randn(K, generator=gen, device="cuda") * 100
    return mean, invstd, gamma, beta, dgamma, dbeta


@gpu
@pytest.mark.parametrize("relu", [True, False], ids=["relu", "norelu"])
@pytest.mark.parametrize("training", [True, False], ids=["train", "eval"])
@pytest.mark.parametrize("name,case", list(DGRAD_CASES.items()), ids=lambda v: v if isinstance(v, str) else "")
def test_conv1x1_dgrad_bnbwd_against_fp64_chain(name, case, training, relu):
    """dz = gamma*invstd*(g - dbeta/n - xhat*dgamma/n), g = dy*(z*sc + sh > 0), dx = W^T.dz, all in float64 from the same
    fp32 inputs; the stored dz and dx pass the precision tier, and neither leaves its buffer."""
    B, Kc, Mc, hw = case
    gen = torch.Generator(device="cuda").manual_seed(5000 + Kc + Mc + hw)
    mean, invstd, gamma, beta, dgamma, dbeta = _bn_coefficients(Kc, gen)
    z = (mean.view(1, Kc, 1) + torch.randn(B, Kc, hw, generator=gen, device="cuda") / invstd.view(1, Kc, 1)).contiguous()
    dy = torch.randn(B, Kc, hw, generator=gen, device="cuda")
    W = scaled_gaussian((Kc, Mc), 1, gen, "cuda")          # conv weight [out = Kc, in = Mc]; A = W^T, rows scaled
    from pinthememory_b200 import capi

    hiT, loT = capi.conv1x1_prep(W, True, torch.float32)
    sc = invstd * gamma
    sh = beta - mean * sc
    assert torch.equal(sc.double(), invstd.double() * gamma.double()) and torch.equal(
        sh.double(), beta.double() - mean.double() * sc.double()), "coefficients not exact"
    dx = Guarded(B * Mc * hw, torch.float32)
    dz = Guarded(B * Kc * hw, torch.float32)
    rc = _lib().pm_conv1x1_dgrad_bnbwd(dy.data_ptr(), z.data_ptr(), hiT.data_ptr(), loT.data_ptr(), dx.t.data_ptr(),
                                       dz.t.data_ptr(), mean.data_ptr(), invstd.data_ptr(), gamma.data_ptr(),
                                       beta.data_ptr(), dgamma.data_ptr(), dbeta.data_ptr(), int(relu), int(training),
                                       B, Kc, Mc, hw, PM_F32, _stream())
    _ok(rc, "pm_conv1x1_dgrad_bnbwd")
    torch.cuda.synchronize()
    dx.check("dx")
    dz.check("dz")
    # float64 chain
    d = lambda t: t.double().view(1, Kc, 1)
    z64, dy64 = z.double(), dy.double()
    gate = (z64 * d(sc) + d(sh) > 0) if relu else torch.ones_like(z64, dtype=torch.bool)
    g = dy64 * gate
    n = float(B * hw)
    xhat = (z64 - d(mean)) * d(invstd)
    k1 = d(dbeta) / n if training else 0.0
    k2 = d(dgamma) / n if training else 0.0
    dz64 = d(sc) * (g - k1 - xhat * k2)
    t = d(sc).abs() * (g.abs() + (d(dbeta).abs() / n if training else 0.0)
                       + ((z64.abs() + d(mean).abs()) * d(invstd) * (d(dgamma).abs() / n) if training else 0.0))
    dzk = dz.t.view(B, Kc, hw).double()
    ratio_dz = float(((dzk - dz64).abs() / (DZ_C * 2.0 ** -24 * t).clamp_min(1e-300)).max())
    A64 = W.double().t()                                   # [Mc, Kc]
    dx64 = torch.matmul(A64, dz64)
    bound = 2.0 ** -24 * (ELEM_C * (Kc + ELEM_K0) * torch.matmul(A64.abs(), dz64.abs())
                          + DZ_C * torch.matmul(A64.abs(), t))
    ratio_dx = float(((dx.t.view(B, Mc, hw).double() - dx64).abs() / bound.clamp_min(1e-300)).max())
    r_dz, r_dx = rel_l2(dzk, dz64), rel_l2(dx.t.view(B, Mc, hw), dx64)
    print("dgrad_bnbwd %s train=%d relu=%d dz rel_l2=%.3e elem/bound=%.3f  dx rel_l2=%.3e elem/bound=%.3f" % (
        name, training, relu, r_dz, ratio_dz, r_dx, ratio_dx))
    assert ratio_dz <= 1.0 and ratio_dx <= 1.0, (ratio_dz, ratio_dx)
    assert r_dz <= TAU(1) and r_dx <= TAU(Kc), (r_dz, r_dx)


# ====================================================================================== operand preparation
PREP_SHAPES = [(32, 8), (96, 40), (160, 24), (288, 256), (512, 1024)]


def _special_weights(M, K, gen):
    """Normal values over 2^-126..2^126 plus TF32 ties (low 13 bits 0x1000, both signs), +-0 and subnormals."""
    W = torch.randn(M, K, generator=gen, device="cuda") * torch.exp2(_ints((M, K), -100, 100, gen))
    bits = W.view(torch.int32)
    pick = torch.rand(M, K, generator=gen, device="cuda")
    tie = (bits & ~0x1FFF) | 0x1000
    sub = torch.randint(1, 1 << 23, (M, K), generator=gen, device="cuda", dtype=torch.int32) | (bits & -(1 << 31))
    bits = torch.where(pick < 0.2, tie, bits)
    bits = torch.where((pick >= 0.2) & (pick < 0.3), sub, bits)
    bits = torch.where((pick >= 0.3) & (pick < 0.33), torch.zeros_like(bits), bits)
    bits = torch.where((pick >= 0.33) & (pick < 0.36), torch.full_like(bits, -(1 << 31)), bits)
    return bits.view(torch.float32).contiguous()


def _check_split(hi, lo, W, what):
    """hi + lo == W, hi has its low 13 bits clear, |lo| <= half a TF32 ulp of W (4096 fp32 ulps)."""
    assert torch.equal(hi + lo, W), what + ": hi + lo != W"
    hb = hi.view(torch.int32)
    assert not bool((hb & 0x1FFF).any()), what + ": hi is not a TF32 value"
    assert torch.equal(hb < 0, W.view(torch.int32) < 0), what + ": hi lost the sign of W"
    a = W.abs()
    ulp = torch.nextafter(a, torch.full_like(a, float("inf"))) - a
    assert bool((lo.abs() <= 4096 * ulp).all()), what + ": |lo| above half a TF32 ulp"


@gpu
@pytest.mark.parametrize("M,K", PREP_SHAPES)
def test_conv1x1_prep_properties(M, K):
    lib = _lib()
    gen = torch.Generator(device="cuda").manual_seed(6000 + M + K)
    W = _special_weights(M, K, gen)
    Mpad = (M + 127) // 128 * 128
    p = lambda g: g.t.data_ptr()
    out = {}
    for dtype in (torch.float32, torch.bfloat16):
        for tr, src in ((0, W), (1, W.t().contiguous())):            # transpose = 1 takes W^T stored [K][M]
            hi = Guarded(Mpad * K, dtype)
            lo = Guarded(Mpad * K, dtype) if dtype == torch.float32 else None
            rc = lib.pm_conv1x1_prep(src.data_ptr(), M, K, tr, _code(dtype), p(hi), None if lo is None else p(lo), _stream())
            _ok(rc, "pm_conv1x1_prep")
            torch.cuda.synchronize()
            hi.check("hi")
            h = hi.t.view(Mpad, K)
            assert bool((h[M:].view(torch.int16 if dtype == torch.bfloat16 else torch.int32) == 0).all()), "padded rows"
            if dtype == torch.float32:
                lo.check("lo")
                l = lo.t.view(Mpad, K)
                assert bool((l[M:].view(torch.int32) == 0).all()), "padded rows of lo"
                _check_split(h[:M], l[:M], W, "fp32 transpose=%d" % tr)
                out[(dtype, tr)] = (h.clone(), l.clone())
            else:
                assert torch.equal(h[:M].view(torch.int16), W.to(torch.bfloat16).view(torch.int16)), "bf16 hi != bf16(W)"
                out[(dtype, tr)] = (h.clone(), None)
    # both layouts in one launch: bitwise the two single launches, and the statistics buffer cleared
    for dtype in (torch.float32, torch.bfloat16):
        R, S = M, K
        f32 = dtype == torch.float32
        bufs = [Guarded((R + 127) // 128 * 128 * S, dtype), Guarded((R + 127) // 128 * 128 * S, dtype) if f32 else None,
                Guarded((S + 127) // 128 * 128 * R, dtype), Guarded((S + 127) // 128 * 128 * R, dtype) if f32 else None]
        zero = Guarded(2 * R + 1, torch.float64)
        rc = lib.pm_conv1x1_prep_both(W.data_ptr(), R, S, _code(dtype), *[None if b is None else p(b) for b in bufs],
                                      p(zero), 2 * R + 1, _stream())
        _ok(rc, "pm_conv1x1_prep_both")
        torch.cuda.synchronize()
        for b in bufs:
            if b is not None:
                b.check("prep_both output")
        zero.check("zero")
        assert bool((zero.t.view(torch.int64) == 0).all()), "statistics buffer not cleared"
        one = {tr: _prep_call(W, tr, dtype) for tr in (0, 1)}
        ib = torch.int32 if f32 else torch.int16
        assert torch.equal(bufs[0].t.view(ib), one[0][0].flatten().view(ib))
        assert torch.equal(bufs[2].t.view(ib), one[1][0].flatten().view(ib))
        if f32:
            assert torch.equal(bufs[1].t.view(ib), one[0][1].flatten().view(ib))
            assert torch.equal(bufs[3].t.view(ib), one[1][1].flatten().view(ib))


def _prep_call(W, transpose, dtype):
    from pinthememory_b200 import capi

    return capi.conv1x1_prep(W, bool(transpose), dtype)


# =================================================================================================== routing
def _launched(fn):
    """Demangled (T, MT, NT, KB, ORD) of every conv1x1_nn_kernel and T of every conv1x1_wgrad_kernel `fn` launches."""
    from torch.profiler import ProfilerActivity, profile

    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    nn, wg = set(), set()
    for e in prof.events():
        if e.device_type != torch.autograd.DeviceType.CUDA:
            continue
        m = re.search(r"conv1x1_nn_kernel<([\w: ]+?), (\d+), (\d+), (\d+), (true|false)>", e.name)
        if m:
            t = "f32" if m.group(1).strip() == "float" else "bf16"
            nn.add((t, int(m.group(2)), int(m.group(3)), int(m.group(4)), m.group(5) == "true"))
        m = re.search(r"conv1x1_wgrad_kernel<([\w: ]+?)>", e.name)
        if m:
            wg.add("f32" if m.group(1).strip() == "float" else "bf16")
    return nn, wg


@gpu
def test_gemm_routing():
    """Each case launches the instantiations it was written for; together they reach all 12 conv1x1_nn_kernel and both
    conv1x1_wgrad_kernel instantiations (the ordered ones through torch's deterministic flag, as the module does)."""
    from pinthememory_b200 import capi

    wrong, reached_nn, reached_wg = [], set(), set()
    for dtype, name, (B, K, M, hw) in GEMM_CASES:
        x = torch.zeros(B, K, 1, hw, dtype=dtype, device="cuda")
        hi, lo = _prep(torch.zeros(M, K, device="cuda"), dtype)
        for ordered in (False, True):
            stats = torch.zeros(2 * M, dtype=torch.float64, device="cuda") if ordered else None
            with deterministic_flag() if ordered else contextlib.nullcontext():
                nn, _ = _launched(lambda: capi.conv1x1_fwd(x, hi, lo, M, stats=stats))
            want = nn_instantiations(dtype, B, K, M, hw, ordered)
            if nn != want:
                wrong.append((str(dtype), name, ordered, sorted(nn), sorted(want)))
            reached_nn |= nn
    for dtype, name, (B, M, N, hw) in WGRAD_CASES:
        dy = torch.zeros(B, M, 1, hw, dtype=dtype, device="cuda")
        x = torch.zeros(B, N, 1, hw, dtype=dtype, device="cuda")
        _, wg = _launched(lambda: capi.conv1x1_wgrad(dy, x))
        want = {"f32" if dtype == torch.float32 else "bf16"}
        if wg != want:
            wrong.append((str(dtype), name, "wgrad", sorted(wg), sorted(want)))
        reached_wg |= wg
    assert not wrong, wrong
    every_nn = {(t, mt, nt, kb, o) for (t, nt, kb) in (("f32", 256, 16), ("f32", 128, 32), ("bf16", 128, 64))
                for mt in (1, 2) for o in (False, True)}
    print("reached conv1x1_nn_kernel:", sorted(reached_nn), "conv1x1_wgrad_kernel:", sorted(reached_wg))
    assert reached_nn == every_nn, sorted(every_nn - reached_nn)
    assert reached_wg == {"f32", "bf16"}


def test_case_tables_reach_every_instantiation():
    """Host side of the routing pin: the shapes above cover all 12 forward instantiations by construction."""
    got = set()
    for dtype, name, (B, K, M, hw) in GEMM_CASES:
        for o in (False, True):
            got |= nn_instantiations(dtype, B, K, M, hw, o)
    assert len(got) == 12
    assert {wgrad_chunks(torch.float32, 80, 256, 36)[0]} == {64}     # one chunk per image when B * mtiles > 148


# =========================================================== CPU: the precision bounds reject the wrong products
# the emulation keeps the dot-product length the bound depends on and the row/channel scales of each GPU case; the
# number of output rows and columns is cut down, since the wrong products' relative error does not depend on it
_EMU_ROWS, _EMU_PX = 64, 512


@pytest.mark.parametrize("kind,name,case", [("fwd", n, c) for n, c in FP32_CASES.items()]
                         + [("wgrad", n, c) for n, c in WGRAD_FP32.items()]
                         + [("dgrad", n, c) for n, c in DGRAD_CASES.items()], ids=lambda v: v if isinstance(v, str) else "")
def test_precision_bound_rejects_wrong_products(kind, name, case):
    """The norm-wise bound rejects 1-pass TF32 and 3xTF32 without the A_lo.x_hi term at each GPU case. (The loose
    element-wise bound is there for row / channel mix-ups: a per-product error of 2^-12 averages down as 1/sqrt(K)
    relative to sum |a||x|, so it cannot see these at large K.)"""
    gen = torch.Generator().manual_seed(sum(case))
    if kind == "wgrad":                   # K = every pixel of the batch; the GPU bound follows the split-K chunk length
        B, M, N, hw = case
        Kd, (kc, _) = B * hw, wgrad_chunks(torch.float32, B, M, hw)
        tau = TAU(kc)
        A, x = scaled_gaussian((16, Kd), 0, gen, "cpu"), scaled_gaussian((Kd, 16), 1, gen, "cpu")
    else:
        Kd = case[1]
        tau = TAU(Kd)
        A, x = scaled_gaussian((_EMU_ROWS, Kd), 0, gen, "cpu"), scaled_gaussian((Kd, _EMU_PX), 0, gen, "cpu")
    one_pass, no_lo_hi = _wrong_products(A, x)
    assert one_pass > tau and no_lo_hi > tau, (one_pass, no_lo_hi, tau)


def _wrong_products(A, x):
    """rel-L2 against float64 of (1-pass TF32, 3xTF32 without A_lo.x_hi), emulated in float64 on the host."""
    Ah, xh = tf32_rn(A), tf32_trunc(x)
    xl = tf32_trunc(x - xh)
    y64 = A.double() @ x.double()
    one_pass = Ah.double() @ xh.double()
    no_lo_hi = one_pass + Ah.double() @ xl.double()
    return rel_l2(one_pass, y64), rel_l2(no_lo_hi, y64)


# =========================================== CPU: every shape the 1x1 block admits is taken by all three of its GEMMs
def test_conv1x1_ok_admits_only_shapes_every_gemm_of_the_block_takes():
    """For every (M, K) capi.conv1x1_ok admits, neither GEMM of the block (forward, input gradient -- plain and with the
    BatchNorm backward --), the weight gradient nor the ordered-statistics scratch rejects the shape: each entry stops
    at its alignment check (misaligned pointers, so nothing runs)."""
    from pinthememory_b200 import capi

    lib = capi.load()
    a16, bad = ctypes.c_void_p(16), ctypes.c_void_p(8)
    admitted = 0
    for dtype, hw in ((torch.float32, 4), (torch.bfloat16, 8)):
        code = _code(dtype)
        for M in range(32, 2049, 32):
            for K in range(8, 2049, 8):
                fake = types.SimpleNamespace(shape=(2, K, 1, hw), is_cuda=True, dtype=dtype, data_ptr=lambda: 0)
                if not capi.conv1x1_ok(fake, M, K):
                    continue
                admitted += 1
                rc = {
                    "forward": lib.pm_conv1x1_fwd(bad, a16, a16, a16, None, 2, K, M, hw, 0, code, None),
                    "forward_affine": lib.pm_conv1x1_fwd_affine(bad, a16, a16, a16, a16, a16, 1, 2, K, M, hw, code, None),
                    "input_gradient": lib.pm_conv1x1_fwd(bad, a16, a16, a16, None, 2, M, K, hw, 1, code, None),
                    "weight_gradient": lib.pm_conv1x1_wgrad(bad, a16, a16, a16, 2, M, K, hw, 0, code, None),
                }
                if dtype == torch.float32:
                    rc["input_gradient_bnbwd"] = lib.pm_conv1x1_dgrad_bnbwd(bad, a16, a16, a16, a16, a16, a16, a16, a16,
                                                                            a16, a16, a16, 1, 1, 2, M, K, hw, code, None)
                wrong = {k: v for k, v in rc.items() if v != PM_ERR_ALIGN}
                assert not wrong, "conv1x1_ok admits M=%d K=%d (%s) but %s" % (M, K, dtype, wrong)
                assert lib.pm_conv1x1_stats_scratch_bytes(2, M, hw, code) > 0, (M, K)
    assert admitted > 0


# ================================================ the 1x1 block with more input channels than the GEMM row limit
@gpu
@pytest.mark.parametrize("cin", [544, 1024])
def test_wide_input_block_trains_like_torch_modules(cin):
    """conv_bn_act on Conv2d(cin -> 256) + BatchNorm2d + ReLU in training mode: forward, backward and running statistics
    as the torch modules compute them (the input-gradient GEMM of such a block has cin output rows)."""
    import copy

    from pinthememory_b200.memory import conv_bn_act

    prev = torch.backends.cudnn.allow_tf32
    torch.backends.cudnn.allow_tf32 = False
    try:
        torch.manual_seed(11)
        conv = torch.nn.Conv2d(cin, 256, 1, bias=False).cuda()
        bn = torch.nn.BatchNorm2d(256).cuda().train()
        with torch.no_grad():
            bn.weight.uniform_(0.5, 1.5)
            bn.bias.normal_(0, 0.2)
        conv_r, bn_r = copy.deepcopy(conv), copy.deepcopy(bn)
        x = torch.randn(2, cin, 12, 16, device="cuda")
        G = torch.randn(2, 256, 12, 16, device="cuda")
        xa, xb = x.clone().requires_grad_(True), x.clone().requires_grad_(True)
        ya = conv_bn_act(conv, bn, xa, None, True)
        z = bn_r(conv_r(xb))
        gate = ya.detach() > 0
        flipped = gate != (z.detach() > 0)
        if bool(flipped.any()):
            assert float(z.detach().abs()[flipped].max()) <= 2e-5 * float(z.detach().abs().max()), "not a rounding tie"
        yb = z * gate.to(z.dtype)
        (ya * G).sum().backward()
        (yb * G).sum().backward()
        torch.cuda.synchronize()
    finally:
        torch.backends.cudnn.allow_tf32 = prev
    assert_close(ya.detach(), yb.detach(), 1e-5, "y")
    assert_close(xa.grad, xb.grad, 2e-5, "dx")
    assert_close(conv.weight.grad, conv_r.weight.grad, 2e-5, "dW")
    assert_close(bn.weight.grad, bn_r.weight.grad, 2e-5, "dgamma")
    assert_close(bn.bias.grad, bn_r.bias.grad, 2e-5, "dbeta")
    assert_close(bn.running_mean, bn_r.running_mean, 1e-6, "running_mean")
    assert_close(bn.running_var, bn_r.running_var, 1e-6, "running_var")
