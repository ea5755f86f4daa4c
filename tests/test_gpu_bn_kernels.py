"""The BatchNorm passes of csrc/pm_bn.cu entry by entry, against float64 torch on the device.

Every entry is run on each of its vector paths, in both dtypes: VN = 0 (scalar rows, hw % 4 != 0), VN = 4 (fp32 with
hw % 4 == 0; bf16 with hw % 8 != 0 or a base only 8-byte aligned) and VN = 8 (bf16, hw % 8 == 0, 16-byte aligned);
`test_bn_routing` pins which instantiation each case launches. Outputs are pre-filled with NaN and sit between guard
bands. Element-wise bounds are a few fp32 roundings of the terms each output is built from, plus half a bf16 ulp for
bf16 outputs; the sums are bounded by the length of the per-thread fp32 partial sums.

The last test measures how well the statistics fused into the GEMM epilogue are conditioned (E[x^2] - m^2 in fp64 over
fp32 tile sums) for conv outputs whose mean is r standard deviations from zero."""
import pytest
import torch

from golden_util import assert_close

gpu = pytest.mark.gpu

PM_F32, PM_BF16 = 0, 1
GUARD_BYTES = 256
U = 2.0 ** -24                 # unit roundoff of fp32

# y = x*sc + sh (+ res): sc = invstd*gamma, sh = beta - mean*sc and the fused multiply-add are each rounded once in fp32
# (measured on the B200: fp32 outputs reach 0.76 of the bound in bn_apply, 0.92 in bn_bwd_apply)
BN_C = 4.0
# bf16 outputs: rounding the fp32 value to bf16 adds at most half an ulp, <= 2^-8 |y|
BF16_HALF_ULP = 2.0 ** -8
# sums: each thread adds about L = hw/256 + VN elements in fp32 before the fp64 block sum. The worst case is L roundings
# of one sign (RED_C = 1); measured on the B200 the errors stay below 0.06 of that, so a quarter keeps a 4x margin
RED_C = 0.25
# mean / invstd / running statistics finalised in fp64 and rounded once to fp32 (plus the fp32 inputs of running stats)
STAT_REL = 2.0 ** -22
# the module's sequence (GEMM statistics -> normalise) against float64 BatchNorm of the same conv output, r <= 10: the
# parity bar of the module (measured on the B200 at r = 10: rel-L2 about 6e-6)
COND_TOL = 1e-5

# (dtype, B, C, hw, base offset in elements, VN the passes must take)
CASES = {
    "f32_vn0_tiny": (torch.float32, 2, 3, 63, 0, 0),
    "f32_vn0": (torch.float32, 4, 64, 63, 0, 0),
    "f32_vn4_tiny": (torch.float32, 2, 3, 36, 0, 4),
    "f32_vn4": (torch.float32, 3, 96, 100, 0, 4),
    "f32_vn4_full": (torch.float32, 16, 512, 9216, 0, 4),
    "bf16_vn0": (torch.bfloat16, 2, 5, 63, 0, 0),
    "bf16_vn4_hw36": (torch.bfloat16, 2, 5, 36, 0, 4),
    "bf16_vn4_offset8": (torch.bfloat16, 3, 64, 200, 4, 4),
    "bf16_vn8_tiny": (torch.bfloat16, 2, 5, 40, 0, 8),
    "bf16_vn8": (torch.bfloat16, 3, 96, 200, 0, 8),
    "bf16_vn8_full": (torch.bfloat16, 16, 512, 9216, 0, 8),
}
CASE_IDS = list(CASES)


class Guarded:
    """`n` elements inside one allocation, with GUARD_BYTES of random bits before and after them (`offset_bytes` more
    in front moves the base off 16-byte alignment). `t` is the inner tensor."""

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

    def check(self, what):
        b, r = self.buf.view(torch.uint8), self.ref.view(torch.uint8)
        esz = self.buf.element_size()
        assert torch.equal(b[: self.lo * esz], r[: self.lo * esz]), what + ": guard band before the buffer overwritten"
        assert torch.equal(b[self.hi * esz:], r[self.hi * esz:]), what + ": guard band after the buffer overwritten"
        if self.t.is_floating_point():
            assert not bool(torch.isnan(self.t).any()), what + ": elements left unwritten (NaN)"


def _placed(t, off_elems):
    """A copy of `t` (4-D) whose base is `off_elems` elements past a 16-byte boundary."""
    g = Guarded(t.numel(), t.dtype, fill=None, offset_bytes=off_elems * t.element_size())
    g.t.copy_(t.flatten())
    return g.t.view(t.shape)


def _out(shape, dtype, off_elems=0):
    n = 1
    for s in shape:
        n *= s
    return Guarded(n, dtype, offset_bytes=off_elems * torch.empty(0, dtype=dtype).element_size())


def _inputs(name, seed):
    dtype, B, C, hw, off, vn = CASES[name]
    g = torch.Generator(device="cuda").manual_seed(seed + B * 1000 + C + hw)
    ch = lambda: torch.randn(C, generator=g, device="cuda")
    mean, invstd = ch() * 0.5, torch.rand(C, generator=g, device="cuda") + 0.5
    gamma, beta = 1 + 0.3 * ch(), 0.3 * ch()
    x = (mean.view(1, C, 1, 1) + torch.randn(B, C, 1, hw, generator=g, device="cuda") / invstd.view(1, C, 1, 1))
    res = torch.randn(B, C, 1, hw, generator=g, device="cuda")
    dy = torch.randn(B, C, 1, hw, generator=g, device="cuda")
    return dict(dtype=dtype, B=B, C=C, hw=hw, off=off, vn=vn, mean=mean, invstd=invstd, gamma=gamma, beta=beta,
                x=_placed(x.to(dtype), off), res=_placed(res.to(dtype), off), dy=_placed(dy.to(dtype), off), g=g)


def _c(t):
    return t.double().view(1, -1, 1, 1)


def _mask_bits(words, B, C, hw):
    """[B, C, 1, 32 * words per row] bool from the packed mask (1 bit per element, 32 per word)."""
    wpr = (hw + 31) // 32
    w = words.view(B * C, wpr).to(torch.int64) & 0xFFFFFFFF
    bits = (w.unsqueeze(-1) >> torch.arange(32, device=w.device)) & 1
    return bits.view(B, C, 1, wpr * 32).bool()


def _ratio(err, bound):
    return float((err / bound.clamp_min(1e-300)).max())


def _apply_ref(d, residual, relu, mean=None, invstd=None):
    mean = d["mean"] if mean is None else mean
    invstd = d["invstd"] if invstd is None else invstd
    x64 = d["x"].double()
    y64 = (x64 - _c(mean)) * _c(invstd) * _c(d["gamma"]) + _c(d["beta"])
    sc = _c(invstd) * _c(d["gamma"])
    mag = (x64 * sc).abs() + (_c(mean) * sc).abs() + _c(d["beta"]).abs()
    if residual:
        y64 = y64 + d["res"].double()
        mag = mag + d["res"].double().abs()
    if relu:
        y64 = y64.clamp_min(0.0)
    return y64, mag


def _check_y(y, y64, mag, dtype, what, c=BN_C):
    bound = c * U * mag
    if dtype == torch.bfloat16:
        bound = bound + BF16_HALF_ULP * y64.abs()
    ratio = _ratio((y.double() - y64).abs(), bound)
    assert ratio <= 1.0, "%s: element-wise bound exceeded by %.2fx" % (what, ratio)
    return ratio


# ============================================================================================== normalise pass
@gpu
@pytest.mark.parametrize("relu", [False, True], ids=["norelu", "relu"])
@pytest.mark.parametrize("residual", [False, True], ids=["nores", "res"])
@pytest.mark.parametrize("name", CASE_IDS)
def test_bn_apply(name, residual, relu):
    from pinthememory_b200 import capi

    d = _inputs(name, 1)
    dtype, B, C, hw, off = d["dtype"], d["B"], d["C"], d["hw"], d["off"]
    y = _out((B, C, 1, hw), dtype, off)
    nw = capi.bn_mask_words(B, C, hw) if (relu and d["vn"]) else 0
    mask = Guarded(nw, torch.int32, fill=None) if nw else None
    capi.bn_apply(d["x"], d["mean"], d["invstd"], d["gamma"], d["beta"], d["res"] if residual else None,
                  y.t.view(B, C, 1, hw), relu, relu_mask=None if mask is None else mask.t)
    torch.cuda.synchronize()
    y.check("y")
    yk = y.t.view(B, C, 1, hw)
    y64, mag = _apply_ref(d, residual, relu)
    r = _check_y(yk, y64, mag, dtype, "y")
    print("bn_apply %s res=%d relu=%d elem/bound=%.3f" % (name, residual, relu, r))
    if mask is not None:
        mask.check("relu mask")
        bits = _mask_bits(mask.t, B, C, hw)
        assert torch.equal(bits[..., :hw], yk > 0), "mask bits differ from y > 0"
        assert not bool(bits[..., hw:].any()), "mask bits set past the end of a row"


@gpu
@pytest.mark.parametrize("residual", [False, True], ids=["nores", "res"])
@pytest.mark.parametrize("name", CASE_IDS)
def test_bn_apply_stats(name, residual):
    """Statistics finalised inside the normalise pass from float64 sums: mean / invstd, running statistics with the
    unbiased n/(n-1), the device-side count, and num_batches_tracked bumped exactly once per call."""
    from pinthememory_b200 import capi

    d = _inputs(name, 2)
    dtype, B, C, hw, off = d["dtype"], d["B"], d["C"], d["hw"], d["off"]
    x64 = d["x"].double()
    n = B * hw
    stats = torch.cat([x64.sum((0, 2, 3)), (x64 * x64).sum((0, 2, 3))])
    m64 = stats[:C] / n
    var64 = (stats[C:] / n - m64 * m64).clamp_min(0.0)
    eps, mom = 1e-5, 0.1
    is64 = 1.0 / torch.sqrt(var64 + eps)
    rm0 = torch.randn(C, generator=d["g"], device="cuda")
    rv0 = torch.rand(C, generator=d["g"], device="cuda") + 0.5
    count_dev = torch.tensor([float(n)], dtype=torch.float64, device="cuda")
    nbt = torch.zeros(3, dtype=torch.int64, device="cuda")
    for call in range(3):
        rm, rv = rm0.clone(), rv0.clone()
        mean_o, inv_o = _out((C,), torch.float32), _out((C,), torch.float32)
        y = _out((B, C, 1, hw), dtype, off)
        # the second and third calls pass a wrong host count: the device count must win
        capi.bn_apply_stats(d["x"], stats, n if call == 0 else 1.0, eps, d["gamma"], d["beta"],
                            d["res"] if residual else None, y.t.view(B, C, 1, hw), True, mean_o.t, inv_o.t, rm, rv, mom,
                            count_dev=None if call == 0 else count_dev, num_batches_tracked=nbt[1:2])
        torch.cuda.synchronize()
        for g_, w in ((y, "y"), (mean_o, "mean"), (inv_o, "invstd")):
            g_.check(w)
        assert ((mean_o.t.double() - m64).abs() <= STAT_REL * m64.abs() + U * 4 * torch.sqrt(var64)).all(), "mean"
        assert ((inv_o.t.double() - is64).abs() <= STAT_REL * is64).all(), "invstd"
        rm64 = (1 - mom) * rm0.double() + mom * m64
        rv64 = (1 - mom) * rv0.double() + mom * var64 * n / (n - 1)
        assert ((rm.double() - rm64).abs() <= STAT_REL * ((1 - mom) * rm0.double().abs() + mom * m64.abs())).all(), "rm"
        assert ((rv.double() - rv64).abs() <= STAT_REL * rv64.abs()).all(), "running_var"
        y64, mag = _apply_ref(d, residual, True, mean=m64, invstd=is64)
        _check_y(y.t.view(B, C, 1, hw), y64, mag, dtype, "y", c=BN_C + 2)   # + the fp32 rounding of mean and invstd
    assert nbt.tolist() == [0, 3, 0], "num_batches_tracked must grow by exactly 1 per call: %s" % nbt.tolist()


# ============================================================================================ backward passes
def _bwd_ref(d, gate, training, dgamma=None, dbeta=None):
    """float64 (dbeta, dgamma) from the gate, and dx from given fp32 sums (the kernel's) or the float64 ones."""
    B, hw = d["B"], d["hw"]
    g = d["dy"].double() * gate
    xhat = (d["x"].double() - _c(d["mean"])) * _c(d["invstd"])
    db64, dg64 = g.sum((0, 2, 3)), (g * xhat).sum((0, 2, 3))
    n = float(B * hw)
    dgk = dg64 if dgamma is None else dgamma.double()
    dbk = db64 if dbeta is None else dbeta.double()
    gi = _c(d["gamma"]) * _c(d["invstd"])
    if training:
        dx64 = gi * (g - _c(dbk) / n - xhat * _c(dgk) / n)
        mag = gi.abs() * (g.abs() + _c(dbk).abs() / n + (xhat.abs() + (d["x"].double().abs() + _c(d["mean"]).abs())
                                                          * _c(d["invstd"])) * _c(dgk).abs() / n)
    else:
        dx64, mag = gi * g, (gi * g).abs()
    return db64, dg64, g, xhat, dx64, mag


def _check_sums(d, dgamma, dbeta, g, xhat, db64, dg64, what):
    L = d["hw"] / 256 + 9
    xs = (d["x"].double().abs() + _c(d["mean"]).abs()) * _c(d["invstd"])
    b_db = RED_C * U * L * g.abs().sum((0, 2, 3)) + U * db64.abs()
    b_dg = RED_C * U * L * (g * xhat).abs().sum((0, 2, 3)) + 3 * U * (g.abs() * xs).sum((0, 2, 3)) + U * dg64.abs()
    r1 = _ratio((dbeta.double() - db64).abs(), b_db)
    r2 = _ratio((dgamma.double() - dg64).abs(), b_dg)
    assert r1 <= 1.0 and r2 <= 1.0, "%s: dbeta %.2fx, dgamma %.2fx of the bound" % (what, r1, r2)
    return max(r1, r2)


def _run_bwd(d, relu, training, y, mask, with_dres=True):
    from pinthememory_b200 import capi

    dtype, B, C, hw, off = d["dtype"], d["B"], d["C"], d["hw"], d["off"]
    dg, db = _out((C,), torch.float32), _out((C,), torch.float32)
    capi.bn_bwd_reduce(d["dy"], y, mask, d["x"], d["mean"], d["invstd"], relu, dg.t, db.t)
    dx = _out((B, C, 1, hw), dtype, off)
    dres = _out((B, C, 1, hw), dtype, off) if with_dres else None
    capi.bn_bwd_apply(d["dy"], y, mask, d["x"], d["mean"], d["invstd"], d["gamma"], dg.t, db.t, relu, training,
                      dx.t.view(B, C, 1, hw), None if dres is None else dres.t.view(B, C, 1, hw))
    torch.cuda.synchronize()
    for g_, w in ((dg, "dgamma"), (db, "dbeta"), (dx, "dx")) + (((dres, "dres"),) if dres is not None else ()):
        g_.check(w)
    return dg.t.clone(), db.t.clone(), dx.t.view(B, C, 1, hw).clone(), None if dres is None else dres.t.view(B, C, 1, hw)


@gpu
@pytest.mark.parametrize("training", [True, False], ids=["train", "eval"])
@pytest.mark.parametrize("relu", [False, True], ids=["norelu", "relu"])
@pytest.mark.parametrize("name", CASE_IDS)
def test_bn_backward(name, relu, training):
    """pm_bn_bwd_reduce_rows and pm_bn_bwd_apply (with dres) against float64, the gate taken from y; where the packed
    mask exists, the mask path gives bitwise the same dgamma / dbeta / dx as the y path."""
    from pinthememory_b200 import capi

    d = _inputs(name, 3)
    dtype, B, C, hw, off = d["dtype"], d["B"], d["C"], d["hw"], d["off"]
    y = _placed(torch.zeros(B, C, 1, hw, dtype=dtype, device="cuda"), off)
    nw = capi.bn_mask_words(B, C, hw) if d["vn"] else 0
    mask = torch.empty(nw, dtype=torch.int32, device="cuda") if (relu and nw) else None
    capi.bn_apply(d["x"], d["mean"], d["invstd"], d["gamma"], d["beta"], None, y, True, relu_mask=mask)
    gate = (y.double() > 0) if relu else torch.ones_like(y, dtype=torch.bool)
    dg, db, dx, dres = _run_bwd(d, relu, training, y, None)
    db64, dg64, g, xhat, _, _ = _bwd_ref(d, gate, training)
    rs = _check_sums(d, dg, db, g, xhat, db64, dg64, name)
    _, _, _, _, dx64, mag = _bwd_ref(d, gate, training, dgamma=dg, dbeta=db)
    rx = _check_y(dx, dx64, mag, dtype, "dx")
    assert torch.equal(dres.double(), g), "dres != dy * gate"
    print("bn_backward %s relu=%d train=%d sums %.3f dx %.3f (of the bounds)" % (name, relu, training, rs, rx))
    if mask is not None:
        dg2, db2, dx2, _ = _run_bwd(d, relu, training, None, mask, with_dres=False)
        assert torch.equal(dg2, dg) and torch.equal(db2, db), "mask path sums differ from the y path"
        ib = torch.int32 if dtype == torch.float32 else torch.int16
        assert torch.equal(dx2.view(ib), dx.view(ib)), "mask path dx differs from the y path"


@gpu
@pytest.mark.parametrize("dtype,hw", [(torch.bfloat16, 40), (torch.bfloat16, 36), (torch.float32, 36)], ids=str)
def test_relu_mask_read_at_another_vector_width(dtype, hw):
    """A mask written by bn_apply is read correctly by a backward that runs at another vector width: bf16 written at
    VN = 8 and read at VN = 4 (dy and dx 8 bytes off alignment); hw = 36, where the last mask word of a row is partial."""
    from pinthememory_b200 import capi

    B, C = 3, 7
    g = torch.Generator(device="cuda").manual_seed(hw)
    x = torch.randn(B, C, 1, hw, generator=g, device="cuda").to(dtype)
    mean, invstd = torch.zeros(C, device="cuda"), torch.ones(C, device="cuda")
    gamma, beta = torch.ones(C, device="cuda"), 0.1 * torch.randn(C, generator=g, device="cuda")
    y = torch.empty_like(x)
    mask = torch.empty(capi.bn_mask_words(B, C, hw), dtype=torch.int32, device="cuda")
    capi.bn_apply(x, mean, invstd, gamma, beta, None, y, True, relu_mask=mask)
    dy = torch.randn(B, C, 1, hw, generator=g, device="cuda").to(dtype)
    d = dict(dtype=dtype, B=B, C=C, hw=hw, off=4 if dtype == torch.bfloat16 else 0, mean=mean, invstd=invstd,
             gamma=gamma, x=_placed(x, 4 if dtype == torch.bfloat16 else 0),
             dy=_placed(dy, 4 if dtype == torch.bfloat16 else 0))
    yo = _placed(y, d["off"])
    dg, db, dx, _ = _run_bwd(d, True, True, None, mask, with_dres=False)
    dg2, db2, dx2, _ = _run_bwd(d, True, True, yo, None, with_dres=False)
    ib = torch.int32 if dtype == torch.float32 else torch.int16
    assert torch.equal(dg, dg2) and torch.equal(db, db2) and torch.equal(dx.view(ib), dx2.view(ib))
    gate = y.double() > 0
    db64, dg64, gg, xhat, _, _ = _bwd_ref(d, gate, True)
    _check_sums(d, dg, db, gg, xhat, db64, dg64, "mask")


@gpu
@pytest.mark.parametrize("B", [1, 4])
def test_bn_rows_scratch_is_reused(B):
    """Three consecutive reductions with different data on the one cached scratch of capi._bn_rows_scratch: each matches
    float64, so the arrival counters are back at zero after every call."""
    from pinthememory_b200 import capi

    C, hw = 33, 100
    bufs = set()
    for call in range(3):
        g = torch.Generator(device="cuda").manual_seed(100 * B + call)
        x = torch.randn(B, C, 1, hw, generator=g, device="cuda") * (call + 1)
        dy = torch.randn(B, C, 1, hw, generator=g, device="cuda")
        y = torch.randn(B, C, 1, hw, generator=g, device="cuda")
        mean, invstd = torch.randn(C, generator=g, device="cuda"), torch.rand(C, generator=g, device="cuda") + 0.5
        bufs.add(capi._bn_rows_scratch(x, B, C).data_ptr())
        d = dict(dtype=torch.float32, B=B, C=C, hw=hw, dy=dy, x=x, mean=mean, invstd=invstd, gamma=torch.ones(C, device="cuda"))
        dg, db = torch.full((C,), float("nan"), device="cuda"), torch.full((C,), float("nan"), device="cuda")
        capi.bn_bwd_reduce(dy, y, None, x, mean, invstd, True, dg, db)
        torch.cuda.synchronize()
        db64, dg64, gg, xhat, _, _ = _bwd_ref(d, y.double() > 0, True)
        _check_sums(d, dg, db, gg, xhat, db64, dg64, "call %d" % call)
    assert len(bufs) == 1


# ================================================================== statistics, finalise, eval-mode affine
@gpu
@pytest.mark.parametrize("name", CASE_IDS)
def test_bn_stats(name):
    """pm_bn_stats: fp32 partial sums per thread (about B*hw/512 elements each), fp64 across threads; the bound on
    invstd follows from the bounds on the two sums."""
    from pinthememory_b200 import capi

    d = _inputs(name, 4)
    B, C, hw = d["B"], d["C"], d["hw"]
    x64 = d["x"].double()
    n = B * hw
    eps, mom = 1e-5, 0.1
    m64 = x64.mean((0, 2, 3))
    var64 = x64.var((0, 2, 3), unbiased=False)
    mean, inv = _out((C,), torch.float32), _out((C,), torch.float32)
    rm, rv = torch.zeros(C, device="cuda"), torch.ones(C, device="cuda")
    capi.bn_stats(d["x"], eps, mean.t, inv.t, rm, rv, mom)
    torch.cuda.synchronize()
    mean.check("mean")
    inv.check("invstd")
    L = n / 512 + 8
    eS = RED_C * U * L * x64.abs().sum((0, 2, 3)) / n
    eQ = RED_C * U * L * (x64 * x64).sum((0, 2, 3)) / n
    evar = eQ + 2 * m64.abs() * eS + U * (var64 + m64 * m64)
    is64 = 1 / torch.sqrt(var64 + eps)
    assert ((mean.t.double() - m64).abs() <= eS + U * m64.abs()).all(), "mean"
    assert ((inv.t.double() - is64).abs() <= is64 * (0.5 * evar / (var64 + eps) + STAT_REL)).all(), "invstd"
    rv64 = (1 - mom) + mom * var64 * n / (n - 1)
    assert ((rm.double() - mom * m64).abs() <= mom * (eS + U * m64.abs()) + U * m64.abs() * mom).all(), "running_mean"
    assert ((rv.double() - rv64).abs() <= mom * evar * n / (n - 1) + STAT_REL * rv64).all(), "running_var"


@gpu
def test_bn_finalize_and_eval_affine():
    from pinthememory_b200 import capi

    C, n = 300, 8 * 9216
    g = torch.Generator(device="cuda").manual_seed(9)
    m = torch.randn(C, generator=g, device="cuda", dtype=torch.float64)
    var = torch.rand(C, generator=g, device="cuda", dtype=torch.float64) + 0.1
    stats = torch.cat([m * n, (var + m * m) * n])
    mean, inv = _out((C,), torch.float32), _out((C,), torch.float32)
    rm0, rv0 = torch.randn(C, generator=g, device="cuda"), torch.rand(C, generator=g, device="cuda") + 0.5
    rm, rv = rm0.clone(), rv0.clone()
    capi.bn_finalize(stats, C, n, 1e-5, mean.t, inv.t, rm, rv, 0.1)
    torch.cuda.synchronize()
    mean.check("mean")
    inv.check("invstd")
    m64, v64 = stats[:C] / n, stats[C:] / n - (stats[:C] / n) ** 2
    is64 = 1 / torch.sqrt(v64 + 1e-5)
    assert ((mean.t.double() - m64).abs() <= STAT_REL * m64.abs()).all()
    assert ((inv.t.double() - is64).abs() <= STAT_REL * is64).all()
    rm64, rv64 = 0.9 * rm0.double() + 0.1 * m64, 0.9 * rv0.double() + 0.1 * v64 * n / (n - 1)
    assert ((rm.double() - rm64).abs() <= STAT_REL * (0.9 * rm0.double().abs() + 0.1 * m64.abs())).all()
    assert ((rv.double() - rv64).abs() <= STAT_REL * rv64).all()
    # eval-mode affine: scale = gamma * rsqrt(var + eps) (rsqrtf: 2 ulp), shift = beta - mean * scale (one fma)
    gamma, beta = torch.randn(C, generator=g, device="cuda"), torch.randn(C, generator=g, device="cuda")
    scale, shift = capi.bn_eval_affine(gamma, beta, rm, rv, 1e-5)
    s64 = gamma.double() / torch.sqrt(rv.double() + 1e-5)
    sh64 = beta.double() - rm.double() * s64
    assert ((scale.double() - s64).abs() <= 4 * U * s64.abs()).all(), "scale"
    assert ((shift.double() - sh64).abs() <= U * (5 * (rm.double() * s64).abs() + beta.double().abs())).all(), "shift"


# ============================================================================================== routing pin
@gpu
def test_bn_routing():
    """Each case launches every BatchNorm kernel at the vector width it was written for; together they reach VN 0, 4
    and 8 in bf16 and VN 0 and 4 in fp32 for all four kernels."""
    import re

    from torch.profiler import ProfilerActivity, profile

    from pinthememory_b200 import capi

    wrong, reached = [], set()
    for name in CASE_IDS:
        d = _inputs(name, 5)
        dtype, B, C, hw, off = d["dtype"], d["B"], d["C"], d["hw"], d["off"]
        y = _placed(torch.zeros(B, C, 1, hw, dtype=dtype, device="cuda"), off)
        dx = _placed(torch.zeros(B, C, 1, hw, dtype=dtype, device="cuda"), off)
        mean, inv = torch.empty(C, device="cuda"), torch.empty(C, device="cuda")
        dg, db = torch.empty(C, device="cuda"), torch.empty(C, device="cuda")
        torch.cuda.synchronize()
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            capi.bn_stats(d["x"], 1e-5, mean, inv, None, None, 0.1)
            capi.bn_apply(d["x"], mean, inv, d["gamma"], d["beta"], None, y, True)
            capi.bn_bwd_reduce(d["dy"], y, None, d["x"], mean, inv, True, dg, db)
            capi.bn_bwd_apply(d["dy"], y, None, d["x"], mean, inv, d["gamma"], dg, db, True, True, dx, None)
            torch.cuda.synchronize()
        got = set()
        for e in prof.events():
            m = re.search(r"(bn_stats_kernel|bn_apply_kernel|bn_bwd_reduce_rows_kernel|bn_bwd_apply_kernel)<([\w: ]+?), (\d+)>",
                          e.name)
            if e.device_type == torch.autograd.DeviceType.CUDA and m:
                got.add((m.group(1), "f32" if m.group(2).strip() == "float" else "bf16", int(m.group(3))))
        t = "f32" if dtype == torch.float32 else "bf16"
        want = {(k, t, d["vn"]) for k in ("bn_stats_kernel", "bn_apply_kernel", "bn_bwd_reduce_rows_kernel",
                                          "bn_bwd_apply_kernel")}
        if got != want:
            wrong.append((name, sorted(got), sorted(want)))
        reached |= got
    assert not wrong, wrong
    assert {(t, vn) for _, t, vn in reached} == {("f32", 0), ("f32", 4), ("bf16", 0), ("bf16", 4), ("bf16", 8)}
    assert len(reached) == 4 * 5


# ==================================== conditioning of the statistics fused into the GEMM epilogue (E[x^2] - m^2)
@gpu
@pytest.mark.parametrize("r", [0, 3, 10, 30, 100])
def test_fused_statistics_conditioning(r):
    """conv1x1_fwd(stats) -> bn_apply_stats, the module's sequence, against float64 BatchNorm of the same fp32 conv
    output, for conv outputs whose per-channel mean is r standard deviations: one constant input channel whose weight is
    r * sigma_row. Asserted for r <= 10; r = 30 and 100 are reported (DESIGN 2)."""
    from pinthememory_b200 import capi

    B, K, M, hw = 8, 64, 256, 9216
    g = torch.Generator(device="cuda").manual_seed(77)
    A = torch.randn(M, K, generator=g, device="cuda") / 8
    A[:, K - 1] = r * A[:, : K - 1].norm(dim=1)
    x = torch.randn(B, K, 96, 96, generator=g, device="cuda")
    x[:, K - 1] = 1.0
    hi, lo = capi.conv1x1_prep(A.contiguous(), False, torch.float32)
    stats = torch.zeros(2 * M, dtype=torch.float64, device="cuda")
    z = capi.conv1x1_fwd(x, hi, lo, M, stats=stats)
    gamma, beta = torch.ones(M, device="cuda"), torch.zeros(M, device="cuda")
    y = torch.empty_like(z)
    mean, inv = torch.empty(M, device="cuda"), torch.empty(M, device="cuda")
    capi.bn_apply_stats(z, stats, B * hw, 1e-5, gamma, beta, None, y, False, mean, inv, None, None, 0.1)
    torch.cuda.synchronize()
    z64 = z.double()
    m64 = z64.mean((0, 2, 3))
    v64 = z64.var((0, 2, 3), unbiased=False)
    is64 = 1 / torch.sqrt(v64 + 1e-5)
    y64 = (z64 - m64.view(1, M, 1, 1)) * is64.view(1, M, 1, 1)
    e_inv = float(((inv.double() - is64).abs() / is64).max())
    print("conditioning r=%d: mean/std %.1f, max rel invstd error %.2e, y max abs error %.2e" % (
        r, float((m64.abs() / v64.sqrt()).median()), e_inv, float((y.double() - y64).abs().max())))
    if r <= 10:
        assert_close(y, y64, COND_TOL, "normalised output at r = %d" % r)
