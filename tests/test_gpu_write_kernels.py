"""The write kernels of csrc/pm_write.cu and csrc/pm_write_tiled.cu kernel by kernel, against float64 torch on the device.

Class sums (pm_write_reduce_fwd[8][_ordered]), the write backward (pm_write_bwd[8]) and the writing net's fused passes
(pm_write_reduce_bn_fwd[_ordered], pm_write_bwd_bn), called through ctypes with the structure and the two tiers of
test_gpu_read_kernels.py (whose host logic this file shares): every case names its route, the routing test pins what each
case launches and that together they launch every write instantiation of the library.

The label geometries are the ones the down-sampling meets: identity, integer ratio, the cfg shapes' 767/95, labels coarser
than the features, a non-integer ratio, h = 1 / w = 1 (scale 0) and Hm = 1 / Wm = 1; the label values include 255, values
out of range (counted as ignore), a class absent from the batch and an image that is all ignore, as int64 and as the
packed uint8 map of pm_labels_pack. The exact tier (four +-1 features, dyadic dS, dyadic tap weights) pins S, D and df bit
for bit in every mode, atomic ones included; SD is pre-filled with a pattern and must come back as pattern + sums, its
unused columns C+1..C+3 untouched."""
from fractions import Fraction

import pytest
import torch

from golden_util import rel_l2
from test_gpu_gemm_kernels import Guarded, _lib, _ok, _stream
from test_gpu_read_kernels import (BF16_SPLIT, BF16_U, DT, N0, NORM_EPS, U24, _code, _guard_in, _shapes, a_ratio, case_id,
                                   family, four_signs, launched_kernels, library_kernels, nchw, rows_of, rw_instantiations,
                                   scaled, sixteenths, unchanged)

gpu = pytest.mark.gpu

WS_WORDS = 40
# Element-wise bounds as in test_gpu_read_kernels.py; each A about twice the largest ratio measured on an NVIDIA B200
# (1000 W power limit) over every case below (DESIGN 2).
A_SD = 0.125   # class sums S and soft counts D     measured 0.056 (S), < 5e-4 (D)
A_DF = 0.3     # df = (dv - v (v.dv)) / |f|, and g  measured 0.14 (df), 0.06 (g)
A_BN = 0.01    # dgamma / dbeta of pm_write_bwd_bn  measured < 5e-4 beyond the summed bound of g


# ------------------------------------------------------------------------------------------------ geometry, labels
def label_dim(kind, n):
    """Label size along an axis of n feature pixels for geometry `kind` (scale = (Hm - 1) / (h - 1))."""
    if n == 1:
        return 5                                   # scale 0 whatever the label size
    return {"identity": n, "x2": 2 * (n - 1) + 1, "cfg": 8 * n,
            "half": (n - 1) // 2 + 1, "x1.5": (3 * (n - 1)) // 2 + 1, "label_line": 1}[kind]


GEOMS = ["identity", "x2", "cfg", "half", "x1.5", "label_line"]


def geometry(kind, h, w):
    Hm = label_dim(kind, h)
    Wm = w if kind == "label_line" else label_dim(kind, w)
    return Hm, Wm


def dyadic(h, w, Hm, Wm):
    """Tap weights exact in fp32: both scales are dyadic rationals (or 0)."""
    for n, m in ((h, Hm), (w, Wm)):
        if n > 1:
            d = Fraction(m - 1, n - 1).denominator
            if d & (d - 1):
                return False
    return True


def axis_taps(n_out, n_in):
    """(i0, i1, lambda) of src_index in fp32, as the kernels form them."""
    scale = (torch.tensor(float(n_in - 1)) / torch.tensor(float(n_out - 1))) if n_out > 1 else torch.tensor(0.0)
    src = scale * torch.arange(n_out, dtype=torch.float32)
    i0 = src.trunc().long().clamp(max=n_in - 1)
    lam = (src - i0.float()).clamp(0.0, 1.0)
    i1 = i0 + (i0 < n_in - 1).long()
    return i0, i1, lam


def soft_weights(cls, K, h, w):
    """omega [B, h*w, K+1] (float64) of the <= 4 bilinear taps, class map `cls` [B, Hm, Wm] in 0..K (K = ignore), weights
    in fp32 as the kernels compute them; and `touch` [B, h*w, K+1]: classes at any of the four tap positions."""
    B, Hm, Wm = cls.shape
    y0, y1, ly = axis_taps(h, Hm)
    x0, x1, lx = axis_taps(w, Wm)
    dev = cls.device
    y0, y1, x0, x1 = y0.to(dev), y1.to(dev), x0.to(dev), x1.to(dev)
    ly, lx = ly.to(dev).view(h, 1), lx.to(dev).view(1, w)
    hy0, hx0 = 1.0 - ly, 1.0 - lx
    wts = [hy0 * hx0, hy0 * lx, ly * hx0, ly * lx]                   # fp32 products
    pos = [(y0, x0), (y0, x1), (y1, x0), (y1, x1)]
    om = torch.zeros(B, h * w, K + 1, dtype=torch.float64, device=dev)
    touch = torch.zeros(B, h * w, K + 1, dtype=torch.bool, device=dev)
    for wt, (yy, xx) in zip(wts, pos):
        c = cls[:, yy][:, :, xx].reshape(B, h * w)
        om.scatter_add_(2, c.unsqueeze(2), wt.double().reshape(1, h * w, 1).expand(B, h * w, 1).contiguous())
        touch.scatter_(2, c.unsqueeze(2), True)
    return om, touch


def make_labels(B, Hm, Wm, K, gen):
    """int64 labels: blocky classes, 255 and out-of-range values sprinkled in, class K-1 absent (K > 1), the last image
    all ignore (B > 1)."""
    dev = "cuda"
    yy = torch.arange(Hm, device=dev).view(Hm, 1) // max(1, Hm // 5)
    xx = torch.arange(Wm, device=dev).view(1, Wm) // max(1, Wm // 7)
    base = torch.stack([((yy * 3 + xx * 5 + b) % K).expand(Hm, Wm) for b in range(B)])
    if K > 1:
        base = torch.where(base == K - 1, torch.zeros_like(base), base)
    r = torch.rand(B, Hm, Wm, generator=gen, device=dev)
    base = torch.where(r < 0.1, torch.full_like(base, 255), base)
    noise = torch.randint(0, K, (B, Hm, Wm), generator=gen, device=dev)
    if K > 1:
        noise = torch.where(noise == K - 1, torch.zeros_like(noise), noise)
    base = torch.where((r >= 0.1) & (r < 0.2), noise, base)
    bad = torch.tensor([K + 3, 1000, -3, 254], device=dev)
    base = torch.where((r >= 0.2) & (r < 0.24), bad[torch.randint(0, 4, (B, Hm, Wm), generator=gen, device=dev)], base)
    if B > 1:
        base[-1] = 255
    return base.long().contiguous()


def class_map(lab, K):
    return torch.where((lab >= 0) & (lab < K), lab, torch.full_like(lab, K))


def pack_labels(lab, K):
    ws = torch.zeros(WS_WORDS, dtype=torch.int64, device="cuda")
    lab8 = torch.empty(lab.shape, dtype=torch.uint8, device="cuda")
    _ok(_lib().pm_labels_pack(lab.data_ptr(), 0, lab.numel(), K, lab8.data_ptr(), ws.data_ptr(), _stream()), "pm_labels_pack")
    torch.cuda.synchronize()
    assert torch.equal(lab8.long(), class_map(lab, K)), "packed map"
    return lab8


# ----------------------------------------------------------------------------------------------------- case tables
def _write_cases():
    cases, i = [], 0
    extra = {"row_h1": (2, 1, 40), "col_w1": (2, 45, 1)}
    for dtype in DT:
        sh = list(_shapes(dtype).items()) + [("row_h1", extra["row_h1"])]
        gsh = [("odd_hw_b3", (3, 7, 9)), ("px_tail", (2, 10, 13)), ("col_w1", extra["col_w1"]), ("aligned_off", (2, 16, 24))]
        for C in (32, 64, 128, 256):
            for KP in (20, 32):
                for ordered in (False, True):
                    K = {20: [19, 1, 7], 32: [20, 31, 25]}[KP][i % 3]
                    name, (B, h, w) = sh[i % len(sh)]
                    geo = "cfg" if name == "cfg2" else GEOMS[i % len(GEOMS)]
                    if dtype == torch.float32:
                        route = {"write_reduce_mma_kernel"}
                    elif C >= 64:
                        route = {"write_reduce_mma16_kernel"}
                    else:
                        route = {"write_reduce_tiled_kernel"}
                    red = {"reduce_partials_kernel"} if ordered else set()
                    cases.append(("write_reduce", dtype, C, K, B, h, w, dict(geo=geo, u8=i % 2 == 0, ordered=ordered), route | red))
                    gname, (B, h, w) = gsh[i % len(gsh)]
                    off = 1 if gname == "aligned_off" else 0
                    cases.append(("write_reduce", dtype, C, {20: [1, 19, 7], 32: [31, 20, 25]}[KP][i % 3], B, h, w,
                                  dict(geo=GEOMS[(i + 2) % len(GEOMS)], u8=i % 2 == 1, ordered=ordered, off=off),
                                  {"write_reduce_kernel"} | red))
                    if not ordered:
                        name, (B, h, w) = sh[(i + 2) % len(sh)]
                        geo = "cfg" if name == "cfg2" else GEOMS[(i + 1) % len(GEOMS)]
                        cases.append(("write_bwd", dtype, C, K, B, h, w, dict(geo=geo, u8=i % 2 == 1), {"write_bwd_tiled_kernel"}))
                        gname, (B, h, w) = gsh[(i + 1) % len(gsh)]
                        off = 1 if gname == "aligned_off" else 0
                        cases.append(("write_bwd", dtype, C, K, B, h, w, dict(geo=GEOMS[(i + 3) % len(GEOMS)], u8=i % 2 == 0, off=off),
                                      {"write_bwd_kernel"}))
                    i += 1
    for C in (32, 64, 128, 256):                   # the writing net's fused passes: fp32, pipelined only
        for j, KP in enumerate((20, 32)):
            K = {20: 19, 32: 31}[KP] if C in (32, 128) else {20: 1, 32: 20}[KP]
            name, (B, h, w) = list(_shapes(torch.float32).items())[(C // 32 + j) % 6]
            geo = "cfg" if name == "cfg2" else GEOMS[(C // 32 + j) % len(GEOMS)]
            cases.append(("write_reduce_bn", torch.float32, C, K, B, h, w, dict(geo=geo, u8=j == 1, ordered=j == 1),
                          {"write_reduce_mma_kernel"} | ({"reduce_partials_kernel"} if j == 1 else set())))
            cases.append(("write_bwd_bn", torch.float32, C, K, B, h, w, dict(geo=geo, u8=j == 0),
                          {"write_bwd_tiled_kernel", "bn_sums_finalize_kernel"}))
    return cases


WRITE_CASES = _write_cases()
REDUCE_CASES = [c for c in WRITE_CASES if c[0] == "write_reduce"]
BWD_CASES = [c for c in WRITE_CASES if c[0] == "write_bwd"]
BN_CASES = [c for c in WRITE_CASES if c[0] in ("write_reduce_bn", "write_bwd_bn")]
WRITE_FAMILIES = {"write_reduce_kernel", "write_bwd_kernel", "write_reduce_tiled_kernel", "write_reduce_mma_kernel",
                  "write_reduce_mma16_kernel", "write_bwd_tiled_kernel", "bn_sums_finalize_kernel"}


def _geo(case):
    entry, dtype, C, K, B, h, w, opts, _ = case
    return geometry(opts["geo"], h, w)


def _exact_ok(case):
    entry, dtype, C, K, B, h, w, opts, _ = case
    return dyadic(h, w, *_geo(case))


def write_route(c):
    entry, dtype, C, K, B, h, w, opts, _ = c
    return rw_instantiations(entry, dtype, C, K, h * w, aligned=not opts.get("off"), ordered=opts.get("ordered", False))


def every_write_instantiation():
    out = {"bn_sums_finalize_kernel"}
    for t in ("f32", "bf16"):
        for KP in (20, 32):
            for C in (32, 64, 128, 256):
                out |= {"write_reduce_kernel<%s,%d,%d,%s>" % (t, C, KP, o) for o in ("false", "true")}
                out |= {"write_bwd_kernel<%s,%d,%d>" % (t, C // 8, KP), "write_bwd_tiled_kernel<%s,%d,%d,false>" % (t, C, KP)}
                if t == "f32":
                    out.add("write_bwd_tiled_kernel<f32,%d,%d,true>" % (C, KP))
            out |= {"write_reduce_tiled_kernel<bf16,32,%d,%s>" % (KP, o) for o in ("false", "true")}
    for C in (32, 64, 128, 256):
        for o in ("false", "true"):
            out |= {"write_reduce_mma_kernel<%d,32,%s,%s>" % (C, o, bn) for bn in ("false", "true")}
            if C >= 64:
                out.add("write_reduce_mma16_kernel<%d,32,%s>" % (C, o))
    return out


# ------------------------------------------------------------------------------------------------- host-side tests
def test_write_case_tables_name_their_routes():
    wrong = [(case_id(c), sorted(c[8]), sorted(write_route(c))) for c in WRITE_CASES
             if {family(n) for n in write_route(c)} != c[8]]
    assert not wrong, wrong
    geos = {(c[7]["geo"], c[5] == 1 or c[6] == 1) for c in WRITE_CASES}
    assert {g for g, _ in geos} == set(GEOMS) and any(line for _, line in geos)
    assert {1, 19, 20, 31} <= {c[3] for c in REDUCE_CASES} and {1, 19, 20, 31} <= {c[3] for c in BWD_CASES}
    assert any(c[4] * c[5] * c[6] == 8 * 96 * 96 for c in REDUCE_CASES)


def test_write_cases_reach_every_write_instantiation():
    reached = set()
    for c in WRITE_CASES:
        reached |= write_route(c)
    reached = {n for n in reached if family(n) in WRITE_FAMILIES}
    every = every_write_instantiation()
    assert reached == every, (sorted(every - reached), sorted(reached - every))
    assert len(every) == 99


def test_write_instantiations_match_the_built_library():
    """No class-sum template compiled that no call can reach (the bf16 run-length kernel exists for C = 32 only), and no
    write template without a case."""
    got = library_kernels(WRITE_FAMILIES)
    if got is None:
        pytest.skip("no built library or no cuobjdump / c++filt")
    every = every_write_instantiation()
    assert got == every, ("in the library, not in the table:", sorted(got - every), "in the table, not built:", sorted(every - got))


def test_weight_emulation_is_torch_bilinear_on_dyadic_geometries():
    """The fp32 tap emulation above equals F.interpolate(align_corners=True) of the one-hot map wherever the weights are
    exact, so the float64 restatement is the reference's down-sampling."""
    import torch.nn.functional as F

    gen = torch.Generator().manual_seed(3)
    for h, w, Hm, Wm in ((7, 9, 13, 17), (9, 5, 5, 3), (1, 6, 4, 11), (5, 8, 1, 8), (96, 96, 191, 191)):
        assert dyadic(h, w, Hm, Wm)
        cls = torch.randint(0, 4, (2, Hm, Wm), generator=gen)
        om, _ = soft_weights(cls, 3, h, w)
        want = F.interpolate(F.one_hot(cls, 4).permute(0, 3, 1, 2).double(), [h, w], mode="bilinear", align_corners=True)
        assert torch.equal(om, want.permute(0, 2, 3, 1).reshape(2, h * w, 4))


# ----------------------------------------------------------------------------------------------- float64 pieces
def _features(case, tier, gen, zero_last=True):
    entry, dtype, C, K, B, h, w, opts, _ = case
    N = B * h * w
    fr = four_signs(N, C, gen, "cuda") if tier == "exact" else rows_of(scaled((B, C, h * w), 1, gen, "cuda"))
    if zero_last:
        fr[-1] = 0                                 # a zero feature vector in the last tile: the norm clamp
    return nchw(fr, B, h * w).to(dtype)


def _labels(case, gen):
    entry, dtype, C, K, B, h, w, opts, _ = case
    Hm, Wm = _geo(case)
    lab = make_labels(B, Hm, Wm, K, gen)
    return lab, (pack_labels(lab, K) if opts.get("u8") else lab), Hm, Wm


def _wtol(case):
    """Tap-weight uncertainty when the scale is not dyadic (the kernel may contract src - i0 into one FMA): half an ulp of
    the source coordinate, both axes, both factors of a weight."""
    if _exact_ok(case):
        return 0.0
    Hm, Wm = _geo(case)
    return 4 * U24 * max(Hm, Wm)


def unit_rows(f):
    """v = f / max(|f|, eps) over the channels of [B, C, hw], float64."""
    fd = f.double()
    return fd / fd.norm(dim=1, keepdim=True).clamp_min(NORM_EPS)


def _reduce_pixels(B, hw):
    """Upper bound of (pixels one CTA sums, CTAs added into SD): the grids are at least min(ntiles, 148)."""
    ntiles = B * -(-hw // 32)
    g = min(ntiles, 148)
    return -(-ntiles // g) * 32, min(ntiles, 4 * 148)


def _sd_pattern(K, C):
    return ((torch.arange((K + 1) * (C + 4), device="cuda", dtype=torch.float32) % 9 - 4) / 4).view(K + 1, C + 4)


def _check_sd(case, tier, SDk, pattern, v, om, touch, exact, split):
    """SD = pattern + [S | D | 0 0 0]: bit for bit in the exact tier, element-wise bound otherwise."""
    entry, dtype, C, K, B, h, w, opts, _ = case
    S64 = torch.einsum("bcp,bpk->kc", v, om)
    D64 = om.sum((0, 1))
    got = SDk.double() - pattern.double()
    assert torch.equal(SDk[:, C + 1:], pattern[:, C + 1:]), "columns C+1..C+3 of SD changed"
    if exact:
        assert torch.equal(got[:, :C], S64), "class sums differ from float64 (exact tier)"
        assert torch.equal(got[:, C], D64), "soft counts differ from float64 (exact tier)"
    # base: the n adds of a CTA (and the C-long norm of v); fixed: the operand split's residual (bf16 tensor-core path), the
    # tap-weight uncertainty of a non-dyadic scale, and the `grid` adds into SD, which starts at the pattern
    n, grid = _reduce_pixels(B, h * w)
    magS = torch.einsum("bcp,bpk->kc", v.abs(), om)
    wt = _wtol(case)
    extraS = wt * torch.einsum("bcp,bpk->kc", v.abs(), touch.double()) if wt else 0.0
    fS = split * magS + extraS + grid * U24 * (magS + pattern[:, :C].double().abs())
    fD = (wt * touch.double().sum((0, 1)) if wt else 0.0) + grid * U24 * (D64 + pattern[:, C].double().abs())
    rS = a_ratio((got[:, :C] - S64).abs(), fS, (n + C + N0) * U24 * magS)
    rD = a_ratio((got[:, C] - D64).abs(), fD, (n + N0) * U24 * D64)
    return rS, rD


def _run_reduce(case, f, lab_arg, Hm, Wm, SD):
    entry, dtype, C, K, B, h, w, opts, _ = case
    lib = _lib()
    u8 = bool(opts.get("u8"))
    scratch = None
    if opts.get("ordered"):
        nbytes = lib.pm_write_reduce_scratch_bytes(B, C, h, w, K)
        assert nbytes > 0 and nbytes % 16 == 0
        scratch = Guarded(nbytes // 4, torch.float32)
        fn = lib.pm_write_reduce_fwd8_ordered if u8 else lib.pm_write_reduce_fwd_ordered
        rc = fn(f.data_ptr(), lab_arg.data_ptr(), SD.t.data_ptr(), scratch.t.data_ptr(), B, C, h, w, Hm, Wm, K, _code(dtype), _stream())
    else:
        fn = lib.pm_write_reduce_fwd8 if u8 else lib.pm_write_reduce_fwd
        rc = fn(f.data_ptr(), lab_arg.data_ptr(), SD.t.data_ptr(), B, C, h, w, Hm, Wm, K, _code(dtype), _stream())
    _ok(rc, "pm_write_reduce_fwd")
    torch.cuda.synchronize()
    SD.check("SD")
    if scratch is not None:
        scratch.check("class-sum scratch", scratch=True)


def _guarded_sd(pattern):
    SD = Guarded(pattern.numel(), torch.float32, fill=None)
    SD.t.copy_(pattern.flatten())
    SD.ref = SD.buf.clone()
    return SD


# ------------------------------------------------------------------------------------------------------ class sums
@gpu
@pytest.mark.parametrize("tier", ["exact", "precision"])
@pytest.mark.parametrize("case", REDUCE_CASES, ids=case_id)
def test_write_reduce(case, tier):
    entry, dtype, C, K, B, h, w, opts, _ = case
    if tier == "exact" and not _exact_ok(case):
        pytest.skip("tap weights of this geometry are not dyadic: precision tier only")
    gen = torch.Generator(device="cuda").manual_seed(500 + C + K + B * h * w)
    f = _features(case, tier, gen)
    lab, lab_arg, Hm, Wm = _labels(case, gen)
    fg = _guard_in(f, opts.get("off", 0))
    pattern = _sd_pattern(K, C)
    SD = _guarded_sd(pattern)
    _run_reduce(case, fg.t, lab_arg, Hm, Wm, SD)
    om, touch = soft_weights(class_map(lab, K), K, h, w)
    v = unit_rows(f)
    split = BF16_SPLIT if (dtype == torch.bfloat16 and C >= 64 and not opts.get("off") and (h * w) % 8 == 0) else 0.0
    rS, rD = _check_sd(case, tier, SD.t.view(K + 1, C + 4), pattern, v, om, touch, tier == "exact", split)
    print("RATIO write_reduce %s %s S=%.3f D=%.3f" % (tier, case_id(case), rS, rD))
    assert rS <= A_SD and rD <= A_SD, (rS, rD)
    if opts.get("ordered"):                                  # bitwise reproducible
        SD2 = _guarded_sd(pattern)
        _run_reduce(case, fg.t, lab_arg, Hm, Wm, SD2)
        assert torch.equal(SD2.t.view(torch.int32), SD.t.view(torch.int32)), "ordered class sums not reproducible"


# -------------------------------------------------------------------------------------------------------- backward
def write_bwd_ref(f, om, touch, dS, K, wtol, C):
    """float64 df of pm_write_bwd on [N, C] rows and its bound (fixed, base): the <= 4 taps' sum dv, the projection and
    1/|f| (base); the tap-weight uncertainty of a non-dyadic scale (fixed)."""
    fd = f.double()
    n = fd.norm(dim=1, keepdim=True)
    ir = 1.0 / n.clamp_min(NORM_EPS)
    v = fd * ir
    dS1 = torch.cat([dS.double(), torch.zeros(1, C, dtype=torch.float64, device=dS.device)])   # ignore row
    dv = om @ dS1
    nz = (n > NORM_EPS).double()
    dot = (v * dv).sum(1, keepdim=True) * nz
    df = (dv - v * dot) * ir
    va = v.abs()
    inner = lambda e: e + va * (va * e).sum(1, keepdim=True) * nz
    fixed = ir * inner(wtol * (touch.double() @ dS1.abs())) if wtol else torch.zeros_like(df)
    base = ir * (inner(8 * U24 * (om @ dS1.abs())) + (C + N0) * U24 * inner(dv.abs()))
    return df, fixed, base


def _dS(K, C, tier, gen):
    return sixteenths((K, C), gen, "cuda") if tier == "exact" else scaled((K, C), 1, gen, "cuda")


@gpu
@pytest.mark.parametrize("tier", ["exact", "precision"])
@pytest.mark.parametrize("case", BWD_CASES, ids=case_id)
def test_write_bwd(case, tier):
    entry, dtype, C, K, B, h, w, opts, _ = case
    if tier == "exact" and not _exact_ok(case):
        pytest.skip("tap weights of this geometry are not dyadic: precision tier only")
    N, hw = B * h * w, h * w
    gen = torch.Generator(device="cuda").manual_seed(600 + C + K + N)
    f = _features(case, tier, gen, zero_last=tier == "precision")   # 1/eps is not a short fp32 value: precision tier only
    lab, lab_arg, Hm, Wm = _labels(case, gen)
    dS = _dS(K, C, tier, gen)
    off = opts.get("off", 0)
    fg = _guard_in(f)
    df = Guarded(B * C * hw, dtype, offset_bytes=off * torch.empty(0, dtype=dtype).element_size())
    fn = _lib().pm_write_bwd8 if opts.get("u8") else _lib().pm_write_bwd
    _ok(fn(dS.data_ptr(), fg.t.data_ptr(), lab_arg.data_ptr(), df.t.data_ptr(), B, C, h, w, Hm, Wm, K, _code(dtype), _stream()),
        "pm_write_bwd")
    torch.cuda.synchronize()
    df.check("df")
    assert unchanged(fg), "f modified"
    om, touch = soft_weights(class_map(lab, K), K, h, w)
    ref, fixed, base = write_bwd_ref(rows_of(f), om.view(N, K + 1), touch.view(N, K + 1), dS, K, _wtol(case), C)
    got = rows_of(df.t.view(B, C, hw))
    if tier == "exact":
        want = ref.to(dtype)
        bad = got != want
        assert not bool(bad.any()), "df differs from float64 (exact tier) at %d elements" % int(bad.sum())
    if dtype == torch.bfloat16:
        fixed = fixed + BF16_U * ref.abs()
    r = a_ratio((got.double() - ref).abs(), fixed, base)
    print("RATIO write_bwd %s %s df=%.3f" % (tier, case_id(case), r))
    assert r <= A_DF, r
    assert rel_l2(got, ref) <= (1e-5 if dtype == torch.float32 else 2 ** -8)


# ------------------------------------------------------------------------------------------ the writing net's passes
def _bn_inputs(case, gen):
    entry, dtype, C, K, B, h, w, opts, _ = case
    z = (scaled((B, C, h * w), 1, gen, "cuda", -2, 2) + 0.25).view(B, C, h, w).contiguous()
    x = torch.randn(B, C, h, w, generator=gen, device="cuda")
    gamma = torch.rand(C, generator=gen, device="cuda") + 0.5
    beta = torch.randn(C, generator=gen, device="cuda") * 0.3
    z64 = z.double()
    stats = torch.cat([z64.sum((0, 2, 3)), (z64 * z64).sum((0, 2, 3)), torch.zeros(1, device="cuda", dtype=torch.float64)])
    return z, x, gamma, beta, stats


def _bn_f(z, x, stats, gamma, beta, n):
    """f = relu(x + BN(z)) and the statistics from pm_bn_apply_stats: the map the fused passes form in shared memory."""
    from pinthememory_b200 import capi

    C = z.shape[1]
    f = torch.empty_like(z)
    mean, inv = torch.empty(C, device="cuda"), torch.empty(C, device="cuda")
    rm, rv = torch.zeros(C, device="cuda"), torch.ones(C, device="cuda")
    capi.bn_apply_stats(z, stats, n, 1e-5, gamma, beta, x, f, True, mean, inv, rm, rv, 0.1)
    torch.cuda.synchronize()
    return f, mean, inv


@gpu
@pytest.mark.parametrize("case", BN_CASES, ids=case_id)
def test_write_bn(case):
    """pm_write_reduce_bn_fwd[_ordered]: class sums of relu(x + BN(z)) against float64 (pattern + sums), the statistics those
    of pm_bn_apply_stats. pm_write_bwd_bn: g = df [f > 0] against float64, dgamma / dbeta against the float64 sums of g."""
    entry, dtype, C, K, B, h, w, opts, _ = case
    N, hw = B * h * w, h * w
    lib = _lib()
    gen = torch.Generator(device="cuda").manual_seed(700 + C + K + N)
    z, x, gamma, beta, stats = _bn_inputs(case, gen)
    lab, lab_arg, Hm, Wm = _labels(case, gen)
    u8 = int(bool(opts.get("u8")))
    f, mean, inv = _bn_f(z, x, stats, gamma, beta, N)
    om, touch = soft_weights(class_map(lab, K), K, h, w)
    zg, xg = _guard_in(z), _guard_in(x)
    if entry == "write_reduce_bn":
        pattern = _sd_pattern(K, C)
        SD = _guarded_sd(pattern)
        mean_o, inv_o = Guarded(C, torch.float32), Guarded(C, torch.float32)
        rm, rv = torch.zeros(C, device="cuda"), torch.ones(C, device="cuda")
        nbt = torch.zeros((), dtype=torch.int64, device="cuda")
        common = (stats.data_ptr(), float(N), None, 1e-5, gamma.data_ptr(), beta.data_ptr(), mean_o.t.data_ptr(), inv_o.t.data_ptr(),
                  rm.data_ptr(), rv.data_ptr(), 0.1, nbt.data_ptr(), B, C, h, w, Hm, Wm, K, _stream())
        scratch = None
        if opts.get("ordered"):
            scratch = Guarded(lib.pm_write_reduce_scratch_bytes(B, C, h, w, K) // 4, torch.float32)
            rc = lib.pm_write_reduce_bn_fwd_ordered(zg.t.data_ptr(), xg.t.data_ptr(), lab_arg.data_ptr(), u8, SD.t.data_ptr(),
                                                    scratch.t.data_ptr(), *common)
        else:
            rc = lib.pm_write_reduce_bn_fwd(zg.t.data_ptr(), xg.t.data_ptr(), lab_arg.data_ptr(), u8, SD.t.data_ptr(), *common)
        _ok(rc, entry)
        torch.cuda.synchronize()
        for g, what in ((SD, "SD"), (mean_o, "mean"), (inv_o, "invstd")):
            g.check(what)
        if scratch is not None:
            scratch.check("scratch", scratch=True)
        assert torch.equal(mean_o.t, mean) and torch.equal(inv_o.t, inv) and int(nbt) == 1
        v = unit_rows(f.view(B, C, hw))
        rS, rD = _check_sd(case, "precision", SD.t.view(K + 1, C + 4), pattern, v, om, touch, False, 0.0)
        print("RATIO write_reduce_bn %s S=%.3f D=%.3f" % (case_id(case), rS, rD))
        assert rS <= A_SD and rD <= A_SD, (rS, rD)
        return
    dS = scaled((K, C), 1, gen, "cuda", -2, 2)
    g = Guarded(N * C, torch.float32)
    dgamma, dbeta = Guarded(C, torch.float32), Guarded(C, torch.float32)
    scratch = Guarded(lib.pm_write_bwd_bn_scratch_bytes(C) // 4, torch.float32)
    rc = lib.pm_write_bwd_bn(dS.data_ptr(), zg.t.data_ptr(), xg.t.data_ptr(), lab_arg.data_ptr(), u8, mean.data_ptr(), inv.data_ptr(),
                             gamma.data_ptr(), beta.data_ptr(), g.t.data_ptr(), dgamma.t.data_ptr(), dbeta.t.data_ptr(),
                             scratch.t.data_ptr(), B, C, h, w, Hm, Wm, K, _stream())
    _ok(rc, entry)
    torch.cuda.synchronize()
    for t, what in ((g, "g"), (dgamma, "dgamma"), (dbeta, "dbeta")):
        t.check(what)
    scratch.check("scratch", scratch=True)
    fr = rows_of(f.view(B, C, hw))
    df64, fixed, base = write_bwd_ref(fr, om.view(N, K + 1), touch.view(N, K + 1), dS, K, _wtol(case), C)
    bound = fixed + A_DF * base
    gate = (fr > 0).double()
    g64 = df64 * gate
    got = rows_of(g.t.view(B, C, hw))
    assert bool((got[fr <= 0] == 0).all()), "g is not 0 where f <= 0"
    r_g = a_ratio((got.double() - g64).abs(), fixed * gate, base * gate)
    mu, isd = mean.double(), inv.double()
    xhat = (rows_of(z.view(B, C, hw)).double() - mu) * isd
    n_cta = -(-B * -(-hw // 32) // min(B * -(-hw // 32), 296)) * 32
    # base: a CTA's fp32 sums over its tiles; fixed: the bound of g itself, summed
    r_b = a_ratio((dbeta.t.double() - g64.sum(0)).abs(), (bound * gate).sum(0), (n_cta + N0) * U24 * g64.abs().sum(0))
    r_gm = a_ratio((dgamma.t.double() - (g64 * xhat).sum(0)).abs(), (bound * gate * xhat.abs()).sum(0),
                   (n_cta + N0) * U24 * (g64 * xhat).abs().sum(0))
    print("RATIO write_bwd_bn %s g=%.3f dbeta=%.3f dgamma=%.3f" % (case_id(case), r_g, r_b, r_gm))
    assert r_g <= A_DF and r_b <= A_BN and r_gm <= A_BN, (r_g, r_b, r_gm)


# ------------------------------------------------------------------------------------------------------- routing
def _dry_write(case):
    entry, dtype, C, K, B, h, w, opts, _ = case
    N, hw = B * h * w, h * w
    lib, code, st = _lib(), _code(dtype), _stream()
    off = opts.get("off", 0)
    Hm, Wm = _geo(case)
    lab = torch.zeros(B, Hm, Wm, dtype=torch.uint8 if opts.get("u8") else torch.int64, device="cuda")
    u8 = int(bool(opts.get("u8")))
    f = torch.zeros(N * C + 8, dtype=dtype, device="cuda")[off:off + N * C]
    SD = torch.zeros(K + 1, C + 4, device="cuda")
    if entry == "write_reduce":
        if opts.get("ordered"):
            scr = torch.zeros(lib.pm_write_reduce_scratch_bytes(B, C, h, w, K) // 4, device="cuda")
            fn = lib.pm_write_reduce_fwd8_ordered if u8 else lib.pm_write_reduce_fwd_ordered
            return lambda: _ok(fn(f.data_ptr(), lab.data_ptr(), SD.data_ptr(), scr.data_ptr(), B, C, h, w, Hm, Wm, K, code, st), entry)
        fn = lib.pm_write_reduce_fwd8 if u8 else lib.pm_write_reduce_fwd
        return lambda: _ok(fn(f.data_ptr(), lab.data_ptr(), SD.data_ptr(), B, C, h, w, Hm, Wm, K, code, st), entry)
    dS = torch.zeros(K, C, device="cuda")
    if entry == "write_bwd":
        df = torch.zeros(N * C, dtype=dtype, device="cuda")
        fn = lib.pm_write_bwd8 if u8 else lib.pm_write_bwd
        return lambda: _ok(fn(dS.data_ptr(), f.data_ptr(), lab.data_ptr(), df.data_ptr(), B, C, h, w, Hm, Wm, K, code, st), entry)
    vec = lambda v: torch.full((C,), v, device="cuda")
    z, x = torch.zeros(N * C, device="cuda"), torch.zeros(N * C, device="cuda")
    if entry == "write_reduce_bn":
        keep = [torch.zeros(2 * C + 1, dtype=torch.float64, device="cuda"), vec(1.0), vec(0.0), vec(0.0), vec(0.0), vec(0.0), vec(1.0)]
        stats, ga, be, mo, io, rm, rv = keep
        common = (stats.data_ptr(), float(N), None, 1e-5, ga.data_ptr(), be.data_ptr(), mo.data_ptr(), io.data_ptr(), rm.data_ptr(),
                  rv.data_ptr(), 0.1, None, B, C, h, w, Hm, Wm, K, st)
        if opts.get("ordered"):
            keep.append(torch.zeros(lib.pm_write_reduce_scratch_bytes(B, C, h, w, K) // 4, device="cuda"))
            return lambda keep=keep: _ok(lib.pm_write_reduce_bn_fwd_ordered(z.data_ptr(), x.data_ptr(), lab.data_ptr(), u8,
                                                                            SD.data_ptr(), keep[-1].data_ptr(), *common), entry)
        return lambda keep=keep: _ok(lib.pm_write_reduce_bn_fwd(z.data_ptr(), x.data_ptr(), lab.data_ptr(), u8, SD.data_ptr(),
                                                                *common), entry)
    gm, gi, ga, be, dg, db = vec(0.0), vec(1.0), vec(1.0), vec(0.0), vec(0.0), vec(0.0)
    g = torch.zeros(N * C, device="cuda")
    scr = torch.zeros(lib.pm_write_bwd_bn_scratch_bytes(C) // 4, device="cuda")
    return lambda: _ok(lib.pm_write_bwd_bn(dS.data_ptr(), z.data_ptr(), x.data_ptr(), lab.data_ptr(), u8, gm.data_ptr(), gi.data_ptr(),
                                           ga.data_ptr(), be.data_ptr(), g.data_ptr(), dg.data_ptr(), db.data_ptr(), scr.data_ptr(),
                                           B, C, h, w, Hm, Wm, K, st), entry)


@gpu
def test_write_routing():
    """Each case launches exactly the predicted instantiations; together: every write instantiation, BN and ORD included."""
    wrong, reached = [], set()
    for case in WRITE_CASES:
        got = launched_kernels(_dry_write(case))
        want = write_route(case)
        if got != want:
            wrong.append((case_id(case), sorted(got), sorted(want)))
        reached |= got
    assert not wrong, wrong
    reached = {n for n in reached if family(n) in WRITE_FAMILIES}
    assert reached == every_write_instantiation(), sorted(every_write_instantiation() - reached)
