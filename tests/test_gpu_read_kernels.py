"""The read kernels of csrc/pm_read.cu and csrc/pm_read_tiled.cu kernel by kernel, against float64 torch on the device.

Entries are called through ctypes, never through the module. Every case names the route it is written to reach (the
generic one-launch kernels, the pipelined tile kernels, the score-plane variants); `rw_instantiations` states which
kernel instantiations a call launches, `test_read_case_tables_name_their_routes` checks the tables against it on the host
and `test_read_routing` against what the profiler sees on the GPU. A pipelined shape reaches the generic kernel when one
pointer is moved off 16-byte alignment by one element inside its guarded buffer.

Two tiers, as for the GEMMs. The exact tier uses feature vectors with four +-1 entries (|x| = 2, 1/|x| = 0.5) and
memory rows in multiples of 1/16, so every TF32 / bf16 split is exact (lo parts 0) and every sum is exact: s, its
padding and the q half of u must equal float64 bit for bit (bf16 outputs: the float64 value rounded to bf16). The
precision tier uses Gaussian data with 2^-8..2^8 scales per channel (and per slot for the memory), so a channel or slot
mix-up shows element by element, and bounds each output element-wise by A * (n + N0) * 2^-24 * mag, mag being the same
expression in float64 on absolute values (DESIGN 2). CPU tests show that these bounds reject the plausible wrong kernels
(1-pass TF32, 3xTF32 without a cross term, bf16 memory without its lo part, exp in bf16 precision) at every shape used.

Every output sits between guard bands that must stay untouched; overwritten outputs are pre-filled with NaN, accumulated
ones (dM) with a known pattern that must come back as pattern + sum."""
import os
import re
import shutil
import subprocess

import pytest
import torch

from golden_util import rel_l2
from test_gpu_gemm_kernels import Guarded, _lib, _ok, _stream

gpu = pytest.mark.gpu

PM_F32, PM_BF16 = 0, 1
NORM_EPS = 1e-12
U24 = 2.0 ** -24
BF16_U = 2.0 ** -8        # half a bf16 ulp, relative
BF16_SPLIT = 2.0 ** -16   # hi + lo bf16 split of an fp32 operand: |v - hi - lo| <= 2^-17 |v|, two operands
PLANES = 32
COLPART_ROWS = 296

# ------------------------------------------------------------------------------------------------- tolerances
# Element-wise bound |y - y64| <= fixed + A * (n + N0) * 2^-24 * mag: `fixed` holds the propagated bounds of the inputs, the
# final bf16 rounding and the adds into a pre-filled output; N0 covers the per-element roundings that do not grow with the
# contraction length n (1/|x|, the softmax's exp and division). Each A is about twice the largest ratio
# (err - fixed) / ((n + N0) 2^-24 mag) measured on an NVIDIA B200 (1000 W power limit) over every case below (DESIGN 2).
N0 = 16
A_S = 0.5      # s = q.M^T and q = x/|x|            measured 0.22 (s), 0.08 (q)
A_P = 0.5      # score_memory = softmax(s + g)      measured 0.22
A_C = 0.5      # p.M, the second half of u          measured 0.19
A_DS = 0.4     # ds = p (dp - p.dp) + scale ds_rl   measured 0.17
A_DX = 0.25    # dx = (dq - q (q.dq)) / |x|         measured 0.11
A_DM = 0.05    # dM = p^T dc + ds^T q               measured 0.025
A_COL = 0.5    # 1/sum of col_partials              measured 0.21


# ----------------------------------------------------------------------------------------------- host logic
def kp_of(K):
    return 20 if K <= 19 else 32


def _tn(dtype):
    return "f32" if dtype == torch.float32 else "bf16"


def rw_instantiations(entry, dtype, C, K, hw, aligned=True, ordered=False, dx_add=False, ds=True, col_partials=False):
    """The kernel instantiations (demangled, types as f32 / bf16, no spaces) one call of `entry` launches, as the
    launchers of pm_read*.cu / pm_write*.cu pick them. `aligned`: every feature pointer 16-byte aligned."""
    T, KP, o = _tn(dtype), kp_of(K), "true" if ordered else "false"
    tiled = aligned and hw % (4 if dtype == torch.float32 else 8) == 0
    red = {"reduce_partials_kernel<f32>"} if ordered else set()

    def dx_kernel():
        if T == "bf16" and C >= 128 and not dx_add:
            return "read_bwd_dx_bf16_kernel<%d,%d,2>" % (C, KP)
        return "read_bwd_dx_tma_kernel<%s,%d,%d,2>" % (T, C, KP)

    if entry in ("read_fwd", "read_fwd_planes"):
        if tiled or entry == "read_fwd_planes":
            return {"read_fwd_tiled_kernel<%s,%d,%d,2>" % (T, C, KP)}
        extra = {"colsoftmax_stats_kernel", "colsoftmax_combine_kernel"} if col_partials else set()
        return {"read_fwd_kernel<%s,%d,%d>" % (T, C // 8, KP)} | extra
    if entry == "read_bwd":
        if not (tiled and ds):
            return {"read_bwd_kernel<%s,%d,%d>" % (T, C // 8, KP)}
        return {"read_bwd_ds_tiled_kernel<%s,%d,%d,2>" % (T, C, KP), dx_kernel()}
    if entry == "read_bwd_planes":
        return {"read_bwd_ds_planes_kernel<%s,%d>" % (T, KP), dx_kernel()}
    if entry == "read_dM":
        return {"read_bwd_dM_kernel<%s,%d,%d,%s>" % (T, C, KP, o)} | red
    if entry == "write_reduce":
        if not tiled:
            k = "write_reduce_kernel<%s,%d,%d,%s>" % (T, C, KP, o)
        elif T == "f32":
            k = "write_reduce_mma_kernel<%d,32,%s,false>" % (C, o)
        elif C >= 64:
            k = "write_reduce_mma16_kernel<%d,32,%s>" % (C, o)
        else:
            k = "write_reduce_tiled_kernel<bf16,32,%d,%s>" % (KP, o)
        return {k} | red
    if entry == "write_bwd":
        return {("write_bwd_tiled_kernel<%s,%d,%d,false>" % (T, C, KP)) if tiled else
                ("write_bwd_kernel<%s,%d,%d>" % (T, C // 8, KP))}
    if entry == "write_reduce_bn":
        return {"write_reduce_mma_kernel<%d,32,%s,true>" % (C, o)} | red
    if entry == "write_bwd_bn":
        return {"write_bwd_tiled_kernel<f32,%d,%d,true>" % (C, KP), "bn_sums_finalize_kernel"}
    raise ValueError(entry)


def family(name):
    return name.split("<")[0]


def normalize_kernel_name(demangled):
    """'void pm::read_fwd_tiled_kernel<__nv_bfloat16, 64, 20, 2>(CUtensorMap_st, ...)' -> 'read_fwd_tiled_kernel<bf16,64,20,2>';
    None for a kernel outside namespace pm."""
    name = re.sub(r"\(.*", "", demangled).replace("void ", "").strip()
    if not name.startswith("pm::"):
        return None
    return name[4:].replace(" ", "").replace("__nv_bfloat16", "bf16").replace("float", "f32")


def library_kernels(families):
    """Normalised names of every kernel of `families` compiled into the built library (cuobjdump's function list), or
    None when the library or the tools are missing."""
    from pinthememory_b200 import build

    lib, tool, filt = build.LIB_PATH, shutil.which("cuobjdump") or "/usr/local/cuda/bin/cuobjdump", shutil.which("c++filt")
    if not (os.path.exists(lib) and os.path.exists(tool) and filt):
        return None
    out = subprocess.run([tool, "-elf", lib], capture_output=True, text=True).stdout
    mangled = sorted(set(re.findall(r"\.text\.(_Z\S+)", out)))
    if not mangled:
        return None
    names = subprocess.run([filt], input="\n".join(mangled), capture_output=True, text=True).stdout.splitlines()
    got = {normalize_kernel_name(n) for n in names}
    return {n for n in got if n is not None and family(n) in families}


def launched_kernels(fn):
    """Normalised names of the pm:: kernels `fn` launches (torch.profiler)."""
    from torch.profiler import ProfilerActivity, profile

    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    got = set()
    for e in prof.events():
        if e.device_type == torch.autograd.DeviceType.CUDA:
            n = normalize_kernel_name(e.name)
            if n is not None:
                got.add(n)
    return got


def tf32_rn(t):
    return ((t.view(torch.int32) + 0x1000) & ~0x1FFF).view(torch.float32)


def tf32_trunc(t):
    return (t.view(torch.int32) & ~0x1FFF).view(torch.float32)


def scaled(shape, axis, gen, device, lo=-8, hi=8):
    """Gaussian values times 2^e, e uniform in lo..hi along `axis`."""
    t = torch.randn(*shape, generator=gen, device=device)
    e = torch.randint(lo, hi + 1, (shape[axis],), generator=gen, device=device).double()
    view = [1] * len(shape)
    view[axis] = shape[axis]
    return (t * torch.exp2(e).float().view(view)).contiguous()


def four_signs(N, C, gen, device):
    """[N, C] rows with exactly four +-1 entries: |x| = 2 exactly."""
    pick = torch.rand(N, C, generator=gen, device=device).argsort(dim=1)[:, :4]
    sign = torch.randint(0, 2, (N, 4), generator=gen, device=device).float() * 2 - 1
    x = torch.zeros(N, C, device=device)
    x.scatter_(1, pick, sign)
    return x


def sixteenths(shape, gen, device, lim=32):
    """Multiples of 1/16 in [-2, 2]: at most 6 significant bits, so TF32 / bf16 hi parts are the values."""
    return torch.randint(-lim, lim + 1, shape, generator=gen, device=device).float() / 16


def nchw(rows, B, hw):
    """[B*hw, C] pixel rows -> [B, C, hw] contiguous."""
    return rows.view(B, hw, -1).permute(0, 2, 1).contiguous()


def rows_of(t):
    """[B, C, hw] -> [B*hw, C]."""
    return t.permute(0, 2, 1).reshape(-1, t.shape[1])


def _code(dtype):
    return PM_F32 if dtype == torch.float32 else PM_BF16


def _esz(dtype):
    return torch.empty(0, dtype=dtype).element_size()


def _guard_in(t, offset_elems=0):
    """A copy of input `t` inside a guarded buffer (optionally one element off 16-byte alignment)."""
    g = Guarded(t.numel(), t.dtype, fill=None, offset_bytes=offset_elems * _esz(t.dtype))
    g.t.copy_(t.flatten())
    g.ref = g.buf.clone()
    return g


def unchanged(g):
    """An input's guarded buffer, guards included, bit for bit as it was filled (the guards' random bits may be NaNs)."""
    return torch.equal(g.buf.view(torch.uint8), g.ref.view(torch.uint8))


def ratio(err, bound):
    return float((err / bound.clamp_min(1e-300)).max()) if err.numel() else 0.0


def a_ratio(err, fixed, base):
    """The smallest A with err <= fixed + A * base everywhere: `fixed` holds what does not scale with the calibrated
    constant (propagated input bounds, the final bf16 rounding, atomics onto a pre-filled output)."""
    return ratio((err - fixed).clamp_min(0.0), base)


FTZ_FLOOR = 2.0 ** -125   # the softmax's ex2.approx.ftz and fp32 products flush results below 2^-126 to zero


# ------------------------------------------------------------------------------------------------ case tables
# A case: (entry, dtype, C, K, B, h, w, opts, route). `opts`: off = the one-element offset that moves a pointer off 16-byte
# alignment (the generic kernel at a pipelined shape), gumbel, colpart, rl (the read-loss term of the backward), dx_add,
# ds_null (pm_read_bwd with ds == NULL), ordered. `route`: the kernel families the case is written to reach.
#
# Shapes: one partly filled tile (hw = 4 / 8, one CTA); tail tiles at image boundaries (hw % 32 != 0, B > 1); ntiles one
# above the persistent grids (296 for the forward and the ds pass: 297 tiles; 148 for the fp32 dx and dM: 149 tiles);
# cfg-2 (B = 8 at 96 x 96: ~8 tiles per CTA, the rings wrap many times); ntiles below the grid. Slots: K = 1, 19 (one pad
# slot of KP = 20), 20 (twelve pad slots of KP = 32), 31 (one pad slot of KP = 32).
def _shapes(dtype):
    f32 = dtype == torch.float32
    return {
        "one_tile": (1, 2, 2) if f32 else (1, 2, 4),
        "tails_b3": (3, 10, 10) if f32 else (3, 8, 13),
        "grid296_plus1": (1, 92, 103) if f32 else (1, 79, 120),     # 296 * 32 + 4 / + 8 pixels: 297 tiles
        "grid148_plus1": (1, 60, 79) if f32 else (1, 8, 593),       # 148 * 32 + 4 / + 8 pixels: 149 tiles
        "cfg2": (8, 96, 96),
        "few_tiles": (2, 8, 16),
    }


GENERIC_SHAPES = {                     # the generic kernels' 64-pixel tiles (the dM kernel: 32-pixel tiles)
    "odd_hw_b3": (3, 7, 9),            # hw = 63: no pipelined variant at all
    "px64_tail": (2, 10, 13),          # hw = 130: a 2-pixel tail tile per image
    "aligned_hw_off": (2, 16, 24),     # hw = 384 (a pipelined shape), reached through the offset pointer
}
K_BY_KP = {20: [19, 1, 7], 32: [20, 31, 25]}
CS = (32, 64, 128, 256)
DT = (torch.float32, torch.bfloat16)


def _read_fwd_cases():
    cases, i = [], 0
    for dtype in DT:
        sh = list(_shapes(dtype).items())
        for C in CS:
            for KP in (20, 32):
                K = K_BY_KP[KP][i % 3]
                name, (B, h, w) = sh[i % len(sh)]
                opts = dict(gumbel=i % 2 == 0, colpart=i % 3 != 1)
                cases.append(("read_fwd", dtype, C, K, B, h, w, opts, {"read_fwd_tiled_kernel"}))
                pname, (B, h, w) = sh[(i + 3) % len(sh)]
                cases.append(("read_fwd_planes", dtype, C, K_BY_KP[KP][(i + 1) % 3], B, h, w, dict(gumbel=i % 2 == 1, colpart=True),
                              {"read_fwd_tiled_kernel"}))
                gname, (B, h, w) = list(GENERIC_SHAPES.items())[i % 3]
                off = 1 if gname == "aligned_hw_off" else 0
                route = {"read_fwd_kernel"} | ({"colsoftmax_stats_kernel", "colsoftmax_combine_kernel"} if i % 2 == 0 else set())
                cases.append(("read_fwd", dtype, C, K_BY_KP[KP][(i + 2) % 3], B, h, w,
                              dict(off=off, gumbel=i % 3 == 0, colpart=i % 2 == 0), route))
                i += 1
    return cases


def _read_bwd_cases():
    cases, i = [], 0
    for dtype in DT:
        sh = list(_shapes(dtype).items())
        for C in CS:
            for KP in (20, 32):
                bf_mma = dtype == torch.bfloat16 and C >= 128
                dx = {"read_bwd_dx_bf16_kernel"} if bf_mma else {"read_bwd_dx_tma_kernel"}
                name, (B, h, w) = sh[i % len(sh)]
                cases.append(("read_bwd", dtype, C, K_BY_KP[KP][i % 3], B, h, w, dict(rl=i % 2 == 0),
                              {"read_bwd_ds_tiled_kernel"} | dx))
                name, (B, h, w) = sh[(i + 2) % len(sh)]
                cases.append(("read_bwd_planes", dtype, C, K_BY_KP[KP][(i + 1) % 3], B, h, w, dict(rl=i % 2 == 1),
                              {"read_bwd_ds_planes_kernel"} | dx))
                name, (B, h, w) = sh[(i + 4) % len(sh)]
                cases.append(("read_bwd_planes", dtype, C, K_BY_KP[KP][(i + 2) % 3], B, h, w, dict(rl=True, dx_add=True),
                              {"read_bwd_ds_planes_kernel", "read_bwd_dx_tma_kernel"}))
                gname, (B, h, w) = list(GENERIC_SHAPES.items())[i % 3]
                off = 1 if gname == "aligned_hw_off" else 0
                cases.append(("read_bwd", dtype, C, K_BY_KP[KP][(i + 1) % 3], B, h, w, dict(off=off, rl=i % 2 == 1),
                              {"read_bwd_kernel"}))
                if i % 4 == 0:
                    name, (B, h, w) = sh[(i + 1) % len(sh)]
                    cases.append(("read_bwd", dtype, C, K_BY_KP[KP][i % 3], B, h, w, dict(ds_null=True, rl=True),
                                  {"read_bwd_kernel"}))
                i += 1
    return cases


def _read_dM_cases():
    cases, i = [], 0
    for dtype in DT:
        sh = list(_shapes(dtype).items()) + list(GENERIC_SHAPES.items())
        for C in CS:
            for KP in (20, 32):
                for ordered in (False, True):
                    name, (B, h, w) = sh[i % len(sh)]
                    cases.append(("read_dM", dtype, C, K_BY_KP[KP][i % 3], B, h, w, dict(ordered=ordered, du_null=i % 3 == 2),
                                  {"read_bwd_dM_kernel"} | ({"reduce_partials_kernel"} if ordered else set())))
                    i += 1
    return cases


READ_FWD_CASES = _read_fwd_cases()
READ_BWD_CASES = _read_bwd_cases()
READ_DM_CASES = _read_dM_cases()
READ_CASES = READ_FWD_CASES + READ_BWD_CASES + READ_DM_CASES
READ_FAMILIES = {"read_fwd_kernel", "read_bwd_kernel", "read_bwd_dM_kernel", "read_fwd_tiled_kernel", "read_bwd_ds_tiled_kernel",
                 "read_bwd_ds_planes_kernel", "read_bwd_dx_tma_kernel", "read_bwd_dx_bf16_kernel"}


def case_id(c):
    entry, dtype, C, K, B, h, w, opts, _ = c
    flags = "-".join(k if v is True else "%s%s" % (k, v) for k, v in sorted(opts.items()) if v)
    return "%s-%s-C%d-K%d-%dx%dx%d%s" % (entry, _tn(dtype), C, K, B, h, w, ("-" + flags) if flags else "")


def case_route(c):
    entry, dtype, C, K, B, h, w, opts, _ = c
    return rw_instantiations(entry, dtype, C, K, h * w, aligned=not opts.get("off"), ordered=opts.get("ordered", False),
                             dx_add=opts.get("dx_add", False), ds=not opts.get("ds_null"), col_partials=opts.get("colpart", False))


def _edges_hit(cases):
    """(entry-independent) which of the shape edges the cases hit: used by the host test below."""
    hit = set()
    for entry, dtype, C, K, B, h, w, opts, _ in cases:
        hw = h * w
        tiles32 = B * -(-hw // 32)
        if B == 1 and hw <= 8:
            hit.add("one_partial_tile")
        if hw % 32 and B > 1:
            hit.add("tails_at_image_boundaries")
        if tiles32 == 297:
            hit.add("grid296_plus1")
        if tiles32 == 149:
            hit.add("grid148_plus1")
        if tiles32 >= 2304:                  # cfg-2: ~8 tiles per CTA of a 296-CTA grid
            hit.add("many_tiles_per_cta")
        if K in (1, 19, 20, 31):
            hit.add("K%d" % K)
    return hit


# ------------------------------------------------------------------------------------------- host-side tests
def test_read_case_tables_name_their_routes():
    """Every case names the kernel families rw_instantiations predicts for it, and the tables hit every edge."""
    wrong = [(case_id(c), sorted(c[8]), sorted(case_route(c))) for c in READ_CASES
             if {family(n) for n in case_route(c)} != c[8]]
    assert not wrong, wrong
    for cases in (READ_FWD_CASES, READ_BWD_CASES, READ_DM_CASES):
        assert {"one_partial_tile", "tails_at_image_boundaries", "K1", "K19", "K20", "K31"} <= _edges_hit(cases)
    assert {"grid296_plus1", "many_tiles_per_cta"} <= _edges_hit(READ_FWD_CASES)
    assert {"grid296_plus1", "grid148_plus1", "many_tiles_per_cta"} <= _edges_hit(READ_BWD_CASES)
    assert {"grid148_plus1", "many_tiles_per_cta"} <= _edges_hit(READ_DM_CASES)


def every_read_instantiation():
    T = ("f32", "bf16")
    out = set()
    for t in T:
        for KP in (20, 32):
            out.add("read_bwd_ds_planes_kernel<%s,%d>" % (t, KP))
            for C in CS:
                out |= {"read_fwd_kernel<%s,%d,%d>" % (t, C // 8, KP), "read_bwd_kernel<%s,%d,%d>" % (t, C // 8, KP),
                        "read_fwd_tiled_kernel<%s,%d,%d,2>" % (t, C, KP), "read_bwd_ds_tiled_kernel<%s,%d,%d,2>" % (t, C, KP),
                        "read_bwd_dx_tma_kernel<%s,%d,%d,2>" % (t, C, KP)}
                out |= {"read_bwd_dM_kernel<%s,%d,%d,%s>" % (t, C, KP, o) for o in ("false", "true")}
                if t == "bf16" and C >= 128:
                    out.add("read_bwd_dx_bf16_kernel<%d,%d,2>" % (C, KP))
    return out


def test_read_cases_reach_every_read_instantiation():
    reached = set()
    for c in READ_CASES:
        reached |= case_route(c)
    reached = {n for n in reached if family(n) in READ_FAMILIES}
    every = every_read_instantiation()
    assert reached == every, (sorted(every - reached), sorted(reached - every))
    assert len(every) == 120


def test_read_instantiations_match_the_built_library():
    """The table of read instantiations is the library's: a template added without a case fails here."""
    got = library_kernels(READ_FAMILIES)
    if got is None:
        pytest.skip("no built library or no cuobjdump / c++filt")
    every = every_read_instantiation()
    assert got == every, ("in the library, not in the table:", sorted(got - every), "in the table, not built:", sorted(every - got))


# ----------------------------------------------------------------------------------------- float64 restatements
def read_fwd_ref(x, M, gm):
    """float64 restatement of pm_read_fwd on [N, C] rows: (q, s, p, c) and the magnitudes of s and c."""
    xd, Md = x.double(), M.double()
    n = xd.norm(dim=1, keepdim=True)
    ir = 1.0 / n.clamp_min(NORM_EPS)
    q = xd * ir
    s = q @ Md.t()
    z = s + (gm.double() if gm is not None else 0.0)
    p = torch.softmax(z, dim=1)
    c = p @ Md
    return dict(q=q, s=s, z=z, p=p, c=c, mag_s=q.abs() @ Md.abs().t(), mag_c=p @ Md.abs())


def s_bound(ref, C, bf16_mma):
    """(fixed, base) of s: C-long dots and the norm (base); the operand split's residual on the bf16 tensor-core path."""
    return (BF16_SPLIT * ref["mag_s"] if bf16_mma else 0.0), (C + N0) * U24 * ref["mag_s"]


def p_bound(ref, sb, K):
    """(fixed, base) of score_memory: the exp of z - max (the argument's rounding grows with |z - max|), the sum and the
    division (base); the propagated bound `sb` of s and the flush of results below 2^-126 (fixed)."""
    p, z = ref["p"], ref["z"]
    dz = (z - z.max(dim=1, keepdim=True).values).abs()
    return p * (sb + (p * sb).sum(dim=1, keepdim=True)) + FTZ_FLOOR, (K + N0 + dz) * U24 * p


def c_bound(ref, pb, M, K):
    """(fixed, base) of p.M given the total bound `pb` of p."""
    return pb @ M.double().abs(), (K + N0) * U24 * ref["mag_c"]


# --------------------------------------------------------------------------------------------------- forward
def _read_fwd_inputs(case, tier, gen):
    entry, dtype, C, K, B, h, w, opts, _ = case
    N = B * h * w
    if tier == "exact":
        xr = four_signs(N, C, gen, "cuda")
        M = sixteenths((K, C), gen, "cuda")
    else:
        xr = rows_of(scaled((B, C, h * w), 1, gen, "cuda"))
        M = scaled((K, C), 0, gen, "cuda")
    xr[-1] = 0                                           # a zero feature vector in the last (tail) tile: the norm clamp
    x = nchw(xr, B, h * w).to(dtype)
    gm = gq = None
    if opts.get("gumbel"):
        gm = -torch.empty(N, K, device="cuda").exponential_(generator=gen).log()
        gq = -torch.empty(N, K, device="cuda").exponential_(generator=gen).log()
    return x, M, gm, gq


def _run_read_fwd(case, x, M, gm, gq, colpart=None):
    entry, dtype, C, K, B, h, w, opts, _ = case
    N, hw, KP = B * h * w, h * w, kp_of(K)
    UC = C + PLANES if entry == "read_fwd_planes" else 2 * C
    off = opts.get("off", 0)
    xg = _guard_in(x, off)
    u = Guarded(B * UC * hw, dtype)
    s = Guarded(N * KP, torch.float32)
    p = Guarded(N * K, torch.float32)
    fn = _lib().pm_read_fwd_planes if entry == "read_fwd_planes" else _lib().pm_read_fwd
    P = lambda t: None if t is None else t.data_ptr()
    rc = fn(xg.t.data_ptr(), M.data_ptr(), P(gm), P(gq), u.t.data_ptr(), s.t.data_ptr(), p.t.data_ptr(),
            None if colpart is None else colpart.t.data_ptr(), B, C, h, w, K, _code(dtype), _stream())
    _ok(rc, entry)
    torch.cuda.synchronize()
    assert unchanged(xg), "input x modified"
    for g, what in ((u, "u"), (s, "s"), (p, "score_memory")):
        g.check(what)
    return u.t.view(B, UC, hw), s.t.view(N, KP), p.t.view(N, K)


def _check_colpart(colpart, ref, gq, K, N, exact):
    """Combined row = float64 column maximum and 1/sum of s + gumbel_q; the ticket row back to zero."""
    cp = colpart.t.view(COLPART_ROWS + 2, 64)
    assert bool((cp[COLPART_ROWS + 1].view(torch.int32) == 0).all()), "ticket row not left zero"
    zq = ref["s"] + (gq.double() if gq is not None else 0.0)
    m64 = zq.max(dim=0).values
    inv64 = 1.0 / torch.exp(zq - m64).sum(dim=0)
    m, inv = cp[COLPART_ROWS, :K].double(), cp[COLPART_ROWS, 32:32 + K].double()
    # the kernel forms s + g in fp32 (one rounding of each side of the maximum); sums of N exp terms in fp32
    sq = ref["mag_s"].max(dim=0).values * (0 if exact else A_S * (64 + N0) * U24)
    r_m = ratio((m - m64).abs(), 2 * U24 * zq.abs().max(dim=0).values + sq + 1e-300)
    dzmax = (zq - m64).abs()
    w = torch.exp(zq - m64)
    spread = ((w * dzmax).sum(0) * inv64)          # exp argument roundings, weighted
    r_i = ratio((inv - inv64).abs() / inv64, A_COL * ((N ** 0.5) * 8 + N0 + spread) * U24 + sq)
    return r_m, r_i


@gpu
@pytest.mark.parametrize("tier", ["exact", "precision"])
@pytest.mark.parametrize("case", READ_FWD_CASES, ids=case_id)
def test_read_fwd(case, tier):
    entry, dtype, C, K, B, h, w, opts, _ = case
    gen = torch.Generator(device="cuda").manual_seed(100 + C + K + B * h * w)
    x, M, gm, gq = _read_fwd_inputs(case, tier, gen)
    N, KP = B * h * w, kp_of(K)
    colpart = None
    if opts.get("colpart"):
        nfl = _lib().pm_colsoftmax_workspace_floats(K)
        assert nfl == (COLPART_ROWS + 2) * 64
        colpart = Guarded(nfl, torch.float32)
        colpart.t[COLPART_ROWS * 64:].zero_()                    # the caller zeroes the ticket row
    u, s, p = _run_read_fwd(case, x, M, gm, gq, colpart)
    if colpart is not None:
        colpart.check("col_partials", scratch=True)
    ref = read_fwd_ref(rows_of(x), M, gm)
    # padding and the score planes
    assert bool((s[:, K:] == 0).all()), "padded columns of s are not 0"
    q_half = rows_of(u[:, :C])
    q_want = ref["q"].to(dtype)
    if entry == "read_fwd_planes":
        pl = rows_of(u[:, C:])
        assert bool((pl[:, K:] == 0).all()), "score planes >= K are not 0"
        c_or_planes = pl[:, :K]
    else:
        c_or_planes = rows_of(u[:, C:])
    if tier == "exact":
        assert torch.equal(s[:, :K].double(), ref["s"]), "s differs from float64 (exact tier)"
        assert torch.equal(q_half, q_want), "q half of u differs from float64 (exact tier)"
    bf16_mma = dtype == torch.bfloat16 and C >= 128 and not opts.get("off") and (h * w) % 8 == 0
    bf16_out = BF16_U if dtype == torch.bfloat16 else 0.0
    sf, sbase = s_bound(ref, C, bf16_mma)
    r_s = a_ratio((s[:, :K].double() - ref["s"]).abs(), sf, sbase)
    pf, pbase = p_bound(ref, sf + A_S * sbase, K)
    r_p = a_ratio((p.double() - ref["p"]).abs(), pf, pbase)
    pb = pf + A_P * pbase
    if entry == "read_fwd_planes":                      # the score planes are p stored in the feature dtype
        r_c = a_ratio((c_or_planes.double() - ref["p"]).abs(), pf + bf16_out * ref["p"], pbase)
    else:
        cf, cbase = c_bound(ref, pb, M, K)
        r_c = a_ratio((c_or_planes.double() - ref["c"]).abs(), cf + bf16_out * ref["c"].abs(), cbase)
    # q = x / |x|: the squared norm is a C-long fp32 sum
    r_q = a_ratio((q_half.double() - ref["q"]).abs(), bf16_out * ref["q"].abs(), (C + N0) * U24 * ref["q"].abs())
    print("RATIO read_fwd %s %s s=%.3f p=%.3f c=%.3f q=%.3f rel_l2(s)=%.2e" % (tier, case_id(case), r_s, r_p, r_c, r_q,
                                                                            rel_l2(s[:, :K], ref["s"])))
    assert r_s <= A_S and r_p <= A_P and r_c <= (A_P if entry == "read_fwd_planes" else A_C) and r_q <= A_S, (r_s, r_p, r_c, r_q)
    tau = 1e-4 if bf16_mma else 1e-5           # norm-wise; the split residual 2^-17 of the bf16 tensor-core path: 3e-5
    assert rel_l2(s[:, :K], ref["s"]) <= tau and rel_l2(p, ref["p"]) <= tau
    if colpart is not None:
        r_m, r_i = _check_colpart(colpart, ref, gq, K, N, tier == "exact")
        first = colpart.t.clone()
        _run_read_fwd(case, x, M, gm, gq, colpart)               # same buffer again: the ticket was left at zero
        colpart.check("col_partials (second launch)", scratch=True)
        assert torch.equal(colpart.t[COLPART_ROWS * 64:].view(torch.int32), first[COLPART_ROWS * 64:].view(torch.int32)), \
            "second launch on the same buffer combined differently"
        print("RATIO colpart %s %s max=%.3f inv=%.3f" % (tier, case_id(case), r_m, r_i))
        assert r_m <= 1.0 and r_i <= 1.0, (r_m, r_i)


# -------------------------------------------------------------------------------------------------- backward
def _read_bwd_inputs(case, gen):
    entry, dtype, C, K, B, h, w, opts, _ = case
    N, hw, KP = B * h * w, h * w, kp_of(K)
    planes = entry == "read_bwd_planes"
    UC = C + PLANES if planes else 2 * C
    xr = rows_of(scaled((B, C, hw), 1, gen, "cuda"))
    xr[-1] = 0
    x = nchw(xr, B, hw).to(dtype)
    M = scaled((K, C), 0, gen, "cuda")
    du = scaled((B, UC, hw), 1, gen, "cuda", -4, 4).to(dtype)
    logits = torch.randn(N, K, generator=gen, device="cuda") * 3
    p = torch.softmax(logits, dim=1)
    ds_rl = g_loss = rl_out = None
    if opts.get("rl"):
        ds_rl = torch.randn(N, KP, generator=gen, device="cuda")
        ds_rl[:, K:] = float("nan")                                  # padding a kernel must not read into ds
        g_loss = torch.tensor([0.75], device="cuda")
        rl_out = torch.tensor([0.0, 2.0 ** -10], device="cuda")
    dx_add = scaled((B, C, hw), 1, gen, "cuda").to(dtype) if opts.get("dx_add") else None
    return x, M, du, p, ds_rl, g_loss, rl_out, dx_add


def read_bwd_ref(x, M, du, p, ds_rl, scale, dx_add, planes, C, K):
    """float64 restatement of pm_read_bwd[_planes] on [N, *] rows: ds, dx and their magnitudes."""
    xd, Md, dud, pd = x.double(), M.double(), du.double(), p.double()
    n = xd.norm(dim=1, keepdim=True)
    ir = 1.0 / n.clamp_min(NORM_EPS)
    q = xd * ir
    dq0 = dud[:, :C]
    if planes:
        dp, mag_dp = dud[:, C:C + K], dud[:, C:C + K].abs()
    else:
        dc = dud[:, C:2 * C]
        dp, mag_dp = dc @ Md.t(), dc.abs() @ Md.abs().t()
    dot = (pd * dp).sum(1, keepdim=True)
    ds = pd * (dp - dot)
    if ds_rl is not None:
        ds = ds + scale * ds_rl[:, :K].double()
    dq = dq0 + ds @ Md
    proj = (q * dq).sum(1, keepdim=True) * (n > NORM_EPS)
    dx = (dq - q * proj) * ir
    if dx_add is not None:
        dx = dx + dx_add.double()
    return dict(q=q, ir=ir, dp=dp, mag_dp=mag_dp, ds=ds, dq=dq, dx=dx, proj=proj, nz=(n > NORM_EPS))


def ds_bound(ref, p, ds_rl, scale, n_dp, K):
    """(fixed, base) of ds: the dp = M.dc contraction (none in planes mode, n_dp = 0) and the softmax backward (base); the
    read-loss term's two roundings (fixed)."""
    pd = p.double()
    dpb = (n_dp + N0) * U24 * ref["mag_dp"]
    mag = pd * (ref["dp"].abs() + (pd * ref["dp"]).abs().sum(1, keepdim=True))
    base = (K + N0) * U24 * mag + pd * (dpb + (pd * dpb).sum(1, keepdim=True))
    fixed = 2 * U24 * abs(scale) * ds_rl[:, :K].double().abs() if ds_rl is not None else 0.0
    return fixed, base


def dx_bound(ref, dsb, M, K, C, split):
    """(fixed, base) of dx given the total bound `dsb` of ds: dq = dq0 + ds.M, then the projection and 1/|x| (base); the
    propagated ds bound and the bf16 split residual (fixed)."""
    Md = M.double().abs()
    q, nz = ref["q"].abs(), ref["nz"].double()
    inner = lambda e: e + q * (q * e).sum(1, keepdim=True) * nz
    mag_dq = ref["dq"].abs() + ref["ds"].abs() @ Md
    fixed = ref["ir"] * inner(dsb @ Md + split * (ref["ds"].abs() @ Md))
    base = ref["ir"] * (inner((K + N0) * U24 * mag_dq) + (C + N0) * U24 * inner(ref["dq"].abs()))
    return fixed, base


@gpu
@pytest.mark.parametrize("case", READ_BWD_CASES, ids=case_id)
def test_read_bwd(case):
    entry, dtype, C, K, B, h, w, opts, _ = case
    N, hw, KP = B * h * w, h * w, kp_of(K)
    planes = entry == "read_bwd_planes"
    gen = torch.Generator(device="cuda").manual_seed(200 + C + K + N)
    x, M, du, p, ds_rl, g_loss, rl_out, dx_add = _read_bwd_inputs(case, gen)
    off = opts.get("off", 0)
    dug, xg = _guard_in(du, off), _guard_in(x)
    dx = Guarded(B * C * hw, dtype)
    ds = None if opts.get("ds_null") else Guarded(N * KP, torch.float32)
    P = lambda t: None if t is None else t.data_ptr()
    args = [dug.t.data_ptr(), xg.t.data_ptr(), M.data_ptr(), p.data_ptr(), P(ds_rl), P(g_loss), P(rl_out), dx.t.data_ptr()]
    if planes:
        rc = _lib().pm_read_bwd_planes(*args, P(dx_add), ds.t.data_ptr(), B, C, h, w, K, _code(dtype), _stream())
    else:
        rc = _lib().pm_read_bwd(*args, None if ds is None else ds.t.data_ptr(), B, C, h, w, K, _code(dtype), _stream())
    _ok(rc, entry)
    torch.cuda.synchronize()
    dx.check("dx")
    if ds is not None:
        ds.check("ds")
    assert unchanged(dug) and unchanged(xg), "inputs modified"
    scale = 0.75 * 2.0 ** -10 if ds_rl is not None else 0.0
    ref = read_bwd_ref(rows_of(x), M, rows_of(du), p, ds_rl, scale, None if dx_add is None else rows_of(dx_add), planes, C, K)
    dsf, dsbase = ds_bound(ref, p, ds_rl, scale, 0 if planes else C, K)
    r_ds = 0.0
    if ds is not None:
        dsk = ds.t.view(N, KP)
        assert bool((dsk[:, K:] == 0).all()), "padded columns of ds are not 0"
        r_ds = a_ratio((dsk[:, :K].double() - ref["ds"]).abs(), dsf, dsbase)
    bf16_dx_mma = dtype == torch.bfloat16 and C >= 128 and dx_add is None and (planes or ds is not None)
    dxf, dxbase = dx_bound(ref, dsf + A_DS * dsbase, M, K, C, BF16_SPLIT if bf16_dx_mma else 0.0)
    if dx_add is not None:
        dxf = dxf + 2 * U24 * (ref["dx"].abs() + rows_of(dx_add).double().abs())
    if dtype == torch.bfloat16:
        dxf = dxf + BF16_U * ref["dx"].abs()
    r_dx = a_ratio((rows_of(dx.t.view(B, C, hw)).double() - ref["dx"]).abs(), dxf, dxbase)
    print("RATIO read_bwd %s ds=%.3f dx=%.3f" % (case_id(case), r_ds, r_dx))
    assert r_ds <= A_DS and r_dx <= A_DX, (r_ds, r_dx)
    if ds is not None:
        assert rel_l2(ds.t.view(N, KP)[:, :K], ref["ds"]) <= 1e-5
    assert rel_l2(dx.t.view(B, C, hw), nchw(ref["dx"], B, hw)) <= (1e-5 if dtype == torch.float32 else 2 ** -8)


# ------------------------------------------------------------------------------------------------------- dM
def dm_pixels_per_sum(B, hw):
    """(pixels one CTA of read_bwd_dM_kernel sums, number of CTAs added into dM)."""
    ntiles = B * -(-hw // 32)
    grid = min(ntiles, 148)
    return -(-ntiles // grid) * 32, grid


@gpu
@pytest.mark.parametrize("case", READ_DM_CASES, ids=case_id)
def test_read_bwd_dM(case):
    entry, dtype, C, K, B, h, w, opts, _ = case
    N, hw, KP = B * h * w, h * w, kp_of(K)
    gen = torch.Generator(device="cuda").manual_seed(300 + C + K + N)
    xr = rows_of(scaled((B, C, hw), 1, gen, "cuda"))
    xr[-1] = 0
    x = nchw(xr, B, hw).to(dtype)
    du = None if opts.get("du_null") else scaled((B, 2 * C, hw), 1, gen, "cuda", -4, 4).to(dtype)
    p = torch.softmax(torch.randn(N, K, generator=gen, device="cuda") * 3, dim=1)
    ds = scaled((N, KP), 1, gen, "cuda", -4, 4)
    ds[:, K:] = float("nan")                                     # the kernel must not read the padding
    pattern = (torch.arange(K * C, device="cuda", dtype=torch.float32) % 7 - 3).view(K, C)
    dM = Guarded(K * C, torch.float32, fill=None)
    dM.t.copy_(pattern.flatten())
    dM.ref = dM.buf.clone()
    P = lambda t: None if t is None else t.data_ptr()
    if opts.get("ordered"):
        nbytes = _lib().pm_read_bwd_dM_scratch_bytes(B, C, h, w, K)
        assert nbytes > 0 and nbytes % 16 == 0
        scratch = Guarded(nbytes // 4, torch.float32)
        rc = _lib().pm_read_bwd_dM_ordered(P(du), x.data_ptr(), p.data_ptr(), ds.data_ptr(), dM.t.data_ptr(), scratch.t.data_ptr(),
                                           B, C, h, w, K, _code(dtype), _stream())
    else:
        scratch = None
        rc = _lib().pm_read_bwd_dM(P(du), x.data_ptr(), p.data_ptr(), ds.data_ptr(), dM.t.data_ptr(), B, C, h, w, K,
                                   _code(dtype), _stream())
    _ok(rc, "pm_read_bwd_dM")
    torch.cuda.synchronize()
    dM.check("dM")
    if scratch is not None:
        scratch.check("dM scratch", scratch=True)
    xd = rows_of(x).double()
    q = xd / xd.norm(dim=1, keepdim=True).clamp_min(NORM_EPS)
    dsd = ds[:, :K].double()
    ref = dsd.t() @ q
    mag = dsd.abs().t() @ q.abs()
    if du is not None:
        dc = rows_of(du[:, C:]).double()
        ref, mag = ref + p.double().t() @ dc, mag + p.double().t() @ dc.abs()
    got = dM.t.view(K, C).double() - pattern.double()
    n, grid = dm_pixels_per_sum(B, hw)
    # base: each CTA's 2n fused adds and the norm of q; fixed: the `grid` adds into dM, which starts at the pattern
    fixed = grid * U24 * (mag + pattern.double().abs())
    r = a_ratio((got - ref).abs(), fixed, (2 * n + C + N0) * U24 * mag)
    print("RATIO read_dM %s dM=%.3f (n=%d, grid=%d)" % (case_id(case), r, n, grid))
    assert r <= A_DM, r
    if opts.get("ordered"):                                         # the ordered entry is bitwise reproducible
        dM2 = Guarded(K * C, torch.float32, fill=None)
        dM2.t.copy_(pattern.flatten())
        _ok(_lib().pm_read_bwd_dM_ordered(P(du), x.data_ptr(), p.data_ptr(), ds.data_ptr(), dM2.t.data_ptr(),
                                          scratch.t.data_ptr(), B, C, h, w, K, _code(dtype), _stream()), "pm_read_bwd_dM_ordered")
        torch.cuda.synchronize()
        assert torch.equal(dM2.t.view(torch.int32), dM.t.view(torch.int32)), "ordered dM not reproducible"


# --------------------------------------------------------------------------------------------------- routing
def _dry_call(case):
    """A closure that makes the case's call on zero data (the routing test only looks at what is launched)."""
    entry, dtype, C, K, B, h, w, opts, _ = case
    N, hw, KP = B * h * w, h * w, kp_of(K)
    lib, code, st = _lib(), _code(dtype), _stream()
    off = opts.get("off", 0)
    z = lambda *s, dt=dtype: torch.zeros(*s, dtype=dt, device="cuda")
    M, p = z(K, C, dt=torch.float32), z(N, K, dt=torch.float32)
    x = z(B * C * hw + 8)[off:off + B * C * hw]
    if entry in ("read_fwd", "read_fwd_planes"):
        UC = C + PLANES if entry == "read_fwd_planes" else 2 * C
        u, s = z(B * UC * hw), z(N, KP, dt=torch.float32)
        cp = z((COLPART_ROWS + 2) * 64, dt=torch.float32) if opts.get("colpart") else None
        fn = lib.pm_read_fwd_planes if entry == "read_fwd_planes" else lib.pm_read_fwd
        return lambda: _ok(fn(x.data_ptr(), M.data_ptr(), None, None, u.data_ptr(), s.data_ptr(), p.data_ptr(),
                              None if cp is None else cp.data_ptr(), B, C, h, w, K, code, st), entry)
    if entry in ("read_bwd", "read_bwd_planes"):
        UC = C + PLANES if entry == "read_bwd_planes" else 2 * C
        du = z(B * UC * hw + 8)[off:off + B * UC * hw]
        dx, ds = z(B * C * hw), z(N, KP, dt=torch.float32)
        if entry == "read_bwd_planes":
            add = z(B * C * hw) if opts.get("dx_add") else None
            return lambda: _ok(lib.pm_read_bwd_planes(du.data_ptr(), x.data_ptr(), M.data_ptr(), p.data_ptr(), None, None, None,
                                                      dx.data_ptr(), None if add is None else add.data_ptr(), ds.data_ptr(),
                                                      B, C, h, w, K, code, st), entry)
        dsp = None if opts.get("ds_null") else ds.data_ptr()
        return lambda: _ok(lib.pm_read_bwd(du.data_ptr(), x.data_ptr(), M.data_ptr(), p.data_ptr(), None, None, None,
                                           dx.data_ptr(), dsp, B, C, h, w, K, code, st), entry)
    if entry == "read_dM":
        du = None if opts.get("du_null") else z(B * 2 * C * hw)
        ds, dM = z(N, KP, dt=torch.float32), z(K, C, dt=torch.float32)
        dup = None if du is None else du.data_ptr()
        if opts.get("ordered"):
            scr = z(lib.pm_read_bwd_dM_scratch_bytes(B, C, h, w, K) // 4, dt=torch.float32)
            return lambda: _ok(lib.pm_read_bwd_dM_ordered(dup, x.data_ptr(), p.data_ptr(), ds.data_ptr(), dM.data_ptr(),
                                                          scr.data_ptr(), B, C, h, w, K, code, st), entry)
        return lambda: _ok(lib.pm_read_bwd_dM(dup, x.data_ptr(), p.data_ptr(), ds.data_ptr(), dM.data_ptr(), B, C, h, w, K,
                                              code, st), entry)
    raise ValueError(entry)


@gpu
def test_read_routing():
    """Each case launches exactly the instantiations rw_instantiations predicts; together they are every read
    instantiation of the library (the ordered dM ones included)."""
    wrong, reached = [], set()
    for case in READ_CASES:
        got = launched_kernels(_dry_call(case))
        want = case_route(case)
        if got != want:
            wrong.append((case_id(case), sorted(got), sorted(want)))
        reached |= got
    assert not wrong, wrong
    reached = {n for n in reached if family(n) in READ_FAMILIES}
    every = every_read_instantiation()
    assert reached == every, sorted(every - reached)


# ===================================================== CPU: the precision bounds reject the plausible wrong kernels
def _emulated_s(q, M, variant):
    """s = q.M^T as a wrong kernel would compute it (float64 emulation on the host)."""
    if variant == "tf32_1pass":
        return tf32_rn(q).double() @ tf32_rn(M).double().t()
    if variant == "3xtf32_no_lo_hi":             # a_hi.b_hi + a_hi.b_lo, the a_lo.b_hi term dropped
        qh, Mh = tf32_trunc(q), tf32_trunc(M)
        Ml = tf32_trunc(M - Mh)
        return qh.double() @ Mh.double().t() + qh.double() @ Ml.double().t()
    if variant == "bf16_M_no_lo":
        return q.double() @ M.to(torch.bfloat16).double().t()
    raise ValueError(variant)


@pytest.mark.parametrize("C,K", sorted({(c[2], c[3]) for c in READ_FWD_CASES}))
def test_read_bounds_reject_wrong_kernels(C, K):
    """At every (C, K) of the forward cases: the s bound rejects 1-pass TF32, 3xTF32 without a cross term and (on the
    bf16 tensor-core route, whose bound is the loosest) a bf16 memory without its lo part; the score_memory bound rejects
    exp evaluated in bf16 precision."""
    gen = torch.Generator().manual_seed(C * 64 + K)
    N = 2048
    x = scaled((N, C), 1, gen, "cpu")
    M = scaled((K, C), 0, gen, "cpu")
    ref = read_fwd_ref(x, M, None)
    qf = ref["q"].float()
    for variant, bf16_mma in (("tf32_1pass", False), ("3xtf32_no_lo_hi", False), ("bf16_M_no_lo", True)):
        s_bad = _emulated_s(qf, M, variant)
        sf, sbase = s_bound(ref, C, bf16_mma)
        r = a_ratio((s_bad - ref["s"]).abs(), sf, sbase)
        assert r > A_S, (variant, r)
    if K == 1:                                   # p = 1 whatever exp does
        return
    # exp in bf16 precision: every term exp(z - max) rounded to bf16 before the sum
    zc = ref["z"] - ref["z"].max(dim=1, keepdim=True).values
    e = torch.exp(zc).to(torch.bfloat16).double()
    p_bad = e / e.sum(dim=1, keepdim=True)
    sf, sbase = s_bound(ref, C, False)
    pf, pbase = p_bound(ref, sf + A_S * sbase, K)
    assert a_ratio((p_bad - ref["p"]).abs(), pf, pbase) > A_P
