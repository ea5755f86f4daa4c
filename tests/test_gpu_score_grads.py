"""Gradients through the score maps of the read and through ``get_score``, as the reference module has them.

In the reference, ``score_query`` / ``score_memory`` are plain torch tensors (``F.softmax`` / ``F.gumbel_softmax`` of
s = q.M^T, memory.py:171,181-187) and all three outputs of ``get_score`` (memory.py:167-189) carry graph, so a loss on
them reaches the query, the memory and (meta-test read) the writing net. Checked here:
  - the module against the oracle evaluated in float64, with a loss that includes both score maps;
  - pm_score_bwd kernel by kernel against float64 torch, for every NULL combination;
  - get_score's three outputs differentiated against the float64 oracle, and its no-grad path unchanged;
  - the two new kernels bitwise repeatable with torch's deterministic flag off and on, whole score-gradient steps with it
    on;
  - a step whose loss does not touch the scores runs exactly the kernels it ran before.
"""
import pytest
import torch

from gate_util import check_ties, oracle_module_like, record_gates
from golden_util import LOSS_WEIGHTS, assert_close, max_abs_over_scale, rel_l2

pytestmark = pytest.mark.gpu

TOL32 = 1e-5
TOL16 = 2e-2


@pytest.fixture(autouse=True)
def _exact_fp32():
    old = (torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32)
    torch.backends.cudnn.allow_tf32 = False
    torch.backends.cuda.matmul.allow_tf32 = False
    yield
    torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32 = old


def _module(K, C, gumbel, dtype=torch.float32, seed=5):
    from pinthememory_b200.memory import Memory_sup

    torch.manual_seed(seed)
    m = Memory_sup(K, C, C, 0.8, 1.0, gumbel).cuda()
    with torch.no_grad():
        m.clsfier.weight.normal_(0, 0.2)
    m = m.to(dtype)
    m.m_items = m.m_items.float()
    return m


def _inputs(B, C, h, w, Hm, Wm, K, seed, labels=True):
    from pinthememory_b200 import synth

    N = B * h * w
    x = synth.make_features(B, C, h, w, seed=seed, device="cuda")
    lab = synth.make_labels(B, Hm, Wm, K, "blocky", seed=seed + 1, device="cuda", block=16) if labels else None
    G = synth.make_upstream_grad((B, C, h, w), seed=seed + 2, device="cuda") / N
    # score_query is a softmax over all N pixels (entries ~1/N), score_memory one over K slots: scaled so that each term
    # moves the similarity gradient about as much as the others
    Gq = synth.make_upstream_grad((B, h, w, K), seed=seed + 3, device="cuda")
    Gm = synth.make_upstream_grad((B, h, w, K), seed=seed + 4, device="cuda") / N
    return x, lab, G, Gq, Gm


def _loss(uq, sq, sm, rl, wl, G, Gq, Gm, terms, labels, writing):
    """<G,uq> + 0.02 readloss + 0.4 div + 0.2 cls + <Gq,score_query> + <Gm,score_memory> (the parts ``terms`` selects)."""
    total = 0
    if terms in ("all", "q", "m"):
        total = (uq.double() * G.double()).sum()
        if labels:
            total = total + LOSS_WEIGHTS["read"] * rl
        if writing:
            total = total + LOSS_WEIGHTS["div"] * wl[0] + LOSS_WEIGHTS["cls"] * wl[1]
    if terms in ("all", "scores", "q"):
        total = total + (sq.double() * Gq.double()).sum()
    if terms in ("all", "scores", "m"):
        total = total + (sm.double() * Gm.double()).sum()
    return total


def _check_ties(relu_gates, dtype):
    """Replayed ReLU gates must be ties at the precision of the module's arithmetic: rounding level in fp32
    (gate_util.check_ties), a few bf16 ulps (2^-8 relative) in bf16."""
    if dtype != torch.bfloat16:
        return check_ties(relu_gates)
    for name, n, numel, ratio in relu_gates.mismatches:
        assert ratio <= 2.0 ** -6, f"{name}: ReLU gate differs where |z|/max|z| = {ratio:.2e} (not a bf16 rounding tie)"
        assert n <= max(3, 1e-3 * numel), f"{name}: {n} of {numel} ReLU gates differ"


def _yardstick(a32, a64):
    return max(rel_l2(a32, a64), max_abs_over_scale(a32, a64))


def _noise(seed, N, K):
    from pinthememory_b200.memory import draw_gumbel_pair

    torch.manual_seed(seed)
    return draw_gumbel_pair(N, K, "cuda")


# B, C, h, w, Hm, Wm, K, dtype, fold, gumbel, labels, writing, two_stream, terms
MODULE_CASES = [
    (2, 64, 12, 16, 48, 64, 19, "f32", False, False, True, True, False, "all"),
    (2, 64, 12, 16, 48, 64, 19, "f32", True, False, True, True, False, "all"),
    (2, 64, 12, 16, 48, 64, 19, "f32", False, True, True, True, False, "all"),
    (2, 64, 12, 16, 48, 64, 19, "f32", True, True, True, True, False, "all"),
    (2, 32, 16, 16, 64, 64, 7, "f32", True, True, True, False, False, "all"),
    (1, 64, 16, 16, 64, 64, 25, "f32", False, True, True, True, False, "all"),
    (1, 64, 16, 16, 64, 64, 25, "f32", True, False, True, False, False, "all"),
    (2, 64, 12, 16, 0, 0, 19, "f32", True, True, False, False, False, "all"),
    (2, 64, 12, 16, 0, 0, 25, "f32", False, False, False, False, False, "all"),
    (2, 64, 12, 16, 48, 64, 19, "f32", True, True, True, True, True, "all"),
    (2, 64, 12, 16, 48, 64, 19, "f32", True, True, True, True, False, "scores"),
    (2, 64, 12, 16, 48, 64, 19, "f32", False, True, True, False, False, "scores"),
    (2, 64, 12, 16, 48, 64, 19, "f32", True, False, True, True, False, "q"),
    (2, 64, 12, 16, 48, 64, 19, "f32", False, True, True, True, False, "m"),
    (2, 64, 12, 16, 48, 64, 19, "bf16", False, True, True, True, False, "all"),
    (2, 64, 12, 16, 48, 64, 19, "bf16", True, False, True, True, False, "all"),
    (1, 64, 16, 16, 64, 64, 25, "bf16", True, True, True, False, False, "scores"),
    (8, 256, 96, 96, 768, 768, 19, "f32", True, True, True, True, False, "all"),   # cfg 2
]


def _case_id(c):
    B, C, h, w, Hm, Wm, K, dt, fold, gum, lab, wr, two, terms = c
    return (f"B{B}_C{C}_{h}x{w}_K{K}_{dt}_{'folded' if fold else 'concat'}_{'gumbel' if gum else 'plain'}"
            f"_{'labels' if lab else 'nolabels'}_{'write' if wr else 'nowrite'}{'_2stream' if two else ''}_{terms}")


@pytest.mark.parametrize("case", MODULE_CASES, ids=_case_id)
def test_module_score_gradients_match_fp64_oracle(case):
    from oracle import memory_oracle as mo

    B, C, h, w, Hm, Wm, K, dt, fold, gumbel, labels, writing, two_stream, terms = case
    dtype = torch.bfloat16 if dt == "bf16" else torch.float32
    N = B * h * w
    mem = _module(K, C, gumbel, dtype)
    mem.fold_memory_into_conv = fold
    mem.fold_min_pixels = 0
    mem.overlap_write = two_stream
    x, lab, G, Gq, Gm = _inputs(B, C, h, w, Hm, Wm, K, seed=31 + K + C, labels=labels)
    x = x.to(dtype)
    noise = _noise(77, N, K) if gumbel else None
    # the fp32 oracle is the yardstick of the output block's parameter gradients (below); both copy the state before the
    # module's forward updates it
    oracles = {dt: oracle_module_like(mem, dtype=dt) for dt in (torch.float64, torch.float32)}

    xm = x.clone().requires_grad_(True)
    torch.manual_seed(77)   # the module draws the same noise (draw_gumbel_pair after the same seed)
    with record_gates() as gates:
        uq, sq, sm, rl, wl = mem(xm, lab, writing, True)
    assert sq.grad_fn is not None and sm.grad_fn is not None
    _loss(uq, sq, sm, rl, wl, G, Gq, Gm, terms, labels, writing).backward()

    ref = {}
    for odt, ora in oracles.items():
        ora.relu_gates = mo.ReluGates(gates)
        xo = x.to(odt).requires_grad_(True)
        no = tuple(t.to(odt) for t in noise) if gumbel else None
        uo, sqo, smo, rlo, wlo = ora(xo, lab, writing, True, noise=no)
        _loss(uo, sqo, smo, rlo, wlo, G, Gq, Gm, terms, labels, writing).backward()
        _check_ties(ora.relu_gates, dtype)
        ref[odt] = dict(score_query=sqo.detach(), grad_x=xo.grad,
                        **{n: p.grad for n, p in ora.named_parameters() if p.grad is not None})
    r64, r32 = ref[torch.float64], ref[torch.float32]

    tol = TOL16 if dtype == torch.bfloat16 else TOL32
    assert_close(sq.detach(), r64["score_query"], tol, "score_query")
    assert_close(xm.grad.double(), r64["grad_x"], tol, "grad_x")
    for n, p in mem.named_parameters():
        assert (p.grad is None) == (n not in r64), n
        if p.grad is None:
            continue
        t = tol
        if n.startswith(("output", "writenet")):
            # the two 1x1-conv blocks' parameter gradients cross their BatchNorm statistics and come out of the
            # weight-gradient GEMM, a reduction over all N pixels: 2e-5 as in test_gpu_parity, 3x the deviation of eager
            # fp32 torch from fp64, or the GEMM's calibrated bound tau(N) = 1e-8 * N (DESIGN §2), whichever is largest.
            # At cfg 2 the module's errors here are the same with and without the score terms in the loss.
            t = max(tol, 2e-5, 3.0 * _yardstick(r32[n], r64[n]), 1e-8 * N)
        assert_close(p.grad.double(), r64[n], t, n)


@pytest.mark.parametrize("shape", [(2, 64, 12, 12, 48, 48, 19), (1, 64, 16, 16, 64, 64, 25)], ids=["K19", "K25"])
@pytest.mark.parametrize("fold", [False, True], ids=["concat", "folded"])
def test_meta_test_read_with_graph_carrying_memory(shape, fold):
    """Case C (train.py:558,570): the memory comes out of a write with graph; the read's score maps are in the loss, so
    their gradient reaches the memory and, through it, the writing net and the classifier."""
    from oracle import memory_oracle as mo

    B, C, h, w, Hm, Wm, K = shape
    mem = _module(K, C, False)
    mem.fold_memory_into_conv = fold
    mem.fold_min_pixels = 0
    xb, labb, _, _, _ = _inputs(B, C, h, w, Hm, Wm, K, seed=101)
    xc, labc, G, Gq, Gm = _inputs(B, C, h, w, Hm, Wm, K, seed=201)

    def run(m, xb, xc, gates=None):
        xb, xc = xb.clone().requires_grad_(True), xc.clone().requires_grad_(True)
        if gates is None:
            m.write(xb, labb, writing_detach=False)
        else:
            f = m.writenet(xb, m.relu_gates)
            m.m_items = mo.write(f, labb, m.m_items, m.momentum, m.clsfier.weight, m.clsfier.bias)["memory_new"]
        M_b = m.m_items
        M_b.retain_grad()
        uq, sq, sm, rl, _ = m(xc, labc, False)
        _loss(uq, sq, sm, rl, None, G, Gq, Gm, "all", True, False).backward()
        return dict(grad_xb=xb.grad, grad_xc=xc.grad, dM=M_b.grad,
                    **{"grad." + n: p.grad for n, p in m.named_parameters() if p.grad is not None})

    # the fp32 oracle is the yardstick of these ill-conditioned gradients; both copy the module's state (memory, running
    # statistics) before its write replaces them
    oracles = {dt: oracle_module_like(mem, dtype=dt) for dt in (torch.float64, torch.float32)}
    with record_gates() as gates:
        got = run(mem, xb, xc)
    results = {}
    for dt, o in oracles.items():
        o.relu_gates = mo.ReluGates(gates)
        results[dt] = run(o, xb.to(dt), xc.to(dt), gates)
        check_ties(o.relu_gates)
    ref, ref32 = results[torch.float64], results[torch.float32]
    assert set(ref) <= set(got) and "grad.writenet.writefeat.0.weight" in got
    for k in set(got) - set(ref):   # (_WriteFn returns the classifier's gradient even when no loss reaches it)
        assert torch.count_nonzero(got[k]) == 0, k
    for k in ref:
        assert_close(got[k].double(), ref[k], max(5e-5, 3.0 * _yardstick(ref32[k], ref[k])), k)


# ---------------------------------------------------------------------------------------- pm_score_bwd kernel


def _score_bwd_ref(pq, gq, pm, gm, ds_rl, scale, K):
    E = torch.zeros(pq.shape[0], ds_rl.shape[1], dtype=torch.float64, device=pq.device)
    if gm is not None:
        E[:, :K] += pm * (gm - (pm * gm).sum(1, keepdim=True))
    if gq is not None:
        E[:, :K] += pq * (gq - (pq * gq).sum(0, keepdim=True))
    if scale is not None:
        E[:, :K] += scale * ds_rl[:, :K]
    return E


@pytest.mark.parametrize("N", [1, 149, 4099, 73728])
@pytest.mark.parametrize("K", [1, 7, 19, 20, 31])
def test_score_bwd_kernel_against_fp64(N, K):
    from pinthememory_b200 import capi

    KP = capi.score_stride(K)
    g = torch.Generator(device="cuda").manual_seed(N * 37 + K)
    s = 3.0 * torch.randn(N, K, device="cuda", generator=g, dtype=torch.float64)
    pq64, pm64 = torch.softmax(s, 0), torch.softmax(s, 1)
    gq64 = torch.randn(N, K, device="cuda", generator=g, dtype=torch.float64)
    gm64 = torch.randn(N, K, device="cuda", generator=g, dtype=torch.float64)
    rl64 = torch.randn(N, KP, device="cuda", generator=g, dtype=torch.float64)
    pq, pm, gq, gm, rl = (t.float().contiguous() for t in (pq64, pm64, gq64, gm64, rl64))
    # the kernel reads what it is given: compare against float64 arithmetic on the same fp32 values
    pq64, pm64, gq64, gm64, rl64 = (t.double() for t in (pq, pm, gq, gm, rl))
    g_loss = torch.tensor([0.7], device="cuda")
    rl_out = torch.tensor([0.0, 1.0 / 3000.0], device="cuda")
    scale = float(g_loss[0].double() * rl_out[1].double())
    for use_q in (False, True):
        for use_m in (False, True):
            for use_rl in (False, True):
                E = torch.full((N, KP), float("nan"), device="cuda")
                capi.score_bwd(pq if use_q else None, gq if use_q else None, pm if use_m else None,
                               gm if use_m else None, E, K, ds_rl=rl if use_rl else None,
                               g_loss=g_loss if use_rl else None, rl_out=rl_out if use_rl else None)
                ref = _score_bwd_ref(pq64, gq64 if use_q else None, pm64, gm64 if use_m else None, rl64,
                                     scale if use_rl else None, K)
                what = f"q={use_q} m={use_m} rl={use_rl}"
                assert torch.isfinite(E).all(), what
                assert torch.equal(E[:, K:], torch.zeros_like(E[:, K:])), what + ": padding columns must be zero"
                if not ref.abs().max() > 0:   # (N = 1 or K = 1: every softmax term is exactly zero)
                    assert torch.count_nonzero(E) == 0, what
                    continue
                assert_close(E.double(), ref, 2e-6, what)


def test_score_bwd_argument_checks():
    import ctypes

    from pinthememory_b200 import capi

    lib = capi.load()
    one = ctypes.c_void_p(16)
    assert lib.pm_score_bwd(None, None, None, None, None, None, None, None, None, 4, 19, None) == -1
    assert lib.pm_score_bwd(one, one, None, None, None, None, None, one, None, 4, 19, None) == -1   # g_q needs workspace
    assert lib.pm_score_bwd(None, None, None, one, None, None, None, one, None, 4, 19, None) == -1  # g_m needs score_m
    assert lib.pm_score_bwd(None, None, None, None, None, None, None, one, None, 4, 32, None) == -4
    assert lib.pm_score_bwd(None, None, None, None, None, None, None, one, None, 0, 19, None) == -5
    assert lib.pm_score_bwd(None, None, None, None, None, None, None, ctypes.c_void_p(4), None, 4, 19, None) == -6
    assert lib.pm_score_nhwc_bwd(None, None, None, None, None, None, 4, 64, 19, None) == -1
    assert lib.pm_score_nhwc_bwd_scratch_bytes(4, 64, 0) == -4


# -------------------------------------------------------------------------------------------------- get_score


@pytest.mark.parametrize("gumbel", [False, True], ids=["plain", "gumbel"])
@pytest.mark.parametrize("K", [19, 25])
def test_get_score_gradients_match_fp64_oracle(K, gumbel, monkeypatch):
    from oracle import memory_oracle as mo

    mem = _module(K, 64, gumbel)
    B, h, w, C = 2, 9, 7, 64
    N = B * h * w
    q0 = torch.nn.functional.normalize(torch.randn(B, h, w, C, device="cuda"), dim=3)
    M0 = mem.m_items.detach().clone()
    labels = torch.randint(0, K, (B, 36, 28), device="cuda")
    labels[0, :5] = 255
    Gq = torch.randn(N, K, device="cuda")
    Gm = torch.randn(N, K, device="cuda") / N
    ora = oracle_module_like(mem, dtype=torch.float64)
    noise = _noise(13, N, K) if gumbel else None
    if gumbel:
        monkeypatch.setattr(mo, "gumbel_noise_pair", lambda s: tuple(t.double() for t in noise))
    for which in range(3):
        for m, dt in ((mem, torch.float32), (ora, torch.float64)):
            q = q0.to(dt, copy=True).requires_grad_(True)
            M = M0.to(dt, copy=True).requires_grad_(True)
            torch.manual_seed(13)
            sq, sm, rl = m.get_score(q, labels, M)
            out = (sq.double() * Gq.double()).sum(), (sm.double() * Gm.double()).sum(), rl.double()
            out[which].backward()
            if m is mem:
                got = (q.grad, M.grad)
            else:
                ref = (q.grad, M.grad)
        for a, b, n in zip(got, ref, ("query", "mem")):
            assert_close(a.double(), b, TOL32, f"d output[{which}] / d {n}")


def test_get_score_without_grad_is_unchanged():
    from pinthememory_b200 import capi

    mem = _module(19, 64, True)
    q = torch.nn.functional.normalize(torch.randn(2, 9, 7, 64, device="cuda"), dim=3)
    labels = torch.randint(0, 19, (2, 36, 28), device="cuda")
    res = []
    for grad_mode in (False, True):
        torch.manual_seed(3)
        n0 = capi.LAUNCHES
        with torch.set_grad_enabled(grad_mode):
            out = mem.get_score(q, labels, mem.m_items)
        res.append((out, capi.LAUNCHES - n0))
        assert all(t.grad_fn is None for t in out)
    (a, na), (b, nb) = res
    assert na == nb
    for x, y in zip(a, b):
        assert torch.equal(x, y)


# ----------------------------------------------------------------------------------------------- determinism


@pytest.fixture(params=[False, True], ids=["flag_off", "flag_on"])
def det_flag(request):
    was, warn_only = torch.are_deterministic_algorithms_enabled(), torch.is_deterministic_algorithms_warn_only_enabled()
    torch.use_deterministic_algorithms(request.param)
    try:
        yield request.param
    finally:
        torch.use_deterministic_algorithms(was, warn_only=warn_only)


def _repeat_equal(fn, n=3):
    outs = [fn() for _ in range(n)]
    for o in outs[1:]:
        assert len(o) == len(outs[0])
        for i, (a, b) in enumerate(zip(o, outs[0])):
            assert torch.equal(a, b), f"output {i} differs between repeats"


def test_score_backward_kernels_are_bitwise_repeatable(det_flag):
    """pm_score_bwd and pm_score_nhwc_bwd add their partials in a fixed order in every mode: with torch's deterministic
    flag off as well as on, repeats give the same bits (cfg-2 pixel count)."""
    from pinthememory_b200 import capi

    N, K = 8 * 96 * 96, 19
    KP = capi.score_stride(K)
    g = torch.Generator(device="cuda").manual_seed(3)
    s = 3.0 * torch.randn(N, K, device="cuda", generator=g)
    pq, pm = torch.softmax(s, 0), torch.softmax(s, 1)
    gq, gm = torch.randn(N, K, device="cuda", generator=g), torch.randn(N, K, device="cuda", generator=g)
    rl = torch.randn(N, KP, device="cuda", generator=g)
    g_loss, rl_out = torch.tensor([0.02], device="cuda"), torch.tensor([0.0, 1e-5], device="cuda")

    def score_bwd():
        E = torch.empty(N, KP, device="cuda")
        capi.score_bwd(pq, gq, pm, gm, E, K, ds_rl=rl, g_loss=g_loss, rl_out=rl_out)
        return [E]

    _repeat_equal(score_bwd)
    mem = _module(K, 256, True)
    q0 = torch.nn.functional.normalize(torch.randn(8, 96, 96, 256, device="cuda", generator=g), dim=3)
    labels = torch.randint(0, K, (8, 768, 768), device="cuda", generator=g)

    def get_score_grads():
        # (the score terms only: the read-loss term's ds_rl comes from the forward's read-loss kernel, whose default
        # instantiation adds with float atomics; pm_score_bwd's handling of it is covered above with fixed inputs)
        q = q0.clone().requires_grad_(True)
        M = mem.m_items.clone().requires_grad_(True)
        torch.manual_seed(5)
        sq, sm, _ = mem.get_score(q, labels, M)
        ((sq * gq).sum() + (sm * gm).sum() / N).backward()
        return [q.grad, M.grad]

    _repeat_equal(get_score_grads)


@pytest.mark.parametrize("fold", [False, True], ids=["concat", "folded"])
def test_score_gradient_steps_are_bitwise_repeatable(fold):
    """A whole score-gradient step with a graph-carrying memory, under torch's deterministic flag: dx, dM and every
    parameter gradient repeat bit for bit. (With the flag off the read loss and dM of the default kernels add partials
    with float atomics, so a whole step repeats only up to rounding; the new kernels are checked in both modes above.)"""
    import copy

    was, warn_only = torch.are_deterministic_algorithms_enabled(), torch.is_deterministic_algorithms_warn_only_enabled()
    torch.use_deterministic_algorithms(True)
    try:
        base = _module(19, 64, True)
        base.fold_memory_into_conv, base.fold_min_pixels = fold, 0
        x, lab, G, Gq, Gm = _inputs(2, 64, 24, 24, 96, 96, 19, seed=7)
        M0 = base.m_items.clone()

        def step():
            m = copy.deepcopy(base)
            m.m_items = M0.clone().requires_grad_(True)
            xm = x.clone().requires_grad_(True)
            torch.manual_seed(5)
            uq, sq, sm, rl, wl = m(xm, lab, False)
            _loss(uq, sq, sm, rl, wl, G, Gq, Gm, "all", True, False).backward()
            return [xm.grad, m.m_items.grad] + [p.grad for p in m.parameters() if p.grad is not None]

        _repeat_equal(step)
    finally:
        torch.use_deterministic_algorithms(was, warn_only=warn_only)


# --------------------------------------------------------------------------------------------- default path


def _kernel_names(fn):
    from pinthememory_b200 import capi

    capi.enable_kernel_timing(True)
    try:
        fn()
        torch.cuda.synchronize()
        return set(capi._timing)
    finally:
        capi.enable_kernel_timing(False)


def _default(mem, x, lab, G):
    """A training step whose loss does not touch the score maps."""
    def run():
        xm = x.clone().requires_grad_(True)
        uq, sq, sm, rl, wl = mem(xm, lab, True, True)
        total = (uq * G).sum() + LOSS_WEIGHTS["read"] * rl + LOSS_WEIGHTS["div"] * wl[0] + LOSS_WEIGHTS["cls"] * wl[1]
        total.backward()
    return run


@pytest.mark.parametrize("fold", [False, True], ids=["concat", "folded"])
def test_default_step_runs_no_score_backward(fold):
    mem = _module(19, 64, True)
    mem.fold_memory_into_conv, mem.fold_min_pixels = fold, 0
    x, lab, G, Gq, Gm = _inputs(2, 64, 24, 24, 96, 96, 19, seed=9)

    def with_scores():
        xm = x.clone().requires_grad_(True)
        uq, sq, sm, rl, wl = mem(xm, lab, True, True)
        _loss(uq, sq, sm, rl, wl, G, Gq, Gm, "all", True, True).backward()

    assert "pm_score_bwd" not in _kernel_names(_default(mem, x, lab, G))
    assert "pm_score_bwd" in _kernel_names(with_scores)


def test_graphed_step_returns_detached_scores_and_no_score_backward():
    from pinthememory_b200 import capi
    from pinthememory_b200.graphed import GraphedStep

    mem = _module(19, 64, False)
    x, lab, G, _, _ = _inputs(2, 64, 24, 24, 96, 96, 19, seed=3)
    names = _kernel_names(_default(mem, x, lab, G))
    n0 = capi.LAUNCHES
    _default(mem, x, lab, G)()
    eager = capi.LAUNCHES - n0
    step = GraphedStep(mem, x, lab, G)
    try:
        assert step.kernels_per_replay == eager
        out = step.replay()
        assert out["score_query"].grad_fn is None and out["score_memory"].grad_fn is None
        assert "pm_score_bwd" not in names
    finally:
        step.release()
