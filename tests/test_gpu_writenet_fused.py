"""The writing net fused into the write (memory.py:74-87 then :206-257, fp32): _WriteNetFn with pm_write_reduce_bn_fwd and
pm_write_bwd_bn against the separate Writingnet + _WriteFn composition, and the two new entries against the kernels they
replace and float64 torch.

The fused class-sum kernel forms f = relu(x + BN(z)) with pm_bn_apply's expression, so with torch's deterministic flag set
(fixed-order sums in both paths) every forward output, the class sums and the new memory are bitwise those of the separate
path. Gradients differ only in the order of the dgamma / dbeta sums."""
import pytest
import torch

from pinthememory_b200 import capi, synth

gpu = pytest.mark.gpu
LOSS_W = (0.02, 0.4, 0.2)
GRAD_REL = 1e-6

# (B, C, h, w, Hm, Wm, K): the default workload, BASELINE config 4, and a map whose last 32-pixel tile is ragged
SHAPES = {
    "cfg2": (8, 256, 96, 96, 768, 768, 19),
    "cfg4": (8, 256, 48, 48, 768, 768, 19),
    "ragged": (2, 64, 10, 14, 37, 53, 19),
    "c128_k25": (3, 128, 20, 28, 81, 113, 25),
}


@pytest.fixture
def deterministic():
    was = torch.are_deterministic_algorithms_enabled()
    warn_only = torch.is_deterministic_algorithms_warn_only_enabled()
    fill = torch.utils.deterministic.fill_uninitialized_memory
    torch.use_deterministic_algorithms(True)
    try:
        yield
    finally:
        torch.use_deterministic_algorithms(was, warn_only=warn_only)
        torch.utils.deterministic.fill_uninitialized_memory = fill


def _module(K, C, seed=5, dtype=torch.float32, fused=True, **attrs):
    from pinthememory_b200.memory import Memory_sup

    torch.manual_seed(seed)
    m = Memory_sup(K, C, C, 0.8, 1.0, False).cuda()
    with torch.no_grad():
        m.clsfier.weight.normal_(0, 0.2)
        bn = m.writenet.writefeat[1]
        bn.weight.uniform_(0.5, 1.5)
        bn.bias.normal_(0, 0.3)
    m = m.to(dtype)
    m.m_items = m.m_items.float()
    if not fused:
        m._writenet_fused = lambda x: False
    for k, v in attrs.items():
        setattr(m, k, v)
    return m


def _inputs(B, C, h, w, Hm, Wm, K, seed=21, dtype=torch.float32):
    x = synth.make_features(B, C, h, w, seed=seed, device="cuda").to(dtype)
    lab = synth.make_labels(B, Hm, Wm, K, "blocky", seed=seed + 1, device="cuda", block=16)
    G = synth.make_upstream_grad((B, C, h, w), seed=seed + 2, device="cuda").to(dtype)
    return x, lab, G


def _step(mem, x, lab, G):
    x = x.detach().clone().requires_grad_(True)
    mem.zero_grad(set_to_none=True)
    uq, sq, sm, rl, wl = mem(x, lab, True, False)
    dev = x.device
    torch.autograd.backward([uq, rl, wl[0], wl[1]], [G] + [torch.tensor(v, device=dev, dtype=rl.dtype) for v in LOSS_W])
    fwd = {"uq": uq, "sq": sq, "sm": sm, "readloss": rl, "div": wl[0], "cls": wl[1], "m_items": mem.m_items,
           "class_sums": mem.last_class_sums}
    fwd.update({"buf." + k: b for k, b in mem.named_buffers()})
    grads = {"dx": x.grad}
    grads.update({"grad." + k: p.grad for k, p in mem.named_parameters()})
    torch.cuda.synchronize()
    return ({k: v.detach().clone() for k, v in fwd.items()}, {k: v.detach().clone() for k, v in grads.items() if v is not None})


def _rel_l2(a, b):
    a, b = a.double(), b.double()
    return float((a - b).norm() / b.norm().clamp_min(1e-30))


def _launched(fn):
    """Names of the C-ABI entries `fn` calls."""
    capi.enable_kernel_timing(True)
    try:
        capi.reset_counters()
        fn()
        return set(capi.kernel_timings_ms())
    finally:
        capi.enable_kernel_timing(False)


@gpu
@pytest.mark.parametrize("shape", list(SHAPES), ids=list(SHAPES))
def test_fused_module_equals_separate_writing_net(deterministic, shape):
    B, C, h, w, Hm, Wm, K = SHAPES[shape]
    x, lab, G = _inputs(B, C, h, w, Hm, Wm, K)
    fused, sep = _module(K, C), _module(K, C, fused=False)
    assert fused._writenet_fused(x) and not sep._writenet_fused(x)
    names = _launched(lambda: _step(_module(K, C), x, lab, G))
    assert "pm_write_reduce_bn_fwd_ordered" in names and "pm_write_bwd_bn" in names
    f_fwd, f_grad = _step(fused, x, lab, G)
    s_fwd, s_grad = _step(sep, x, lab, G)
    assert set(f_fwd) == set(s_fwd) and set(f_grad) == set(s_grad)
    for k in s_fwd:
        assert torch.equal(f_fwd[k], s_fwd[k]), (k, float((f_fwd[k].double() - s_fwd[k].double()).abs().max()))
    for k in s_grad:
        assert _rel_l2(f_grad[k], s_grad[k]) <= GRAD_REL, (k, _rel_l2(f_grad[k], s_grad[k]))


@gpu
def test_running_statistics_and_counter_bumped_once(deterministic):
    B, C, h, w, Hm, Wm, K = SHAPES["ragged"]
    x, lab, G = _inputs(B, C, h, w, Hm, Wm, K)
    fused, sep = _module(K, C), _module(K, C, fused=False)
    for _ in range(2):
        _step(fused, x, lab, G)
        _step(sep, x, lab, G)
    bf, bs = fused.writenet.writefeat[1], sep.writenet.writefeat[1]
    assert int(bf.num_batches_tracked) == 2 == int(bs.num_batches_tracked)
    assert torch.equal(bf.running_mean, bs.running_mean) and torch.equal(bf.running_var, bs.running_var)


@gpu
def test_fused_steps_are_bitwise_reproducible(deterministic):
    B, C, h, w, Hm, Wm, K = SHAPES["cfg4"]
    x, lab, G = _inputs(B, C, h, w, Hm, Wm, K)
    runs = []
    for _ in range(3):
        m = _module(K, C)
        for _ in range(2):
            out = _step(m, x, lab, G)
        runs.append(out)
    for fwd, grads in runs[1:]:
        for a, b in ((fwd, runs[0][0]), (grads, runs[0][1])):
            for k in b:
                assert torch.equal(a[k], b[k]), k


@gpu
@pytest.mark.parametrize("shape", ["cfg2", "ragged"])
def test_kernels_against_separate_passes_and_float64(shape):
    """pm_write_reduce_bn_fwd / pm_write_bwd_bn entry by entry: f (through the class sums) and the statistics bitwise those of
    pm_bn_apply_stats + pm_write_reduce_fwd; g bitwise df * [f > 0] of pm_write_bwd; dgamma / dbeta / dz against float64."""
    B, C, h, w, Hm, Wm, K = SHAPES[shape]
    gen = torch.Generator(device="cuda").manual_seed(7)
    z = torch.randn(B, C, h, w, device="cuda", generator=gen) * 2 + 0.5
    x = torch.randn(B, C, h, w, device="cuda", generator=gen)
    lab = synth.make_labels(B, Hm, Wm, K, "blocky", seed=3, device="cuda", block=16)
    gamma = torch.rand(C, device="cuda", generator=gen) + 0.5
    beta = torch.randn(C, device="cuda", generator=gen) * 0.3
    z64 = z.double()
    stats = torch.cat([z64.sum((0, 2, 3)), (z64 * z64).sum((0, 2, 3)), torch.zeros(1, device="cuda", dtype=torch.float64)])
    n = B * h * w

    def fresh():
        return [torch.zeros(C, device="cuda"), torch.ones(C, device="cuda"), torch.zeros((), dtype=torch.int64, device="cuda")]

    # separate passes
    rm_s, rv_s, nbt_s = fresh()
    mean_s, inv_s = torch.empty(C, device="cuda"), torch.empty(C, device="cuda")
    f = torch.empty_like(z)
    capi.bn_apply_stats(z, stats, n, 1e-5, gamma, beta, x, f, True, mean_s, inv_s, rm_s, rv_s, 0.1, num_batches_tracked=nbt_s)
    SD_s = torch.zeros(K + 1, C + 4, device="cuda")
    capi.write_reduce_fwd(f, lab, SD_s, K)
    # fused
    rm_f, rv_f, nbt_f = fresh()
    mean_f, inv_f = torch.empty(C, device="cuda"), torch.empty(C, device="cuda")
    SD_f = torch.zeros(K + 1, C + 4, device="cuda")
    capi.write_reduce_bn_fwd(z, x, lab, SD_f, K, stats, n, 1e-5, gamma, beta, mean_f, inv_f, rm_f, rv_f, 0.1,
                             num_batches_tracked=nbt_f)
    torch.cuda.synchronize()
    for a, b in ((mean_f, mean_s), (inv_f, inv_s), (rm_f, rm_s), (rv_f, rv_s), (nbt_f, nbt_s)):
        assert torch.equal(a, b)
    assert int(nbt_f) == 1
    # same f -> same per-CTA MMA partials; only the float-atomic order of the two launches may differ
    assert _rel_l2(SD_f, SD_s) <= 1e-6
    # backward
    dS = torch.randn(K, C, device="cuda", generator=gen) * 0.1
    df = torch.empty_like(z)
    capi.write_bwd(dS, f, lab, df, K)
    g = torch.full_like(z, float("nan"))
    dgamma, dbeta = torch.empty(C, device="cuda"), torch.empty(C, device="cuda")
    capi.write_bwd_bn(dS, z, x, lab, mean_f, inv_f, gamma, beta, g, dgamma, dbeta, K)
    torch.cuda.synchronize()
    ref = torch.where(f > 0, df, torch.zeros_like(df))
    assert torch.equal(g == 0, ref == 0) and _rel_l2(g, ref) <= 1e-6
    xhat = (z64 - mean_f.double().view(1, C, 1, 1)) * inv_f.double().view(1, C, 1, 1)
    g64 = g.double()
    db64, dg64 = g64.sum((0, 2, 3)), (g64 * xhat).sum((0, 2, 3))
    scale = g64.abs().sum((0, 2, 3)) + 1e-30
    assert float(((dbeta.double() - db64).abs() / scale).max()) < 1e-5
    assert float(((dgamma.double() - dg64).abs() / (g64 * xhat).abs().sum((0, 2, 3)).clamp_min(1e-30)).max()) < 1e-5
    dz = torch.empty_like(z)
    capi.bn_bwd_apply(g, None, None, z, mean_f, inv_f, gamma, dgamma, dbeta, False, True, dz, None)
    gi = (gamma.double() * inv_f.double()).view(1, C, 1, 1)
    dz64 = gi * (g64 - db64.view(1, C, 1, 1) / n - xhat * dg64.view(1, C, 1, 1) / n)
    assert _rel_l2(dz, dz64) < 1e-5


@gpu
def test_two_stream_graph_replay_equals_eager(deterministic):
    from pinthememory_b200.graphed import GraphedStep

    B, C, h, w, Hm, Wm, K = 2, 256, 48, 48, 384, 384, 19
    batches = [_inputs(B, C, h, w, Hm, Wm, K, seed=s) for s in (3, 40)]
    eager, graphed = _module(K, C, overlap_write=True), _module(K, C, overlap_write=True)
    step = GraphedStep(graphed, *batches[0], loss_weights=LOSS_W, memory_writing=True, writing_detach=False)
    for x, lab, G in batches:
        fwd, grads = _step(eager, x, lab, G)
        step(x, lab, G)
        torch.cuda.synchronize()
        assert torch.equal(step.query_grad, grads["dx"])
        assert torch.equal(graphed.m_items, fwd["m_items"])
        for k, p in graphed.named_parameters():
            assert torch.equal(p.grad, grads["grad." + k]), k
    step.release()


@gpu
def test_launch_list_and_kernels_per_replay():
    """The default step runs no normalise pass and no BatchNorm-sums pass for the writing net: one pm_bn_apply_stats and one
    pm_bn_bwd_reduce_rows (the output block's) instead of two each, and one kernel less per replay."""
    from pinthememory_b200.graphed import GraphedStep

    B, C, h, w, Hm, Wm, K = 2, 256, 48, 48, 384, 384, 19
    x, lab, G = _inputs(B, C, h, w, Hm, Wm, K)
    counts = {}
    per_replay = {}
    for fused in (True, False):
        m = _module(K, C, fused=fused)
        capi.enable_kernel_timing(True)
        try:
            capi.reset_counters()
            _step(m, x, lab, G)
            counts[fused] = {k: len(v) for k, v in capi.kernel_timings_ms().items()}
        finally:
            capi.enable_kernel_timing(False)
        g = _module(K, C, fused=fused, overlap_write=True)
        step = GraphedStep(g, x, lab, G, loss_weights=LOSS_W, memory_writing=True, writing_detach=False)
        per_replay[fused] = step.kernels_per_replay
        step.release()
    assert counts[True].get("pm_bn_apply_stats", 0) == counts[False]["pm_bn_apply_stats"] - 1
    assert counts[True].get("pm_bn_bwd_reduce_rows", 0) == counts[False]["pm_bn_bwd_reduce_rows"] - 1
    assert "pm_write_reduce_fwd" not in counts[True] and "pm_write_bwd" not in counts[True]
    assert per_replay[True] == per_replay[False] - 1


@gpu
def test_bf16_keeps_the_separate_kernels():
    B, C, h, w, Hm, Wm, K = 2, 256, 48, 48, 384, 384, 19   # bf16 rows of 16-byte multiples: the GEMM path, not the library
    x, lab, G = _inputs(B, C, h, w, Hm, Wm, K, dtype=torch.bfloat16)
    m = _module(K, C, dtype=torch.bfloat16)
    assert not m._writenet_fused(x)
    names = _launched(lambda: _step(m, x, lab, G))
    assert "pm_write_reduce_bn_fwd" not in names and "pm_write_bwd_bn" not in names
    assert "pm_bn_apply_stats" in names
