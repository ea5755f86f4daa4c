"""Bitwise reproducibility under ``torch.use_deterministic_algorithms(True)``.

With torch's flag set, the package calls the ordered entries (per-CTA partials added in a fixed order) instead of the
kernels that combine partials with float atomics, so repeating a step from the same state on the same inputs gives
identical bits. The CPU tests at the end check the argument validation of those entries without a GPU.
"""
import ctypes

import pytest
import torch

from pinthememory_b200 import capi, synth

W = (0.02, 0.4, 0.2)
gpu = pytest.mark.gpu


@pytest.fixture
def deterministic():
    was = torch.are_deterministic_algorithms_enabled()
    warn_only = torch.is_deterministic_algorithms_warn_only_enabled()
    fill = torch.utils.deterministic.fill_uninitialized_memory
    tf32 = (torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32)
    torch.use_deterministic_algorithms(True)
    torch.backends.cudnn.allow_tf32 = False
    torch.backends.cuda.matmul.allow_tf32 = False
    try:
        yield
    finally:
        torch.use_deterministic_algorithms(was, warn_only=warn_only)
        torch.utils.deterministic.fill_uninitialized_memory = fill
        torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32 = tf32


def _module(K, C, dtype=torch.float32, seed=5, **attrs):
    from pinthememory_b200.memory import Memory_sup

    torch.manual_seed(seed)
    m = Memory_sup(K, C, C, 0.8, 1.0, False).cuda()
    with torch.no_grad():
        m.clsfier.weight.normal_(0, 0.2)
    m = m.to(dtype)
    m.m_items = m.m_items.float()
    for k, v in attrs.items():
        setattr(m, k, v)
    return m


def _clone_module(src):
    import copy

    m = copy.deepcopy(src)
    m.m_items = src.m_items.clone()
    return m


def _inputs(B, C, h, w, Hm, Wm, K, dtype=torch.float32, labels_u8=False, seed=21, block=32):
    x = synth.make_features(B, C, h, w, seed=seed, device="cuda").to(dtype)
    lab = synth.make_labels(B, Hm, Wm, K, "blocky", seed=seed + 1, device="cuda", block=block)
    if labels_u8:
        lab = lab.to(torch.uint8)
    G = synth.make_upstream_grad((B, C, h, w), seed=seed + 2, device="cuda").to(dtype)
    return x, lab, G


def _step(mem, x, lab, G):
    """One training step of the module (read + write, forward + backward); everything it produces."""
    x = x.detach().clone().requires_grad_(True)
    mem.zero_grad(set_to_none=True)
    uq, sq, sm, rl, wl = mem(x, lab, True, False)
    dev = x.device
    torch.autograd.backward([uq, rl, wl[0], wl[1]], [G] + [torch.tensor(v, device=dev, dtype=rl.dtype) for v in W])
    out = {"uq": uq, "sq": sq, "sm": sm, "readloss": rl, "div": wl[0], "cls": wl[1], "m_items": mem.m_items, "dx": x.grad,
           "class_sums": mem.last_class_sums}
    for k, p in mem.named_parameters():
        out["grad." + k] = p.grad
    for k, b in mem.named_buffers():
        out["buf." + k] = b
    torch.cuda.synchronize()
    return {k: v.detach().clone() for k, v in out.items() if torch.is_tensor(v)}


def _assert_equal(a, b, what=""):
    assert set(a) == set(b), what
    for k in a:
        assert a[k].dtype == b[k].dtype and a[k].shape == b[k].shape, (what, k)
        assert torch.equal(a[k], b[k]), (what, k, float((a[k].double() - b[k].double()).abs().max()))


def _repeats(make, x, lab, G, n=3, steps=1):
    """n independent runs of `steps` steps from identical state and inputs."""
    runs = []
    for _ in range(n):
        mem = make()
        for _ in range(steps):
            res = _step(mem, x, lab, G)
        runs.append(res)
    return runs


@gpu
@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16], ids=["fp32", "bf16"])
def test_cfg2_steps_are_bitwise_reproducible(deterministic, dtype):
    B, C, h, w, Hm, Wm, K = 8, 256, 96, 96, 768, 768, 19
    base = _module(K, C, dtype)
    x, lab, G = _inputs(B, C, h, w, Hm, Wm, K, dtype)
    runs = _repeats(lambda: _clone_module(base), x, lab, G, n=3, steps=3)
    for r in runs[1:]:
        _assert_equal(runs[0], r, "cfg2")


PATHS = {
    # name: (B, C, h, w, Hm, Wm, K, module attributes, uint8 labels)
    "readloss8_ratio2": (2, 64, 24, 24, 48, 48, 19, {}, False),
    "w1": (2, 64, 16, 1, 64, 4, 19, {}, False),
    "K25_first_kernel": (2, 64, 24, 24, 96, 96, 25, {}, False),
    "hw_not_mult4": (2, 64, 13, 15, 52, 60, 19, {}, False),
    "folded_small": (2, 64, 24, 24, 96, 96, 19, {"fold_min_pixels": 0}, False),
    "unfolded": (2, 128, 48, 48, 192, 192, 19, {"fold_memory_into_conv": False}, False),
    "uint8_labels": (2, 64, 24, 24, 96, 96, 19, {"fold_min_pixels": 0}, True),
}


@gpu
@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16], ids=["fp32", "bf16"])
@pytest.mark.parametrize("name", list(PATHS))
def test_other_paths_are_bitwise_reproducible(deterministic, name, dtype):
    B, C, h, w, Hm, Wm, K, attrs, u8 = PATHS[name]
    base = _module(K, C, dtype, **attrs)
    x, lab, G = _inputs(B, C, h, w, Hm, Wm, K, dtype, labels_u8=u8, block=8)
    runs = _repeats(lambda: _clone_module(base), x, lab, G, n=2, steps=2)
    _assert_equal(runs[0], runs[1], name)


@gpu
def test_get_score_is_bitwise_reproducible(deterministic):
    import torch.nn.functional as F

    mem = _module(19, 64)
    for K, (Hm, Wm) in ((19, (96, 96)), (25, (96, 96))):
        q = F.normalize(torch.randn(2, 24, 24, 64, device="cuda"), dim=-1)
        lab = synth.make_labels(2, Hm, Wm, K, "blocky", seed=3, device="cuda", block=8)
        M = F.normalize(torch.randn(K, 64, device="cuda"), dim=1)
        a = mem.get_score(q, lab, M)
        b = mem.get_score(q, lab, M)
        for u, v in zip(a, b):
            assert torch.equal(u, v)


@gpu
def test_meta_step_with_dM_is_bitwise_reproducible(deterministic):
    from pinthememory_b200.memory import Memory_sup
    from pinthememory_b200.metastep import meta_step

    B, C, h, w, Hm, Wm, K = 4, 256, 48, 48, 192, 192, 19
    x_tr = synth.make_features(B, C, h, w, seed=11, device="cuda")
    x_te = synth.make_features(B, C, h, w, seed=12, device="cuda")
    lab_tr = synth.make_labels(B, Hm, Wm, K, "blocky", seed=13, device="cuda", block=16)
    lab_te = synth.make_labels(B, Hm, Wm, K, "blocky", seed=14, device="cuda", block=16)
    G_tr = synth.make_upstream_grad((B, C, h, w), seed=15, device="cuda") / (B * h * w)
    G_te = synth.make_upstream_grad((B, C, h, w), seed=16, device="cuda") / (B * h * w)
    results = []
    for _ in range(2):
        mods = []
        for _ in range(3):
            torch.manual_seed(7)
            m = Memory_sup(K, C, C, 0.8, 1.0, False).cuda()
            with torch.no_grad():
                m.clsfier.weight.normal_(0, 0.2)
            m.train()
            mods.append(m)
        for m in mods[1:]:
            m.load_state_dict(mods[0].state_dict())
            m.m_items = mods[0].m_items.clone()
        got = meta_step(*mods, x_tr, lab_tr, x_te, lab_te, G_tr, G_te, inner_lr=0.01)
        torch.cuda.synchronize()
        flat = {}
        for k, v in got.items():
            if isinstance(v, dict):
                flat.update({k + "." + kk: vv.detach().clone() for kk, vv in v.items()})
            elif torch.is_tensor(v):
                flat[k] = v.detach().clone()
        assert any(k.startswith("grads.") for k in flat)
        results.append(flat)
    _assert_equal(results[0], results[1], "meta step")


@gpu
def test_callers_are_bitwise_reproducible(deterministic):
    from pinthememory_b200 import callers

    # PrototypePool over several batches
    sums = []
    for _ in range(2):
        pool = callers.PrototypePool(19, 256)
        for s in range(3):
            f = synth.make_features(4, 256, 48, 48, seed=30 + s, device="cuda")
            lab = synth.make_labels(4, 192, 192, 19, "blocky", seed=40 + s, device="cuda", block=16)
            pool.add(f, lab)
        sums.append((pool.sums_counts.clone(), pool.finalize()))
    assert torch.equal(sums[0][0], sums[1][0]) and torch.equal(sums[0][1], sums[1][1])
    # upsampled_cross_entropy at 192^2 -> 768^2
    logits = torch.randn(2, 19, 192, 192, device="cuda")
    lab = synth.make_labels(2, 768, 768, 19, "blocky", seed=5, device="cuda", block=16)
    outs = []
    for _ in range(2):
        lg = logits.clone().requires_grad_(True)
        loss = callers.upsampled_cross_entropy(lg, lab)
        loss.backward()
        outs.append((loss.detach().clone(), lg.grad.clone()))
    assert torch.equal(outs[0][0], outs[1][0]) and torch.equal(outs[0][1], outs[1][1])
    # class_mean_vectors
    f = synth.make_features(2, 64, 48, 48, seed=8, device="cuda")
    lab = synth.make_labels(2, 192, 192, 19, "blocky", seed=9, device="cuda", block=16)
    a = callers.class_mean_vectors(f, lab, 19)
    b = callers.class_mean_vectors(f, lab, 19)
    assert torch.equal(a[0], b[0]) and torch.equal(a[1], b[1])


@gpu
def test_graph_replay_equals_eager_launches(deterministic):
    from pinthememory_b200.graphed import GraphedStep

    B, C, h, w, Hm, Wm, K = 2, 256, 48, 48, 384, 384, 19
    base = _module(K, C, overlap_write=True)
    batches = [_inputs(B, C, h, w, Hm, Wm, K, seed=s, block=16) for s in (3, 40)]
    eager, graphed = _clone_module(base), _clone_module(base)
    step = GraphedStep(graphed, *batches[0], loss_weights=W, memory_writing=True, writing_detach=False)
    for x, lab, G in batches:
        ref = _step(eager, x, lab, G)
        step(x, lab, G)
        torch.cuda.synchronize()
        assert torch.equal(step.query_grad, ref["dx"])
        assert torch.equal(graphed.m_items, ref["m_items"])
        for k, p in graphed.named_parameters():
            assert torch.equal(p.grad, ref["grad." + k]), k
    step.release()


@gpu
def test_schedule_and_fill_independence(deterministic):
    B, C, h, w, Hm, Wm, K = 4, 256, 48, 48, 384, 384, 19
    base = _module(K, C)
    x, lab, G = _inputs(B, C, h, w, Hm, Wm, K, block=16)
    results = {}
    for overlap in (False, True):
        for fill in (True, False):
            torch.utils.deterministic.fill_uninitialized_memory = fill
            mem = _clone_module(base)
            mem.overlap_write = overlap
            results[(overlap, fill)] = _step(mem, x, lab, G)
    first = results[(False, True)]
    for key, r in results.items():
        _assert_equal(first, r, str(key))


@gpu
@pytest.mark.parametrize("precision", ["fp32", "bf16"])
def test_oracle_parity_holds_under_the_flag(deterministic, precision):
    import test_gpu_parity as parity

    # the oracle's own torch ops (nll_loss2d) have no deterministic CUDA kernel: let torch warn for those; the flag stays
    # set, so the module takes its ordered entries
    torch.use_deterministic_algorithms(True, warn_only=True)

    cases = parity.CORE_CASES if precision == "fp32" else parity.CORE_CASES[:3] + parity.CORE_CASES[4:6]
    fn = parity.test_core_fp32_matches_oracle if precision == "fp32" else parity.test_core_bf16_matches_oracle
    for case in cases:
        fn(case)


@gpu
@pytest.mark.parametrize("fold", [False, True], ids=["concat", "folded"])
def test_reference_fixtures_hold_under_the_flag(deterministic, fold, monkeypatch):
    import test_gpu_parity as parity
    from golden_util import golden_names

    torch.use_deterministic_algorithms(True, warn_only=True)   # (the oracle's nll_loss2d, as above)

    for name in golden_names():
        parity.test_module_reproduces_reference_fixture(name, fold, monkeypatch)


class _StandInHead(torch.nn.Module):
    """The stand-in DeepLabV3+ head of test_gpu_head_standin.py with the package's callers around the memory: the decoder
    concatenates the up-sampled memory output with the fine features (upsample_concat, deepv3plus.py:569-572) and the main
    loss is upsampled_cross_entropy (deepv3plus.py:575-578). Its own layers are cuDNN convolutions and BatchNorm."""

    def __init__(self, memory, c_in, c_low, c_fine, c_mem, num_classes):
        super().__init__()
        nn = torch.nn
        self.bot_aspp = nn.Conv2d(c_in, c_mem, kernel_size=1, bias=False)
        self.bot_fine = nn.Conv2d(c_low, c_fine, kernel_size=1, bias=False)
        self.memory = memory
        self.final = nn.Sequential(nn.Conv2d(c_fine + c_mem, c_mem, kernel_size=3, padding=1, bias=False),
                                   nn.BatchNorm2d(c_mem), nn.ReLU(inplace=True),
                                   nn.Conv2d(c_mem, num_classes, kernel_size=1, bias=False))

    def forward(self, aspp, low, gts):
        from pinthememory_b200 import upsample_concat, upsampled_cross_entropy

        mem_output = self.memory(self.bot_aspp(aspp), gts, True, False)
        dec0 = upsample_concat(self.bot_fine(low), mem_output[0])
        loss1 = upsampled_cross_entropy(self.final(dec0), gts)
        readloss, writeloss = mem_output[3], mem_output[4]
        return loss1 + 0.02 * readloss + 0.4 * writeloss[0] + 0.2 * writeloss[1]   # train.py:1213-1215


@gpu
def test_stand_in_head_trains_bitwise_reproducibly(deterministic):
    B, Cin, Clow, Cf, C, h, w, Hm, Wm, K = 2, 96, 48, 48, 64, 12, 16, 96, 128, 19
    torch.manual_seed(11)
    mem = _module(K, C, fold_min_pixels=0)
    base = _StandInHead(mem, Cin, Clow, Cf, C, K).cuda().train()
    aspp = synth.make_features(B, Cin, h, w, seed=41, device="cuda")
    low = synth.make_features(B, Clow, 4 * h, 4 * w, seed=43, device="cuda")
    gts = synth.make_labels(B, Hm, Wm, K, "blocky", seed=42, device="cuda")
    runs = []
    for _ in range(2):
        import copy

        head = copy.deepcopy(base)
        head.memory.m_items = base.memory.m_items.clone()
        opt = torch.optim.SGD(head.parameters(), lr=0.01, momentum=0.9)
        res = {}
        for step in range(2):
            opt.zero_grad(set_to_none=True)
            a = aspp.clone().requires_grad_(True)
            loss = head(a, low, gts)
            loss.backward()
            res[f"loss{step}"] = loss.detach().clone()
            res[f"d_aspp{step}"] = a.grad.clone()
            res[f"memory{step}"] = head.memory.m_items.detach().clone()
            res.update({f"grad{step} {n}": p.grad.clone() for n, p in head.named_parameters()})
            opt.step()
        res.update({"param " + n: p.detach().clone() for n, p in head.named_parameters()})
        res.update({"buffer " + n: b.clone() for n, b in head.named_buffers()})
        torch.cuda.synchronize()
        runs.append(res)
    assert any(k.startswith("grad1 bot_fine") for k in runs[0])
    _assert_equal(runs[0], runs[1], "stand-in head")


def _sharded_worker(rank, world, port, out):
    import os

    import torch.distributed as dist

    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    os.environ.pop("PINMEM_B200_NCCL_EXCHANGE", None)
    torch.cuda.set_device(rank)
    dev = torch.device("cuda", rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=dev)
    try:
        torch.use_deterministic_algorithms(True)
        torch.backends.cudnn.allow_tf32 = False
        torch.backends.cuda.matmul.allow_tf32 = False
        from pinthememory_b200 import sharding
        from pinthememory_b200.memory import Memory_sup

        B, C, h, w, Hm, Wm, K = 4, 256, 48, 48, 384, 384, 19
        torch.manual_seed(7)   # the same initial state on every rank (CPU generator)
        mem = Memory_sup(K, C, C, 0.8, 1.0, False).to(dev).train()
        mem.m_items = mem.m_items.to(dev)
        state = {k: v.clone() for k, v in mem.state_dict().items()}
        mem0 = mem.m_items.clone()
        shard = sharding.enable_sharded_update(mem)
        x = synth.make_features(B, C, h, w, seed=21 + rank, device=dev)
        lab = synth.make_labels(B, Hm, Wm, K, "blocky", seed=31 + rank, device=dev, block=16)
        G = synth.make_upstream_grad((B, C, h, w), seed=41 + rank, device=dev)
        repeats = []
        for _ in range(2):
            mem.load_state_dict(state)
            mem.m_items = mem0.clone()
            res = {}
            for step in range(2):
                r = _step(mem, x, lab, G)
                res.update({f"{k}{step}": v.cpu() for k, v in r.items()})
            repeats.append(res)
        out[rank] = dict(repeats=repeats, peer=shard.peer is not None, peer_error=shard.peer_error)
    finally:
        dist.destroy_process_group()


@gpu
@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs 2 GPUs")
def test_sharded_peer_update_is_bitwise_reproducible():
    """Two ranks, the class sums exchanged inside the update kernels over peer memory: two repeats of two training steps
    give identical bits on each rank, and the memory is identical on both ranks."""
    import socket

    import torch.multiprocessing as mp

    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    port = s.getsockname()[1]
    s.close()
    world = 2
    out = mp.get_context("spawn").Manager().dict()
    mp.spawn(_sharded_worker, args=(world, port, out), nprocs=world, join=True)
    if not out[0]["peer"]:
        pytest.skip("no symmetric-memory peer exchange on this box: %s" % out[0]["peer_error"])
    for r in range(world):
        _assert_equal(out[r]["repeats"][0], out[r]["repeats"][1], f"rank {r}")
    for step in range(2):
        assert torch.equal(out[0]["repeats"][0][f"m_items{step}"], out[1]["repeats"][0][f"m_items{step}"]), step


# ----------------------------------------------------------------------------- CPU: argument checks of the new entries

def _lib():
    return capi.load()


def _buf():
    return ctypes.c_void_p(256)   # a non-NULL, 16-byte aligned address: the checks below fail before any dereference


def test_ordered_entries_check_arguments_without_a_gpu():
    lib = _lib()
    p, z = _buf(), None
    # NULL scratch / outputs
    assert lib.pm_readloss_fwd8_ordered(p, p, 1.0, 2, 8, 8, 32, 32, 19, p, p, p, z, z) == -1
    assert lib.pm_readloss_fwd_ordered(p, p, 1.0, 2, 8, 8, 32, 32, 25, p, p, p, z, z) == -1
    assert lib.pm_write_reduce_fwd_ordered(p, p, p, z, 2, 64, 8, 8, 32, 32, 19, 0, z) == -1
    assert lib.pm_write_reduce_fwd8_ordered(p, p, z, p, 2, 64, 8, 8, 32, 32, 19, 0, z) == -1
    assert lib.pm_read_bwd_dM_ordered(z, p, p, p, p, z, 2, 64, 8, 8, 19, 0, z) == -1
    assert lib.pm_conv1x1_fwd_ordered(p, p, p, p, p, z, 2, 64, 64, 64, 0, z) == -1
    # slots, shapes, channels, dtype, alignment
    assert lib.pm_readloss_fwd8_ordered(p, p, 1.0, 2, 8, 8, 32, 32, 20, p, p, p, p, z) == -4
    assert lib.pm_readloss_fwd_ordered(p, p, 1.0, 2, 8, 8, 32, 32, 32, p, p, p, p, z) == -4
    assert lib.pm_readloss_fwd8_ordered(p, p, 0.0, 2, 8, 8, 32, 32, 19, p, p, p, p, z) == -5
    assert lib.pm_readloss_fwd_ordered(p, p, 1.0, 0, 8, 8, 32, 32, 19, p, p, p, p, z) == -5
    assert lib.pm_readloss_fwd8_ordered(p, p, 1.0, 2, 8, 8, 32, 32, 19, p, p, p, ctypes.c_void_p(260), z) == -6
    assert lib.pm_write_reduce_fwd_ordered(p, p, p, p, 2, 48, 8, 8, 32, 32, 19, 0, z) == -3
    assert lib.pm_write_reduce_fwd8_ordered(p, p, p, p, 2, 64, 8, 8, 32, 32, 19, 7, z) == -2
    assert lib.pm_write_reduce_fwd_ordered(p, p, p, ctypes.c_void_p(260), 2, 64, 8, 8, 32, 32, 19, 0, z) == -6
    assert lib.pm_read_bwd_dM_ordered(z, p, p, p, p, p, 2, 64, 8, 8, 0, 0, z) == -4
    assert lib.pm_read_bwd_dM_ordered(z, p, p, p, p, ctypes.c_void_p(260), 2, 64, 8, 8, 19, 0, z) == -6
    assert lib.pm_conv1x1_fwd_ordered(p, p, p, p, p, ctypes.c_void_p(260), 2, 64, 64, 64, 0, z) == -6
    assert lib.pm_conv1x1_fwd_ordered(p, p, p, p, p, p, 2, 64, 48, 64, 0, z) == -5
    assert lib.pm_conv1x1_fwd_ordered(p, p, p, p, p, p, 2, 64, 64, 64, 3, z) == -2
    # scratch-size queries
    assert lib.pm_readloss_scratch_bytes(2, 8, 8, 32, 32, 20, 1) == -4
    assert lib.pm_readloss_scratch_bytes(2, 8, 0, 32, 32, 19, 0) == -5
    assert lib.pm_write_reduce_scratch_bytes(2, 48, 8, 8, 19) == -3
    assert lib.pm_read_bwd_dM_scratch_bytes(2, 64, 8, 8, 32) == -4
    assert lib.pm_conv1x1_stats_scratch_bytes(2, 64, 64, 5) == -2


def test_scratch_sizes_follow_the_partials():
    lib = _lib()
    # class sums: min(296, 32-pixel tiles) CTAs x [K+1][C+4] floats; 6.2 MB at cfg 2
    assert lib.pm_write_reduce_scratch_bytes(8, 256, 96, 96, 19) == 296 * 20 * 260 * 4
    assert lib.pm_write_reduce_scratch_bytes(1, 64, 8, 8, 19) == 2 * 20 * 68 * 4
    # dM: min(148, tiles) CTAs x [K][C]
    assert lib.pm_read_bwd_dM_scratch_bytes(4, 256, 48, 48, 19) == 148 * 19 * 256 * 4
    # BatchNorm statistics: one fp64 [sum | sq] row pair per GEMM CTA
    assert lib.pm_conv1x1_stats_scratch_bytes(8, 256, 96 * 96, 0) == 148 * 2 * 256 * 8
    assert lib.pm_conv1x1_stats_scratch_bytes(1, 64, 256, 1) == 2 * 2 * 64 * 8
    # read loss: N*KP floats plus the halos -- between 1x and 2x the ds_rl buffer at cfg 2
    n = lib.pm_readloss_scratch_bytes(8, 96, 96, 768, 768, 19, 1)
    assert 8 * 96 * 96 * 20 * 4 < n < 2 * 8 * 96 * 96 * 20 * 4
    n = lib.pm_readloss_scratch_bytes(8, 96, 96, 768, 768, 25, 0)
    assert 8 * 96 * 96 * 32 * 4 < n < 2 * 8 * 96 * 96 * 32 * 4
