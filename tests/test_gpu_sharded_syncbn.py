"""GPU, 2 ranks: SyncBatchNorm (``convert_sync_batchnorm``, the reference under --syncbn) over the sharded update's peer
memory.

Needs >= 2 CUDA devices (skipped otherwise). With ``enable_sharded_update`` and its peer exchange, both SyncBatchNorm layers
of the module (the output block and the writing net) sum their batch statistics and backward sums over the same symmetric
buffer as the class sums, in rank order, with no NCCL call. The checker is the oracle with plain BatchNorm2d on the
concatenated batch. Objective of rank r: <uq_r, G_r> + 0.4 div + 0.2 cls, so rank r's dx is the slice of the gradient of
<uq, G> + 2 (0.4 div + 0.2 cls) on the whole batch, and the ranks' parameter gradients add up to that objective's gradient.
"""
import os
import socket

import pytest
import torch

pytestmark = [pytest.mark.gpu, pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs 2 GPUs")]

WORLD = 2
K, C, h, w, Hm, Wm = 19, 64, 12, 16, 48, 64
SPLIT = (3, 5)
B = sum(SPLIT)
LW = dict(div=0.4, cls=0.2)


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def _slices(split):
    out, a = [], 0
    for n in split:
        out.append(slice(a, a + n))
        a += n
    return out


def _inputs(device, dtype=torch.float32):
    from pinthememory_b200 import synth

    x = synth.make_features(B, C, h, w, seed=21, device=device).to(dtype)
    labels = synth.make_labels(B, Hm, Wm, K, "blocky", seed=22, device=device, block=8)
    G = synth.make_upstream_grad((B, C, h, w), seed=23, device=device).to(dtype)
    return x, labels, G


def _state(device):
    from oracle import memory_oracle as mo

    torch.manual_seed(7)
    ora = mo.OracleMemorySup(K, C, C, 0.8, 1.0, False)
    with torch.no_grad():
        ora.clsfier.weight.normal_(0, 0.2)
        for m in ora.modules():
            if isinstance(m, torch.nn.BatchNorm2d):
                m.running_mean.normal_(0, 0.1)
                m.running_var.uniform_(0.5, 1.5)
    ora = ora.to(device).train()
    ora.m_items = ora.m_items.to(device)
    return ora


# ------------------------------------------------------------------------------------------------------------- ranks


def _module(ora, dev, peer_exchange=True, overlap=False, unfused=False, sync_first=True):
    from pinthememory_b200 import sharding
    from pinthememory_b200.memory import Memory_sup

    mem = Memory_sup(K, C, C, 0.8, 1.0, False).to(dev)
    mem.load_state_dict(ora.state_dict())
    mem.m_items = ora.m_items.clone()
    mem.fold_min_pixels = 0
    mem.overlap_write = overlap
    if unfused:   # a hooked writing net runs as Writingnet + _WriteFn
        mem.writenet.register_forward_hook(lambda mod, i, o: None)
    if sync_first:
        mem = torch.nn.SyncBatchNorm.convert_sync_batchnorm(mem)
        shard = sharding.enable_sharded_update(mem, peer_exchange=peer_exchange)
    else:         # the order must not matter: the path is chosen per call from the live layer
        shard = sharding.enable_sharded_update(mem, peer_exchange=peer_exchange)
        mem = torch.nn.SyncBatchNorm.convert_sync_batchnorm(mem)
    return mem.train(), shard


def _step(mem, xr, lr, Gr):
    xr = xr.clone().requires_grad_(True)
    mem.zero_grad(set_to_none=True)
    uq, _, _, _, wl = mem(xr, lr, True, False)
    ((uq.float() * Gr.float()).sum() + LW["div"] * wl[0] + LW["cls"] * wl[1]).backward()
    return dict(uq=uq.detach().float().cpu(), dx=xr.grad.float().cpu(), m_items=mem.m_items.detach().cpu(),
                grads={k: p.grad.float().cpu() for k, p in mem.named_parameters() if p.grad is not None},
                rm=[mem.output[1].running_mean.cpu(), mem.writenet.writefeat[1].running_mean.cpu()],
                rv=[mem.output[1].running_var.cpu(), mem.writenet.writefeat[1].running_var.cpu()])


def _cuda_kernels(fn):
    from torch.autograd import DeviceType
    from torch.profiler import ProfilerActivity, profile

    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    return [e.name for e in prof.events() if e.device_type == DeviceType.CUDA]


def _worker(rank, world, port, out):
    import torch.distributed as dist

    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    os.environ.pop("PINMEM_B200_NCCL_EXCHANGE", None)
    torch.cuda.set_device(rank)
    dev = torch.device("cuda", rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=dev)
    try:
        torch.backends.cudnn.allow_tf32 = False
        torch.backends.cuda.matmul.allow_tf32 = False
        from pinthememory_b200.graphed import GraphedStep

        res = {}
        ora = _state(dev)
        sl = _slices(SPLIT)[rank]
        x, labels, G = _inputs(dev)
        xr, lr, Gr = x[sl].contiguous(), labels[sl].contiguous(), G[sl].contiguous()

        mem, shard = _module(ora, dev)
        res["peer"], res["peer_error"] = shard.peer is not None, shard.peer_error
        res["fused"] = _step(mem, xr, lr, Gr)
        res["epochs"] = shard.peer.epochs.cpu() if shard.peer is not None else None
        mem, _ = _module(ora, dev, unfused=True)
        res["unfused"] = _step(mem, xr, lr, Gr)
        mem, _ = _module(ora, dev, sync_first=False)
        res["enable_first"] = _step(mem, xr, lr, Gr)
        mem, _ = _module(ora, dev, overlap=True)
        res["two_stream"] = _step(mem, xr, lr, Gr)
        mem, _ = _module(ora, dev, peer_exchange=False)
        res["nccl"] = _step(mem, xr, lr, Gr)
        xb, _, Gb = _inputs(dev, torch.bfloat16)
        mem, _ = _module(ora, dev)
        res["bf16"] = _step(mem, xb[sl].contiguous(), lr, Gb[sl].contiguous())

        # deterministic algorithms: two identical steps, identical bits
        torch.use_deterministic_algorithms(True)
        try:
            reps = []
            for _ in range(2):
                mem, _ = _module(ora, dev, overlap=True)
                reps.append(_step(mem, xr, lr, Gr))
            res["deterministic"] = reps
        finally:
            torch.use_deterministic_algorithms(False)

        # GraphedStep: three replays equal three eager steps (memory carried)
        eager_mem, _ = _module(ora, dev, overlap=True)
        graph_mem, _ = _module(ora, dev, overlap=True)
        gs = GraphedStep(graph_mem, xr, lr, Gr, loss_weights=(0.0, LW["div"], LW["cls"]))
        rows = []
        for _ in range(3):
            xq = xr.clone().requires_grad_(True)
            eager_mem.zero_grad(set_to_none=True)
            uq, _, _, rl, wl = eager_mem(xq, lr, True, True)
            torch.autograd.backward([uq, wl[0], wl[1]], [Gr, *(torch.tensor(LW[k], device=dev) for k in ("div", "cls"))])
            eager_mem.m_items = eager_mem.m_items.detach()
            o = gs.replay()
            rows.append(dict(e_uq=uq.detach().cpu(), g_uq=o["updated_query"].cpu(), e_dx=xq.grad.cpu(),
                             g_dx=gs.query_grad.cpu(), e_m=eager_mem.m_items.cpu(), g_m=o["memory"].cpu()))
        gs.release()
        res["graphed"] = rows

        # the kernels of one step: no NCCL kernel on the peer path; the NCCL path keeps its all-reduces
        for name, kw in (("trace_peer", {}), ("trace_nccl", dict(peer_exchange=False))):
            mem, _ = _module(ora, dev, **kw)
            _step(mem, xr, lr, Gr)
            res[name] = _cuda_kernels(lambda: _step(mem, xr, lr, Gr))
        out[rank] = res
    finally:
        dist.destroy_process_group()


@pytest.fixture(scope="module")
def ranks():
    import torch.multiprocessing as mp

    out = mp.get_context("spawn").Manager().dict()
    mp.spawn(_worker, args=(WORLD, _free_port(), out), nprocs=WORLD, join=True)
    res = {r: out[r] for r in range(WORLD)}
    if not res[0]["peer"]:
        pytest.skip("no symmetric-memory peer exchange on this box: %s" % res[0]["peer_error"])
    return res


# ---------------------------------------------------------------------------------------------------------- checker


def _oracle(dtype=torch.float32):
    """The oracle with plain BatchNorm2d on the concatenated batch (fp32; a bf16 run is compared to it at bf16's bar)."""
    from oracle import memory_oracle as mo

    torch.backends.cudnn.allow_tf32 = False
    torch.backends.cuda.matmul.allow_tf32 = False
    dev = torch.device("cuda", 0)
    ora = _state(dev)
    x, labels, G = _inputs(dev, dtype)
    xa = x.float().clone().requires_grad_(True)
    M0 = ora.m_items.clone()
    rd = mo.read(xa, M0, None, 1.0)
    uq = ora.output(rd["u"])
    wr = mo.write(ora.writenet(xa), labels, M0, 0.8, ora.clsfier.weight, ora.clsfier.bias)
    ((uq * G.float()).sum() + WORLD * (LW["div"] * wr["div_loss"] + LW["cls"] * wr["cls_loss"])).backward()
    return dict(uq=uq.detach().cpu(), dx=xa.grad.cpu(), m_items=wr["memory_new"].detach().cpu(),
                grads={k: p.grad.cpu() for k, p in ora.named_parameters() if p.grad is not None},
                rm=[ora.output[1].running_mean.cpu(), ora.writenet.writefeat[1].running_mean.cpu()],
                rv=[ora.output[1].running_var.cpu(), ora.writenet.writefeat[1].running_var.cpu()])


def _check(ranks, key, ref, tol_out=1e-5, tol_grad=5e-5):
    from golden_util import assert_close

    assert torch.equal(ranks[0][key]["m_items"], ranks[1][key]["m_items"]), "ranks must hold bit-identical memory"
    for r, sl in enumerate(_slices(SPLIT)):
        got = ranks[r][key]
        assert_close(got["uq"], ref["uq"][sl], tol_out, "%s updated_query rank %d" % (key, r))
        assert_close(got["dx"], ref["dx"][sl], tol_grad, "%s dx rank %d" % (key, r))
        assert_close(got["m_items"], ref["m_items"], tol_out, "%s m_items rank %d" % (key, r))
        for i in range(2):
            assert_close(got["rm"][i], ref["rm"][i], tol_out, "%s running_mean %d rank %d" % (key, i, r))
            assert_close(got["rv"][i], ref["rv"][i], tol_out, "%s running_var %d rank %d" % (key, i, r))
    for k, g in ref["grads"].items():
        assert_close(sum(ranks[r][key]["grads"][k] for r in range(WORLD)), g, tol_grad, "%s grad %s" % (key, k))


# ------------------------------------------------------------------------------------------------------------ tests


@pytest.mark.parametrize("key", ["fused", "unfused", "enable_first", "two_stream"])
def test_peer_path_equals_the_global_batch(ranks, key):
    """3 + 5 images; the fused and the unfused writing net; convert_sync_batchnorm before or after enable_sharded_update;
    one and two streams."""
    _check(ranks, key, _oracle())


def test_bf16_peer_path_equals_the_global_batch(ranks):
    _check(ranks, "bf16", _oracle(torch.bfloat16), tol_out=3e-2, tol_grad=5e-2)


def test_all_four_exchanges_ran_over_peer_memory(ranks):
    # [update fwd, update bwd, read fwd, read bwd, output BN fwd, bwd, writing net BN fwd, bwd] after the first step
    assert ranks[0]["epochs"].tolist() == [1, 1, 0, 0, 1, 1, 1, 1]


def test_peer_path_agrees_with_the_nccl_path(ranks):
    from golden_util import assert_close

    for r in range(WORLD):
        a, b = ranks[r]["fused"], ranks[r]["nccl"]
        for k in ("uq", "dx", "m_items"):
            assert_close(a[k], b[k], 1e-5, "%s rank %d" % (k, r))
        for k in a["grads"]:
            assert_close(a["grads"][k], b["grads"][k], 5e-5, "grad %s rank %d" % (k, r))


def test_deterministic_steps_are_bitwise_identical_and_the_statistics_agree_across_ranks(ranks):
    for r in range(WORLD):
        a, b = ranks[r]["deterministic"]
        for k in ("uq", "dx", "m_items"):
            assert torch.equal(a[k], b[k]), (r, k)
        for k in a["grads"]:
            assert torch.equal(a["grads"][k], b["grads"][k]), (r, k)
    for i in range(2):   # the normalised statistics: the same global sums on both ranks
        assert torch.equal(ranks[0]["deterministic"][0]["rm"][i], ranks[1]["deterministic"][0]["rm"][i])
        assert torch.equal(ranks[0]["deterministic"][0]["rv"][i], ranks[1]["deterministic"][0]["rv"][i])


def test_graphed_step_replays_equal_the_eager_steps(ranks):
    from golden_util import assert_close

    for r in range(WORLD):
        for i, row in enumerate(ranks[r]["graphed"]):
            for k in ("uq", "dx", "m"):
                assert_close(row["g_" + k], row["e_" + k], 1e-5, "rank %d replay %d %s" % (r, i, k))


def test_no_nccl_kernel_on_the_peer_path(ranks):
    for r in range(WORLD):
        peer = [n for n in ranks[r]["trace_peer"] if "nccl" in n.lower()]
        assert peer == [], peer
        nccl = [n for n in ranks[r]["trace_nccl"] if "nccl" in n.lower() and "allreduce" in n.lower()]
        assert len(nccl) >= 4, ranks[r]["trace_nccl"]
