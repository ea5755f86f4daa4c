"""GPU, 2 ranks over NCCL: the global-batch read (``enable_sharded_update(global_read=True)``).

Needs >= 2 CUDA devices (skipped otherwise). The read loss becomes the mean over the valid label pixels of all ranks and
score_query the softmax over all ranks' pixels; the backward sums the ranks' gradients of both. The checker is the oracle
on the concatenated batch in one process. Every check runs once with the exchange over NVLink peer memory ("peer") and
once over NCCL all-gathers ("nccl"); the two ranks run all scenarios in one spawn per exchange.

Objective of the gradient checks: each rank backpropagates its own
    <uq_r, G_r> + <score_query_r, Gq_r> + 0.02 readloss + 0.4 div + 0.2 cls,
so rank r's dx is the slice of the single-process gradient of
    sum_r (<uq_r, G_r> + <score_query_r, Gq_r>) + W (0.02 readloss + 0.4 div + 0.2 cls)
and the ranks' parameter gradients add up to that objective's gradient (DDP's mean then gives the global-batch one).
"""
import os
import socket

import pytest
import torch

pytestmark = [pytest.mark.gpu, pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs 2 GPUs")]

WORLD = 2
K, C, B, h, w, Hm, Wm = 19, 64, 4, 12, 16, 48, 64
SPLIT = (3, 1)            # uneven batch split: images [0,3) on rank 0, [3,4) on rank 1
LW = dict(read=0.02, div=0.4, cls=0.2)
GUMBEL_SEED = 1234


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


def _inputs(device, empty_rank1=False):
    """Blocky labels; rank 0's images are mostly ignore label, so V_0 != V_1. ``empty_rank1``: rank 1 has none valid."""
    from pinthememory_b200 import synth

    x = synth.make_features(B, C, h, w, seed=21, device=device)
    labels = synth.make_labels(B, Hm, Wm, K, "blocky", seed=22, device=device, block=8)
    labels[:3, : 3 * Hm // 4] = 255
    if empty_rank1:
        labels[3:] = 255
    G = synth.make_upstream_grad((B, C, h, w), seed=23, device=device)
    Gq = synth.make_upstream_grad((B, h, w, K), seed=24, device=device) * 1e3   # score_query entries are ~1/N
    return x, labels, G, Gq


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
    ora = ora.to(device).eval()
    ora.m_items = ora.m_items.to(device)
    return ora


# ------------------------------------------------------------------------------------------------------------- ranks


def _module(ora, dev, group=None, global_read=True, syncbn=False, train=False, overlap=False, gumbel=False):
    from pinthememory_b200 import sharding
    from pinthememory_b200.memory import Memory_sup

    mem = Memory_sup(K, C, C, 0.8, 1.0, gumbel).to(dev)
    mem.load_state_dict(ora.state_dict())
    mem.m_items = ora.m_items.clone()
    if syncbn:
        mem = torch.nn.SyncBatchNorm.convert_sync_batchnorm(mem)
    mem = mem.train() if train else mem.eval()
    mem.overlap_write = overlap
    shard = sharding.enable_sharded_update(mem, group=group, global_read=global_read)
    return mem, shard


def _step(mem, xr, lr, Gr, Gqr, writing=True, meta_memory=None):
    """One forward + backward of the rank's objective; returns CPU copies of everything the checks compare."""
    xr = xr.clone().requires_grad_(True)
    mem.zero_grad(set_to_none=True)
    if meta_memory is not None:
        mem.m_items = meta_memory * 1.0   # a memory that carries graph (meta-test read)
    uq, sq, sm, rl, wl = mem(xr, lr, writing, False)
    loss = (uq * Gr).sum() + (sq * Gqr).sum() + LW["read"] * rl
    if writing:
        loss = loss + LW["div"] * wl[0] + LW["cls"] * wl[1]
    loss.backward()
    out = dict(uq=uq.detach().cpu(), sq=sq.detach().cpu(), rl=rl.detach().cpu(), dx=xr.grad.cpu(),
               grads={k: p.grad.cpu() for k, p in mem.named_parameters() if p.grad is not None})
    if writing:
        out["m_items"] = mem.m_items.detach().cpu()
    if meta_memory is not None:
        out["dM"] = meta_memory.grad.cpu()
    return out


def _worker(rank, world, port, out, exchange):
    import torch.distributed as dist

    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    if exchange == "nccl":
        os.environ["PINMEM_B200_NCCL_EXCHANGE"] = "1"
    else:
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
        x, labels, G, Gq = _inputs(dev)
        sl = _slices(SPLIT)[rank]
        xr, lr, Gr, Gqr = x[sl].contiguous(), labels[sl].contiguous(), G[sl].contiguous(), Gq[sl].contiguous()

        # uneven shards, BatchNorm in eval mode, one and two streams
        for overlap in (False, True):
            mem, shard = _module(ora, dev, overlap=overlap)
            res["uneven_two_stream" if overlap else "uneven"] = _step(mem, xr, lr, Gr, Gqr)
        res["peer"] = shard.peer is not None
        res["peer_error"] = shard.peer_error

        # Gumbel read: each rank's noise from GUMBEL_SEED + rank (the checker redraws it with draw_gumbel_pair)
        mem, _ = _module(ora, dev, gumbel=True)
        torch.cuda.manual_seed(GUMBEL_SEED + rank)
        res["gumbel"] = _step(mem, xr, lr, Gr, Gqr)

        # no-grad eval reads (validation's net(inputs), memory_initalize): rank-local, no exchange
        mem, _ = _module(ora, dev)
        with torch.no_grad():
            uq, sq, _, rl, _ = mem(xr, lr, False)
            uq2, sq2, _, rl2, _ = mem(xr, None, False)
        res["no_grad"] = dict(uq=uq.cpu(), sq=sq.cpu(), rl=rl.cpu(), uq2=uq2.cpu(), sq2=sq2.cpu())

        # meta-test read on a memory that carries graph
        mem, _ = _module(ora, dev)
        M = ora.m_items.clone().requires_grad_(True)
        res["meta"] = _step(mem, xr, lr, Gr, Gqr, writing=False, meta_memory=M)

        # rank 1 has no valid label pixel
        _, lab_e, _, _ = _inputs(dev, empty_rank1=True)
        mem, _ = _module(ora, dev)
        res["empty_rank"] = _step(mem, xr, lab_e[sl].contiguous(), Gr, Gqr)

        # GPU-count invariance: SyncBatchNorm + sharded update + global read in training mode, two-stream mode
        even = _slices((2, 2))[rank]
        xe, le, Ge, Gqe = x[even].contiguous(), labels[even].contiguous(), G[even].contiguous(), Gq[even].contiguous()
        mem, _ = _module(ora, dev, syncbn=True, train=True, overlap=True)
        mem.fold_min_pixels = 0
        res["invariance"] = _step(mem, xe, le, Ge, Gqe)

        # determinism: two identical steps, identical bits
        torch.use_deterministic_algorithms(True)
        try:
            reps = []
            for _ in range(2):
                mem, _ = _module(ora, dev, syncbn=True, train=True, overlap=True)
                reps.append(_step(mem, xe, le, Ge, Gqe))
            res["deterministic"] = reps
            # one rank per group: global_read=True is the plain (rank-local) module, bit for bit
            groups = [dist.new_group([r]) for r in range(world)]
            one = []
            for grp in (groups[rank], None):
                mem, _ = _module(ora, dev, group=grp, global_read=True)
                if grp is None:
                    mem.shard_group = None
                one.append(_step(mem, xr, lr, Gr, Gqr))
            res["world1"] = one
        finally:
            torch.use_deterministic_algorithms(False)

        # GraphedStep: replays equal the eager steps (two steps, memory carried)
        eager_mem, _ = _module(ora, dev, syncbn=True, train=True, overlap=True)
        graph_mem, _ = _module(ora, dev, syncbn=True, train=True, overlap=True)
        gs = GraphedStep(graph_mem, xe, le, Ge, loss_weights=(LW["read"], LW["div"], LW["cls"]))
        rows = []
        for _ in range(2):
            xq = xe.clone().requires_grad_(True)
            eager_mem.zero_grad(set_to_none=True)
            uq, sq, sm, rl, wl = eager_mem(xq, le, True, True)
            torch.autograd.backward([uq, rl, wl[0], wl[1]], [Ge, *(torch.tensor(LW[k], device=dev) for k in ("read", "div", "cls"))])
            eager_mem.m_items = eager_mem.m_items.detach()
            o = gs.replay()
            rows.append(dict(e_uq=uq.detach().cpu(), g_uq=o["updated_query"].cpu(), e_sq=sq.detach().cpu(),
                             g_sq=o["score_query"].cpu(), e_rl=rl.detach().cpu(), g_rl=o["readloss"].cpu(),
                             e_dx=xq.grad.cpu(), g_dx=gs.query_grad.cpu(), e_m=eager_mem.m_items.cpu(), g_m=o["memory"].cpu()))
        gs.release()
        res["graphed"] = rows
        out[rank] = res
    finally:
        dist.destroy_process_group()


@pytest.fixture(scope="module", params=["peer", "nccl"])
def ranks(request):
    import torch.multiprocessing as mp

    out = mp.get_context("spawn").Manager().dict()
    mp.spawn(_worker, args=(WORLD, _free_port(), out, request.param), nprocs=WORLD, join=True)
    res = {r: out[r] for r in range(WORLD)}
    if request.param == "peer" and not res[0]["peer"]:
        pytest.skip("no symmetric-memory peer exchange on this box: %s" % res[0]["peer_error"])
    assert res[0]["peer"] == (request.param == "peer")
    return res


# ---------------------------------------------------------------------------------------------------------- checker


def _oracle(labels_fn=_inputs, train=False, gumbel=False, writing=True, meta=False):
    """The oracle on the concatenated batch; returns outputs and gradients of the global objective."""
    from oracle import memory_oracle as mo
    from pinthememory_b200.memory import draw_gumbel_pair

    torch.backends.cudnn.allow_tf32 = False
    torch.backends.cuda.matmul.allow_tf32 = False
    dev = torch.device("cuda", 0)
    ora = _state(dev)
    if train:
        ora = ora.train()
    x, labels, G, Gq = labels_fn(dev)
    xa = x.clone().requires_grad_(True)
    M0 = ora.m_items.clone().requires_grad_(meta)
    noise = None
    if gumbel:
        pairs = []
        for r, sl in enumerate(_slices(SPLIT)):
            torch.cuda.manual_seed(GUMBEL_SEED + r)
            pairs.append(draw_gumbel_pair((sl.stop - sl.start) * h * w, K, dev))
        noise = (torch.cat([p[0] for p in pairs]), torch.cat([p[1] for p in pairs]))
    rd = mo.read(xa, M0, labels, 1.0, noise)
    uq = ora.output(rd["u"])
    J = (uq * G).sum() + (rd["score_query"] * Gq).sum() + WORLD * LW["read"] * rd["readloss"]
    res = dict(uq=uq.detach().cpu(), sq=rd["score_query"].detach().cpu(), rl=rd["readloss"].detach().cpu())
    if writing:
        wr = mo.write(ora.writenet(xa), labels, M0.detach(), 0.8, ora.clsfier.weight, ora.clsfier.bias)
        J = J + WORLD * (LW["div"] * wr["div_loss"] + LW["cls"] * wr["cls_loss"])
        res["m_items"] = wr["memory_new"].detach().cpu()
    J.backward()
    res["dx"] = xa.grad.cpu()
    res["grads"] = {k: p.grad.cpu() for k, p in ora.named_parameters() if p.grad is not None}
    if meta:
        res["dM"] = M0.grad.cpu()
    return res


def _check(ranks, key, ref, split=SPLIT, grads=True):
    from golden_util import assert_close

    assert torch.equal(ranks[0][key]["rl"], ranks[1][key]["rl"]), "readloss must be bit-identical on every rank"
    assert_close(ranks[0][key]["rl"], ref["rl"], 1e-5, key + " readloss")
    for r, sl in enumerate(_slices(split)):
        got = ranks[r][key]
        assert_close(got["sq"], ref["sq"][sl], 1e-5, "%s score_query rank %d" % (key, r))
        assert_close(got["uq"], ref["uq"][sl], 1e-5, "%s updated_query rank %d" % (key, r))
        if "m_items" in ref:
            assert_close(got["m_items"], ref["m_items"], 1e-5, "%s m_items rank %d" % (key, r))
        if grads:
            assert_close(got["dx"], ref["dx"][sl], 5e-5, "%s dx rank %d" % (key, r))
    if "m_items" in ref:
        assert torch.equal(ranks[0][key]["m_items"], ranks[1][key]["m_items"])
    if grads:
        for k, g in ref["grads"].items():
            assert_close(sum(ranks[r][key]["grads"][k] for r in range(WORLD)), g, 5e-5, "%s grad %s" % (key, k))


# ------------------------------------------------------------------------------------------------------------ tests


def test_uneven_shards_equal_the_global_batch(ranks):
    """3 + 1 images, rank 0's mostly ignore label (V_0 != V_1), BatchNorm in eval mode."""
    _check(ranks, "uneven", _oracle())


def test_two_stream_mode_equals_the_global_batch(ranks):
    """overlap_write=True: the exchange runs on the column softmax's side stream."""
    _check(ranks, "uneven_two_stream", _oracle())


def test_gumbel_score_query_equals_the_global_batch(ranks):
    _check(ranks, "gumbel", _oracle(gumbel=True))


def test_meta_test_read_dM_on_a_graph_carrying_memory(ranks):
    from golden_util import assert_close

    ref = _oracle(writing=False, meta=True)
    _check(ranks, "meta", ref)
    assert_close(ranks[0]["meta"]["dM"] + ranks[1]["meta"]["dM"], ref["dM"], 5e-5, "dM")


def test_rank_without_valid_pixels_gets_the_global_readloss(ranks):
    rl = ranks[1]["empty_rank"]["rl"]
    assert torch.isfinite(rl).all()
    _check(ranks, "empty_rank", _oracle(labels_fn=lambda d: _inputs(d, empty_rank1=True)))


def test_module_outputs_and_gradients_are_independent_of_the_gpu_count(ranks):
    """convert_sync_batchnorm + sharded update + global read, training mode, two-stream mode: 2 ranks of 2 images each
    against one process with plain BatchNorm2d on all 4."""
    _check(ranks, "invariance", _oracle(train=True), split=(2, 2))


def test_deterministic_steps_are_bitwise_identical(ranks):
    for r in range(WORLD):
        a, b = ranks[r]["deterministic"]
        for k in ("uq", "sq", "rl", "dx", "m_items"):
            assert torch.equal(a[k], b[k]), (r, k)
        for k in a["grads"]:
            assert torch.equal(a["grads"][k], b["grads"][k]), (r, k)


def test_one_rank_global_read_is_the_rank_local_module_bit_for_bit(ranks):
    for r in range(WORLD):
        a, b = ranks[r]["world1"]
        for k in ("uq", "sq", "rl", "dx", "m_items"):
            assert torch.equal(a[k], b[k]), (r, k)


def test_graphed_step_replays_equal_the_eager_steps(ranks):
    from golden_util import assert_close

    for r in range(WORLD):
        for i, row in enumerate(ranks[r]["graphed"]):
            for k in ("uq", "sq", "rl", "dx", "m"):
                assert_close(row["g_" + k], row["e_" + k], 1e-5, "rank %d replay %d %s" % (r, i, k))
    for i in range(2):
        assert torch.equal(ranks[0]["graphed"][i]["g_rl"], ranks[1]["graphed"][i]["g_rl"])


def test_no_grad_eval_read_stays_rank_local(ranks):
    """A read under torch.no_grad exchanges nothing: each rank's readloss and score_query are those of its own images (the
    oracle on the rank's slice), with and without labels."""
    from golden_util import assert_close
    from oracle import memory_oracle as mo

    dev = torch.device("cuda", 0)
    ora = _state(dev)
    x, labels, _, _ = _inputs(dev)
    with torch.no_grad():
        for r, sl in enumerate(_slices(SPLIT)):
            rd = mo.read(x[sl], ora.m_items, labels[sl], 1.0)
            got = ranks[r]["no_grad"]
            assert_close(got["rl"], rd["readloss"].cpu(), 1e-5, "rank-local readloss rank %d" % r)
            assert_close(got["sq"], rd["score_query"].cpu(), 1e-5, "rank-local score_query rank %d" % r)
            assert_close(got["sq2"], rd["score_query"].cpu(), 1e-5, "rank-local score_query (no labels) rank %d" % r)
            assert_close(got["uq"], ora.output(rd["u"]).cpu(), 1e-5, "updated_query rank %d" % r)
