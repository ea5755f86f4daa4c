"""GPU (one device): the global-read exchange kernels of csrc/pm_exchange.cu and pm_score_bwd_global, entry by entry.

Two "ranks" live on one GPU: each has its own score map, read-loss workspace and column-softmax partials. The gathered path
combines rows stacked in rank order (what the NCCL all-gather produces); the peer path runs the two ranks' one-CTA kernels
on two streams over two buffers laid out like the symmetric peer buffers, for several launches in a row (epochs, the
deferred "done" round). Both must give what one call over the concatenated pixels gives, identically on both ranks, and
the two paths must agree bit for bit.

The peer-path checks need both ranks' one-CTA kernels resident on the GPU at the same time, as they are on separate GPUs.
CUDA does not promise that for two streams of one device; it holds when launches are asynchronous and the device is not
full, which is the case here (two 64-thread CTAs, nothing else running). With CUDA_LAUNCH_BLOCKING set, launches are
serialised and the first rank's kernel would wait for a peer that cannot start: those checks are skipped then.
"""
import os
import types

import pytest
import torch

pytestmark = pytest.mark.gpu

K, T = 19, 0.7
SHAPES = ((3, 12, 16), (1, 12, 16))   # (B, h, w) of the two ranks: an uneven split
Hm, Wm = 48, 64


def _rank_inputs(r, B, h, w, dev, empty=False):
    from pinthememory_b200 import capi, synth

    KP = capi.score_stride(K)
    g = torch.Generator(device="cpu").manual_seed(10 + r)
    s = torch.zeros(B * h * w, KP, dtype=torch.float32)
    s[:, :K] = torch.randn(B * h * w, K, generator=g) * 2.0
    s = s.to(dev)
    labels = synth.make_labels(B, Hm, Wm, K, "blocky", seed=20 + r, device=dev, block=8)
    if r == 0:
        labels[:, : 3 * Hm // 4] = 255
    if empty:
        labels[:] = 255
    return s, labels


def _forward_one_rank(s, labels, B, h, w):
    """The rank's own statistics: column partials (combined row filled) and the read-loss workspace / out."""
    from pinthememory_b200 import capi

    N = B * h * w
    KP = capi.score_stride(K)
    cp = torch.zeros(capi.colsoftmax_workspace_floats(K), dtype=torch.float32, device=s.device)
    sq_local = torch.empty(N, K, dtype=torch.float32, device=s.device)
    capi.colsoftmax(s, None, sq_local, cp, N, K)
    buf = torch.zeros(N * KP + 2 * capi.WS_WORDS + 4, dtype=torch.float32, device=s.device)
    ds_rl, ws, out = buf[: N * KP], buf[N * KP: N * KP + 2 * capi.WS_WORDS], buf[N * KP + 2 * capi.WS_WORDS:]
    capi.readloss(s, labels, T, B, h, w, K, ds_rl, ws, out)
    return cp, ws, out, ds_rl


def _fake_peers(dev, world):
    from pinthememory_b200 import capi

    bufs = [torch.zeros(capi.PEER_BYTES // 4, dtype=torch.float32, device=dev) for _ in range(world)]
    ptrs = torch.tensor([b.data_ptr() for b in bufs], dtype=torch.int64, device=dev)
    peers = [types.SimpleNamespace(bufs_dev=ptrs.data_ptr(), rank=r, world_size=world,
                                   epochs=torch.zeros(4, dtype=torch.int32, device=dev)) for r in range(world)]
    return peers, (bufs, ptrs)


def _require_concurrent_launches():
    if os.environ.get("CUDA_LAUNCH_BLOCKING", "0") not in ("", "0"):
        pytest.skip("CUDA_LAUNCH_BLOCKING serialises launches: the two simulated ranks could not run at the same time")


def _on_rank_streams(streams, fns):
    """fns[r]() on streams[r]: the ranks' kernels run concurrently, as on separate GPUs."""
    cur = torch.cuda.current_stream()
    for st in streams:
        st.wait_stream(cur)
    for st, fn in zip(streams, fns):
        with torch.cuda.stream(st):
            fn()
    for st in streams:
        cur.wait_stream(st)


def _global_reference(ss, labs):
    from oracle import memory_oracle as mo

    s_all = torch.cat([s[:, :K] for s in ss]).double()
    sq = torch.softmax(s_all, dim=0)
    maps = [s[:, :K].reshape(B, h, w, K) for s, (B, h, w) in zip(ss, SHAPES)]
    # the read loss of the concatenated batch: every rank's maps share h, w
    rl = mo.feature_cohesion_loss(torch.cat(maps).double(), torch.cat(labs), T)
    return sq, rl


@pytest.mark.parametrize("empty_rank1", [False, True])
def test_forward_exchange_gathered_and_peer(empty_rank1):
    from golden_util import assert_close
    from pinthememory_b200 import capi

    dev = torch.device("cuda")
    world = 2
    ins = [_rank_inputs(r, *SHAPES[r], dev, empty=(empty_rank1 and r == 1)) for r in range(world)]
    ref_sq, ref_rl = _global_reference([i[0] for i in ins], [i[1] for i in ins])
    base = [_forward_one_rank(s, lab, *SHAPES[r]) for r, (s, lab) in enumerate(ins)]

    # gathered rows (the NCCL fallback's layout)
    cps = [b[0].clone() for b in base]
    wss = [b[1].clone() for b in base]
    outs = [b[2].clone() for b in base]
    rows = torch.empty(world, capi.READ_ROW_FLOATS, dtype=torch.float32, device=dev)
    for r in range(world):
        capi.read_row_fwd(cps[r], wss[r], rows[r], K)
    sq_g = []
    for r in range(world):
        capi.read_exchange_fwd(None, rows, world, cps[r], wss[r], T, outs[r], K)
        N = SHAPES[r][0] * SHAPES[r][1] * SHAPES[r][2]
        sq = torch.empty(N, K, dtype=torch.float32, device=dev)
        capi.colsoftmax_apply(ins[r][0], None, cps[r], sq, N, K)
        sq_g.append(sq)
    torch.cuda.synchronize()
    assert torch.equal(outs[0], outs[1])
    assert torch.isfinite(outs[1][0])
    assert_close(outs[0][0:1].double(), ref_rl.reshape(1), 1e-5, "readloss")
    V = sum(int((lab < K).sum()) for _, lab in ins)
    assert_close(outs[0][1:2].double(), torch.tensor([1.0 / (V * T)], dtype=torch.float64, device=dev), 1e-7, "scale")
    assert_close(torch.cat(sq_g).double(), ref_sq, 1e-5, "score_query")

    # peer memory: three launches in a row on the two ranks' streams (epochs 1..3, the done round between them)
    _require_concurrent_launches()
    peers, keep = _fake_peers(dev, world)
    streams = [torch.cuda.Stream() for _ in range(world)]
    for rep in range(3):
        cps_p = [b[0].clone() for b in base]
        outs_p = [b[2].clone() for b in base]
        _on_rank_streams(streams, [lambda r=r: capi.read_exchange_fwd(peers[r], None, world, cps_p[r], base[r][1], T,
                                                                      outs_p[r], K) for r in range(world)])
        torch.cuda.synchronize()
        for r in range(world):
            assert torch.equal(outs_p[r], outs[r]), (rep, r)
            assert torch.equal(cps_p[r], cps[r]), (rep, r)
    for p in peers:
        assert int(p.epochs[2]) == 3 and int(p.epochs[3]) == 0


def test_forward_exchange_without_labels_changes_only_the_column_statistics():
    from pinthememory_b200 import capi

    dev = torch.device("cuda")
    ins = [_rank_inputs(r, *SHAPES[r], dev) for r in range(2)]
    cps = [_forward_one_rank(s, lab, *SHAPES[r])[0] for r, (s, lab) in enumerate(ins)]
    rows = torch.empty(2, capi.READ_ROW_FLOATS, dtype=torch.float32, device=dev)
    for r in range(2):
        capi.read_row_fwd(cps[r], None, rows[r], K)
    torch.cuda.synchronize()
    assert float(rows[:, 64:68].abs().sum()) == 0.0   # the two doubles: no loss sum, no valid count
    ref_sq, _ = _global_reference([i[0] for i in ins], [i[1] for i in ins])
    sqs = []
    for r in range(2):
        capi.read_exchange_fwd(None, rows, 2, cps[r], None, T, None, K)
        N = SHAPES[r][0] * SHAPES[r][1] * SHAPES[r][2]
        sq = torch.empty(N, K, dtype=torch.float32, device=dev)
        capi.colsoftmax_apply(ins[r][0], None, cps[r], sq, N, K)
        sqs.append(sq)
    from golden_util import assert_close

    assert_close(torch.cat(sqs).double(), ref_sq, 1e-5, "score_query")


def test_backward_exchange_and_score_bwd_global():
    """c_k summed over both ranks, the readloss gradients summed; pm_score_bwd_global on each rank's pixels equals
    pm_score_bwd over the concatenated pixels."""
    from golden_util import assert_close
    from pinthememory_b200 import capi

    dev = torch.device("cuda")
    world = 2
    KP = capi.score_stride(K)
    gen = torch.Generator(device="cpu").manual_seed(3)
    Ns = [B * h * w for B, h, w in SHAPES]
    p = [torch.softmax(torch.randn(n, K, generator=gen), 0).to(dev) for n in Ns]
    g = [torch.randn(n, K, generator=gen).to(dev) for n in Ns]
    pm = [torch.softmax(torch.randn(n, K, generator=gen), 1).to(dev) for n in Ns]
    gm = [torch.randn(n, K, generator=gen).to(dev) for n in Ns]
    ds = [torch.zeros(n, KP, device=dev) for n in Ns]
    for d in ds:
        d[:, :K] = torch.randn(d.shape[0], K, generator=gen).to(dev)
    g_loss = [torch.tensor([0.02], device=dev), torch.tensor([0.03], device=dev)]
    rl_out = torch.tensor([0.0, 1e-3], device=dev)

    parts = [capi.score_bwd_partials(p[r], g[r], K) for r in range(world)]
    rows = torch.empty(world, capi.READ_ROW_FLOATS, dtype=torch.float32, device=dev)
    for r in range(world):
        capi.read_row_bwd(parts[r], g_loss[r], rows[r], K)
    res = []
    for r in range(world):
        buf = torch.empty(33, dtype=torch.float64, device=dev)
        colsums, gsum = buf[:32], buf[32:].view(torch.float32)[:1]
        capi.read_exchange_bwd(None, rows, world, parts[r], g_loss[r], gsum, colsums, K)
        res.append((gsum, colsums))
    torch.cuda.synchronize()
    assert torch.equal(res[0][0], res[1][0]) and torch.equal(res[0][1], res[1][1])
    assert float(res[0][0]) == pytest.approx(0.05, rel=1e-7)
    c_ref = sum((pi.double() * gi.double()).sum(0) for pi, gi in zip(p, g))
    assert_close(res[0][1][:K], c_ref, 1e-12, "column sums")
    assert float(res[0][1][K:].abs().sum()) == 0.0

    # the peer path: same bits, over three launches
    _require_concurrent_launches()
    peers, keep = _fake_peers(dev, world)
    streams = [torch.cuda.Stream() for _ in range(world)]
    for rep in range(3):
        out_p = [(torch.empty(1, device=dev), torch.empty(32, dtype=torch.float64, device=dev)) for _ in range(world)]
        _on_rank_streams(streams, [lambda r=r: capi.read_exchange_bwd(peers[r], None, world, parts[r], g_loss[r], out_p[r][0],
                                                                      out_p[r][1], K) for r in range(world)])
        torch.cuda.synchronize()
        for r in range(world):
            assert torch.equal(out_p[r][0], res[r][0]) and torch.equal(out_p[r][1], res[r][1]), (rep, r)

    # E per rank with the global sums == E of one call over all pixels (with the summed readloss gradient)
    E_all = torch.empty(sum(Ns), KP, device=dev)
    capi.score_bwd(torch.cat(p), torch.cat(g), torch.cat(pm), torch.cat(gm), E_all, K, ds_rl=torch.cat(ds),
                   g_loss=res[0][0], rl_out=rl_out)
    Es = []
    for r in range(world):
        E = torch.empty(Ns[r], KP, device=dev)
        capi.score_bwd_global(p[r], g[r], pm[r], gm[r], E, K, res[r][1], ds_rl=ds[r], g_loss=res[r][0], rl_out=rl_out)
        Es.append(E)
    torch.cuda.synchronize()
    assert_close(torch.cat(Es), E_all, 1e-6, "E")
    # and a single rank's global form with its own sums is pm_score_bwd bit for bit
    own = torch.empty(33, dtype=torch.float64, device=dev)
    capi.read_exchange_bwd(None, rows[:1], 1, parts[0], g_loss[0], own[32:].view(torch.float32)[:1], own[:32], K)
    E0, E1 = torch.empty(Ns[0], KP, device=dev), torch.empty(Ns[0], KP, device=dev)
    capi.score_bwd(p[0], g[0], pm[0], gm[0], E0, K, ds_rl=ds[0], g_loss=g_loss[0], rl_out=rl_out)
    capi.score_bwd_global(p[0], g[0], pm[0], gm[0], E1, K, own[:32], ds_rl=ds[0], g_loss=own[32:].view(torch.float32)[:1],
                          rl_out=rl_out)
    torch.cuda.synchronize()
    assert torch.equal(E0, E1)


def test_only_grad_mode_reads_exchange(monkeypatch):
    """A read under torch.no_grad (validation, memory_initalize) stays rank-local and launches no exchange, so ranks need
    not make such reads in lock-step; a grad-mode read of the same module does exchange. The shard group is a stand-in
    (two ranks, no peers) whose exchange records the call instead of running it."""
    from pinthememory_b200 import sharding, synth
    from pinthememory_b200.memory import Memory_sup

    dev = torch.device("cuda")
    calls = []

    def record(*args, **kwargs):
        calls.append(1)
        raise RuntimeError("exchange called")

    monkeypatch.setattr(sharding, "read_exchange_fwd", record)
    torch.manual_seed(7)
    mem = Memory_sup(K, 64, 64, 0.8, 1.0, False).to(dev).eval()
    mem.m_items = mem.m_items.to(dev)
    mem.shard_group = types.SimpleNamespace(global_read=True, world_size=2, rank=0, peer=None, group=None)
    x = synth.make_features(2, 64, 12, 16, seed=1, device=dev)
    lab = synth.make_labels(2, Hm, Wm, K, "blocky", seed=2, device=dev)
    with torch.no_grad():
        mem(x, lab, False)
        mem(x, None, False)
    assert calls == []
    with pytest.raises(RuntimeError, match="exchange called"):
        mem(x.clone().requires_grad_(True), lab, False)
    assert calls == [1]
