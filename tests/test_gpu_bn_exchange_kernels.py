"""GPU (one device): the SyncBatchNorm exchanges of csrc/pm_bn_exchange.cu, entry by entry.

Two or four "ranks" live on one GPU, each with its own buffer laid out like the symmetric peer buffers and its own launch
counters; their one-CTA kernels run on separate streams. The forward must leave on every rank the rank-order fp64 sum of
all ranks' [sum | sum of squares | count] bit for bit, the backward the rank-order fp64 sum of (dgamma, dbeta) times
local / global count, rounded once; over several launches in a row (epochs, the deferred "done" round) and with the two
slots in flight at the same time on different streams.

As in test_gpu_read_exchange_kernels.py, these checks need the ranks' kernels resident on the GPU at the same time, as they
are on separate GPUs: CUDA does not promise that for streams of one device, but it holds with asynchronous launches on an
otherwise idle device. With CUDA_LAUNCH_BLOCKING set launches are serialised, and the checks are skipped.
"""
import os

import pytest
import torch

pytestmark = pytest.mark.gpu


def _require_concurrent_launches():
    if os.environ.get("CUDA_LAUNCH_BLOCKING", "0") not in ("", "0"):
        pytest.skip("CUDA_LAUNCH_BLOCKING serialises launches: the simulated ranks could not run at the same time")


def _fake_peers(dev, world):
    """PeerExchange objects of `world` simulated ranks on one device: buffers, the device array of their addresses, and the
    eight launch counters of sharding.PeerExchange."""
    from pinthememory_b200 import capi, sharding

    bufs = [torch.zeros(capi.PEER_BYTES // 4, dtype=torch.float32, device=dev) for _ in range(world)]
    ptrs = torch.tensor([b.data_ptr() for b in bufs], dtype=torch.int64, device=dev)
    peers = []
    for r in range(world):
        p = object.__new__(sharding.PeerExchange)
        p.buffer, p.rank, p.world_size, p.bufs_dev = bufs[r], r, world, ptrs.data_ptr()
        p.epochs = torch.zeros(8, dtype=torch.int32, device=dev)
        peers.append(p)
    return peers, (bufs, ptrs)


def _on_streams(streams, fns):
    cur = torch.cuda.current_stream()
    for st in streams:
        st.wait_stream(cur)
    for st, fn in zip(streams, fns):
        with torch.cuda.stream(st):
            fn()
    for st in streams:
        cur.wait_stream(st)


def _fwd_inputs(world, M, dev, seed):
    g = torch.Generator(device="cpu").manual_seed(seed)
    counts = [float(192 * (2 * r + 3)) for r in range(world)]          # uneven: 3, 5, 7, 9 images of 192 pixels
    stats = []
    for r in range(world):
        s = torch.empty(2 * M + 1, dtype=torch.float64)
        s[:M] = torch.randn(M, generator=g, dtype=torch.float64) * counts[r]
        s[M:2 * M] = torch.rand(M, generator=g, dtype=torch.float64) * counts[r] * 3.0
        s[2 * M] = -1.0                                                 # overwritten with the count by the kernel
        stats.append(s.to(dev))
    ref = torch.zeros(2 * M + 1, dtype=torch.float64)
    for r in range(world):                                              # rank order, fp64
        row = stats[r].cpu().clone()
        row[2 * M] = counts[r]
        ref += row
    return stats, counts, ref


def _bwd_inputs(world, M, dev, seed, counts):
    g = torch.Generator(device="cpu").manual_seed(seed)
    dg = [torch.randn(M, generator=g).to(dev) for _ in range(world)]
    db = [torch.randn(M, generator=g).to(dev) for _ in range(world)]
    glob = sum(counts)
    acc = torch.zeros(2 * M, dtype=torch.float64)
    for r in range(world):
        acc += torch.cat([dg[r], db[r]]).cpu().double()
    refs = [(acc * (counts[r] / glob)).float() for r in range(world)]  # fp64 sum x local / global, rounded once
    return dg, db, torch.tensor([glob], dtype=torch.float64, device=dev), refs


@pytest.mark.parametrize("world", [2, 4])
@pytest.mark.parametrize("M", [64, 256])
def test_forward_and_backward_exchange_equal_the_rank_order_sums(world, M):
    from pinthememory_b200 import capi

    _require_concurrent_launches()
    dev = torch.device("cuda")
    peers, keep = _fake_peers(dev, world)
    streams = [torch.cuda.Stream() for _ in range(world)]
    stats0, counts, ref = _fwd_inputs(world, M, dev, seed=world * 1000 + M)
    for rep in range(3):                                                # epochs 1..3 and the done round between them
        for slot in (0, 1):
            stats = [s.clone() for s in stats0]
            _on_streams(streams, [lambda r=r: capi.bn_exchange_fwd(peers[r], slot, stats[r], counts[r], M) for r in range(world)])
            torch.cuda.synchronize()
            for r in range(world):
                assert torch.equal(stats[r].cpu(), ref), (rep, slot, r)
    dg, db, glob, refs = _bwd_inputs(world, M, dev, seed=world + M, counts=counts)
    for rep in range(3):
        for slot in (0, 1):
            outs = [torch.full((2 * M,), float("nan"), device=dev) for _ in range(world)]
            _on_streams(streams, [lambda r=r: capi.bn_exchange_bwd(peers[r], slot, dg[r], db[r], glob, counts[r], outs[r][:M],
                                                                   outs[r][M:], M) for r in range(world)])
            torch.cuda.synchronize()
            for r in range(world):
                assert torch.equal(outs[r].cpu(), refs[r]), (rep, slot, r)
    for p in peers:
        assert p.epochs.tolist() == [0, 0, 0, 0, 3, 3, 3, 3]


def test_two_slots_in_flight_on_different_streams():
    """The output block's and the writing net's exchanges of one step overlap (two-stream mode): slot 0 on one stream, slot 1
    on another, per rank, for three steps; every result equals the one-slot-at-a-time result."""
    from pinthememory_b200 import capi

    _require_concurrent_launches()
    dev = torch.device("cuda")
    world, Ms = 2, (256, 64)
    peers, keep = _fake_peers(dev, world)
    streams = [torch.cuda.Stream() for _ in range(world * 2)]
    ins = [_fwd_inputs(world, M, dev, seed=40 + M) for M in Ms]
    bw = [_bwd_inputs(world, M, dev, seed=50 + M, counts=ins[s][1]) for s, M in enumerate(Ms)]
    for rep in range(3):
        stats = [[t.clone() for t in ins[s][0]] for s in range(2)]
        fns = [lambda r=r, s=s: capi.bn_exchange_fwd(peers[r], s, stats[s][r], ins[s][1][r], Ms[s])
               for r in range(world) for s in range(2)]
        _on_streams(streams, fns)
        torch.cuda.synchronize()
        for s in range(2):
            for r in range(world):
                assert torch.equal(stats[s][r].cpu(), ins[s][2]), (rep, s, r)
        outs = [[torch.empty(2 * M, device=dev) for _ in range(world)] for M in Ms]
        fns = [lambda r=r, s=s: capi.bn_exchange_bwd(peers[r], s, bw[s][0][r], bw[s][1][r], bw[s][2], ins[s][1][r],
                                                     outs[s][r][:Ms[s]], outs[s][r][Ms[s]:], Ms[s])
               for r in range(world) for s in range(2)]
        _on_streams(streams, fns)
        torch.cuda.synchronize()
        for s in range(2):
            for r in range(world):
                assert torch.equal(outs[s][r].cpu(), bw[s][3][r]), (rep, s, r)
    for p in peers:
        assert p.epochs.tolist()[4:] == [3, 3, 3, 3]
