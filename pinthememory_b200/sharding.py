"""Batch sharding of the memory path across the GPUs of one box (SURVEY.md 8e).

Read (including the read loss) is per-pixel independent given the memory, so ranks just process their own
images. The write has ONE exchange step: the packed per-class sums|counts ``[K+1, C+4]`` fp32 (~21 KB)
are all-reduced (sum) over NCCL/NVLink before the momentum update, and -- the autograd mirror -- the
gradient w.r.t. the class sums ``[K, C]`` is all-reduced in the backward. Every rank then holds a
bit-identical ``m_items`` equal to the single-process update on the concatenated global batch.
The reference has no such collective (each rank silently keeps its own memory, SURVEY.md 2.1).

Opt-in (``global_read=True``): the read loss and score_query, the read's two reductions over pixels, are also taken over
the global batch -- one small row per rank exchanged before the column softmax and one in the backward
(csrc/pm_exchange.cu).

SyncBatchNorm layers (``convert_sync_batchnorm``) that reduce over the shard group sum their batch statistics and backward
sums over the same peer buffers (csrc/pm_bn_exchange.cu; ``bn_peer``), else with NCCL all-reduces.
"""
import torch
import torch.distributed as dist


class PeerExchange:
    """Symmetric (peer-mapped) buffer of one module for the exchange fused into the update kernels (pm_update_fwd_peer /
    pm_update_bwd_peer, include/pinmem_b200.h): every rank allocates ``PM_PEER_BYTES`` through
    ``torch.distributed._symmetric_memory``, the rendezvous hands every rank the others' addresses, and the kernels read
    the class sums / their gradient straight out of the peers' buffers over NVLink -- no NCCL launch on the step."""

    def __init__(self, group, device):
        import torch.distributed._symmetric_memory as symm

        from . import capi

        pg = group if group is not None else dist.group.WORLD
        self.buffer = symm.empty(capi.PEER_BYTES // 4, dtype=torch.float32, device=device)
        self.buffer.zero_()
        self.handle = symm.rendezvous(self.buffer, pg.group_name)
        self.rank, self.world_size = self.handle.rank, self.handle.world_size
        self.bufs_dev = int(self.handle.buffer_ptrs_dev)      # device array of all ranks' buffer addresses
        # one launch counter per kernel kind: update fwd, update bwd, global-read fwd, global-read bwd, then the SyncBatchNorm
        # exchanges: output block fwd, bwd, writing net fwd, bwd (capi.bn_exchange_*)
        self.epochs = torch.zeros(8, dtype=torch.int32, device=device)
        torch.cuda.synchronize(device)
        dist.barrier(group=group)                              # every rank's flags are zero before anyone signals

    def sums_view(self, K, C):
        """This rank's [K+1, C+4] sums|counts region (pm_write_reduce_fwd accumulates into it; zero it first)."""
        return self.buffer[: (K + 1) * (C + 4)].view(K + 1, C + 4)


class ShardGroup:
    """Handle for the process group the class sums are reduced over (``None`` group = WORLD)."""

    def __init__(self, group=None):
        if not dist.is_available() or not dist.is_initialized():
            raise RuntimeError("pinmem_b200.sharding: torch.distributed is not initialised")
        self.group = group
        self.world_size = dist.get_world_size(group)
        self.rank = dist.get_rank(group)
        self.peer = None          # a PeerExchange when the fused exchange is available (CUDA, NVLink peers, <= 16 ranks)
        self.peer_error = None    # why it is not (the NCCL all-reduce is used then)
        self.global_read = False  # read loss and score_query over the global batch (enable_sharded_update(global_read=True))

    def enable_peer_exchange(self, device):
        """Try to set up the fused peer-memory exchange; on any failure keep the NCCL all-reduces (and remember why).
        Collective: every rank of the group must call it."""
        import os

        ok = 0
        if self.world_size > 1 and self.world_size <= 16 and not os.environ.get("PINMEM_B200_NCCL_EXCHANGE"):
            try:
                self.peer = PeerExchange(self.group, device)
                ok = 1
            except Exception as e:  # no symmetric-memory support / no peer access: fall back, identically on all ranks
                self.peer, self.peer_error = None, repr(e)[:300]
        flag = torch.tensor([ok], device=device, dtype=torch.int32)
        dist.all_reduce(flag, op=dist.ReduceOp.MIN, group=self.group)
        if int(flag.item()) == 0:
            self.peer = None
        return self.peer is not None


def all_reduce_sum_(t, shard):
    """In-place sum all-reduce on the caller's current stream; a no-op for a single rank."""
    if shard is None or shard.world_size == 1:
        return t
    dist.all_reduce(t, op=dist.ReduceOp.SUM, group=shard.group)
    return t


class AllReduceSum(torch.autograd.Function):
    """Autograd-aware sum all-reduce: forward sums over ranks, backward sums the gradients over ranks.

    This is the exchange step as a differentiable op; ``Memory_sup`` issues the same two collectives
    around its update kernel. Exposed so host-side logic (and the gloo CPU tests) can compose it.
    """

    @staticmethod
    def forward(ctx, t, shard):
        ctx.shard = shard
        return all_reduce_sum_(t.clone(), shard)

    @staticmethod
    def backward(ctx, g):
        return all_reduce_sum_(g.contiguous().clone(), ctx.shard), None


def enable_sharded_update(module, group=None, peer_exchange=True, global_read=False):
    """Turn on the all-reduce of class sums for every ``Memory_sup`` inside ``module``.

    Call after ``init_process_group`` (and after DDP wrapping, or on the bare net) on EVERY rank (collective). Returns
    the (last) ``ShardGroup``. Without this call the module keeps the reference's rank-local update. With
    ``peer_exchange`` (default) the exchange is fused into the update kernels over NVLink peer memory when the platform
    supports it (``ShardGroup.peer``), else two NCCL all-reduces per step are issued.

    ``global_read=True`` also makes the read's two reductions over pixels global: the read loss becomes the mean over the
    valid label pixels of ALL ranks (memory.py:173-176) and score_query the softmax over all ranks' pixels
    (memory.py:183,186-187), each bit-identical across ranks; the backward sums the ranks' gradients of both (the autograd
    mirror of an all-reduce, as for the class sums). Together with the sharded update and SyncBatchNorm, every output and
    gradient of the module is then independent of the number of GPUs the global batch is split over. It costs two small
    exchanges per read (one forward, one backward), over the same peer buffers or, without them, NCCL all-gathers. All
    ranks must pass the same value (checked). ``get_score`` stays rank-local.

    Only reads made with grad mode on exchange (training steps, the meta-test read); a read under ``torch.no_grad()``
    (validation's ``net(inputs)``, ``memory_initalize``) stays rank-local and needs nothing from the other ranks. Every
    grad-mode forward of the module is then a collective: all ranks must make the same number of them, in the same order
    (a training step with the sharded update or SyncBatchNorm already is one; with global_read a grad-mode read without a
    write is one too). A rank that makes one fewer leaves its peers
    waiting: on the peer path their exchange kernel gives up after a bounded spin with a device trap (an unrecoverable CUDA
    error in those processes), on the NCCL path their all-gather waits for NCCL's own timeout.
    """
    from .memory import Memory_sup

    if not isinstance(global_read, bool):
        raise TypeError(f"enable_sharded_update: global_read must be a bool, got {type(global_read).__name__}")
    mems = [m for m in module.modules() if isinstance(m, Memory_sup)]
    if not mems:
        raise RuntimeError("enable_sharded_update: no Memory_sup inside the given module")
    shard = None
    for m in mems:   # one exchange buffer per memory module (each has its own sums and step order)
        shard = ShardGroup(group)
        _check_same_on_all_ranks(global_read, shard, m.m_items.device)
        shard.global_read = global_read
        if peer_exchange and m.m_items.is_cuda:
            shard.enable_peer_exchange(m.m_items.device)
        m.shard_group = shard
    return shard


def _check_same_on_all_ranks(flag, shard, device):
    """Raise on every rank when the ranks passed different values of a collective switch (a rank that exchanges while
    another does not would wait for a peer that never arrives)."""
    if shard.world_size == 1:
        return
    t = torch.tensor([int(flag), -int(flag)], dtype=torch.int32, device=device)
    dist.all_reduce(t, op=dist.ReduceOp.MAX, group=shard.group)
    if int(t[0]) != -int(t[1]):
        raise ValueError("enable_sharded_update: global_read must be the same on every rank")


def global_read(shard):
    """True when a read under this shard group exchanges its reductions (global_read on, more than one rank)."""
    return shard is not None and shard.global_read and shard.world_size > 1


def gather_rows(row, shard):
    """[world, n] tensor of every rank's row ``row`` [n], in rank order (one all-gather on the current stream): the
    layout the exchange kernels read when there is no peer memory."""
    out = torch.empty(shard.world_size * row.numel(), dtype=row.dtype, device=row.device)
    dist.all_gather_into_tensor(out, row.contiguous(), group=shard.group)
    return out.view(shard.world_size, row.numel())


def read_exchange_fwd(shard, col_partials, ws, temperature, out, K):
    """Forward exchange of the global read: col_partials' combined row (and, with the read-loss workspace ws and its
    out[2], the read loss and its gradient scale) become those of the global batch."""
    from . import capi

    if shard.peer is not None:
        capi.read_exchange_fwd(shard.peer, None, shard.world_size, col_partials, ws, temperature, out, K)
        return
    row = torch.empty(capi.READ_ROW_FLOATS, dtype=torch.float32, device=col_partials.device)
    capi.read_row_fwd(col_partials, ws, row, K)
    capi.read_exchange_fwd(None, gather_rows(row, shard), shard.world_size, col_partials, ws, temperature, out, K)


def read_exchange_bwd(shard, partials, g_loss, K, device):
    """Backward exchange of the global read: (sum over ranks of readloss's upstream gradient, fp32 [1]; global column sums
    of score_query's backward, fp64 [32]). ``partials`` (capi.score_bwd_partials) and ``g_loss`` may be None (zero)."""
    from . import capi

    buf = torch.empty(33, dtype=torch.float64, device=device)
    colsums, g_sum = buf[:32], buf[32:].view(torch.float32)[:1]
    if shard.peer is not None:
        capi.read_exchange_bwd(shard.peer, None, shard.world_size, partials, g_loss, g_sum, colsums, K)
        return g_sum, colsums
    row = torch.empty(capi.READ_ROW_FLOATS, dtype=torch.float32, device=device)
    capi.read_row_bwd(partials, g_loss, row, K)
    capi.read_exchange_bwd(None, gather_rows(row, shard), shard.world_size, partials, g_loss, g_sum, colsums, K)
    return g_sum, colsums


def same_group(a, b):
    """True when two process-group handles name the same group; ``None`` and ``dist.group.WORLD`` are the same group."""
    if a is b:
        return True
    world = dist.group.WORLD if dist.is_available() and dist.is_initialized() else None
    return (a is None or a is world) and (b is None or b is world)


def bn_peer(shard, group, channels):
    """The PeerExchange a SyncBatchNorm layer of ``channels`` channels that reduces over ``group`` sums through, or None for
    the NCCL all-reduces. It is the shard group's buffer when that group has one (``enable_sharded_update`` with the peer
    exchange available), the layer reduces over that same group and has at most capi.BN_MAX_C channels. Decided per call
    from the live layer, so it does not matter whether ``convert_sync_batchnorm`` ran before or after
    ``enable_sharded_update``."""
    from . import capi

    if shard is None or shard.peer is None or shard.world_size < 2 or channels > capi.BN_MAX_C:
        return None
    return shard.peer if same_group(group, shard.group) else None


def bn_stats_exchange(stats, count, M, group, peer, slot):
    """SyncBatchNorm forward: stats [2M+1] fp64, the rank's [sum | sum of squares] in [0, 2M), become the sums over the
    ranks of ``group`` with the global pixel count in stats[2M] (``count`` is the rank's). Over ``peer`` memory when given
    (slot 0: the output block, 1: the writing net), else one NCCL all-reduce. Returns stats[2M:], the device count the
    normalise pass takes."""
    from . import capi

    if peer is not None:
        capi.bn_exchange_fwd(peer, slot, stats, count, M)
    else:
        stats[2 * M:].fill_(float(count))   # (a fill kernel: capturable, unlike a scalar copy from the host)
        dist.all_reduce(stats, group=group)
    return stats[2 * M:]


def bn_grad_exchange(dgamma, dbeta, local_count, count, group, peer, slot):
    """SyncBatchNorm backward: (sg, sb), the sums of the rank's dgamma, dbeta [M] over the ranks, scaled by local_count /
    count (``count`` the device global count of bn_stats_exchange): the input-gradient passes divide by the LOCAL pixel
    count. The parameter gradients themselves stay local (DDP averages them, as for torch's own SyncBatchNorm)."""
    from . import capi

    M = dgamma.numel()
    if peer is not None:
        out = torch.empty(2 * M, dtype=torch.float32, device=dgamma.device)
        capi.bn_exchange_bwd(peer, slot, dgamma, dbeta, count, local_count, out[:M], out[M:], M)
        return out[:M], out[M:]
    sums = torch.cat([dgamma, dbeta])
    dist.all_reduce(sums, group=group)
    sums = sums * (float(local_count) / count).to(torch.float32)
    return sums[:M].contiguous(), sums[M:].contiguous()


def broadcast_memory(module, src=0, group=None):
    """Make ``m_items`` identical on all ranks (e.g. right after construction / checkpoint restore)."""
    from .memory import Memory_sup

    for m in module.modules():
        if isinstance(m, Memory_sup):
            t = m.m_items.detach().clone()
            dist.broadcast(t, src=src, group=group)
            m.m_items = t
