"""B200-native drop-in for the reference's ``network/memory.py`` (``Memory_sup``, ``Writingnet``).

Same constructor, attributes, sub-module names (``output``, ``writenet.writefeat``, ``clsfier`` -- so
``state_dict`` keys, ``SyncBatchNorm`` conversion and the meta-learning ``put_theta`` of train.py:246-277
keep working), same 5-tuple from ``forward`` and the same ``m_items`` aliasing rules as the reference
(memory.py:94-122, 167-257, 317-336); the arithmetic between the two 1x1-conv blocks runs in the
hand-written sm_100a kernels of ``csrc/`` reached through the C ABI of ``include/pinmem_b200.h``.
There is no CPU path and no torch fallback: tensors off the GPU raise.

Install under the reference's module name with ``pinthememory_b200.install()`` (see INTEGRATION.md).
"""
import os

import torch
import torch.nn as nn
import torch.nn.functional as F

from . import capi
from . import sharding

IGNORE_LABEL = 255


def initialize_weights(*models):
    """memory.py:9-19: conv kaiming-normal, BN weight 1 / bias 1e-4, Linear N(0, 1e-4) / bias 0."""
    for model in models:
        for module in model.modules():
            if isinstance(module, nn.Conv2d):
                nn.init.kaiming_normal_(module.weight, nonlinearity="relu")
            elif isinstance(module, nn.BatchNorm2d):
                module.weight.data.fill_(1.0)
                module.bias.data.fill_(1e-4)
            elif isinstance(module, nn.Linear):
                module.weight.data.normal_(0.0, 0.0001)
                module.bias.data.zero_()


def _check_labels(mask, B):
    if mask.dtype not in (torch.int64, torch.uint8):
        raise RuntimeError(f"pinmem_b200: labels must be int64 like the reference's (or uint8 class ids with 255 = ignore), "
                           f"got {mask.dtype}")
    if mask.dim() != 3 or mask.shape[0] != B:
        raise RuntimeError(f"pinmem_b200: labels must be [B,Hm,Wm] with B={B}, got {tuple(mask.shape)}")
    capi.require_cuda(mask)
    return mask.contiguous()


def _check_features(x, what):
    capi.require_cuda(x)
    if x.dim() != 4:
        raise RuntimeError(f"pinmem_b200: {what} must be [B,C,h,w], got {tuple(x.shape)}")
    capi.dtype_code(x)
    return x.contiguous()


def draw_gumbel_pair(N, K, device):
    """The two noise tensors of ``F.gumbel_softmax`` in the reference's order (memory.py:183-184):
    the dim-0 (score_query) draw first, then the dim-1 (score_memory) draw, each
    ``-empty_like(score).exponential_().log()`` on an fp32 [N,K] tensor, so the device generator stays
    aligned with the reference module."""
    probe = torch.empty(N, K, dtype=torch.float32, device=device)
    g_query = -torch.empty_like(probe, memory_format=torch.legacy_contiguous_format).exponential_().log()
    g_memory = -torch.empty_like(probe, memory_format=torch.legacy_contiguous_format).exponential_().log()
    return g_query, g_memory


_SIDE_STREAMS = {}  # device -> stream of the write branch (module-level: modules stay deep-copyable)
_AUX_STREAMS = {}   # device -> second side stream (the column softmax of a branched read)


def _stream_of(table, device):
    st = table.get(device)
    if st is None:
        st = table[device] = torch.cuda.Stream(device=device)
    return st


class _ReadFn(torch.autograd.Function):
    """x, M (, labels, noise) -> u = [q ; p.M], score_query, score_memory, readloss, label histogram.

    ``planes=True``: u = [q ; score_memory as 32 channel planes] for a caller that folds the memory into the
    1x1 convolution that follows (include/pinmem_b200.h, pm_read_fwd_planes); the returned dM then only holds
    the similarity term, the other one reaches M through the folded weight in autograd.
    """

    last_bad = None   # device int64 scalar: label values outside [0,K) u {255} seen by the last read with labels
    last_lab8 = None  # the packed uint8 class map that read produced (None when the first-generation kernel ran)

    @staticmethod
    def forward(ctx, x, M, labels, g_query, g_memory, temperature, K, planes=False, tee=False, branch=False, xg=None):
        """``tee=True`` appends x itself to the outputs: a caller that feeds the same features to a second branch (the
        writing net) hands that branch the tee, so its gradient arrives HERE as an input of backward() and the dx kernel
        sums it in (``dx_add``) -- instead of autograd adding two feature-sized gradients with an element-wise kernel.

        ``xg``: the shard group of a global read (sharding.enable_sharded_update(global_read=True), more than one rank) or
        None. The read loss then runs before the column softmax, and one exchange between them turns the rank's column
        statistics and read-loss sum / valid count into the global batch's (sharding.read_exchange_fwd)."""
        B, C, h, w = x.shape
        N = B * h * w
        dev = x.device
        KP = capi.score_stride(K)
        UC = C + capi.PLANES if planes else 2 * C
        u = torch.empty(B, UC, h, w, dtype=x.dtype, device=dev)
        # deterministic mode: torch may fill `empty` with NaN; the read-loss kernels read whole padded rows of s, so its
        # padding columns must be finite -- zero them rather than depend on what the allocation held
        s = (torch.zeros if capi.deterministic() else torch.empty)(N, KP, dtype=torch.float32, device=dev)
        score_m = torch.empty(N, K, dtype=torch.float32, device=dev)
        score_q = torch.empty(N, K, dtype=torch.float32, device=dev)
        M = M.contiguous()
        # one zeroed allocation: [ds_rl (N*KP floats, with labels) | workspace (40 x 8 bytes) | out (4 floats) | column
        # partials (their ticket row must be zero)]
        n_rl = N * KP if labels is not None else 0
        n_cp = capi.colsoftmax_workspace_floats(K)
        buf = torch.zeros(n_rl + 2 * capi.WS_WORDS + 4 + n_cp, dtype=torch.float32, device=dev)
        col_partials = buf[n_rl + 2 * capi.WS_WORDS + 4:]
        # ``branch`` (the module's two-stream mode): the label pass needs nothing from the read and nothing on the step's
        # critical path needs the column softmax, so the pack runs on the write branch's stream UNDER read_fwd (which also
        # orders it before the write kernels that consume the packed map) and the column softmax on a second side stream
        # under the read loss: two small kernels (17 + 11 us at cfg 2) leave the main chain. Captured, they are parallel
        # branches of the graph.
        use_pack = labels is not None and K <= 19
        branch = bool(branch) and x.is_cuda
        lab8 = None
        if branch:
            cur = torch.cuda.current_stream(dev)
            side, aux = _stream_of(_SIDE_STREAMS, dev), _stream_of(_AUX_STREAMS, dev)
        if branch and use_pack:
            ws = buf[N * KP: N * KP + 2 * capi.WS_WORDS]
            side.wait_stream(cur)                      # (after the zero fill of the workspace)
            with torch.cuda.stream(side):
                lab8 = capi.labels_pack(labels, K, ws)
            buf.record_stream(side)
            labels.record_stream(side)
            lab8.record_stream(cur)
        capi.read_fwd(x, M, g_memory, u, s, score_m, K, gumbel_q=g_query, col_partials=col_partials, planes=planes)

        def column_softmax():
            if xg is not None:
                rl_ws = buf[N * KP: N * KP + 2 * capi.WS_WORDS] if labels is not None else None
                rl_res = buf[N * KP + 2 * capi.WS_WORDS: N * KP + 2 * capi.WS_WORDS + 4] if labels is not None else None
                sharding.read_exchange_fwd(xg, col_partials, rl_ws, temperature, rl_res, K)
            capi.colsoftmax_apply(s, g_query, col_partials, score_q, N, K)

        def column_softmax_on_stream():
            if branch:
                aux.wait_stream(cur)
                with torch.cuda.stream(aux):
                    column_softmax()
                for t in (s, g_query, buf, score_q):
                    if torch.is_tensor(t):
                        t.record_stream(aux)
            else:
                column_softmax()

        if xg is None:
            column_softmax_on_stream()
        if labels is not None:
            ds_rl = buf[: N * KP]
            ws = buf[N * KP: N * KP + 2 * capi.WS_WORDS]
            rl_out = buf[N * KP + 2 * capi.WS_WORDS: N * KP + 2 * capi.WS_WORDS + 4]
            if lab8 is not None:
                cur.wait_stream(side)                  # the packed map and its histogram
                capi.readloss_fwd8(s, lab8, temperature, B, h, w, K, ds_rl, ws, rl_out)
                _ReadFn.last_lab8 = lab8
            elif use_pack and x.is_cuda:
                # one pass over the labels (packed uint8 classes + histogram + bad-label count), then the read loss on it
                lab8 = capi.labels_pack(labels, K, ws)
                capi.readloss_fwd8(s, lab8, temperature, B, h, w, K, ds_rl, ws, rl_out)
                _ReadFn.last_lab8 = lab8
            else:
                _ReadFn.last_lab8 = capi.readloss(s, labels, temperature, B, h, w, K, ds_rl, ws, rl_out)
            readloss = rl_out[0]
            hist = ws.view(torch.int64)[capi.WS_HIST: capi.WS_HIST + K + 1]
            _ReadFn.last_bad = ws.view(torch.int64)[capi.WS_BAD]
        else:
            ds_rl = rl_out = None
            readloss = torch.zeros((), dtype=torch.float32, device=dev)
            hist = torch.zeros(K + 1, dtype=torch.int64, device=dev)
        if xg is not None:   # after the read loss: the exchange carries its sum and valid count too
            column_softmax_on_stream()
        ctx.K, ctx.planes, ctx.UC, ctx.xg = K, planes, UC, xg
        ctx.has_loss = labels is not None
        ctx.set_materialize_grads(False)  # unused outputs (scores, histogram) arrive as None, not as zero fills
        # score_q is kept for the gradient of score_query (N*K*4 bytes, 5.6 MB at cfg 2: the one cost of differentiable
        # scores on a step that does not use them)
        ctx.save_for_backward(x, M, score_m, ds_rl, rl_out, score_q)
        ctx.mark_non_differentiable(hist)
        if branch:
            cur.wait_stream(aux)                       # join: score_query is ready for whoever reads it on this stream
        outs = (u, score_q.view(B, h, w, K), score_m.view(B, h, w, K), readloss, hist)
        return outs + (x,) if tee else outs

    @staticmethod
    def backward(ctx, du, g_sq, g_sm, g_loss, _g_hist, g_tee=None):
        x, M, score_m, ds_rl, rl_out, score_q = ctx.saved_tensors
        B, C, h, w = x.shape
        K = ctx.K
        N = B * h * w
        need_dM = ctx.needs_input_grad[1]
        if du is None:
            du = torch.zeros(B, ctx.UC, h, w, dtype=x.dtype, device=x.device)
        du = du.to(x.dtype).contiguous()
        if ctx.has_loss and g_loss is not None:
            g_loss = g_loss.to(torch.float32).contiguous()
        else:
            g_loss = None
        dense = lambda g: None if g is None else g.reshape(N, K).to(torch.float32).contiguous()
        colsums = None
        if ctx.xg is not None and (ctx.has_loss or g_sq is not None):
            # global read: the ranks' upstream gradients of readloss and the column sums of score_query's backward are
            # summed over the ranks (the autograd mirror of the forward's exchange)
            g_sq = dense(g_sq)
            partials = capi.score_bwd_partials(score_q, g_sq, K) if g_sq is not None else None
            g_sum, colsums = sharding.read_exchange_bwd(ctx.xg, partials, None if g_loss is None else g_loss.reshape(1), K,
                                                        x.device)
            if ctx.has_loss:
                g_loss = g_sum
        if g_loss is None:
            ds_rl = rl_out = None
        if g_sq is not None or g_sm is not None:
            # gradients of score_query / score_memory: their softmax backward (plus the scaled read-loss term) forms one
            # additive similarity gradient E, which the read backward takes in place of ds_rl with a unit scale
            E = torch.empty(N, capi.score_stride(K), dtype=torch.float32, device=x.device)
            if colsums is not None and g_sq is not None:
                capi.score_bwd_global(score_q, g_sq, score_m if g_sm is not None else None, dense(g_sm), E, K, colsums,
                                      ds_rl=ds_rl, g_loss=g_loss, rl_out=rl_out)
            else:
                capi.score_bwd(score_q if g_sq is not None else None, dense(g_sq), score_m if g_sm is not None else None,
                               dense(g_sm), E, K, ds_rl=ds_rl, g_loss=g_loss, rl_out=rl_out)
            ds_rl = E
            g_loss = rl_out = torch.ones(2, dtype=torch.float32, device=x.device)
        dx = torch.empty_like(x)
        ds = torch.empty(N, capi.score_stride(K), dtype=torch.float32, device=x.device)
        fused_add = g_tee is not None and ctx.planes and g_tee.dtype == x.dtype and g_tee.shape == x.shape
        capi.read_bwd(du, x, M, score_m, ds_rl, g_loss, rl_out, dx, ds, K, planes=ctx.planes,
                      dx_add=g_tee.contiguous() if fused_add else None)
        if g_tee is not None and not fused_add:
            dx = dx + g_tee.to(dx.dtype)
        dM = None
        if need_dM:
            dM = torch.zeros_like(M)
            capi.read_bwd_dM(None if ctx.planes else du, x, score_m, ds, dM, K)
        return dx, dM, None, None, None, None, None, None, None, None, None


class _FoldWeightFn(torch.autograd.Function):
    """W [Co,2C,1,1], M [K,C] -> W' = [W1 | W2.M^T | 0] [Co, C+32, 1, 1] (pm_fold_weight_fwd / _bwd)."""

    @staticmethod
    def forward(ctx, W, M):
        Co, C2 = W.shape[0], W.shape[1]
        C, K = C2 // 2, M.shape[0]
        W32 = W.detach().to(torch.float32).contiguous()
        M32 = M.detach().to(torch.float32).contiguous()
        Wp = torch.empty(Co, C + capi.PLANES, 1, 1, dtype=torch.float32, device=W.device)
        capi.fold_weight_fwd(W32, M32, Wp, Co, C, K)
        ctx.save_for_backward(W32, M32)
        ctx.wdtype = W.dtype
        return Wp.to(W.dtype)

    @staticmethod
    def backward(ctx, dWp):
        W32, M32 = ctx.saved_tensors
        Co, C, K = W32.shape[0], M32.shape[1], M32.shape[0]
        dWp = dWp.to(torch.float32).contiguous()
        dW = dM = None
        if ctx.needs_input_grad[0]:
            dW = torch.empty_like(W32)
            capi.fold_weight_bwd(dWp, M32, dW, Co, C, K)
            dW = dW.to(ctx.wdtype)
        if ctx.needs_input_grad[1]:  # meta-test read: the p (x) dc term of dM
            dM = dWp[:, C:C + K, 0, 0].t() @ W32[:, C:, 0, 0]
        return dW, dM


class _WriteFn(torch.autograd.Function):
    """f, labels, M_old, classifier -> new memory, divergence loss, classification loss.

    With a shard group the packed class sums|counts are all-reduced before the update and the gradient
    w.r.t. the sums is all-reduced in the backward (SURVEY.md 8e), so every rank computes the update of
    the concatenated global batch.
    """

    @staticmethod
    def forward(ctx, f, labels, M_old, W, b, momentum, K, group):
        C = f.shape[1]
        M_new, losses, saved, W, b, SD = _write_update_fwd(lambda sd: capi.write_reduce_fwd(f, labels, sd, K), M_old, W, b,
                                                           momentum, C, K, group, f.device)
        ctx.K, ctx.momentum, ctx.group = K, momentum, group
        ctx.set_materialize_grads(False)
        ctx.save_for_backward(f, labels, M_new, saved, W, b)
        ctx.mark_non_differentiable(SD)
        return M_new, losses[0], losses[1], SD

    @staticmethod
    def backward(ctx, dM_new, g_div, g_cls, _g_sd):
        f, labels, M_new, saved, W, b = ctx.saved_tensors
        K = ctx.K
        dS, dW, db = _write_update_bwd(ctx, dM_new, g_div, g_cls, M_new, saved, W, b, f.shape[1], K)
        df = None
        if ctx.needs_input_grad[0]:
            df = torch.empty_like(f)
            capi.write_bwd(dS, f, labels, df, K)
        return df, None, None, dW, db, None, None, None


def _write_update_fwd(reduce, M_old, W, b, momentum, C, K, group, dev):
    """reduce(sums) adds the class sums|counts into `sums`; then the update (plain, all-reduced or over peer memory).
    Returns (M_new, losses, saved, W fp32, b fp32, SD)."""
    peer = group.peer if (group is not None and group.world_size > 1) else None
    # one zeroed allocation: the class sums|counts [K+1, C+4] and the update kernel's scratch
    nsd = (K + 1) * (C + 4)
    zbuf = torch.zeros(nsd + capi.update_aux_floats(K), dtype=torch.float32, device=dev)
    SD, aux = zbuf[:nsd].view(K + 1, C + 4), zbuf[nsd:]
    M_old = M_old.detach().contiguous()
    W = W.detach().to(torch.float32).contiguous()
    b = b.detach().to(torch.float32).contiguous()
    M_new = torch.empty(K, C, dtype=torch.float32, device=dev)
    losses = torch.empty(2, dtype=torch.float32, device=dev)
    saved = torch.empty(2 * K, dtype=torch.float32, device=dev)
    if peer is not None:
        # the rank's sums go into its peer-mapped buffer; the update kernel itself gathers and sums all ranks' rows
        # over NVLink (and leaves the all-reduced sums in SD for the host side)
        mine = peer.sums_view(K, C)
        mine.zero_()
        reduce(mine)
        capi.update_fwd_peer(peer, SD, M_old, momentum, W, b, M_new, losses, saved, C, K, aux=aux)
    else:
        reduce(SD)
        if group is not None:
            sharding.all_reduce_sum_(SD, group)
        capi.update_fwd(SD, M_old, momentum, W, b, M_new, losses, saved, C, K, aux=aux)
    return M_new, losses, saved, W, b, SD


def _write_update_bwd(ctx, dM_new, g_div, g_cls, M_new, saved, W, b, C, K):
    """(dS, dW, db) of the update; ctx carries momentum and group."""
    dev = M_new.device
    as32 = lambda t: None if t is None else t.to(torch.float32).contiguous()
    dS = torch.empty(K, C, dtype=torch.float32, device=dev)
    dW = torch.empty(K, C, dtype=torch.float32, device=dev)
    db = torch.empty(K, dtype=torch.float32, device=dev)
    peer = ctx.group.peer if (ctx.group is not None and ctx.group.world_size > 1) else None
    if peer is not None:
        capi.update_bwd_peer(peer, as32(dM_new), as32(g_div), as32(g_cls), M_new, saved, W, b, ctx.momentum, dS, dW, db, C, K)
    else:
        capi.update_bwd(as32(dM_new), as32(g_div), as32(g_cls), M_new, saved, W, b, ctx.momentum, dS, dW, db, C, K)
        if ctx.group is not None:
            sharding.all_reduce_sum_(dS, ctx.group)
    return dS, dW, db


class _WriteNetFn(torch.autograd.Function):
    """Writingnet then _WriteFn in one Function (fp32): z = conv1x1(x, Wc) with the batch statistics in the GEMM epilogue, then
    the class sums of f = relu(x + BatchNorm(z)) with f formed inside the class-sum kernel (pm_write_reduce_bn_fwd), then the
    update. f and its ReLU mask are never stored; the backward forms f again from (z, x) inside the write backward, which
    also leaves g = df * [f > 0] and the BatchNorm sums (pm_write_bwd_bn), so the BatchNorm backward is one pass
    (pm_bn_bwd_apply on (g, z)) and the input-gradient GEMM accumulates into g. Saves x and z."""

    @staticmethod
    def forward(ctx, x, labels, M_old, Wc, gamma, beta, running_mean, running_var, factor, eps, num_batches_tracked, sync_group,
                W, b, momentum, K, group):
        B, C, h, w = x.shape
        dev = x.device
        W2 = Wc.detach().reshape(C, C).to(torch.float32).contiguous()
        g32 = gamma.detach().to(torch.float32).contiguous()
        b32 = beta.detach().to(torch.float32).contiguous()
        # [sum | sum of squares | element count], cleared by the launch that also splits W and W^T for the two GEMMs
        stats = torch.empty(2 * C + 1, dtype=torch.float64, device=dev)
        ctx.tf32 = capi.tf32()   # decided once: the backward's operand W^T is prepared here, in the same mode
        (hi, lo), ctx.preT = capi.conv1x1_prep_both(W2, torch.float32, zero=stats, tf32=ctx.tf32)
        z = capi.conv1x1_fwd(x, hi, lo, C, stats=stats)
        count = None
        ctx.bn_peer = None
        if sync_group is not None:   # as _ConvBnActFn: global statistics (slot 1 of the shard group's peer buffer)
            ctx.bn_peer = sharding.bn_peer(group, sync_group, C)
            count = sharding.bn_stats_exchange(stats, B * h * w, C, sync_group, ctx.bn_peer, 1)
        mean = torch.empty(C, dtype=torch.float32, device=dev)
        invstd = torch.empty(C, dtype=torch.float32, device=dev)
        M_new, losses, saved, W, b, SD = _write_update_fwd(
            lambda sd: capi.write_reduce_bn_fwd(z, x, labels, sd, K, stats, B * h * w, eps, g32, b32, mean, invstd,
                                                running_mean, running_var, factor, count_dev=count,
                                                num_batches_tracked=num_batches_tracked),
            M_old, W, b, momentum, C, K, group, dev)
        if GATE_LOG is not None:   # debug only: the gate the kernels applied, formed with the same expression
            y = torch.empty_like(z)
            capi.bn_apply(z, mean, invstd, g32, b32, x, y, True)
            GATE_LOG.setdefault("writenet", []).append(y > 0)
        ctx.K, ctx.momentum, ctx.group, ctx.sync_group = K, momentum, group, sync_group
        ctx.wshape, ctx.wdtype = Wc.shape, Wc.dtype
        ctx.set_materialize_grads(False)
        ctx.save_for_backward(x, z, labels, M_new, saved, W, b, mean, invstd, g32, b32, count)
        ctx.mark_non_differentiable(SD)
        return M_new, losses[0], losses[1], SD

    @staticmethod
    def backward(ctx, dM_new, g_div, g_cls, _g_sd):
        x, z, labels, M_new, saved, W, b, mean, invstd, g32, b32, count = ctx.saved_tensors
        K = ctx.K
        B, C, h, w = x.shape
        dev = x.device
        dS, dW, db = _write_update_bwd(ctx, dM_new, g_div, g_cls, M_new, saved, W, b, C, K)
        dx = dWc = dgamma = dbeta = None
        if any(ctx.needs_input_grad[i] for i in (0, 3, 4, 5)):
            g = torch.empty_like(z)
            dgamma = torch.empty(C, dtype=torch.float32, device=dev)
            dbeta = torch.empty(C, dtype=torch.float32, device=dev)
            capi.write_bwd_bn(dS, z, x, labels, mean, invstd, g32, b32, g, dgamma, dbeta, K)
            sg, sb = dgamma, dbeta
            if ctx.sync_group is not None:   # as _ConvBnActFn.backward: input gradient from the sums over all ranks
                sg, sb = sharding.bn_grad_exchange(dgamma, dbeta, B * h * w, count, ctx.sync_group, ctx.bn_peer, 1)
            dz = torch.empty_like(z)
            capi.bn_bwd_apply(g, None, None, z, mean, invstd, g32, sg, sb, False, True, dz, None)
            if ctx.needs_input_grad[0]:
                # dx = g + W^T . dz; before the weight gradient, so that a consumer of dx (the read's backward) is not
                # queued behind it
                hiT, loT = ctx.preT
                dx = capi.conv1x1_fwd(dz, hiT, loT, C, y=g, accumulate=True)
            if ctx.needs_input_grad[3]:
                dWc = capi.conv1x1_wgrad(dz, x, tf32=ctx.tf32).view(ctx.wshape).to(ctx.wdtype)
        return (dx, None, None, dWc, dgamma, dbeta, None, None, None, None, None, None, dW, db, None, None, None)


class _MemoryLossFn(torch.autograd.Function):
    """(div, cls) of an arbitrary memory: memory.py:264-272 and :259-262 (pm_memory_losses_fwd / _bwd).
    W/b None -> divergence loss only (cls is returned as 0)."""

    @staticmethod
    def forward(ctx, mem, W, b):
        K, C = mem.shape
        dev = mem.device
        m32 = mem.detach().to(torch.float32).contiguous()
        W32 = None if W is None else W.detach().to(torch.float32).contiguous()
        b32 = None if b is None else b.detach().to(torch.float32).contiguous()
        out = torch.empty(2, dtype=torch.float32, device=dev)
        gram = torch.empty(K * K, dtype=torch.float32, device=dev)
        prob = torch.empty(K * K, dtype=torch.float32, device=dev) if W is not None else None
        capi.memory_losses_fwd(m32, W32, b32, out, gram, prob)
        ctx.has_cls = W is not None
        ctx.save_for_backward(m32, W32, gram, prob)
        return out[0], out[1]

    @staticmethod
    def backward(ctx, g_div, g_cls):
        m32, W32, gram, prob = ctx.saved_tensors
        as32 = lambda t: None if t is None else t.to(torch.float32).contiguous()
        dmem = torch.empty_like(m32)
        dW = torch.empty_like(W32) if ctx.has_cls else None
        db = torch.empty(m32.shape[0], dtype=torch.float32, device=m32.device) if ctx.has_cls else None
        capi.memory_losses_bwd(m32, W32, gram, prob, as32(g_div), as32(g_cls), dmem, dW, db)
        return dmem, dW, db


class _BnActFn(torch.autograd.Function):
    """y = [relu](BatchNorm2d(xc) [+ residual]) with batch (training) or given (eval) statistics."""

    @staticmethod
    def forward(ctx, xc, gamma, beta, residual, running_mean, running_var, use_batch_stats, factor, eps, relu):
        C = xc.shape[1]
        dev = xc.device
        g32 = gamma.detach().to(torch.float32).contiguous()
        b32 = beta.detach().to(torch.float32).contiguous()
        if use_batch_stats:
            mean = torch.empty(C, dtype=torch.float32, device=dev)
            invstd = torch.empty(C, dtype=torch.float32, device=dev)
            capi.bn_stats(xc, eps, mean, invstd, running_mean, running_var, factor)
        else:
            mean = running_mean.to(torch.float32).contiguous()
            invstd = (running_var.to(torch.float32) + eps).rsqrt_()
        y = torch.empty_like(xc)
        # packed ReLU mask (1 bit per element) for the backward, so that it does not have to re-read y
        nwords = capi.bn_mask_words(xc.shape[0], C, xc.shape[2] * xc.shape[3]) if relu else 0
        vec_ok = nwords > 0 and all(t is None or t.data_ptr() % 16 == 0 for t in (xc, y, residual))
        mask = torch.empty(nwords, dtype=torch.int32, device=dev) if vec_ok else None
        capi.bn_apply(xc, mean, invstd, g32, b32, residual, y, relu, relu_mask=mask)
        ctx.relu, ctx.training, ctx.has_res = relu, use_batch_stats, residual is not None
        ctx.use_mask = mask is not None
        ctx.save_for_backward(xc, mask if mask is not None else y, mean, invstd, g32)
        return y

    @staticmethod
    def backward(ctx, dy):
        xc, y_or_mask, mean, invstd, g32 = ctx.saved_tensors
        y, mask = (None, y_or_mask) if ctx.use_mask else (y_or_mask, None)
        C = xc.shape[1]
        dy = dy.to(xc.dtype).contiguous()
        dgamma = torch.empty(C, dtype=torch.float32, device=xc.device)
        dbeta = torch.empty(C, dtype=torch.float32, device=xc.device)
        dx = torch.empty_like(xc)
        dres = torch.empty_like(xc) if (ctx.has_res and ctx.needs_input_grad[3]) else None
        if mask is not None and any(t is not None and t.data_ptr() % 16 for t in (dy, dx, dres)):
            raise RuntimeError("pinmem_b200: misaligned gradient buffer on the packed-mask BatchNorm path")
        capi.bn_bwd_reduce(dy, y, mask, xc, mean, invstd, ctx.relu, dgamma, dbeta)
        capi.bn_bwd_apply(dy, y, mask, xc, mean, invstd, g32, dgamma, dbeta, ctx.relu, ctx.training, dx, dres)
        return dx, dgamma, dbeta, dres, None, None, None, None, None, None


class _ConvBnActFn(torch.autograd.Function):
    """y = [relu](BatchNorm2d(conv1x1(x, W)) [+ residual]) -- memory.py:74-87 (Writingnet) and :103-107 (self.output).

    The convolution, its input gradient and its weight gradient are the tcgen05 GEMMs of csrc/pm_gemm.cu (3xTF32 in
    fp32 -- one TF32 pass when torch's TF32 switches allow it (capi.tf32), decided once in the forward --, bf16
    otherwise); the forward GEMM's epilogue produces the batch statistics, so the BatchNorm costs one
    normalise pass instead of a statistics pass + a normalise pass; when the residual IS the convolution input
    (Writingnet) the input-gradient GEMM accumulates into the residual gradient (TMA reduce-add) instead of leaving an
    element-wise add to autograd."""

    @staticmethod
    def forward(ctx, x, W, gamma, beta, residual, running_mean, running_var, use_batch_stats, factor, eps, relu,
                res_is_x, sync_group=None, num_batches_tracked=None, pre=None, shard=None, slot=0):
        B, K, h, w = x.shape
        M = W.shape[0]
        dev = x.device
        W2 = W.detach().reshape(M, K).to(torch.float32).contiguous()
        g32 = gamma.detach().to(torch.float32).contiguous()
        b32 = beta.detach().to(torch.float32).contiguous()
        ctx.preT = None
        ctx.bn_peer, ctx.slot = None, slot
        stats = None
        tf32 = x.dtype == torch.float32 and capi.tf32()
        if pre is not None and (pre[0][0].dtype != x.dtype or capi.operands_tf32(pre[0]) != tf32):
            pre = None                # prepared for another compute dtype (autocast) or TF32 mode: redo it here
        ctx.w_on_aux = pre is not None
        if pre is not None:           # operands (and the cleared statistics buffer) prepared ahead of time on a side stream
            (hi, lo), ctx.preT, stats = pre
            if not use_batch_stats:
                stats = None
        elif ctx.needs_input_grad[0]:   # the input-gradient GEMM's operand W^T comes out of the same launch ...
            if use_batch_stats:       # ... which also clears the statistics buffer (no fill kernel)
                stats = torch.empty(2 * M + 1, dtype=torch.float64, device=dev)
            (hi, lo), ctx.preT = capi.conv1x1_prep_both(W2, x.dtype, zero=stats, tf32=tf32)
        else:
            hi, lo = capi.conv1x1_prep(W2, False, x.dtype, tf32=tf32)
        if use_batch_stats:
            # [sum | sum of squares | element count]: the GEMM epilogue fills the first 2M; with SyncBatchNorm the whole
            # vector is summed over the ranks (fp64; over the shard group's peer memory when the layer reduces over that
            # group, else one small all-reduce) and the normalise pass finalises GLOBAL statistics
            if stats is None:
                stats = torch.zeros(2 * M + 1, dtype=torch.float64, device=dev)
            xc = capi.conv1x1_fwd(x, hi, lo, M, stats=stats)
            count = None
            if sync_group is not None:
                ctx.bn_peer = sharding.bn_peer(shard, sync_group, M)
                count = sharding.bn_stats_exchange(stats, B * h * w, M, sync_group, ctx.bn_peer, slot)
            mean = torch.empty(M, dtype=torch.float32, device=dev)
            invstd = torch.empty(M, dtype=torch.float32, device=dev)
        else:
            xc = capi.conv1x1_fwd(x, hi, lo, M)
            mean = running_mean.to(torch.float32).contiguous()
            invstd = (running_var.to(torch.float32) + eps).rsqrt_()
        res = x if res_is_x else residual
        y = torch.empty_like(xc)
        nwords = capi.bn_mask_words(B, M, h * w) if relu else 0
        vec_ok = nwords > 0 and all(t is None or t.data_ptr() % 16 == 0 for t in (xc, y, res))
        mask = torch.empty(nwords, dtype=torch.int32, device=dev) if vec_ok else None
        if use_batch_stats:  # mean / invstd / running statistics are finalised inside the normalise pass
            capi.bn_apply_stats(xc, stats, B * h * w, eps, g32, b32, res, y, relu, mean, invstd, running_mean, running_var,
                                factor, relu_mask=mask, count_dev=count, num_batches_tracked=num_batches_tracked)
        else:
            if num_batches_tracked is not None:
                num_batches_tracked.add_(1)
            capi.bn_apply(xc, mean, invstd, g32, b32, res, y, relu, relu_mask=mask)
        ctx.relu, ctx.training, ctx.res_is_x, ctx.has_res = relu, use_batch_stats, res_is_x, res is not None
        ctx.use_mask = mask is not None
        ctx.wshape, ctx.wdtype = W.shape, W.dtype
        ctx.tf32 = tf32
        ctx.sync_group = sync_group if use_batch_stats else None
        ctx.beta32 = b32   # (a detached fp32 copy: only the fused BatchNorm-backward GEMM reads it, to recompute the ReLU gate)
        ctx.save_for_backward(x, W2, xc, mask if mask is not None else y, mean, invstd, g32,
                              count if (use_batch_stats and sync_group is not None) else None)
        return y

    @staticmethod
    def backward(ctx, dy):
        x, W2, xc, y_or_mask, mean, invstd, g32, count = ctx.saved_tensors
        y, mask = (None, y_or_mask) if ctx.use_mask else (y_or_mask, None)
        M, K = W2.shape
        dy = dy.to(xc.dtype).contiguous()
        dgamma = torch.empty(M, dtype=torch.float32, device=xc.device)
        dbeta = torch.empty(M, dtype=torch.float32, device=xc.device)
        dxc = torch.empty_like(xc)
        need_x = ctx.needs_input_grad[0]
        need_res = ctx.has_res and (need_x if ctx.res_is_x else ctx.needs_input_grad[4])
        dres = torch.empty_like(xc) if need_res else None
        if mask is not None and any(t is not None and t.data_ptr() % 16 for t in (dy, dxc, dres)):
            raise RuntimeError("pinmem_b200: misaligned gradient buffer on the packed-mask BatchNorm path")
        capi.bn_bwd_reduce(dy, y, mask, xc, mean, invstd, ctx.relu, dgamma, dbeta)
        sg, sb = dgamma, dbeta
        if ctx.sync_group is not None:
            # SyncBatchNorm: the input gradient needs the sums over ALL ranks' pixels (the parameter gradients stay
            # local, DDP averages them -- torch's own SyncBatchNorm does the same); the kernel divides by the LOCAL pixel
            # count, so the global sums come pre-scaled by local / global
            sg, sb = sharding.bn_grad_exchange(dgamma, dbeta, xc.shape[0] * xc.shape[2] * xc.shape[3], count, ctx.sync_group,
                                               ctx.bn_peer, ctx.slot)
        if need_x and not ctx.has_res and xc.dtype == torch.float32 and M % 32 == 0 and ctx.beta32 is not None:
            # blocks without a residual (self.output): the BatchNorm backward rides in the operand path of the
            # input-gradient GEMM, which also stores dz for the weight-gradient GEMM -- no bn_bwd_apply pass
            hiT, loT = ctx.preT if ctx.preT is not None else capi.conv1x1_prep(W2, True, x.dtype, tf32=ctx.tf32)
            dx, dxc = capi.conv1x1_dgrad_bnbwd(dy, xc, hiT, loT, K, mean, invstd, g32, sg, sb, ctx.beta32, ctx.relu,
                                               ctx.training)
            dW = None
            if ctx.needs_input_grad[1]:
                if getattr(ctx, "w_on_aux", False):
                    # two-stream mode: the weight came from the second side stream (folded there, so its backward runs there):
                    # the weight-gradient GEMM goes to that stream too -- the read's backward, next on this stream, only
                    # needs dx
                    cur = torch.cuda.current_stream(x.device)
                    aux = _stream_of(_AUX_STREAMS, x.device)
                    aux.wait_stream(cur)
                    with torch.cuda.stream(aux):
                        dW = capi.conv1x1_wgrad(dxc, x, tf32=ctx.tf32).view(ctx.wshape).to(ctx.wdtype)
                    dxc.record_stream(aux)
                    x.record_stream(aux)
                else:
                    dW = capi.conv1x1_wgrad(dxc, x, tf32=ctx.tf32).view(ctx.wshape).to(ctx.wdtype)
            return dx, dW, dgamma, dbeta, None, None, None, None, None, None, None, None, None, None, None, None, None
        capi.bn_bwd_apply(dy, y, mask, xc, mean, invstd, g32, sg, sb, ctx.relu, ctx.training, dxc, dres)
        dW = None
        if ctx.needs_input_grad[1]:
            dW = capi.conv1x1_wgrad(dxc, x, tf32=ctx.tf32).view(ctx.wshape).to(ctx.wdtype)
        dx = None
        if need_x:
            hiT, loT = ctx.preT if ctx.preT is not None else capi.conv1x1_prep(W2, True, x.dtype, tf32=ctx.tf32)
            if ctx.res_is_x:
                dx = capi.conv1x1_fwd(dxc, hiT, loT, K, y=dres, accumulate=True)   # dres += W^T . dxc
                dres = None
            else:
                dx = capi.conv1x1_fwd(dxc, hiT, loT, K)
        return (dx, dW, dgamma, dbeta, (None if ctx.res_is_x else dres), None, None, None, None, None, None, None, None, None, None,
                None, None)


def _plain(m):
    return not (m._forward_hooks or m._forward_pre_hooks or m._backward_hooks)


def _foldable(conv, C):
    """The 1x1, bias-free, ungrouped 2C -> * convolution of the reference (memory.py:104)."""
    return _pointwise(conv) and conv.in_channels == 2 * C


def _pointwise(conv):
    return (type(conv) is nn.Conv2d and conv.kernel_size == (1, 1) and conv.stride == (1, 1) and conv.padding == (0, 0)
            and conv.dilation == (1, 1) and conv.groups == 1 and conv.bias is None and conv.padding_mode == "zeros")


# Debug hook for parity tests: a dict name -> list; when set, every ReLU of the two conv blocks appends its gate
# (output > 0) under "output" / "writenet" in call order, so a checker can replay the decisions at rounding-level ties
# (oracle/memory_oracle.py::ReluGates). None (the default) costs nothing.
GATE_LOG = None

_warned = set()


def _warn_once(key, msg):
    if key not in _warned:
        _warned.add(key)
        import warnings

        warnings.warn("pinmem_b200: " + msg, RuntimeWarning, stacklevel=3)


def _bn_args(bn, defer_counter=False):
    """(use_batch_stats, running_mean, running_var, momentum factor) of one nn.BatchNorm2d call, with the module's
    own side effect (num_batches_tracked += 1) applied -- or, with ``defer_counter``, left to the normalise kernel: then a
    fifth element is returned, the counter tensor that launch must bump (None when there is nothing to bump)."""
    nbt = None
    use_batch = bn.training or bn.running_mean is None
    factor = 0.0
    rm = rv = None
    if bn.training and bn.track_running_stats and bn.running_mean is not None:
        rm, rv = bn.running_mean, bn.running_var
        if bn.num_batches_tracked is not None:
            t = bn.num_batches_tracked
            if (defer_counter and bn.momentum is not None and t.dtype == torch.int64 and t.is_cuda and t.is_contiguous()
                    and rm.dtype == torch.float32 and rv.dtype == torch.float32):
                nbt = t
            else:
                t.add_(1)
        factor = bn.momentum if bn.momentum is not None else 1.0 / float(bn.num_batches_tracked)
        if rm.dtype != torch.float32 or rv.dtype != torch.float32:
            rm = rv = None  # keep exotic buffer dtypes out of the kernel (statistics are still exact)
    elif not use_batch:
        rm, rv = bn.running_mean, bn.running_var
    if defer_counter:
        return use_batch, rm, rv, float(factor), nbt
    return use_batch, rm, rv, float(factor)


def _bn_fast(bn, xc):
    return (type(bn) in (nn.BatchNorm2d, nn.SyncBatchNorm) and bn.affine and _plain(bn) and xc.is_cuda and xc.dim() == 4
            and xc.dtype in (torch.float32, torch.bfloat16) and bn.weight.is_cuda)


def _sync_group(bn):
    """The process group whose ranks share this layer's batch statistics: ``nn.SyncBatchNorm`` in training mode with
    more than one rank (what ``convert_sync_batchnorm`` makes of the module's two BatchNorm2d under ``--syncbn``,
    train.py:95). Returns None when the layer behaves like a plain BatchNorm2d (eval mode, one rank, not initialised)."""
    if type(bn) is not nn.SyncBatchNorm or not (bn.training or bn.running_mean is None):
        return None
    import torch.distributed as dist

    if not (dist.is_available() and dist.is_initialized()):
        return None
    group = bn.process_group if bn.process_group is not None else dist.group.WORLD
    return group if dist.get_world_size(group) > 1 else None


def weight_bn_act(W, bn, x, residual, relu, name=None, prepared=None, affine=None, pre=None, shard=None, slot=0):
    """[relu](BatchNorm2d(conv1x1(x, W)) [+ residual]) for a [M,K,1,1] weight: everything in this package's kernels
    (tcgen05 GEMM with the statistics in its epilogue + one normalise pass) when the shapes allow, else the library
    convolution followed by the fused BatchNorm passes. ``shard`` / ``slot``: the module's shard group and which of its two
    blocks this is (0 output, 1 writing net): a SyncBatchNorm over the shard group exchanges over its peer memory."""
    y = _weight_bn_act(W, bn, x, residual, relu, prepared, affine, pre, shard, slot)
    if GATE_LOG is not None and relu and name is not None:
        GATE_LOG.setdefault(name, []).append(y.detach() > 0)
    return y


def _eval_affine(bn):
    return capi.bn_eval_affine(bn.weight.detach().float().contiguous(), bn.bias.detach().float().contiguous(),
                               bn.running_mean, bn.running_var, bn.eps)


def _inference_block(bn, x, residual):
    """conv + eval-mode BN (+ ReLU) can run as ONE kernel: no batch statistics, no residual, nothing to differentiate."""
    return (_bn_fast(bn, x) and not bn.training and bn.running_mean is not None and residual is None
            and not torch.is_grad_enabled() and bn.running_mean.dtype == torch.float32
            and bn.running_var.dtype == torch.float32)


def _weight_bn_act(W, bn, x, residual, relu, prepared=None, affine=None, pre=None, shard=None, slot=0):
    if torch.is_autocast_enabled("cuda"):  # the nn.Conv2d this replaces would run in the autocast dtype
        x = x.to(torch.get_autocast_dtype("cuda"))
    M, K = W.shape[0], W.shape[1]
    if _bn_fast(bn, x) and capi.conv1x1_ok(x, M, K):
        x = x.contiguous()
        if _inference_block(bn, x, residual):
            # inference read (BASELINE config 5): the eval-mode BatchNorm and the ReLU ride in the GEMM epilogue
            hi, lo = prepared if prepared is not None else capi.conv1x1_prep(
                W.detach().reshape(M, K).to(torch.float32).contiguous(), False, x.dtype, tf32=capi.tf32())
            scale, shift = affine if affine is not None else _eval_affine(bn)
            return capi.conv1x1_fwd_affine(x, hi, lo, M, scale, shift, relu)
        res_is_x = residual is x or (residual is not None and residual.data_ptr() == x.data_ptr()
                                     and residual.shape == x.shape and residual.dtype == x.dtype)
        if residual is not None and not res_is_x:
            residual = residual.to(x.dtype).contiguous()
        use_batch, rm, rv, factor, nbt = _bn_args(bn, defer_counter=True)
        return _ConvBnActFn.apply(x, W, bn.weight, bn.bias, None if res_is_x else residual, rm, rv, use_batch, factor,
                                  float(bn.eps), relu, res_is_x, _sync_group(bn), nbt, pre, shard, slot)
    _warn_once("libconv", "a 1x1 convolution fell back to the library GEMM (feature rows not 16-byte aligned, or an "
                          "unsupported channel count); the BatchNorm passes stay fused")
    return bn_act(F.conv2d(x, W.to(x.dtype)), bn, residual, relu)


def conv_bn_act(conv, bn, x, residual, relu, name=None, shard=None, slot=0):
    """conv -> BatchNorm2d (-> + residual) (-> ReLU) for the module's 1x1 blocks (``shard``, ``slot``: see weight_bn_act)."""
    if _pointwise(conv) and _plain(conv):
        return weight_bn_act(conv.weight, bn, x, residual, relu, name, shard=shard, slot=slot)
    y = bn_act(conv(x), bn, residual, relu)
    if GATE_LOG is not None and relu and name is not None:
        GATE_LOG.setdefault(name, []).append(y.detach() > 0)
    return y


def bn_act(xc, bn, residual, relu):
    """BatchNorm2d (-> + residual) (-> ReLU) of an already convolved tensor (see conv_bn_act)."""
    if not _bn_fast(bn, xc) or _sync_group(bn) is not None:   # (cross-rank statistics exist on the fused conv path only)
        y = bn(xc)
        if residual is not None:
            y = residual + y
        return F.relu(y) if relu else y
    use_batch, rm, rv, factor = _bn_args(bn)
    xc = xc.contiguous()
    if residual is not None:
        residual = residual.to(xc.dtype).contiguous()
    return _BnActFn.apply(xc, bn.weight, bn.bias, residual, rm, rv, use_batch, factor, float(bn.eps), relu)


class Writingnet(nn.Module):
    """relu(x + BN(conv1x1(x))) -- memory.py:67-87; conv, BN, residual and ReLU in this package's kernels."""

    def __init__(self, input_feature_dim, feature_dim):
        super().__init__()
        assert input_feature_dim == feature_dim, \
            "Should match when residual mode is on ({} != {})".format(input_feature_dim, feature_dim)
        self.writefeat = nn.Sequential(
            nn.Conv2d(input_feature_dim, feature_dim, kernel_size=1, stride=1, bias=False),
            nn.BatchNorm2d(feature_dim),
        )
        self.relu = nn.ReLU(inplace=True)
        initialize_weights(self)

    def forward(self, x):
        if x.is_cuda and _plain(self.writefeat) and _plain(self.writefeat[0]):
            # _shard_group: the owning Memory_sup's shard group, set by its write() (a plain attribute: not in state_dict)
            return conv_bn_act(self.writefeat[0], self.writefeat[1], x, x, True, "writenet",
                               shard=getattr(self, "_shard_group", None), slot=1)
        return self.relu(x + self.writefeat(x))


class Memory_sup(nn.Module):
    """Categorical class memory with the reference's interface (memory.py:93-257, 317-336)."""

    def __init__(self, memory_size, input_feature_dim, feature_dim, momentum, temperature, gumbel_read,
                 device=None):
        super().__init__()
        self.memory_size = memory_size
        self.feature_dim = feature_dim
        self.momentum = momentum
        self.initial_momentum = momentum
        self.temperature = temperature
        self.output = nn.Sequential(
            nn.Conv2d(feature_dim * 2, input_feature_dim, kernel_size=1, stride=1, bias=False),
            nn.BatchNorm2d(input_feature_dim),
            nn.ReLU(inplace=True),
        )
        self.writenet = Writingnet(input_feature_dim, feature_dim)
        # the reference puts its state on the GPU unconditionally (memory.py:111,121); ``device`` (or the
        # PINMEM_B200_DEVICE environment variable) exists only so host-side logic can be unit-tested
        # without one -- forward() still refuses CPU tensors.
        dev = torch.device(device if device is not None else os.environ.get("PINMEM_B200_DEVICE", "cuda"))
        self.mem_cls = torch.arange(self.memory_size, device=dev)
        self.clsfier = nn.Linear(in_features=self.feature_dim, out_features=self.memory_size, bias=True)
        self.celoss = nn.CrossEntropyLoss(ignore_index=IGNORE_LABEL)
        self.gumbel_read = gumbel_read
        self.writeTF = lambda x: x.clone()
        self.m_items = F.normalize(torch.rand((memory_size, feature_dim), dtype=torch.float), dim=1).to(dev)
        initialize_weights(self)
        # extras (not in the reference)
        self.overlap_write = False     # run the write branch on a side stream next to the read (see forward)
        self.fold_memory_into_conv = True  # read hands [q ; score planes] to a convolution with the memory folded in
        self.fuse_grad_sum = True      # the write branch's d/d(query) is summed inside the read's dx kernel (see read())
        self.fold_min_pixels = 32768       # ... for feature maps of at least this many pixels per call
        self.shard_group = None        # set by sharding.enable_sharded_update()
        self.last_label_hist = None    # int64 [K+1] label histogram of the last read with labels
        self.last_bad_labels = None    # device int64 scalar: out-of-range label values of that read (counted as ignore)
        self.debug_labels = False      # True: raise when last_bad_labels != 0 (costs a device synchronisation per read)
        self.last_class_sums = None    # fp32 [K+1, C+4] sums|counts of the last write (after all-reduce)

    # ------------------------------------------------------------------------------------- forward

    def forward(self, query, mask=None, memory_writing=True, writing_detach=True):
        if memory_writing and self.overlap_write and query.is_cuda:
            return self._forward_two_streams(query, mask, writing_detach)
        updated_query, score_query, score_memory, readloss = self.read(query, mask, memory_writing, _tee=memory_writing)
        if memory_writing:
            tee, self._tee = getattr(self, "_tee", None), None
            writeloss = self.write(query if tee is None else tee, mask, writing_detach)
        else:
            writeloss = [0, 0]
        return updated_query, score_query, score_memory, readloss, writeloss

    def _forward_two_streams(self, query, mask, writing_detach):
        """Read and write only share their inputs (the query, the labels, the OLD memory), so the write runs on a
        side stream next to the read; autograd replays each branch's backward on the stream of its forward. Under
        CUDA-graph capture the two become parallel branches of the graph -- small-grid kernels of one branch
        (update, BatchNorm statistics, the 1x1-conv GEMMs) fill the SMs the other leaves idle."""
        cur = torch.cuda.current_stream(query.device)
        side = _SIDE_STREAMS.get(query.device)
        if side is None:
            side = _SIDE_STREAMS[query.device] = torch.cuda.Stream(device=query.device)
        side.wait_stream(cur)                     # fork: the write depends only on what precedes this call
        memory_in = self.m_items
        # the read's label pass runs on `side` too (before the write kernels that consume the packed map: stream order is
        # the dependency), its column softmax on a second side stream
        updated_query, score_query, score_memory, readloss = self.read(query, mask, True, _tee=True, _branch=True)
        memory_after_read = self.m_items          # the detached view read() installed (memory.py:323-324)
        tee, self._tee = getattr(self, "_tee", None), None
        with torch.cuda.stream(side):
            self.m_items = memory_after_read
            writeloss = self.write(query if tee is None else tee, mask, writing_detach)
            for t in (query, mask, memory_in, memory_after_read):
                if torch.is_tensor(t):
                    t.record_stream(side)
        cur.wait_stream(side)
        for t in (self.m_items, self.last_class_sums, writeloss[0], writeloss[1]):
            if torch.is_tensor(t):
                t.record_stream(cur)
        return updated_query, score_query, score_memory, readloss, writeloss

    def _inference_weights(self, M, u):
        """Folded + split weight of the output convolution for the inference read, cached while neither the weight nor
        the memory changes (same tensor objects, same in-place version counters). Never used while a CUDA graph is being
        captured: a replay must recompute it from whatever the memory buffer holds then."""
        W = self.output[0].weight
        Co, C, K = W.shape[0], self.feature_dim, self.memory_size
        self._folded_shape = torch.empty(Co, C + capi.PLANES, 0, 0, device="meta")  # shape carrier only (M, K of the GEMM)
        key = (W, W._version, M, M._version, u.dtype, capi.tf32())   # (an operand split for 3xTF32 has a lo part, one-pass not)
        cached = getattr(self, "_infer_cache", None)
        capturing = torch.cuda.is_current_stream_capturing()
        if (not capturing and cached is not None and cached[0][0] is W and cached[0][2] is M and cached[0][1] == key[1]
                and cached[0][3] == key[3] and cached[0][4] == key[4] and cached[0][5] == key[5]):
            return cached[1]
        W32 = W.detach().to(torch.float32).contiguous()
        Wp = torch.empty(Co, C + capi.PLANES, dtype=torch.float32, device=W.device)
        capi.fold_weight_fwd(W32, M.detach().to(torch.float32).contiguous(), Wp, Co, C, K)
        prepared = capi.conv1x1_prep(Wp, False, u.dtype, tf32=key[5])
        if not capturing:
            self._infer_cache = (key, prepared)
        return prepared

    def _memory_for_kernels(self, device):
        M = self.m_items
        if not M.is_cuda:
            raise RuntimeError("pinmem_b200 has no CPU path: m_items must live on a CUDA device")
        if M.dtype != torch.float32:
            raise RuntimeError("pinmem_b200: m_items must be float32")
        if M.shape != (self.memory_size, self.feature_dim):
            raise RuntimeError(f"pinmem_b200: m_items must be [{self.memory_size},{self.feature_dim}]")
        return M

    def read(self, query, mask, memory_writing, _tee=False, _branch=False):
        """memory.py:317-336. Returns (updated_query, score_query, score_memory, readloss)."""
        query = _check_features(query, "query")
        B, C, h, w = query.shape
        if C != self.feature_dim:
            raise RuntimeError(f"pinmem_b200: query has {C} channels, memory has {self.feature_dim}")
        if memory_writing:  # memory.py:323-324: cut the gradient into the memory when it is about to be rewritten
            self.m_items = self.m_items.detach()
        M = self._memory_for_kernels(query.device)
        labels = _check_labels(mask, B) if mask is not None else None
        g_query = g_memory = None
        if self.gumbel_read:
            g_query, g_memory = draw_gumbel_pair(B * h * w, self.memory_size, query.device)
        plain = _plain(self.output) and _plain(self.output[0]) and _plain(self.output[2])
        # pays once the GEMMs are big enough to be compute- rather than launch-bound (break-even ~ 3e4 pixels)
        planes = (plain and self.fold_memory_into_conv and B * h * w >= self.fold_min_pixels
                  and _foldable(self.output[0], C) and capi.planes_ok(query))
        # fp32 score-plane read about to be followed by a write on the same features: tee the features through the read so
        # that the write branch's gradient is summed inside the read's dx kernel (pm_read_bwd_planes, dx_add)
        tee = (_tee and memory_writing and planes and self.fuse_grad_sum and torch.is_grad_enabled()
               and query.requires_grad and query.dtype == torch.float32)
        # Inference read (BASELINE config 5): the folded + split weight and the BatchNorm affine depend on parameters only, so
        # their three small kernels run on a side stream -- a parallel branch of a captured graph -- under the read kernels
        # instead of between them and the convolution (27 us of a 108 us step at one 1024x2048 image per GPU)
        pre = None
        if planes and _inference_block(self.output[1], query, None) and query.dtype in (torch.float32, torch.bfloat16):
            cur = torch.cuda.current_stream(query.device)
            side = _SIDE_STREAMS.get(query.device)
            if side is None:
                side = _SIDE_STREAMS[query.device] = torch.cuda.Stream(device=query.device)
            side.wait_stream(cur)
            with torch.cuda.stream(side):
                pre = (self._inference_weights(M, query), _eval_affine(self.output[1]))
            for t in (*pre[0], *pre[1]):
                if torch.is_tensor(t):
                    t.record_stream(cur)
        # Two-stream mode, training: the output convolution's weight work (fold the memory in, split both operand layouts,
        # clear the statistics buffer: two small launches) depends on parameters only -- it runs on the second side stream
        # under read_fwd instead of between the read loss and the convolution
        wpre = None
        if (_branch and planes and pre is None and torch.is_grad_enabled() and self.output[1].training
                and _bn_fast(self.output[1], query) and query.dtype in (torch.float32, torch.bfloat16)
                and capi.conv1x1_ok(query, self.output[0].weight.shape[0], C + capi.PLANES)):
            cur = torch.cuda.current_stream(query.device)
            aux = _stream_of(_AUX_STREAMS, query.device)
            aux.wait_stream(cur)
            with torch.cuda.stream(aux):
                Wp_early = _FoldWeightFn.apply(self.output[0].weight, M)
                Co = Wp_early.shape[0]
                stats = torch.empty(2 * Co + 1, dtype=torch.float64, device=query.device)
                cdt = torch.get_autocast_dtype("cuda") if torch.is_autocast_enabled("cuda") else query.dtype
                ops, opsT = capi.conv1x1_prep_both(Wp_early.detach().reshape(Co, C + capi.PLANES).to(torch.float32).contiguous(),
                                                   cdt, zero=stats, tf32=capi.tf32())
            wpre = (Wp_early, (ops, opsT, stats))
            for t in (Wp_early, stats, *ops, *opsT):
                if torch.is_tensor(t):
                    t.record_stream(cur)
        # the global read exchanges only for reads that can feed a training gradient: a read under no_grad (validation,
        # memory_initalize, a forward-only GraphedStep) stays rank-local, so ranks need not make such reads in lock-step
        xg = self.shard_group if (torch.is_grad_enabled() and sharding.global_read(self.shard_group)) else None
        outs = _ReadFn.apply(query, M, labels, g_query, g_memory, float(self.temperature), self.memory_size, planes, tee,
                             _branch, xg)
        if wpre is not None:   # (a branched _ReadFn joins the aux stream itself; this covers the read without labels / K > 19)
            torch.cuda.current_stream(query.device).wait_stream(_stream_of(_AUX_STREAMS, query.device))
        u, score_query, score_memory, readloss, hist = outs[:5]
        if pre is not None:
            torch.cuda.current_stream(query.device).wait_stream(_SIDE_STREAMS[query.device])
        self._tee = outs[5] if tee else None
        if labels is None:
            readloss = 0  # memory.py:178
        else:
            self.last_label_hist = hist
            self.last_bad_labels = _ReadFn.last_bad
            # the write of the same forward() reads the packed map instead of the int64 one (1/8 of the bytes)
            self._packed = (mask, _ReadFn.last_lab8) if _ReadFn.last_lab8 is not None else None
            if self.debug_labels and int(self.last_bad_labels) != 0:   # synchronises: debugging aid only
                raise RuntimeError(f"pinmem_b200: {int(self.last_bad_labels)} label values outside [0,{self.memory_size}) "
                                   "and != 255 (torch's one_hot / CrossEntropyLoss would raise a device assert)")
        if planes:
            # conv(W, [q ; p.M]) = W1.q + (W2.M^T).p : the memory is folded into the weight (a [C_out, 32] block) and
            # the convolution runs on [q ; score planes] -- C+32 input channels instead of 2C
            # (`pre` exists exactly when this is an inference block: u has the query's device, rank and dtype)
            infer = pre is not None and capi.conv1x1_ok(u, self.output[0].weight.shape[0], C + capi.PLANES)
            prepared = pre[0] if infer else None
            if prepared is not None:
                Wp = self._folded_shape
            elif wpre is not None:
                Wp = wpre[0]
            else:
                Wp = _FoldWeightFn.apply(self.output[0].weight, M)
            updated_query = weight_bn_act(Wp, self.output[1], u, None, True, "output", prepared,   # Wp [C_out, C+32, 1, 1]
                                          pre[1] if infer else None,
                                          wpre[1] if (wpre is not None and prepared is None) else None,
                                          shard=self.shard_group, slot=0)
        elif plain:
            updated_query = conv_bn_act(self.output[0], self.output[1], u, None, True, "output", shard=self.shard_group,
                                        slot=0)
        else:
            updated_query = self.output(u)
        return updated_query, score_query, score_memory, readloss

    def write(self, input, mask, writing_detach=True):
        """memory.py:206-257. Rebinds ``m_items`` to a fresh tensor; returns [div_loss, cls_loss]."""
        query = _check_features(input, "input")
        B = query.shape[0]
        if mask is None:
            raise RuntimeError("pinmem_b200: memory_writing=True needs labels (the reference crashes at memory.py:208)")
        labels = _check_labels(mask, B)
        packed = getattr(self, "_packed", None)
        if packed is not None and packed[0] is mask:   # same label tensor as the read of this forward(): reuse its pack
            labels = packed[1]
        self._packed = None
        M_old = self._memory_for_kernels(query.device)
        if M_old.requires_grad and torch.is_grad_enabled():
            # memory.py:236 blends the NON-detached self.m_items[slot]; forward() never gets here with a grad-carrying
            # memory (read() detaches it first when writing, memory.py:323-324). A direct write() on one would silently
            # drop d loss / d m_items: refuse instead of returning a wrong gradient.
            raise RuntimeError("pinmem_b200: write() on a grad-carrying m_items is not differentiable w.r.t. the old memory "
                               "here; detach it first (forward(..., memory_writing=True) does)")
        if self._writenet_fused(query):
            conv, bn = self.writenet.writefeat[0], self.writenet.writefeat[1]
            use_batch, rm, rv, factor, nbt = _bn_args(bn, defer_counter=True)
            M_new, div_loss, cls_loss, SD = _WriteNetFn.apply(
                query.contiguous(), labels, M_old, conv.weight, bn.weight, bn.bias, rm, rv, factor, float(bn.eps), nbt,
                _sync_group(bn), self.clsfier.weight, self.clsfier.bias, float(self.momentum), self.memory_size,
                self.shard_group)
        else:
            if isinstance(self.writenet, Writingnet):
                self.writenet._shard_group = self.shard_group   # its SyncBatchNorm exchanges over this group's peer memory
            f = self.writenet(query)
            f = _check_features(f, "write feature")
            M_new, div_loss, cls_loss, SD = _WriteFn.apply(f, labels, M_old, self.clsfier.weight, self.clsfier.bias,
                                                           float(self.momentum), self.memory_size, self.shard_group)
        self.last_class_sums = SD
        self.m_items = M_new.detach() if writing_detach else M_new
        return [div_loss, cls_loss]

    def _writenet_fused(self, x):
        """The writing net can ride in the write's kernels (_WriteNetFn): an unhooked Writingnet of a 1x1 convolution and a
        training-mode BatchNorm2d / SyncBatchNorm, fp32 features on the pipelined kernels' alignment. Anything else (bf16,
        autocast, eval-mode statistics, hooks, odd shapes) runs the Writingnet and _WriteFn as separate steps."""
        wn = self.writenet
        if not (type(wn) is Writingnet and _plain(wn) and _plain(wn.writefeat) and len(wn.writefeat) == 2):
            return False
        conv, bn = wn.writefeat[0], wn.writefeat[1]
        C = x.shape[1]
        return (_pointwise(conv) and _plain(conv) and conv.in_channels == C and conv.out_channels == C and _bn_fast(bn, x)
                and bn.training and not torch.is_autocast_enabled("cuda") and x.dtype == torch.float32
                and C in (32, 64, 128, 256) and capi.conv1x1_ok(x, C, C) and capi.planes_ok(x))

    # ----------------------------------------------------------------------- external entry points

    def classification_loss(self, mem):
        """memory.py:259-262: CE of the slot classifier on ``mem`` against the slot indices (differentiable w.r.t.
        ``mem`` and the classifier). write() computes the same loss fused into the update kernel."""
        capi.require_cuda(mem)
        return _MemoryLossFn.apply(mem, self.clsfier.weight, self.clsfier.bias)[1]

    def diversityloss(self, mem):
        """memory.py:264-272: mean positive off-diagonal cosine of ``mem`` (differentiable w.r.t. ``mem``)."""
        capi.require_cuda(mem)
        return _MemoryLossFn.apply(mem, None, None)[0]

    def get_score(self, query, mask, mem):
        """memory.py:167-189 on an already normalised NHWC query (validation, train.py:891-896).

        Returns (score_query [N,K], score_memory [N,K], readloss), readloss the int 0 without labels. As in the reference,
        all three are differentiable with respect to ``query`` and ``mem`` when either requires grad (and grad mode is on);
        otherwise the same kernels run without saving anything for a backward.
        """
        capi.require_cuda(query, mem)
        Bq = query.shape[0]
        labels = _check_labels(mask, Bq) if mask is not None else None
        if torch.is_grad_enabled() and (query.requires_grad or mem.requires_grad):
            score_query, score_memory, readloss = _ScoreFn.apply(query, mem, labels, float(self.temperature), self.gumbel_read)
            hist = _ScoreFn.last_hist
        else:
            with torch.no_grad():
                score_query, score_memory, readloss, hist = _score_kernels(
                    query.detach().to(torch.float32).contiguous(), mem.detach().to(torch.float32).contiguous(), labels,
                    float(self.temperature), self.gumbel_read)[:4]
        if labels is not None:
            self.last_label_hist = hist
        return score_query, score_memory, (readloss if labels is not None else 0)


def _score_kernels(q, M, labels, temperature, gumbel):
    """The kernels of get_score on a contiguous fp32 NHWC query [B,h,w,C] and memory [K,C]. Returns (score_query,
    score_memory, readloss, label histogram, ds_rl, rl_out); the last four are None without labels."""
    Bq, h, w, C = q.shape
    K = M.shape[0]
    N = Bq * h * w
    dev = q.device
    KP = capi.score_stride(K)
    s = (torch.zeros if capi.deterministic() else torch.empty)(N, KP, dtype=torch.float32, device=dev)   # (see _ReadFn)
    capi.score_nhwc(q, M, s, N, C, K)
    readloss = hist = ds_rl = rl_out = None
    if labels is not None:
        buf = torch.zeros(N * KP + 2 * capi.WS_WORDS + 4, dtype=torch.float32, device=dev)
        ws = buf[N * KP: N * KP + 2 * capi.WS_WORDS]
        ds_rl, rl_out = buf[: N * KP], buf[N * KP + 2 * capi.WS_WORDS:]
        capi.readloss(s, labels, temperature, Bq, h, w, K, ds_rl, ws, rl_out)
        readloss = rl_out[0]
        hist = ws.view(torch.int64)[capi.WS_HIST: capi.WS_HIST + K + 1]
    g_query = g_memory = None
    if gumbel:
        g_query, g_memory = draw_gumbel_pair(N, K, dev)
    score_query = torch.empty(N, K, dtype=torch.float32, device=dev)
    score_memory = torch.empty(N, K, dtype=torch.float32, device=dev)
    cs_ws = torch.empty(capi.colsoftmax_workspace_floats(K), dtype=torch.float32, device=dev)
    capi.colsoftmax(s, g_query, score_query, cs_ws, N, K)
    capi.rowsoftmax(s, g_memory, score_memory, N, K)
    return score_query, score_memory, readloss, hist, ds_rl, rl_out


class _ScoreFn(torch.autograd.Function):
    """get_score with its autograd: query [B,h,w,C], mem [K,C] -> score_query, score_memory [N,K], readloss.

    Backward: E = pm_score_bwd (both softmaxes and the read loss), then dq = E.M and dM = E^T.q (pm_score_nhwc_bwd). There is
    no normalisation to differentiate: get_score takes the query as it is."""

    last_hist = None  # the label histogram of the last call with labels

    @staticmethod
    def forward(ctx, query, mem, labels, temperature, gumbel):
        q = query.detach().to(torch.float32).contiguous()
        M = mem.detach().to(torch.float32).contiguous()
        score_query, score_memory, readloss, _ScoreFn.last_hist, ds_rl, rl_out = _score_kernels(q, M, labels, temperature,
                                                                                                gumbel)
        if readloss is None:
            readloss = torch.zeros((), dtype=torch.float32, device=q.device)
        ctx.set_materialize_grads(False)
        ctx.has_loss = labels is not None
        ctx.qshape, ctx.qdtype, ctx.mdtype = query.shape, query.dtype, mem.dtype
        ctx.save_for_backward(q, M, score_query, score_memory, ds_rl, rl_out)
        return score_query, score_memory, readloss

    @staticmethod
    def backward(ctx, g_sq, g_sm, g_rl):
        q, M, score_query, score_memory, ds_rl, rl_out = ctx.saved_tensors
        N, K = score_query.shape
        C = q.shape[-1]
        q = q.view(N, C)
        dense = lambda g: None if g is None else g.reshape(N, K).to(torch.float32).contiguous()
        if ctx.has_loss and g_rl is not None:
            g_rl = g_rl.reshape(1).to(torch.float32).contiguous()
        else:
            g_rl = ds_rl = rl_out = None
        E = torch.empty(N, capi.score_stride(K), dtype=torch.float32, device=q.device)
        capi.score_bwd(score_query if g_sq is not None else None, dense(g_sq), score_memory if g_sm is not None else None,
                       dense(g_sm), E, K, ds_rl=ds_rl, g_loss=g_rl, rl_out=rl_out)
        dq = torch.empty(N, C, dtype=torch.float32, device=q.device) if ctx.needs_input_grad[0] else None
        dM = torch.zeros(K, C, dtype=torch.float32, device=q.device) if ctx.needs_input_grad[1] else None
        capi.score_nhwc_bwd(q, M, E, dq, dM, K)
        if dq is not None:
            dq = dq.view(ctx.qshape).to(ctx.qdtype)
        if dM is not None:
            dM = dM.to(ctx.mdtype)
        return dq, dM, None, None, None
