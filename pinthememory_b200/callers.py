"""The callers either side of the memory path, on the same kernels (SURVEY.md 8f rows 2, 3 and 5).

* ``PrototypePool`` / ``initialize_memory`` -- the reference's ``Trainer.memory_initalize``
  (train.py:1000-1042): class prototypes pooled over the training set. One ``pm_write_reduce_fwd`` launch
  per batch accumulates the packed class sums|counts in place (the kernel only ever adds into its output);
  with a shard group the sums are all-reduced once at the end, so every rank starts from the same memory.
* ``upsampled_cross_entropy`` -- the head's main loss ``criterion(Upsample(logits, size), gts)``
  (network/deepv3plus.py:575-578, mynn.py:57-62, loss.py:167-180) through ``pm_readloss_fwd``: the
  ``[B,K,Hm,Wm]`` up-sampled logits and their log-softmax never exist in memory (for K=19 at 768x768 and
  batch 8 that is 358 MB written and re-read several times by the eager path).

* ``class_mean_vectors`` -- the t-SNE tooling's per-class mean of the UP-SAMPLED normalised features
  (tsnelib.py:48-74 ``input2basket``): sum over the label pixels of class k of bilinear_up(x/|x|), divided by the pixel
  count. The bilinear weights are transposed onto the feature grid by ``pm_readloss_fwd`` (with all-zero logits and one
  spare slot its gradient IS ``W/K' - onehot`` scattered back), and ``pm_read_bwd_dM`` contracts them with the
  normalised features -- the [B,C,Hm,Wm] up-sampled map (1.2 GB at 8 x 768 x 768) never exists.
* ``SegMetrics`` -- validation (train.py:847-939, eval.py:277-286,304-337): the criterion on the up-sampled head output,
  its argmax and ``fast_hist`` (utils/misc.py:65-73) in one ``pm_seg_eval`` launch per batch; the confusion matrix stays
  on the device and is all-reduced once at the end (train.py:927-929). At a Cityscapes validation image that removes
  160 MB of up-sampled logits, a 16.8 MB prediction copy to the host and a NumPy bincount over 2.1 M pixels.
* ``upsample_concat`` -- the decoder step after the memory module (network/deepv3plus.py:569-572):
  ``cat([dec0_fine, Upsample(dec0_up, low_level.size()[2:])], 1)`` as one ``pm_upcat_fwd`` launch that writes the
  up-sampled channels straight into the concatenated map, and a deterministic gather backward (``pm_upcat_bwd``) that
  reads the gradient's coarse channels in place. torch's own backward uses atomics and raises under
  ``torch.use_deterministic_algorithms(True)``.

CUDA only, like the rest of the package.
"""
import os

import torch
import torch.nn.functional as F

from . import capi, sharding


class PrototypePool:
    """Accumulates per-class sums of L2-normalised features weighted by the down-sampled one-hot labels."""

    def __init__(self, memory_size, feature_dim, device="cuda", group=None):
        self.K, self.C, self.group = int(memory_size), int(feature_dim), group
        self.sums_counts = torch.zeros(self.K + 1, self.C + 4, dtype=torch.float32, device=device)  # [K+1, C | count,0,0,0]
        self.batches = 0

    def add(self, features, labels):
        """features [B,C,h,w] fp32|bf16 (un-normalised: train.py:1019 normalises, so does the kernel),
        labels [B,Hm,Wm] int64 with 255 = ignore."""
        capi.require_cuda(features, labels)
        if features.dim() != 4 or features.shape[1] != self.C:
            raise RuntimeError(f"pinmem_b200: features must be [B,{self.C},h,w], got {tuple(features.shape)}")
        if labels.dtype != torch.int64 or labels.dim() != 3 or labels.shape[0] != features.shape[0]:
            raise RuntimeError("pinmem_b200: labels must be int64 [B,Hm,Wm]")
        capi.write_reduce_fwd(features.detach().contiguous(), labels.contiguous(), self.sums_counts, self.K)
        self.batches += 1
        return self

    def finalize(self):
        """train.py:1037-1040: ``normalize(basket / count)`` with empty classes' counts set to 1 (zero rows)."""
        sd = self.sums_counts
        if self.group is not None:
            sd = sharding.all_reduce_sum_(sd.clone(), self.group)
        sums, counts = sd[: self.K, : self.C], sd[: self.K, self.C]
        counts = torch.where(counts == 0, torch.ones_like(counts), counts)
        return F.normalize(sums / counts.unsqueeze(1), dim=1)


def initialize_memory(module, batches, group=None):
    """``module.m_items <- prototypes`` from an iterable of (features, labels); returns the pool."""
    pool = PrototypePool(module.memory_size, module.feature_dim, module.m_items.device,
                         group if group is not None else getattr(module, "shard_group", None))
    for features, labels in batches:
        pool.add(features, labels)
    module.m_items = pool.finalize()
    return pool


class _UpsampledCE(torch.autograd.Function):
    @staticmethod
    def forward(ctx, logits, labels):
        B, K, h, w = logits.shape
        N = B * h * w
        KP = capi.score_stride(K)
        dev = logits.device
        s = torch.zeros(N, KP, dtype=torch.float32, device=dev)
        s[:, :K] = logits.detach().permute(0, 2, 3, 1).reshape(N, K)
        buf = torch.zeros(N * KP + 2 * capi.WS_WORDS + 4, dtype=torch.float32, device=dev)
        ds = buf[: N * KP]
        ws = buf[N * KP: N * KP + 2 * capi.WS_WORDS]
        out = buf[N * KP + 2 * capi.WS_WORDS:]
        capi.readloss(s, labels, 1.0, B, h, w, K, ds, ws, out)
        ctx.save_for_backward(ds, out)
        ctx.shape, ctx.dtype = (B, K, h, w), logits.dtype
        return out[0].to(logits.dtype)

    @staticmethod
    def backward(ctx, g):
        ds, out = ctx.saved_tensors
        B, K, h, w = ctx.shape
        grad = (ds.view(B, h, w, -1)[..., :K] * (g.to(torch.float32) * out[1])).permute(0, 3, 1, 2)
        return grad.to(ctx.dtype).contiguous(), None


def upsampled_cross_entropy(logits, labels):
    """``CrossEntropyLoss2d(ignore_index=255)(Upsample(logits, labels.shape[-2:]), labels)`` fused.

    logits [B,K,h,w] (K <= 31) fp32|bf16 CUDA, labels [B,Hm,Wm] int64. Mean over the non-ignored pixels
    (NaN if there is none, like torch). Differentiable w.r.t. ``logits``.
    """
    capi.require_cuda(logits, labels)
    if logits.dim() != 4 or labels.dim() != 3 or labels.shape[0] != logits.shape[0]:
        raise RuntimeError("pinmem_b200: logits must be [B,K,h,w] and labels [B,Hm,Wm]")
    if labels.dtype not in (torch.int64, torch.uint8):
        raise RuntimeError("pinmem_b200: labels must be int64 (or uint8 class ids)")
    if not 1 <= logits.shape[1] <= 31:
        raise RuntimeError("pinmem_b200: upsampled_cross_entropy supports 1..31 classes")
    return _UpsampledCE.apply(logits, labels.contiguous())


def class_mean_vectors(features, labels, num_class):
    """tsnelib.py:48-74: ``(means [K,C], counts [K])`` with ``means[k] = sum_{label px of class k} up(x/|x|)[px] / counts[k]``
    (zero rows where a class has no pixel), ``up`` = bilinear, align_corners=True, to the label size. The reference
    appends ``means[k]`` for every selected class with ``counts[k] != 0`` to its basket.

    features [B,C,h,w] fp32|bf16 CUDA (C in 32/64/128/256), labels [B,Hm,Wm] int64, num_class <= 30.
    """
    capi.require_cuda(features, labels)
    if features.dim() != 4 or labels.dim() != 3 or labels.shape[0] != features.shape[0]:
        raise RuntimeError("pinmem_b200: features must be [B,C,h,w] and labels [B,Hm,Wm]")
    if labels.dtype != torch.int64:
        raise RuntimeError("pinmem_b200: labels must be int64")
    K = int(num_class)
    if not 1 <= K <= 30:
        raise RuntimeError("pinmem_b200: class_mean_vectors supports 1..30 classes")
    B, C, h, w = features.shape
    N, dev = B * h * w, features.device
    x = features.detach().contiguous()
    labels = labels.contiguous()
    K1 = K + 1                      # one spare slot no pixel is labelled with: its "gradient" is the plain tap weight / K1
    KP = capi.score_stride(K1)
    s = torch.zeros(N, KP, dtype=torch.float32, device=dev)       # all logits equal -> softmax = 1/K1 everywhere
    buf = torch.zeros(N * KP + 2 * capi.WS_WORDS + 4, dtype=torch.float32, device=dev)
    ds, ws, out = buf[: N * KP], buf[N * KP: N * KP + 2 * capi.WS_WORDS], buf[N * KP + 2 * capi.WS_WORDS:]
    # labels >= K (and 255) are "ignore" for the K1-slot loss exactly as for the reference's one_hot(K+1) trick
    capi.readloss_fwd(s, labels, 1.0, B, h, w, K1, ds, ws, out)
    ds = ds.view(N, KP)
    # ds[n,k] = sum_px w(px->n) (1/K1 - [label(px) = k]); slot K is never labelled: ds[n,K] = sum_px w(px->n) / K1
    omega = torch.zeros(N, KP, dtype=torch.float32, device=dev)
    omega[:, :K] = ds[:, K:K1] - ds[:, :K]                          # transposed bilinear weights per class
    sums = torch.zeros(K1, C, dtype=torch.float32, device=dev)
    score_dummy = torch.zeros(N, K1, dtype=torch.float32, device=dev)
    capi.read_bwd_dM(None, x, score_dummy, omega, sums, K1)          # sums[k] = sum_n omega[n,k] x[n]/|x[n]|
    counts = ws.view(torch.int64)[capi.WS_HIST: capi.WS_HIST + K].to(torch.float32)
    safe = torch.where(counts == 0, torch.ones_like(counts), counts)
    return sums[:K] / safe.unsqueeze(1), counts


class SegMetrics:
    """Validation metrics of a segmentation head: mean cross-entropy per batch and the accumulated ``[K,K]`` confusion
    matrix (rows = label, columns = prediction, ``fast_hist``'s layout), both computed on the device.

    ``group``: a ``sharding.ShardGroup`` whose ranks' matrices ``finalize`` sums, or None (this process only).
    ``device`` defaults to CUDA (``PINMEM_B200_DEVICE`` only serves CPU unit tests of ``finalize``'s host logic).
    """

    def __init__(self, num_classes, device=None, group=None):
        self.K, self.group = int(num_classes), group
        if not 1 <= self.K <= 31:
            raise RuntimeError("pinmem_b200: SegMetrics supports 1..31 classes")
        dev = torch.device(device if device is not None else os.environ.get("PINMEM_B200_DEVICE", "cuda"))
        self.confusion = torch.zeros(self.K, self.K, dtype=torch.int64, device=dev)
        self.last_bad_labels = None   # device int64 scalar: label values of the last batch outside [0,K) and != 255

    def add(self, logits, labels, predictions=False):
        """logits [B,K,h,w] fp32|bf16 (before the head's up-sampling, or already at label size), labels [B,Hm,Wm] int64|uint8
        with 255 = ignore, Hm >= h, Wm >= w. Returns the batch's mean cross-entropy over its valid label pixels (0-d fp32
        device tensor, NaN when there is none); with ``predictions`` also the argmax map [B,Hm,Wm] uint8."""
        capi.require_cuda(logits, labels)
        if logits.device != self.confusion.device or labels.device != self.confusion.device:
            raise RuntimeError(f"pinmem_b200: SegMetrics lives on {self.confusion.device}, got tensors on {logits.device} "
                               f"and {labels.device}")
        if logits.dim() != 4 or labels.dim() != 3 or labels.shape[0] != logits.shape[0] or logits.shape[1] != self.K:
            raise RuntimeError(f"pinmem_b200: logits must be [B,{self.K},h,w] and labels [B,Hm,Wm], got "
                               f"{tuple(logits.shape)} and {tuple(labels.shape)}")
        if labels.dtype not in (torch.int64, torch.uint8):
            raise RuntimeError("pinmem_b200: labels must be int64 (or uint8 class ids)")
        capi.dtype_code(logits)
        if labels.shape[1] < logits.shape[2] or labels.shape[2] < logits.shape[3]:
            raise RuntimeError("pinmem_b200: SegMetrics up-samples only: labels must be at least the logits' size")
        dev = logits.device
        buf = torch.zeros(capi.SEG_WS_WORDS + 1, dtype=torch.int64, device=dev)   # workspace words | loss (fp32 bits)
        ws, out = buf[: capi.SEG_WS_WORDS], buf[capi.SEG_WS_WORDS:].view(torch.float32)
        pred = torch.empty(labels.shape, dtype=torch.uint8, device=dev) if predictions else None
        capi.seg_eval(logits.detach().contiguous(), labels.contiguous(), self.confusion, pred, ws, out)
        self.last_bad_labels = ws[capi.SEG_WS_BAD]
        loss = out[0]
        return (loss, pred) if predictions else loss

    def reset(self):
        self.confusion.zero_()

    def finalize(self):
        """(confusion [K,K] int64 summed over the group, iou [K] float64, mean_iou): iou = diag / (rowsum + colsum - diag),
        NaN for a class absent from both labels and predictions; mean_iou = nanmean(iou) (0-d float64)."""
        conf = self.confusion
        if self.group is not None:
            conf = sharding.all_reduce_sum_(conf.clone(), self.group)
        iou = segmentation_iou(conf)
        return conf, iou, iou.nanmean()


def segmentation_iou(confusion):
    """Per-class IoU of a [K,K] confusion matrix (rows = label, columns = prediction) in float64."""
    c = confusion.to(torch.float64)
    diag = c.diagonal()
    return diag / (c.sum(1) + c.sum(0) - diag)


class _UpsampleConcat(torch.autograd.Function):
    @staticmethod
    def forward(ctx, fine, coarse):
        B, Cf, H, W = fine.shape
        out = torch.empty(B, Cf + coarse.shape[1], H, W, dtype=fine.dtype, device=fine.device)
        capi.upcat_fwd(fine.detach().contiguous(), coarse.detach().contiguous(), out)
        ctx.Cf, ctx.coarse_shape = Cf, coarse.shape   # shapes only: the backward needs no saved tensor
        return out

    @staticmethod
    def backward(ctx, g):
        if not g.is_contiguous():
            g = g.contiguous()
        d_coarse = None
        if ctx.needs_input_grad[1]:
            d_coarse = torch.empty(ctx.coarse_shape, dtype=g.dtype, device=g.device)
            capi.upcat_bwd(g, d_coarse, ctx.Cf)
        d_fine = g.narrow(1, 0, ctx.Cf) if ctx.needs_input_grad[0] else None
        return d_fine, d_coarse


def upsample_concat(fine, coarse):
    """``torch.cat([fine, F.interpolate(coarse, fine.shape[-2:], mode="bilinear", align_corners=True)], 1)`` fused.

    fine [B,Cf,H,W] and coarse [B,Cc,h,w]: CUDA, the same device, dtype (fp32|bf16) and batch, H >= h, W >= w; Cf may
    be 0. The forward equals torch's bit for bit. Differentiable w.r.t. both inputs: the gradient of ``fine`` is the
    incoming gradient's first Cf channels (a view, as with torch.cat), that of ``coarse`` comes from a deterministic
    kernel (fp32 accumulation in a fixed order, no atomics).
    """
    capi.require_cuda(fine, coarse)
    if fine.dim() != 4 or coarse.dim() != 4:
        raise RuntimeError(f"pinmem_b200: upsample_concat takes [B,C,H,W] tensors, got {tuple(fine.shape)} and "
                           f"{tuple(coarse.shape)}")
    if fine.device != coarse.device:
        raise RuntimeError(f"pinmem_b200: upsample_concat got tensors on {fine.device} and {coarse.device}")
    if fine.dtype != coarse.dtype:
        raise RuntimeError(f"pinmem_b200: upsample_concat got {fine.dtype} and {coarse.dtype}")
    capi.dtype_code(fine)
    if fine.shape[0] != coarse.shape[0]:
        raise RuntimeError(f"pinmem_b200: upsample_concat got batches of {fine.shape[0]} and {coarse.shape[0]}")
    if fine.shape[2] < coarse.shape[2] or fine.shape[3] < coarse.shape[3]:
        raise RuntimeError("pinmem_b200: upsample_concat up-samples only: fine must be at least coarse's size")
    return _UpsampleConcat.apply(fine, coarse)
