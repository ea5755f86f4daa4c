"""SegMetrics / pm_seg_eval: up-sampling, argmax, cross-entropy and the fast_hist confusion matrix in one label pass.

The checker is ``segmentation_confusion`` below (F.interpolate, argmax, the fast_hist restatement of
utils/misc.py:65-73); bf16 logits are checked with fp32 maths on their values. CPU tests cover the host-side IoU maths,
the C entry's argument checks and the group reduction of ``finalize`` over gloo.
"""
import ctypes
import os
import socket

import numpy as np
import pytest
import torch
import torch.nn.functional as F

K19 = 19


def fast_hist(pred, gt, K):
    """utils/misc.py:65-73 restated: ``bincount(K * gt[m] + pred[m], minlength=K*K).reshape(K, K)`` with
    ``m = (gt >= 0) & (gt < K)`` -- rows = label, columns = prediction. Works on torch tensors (CPU or CUDA)."""
    m = (gt >= 0) & (gt < K)
    return torch.bincount(K * gt[m].to(torch.int64) + pred[m].to(torch.int64), minlength=K * K).view(K, K)


def upsample_logits(logits, size):
    """The head's output at label size: bilinear, align_corners=True; equal sizes are a copy (as in torch)."""
    if tuple(logits.shape[-2:]) == tuple(size):
        return logits
    return F.interpolate(logits, size=tuple(size), mode="bilinear", align_corners=True)


def segmentation_confusion(logits, labels, K):
    """One validation batch of train.py:847-939 / eval.py:277-286,304-337: ``(confusion [K,K] int64, pred [B,Hm,Wm]
    int64, mean CE)``. The logits are up-sampled (``upsample_logits``), ``pred = argmax(1)`` (first maximal class),
    the confusion matrix is ``fast_hist`` of utils/misc.py:65-73 and the loss is CrossEntropyLoss2d(ignore_index=255)
    (mean over the label pixels in [0,K); NaN when there is none).

    The reference tree is not part of this checkout: this restatement of ``fast_hist`` (utils/misc.py:65-73) and the
    loop around it is the contract the fused kernel is checked against. Computed in the logits' dtype (pass
    ``.double()`` for an fp64 loss).
    """
    labels = labels.to(torch.int64)
    up = upsample_logits(logits, labels.shape[-2:])
    pred = up.argmax(1)
    conf = fast_hist(pred, labels, K)
    m = (labels >= 0) & (labels < K)
    lsm = F.log_softmax(up, dim=1)
    nll = -lsm.gather(1, torch.where(m, labels, torch.zeros_like(labels)).unsqueeze(1)).squeeze(1)
    loss = nll[m].mean() if bool(m.any()) else torch.tensor(float("nan"), dtype=up.dtype, device=up.device)
    return conf, pred, loss


def top2_gap(logits, size):
    """Per label pixel: the largest minus the second largest up-sampled logit (where a fused argmax may legitimately
    differ from torch's by rounding); +inf for K == 1."""
    up = upsample_logits(logits, size)
    if up.shape[1] == 1:
        return torch.full_like(up[:, 0], float("inf"))
    t = up.topk(2, dim=1).values
    return t[:, 0] - t[:, 1]


# ----------------------------------------------------------------------------------------------------------------- CPU


def _numpy_fast_hist(pred, gt, K):
    """utils/misc.py:65-73 as the reference writes it, on NumPy arrays."""
    mask = (gt >= 0) & (gt < K)
    return np.bincount(K * gt[mask].astype(int) + pred[mask], minlength=K ** 2).reshape(K, K)


def test_fast_hist_and_iou_restatement_match_numpy():
    from pinthememory_b200.callers import segmentation_iou

    g = torch.Generator().manual_seed(5)
    K = 7
    gt = torch.randint(0, K, (3, 20, 24), generator=g)
    gt[0, :4] = 255
    gt[1, 2, :5] = 9        # out of range: excluded
    gt[2, 3, :3] = -1       # negative: excluded
    pred = torch.randint(0, K, (3, 20, 24), generator=g)
    pred[gt == 3] = 3       # a class predicted perfectly
    conf = fast_hist(pred, gt, K)
    ref = _numpy_fast_hist(pred.numpy().ravel(), gt.numpy().ravel(), K)
    assert np.array_equal(conf.numpy(), ref)
    conf[6, :] = 0
    conf[:, 6] = 0          # class 6 absent from labels and predictions -> NaN
    iou = segmentation_iou(conf).numpy()
    c = conf.numpy().astype(np.float64)
    with np.errstate(invalid="ignore"):
        want = np.diag(c) / (c.sum(1) + c.sum(0) - np.diag(c))
    assert np.isnan(iou[6]) and np.allclose(iou[:6], want[:6], rtol=0, atol=0)
    assert abs(float(torch.tensor(iou).nanmean()) - float(np.nanmean(want))) < 1e-15


def test_seg_eval_argument_checks_run_without_a_gpu():
    """Rejected arguments return negative status codes before any CUDA call."""
    from pinthememory_b200 import capi

    lib = capi.load()
    p = ctypes.c_void_p(256)
    ok = (p, 0, 2, 19, 8, 8, p, 0, 32, 32, p, None, p, p, None)

    def call(**kw):
        a = list(ok)
        names = ("logits", "dtype", "B", "K", "h", "w", "labels", "u8", "Hm", "Wm", "conf", "pred", "ws", "out", "stream")
        for k, v in kw.items():
            a[names.index(k)] = v
        return lib.pm_seg_eval(*a)

    assert call(logits=None) == -1
    assert call(labels=None) == -1
    assert call(conf=None) == -1
    assert call(ws=None) == -1
    assert call(out=None) == -1
    assert call(dtype=2) == -2
    assert call(K=0) == -4 and call(K=32) == -4
    assert call(B=0) == -5 and call(h=0) == -5 and call(w=0) == -5
    assert call(Hm=7) == -5 and call(Wm=7) == -5          # labels smaller than the logits
    assert call(conf=ctypes.c_void_p(260)) == -6
    assert call(ws=ctypes.c_void_p(4)) == -6


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def _hand_confusion(rank, K=5):
    g = torch.Generator().manual_seed(40 + rank)
    c = torch.randint(0, 1000, (K, K), generator=g, dtype=torch.int64)
    c[4, :] = 0
    c[:, 4] = 0     # class 4 absent everywhere -> NaN IoU
    return c


def _gloo_worker(rank, world, port, out):
    import torch.distributed as dist

    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), PINMEM_B200_DEVICE="cpu")
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        from pinthememory_b200 import sharding
        from pinthememory_b200.callers import SegMetrics

        sm = SegMetrics(5, group=sharding.ShardGroup())
        sm.confusion += _hand_confusion(rank)
        conf, iou, miou = sm.finalize()
        out[rank] = dict(conf=conf, iou=iou, miou=miou, local=sm.confusion.clone())
    finally:
        dist.destroy_process_group()


def test_finalize_reduces_over_the_group_gloo():
    import torch.multiprocessing as mp

    world = 2
    mgr = mp.get_context("spawn").Manager()
    out = mgr.dict()
    mp.spawn(_gloo_worker, args=(world, _free_port(), out), nprocs=world, join=True)
    total = _hand_confusion(0) + _hand_confusion(1)
    c = total.double()
    iou = c.diagonal() / (c.sum(0) + c.sum(1) - c.diagonal())
    for r in range(world):
        assert torch.equal(out[r]["conf"], total)
        assert torch.equal(out[r]["local"], _hand_confusion(r)), "finalize must not modify the local matrix"
        assert torch.isnan(out[r]["iou"][4]) and torch.allclose(out[r]["iou"][:4], iou[:4], rtol=0, atol=1e-15)
        assert abs(float(out[r]["miou"]) - float(iou[:4].mean())) < 1e-15
    assert torch.equal(out[0]["iou"].nan_to_num(-1), out[1]["iou"].nan_to_num(-1))


def test_rejects_cpu_tensors_and_bad_class_counts():
    from pinthememory_b200.callers import SegMetrics

    with pytest.raises(RuntimeError):
        SegMetrics(0, device="cpu")
    with pytest.raises(RuntimeError):
        SegMetrics(32, device="cpu")
    sm = SegMetrics(4, device="cpu")
    with pytest.raises(RuntimeError, match="no CPU path"):
        sm.add(torch.zeros(1, 4, 2, 2), torch.zeros(1, 4, 4, dtype=torch.int64))


# ----------------------------------------------------------------------------------------------------------------- GPU

DTYPES = [torch.float32, torch.bfloat16]


def _logits(B, K, h, w, seed, dtype, scale=3.0):
    from pinthememory_b200 import synth

    return (scale * synth.make_features(B, K, h, w, seed=seed, device="cuda")).to(dtype)


def _check(logits, labels, K, loss, pred, conf_delta, exact=False, tag=""):
    """pred vs torch's argmax (differences only at rounding-level top-2 gaps), the confusion increment vs fast_hist of
    the kernel's own pred, the loss vs the fp64 oracle and the fused training loss. Returns the number of differing
    pixels."""

    x = logits.float()
    size = labels.shape[-2:]
    conf_t, pred_t, _ = segmentation_confusion(x, labels, K)
    diff = pred.long() != pred_t
    n = int(diff.sum())
    if exact:
        assert n == 0, (tag, n)
        assert torch.equal(conf_delta, conf_t), tag
    else:
        gap = top2_gap(x, size)
        tol = 2e-6 * float(upsample_logits(x, size).abs().max())
        assert bool((gap[diff] <= tol).all()), (tag, "argmax differs away from a near-tie")
        assert n <= 1e-5 * pred.numel(), (tag, n)
    assert torch.equal(conf_delta, fast_hist(pred.long(), labels.long(), K)), tag
    _, _, loss64 = segmentation_confusion(x.double(), labels, K)
    if torch.isnan(loss64):
        assert torch.isnan(loss), tag
    else:
        assert abs(float(loss) - float(loss64)) <= 1e-5 * abs(float(loss64)) + 1e-7, (tag, float(loss), float(loss64))
    return n


def _run(logits, labels, K, exact=False, tag=""):
    from pinthememory_b200.callers import SegMetrics

    sm = SegMetrics(K)
    loss, pred = sm.add(logits, labels, predictions=True)
    n = _check(logits, labels, K, loss, pred, sm.confusion, exact=exact, tag=tag)
    return sm, loss, pred, n


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", DTYPES)
def test_identity_mode_is_bit_exact(dtype):
    from pinthememory_b200 import synth

    B, K, H, W = 2, K19, 96, 160
    x = _logits(B, K, H, W, 11, dtype)
    lab = synth.make_labels(B, H, W, K, "blocky", seed=12, device="cuda", block=8)
    sm, loss, pred, _ = _run(x, lab, K, exact=True, tag="identity")
    assert torch.equal(pred.long(), x.argmax(1))
    m = (lab >= 0) & (lab < K)
    want = torch.bincount(K * lab[m] + x.argmax(1)[m], minlength=K * K).view(K, K)
    assert torch.equal(sm.confusion, want)


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", DTYPES)
def test_upsampling_with_exact_arithmetic_is_bit_exact(dtype):
    """(Hm-1) = 4(h-1) and logits on a 1/64 grid: every interpolated value is exact, ties included (first class wins)."""
    from pinthememory_b200 import synth

    B, K, h, w = 2, K19, 17, 25
    Hm, Wm = 4 * (h - 1) + 1, 4 * (w - 1) + 1
    g = torch.Generator().manual_seed(13)
    x = (torch.randint(-256, 257, (B, K, h, w), generator=g).float() / 64).to(device="cuda", dtype=dtype)
    lab = synth.make_labels(B, Hm, Wm, K, "iid", seed=14, device="cuda")
    _run(x, lab, K, exact=True, tag="exact")


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("kind", ["blocky", "iid"])
@pytest.mark.parametrize("shape", [(1, 256, 512, 1024, 2048), (2, 192, 192, 768, 768)], ids=["cityscapes_val", "crop"])
def test_full_size(shape, kind, dtype):
    from pinthememory_b200 import synth
    from pinthememory_b200.callers import upsampled_cross_entropy

    B, h, w, Hm, Wm = shape
    x = _logits(B, K19, h, w, 15, dtype)
    lab = synth.make_labels(B, Hm, Wm, K19, kind, seed=16, device="cuda")
    _, loss, _, n = _run(x, lab, K19, tag=f"{shape} {kind} {dtype}")
    print(f"pred differs from torch at {n} of {B * Hm * Wm} pixels")
    ref = upsampled_cross_entropy(x.float(), lab)
    assert abs(float(loss) - float(ref)) <= 1e-5 * abs(float(ref))


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("K,B,h,w,Hm,Wm", [
    (1, 2, 9, 11, 33, 41),
    (31, 2, 9, 11, 33, 41),
    (5, 2, 1, 13, 7, 50),
    (5, 2, 13, 1, 50, 7),
    (5, 2, 1, 1, 1, 9),
    (5, 2, 1, 9, 1, 40),
    (5, 2, 9, 1, 40, 1),
    (K19, 1, 97, 131, 389, 521),
    (K19, 2, 97, 131, 97, 521),   # equal heights, up-sampled widths
    (27, 1, 40, 40, 41, 43),      # ratio ~1: the largest shared-memory footprint
    (31, 1, 40, 40, 41, 43),
])
def test_edge_shapes(K, B, h, w, Hm, Wm, dtype):
    from pinthememory_b200 import synth

    x = _logits(B, K, h, w, 17, dtype)
    # (iid maps ignore their top 1/16 of rows: all of a one-row map)
    lab = synth.make_labels(B, Hm, Wm, K, "iid" if Hm > 1 else "blocky", seed=18, device="cuda", block=3)
    _run(x, lab, K, tag=f"K={K} {h}x{w}->{Hm}x{Wm}")


@pytest.mark.gpu
def test_uint8_labels_equal_int64_and_bad_labels_are_counted():
    from pinthememory_b200 import synth
    from pinthememory_b200.callers import SegMetrics

    B, K, h, w, Hm, Wm = 2, K19, 24, 32, 96, 128
    x = _logits(B, K, h, w, 19, torch.float32)
    lab = synth.make_labels(B, Hm, Wm, K, "blocky", seed=20, device="cuda", block=8)
    lab[0, 5, :7] = 19          # == K: bad
    lab[1, 9, :3] = 200         # bad
    lab[1, 10, :4] = 255        # ignore, not bad
    a, b = SegMetrics(K), SegMetrics(K)
    la, pa = a.add(x, lab, predictions=True)
    lb, pb = b.add(x, lab.to(torch.uint8), predictions=True)
    assert torch.equal(a.confusion, b.confusion) and torch.equal(pa, pb) and torch.equal(la, lb)
    assert int(a.last_bad_labels) == 10 and int(b.last_bad_labels) == 10
    _check(x, lab, K, la, pa, a.confusion, tag="bad labels")
    neg = lab.clone()
    neg[0, 0, :6] = -3          # negative int64: excluded and counted
    c = SegMetrics(K)
    lc, pc = c.add(x, neg, predictions=True)
    assert int(c.last_bad_labels) == 16
    _check(x, neg, K, lc, pc, c.confusion, tag="negative labels")


@pytest.mark.gpu
def test_all_ignore_batch_leaves_confusion_and_gives_nan():
    from pinthememory_b200.callers import SegMetrics

    K = K19
    x = _logits(1, K, 8, 8, 21, torch.float32)
    sm = SegMetrics(K)
    sm.add(x, torch.randint(0, K, (1, 32, 32), device="cuda"))
    before = sm.confusion.clone()
    loss = sm.add(x, torch.full((1, 32, 32), 255, dtype=torch.int64, device="cuda"))
    assert torch.isnan(loss) and torch.equal(sm.confusion, before) and int(sm.last_bad_labels) == 0


@pytest.mark.gpu
def test_rejections():
    from pinthememory_b200.callers import SegMetrics

    sm = SegMetrics(K19)
    x = _logits(1, K19, 16, 16, 22, torch.float32)
    with pytest.raises(RuntimeError, match="at least"):
        sm.add(x, torch.zeros(1, 8, 32, dtype=torch.int64, device="cuda"))
    with pytest.raises(RuntimeError):
        sm.add(x.half(), torch.zeros(1, 16, 16, dtype=torch.int64, device="cuda"))
    with pytest.raises(RuntimeError):
        sm.add(x[:, :5], torch.zeros(1, 16, 16, dtype=torch.int64, device="cuda"))
    with pytest.raises(RuntimeError):
        sm.add(x, torch.zeros(1, 16, 16, dtype=torch.int32, device="cuda"))
    with pytest.raises(RuntimeError):
        sm.add(x, torch.zeros(2, 16, 16, dtype=torch.int64, device="cuda"))
    assert int(sm.confusion.sum()) == 0
    if torch.cuda.device_count() < 2:
        pytest.skip("one GPU: the cross-device rejection needs two")
    with pytest.raises(RuntimeError):
        sm.add(x.to("cuda:1"), torch.zeros(1, 16, 16, dtype=torch.int64, device="cuda:1"))


@pytest.mark.gpu
def test_two_adds_equal_one_add_of_the_concatenated_batch():
    from pinthememory_b200 import synth
    from pinthememory_b200.callers import SegMetrics

    x = _logits(4, K19, 24, 24, 23, torch.float32)
    lab = synth.make_labels(4, 96, 96, K19, "iid", seed=24, device="cuda")
    one, two = SegMetrics(K19), SegMetrics(K19)
    one.add(x, lab)
    two.add(x[:2], lab[:2])
    two.add(x[2:], lab[2:])
    assert torch.equal(one.confusion, two.confusion)
    c1, iou1, m1 = one.finalize()
    c2, iou2, m2 = two.finalize()
    assert torch.equal(c1, c2) and torch.equal(iou1.nan_to_num(-1), iou2.nan_to_num(-1)) and torch.equal(m1, m2)


@pytest.mark.gpu
def test_cuda_graph_replay_equals_eager():
    from pinthememory_b200 import synth
    from pinthememory_b200.callers import SegMetrics

    x = _logits(2, K19, 24, 32, 25, torch.float32)
    lab = synth.make_labels(2, 96, 128, K19, "blocky", seed=26, device="cuda", block=8)
    eager = SegMetrics(K19)
    le, pe = eager.add(x, lab, predictions=True)
    eager.add(x, lab)
    graphed = SegMetrics(K19)
    graphed.add(x, lab)             # warm-up outside the capture (module load)
    graphed.reset()
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        lg, pg = graphed.add(x, lab, predictions=True)
    g.replay()
    g.replay()
    torch.cuda.synchronize()
    assert torch.equal(graphed.confusion, eager.confusion)
    assert torch.equal(lg, le) and torch.equal(pg, pe)


def _nccl_worker(rank, world, port, out):
    import torch.distributed as dist

    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    torch.cuda.set_device(rank)
    dev = torch.device("cuda", rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=dev)
    try:
        from pinthememory_b200 import sharding, synth
        from pinthememory_b200.callers import SegMetrics

        x = (3.0 * synth.make_features(4, K19, 24, 24, seed=27)).to(dev)
        lab = synth.make_labels(4, 96, 96, K19, "iid", seed=28, device=dev)
        sm = SegMetrics(K19, device=dev, group=sharding.ShardGroup())
        sm.add(x[2 * rank: 2 * rank + 2], lab[2 * rank: 2 * rank + 2])
        conf, iou, miou = sm.finalize()
        out[rank] = dict(conf=conf.cpu(), iou=iou.cpu(), miou=float(miou))
    finally:
        dist.destroy_process_group()


@pytest.mark.gpu
def test_two_gpu_finalize_equals_single_process():
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    import torch.multiprocessing as mp

    from pinthememory_b200 import synth
    from pinthememory_b200.callers import SegMetrics

    mgr = mp.get_context("spawn").Manager()
    out = mgr.dict()
    mp.spawn(_nccl_worker, args=(2, _free_port(), out), nprocs=2, join=True)
    x = (3.0 * synth.make_features(4, K19, 24, 24, seed=27)).cuda()
    lab = synth.make_labels(4, 96, 96, K19, "iid", seed=28, device="cuda")
    sm = SegMetrics(K19)
    sm.add(x, lab)
    conf, iou, miou = sm.finalize()
    for r in range(2):
        assert torch.equal(out[r]["conf"], conf.cpu())
        assert torch.equal(out[r]["iou"].nan_to_num(-1), iou.cpu().nan_to_num(-1))
    assert out[0]["miou"] == out[1]["miou"] == float(miou)
