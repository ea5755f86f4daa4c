"""The read-loss kernels against a float64 torch restatement of memory.py:173-176. `pm_readloss_fwd8` runs the cells kernel
(a lane pair per cell) when the label map is at least 3x the feature map and the one-thread-per-cell kernel otherwise, or
when the cells are too large for the cells kernel's fixed-point one-hot tile; `capi.readloss` runs the first kernel
(int64 labels) for K > 19. Every kernel is reached through the shapes that select it, and the shapes cover their edge
handling: ragged maps, non-integer label/feature ratios, few slots, ignore labels, tiny temperatures (the exact per-pixel
path) and small grids (the row split of the cells kernel)."""
import pytest
import torch
import torch.nn.functional as F

pytestmark = pytest.mark.gpu

# B, h, w, Hm, Wm, K, T, ignore share
CELLS_CASES = [
    (2, 24, 24, 192, 192, 19, 1.0, 0.1),     # ratio 8, the cfg-2 geometry
    (1, 12, 37, 97, 300, 19, 1.0, 0.2),      # ragged, non-integer ratios (8.7 / 8.3)
    (2, 16, 16, 256, 256, 19, 1.0, 0.0),     # ratio 17: small grid -> row split
    (1, 33, 18, 100, 55, 5, 0.5, 0.3),       # ratio 3.1 / 3.2, five slots
    (2, 20, 28, 160, 224, 19, 0.02, 0.1),    # tiny temperature: per-pixel maximum path
    (1, 9, 9, 72, 72, 1, 1.0, 0.5),          # one slot
    (1, 8, 40, 64, 320, 19, 1.0, 1.0),       # every label ignored: loss = 0/0 = NaN like torch, zero gradient
]
CELL_THREAD_CASES = [
    (2, 24, 24, 48, 48, 19, 1.0, 0.1),       # ratio 2
    (1, 12, 37, 29, 90, 19, 1.0, 0.2),       # ragged, ratio about 2.5
    (2, 16, 16, 16, 16, 19, 1.0, 0.1),       # identity
    (1, 10, 1, 40, 7, 19, 1.0, 0.1),         # w == 1: one feature column
    (1, 2, 2, 300, 300, 19, 1.0, 0.1),       # cells too large for the cells kernel's fixed-point tile
    (2, 20, 28, 40, 56, 19, 0.02, 0.1),      # tiny temperature
    (1, 8, 40, 16, 80, 19, 1.0, 1.0),        # every label ignored
]
FIRST_CASES = [
    (1, 12, 20, 96, 160, 25, 1.0, 0.1),      # K > 19: int64 labels, 32-float rows
]
KERNEL = {"cells": "readloss_cells_kernel", "cell_thread": "readloss8_kernel", "first": "readloss_kernel"}
ROUTES = [(c, "cells") for c in CELLS_CASES] + [(c, "cell_thread") for c in CELL_THREAD_CASES] + \
         [(c, "first") for c in FIRST_CASES]


def _reference(s, labels, T, B, h, w, K):
    z = (s[:, :K].double().view(B, h, w, K).permute(0, 3, 1, 2) / T).requires_grad_(True)
    up = F.interpolate(z, size=labels.shape[1:], mode="bilinear", align_corners=True)
    lab = labels.clone()
    loss_sum = F.cross_entropy(up, lab, ignore_index=255, reduction="sum")
    V = int((lab != 255).sum())
    (g,) = torch.autograd.grad(loss_sum, z)
    # d(loss_sum)/d(s/T) in the kernels' [N, KP] layout
    return (loss_sum / V if V else torch.tensor(float("nan"))), g.permute(0, 2, 3, 1).reshape(B * h * w, K), V


def _inputs(case, dev="cuda"):
    from pinthememory_b200 import capi

    B, h, w, Hm, Wm, K, T, ign = case
    KP = capi.score_stride(K)
    g = torch.Generator(device="cpu").manual_seed(hash(case) % (2 ** 31))
    N = B * h * w
    s = torch.zeros(N, KP, device=dev)
    s[:, :K] = (torch.rand(N, K, generator=g) * 2 - 1).to(dev)
    labels = torch.randint(0, K, (B, Hm, Wm), generator=g)
    # piecewise-constant regions with some ignore
    blocks = torch.randint(0, K, (B, (Hm + 15) // 16, (Wm + 15) // 16), generator=g)
    labels = torch.where(torch.rand(B, Hm, Wm, generator=g) < 0.5,
                         blocks.repeat_interleave(16, 1).repeat_interleave(16, 2)[:, :Hm, :Wm], labels)
    labels[torch.rand(B, Hm, Wm, generator=g) < ign] = 255
    return s, labels.to(dev)


def _run(case, s, labels):
    """The read loss as the module runs it: label pack + pm_readloss_fwd8 for K <= 19, pm_readloss_fwd above."""
    from pinthememory_b200 import capi

    B, h, w, Hm, Wm, K, T, ign = case
    N, KP = s.shape
    buf = torch.zeros(N * KP + 2 * capi.WS_WORDS + 4, dtype=torch.float32, device=s.device)
    ds, ws, out = buf[: N * KP], buf[N * KP: N * KP + 2 * capi.WS_WORDS], buf[N * KP + 2 * capi.WS_WORDS:]
    capi.readloss(s, labels, T, B, h, w, K, ds, ws, out)
    return ds.view(N, KP), out


@pytest.mark.parametrize("case,route", ROUTES)
def test_readloss_kernel_matches_reference(case, route):
    B, h, w, Hm, Wm, K, T, ign = case
    s, labels = _inputs(case)
    ref_loss, ref_g, V = _reference(s, labels, T, B, h, w, K)
    ds, out = _run(case, s, labels)
    torch.cuda.synchronize()
    loss, dsg = out[0].item(), ds[:, :K].double()
    assert ds[:, K:].abs().max().item() == 0.0, "padded slots received gradient"
    if V == 0:
        assert loss != loss and dsg.abs().max().item() == 0.0
        return
    # the gradient is the difference of two sums of ~(Hm/h)*(Wm/w) bilinear weights per feature pixel (softmax part minus
    # one-hot part): with one slot it is exactly zero in the reference, so the error is measured against that natural scale
    area = (Hm / h) * (Wm / w)
    scale = max(ref_g.abs().max().item(), area)
    assert abs(loss - ref_loss.item()) <= 1e-5 * max(1.0, abs(ref_loss.item())), (loss, ref_loss.item())
    err = (dsg - ref_g).abs().max().item() / scale                # max-abs over max(|ref|, weights per feature pixel)
    rel = ((dsg - ref_g).norm() / max(ref_g.norm().item(), area)).item()   # relative L2
    assert err <= 1e-5 and rel <= 1e-5, (err, rel)


def test_readloss_routing():
    """Each shape class launches the read-loss kernel that serves it, and only that one."""
    from torch.profiler import ProfilerActivity, profile

    runs = []
    for case, route in ROUTES:
        s, labels = _inputs(case)
        torch.cuda.synchronize()
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            _run(case, s, labels)
            torch.cuda.synchronize()
        names = [e.name for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA]
        # (no kernel name is a substring of another)
        launched = {k for k, kern in KERNEL.items() if any(kern in n for n in names)}
        runs.append((case, route, launched))
    assert all(launched == {route} for case, route, launched in runs), \
        [(case, route, launched) for case, route, launched in runs if launched != {route}]
