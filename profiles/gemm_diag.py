"""Diagnostic: where are the wrong elements of conv1x1_fwd for a given shape? (bring-up tool)"""
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
from pinthememory_b200 import capi

dev = "cuda"


def diag(B, K, M, h, w, transpose, reps=3, pre=None):
    hw = h * w
    torch.manual_seed(1)
    x = torch.randn(B, K, h, w, device=dev)
    W = torch.randn((K, M) if transpose else (M, K), device=dev) / K ** 0.5
    Wm = W.t() if transpose else W
    ref = torch.einsum("mk,bkp->bmp", Wm.double(), x.double().view(B, K, hw))
    for r in range(reps):
        if pre is not None:
            pre()
        hi, lo = capi.conv1x1_prep(W, transpose, torch.float32)
        y = torch.full((B, M, h, w), float("nan"), device=dev)
        capi.conv1x1_fwd(x, hi, lo, M, y=y)
        torch.cuda.synchronize()
        err = (y.view(B, M, hw).double() - ref).abs()
        bad = ~(err <= 1e-4 * ref.abs().max())
        n = int(bad.sum())
        print(f"B={B} K={K} M={M} hw={hw} T={int(transpose)} rep {r}: bad={n} nan={int(torch.isnan(y).sum())}", flush=True)
        if n:
            idx = bad.nonzero()
            bs, ms, ps = idx[:, 0], idx[:, 1], idx[:, 2]
            print("  images", sorted(set(bs.tolist()))[:10], "row blocks(32)", sorted(set((ms // 32).tolist()))[:16],
                  "px blocks(32)", sorted(set((ps // 32).tolist()))[:40])
            tiles = sorted(set((bs * ((hw + 127) // 128) + ps // 128).tolist()))
            print("  tiles", tiles[:40], "of", B * ((hw + 127) // 128))


def noise():
    a = torch.randn(8, 256, 48, 48, device=dev)
    b = torch.randn(8, 256, 48, 48, device=dev)
    capi.conv1x1_wgrad(a, b)


diag(8, 256, 256, 48, 48, False)
diag(8, 256, 256, 48, 48, True)
diag(8, 256, 256, 48, 48, True, pre=noise)
diag(8, 288, 256, 96, 96, False)
diag(8, 256, 288, 96, 96, True, pre=noise)
diag(4, 64, 64, 12, 20, True, pre=None)
