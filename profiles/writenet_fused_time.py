"""The writing net's element-wise chain, separate passes against the fused ones, timed launch by launch with CUDA events.

separate (Writingnet + _WriteFn): pm_bn_apply_stats (f and its ReLU mask) -> pm_write_reduce_fwd8 -> pm_write_bwd8 ->
    pm_bn_bwd_reduce_rows -> pm_bn_bwd_apply (dz and the residual gradient)
fused (_WriteNetFn): pm_write_reduce_bn_fwd -> pm_write_bwd_bn (g, dgamma / dbeta) -> pm_bn_bwd_apply (dz)

Feature maps are B x 256 x 96 x 96 fp32 with B = 24 by default (226 MB per map, above the 126 MB L2), K = 19, packed
labels as the module step uses them. MB are the algorithmic feature-map bytes of each launch (labels and per-channel
vectors left out); GB/s = MB / time.

    python profiles/writenet_fused_time.py [--batch 24] [--hw 96 96] [--reps 20] [--out FILE]
"""
import argparse
import json
import subprocess
import sys

import torch

sys.path.insert(0, __import__("os").path.dirname(__import__("os").path.dirname(__import__("os").path.abspath(__file__))))
from pinthememory_b200 import capi, synth  # noqa: E402


def card():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip().splitlines()
        return out[torch.cuda.current_device()] if out else "unknown"
    except Exception as e:  # noqa: BLE001
        return "unknown (%s)" % e


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batch", type=int, default=24)
    ap.add_argument("--hw", type=int, nargs=2, default=(96, 96), metavar=("H", "W"))
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    (h, w), C, Hm, Wm, K = args.hw, 256, 768, 768, 19
    B = args.batch
    dev = torch.device("cuda")
    g = torch.Generator(device="cuda").manual_seed(1)
    z = torch.randn(B, C, h, w, device=dev, generator=g) * 2 + 0.3
    x = torch.randn(B, C, h, w, device=dev, generator=g)
    lab8 = synth.make_labels(B, Hm, Wm, K, "blocky", seed=2, device=dev).to(torch.uint8)
    gamma = torch.rand(C, device=dev, generator=g) + 0.5
    beta = torch.randn(C, device=dev, generator=g) * 0.3
    z64 = z.double()
    stats = torch.cat([z64.sum((0, 2, 3)), (z64 * z64).sum((0, 2, 3)), torch.zeros(1, device=dev, dtype=torch.float64)])
    del z64
    n = B * h * w
    rm, rv = torch.zeros(C, device=dev), torch.ones(C, device=dev)
    mean, invstd = torch.empty(C, device=dev), torch.empty(C, device=dev)
    dS = torch.randn(K, C, device=dev, generator=g) * 0.1
    SD = torch.zeros(K + 1, C + 4, device=dev)
    dgamma, dbeta = torch.empty(C, device=dev), torch.empty(C, device=dev)
    f, df, dz, dres = (torch.empty_like(z) for _ in range(4))
    mask = torch.empty(capi.bn_mask_words(B, C, h * w), dtype=torch.int32, device=dev)
    N = z.numel() * 4 / 1e6          # MB of one feature map
    Mk = mask.numel() * 4 / 1e6       # MB of the ReLU mask

    separate = [
        ("pm_bn_apply_stats", 3 * N + Mk, lambda: capi.bn_apply_stats(z, stats, n, 1e-5, gamma, beta, x, f, True, mean, invstd,
                                                                       rm, rv, 0.1, relu_mask=mask)),
        ("pm_write_reduce_fwd8", N, lambda: capi.write_reduce_fwd(f, lab8, SD, K)),
        ("pm_write_bwd8", 2 * N, lambda: capi.write_bwd(dS, f, lab8, df, K)),
        ("pm_bn_bwd_reduce_rows", 2 * N + Mk, lambda: capi.bn_bwd_reduce(df, None, mask, z, mean, invstd, True, dgamma, dbeta)),
        ("pm_bn_bwd_apply", 4 * N + Mk, lambda: capi.bn_bwd_apply(df, None, mask, z, mean, invstd, gamma, dgamma, dbeta, True, True,
                                                                 dz, dres)),
    ]
    fused = [
        ("pm_write_reduce_bn_fwd", 2 * N, lambda: capi.write_reduce_bn_fwd(z, x, lab8, SD, K, stats, n, 1e-5, gamma, beta, mean,
                                                                           invstd, rm, rv, 0.1)),
        ("pm_write_bwd_bn", 3 * N, lambda: capi.write_bwd_bn(dS, z, x, lab8, mean, invstd, gamma, beta, dres, dgamma, dbeta, K)),
        ("pm_bn_bwd_apply", 3 * N, lambda: capi.bn_bwd_apply(dres, None, None, z, mean, invstd, gamma, dgamma, dbeta, False, True,
                                                            dz, None)),
    ]

    def run(chain):
        for _ in range(3):
            for _, _, fn in chain:
                fn()
        torch.cuda.synchronize()
        ev = [[(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in chain]
              for _ in range(args.reps)]
        for r in range(args.reps):
            for (a, b), (_, _, fn) in zip(ev[r], chain):
                a.record()
                fn()
                b.record()
        torch.cuda.synchronize()
        rows = []
        for i, (name, mb, _) in enumerate(chain):
            ts = sorted(ev[r][i][0].elapsed_time(ev[r][i][1]) * 1e3 for r in range(args.reps))
            us = ts[len(ts) // 2]
            rows.append({"launch": name, "us_median": round(us, 1), "MB": round(mb, 1), "GB_per_s": round(mb / us * 1e3)})
        return {"launches": rows, "us_total": round(sum(r["us_median"] for r in rows), 1),
                "MB_total": round(sum(r["MB"] for r in rows), 1)}

    res = {"card": card(), "shape": {"B": B, "C": C, "h": h, "w": w, "K": K, "labels": "packed uint8, 768x768"},
           "reps": args.reps, "timing": "CUDA events around each launch, median over reps; inputs above L2",
           "separate": run(separate), "fused": run(fused)}
    # alternate once more so that neither chain is measured only first
    res["separate_again"] = run(separate)
    line = json.dumps(res, indent=1)
    print(line)
    if args.out:
        with open(args.out, "w") as fh:
            fh.write(line + "\n")


if __name__ == "__main__":
    main()
