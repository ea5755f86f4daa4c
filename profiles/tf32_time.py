"""What one-pass TF32 (torch's TF32 switches on, capi.tf32) buys against the default 3xTF32 GEMMs.

    python profiles/tf32_time.py [--seconds 1.0] [--rounds 5] [--out profiles/tf32_time_b200.json]

GEMM forms at BASELINE config 2 (B=8, 96x96, the folded output convolution 288 -> 256 and its gradients, the writing
net's 256 -> 256), each 3-pass (PM_F32) and one-pass (PM_F32_TF32), next to cuDNN with TF32 on for the same product:
  fwd_288_256          pm_conv1x1_fwd with the BatchNorm statistics in its epilogue   | F.conv2d
  dgrad_bnbwd_256_288  pm_conv1x1_dgrad_bnbwd (input gradient + BatchNorm backward)   | convolution_backward (input)
  dgrad_256_288        pm_conv1x1_fwd on W^T (input gradient alone)                   | convolution_backward (input)
  wgrad_256_288        pm_conv1x1_wgrad (+ its reduce kernel)                         | convolution_backward (weight)
  fwd_256_256          the writing net's forward GEMM                                 | F.conv2d
Module step: the cfg-2 fp32 training step (read + write, forward + backward, two-stream mode) captured as a CUDA graph
once per mode (GraphedStep fixes the mode at capture) and replayed; the two graphs are timed alternately, --rounds
windows each, so drift on the shared machine lands on both. Every figure is CUDA-event time over a window of at least
--seconds divided by the calls in it, after a warm-up. Prints one JSON line and writes it to --out.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys

import torch
import torch.nn.functional as F

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

from pinthememory_b200 import capi, synth  # noqa: E402
from pinthememory_b200.graphed import GraphedStep  # noqa: E402
from pinthememory_b200.memory import Memory_sup  # noqa: E402


def gpu_info():
    info = {"name": torch.cuda.get_device_name(0), "power_limit_w": None}
    try:
        r = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader,nounits", "-i", "0"],
                           capture_output=True, text=True, timeout=30)
        info["power_limit_w"] = float(r.stdout.strip().splitlines()[0])
    except Exception as e:  # noqa: BLE001
        info["power_limit_error"] = repr(e)[:200]
    return info


def set_tf32(on):
    torch.backends.cuda.matmul.allow_tf32 = on
    torch.backends.cudnn.allow_tf32 = on


def timed(fn, seconds):
    """Mean time per call (us) over a window of at least `seconds`, CUDA events around the whole window."""
    for _ in range(3):
        fn()
    torch.cuda.synchronize()
    n = 1
    while True:
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for _ in range(n):
            fn()
        b.record()
        b.synchronize()
        ms = a.elapsed_time(b)
        if ms >= 1000.0 * seconds:
            return 1000.0 * ms / n
        n = max(n * 2, int(n * 1.2 * 1000.0 * seconds / max(ms, 1e-3)))


def gemm_forms(seconds):
    B, hw, C, Cin = 8, 96 * 96, 256, 256 + capi.PLANES
    g = torch.Generator(device="cuda").manual_seed(3)
    x = torch.randn(B, Cin, 96, 96, generator=g, device="cuda")
    xw = torch.randn(B, C, 96, 96, generator=g, device="cuda")
    dy = torch.randn(B, C, 96, 96, generator=g, device="cuda")
    z = torch.randn(B, C, 96, 96, generator=g, device="cuda")
    W = torch.randn(C, Cin, generator=g, device="cuda") * 0.05
    Ww = torch.randn(C, C, generator=g, device="cuda") * 0.05
    v = torch.rand(C, generator=g, device="cuda") + 0.5
    stats = torch.zeros(2 * C, dtype=torch.float64, device="cuda")
    out = {}
    for tf32 in (False, True):
        (hi, lo), (hiT, loT) = capi.conv1x1_prep_both(W, torch.float32, tf32=tf32)
        (hw_, lw_), _ = capi.conv1x1_prep_both(Ww, torch.float32, tf32=tf32)
        key = "one_pass" if tf32 else "three_pass"
        out.setdefault("fwd_288_256", {})[key] = timed(lambda: capi.conv1x1_fwd(x, hi, lo, C, stats=stats), seconds)
        out.setdefault("dgrad_bnbwd_256_288", {})[key] = timed(
            lambda: capi.conv1x1_dgrad_bnbwd(dy, z, hiT, loT, Cin, v, v, v, v, v, v, True, True), seconds)
        out.setdefault("dgrad_256_288", {})[key] = timed(lambda: capi.conv1x1_fwd(dy, hiT, loT, Cin), seconds)
        out.setdefault("wgrad_256_288", {})[key] = timed(lambda: capi.conv1x1_wgrad(dy, x, tf32=tf32), seconds)
        out.setdefault("fwd_256_256", {})[key] = timed(lambda: capi.conv1x1_fwd(xw, hw_, lw_, C, stats=stats), seconds)
    set_tf32(True)
    W4, Ww4 = W.view(C, Cin, 1, 1), Ww.view(C, C, 1, 1)
    cb = torch.ops.aten.convolution_backward
    args = ([1, 1], [0, 0], [1, 1], False, [0, 0], 1)
    out["fwd_288_256"]["cudnn_tf32"] = timed(lambda: F.conv2d(x, W4), seconds)
    out["dgrad_bnbwd_256_288"]["cudnn_tf32"] = out["dgrad_256_288"]["cudnn_tf32"] = timed(
        lambda: cb(dy, x, W4, None, *args, [True, False, False]), seconds)
    out["wgrad_256_288"]["cudnn_tf32"] = timed(lambda: cb(dy, x, W4, None, *args, [False, True, False]), seconds)
    out["fwd_256_256"]["cudnn_tf32"] = timed(lambda: F.conv2d(xw, Ww4), seconds)
    set_tf32(False)
    return {k: {m: round(t, 1) for m, t in d.items()} for k, d in out.items()}


def module_step(seconds, rounds):
    B, C, h, w, Hm, Wm, K = 8, 256, 96, 96, 768, 768, 19
    x = synth.make_features(B, C, h, w, seed=1, device="cuda")
    lab = synth.make_labels(B, Hm, Wm, K, "blocky", seed=2, device="cuda")
    G = synth.make_upstream_grad((B, C, h, w), seed=3, device="cuda")
    steps = {}
    for tf32 in (False, True):
        set_tf32(tf32)
        torch.manual_seed(5)
        m = Memory_sup(K, C, C, 0.8, 1.0, False).cuda()
        m.overlap_write = True
        steps[tf32] = GraphedStep(m, x, lab, G, loss_weights=(0.02, 0.4, 0.2), memory_writing=True, writing_detach=False)
    set_tf32(False)
    times = {False: [], True: []}
    try:
        for _ in range(rounds):
            for tf32 in (False, True):
                times[tf32].append(timed(lambda: steps[tf32](x, lab, G), seconds))
    finally:
        for s in steps.values():
            s.release()
    med = {k: statistics.median(v) for k, v in times.items()}
    return {"three_pass_us": [round(t, 1) for t in times[False]], "one_pass_us": [round(t, 1) for t in times[True]],
            "three_pass_median_us": round(med[False], 1), "one_pass_median_us": round(med[True], 1),
            "one_pass_gain": round(1.0 - med[True] / med[False], 4)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--seconds", type=float, default=1.0)
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "tf32_time_b200.json"))
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("tf32_time.py needs a CUDA device")
    set_tf32(False)
    res = {"gpu": gpu_info(), "window_s": args.seconds, "gemm_us": gemm_forms(args.seconds),
           "cfg2_fp32_graph_step": module_step(args.seconds, args.rounds)}
    line = json.dumps(res)
    print(line)
    if args.out:
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
