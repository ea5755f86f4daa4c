"""Cost of torch.use_deterministic_algorithms(True) for the module: the ordered entries (per-CTA partials added in a fixed
order, readloss8_kernel instead of the cells kernel) and torch's NaN fill of uninitialised allocations.

    python profiles/deterministic_time.py [--seconds 1.0] [--out profiles/deterministic_time_b200.json]

Workloads:
  cfg2_fp32 / cfg2_bf16  the module's training step (read + write, forward + backward) at B=8, 96x96, C=256, K=19,
                         768x768 blocky int64 labels, captured once as a CUDA graph (GraphedStep) and replayed
  cfg3_meta              the module's part of a meta-train step (pinthememory_b200/metastep.py) at B=4, 48x48, C=256,
                         K=19, 192x192 labels, launched eagerly (host overhead included, the same in every mode)
Modes: `off` (the default kernels), `on` (the flag set: ordered kernels and torch's NaN fill of `empty`), `on_nofill`
(the flag set with torch.utils.deterministic.fill_uninitialized_memory = False). GraphedStep fixes the choice at capture,
so each mode captures its own graph. Each figure is CUDA-event time over a window of at least --seconds, divided by the
number of steps in it, after a warm-up of every shape. Prints one JSON line and writes it to --out.
"""
import argparse
import json
import os
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

from pinthememory_b200 import synth  # noqa: E402
from pinthememory_b200.graphed import GraphedStep  # noqa: E402
from pinthememory_b200.memory import Memory_sup  # noqa: E402
from pinthememory_b200.metastep import meta_step  # noqa: E402

MODES = ("off", "on", "on_nofill")


def gpu_info():
    info = {"name": torch.cuda.get_device_name(0), "power_limit_w": None}
    try:
        r = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader,nounits", "-i", "0"],
                           capture_output=True, text=True, timeout=30)
        info["power_limit_w"] = float(r.stdout.strip().splitlines()[0])
    except Exception as e:  # noqa: BLE001
        info["power_limit_error"] = repr(e)[:200]
    return info


def set_mode(mode):
    torch.use_deterministic_algorithms(mode != "off")
    torch.utils.deterministic.fill_uninitialized_memory = mode != "on_nofill"


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


def module(K, C, dtype):
    torch.manual_seed(5)
    m = Memory_sup(K, C, C, 0.8, 1.0, False).cuda().to(dtype)
    m.m_items = m.m_items.float()
    return m


def cfg2(dtype, mode, seconds):
    B, C, h, w, Hm, Wm, K = 8, 256, 96, 96, 768, 768, 19
    set_mode(mode)
    m = module(K, C, dtype)
    m.overlap_write = True
    x = synth.make_features(B, C, h, w, seed=1, device="cuda").to(dtype)
    lab = synth.make_labels(B, Hm, Wm, K, "blocky", seed=2, device="cuda")
    G = synth.make_upstream_grad((B, C, h, w), seed=3, device="cuda").to(dtype)
    step = GraphedStep(m, x, lab, G, loss_weights=(0.02, 0.4, 0.2), memory_writing=True, writing_detach=False)
    try:
        return timed(lambda: step(x, lab, G), seconds)
    finally:
        step.release()


def cfg3_meta(mode, seconds):
    B, C, h, w, Hm, Wm, K = 4, 256, 48, 48, 192, 192, 19
    set_mode(mode)
    mods = [module(K, C, torch.float32) for _ in range(3)]
    x_tr = synth.make_features(B, C, h, w, seed=11, device="cuda")
    x_te = synth.make_features(B, C, h, w, seed=12, device="cuda")
    lab_tr = synth.make_labels(B, Hm, Wm, K, "blocky", seed=13, device="cuda", block=16)
    lab_te = synth.make_labels(B, Hm, Wm, K, "blocky", seed=14, device="cuda", block=16)
    G_tr = synth.make_upstream_grad((B, C, h, w), seed=15, device="cuda") / (B * h * w)
    G_te = synth.make_upstream_grad((B, C, h, w), seed=16, device="cuda") / (B * h * w)
    mem0 = mods[0].m_items.clone()

    def once():
        mods[0].m_items = mem0.clone()
        meta_step(*mods, x_tr, lab_tr, x_te, lab_te, G_tr, G_te, inner_lr=0.01)

    return timed(once, seconds)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--seconds", type=float, default=1.0)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "deterministic_time_b200.json"))
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("deterministic_time.py needs a CUDA device")
    torch.backends.cudnn.allow_tf32 = False
    torch.backends.cuda.matmul.allow_tf32 = False
    res = {"gpu": gpu_info(), "window_s": args.seconds, "us_per_step": {}}
    try:
        for mode in MODES:
            res["us_per_step"].setdefault("cfg2_fp32_graph", {})[mode] = round(cfg2(torch.float32, mode, args.seconds), 1)
            res["us_per_step"].setdefault("cfg2_bf16_graph", {})[mode] = round(cfg2(torch.bfloat16, mode, args.seconds), 1)
            res["us_per_step"].setdefault("cfg3_meta_eager", {})[mode] = round(cfg3_meta(mode, args.seconds), 1)
    finally:
        set_mode("off")
        torch.utils.deterministic.fill_uninitialized_memory = True
    line = json.dumps(res)
    print(line)
    if args.out:
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
