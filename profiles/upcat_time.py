"""Decoder up-sample + concat: the fused ``upsample_concat`` (pm_upcat_fwd / pm_upcat_bwd) against eager
``torch.cat([fine, F.interpolate(coarse, align_corners=True)], 1)`` and its autograd backward, on three workloads.
Prints one JSON line (and writes it to ``--out`` if given).

    python profiles/upcat_time.py [--reps 40] [--out upcat_time.json]

Workloads (Cf = 48 bot_fine channels, Cc = 256 memory-output channels, DeepLabV3+ decoder):
  a  reference crop, fp32: B=8, 48x48 -> 192x192
  b  the same in bf16
  c  validation image, fp32: B=1, 64x128 -> 256x512

Paths, each through autograd as a training step calls it (the backward returns both input gradients):
  fwd       forward only
  fwd_bwd   forward + backward with respect to both inputs
Times are CUDA events around CUDA-graph replays of the calls (device time; `*_graph_us`) and around eager calls
(`*_eager_us`, host overhead of the Python call included). Every repetition reads a different set of input buffers
from a rotation larger than the 126 MB L2, so inputs come from HBM. Algorithmic bytes of the fused path: forward =
read fine + coarse, write out; backward = read the gradient's coarse channels, write d_coarse. Those of the eager path
count each of its feature-sized passes (interpolate write; cat read + write; backward: slice copy read + write,
zero-fill, scatter read + atomic updates).
"""
import argparse
import json
import math
import os
import subprocess
import sys

import torch
import torch.nn.functional as F

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

from pinthememory_b200 import upsample_concat  # noqa: E402

L2_BYTES = 126 * 2 ** 20
CF, CC = 48, 256
WORKLOADS = {"a_crop_fp32": (8, 48, 48, 192, 192, torch.float32), "b_crop_bf16": (8, 48, 48, 192, 192, torch.bfloat16),
             "c_val_fp32": (1, 64, 128, 256, 512, torch.float32)}


def card():
    info = {"name": torch.cuda.get_device_name(0), "power_limit_w": None}
    try:   # read-only query
        r = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader,nounits", "-i", "0"],
                           capture_output=True, text=True, timeout=30)
        info["power_limit_w"] = float(r.stdout.strip().splitlines()[0])
    except Exception as e:  # noqa: BLE001
        info["power_limit_error"] = repr(e)[:200]
    return info


def eager_cat(fine, coarse):
    return torch.cat([fine, F.interpolate(coarse, size=fine.shape[-2:], mode="bilinear", align_corners=True)], 1)


def event_time_ms(fn, sets, reps):
    for s in sets:   # warm every shape and buffer
        fn(*s)
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for i in range(reps):
        fn(*sets[i % len(sets)])
    b.record()
    b.synchronize()
    return a.elapsed_time(b) / reps


def graph_time_ms(fn, sets, reps):
    """Per-call device time of ``fn``: one call per buffer set captured in a CUDA graph, replayed."""
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        for st in sets:
            fn(*st)
    torch.cuda.current_stream().wait_stream(side)
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        for st in sets:
            fn(*st)
    g.replay()
    torch.cuda.synchronize()
    n = max(1, reps // len(sets))
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(n):
        g.replay()
    b.record()
    b.synchronize()
    del g
    return a.elapsed_time(b) / (n * len(sets))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=40)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("upcat_time.py needs a CUDA device")
    dev = torch.device("cuda:0")
    res = {"what": "upcat_time", "Cf": CF, "Cc": CC, "card": card(),
           "inputs": "rotated buffers larger than the 126 MB L2 (HBM reads)", "workloads": {}}
    for name, (B, h, w, H, W, dt) in WORKLOADS.items():
        esz = torch.empty(0, dtype=dt).element_size()
        n_fine, n_coarse, n_up, n_out = B * CF * H * W, B * CC * h * w, B * CC * H * W, B * (CF + CC) * H * W
        bytes_fwd = (n_fine + n_coarse + n_out) * esz
        bytes_bwd = (n_up + n_coarse) * esz
        bytes_eager_fwd = (n_coarse + n_up + n_fine + n_up + n_out) * esz
        bytes_eager_bwd = (2 * n_up + n_coarse + n_up + 2 * n_coarse) * esz
        set_bytes = (n_fine + n_coarse + n_out) * esz
        nsets = max(2, math.ceil(2 * L2_BYTES / set_bytes))
        gen = torch.Generator(device=dev).manual_seed(7)
        sets = []
        for _ in range(nsets):
            fine = torch.randn(B, CF, H, W, device=dev, generator=gen).to(dt).requires_grad_(True)
            coarse = torch.randn(B, CC, h, w, device=dev, generator=gen).to(dt).requires_grad_(True)
            g = torch.randn(B, CF + CC, H, W, device=dev, generator=gen).to(dt)
            sets.append((fine, coarse, g))

        def fwd(op):
            return lambda f, c, g: op(f, c)

        def fwd_bwd(op):
            return lambda f, c, g: torch.autograd.grad(op(f, c), (f, c), g)

        row = {"B": B, "coarse": [h, w], "out": [H, W], "dtype": str(dt).replace("torch.", ""), "buffer_sets": nsets,
               "algorithmic_bytes": {"fused_fwd": bytes_fwd, "fused_bwd": bytes_bwd, "eager_fwd": bytes_eager_fwd,
                                     "eager_bwd": bytes_eager_bwd}}
        for path, mk in (("fwd", fwd), ("fwd_bwd", fwd_bwd)):
            for arm, op in (("fused", upsample_concat), ("eager", eager_cat)):
                t_g = graph_time_ms(mk(op), sets, args.reps)
                t_e = event_time_ms(mk(op), sets, args.reps)
                row[f"{arm}_{path}_graph_us"] = round(t_g * 1e3, 2)
                row[f"{arm}_{path}_eager_us"] = round(t_e * 1e3, 2)
                nbytes = bytes_fwd if arm == "fused" else bytes_eager_fwd
                if path == "fwd_bwd":
                    nbytes += bytes_bwd if arm == "fused" else bytes_eager_bwd
                row[f"{arm}_{path}_GBps"] = round(nbytes / (t_g * 1e-3) / 1e9, 1)
        tf, tb = row["fused_fwd_graph_us"], row["fused_fwd_bwd_graph_us"] - row["fused_fwd_graph_us"]
        row["fused_bwd_only_us_by_difference"] = round(tb, 2)
        row["speedup_fwd"] = round(row["eager_fwd_graph_us"] / tf, 2)
        row["speedup_fwd_bwd"] = round(row["eager_fwd_bwd_graph_us"] / row["fused_fwd_bwd_graph_us"], 2)
        # parity at the timed size: the forward bit for bit, d_coarse against torch's (atomic) fp32/bf16 backward
        f, c, g = sets[0]
        out_f, out_e = upsample_concat(f, c), eager_cat(f, c)
        dc_f = torch.autograd.grad(out_f, c, g)[0]
        dc_e = torch.autograd.grad(out_e, c, g)[0]
        row["parity"] = {"forward_bit_equal": bool(torch.equal(out_f, out_e)),
                         "d_coarse_max_abs_diff_vs_torch": float((dc_f.float() - dc_e.float()).abs().max()),
                         "d_coarse_max_abs": float(dc_e.float().abs().max())}
        res["workloads"][name] = row
        del sets, out_f, out_e, dc_f, dc_e
        torch.cuda.empty_cache()
    line = json.dumps(res)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
