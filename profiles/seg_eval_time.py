"""Validation metrics per batch: the fused ``SegMetrics.add`` (pm_seg_eval) against the torch GPU sequence and the
reference's host path, on three workloads. Prints one JSON line (and writes it to ``--out`` if given).

    python profiles/seg_eval_time.py [--reps 50] [--out seg_eval_time.json]

Workloads (synthetic ``blocky`` int64 labels, K = 19):
  a  Cityscapes validation image: B=1, logits 256x512 -> labels 1024x2048
  b  training-crop size:          B=2, logits 192x192 -> labels 768x768
  c  identity mode:               B=1, logits 1024x2048 at label size (the unmodified head's output)

Paths:
  fused   SegMetrics.add (workspace memset + one kernel), with and without the uint8 prediction map; CUDA events
          around eager calls (host overhead of the Python call included), and around CUDA-graph replays of the same
          calls (device time only)
  torch   F.interpolate + F.cross_entropy + argmax + torch.bincount (masked with torch.where, no boolean indexing) into a
          device confusion matrix; CUDA events
  host    the reference's validation loop: interpolate + argmax, .cpu(), NumPy fast_hist (utils/misc.py:65-73); wall
          clock around a device synchronise
Every timed repetition reads a different set of input buffers from a rotation larger than the 126 MB L2, so inputs
come from HBM. Algorithmic bytes: labels (8 B/pixel int64) + logits (K * element size per logit pixel) + 1 B/pixel
when the prediction map is written.
"""
import argparse
import json
import math
import os
import subprocess
import sys
import time

import numpy as np
import torch
import torch.nn.functional as F

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

from pinthememory_b200 import synth  # noqa: E402
from pinthememory_b200.callers import SegMetrics  # noqa: E402

K = 19
L2_BYTES = 126 * 2 ** 20
WORKLOADS = {"a_cityscapes_val": (1, 256, 512, 1024, 2048), "b_crop": (2, 192, 192, 768, 768),
             "c_identity": (1, 1024, 2048, 1024, 2048)}


def card():
    info = {"name": torch.cuda.get_device_name(0), "power_limit_w": None}
    try:   # read-only query
        r = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader,nounits", "-i", "0"],
                           capture_output=True, text=True, timeout=30)
        info["power_limit_w"] = float(r.stdout.strip().splitlines()[0])
    except Exception as e:  # noqa: BLE001
        info["power_limit_error"] = repr(e)[:200]
    return info


def fast_hist(a, b, n):
    """utils/misc.py:65-73 (a = label, b = prediction)."""
    k = (a >= 0) & (a < n)
    return np.bincount(n * a[k].astype(int) + b[k], minlength=n ** 2).reshape(n, n)


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
    """Per-call device time of ``fn`` with the host out of the loop: one call per buffer set captured in a CUDA graph."""
    for st in sets:
        fn(*st)
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
    return a.elapsed_time(b) / (n * len(sets))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=50)
    ap.add_argument("--host-reps", type=int, default=5)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("seg_eval_time.py needs a CUDA device")
    dev = torch.device("cuda:0")
    res = {"what": "seg_eval_time", "K": K, "card": card(), "inputs": "rotated buffers larger than the 126 MB L2 (HBM reads)",
           "workloads": {}}
    for name, (B, h, w, Hm, Wm) in WORKLOADS.items():
        x0 = 3.0 * synth.make_features(B, K, h, w, seed=101, device=dev)
        lab0 = synth.make_labels(B, Hm, Wm, K, "blocky", seed=102, device=dev)
        set_bytes = x0.numel() * 4 + lab0.numel() * 8
        nsets = max(2, math.ceil(2 * L2_BYTES / set_bytes))
        sets = [(x0.roll(i, dims=-1).contiguous(), lab0.roll(i, dims=-1).contiguous()) for i in range(nsets)]
        npx, nlog = B * Hm * Wm, B * h * w
        bytes_fused = npx * 8 + nlog * K * 4
        sm = SegMetrics(K, device=dev)

        t_fused = event_time_ms(lambda x, l: sm.add(x, l), sets, args.reps)
        t_fused_pred = event_time_ms(lambda x, l: sm.add(x, l, predictions=True), sets, args.reps)
        t_fused_graph = graph_time_ms(lambda x, l: sm.add(x, l), sets, 4 * args.reps)
        conf = torch.zeros(K, K, dtype=torch.int64, device=dev)

        def torch_seq(x, lab):
            up = x if (h, w) == (Hm, Wm) else F.interpolate(x, size=(Hm, Wm), mode="bilinear", align_corners=True)
            loss = F.cross_entropy(up, lab, ignore_index=255)
            pred = up.argmax(1)
            m = (lab >= 0) & (lab < K)
            idx = torch.where(m, K * lab + pred, K * K)
            conf.add_(torch.bincount(idx.view(-1), minlength=K * K + 1)[: K * K].view(K, K))
            return loss

        t_torch = event_time_ms(torch_seq, sets, max(5, args.reps // 5))
        # parity on the first set, at the size timed
        sm_chk = SegMetrics(K, device=dev)
        lf, pf = sm_chk.add(*sets[0], predictions=True)
        conf.zero_()
        lt = torch_seq(*sets[0])
        x, lab = sets[0]
        up = x if (h, w) == (Hm, Wm) else F.interpolate(x, size=(Hm, Wm), mode="bilinear", align_corners=True)
        pred_diff = int((pf.long() != up.argmax(1)).sum())
        del up

        def host_path(x, lab):
            up = x if (h, w) == (Hm, Wm) else F.interpolate(x, size=(Hm, Wm), mode="bilinear", align_corners=True)
            p = up.argmax(1).cpu().numpy()
            return fast_hist(lab.cpu().numpy().ravel(), p.ravel(), K)

        host_path(*sets[0])
        times = []
        for i in range(args.host_reps):
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            host_path(*sets[i % nsets])
            torch.cuda.synchronize()
            times.append((time.perf_counter() - t0) * 1e3)
        res["workloads"][name] = {
            "B": B, "logits": [h, w], "labels": [Hm, Wm], "buffer_sets": nsets,
            "algorithmic_bytes": bytes_fused, "algorithmic_bytes_with_pred": bytes_fused + npx,
            "fused_add_us": round(t_fused * 1e3, 2), "fused_add_pred_us": round(t_fused_pred * 1e3, 2),
            "fused_add_graph_us": round(t_fused_graph * 1e3, 2),
            "fused_GBps": round(bytes_fused / (t_fused * 1e-3) / 1e9, 1),
            "fused_graph_GBps": round(bytes_fused / (t_fused_graph * 1e-3) / 1e9, 1),
            "fused_pred_GBps": round((bytes_fused + npx) / (t_fused_pred * 1e-3) / 1e9, 1),
            "torch_gpu_sequence_us": round(t_torch * 1e3, 2),
            "host_path_ms_median": round(float(np.median(times)), 3),
            "speedup_vs_torch": round(t_torch / t_fused, 2),
            "parity": {"loss_fused": float(lf), "loss_torch": float(lt), "confusion_equal": bool(torch.equal(sm_chk.confusion, conf)),
                       "pred_differs_px": pred_diff},
        }
        del sets, sm, sm_chk
        torch.cuda.empty_cache()
    line = json.dumps(res)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
