"""Cost of differentiable score maps: a cfg-2 module step with and without the two score terms in its loss, and
pm_score_bwd on its own against its algorithmic bytes.

    python profiles/score_grad_time.py [--seconds 1.0] [--out profiles/score_grad_time_b200.json]

Workloads:
  cfg2_{fp32,bf16}_graph  the module's training step (read + write, forward + backward, two-stream mode) at B=8, 96x96,
                          C=256, K=19, 768x768 blocky int64 labels, captured once as a CUDA graph and replayed. `default`:
                          loss <G,updated_query> + 0.02 readloss + 0.4 div + 0.2 cls; `scores`: the same plus
                          <G_q,score_query> + <G_m,score_memory>.
  pm_score_bwd            both score terms and the read-loss term at N = 73728, K = 19 (stride 20). Algorithmic bytes:
                          2*N*K*4 for the column sums, 4*N*K*4 + 2*N*stride*4 for the element-wise pass (about 45 MB).
                          Four input/output sets (180 MB > the 126 MB L2) are run in turn from one CUDA graph.
Each time is CUDA-event time over a window of at least --seconds, divided by the number of calls in it, after a warm-up.
Prints one JSON line and writes it to --out.
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

from pinthememory_b200 import capi, synth  # noqa: E402
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


def cfg2_step(dtype, with_scores, seconds):
    B, C, h, w, Hm, Wm, K = 8, 256, 96, 96, 768, 768, 19
    N = B * h * w
    torch.manual_seed(5)
    m = Memory_sup(K, C, C, 0.8, 1.0, False).cuda().to(dtype)
    m.overlap_write = True
    memory = m.m_items.float().clone()
    x = synth.make_features(B, C, h, w, seed=1, device="cuda").to(dtype).requires_grad_(True)
    lab = synth.make_labels(B, Hm, Wm, K, "blocky", seed=2, device="cuda")
    G = synth.make_upstream_grad((B, C, h, w), seed=3, device="cuda").to(dtype)
    Gq = synth.make_upstream_grad((B, h, w, K), seed=4, device="cuda")
    Gm = synth.make_upstream_grad((B, h, w, K), seed=5, device="cuda") / N
    wts = [torch.tensor(v, device="cuda") for v in (0.02, 0.4, 0.2)]
    params = [p for p in m.parameters() if p.requires_grad]

    def run():
        x.grad = None
        for p in params:
            p.grad = None
        m.m_items = memory
        uq, sq, sm, rl, wl = m(x, lab, True, True)
        outs, grads = [uq, rl, wl[0], wl[1]], [G, *wts]
        if with_scores:
            outs += [sq, sm]
            grads += [Gq, Gm]
        torch.autograd.backward(outs, grads)

    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        for _ in range(3):
            run()
    torch.cuda.current_stream().wait_stream(side)
    torch.cuda.synchronize()
    x.grad = None
    for p in params:
        p.grad = None
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        run()
    try:
        return timed(graph.replay, seconds)
    finally:
        torch.cuda.synchronize()
        graph.reset()


def score_bwd_alone(seconds, sets=4):
    N, K = 8 * 96 * 96, 19
    KP = capi.score_stride(K)
    g = torch.Generator(device="cuda").manual_seed(1)
    bufs = []
    for _ in range(sets):
        s = 3.0 * torch.randn(N, K, device="cuda", generator=g)
        bufs.append(dict(pq=torch.softmax(s, 0), gq=torch.randn(N, K, device="cuda", generator=g), pm=torch.softmax(s, 1),
                         gm=torch.randn(N, K, device="cuda", generator=g), rl=torch.randn(N, KP, device="cuda", generator=g),
                         E=torch.empty(N, KP, device="cuda")))
    g_loss = torch.tensor([0.02], device="cuda")
    rl_out = torch.tensor([0.0, 1e-6], device="cuda")

    def calls():
        for b in bufs:
            capi.score_bwd(b["pq"], b["gq"], b["pm"], b["gm"], b["E"], K, ds_rl=b["rl"], g_loss=g_loss, rl_out=rl_out)

    # one graph launches the `sets` calls back to back: device time, not the host's launch rate
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        calls()
    torch.cuda.current_stream().wait_stream(side)
    torch.cuda.synchronize()
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        calls()
    us = timed(graph.replay, seconds) / sets
    graph.reset()
    nbytes = 2 * N * K * 4 + 4 * N * K * 4 + 2 * N * KP * 4
    return {"N": N, "K": K, "us": round(us, 2), "alg_MB": round(nbytes / 1e6, 2), "GBps": round(nbytes / us / 1e3, 1)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--seconds", type=float, default=1.0)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "score_grad_time_b200.json"))
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("score_grad_time.py needs a CUDA device")
    res = {"gpu": gpu_info(), "window_s": args.seconds, "us_per_step": {}}
    for name, dt in (("cfg2_fp32_graph", torch.float32), ("cfg2_bf16_graph", torch.bfloat16)):
        res["us_per_step"][name] = {mode: round(cfg2_step(dt, mode == "scores", args.seconds), 1)
                                    for mode in ("default", "scores")}
    res["pm_score_bwd"] = score_bwd_alone(args.seconds)
    line = json.dumps(res)
    print(line)
    if args.out:
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
