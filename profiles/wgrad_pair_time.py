"""The weight-gradient GEMM as SM pairs against the single-CTA kernel it replaced, in one process.

    python profiles/wgrad_pair_time.py --parent-lib OLD/libpinmem_b200.so [--seconds 1.0] [--rounds 3]
                                       [--out profiles/wgrad_pair_time_b200.json]

Times pm_conv1x1_wgrad (the GEMM and its wgrad_reduce_kernel) of this tree's library and of an earlier build given by
--parent-lib, both loaded through ctypes, at the two products of BASELINE config 2 (B = 8, 96x96): 256x288 (the folded
output convolution) and 256x256 (the writing net), each in 3xTF32 (PM_F32), one-pass TF32 (PM_F32_TF32) and bf16.
Every call reads the next of several input sets whose sum exceeds the 126 MB L2, so operands come from HBM as in the
training step. The two libraries are timed alternately, --rounds windows each of at least --seconds (CUDA events around
the window, divided by the calls in it), after a warm-up; the median window is reported. The outputs of both libraries
on the same inputs are compared bit for bit. Prints one JSON line and writes it to --out.
"""
import argparse
import ctypes
import json
import os
import statistics
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PM_F32, PM_BF16, PM_F32_TF32 = 0, 1, 2
L2_BYTES = 126 << 20


def gpu_info():
    info = {"name": torch.cuda.get_device_name(0), "power_limit_w": None}
    try:
        r = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader,nounits", "-i", "0"],
                           capture_output=True, text=True, timeout=30)
        info["power_limit_w"] = float(r.stdout.strip().splitlines()[0])
    except Exception as e:  # noqa: BLE001
        info["power_limit_error"] = repr(e)[:200]
    return info


def load(path):
    lib = ctypes.CDLL(path)
    lib.pm_conv1x1_wgrad.argtypes = [ctypes.c_void_p] * 4 + [ctypes.c_int] * 6 + [ctypes.c_void_p]
    lib.pm_conv1x1_wgrad.restype = ctypes.c_int
    lib.pm_conv1x1_wgrad_workspace_floats.argtypes = [ctypes.c_int] * 5
    lib.pm_conv1x1_wgrad_workspace_floats.restype = ctypes.c_int
    return lib


def window(fn, n):
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(n):
        fn()
    b.record()
    b.synchronize()
    return a.elapsed_time(b)


def calls_for(fn, seconds):
    """Number of calls that fill a window of at least `seconds` (after a warm-up)."""
    for _ in range(5):
        fn()
    torch.cuda.synchronize()
    n = 4
    while True:
        ms = window(fn, n)
        if ms >= 1000.0 * seconds:
            return n
        n = max(n * 2, int(n * 1.2 * 1000.0 * seconds / max(ms, 1e-3)))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--parent-lib", required=True)
    ap.add_argument("--lib", default=os.path.join(ROOT, "pinthememory_b200", "_lib", "libpinmem_b200.so"))
    ap.add_argument("--seconds", type=float, default=1.0)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "wgrad_pair_time_b200.json"))
    args = ap.parse_args()
    assert torch.cuda.is_available(), "needs a CUDA device"
    libs = {"parent": load(args.parent_lib), "pairs": load(args.lib)}
    stream = torch.cuda.current_stream().cuda_stream
    B, hw, M = 8, 96 * 96, 256
    res = {}
    for N in (288, 256):
        for dname, code, dtype in (("three_pass", PM_F32, torch.float32), ("one_pass", PM_F32_TF32, torch.float32),
                                   ("bf16", PM_BF16, torch.bfloat16)):
            g = torch.Generator(device="cuda").manual_seed(N + code)
            set_bytes = B * (M + N) * hw * dtype.itemsize
            nsets = L2_BYTES // set_bytes + 2
            sets = [(torch.randn(B, M, hw, generator=g, device="cuda").to(dtype),
                     torch.randn(B, N, hw, generator=g, device="cuda").to(dtype)) for _ in range(nsets)]
            nws = libs["pairs"].pm_conv1x1_wgrad_workspace_floats(B, M, N, hw, code)
            assert nws == libs["parent"].pm_conv1x1_wgrad_workspace_floats(B, M, N, hw, code)
            ws = torch.empty(nws, device="cuda")
            dW = torch.empty(M * N, device="cuda")
            outs = {}
            for key, lib in libs.items():
                dy, x = sets[0]
                rc = lib.pm_conv1x1_wgrad(dy.data_ptr(), x.data_ptr(), ws.data_ptr(), dW.data_ptr(), B, M, N, hw, 0, code, stream)
                assert rc == 0, (key, rc)
                torch.cuda.synchronize()
                outs[key] = dW.clone()
            diff = float((outs["pairs"] - outs["parent"]).abs().max())
            bitwise = bool(torch.equal(outs["pairs"].view(torch.int32), outs["parent"].view(torch.int32)))

            def caller(lib):
                it = [0]  # rotation through the input sets

                def fn():
                    dy, x = sets[it[0] % nsets]
                    it[0] += 1
                    lib.pm_conv1x1_wgrad(dy.data_ptr(), x.data_ptr(), ws.data_ptr(), dW.data_ptr(), B, M, N, hw, 0, code, stream)
                return fn

            fns = {k: caller(lib) for k, lib in libs.items()}
            n = {k: calls_for(f, args.seconds) for k, f in fns.items()}
            times = {k: [] for k in libs}
            for _ in range(args.rounds):
                for k, f in fns.items():
                    times[k].append(round(1000.0 * window(f, n[k]) / n[k], 2))
            med = {k: statistics.median(v) for k, v in times.items()}
            res["wgrad_%dx%d_%s" % (M, N, dname)] = {
                "parent_us": times["parent"], "pairs_us": times["pairs"], "parent_median_us": med["parent"],
                "pairs_median_us": med["pairs"], "gain": round(1.0 - med["pairs"] / med["parent"], 3),
                "bitwise_equal": bitwise, "max_abs_diff": diff, "input_sets": nsets}
            del sets, ws, dW
            torch.cuda.empty_cache()
    out = {"gpu": gpu_info(), "window_s": args.seconds, "rounds": args.rounds, "B": B, "hw": hw, "wgrad_with_reduce": res}
    line = json.dumps(out)
    print(line)
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        f.write(line + "\n")


if __name__ == "__main__":
    sys.exit(main())
