"""The weight-gradient GEMM as tcgen05 SM pairs (conv1x1_wgrad_kernel, cta_group::2), at the shapes the pair layout adds.

A pair runs row tiles 2p and 2p+1 of one chunk; each CTA stages half of every X box (NW/2 rows) and the leader's MMAs
read both. The shapes below reach what the single-CTA kernel did not have: a pair whose second CTA has no row tile of its
own (M = 384, M = 96), every width per instruction the split takes (NW = 32, 64, 144, 256), two instructions per stage
(N = 288) next to a one-instruction column block (256 + 288), and more clusters than fit at once (B = 80). Each runs in
the exact tier (integer operands, bitwise against float64) and the precision tier of test_gpu_gemm_kernels.py and
test_gpu_tf32_gemm.py, with their bounds and guarded buffers; plus repeat-equality and replay inside a CUDA graph. A CPU
test checks that every instantiation compiles without spills to pair MMAs and multicast commits only."""
import os
import re
import shutil
import subprocess

import pytest
import torch

from golden_util import rel_l2
from test_gpu_gemm_kernels import (ELEM_C, ELEM_K0, PM_BF16, PM_F32, TAU, Guarded, _ints, _lib, _ok, _run_wgrad, _stream,
                                   _wgrad_ref, scaled_gaussian, wgrad_chunks)
from test_gpu_tf32_gemm import PM_F32_TF32, _run_wgrad1, tf32_bound

gpu = pytest.mark.gpu

# (B, M, N, hw); hw % 8 == 0 so that every case also runs in bf16 (16-byte rows)
PAIR_CASES = {
    "m384_idle_half": (2, 384, 288, 1296),       # 3 row tiles: the second pair's rank 1 has rows >= Mpad
    "m96_nw32": (2, 96, 32, 104),                # one row tile (idle rank 1), 16 X rows per CTA, pixel tail
    "m96_nw64": (3, 96, 64, 1296),
    "m96_nw144": (2, 96, 288, 1296),             # N = 288: two 144-wide instructions, 72 X rows per CTA
    "m96_nw256": (2, 96, 256, 1296),
    "ni2": (3, 256, 288, 1296),
    "cols_256_288": (2, 256, 544, 2304),         # column blocks of 256 (NI = 1) + 288 (NI = 2)
    "b80_second_wave": (80, 256, 288, 1024),     # one chunk per image: 80 clusters of 2, more than 148 SMs hold at once
    "b80_m384": (80, 384, 64, 40),               # 160 clusters, idle halves in every second one
}
DTYPES = {"f32": PM_F32, "tf32": PM_F32_TF32, "bf16": PM_BF16}
CASES = [(d, n, c) for d in DTYPES for n, c in PAIR_CASES.items()]


def _run(dt, dY, X, B, M, N, hw):
    if dt == "tf32":
        return _run_wgrad1(dY, X, B, M, N, hw)
    return _run_wgrad(torch.bfloat16 if dt == "bf16" else torch.float32, dY, X, B, M, N, hw)


@gpu
@pytest.mark.parametrize("dt,name,case", CASES, ids=lambda v: v if isinstance(v, str) else "")
def test_wgrad_pair_exact(dt, name, case):
    """Integer operands, |dW| <= 49 B hw < 2^24: bitwise equal to float64, and to a second call."""
    B, M, N, hw = case
    gen = torch.Generator(device="cuda").manual_seed(12000 + M + N + hw + B)
    dtype = torch.bfloat16 if dt == "bf16" else torch.float32
    dY, X = _ints((B, M, hw), -7, 7, gen).to(dtype), _ints((B, N, hw), -7, 7, gen).to(dtype)
    dY[:, 0] = 0
    ref = _wgrad_ref(dY, X)
    dW = _run(dt, dY, X, B, M, N, hw)
    bad = dW.double() != ref
    assert not bool(bad.any()), "%d elements differ, first at %s" % (int(bad.sum()), bad.nonzero()[0].tolist())
    assert torch.equal(_run(dt, dY, X, B, M, N, hw).view(torch.int32), dW.view(torch.int32)), "not reproducible"


@gpu
@pytest.mark.parametrize("dt,name,case", CASES, ids=lambda v: v if isinstance(v, str) else "")
def test_wgrad_pair_precision(dt, name, case):
    """Gaussian data with 2^-8..2^8 channel scales; the bounds of the existing weight-gradient precision tests."""
    B, M, N, hw = case
    gen = torch.Generator(device="cuda").manual_seed(13000 + M + N + hw + B)
    dtype = torch.bfloat16 if dt == "bf16" else torch.float32
    dY = scaled_gaussian((B, M, hw), 1, gen, "cuda").to(dtype)
    X = scaled_gaussian((B, N, hw), 1, gen, "cuda").to(dtype)
    dW = _run(dt, dY, X, B, M, N, hw)
    ref = _wgrad_ref(dY, X)
    mag = torch.einsum("bmp,bnp->mn", dY.double().abs(), X.double().abs())
    kc, nch = wgrad_chunks(dtype, B, M, hw)
    if dt == "tf32":
        bound = tf32_bound(kc + nch, mag)
    else:
        bound = ELEM_C * (kc + nch + ELEM_K0) * 2.0 ** -24 * mag
    ratio = float(((dW.double() - ref).abs() / bound.clamp_min(1e-300)).max())
    r = rel_l2(dW, ref)
    print("pair wgrad %s %s chunk=%d x %d rel_l2=%.3e elem/bound=%.3f" % (dt, name, kc, nch, r, ratio))
    assert ratio <= 1.0, "element-wise bound exceeded by %.2fx" % ratio
    if dt != "tf32":
        assert r <= TAU(kc), "rel_l2 %.3e > tau(%d) = %.1e" % (r, kc, TAU(kc))


@gpu
@pytest.mark.parametrize("dt", list(DTYPES))
def test_wgrad_pair_graph_replay(dt):
    """The cluster launch captured in a CUDA graph: a replay equals the eager call, also after the inputs change in place."""
    B, M, N, hw = 3, 384, 544, 1296
    lib = _lib()
    dtype = torch.bfloat16 if dt == "bf16" else torch.float32
    gen = torch.Generator(device="cuda").manual_seed(14000)
    dY = scaled_gaussian((B, M, hw), 1, gen, "cuda").to(dtype)
    X = scaled_gaussian((B, N, hw), 1, gen, "cuda").to(dtype)
    nws = lib.pm_conv1x1_wgrad_workspace_floats(B, M, N, hw, DTYPES[dt])
    ws = Guarded(nws, torch.float32)
    dW = Guarded(M * N, torch.float32)

    def call():
        _ok(lib.pm_conv1x1_wgrad(dY.data_ptr(), X.data_ptr(), ws.t.data_ptr(), dW.t.data_ptr(), B, M, N, hw, 0, DTYPES[dt],
                                 _stream()), "pm_conv1x1_wgrad")

    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        call()                                   # warm-up outside the capture (tensor maps, function attributes)
    torch.cuda.current_stream().wait_stream(s)
    torch.cuda.synchronize()
    eager = _run(dt, dY, X, B, M, N, hw)
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        call()
    for step in range(2):
        if step == 1:                            # new inputs at the same addresses
            dY.copy_(scaled_gaussian((B, M, hw), 1, gen, "cuda").to(dtype))
            X.copy_(scaled_gaussian((B, N, hw), 1, gen, "cuda").to(dtype))
            eager = _run(dt, dY, X, B, M, N, hw)
        dW.t.fill_(float("nan"))
        g.replay()
        torch.cuda.synchronize()
        ws.check("workspace", scratch=True)
        dW.check("dW")
        assert torch.equal(dW.t.view(M, N).view(torch.int32), eager.view(torch.int32)), "replay %d differs" % step


@pytest.mark.skipif(shutil.which("nvcc") is None and not os.path.exists("/usr/local/cuda/bin/nvcc"), reason="no nvcc")
def test_wgrad_kernel_compiles_to_pairs_without_spills(tmp_path):
    """Every conv1x1_wgrad_kernel instantiation: no spill bytes, and in SASS only pair MMAs (UTCHMMA.2CTA) and multicast
    pair commits (UTCBAR.2CTA.MULTICAST)."""
    from pinthememory_b200 import build

    obj = str(tmp_path / "g.o")
    cmd = [build._nvcc(), *build.ARCH_FLAGS, "-O3", "-std=c++17", "-Xptxas=-v", "-c", os.path.join(build.CSRC, "pm_gemm.cu"),
           "-o", obj]
    r = subprocess.run(cmd, capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    entries = re.findall(r"Compiling entry function '(\w*conv1x1_wgrad_kernel\w*)'.*?(\d+) bytes spill stores, (\d+) bytes spill loads",
                         r.stderr, flags=re.S)
    assert len(entries) == 3, r.stderr          # float, Tf32OnePass<false>, __nv_bfloat16
    for name, st, ld in entries:
        assert st == "0" and ld == "0", name
    cuobjdump = os.path.join(os.path.dirname(build._nvcc()), "cuobjdump")
    if not os.path.exists(cuobjdump):
        return
    sass = subprocess.run([cuobjdump, "-sass", obj], capture_output=True, text=True)
    assert sass.returncode == 0, sass.stderr
    funcs = [f for f in re.split(r"\n\s*Function : ", sass.stdout) if "conv1x1_wgrad_kernel" in f.split("\n", 1)[0]]
    assert len(funcs) == 3
    for f in funcs:
        mma = re.findall(r"\bUTC\w*MMA[\w.]*", f)
        bars = re.findall(r"\bUTCBAR[\w.]*", f)
        assert mma and all(m.startswith("UTCHMMA.2CTA") for m in mma), (f.split("\n", 1)[0], sorted(set(mma)))
        assert bars and all(b.startswith("UTCBAR.2CTA.MULTICAST") for b in bars), (f.split("\n", 1)[0], sorted(set(bars)))
