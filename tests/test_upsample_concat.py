"""upsample_concat / pm_upcat_fwd / pm_upcat_bwd: the DeepLabV3+ decoder step after the memory module
(network/deepv3plus.py:569-572), ``cat([fine, Upsample(coarse, fine.shape[-2:])], 1)``.

The forward is checked bit for bit against torch. The gradient of ``coarse`` is checked against the fp64 transpose of
the forward's own taps (the fp32 source coordinates ATen and the kernel use), and against torch's fp64 autograd with a
bound that allows for those fp32 coordinates. CPU tests cover the C entries' argument checks.
"""
import ctypes

import numpy as np
import pytest
import torch
import torch.nn as nn
import torch.nn.functional as F

from golden_util import assert_close, max_abs_over_scale, rel_l2

# (B, Cf, Cc, h, w, H, W)
SHAPES = {
    "crop": (8, 48, 256, 48, 48, 192, 192),          # the reference crop: DR50V3P, OS16, 768^2
    "os8": (8, 48, 256, 96, 96, 192, 192),
    "eval": (1, 48, 256, 64, 128, 256, 512),         # a Cityscapes validation image at OS16
    "ragged": (2, 5, 3, 13, 17, 50, 61),             # non-integer scales, odd channels, rows not 16-byte multiples
    "identity": (2, 5, 3, 20, 23, 20, 23),
    "h1": (2, 5, 3, 1, 17, 7, 50),
    "w1": (2, 5, 3, 13, 1, 50, 7),
    "one": (2, 5, 3, 1, 1, 1, 1),
    "cf0": (2, 0, 7, 13, 17, 50, 61),
}
SMALL = ["ragged", "identity", "h1", "w1", "one", "cf0"]
DTYPES = [torch.float32, torch.bfloat16]


def reference(fine, coarse):
    return torch.cat([fine, F.interpolate(coarse, size=fine.shape[-2:], mode="bilinear", align_corners=True)], 1)


def interp_matrix(n_out, n_in, device):
    """[n_out, n_in] float64: the forward's bilinear weights along one axis, with ATen's fp32 source coordinates
    (src = scale * dst, i0 = trunc(src), lambda = src - i0, the second tap clamped at the last index)."""
    # (in - 1) / (out - 1) divided in fp32 (IEEE division, as ATen does it on the host), 0 when out == 1
    scale = float(np.float32(n_in - 1) / np.float32(n_out - 1)) if n_out > 1 else 0.0
    src = torch.arange(n_out, device=device, dtype=torch.float32) * scale   # scale is exact in fp32
    i0 = src.trunc().long().clamp(max=n_in - 1)
    lam = src - i0.float()
    i1 = torch.where(i0 < n_in - 1, i0 + 1, i0)
    m = torch.zeros(n_out, n_in, dtype=torch.float64, device=device)
    rows = torch.arange(n_out, device=device)
    m.index_put_((rows, i0), (1 - lam).double(), accumulate=True)
    m.index_put_((rows, i1), lam.double(), accumulate=True)
    return m


def transpose64(g, Cf, h, w):
    """fp64 d_coarse = Wy^T g[:, Cf:] Wx with the forward's fp32 taps."""
    H, W = g.shape[-2:]
    wy, wx = interp_matrix(H, h, g.device), interp_matrix(W, w, g.device)
    return torch.einsum("yi,bcyx,xj->bcij", wy, g[:, Cf:].double(), wx)


def _inputs(shape, dtype, seed):
    B, Cf, Cc, h, w, H, W = shape
    gen = torch.Generator(device="cuda").manual_seed(seed)
    fine = torch.randn(B, Cf, H, W, device="cuda", generator=gen).to(dtype)
    coarse = torch.randn(B, Cc, h, w, device="cuda", generator=gen).to(dtype)
    g = torch.randn(B, Cf + Cc, H, W, device="cuda", generator=gen).to(dtype)
    return fine, coarse, g


# ----------------------------------------------------------------------------------------------------------------- CPU


def test_upcat_argument_checks_run_without_a_gpu():
    """Rejected arguments return negative status codes before any CUDA call."""
    from pinthememory_b200 import capi

    lib = capi.load()
    p = ctypes.c_void_p(256)
    sizes = dict(dtype=0, B=2, Cf=48, Cc=256, h=12, w=12, H=48, W=48, stream=None)

    def fwd(**kw):
        a = dict(fine=p, coarse=p, out=p, **sizes)
        a.update(kw)
        return lib.pm_upcat_fwd(*a.values())

    def bwd(**kw):
        a = dict(g=p, d_coarse=p, **sizes)
        a.update(kw)
        return lib.pm_upcat_bwd(*a.values())

    assert fwd(coarse=None) == -1 and fwd(out=None) == -1 and fwd(fine=None) == -1
    assert bwd(g=None) == -1 and bwd(d_coarse=None) == -1
    for call in (fwd, bwd):
        assert call(dtype=2) == -2 and call(dtype=-1) == -2
        assert call(B=0) == -5 and call(Cc=0) == -5 and call(Cf=-1) == -5
        assert call(h=0) == -5 and call(w=0) == -5 and call(H=0) == -5 and call(W=0) == -5
        assert call(H=11) == -5 and call(W=11) == -5          # down-sampling
        assert call(B=65536) == -5 and call(Cf=65000, Cc=536) == -5
        assert call(H=65536, W=65536, h=1, w=1) == -5          # plane of 2^32 elements
    assert fwd(Cf=0, fine=None, dtype=5) == -2                  # a NULL fine is allowed with Cf = 0


# ----------------------------------------------------------------------------------------------------------------- GPU


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("name", list(SHAPES))
def test_forward_is_bit_exact(name, dtype):
    from pinthememory_b200 import upsample_concat

    fine, coarse, _ = _inputs(SHAPES[name], dtype, 1)
    out = upsample_concat(fine, coarse)
    assert out.dtype == dtype and out.is_contiguous()
    assert torch.equal(out, reference(fine, coarse)), name


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("name", list(SHAPES))
def test_backward_against_fp64(name, dtype):
    from pinthememory_b200 import upsample_concat

    B, Cf, Cc, h, w, H, W = SHAPES[name]
    fine, coarse, g = _inputs(SHAPES[name], dtype, 2)
    f, c = fine.clone().requires_grad_(True), coarse.clone().requires_grad_(True)
    upsample_concat(f, c).backward(g)
    assert torch.equal(f.grad, g[:, :Cf]), "d_fine must be g's first Cf channels"
    assert c.grad.dtype == dtype
    # the exact transpose of the forward: fp32 accumulation error only (bf16: plus one rounding of the result)
    tol = 1e-6 if dtype == torch.float32 else 4e-3
    assert_close(c.grad, transpose64(g, Cf, h, w), tol, f"{name} {dtype} d_coarse vs the fp64 transpose")
    # torch's fp64 autograd: its fp64 source coordinates differ from the fp32 ones by up to ~max(h,w) * 2^-24 in lambda
    c64 = coarse.double().requires_grad_(True)
    reference(fine.double(), c64).backward(g.double())
    tol64 = tol + 4 * max(h, w) * 2.0 ** -24
    assert_close(c.grad, c64.grad, tol64, f"{name} {dtype} d_coarse vs torch fp64")
    ct = coarse.clone().requires_grad_(True)
    reference(fine, ct).backward(g)
    print(f"{name} {dtype}: fused rel_l2 {rel_l2(c.grad, c64.grad):.2e} max/scale {max_abs_over_scale(c.grad, c64.grad):.2e}"
          f" | torch rel_l2 {rel_l2(ct.grad, c64.grad):.2e} max/scale {max_abs_over_scale(ct.grad, c64.grad):.2e}")


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("name", SMALL)
def test_adjoint_identity(name, dtype):
    """<g, upcat(f, c)> = <d_f, f> + <d_c, c> in fp64: a wrong tap at a border row or column breaks it."""
    from pinthememory_b200 import upsample_concat

    fine, coarse, g = _inputs(SHAPES[name], dtype, 3)
    f, c = fine.clone().requires_grad_(True), coarse.clone().requires_grad_(True)
    out = upsample_concat(f, c)
    out.backward(g)
    g64, o64 = g.double(), out.detach().double()
    lhs = (g64 * o64).sum()
    rhs = (f.grad.double() * fine.double()).sum() + (c.grad.double() * coarse.double()).sum()
    mag = (g64 * o64).abs().sum() + (c.grad.double() * coarse.double()).abs().sum()
    eps = 1e-6 if dtype == torch.float32 else 2.0 ** -8   # fp32 accumulation / one bf16 rounding of out and of d_c
    assert abs(float(lhs - rhs)) <= eps * float(mag), (name, float(lhs), float(rhs), float(mag))


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", DTYPES)
def test_deterministic_mode(dtype):
    from pinthememory_b200 import upsample_concat

    fine, coarse, g = _inputs(SHAPES["crop"], dtype, 4)
    was = torch.are_deterministic_algorithms_enabled()
    torch.use_deterministic_algorithms(True)
    try:
        grads = []
        for _ in range(2):
            f, c = fine.clone().requires_grad_(True), coarse.clone().requires_grad_(True)
            upsample_concat(f, c).backward(g)
            grads.append((f.grad, c.grad))
    finally:
        torch.use_deterministic_algorithms(was)
    assert torch.are_deterministic_algorithms_enabled() == was
    assert torch.equal(grads[0][0], grads[1][0]) and torch.equal(grads[0][1], grads[1][1])


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", DTYPES)
def test_cuda_graph_replay_equals_eager(dtype):
    from pinthememory_b200 import upsample_concat

    fine, coarse, g = _inputs(SHAPES["ragged"], dtype, 5)
    f, c = fine.clone().requires_grad_(True), coarse.clone().requires_grad_(True)

    def step():
        out = upsample_concat(f, c)
        df, dc = torch.autograd.grad(out, (f, c), g)
        return out, df, dc

    # warm-up on a side stream, as GraphedStep does, so that first-use set-up stays outside the capture
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        for _ in range(3):
            step()
    torch.cuda.current_stream().wait_stream(side)
    torch.cuda.synchronize()
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        captured = step()
    captured[0].zero_()
    captured[2].zero_()   # (captured[1], d_fine, is a view of g)
    graph.replay()
    torch.cuda.synchronize()
    eager = step()
    for a, b in zip(captured, eager):
        assert torch.equal(a, b)


class Decoder(nn.Module):
    """The DeepLabV3+ decoder around the module's output (deepv3plus.py:569-578): bot_fine on the low-level map, the
    (memory) output up-sampled and concatenated, final1 (conv + BN + ReLU), the classifier, the main loss."""

    def __init__(self, c_low, c_in, c_coarse, num_classes, fused):
        super().__init__()
        self.fused = fused
        self.bot_fine = nn.Conv2d(c_low, 48, kernel_size=1, bias=False)
        self.bot_aspp = nn.Conv2d(c_in, c_coarse, kernel_size=1, bias=False)
        self.final1 = nn.Sequential(nn.Conv2d(48 + c_coarse, c_coarse, kernel_size=3, padding=1, bias=False),
                                    nn.BatchNorm2d(c_coarse), nn.ReLU(inplace=True))
        self.final2 = nn.Conv2d(c_coarse, num_classes, kernel_size=1, bias=False)

    def forward(self, low_level, aspp, gts):
        from pinthememory_b200 import upsample_concat, upsampled_cross_entropy

        dec0_fine = self.bot_fine(low_level)
        dec0_up = self.bot_aspp(aspp)
        dec0 = upsample_concat(dec0_fine, dec0_up) if self.fused else reference(dec0_fine, dec0_up)
        return upsampled_cross_entropy(self.final2(self.final1(dec0)), gts)


@pytest.mark.gpu
def test_decoder_standin_matches_interpolate_and_cat():
    from pinthememory_b200 import synth

    old = (torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32)
    torch.backends.cudnn.allow_tf32 = torch.backends.cuda.matmul.allow_tf32 = False
    try:
        B, c_low, c_in, c_coarse, K, h, H = 2, 64, 96, 64, 19, 12, 48
        torch.manual_seed(21)
        fused = Decoder(c_low, c_in, c_coarse, K, True).cuda().train()
        plain = Decoder(c_low, c_in, c_coarse, K, False).cuda().train()
        plain.load_state_dict(fused.state_dict())
        low = synth.make_features(B, c_low, H, H, seed=22, device="cuda")
        aspp = synth.make_features(B, c_in, h, h, seed=23, device="cuda")
        gts = synth.make_labels(B, 4 * H, 4 * H, K, "blocky", seed=24).cuda()
        res = []
        for net in (fused, plain):
            lo, asp = low.clone().requires_grad_(True), aspp.clone().requires_grad_(True)
            loss = net(lo, asp, gts)
            loss.backward()
            res.append((loss.detach(), lo.grad, asp.grad, {n: p.grad for n, p in net.named_parameters()}))
    finally:
        torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32 = old
    (l1, dl1, da1, g1), (l2, dl2, da2, g2) = res
    assert_close(l1, l2, 2e-5, "loss")
    assert_close(dl1, dl2, 2e-5, "d low-level")
    assert_close(da1, da2, 2e-5, "d ASPP")
    for n in g2:
        assert_close(g1[n], g2[n], 2e-5, "grad " + n)


@pytest.mark.gpu
def test_rejections():
    from pinthememory_b200 import upsample_concat

    fine = torch.randn(2, 4, 16, 16, device="cuda")
    coarse = torch.randn(2, 3, 8, 8, device="cuda")
    with pytest.raises(RuntimeError, match="no CPU path"):
        upsample_concat(fine.cpu(), coarse.cpu())
    with pytest.raises(RuntimeError, match="pinmem_b200"):
        upsample_concat(fine.half(), coarse.half())
    with pytest.raises(RuntimeError, match="pinmem_b200"):
        upsample_concat(fine, coarse.bfloat16())
    with pytest.raises(RuntimeError, match="pinmem_b200"):
        upsample_concat(fine, coarse[:1])
    with pytest.raises(RuntimeError, match="up-samples only"):
        upsample_concat(fine[..., :8, :8], torch.randn(2, 3, 9, 8, device="cuda"))
    with pytest.raises(RuntimeError, match="pinmem_b200"):
        upsample_concat(fine[0], coarse[0])
    if torch.cuda.device_count() < 2:
        pytest.skip("one GPU: the cross-device rejection needs two")
    with pytest.raises(RuntimeError, match="pinmem_b200"):
        upsample_concat(fine, coarse.to("cuda:1"))
