"""The module with torch's TF32 switches on (capi.tf32): its fp32 1x1-convolution GEMMs run one TF32 pass.

Accuracy: the checker is the fp64 oracle with the module's ReLU gates replayed; the yardstick is the same oracle in fp32
with torch's own TF32 convolutions (cuDNN, the reference's Conv2d under these switches; its matmuls stay fp32) against
its fp64 self. Each tensor's error (the larger of rel-L2 and max-abs/scale) must be within C_YARD times the yardstick's,
or FLOOR. The measured errors are printed.

Mode: decided once per autograd Function in its forward, stored with it and in the operands it prepares; a captured
GraphedStep keeps the mode of its capture."""
import contextlib

import pytest
import torch

from golden_util import LOSS_WEIGHTS, max_abs_over_scale, rel_l2
from gate_util import oracle_module_like, record_gates
from test_gpu_deterministic import _clone_module, _module

pytestmark = pytest.mark.gpu

C_YARD, FLOOR = 3.0, 1e-4
# ReLU ties at TF32 level: a one-pass product is ~2^-11 of sum |a||x| off, so a pre-activation within a few 1e-4 of the
# map's largest can land on either side in two correct TF32 implementations
TF32_TIE_RATIO = 2e-3
TF32_TIE_FRACTION = 2e-3


@contextlib.contextmanager
def torch_tf32_convs():
    """The yardstick's mode: torch's cuDNN convolutions in TF32, its matmuls (the oracle's read and write contractions,
    which the module's kernels keep in 3xTF32) in fp32."""
    old = (torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32)
    torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32 = True, False
    try:
        yield
    finally:
        torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32 = old


@contextlib.contextmanager
def tf32(on):
    old = (torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32)
    torch.backends.cudnn.allow_tf32 = torch.backends.cuda.matmul.allow_tf32 = on
    try:
        yield
    finally:
        torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32 = old


def check_tf32_ties(relu_gates):
    for name, n, numel, ratio in relu_gates.mismatches:
        assert ratio <= TF32_TIE_RATIO, f"{name}: ReLU gate differs where |z|/max|z| = {ratio:.2e} (not a TF32 tie)"
        assert n <= max(3, TF32_TIE_FRACTION * numel), f"{name}: {n} of {numel} ReLU gates differ"


def _err(a, b):
    return max(rel_l2(a, b), max_abs_over_scale(a, b))


def _judge(got, ref64, ref32, what):
    """got and the yardstick ref32 against ref64: dicts of tensors with the same keys."""
    worst = []
    for k in ref64:
        e, y = _err(got[k], ref64[k]), _err(ref32[k], ref64[k])
        print("%s %-40s tf32 kernels %.2e  torch tf32 %.2e  ratio %.2f" % (what, k, e, y, e / max(y, 1e-30)))
        if e > max(FLOOR, C_YARD * y):
            worst.append((k, e, y))
    assert not worst, worst


def _step(m, x, labels, G):
    """forward with write + backward of the three weighted losses; returns every output and gradient by name."""
    x = x.clone().requires_grad_(True)
    uq, sq, sm, rl, wl = m(x, labels, True, True)
    total = (uq * G).sum() + LOSS_WEIGHTS["read"] * rl + LOSS_WEIGHTS["div"] * wl[0] + LOSS_WEIGHTS["cls"] * wl[1]
    total.backward()
    out = {"updated_query": uq, "score_query": sq, "score_memory": sm, "readloss": rl.reshape(1), "div_loss": wl[0].reshape(1),
           "cls_loss": wl[1].reshape(1), "m_items": m.m_items, "grad_x": x.grad}
    for n, p in m.named_parameters():
        if p.grad is not None:
            out["grad." + n] = p.grad
    return {k: v.detach().double() for k, v in out.items()}


def _oracle_step(o, x, labels, G):
    x = x.clone().requires_grad_(True)
    uq, sq, sm, rl, wl = o(x, labels, True, True)
    total = (uq * G).sum() + LOSS_WEIGHTS["read"] * rl + LOSS_WEIGHTS["div"] * wl[0] + LOSS_WEIGHTS["cls"] * wl[1]
    total.backward()
    out = {"updated_query": uq, "score_query": sq, "score_memory": sm, "readloss": rl.reshape(1), "div_loss": wl[0].reshape(1),
           "cls_loss": wl[1].reshape(1), "m_items": o.m_items, "grad_x": x.grad}
    for n, p in o.named_parameters():
        if p.grad is not None:
            out["grad." + n] = p.grad
    return {k: v.detach().double() for k, v in out.items()}


CFG2 = (8, 256, 96, 96, 768, 768)


@pytest.mark.parametrize("two_stream", [False, True], ids=["one_stream", "two_stream"])
def test_cfg2_step_against_fp64_oracle(two_stream):
    """BASELINE config 2 shapes (folded output convolution, writing net inside the write), fp32, TF32 on."""
    from oracle import memory_oracle as mo
    from pinthememory_b200 import synth

    B, C, h, w, Hm, Wm = CFG2
    K = 19
    m = _module(K, C, overlap_write=two_stream)
    o64 = oracle_module_like(m, dtype=torch.float64)
    o32 = oracle_module_like(m)
    x = synth.make_features(B, C, h, w, seed=31, device="cuda")
    labels = synth.make_labels(B, Hm, Wm, K, "blocky", seed=32, device="cuda")
    G = synth.make_upstream_grad((B, C, h, w), seed=33, device="cuda") / (B * h * w)
    with tf32(True), record_gates() as gates:
        got = _step(m, x, labels, G)
    o32.relu_gates = mo.ReluGates(gates)
    with torch_tf32_convs():
        ref32 = _oracle_step(o32, x, labels, G)
    o64.relu_gates = mo.ReluGates(gates)
    ref64 = _oracle_step(o64, x.double(), labels, G.double())
    check_tf32_ties(o64.relu_gates)
    keys = set(got) & set(ref64)
    assert {"grad_x", "grad.output.0.weight", "grad.writenet.writefeat.0.weight"} <= keys, sorted(keys)
    _judge({k: got[k] for k in keys}, {k: ref64[k] for k in keys}, ref32, "cfg2" + ("-2s" if two_stream else ""))


def test_cfg3_meta_step_against_fp64_oracle():
    """BASELINE config 3 (the meta-train step at OS16), TF32 on; as test_gpu_meta_step.py with the TF32 yardstick."""
    from oracle import memory_oracle as mo
    from pinthememory_b200 import synth
    from pinthememory_b200.memory import Memory_sup
    from pinthememory_b200.metastep import meta_step
    from test_gpu_meta_step import _trio

    B, C, h, w, Hm, Wm = 4, 256, 48, 48, 192, 192
    K = 19
    net, upd, upd2 = _trio(Memory_sup, K, C)
    with torch.no_grad():
        net.clsfier.weight.normal_(0, 0.2)
    state = {k: v.clone() for k, v in net.state_dict().items()}
    mem0 = net.m_items.clone()
    x_tr = synth.make_features(B, C, h, w, seed=11, device="cuda")
    x_te = synth.make_features(B, C, h, w, seed=12, device="cuda")
    lab_tr = synth.make_labels(B, Hm, Wm, K, "blocky", seed=13, device="cuda", block=16)
    lab_te = synth.make_labels(B, Hm, Wm, K, "blocky", seed=14, device="cuda", block=16)
    G_tr = synth.make_upstream_grad((B, C, h, w), seed=15, device="cuda") / (B * h * w)
    G_te = synth.make_upstream_grad((B, C, h, w), seed=16, device="cuda") / (B * h * w)
    with tf32(True), record_gates() as gates:
        got = meta_step(net, upd, upd2, x_tr, lab_tr, x_te, lab_te, G_tr, G_te, inner_lr=0.01)
    f_trio = _trio(mo.OracleMemorySup, K, C, state, mem0)
    shared32 = mo.ReluGates(gates)
    for o in f_trio:
        o.relu_gates = shared32
    with torch_tf32_convs():
        ref32 = meta_step(*f_trio, x_tr, lab_tr, x_te, lab_te, G_tr, G_te, inner_lr=0.01)
    o_trio = _trio(mo.OracleMemorySup, K, C, {k: v.double() for k, v in state.items()}, mem0, torch.float64)
    shared = mo.ReluGates(gates)
    for o in o_trio:
        o.relu_gates = shared
    ref = meta_step(*o_trio, x_tr.double(), lab_tr, x_te.double(), lab_te, G_tr.double(), G_te.double(), inner_lr=0.01)
    check_tf32_ties(shared)

    def flat(r):
        out = {k: r[k].reshape(-1) for k in ("inner_loss", "outer_loss", "readloss_a", "div_a", "cls_a", "readloss_c",
                                             "uq_c", "memory_b", "memory_final")}
        for name in ("inner_grads", "grads"):
            out.update({name + " " + k: v for k, v in r[name].items()})
        return {k: v.detach().double() for k, v in out.items()}

    _judge(flat(got), flat(ref), flat(ref32), "cfg3")


# ================================================================================================ mode handling
def _kernels(fn):
    """(3-pass, one-pass) sets of the GEMM kernel names `fn` launches."""
    from torch.profiler import ProfilerActivity, profile

    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    three, one = set(), set()
    for e in prof.events():
        if e.device_type != torch.autograd.DeviceType.CUDA or "conv1x1_" not in e.name:
            continue
        if "Tf32OnePass" in e.name:
            one.add(e.name.split("(")[0])
        elif "conv1x1_nn_kernel<float" in e.name or "conv1x1_wgrad_kernel<float" in e.name:
            three.add(e.name.split("(")[0])
    return three, one


def _small_inputs(K=19, C=256, seed=41):
    from pinthememory_b200 import synth

    x = synth.make_features(2, C, 96, 96, seed=seed, device="cuda").requires_grad_(True)
    lab = synth.make_labels(2, 384, 384, K, "blocky", seed=seed + 1, device="cuda")
    G = synth.make_upstream_grad((2, C, 96, 96), seed=seed + 2, device="cuda")
    return x, lab, G


def _fwd(m, x, lab):
    uq, sq, sm, rl, wl = m(x, lab, True, True)
    return uq, rl, wl


def _bwd(outs, G):
    uq, rl, wl = outs
    ((uq * G).sum() + 0.02 * rl + 0.4 * wl[0] + 0.2 * wl[1]).backward()


def test_switch_read_per_call():
    """Flipping the switches between two steps changes the kernels the next step launches (forward and backward)."""
    m = _module(19, 256)
    x, lab, G = _small_inputs()
    for on in (True, False, True):
        with tf32(on):
            three, one = _kernels(lambda: _bwd(_fwd(m, x, lab), G))
        assert bool(one) == on and bool(three) != on, (on, sorted(three), sorted(one))


@pytest.mark.parametrize("fwd_on", [True, False], ids=["fwd_tf32", "fwd_3pass"])
def test_backward_keeps_the_forward_mode(fwd_on):
    """Flipping the switches between a forward and its backward does not change the backward's GEMMs."""
    m = _module(19, 256, overlap_write=True)   # (two-stream: the weight operands are prepared on a side stream too)
    x, lab, G = _small_inputs()
    with tf32(fwd_on):
        outs = _fwd(m, x, lab)
    with tf32(not fwd_on):
        three, one = _kernels(lambda: _bwd(outs, G))
    assert bool(one) == fwd_on and bool(three) != fwd_on, (sorted(three), sorted(one))


def test_inference_cache_not_shared_between_modes():
    """The inference read's cached weight operand is per mode: a 3-pass read after a TF32 read (and back) gives the bits
    a module that never ran in the other mode gives."""
    from pinthememory_b200 import synth

    m = _module(19, 256).eval()
    fresh = {on: _clone_module(m) for on in (False, True)}
    x = synth.make_features(1, 256, 128, 256, seed=51, device="cuda")
    want = {}
    with torch.no_grad():
        for on in (False, True):
            with tf32(on):
                want[on] = fresh[on](x, None, False)[0]
        for on in (True, False, True, False):
            with tf32(on):
                three, one = _kernels(lambda: m(x, None, False))
                got = m(x, None, False)[0]
            assert bool(one) == on and bool(three) != on, (on, sorted(three), sorted(one))
            assert torch.equal(got.view(torch.int32), want[on].view(torch.int32)), on
            assert m._infer_cache[0][5] is on and (m._infer_cache[1][1] is None) == on


@pytest.mark.parametrize("capture_on", [True, False], ids=["captured_tf32", "captured_3pass"])
def test_graphed_step_keeps_its_capture_mode(capture_on):
    from pinthememory_b200.graphed import GraphedStep

    m = _module(19, 256)
    x, lab, G = _small_inputs()
    with tf32(capture_on):
        step = GraphedStep(m, x.detach(), lab, G)
        three, one = _kernels(step.replay)
        assert bool(one) == capture_on and bool(three) != capture_on, (sorted(three), sorted(one))
    with tf32(not capture_on):
        three, one = _kernels(step.replay)
    step.release()
    assert bool(one) == capture_on and bool(three) != capture_on, (sorted(three), sorted(one))


def test_tf32_deterministic_repeats_bitwise():
    """TF32 together with torch.use_deterministic_algorithms(True): two steps from the same state give the same bits."""
    was = torch.are_deterministic_algorithms_enabled()
    base = _module(19, 256, overlap_write=True)
    x, lab, G = _small_inputs()
    runs = []
    try:
        torch.use_deterministic_algorithms(True)
        with tf32(True):
            for _ in range(2):
                m = _clone_module(base)
                xi = x.detach().clone().requires_grad_(True)
                outs = _fwd(m, xi, lab)
                three, one = _kernels(lambda: _bwd(outs, G))
                assert one and not three
                runs.append([outs[0].detach(), outs[1].detach(), outs[2][0].detach(), outs[2][1].detach(),
                             m.m_items.detach(), xi.grad] + [p.grad for p in m.parameters() if p.grad is not None])
    finally:
        torch.use_deterministic_algorithms(was)
    for a, b in zip(*runs):
        assert torch.equal(a.view(torch.int32), b.view(torch.int32))
