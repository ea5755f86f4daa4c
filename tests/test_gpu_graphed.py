"""The CUDA-graph captured step gives the results of the eagerly launched one (pinthememory_b200/graphed.py)."""
import pytest
import torch

from golden_util import assert_close
from pinthememory_b200 import synth

pytestmark = pytest.mark.gpu


@pytest.fixture(autouse=True)
def _exact_fp32_convs():
    old = (torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32)
    torch.backends.cudnn.allow_tf32 = False
    torch.backends.cuda.matmul.allow_tf32 = False
    yield
    torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32 = old


def _pair(K=19, C=64, gumbel=False):
    from pinthememory_b200.memory import Memory_sup

    torch.manual_seed(11)
    a = Memory_sup(K, C, C, 0.8, 1.0, gumbel).cuda()
    with torch.no_grad():
        a.clsfier.weight.normal_(0, 0.2)
    b = Memory_sup(K, C, C, 0.8, 1.0, gumbel).cuda()
    b.load_state_dict(a.state_dict())
    b.m_items = a.m_items.clone()
    return a, b


W = (0.02, 0.4, 0.2)


def _eager_step(mem, x, lab, G):
    x = x.detach().clone().requires_grad_(True)
    mem.zero_grad(set_to_none=True)
    uq, sq, sm, rl, wl = mem(x, lab, True, False)
    dev = x.device
    torch.autograd.backward([uq, rl, wl[0], wl[1]], [G] + [torch.tensor(v, device=dev) for v in W])
    return uq, sq, sm, rl, wl, x.grad


def test_graphed_training_steps_match_eager_steps():
    from pinthememory_b200.graphed import GraphedStep

    B, C, h, w, Hm, Wm, K = 2, 64, 12, 16, 48, 64, 19
    eager, graphed = _pair(K, C)
    batches = [(synth.make_features(B, C, h, w, seed=s, device="cuda"),
                synth.make_labels(B, Hm, Wm, K, "blocky", seed=s + 1).cuda(),
                synth.make_upstream_grad((B, C, h, w), seed=s + 2, device="cuda")) for s in (3, 40, 77)]
    step = GraphedStep(graphed, *batches[0], loss_weights=W, memory_writing=True, writing_detach=False)
    assert step.kernels_per_replay >= 15
    # capturing (and its warm-up) must not have advanced any state
    for (k, va), vb in zip(eager.state_dict().items(), graphed.state_dict().values()):
        assert torch.equal(va, vb), k
    assert torch.equal(eager.m_items, graphed.m_items)

    for x, lab, G in batches:
        uq, sq, sm, rl, wl, dx = _eager_step(eager, x, lab, G)
        out = step(x, lab, G)
        assert_close(out["updated_query"], uq, 1e-5, "updated_query")
        assert_close(out["score_query"], sq, 1e-5, "score_query")
        assert_close(out["score_memory"], sm, 1e-5, "score_memory")
        assert_close(out["readloss"], rl, 1e-5, "readloss")
        assert_close(out["writeloss"][0], wl[0], 1e-5, "div")
        assert_close(out["writeloss"][1], wl[1], 1e-5, "cls")
        assert_close(step.query_grad, dx, 1e-5, "dx")
        assert_close(graphed.m_items, eager.m_items, 1e-5, "memory")  # carried from step to step
        assert graphed.m_items.data_ptr() == step.memory.data_ptr()
        for (n, pa), pb in zip(eager.named_parameters(), graphed.parameters()):
            assert_close(pb.grad, pa.grad, 1e-4, "grad " + n)
    for (k, va), vb in zip(eager.state_dict().items(), graphed.state_dict().values()):
        assert_close(vb.float(), va.float(), 1e-5, k)  # BatchNorm running statistics advanced alike
    assert torch.equal(graphed.last_label_hist, eager.last_label_hist)


def test_graphed_eval_read_matches_eager():
    from pinthememory_b200.graphed import GraphedStep

    B, C, h, w, K = 1, 64, 16, 32, 19
    eager, graphed = _pair(K, C)
    eager.eval(), graphed.eval()
    x0 = synth.make_features(B, C, h, w, seed=1, device="cuda")
    step = GraphedStep(graphed, x0, None, memory_writing=False)
    m0 = eager.m_items.clone()
    for s in (5, 6):
        x = synth.make_features(B, C, h, w, seed=s, device="cuda")
        with torch.no_grad():
            uq, sq, sm, rl, wl = eager(x, None, False)
        out = step(x)
        assert_close(out["updated_query"], uq, 1e-5, "updated_query")
        assert_close(out["score_memory"], sm, 1e-5, "score_memory")
        assert out["readloss"] == 0 and out["writeloss"] == [0, 0]
    assert torch.equal(graphed.m_items, m0)


def test_graphed_gumbel_read_draws_fresh_noise_each_replay():
    from pinthememory_b200.graphed import GraphedStep

    B, C, h, w, K = 1, 64, 8, 8, 19
    _, graphed = _pair(K, C, gumbel=True)
    graphed.eval()
    x = synth.make_features(B, C, h, w, seed=1, device="cuda")
    step = GraphedStep(graphed, x, None, memory_writing=False)
    a = step(x)["score_memory"].clone()
    b = step(x)["score_memory"].clone()
    assert not torch.equal(a, b)
    assert_close(a.sum(-1), torch.ones_like(a.sum(-1)), 1e-5, "rows sum to one")


@pytest.mark.parametrize("graphed", [False, True])
def test_two_stream_forward_matches_single_stream(graphed):
    """overlap_write: the write branch on a side stream (a parallel branch when captured) changes nothing, with the read's
    own branches (label pass on the write stream, column softmax / weight work on a second side stream)."""
    from pinthememory_b200.graphed import GraphedStep

    B, C, h, w, Hm, Wm, K = 2, 64, 12, 16, 48, 64, 19
    plain, forked = _pair(K, C)
    forked.overlap_write = True
    batches = [(synth.make_features(B, C, h, w, seed=s, device="cuda"),
                synth.make_labels(B, Hm, Wm, K, "blocky", seed=s + 1).cuda(),
                synth.make_upstream_grad((B, C, h, w), seed=s + 2, device="cuda")) for s in (3, 40, 77)]
    step = GraphedStep(forked, *batches[0], loss_weights=W, memory_writing=True, writing_detach=False) if graphed else None
    for x, lab, G in batches:
        uq, sq, sm, rl, wl, dx = _eager_step(plain, x, lab, G)
        if graphed:
            out = step(x, lab, G)
            uq2, rl2, wl2, dx2 = out["updated_query"], out["readloss"], out["writeloss"], step.query_grad
        else:
            uq2, _, _, rl2, wl2, dx2 = _eager_step(forked, x, lab, G)
        torch.cuda.synchronize()
        assert_close(uq2, uq, 1e-5, "updated_query")
        assert_close(rl2, rl, 1e-5, "readloss")
        assert_close(wl2[0], wl[0], 1e-5, "div")
        assert_close(wl2[1], wl[1], 1e-5, "cls")
        assert_close(dx2, dx, 1e-5, "dx")
        assert_close(forked.m_items, plain.m_items, 1e-5, "memory")
        for (n, pa), pb in zip(plain.named_parameters(), forked.parameters()):
            assert_close(pb.grad, pa.grad, 1e-4, "grad " + n)
