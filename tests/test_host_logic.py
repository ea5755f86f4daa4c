"""CPU: host-side mirror of the reference interface (names, attributes, aliasing rules, install hook)."""
import sys

import pytest
import torch

from golden_util import load_golden
from oracle.ref_loader import build_reference_memory, reference_available


def _mem(K=19, C=64, **kw):
    from pinthememory_b200.memory import Memory_sup

    return Memory_sup(K, C, C, 0.8, 1.0, False, device="cpu", **kw)


def test_state_dict_keys_and_shapes_match_the_reference_fixture():
    meta, fx = load_golden("train_write_c64_blocky")
    mem = _mem(meta["K"], meta["C"])
    ref_keys = [k[len("state."):] for k in fx if k.startswith("state.")]
    sd = mem.state_dict()
    assert sorted(sd.keys()) == sorted(ref_keys)
    for k in ref_keys:
        assert tuple(sd[k].shape) == tuple(fx["state." + k].shape), k
    assert "m_items" not in sd
    mem.load_state_dict({k: fx["state." + k] for k in ref_keys})


def test_parameters_live_only_in_leaf_modules():
    """train.py:262-277 (put_theta) rewrites _parameters of child-less modules only."""
    mem = _mem()
    assert len(mem._parameters) == 0 and len(mem.writenet._parameters) == 0
    names = [n for n, _ in mem.named_parameters()]
    assert names == ["output.0.weight", "output.1.weight", "output.1.bias", "writenet.writefeat.0.weight",
                     "writenet.writefeat.1.weight", "writenet.writefeat.1.bias", "clsfier.weight", "clsfier.bias"]


def test_reference_initialisation():
    torch.manual_seed(0)
    mem = _mem(19, 256)
    assert torch.all(mem.output[1].weight == 1) and torch.allclose(mem.output[1].bias, torch.tensor(1e-4))
    assert float(mem.clsfier.bias.detach().abs().max()) == 0 and 5e-5 < float(mem.clsfier.weight.detach().std()) < 2e-4
    assert torch.allclose(mem.m_items.norm(dim=1), torch.ones(19), atol=1e-6)
    assert mem.m_items.dtype == torch.float32 and not mem.m_items.requires_grad
    assert (mem.momentum, mem.memory_size, mem.feature_dim, mem.temperature, mem.gumbel_read) == (0.8, 19, 256, 1.0, False)
    with pytest.raises(AssertionError):
        from pinthememory_b200.memory import Memory_sup

        Memory_sup(19, 128, 256, 0.8, 1.0, False, device="cpu")


def test_no_cpu_fallback():
    mem = _mem()
    x = torch.randn(1, 64, 4, 4)
    with pytest.raises(RuntimeError, match="no CPU path"):
        mem(x, None, False)
    with pytest.raises(RuntimeError, match="no CPU path"):
        mem.get_score(torch.randn(1, 4, 4, 64), None, mem.m_items)


def test_install_replaces_the_reference_module_name():
    import pinthememory_b200

    saved = {k: sys.modules.get(k) for k in ("network", "network.memory")}
    try:
        import types

        pkg = types.ModuleType("network")
        pkg.__path__ = []
        sys.modules["network"] = pkg
        mod = pinthememory_b200.install()
        from network import memory  # the import line of deepv3plus.py:32 / deepv2.py:32

        assert memory is mod and memory.Memory_sup is pinthememory_b200.Memory_sup
        for sym in ("Memory_sup", "Writingnet", "initialize_weights"):
            assert hasattr(memory, sym)
    finally:
        for k, v in saved.items():
            if v is None:
                sys.modules.pop(k, None)
            else:
                sys.modules[k] = v


def test_product_never_imports_the_oracle():
    import os

    root = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "pinthememory_b200")
    for fn in os.listdir(root):
        if fn.endswith(".py"):
            src = open(os.path.join(root, fn)).read()
            imports = [ln for ln in src.splitlines() if ln.lstrip().startswith(("import ", "from "))]
            assert not any("oracle" in ln for ln in imports), fn + " must not import oracle/"


def _surface(m):
    import inspect

    return {"named_modules": [n for n, _ in m.named_modules()], "forward": list(inspect.signature(m.forward).parameters),
            "init": list(inspect.signature(type(m).__init__).parameters)}


def test_attribute_surface_matches_the_live_reference():
    """Against the reference's surface stored in tests/golden/reference_surface.json, and against the live reference
    module as well where its source tree is mounted (PINMEM_REFERENCE_ROOT)."""
    import json
    import os

    with open(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "reference_surface.json")) as fh:
        ref = json.load(fh)
    if reference_available():
        live = build_reference_memory(19, 64)
        assert all(hasattr(live, name) for name in ref["attributes"])
        assert _surface(live) == {k: ref[k] for k in ("named_modules", "forward", "init")}
    mem = _mem()
    for name in ref["attributes"]:
        assert hasattr(mem, name), name
    for m in ("forward", "read", "write", "get_score"):
        assert callable(getattr(mem, m))
    got = _surface(mem)
    assert got["named_modules"] == ref["named_modules"]
    assert got["forward"] == ref["forward"]
    assert got["init"][:-1] == ref["init"] and got["init"][-1] == "device"


def test_bn_args_counter_is_bumped_once_and_only_deferred_for_cuda_buffers():
    """_bn_args applies nn.BatchNorm2d's own side effect (num_batches_tracked += 1) itself unless the normalise kernel can
    do it (CUDA int64 counter, fixed momentum): on CPU buffers it must never defer."""
    import torch
    import torch.nn as nn

    from pinthememory_b200.memory import _bn_args

    bn = nn.BatchNorm2d(8)
    bn.train()
    use_batch, rm, rv, factor, nbt = _bn_args(bn, defer_counter=True)
    assert use_batch and nbt is None and int(bn.num_batches_tracked) == 1 and factor == bn.momentum
    assert rm is bn.running_mean and rv is bn.running_var
    use_batch, rm, rv, factor = _bn_args(bn)
    assert int(bn.num_batches_tracked) == 2
    bn.momentum = None                       # cumulative average: the factor needs the bumped counter on the host
    *_, factor, nbt = _bn_args(bn, defer_counter=True)
    assert nbt is None and int(bn.num_batches_tracked) == 3 and abs(factor - 1.0 / 3.0) < 1e-12
    bn.eval()
    use_batch, rm, rv, factor, nbt = _bn_args(bn, defer_counter=True)
    assert not use_batch and nbt is None and int(bn.num_batches_tracked) == 3 and rm is bn.running_mean
