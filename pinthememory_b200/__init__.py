"""pinthememory_b200 -- B200-native categorical class memory (drop-in for the reference's network/memory.py)."""
import sys

__all__ = ["Memory_sup", "Writingnet", "initialize_weights", "install", "enable_sharded_update", "GraphedStep", "PrototypePool", "initialize_memory",
           "upsampled_cross_entropy", "SegMetrics", "upsample_concat"]


def __getattr__(name):
    # lazy: importing the package (e.g. for synth / build) must not require the CUDA library
    if name in ("Memory_sup", "Writingnet", "initialize_weights"):
        from . import memory

        return getattr(memory, name)
    if name == "enable_sharded_update":
        from .sharding import enable_sharded_update

        return enable_sharded_update
    if name in ("PrototypePool", "initialize_memory", "upsampled_cross_entropy", "SegMetrics", "upsample_concat"):
        from . import callers

        return getattr(callers, name)
    if name == "GraphedStep":
        from .graphed import GraphedStep

        return GraphedStep
    raise AttributeError(name)


def install(module_name="network.memory"):
    """Make ``from network import memory`` / ``import network.memory`` resolve to this implementation.

    Call BEFORE the reference's head modules are imported (network/deepv3plus.py:32, deepv2.py:32 do
    ``from network import memory``), e.g. at the top of train.py / eval.py. If the ``network`` package is
    already imported its ``memory`` attribute is rebound as well.
    """
    from . import memory

    sys.modules[module_name] = memory
    pkg, _, attr = module_name.rpartition(".")
    if pkg and pkg in sys.modules:
        setattr(sys.modules[pkg], attr, memory)
    return memory
