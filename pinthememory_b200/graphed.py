"""CUDA-graph capture of a ``Memory_sup`` step.

One training step of the memory (forward, the weighted losses, backward) is ~45 short kernels; launched
one by one from Python the GPU idles ~20 % of the step waiting for the host. Every kernel of this package
is stream-ordered, allocates nothing and never synchronises, so the whole step can be captured once into
a CUDA graph and replayed with a single launch. The same holds for the whole segmentation network around
it (``torch.cuda.graph`` / ``make_graphed_callables`` over the reference's ``net(...)``); this helper is
the module-level version used by ``bench.py`` and the tests.

Static-shape contract (the usual CUDA-graph one): inputs are written into ``step.query`` / ``step.mask``
/ ``step.grad_updated_query`` (or passed to ``__call__``, which copies them there), results are read from
the returned static tensors and are overwritten by the next replay.

Memory state: the reference rebinds ``m_items`` to a fresh tensor on every write (memory.py:252-257). A
replayed graph reads and writes fixed addresses, so here the module's ``m_items`` is bound to the static
buffer ``step.memory`` and the captured step ends with ``memory <- updated memory`` (after the backward,
which still needs the old rows). Take ``step.memory.clone()`` for a snapshot (e.g. ``mem_t``, train.py:530).
"""
import torch

from . import capi


class GraphedStep:
    """Capture ``module(query, mask, memory_writing, writing_detach)`` (+ backward) and replay it.

    Parameters
    ----------
    module : Memory_sup (already on the device; train()/eval() mode is frozen into the graph)
    query : example features ``[B,C,h,w]`` (values are used for the warm-up runs)
    mask : example labels ``[B,Hm,Wm]`` int64, or None for a read without labels
    grad_updated_query : upstream gradient ``[B,C,h,w]`` of ``updated_query``; None captures forward only
    loss_weights : (read, div, cls) weights of the three auxiliary losses in the backward
                   (train.py:1213-1215 uses 0.02 / 0.4 / 0.2)
    carry_memory : end the step with ``memory <- updated memory`` (training); False replays from the
                   same memory every time
    autocast_dtype : run the module under ``torch.autocast`` (bf16 feature tensors)

    The modes the module reads from torch at call time -- deterministic algorithms, the TF32 switches (``capi.tf32``) --
    are fixed when the step is captured; changing them afterwards does not change what a replay runs.
    """

    def __init__(self, module, query, mask=None, grad_updated_query=None, loss_weights=(0.02, 0.4, 0.2),
                 memory_writing=True, writing_detach=True, carry_memory=True, autocast_dtype=None, warmup=3):
        capi.require_cuda(query)
        if capi._timing is not None:
            raise RuntimeError("pinmem_b200: per-kernel event timing cannot be on while capturing a graph")
        if memory_writing and mask is None:
            raise RuntimeError("pinmem_b200: memory_writing=True needs labels")
        dev = query.device
        self.module = module
        self.backward = grad_updated_query is not None
        self.memory_writing, self.writing_detach = memory_writing, writing_detach
        self.carry_memory = carry_memory and memory_writing
        self._autocast = autocast_dtype
        self.query = query.detach().clone().requires_grad_(self.backward)
        self.mask = mask.detach().clone() if mask is not None else None
        self.grad_updated_query = grad_updated_query.detach().clone() if self.backward else None
        self.memory = module.m_items.detach().clone()
        self._w = [torch.tensor(float(v), device=dev) for v in loss_weights]
        self._params = [p for p in module.parameters() if p.requires_grad]

        side = torch.cuda.Stream(device=dev)
        side.wait_stream(torch.cuda.current_stream(dev))
        with torch.cuda.stream(side):
            # warm-up outside the capture: library handles, cuDNN algorithm choice, allocator pools.
            # State that the step mutates is put back afterwards so that capturing has no side effect
            # beyond the single step the capture itself records but does not run.
            state = {k: v.detach().clone() for k, v in module.state_dict().items()}
            memory0 = self.memory.clone()
            for _ in range(warmup):
                self._run()
            module.load_state_dict(state)
            self.memory.copy_(memory0)
        torch.cuda.current_stream(dev).wait_stream(side)
        torch.cuda.synchronize(dev)

        self._clear_grads()
        self.graph = torch.cuda.CUDAGraph()
        n0 = capi.LAUNCHES
        with torch.cuda.graph(self.graph):
            self.outputs = self._run()
        self.kernels_per_replay = capi.LAUNCHES - n0  # this package's kernels inside one replay
        module.m_items = self.memory
        self.query_grad = self.query.grad if self.backward else None
        self.param_grads = [p.grad for p in self._params]  # static: rewritten (not accumulated) by every replay

    # ------------------------------------------------------------------------------------------

    def _clear_grads(self):
        self.query.grad = None
        for p in self._params:
            p.grad = None

    def _run(self):
        m = self.module
        m.m_items = self.memory
        if self.backward:
            self._clear_grads()
        ctx = torch.autocast("cuda", dtype=self._autocast, enabled=self._autocast is not None)
        with torch.set_grad_enabled(self.backward), ctx:
            uq, sq, sm, rl, wl = m(self.query, self.mask, self.memory_writing, self.writing_detach)
        if self.backward:
            outs, grads = [uq], [self.grad_updated_query.to(uq.dtype)]
            if torch.is_tensor(rl):
                outs.append(rl), grads.append(self._w[0])
            if self.memory_writing:
                outs += [wl[0], wl[1]]
                grads += [self._w[1], self._w[2]]
            torch.autograd.backward(outs, grads)
        new_memory = m.m_items.detach()
        if self.carry_memory:
            # after the backward: the read's saved memory IS self.memory
            self.memory.copy_(new_memory)
            new_memory = self.memory
        return {"updated_query": uq.detach(), "score_query": sq.detach(), "score_memory": sm.detach(),
                "readloss": rl.detach() if torch.is_tensor(rl) else rl,
                "writeloss": [w.detach() if torch.is_tensor(w) else w for w in wl],
                "memory": new_memory}

    def replay(self):
        """Run the captured step on whatever the static input buffers hold; returns the static outputs."""
        if self.graph is None:
            raise RuntimeError("pinmem_b200: this GraphedStep was released")
        self.graph.replay()
        self.module.m_items = self.memory
        if self.backward:
            self.query.grad = self.query_grad
            for p, g in zip(self._params, self.param_grads):
                p.grad = g
        return self.outputs

    def release(self):
        """Free the captured graph. Required before ``destroy_process_group()`` when the step contains the
        sharded update: NCCL will not tear down a communicator that a live graph still references (it hangs)."""
        if self.graph is not None:
            torch.cuda.synchronize()
            self.graph.reset()
            self.graph = None
        self.outputs = None

    def __call__(self, query=None, mask=None, grad_updated_query=None):
        if query is not None:
            self.query.data.copy_(query, non_blocking=True)
        if mask is not None:
            self.mask.copy_(mask, non_blocking=True)
        if grad_updated_query is not None:
            self.grad_updated_query.copy_(grad_updated_query, non_blocking=True)
        return self.replay()
