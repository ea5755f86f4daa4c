#!/usr/bin/env python
"""Benchmark of the categorical-memory hot path (BASELINE.json metric) on B200.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dtype f32|bf16]
                    [--workload cfg2_module_os8_b8] [--labels blocky|iid] [--dump-outputs DIR]

One "step" = one pass of the hot path over one batch of synthetic input: ``Memory_sup.forward(query, labels,
memory_writing=True, writing_detach=False)`` + backward of ``<G, updated_query> + 0.02*readloss + 0.4*div +
0.2*cls`` (loss weights train.py:1213-1215), i.e. memory read + update, forward + backward, BN in train mode.
The metric is feature-map Mpixels/s. Prints ONE JSON line (rank 0).

* ``value``      whole module (every kernel ours, incl. the two 1x1 convolutions as tcgen05 GEMMs), inputs resident in HBM
* ``e2e``        the same call with HOST (pinned) inputs: H2D of features+labels and D2H of losses+memory per step
* ``core``       only the hand-written kernels (write feature f and upstream du given), with the aggregate
                 fraction of the HBM roofline for A_train bytes/pixel (SURVEY.md 8d)
* ``roofline``   the dominant kernel: algorithmic bytes / its CUDA-event duration measured inside the timed region
* ``cpu_baseline`` the reference's own module (byte-compiled into oracle/_ref/, else the oracle/ port) timed on this host's cores on a bounded sample
``--impl reference`` times that CPU arm instead (all host threads, the workload's full batch) and prints the same
line shape. Each timed region of the workload runs exactly ``--steps`` steps after ``--warmup`` untimed ones (``e2e``
half as many, at least 5, after 3); the short runs of the other configs repeat fixed blocks and report the median block
(``timing`` gives each region's blocks and their milliseconds). ``--impl reference`` is the exception: it warms up with
at most 2 steps (the eval read with exactly 2), and on the training workloads it stops timing after 120 s (at least 3
steps), since a full-batch CPU step can take seconds; ``sample`` reports the steps it timed.
``--dump-outputs DIR`` writes what the headline path computed in its last timed step; the inputs are seeded, so two
builds run with the same arguments can be compared output for output.
Under torchrun (N>1) every rank runs its own batch (weak scaling); the write path all-reduces the class sums.
"""
import argparse
import json
import os
import statistics
import sys
import threading
import time

import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

from pinthememory_b200 import synth  # noqa: E402

METRIC = "memory read+update fwd+bwd Mpixels/s"
UNIT = "Mpixels/s"
K, C = 19, 256
LOSS_W = dict(read=0.02, div=0.4, cls=0.2)


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    # 600 steps of the ~0.83 ms default step keep the headline's single timed window at about 0.5 s
    ap.add_argument("--steps", type=int, default=600)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--dtype", default="f32", choices=["f32", "bf16"])
    ap.add_argument("--workload", default="cfg2_module_os8_b8", choices=sorted(synth.WORKLOADS))
    ap.add_argument("--labels", default="blocky", choices=["blocky", "iid"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-callers", action="store_true", help="skip the timings of the callers (main loss, prototype pooling)")
    ap.add_argument("--core-serial", action="store_true", help="core graph as one linear chain (no parallel write branch)")
    ap.add_argument("--overlap-write", action="store_true", help="write branch on a side stream (parallel graph branch)")
    ap.add_argument("--no-graph", action="store_true", help="headline = kernel-by-kernel launches instead of the CUDA graph")
    ap.add_argument("--no-extra", action="store_true", help="skip the short runs of the other BASELINE configs (cfg 3/4/5)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write what the headline path computed in its last timed step as DIR/<name>.npy (float32, or "
                         "float64 where the output is); outputs above %d elements are replaced by a fixed seeded sample "
                         "of %d of their elements" % (DUMP_FULL_MAX, DUMP_SAMPLE))
    args = ap.parse_args()
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes the outputs of --impl ours")
    return args


# ------------------------------------------------------------------------------------------ output dump

DUMP_FULL_MAX = 1 << 21   # outputs up to this many elements are written whole
DUMP_SAMPLE = 1 << 20     # larger ones as this many elements at seeded flat positions (the same for every run)
DUMP_MAX_BYTES = 64 << 20


def dump_arrays(named):
    """{name: tensor} -> {name: float32 | float64 numpy array}, sampled as --dump-outputs describes. Call right after the
    timed steps: the tensors are the step's static outputs and the next step overwrites them."""
    out = {}
    for name, t in named.items():
        if t.numel() > DUMP_FULL_MAX:
            g = torch.Generator().manual_seed(synth.SEED)
            idx = torch.randint(t.numel(), (DUMP_SAMPLE,), generator=g).sort().values
            t = t.reshape(-1)[idx.to(t.device)]
        out[name] = t.to(torch.float64 if t.dtype == torch.float64 else torch.float32).cpu().numpy()
    total = sum(a.nbytes for a in out.values())
    if total > DUMP_MAX_BYTES:
        raise RuntimeError("--dump-outputs: %d bytes exceed the %d byte bound" % (total, DUMP_MAX_BYTES))
    return out


def write_dump(out_dir, arrays):
    import numpy as np

    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)


def step_outputs(uq, sq, sm, rl, wl, memory=None, grad_query=None, param_grads=()):
    """The arrays a caller of Memory_sup.forward (+ backward) receives, by name; int zeros of an absent loss are left out.
    Detached: a kept reference to the step's autograd graph would keep its AccumulateGrad nodes alive, and a later CUDA
    graph capture of the same parameters on another stream then fails."""
    named = {"updated_query": uq, "score_query": sq, "score_memory": sm}
    for n, v in (("readloss", rl), ("div_loss", wl[0]), ("cls_loss", wl[1]), ("m_items", memory), ("grad_query", grad_query)):
        if torch.is_tensor(v):
            named[n] = v
    for n, g in param_grads:
        if g is not None:
            named["grad." + n] = g
    return {n: t.detach() for n, t in named.items()}


def tensor_peak(dt):
    """Dense tensor peak for the GEMMs: MEASURED_PEAKS.json's cuBLAS bf16 burst figure; TF32 runs at half the bf16 rate."""
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    try:
        with open(path) as fh:
            bf16 = float(json.load(fh)["bf16_tflops"])
        src = "measured bf16 burst (MEASURED_PEAKS.json)"
    except Exception:
        bf16, src = 1590.0, "fallback (B200_PROFILING.md 1.59 PFLOP/s)"
    if dt == torch.float32:
        return bf16 / 2.0, src + " / 2 for TF32"
    return bf16, src


def exchange_name(module):
    """Which exchange a sharded module uses for the class sums / their gradient."""
    g = getattr(module, "shard_group", None)
    if g is None or g.world_size <= 1:
        return "none (single rank)"
    if getattr(g, "peer", None) is not None:
        return "fused into the update kernels over NVLink peer memory (pm_update_fwd_peer / pm_update_bwd_peer), no NCCL node"
    return "two NCCL all-reduces (%s)" % (getattr(g, "peer_error", None) or "peer exchange disabled")


def measured_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    try:
        with open(path) as fh:
            return float(json.load(fh)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


# ------------------------------------------------------------------------------------- clock sampler


class ClockSampler:
    """Samples SM clock and throttle reasons through NVML while the timed region runs."""

    def __init__(self, index):
        self.samples, self.reasons, self.max_mhz = [], set(), None
        self._stop = threading.Event()
        self._thread = None
        try:
            import pynvml

            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
        except Exception:
            self.nv = None

    def _loop(self):
        nv = self.nv
        names = {"hw_slowdown": 0x8, "sw_thermal_slowdown": 0x20, "hw_thermal_slowdown": 0x40,
                 "hw_power_brake": 0x80, "sw_power_cap": 0x4, "sync_boost": 0x10, "applications_clocks": 0x2}
        while not self._stop.is_set():
            try:
                self.samples.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                for n, bit in names.items():
                    if r & bit:
                        self.reasons.add(n)
            except Exception:
                pass
            time.sleep(0.005)

    def __enter__(self):
        if self.nv is not None:
            self._thread = threading.Thread(target=self._loop, daemon=True)
            self._thread.start()
        return self

    def __exit__(self, *a):
        self._stop.set()
        if self._thread is not None:
            self._thread.join()

    def summary(self):
        if not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": self.max_mhz, "reasons": ["unavailable"]}
        return {"sm_mhz": statistics.median(self.samples), "sm_max_mhz": self.max_mhz,
                "reasons": sorted(self.reasons), "samples": len(self.samples)}


def _bind_to_gpu_numa_node(index):
    """Run this rank (and first-touch its pinned staging buffers) on the CPUs next to its GPU, so that N ranks
    uploading at once do not all cross the same socket link (e2e with host buffers is PCIe/host-memory bound)."""
    try:
        import pynvml

        pynvml.nvmlInit()
        pynvml.nvmlDeviceSetCpuAffinity(pynvml.nvmlDeviceGetHandleByIndex(index))
    except Exception:
        pass


# ------------------------------------------------------------------------------------ CPU reference


def host_threads():
    """All the cores this process may use (torchrun exports OMP_NUM_THREADS=1: undo it explicitly)."""
    try:
        n = len(os.sched_getaffinity(0))
    except Exception:
        n = os.cpu_count() or 1
    torch.set_num_threads(max(1, n))
    return torch.get_num_threads()


def reference_module(device, gumbel=False):
    """The reference's OWN ``Memory_sup`` (unmodified, byte-compiled into oracle/_ref/ by oracle/build_ref.py, or loaded from
    /root/reference where that is mounted) on ``device``; None when neither is there (the oracle port is used then)."""
    try:
        from oracle import ref_loader

        if not (ref_loader.reference_available() or ref_loader.compiled_reference_available()):
            return None
        cpu = torch.device(device).type == "cpu"
        m = ref_loader.build_reference_memory(K, C, 0.8, 1.0, gumbel, force_cpu=cpu)
        if not cpu:
            m = m.to(device)
            m.m_items = m.m_items.to(device)
            m.mem_cls = m.mem_cls.to(device)
        return m
    except Exception:
        return None


def cpu_reference_run(wl, kind, steps, warmup, sample_B=None, budget_s=120.0):
    """The reference module on the host cores, on the workload's own batch (or a bounded sample of it), all host threads:
    the reference's own ``network/memory.py`` when oracle/_ref holds it (``kind: "reference"``), else the oracle port
    (``kind: "port"``). Stops early when the time budget is spent (the step count actually timed is reported)."""
    from oracle import memory_oracle as mo
    from oracle import ref_loader

    cores = host_threads()
    torch.manual_seed(synth.SEED)
    B = wl["B"] if sample_B is None else min(sample_B, wl["B"])
    mem = reference_module("cpu")
    impl_kind = "reference" if mem is not None else "port"
    if mem is None:
        mem = mo.OracleMemorySup(K, C, C, 0.8, 1.0, False)
    mem.train()
    x = synth.make_features(B, C, wl["h"], wl["w"]).requires_grad_(True)
    labels = synth.make_labels(B, wl["Hm"], wl["Wm"], K, kind)
    G = synth.make_upstream_grad((B, C, wl["h"], wl["w"]))
    M0 = mem.m_items.clone()
    times = []
    t_start = time.perf_counter()
    for i in range(warmup + steps):
        mem.m_items = M0
        x.grad = None
        mem.zero_grad(set_to_none=True)
        t0 = time.perf_counter()
        with ref_loader.cuda_identity(force=True):   # the reference calls .cuda() inside write() (memory.py:246)
            uq, _, _, rl, wlss = mem(x, labels, True, False)
            torch.autograd.backward([uq, rl, wlss[0], wlss[1]],
                                    [G, torch.tensor(LOSS_W["read"]), torch.tensor(LOSS_W["div"]),
                                     torch.tensor(LOSS_W["cls"])])
        t1 = time.perf_counter()
        if i >= warmup:
            times.append(t1 - t0)
        if len(times) >= 3 and t1 - t_start > budget_s:
            break
    px = B * wl["h"] * wl["w"]
    total = sum(times)
    return dict(value=px * len(times) / total / 1e6, ms_per_step=1e3 * total / len(times), cores=cores,
                same_config=(B == wl["B"]), kind=impl_kind,
                sample="B=%d of the workload's %d images per step (%dx%d features, %dx%d labels), %d timed steps, %d threads" %
                       (B, wl["B"], wl["h"], wl["w"], wl["Hm"], wl["Wm"], len(times), cores))


# ------------------------------------------------------------------------- eval read (BASELINE cfg 5)


def eval_read_main(args, wl):
    """`--workload cfg5_dr101v2_eval_b1`: the eval-mode memory read (no labels, no write, Gumbel read on as in
    the reference's default) on one full-resolution Cityscapes feature map per GPU. No collective: replicas."""
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    B, h, w = wl["B"], wl["h"], wl["w"]
    N = B * h * w
    line = {"metric": "memory read fwd (eval, no labels) Mpixels/s", "unit": UNIT, "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "data": "synthetic", "dtype": args.dtype,
            "config": {"workload": "%s: per-GPU batch %d, %dx%d feature map (OS8 of 1024x2048), C=%d, K=%d, no labels, "
                                   "gumbel read on, eval-mode BatchNorm; replicas only (no collective)" %
                                   (args.workload, B, h, w, C, K),
                       "l2": "L2 flushed between timed steps by writing a 256 MB buffer (the 100 MB working set fits L2)"}}
    if args.impl == "reference":
        if rank != 0:
            return
        from oracle import memory_oracle as mo

        from oracle import ref_loader

        host_threads()
        torch.manual_seed(synth.SEED)
        ora = reference_module("cpu", gumbel=True)      # the reference's own module when oracle/_ref holds it
        kind_ = "reference" if ora is not None else "port"
        if ora is None:
            ora = mo.OracleMemorySup(K, C, C, 0.8, 1.0, True)
        ora.eval()
        x = synth.make_features(B, C, h, w)
        times = []
        with torch.no_grad(), ref_loader.cuda_identity(force=True):
            for i in range(2 + args.steps):
                t0 = time.perf_counter()
                ora(x, None, False)
                if i >= 2:
                    times.append(time.perf_counter() - t0)
        v = N * len(times) / sum(times) / 1e6
        line.update({"impl": "reference", "value": v, "ms_per_step": 1e3 * sum(times) / len(times), "dtype": "f32",
                     "gpu_launches": 0,
                     "cpu_baseline": {"value": v, "unit": UNIT, "cores": torch.get_num_threads(), "kind": kind_,
                                      "sample": "the full per-GPU step (B=%d), %d timed steps" % (B, len(times))},
                     "e2e": {"value": v, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}})
        print(json.dumps(line))
        return
    if not torch.cuda.is_available():
        raise SystemExit("bench.py --impl ours needs a CUDA device (no CPU fallback)")
    import torch.distributed as dist

    from pinthememory_b200 import capi
    from pinthememory_b200.graphed import GraphedStep
    from pinthememory_b200.memory import Memory_sup

    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    dt = torch.float32 if args.dtype == "f32" else torch.bfloat16
    esz = 4 if dt == torch.float32 else 2
    torch.manual_seed(synth.SEED)
    mem = Memory_sup(K, C, C, 0.8, 1.0, True).to(dev).eval()
    x_host = synth.make_features(B, C, h, w, seed=synth.SEED + 100 * rank, dtype=dt).pin_memory()
    x = x_host.to(dev)
    flush = torch.empty(64 * 1024 * 1024, dtype=torch.float32, device=dev)
    autocast = torch.autocast("cuda", dtype=torch.bfloat16, enabled=(dt == torch.bfloat16))

    def eager_step(xin=x):
        with torch.no_grad(), autocast:
            return mem(xin, None, False)

    def run(fn, steps, warmup, clocks=False):
        """Each timed step is bracketed by its own events; the L2 flush between steps is not counted."""
        for _ in range(warmup):
            fn()
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        sampler = ClockSampler(local_rank) if clocks else None
        if sampler:
            sampler.__enter__()
        evs = []
        for _ in range(steps):
            flush.zero_()
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            fn()
            b.record()
            evs.append((a, b))
        torch.cuda.synchronize()
        if sampler:
            sampler.__exit__()
        ms = sum(a.elapsed_time(b) for a, b in evs)
        if world > 1:
            t = torch.tensor([ms], device=dev, dtype=torch.float64)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = float(t.item())
        return ms / steps, (sampler.summary() if sampler else None)

    ms_eager, _ = run(eager_step, args.steps, args.warmup)
    capi.enable_kernel_timing(True)
    capi.reset_counters()

    def eager_step_queued():   # behind a device-side sleep: the events bracket the kernels, not the Python between launches
        torch.cuda._sleep(2_000_000)
        eager_step()

    run(eager_step_queued, 20, 2)
    ktimes = capi.kernel_timings_ms()
    launches_per_step = capi.LAUNCHES / 22.0
    capi.enable_kernel_timing(False)
    gstep = GraphedStep(mem, x, None, memory_writing=False, autocast_dtype=torch.bfloat16 if dt == torch.bfloat16 else None)
    ms_graph, clocks = run(gstep.replay, args.steps, args.warmup, clocks=True)
    if args.dump_outputs and rank == 0:
        o = gstep.outputs
        write_dump(args.dump_outputs, dump_arrays(step_outputs(o["updated_query"], o["score_query"], o["score_memory"],
                                                               o["readloss"], o["writeloss"])))

    res_host = torch.empty(N, dtype=torch.uint8).pin_memory()

    def e2e_step():
        xin = x_host.to(dev, non_blocking=True)
        out = eager_step(xin)
        res_host.copy_(out[2].view(N, K).argmax(1).to(torch.uint8), non_blocking=True)

    ms_e2e, _ = run(e2e_step, max(args.steps // 2, 5), 3)
    peak, peak_src = measured_peaks()
    kavg = {k: sum(v) / len(v) for k, v in ktimes.items()}
    alg = {"pm_read_fwd": N * (3 * C * esz + 4 * 20 + 4 * K + 4 * K),      # x -> u, s, score_memory; Gumbel noise in
           "pm_colsoftmax_apply": N * (4 * 20 + 4 * K + 4 * K),
           "pm_bn_apply": N * C * esz * 2}
    kernels = {k: {"ms": round(t, 5), **({"alg_MB": round(alg[k] / 1e6, 2), "GBps": round(alg[k] / t / 1e6, 1),
                                          "frac": round(alg[k] / t / 1e6 / peak, 4)} if k in alg else {})}
               for k, t in kavg.items()}
    dom = max((k for k in kavg if k in alg), key=lambda k: kavg[k])
    a_eval = 3 * C * esz + 8 * K
    line.update({"value": world * N / (ms_graph * 1e-3) / 1e6, "ms_per_step": ms_graph,
                 "gpu_launches": int(gstep.kernels_per_replay * args.steps), "clocks": clocks,
                 "eager_launch": {"value": world * N / (ms_eager * 1e-3) / 1e6, "ms_per_step": ms_eager,
                                  "gpu_launches_per_step": launches_per_step},
                 "cuda_graph": {"kernels_per_replay": gstep.kernels_per_replay},
                 "e2e": {"value": world * N / (ms_e2e * 1e-3) / 1e6, "unit": UNIT, "ms_per_step": ms_e2e,
                         "h2d_bytes_per_step": x_host.numel() * x_host.element_size(), "d2h_bytes_per_step": N,
                         "what": "pinned-host features in, per-pixel memory-slot argmax (uint8) out, every step"},
                 "roofline": {"bound": "hbm", "kernel": dom, "achieved": kernels[dom]["GBps"], "peak": peak, "unit": "GB/s",
                              "frac": kernels[dom]["frac"], "traffic": None, "peak_source": peak_src,
                              "alg_bytes_per_launch": alg[dom], "launch_ms": kernels[dom]["ms"]},
                 "module_frac_of_peak": {"a_eval_bytes_per_pixel": a_eval,
                                         "frac": N * a_eval / (ms_graph * 1e-3) / 1e9 / peak},
                 "kernels": kernels})
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        from oracle import memory_oracle as mo

        from oracle import ref_loader

        host_threads()
        ora = reference_module("cpu", gumbel=True)
        kind_ = "reference" if ora is not None else "port"
        if ora is None:
            ora = mo.OracleMemorySup(K, C, C, 0.8, 1.0, True)
        ora.eval()
        xc = x_host.float()
        times = []
        with torch.no_grad(), ref_loader.cuda_identity(force=True):
            for i in range(5):
                t0 = time.perf_counter()
                ora(xc, None, False)
                if i >= 2:
                    times.append(time.perf_counter() - t0)
        line["cpu_baseline"] = {"value": N * len(times) / sum(times) / 1e6, "unit": UNIT, "cores": torch.get_num_threads(),
                                "kind": kind_, "sample": "the full per-GPU step (B=%d), 3 timed steps" % B}
    if rank == 0:
        print(json.dumps(line), flush=True)
    gstep.release()
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


# ------------------------------------------------------------ the other BASELINE configs (short runs)


def extra_configs(args, dev, dt, world, rank, mem0, timed):
    """cfg 4 (data-parallel OS16, GLOBAL batch 64 -> 64/N images per GPU, sharded update), cfg 5 (eval read of one
    1024x2048 image per GPU, replicas) and cfg 3 (the module's share of one GS meta-train step, 4 forwards + 3
    backwards, OS16 batch 4) -- each a short timed run on the same kernels, reported next to the headline."""
    import torch.distributed as dist

    from pinthememory_b200 import sharding
    from pinthememory_b200.graphed import GraphedStep
    from pinthememory_b200.memory import Memory_sup
    from pinthememory_b200.metastep import meta_step

    out = {}
    ac = torch.bfloat16 if dt == torch.bfloat16 else None
    state = {k: v.detach().clone() for k, v in mem0.state_dict().items()}

    def fresh(gumbel=False, shard=False):
        m = Memory_sup(K, C, C, 0.8, 1.0, gumbel).to(dev)
        m.load_state_dict(state)
        m.m_items = mem0.m_items.detach().clone()
        if shard and world > 1:
            sharding.enable_sharded_update(m)
            m.overlap_write = True
        return m

    try:   # ---- cfg 4
        Bg = 64
        Bl = max(Bg // world, 1)
        w4 = synth.WORKLOADS["cfg4_dp_os16_b8"]
        m = fresh(shard=True)
        if world > 1:   # the reference's multi-GPU scripts pass --syncbn (train.py:95): batch statistics of the GLOBAL batch
            m = torch.nn.SyncBatchNorm.convert_sync_batchnorm(m)
        m = m.train()
        seed = synth.SEED + 100 * rank + 7
        x4 = synth.make_features(Bl, C, w4["h"], w4["w"], seed=seed, dtype=dt, device=dev)
        l4 = synth.make_labels(Bl, w4["Hm"], w4["Wm"], K, args.labels, seed=seed + 2, device=dev)
        G4 = synth.make_upstream_grad((Bl, C, w4["h"], w4["w"]), seed=seed + 3, dtype=dt, device=dev)
        m.overlap_write = True
        gs = GraphedStep(m, x4, l4, G4, loss_weights=(LOSS_W["read"], LOSS_W["div"], LOSS_W["cls"]), memory_writing=True,
                         writing_detach=False, carry_memory=True, autocast_dtype=ac)
        ms, _, _, _ = timed(gs.replay, 20, 3, min_total_ms=100.0)
        ms /= 20
        out["cfg4_dp_os16_global_batch_64"] = {
            "ms_per_step": ms, "value": Bg * w4["h"] * w4["w"] / (ms * 1e-3) / 1e6, "unit": UNIT, "scaling": "strong",
            "per_gpu_batch": Bl, "what": "DR50V3P shape (48x48 features, 768x768 labels), global batch 64 split over %d "
                                         "GPU(s), class sums|counts exchanged before the update (%s), %s, CUDA graph "
                                         "replay" % (world, exchange_name(m),
                                                     "SyncBatchNorm as under --syncbn (statistics all-reduced out of the GEMM "
                                                     "epilogue, 4 small NCCL all-reduces per step)" if world > 1 else
                                                     "BatchNorm2d")}
        gs.release()
        del gs, m, x4, l4, G4
    except Exception as e:
        out["cfg4_dp_os16_global_batch_64"] = {"error": str(e)[:300]}

    try:   # ---- cfg 5: replicas, no collective
        w5 = synth.WORKLOADS["cfg5_dr101v2_eval_b1"]
        m = fresh(gumbel=True).eval()
        x5 = synth.make_features(w5["B"], C, w5["h"], w5["w"], seed=synth.SEED + 100 * rank + 9, dtype=dt, device=dev)
        gs = GraphedStep(m, x5, None, memory_writing=False, autocast_dtype=ac)
        flush = torch.empty(64 * 1024 * 1024, dtype=torch.float32, device=dev)
        for _ in range(3):
            gs.replay()
        evs = []
        for _ in range(20):
            flush.zero_()
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            gs.replay()
            b.record()
            evs.append((a, b))
        torch.cuda.synchronize()
        ms = statistics.median(a.elapsed_time(b) for a, b in evs)
        if world > 1:
            t = torch.tensor([ms], device=dev, dtype=torch.float64)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = float(t.item())
        n5 = w5["B"] * w5["h"] * w5["w"]
        a_eval = 3 * C * (4 if dt == torch.float32 else 2) + 8 * K
        out["cfg5_dr101v2_eval_read"] = {
            "ms_per_image": ms, "value": world * n5 / (ms * 1e-3) / 1e6, "unit": UNIT,
            "frac_of_hbm_roofline": n5 * a_eval / (ms * 1e-3) / 1e9 / measured_peaks()[0],
            "what": "eval-mode read of one 128x256 feature map (1024x2048 image) per GPU, gumbel read on, L2 flushed "
                    "between images, CUDA graph replay; %d replica(s), no collective" % world}
        gs.release()
        del gs, m, x5, flush
    except Exception as e:
        out["cfg5_dr101v2_eval_read"] = {"error": str(e)[:300]}

    if world == 1:
        try:   # ---- cfg 3: the memory module's part of one meta-train step (pinthememory_b200/metastep.py)
            w3 = synth.WORKLOADS["cfg3_meta_os16_b4"]
            net, upd, upd2 = fresh().train(), fresh().train(), fresh().train()
            mk = lambda sd: synth.make_features(w3["B"], C, w3["h"], w3["w"], seed=sd, dtype=dt, device=dev)
            x_tr, x_te = mk(21), mk(22)
            l_tr = synth.make_labels(w3["B"], w3["Hm"], w3["Wm"], K, args.labels, seed=23, device=dev)
            l_te = synth.make_labels(w3["B"], w3["Hm"], w3["Wm"], K, args.labels, seed=24, device=dev)
            Gt = synth.make_upstream_grad((w3["B"], C, w3["h"], w3["w"]), seed=25, dtype=dt, device=dev)
            mem_start = net.m_items.detach().clone()

            def step3():
                net.m_items = mem_start
                with torch.autocast("cuda", dtype=torch.bfloat16, enabled=ac is not None):
                    meta_step(net, upd, upd2, x_tr, l_tr, x_te, l_te, Gt, Gt, inner_lr=0.01)

            ms, _, _, _ = timed(step3, 5, 2, min_total_ms=100.0)
            ms /= 5
            n3 = 2 * w3["B"] * w3["h"] * w3["w"]
            graphed = None
            if not args.no_graph:   # the same seven passes captured once and replayed (no host work between kernels)
                try:
                    # fresh modules that only ever ran on the warm-up / capture stream: the AccumulateGrad nodes of
                    # parameters that stepped on the main stream would pull that stream into the capture
                    side = torch.cuda.Stream(device=dev)
                    side.wait_stream(torch.cuda.current_stream(dev))
                    with torch.cuda.stream(side):
                        net_g, upd_g, upd2_g = fresh().train(), fresh().train(), fresh().train()
                        mem_g = net_g.m_items.detach().clone()

                        def step3g():
                            net_g.m_items = mem_g
                            with torch.autocast("cuda", dtype=torch.bfloat16, enabled=ac is not None):
                                meta_step(net_g, upd_g, upd2_g, x_tr, l_tr, x_te, l_te, Gt, Gt, inner_lr=0.01)

                        for _ in range(2):
                            step3g()
                    torch.cuda.current_stream(dev).wait_stream(side)
                    torch.cuda.synchronize()
                    g3 = torch.cuda.CUDAGraph()
                    with torch.cuda.graph(g3, stream=side):
                        step3g()
                    msg, _, _, _ = timed(g3.replay, 10, 3, min_total_ms=100.0)
                    step3()             # the eagerly launched step on its own modules, same inputs and state
                    g3.replay()
                    torch.cuda.synchronize()
                    worst = 0.0
                    ge = dict(net.named_parameters())
                    for k, p in net_g.named_parameters():
                        a, b = p.grad.float(), ge[k].grad.float()
                        worst = max(worst, float((a - b).norm() / b.norm().clamp_min(1e-30)))
                    worst = max(worst, float((net_g.m_items - net.m_items).norm() / net.m_items.norm()))
                    graphed = {"ms_per_step": msg / 10, "value": n3 / (msg / 10 * 1e-3) / 1e6,
                               "max_rel_l2_vs_eager_launch": worst,
                               "what": "the same step captured as one CUDA graph and replayed; gradients of all parameters "
                                       "and the final memory compared with the eagerly launched step"}
                    g3.reset()
                    del g3
                except Exception as e:
                    graphed = {"error": str(e)[:200]}
            out["cfg3_meta_train_step"] = {
                "ms_per_step": ms, "value": n3 / (ms * 1e-3) / 1e6, "unit": UNIT, "cuda_graph": graphed,
                "what": "4 forwards + 3 backwards of the module per step as in train.py:530-583 (write with graph + "
                        "backward(retain_graph), functional theta' through _parameters, write on the saved memory, read of "
                        "the graph-carrying memory + backward, no-grad eval write), OS16 batch 4 meta-train + 4 meta-test "
                        "images; launched kernel by kernel (host-bound); pixels = meta-train + meta-test feature pixels"}
        except Exception as e:
            out["cfg3_meta_train_step"] = {"error": str(e)[:300]}
    return out


# -------------------------------------------------------------------------------------------- main


def main():
    args = parse()
    wl = synth.WORKLOADS[args.workload]
    if wl["Hm"] == 0:
        return eval_read_main(args, wl)
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    workload_desc = ("%s: per-GPU batch %d, %dx%d feature map, C=%d, K=%d, labels %dx%d int64 (%s), gumbel off, "
                     "momentum 0.8, T=1" % (args.workload, wl["B"], wl["h"], wl["w"], C, K, wl["Hm"], wl["Wm"],
                                            args.labels))
    base = {"metric": METRIC, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "data": "synthetic",
            "dtype": args.dtype,
            "config": {"workload": workload_desc,
                       "l2": "no flush: per-step working set (x,f,u,du,dx,df + labels ~ %d MB in fp32) exceeds the 126 MB L2"
                             % round((10 * C * 4 + 8 * wl["Hm"] * wl["Wm"] / (wl["h"] * wl["w"])) * wl["B"] * wl["h"] * wl["w"] / 1e6)}}

    if args.impl == "reference":
        if rank != 0:
            return
        r = cpu_reference_run(wl, args.labels, args.steps, min(args.warmup, 2))
        line = dict(base)
        line.update({"impl": "reference", "value": r["value"], "ms_per_step": r["ms_per_step"], "n_gpus": args.gpus,
                     "dtype": "f32", "gpu_launches": 0, "same_config": r["same_config"],
                     "cpu_baseline": {"value": r["value"], "unit": UNIT, "cores": r["cores"], "kind": r["kind"],
                                      "sample": r["sample"]},
                     "e2e": {"value": r["value"], "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
                     "note": ("reference's own CPU path = %s; torch %s, %d threads; one rank's batch (the metric is "
                              "per-pixel throughput, the CPU arm does not scale with --gpus)" %
                              ("the reference's unmodified network/memory.py::Memory_sup, byte-compiled into oracle/_ref/ "
                               "(oracle/build_ref.py)" if r["kind"] == "reference" else
                               "oracle/ port of network/memory.py (oracle/_ref/ is not on this box)",
                               torch.__version__, r["cores"]))})
        print(json.dumps(line))
        return

    if not torch.cuda.is_available():
        raise SystemExit("bench.py --impl ours needs a CUDA device (no CPU fallback)")
    import torch.distributed as dist

    from pinthememory_b200 import capi, sharding
    from pinthememory_b200.memory import Memory_sup, _ReadFn, _WriteFn

    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    # the configuration the parity tests check: no TF32 in any torch/cuDNN op (this package's own GEMMs are 3xTF32 with
    # fp32-level accuracy whatever these flags say; they matter only for the eager-torch comparator below)
    torch.backends.cudnn.allow_tf32 = False
    torch.backends.cuda.matmul.allow_tf32 = False
    _bind_to_gpu_numa_node(local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    dt = torch.float32 if args.dtype == "f32" else torch.bfloat16
    B, h, w, Hm, Wm = wl["B"], wl["h"], wl["w"], wl["Hm"], wl["Wm"]
    N = B * h * w
    esz = 4 if dt == torch.float32 else 2

    torch.manual_seed(synth.SEED)
    mem = Memory_sup(K, C, C, 0.8, 1.0, False).to(dev)
    mem.train()
    # sharded runs: the write branch (with its two small all-reduces) goes on a side stream, i.e. a parallel branch
    # of the captured graph, so the exchange latency hides under the read path (2 GPUs: 0.892 -> 0.852 ms/step)
    mem.overlap_write = bool(args.overlap_write) or world > 1
    if world > 1:
        for p in mem.parameters():
            dist.broadcast(p.data, 0)
        sharding.broadcast_memory(mem)
        sharding.enable_sharded_update(mem)
    seed = synth.SEED + 100 * rank
    x_host = synth.make_features(B, C, h, w, seed=seed, dtype=dt).pin_memory()
    lab_host = synth.make_labels(B, Hm, Wm, K, args.labels, seed=seed + 2).pin_memory()
    x = x_host.to(dev).requires_grad_(True)
    labels = lab_host.to(dev)
    G = synth.make_upstream_grad((B, C, h, w), seed=seed + 3, dtype=dt, device=dev)
    f_core = synth.make_features(B, C, h, w, seed=seed + 5, dtype=dt, device=dev).abs_().requires_grad_(True)
    Gu = synth.make_upstream_grad((B, 2 * C, h, w), seed=seed + 6, dtype=dt, device=dev)
    M0 = mem.m_items.clone()
    gw = [torch.tensor(LOSS_W[k], device=dev) for k in ("read", "div", "cls")]
    autocast = torch.autocast("cuda", dtype=torch.bfloat16, enabled=(dt == torch.bfloat16))
    # --dump-outputs: module_step records its outputs on the call that counts "calls_left" down to 0
    last_step = {"calls_left": 0}

    def module_step(xin, lab):
        mem.m_items = M0
        xin.grad = None
        mem.zero_grad(set_to_none=True)
        with autocast:
            uq, sq, sm, rl, wlss = mem(xin, lab, True, False)
        torch.autograd.backward([uq, rl, wlss[0], wlss[1]], [G.to(uq.dtype), gw[0], gw[1], gw[2]])
        if last_step["calls_left"]:
            last_step["calls_left"] -= 1
            if last_step["calls_left"] == 0:
                last_step["outputs"] = step_outputs(uq, sq, sm, rl, wlss, mem.m_items, xin.grad,
                                                    [(n, p.grad) for n, p in mem.named_parameters()])
        return rl, wlss

    Wc, bc = mem.clsfier.weight, mem.clsfier.bias

    core_side = [None]

    def core_step(xi=None, fi=None, Wi=None, bi=None):
        xi = x if xi is None else xi
        fi = f_core if fi is None else fi
        Wi = Wc if Wi is None else Wi
        bi = bc if bi is None else bi
        xi.grad = None
        fi.grad = None
        u, _, _, rl, _ = _ReadFn.apply(xi, M0, labels, None, None, 1.0, K)
        if core_side[0] is not None:      # write branch as a parallel branch (its backward follows it onto that stream)
            cur = torch.cuda.current_stream(dev)
            core_side[0].wait_stream(cur)
            with torch.cuda.stream(core_side[0]):
                M_new, div, cls, _ = _WriteFn.apply(fi, labels, M0, Wi, bi, 0.8, K, mem.shard_group)
            cur.wait_stream(core_side[0])
        else:
            M_new, div, cls, _ = _WriteFn.apply(fi, labels, M0, Wi, bi, 0.8, K, mem.shard_group)
        torch.autograd.backward([u, rl, div, cls], [Gu, gw[0], gw[1], gw[2]])

    res_host = torch.empty(3 + K * C, dtype=torch.float32).pin_memory()

    def e2e_step():
        xin = x_host.to(dev, non_blocking=True).requires_grad_(True)
        lab = lab_host.to(dev, non_blocking=True)
        rl, wlss = module_step(xin, lab)
        res = torch.cat([rl.detach().reshape(1), wlss[0].detach().reshape(1), wlss[1].detach().reshape(1),
                         mem.m_items.detach().reshape(-1)])
        res_host.copy_(res, non_blocking=True)

    # the same, as a training loop would run it: the next batch is uploaded on a copy stream (double-buffered
    # device staging) while the current one is processed; every step still moves its own inputs and results
    copy_stream = torch.cuda.Stream(device=dev)
    stage_x = [torch.empty_like(x) for _ in range(2)]
    stage_l = [torch.empty_like(labels) for _ in range(2)]
    lab_src = [lab_host]
    ready = [torch.cuda.Event() for _ in range(2)]
    consumed = [torch.cuda.Event() for _ in range(2)]
    slot = [0]

    def upload(i):
        with torch.cuda.stream(copy_stream):
            copy_stream.wait_event(consumed[i])
            stage_x[i].copy_(x_host, non_blocking=True)
            stage_l[i].copy_(lab_src[0], non_blocking=True)
            ready[i].record(copy_stream)

    def e2e_pipelined_step():
        i = slot[0]
        upload(i ^ 1)  # prefetch the next batch
        torch.cuda.current_stream().wait_event(ready[i])
        xin = stage_x[i].detach().requires_grad_(True)
        rl, wlss = module_step(xin, stage_l[i])
        res = torch.cat([rl.detach().reshape(1), wlss[0].detach().reshape(1), wlss[1].detach().reshape(1),
                         mem.m_items.detach().reshape(-1)])
        res_host.copy_(res, non_blocking=True)
        consumed[i].record()
        slot[0] = i ^ 1

    timing_info = {}

    def timed(fn, steps, warmup, sample_clocks=False, kernel_timing=False, min_total_ms=0.0, tag=None):
        """W warm-up steps, then blocks of EXACTLY `steps` steps, each bracketed by barrier + synchronize and timed
        with CUDA events on the launching stream (max over ranks per block); blocks repeat until `min_total_ms` of timed
        work has accumulated and the MEDIAN block is returned. The measurements that --steps sizes run one block, so that
        --steps is the number of timed steps."""
        for _ in range(warmup):
            fn()
        torch.cuda.synchronize()
        capi.enable_kernel_timing(kernel_timing)
        capi.reset_counters()
        sampler = ClockSampler(local_rank) if sample_clocks else None
        if sampler:
            sampler.__enter__()
        blocks, total, launches = [], 0.0, 0
        while True:
            if world > 1:
                dist.barrier()
            torch.cuda.synchronize()
            n0 = capi.LAUNCHES
            ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            ev0.record()
            for _ in range(steps):
                fn()
            ev1.record()
            torch.cuda.synchronize()
            ms = ev0.elapsed_time(ev1)
            launches = capi.LAUNCHES - n0
            if world > 1:
                t = torch.tensor([ms], device=dev, dtype=torch.float64)
                dist.all_reduce(t, op=dist.ReduceOp.MAX)   # also keeps the ranks' block counts in step
                ms = float(t.item())
            blocks.append(ms)
            total += ms
            if total >= min_total_ms or len(blocks) >= 200 or kernel_timing:
                break
        if sampler:
            sampler.__exit__()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        ktimes = capi.kernel_timings_ms() if kernel_timing else {}
        capi.enable_kernel_timing(False)
        ms = statistics.median(blocks)
        if tag:
            timing_info[tag] = {"blocks": len(blocks), "steps_per_block": steps, "block_ms_min": round(min(blocks), 4),
                                "block_ms_median": round(ms, 4), "block_ms_max": round(max(blocks), 4)}
        return ms, launches, ktimes, (sampler.summary() if sampler else None)

    # whole module, device-resident inputs, one Python-side launch per kernel
    last_step["calls_left"] = args.warmup + args.steps if args.dump_outputs else 0
    ms, launches, _, clocks = timed(lambda: module_step(x, labels), args.steps, args.warmup, sample_clocks=True,
                                    tag="eager_launch")
    ms_per_step = ms / args.steps
    value = world * N / (ms_per_step * 1e-3) / 1e6
    eager_launch = {"value": value, "unit": UNIT, "ms_per_step": ms_per_step, "gpu_launches": launches,
                    "what": "the same step launched kernel by kernel from Python (no CUDA graph)"}

    # headline: the same step captured once into a CUDA graph (pinthememory_b200.graphed.GraphedStep: forward,
    # the weighted losses, backward, memory carried from step to step) and replayed -- identical kernels and
    # work, without the host launch gaps
    graph_info = gstep = None
    if not args.no_graph:
        try:
            from pinthememory_b200.graphed import GraphedStep

            mem.m_items = M0.clone()
            # captured, the write branch is a parallel branch of the graph (a side stream); launched kernel by kernel
            # the extra stream only costs host time, so the eager measurements keep a single stream at N = 1
            overlap_eager = mem.overlap_write
            mem.overlap_write = True
            gstep = GraphedStep(mem, x, labels, G, loss_weights=(LOSS_W["read"], LOSS_W["div"], LOSS_W["cls"]),
                                memory_writing=True, writing_detach=False, carry_memory=True,
                                autocast_dtype=torch.bfloat16 if dt == torch.bfloat16 else None)
            mem.overlap_write = overlap_eager
            ms_g, _, _, clocks_g = timed(gstep.replay, args.steps, args.warmup, sample_clocks=True, tag="value")
            if args.dump_outputs:
                o = gstep.outputs
                names = [n for n, p in mem.named_parameters() if p.requires_grad]   # GraphedStep's order of param_grads
                last_step["outputs"] = step_outputs(o["updated_query"], o["score_query"], o["score_memory"], o["readloss"],
                                                    o["writeloss"], o["memory"], gstep.query_grad,
                                                    zip(names, gstep.param_grads))
            graph_info = {"kernels_per_replay": gstep.kernels_per_replay}
            ms_per_step = ms_g / args.steps
            value = world * N / (ms_per_step * 1e-3) / 1e6
            launches = gstep.kernels_per_replay * args.steps
            clocks = clocks_g
        except Exception as e:  # report the eagerly launched number rather than nothing
            graph_info = {"error": str(e)[:300]}
            mem.overlap_write = bool(args.overlap_write) or world > 1
    if args.dump_outputs and rank == 0:
        write_dump(args.dump_outputs, dump_arrays(last_step["outputs"]))
    last_step.pop("outputs", None)

    # per-kernel durations measured live (events around every C-ABI launch) in a second timed region
    # (each step starts behind a ~3 ms device-side sleep so that the host has queued the whole step before the first kernel
    # runs: the event pair around a launch then brackets the kernel alone, not the Python time between the two records)
    def timed_kernels_step():
        torch.cuda._sleep(6_000_000)
        module_step(x, labels)

    ms_k, _, ktimes, _ = timed(timed_kernels_step, args.steps, 2, kernel_timing=True)
    kavg = {k: sum(v) / len(v) for k, v in ktimes.items()}  # ms per call
    r = Hm * Wm / float(h * w)
    KP = 20
    alg_bytes = {  # ALGORITHMIC bytes per launch (DESIGN.md section 4)
        "pm_read_fwd": N * (3 * C * esz + 4 * KP + 4 * K),
        "pm_read_bwd": N * (4 * C * esz + 4 * KP + 4 * K),
        # score-plane read (the module's default: the memory folded into the output convolution)
        "pm_read_fwd_planes": N * ((2 * C + 32) * esz + 4 * KP + 4 * K),
        "pm_read_bwd_planes": N * ((3 * C + K) * esz + 2 * 4 * KP + 4 * K),
        "pm_readloss_fwd": N * (8 * r + 2 * 4 * KP),
        # second-generation read loss: the label pass (int64 in, uint8 out, histogram) + the loss on the packed map; the
        # pair is what SURVEY 8d budgets as ONE read of the int64 labels (8r) + the score / gradient rows
        "pm_labels_pack": N * r * 9,
        "pm_readloss_fwd8": N * (r + 2 * 4 * KP),
        "pm_readloss (pm_labels_pack + pm_readloss_fwd8)": N * (8 * r + 2 * 4 * KP),
        "pm_write_reduce_fwd": N * (C * esz),
        "pm_write_bwd": N * (2 * C * esz),
        "pm_write_reduce_fwd8": N * (C * esz),
        "pm_write_bwd8": N * (2 * C * esz),
        "pm_colsoftmax_apply": N * (4 * KP + 4 * K),
        # the fused BatchNorm passes run once per conv block (2 per step); bytes are the mean of the two calls
        "pm_bn_stats": N * C * esz,
        "pm_bn_apply": N * C * esz * 2.5,        # x (+ residual in one of the two blocks) -> y
        "pm_bn_apply_stats": N * C * esz * 2.5,  # the same pass with the statistics finalised in-kernel
        "pm_bn_bwd_reduce": N * C * esz * 2,     # dy, x (+ the packed ReLU mask, 1/32)
        "pm_bn_bwd_reduce_rows": N * C * esz * 2,
        "pm_bn_bwd_apply": N * C * esz * 3.5,    # dy, x -> dx (+ dres in one of the two blocks)
    }
    if "pm_labels_pack" in kavg and "pm_readloss_fwd8" in kavg:
        kavg["pm_readloss (pm_labels_pack + pm_readloss_fwd8)"] = kavg["pm_labels_pack"] + kavg["pm_readloss_fwd8"]
    bound_note = {
        "pm_readloss (pm_labels_pack + pm_readloss_fwd8)":
            "two launches reported as one logical kernel (time and bytes are their sums; bytes as SURVEY 8d counts them: "
            "int64 labels read once). Not HBM-bound by nature: ~2 x 55 instructions per LABEL pixel (64 label pixels per "
            "feature pixel; a lane pair per bilinear cell, half of the 20 slots each) plus the per-row exp2 set-up, 16 "
            "warps per SM -- instruction-issue bound (ncu: issue slots 61 % busy), see DESIGN.md 6; DRAM traffic = "
            "algorithmic bytes (no re-reads)",
        "pm_readloss_fwd": "not HBM-bound by nature: ~19 ex2 + ~60 FMA per LABEL pixel (64 label pixels per feature "
                           "pixel) make it FP32/MUFU-issue bound; the HBM fraction is reported because the contract asks "
                           "for it, see DESIGN.md 4/6",
        "pm_read_bwd": "one C-ABI call = two kernels (score gradients, then dx); bytes and time are their sums",
        "pm_read_bwd_planes": "one C-ABI call = two kernels (score gradients, then dx); bytes and time are their sums",
    }
    peak, peak_src = measured_peaks()
    # the two 1x1 convolutions: tensor-bound. ALGORITHMIC FLOPs per step (2*M*N*K of the fp32 product, one pass): forward
    # of both blocks + input gradient of both blocks for pm_conv1x1_fwd (the same kernel; the 288-row input gradient of
    # the folded output convolution is two launches), both weight gradients for pm_conv1x1_wgrad. fp32 I/O EXECUTES
    # three TF32 passes per product (3xTF32 error compensation) -- reported separately as executed_*.
    passes = 3 if dt == torch.float32 else 1
    calls = {k: len(v) / float(args.steps) for k, v in ktimes.items()}          # launches per step
    kstep = {k: sum(v) / float(args.steps) for k, v in ktimes.items()}          # ms per step
    conv_flops_step = {"pm_conv1x1_fwd": 2.0 * N * C * (4 * C + 64), "pm_conv1x1_wgrad": 2.0 * N * C * (2 * C + 32)}
    if "pm_conv1x1_dgrad_bnbwd" in kstep:
        # the input gradient of the output block (C+32 rows) runs inside pm_conv1x1_dgrad_bnbwd (BatchNorm backward in the
        # GEMM's operand path): its flops leave the pm_conv1x1_fwd budget
        conv_flops_step["pm_conv1x1_dgrad_bnbwd"] = 2.0 * N * C * (C + 32)
        conv_flops_step["pm_conv1x1_fwd"] -= conv_flops_step["pm_conv1x1_dgrad_bnbwd"]
    tpeak, tpeak_src = tensor_peak(dt)
    kernels = {}
    for k, t_ms in kavg.items():
        ent = {"ms": round(t_ms, 5)}
        if k in calls:
            ent["launches_per_step"] = round(calls[k], 2)
            ent["ms_per_step"] = round(kstep[k], 5)
        if k in conv_flops_step and k in kstep:
            alg = conv_flops_step[k] / (kstep[k] * 1e-3) / 1e12
            ent["bound"] = "tensor"
            ent["TFLOPs"] = round(alg, 1)
            ent["executed_TFLOPs"] = round(alg * passes, 1)
            ent["tensor_peak_TFLOPs"] = tpeak
            ent["frac"] = round(alg / tpeak, 4)
            ent["executed_frac"] = round(alg * passes / tpeak, 4)
            ent["note"] = ("%d-pass %s tcgen05 GEMM; TFLOPs = algorithmic 2MNK per launch / launch time, executed_* = "
                           "x%d passes; peak = %s" % (passes, "TF32" if passes == 3 else "bf16", passes, tpeak_src))
        if k in alg_bytes:
            ent["alg_MB"] = round(alg_bytes[k] / 1e6, 3)
            ent["GBps"] = round(alg_bytes[k] / (t_ms * 1e-3) / 1e9, 1)
            ent["frac"] = round(ent["GBps"] / peak, 4)
        kernels[k] = ent
    comb = "pm_readloss (pm_labels_pack + pm_readloss_fwd8)"
    if comb in kavg:
        kstep[comb] = kstep["pm_labels_pack"] + kstep["pm_readloss_fwd8"]
    # the DOMINANT kernel = the one with the largest share of the step (launches x duration), among those with a budget
    cand = [k for k in kstep if (k in alg_bytes or k in conv_flops_step) and k not in ("pm_labels_pack", "pm_readloss_fwd8")]
    dom = max(cand, key=lambda k: kstep[k])
    dom_hbm = max((k for k in cand if k in alg_bytes), key=lambda k: kstep[k])
    tr = {}
    try:
        with open(os.path.join(ROOT, "profiles", "ncu_traffic.json")) as fh:
            tr = json.load(fh).get(args.dtype, {})
    except Exception:
        pass

    def traffic_of(k):
        if k.startswith("pm_readloss ("):
            return (tr.get("pm_labels_pack", 0.0) + tr.get("pm_readloss_fwd8", 0.0)) or None
        for cand_k in (k, k.replace("_planes", ""), k.rstrip("8"), k.replace("_apply_stats", "_apply")):
            if cand_k in tr:
                return tr[cand_k]
        return None

    def hbm_entry(k):
        ent = {"bound": "hbm", "kernel": k, "achieved": kernels[k]["GBps"], "peak": peak, "unit": "GB/s",
               "frac": kernels[k]["frac"], "traffic": traffic_of(k), "peak_source": peak_src,
               "alg_bytes_per_launch": alg_bytes[k], "launch_ms": kernels[k]["ms"],
               "share_of_step": round(kstep[k] / sum(v for q, v in kstep.items() if q != comb), 4)}
        if k in bound_note:
            ent["note"] = bound_note[k]
        return ent

    if dom in conv_flops_step:
        e = kernels[dom]
        roofline = {"bound": "tensor", "kernel": dom, "achieved": e["TFLOPs"], "peak": tpeak, "unit": "TFLOP/s",
                    "frac": e["frac"], "traffic": traffic_of(dom), "peak_source": tpeak_src,
                    "alg_flops_per_launch": conv_flops_step[dom] / calls[dom], "launch_ms": e["ms"],
                    "launches_per_step": e["launches_per_step"],
                    "share_of_step": round(kstep[dom] / sum(v for q, v in kstep.items() if q != comb), 4),
                    "executed_TFLOPs": e["executed_TFLOPs"], "executed_frac": e["executed_frac"],
                    "note": "dominant by share of the step (launches x duration). achieved = ALGORITHMIC flops (2MNK of "
                            "the fp32 product, averaged over the step's launches of this kernel) / mean launch time. "
                            + ("fp32 I/O computes every product as three TF32 tensor-core passes (hi*hi + hi*lo + lo*hi) "
                               "to hold the 1e-5 parity bar, so the algorithmic fraction is bounded by 1/3 of the TF32 "
                               "peak; executed_* counts the three passes (tensor-pipe view). " if passes == 3 else "")
                            + "The streaming kernels' HBM rooflines are in `hbm_dominant`, `core` and `kernels`.",
                    "hbm_dominant": hbm_entry(dom_hbm)}
    else:
        roofline = hbm_entry(dom)

    # core: hand-written kernels only, one Python-side launch per kernel (host-launch bound at ~0.4 ms: capturing this
    # autograd fragment separately was tried and disturbs the measurements that follow; the headline step IS captured)
    core_graph = None
    core_launch = "one Python-side launch per kernel"
    core_fn = core_step
    if not args.no_graph:
        try:  # the same 9 launches captured once and replayed (removes the host launch gaps, as for the headline)
            side = torch.cuda.Stream(device=dev)
            side.wait_stream(torch.cuda.current_stream(dev))
            with torch.cuda.stream(side):
                # fresh leaves: the AccumulateGrad nodes of x / f_core were created on the main stream by earlier steps and
                # would pull that stream into the capture
                xg = x.detach().clone().requires_grad_(True)
                fg = f_core.detach().clone().requires_grad_(True)
                Wg = Wc.detach().clone().requires_grad_(True)
                bg = bc.detach().clone().requires_grad_(True)
                for _ in range(3):
                    core_step(xg, fg, Wg, bg)
            torch.cuda.current_stream(dev).wait_stream(side)
            torch.cuda.synchronize()
            xg.grad = fg.grad = Wg.grad = bg.grad = None
            core_graph = torch.cuda.CUDAGraph()
            n0 = capi.LAUNCHES
            core_side[0] = None if args.core_serial else torch.cuda.Stream(device=dev)
            with torch.cuda.graph(core_graph):
                core_step(xg, fg, Wg, bg)
            core_side[0] = None
            core_launches_per_replay = capi.LAUNCHES - n0
            core_fn = core_graph.replay
            core_launch = "CUDA graph replay of the %d launches%s" % (
                core_launches_per_replay, "" if args.core_serial else
                "; the write branch (class sums, update and their backward) is a parallel branch of the graph, as in the "
                "captured module step")
        except Exception as e:
            core_graph, core_fn = None, core_step
            core_launch = "one Python-side launch per kernel (capture failed: %s)" % str(e)[:120]
    ms_c, launches_c, _, _ = timed(core_fn, args.steps, args.warmup, tag="core")
    ms_core = ms_c / args.steps
    a_train = 10 * C * esz + 8 * r + 8 * K
    core_gbps = N * a_train / (ms_core * 1e-3) / 1e9
    core = {"value": world * N / (ms_core * 1e-3) / 1e6, "unit": UNIT, "ms_per_step": ms_core,
            "a_train_bytes_per_pixel": a_train, "GBps": core_gbps, "frac_of_peak": core_gbps / peak,
            "gpu_launches_per_step": (core_launches_per_replay if core_graph is not None else launches_c / args.steps),
            "launch": core_launch,
            "what": "read_fwd+colsoftmax+readloss+write_reduce+update fwd, update+write+read bwd; f and du given"}

    # e2e: host (pinned) inputs through the public module API
    n_e = max(args.steps // 2, 5)
    ms_e, _, _, _ = timed(e2e_step, n_e, 3)
    ms_e2e_serial = ms_e / n_e
    for i in range(2):
        consumed[i].record()
    upload(0)
    ms_e, _, _, _ = timed(e2e_pipelined_step, n_e, 3, tag="e2e")
    ms_e2e = ms_e / n_e
    # the same with the labels handed over as uint8 class ids (the module accepts both; 1/8 of the label bytes on the bus)
    e2e_u8 = None
    try:
        lab_host8 = lab_host.to(torch.uint8).pin_memory()
        lab_src[0] = lab_host8
        for i in range(2):
            stage_l[i] = torch.empty(labels.shape, dtype=torch.uint8, device=dev)
        torch.cuda.synchronize()
        for i in range(2):
            consumed[i].record()
        slot[0] = 0
        upload(0)
        ms_u8, _, _, _ = timed(e2e_pipelined_step, n_e, 3)
        ms_u8 /= n_e
        e2e_u8 = {"value": world * N / (ms_u8 * 1e-3) / 1e6, "ms_per_step": ms_u8,
                  "h2d_bytes_per_step": x_host.numel() * x_host.element_size() + lab_host8.numel(),
                  "what": "labels uploaded as uint8 class ids (255 = ignore) instead of int64"}
    except Exception as e:
        e2e_u8 = {"error": str(e)[:200]}
    e2e = {"value": world * N / (ms_e2e * 1e-3) / 1e6, "unit": UNIT, "ms_per_step": ms_e2e, "uint8_labels": e2e_u8,
           "h2d_bytes_per_step": x_host.numel() * x_host.element_size() + lab_host.numel() * 8,
           "d2h_bytes_per_step": res_host.numel() * 4,
           "serial": {"value": world * N / (ms_e2e_serial * 1e-3) / 1e6, "ms_per_step": ms_e2e_serial,
                      "what": "copy-in, compute, copy-out back to back on one stream"},
           "what": "Memory_sup.forward+backward per step with that step's pinned-host features and int64 labels copied "
                   "in and losses + new memory copied out; the upload of the next batch runs on a copy stream under "
                   "the current step's compute (PCIe-bound: %.0f MB per step)" %
                   ((x_host.numel() * x_host.element_size() + lab_host.numel() * 8) / 1e6)}

    line = dict(base)
    line.update({"value": value, "ms_per_step": ms_per_step, "gpu_launches": launches, "clocks": clocks,
                 "e2e": e2e, "roofline": roofline, "core": core, "kernels": kernels, "eager_launch": eager_launch,
                 "cuda_graph": graph_info, "timing": timing_info,
                 "gpu_launches_what": "kernels of this package (C-ABI launches) inside the timed region = per-replay count "
                                      "x steps; since round 2 there are no library GEMM kernels on the step (the 1x1 "
                                      "convolutions are pm_conv1x1_*); the few remaining torch element-wise kernels "
                                      "(gradient accumulation, fills, the memory copy) are not counted",
                 "tf32": "disabled for torch/cuDNN (allow_tf32=False), as in the parity tests"})
    line["config"]["launch"] = ("CUDA graph replay of the whole step (GraphedStep)" if graph_info and "error" not in graph_info
                                else "one Python-side launch per kernel")
    if graph_info and "error" not in graph_info:
        line["config"]["launch"] += "; write branch (incl. the all-reduces when sharded) as a parallel graph branch"

    # ---- sharded == global batch, checked on this very job (the 2-GPU pytest cannot run on a 1-GPU test box) ----------
    if world > 1:
        try:
            from oracle import memory_oracle as mo

            with torch.no_grad():
                f_loc = f_core.detach().float()
                Mn, _, _, SDn = _WriteFn.apply(f_core.detach(), labels, M0, Wc, bc, 0.8, K, mem.shard_group)
                gat = [torch.empty_like(Mn) for _ in range(world)]
                dist.all_gather(gat, Mn.contiguous())
                identical = all(torch.equal(g, gat[0]) for g in gat)
                f_all = [torch.empty_like(f_loc) for _ in range(world)]
                l_all = [torch.empty_like(labels) for _ in range(world)]
                dist.all_gather(f_all, f_loc.contiguous())
                dist.all_gather(l_all, labels)
                rel = None
                if rank == 0:   # the oracle's update of the CONCATENATED batch, one image at a time (sums are additive)
                    S = torch.zeros(K + 1, C, device=dev, dtype=torch.float64)
                    D = torch.zeros(K + 1, device=dev, dtype=torch.float64)
                    for fr, lr in zip(f_all, l_all):
                        for i in range(fr.shape[0]):
                            s_i, d_i = mo.class_sums(fr[i:i + 1].double(), lr[i:i + 1], K)
                            S += s_i
                            D += d_i
                    M_ref = mo.momentum_update(M0.double(), S, D, 0.8)
                    rel = float((Mn.double() - M_ref).norm() / M_ref.norm())
            line["sharded_parity"] = {"memory_bit_identical_across_ranks": bool(identical),
                                      "memory_vs_oracle_global_batch_rel_l2": rel, "images": world * B,
                                      "exchange": exchange_name(mem),
                                      "what": "pm_write_reduce_fwd on each rank's shard + exchange of the [K+1,C+4] "
                                              "sums|counts + update, against the fp64 oracle update of the "
                                              "concatenated %d-image batch (write features given)" % (world * B)}
            line["exchange"] = exchange_name(mem)
        except Exception as e:
            line["sharded_parity"] = {"error": str(e)[:300]}

    # ---- the other BASELINE configs on the same kernels (short runs; parity for these shapes is in tests/) -----------
    if not args.no_extra:
        line["configs"] = extra_configs(args, dev, dt, world, rank, mem, timed)

    if rank == 0 and world == 1 and not args.no_callers:
        # the callers either side of the path that run on the same kernels (SURVEY.md 8f rows 2 and 5)
        try:
            import torch.nn.functional as F

            from pinthememory_b200.callers import PrototypePool, upsampled_cross_entropy

            lg = (torch.randn(B, K, Hm // 4, Wm // 4, device=dev) * 3).requires_grad_(True)

            def fused_loss():
                lg.grad = None
                upsampled_cross_entropy(lg, labels).backward()

            def eager_loss():
                lg.grad = None
                up = F.interpolate(lg, size=(Hm, Wm), mode="bilinear", align_corners=True)
                F.cross_entropy(up, labels, ignore_index=255).backward()

            ms_f, _, _, _ = timed(fused_loss, 10, 3)
            ms_t, _, _, _ = timed(eager_loss, 10, 3)
            pool = PrototypePool(K, C, dev)
            ms_p, _, _, _ = timed(lambda: pool.add(x, labels), 10, 3)
            line["callers"] = {
                "main_loss_fwd_bwd": {"fused_ms": ms_f / 10, "torch_eager_ms": ms_t / 10,
                                      "what": "CE(bilinear_up(logits [%d,%d,%d,%d] -> %dx%d), labels) forward+backward; "
                                              "pm_readloss_fwd vs F.interpolate+F.cross_entropy on this GPU"
                                              % (B, K, Hm // 4, Wm // 4, Hm, Wm)},
                "prototype_pool_add": {"ms": ms_p / 10, "Mpixels_per_s": N / (ms_p / 10 * 1e-3) / 1e6,
                                       "what": "memory_initalize pooling of one batch (pm_write_reduce_fwd accumulating)"}}
        except Exception as e:
            line["callers"] = {"error": str(e)[:300]}

    if rank == 0 and world == 1:
        # like-for-like GPU comparison: the oracle restatement (eager torch ops) on the same B200
        try:
            from oracle import memory_oracle as mo

            ora = mo.OracleMemorySup(K, C, C, 0.8, 1.0, False).to(dev)
            ora.load_state_dict(mem.state_dict())
            ora.train()

            def eager_step():
                ora.m_items = M0
                x.grad = None
                ora.zero_grad(set_to_none=True)
                with autocast:
                    uq, _, _, rl, wlss = ora(x, labels, True, False)
                torch.autograd.backward([uq, rl, wlss[0], wlss[1]], [G.to(uq.dtype), gw[0], gw[1], gw[2]])

            ms_o, _, _, _ = timed(eager_step, 10, 3)
            line["torch_eager_same_gpu"] = {"value": N / (ms_o / 10 * 1e-3) / 1e6, "unit": UNIT, "ms_per_step": ms_o / 10,
                                            "what": "oracle restatement of the reference module, eager PyTorch ops, fp32"
                                            if dt == torch.float32 else "oracle restatement under bf16 autocast (speed only)"}
        except Exception as e:  # the comparison is informative only
            line["torch_eager_same_gpu"] = {"error": str(e)[:200]}
        if dt == torch.float32:
            try:   # the reference's OWN module (unmodified, oracle/_ref), eagerly on this GPU
                refm = reference_module(dev)
                if refm is not None:
                    refm.load_state_dict(mem.state_dict())
                    refm.train()

                    def ref_step():
                        refm.m_items = M0
                        x.grad = None
                        refm.zero_grad(set_to_none=True)
                        uq, _, _, rl, wlss = refm(x, labels, True, False)
                        torch.autograd.backward([uq, rl, wlss[0], wlss[1]], [G.to(uq.dtype), gw[0], gw[1], gw[2]])

                    ms_r, _, _, _ = timed(ref_step, 10, 3)
                    line["reference_eager_same_gpu"] = {
                        "value": N / (ms_r / 10 * 1e-3) / 1e6, "unit": UNIT, "ms_per_step": ms_r / 10,
                        "what": "the reference's unmodified network/memory.py::Memory_sup (oracle/_ref), eager PyTorch on this "
                                "GPU, fp32 with TF32 off (the parity configuration)"}
                    del refm
            except Exception as e:
                line["reference_eager_same_gpu"] = {"error": str(e)[:200]}
        if not args.no_cpu_baseline:
            cb = cpu_reference_run(wl, args.labels, 6, 1, None, budget_s=25.0)
            line["cpu_baseline"] = {"value": cb["value"], "unit": UNIT, "cores": cb["cores"], "kind": cb["kind"],
                                    "sample": cb["sample"], "ms_per_step": cb["ms_per_step"], "same_config": cb["same_config"]}
    if rank == 0:
        print(json.dumps(line), flush=True)
    if world > 1:
        # a live graph that captured the all-reduce keeps the NCCL communicator busy: release it first, and
        # never let a stuck teardown hold the job (the result line is already out)
        import threading

        threading.Timer(30.0, lambda: os._exit(0)).start()
        if gstep is not None:
            gstep.release()
        if core_graph is not None:
            torch.cuda.synchronize()
            core_graph.reset()
        torch.cuda.synchronize()
        dist.barrier()
        dist.destroy_process_group()
        os._exit(0)


if __name__ == "__main__":
    main()
