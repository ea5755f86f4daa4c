"""SyncBatchNorm over the sharded update's peer memory against the NCCL all-reduces, in the BASELINE cfg-4 step.

    python profiles/syncbn_exchange_time.py [--worlds 2 8] [--steps 50] [--rounds 5] [--out profiles/syncbn_exchange_time_b200.json]

Workload: the module's training step (read + write, forward + backward) at the DR50V3P cfg-4 shape -- 48x48 features,
768x768 blocky int64 labels, C=256, K=19, global batch 64 split over W GPUs (64/W images each) -- with SyncBatchNorm
(convert_sync_batchnorm, as under --syncbn), the sharded update and two-stream mode, captured once as a CUDA graph
(GraphedStep) per mode and replayed. Modes: `peer` (both SyncBatchNorm layers exchange over the shard group's symmetric
buffer) and `nccl` (the layers reduce over another process group of the same ranks: their four small NCCL all-reduces per
step); the class sums go over peer memory in both. The two graphs
are timed alternately in one job, --rounds times each, every round --steps replays between CUDA events on rank 0 (the
graphs hold collectives, so the ranks move in lock-step); the median round is reported. The card's name and power limit
are read in the same run. Needs at least max(--worlds) GPUs; a world that does not fit is an error, not skipped.
"""
import argparse
import json
import os
import socket
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

K, C, GLOBAL_B = 19, 256, 64
MODES = ("peer", "nccl")


def gpu_info():
    info = {"name": torch.cuda.get_device_name(0), "power_limit_w": None}
    try:
        r = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader,nounits", "-i", "0"],
                           capture_output=True, text=True, timeout=30)
        info["power_limit_w"] = float(r.stdout.strip().splitlines()[0])
    except Exception as e:  # noqa: BLE001
        info["power_limit_error"] = repr(e)[:200]
    return info


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def _worker(rank, world, port, steps, rounds, out):
    import torch.distributed as dist

    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    torch.cuda.set_device(rank)
    dev = torch.device("cuda", rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=dev)
    try:
        torch.backends.cudnn.allow_tf32 = False
        torch.backends.cuda.matmul.allow_tf32 = False
        from pinthememory_b200 import sharding, synth
        from pinthememory_b200.graphed import GraphedStep
        from pinthememory_b200.memory import Memory_sup

        wl = synth.WORKLOADS["cfg4_dp_os16_b8"]
        Bl = GLOBAL_B // world
        seed = synth.SEED + 100 * rank + 7
        x = synth.make_features(Bl, C, wl["h"], wl["w"], seed=seed, device=dev)
        lab = synth.make_labels(Bl, wl["Hm"], wl["Wm"], K, "blocky", seed=seed + 2, device=dev)
        G = synth.make_upstream_grad((Bl, C, wl["h"], wl["w"]), seed=seed + 3, device=dev)
        steps_by_mode = {}
        for mode in MODES:
            torch.manual_seed(synth.SEED)
            m = Memory_sup(K, C, C, 0.8, 1.0, False).to(dev)
            # nccl: the layers reduce over a group of the same ranks that is not the shard group, so only they leave the
            # peer path
            bn_group = dist.new_group(list(range(world))) if mode == "nccl" else None
            m = torch.nn.SyncBatchNorm.convert_sync_batchnorm(m, process_group=bn_group).train()
            shard = sharding.enable_sharded_update(m)
            if shard.peer is None:
                raise RuntimeError("no symmetric-memory peer exchange on this box: %s" % shard.peer_error)
            m.overlap_write = True
            steps_by_mode[mode] = GraphedStep(m, x, lab, G, loss_weights=(0.02, 0.4, 0.2), memory_writing=True,
                                              writing_detach=False)
        times = {mode: [] for mode in MODES}
        for _ in range(rounds):
            for mode in MODES:
                gs = steps_by_mode[mode]
                for _ in range(3):
                    gs.replay()
                torch.cuda.synchronize()
                a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                a.record()
                for _ in range(steps):
                    gs.replay()
                b.record()
                b.synchronize()
                times[mode].append(1000.0 * a.elapsed_time(b) / steps)
        for gs in steps_by_mode.values():
            gs.release()
        if rank == 0:
            med = {mode: sorted(v)[len(v) // 2] for mode, v in times.items()}
            out[world] = {"per_gpu_batch": Bl, "us_per_step_median": {k: round(v, 1) for k, v in med.items()},
                          "us_per_step_rounds": {k: [round(t, 1) for t in v] for k, v in times.items()},
                          "peer_saves_us": round(med["nccl"] - med["peer"], 1)}
    finally:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--worlds", type=int, nargs="+", default=[2, 8])
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "syncbn_exchange_time_b200.json"))
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("syncbn_exchange_time.py needs CUDA devices")
    have = torch.cuda.device_count()
    if max(args.worlds) > have:
        raise SystemExit("syncbn_exchange_time.py: --worlds %s needs %d GPUs, this box has %d" % (args.worlds, max(args.worlds), have))
    import torch.multiprocessing as mp

    res = {"gpu": gpu_info(), "workload": "cfg4: 48x48 features, 768x768 blocky labels, C=%d, K=%d, global batch %d, "
                                          "SyncBatchNorm, sharded update, two-stream mode, CUDA graph replay" % (C, K, GLOBAL_B),
           "steps_per_round": args.steps, "rounds": args.rounds, "worlds": {}}
    for world in args.worlds:
        out = mp.get_context("spawn").Manager().dict()
        mp.spawn(_worker, args=(world, _free_port(), args.steps, args.rounds, out), nprocs=world, join=True)
        res["worlds"][str(world)] = out[world]
    line = json.dumps(res)
    print(line)
    if args.out:
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
