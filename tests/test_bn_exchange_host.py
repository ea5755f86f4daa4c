"""CPU: SyncBatchNorm over the sharded update's peer buffers -- the buffer layout of the two new exchanges, header and binding
agreement, the argument checks of pm_bn_exchange_fwd / _bwd, and which layers take the peer path (over gloo)."""
import ctypes
import os
import re
import shutil
import socket
import subprocess
import types

import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _header_defines():
    src = open(os.path.join(ROOT, "include", "pinmem_b200.h")).read()
    return {m.group(1): int(m.group(2)) for m in re.finditer(r"#define (PM_\w+) (\d+)", src)}


def test_header_and_binding_agree():
    from pinthememory_b200 import capi

    d = _header_defines()
    assert d["PM_ABI_VERSION"] == capi.ABI_VERSION == 215
    assert capi.BN_MAX_C == d["PM_BN_MAX_C"] == 256
    assert capi.PEER_BN_FLAG_OFF == d["PM_PEER_BN_FLAG_OFF"]
    assert (capi.PEER_BN_FWD_OFF, capi.BN_FWD_ROW_BYTES) == (d["PM_PEER_BN_FWD_OFF"], d["PM_BN_FWD_ROW_BYTES"])
    assert (capi.PEER_BN_BWD_OFF, capi.BN_BWD_ROW_BYTES) == (d["PM_PEER_BN_BWD_OFF"], d["PM_BN_BWD_ROW_BYTES"])
    assert capi.load().pm_version() == 215


def test_peer_buffer_layout_of_the_syncbn_exchanges():
    """Every region of the 128 KB peer buffer, the four new rows (M = 256) and the new flags (4 exchanges x {arrival, done} x
    16 ranks of u32) included, is disjoint from every other, inside PM_PEER_BYTES and 16-byte aligned."""
    d = _header_defines()
    M, ranks = d["PM_BN_MAX_C"], 16
    assert (d["PM_PEER_DS_OFF"], d["PM_PEER_FLAG_OFF"], d["PM_PEER_BYTES"]) == (36864, 73728, 131072)
    assert d["PM_BN_FWD_ROW_BYTES"] >= (2 * M + 1) * 8 and d["PM_BN_BWD_ROW_BYTES"] >= 2 * M * 4
    regions = {
        "sums": (0, d["PM_PEER_DS_OFF"]),
        "dS": (d["PM_PEER_DS_OFF"], d["PM_PEER_FLAG_OFF"]),
        "flags kinds 0..7": (d["PM_PEER_FLAG_OFF"], d["PM_PEER_FLAG_OFF"] + 8 * 32 * 16 * 4),
        "bn flags": (d["PM_PEER_BN_FLAG_OFF"], d["PM_PEER_BN_FLAG_OFF"] + 4 * 2 * ranks * 4),
        "read fwd": (d["PM_PEER_READ_FWD_OFF"], d["PM_PEER_READ_FWD_OFF"] + d["PM_READ_ROW_FLOATS"] * 4),
        "read bwd": (d["PM_PEER_READ_BWD_OFF"], d["PM_PEER_READ_BWD_OFF"] + d["PM_READ_ROW_FLOATS"] * 4),
    }
    for slot in (0, 1):
        a = d["PM_PEER_BN_FWD_OFF"] + slot * d["PM_BN_FWD_ROW_BYTES"]
        regions["bn fwd slot %d" % slot] = (a, a + (2 * M + 1) * 8)
        b = d["PM_PEER_BN_BWD_OFF"] + slot * d["PM_BN_BWD_ROW_BYTES"]
        regions["bn bwd slot %d" % slot] = (b, b + 2 * M * 4)
    items = sorted(regions.items(), key=lambda kv: kv[1][0])
    for (n0, (a0, e0)), (n1, (a1, _)) in zip(items, items[1:]):
        assert e0 <= a1, "%s overlaps %s" % (n0, n1)
    for name, (a, e) in items:
        assert 0 <= a < e <= d["PM_PEER_BYTES"], name
        assert a % 16 == 0, name
    # the new flags are rows 0..7 of flag kind 8, which the kernels address as peer_flag(base, 8, row, rank)
    assert d["PM_PEER_BN_FLAG_OFF"] == d["PM_PEER_FLAG_OFF"] + (8 * 32 * 16) * 4
    # the new rows live in what was free space after the read rows
    assert regions["bn fwd slot 0"][0] >= regions["read bwd"][1]


def test_exchange_entries_check_arguments_without_a_gpu():
    from pinthememory_b200 import capi

    lib = capi.load()
    p = ctypes.c_void_p(256)
    c = ctypes.c_double(8.0)
    fwd, bwd = lib.pm_bn_exchange_fwd, lib.pm_bn_exchange_bwd
    assert fwd(None, 0, 2, p, 0, p, c, 64, None) == -1                 # no peer buffers
    assert fwd(p, 0, 2, None, 0, p, c, 64, None) == -1                 # no epoch
    assert fwd(p, 0, 2, p, 0, None, c, 64, None) == -1                 # no stats
    assert fwd(p, 0, 2, p, 0, p, c, 0, None) == -5                     # M < 1
    assert fwd(p, 0, 2, p, 0, p, c, 257, None) == -5                   # M > 256
    assert fwd(p, 0, 1, p, 0, p, c, 64, None) == -5                    # one rank
    assert fwd(p, 0, 17, p, 0, p, c, 64, None) == -5                   # more than 16 ranks
    assert fwd(p, 2, 2, p, 0, p, c, 64, None) == -5                    # rank outside the group
    assert fwd(p, 0, 2, p, 2, p, c, 64, None) == -5                    # slot
    assert fwd(p, 0, 2, p, -1, p, c, 64, None) == -5
    assert fwd(p, 0, 2, p, 0, ctypes.c_void_p(260), c, 64, None) == -6  # stats not 8-byte aligned
    assert bwd(p, 0, 2, p, 0, p, p, None, c, p, p, 64, None) == -1     # no count_global
    assert bwd(p, 0, 2, p, 0, None, p, p, c, p, p, 64, None) == -1     # no dgamma
    assert bwd(p, 0, 2, p, 0, p, p, p, c, p, None, 64, None) == -1     # no sb
    assert bwd(p, 0, 2, p, 0, p, p, p, c, p, p, 0, None) == -5
    assert bwd(p, 0, 2, p, 0, p, p, p, c, p, p, 300, None) == -5
    assert bwd(p, 0, 17, p, 0, p, p, p, c, p, p, 64, None) == -5
    assert bwd(p, 0, 2, p, 3, p, p, p, c, p, p, 64, None) == -5
    assert bwd(p, 0, 2, p, 0, p, p, ctypes.c_void_p(260), c, p, p, 64, None) == -6
    assert bwd(p, 0, 2, p, 0, p, ctypes.c_void_p(258), p, c, p, p, 64, None) == -6


@pytest.mark.skipif(shutil.which("nvcc") is None and not os.path.exists("/usr/local/cuda/bin/nvcc"), reason="no nvcc")
def test_exchange_kernels_compile_without_spills(tmp_path):
    from pinthememory_b200 import build

    cmd = [build._nvcc(), *build.ARCH_FLAGS, "-O3", "-std=c++17", "-Xptxas=-v", "-c",
           os.path.join(build.CSRC, "pm_bn_exchange.cu"), "-o", str(tmp_path / "x.o")]
    r = subprocess.run(cmd, capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    entries = re.findall(r"Compiling entry function '(\w+)'.*?(\d+) bytes spill stores, (\d+) bytes spill loads", r.stderr,
                         flags=re.S)
    assert len(entries) == 2, r.stderr
    for name, st, ld in entries:
        assert st == "0" and ld == "0", name


# ------------------------------------------------------------------------------------------------ which path a layer takes


def _fake_shard(group, world=2, peer=True):
    return types.SimpleNamespace(group=group, world_size=world, rank=0, peer=object() if peer else None)


def test_peer_only_for_the_shard_group_with_peer_memory():
    from pinthememory_b200 import sharding

    g, other = object(), object()
    sh = _fake_shard(g)
    assert sharding.bn_peer(sh, g, 64) is sh.peer
    assert sharding.bn_peer(sh, other, 64) is None                     # the layer reduces over another group
    assert sharding.bn_peer(_fake_shard(g, peer=False), g, 64) is None  # no symmetric memory / NCCL exchange requested
    assert sharding.bn_peer(None, g, 64) is None                       # no sharded update
    assert sharding.bn_peer(_fake_shard(g, world=1), g, 64) is None
    assert sharding.bn_peer(sh, g, 257) is None                        # wider than a row
    assert sharding.bn_peer(_fake_shard(None), None, 64) is not None


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def _worker(rank, world, port, out):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        from pinthememory_b200 import memory, sharding

        res = {}
        W = dist.group.WORLD
        sub = dist.new_group([0, 1])
        res["same"] = [sharding.same_group(None, W), sharding.same_group(W, None), sharding.same_group(None, None),
                       sharding.same_group(sub, sub)]
        res["differ"] = [sharding.same_group(sub, W), sharding.same_group(None, sub)]

        bn = torch.nn.SyncBatchNorm(64).train()
        sync = memory._sync_group(bn)   # the live layer's group: WORLD for process_group None
        res["sync_is_world"] = sync is W
        for shard_group in (None, W):   # enable_sharded_update(group=None) or (group=WORLD): the same group
            sh = types.SimpleNamespace(group=shard_group, world_size=world, rank=rank, peer=object())
            res.setdefault("peer_for_world", []).append(sharding.bn_peer(sh, sync, 64) is sh.peer)
        sh = types.SimpleNamespace(group=sub, world_size=world, rank=rank, peer=object())
        res["peer_for_other_group"] = sharding.bn_peer(sh, sync, 64) is not None
        bn.process_group = sub
        res["sub_layer_on_sub_shard"] = sharding.bn_peer(sh, memory._sync_group(bn), 64) is sh.peer
        res["eval_sync_group"] = memory._sync_group(torch.nn.SyncBatchNorm(64).eval())

        # PINMEM_B200_NCCL_EXCHANGE=1: no peer buffer is set up, so every SyncBatchNorm stays on NCCL
        os.environ["PINMEM_B200_NCCL_EXCHANGE"] = "1"
        try:
            shard = sharding.ShardGroup(None)
            res["env_enabled"] = shard.enable_peer_exchange(torch.device("cpu"))
            res["env_peer"] = sharding.bn_peer(shard, sync, 64)
        finally:
            del os.environ["PINMEM_B200_NCCL_EXCHANGE"]
        out[rank] = res
    finally:
        dist.destroy_process_group()


def test_layer_selection_over_gloo():
    """None and WORLD name the same group; a layer on another group, the NCCL switch and eval mode keep the peer path off."""
    world = 2
    out = mp.get_context("spawn").Manager().dict()
    mp.spawn(_worker, args=(world, _free_port(), out), nprocs=world, join=True)
    for r in range(world):
        res = out[r]
        assert all(res["same"]) and not any(res["differ"])
        assert res["sync_is_world"]
        assert res["peer_for_world"] == [True, True]
        assert not res["peer_for_other_group"]
        assert res["sub_layer_on_sub_shard"]
        assert res["eval_sync_group"] is None          # eval mode: the layer exchanges nothing
        assert res["env_enabled"] is False and res["env_peer"] is None
