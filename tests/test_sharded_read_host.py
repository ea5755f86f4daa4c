"""CPU: host logic of the global-batch read (``enable_sharded_update(global_read=True)``): argument validation, the agreement
check across ranks, the rank-ordered row layout of the NCCL fallback (over gloo), the peer-buffer layout constants and the
argument checks of the new C entries."""
import ctypes
import os
import re
import shutil
import socket
import subprocess

import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def _cpu_module():
    from pinthememory_b200.memory import Memory_sup

    return Memory_sup(19, 32, 32, 0.8, 1.0, False, device="cpu")


def test_global_read_must_be_a_bool():
    from pinthememory_b200 import sharding

    for bad in ("yes", 1, None):
        with pytest.raises(TypeError, match="global_read"):
            sharding.enable_sharded_update(_cpu_module(), global_read=bad)


def test_global_read_off_for_no_group_or_one_rank():
    from pinthememory_b200 import sharding

    class One:
        global_read, world_size = True, 1

    assert not sharding.global_read(None)
    assert not sharding.global_read(One())


def _worker(rank, world, port, flags, out):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        from pinthememory_b200 import capi, sharding

        res = {}
        try:
            shard = sharding.enable_sharded_update(_cpu_module(), global_read=flags[rank])
            res["global_read"] = shard.global_read
            res["active"] = sharding.global_read(shard)
            res["peer"] = shard.peer is not None
            row = torch.arange(capi.READ_ROW_FLOATS, dtype=torch.float32) + 1000.0 * rank
            res["gathered"] = sharding.gather_rows(row, shard)
        except ValueError as e:
            res["error"] = str(e)
        out[rank] = res
    finally:
        dist.destroy_process_group()


def _run(flags):
    world = len(flags)
    out = mp.get_context("spawn").Manager().dict()
    mp.spawn(_worker, args=(world, _free_port(), flags, out), nprocs=world, join=True)
    return [out[r] for r in range(world)]


def test_ranks_that_disagree_on_global_read_all_raise():
    res = _run([True, False])
    for r in res:
        assert "same on every rank" in r["error"]


def test_gather_layout_is_rank_ordered_rows():
    from pinthememory_b200 import capi

    res = _run([True, True])
    for r in res:
        assert r["global_read"] and r["active"] and not r["peer"]
        g = r["gathered"]
        assert g.shape == (2, capi.READ_ROW_FLOATS) and g.is_contiguous()
        for rank in range(2):
            assert torch.equal(g[rank], torch.arange(capi.READ_ROW_FLOATS, dtype=torch.float32) + 1000.0 * rank)


def _header_defines():
    src = open(os.path.join(ROOT, "include", "pinmem_b200.h")).read()
    return {m.group(1): int(m.group(2)) for m in re.finditer(r"#define (PM_\w+) (\d+)", src)}


def test_peer_buffer_layout():
    """The read rows sit in free space of the peer buffer: after the flag area (8 kinds x 32 rows x 16 ranks of u32),
    apart from each other, inside the buffer; the update kernels' offsets are where they were."""
    from pinthememory_b200 import capi

    d = _header_defines()
    assert (d["PM_PEER_DS_OFF"], d["PM_PEER_FLAG_OFF"], d["PM_PEER_BYTES"]) == (36864, 73728, 131072)
    assert (capi.PEER_DS_OFF, capi.PEER_FLAG_OFF, capi.PEER_BYTES) == (36864, 73728, 131072)
    row = d["PM_READ_ROW_FLOATS"] * 4
    assert capi.READ_ROW_FLOATS == d["PM_READ_ROW_FLOATS"]
    assert (capi.PEER_READ_FWD_OFF, capi.PEER_READ_BWD_OFF) == (d["PM_PEER_READ_FWD_OFF"], d["PM_PEER_READ_BWD_OFF"])
    assert d["PM_PEER_FLAG_OFF"] + 8 * 32 * 16 * 4 <= d["PM_PEER_READ_FWD_OFF"]
    assert d["PM_PEER_READ_FWD_OFF"] + row <= d["PM_PEER_READ_BWD_OFF"]
    assert d["PM_PEER_READ_BWD_OFF"] + row <= d["PM_PEER_BYTES"]
    assert d["PM_PEER_READ_FWD_OFF"] % 16 == 0 and d["PM_PEER_READ_BWD_OFF"] % 16 == 0
    # a forward row: 64 floats of column statistics and two doubles; a backward row: 1 + 31 doubles
    assert 64 * 4 + 2 * 8 <= row and (1 + 31) * 8 <= row


def test_exchange_entries_check_arguments_without_a_gpu():
    from pinthememory_b200 import capi

    lib = capi.load()
    p = ctypes.c_void_p(256)
    f = ctypes.c_float(1.0)
    fwd, bwd = lib.pm_read_exchange_fwd, lib.pm_read_exchange_bwd
    assert fwd(None, 0, 2, None, p, None, None, f, None, 19, None) == -1            # no col_partials
    assert fwd(None, 0, 2, None, p, p, p, f, None, 19, None) == -1                  # ws without out
    assert fwd(None, 0, 2, None, None, p, None, f, None, 19, None) == -1            # neither peers nor gathered rows
    assert fwd(p, 0, 2, None, None, p, None, f, None, 19, None) == -1               # peers without an epoch
    assert fwd(None, 0, 2, None, p, p, None, f, None, 0, None) == -4
    assert fwd(None, 0, 17, None, p, p, None, f, None, 19, None) == -5
    assert fwd(p, 2, 2, p, None, p, None, f, None, 19, None) == -5                  # rank outside the group
    assert fwd(None, 0, 2, None, ctypes.c_void_p(260), p, None, f, None, 19, None) == -6
    assert bwd(None, 0, 2, None, p, None, None, None, p, 19, None) == -1
    assert bwd(None, 0, 2, None, p, None, None, p, p, 32, None) == -4
    assert bwd(None, 0, 2, None, p, ctypes.c_void_p(260), None, p, p, 19, None) == -6
    assert lib.pm_read_row_fwd(None, None, p, 19, None) == -1
    assert lib.pm_read_row_bwd(None, None, ctypes.c_void_p(260), 19, None) == -6
    assert lib.pm_score_bwd_partials(p, None, p, 10, 19, None) == -1
    assert lib.pm_score_bwd_global(p, p, None, None, None, None, None, None, p, 10, 19, None) == -1   # g_q without colsums
    assert lib.pm_score_bwd_global(None, None, None, None, None, None, None, None, p, 0, 19, None) == -5


@pytest.mark.skipif(shutil.which("nvcc") is None and not os.path.exists("/usr/local/cuda/bin/nvcc"), reason="no nvcc")
def test_exchange_kernels_compile_without_spills(tmp_path):
    from pinthememory_b200 import build

    cmd = [build._nvcc(), *build.ARCH_FLAGS, "-O3", "-std=c++17", "-Xptxas=-v", "-c",
           os.path.join(build.CSRC, "pm_exchange.cu"), "-o", str(tmp_path / "x.o")]
    r = subprocess.run(cmd, capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    entries = re.findall(r"Compiling entry function '(\w+)'.*?(\d+) bytes spill stores, (\d+) bytes spill loads", r.stderr,
                         flags=re.S)
    assert len(entries) == 6, r.stderr
    for name, st, ld in entries:
        assert st == "0" and ld == "0", name
