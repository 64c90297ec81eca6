"""Host-side logic of the multi-GPU path on CPU: frame partitioning and the variable-length gather,
world_size 2 over gloo.  The per-rank compressor here is the ORACLE (tests may use it); on GPUs the
same code runs with libzstd_b200 and NCCL (bench.py --gpus N)."""
import os
import socket

import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

import zref
from zstd_b200.sharding import gather_frame_sizes, gather_compressed, partition_frames, split_into_frames


def test_partition_is_contiguous_and_balanced():
    sizes = [64 << 20] * 16
    parts = partition_frames(sizes, 8)
    assert parts == [(2 * i, 2 * i + 2) for i in range(8)]
    sizes = [5, 1, 1, 1, 8, 2, 2, 4, 3, 9]
    for ws in (1, 2, 3, 4, 7):
        parts = partition_frames(sizes, ws)
        assert parts[0][0] == 0 and parts[-1][1] == len(sizes)
        assert all(parts[i][1] == parts[i + 1][0] for i in range(ws - 1))
    assert split_into_frames(10, 4) == [(0, 4), (4, 4), (8, 2)]
    assert split_into_frames(0, 4) == [(0, 0)]


def _worker(rank, world, port, q):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    src = zref.synthetic(3 * (1 << 20) + 777, 42)
    frames = split_into_frames(len(src), 1 << 20)
    b, e = partition_frames([s for _, s in frames], world)[rank]
    local = b"".join(zref.oracle_compress(src[o:o + s], 1) for o, s in frames[b:e])
    sizes, cat, _ = gather_compressed(torch.frombuffer(bytearray(local), dtype=torch.uint8), dst=0)
    # per-frame sizes of all ranks, for one seek table over the gathered frames (contrib/seekable_format)
    mine = [zref.oracle_compress(src[o:o + s], 1) for o, s in frames[b:e]]
    gathered = gather_frame_sizes([len(f) for f in mine], [s for _, s in frames[b:e]], dst=0)
    if rank == 0:
        out = bytes(cat.numpy())
        ok = sum(sizes) == len(out) and zref.ref_decodes(out, src)
        whole = b"".join(zref.oracle_compress(src[o:o + s], 1) for o, s in frames)
        cs, ds = gathered
        ok = ok and sum(cs) == len(out) and ds == [s for _, s in frames]
        import zstd_b200
        seekable = out + zstd_b200.seek_table(cs, ds)
        ok = ok and seekable[-4:] == bytes.fromhex("b1ea928f")
        ok = ok and zref.ref_decodes(seekable, src)                           # the table is a skippable frame
        q.put(bool(ok and out == whole))
    dist.destroy_process_group()


def test_gather_world_size_2_gloo():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    port = s.getsockname()[1]
    s.close()
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    procs = [ctx.Process(target=_worker, args=(r, 2, port, q)) for r in range(2)]
    for p in procs:
        p.start()
    for p in procs:
        p.join(120)
        assert p.exitcode == 0
    assert q.get(timeout=5) is True


def test_split_one_frame_shares():
    """shares of one frame for ZSTDB200_compressFramePart: aligned starts, contiguous, complete; idle ranks marked"""
    from zstd_b200.sharding import split_one_frame
    A = 512 << 10
    for size, world in ((1 << 30, 8), (5 * A + 12345, 3), (3 << 20, 8), (400_000, 2), (0, 2), (A, 1), (A + 1, 4)):
        parts = split_one_frame(size, world, A)
        assert len(parts) == world
        pos = 0
        for b, n in parts:
            if b < 0:
                assert n == 0
                continue
            assert b == pos and b % A == 0
            pos += n
        assert pos == size
        assert sum(1 for b, n in parts if b >= 0) >= 1
