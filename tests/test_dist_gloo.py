"""world_size-2 gloo tests (CPU) of the multi-rank host logic: payload layout, variable
length all-gather, blend order, collector ordering / assembly."""
import os
import socket

import numpy as np
import pytest
import torch
import torch.distributed as td
import torch.multiprocessing as mp

import usdu_oracle as orc
from __graft_entry__ import load_package

load_package()
from comfyui_distributed_b200 import dist as udist  # noqa: E402
from comfyui_distributed_b200 import planner  # noqa: E402
from comfyui_distributed_b200.nodes.collector import collect_images, combine_audio  # noqa: E402


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def _run(fn, world, *args):
    port = _free_port()
    mp.spawn(_entry, args=(world, port, fn, args), nprocs=world, join=True)


def _entry(rank, world, port, fn, args):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world))
    load_package()
    td.init_process_group("gloo", rank=rank, world_size=world)
    try:
        fn(rank, world, *args)
    finally:
        td.destroy_process_group()


# ---- pure host logic ------------------------------------------------------------------------
def test_payload_layout_and_blend_order():
    p = planner.get_plan(1600, 1200, 512, 512, 32, 8, True)
    asg = p.partition(2)
    where, sizes = udist.tile_payload_layout(p, asg, B=1)
    assert sorted(where) == list(range(len(p.tiles)))
    for r, tiles in enumerate(asg):
        cur = 0
        for t in tiles:                                   # owner order, 16-byte aligned slots, no overlap
            assert where[t] == (r, cur)
            cur += (p.tiles[t].ph * p.tiles[t].pw * 3 + 15) // 16 * 16
        assert sizes[r] == cur
    assert udist.final_blend_order(asg) == sorted(asg[1])
    assert udist.final_blend_order([[0, 1], [5, 2], [4, 3]]) == [2, 3, 4, 5]


def test_collector_order_matches_reference_rules():
    # master first, then enabled order with repeated ids dropped (the node de-duplicates before assembling,
    # collector.py:245-253; the raw assembly loop is pinned by tests/test_collector_vs_reference.py),
    # unknown ids sorted last
    ids = ["", "w_b", "w_a", "zz", "w_c"]
    assert udist.collector_order(5, ["w_a", "w_b", "w_a", "w_x"], ids) == [0, 2, 1, 4, 3]
    assert udist.collector_order(1, [], [""]) == [0]


def test_oracle_collector_combine():
    m = np.full((1, 2, 2, 3), 0.123456, np.float32)
    w = {"b": np.full((2, 2, 2, 3), 0.5, np.float32), "a": np.full((1, 2, 2, 3), 0.25, np.float32)}
    out = orc.collector_combine(m, w, ["a", "b"])
    assert out.shape == (4, 2, 2, 3)
    assert out[0, 0, 0, 0] == np.float32(0.123456)                       # master keeps full precision
    assert out[1, 0, 0, 0] == np.float32(63) / np.float32(255)           # workers are truncated to u8
    assert out[2, 0, 0, 0] == np.float32(127) / np.float32(255)


def test_combine_audio():
    e = {"waveform": torch.zeros(1, 2, 1), "sample_rate": 44100}
    a = {"waveform": torch.ones(1, 2, 5), "sample_rate": 48000}
    b = {"waveform": torch.ones(1, 2, 3) * 2, "sample_rate": 48000}
    out = combine_audio([a, None, b], e)
    assert out["waveform"].shape == (1, 2, 8) and out["sample_rate"] == 48000
    assert combine_audio([None, None], e) is e


# ---- 2 processes, gloo ------------------------------------------------------------------------
def _w_all_gather_bytes(rank, world):
    n = 1000 + 777 * rank                                 # different sizes per rank
    payload = torch.arange(n, dtype=torch.int64).remainder(251).to(torch.uint8) + rank
    buf, sizes = udist.all_gather_bytes(payload)
    assert sizes == [1000 + 777 * r for r in range(world)]
    assert buf.shape[0] == world and buf.shape[1] % 16 == 0
    for r in range(world):
        ref = torch.arange(sizes[r], dtype=torch.int64).remainder(251).to(torch.uint8) + r
        assert torch.equal(buf[r, : sizes[r]], ref)


def test_all_gather_bytes_two_ranks():
    _run(_w_all_gather_bytes, 2)


def _pack_cpu(images):     # test double of the GPU pack kernel (same arithmetic as the oracle)
    return torch.from_numpy(orc.quantize_u8(images.numpy()))


def _unpack_cpu(q):
    return torch.from_numpy(orc.dequantize_u8(q.numpy()))


def _w_collect(rank, world):
    g = torch.Generator().manual_seed(100 + rank)
    images = torch.rand(1 + rank, 6, 5, 3, generator=g)  # different batch sizes per rank
    combined, order, _ = collect_images(images, ["w1"], "" if rank == 0 else "w1", pack=_pack_cpu, unpack=_unpack_cpu)
    if rank != 0:
        assert combined is None
        return
    assert order == [0, 1]
    g1 = torch.Generator().manual_seed(101)
    w = torch.rand(2, 6, 5, 3, generator=g1)
    ref = orc.collector_combine(images.numpy(), {"w1": w.numpy()}, ["w1"])
    assert np.array_equal(combined.numpy(), ref)


def test_collector_two_ranks():
    _run(_w_collect, 2)


def _w_delegate(rank, world):
    images = torch.full((1, 4, 4, 3), 0.1 * (rank + 1))
    combined, order, _ = collect_images(images, ["w1"], "" if rank == 0 else "w1", delegate_only=True, pack=_pack_cpu,
                                     unpack=_unpack_cpu)
    if rank == 0:
        assert combined.shape[0] == 1                    # master excluded (collector.py:270-274)
        assert np.array_equal(combined.numpy(), orc.dequantize_u8(orc.quantize_u8(np.full((1, 4, 4, 3), 0.2, np.float32))))


def test_collector_delegate_only_two_ranks():
    _run(_w_delegate, 2)


def _w_static_bookkeeping(rank, world):
    """The transport half of static mode on CPU tensors: every rank ships a payload laid out
    by tile_payload_layout; rank 0 finds each worker tile at rank*cap + offset."""
    p = planner.get_plan(1000, 900, 256, 256, 16, 8, True)
    asg = p.partition(world)
    where, sizes = udist.tile_payload_layout(p, asg, 1)
    payload = torch.zeros(sizes[rank], dtype=torch.uint8)
    for t in asg[rank]:
        n = p.tiles[t].ph * p.tiles[t].pw * 3
        payload[where[t][1]: where[t][1] + n] = t % 251   # tile id as content
    buf, got = udist.all_gather_bytes(payload)
    assert got == sizes
    cap = buf.shape[1]
    flat = buf.view(-1)
    for t in udist.final_blend_order(asg):
        r, off = where[t]
        n = p.tiles[t].ph * p.tiles[t].pw * 3
        seg = flat[r * cap + off: r * cap + off + n]
        assert int(seg.min()) == int(seg.max()) == t % 251


def test_static_transport_two_ranks():
    _run(_w_static_bookkeeping, 2)


def test_peer_offsets_address_every_owner_buffer():
    """Offsets handed to the blend kernel in peer mode = distance between the buffers' device
    addresses (as mapped on the reading rank) + the tile's slot inside its owner's payload."""
    from comfyui_distributed_b200 import dist as udist
    where = {0: (0, 0), 1: (1, 0), 2: (2, 16), 3: (1, 4096), 4: (0, 2048)}
    ptrs = [0x7F0000000000, 0x7F0040000000, 0x7E0000000000]          # rank 2's buffer is mapped BELOW the reader's
    offs = udist.peer_offsets([1, 2, 3], where, ptrs, own_rank=0)
    assert offs.dtype == np.int64
    assert list(offs) == [0x40000000, 0x7E0000000000 - 0x7F0000000000 + 16, 0x40000000 + 4096]
    assert list(udist.peer_offsets([0, 4], where, ptrs, own_rank=0)) == [0, 2048]
    assert list(udist.peer_offsets([1], where, ptrs, own_rank=1)) == [0]


def _w_shared_host(rank, world):
    import glob
    sh = udist.SharedHost.get(None)
    sh.MAX_MAPPED = 3
    assert sh.pin == torch.cuda.is_available()            # buffers are page-locked wherever there is a device
    sh.pin = False                                        # the hand-shakes and the mapping policy only, with or without one
    held = None
    rows = [100, 200, 100, 300, 400, 500, 100, 200]
    for j, n in enumerate(rows):
        out = sh.begin((1, n, 4, 3), touch=(rank * (n // 2) * 12, (rank + 1) * (n // 2) * 12))
        out[0, rank * (n // 2):(rank + 1) * (n // 2)] = 10 * j + rank     # this rank's slab
        sh.finish()
        if rank == 0:
            assert torch.equal(out[0, :n // 2], torch.full((n // 2, 4, 3), 10.0 * j))
            assert torch.equal(out[0, n // 2:], torch.full((n // 2, 4, 3), 10.0 * j + 1))
            if j == 1:
                held = out                                # a consumer that keeps its result: never recycled, never unmapped
        assert sh.mapped() <= 3, (j, sh.mapped())
        if j == 2:
            assert sh.mapped() == 2                       # the dropped 100-row buffer was recycled, not mapped again
        del out
        td.barrier()
        assert glob.glob(f"/dev/shm/usdu_b200_{sh.uid}_*") == []          # rank 0 unlinked it once everybody had mapped it
        td.barrier()                                                      # (rank 0 creates the next job's file after this)
    if rank == 0:
        assert torch.equal(held[0, 100:], torch.full((100, 4, 3), 11.0))
        assert sh.bufs[200 * 12][0] is not None and sh.bufs[200 * 12][1] is not None     # the second 200-row job got its own buffer
    assert sorted(k for k in sh.last_use) == sorted((n, i) for n, lst in sh.bufs.items() for i in range(len(lst)) if lst[i] is not None)


def test_shared_host_buffers_are_bounded_unlinked_and_never_taken_from_a_consumer():
    _run(_w_shared_host, 2)
