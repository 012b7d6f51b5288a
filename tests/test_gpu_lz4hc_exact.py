"""LZ4 HC frames written on the GPU (lz4hc_blocks.cuh) byte for byte against the serial restatement of tests/lz4hc_ref.py:
every level, a context whose small scratch splits the HC blocks over many rounds, the multi-GPU group; and an HC-packed
multi-MiB entry read back through the block-sharded paths.  Large entries are checked on a sample of their blocks, and
their frame layout around the GPU's own payloads, so that the serial reference stays within a few minutes."""
import numpy as np
import pytest

import lz4hc_ref as R
from test_gpu_lz4hc import _layout, _pack_device, hc_ctx  # noqa: F401  (hc_ctx: the fixture)
from zpack_b200 import corpus, shard
from zpack_b200 import lib as zlib

pytestmark = pytest.mark.gpu

LEVELS = list(range(3, 13)) + [16]


def assert_frame(data, frame, level, sample=None):
    """frame == the reference's frame of data at level, on the blocks in sample (all of them if None)"""
    b, K = bytes(data), R.links(level)
    got = R.frame_blocks(bytes(frame))
    nblk = (len(b) + R.BLOCK - 1) // R.BLOCK
    assert len(got) == nblk and bytes(frame) == R.frame_from_blocks(b, got), (len(b), level)
    for k in (range(nblk) if sample is None else sample):
        blk = b[k * R.BLOCK:(k + 1) * R.BLOCK]
        c, payload = got[k]
        assert (c, payload) == R.ref_block(blk, K), f"block {k} of {len(b)}: " + R.explain(blk, K, c, payload)


@pytest.mark.parametrize("level", LEVELS)
def test_levels_equal_the_reference(hc_ctx, level):
    sizes = [0, 13, 4095, 65537, 200001]
    bufs = [corpus.entry_bytes(8 * level + j, s) for j, s in enumerate(sizes)]
    frames, comp, digest, status = _pack_device(hc_ctx, bufs, [2] * len(bufs), [level] * len(bufs))
    assert (status == 0).all(), status
    for b, fr in zip(bufs, frames):
        assert_frame(b, fr, level, sample=[level % 3, 3] if len(b) == 200001 else None)


def _mixed_batch():
    """HC files of several levels among fast LZ4, zstd and stored ones -> bufs, methods, levels"""
    hc = [(200001, 3), (131072, 9), (70000, 12), (65536, 16), (13, 5), (4095, 7), (0, 10), (140000, 6)]
    other = [(150000, 2, 1), (65536, 2, 0), (1000, 2, 2), (100000, 1, 3), (300000, 1, 3), (5000, 0, 0)]
    spec = []
    for i in range(max(len(hc), len(other))):
        if i < len(hc):
            spec.append((hc[i][0], 2, hc[i][1]))
        if i < len(other):
            spec.append(other[i])
    bufs = [corpus.entry_bytes(500 + i, s) for i, (s, _, _) in enumerate(spec)]
    return bufs, [m for _, m, _ in spec], [lv for _, _, lv in spec]


def test_many_rounds_of_four_hc_blocks_equal_the_reference(hc_ctx, monkeypatch):
    """ZPB_PACK_SCRATCH_MB=1: 16 block slots per round, at most 4 of them HC: the HC blocks of one call go through
    several rounds.  The HC frames equal the reference; every frame equals the default context's."""
    import zpack_b200
    bufs, methods, levels = _mixed_batch()
    monkeypatch.setenv("ZPB_PACK_SCRATCH_MB", "1")
    small = zpack_b200.Context(0)
    monkeypatch.delenv("ZPB_PACK_SCRATCH_MB")
    try:
        small.set_lz4hc(True)
        n0 = small.launch_count
        frames, comp, digest, status = _pack_device(small, bufs, methods, levels)
        hc_blocks = sum((len(b) + 65535) >> 16 for b, m, lv in zip(bufs, methods, levels) if m == 2 and lv >= 3)
        assert small.launch_count - n0 >= 2 * ((hc_blocks + 3) // 4)        # two HC launches per round
    finally:
        small.close()
    assert (status == 0).all(), status
    ref = _pack_device(hc_ctx, bufs, methods, levels)
    assert np.array_equal(comp, ref[1]) and np.array_equal(digest, ref[2])
    for i, (b, fr) in enumerate(zip(bufs, frames)):
        assert np.array_equal(fr, ref[0][i]), i
        if methods[i] == 2 and levels[i] >= 3:
            assert_frame(b, fr, levels[i])


def test_hc_entry_reads_through_the_block_sharded_paths(hc_ctx, oracle, monkeypatch):
    """A multi-MiB entry packed at level 9 decodes through zpb_unpack_entry_blocks_host (1 MiB chunks, so several
    chunks and workers) and through zpb_unpack_blocks_device + zpb_blocks_digest relayed over three shards."""
    import torch
    import zpack_b200
    total = (6 << 20) + 777
    data = corpus.big_entry(total, piece=1 << 20, first=1)
    want = oracle.xxh3_port(data)
    [frame], comp, digest, status = _pack_device(hc_ctx, [data], [2], [9])
    assert status[0] == 0 and int(digest[0]) == want
    assert len(frame) < total // 2
    assert_frame(data, frame, 9, sample=[0, 37, len(data) >> 16])
    monkeypatch.setenv("ZPB_HOST_CHUNK_MB", "1")
    ctx = zpack_b200.Context(0)
    monkeypatch.delenv("ZPB_HOST_CHUNK_MB")
    try:
        out = np.zeros(total + 5, np.uint8)
        assert ctx.unpack_entry_blocks_host(frame, len(frame), out, total + 5, total, want) == (0, want)
        assert np.array_equal(out[:total], data)
    finally:
        ctx.close()
    blocks, bs, _ = zlib.lz4_frame_index(frame, archive_off=10)
    arch = np.concatenate([np.zeros(10, np.uint8), frame])
    d_arch = torch.from_numpy(arch).cuda()
    out = np.zeros(total, np.uint8)
    acc, got = None, None
    for lo, hi in shard.split_blocks(len(blocks), 3, bs, total):
        pos, size = lo * bs, min(total, hi * bs) - lo * bs
        d_out = torch.zeros(size + 16, dtype=torch.uint8, device="cuda")
        assert hc_ctx.unpack_blocks_device(d_arch, len(arch), d_out, size, np.ascontiguousarray(blocks[lo:hi]), bs, size) == 0
        acc, dg = hc_ctx.blocks_digest(acc, pos, total, d_out)
        out[pos:pos + size] = d_out[:size].cpu().numpy()
        got = dg if dg is not None else got
    assert got == want and np.array_equal(out, data)


def test_group_created_with_the_switch_packs_the_same_bytes(hc_ctx, monkeypatch):
    """zpb_group_create reads ZPB_LZ4HC like zpb_create: its contexts pack HC files, to the single context's bytes."""
    import zpack_b200
    bufs, methods, levels = _mixed_batch()
    monkeypatch.setenv("ZPB_LZ4HC", "1")
    g = zpack_b200.Group(None)
    monkeypatch.delenv("ZPB_LZ4HC")
    try:
        f, h_in, out_size = _layout(hc_ctx, bufs, methods, levels)
        h_out = np.zeros(out_size, np.uint8)
        comp, digest, status = g.pack_host(h_in, len(h_in), h_out, out_size, f)
    finally:
        g.close()
    assert (status == 0).all(), status
    frames, comp1, digest1, _ = _pack_device(hc_ctx, bufs, methods, levels)
    assert np.array_equal(comp, comp1) and np.array_equal(digest, digest1)
    for i, fr in enumerate(frames):
        o = int(f["dst_off"][i])
        assert np.array_equal(h_out[o:o + int(comp[i])], fr), i
    for i, b in enumerate(bufs):
        if methods[i] == 2 and levels[i] >= 3 and len(b) <= 65536:
            assert_frame(b, frames[i], levels[i])
