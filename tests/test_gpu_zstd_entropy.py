"""The zstd writer's entropy switch (zpb_set_zstd_entropy) on the device: literal-only blocks and full-alphabet Huffman
literals.  Frames decode in the oracle's port, in zpb_unpack_device and in the reference when it is built; LZ4, HC,
stored files and blocks of bytes 0..128 come out as with the switch off, and no zstd frame is larger; the switch reaches
the pipelined host path, Group contexts and multi-round calls; the launch count does not change."""
import numpy as np
import pytest

import entropy_data as ED
from test_gpu_lz4hc import _layout, _pack_device
from zpack_b200 import container, corpus
from zpack_b200 import lib as zlib

pytestmark = pytest.mark.gpu

NONE, ZSTD, LZ4 = 0, 1, 2
SIZES = (0, 1, 12, 13, 4095, 65535, 65536, 65537, 131072, 200001, 262144)


@pytest.fixture(scope="module")
def ent_ctx():
    import zpack_b200
    ctx = zpack_b200.Context(0)
    ctx.set_zstd_entropy(True)
    yield ctx
    ctx.close()


def _unpack_device(ctx, bufs, frames, digest, methods):
    import torch
    arch = container.assemble([f"e{i}" for i in range(len(bufs))], frames, [len(b) for b in bufs], digest, list(methods))
    e = container.parse(arch).entries()
    out_size = int((e["dst_off"] + e["dst_cap"]).max()) + 16
    d_arch = torch.from_numpy(np.ascontiguousarray(arch)).cuda()
    d_out = torch.zeros(out_size, dtype=torch.uint8, device="cuda")
    status, _ = ctx.unpack_device(d_arch, len(arch), d_out, out_size, e)
    assert (status == 0).all(), status
    out = d_out.cpu().numpy()
    for i, b in enumerate(bufs):
        o = int(e["dst_off"][i])
        assert np.array_equal(out[o:o + len(b)], b), i


def _raw_blocks(frame):
    """block types of a zstd frame as pack_kernel.cuh writes it (14-byte header)"""
    p, types = 14, []
    while p < len(frame):
        h = int(frame[p]) | int(frame[p + 1]) << 8 | int(frame[p + 2]) << 16
        types.append((h >> 1) & 3)
        p += 3 + (h >> 3)
        if h & 1:
            break
    return types


@pytest.mark.parametrize("cls", ED.CLASSES)
def test_every_class_and_size_decodes(ent_ctx, oracle, cls):
    bufs = [ED.class_bytes(cls, n, seed=n) for n in SIZES]
    frames, comp, digest, status = _pack_device(ent_ctx, bufs, [ZSTD] * len(bufs), [3] * len(bufs))
    assert (status == 0).all(), status
    for b, fr, dg in zip(bufs, frames, digest):
        assert int(dg) == oracle.xxh3_port(b)
        rc, got = oracle.zstd_decode_port(fr, len(b))
        assert rc == 0 and np.array_equal(got[:len(b)], b), (cls, len(b))
        if oracle.have_ref() and len(b):
            assert np.array_equal(oracle.zstd_decompress_ref(fr, len(b)), b)
    _unpack_device(ent_ctx, bufs, frames, digest, [ZSTD] * len(bufs))
    if cls != "int8rep":
        assert all(2 in _raw_blocks(fr) for b, fr in zip(bufs, frames) if len(b) >= 65536)


def _mixed():
    """LZ4 level 0, zstd of text / runs / random and of the new classes, stored, LZ4 HC"""
    spec = [(corpus.entry_bytes(1, 150000), LZ4, 0), (corpus.entry_bytes(5, 131072), ZSTD, 3), (ED.class_bytes("bf16", 131072), ZSTD, 3),
            (corpus.entry_bytes(0, 70000), ZSTD, 1), (corpus.entry_bytes(2, 100000), ZSTD, 3), (ED.class_bytes("int8", 200001), ZSTD, 3),
            (corpus.entry_bytes(3, 5000), NONE, 0), (corpus.entry_bytes(9, 140000), LZ4, 9), (ED.class_bytes("int8rep", 131072), ZSTD, 3),
            (corpus.entry_bytes(7, 65536), LZ4, 1), (ED.class_bytes("fp32", 65537), ZSTD, 19), (corpus.entry_bytes(13, 40000), ZSTD, 3)]
    return [s[0] for s in spec], [s[1] for s in spec], [s[2] for s in spec]


def test_mixed_batch_against_the_switch_off(oracle):
    import zpack_b200
    bufs, methods, levels = _mixed()
    ctxs = [zpack_b200.Context(0), zpack_b200.Context(0)]
    try:
        for c in ctxs:
            c.set_lz4hc(True)
        ctxs[1].set_zstd_entropy(True)
        off, on = [_pack_device(c, bufs, methods, levels) for c in ctxs]
    finally:
        for c in ctxs:
            c.close()
    assert (off[3] == 0).all() and (on[3] == 0).all()
    assert np.array_equal(off[2], on[2])
    for i, (b, m) in enumerate(zip(bufs, methods)):
        a, z = off[0][i], on[0][i]
        if m != ZSTD or int(b.max()) <= 128 or i == 3:
            assert np.array_equal(a, z), i                 # LZ4, HC, stored, zstd of bytes 0..128 and random: unchanged
        assert len(z) <= len(a), i
        if m == ZSTD:
            rc, got = oracle.zstd_decode_port(z, len(b))
            assert rc == 0 and np.array_equal(got[:len(b)], b), i
    assert sum(len(z) < len(a) for a, z in zip(off[0], on[0])) >= 4


def test_ratio_gates(ent_ctx, oracle):
    """128 KiB entries of each class: at least 0.97 of the order-0 Huffman bound; next to ZSTD_compress level 3 when the
    reference is built (0.95 of it for bf16 and int8)."""
    for cls in ED.CLASSES:
        bufs = [ED.class_bytes(cls, 131072, seed=s) for s in range(8)]
        frames, comp, digest, status = _pack_device(ent_ctx, bufs, [ZSTD] * len(bufs), [3] * len(bufs))
        assert (status == 0).all()
        data = np.concatenate(bufs)
        ratio, bound = len(data) / int(comp.sum()), ED.huffman_bound(data)
        line = f"{cls}: ratio {ratio:.3f}, order-0 Huffman bound {bound:.3f}"
        if oracle.have_ref():
            l3 = len(data) / sum(len(oracle.zstd_compress_ref(b, 3)) for b in bufs)
            line += f", ZSTD_compress level 3 {l3:.3f}"
            if cls in ("bf16", "int8"):
                assert ratio >= 0.95 * l3, line
        print("\n" + line)
        assert ratio >= 0.97 * bound, line


def _batch():
    bufs = [ED.class_bytes(c, n, seed=k) for k, (c, n) in enumerate((("bf16", 1 << 20), ("int8rep", 700000), ("fp16", 1 << 19),
                                                                   ("int8", 900001), ("fp32", 300000)))]
    bufs += [corpus.entry_bytes(i, 400000) for i in range(4)]
    return bufs, [ZSTD] * len(bufs), [3] * len(bufs)


def test_settings_reach_every_path(ent_ctx, monkeypatch):
    import zpack_b200
    bufs, methods, levels = _batch()
    ref_frames, ref_comp, ref_dig, ref_st = _pack_device(ent_ctx, bufs, methods, levels)
    assert (ref_st == 0).all()
    f, h_in, out_size = _layout(ent_ctx, bufs, methods, levels)

    def check_host(comp, digest, status, h_out):
        assert (status == 0).all() and np.array_equal(comp, ref_comp) and np.array_equal(digest, ref_dig)
        for i in range(len(bufs)):
            o = int(f["dst_off"][i])
            assert np.array_equal(h_out[o:o + int(comp[i])], ref_frames[i]), i

    # the pipelined host path: 1 MiB chunks over three workers, which take the caller's settings
    monkeypatch.setenv("ZPB_HOST_CHUNK_MB", "1")
    monkeypatch.setenv("ZPB_HOST_WORKERS", "3")
    ctx = zpack_b200.Context(0)
    try:
        ctx.set_zstd_entropy(True)
        h_out = np.zeros(out_size, np.uint8)
        check_host(*ctx.pack_host(h_in, len(h_in), h_out, out_size, f), h_out)
    finally:
        ctx.close()
    monkeypatch.delenv("ZPB_HOST_CHUNK_MB")
    monkeypatch.delenv("ZPB_HOST_WORKERS")
    # a Group created with the switch in the environment
    monkeypatch.setenv("ZPB_ZSTD_ENTROPY", "1")
    g = zpack_b200.Group(None)
    try:
        h_out = np.zeros(out_size, np.uint8)
        check_host(*g.pack_host(h_in, len(h_in), h_out, out_size, f), h_out)
    finally:
        g.close()
    # several rounds: 16 block slots each
    monkeypatch.setenv("ZPB_PACK_SCRATCH_MB", "1")
    small = zpack_b200.Context(0)
    monkeypatch.delenv("ZPB_PACK_SCRATCH_MB")
    monkeypatch.delenv("ZPB_ZSTD_ENTROPY")
    try:
        frames, comp, digest, status = _pack_device(small, bufs, methods, levels)
    finally:
        small.close()
    assert (status == 0).all() and np.array_equal(comp, ref_comp)
    for i in range(len(bufs)):
        assert np.array_equal(frames[i], ref_frames[i]), i


def test_default_context_writes_raw_blocks(gpu_ctx):
    bufs = [ED.class_bytes("bf16", 262144, seed=1)]
    frames, comp, digest, status = _pack_device(gpu_ctx, bufs, [ZSTD], [3])
    assert (status == 0).all()
    assert _raw_blocks(frames[0]) == [0, 0, 0, 0] and int(comp[0]) == 14 + 4 * 3 + 262144


def test_launch_count_is_the_same(ent_ctx, gpu_ctx):
    bufs, methods, levels = _batch()
    counts = []
    for c in (gpu_ctx, ent_ctx):
        n0 = c.launch_count
        _pack_device(c, bufs, methods, levels)
        counts.append(c.launch_count - n0)
    assert counts[0] == counts[1] and counts[0] > 0


def test_switch_is_exported():
    assert "zpb_set_zstd_entropy" in zlib.EXPORTS
