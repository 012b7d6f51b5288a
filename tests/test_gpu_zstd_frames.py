"""GPU side of large zstd entries written as one frame per 64 KB (ZPB_ZSTD_FRAMED_MIN and up): the writer's layout
(frame k = the blocks of piece k packed alone, behind a single-segment header), decoding in the oracle's port, the
reference and zpb_unpack_device, and the frame-parallel read — zpb_unpack_blocks_device + zpb_blocks_digest with the
XXH3 relay, zpb_unpack_entry_blocks_host over worker streams, and the drop-in's zpack_read_file."""
import ctypes as C
import os

import numpy as np
import pytest

import entropy_data as ED
from test_gpu_lz4hc import _pack_device
from zpack_b200 import corpus, shard
from zpack_b200 import lib as zlib

pytestmark = pytest.mark.gpu

K64 = 65536
T = zlib.ZSTD_FRAMED_MIN
SIZES = [T - 1, T, T + 1, (12 << 20) + 777, 64 << 20]


@pytest.fixture(scope="module")
def ctxs():
    """zstd_entropy off and on; 1 MiB host chunks, so that one entry spans several chunks and workers"""
    import zpack_b200
    os.environ["ZPB_HOST_CHUNK_MB"] = "1"
    try:
        off, on = zpack_b200.Context(0), zpack_b200.Context(0)
    finally:
        del os.environ["ZPB_HOST_CHUNK_MB"]
    on.set_zstd_entropy(True)
    yield {"mix": off, "bf16": on}
    off.close()
    on.close()


def _data(kind, total):
    return corpus.big_entry(total, piece=1 << 20, first=1) if kind == "mix" else ED.class_bytes("bf16", total)


def _pack(ctx, data):
    frames, _, digest, status = _pack_device(ctx, [data], [1], [3])
    assert status[0] == 0
    return frames[0], int(digest[0])


def _pieces(data):
    return [data[p:p + K64] for p in range(0, len(data), K64)]


@pytest.mark.parametrize("kind", ["mix", "bf16"])
@pytest.mark.parametrize("total", SIZES)
def test_layout_and_decoders(ctxs, oracle, kind, total):
    ctx = ctxs[kind]
    data = _data(kind, total)
    entry, digest = _pack(ctx, data)
    want = oracle.xxh3_port(data)
    assert digest == want
    idx = zlib.zstd_frame_index(entry)
    if total < T:                                                   # today's single frame, 14-byte header
        assert idx is None and entry[4] == 0xC0 and int.from_bytes(entry[6:14].tobytes(), "little") == total
    else:
        frames, content = idx
        pieces = _pieces(data)
        assert content == total and len(frames) == len(pieces)
        assert int(frames["src_off"][0]) == 0 and int(frames["src_off"][-1] + frames["comp_size"][-1]) == len(entry)
        alone, _, _, st = _pack_device(ctx, pieces, [1] * len(pieces), [3] * len(pieces))
        assert (st == 0).all()
        for k, (f, piece) in enumerate(zip(frames, pieces)):
            fr = entry[int(f["src_off"]):int(f["src_off"]) + int(f["comp_size"])]
            h = 6 if len(piece) < 256 else 7
            assert fr[4] == (0x20 if h == 6 else 0x60), k           # single segment, smallest FCS field
            assert np.array_equal(fr[h:], alone[k][14:]), k         # the same blocks as piece k packed alone
            rc, out = oracle.zstd_decode_port(fr, len(piece))
            assert rc == 0 and np.array_equal(out, piece), k
    rc, out = oracle.zstd_decode_port(entry, total)
    assert rc == 0 and np.array_equal(out, data)
    if oracle.have_ref():
        assert np.array_equal(oracle.zstd_decompress_ref(entry, total), data)
    if total <= T + 1 or kind == "bf16":                            # the whole entry as one zpb_unpack_host entry (one warp)
        e = np.zeros(1, zlib.Entry)
        e["comp_size"], e["dst_cap"], e["uncomp_size"], e["hash"], e["method"] = len(entry), total, total, want, 1
        out = np.zeros(total, np.uint8)
        st, dg = ctx.unpack_host(entry, len(entry), out, total, e)
        assert st[0] == 0 and int(dg[0]) == want and np.array_equal(out, data)
    if total >= T:                                                  # frame-parallel, host buffers
        out = np.zeros(total, np.uint8)
        assert ctx.unpack_entry_blocks_host(entry, len(entry), out, total, total, want) == (0, want)
        assert np.array_equal(out, data)


def _decode_sharded(ctx, entry, total, world, archive_off=0):
    """world shards decoded and chained in shard order on one GPU (what N ranks do with a 64-byte relay)"""
    import torch
    frames, content = zlib.zstd_frame_index(entry, archive_off=archive_off)
    assert content == total
    arch = np.concatenate([np.zeros(archive_off, np.uint8), entry])
    d_arch = torch.from_numpy(arch).cuda()
    out = np.zeros(total, np.uint8)
    acc, digest = None, None
    for lo, hi in shard.split_blocks(len(frames), world, K64, total):
        if hi == lo:
            continue
        pos = lo * K64
        size = min(total, hi * K64) - pos
        d_out = torch.zeros(size + 16, dtype=torch.uint8, device="cuda")
        st = ctx.unpack_blocks_device(d_arch, len(arch), d_out, size, np.ascontiguousarray(frames[lo:hi]), K64, size)
        assert st == 0
        acc, dg = ctx.blocks_digest(acc, pos, total, d_out)
        out[pos:pos + size] = d_out[:size].cpu().numpy()
        if dg is not None:
            digest = dg
    return out, digest


@pytest.mark.parametrize("world", [1, 2, 3])
def test_shards_relay_the_digest(ctxs, oracle, world):
    total = (12 << 20) + 777
    data = _data("mix", total)
    entry, _ = _pack(ctxs["mix"], data)
    out, digest = _decode_sharded(ctxs["mix"], entry, total, world, archive_off=5)
    assert np.array_equal(out, data) and digest == oracle.xxh3_port(data)


def test_entry_blocks_host_contract(ctxs, oracle):
    ctx = ctxs["mix"]
    total = (12 << 20) + 777
    data = _data("mix", total)
    entry, want = _pack(ctx, data)
    out = np.zeros(total + 5, np.uint8)
    assert ctx.unpack_entry_blocks_host(entry, len(entry), out, total + 5, total, want) == (0, want)
    assert np.array_equal(out[:total], data) and not out[total:].any()
    assert ctx.unpack_entry_blocks_host(entry, len(entry), out, total, total, want ^ 1) == (zlib.ST_HASH_MISMATCH, want)
    assert ctx.unpack_entry_blocks_host(entry, len(entry), out, total - 1, total, want)[0] == zlib.ST_BUFFER_TOO_SMALL
    out[:] = 0
    assert ctx.unpack_entry_blocks_host(entry, len(entry), out, total, total, want, flags=zlib.F_DISCARD) == (0, want)
    assert not out.any()                                            # verdict only: nothing copied back
    # not eligible -> None (the caller goes through zpb_unpack_host): a single frame, a wrong declared size
    small = data[:T - 1]
    one, dg1 = _pack(ctx, small)
    assert ctx.unpack_entry_blocks_host(one, len(one), out, total, T - 1, dg1) is None
    assert ctx.unpack_entry_blocks_host(entry, len(entry), out, total, total - K64, want) is None


def _block_types(entry, f):
    """(header position, type, size) of every block of the frame at f"""
    p = int(f["src_off"])
    p += 6 if entry[p + 4] == 0x20 else 7
    out = []
    while True:
        bh = int.from_bytes(entry[p:p + 3].tobytes(), "little")
        out.append((p, (bh >> 1) & 3, bh >> 3))
        p += 3 + (1 if (bh >> 1) & 3 == 1 else bh >> 3)
        if bh & 1:
            return out


def test_a_corrupted_frame_gets_the_general_verdict(ctxs, oracle):
    import torch
    ctx = ctxs["mix"]
    total = (12 << 20) + 777
    data = _data("mix", total)
    entry, want = _pack(ctx, data)
    frames, _ = zlib.zstd_frame_index(entry)
    mid = len(frames) // 2
    e = np.zeros(1, zlib.Entry)
    e["comp_size"], e["dst_cap"], e["uncomp_size"], e["hash"], e["method"] = len(entry), total, total, want, 1
    out = np.zeros(total, np.uint8)

    def verdicts(bad):
        st, _ = ctx.unpack_host(bad, len(bad), out, total, e)
        blk = ctx.unpack_entry_blocks_host(bad, len(bad), out, total, total, want)
        rc, _, _ = oracle.read_entry_port(1, bad, total, total, want)
        return int(st[0]), blk, rc

    # a Compressed_Block's body zeroed: the headers still index, the frame fails on the device and the shard declines
    k = next(k for k in range(mid, len(frames)) if any(t == 2 for _, t, _ in _block_types(entry, frames[k])))
    p, _, size = next(b for b in _block_types(entry, frames[k]) if b[1] == 2)
    bad = entry.copy()
    bad[p + 3:p + 3 + size] = 0
    st, blk, rc = verdicts(bad)
    assert blk is None and st == rc == zlib.ST_DECOMPRESS_FAILED
    d_arch = torch.from_numpy(bad).cuda()
    d_out = torch.zeros(total, dtype=torch.uint8, device="cuda")
    assert ctx.unpack_blocks_device(d_arch, len(bad), d_out, total, frames, K64, total) == zlib.ST_NOT_AVAILABLE
    # a byte of a Raw_Block flipped: decodes, digest differs — on both paths
    k = next(k for k in range(mid, len(frames)) if any(t == 0 for _, t, _ in _block_types(entry, frames[k])))
    p, _, _ = next(b for b in _block_types(entry, frames[k]) if b[1] == 0)
    bad = entry.copy()
    bad[p + 10] ^= 0x40
    st, blk, rc = verdicts(bad)
    assert st == rc == zlib.ST_HASH_MISMATCH and blk[0] == zlib.ST_HASH_MISMATCH


def test_argument_contract(ctxs):
    import torch
    ctx = ctxs["mix"]
    data = _data("mix", T)
    entry, _ = _pack(ctx, data)
    frames, _ = zlib.zstd_frame_index(entry)
    d_arch = torch.from_numpy(entry).cuda()
    d_out = torch.zeros(T, dtype=torch.uint8, device="cuda")
    mixed = frames[:2].copy()
    mixed["flags"][1] = 0                                           # an LZ4 block next to a zstd frame
    with pytest.raises(zlib.ZpbError):
        ctx.unpack_blocks_device(d_arch, len(entry), d_out, 2 * K64, mixed, K64, 2 * K64)
    e = np.zeros(1, zlib.Entry)                                     # the internal frame method is not an archive method
    e["comp_size"], e["dst_cap"], e["uncomp_size"], e["method"] = 100, 100, 100, 0x103
    status, _ = ctx.unpack_device(d_arch, len(entry), d_out, T, e)
    assert status[0] == zlib.ST_METHOD_INVALID


def test_drop_in_writes_and_reads_a_framed_entry(oracle):
    from test_host_lib import Options, Reader, Writer, ZFile, _lib
    lib = _lib()
    total = 12 << 20
    data = corpus.big_entry(total, piece=1 << 20)
    opt = Options(1, 3)
    w = Writer()
    assert lib.zpack_init_writer_heap(C.byref(w), C.c_size_t(0)) == 0
    files = (ZFile * 1)()
    files[0].filename, files[0].buffer, files[0].size, files[0].options = b"big.bin", data.ctypes.data, total, C.pointer(opt)
    assert lib.zpack_write_archive(C.byref(w), files, C.c_uint64(1)) == 0
    arch = np.ctypeslib.as_array(C.cast(w.buffer, C.POINTER(C.c_uint8)), shape=(w.file_size,)).copy()
    lib.zpack_close_writer(C.byref(w))
    r = Reader()
    assert lib.zpack_init_reader_memory_shared(C.byref(r), arch.ctypes.data_as(C.c_void_p), C.c_size_t(len(arch))) == 0
    e = r.file_entries[0]
    assert e.comp_method == 1 and e.uncomp_size == total and e.hash == oracle.xxh3_port(data)
    frame = arch[e.offset:e.offset + e.comp_size]
    frames, _ = zlib.zstd_frame_index(frame)                        # eligible: this read is frame-parallel
    out = np.zeros(total, np.uint8)
    assert lib.zpack_read_file(C.byref(r), C.byref(e), out.ctypes.data_as(C.c_void_p), C.c_size_t(total), None) == 0
    assert np.array_equal(out, data)
    p, _, _ = next(b for k in range(len(frames)) for b in _block_types(frame, frames[k]) if b[1] == 0)
    arch[e.offset + p + 10] ^= 0x40                                 # inside a Raw_Block: decodes, digest differs
    assert lib.zpack_read_file(C.byref(r), C.byref(e), out.ctypes.data_as(C.c_void_p), C.c_size_t(total), None) == 15
    arch[e.offset + p + 10] ^= 0x40
    lib.zpack_close_reader(C.byref(r))
    if oracle.have_ref():
        rd = oracle.RefReader(arch)
        rc, ref_out = rd.read(0)
        assert rc == 0 and np.array_equal(ref_out[:total], data)
        rd.close()


def _one_frame(entry, total):
    """The same blocks as one frame with the 14-byte header the writer uses below ZPB_ZSTD_FRAMED_MIN — the layout every
    large zstd entry had before the 64 KB frames, and the shape of the reference's (one frame, dependent blocks)."""
    frames, _ = zlib.zstd_frame_index(entry)
    out = [np.frombuffer(b"\x28\xb5\x2f\xfd\xc0\x38" + int(total).to_bytes(8, "little"), np.uint8)]
    for k, f in enumerate(frames):
        for p, t, size in _block_types(entry, f):
            blk = entry[p:p + 3 + (1 if t == 1 else size)].copy()
            if k + 1 < len(frames):
                blk[0] &= 0xFE                                      # Last_Block only on the entry's final block
            out.append(blk)
    return np.concatenate(out)


def _reader(arch):
    from test_host_lib import Reader, _lib
    lib = _lib()
    r = Reader()
    assert lib.zpack_init_reader_memory_shared(C.byref(r), arch.ctypes.data_as(C.c_void_p), C.c_size_t(len(arch))) == 0
    return lib, r


def _timed_reads(lib, r, order, bufs):
    import time
    t = time.perf_counter()
    for i in order:
        out = np.zeros(len(bufs[i]), np.uint8)
        rc = lib.zpack_read_file(C.byref(r), C.byref(r.file_entries[i]), out.ctypes.data_as(C.c_void_p),
                                 C.c_size_t(len(out)), None)
        assert rc == 0 and np.array_equal(out, bufs[i]), i
    return time.perf_counter() - t


def test_drop_in_reads_64k_frames_frame_parallel_and_one_frame_on_one_warp(ctxs, oracle):
    """zpack_read_file on the same 64 MiB as 64 KB frames and as one frame: both decode; the first takes the
    frame-parallel path, which is many times faster than the one warp the second gets."""
    from zpack_b200 import container
    total = 64 << 20
    data = _data("mix", total)
    framed, want = _pack(ctxs["mix"], data)
    single = _one_frame(framed, total)
    assert zlib.zstd_frame_index(single) is None
    rc, out = oracle.zstd_decode_port(single, total)
    assert rc == 0 and np.array_equal(out, data)
    warm = data[:1 << 20]
    arch = container.assemble(["warm", "framed", "single"], [_pack(ctxs["mix"], warm)[0], framed, single],
                              [len(warm), total, total], [oracle.xxh3_port(warm), want, want], [1, 1, 1])
    lib, r = _reader(arch)
    bufs = [warm, data, data]
    _timed_reads(lib, r, [0], bufs)                                 # context creation and first launches
    t_framed = _timed_reads(lib, r, [1], bufs)
    t_single = _timed_reads(lib, r, [2], bufs)
    lib.zpack_close_reader(C.byref(r))
    assert t_framed * 4 < t_single, (t_framed, t_single)


def test_large_one_frame_entries_stay_in_the_read_ahead(ctxs, oracle):
    """Large zstd entries that are one frame (the reference's layout, and this library's before the 64 KB frames) read in
    order are still decoded together by the read-ahead, one warp each at the same time: in order they take a fraction
    of the time the same reads take out of order (one entry per call)."""
    from zpack_b200 import container
    n, total = 12, T + 1000
    bufs = [corpus.big_entry(total, piece=1 << 20, first=3 * i) for i in range(n)]
    frames, _, digest, st = _pack_device(ctxs["mix"], bufs, [1] * n, [3] * n)
    assert (st == 0).all()
    singles = [_one_frame(f, total) for f in frames]
    if oracle.have_ref():
        singles[-1] = oracle.zstd_compress_ref(bufs[-1], 3)
    arch = container.assemble([f"f{i}" for i in range(n)], singles, [total] * n, [int(d) for d in digest], [1] * n)
    lib, r = _reader(arch)
    _timed_reads(lib, r, [0], bufs)                                 # context creation and first launches
    t_apart = _timed_reads(lib, r, list(range(0, n, 2)) + list(range(1, n, 2)), bufs)
    t_order = _timed_reads(lib, r, range(n), bufs)
    lib.zpack_close_reader(C.byref(r))
    assert t_order * 2 < t_apart, (t_order, t_apart)
