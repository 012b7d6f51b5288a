"""Host side of the frame-parallel zstd path on CPU: zpb_zstd_frame_index (pure framing, no GPU) on entries of 64 KB
frames against an independent walk of zstd_compression_format.md, the shapes it declines, and zpb_pack_bound around
ZPB_ZSTD_FRAMED_MIN."""
import numpy as np
import pytest

from zpack_b200 import corpus
from zpack_b200 import lib as zlib

MAGIC = b"\x28\xb5\x2f\xfd"
K64 = 65536


def _frame(data, single=True, fcs=True, checksum=False, dict_id=False, block=20000):
    """A zstd frame of Raw_Blocks and RLE_Blocks (a piece of one repeated byte) of at most `block` bytes each."""
    n = len(data)
    if single:
        code = 0 if n < 256 else 1 if n < K64 + 256 else 2
    else:
        code = 2 if fcs else 0
    hdr = bytearray(MAGIC) + bytes([(code << 6) | (single << 5) | (checksum << 2) | (1 if dict_id else 0)])
    if not single:
        hdr.append(0x38)                                            # window 128 KB
    if dict_id:
        hdr.append(7)
    if single or fcs:
        v = n - 256 if code == 1 else n
        hdr += v.to_bytes({0: 1, 1: 2, 2: 4}[code], "little")
    pieces = [data[p:p + block] for p in range(0, n, block)] or [data[:0]]
    for k, piece in enumerate(pieces):
        last = k + 1 == len(pieces)
        rle = len(piece) > 1 and (piece == piece[0]).all()
        hdr += (int(last) | ((1 if rle else 0) << 1) | (len(piece) << 3)).to_bytes(3, "little")
        hdr += piece[:1].tobytes() if rle else piece.tobytes()
    if checksum:
        hdr += b"\x00\x00\x00\x00"
    return np.frombuffer(bytes(hdr), np.uint8)


def _framed(data, **kw):
    return np.concatenate([_frame(data[p:p + K64], **kw) for p in range(0, len(data), K64)])


def _walk(entry):
    """Independent restatement of the frame and block-header chain: [(frame start, frame bytes, content size)]."""
    out, p = [], 0
    while p < len(entry):
        assert entry[p:p + 4].tobytes() == MAGIC
        fhd = int(entry[p + 4])
        code, single = fhd >> 6, (fhd >> 5) & 1
        q = p + 5 + (0 if single else 1)
        size = {0: 1, 1: 2, 2: 4, 3: 8}[code]
        fcs = int.from_bytes(entry[q:q + size].tobytes(), "little") + (256 if code == 1 else 0)
        q += size
        while True:
            bh = int.from_bytes(entry[q:q + 3].tobytes(), "little")
            q += 3 + (1 if (bh >> 1) & 3 == 1 else bh >> 3)
            if bh & 1:
                break
        out.append((p, q - p, fcs))
        p = q
    assert p == len(entry)
    return out


def _data(total):
    data = corpus.big_entry(total, piece=K64 + 4321, first=1)
    data[K64 + 100:K64 + 30000] = 0x41                              # RLE blocks in frame 1
    return data


@pytest.mark.parametrize("total", [K64, K64 + 1, 3 * K64 + 255, 3 * K64 + 256, 5 * K64 + 1234, 6 * K64 - 1, 6 * K64])
def test_index_matches_the_frame_chain(total):
    data = _data(total)
    entry = _framed(data)
    got = zlib.zstd_frame_index(entry, archive_off=10)
    assert got is not None
    frames, content = got
    want = _walk(entry)
    assert content == total and len(frames) == len(want) == (total + K64 - 1) // K64
    assert [(int(f["src_off"]) - 10, int(f["comp_size"])) for f in frames] == [w[:2] for w in want]
    assert (frames["flags"] == zlib.BLK_ZSTD).all()
    assert [w[2] for w in want] == [min(K64, total - k * K64) for k in range(len(want))]


def test_index_takes_frames_with_a_window_descriptor_and_an_fcs():
    data = _data(3 * K64 + 7)
    entry = _framed(data, single=False)
    frames, content = zlib.zstd_frame_index(entry)
    assert content == len(data) and [int(f["comp_size"]) for f in frames] == [w[1] for w in _walk(entry)]


def test_index_on_reference_written_frames(oracle):
    if not oracle.have_ref():
        pytest.skip("oracle/_ref not built")
    total = 7 * K64 + 999
    data = corpus.big_entry(total, piece=2 * K64, first=1)
    entry = np.concatenate([oracle.zstd_compress_ref(data[p:p + K64], 3) for p in range(0, total, K64)])
    frames, content = zlib.zstd_frame_index(entry, archive_off=3)
    assert content == total
    assert [(int(f["src_off"]) - 3, int(f["comp_size"])) for f in frames] == [w[:2] for w in _walk(entry)]
    assert zlib.zstd_frame_index(oracle.zstd_compress_ref(data, 3)) is None     # one frame of more than 64 KB


def test_index_declines_every_other_shape():
    data = _data(4 * K64 + 5000)
    ok = _framed(data)
    assert zlib.zstd_frame_index(ok) is not None
    skippable = np.frombuffer(b"\x50\x2a\x4d\x18\x04\x00\x00\x00abcd", np.uint8)
    short = _frame(data[:K64 - 1])
    bad = {
        "one frame > 64 KB": _frame(data),
        "skippable first": np.concatenate([skippable, ok]),
        "skippable last": np.concatenate([ok, skippable]),
        "no FCS": _framed(data, single=False, fcs=False),
        "checksum": _framed(data, checksum=True),
        "dictionary ID": _framed(data, dict_id=True),
        "short frame not last": np.concatenate([short, ok]),
        "trailing bytes": np.concatenate([ok, np.zeros(3, np.uint8)]),
        "empty frame": _frame(data[:0]),
        "empty entry": ok[:0],
    }
    for name, entry in bad.items():
        assert zlib.zstd_frame_index(entry) is None, name
    for cut in (1, 4, 5, 6, 8, 2000, K64 + 9, len(ok) // 2, len(ok) - 1, len(ok) - 3):
        assert zlib.zstd_frame_index(ok[:cut]) is None, cut
    reserved = ok.copy()
    reserved[4] |= 8                                                # reserved bit of the frame header descriptor
    assert zlib.zstd_frame_index(reserved) is None
    btype = ok.copy()
    btype[7] |= 6                                                   # first block: Block_Type 3 (reserved)
    assert zlib.zstd_frame_index(btype) is None
    assert zlib.zstd_frame_index(corpus.big_entry(K64, piece=K64)) is None      # not zstd at all


def test_pack_bound_around_the_framed_threshold():
    bound = zlib.load_library().zpb_pack_bound
    T = zlib.ZSTD_FRAMED_MIN
    for size in (0, 1, K64 - 1, K64, K64 + 1, 1 << 20, T - K64, T - 1):
        nb = max(1, (size + K64 - 1) // K64)
        assert bound(1, size) == 14 + 3 * nb + size, size          # unchanged below the threshold
    for size in (T, T + 1, T + 255, T + 256, T + K64 - 1, (12 << 20) + 777, 1 << 30):
        # the writer's worst case: every 64 KB is a frame (6-byte header below 256 bytes, else 7) + one Raw_Block
        worst = sum((6 if min(K64, size - p) < 256 else 7) + 3 + min(K64, size - p) for p in range(0, size, K64))
        assert bound(1, size) >= worst, size
        assert bound(1, size) == 10 * ((size + K64 - 1) // K64) + size
    assert bound(2, T) == 7 + 4 * (T // K64) + T + 4                # LZ4 is not affected
