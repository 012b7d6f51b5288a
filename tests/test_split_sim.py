"""The pre-pass that cuts a large entry of a batch into 64 KB pseudo-rows (split_index_kernel, zpack_b200/csrc/
split_entries.cuh) on the CPU emulation (tests/sim/sim_rt.h): for every input its verdict and its rows equal what the
host index functions (zpb_lz4_frame_index / zpb_zstd_frame_index) say about the same bytes."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

from zpack_b200 import corpus
from zpack_b200 import lib as zlib
from zpack_b200.lib import Entry

HERE = os.path.dirname(os.path.abspath(__file__))
SIM = os.path.join(HERE, "sim")
LIB = os.path.join(SIM, "libsplit_sim.so")
CSRC = os.path.join(os.path.dirname(HERE), "zpack_b200", "csrc")

K64 = 65536
T = zlib.ZSTD_FRAMED_MIN
M_LZ4_BLOCK, M_ZSTD_FRAME, M_SPLIT, F_STORED_BLK = 0x102, 0x103, 0x104, 0x100
DESC_PER_BLOCK = 2060
FastAux = np.dtype([("desc_base", "<u8"), ("slot_base", "<u4"), ("nslots", "<u4")])


def _build():
    deps = [os.path.join(SIM, f) for f in ("split_sim.cpp", "sim_rt.h", "sim_cuda.h")]
    deps += [os.path.join(CSRC, f) for f in ("split_entries.cuh", "lz4_fast.cuh", "ptx.cuh", "common.cuh")]
    if os.path.exists(LIB) and all(os.path.getmtime(d) <= os.path.getmtime(LIB) for d in deps):
        return
    subprocess.run(["g++", "-O1", "-g", "-std=c++17", "-DZPB_SIM", "-shared", "-fPIC", "-w",
                    os.path.join(SIM, "split_sim.cpp"), "-o", LIB], check=True)


@pytest.fixture(scope="module")
def sim():
    _build()
    lib = C.CDLL(LIB)
    vp = C.c_void_p
    lib.sim_split_index.argtypes = [vp, vp, C.c_uint64, C.c_uint64, C.c_uint32, vp, vp, C.c_uint64]
    return lib


# ---- inputs ------------------------------------------------------------------------------------------------------

def _lz4_frame(blocks, content=None, independent=True):
    """An LZ4 frame of stored 64 KB blocks (the framing is what the pre-pass reads; block bodies are not decoded)."""
    flg = 0x40 | (0x20 if independent else 0) | (0x08 if content is not None else 0)
    desc = bytes([flg, 0x40]) + (content.to_bytes(8, "little") if content is not None else b"")
    hc = (zlib_xxh32(desc) >> 8) & 0xFF
    out = bytearray(b"\x04\x22\x4d\x18") + desc + bytes([hc])
    for b in blocks:
        out += (len(b) | (1 << 31)).to_bytes(4, "little") + b.tobytes()
    out += b"\x00\x00\x00\x00"
    return np.frombuffer(bytes(out), np.uint8)


def zlib_xxh32(data, seed=0):
    P1, P2, P3, P4, P5 = 0x9E3779B1, 0x85EBCA77, 0xC2B2AE3D, 0x27D4EB2F, 0x165667B1
    m = 0xFFFFFFFF
    rotl = lambda v, r: ((v << r) | (v >> (32 - r))) & m  # noqa: E731
    h = (seed + P5 + len(data)) & m
    i = 0
    while i + 4 <= len(data):
        h = rotl((h + int.from_bytes(data[i:i + 4], "little") * P3) & m, 17) * P4 & m
        i += 4
    while i < len(data):
        h = rotl((h + data[i] * P5) & m, 11) * P1 & m
        i += 1
    h ^= h >> 15; h = h * P2 & m; h ^= h >> 13; h = h * P3 & m; h ^= h >> 16
    return h


def _zstd_frame(data, checksum=False, dict_id=False, block=20000):
    """One single-segment zstd frame of Raw_Blocks of at most `block` bytes (the writer's header layout)."""
    n = len(data)
    code = 0 if n < 256 else 1 if n < K64 + 256 else 2
    hdr = bytearray(b"\x28\xb5\x2f\xfd") + bytes([(code << 6) | 0x20 | (checksum << 2) | (1 if dict_id else 0)])
    if dict_id:
        hdr.append(7)
    hdr += (n - 256 if code == 1 else n).to_bytes({0: 1, 1: 2, 2: 4}[code], "little")
    pieces = [data[p:p + block] for p in range(0, n, block)]
    for k, piece in enumerate(pieces):
        hdr += (int(k + 1 == len(pieces)) | (len(piece) << 3)).to_bytes(3, "little") + piece.tobytes()
    if checksum:
        hdr += b"\x00\x00\x00\x00"
    return np.frombuffer(bytes(hdr), np.uint8)


def _zstd_framed(data, frame=K64, **kw):
    return np.concatenate([_zstd_frame(data[p:p + frame], **kw) for p in range(0, len(data), frame)])


def _data(total, seed=1):
    return corpus.big_entry(total, piece=K64 + 4321, first=seed)


def _lz4(total, **kw):
    data = _data(total)
    return _lz4_frame([data[p:p + K64] for p in range(0, total, K64)], **kw), total


# ---- the comparison ----------------------------------------------------------------------------------------------

def _host_view(entry, uncomp, src_off, method):
    """What the host index functions accept: the rows they imply, or None."""
    nrows = (uncomp + K64 - 1) // K64
    if method == 2:
        got = zlib.lz4_frame_index(entry, archive_off=src_off)
        if got is None:
            return None
        blocks, _, content = got
        if len(blocks) != nrows or (content is not None and content != uncomp):
            return None
        sizes = [K64] * (nrows - 1) + [uncomp - K64 * (nrows - 1)]
        return [(int(b["src_off"]), int(b["comp_size"]), sizes[k], F_STORED_BLK if b["flags"] & zlib.BLK_STORED else 0)
                for k, b in enumerate(blocks)]
    got = zlib.zstd_frame_index(entry, archive_off=src_off)
    if got is None or got[1] != uncomp:
        return None
    frames = got[0]
    sizes = [K64] * (len(frames) - 1) + [uncomp - K64 * (len(frames) - 1)]
    return [(int(f["src_off"]), int(f["comp_size"]), sizes[k], 0) for k, f in enumerate(frames)]


def check(sim, entry, uncomp, method, skew=0, seed=1):
    """The entry at archive offset 48 + skew; the pre-pass must agree with the host index on every field."""
    src_off = 48 + skew
    arch = np.zeros(src_off + len(entry) + 64, np.uint8)
    arch[src_off:src_off + len(entry)] = entry
    arch[src_off + len(entry):] = 0xA5                  # bytes after the entry: never part of a row
    parent = np.zeros(1, Entry)
    parent[0] = (src_off, len(entry), 1 << 30, uncomp, uncomp, 1234, method, 0, 0)
    nrows = (uncomp + K64 - 1) // K64
    rows = np.zeros(nrows + 1, Entry)
    aux = np.zeros(nrows + 1, FastAux)
    ok = sim.sim_split_index(arch.ctypes.data, parent.ctypes.data, 100, 4000, 7, rows.ctypes.data, aux.ctypes.data,
                             seed)
    want = _host_view(entry, uncomp, src_off, method)
    assert bool(ok) == (want is not None)
    if want is None:
        assert int(rows[0]["method"]) == method
        assert (rows["comp_size"][1:] == 0).all()        # inert: the scan kernel reports them OK and nothing else
        return False
    assert int(rows[0]["method"]) == M_SPLIT
    r = rows[1:]
    assert [(int(x["src_off"]), int(x["comp_size"]), int(x["uncomp_size"]), int(x["flags"])) for x in r] == want
    assert (r["dst_cap"] == r["uncomp_size"]).all() and (r["hash"] == 0).all()
    assert (r["dst_off"] == (1 << 30) + K64 * np.arange(nrows, dtype=np.uint64)).all()
    assert (r["reserved"] == 100 + 64 * np.arange(nrows, dtype=np.uint64)).all()
    assert (r["method"] == (M_LZ4_BLOCK if method == 2 else M_ZSTD_FRAME)).all()
    if method == 2:                                      # fast_scan_lz4's descriptor layout inside the reservation
        ip = r["src_off"].astype(np.int64) - src_off
        k = np.arange(nrows)
        assert (aux[1:]["desc_base"] == 4000 + ((ip // 3 + DESC_PER_BLOCK * k + 3) & ~3)).all()
        assert (aux[1:]["slot_base"] == 7 + k).all() and (aux[1:]["nslots"] == 1).all()
    return True


SIZES = [T - 1, T, T + 1, 12 * 2**20 + 777]


@pytest.mark.parametrize("total", SIZES)
@pytest.mark.parametrize("skew", [0, 5])
def test_lz4_writer_shape(sim, total, skew):
    entry, uncomp = _lz4(total, content=total if total % 2 else None)
    assert check(sim, entry, uncomp, 2, skew=skew)


@pytest.mark.parametrize("total", SIZES)
@pytest.mark.parametrize("skew", [0, 11])
def test_zstd_writer_shape(sim, total, skew):
    data = _data(total)
    assert check(sim, _zstd_framed(data), total, 1, skew=skew)


def test_64_mib(sim):
    total = 64 << 20
    assert check(sim, *_lz4(total), 2, skew=3)
    assert check(sim, _zstd_framed(_data(total), block=K64), total, 1, skew=9)


def test_linked_lz4_and_one_frame_zstd_decline(sim):
    entry, uncomp = _lz4(T + 5, independent=False)
    assert not check(sim, entry, uncomp, 2)
    data = _data(T + 5)
    assert not check(sim, _zstd_frame(data, block=100000), T + 5, 1)   # one frame of 4 MiB: FCS > 64 KB


def _lz4_blocks(total):
    data = _data(total)
    return [data[p:p + K64] for p in range(0, total, K64)]


def test_lz4_crafted_declines(sim):
    total = T + 999
    blocks = _lz4_blocks(total)
    good = _lz4_frame(blocks)
    # a block header of more than 64 KB (the size field is the real one: the walk stays in bounds)
    big = blocks[:3] + [np.concatenate([blocks[3], blocks[4][:1]])] + blocks[5:]
    assert not check(sim, _lz4_frame(big), total + 1, 2)
    # a truncated last block, and a frame cut before its end mark
    assert not check(sim, good[:-10], total, 2)
    assert not check(sim, good[:-4], total, 2)
    # trailing bytes after the end mark
    assert not check(sim, np.concatenate([good, np.zeros(7, np.uint8)]), total, 2)
    # content size that disagrees with the entry's uncomp_size, and a block count that does
    assert not check(sim, _lz4_frame(blocks, content=total + 1), total, 2)
    assert not check(sim, good, total + K64, 2)
    assert not check(sim, good, total - 1000, 2)
    # a header checksum byte that does not match
    bad = good.copy()
    bad[6] ^= 1
    assert not check(sim, bad, total, 2)


def test_zstd_crafted_declines(sim):
    total = T + 999
    data = _data(total)
    good = _zstd_framed(data)
    assert not check(sim, _zstd_framed(data, checksum=True), total, 1)
    assert not check(sim, _zstd_framed(data, dict_id=True), total, 1)
    # a frame of other than 64 KB before the last
    odd = np.concatenate([_zstd_frame(data[:K64 - 16]), _zstd_framed(data[K64 - 16:])])
    assert not check(sim, odd, total, 1)
    assert not check(sim, good[:-5], total, 1)                           # truncated last block
    assert not check(sim, np.concatenate([good, np.zeros(3, np.uint8)]), total, 1)   # trailing bytes
    assert not check(sim, good, total + 1, 1)                            # content-size mismatch
    bad = good.copy()
    bad[len(_zstd_frame(data[:K64])) + 5 + 4] |= 6                       # second frame's first block: reserved type
    assert not check(sim, bad, total, 1)
