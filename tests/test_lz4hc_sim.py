"""The LZ4 HC block compressor (zpack_b200/csrc/lz4hc_blocks.cuh: chains + search kernel, then the parse kernel) on the
CPU emulation of tests/sim: every block it emits is wrapped into an LZ4 frame and decoded by the oracle, its sequences are
checked against the block format's rules, its bytes must not depend on the scheduling, and its size is compared with the
reference algorithm at level 0 (oracle port of LZ4F_compressFrame).  The GPU tests (tests/test_gpu_lz4hc.py) cover the
real library."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

from zpack_b200 import corpus

HERE = os.path.dirname(os.path.abspath(__file__))
SIM = os.path.join(HERE, "sim")
LIB = os.path.join(SIM, "liblz4hc_sim.so")
CSRC = os.path.join(os.path.dirname(HERE), "zpack_b200", "csrc")

LINKS_LEVEL9 = 32          # hc_links(9) in zpack_b200/csrc/pack_api.inl


def _build():
    deps = [os.path.join(SIM, f) for f in ("lz4hc_sim.cpp", "sim_rt.h", "sim_cuda.h")]
    deps += [os.path.join(CSRC, f) for f in ("lz4hc_blocks.cuh", "pack_blocks.cuh", "ptx.cuh", "common.cuh")]
    if os.path.exists(LIB) and all(os.path.getmtime(d) <= os.path.getmtime(LIB) for d in deps):
        return
    subprocess.run(["g++", "-O1", "-g", "-std=c++17", "-DZPB_SIM", "-shared", "-fPIC", "-w",
                    os.path.join(SIM, "lz4hc_sim.cpp"), "-o", LIB], check=True)


@pytest.fixture(scope="module")
def sim():
    _build()
    lib = C.CDLL(LIB)
    vp = C.c_void_p
    lib.sim_lz4hc_pack_blocks.argtypes = [vp, vp, vp, vp, C.c_uint32, vp, vp, C.c_int, C.c_uint64]
    return lib


def pack_blocks(sim, bufs, links=LINKS_LEVEL9, seed=1, grid=2, misalign=0):
    """bufs: list of byte arrays (each <= 64 KB) -> list of (csize, payload)"""
    offs, total = [], misalign
    for b in bufs:
        offs.append(total)
        total += len(b) + (3 if misalign else 0)
    inp = np.zeros(total + 64, np.uint8)
    for o, b in zip(offs, bufs):
        inp[o:o + len(b)] = b
    n = len(bufs)
    so = np.array(offs, np.uint64)
    ln = np.array([len(b) for b in bufs], np.uint32)
    lk = np.full(n, links, np.uint32)
    scratch = np.full(n * 65536 + 64, 0xEE, np.uint8)
    csize = np.full(n, 0xFFFFFFFF, np.uint32)
    sim.sim_lz4hc_pack_blocks(inp.ctypes.data, so.ctypes.data, ln.ctypes.data, lk.ctypes.data, n, scratch.ctypes.data,
                              csize.ctypes.data, grid, seed)
    assert (scratch[n * 65536:] == 0xEE).all()
    return [(int(csize[i]), scratch[i * 65536:i * 65536 + int(csize[i])].copy()) for i in range(n)]


def decode_block(oracle, payload, n):
    hdr = bytes(oracle.lz4f_encode_port(np.zeros(0, np.uint8), 0, independent=True)[:7])
    fr = hdr + len(payload).to_bytes(4, "little") + bytes(payload) + b"\0\0\0\0"
    return oracle.lz4f_decode_port(np.frombuffer(fr, np.uint8), n)


def walk(payload, n):
    """The block's sequences against the format's rules: offsets in 1 .. min(65535, position), no match starting in the
    last 12 bytes or reaching into the last 5, the block ends with a literals-only sequence that covers it exactly."""
    p = pos = 0
    m = len(payload)
    while True:
        tok = int(payload[p]); p += 1
        lit = tok >> 4
        if lit == 15:
            while True:
                b = int(payload[p]); p += 1; lit += b
                if b != 255:
                    break
        p += lit; pos += lit
        if p == m:
            assert pos == n, (pos, n)
            return
        off = int(payload[p]) | int(payload[p + 1]) << 8; p += 2
        ml = (tok & 15) + 4
        if tok & 15 == 15:
            while True:
                b = int(payload[p]); p += 1; ml += b
                if b != 255:
                    break
        assert 1 <= off <= min(65535, pos), (off, pos)
        assert pos <= n - 12 and pos + ml <= n - 5, (pos, ml, n)
        pos += ml


def check(sim, oracle, bufs, **kw):
    res = pack_blocks(sim, bufs, **kw)
    for i, (b, (c, payload)) in enumerate(zip(bufs, res)):
        assert c < max(len(b), 1), (i, c, len(b))              # compressed only if smaller, else 0 = stored
        if c:
            walk(payload, len(b))
            rc, out = decode_block(oracle, payload, len(b))
            assert rc == 0 and np.array_equal(out[:len(b)], b), (i, len(b), c)
    return res


def _shapes():
    rng = np.random.default_rng(7)
    bufs = [np.frombuffer((b"abcdefghijklm" * 6000)[:s], np.uint8) for s in range(14)]       # sizes 0-13
    bufs += [corpus.entry_bytes(50 + i, s) for i, s in enumerate((4095, 65535, 65536))]
    bufs += [np.zeros(65536, np.uint8)]
    bufs += [np.tile(rng.integers(0, 256, k, dtype=np.uint8), 65536 // k + 1)[:16384] for k in range(1, 8)]   # periods 1-7
    bufs += [rng.integers(0, 256, 65536, dtype=np.uint8)]
    far = rng.integers(0, 256, 65536, dtype=np.uint8)                                        # a repeat at distance 65535
    far[65535] = far[0]
    far[65520:65531] = far[0:11]                                                             # and one at 65520
    bufs += [far]
    return bufs


def test_shapes_decode_walk_and_do_not_depend_on_the_scheduling(sim, oracle):
    bufs = _shapes()
    a = check(sim, oracle, bufs, misalign=1)
    b = check(sim, oracle, bufs, seed=9, grid=3)
    assert [x[0] for x in a] == [x[0] for x in b]
    assert all(np.array_equal(x[1], y[1]) for x, y in zip(a, b))
    c = dict(enumerate(a))
    assert c[17][0] and c[17][0] < 400                                                     # all-zero: one long match
    assert c[25][0] == 0                                                                   # random: stored


def test_corpus_classes_ratio_against_the_reference_level0(sim, oracle):
    """Blocks of the four corpus classes (entry i has class i mod 4) at the level-9 search depth, two schedules."""
    bufs = [corpus.entry_bytes(i, 65536) for i in range(1, 12) if i % 4]
    res = check(sim, oracle, bufs)
    res2 = check(sim, oracle, bufs[:3], seed=5, grid=1)
    assert all(np.array_equal(x[1], y[1]) for x, y in zip(res, res2))
    ours, ref = {}, {}
    for i, b, (c, _) in zip([i for i in range(1, 12) if i % 4], bufs, res):
        cls = ("text", "runs", "records")[i % 4 - 1]
        ours[cls] = ours.get(cls, 0) + (c if c else len(b))
        ref[cls] = ref.get(cls, 0) + len(oracle.lz4f_encode_port(b, 0, independent=True)) - 15
    gain = {k: ref[k] / ours[k] for k in ours}
    print("\nLZ4 HC (level-9 depth) vs the reference algorithm at level 0, by class:",
          {k: round(v, 3) for k, v in gain.items()})
    assert gain["text"] >= 1.08
    assert gain["runs"] >= 1.0 and gain["records"] >= 1.0
