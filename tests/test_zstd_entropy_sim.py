"""The zstd writer's entropy switch (zpb_set_zstd_entropy) on the CPU emulation of tests/sim: full-alphabet Huffman
literals with FSE-compressed weights, and literal-only blocks where the LZ4 block compressor stored the block.  Every
frame is laid out as pack_kernel.cuh lays it out and must decode in the oracle's zstd port, in the product decoder's CPU
build (tests/sim/zstd_sim.cpp) and in the unmodified reference when it is built.  With the switch on, blocks whose
literals are bytes 0..128 and incompressible blocks must come out byte for byte as with it off, and no block larger.
The GPU tests (tests/test_gpu_zstd_entropy.py) cover the real library."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

from zpack_b200 import corpus

import entropy_data as ED

HERE = os.path.dirname(os.path.abspath(__file__))
SIM = os.path.join(HERE, "sim")
LIB = os.path.join(SIM, "libzstd_entropy_sim.so")
DEC_LIB = os.path.join(SIM, "libzstd_sim.so")
CSRC = os.path.join(os.path.dirname(HERE), "zpack_b200", "csrc")
ZE_SLOT = 65536 + 16384 + 512
ZE_FAIL = 0xFFFFFFFF
CARRIER_FIRST = 0xFFFFFFFF


def _stale(lib, deps):
    return not os.path.exists(lib) or any(os.path.getmtime(d) > os.path.getmtime(lib) for d in deps)


@pytest.fixture(scope="module")
def sim():
    deps = [os.path.join(SIM, f) for f in ("zstd_entropy_sim.cpp", "sim_rt.h", "sim_cuda.h")]
    deps += [os.path.join(CSRC, f) for f in ("pack_blocks.cuh", "zstd_encode.cuh", "ptx.cuh", "common.cuh")]
    if _stale(LIB, deps):
        subprocess.run(["g++", "-O1", "-g", "-std=c++17", "-DZPB_SIM", "-shared", "-fPIC", "-w",
                        os.path.join(SIM, "zstd_entropy_sim.cpp"), "-o", LIB], check=True)
    lib = C.CDLL(LIB)
    vp = C.c_void_p
    lib.sim_zstd_pack_blocks.argtypes = [vp, vp, vp, C.c_uint32, C.c_int, C.c_int, C.c_uint64, vp, vp, vp, vp, vp, vp]
    lib.sim_huf_build.argtypes = [vp, C.c_int, vp, vp]
    lib.sim_huf_build.restype = C.c_uint32
    lib.sim_huf_weights_fse.argtypes = [vp, C.c_int, vp]
    lib.sim_huf_weights_fse.restype = C.c_uint32
    return lib


@pytest.fixture(scope="module")
def product_decode():
    """zstd_decode.cuh compiled for the host (the decoder K4 runs)."""
    src = os.path.join(SIM, "zstd_sim.cpp")
    if _stale(DEC_LIB, [src, os.path.join(CSRC, "zstd_decode.cuh")]):
        subprocess.run(["g++", "-O2", "-fPIC", "-shared", "-w", "-o", DEC_LIB, src], check=True)
    lib = C.CDLL(DEC_LIB)
    lib.zs_sim_decode.restype = C.c_int
    lib.zs_sim_decode.argtypes = [C.c_void_p, C.c_uint64, C.c_void_p, C.c_uint64, C.POINTER(C.c_uint64)]

    def decode(comp, cap):
        comp = np.ascontiguousarray(comp, np.uint8)
        out = np.zeros(max(cap, 1), np.uint8)
        n = C.c_uint64(0)
        rc = lib.zs_sim_decode(comp.ctypes.data, len(comp), out.ctypes.data, cap, C.byref(n))
        return rc, out[:n.value]
    return decode


def pack(sim, blocks, entropy, seed=1, grid=2):
    """One round of zstd blocks (each <= 64 KB) -> per block: (list of Compressed_Block bodies, or None = Raw_Block,
    modes of the windows, (description bytes, carrier))."""
    offs, total = [], 0
    for b in blocks:
        offs.append(total)
        total += len(b) + 5                                    # odd offsets: the literals are read in place
    inp = np.zeros(total + 64, np.uint8)
    for o, b in zip(offs, blocks):
        inp[o:o + len(b)] = b
    n = len(blocks)
    so, ln = np.array(offs, np.uint64), np.array([len(b) for b in blocks], np.uint32)
    csize, winop = np.zeros(n, np.uint32), np.zeros(n * 17, np.uint32)
    zbody, modes, huf = np.zeros(n * 16, np.uint32), np.zeros(n * 16, np.uint32), np.zeros(2 * n, np.uint32)
    zslot = np.zeros(n * ZE_SLOT + 64, np.uint8)
    sim.sim_zstd_pack_blocks(inp.ctypes.data, so.ctypes.data, ln.ctypes.data, n, int(entropy), grid, seed, csize.ctypes.data,
                             winop.ctypes.data, zbody.ctypes.data, zslot.ctypes.data, modes.ctypes.data, huf.ctypes.data)
    out = []
    for k, b in enumerate(blocks):
        zw = zbody[16 * k:16 * k + 16]
        subs = None
        ztotal = sum(int(z) + 3 for z in zw if z and z != ZE_FAIL)
        if len(b) and not (zw == ZE_FAIL).any() and ztotal and ztotal < len(b):     # pack_kernel.cuh's choice
            nwin = (len(b) - 12) // 4096 + 1
            subs = []
            for w in range(nwin):
                if zw[w]:
                    o = k * ZE_SLOT + int(winop[17 * k + w]) + (int(winop[17 * k + w]) >> 2) + 24 * w
                    subs.append(zslot[o:o + int(zw[w])].copy())
        out.append((subs, modes[16 * k:16 * k + 16].copy(), (int(huf[2 * k]), int(huf[2 * k + 1]))))
    return out


def frame(subs_list, blocks):
    """A zstd frame as pack_kernel.cuh writes it: FHD 0xC0 (8-byte content size), window 128 KB, 3-byte block headers."""
    total = sum(len(b) for b in blocks)
    fr = bytearray([0x28, 0xB5, 0x2F, 0xFD, 0xC0, 0x38]) + total.to_bytes(8, "little")
    for k, (subs, raw) in enumerate(zip(subs_list, blocks)):
        last_block = k + 1 == len(blocks)
        if subs is None:
            fr += ((1 if last_block else 0) | (len(raw) << 3)).to_bytes(3, "little") + bytes(raw)
        else:
            for j, body in enumerate(subs):
                last = 1 if last_block and j + 1 == len(subs) else 0
                fr += (last | (2 << 1) | (len(body) << 3)).to_bytes(3, "little") + bytes(body)
    return np.frombuffer(bytes(fr), np.uint8)


def check_decodes(oracle, product_decode, fr, plain, what):
    rc, got = oracle.zstd_decode_port(fr, len(plain))
    assert rc == 0 and np.array_equal(got[:len(plain)], plain), ("oracle port", what)
    rc, got = product_decode(fr, len(plain))
    assert rc == 0 and np.array_equal(got, plain), ("product decoder", what)
    if oracle.have_ref():
        assert np.array_equal(oracle.zstd_decompress_ref(fr, len(plain)), plain), ("reference", what)


def block_frames(res, blocks):
    return [frame([r[0]], [b]) for r, b in zip(res, blocks)]


def _shaped(rng, probs, n):
    return rng.choice(len(probs), n, p=np.asarray(probs, float) / np.sum(probs)).astype(np.uint8)


def test_weight_descriptions(sim, oracle, product_decode):
    """Full-alphabet codes: 129 to 256 symbols of flat, Zipf, two-peak and one-dominant shapes, codes at the 11-bit limit,
    odd and even weight counts.  Each description is FSE-compressed (header byte < 128), and the literal-only block it
    codes decodes everywhere."""
    rng = np.random.default_rng(7)
    shapes = {
        "sparse129": np.r_[np.tile([1.0, 0.0], 127), [1.0, 1.0]], "flat130": np.ones(130), "flat200": np.ones(200),
        "flat201": np.ones(201), "flat255": np.ones(255),
        "zipf256": 1.0 / np.arange(1, 257) ** 1.1, "zipf_steep": 1.0 / np.arange(1, 201) ** 2.2,
        "two_peaks": np.exp(-0.5 * ((np.arange(256) - 40) / 6.0) ** 2) + np.exp(-0.5 * ((np.arange(256) - 200) / 9.0) ** 2) + 1e-3,
        "dominant": np.r_[np.full(180, 0.2), [400.0]],
    }
    blocks, seen_limit, parity = [], False, set()
    for name, p in shapes.items():
        b = _shaped(rng, p, 65536)
        present = np.nonzero(p)[0]
        b[:len(present)] = present                           # every symbol of the alphabet occurs
        hist = np.bincount(b, minlength=256).astype(np.uint32)
        desc, lens = np.zeros(128, np.uint8), np.zeros(256, np.uint8)
        n = sim.sim_huf_build(hist.ctypes.data, 1, desc.ctypes.data, lens.ctypes.data)
        last = int(np.nonzero(hist)[0].max())
        blocks.append(b)
        if name == "flat255":                               # 7.99 bits a byte: refused before the build (entropy)
            assert n == 0
            continue
        assert last >= 129 and len(present) >= 129 and 2 <= n <= 128 and desc[0] < 128 and desc[0] == n - 1, name
        assert sim.sim_huf_build(hist.ctypes.data, 0, desc.ctypes.data, lens.ctypes.data) == 0, name     # switch off: no table
        seen_limit |= int(lens.max()) == 11
        parity.add(last & 1)
    assert seen_limit and parity == {0, 1}
    res = pack(sim, blocks, True)
    for (subs, modes, (dl, carrier)), b, name in zip(res, blocks, shapes):
        if name == "flat255":                               # the block stays raw
            assert subs is None and dl == 0, name
            continue
        assert subs is not None and dl and carrier != CARRIER_FIRST and 2 in modes, name
        check_decodes(oracle, product_decode, frame([subs], [b]), b, name)


def test_weight_description_refusals(sim):
    """No description when every weight is the same (the reference writes none either) or when it would take 128 bytes
    or more, which the header byte cannot express."""
    hist = np.full(256, 256, np.uint32)                      # all 256 symbols equally often: every length 8, every weight 1
    desc, lens = np.zeros(128, np.uint8), np.zeros(256, np.uint8)
    assert sim.sim_huf_build(hist.ctypes.data, 1, desc.ctypes.data, lens.ctypes.data) == 0
    out = np.zeros(128, np.uint8)
    same = np.full(255, 3, np.uint8)
    assert sim.sim_huf_weights_fse(same.ctypes.data, 255, out.ctypes.data) == 0
    rng = np.random.default_rng(3)
    # 255 weights spread evenly over 0..11 are the most a real code can need, and they fit; the size guard itself is
    # exercised with a longer weight array
    wt = rng.permutation(np.arange(255) % 12).astype(np.uint8)
    n = sim.sim_huf_weights_fse(wt.ctypes.data, 255, out.ctypes.data)
    assert 100 < n <= 128 and out[0] == n - 1
    wt = rng.permutation(np.arange(320) % 12).astype(np.uint8)
    assert sim.sim_huf_weights_fse(wt.ctypes.data, 320, out.ctypes.data) == 0
    wt = np.r_[np.full(200, 1), np.full(55, 2)].astype(np.uint8)
    assert 2 <= sim.sim_huf_weights_fse(wt.ctypes.data, 255, out.ctypes.data) < 40


SIZES = (13, 14, 4095, 4096, 4097, 4107, 4108, 4109, 8204, 65535, 65536)


@pytest.mark.parametrize("cls", ED.CLASSES)
def test_literal_only_block_sizes(sim, oracle, product_decode, cls):
    """Blocks of every window-boundary size: each frame decodes, with the switch on and off."""
    blocks = [ED.class_bytes(cls, n, seed=n) for n in SIZES]
    for entropy in (False, True):
        res = pack(sim, blocks, entropy)
        for fr, b in zip(block_frames(res, blocks), blocks):
            check_decodes(oracle, product_decode, fr, b, (cls, len(b), entropy))
    big = [r for r, b in zip(res, blocks) if len(b) >= 8204 and cls != "int8rep"]
    assert all(r[0] is not None for r in big), cls                   # the switch on: these are no longer Raw_Blocks


def _corpus_text_and_skew():
    rng = np.random.default_rng(5)
    skew = (rng.geometric(0.35, 65536) % 100).astype(np.uint8)       # the skewed block of test_pack_sim.py
    skew[::97] = 120
    for q in range(4096, 65536, 256):
        skew[q:q + 96] = skew[q - 4096:q - 4000]
    return [corpus.entry_bytes(i, 65536) for i in (1, 5, 2, 3, 7)] + [corpus.entry_bytes(21, 40000), skew]


def test_blocks_of_bytes_0_to_128_are_unchanged(sim, oracle, product_decode):
    blocks = _corpus_text_and_skew()
    assert all(int(b.max()) <= 128 for b in blocks[:2] + blocks[-1:])
    off, on = pack(sim, blocks, False), pack(sim, blocks, True)
    fo, fn = block_frames(off, blocks), block_frames(on, blocks)
    for a, b, plain in zip(fo, fn, blocks):
        assert np.array_equal(a, b)
        check_decodes(oracle, product_decode, b, plain, "text")
    assert sum(r[0] is not None for r in on) >= 5


def test_random_data_is_unchanged(sim):
    rng = np.random.default_rng(9)
    blocks = [corpus.entry_bytes(i, 65536) for i in (0, 4, 8)] + [rng.integers(0, 256, n, dtype=np.uint8) for n in (65536, 5000, 13)]
    off, on = pack(sim, blocks, False), pack(sim, blocks, True)
    for a, b in zip(block_frames(off, blocks), block_frames(on, blocks)):
        assert np.array_equal(a, b)
    assert all(r[0] is None for r in on)


def test_never_larger(sim, oracle, product_decode):
    """Every block of every kind: with the switch on no frame is larger than with it off."""
    rng = np.random.default_rng(13)
    blocks = _corpus_text_and_skew() + [corpus.entry_bytes(i, 65536) for i in range(8)]
    blocks += [ED.class_bytes(c, 65536, seed=3) for c in ED.CLASSES]
    mixed = ED.class_bytes("int8", 65536, seed=4)                  # int8 with a text run: matches and literals above 128
    mixed[20000:30000] = corpus.entry_bytes(1, 10000)
    mixed[40000:50000] = mixed[20000:30000]
    blocks += [mixed, rng.integers(100, 200, 65536, dtype=np.uint8)]
    off, on = pack(sim, blocks, False), pack(sim, blocks, True)
    for k, (a, b) in enumerate(zip(block_frames(off, blocks), block_frames(on, blocks))):
        assert len(b) <= len(a), (k, len(a), len(b))
        check_decodes(oracle, product_decode, b, blocks[k], k)
    fr = frame([r[0] for r in on], blocks)                         # and all of them as one frame
    check_decodes(oracle, product_decode, fr, np.concatenate(blocks), "all")


@pytest.mark.parametrize("cls", ED.CLASSES)
def test_ratio_against_the_huffman_bound(sim, oracle, cls):
    data = ED.class_bytes(cls, 1 << 20, seed=1)
    blocks = [data[o:o + 65536] for o in range(0, len(data), 65536)]
    res = pack(sim, blocks, True)
    fr = frame([r[0] for r in res], blocks)
    rc, got = oracle.zstd_decode_port(fr, len(data))
    assert rc == 0 and np.array_equal(got[:len(data)], data)
    ratio, bound = len(data) / len(fr), ED.huffman_bound(data)
    off = len(data) / len(frame([r[0] for r in pack(sim, blocks, False)], blocks))
    print(f"\n{cls}: ratio {ratio:.3f} (switch off {off:.3f}), order-0 Huffman bound {bound:.3f}")
    assert ratio >= 0.97 * bound, (ratio, bound)
