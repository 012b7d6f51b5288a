"""Regenerates tests/golden/ from the reference's own fixtures and from oracle/_ref.

Run in the build container (needs /root/reference and `make -C oracle ref`):
    python tests/golden/make_golden.py
Outputs (all small, committed):
  archive_{none,zstd,lz4}.zpk, file1.txt, file2.txt  — byte copies of the reference's golden
        archives / plaintexts (/root/reference/tests/workdir, mirrored in tests/archive.h:9-158)
  xxh3_kat.json      — XXH3-64 seed-0 known answers: the upstream table
        (/root/reference/externals/xxHash/xxhsum.c:1246-1272, buffer generator :585-596) plus
        digests computed by the unmodified reference for more lengths
  xxh3_random.json   — XXH3-64 of seeded random buffers (tests/test_oracle.py)
  lz4_cases.npz      — LZ4 frames written by the unmodified reference (LZ4F_compressFrame) for
        hand-picked inputs: linked / independent, stored blocks, checksums, content size, multi-block
  zstd_cases.npz     — zstd frames written by the unmodified reference (ZSTD_compress), several levels
"""
import json
import os
import shutil
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
from oracle import oracle as O  # noqa: E402
from zpack_b200 import corpus  # noqa: E402

HERE = os.path.dirname(os.path.abspath(__file__))
REF = "/root/reference"


def xxh_buffer(n):
    """xxhsum.c:585-596 sanity buffer: byteGen = PRIME32; buf[i] = byteGen >> 56; byteGen *= PRIME64."""
    P32, P64 = 2654435761, 11400714785074694797
    g, out = P32, bytearray(n)
    for i in range(n):
        out[i] = (g >> 56) & 0xFF
        g = (g * P64) & 0xFFFFFFFFFFFFFFFF
    return bytes(out)


def main():
    for f in ("archive_none.zpk", "archive_zstd.zpk", "archive_lz4.zpk", "file1.txt", "file2.txt"):
        shutil.copyfile(os.path.join(REF, "tests/workdir", f), os.path.join(HERE, f))

    # upstream KAT rows {len: XXH3_64bits(seed 0)} copied as data from xxhsum.c:1246-1272
    upstream = {0: 0x2D06800538D394C2, 1: 0xC44BDFF4074EECDB, 6: 0x27B56A84CD2D7325,
                12: 0xA713DAF0DFBB77E7, 24: 0xA3FE70BF9D3510EB, 48: 0x397DA259ECBA1F11,
                80: 0xBCDEFBBB2C47C90A, 195: 0xCD94217EE362EC3A, 403: 0xCDEB804D65C6DEA4,
                512: 0x617E49599013CB6B, 2048: 0xDD59E2C3A5F038E0, 2240: 0x6E73A90539CF2948,
                2367: 0xCB37AEB9E5D361ED}
    buf = xxh_buffer(70000)
    kat = {"generator": "xxhsum.c:585-596", "upstream": {}, "reference_run": {}}
    for n, h in upstream.items():
        assert O.xxh3_ref(buf[:n]) == h, (n, hex(O.xxh3_ref(buf[:n])), hex(h))
        kat["upstream"][str(n)] = f"{h:016x}"
    extra = list(range(0, 260)) + [1023, 1024, 1025, 1087, 1088, 1089, 2047, 2049, 4096, 4097, 65535, 65536, 65537, 69999]
    for n in extra:
        kat["reference_run"][str(n)] = f"{O.xxh3_ref(buf[:n]):016x}"
    json.dump(kat, open(os.path.join(HERE, "xxh3_kat.json"), "w"), indent=0)

    # XXH3-64 of random buffers at the lengths tests/test_oracle.py::test_ref_agrees_on_xxh3_random_lengths draws.
    # (The committed table was written with upstream xxHash 0.8.2, whose XXH3_64bits reproduces every digest of
    # xxh3_kat.json; XXH3's output is frozen since 0.8.0, the version the reference pins.)
    rng = np.random.default_rng(7)
    rbuf = rng.integers(0, 256, 300000, dtype=np.uint8)
    lengths = list(range(0, 300)) + [int(x) for x in rng.integers(300, 300000, 60)]
    json.dump({"generator": "buf = numpy default_rng(7).integers(0, 256, 300000, uint8); lengths 0..299, then 60 of the same "
                            "generator's integers(300, 300000)",
               "xxh3_64": [[n, f"{O.xxh3_ref(rbuf[:n]):016x}"] for n in lengths]},
              open(os.path.join(HERE, "xxh3_random.json"), "w"), indent=0)

    rng = np.random.default_rng(1234)
    inputs = {
        "empty": np.zeros(0, np.uint8),
        "one": np.array([65], np.uint8),
        "tiny12": np.frombuffer(b"abcabcabcabc", np.uint8),
        "text_5k": corpus.entry_bytes(1, 5000),
        "runs_70k": corpus.entry_bytes(2, 70000),
        "records_64k": corpus.entry_bytes(3, 65536),
        "random_66k": corpus.entry_bytes(0, 66000),
        "text_200k": corpus.entry_bytes(5, 200000),
        "mixed_300k": np.concatenate([corpus.entry_bytes(i, 75000) for i in range(4)]),
        "zeros_100k": np.zeros(100000, np.uint8),
        "short_period": np.tile(np.frombuffer(b"abcde", np.uint8), 3000),
        "noise_lowent": rng.integers(0, 4, 40000, dtype=np.uint8),
    }
    lz4 = {}
    for name, data in inputs.items():
        lz4[f"{name}__in"] = data
        lz4[f"{name}__linked"] = O.lz4f_compress_ref(data, level=0)                 # what ZPack writes
        lz4[f"{name}__indep"] = O.lz4f_compress_ref(data, level=0, block_mode=1)
    lz4["text_200k__hc9"] = O.lz4f_compress_ref(inputs["text_200k"], level=9)
    lz4["text_200k__accel"] = O.lz4f_compress_ref(inputs["text_200k"], level=-4)
    lz4["mixed_300k__sums"] = O.lz4f_compress_ref(inputs["mixed_300k"], content_checksum=1, block_checksum=1,
                                                  content_size=len(inputs["mixed_300k"]))
    lz4["mixed_300k__256k"] = O.lz4f_compress_ref(inputs["mixed_300k"], block_size_id=5)
    lz4["runs_70k__4m_indep"] = O.lz4f_compress_ref(inputs["runs_70k"], block_size_id=7, block_mode=1)
    np.savez_compressed(os.path.join(HERE, "lz4_cases.npz"), **lz4)

    zs = {}
    for name, data in inputs.items():
        zs[f"{name}__in"] = data
        zs[f"{name}__l3"] = O.zstd_compress_ref(data, 3)
    for lvl in (1, 5, 9, 19):
        zs[f"text_200k__l{lvl}"] = O.zstd_compress_ref(inputs["text_200k"], lvl)
        zs[f"mixed_300k__l{lvl}"] = O.zstd_compress_ref(inputs["mixed_300k"], lvl)
    np.savez_compressed(os.path.join(HERE, "zstd_cases.npz"), **zs)

    # zstd stress frames: zstd's own generator (externals/zstd/tests/decodecorpus.c, built by oracle/Makefile as
    # oracle/_ref/decodecorpus), seeded, content up to 128 KiB; plus the upstream golden frame whose first block is RLE.
    # Stored: the frame, and of the original its size and XXH3-64 (the unmodified reference decoder's output is the truth).
    import subprocess
    import tempfile
    gen = os.path.join(ROOT, "oracle", "_ref", "decodecorpus")
    zc = {}
    with tempfile.TemporaryDirectory() as td:
        zdir, odir = os.path.join(td, "z"), os.path.join(td, "o")
        os.mkdir(zdir); os.mkdir(odir)
        subprocess.run([gen, "-n240", "-s20261018", "--max-content-size-log=17", f"-p{zdir}", f"-o{odir}"], check=True,
                       stdout=subprocess.DEVNULL, stderr=subprocess.DEVNULL)
        names = sorted(os.listdir(zdir))
        sizes, digests = [], []
        for k, nm in enumerate(names):
            fr = np.fromfile(os.path.join(zdir, nm), np.uint8)
            orig = np.fromfile(os.path.join(odir, nm.replace("z", "o", 1).replace(".zst", "")), np.uint8) if os.path.exists(
                os.path.join(odir, nm.replace("z", "o", 1).replace(".zst", ""))) else None
            got = O.zstd_decompress_ref(fr, 1 << 18)
            if orig is not None:
                assert np.array_equal(got, orig), nm
            zc[f"f{k:03d}"] = fr
            sizes.append(len(got)); digests.append(O.xxh3_ref(got))
    rle = np.fromfile(os.path.join(REF, "externals/zstd/tests/golden-decompression/rle-first-block.zst"), np.uint8)
    got = O.zstd_decompress_ref(rle, 1 << 22)
    zc["rle_first_block"] = rle
    sizes.append(len(got)); digests.append(O.xxh3_ref(got))
    zc["__names"] = np.array([f"f{k:03d}" for k in range(len(sizes) - 1)] + ["rle_first_block"])
    zc["__sizes"] = np.array(sizes, np.uint64)
    zc["__xxh3"] = np.array(digests, np.uint64)
    np.savez_compressed(os.path.join(HERE, "zstd_corpus.npz"), **zc)
    print("golden fixtures written:", sorted(os.listdir(HERE)))


if __name__ == "__main__":
    main()
