"""LZ4 HC levels on the GPU writer (zpb_set_lz4hc / ZPB_LZ4HC, lz4hc_blocks.cuh): frames of every level decode in the
oracle's port and on the GPU reader, carry the right XXH3-64, do not depend on the call, leave the other methods of a
batch byte-identical, and compress better than the GPU's level 0 of the same call.  Every test uses its own context
with the switch on; the shared one keeps the default (levels >= 3 refused, tests/test_gpu_pack.py)."""
import os
import subprocess
import sys

import numpy as np
import pytest

from zpack_b200 import container, corpus
from zpack_b200 import lib as zlib

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SIZES = [0, 1, 5, 12, 13, 14, 64, 1000, 4095, 65535, 65536, 65537, 131072, 200001, 262144]   # as tests/test_gpu_pack.py
HEADER = bytes([0x04, 0x22, 0x4D, 0x18, 0x60, 0x40])


@pytest.fixture(scope="module")
def hc_ctx():
    import zpack_b200
    ctx = zpack_b200.Context(0)
    ctx.set_lz4hc(True)
    yield ctx
    ctx.close()


def _layout(ctx, bufs, methods, levels):
    f = np.zeros(len(bufs), zlib.File)
    in_off = out_off = 0
    for i, b in enumerate(bufs):
        cap = ctx.pack_bound(int(methods[i]), len(b))
        f["src_off"][i], f["size"][i], f["dst_off"][i], f["dst_cap"][i] = in_off, len(b), out_off, cap
        f["method"][i], f["level"][i] = methods[i], levels[i]
        in_off += (len(b) + 15) & ~15
        out_off += (cap + 15) & ~15
    h_in = np.zeros(max(in_off, 16), np.uint8)
    for i, b in enumerate(bufs):
        h_in[int(f["src_off"][i]):int(f["src_off"][i]) + len(b)] = b
    return f, h_in, max(out_off, 16)


def _pack_device(ctx, bufs, methods, levels):
    import torch
    f, h_in, out_size = _layout(ctx, bufs, methods, levels)
    d_in = torch.from_numpy(h_in).cuda()
    d_out = torch.zeros(out_size, dtype=torch.uint8, device="cuda")
    comp, digest, status = ctx.pack_device(d_in, len(h_in), d_out, out_size, f)
    h_out = d_out.cpu().numpy()
    frames = [h_out[int(f["dst_off"][i]):int(f["dst_off"][i] + comp[i])].copy() for i in range(len(bufs))]
    return frames, comp, digest, status


def _gpu_unpack(ctx, bufs, frames, digest, methods):
    arch = container.assemble([f"h{i}" for i in range(len(bufs))], frames, [len(b) for b in bufs], digest, list(methods))
    e = container.parse(arch).entries()
    out = np.zeros(int((e["dst_off"] + e["dst_cap"]).max()) + 16, np.uint8)
    st, _ = ctx.unpack_host(arch, len(arch), out, len(out), e)
    assert (st == 0).all(), st
    for i, b in enumerate(bufs):
        o = int(e["dst_off"][i])
        assert np.array_equal(out[o:o + len(b)], b), i
    return arch


@pytest.mark.parametrize("level", [3, 6, 9, 12, 16])
def test_levels_decode_with_the_oracle_and_the_gpu_reader(hc_ctx, oracle, level):
    bufs = [corpus.entry_bytes(i, s) for i, s in enumerate(SIZES * 2)]
    frames, comp, digest, status = _pack_device(hc_ctx, bufs, [2] * len(bufs), [level] * len(bufs))
    assert (status == 0).all(), status
    for i, (b, fr) in enumerate(zip(bufs, frames)):
        assert len(fr) <= hc_ctx.pack_bound(2, len(b))
        assert bytes(fr[:6]) == HEADER
        rc, out = oracle.lz4f_decode_port(fr, len(b))
        assert rc == 0 and np.array_equal(out, b), (i, len(b))
        assert int(digest[i]) == oracle.xxh3_port(b)
    _gpu_unpack(hc_ctx, bufs, frames, digest, [2] * len(bufs))


def test_files_of_varied_statistics_round_trip(hc_ctx, oracle):
    """As tests/test_gpu_pack.py::test_files_of_varied_statistics_round_trip, at HC levels."""
    rng = np.random.default_rng(321)
    bufs = []
    for t in range(40):
        n = int(rng.choice([1, 12, 13, 4095, 4109, 65535, 65536, 65537, 100000, 200000, 262144]))
        alpha = int(rng.choice([2, 5, 16, 64, 120, 256]))
        b = rng.integers(0, alpha, n, dtype=np.uint8) if t % 3 else (rng.zipf(1.3, n) % alpha).astype(np.uint8)
        for _ in range(int(rng.choice([0, 50, 400, 3000]))):
            ln = int(rng.choice([4, 5, 8, 20, 70, 300]))
            if n <= 2 * ln + 2:
                break
            p = int(rng.integers(ln + 1, n - ln))
            d = min(int(rng.choice([1, 2, 3, 7, 64, 1000, 60000])), p)
            for k in range(ln):
                b[p + k] = b[p + k - d]
        bufs.append(b)
    levels = [3 + t % 10 for t in range(len(bufs))]
    f, h_in, out_size = _layout(hc_ctx, bufs, [2] * len(bufs), levels)
    h_out = np.zeros(out_size, np.uint8)
    comp, digest, status = hc_ctx.pack_host(h_in, len(h_in), h_out, out_size, f)
    assert (status == 0).all(), status
    frames = [h_out[int(f["dst_off"][i]):int(f["dst_off"][i] + comp[i])].copy() for i in range(len(bufs))]
    for i, (b, fr) in enumerate(zip(bufs, frames)):
        assert int(digest[i]) == oracle.xxh3_port(b)
        rc, got = oracle.lz4f_decode_port(fr, len(b))
        assert rc == 0 and np.array_equal(got[:len(b)], b), (i, len(b))
    _gpu_unpack(hc_ctx, bufs, frames, digest, [2] * len(bufs))


def test_mixed_batch_leaves_the_other_methods_unchanged_and_two_calls_agree(hc_ctx, oracle):
    """Fast LZ4, HC, zstd and stored files in one call: the non-HC frames equal those of the same files packed without
    the HC files; a second call gives the same bytes."""
    n = 48
    sizes = [131072 if i % 5 else 70001 + i for i in range(n)]
    bufs = [corpus.entry_bytes(200 + i, s) for i, s in enumerate(sizes)]
    methods = [(2, 0, 1, 2)[i % 4] for i in range(n)]
    levels = [(1, 0, 3, 9)[i % 4] for i in range(n)]          # i % 4 == 3: LZ4 level 9, the HC files
    frames, comp, digest, status = _pack_device(hc_ctx, bufs, methods, levels)
    assert (status == 0).all(), status
    again = _pack_device(hc_ctx, bufs, methods, levels)
    assert np.array_equal(comp, again[1]) and np.array_equal(digest, again[2])
    assert all(np.array_equal(a, b) for a, b in zip(frames, again[0]))
    keep = [i for i in range(n) if i % 4 != 3]
    alone = _pack_device(hc_ctx, [bufs[i] for i in keep], [methods[i] for i in keep], [levels[i] for i in keep])
    for k, i in enumerate(keep):
        assert np.array_equal(frames[i], alone[0][k]), i
    for i in range(3, n, 4):
        rc, got = oracle.lz4f_decode_port(frames[i], len(bufs[i]))
        assert rc == 0 and np.array_equal(got, bufs[i]), i
    _gpu_unpack(hc_ctx, bufs, frames, digest, methods)


def test_pipelined_pack_host_matches_the_device_path(oracle, monkeypatch):
    """The worker sub-contexts of zpb_pack_host get the caller's switch: tiny chunks over three workers, HC files among
    fast / zstd / stored ones, equal to the single-launch device path."""
    import torch
    import zpack_b200
    monkeypatch.setenv("ZPB_HOST_CHUNK_MB", "1")
    monkeypatch.setenv("ZPB_HOST_WORKERS", "3")
    monkeypatch.delenv("ZPB_LZ4HC", raising=False)
    ctx = zpack_b200.Context(0)
    try:
        ctx.set_lz4hc(True)
        n = 60
        sizes = [0 if i == 11 else (131072 if i % 3 else 50001 + i) for i in range(n)]
        bufs = [corpus.entry_bytes(i, s) for i, s in enumerate(sizes)]
        methods = [0 if i % 7 == 5 else (1 if i % 7 == 3 else 2) for i in range(n)]
        levels = [(9 if i % 2 else 12) if m == 2 and i % 3 != 1 else 0 for i, m in enumerate(methods)]
        f, h_in, out_size = _layout(ctx, bufs, methods, levels)
        h_out = np.zeros(out_size, np.uint8)
        comp, digest, status = ctx.pack_host(h_in, len(h_in), h_out, out_size, f)
        d_in = torch.from_numpy(h_in).cuda()
        d_out = torch.zeros(out_size, dtype=torch.uint8, device="cuda")
        comp_d, digest_d, status_d = ctx.pack_device(d_in, len(h_in), d_out, out_size, f)
        ref = d_out.cpu().numpy()
        assert (status == 0).all() and np.array_equal(status, status_d)
        assert np.array_equal(comp, comp_d) and np.array_equal(digest, digest_d)
        for k in range(n):
            o, c = int(f["dst_off"][k]), int(comp[k])
            assert np.array_equal(h_out[o:o + c], ref[o:o + c]), k
            assert digest[k] == oracle.xxh3_port(bufs[k])
    finally:
        ctx.close()


def test_archive_round_trips_through_the_gpu_and_the_reference_reader(hc_ctx, oracle, tmp_path):
    n, size = 32, 131072
    bufs = [corpus.entry_bytes(300 + i, size) for i in range(n)]
    frames, comp, digest, status = _pack_device(hc_ctx, bufs, [2] * n, [9] * n)
    assert (status == 0).all()
    arch = _gpu_unpack(hc_ctx, bufs, frames, digest, [2] * n)
    if not oracle.have_ref():
        pytest.skip("oracle/_ref not present: GPU reader only")
    rd = oracle.RefReader(arch)
    for i in range(n):
        rc, out = rd.read(i)
        assert rc == 0 and np.array_equal(out, bufs[i]), (i, rc)
    rd.close()
    p = tmp_path / "hc.zpk"
    arch.tofile(p)
    r = subprocess.run([oracle.REF_CLI, "t", str(p)], capture_output=True, text=True)
    assert r.returncode == 0 and f"Corrupted files: 0/{n}" in r.stdout, r.stdout[-300:] + r.stderr


def test_ratio_against_the_gpu_level0_of_the_same_call(hc_ctx):
    """256 x 128 KiB corpus entries at levels 0, 3, 9 and 12 in one call."""
    n, size = 256, 131072
    bufs = [corpus.entry_bytes(i, size) for i in range(n)]
    lv = [0, 3, 9, 12]
    frames, comp, digest, status = _pack_device(hc_ctx, bufs * len(lv), [2] * (n * len(lv)), [l for l in lv for _ in range(n)])
    assert (status == 0).all()
    comp = comp.astype(np.float64).reshape(len(lv), n)
    cls = np.arange(n) % 4
    total = {l: n * size / comp[k].sum() for k, l in enumerate(lv)}
    by_class = {l: [float(comp[0][cls == c].sum() / comp[k][cls == c].sum()) for c in range(4)] for k, l in enumerate(lv)}
    print("\nLZ4 HC on the GPU, ratio by level:", {l: round(v, 3) for l, v in total.items()},
          "gain over level 0 by class (random, text, runs, records):", {l: [round(x, 3) for x in v] for l, v in by_class.items()})
    assert total[9] >= 1.03 * total[0]
    assert by_class[9][1] >= 1.08
    for l in lv[1:]:
        assert min(by_class[l]) >= 1.0, (l, by_class[l])
    assert total[12] >= total[9] >= total[3]


def test_dropin_writes_and_reads_an_lz4_level9_archive(tmp_path):
    """libzpack.so in a process started with ZPB_LZ4HC=1: zpack_write_archive with lz4:9, then zpack_read_file."""
    script = r'''
import ctypes as C, sys
import numpy as np
sys.path[:0] = [sys.argv[1], sys.argv[1] + "/tests"]
import test_host_lib as H
from zpack_b200 import corpus
from oracle import oracle as O
lib = H._lib()
bufs = [corpus.entry_bytes(i, s) for i, s in enumerate([169, 70000, 0, 131072, 262144])]
names = [f"f{i}.bin".encode() for i in range(len(bufs))]
opt = H.Options(2, 9)
w = H.Writer()
assert lib.zpack_init_writer(C.byref(w), sys.argv[2].encode()) == 0
files = (H.ZFile * len(bufs))()
for i, b in enumerate(bufs):
    files[i].filename, files[i].buffer, files[i].size = names[i], b.ctypes.data if len(b) else None, len(b)
    files[i].options = C.pointer(opt)
assert lib.zpack_write_archive(C.byref(w), files, C.c_uint64(len(bufs))) == 0
lib.zpack_close_writer(C.byref(w))
arch = np.fromfile(sys.argv[2], np.uint8)
r = H.Reader()
assert lib.zpack_init_reader_memory_shared(C.byref(r), arch.ctypes.data_as(C.c_void_p), C.c_size_t(len(arch))) == 0
assert r.file_count == len(bufs)
for i, b in enumerate(bufs):
    e = r.file_entries[i]
    assert e.comp_method == 2 and e.uncomp_size == len(b) and e.hash == O.xxh3_port(b)
    out = np.zeros(max(len(b), 1), np.uint8)
    assert lib.zpack_read_file(C.byref(r), C.byref(e), out.ctypes.data_as(C.c_void_p), C.c_size_t(len(b)), None) == 0
    assert np.array_equal(out[:len(b)], b)
lib.zpack_close_reader(C.byref(r))
print("HC-ARCHIVE-OK", len(arch), sum(len(b) for b in bufs))
'''
    env = dict(os.environ, ZPB_LZ4HC="1")
    r = subprocess.run([sys.executable, "-c", script, ROOT, str(tmp_path / "hc9.zpk")], capture_output=True, text=True,
                       timeout=600, env=env)
    assert r.returncode == 0 and "HC-ARCHIVE-OK" in r.stdout, r.stdout[-2000:] + r.stderr[-3000:]
    ok = r.stdout.split()
    assert int(ok[-2]) < int(ok[-1])                      # it compressed
