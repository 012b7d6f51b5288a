"""Large entries inside batched calls: an LZ4 frame of independent 64 KB blocks or a zstd entry of 64 KB frames of at
least ZPB_ZSTD_FRAMED_MIN bytes is cut into 64 KB pseudo-rows on the device (split_entries.cuh) and decoded
block-parallel inside zpb_unpack_device, zpb_unpack_host, zpb_group_unpack_host and the drop-in's zpack_read_files.
Every byte and digest is compared with the plaintext and oracle.xxh3_port, every decline with the reference reader."""
import ctypes as C
import os

import numpy as np
import pytest

import entropy_data as ED
from test_gpu_lz4hc import _pack_device
from test_split_sim import _zstd_frame
from zpack_b200 import container, corpus
from zpack_b200 import lib as zlib

pytestmark = pytest.mark.gpu

K64 = 65536
T = zlib.ZSTD_FRAMED_MIN
BIG = [T - 1, T, T + 1, (12 << 20) + 777, 64 << 20] + [T + t for t in (1, 63, 64, 1023, 1024, 1025)]


@pytest.fixture(scope="module")
def ctxs():
    import zpack_b200
    os.environ["ZPB_HOST_CHUNK_MB"] = "1"
    try:
        plain, chunked, entropy = zpack_b200.Context(0), zpack_b200.Context(0), zpack_b200.Context(0)
    finally:
        del os.environ["ZPB_HOST_CHUNK_MB"]
    entropy.set_zstd_entropy(True)
    yield {"plain": plain, "chunked": chunked, "entropy": entropy}
    for c in (plain, chunked, entropy):
        c.close()


def _gpu_frames(ctx, bufs, method):
    frames, _, _, status = _pack_device(ctx, bufs, [method] * len(bufs), [1 if method == 2 else 3] * len(bufs))
    assert (status == 0).all()
    return frames


@pytest.fixture(scope="module")
def items(ctxs, oracle):
    """(frame, plaintext, method, is_candidate) of the mixed batch"""
    small = [corpus.entry_bytes(i, 131072) for i in range(32)]
    out = []
    out += [(oracle.lz4f_encode_port(b, 0, independent=k % 2 == 0), b, 2, False) for k, b in enumerate(small[:16])]
    out += [(f, b, 1, False) for f, b in zip(_gpu_frames(ctxs["plain"], small[16:24], 1), small[16:24])]
    out += [(b.copy(), b, 0, False) for b in small[24:]]
    big = [corpus.big_entry(s, piece=(1 << 20) + 333, first=k + 3) for k, s in enumerate(BIG)]
    out += [(f, b, 2, True) for f, b in zip(_gpu_frames(ctxs["plain"], big, 2), big)]
    out += [(f, b, 1, True) for f, b in zip(_gpu_frames(ctxs["plain"], big[:6], 1), big[:6])]
    bf = [ED.class_bytes("bf16", s) for s in (T + 1025, 12 << 20)]
    out += [(f, b, 1, True) for f, b in zip(_gpu_frames(ctxs["entropy"], bf, 1), bf)]
    # reference-shaped large entries: a block-linked LZ4 frame and one zstd frame (kept on today's path)
    lb = corpus.big_entry(T + 4321, piece=1 << 20, first=9)
    out.append((oracle.lz4f_encode_port(lb, 0, independent=False), lb, 2, False))
    zb = corpus.big_entry(T + 999, piece=1 << 20, first=11)
    out.append((_zstd_frame(zb, block=100000), zb, 1, False))          # one frame of raw blocks, 4 MiB window
    if oracle.have_ref():
        out.append((oracle.zstd_compress_ref(zb, 3), zb, 1, False))
    return out


def _archive(items, oracle, seed=0, hashes=None):
    """Archive in item order; the returned rows are shuffled and their output slots are in yet another order, with gaps."""
    n = len(items)
    hashes = hashes or [oracle.xxh3_port(p) for _, p, _, _ in items]
    arch = container.assemble([f"e{i}" for i in range(n)], [f for f, _, _, _ in items], [len(p) for _, p, _, _ in items],
                              hashes, [m for _, _, m, _ in items])
    e = container.parse(arch).entries()
    rng = np.random.default_rng(seed)
    perm = rng.permutation(n)
    e = e[perm]
    off = 0
    for r in rng.permutation(n):
        e["dst_off"][r] = off
        e["dst_cap"][r] = e["uncomp_size"][r] + int(rng.integers(0, 3)) * 16
        off += (int(e["dst_cap"][r]) + 4096 + 15) & ~15
    return arch, e, perm, off


def _check(items, oracle, e, perm, out, status, digest, want_status=None):
    for r, i in enumerate(perm):
        _, p, _, _ = items[i]
        st = 0 if want_status is None else want_status[i]
        assert int(status[r]) == st, (i, len(p), int(status[r]), st)
        if st in (0, 15):
            assert int(digest[r]) == oracle.xxh3_port(p), i
        if st == 0 and out is not None:
            o = int(e["dst_off"][r])
            assert np.array_equal(out[o:o + len(p)], p), (i, len(p))


def _device(ctx, arch, e, out_size):
    import torch
    d_arch = torch.from_numpy(arch).cuda()
    d_out = torch.zeros(out_size + 64, dtype=torch.uint8, device="cuda")
    status, digest = ctx.unpack_device(d_arch, len(arch), d_out, out_size, e)
    return status, digest, d_out.cpu().numpy()


def test_mixed_batch_on_the_device(ctxs, items, oracle):
    ctx = ctxs["plain"]
    assert sum(c for _, _, _, c in items) >= 19
    arch, e, perm, out_size = _archive(items, oracle)
    status, digest, out = _device(ctx, arch, e, out_size)
    _check(items, oracle, e, perm, out, status, digest)


def test_same_batch_through_the_host_calls(ctxs, items, oracle):
    import zpack_b200
    arch, e, perm, out_size = _archive(items, oracle, seed=1)
    for ctx in (ctxs["plain"], ctxs["chunked"]):
        out = np.zeros(out_size + 64, np.uint8)
        status, digest = ctx.unpack_host(arch, len(arch), out, len(out), e)
        _check(items, oracle, e, perm, out, status, digest)
    g = zpack_b200.Group(None)
    try:
        out = np.zeros(out_size + 64, np.uint8)
        status, digest = g.unpack_host(arch, len(arch), out, len(out), e)
        _check(items, oracle, e, perm, out, status, digest)
    finally:
        g.close()
    # ZPB_F_DISCARD: verdicts and digests only; ZPB_F_NO_VERIFY with wrong hashes: OK and the true digest
    d = e.copy()
    d["flags"] |= zlib.F_DISCARD
    out = np.zeros(out_size + 64, np.uint8)
    status, digest = ctxs["chunked"].unpack_host(arch, len(arch), out, len(out), d)
    _check(items, oracle, e, perm, None, status, digest)
    assert not out.any()


def test_wrong_hashes(ctxs, items, oracle):
    hashes = [oracle.xxh3_port(p) ^ (1 if c else 0) for _, p, _, c in items]
    arch, e, perm, out_size = _archive(items, oracle, seed=2, hashes=hashes)
    want = [15 if c else 0 for _, _, _, c in items]
    status, digest, out = _device(ctxs["plain"], arch, e, out_size)
    _check(items, oracle, e, perm, out, status, digest, want)
    nv = e.copy()
    nv["flags"] |= zlib.F_NO_VERIFY
    status, digest, out = _device(ctxs["plain"], arch, nv, out_size)
    _check(items, oracle, e, perm, out, status, digest)


def test_drop_in_batched_read(items, oracle):
    import test_host_lib as H
    lib = H._lib()
    arch, e, perm, out_size = _archive(items, oracle, seed=3)
    r = H.Reader()
    assert lib.zpack_init_reader_memory_shared(C.byref(r), arch.ctypes.data_as(C.c_void_p), C.c_size_t(len(arch))) == 0
    n = int(r.file_count)
    sizes = [int(r.file_entries[i].uncomp_size) for i in range(n)]
    off = np.zeros(n, np.uint64)
    off[1:] = np.cumsum([(s + 4111) & ~15 for s in sizes])[:-1]
    out = np.zeros(int(off[-1]) + sizes[-1] + 64, np.uint8)
    cap = np.array(sizes, np.uint64)
    st = np.full(n, -1, np.int32)
    lib.zpack_read_files.argtypes = [C.c_void_p, C.c_void_p, C.c_uint64, C.c_void_p, C.c_uint64, C.c_void_p, C.c_void_p, C.c_void_p]
    assert lib.zpack_read_files(C.byref(r), r.file_entries, n, out.ctypes.data, len(out), off.ctypes.data,
                                cap.ctypes.data, st.ctypes.data) == 0
    assert (st == 0).all()
    for i in range(n):
        assert np.array_equal(out[int(off[i]):int(off[i]) + sizes[i]], items[i][1]), i
    lib.zpack_close_reader(C.byref(r))


def test_declines_match_the_reference(ctxs, items, oracle):
    import zpack_b200
    """Damaged candidates in a batch with good entries: each status is the one the whole-entry decoders give (a context
    with the fast path off never splits), which for bit flips and truncation is the reference's zpack_read_file (its
    restatement in the oracle, the unmodified reference too where it is built); the other entries are unaffected."""
    bad = list(items)
    cands = [i for i, it in enumerate(items) if it[3]]
    rng = np.random.default_rng(5)
    for k, i in enumerate(cands[:8]):
        f, p, m, c = bad[i]
        f = f.copy()
        if k % 4 == 0:
            f[len(f) // 2 + int(rng.integers(0, 1000))] ^= 0x5A            # bit flips inside a payload
        elif k % 4 == 1:
            f = f[:-777]                                                    # truncation
        elif k % 4 == 2:
            f = np.concatenate([f, np.zeros(9, np.uint8)])                  # trailing bytes
        else:
            f[len(f) // 3] ^= 0x80
        bad[i] = (f, p, m, c)
    hashes = [oracle.xxh3_port(p) for _, p, _, _ in items]
    arch, e, perm, out_size = _archive(bad, oracle, seed=6, hashes=hashes)
    whole = zpack_b200.Context(0)
    whole.set_fast_path(False)
    try:
        st_whole, dg_whole, _ = _device(whole, arch, e, out_size)
    finally:
        whole.close()
    want = [0] * len(bad)
    for r, i in enumerate(perm):
        want[i] = int(st_whole[r])
    port = [oracle.read_entry_port(m, f, len(p), len(p), h)[0] for (f, p, m, _), h in zip(bad, hashes)]
    for k, i in enumerate(cands[:8]):
        if k % 4 != 2:                                                      # trailing bytes: see the docstring
            assert want[i] == port[i], (i, k)
    if oracle.have_ref():
        rd = oracle.RefReader(arch)
        ref = [rd.read(i)[0] for i in range(len(bad))]
        rd.close()
        assert all(want[i] == ref[i] for k, i in enumerate(cands[:8]) if k % 4 != 2)
    assert sum(w != 0 for w in want) >= 6
    status, digest, out = _device(ctxs["plain"], arch, e, out_size)
    assert (status == st_whole).all() and (digest == dg_whole).all()   # a damaged entry's digest is of what it decoded to
    damaged = set(cands[:8])
    keep = np.array([i not in damaged for i in perm])
    _check(bad, oracle, e[keep], perm[keep], out, status[keep], digest[keep], want)


def test_no_interference_with_the_blocks_path_and_launch_counts(ctxs, items, oracle):
    import torch
    ctx = ctxs["plain"]
    data = corpus.big_entry(12 << 20, piece=1 << 20, first=21)
    frame = _gpu_frames(ctx, [data], 2)[0]
    blocks, bs, _ = zlib.lz4_frame_index(frame)
    d_frame = torch.from_numpy(frame).cuda()
    d_big = torch.zeros(len(data) + 64, dtype=torch.uint8, device="cuda")
    assert ctx.unpack_blocks_device(d_frame, len(frame), d_big, len(data), blocks, bs, len(data)) == 0
    arch, e, perm, out_size = _archive(items, oracle, seed=7)
    status, digest, out = _device(ctx, arch, e, out_size)
    _check(items, oracle, e, perm, out, status, digest)
    _, dg = ctx.blocks_digest(None, 0, len(data), d_big)
    assert dg == oracle.xxh3_port(data)
    # a batch without candidates launches what it launched before large entries were split
    small = [it for it in items if not it[3] and len(it[1]) < T]
    arch, e, perm, out_size = _archive(small, oracle, seed=8)
    before = ctx.launch_count
    status, digest, out = _device(ctx, arch, e, out_size)
    _check(small, oracle, e, perm, out, status, digest)
    n_small = ctx.launch_count - before
    withbig = small + [it for it in items if it[3] and it[2] == 2 and len(it[1]) >= T][:1]
    arch, e, perm, out_size = _archive(withbig, oracle, seed=8)
    before = ctx.launch_count
    status, digest, out = _device(ctx, arch, e, out_size)
    _check(withbig, oracle, e, perm, out, status, digest)
    assert ctx.launch_count - before == n_small + 2                     # the pre-pass and the batched chain


def test_candidate_of_more_than_2_gib(ctxs, oracle):
    import torch
    ctx = ctxs["plain"]
    base = corpus.big_entry(64 << 20, piece=(1 << 20) + 77, first=31)
    frame = oracle.lz4f_encode_port(base, 0, independent=True)
    flg = int(frame[4])
    hs = 7 + (8 if flg & 8 else 0)
    assert not flg & 8
    body = frame[hs:-4]
    reps = 33
    big = np.concatenate([frame[:hs]] + [body] * reps + [frame[-4:]])
    plain = np.tile(base, reps)
    assert len(plain) > 2 << 30
    dg = oracle.xxh3_port(plain)
    arch = container.assemble(["big", "small"], [big, base[:1000]], [len(plain), 1000], [dg, oracle.xxh3_port(base[:1000])],
                              [2, 0])
    e = container.parse(arch).entries()
    del big
    d_arch = torch.from_numpy(arch).cuda()
    out_size = int((e["dst_off"] + e["dst_cap"]).max())
    d_out = torch.zeros(out_size + 64, dtype=torch.uint8, device="cuda")
    status, digest = ctx.unpack_device(d_arch, len(arch), d_out, out_size, e)
    assert list(status) == [0, 0] and int(digest[0]) == dg
    o = int(e["dst_off"][0])
    for k in (0, reps // 2, reps - 1):
        got = d_out[o + k * len(base):o + (k + 1) * len(base)].cpu().numpy()
        assert np.array_equal(got, base), k
