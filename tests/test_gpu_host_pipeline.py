"""The pipelined host calls (zpb_unpack_host, zpb_pack_host, zpb_unpack_entry_blocks_host) and the group calls over
them: worker sub-contexts run with their caller's settings, the group's pack call leaves null output arrays null, and
both group calls record each device's wall time.  Launch counts (zpb_launch_count) show which kernels the workers ran."""
import numpy as np
import pytest

from zpack_b200 import container, corpus
from zpack_b200 import lib as zlib

pytestmark = pytest.mark.gpu

CHUNK = 1 << 20   # ZPB_HOST_CHUNK_MB=1: several chunks per call, dealt over ZPB_HOST_WORKERS=3


@pytest.fixture
def pipeline_env(monkeypatch):
    monkeypatch.setenv("ZPB_HOST_CHUNK_MB", "1")
    monkeypatch.setenv("ZPB_HOST_WORKERS", "3")
    for v in ("ZPB_OVERLAP", "ZPB_FAST", "ZPB_LZ4HC", "ZPB_PACK_SCRATCH_MB", "ZPB_EXEC_CTAS", "ZPB_EARLY_CTAS"):
        monkeypatch.delenv(v, raising=False)
    return monkeypatch


def _context():
    import zpack_b200
    return zpack_b200.Context(0)


def _launches(ctx, call):
    before = ctx.launch_count
    out = call()
    return ctx.launch_count - before, out


def _lz4_archive(oracle, n, size):
    bufs = [corpus.entry_bytes(i, size) for i in range(n)]
    frames = [oracle.lz4f_encode_port(b, 0, independent=bool(i & 1)) for i, b in enumerate(bufs)]
    hashes = [oracle.xxh3_port(b) for b in bufs]
    arch = container.assemble([corpus.entry_name(i) for i in range(n)], frames, [size] * n, hashes, [2] * n)
    return bufs, hashes, arch


def _files(ctx, bufs, method, level):
    f = np.zeros(len(bufs), zlib.File)
    in_off = out_off = 0
    for i, b in enumerate(bufs):
        cap = ctx.pack_bound(method, len(b))
        f["src_off"][i], f["size"][i], f["dst_off"][i], f["dst_cap"][i] = in_off, len(b), out_off, cap
        f["method"][i], f["level"][i] = method, level
        in_off += (len(b) + 15) & ~15
        out_off += (cap + 15) & ~15
    h_in = np.zeros(in_off + 16, np.uint8)
    for i, b in enumerate(bufs):
        h_in[int(f["src_off"][i]):int(f["src_off"][i]) + len(b)] = b
    return f, h_in, out_off + 16


def _frames(f, h_out, comp):
    return [h_out[int(f["dst_off"][i]):int(f["dst_off"][i] + comp[i])].tobytes() for i in range(len(f))]


def test_unpack_host_workers_follow_the_callers_overlap(pipeline_env, oracle):
    """The execute kernel's late third and its pass over put-aside entries are the two launches the overlap adds, per
    chunk; the workers follow the caller's zpb_set_overlap."""
    n, size = 48, 131072
    bufs, hashes, arch = _lz4_archive(oracle, n, size)
    e = container.parse(arch).entries()
    nchunks = -(-n * size // CHUNK)            # entries of equal size in archive order, cut after every CHUNK bytes
    out_size = int((e["dst_off"] + e["dst_cap"]).max()) + 16
    ctx = _context()
    try:
        outs, launches = [], []
        for overlap in (True, False):
            ctx.set_overlap(overlap)
            out = np.zeros(out_size, np.uint8)
            k, (st, dg) = _launches(ctx, lambda: ctx.unpack_host(arch, len(arch), out, out_size, e))
            assert (st == 0).all() and np.array_equal(dg, np.array(hashes, np.uint64))
            outs.append(out)
            launches.append(k)
        assert launches[0] - launches[1] == 2 * nchunks, launches
        assert np.array_equal(outs[0], outs[1])
        for i, b in enumerate(bufs):
            o = int(e["dst_off"][i])
            assert np.array_equal(outs[1][o:o + size], b), i
    finally:
        ctx.close()


def test_entry_blocks_host_workers_follow_the_callers_overlap(pipeline_env, oracle):
    """The same for the block-sharded host call, whose workers used to keep the settings they were created with."""
    total = 5 << 20
    data = corpus.big_entry(total, piece=1 << 20, first=1)
    frame = oracle.lz4f_encode_port(data, 0, independent=True)
    want = oracle.xxh3_port(data)
    nblocks = -(-total // 65536)
    nchunks = -(-nblocks // (CHUNK // 65536))
    ctx = _context()
    try:
        outs, launches = [], []
        for overlap in (True, False):
            ctx.set_overlap(overlap)
            out = np.zeros(total, np.uint8)
            k, res = _launches(ctx, lambda: ctx.unpack_entry_blocks_host(frame, len(frame), out, total, total, want))
            assert res == (0, want)
            outs.append(out)
            launches.append(k)
        assert launches[0] - launches[1] == 2 * nchunks, launches
        assert np.array_equal(outs[0], data) and np.array_equal(outs[1], data)
    finally:
        ctx.close()


def test_pack_host_workers_keep_the_environment_of_the_callers_creation(pipeline_env, oracle):
    """ZPB_PACK_SCRATCH_MB=1 (16 block slots, at most 4 HC blocks a round) set when the caller's context was created and
    unset before its first pipelined call: the workers pack in as many rounds as when the variable is still set."""
    bufs = [corpus.entry_bytes(i, 131072 if i % 5 else 70001) for i in range(40)]

    def pack(unset_before_call):
        pipeline_env.setenv("ZPB_PACK_SCRATCH_MB", "1")
        ctx = _context()
        try:
            ctx.set_lz4hc(True)
            if unset_before_call:
                pipeline_env.delenv("ZPB_PACK_SCRATCH_MB")
            f, h_in, out_size = _files(ctx, bufs, 2, 9)
            h_out = np.zeros(out_size, np.uint8)
            k, (comp, dg, st) = _launches(ctx, lambda: ctx.pack_host(h_in, len(h_in), h_out, out_size, f))
            assert (st == 0).all()
            return k, _frames(f, h_out, comp), dg
        finally:
            ctx.close()
            pipeline_env.delenv("ZPB_PACK_SCRATCH_MB", raising=False)

    k_set, frames_set, dg_set = pack(False)
    k_unset, frames_unset, dg_unset = pack(True)
    assert k_unset == k_set
    assert frames_unset == frames_set and np.array_equal(dg_unset, dg_set)
    for b, fr, d in zip(bufs, frames_set, dg_set):
        rc, got = oracle.lz4f_decode_port(np.frombuffer(fr, np.uint8), len(b))
        assert rc == 0 and np.array_equal(got[:len(b)], b) and int(d) == oracle.xxh3_port(b)
    ctx = _context()   # the default scratch packs the same batch in fewer rounds: the setting is what the count shows
    try:
        ctx.set_lz4hc(True)
        f, h_in, out_size = _files(ctx, bufs, 2, 9)
        k_default, _ = _launches(ctx, lambda: ctx.pack_host(h_in, len(h_in), np.zeros(out_size, np.uint8), out_size, f))
        assert k_default < k_set
    finally:
        ctx.close()


def _group_pack_raw(g, h_in, h_out, f, comp, digest, status):
    p = lambda a: None if a is None else a.ctypes.data   # noqa: E731
    return g.lib.zpb_group_pack_host(g.h, h_in.ctypes.data, len(h_in), h_out.ctypes.data, len(h_out), f.ctypes.data,
                                     len(f), p(comp), p(digest), p(status))


def test_group_pack_leaves_null_output_arrays_null():
    """digest / status NULL: every device packs its files and returns their sizes; comp_size NULL: refused on every
    device, as zpb_pack_host refuses it."""
    import torch
    import zpack_b200
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two or more GPUs")
    g = zpack_b200.Group(None)
    ctx = _context()
    try:
        bufs = [corpus.entry_bytes(i, 131072) for i in range(24)]
        f, h_in, out_size = _files(ctx, bufs, 2, 0)
        h_ref = np.zeros(out_size, np.uint8)
        comp_ref, _, st_ref = g.pack_host(h_in, len(h_in), h_ref, out_size, f)
        assert (st_ref == 0).all()
        h_out = np.zeros(out_size, np.uint8)
        comp = np.zeros(len(f), np.uint64)
        assert _group_pack_raw(g, h_in, h_out, f, comp, None, None) == 0
        assert np.array_equal(comp, comp_ref) and _frames(f, h_out, comp) == _frames(f, h_ref, comp_ref)
        assert _group_pack_raw(g, h_in, h_out, f, None, None, None) == -3   # ZPB_E_ARG
    finally:
        ctx.close()
        g.close()


def test_group_calls_record_each_devices_time(oracle):
    """last_ms after either call, on a group of one device too, and on every device that had work (each group is fresh
    for its first call, so a time that was not recorded reads 0)."""
    import zpack_b200
    for first in ("pack", "unpack"):
        for devices in ([0], None):
            g = zpack_b200.Group(devices)
            ctx = _context()
            try:
                calls = {"pack": lambda: _group_pack(g, ctx), "unpack": lambda: _group_unpack(g, oracle)}
                for name in (first, "unpack" if first == "pack" else "pack"):
                    calls[name]()
                    assert all(ms > 0 for ms in g.last_ms()), (name, g.last_ms())
            finally:
                ctx.close()
                g.close()


def _group_pack(g, ctx):
    bufs = [corpus.entry_bytes(i, 65536) for i in range(8 * g.size)]
    f, h_in, out_size = _files(ctx, bufs, 2, 0)
    _, _, st = g.pack_host(h_in, len(h_in), np.zeros(out_size, np.uint8), out_size, f)
    assert (st == 0).all()


def _group_unpack(g, oracle):
    _, _, arch = _lz4_archive(oracle, 8 * g.size, 65536)
    e = container.parse(arch).entries()
    out_size = int((e["dst_off"] + e["dst_cap"]).max()) + 16
    st, _ = g.unpack_host(arch, len(arch), np.zeros(out_size, np.uint8), out_size, e)
    assert (st == 0).all()
