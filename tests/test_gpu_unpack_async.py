"""zpb_unpack_device_async: the unpack of a device-resident batch enqueued on the caller's stream, statuses and digests
left in device memory.  Every result is compared with zpb_unpack_device's for the same batch and with the plaintext and
oracle.xxh3_port; the tests also check that the call returns while its stream is still busy, that queued calls on one
context and on two streams stay correct, and that argument errors enqueue nothing."""
import numpy as np
import pytest

from test_gpu_split_batch import _archive, _gpu_frames
from zpack_b200 import corpus
from zpack_b200 import lib as zlib

pytestmark = pytest.mark.gpu

T = zlib.ZSTD_FRAMED_MIN
SLEEP_CYCLES = 1 << 30          # torch.cuda._sleep: about half a second at B200 clocks, bounded
ST_TOO_SMALL, ST_HASH_MISMATCH = 12, 15


@pytest.fixture(scope="module")
def ctx():
    import zpack_b200
    c = zpack_b200.Context(0)
    yield c
    c.close()


@pytest.fixture(scope="module")
def items(ctx, oracle):
    """(frame, plaintext, method, is_candidate): reference-format LZ4 (linked and independent), GPU-written zstd,
    stored and empty entries, and GPU-written LZ4 and zstd entries of 64 KB blocks / frames around ZPB_ZSTD_FRAMED_MIN"""
    small = [corpus.entry_bytes(i, 131072) for i in range(24)]
    out = [(oracle.lz4f_encode_port(b, 0, independent=k % 2 == 0), b, 2, False) for k, b in enumerate(small[:10])]
    out += [(f, b, 1, False) for f, b in zip(_gpu_frames(ctx, small[10:16], 1), small[10:16])]
    out += [(b.copy(), b, 0, False) for b in small[16:]]
    out += [(np.zeros(0, np.uint8), np.zeros(0, np.uint8), 0, False)] * 2
    big = [corpus.big_entry(s, piece=(1 << 20) + 333, first=k + 3) for k, s in enumerate((T - 1, T, T + 1025, 9 << 20))]
    out += [(f, b, 2, len(b) >= T) for f, b in zip(_gpu_frames(ctx, big, 2), big)]
    out += [(f, b, 1, len(b) >= T) for f, b in zip(_gpu_frames(ctx, big, 1), big)]
    return out


def _batch(items, oracle, seed, wrong=(), tight=()):
    """An archive of `items`, rows shuffled; items in `wrong` carry a wrong hash, items in `tight` a slot 16 bytes short.
    Returns (arch, entries, perm, out_size, want) with want[i] = the status item i must get."""
    hashes = [oracle.xxh3_port(p) ^ (1 if i in wrong else 0) for i, (_, p, _, _) in enumerate(items)]
    arch, e, perm, out_size = _archive(items, oracle, seed=seed, hashes=hashes)
    want = [ST_HASH_MISMATCH if i in wrong else 0 for i in range(len(items))]
    for r, i in enumerate(perm):
        if i in tight and len(items[i][1]) >= 32:
            e["dst_cap"][r] = e["uncomp_size"][r] - 16
            want[i] = ST_TOO_SMALL
    return arch, e, perm, out_size, want


def _check_oracle(items, oracle, e, perm, out, status, digest, want):
    for r, i in enumerate(perm):
        p = items[i][1]
        assert int(status[r]) == want[i], (i, len(p), int(status[r]), want[i])
        if want[i] in (0, ST_HASH_MISMATCH) and len(p):
            assert int(digest[r]) == oracle.xxh3_port(p), i
        if want[i] == 0:
            o = int(e["dst_off"][r])
            assert np.array_equal(out[o:o + len(p)], p), (i, len(p))


class Dev:
    """One batch resident on the device, with its output and result buffers"""

    def __init__(self, arch, e, out_size):
        import torch
        self.arch, self.e, self.out_size = arch, e, out_size
        self.d_arch = torch.from_numpy(arch).cuda()
        self.d_out = torch.zeros(out_size + 64, dtype=torch.uint8, device="cuda")
        self.d_status = torch.full((len(e),), -1, dtype=torch.int32, device="cuda")
        self.d_digest = torch.zeros(len(e), dtype=torch.int64, device="cuda")
        torch.cuda.synchronize()

    def run_async(self, ctx, stream, entries=None):
        ctx.unpack_device_async(self.d_arch, len(self.arch), self.d_out, self.out_size, self.e if entries is None else entries,
                                self.d_status, self.d_digest, stream.cuda_stream)

    def results(self):
        return (self.d_status.cpu().numpy(), self.d_digest.cpu().numpy().view(np.uint64), self.d_out.cpu().numpy())

    def run_sync(self, ctx):
        import torch
        d_out = torch.zeros(self.out_size + 64, dtype=torch.uint8, device="cuda")
        status, digest = ctx.unpack_device(self.d_arch, len(self.arch), d_out, self.out_size, self.e)
        return status, digest, d_out.cpu().numpy()


def _same(perm, items, e, a, b):
    """async and sync results agree: statuses, digests, and the bytes of every entry that decoded"""
    assert (a[0] == b[0]).all() and (a[1] == b[1]).all()
    for r, i in enumerate(perm):
        if int(a[0][r]) == 0:
            o, k = int(e["dst_off"][r]), len(items[i][1])
            assert np.array_equal(a[2][o:o + k], b[2][o:o + k]), i


def test_parity_with_the_sync_call_and_the_oracle(ctx, items, oracle):
    import torch
    cands = [i for i, it in enumerate(items) if it[3]]
    assert len(cands) >= 6
    wrong = {0, 11, 17} | set(cands[::2])
    tight = {3, 12, 18, cands[1]}
    arch, e, perm, out_size, want = _batch(items, oracle, seed=11, wrong=wrong, tight=tight)
    d = Dev(arch, e, out_size)
    sync = d.run_sync(ctx)
    _check_oracle(items, oracle, e, perm, sync[2], sync[0], sync[1], want)
    s = torch.cuda.Stream()
    d.run_async(ctx, s)
    s.synchronize()
    got = d.results()
    _check_oracle(items, oracle, e, perm, got[2], got[0], got[1], want)
    _same(perm, items, e, got, sync)


def test_split_retry_on_the_device(ctx, items, oracle):
    """Large LZ4 and zstd entries damaged in a later 64 KB piece: the device-side retry gives the status and digest
    zpb_unpack_device's host-side retry gives; a batch without candidates launches what the sync call launches."""
    import torch
    bad = list(items)
    cands = [i for i, it in enumerate(items) if it[3]]
    damaged = []
    for k, i in enumerate(cands):
        f, p, m, c = bad[i]
        f = f.copy()
        at = len(f) * 3 // 4 + 17 * k
        if k % 2:
            f[at:at + 64] ^= 0x5A                                           # a run of flipped bytes late in the entry
        else:
            f[at] ^= 0x80
        bad[i] = (f, p, m, c)
        damaged.append(i)
    assert {bad[i][2] for i in damaged} == {1, 2}
    arch, e, perm, out_size, _ = _batch(bad, oracle, seed=12)
    d = Dev(arch, e, out_size)
    sync = d.run_sync(ctx)
    # a piece that did not decode: the entry's final status is a decode failure, not a hash mismatch
    failed = {bad[i][2] for r, i in enumerate(perm) if i in damaged and int(sync[0][r]) not in (0, ST_HASH_MISMATCH)}
    assert failed == {1, 2}
    s = torch.cuda.Stream()
    d.run_async(ctx, s)
    s.synchronize()
    _same(perm, bad, e, d.results(), sync)

    small = [it for it in items if not it[3]]
    arch, e, perm, out_size, want = _batch(small, oracle, seed=13)
    d = Dev(arch, e, out_size)
    before = ctx.launch_count
    d.run_sync(ctx)
    n_sync = ctx.launch_count - before
    before = ctx.launch_count
    d.run_async(ctx, s)
    s.synchronize()
    assert ctx.launch_count - before == n_sync
    got = d.results()
    _check_oracle(small, oracle, e, perm, got[2], got[0], got[1], want)


def test_returns_while_the_stream_is_busy(ctx, items, oracle):
    import torch
    arch, e, perm, out_size, want = _batch(items, oracle, seed=14)
    d = Dev(arch, e, out_size)
    s = torch.cuda.Stream()
    d.run_async(ctx, s)                                                     # sizes the scratch for this batch
    s.synchronize()
    d.d_status.fill_(-1)
    d.d_out.zero_()
    torch.cuda.synchronize()
    with torch.cuda.stream(s):
        torch.cuda._sleep(SLEEP_CYCLES)
    d.run_async(ctx, s)
    busy = not s.query()
    s.synchronize()
    assert busy
    got = d.results()
    _check_oracle(items, oracle, e, perm, got[2], got[0], got[1], want)
    assert ctx.last_kernel_ms()["unpack_ms"] > 0


def test_queued_calls_on_one_stream(ctx, items, oracle):
    import torch
    batches = []
    for k in range(3):
        sub = items[k::2] if k < 2 else items
        arch, e, perm, out_size, want = _batch(sub, oracle, seed=20 + k, wrong={1}, tight={2})
        batches.append((sub, Dev(arch, e, out_size), perm, want))
    s = torch.cuda.Stream()
    for _, d, _, _ in batches:
        table = d.e.copy()
        d.run_async(ctx, s, table)
        table[:] = np.frombuffer(np.random.default_rng(1).bytes(table.nbytes), zlib.Entry)   # reused at once
    s.synchronize()
    for sub, d, perm, want in batches:
        got = d.results()
        _check_oracle(sub, oracle, d.e, perm, got[2], got[0], got[1], want)


def test_two_streams_one_context(ctx, items, oracle):
    import torch
    runs = []
    for k in range(2):
        arch, e, perm, out_size, want = _batch(items, oracle, seed=30 + k)
        runs.append((Dev(arch, e, out_size), perm, want, torch.cuda.Stream()))
    for d, _, _, s in runs:
        d.run_async(ctx, s)
    for d, perm, want, s in runs:
        s.synchronize()
        got = d.results()
        _check_oracle(items, oracle, d.e, perm, got[2], got[0], got[1], want)


def test_argument_errors_enqueue_nothing(ctx, items, oracle):
    import torch
    small = [it for it in items if not it[3]][:8]
    arch, e, perm, out_size, _ = _batch(small, oracle, seed=40)
    d = Dev(arch, e, out_size)
    s = torch.cuda.Stream()
    lib = ctx.lib

    def call(entries, n=None, status=None, digest=None, out_size_=None):
        return lib.zpb_unpack_device_async(ctx.h, d.d_arch.data_ptr(), len(arch), d.d_out.data_ptr(),
                                           out_size if out_size_ is None else out_size_, entries.ctypes.data,
                                           len(entries) if n is None else n,
                                           d.d_status.data_ptr() if status is None else status,
                                           d.d_digest.data_ptr() if digest is None else digest, s.cuda_stream)

    outside = e.copy()
    outside["dst_off"][3] = out_size - 16
    unaligned = e.copy()
    unaligned["dst_off"][2] += 8
    cases = [call(e, status=0), call(e, digest=0), call(outside), call(unaligned), call(e, n=1 << 31),
             call(e, out_size_=int(e["dst_off"].max()))]
    assert cases == [-3] * len(cases)
    assert s.query()
    torch.cuda.synchronize()
    assert (d.d_status.cpu().numpy() == -1).all()
    assert call(e) == 0                                                     # the context is usable afterwards
    s.synchronize()
    assert (d.d_status.cpu().numpy() == 0).all()
