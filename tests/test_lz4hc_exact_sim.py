"""The LZ4 HC block compressor (zpack_b200/csrc/lz4hc_blocks.cuh) on the CPU emulation, byte for byte against the serial
restatement of tests/lz4hc_ref.py, at search depths K = 1 .. 65535 and under two schedules, on inputs aimed at the parts
where a kernel can go wrong and still write a valid block: chain links (hash collisions K and K + 1 links back), the
compare limit and the length carried past it, ties between candidates and between costs, the end of the block.  The
restatement itself is checked first: against a brute-force match search, the cost model's own accounting, the oracle's
decoder and the block-format walk."""
import numpy as np
import pytest

import lz4hc_ref as R
from zpack_b200 import corpus
from test_lz4hc_sim import decode_block, pack_blocks, sim, walk  # noqa: F401  (sim: the fixture)

DEPTHS = [1, 4, 32, 96, 65535]
SCHEDULES = [dict(grid=2, seed=1), dict(grid=3, seed=9, misalign=1)]
INV_MUL = pow(2654435761, -1, 1 << 32)


def _rand(rng, n, alpha=256):
    return rng.integers(0, alpha, n, dtype=np.uint8)


def _with_copy(rng, n, src, dst, length):
    """random bytes with b[dst : dst + length] = b[src : src + length], a match of exactly `length` at dst"""
    b = _rand(rng, n)
    b[dst:dst + length] = b[src:src + length]
    b[dst + length] = b[src + length] ^ 0x5A
    b[dst - 1] = b[src - 1] ^ 0xA5
    return b


def collision_block(K, h=0x2A5, tail=20):
    """A 4-byte word W and `tail` random bytes S, then K 4-aligned words of W's hash but other bytes, then W S again:
    the second W's only match is K + 1 links back, behind K links that all fail the 4-byte compare (the words
    ((h << 18) | r) * inverse of the multiplier all hash to h).  -> (block, position of the second W)"""
    rng = np.random.default_rng(1000 + K)
    words = [(((h << 18) | r) * INV_MUL) & 0xFFFFFFFF for r in range(K + 1)]
    head = b"".join(w.to_bytes(4, "little") for w in words)
    S = bytes(_rand(rng, tail))
    b = head[:4] + S + head[4:] + head[:4] + S + bytes(_rand(rng, 16))
    return np.frombuffer(b, np.uint8), 4 * (K + 1) + tail


def _inputs():
    """name -> block"""
    rng = np.random.default_rng(2024)
    bufs = {f"size{s}": np.frombuffer((b"abcdefghijklm" * 4)[:s], np.uint8) for s in range(13, 41)}
    bufs["size13_run"] = np.zeros(13, np.uint8)
    bufs["size40_run"] = np.full(40, 7, np.uint8)
    bufs["size4095"] = corpus.entry_bytes(61, 4095)                          # text
    bufs["size65535"] = corpus.entry_bytes(57, 65535)                        # text
    far = _rand(rng, 65536)                                                  # size 65536, a repeat at distance 65524
    far[65524:] = far[:12]
    bufs["far65524"] = far
    for i in range(4):                                                        # random, text, runs, records
        bufs[f"class{i}"] = corpus.entry_bytes(40 + i, 16384)
    bufs["zeros"] = np.zeros(20000, np.uint8)
    for k in range(1, 8):
        bufs[f"period{k}"] = np.tile(_rand(rng, k), 3000 // k + 1)[:3000]
    for L in (18, 19, 127, 128, 129, 274):
        bufs[f"len{L}"] = _with_copy(rng, 1500, 100, 900, L)
    eq = _rand(rng, 2000)                                                    # the same 40 bytes at 300 and 900, then at 1500
    eq[900:940] = eq[300:340]
    eq[1500:1540] = eq[300:340]
    eq[340], eq[940], eq[1540] = 1, 2, 3
    bufs["equal_len"] = eq
    adv = _rand(rng, 8192)                                                   # a nearer copy of a later piece:
    r = _rand(rng, 700)
    adv[500:1200] = r
    adv[2000:2699] = r[1:]                                                   # 3000 matches 500 only, 3001 .. match 2000
    adv[3000:3700] = r
    bufs["nearer_piece"] = adv
    for K in (1, 4, 32, 96):
        bufs[f"collide{K}"] = collision_block(K)[0]
    return bufs


INPUTS = _inputs()
_REF = {}


def ref(name, K):
    """ref_block_trace of an input, cached; a walk that K did not cut gives the same result at every larger K"""
    if (name, K) not in _REF:
        for (nm, k), v in list(_REF.items()):
            if nm == name and k < K and not v[-1]:
                _REF[(name, K)] = v
                break
        else:
            _REF[(name, K)] = R.ref_block_trace(INPUTS[name], K)
    return _REF[(name, K)]


def assert_same(name, K, c, payload):
    trace = ref(name, K)
    assert (c, bytes(payload)) == trace[:2], name + ": " + R.explain(INPUTS[name], K, c, payload, trace)


# ---- the reference on its own -------------------------------------------------------------------------------------------

def _brute_records(b):
    """longest match of at most lim bytes at every p <= mflimit over every earlier position, the nearest among equals"""
    n = len(b)
    mflimit, matchlimit = n - 12, n - 5
    pad = np.concatenate([b, np.zeros(R.CMP, np.uint8)])
    win = np.lib.stride_tricks.sliding_window_view(pad, R.CMP)
    out = []
    for p in range(mflimit + 1):
        lim = min(matchlimit - p, R.CMP)
        if p == 0:
            out.append((0, 0))
            continue
        eq = win[:p, :lim] == win[p, :lim]
        run = np.where(eq.all(axis=1), lim, np.argmin(eq, axis=1))
        best = int(run.max())
        if best < 4:
            out.append((0, 0))
        else:
            out.append((best, p - int(np.flatnonzero(run == best)[-1])))
    return out


def test_reference_search_with_unlimited_links_is_the_longest_nearest_match():
    rng = np.random.default_rng(5)
    bufs = [_rand(rng, 13, 2), _rand(rng, 40, 3), _rand(rng, 300, 4), _with_copy(rng, 1000, 50, 500, 200),
            np.tile(_rand(rng, 5), 400)[:2000], _rand(rng, 2000, 16), INPUTS["equal_len"], INPUTS["len129"]]
    for b in bufs:
        rec, cut = R.search(bytes(b), 1 << 30)
        assert not cut
        want = _brute_records(b)
        bad = [p for p in range(len(rec)) if rec[p] != want[p]]
        assert not bad, (len(b), bad[0], rec[bad[0]], want[bad[0]])


def test_reference_payload_size_is_the_cost_model_and_decodes(oracle):
    for name in ["size13", "size40_run", "size4095", "zeros", "period3", "len274", "equal_len", "nearer_piece",
                 "collide4", "class1", "class3", "far65524"]:
        b = INPUTS[name]
        c, payload, rec, cost, dec, _ = ref(name, 32)
        if not c:
            continue
        ext = sum((s[0] - prev_end - 15) // 255 + 1 for s, prev_end in _literal_runs(payload) if s[0] - prev_end >= 15)
        assert c == cost[0] + 1 + ext, (name, c, cost[0], ext)
        walk(np.frombuffer(payload, np.uint8), len(b))
        rc, out = decode_block(oracle, np.frombuffer(payload, np.uint8), len(b))
        assert rc == 0 and np.array_equal(out[:len(b)], b), name


def _literal_runs(payload):
    """(sequence, end of the previous match) of each sequence"""
    end = 0
    for s in R.sequences(payload):
        yield s, end
        end = s[0] + s[1]


def test_reference_frame_decodes_and_has_the_oracles_header(oracle):
    assert R.FRAME_HEADER == bytes(oracle.lz4f_encode_port(np.zeros(0, np.uint8), 0, independent=True)[:7])
    for size, level in ((0, 3), (12, 9), (13, 12), (65537, 5), (140000, 16)):
        b = corpus.entry_bytes(size % 7, size)
        fr = R.ref_frame(b, level)
        rc, out = oracle.lz4f_decode_port(np.frombuffer(fr, np.uint8), len(b))
        assert rc == 0 and np.array_equal(out[:len(b)], b), (size, level)
        assert R.frame_from_blocks(bytes(b), R.frame_blocks(fr)) == fr


def test_the_inputs_reach_the_cases_they_are_for():
    """the carry, its refusal on a changed distance, a tie of two distances, the farthest distance, the collisions"""
    rec = ref("len274", 32)[2]
    assert (128, 800) in rec and rec.count((128, 800)) > 100
    rec = ref("nearer_piece", 32)[2]
    assert any(rec[p][0] == R.CMP and rec[p + 1][0] and rec[p + 1][1] != rec[p][1] for p in range(len(rec) - 1))
    assert ref("equal_len", 65535)[2][1500] == (40, 600)
    assert ref("far65524", 65535)[2][65524] == (7, 65524)
    for K in (1, 4, 32, 96):
        b, P = collision_block(K)
        prev = R.chains(bytes(b))
        q, links = P, 0
        while prev[q]:
            q -= prev[q]; links += 1
        assert (q, links) == (0, K + 1), (K, q, links)
        assert ref(f"collide{K}", K)[2][P] == (0, 0)
        assert R.search(bytes(b), K + 1)[0][P][1] == P


# ---- the kernels against the reference ------------------------------------------------------------------------------------

@pytest.mark.parametrize("K", DEPTHS)
def test_sim_equals_the_reference(sim, K):
    names = list(INPUTS)
    bufs = [INPUTS[nm] for nm in names]
    for sched in SCHEDULES:
        for nm, (c, payload) in zip(names, pack_blocks(sim, bufs, links=K, **sched)):
            assert_same(nm, K, c, payload)


def test_sim_finds_the_collision_match_exactly_one_link_further(sim):
    """each collision block at the depth that misses its match and at the one that finds it"""
    for K in (1, 4, 32, 96):
        nm = f"collide{K}"
        for k in (K, K + 1):
            for sched in SCHEDULES:
                [(c, payload)] = pack_blocks(sim, [INPUTS[nm]], links=k, **sched)
                assert_same(nm, k, c, payload)
