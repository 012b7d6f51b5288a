"""A serial restatement of the LZ4 HC block compressor (zpack_b200/csrc/lz4hc_blocks.cuh), position by position, so that
the CPU emulation and the GPU can be held to its exact bytes (tests/test_lz4hc_exact_sim.py, test_gpu_lz4hc_exact.py).
It is written from the compressor's rules, not from its kernels: no warps, no chunking, no caches.

Per block of n <= 65536 bytes, mflimit = n - 12 and matchlimit = n - 5:
  chains  prev[p] = distance to the nearest earlier q <= mflimit with the same 14-bit hash of its 4 bytes (0: none)
  search  at most K links (every link counts, matching or not); a candidate whose 4 bytes equal p's has the length
          min(common prefix, lim), lim = min(matchlimit - p, CMP); only a strictly longer one is kept (the nearest wins
          ties); the walk stops once the best reaches lim; the record is (len, dist) if len >= 4
  parse   cost[p] from mflimit down to 0: a length cut at CMP is carried on from p + 1 when that position's match has the
          same distance; the literal, every L = 4 .. min(t, WIN) (cheapest first, then the literal, then the shortest), and
          the full t > WIN when it costs no more
  emit    the chosen sequences from 0, then the closing literals; a block whose payload exceeds n - 1 bytes is stored"""

CMP = 128                     # HC_CMP: the longest compare of one candidate
WIN = 18                      # HC_WIN: every L <= WIN is a candidate of the parse, beyond it only the full length
HASH_LOG = 14
LINKS = {3: 4, 4: 6, 5: 8, 6: 12, 7: 16, 8: 24, 9: 32, 10: 48, 11: 64, 12: 96}   # hc_links in pack_api.inl
FRAME_HEADER = bytes([0x04, 0x22, 0x4D, 0x18, 0x60, 0x40, 0x82])    # magic, FLG (v01, B.Indep), BD (64 KB), HC
BLOCK = 65536


def links(level: int) -> int:
    """Chain links searched at an LZ4 HC level (levels above 12 act as 12)."""
    return LINKS[min(max(level, 3), 12)]


def hash4(word: int) -> int:
    return ((word * 2654435761) & 0xFFFFFFFF) >> (32 - HASH_LOG)


def chains(b: bytes):
    """prev[p] for p = 0 .. mflimit"""
    mflimit = len(b) - 12
    head, prev = {}, []
    for p in range(mflimit + 1):
        h = hash4(int.from_bytes(b[p:p + 4], "little"))
        prev.append(p - head[h] if h in head else 0)
        head[h] = p
    return prev


def search(b: bytes, K: int, prev=None):
    """-> (records: [(len, dist)] for p = 0 .. mflimit, (0, 0) for none; True if some walk was cut by K, i.e. a larger K
    could give other records)"""
    n = len(b)
    mflimit, matchlimit = n - 12, n - 5
    prev = chains(b) if prev is None else prev
    rec, cut = [], False
    for p in range(mflimit + 1):
        lim = min(matchlimit - p, CMP)
        best = bd = 0
        q, d, j = p, prev[p], 0
        while d:
            if j == K:
                cut = True
                break
            q -= d
            j += 1
            need = max(best + 1, 4)                  # a candidate is kept only if it matches beyond the best so far
            if b[q:q + need] == b[p:p + need]:
                L = need
                while L < lim and b[q + L] == b[p + L]:
                    L += 1
                best, bd = L, p - q
                if best >= lim:
                    break
            d = prev[q]
        rec.append((best, bd) if best >= 4 else (0, 0))
    return rec, cut


def parse(n: int, rec):
    """-> (cost[0 .. n], decisions: [(L, dist)] for p = 0 .. mflimit, (0, 0) for a literal)"""
    mflimit = n - 12
    cost = [0] * (n + 1)
    for p in range(mflimit + 1, n):
        cost[p] = n - p
    dec = [(0, 0)] * (mflimit + 1)
    tn = dn = 0                                      # the match at p + 1, after carrying on
    for p in range(mflimit, -1, -1):
        t, d = rec[p]
        if t == CMP and d == dn and tn + 1 > t:
            t = tn + 1
        best, L = cost[p + 1] + 1, 0
        for l in range(4, min(t, WIN) + 1):
            if cost[p + l] + 3 < best:
                best, L = cost[p + l] + 3, l
        if t > WIN:
            c = cost[p + t] + 3 + (t - 19) // 255 + 1
            if c <= best:
                best, L = c, t
        cost[p] = best
        dec[p] = (L, d) if L else (0, 0)
        tn, dn = t, d
    return cost, dec


def _length(out: bytearray, v: int):
    while v >= 255:
        out.append(255)
        v -= 255
    out.append(v)


def sequence(out: bytearray, lits: bytes, off: int, ml: int):
    """One LZ4 sequence (ml = 0: the closing literals-only one)."""
    lit = len(lits)
    out.append(min(lit, 15) << 4 | (min(ml - 4, 15) if ml else 0))
    if lit >= 15:
        _length(out, lit - 15)
    out += lits
    if ml:
        out += off.to_bytes(2, "little")
        if ml >= 19:
            _length(out, ml - 19)


def emit(b: bytes, dec) -> bytes:
    out = bytearray()
    p = anchor = 0
    while p < len(dec):
        L, d = dec[p]
        if not L:
            p += 1
            continue
        sequence(out, b[anchor:p], d, L)
        p += L
        anchor = p
    sequence(out, b[anchor:], 0, 0)
    return bytes(out)


def ref_block_trace(data, K: int):
    """-> (csize, payload, records, cost, decisions, cut); csize 0 = stored (payload b"")"""
    b = bytes(data)
    n = len(b)
    assert n <= BLOCK
    if n < 13:
        return 0, b"", [], [], [], False
    rec, cut = search(b, K)
    cost, dec = parse(n, rec)
    out = emit(b, dec)
    return (len(out), out, rec, cost, dec, cut) if len(out) <= n - 1 else (0, b"", rec, cost, dec, cut)


def ref_block(data, K: int):
    """-> (csize, payload); csize 0 = the block is stored"""
    return ref_block_trace(data, K)[:2]


def ref_frame(data, level: int) -> bytes:
    """The GPU writer's LZ4 frame of `data` at an HC level: header, then per 64 KB block its payload or the stored block
    (bit 31 of the size set), then the EndMark."""
    K = links(level)
    b = bytes(data)
    return frame_from_blocks(b, [ref_block(b[k:k + BLOCK], K) for k in range(0, len(b), BLOCK)])


def frame_from_blocks(b: bytes, blocks) -> bytes:
    """The frame of `b` from the (csize, payload) of each of its 64 KB blocks."""
    out = bytearray(FRAME_HEADER)
    for k, (c, payload) in enumerate(blocks):
        raw = b[k * BLOCK:(k + 1) * BLOCK]
        if c:
            out += c.to_bytes(4, "little") + payload
        else:
            out += (len(raw) | 0x80000000).to_bytes(4, "little") + raw
    return bytes(out + b"\0\0\0\0")


def sequences(payload: bytes):
    """(position, match length, offset) of each sequence of a block payload, the closing one with length 0"""
    out, p, pos = [], 0, 0
    while True:
        tok = payload[p]
        p += 1
        lit = tok >> 4
        if lit == 15:
            while True:
                lit += payload[p]
                p += 1
                if payload[p - 1] != 255:
                    break
        p += lit
        pos += lit
        if p == len(payload):
            out.append((pos, 0, 0))
            return out
        off = payload[p] | payload[p + 1] << 8
        p += 2
        ml = (tok & 15) + 4
        if tok & 15 == 15:
            while True:
                ml += payload[p]
                p += 1
                if payload[p - 1] != 255:
                    break
        out.append((pos, ml, off))
        pos += ml


def explain(data, K: int, csize: int, payload: bytes, trace=None) -> str:
    """Where a block written by a kernel leaves the reference: the first sequence that differs, and the reference's
    record, cost and decision at that position."""
    rc, rp, rec, cost, dec, _ = trace or ref_block_trace(data, K)
    msg = f"block of {len(data)} bytes, K={K}: csize {csize}, reference {rc}"
    if csize and rc:
        a, b = sequences(bytes(payload)), sequences(rp)
        i = 0
        while i < len(a) and i < len(b) and a[i] == b[i]:
            i += 1
        if i < len(a) and i < len(b):
            p = min(a[i][0], b[i][0])
            at = lambda v: v[p] if p < len(v) else None
            msg += (f"; sequence {i} (position, length, offset): kernel {a[i]}, reference {b[i]}; at {p} the reference has"
                    f" the record {at(rec)}, the cost {at(cost)}, the decision {at(dec)}")
    return msg


def frame_blocks(frame: bytes):
    """The (csize, payload) of each block of a frame that frame_from_blocks lays out (0, b"" for a stored block)."""
    assert frame[:7] == FRAME_HEADER
    p, blocks = 7, []
    while True:
        h = int.from_bytes(frame[p:p + 4], "little")
        p += 4
        if h == 0:
            assert p == len(frame)
            return blocks
        size = h & 0x7FFFFFFF
        blocks.append((0, b"") if h >> 31 else (size, frame[p:p + size]))
        p += size
