// pack_blocks.cuh — LZ4 block compressor, stage 1 of the pack path: one CTA of four warps per independent 64 KB block,
// the block resident in shared memory.
//
// Restates the greedy single-probe hash-table matcher of LZ4_compress_generic_validated
// (/root/reference/externals/lz4/lib/lz4.c:851-1240; table of 8192 16-bit positions as for inputs below 64 KB, 4-byte
// minimum match, backward catch-up, the end-of-block rules of lz4.c:883-884 / lz4_Block_format.md), with the serial part
// of the reference — "walk forward, take the first match, skip it" — spread over lanes and warps:
//
//   The block is brought into shared memory by one bulk asynchronous copy (cp.async.bulk + mbarrier): every later read
//   of the input — probing, verifying, extending, copying literals — is a shared-memory access.  It is then processed
//   in windows of P2_WIN = 4096 positions, window w by warp w mod 4:
//   (1a) HASH of every position, 32 per step (no order needed).
//   (1b) PROBE, the only part that has to see the positions in ascending order, as the reference does: hash -> the
//        table's previous position, the table takes the new one.  Windows are probed strictly one after the other: a
//        token in shared memory goes from the warp of window w to the warp of window w + 1.
//   (1c) VERIFY: candidate -> match distance of every position (0 = none), independent loads.  The table cannot hold
//        distances below 32 when a step reads it; the one short distance that matters — 1, inside a byte run — is
//        recognised from the word itself (four equal bytes).
//   (2)  WALK, one lane per 128-byte sub-chunk: the greedy walk (first position with a candidate, extend both ways,
//        emit, skip) runs in all 32 sub-chunks at once; a match stops at its sub-chunk's end.  A lane stages its
//        sequences in shared memory (over the part of the distance array it has already consumed) — except its FIRST
//        one, whose literal run starts in an earlier sub-chunk, and a LAST one that was cut by the sub-chunk's end.
//   (3)  JOIN: the held-back sequences are completed in lane order — a cut match is continued by the next sub-chunk's
//        first match when that starts where it ended with the same offset — and emitted by the whole warp, the staged
//        bytes appended, into the block's scratch slot in HBM.  The window's size is counted first; a second token
//        carries the output position and the start of the pending literal run from window to window and is held for a
//        few instructions only, so the windows of a block are written concurrently.
//   While one warp probes window w, the others hash / verify / walk / join the windows around it.
//
// A block that does not shrink is reported as stored (size 0): the framing stage copies it, as LZ4F_makeBlock does
// (lz4frame.c:750-754).  The compressed bytes are valid LZ4 but not the reference's bytes (every position is probed: no
// skip acceleration — a block whose first 16 KB or more save less than 1/64 is stored instead —, negative levels compress
// like level 0; matches are cut at 128-byte sub-chunk ends unless rejoined, and at window ends);
// the ratio is reported next to the reference's by the tests and the bench.
#pragma once
#include "common.cuh"
#include "ptx.cuh"

#define P2_HASH_LOG 13      // LZ4_HASHLOG + 1: what the reference uses for inputs below 64 KB (lz4.c:739, byU16)
#define P2_WIN      4096u
#define P2_SUB      128u
#define P2_WARPS    4u
#define P2_DIST_N   (P2_WIN + 2u * (P2_WIN / P2_SUB))       // distance array, 2 entries of padding per sub-chunk (banks)
#define P2_LANE_B   (2u * (P2_SUB + 2u))                    // bytes of a lane's part of the distance array = its staging
#define P2_OFF_TABLE 64u                                    // [0, 64): mbarrier, tokens, join state
#define P2_OFF_DIST (P2_OFF_TABLE + 2u * (1u << P2_HASH_LOG) + 16u)       // the table has one spare entry (positions past the last probe)
#define P2_OFF_DATA (P2_OFF_DIST + P2_WARPS * 2u * P2_DIST_N)
#define P2_SMEM     (P2_OFF_DATA + 65536u + 32u)            // 115312 B: two CTAs per SM

struct PackBlock {      // host -> device, one per 64 KB block of an LZ4 file
    u64 src_off;        // where the block's bytes are in the input buffer
    u32 len;            // 1 .. 65536
    u32 pad;            // != 0: the block belongs to a zstd file (zstd_encode.cuh turns its matches into a zstd block)
};

// Shared memory is addressed by byte offsets from the start of the dynamic window (`sm`): 32-bit address arithmetic,
// LDS / STS without generic-pointer conversions.
#define P2_U16(off) (*reinterpret_cast<u16 *>(sm + (off)))
ZPB_DEVINL u32 p2_load32(const u8 *sm, u32 off) {   // unaligned 4-byte load
    const u32 *s = reinterpret_cast<const u32 *>(sm + (off & ~3u));
    return __funnelshift_r(s[0], s[1], (off & 3u) * 8u);
}
// bytes of one sequence in the output (token, length extensions, literals, offset)
ZPB_DEVINL u32 p2_seq_bytes(u32 lit, u32 ml) {
    return 1u + lit + (lit >= 15u ? (lit - 15u) / 255u + 1u : 0u) + (ml ? 2u + (ml - 4u >= 15u ? (ml - 19u) / 255u + 1u : 0u) : 0u);
}
// warp-wide: one sequence at dst (all arguments uniform); literals are block bytes at shared-memory offset `lits`
ZPB_DEVINL u32 p2_emit_coop(u8 *dst, u32 op, const u8 *sm, u32 lits, u32 lit, u32 off, u32 ml, u32 lane) {
    const u32 mlc = ml ? ml - 4u : 0u;
    if (ml && lit < 15u && mlc < 15u) {          // the common short sequence: token, literals, offset
        if (lane == 0) dst[op] = (u8)((lit << 4) | mlc);
        if (lane < lit) dst[op + 1u + lane] = sm[lits + lane];
        if (lane == 31) { dst[op + 1u + lit] = (u8)off; dst[op + 2u + lit] = (u8)(off >> 8); }
        return op + 3u + lit;
    }
    if (lane == 0) dst[op] = (u8)(((lit < 15u ? lit : 15u) << 4) | (mlc < 15u ? mlc : 15u));
    ++op;
    if (lit >= 15u) {
        const u32 r = lit - 15u, n255 = r / 255u;
        for (u32 i = lane; i < n255; i += 32) dst[op + i] = 255;
        if (lane == 0) dst[op + n255] = (u8)(r - n255 * 255u);
        op += n255 + 1u;
    }
    for (u32 i = lane; i < lit; i += 32) dst[op + i] = sm[lits + i];
    op += lit;
    if (ml) {
        if (lane == 0) { dst[op] = (u8)off; dst[op + 1] = (u8)(off >> 8); }
        op += 2u;
        if (mlc >= 15u) {
            const u32 r = mlc - 15u, n255 = r / 255u;
            for (u32 i = lane; i < n255; i += 32) dst[op + i] = 255;
            if (lane == 0) dst[op + n255] = (u8)(r - n255 * 255u);
            op += n255 + 1u;
        }
    }
    return op;
}

// The block into shared memory at window offset D (the caller keeps D congruent to src mod 16): its 16-byte units by one
// bulk copy that thread 0 issues (completion on the mbarrier `bar`), the unaligned ends by ordinary loads of all
// `nthreads` threads.  The caller waits on `bar` after a __syncthreads.
ZPB_DEVINL void p2_stage_block(u8 *sm, u32 D, const u8 *src, u32 n, u32 bar, u32 nthreads) {
    u32 head = (16u - ((u32)(uintptr_t)src & 15u)) & 15u;
    if (head > n) head = n;
    const u32 al = (n - head) & ~15u;
    if (threadIdx.x == 0) {
        mbar_arrive_expect_tx(bar, al);
        for (u32 o = 0; o < al; o += 16384u) bulk_g2s(bar + D + head + o, src + head + o, al - o < 16384u ? al - o : 16384u, bar);
    }
    for (u32 i = threadIdx.x; i < head; i += nthreads) sm[D + i] = src[i];
    for (u32 i = head + al + threadIdx.x; i < n; i += nthreads) sm[D + i] = src[i];
}

// the warp waits until the token is `want` (true) or the block is given up (false).  Every lane polls, lane 0's view
// decides: the warp stays converged and the answer is the same in every lane.
ZPB_DEVINL bool p2_wait(volatile u32 *token, u32 want, volatile u32 *stop) {
    for (;;) {
        const u32 v = __shfl_sync(0xffffffffu, (*token << 1) | (*stop != 0), 0);
        if (v & 1u) return false;
        if ((v >> 1) == want) break;
        spin_pause();
    }
    __threadfence_block();
    return true;
}

// One window's sequences in lane order, at dst + op (WRITE) or only counted (!WRITE): the first literal run starts at
// block position `anchor`.  One sequence is always held back (pv, p_*): the next lane's first match continues it when it
// starts where that one ended with the same offset (a match cut at a sub-chunk end).  Returns the new output position.
template <bool WRITE>
ZPB_DEVINL u32 p2_join(u8 *dst, u32 op, u32 anchor, const u8 *sm, u32 D, u32 dso, u32 lane, bool has, u32 f_pos, u32 f_off,
                       u32 f_len, u32 so, u32 l_pos, u32 l_off, u32 l_len, u32 l_ls, u32 la) {
    bool pv = false;
    u32 p_ls = 0, p_pos = 0, p_off = 0, p_len = 0;
    u32 m = __ballot_sync(0xffffffffu, has);
    while (m) {
        const int k = __ffs(m) - 1;
        m &= m - 1;
        const u32 P = __shfl_sync(0xffffffffu, f_pos, k), O = __shfl_sync(0xffffffffu, f_off, k),
                  L = __shfl_sync(0xffffffffu, f_len, k), SO = __shfl_sync(0xffffffffu, so, k),
                  LL = __shfl_sync(0xffffffffu, l_len, k);
        if (pv && P == anchor && O == p_off) p_len += L;
        else {
            if (pv) op = WRITE ? p2_emit_coop(dst, op, sm, D + p_ls, p_pos - p_ls, p_off, p_len, lane) : op + p2_seq_bytes(p_pos - p_ls, p_len);
            pv = true; p_ls = anchor; p_pos = P; p_off = O; p_len = L;
        }
        anchor = P + L;
        if (SO || LL) {
            op = WRITE ? p2_emit_coop(dst, op, sm, D + p_ls, p_pos - p_ls, p_off, p_len, lane) : op + p2_seq_bytes(p_pos - p_ls, p_len);
            if (WRITE) {
                const u32 sk = dso + (u32)k * P2_LANE_B;
                for (u32 i = lane; i < SO; i += 32) dst[op + i] = sm[sk + i];
            }
            op += SO;
            pv = LL != 0;
            if (pv) {
                p_ls = __shfl_sync(0xffffffffu, l_ls, k); p_pos = __shfl_sync(0xffffffffu, l_pos, k);
                p_off = __shfl_sync(0xffffffffu, l_off, k); p_len = LL;
            }
            anchor = __shfl_sync(0xffffffffu, la, k);
        }
    }
    if (pv) op = WRITE ? p2_emit_coop(dst, op, sm, D + p_ls, p_pos - p_ls, p_off, p_len, lane) : op + p2_seq_bytes(p_pos - p_ls, p_len);
    return op;
}

// Compressed size of every block -> csize[b] (0: store it), payload -> scratch + b * 65536 (at most len - 1 bytes).
// winop (optional, P2_WINOPS entries per block): the payload offset at which each window's sequences start, and behind the
// last window the offset of the closing literals-only sequence — the zstd encoder reads the payload window by window.
#define P2_WINOPS 17u
ZPB_DEVINL void
lz4_pack_blocks_body(const u8 *__restrict__ in, const PackBlock *__restrict__ blocks, u32 nblocks, u32 *counter, u8 *scratch, u32 *csize,
                     u32 *winop) {
    ZPB_DYN_SMEM(p2_smem);
    u8 *sm = reinterpret_cast<u8 *>(p2_smem);
    volatile u32 *ctl = reinterpret_cast<volatile u32 *>(sm);     // [0,1] mbarrier  [2] probe token  [3] join token  [4] block  [5] given up  [8..15] join state
    const u32 lane = threadIdx.x & 31u, warp = threadIdx.x >> 5;
    const u32 tab = P2_OFF_TABLE;                                 // u16 table: last position of each hash
    const u32 dso = P2_OFF_DIST + warp * 2u * P2_DIST_N;          // this warp's window (u16 per position): hash, then candidate, then distance
    const u32 stg = dso + lane * P2_LANE_B;                       // this lane's emitted bytes of the window (over distances it has consumed)
    const u32 bar = smem_window(sm);
    if (threadIdx.x == 0) { mbar_init(bar, 1); mbar_fence_init(); }
    u32 parity = 0;

    for (;;) {
        __syncthreads();                             // the previous block is finished by every warp
        if (threadIdx.x == 0) ctl[4] = atomicAdd(counter, 1u);
        __syncthreads();
        const u32 b = ctl[4];
        if (b >= nblocks) break;
        const PackBlock pb = blocks[b];
        const u8 *__restrict__ src = in + pb.src_off;
        const u32 n = pb.len;
        if (n < 13u) {                               // lz4.c:883: all literals, one byte more than stored
            if (threadIdx.x == 0) csize[b] = 0;
            continue;
        }
        // ---- the block into shared memory, at the same offset mod 16 as in HBM: 16-byte units by one bulk copy
        // (cp.async.bulk, completion on the mbarrier), the unaligned ends by ordinary loads
        const u32 D = P2_OFF_DATA + ((u32)(uintptr_t)src & 15u);  // block byte i is sm[D + i]
        if (threadIdx.x == 0) {
            ctl[2] = 0; ctl[3] = 0; ctl[5] = 0;
            for (u32 i = 8; i < 15; ++i) ctl[i] = 0;
            ctl[15] = 1;                             // fits
        }
        p2_stage_block(sm, D, src, n, bar, 32 * P2_WARPS);
        for (u32 i = threadIdx.x; i < (1u << P2_HASH_LOG) / 2; i += 32 * P2_WARPS) reinterpret_cast<u32 *>(sm + tab)[i] = 0;   // position 0 is a harmless candidate: all are verified
        __syncthreads();
        mbar_wait(bar, parity);
        parity ^= 1u;

        u8 *dst = scratch + (u64)b * 65536u;
        const u32 cap = n - 1u;                      // LZ4F_makeBlock: compressed only if it is smaller (lz4frame.c:747-754)
        const u32 mflimit = n - 12u, matchlimit = n - 5u;
        const u32 nwin = mflimit / P2_WIN + 1u;
        for (u32 w = warp; w < nwin; w += P2_WARPS) {
            const u32 w0 = w * P2_WIN;
            if (__shfl_sync(0xffffffffu, ctl[5], 0)) break;                   // the block was given up (see the join)
            // ---- (1a) hash of every position of the window (no order needed: runs while other warps hold the token);
            // positions past the last probe get the table's spare entry
            for (u32 s = 0; s < P2_WIN; s += 128) {
                const u32 e = dso + 2u * (s + 2u * (s >> 7) + lane);
                u32 wd[4];
#pragma unroll
                for (u32 k = 0; k < 4; ++k) {
                    const u32 p = w0 + s + 32 * k + lane;
                    wd[k] = p2_load32(sm, D + (p <= mflimit ? p : 0u));
                }
#pragma unroll
                for (u32 k = 0; k < 4; ++k) {
                    const u32 p = w0 + s + 32 * k + lane;
                    P2_U16(e + 64 * k) = (u16)(p <= mflimit ? (wd[k] * 2654435761u) >> (32 - P2_HASH_LOG) : 1u << P2_HASH_LOG);
                }
            }
            __syncwarp();
            // ---- (1b) probe, the only part that has to see the positions in order: hash -> the table's previous position,
            // the table takes the new one.  A token goes from window to window.
            if (!p2_wait(ctl + 2, w, ctl + 5)) break;
            for (u32 s = 0; s < P2_WIN; s += 128) {
                const u32 e = dso + 2u * (s + 2u * (s >> 7) + lane);
                u32 h[4], c[4];
#pragma unroll
                for (u32 k = 0; k < 4; ++k) h[k] = tab + 2u * P2_U16(e + 64 * k);
#pragma unroll
                for (u32 k = 0; k < 4; ++k) {
                    c[k] = P2_U16(h[k]);
                    __syncwarp();
                    P2_U16(h[k]) = (u16)(w0 + s + 32 * k + lane);
                    __syncwarp();
                }
#pragma unroll
                for (u32 k = 0; k < 4; ++k) P2_U16(e + 64 * k) = (u16)c[k];
            }
            __syncwarp();
            if (lane == 0) { __threadfence_block(); ctl[2] = w + 1u; }
            // ---- (1c) verify: candidate -> match distance (0 = none).  The four ballots of one round are the "has a match" bits of
            // the 128 positions of ONE sub-chunk: the lane that will walk it keeps them (mk), and skips from match to match
            // with a find-first-set instead of reading distance after distance.
            u32 nmatch = 0;
            u32 mk[4] = {0u, 0u, 0u, 0u};
            for (u32 s = 0; s < P2_WIN; s += 128) {
                const u32 e = dso + 2u * (s + 2u * (s >> 7) + lane);
                u32 c[4], x[4], y[4];
#pragma unroll
                for (u32 k = 0; k < 4; ++k) c[k] = P2_U16(e + 64 * k);
#pragma unroll
                for (u32 k = 0; k < 4; ++k) {
                    const u32 p = w0 + s + 32 * k + lane;
                    x[k] = p2_load32(sm, D + (p <= mflimit ? p : 0u));
                }
#pragma unroll
                for (u32 k = 0; k < 4; ++k) {
                    const u32 p = w0 + s + 32 * k + lane;
                    if (x[k] == __funnelshift_r(x[k], x[k], 8) && p) c[k] = p - 1u;   // four equal bytes: inside a byte run the byte before is the candidate
                    if (p > mflimit) c[k] = 0;
                    y[k] = p2_load32(sm, D + c[k]);
                }
#pragma unroll
                for (u32 k = 0; k < 4; ++k) {
                    const u32 p = w0 + s + 32 * k + lane;
                    const bool hit = x[k] == y[k] && p <= mflimit;            // c < p, or c == p == 0: distance 0 = none
                    const u32 dv = hit ? p - c[k] : 0u;
                    P2_U16(e + 64 * k) = (u16)dv;
                    const u32 bal = __ballot_sync(0xffffffffu, dv != 0u);
                    if (lane == (s >> 7)) mk[k] = bal;
                    nmatch |= bal;
                }
            }
            __syncwarp();
            // ---- (2) walk: every lane its own 128-byte sub-chunk, greedy
            const u32 s0 = w0 + lane * P2_SUB;
            const u32 s1 = s0 + P2_SUB < n ? s0 + P2_SUB : n;
            u32 p = s0, la = s0;                 // position; start of this lane's pending literals
            u32 f_pos = 0, f_off = 0, f_len = 0; // this lane's first sequence (emitted in the join)
            u32 l_pos = 0, l_off = 0, l_len = 0, l_ls = 0;   // its last one, kept back when the sub-chunk end cut it
            u32 so = 0;                          // staged bytes
            bool has = false;
            const u32 mlim = s1 < matchlimit ? s1 : matchlimit;
            const bool any = nmatch != 0;
            // Every loop below has ONE exit, so the 32 lanes — each on its own sub-chunk — come back together after each of
            // them: an iteration of the outer loop costs the longest skip + the longest extension + the longest literal
            // run among the lanes, not their sum.
            bool live = any;
            while (live) {
                // (a) on to the next position that has a match: find-first-set over the sub-chunk's bits
                u32 r = p - s0;
                bool found = false;
                while (!found && r < P2_SUB) {
                    const u32 wsel = r < 64u ? (r < 32u ? mk[0] : mk[1]) : (r < 96u ? mk[2] : mk[3]);
                    const u32 wv = wsel >> (r & 31u);
                    if (wv) { r += (u32)__ffs(wv) - 1u; found = true; }
                    else r = (r | 31u) + 1u;
                }
                p = s0 + r;
                found = found && p + 4u <= mlim;       // a match too close to the end of the sub-chunk (or of the block): nothing behind it can be used either
                const u32 d = found ? P2_U16(stg + 2u * r) : 0u;
                live = found;
                if (live) {
                    // (b) extend forwards, four bytes at a time, then byte-wise up to the limit
                    u32 len = 4;
                    bool go = true, tail = false;
                    while (go) {
                        if (p + len + 4u > mlim) { go = false; tail = true; }
                        else {
                            const u32 x = p2_load32(sm, D + p + len) ^ p2_load32(sm, D + p + len - d);
                            if (x) { len += (u32)(__ffs(x) - 1) >> 3; go = false; }
                            else len += 4u;
                        }
                    }
                    while (tail && p + len < mlim && sm[D + p + len] == sm[D + p + len - d]) ++len;
                    while (p > la && p > d && sm[D + p - 1] == sm[D + p - 1 - d]) { --p; ++len; }   // catch up (lz4.c:1051-1054), within the sub-chunk
                    if (!has) { has = true; f_pos = p; f_off = d; f_len = len; }
                    else if (p + len == s1) { l_pos = p; l_off = d; l_len = len; l_ls = la; }   // may go on in the next sub-chunk
                    else {
                        // staged over this lane's distances: the bytes written stay behind the next index read (a sequence
                        // of lit + len input bytes takes at most lit + 5, and advances the reads by 2 * (lit + len))
                        const u32 lit = p - la, mlc = len - 4u;
                        sm[stg + so++] = (u8)(((lit < 15u ? lit : 15u) << 4) | (mlc < 15u ? mlc : 15u));
                        if (lit >= 15u) sm[stg + so++] = (u8)(lit - 15u);         // lit < 128: one extension byte
                        u32 i = 0;
                        for (; i + 4u <= lit; i += 4u) {                              // four literals per unaligned word load
                            const u32 x = p2_load32(sm, D + la + i);
                            sm[stg + so] = (u8)x; sm[stg + so + 1u] = (u8)(x >> 8); sm[stg + so + 2u] = (u8)(x >> 16); sm[stg + so + 3u] = (u8)(x >> 24);
                            so += 4u;
                        }
                        for (; i < lit; ++i) sm[stg + so++] = sm[D + la + i];
                        sm[stg + so++] = (u8)d; sm[stg + so++] = (u8)(d >> 8);
                        if (mlc >= 15u) sm[stg + so++] = (u8)(mlc - 15u);         // len <= 128: one extension byte
                    }
                    p += len;
                    la = p;
                }
            }
            __syncwarp();
            // ---- (3) join.  What the window emits is counted first (its first literal run taken as empty); the output
            // position and the start of that literal run then come from the window before — a token again, held for a few
            // instructions only — and the warp writes its sequences while the next windows do the same.
            const u32 hm = __ballot_sync(0xffffffffu, has);
            const u32 P0 = __shfl_sync(0xffffffffu, f_pos, hm ? __ffs(hm) - 1 : 0);
            const u32 bytes0 = hm ? p2_join<false>(dst, 0u, P0, sm, D, dso, lane, has, f_pos, f_off, f_len, so, l_pos, l_off, l_len, l_ls, la) : 0u;
            const u32 a_last = __shfl_sync(0xffffffffu, la, hm ? 31 - __clz(hm) : 0);
            if (!p2_wait(ctl + 3, w, ctl + 5)) break;
            const u32 op = ctl[8], anchor = ctl[9];
            const u32 lit0 = P0 - anchor;                                     // the literals in front of the window's first match
            const u32 bytes = hm ? bytes0 + lit0 + (lit0 >= 15u ? (lit0 - 15u) / 255u + 1u : 0u) : 0u;
            const u32 a_out = hm ? a_last : anchor;
            bool fits = op + bytes + 16u <= cap;
            // the reference's answer to incompressible input is its growing search step (lz4.c:634,957); here: a block whose
            // first 16 KB or more saved less than 1/64 so far is stored
            const u32 seen = w0 + P2_WIN;
            if (seen >= 16384u && seen < n && op + bytes + (seen - a_out) + (seen >> 6) > seen) fits = false;
            __syncwarp();
            if (lane == 0) {
                if (!fits) { ctl[5] = 1; ctl[15] = 0; }
                ctl[8] = op + bytes; ctl[9] = a_out;
                if (winop) winop[(u64)b * P2_WINOPS + w] = op;
                __threadfence_block();
                ctl[3] = w + 1u;
            }
            if (!fits) break;
            if (hm) p2_join<true>(dst, op, anchor, sm, D, dso, lane, has, f_pos, f_off, f_len, so, l_pos, l_off, l_len, l_ls, la);
        }
        __syncthreads();
        // ---- the last literals (lz4.c:1224-1240): everything behind the last match
        if (warp == 0) {
            u32 op = ctl[8];
            const u32 anchor = ctl[9];
            bool fits = ctl[15] != 0 && ctl[5] == 0;
            if (winop && lane == 0) winop[(u64)b * P2_WINOPS + nwin] = op;
            if (fits) {
                const u32 lit = n - anchor;
                if (op + p2_seq_bytes(lit, 0) > cap) fits = false;
                else op = p2_emit_coop(dst, op, sm, D + anchor, lit, 0, 0, lane);
            }
            __syncwarp();
            if (lane == 0) csize[b] = fits ? op : 0u;
        }
    }
}

__global__ void __launch_bounds__(32 * P2_WARPS)
lz4_pack_blocks_kernel(const u8 *__restrict__ in, const PackBlock *__restrict__ blocks, u32 nblocks, u32 *counter, u8 *scratch, u32 *csize,
                       u32 *winop) {
    lz4_pack_blocks_body(in, blocks, nblocks, counter, scratch, csize, winop);
}
