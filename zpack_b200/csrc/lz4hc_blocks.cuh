// lz4hc_blocks.cuh — LZ4 HC block compressor (levels 3-12), the alternative stage 1 of the pack path for LZ4 files of
// level >= 3 when the context's HC switch is on (zpb_set_lz4hc / ZPB_LZ4HC).
//
// Same contract as lz4_pack_blocks_kernel (pack_blocks.cuh): one independent block of at most 64 KB in, its payload
// into the block's 64 KB scratch slot, csize[b] = payload bytes or 0 = store the block.  The framing kernel
// (pack_kernel.cuh) cannot tell the two compressors apart, so frames stay B.Indep with 64 KB blocks.
//
// The reference (lz4hc.c) walks hash chains serially, position by position, and parses greedily with lookahead (levels
// 3-9) or optimally (10-12).  Here the work is split into stages that are each parallel, except the parse, which is
// serial per block but runs many blocks at once in a kernel of its own:
//
//   lz4hc_match_kernel, one CTA of HC_THREADS per block (persistent), the block resident in shared memory:
//   (a) CHAINS: prev[p] = distance to the nearest earlier position with the same 14-bit hash of its 4 bytes.  One warp
//       walks the block 32 positions per step: __match_any_sync links the positions of the step among themselves, the
//       first position of each hash group takes the head table's entry, the last one replaces it.
//   (b) SEARCH: one thread per position follows at most K links of its chain (K from the level, hc_links in
//       pack_api.inl) and keeps the longest match, compared up to HC_CMP bytes: (length, distance) -> a per-position
//       record in a global scratch slot (256 KB per block).
//   lz4hc_parse_kernel, one warp per block, nothing in shared memory:
//   (c) PARSE: a backward cost DP, cost[p] = min(cost[p+1] + 1, cost[p+L] + 3 + ext(L)) over L = 4 .. min(T, HC_WIN)
//       and L = T, where T is the match length found at p (a length cut at HC_CMP is carried on from p + 1 when that
//       position's match has the same distance); then a forward walk emits the chosen sequences (p2_emit_coop).
//   Every lane of the parse warp computes the same DP (records and decisions move 32 at a time, one per lane): the
//   block's decisions depend on nothing but its bytes, so the output is the same whatever the scheduling.
//
// The end-of-block rules are those of the fast compressor: no match starts within the last 12 bytes, the last 5 bytes
// are literals (lz4.c:883-884 / lz4_Block_format.md).  A block whose payload is not smaller than the block is stored.
#pragma once
#include "pack_blocks.cuh"

#define HC_THREADS   512u
#define HC_HASH_LOG  14
#define HC_CMP       128u                                   // longest compare of one candidate (longer: carried on in the parse)
#define HC_WIN       18u                                    // every L <= 18 is tried (token-only lengths), beyond only the full one
#define HC_OFF_HEAD  64u                                    // [0, 64): mbarrier, block index
#define HC_OFF_PREV  (HC_OFF_HEAD + 2u * (1u << HC_HASH_LOG))
#define HC_OFF_DATA  (HC_OFF_PREV + 2u * 65536u)
#define HC_SMEM      (HC_OFF_DATA + 65536u + 32u)            // 229472 B: one CTA per SM
#define HC_REC_WORDS (2u * 65536u)                          // per block in global memory: records, then costs

#define HC_U16(off) (*reinterpret_cast<u16 *>(sm + (off)))

// blocks[k].pad: chain links to follow (K); the records of block k go to hrec + k * HC_REC_WORDS
ZPB_DEVINL void lz4hc_match_body(const u8 *__restrict__ in, const PackBlock *__restrict__ blocks, u32 nblocks, u32 *counter, u32 *hrec) {
    ZPB_DYN_SMEM(hc_smem);
    u8 *sm = reinterpret_cast<u8 *>(hc_smem);
    volatile u32 *ctl = reinterpret_cast<volatile u32 *>(sm);     // [0,1] mbarrier  [4] block
    const u32 lane = threadIdx.x & 31u, warp = threadIdx.x >> 5;
    const u32 bar = smem_window(sm);
    if (threadIdx.x == 0) { mbar_init(bar, 1); mbar_fence_init(); }
    u32 parity = 0;
    for (;;) {
        __syncthreads();
        if (threadIdx.x == 0) ctl[4] = atomicAdd(counter, 1u);
        __syncthreads();
        const u32 k = ctl[4];
        if (k >= nblocks) break;
        const PackBlock pb = blocks[k];
        const u32 n = pb.len;
        if (n < 13u) continue;                                     // all literals: the parse stores it
        const u8 *__restrict__ src = in + pb.src_off;
        const u32 D = HC_OFF_DATA + ((u32)(uintptr_t)src & 15u);  // block byte i is sm[D + i]
        p2_stage_block(sm, D, src, n, bar, HC_THREADS);
        for (u32 i = threadIdx.x; i < (1u << HC_HASH_LOG) / 2; i += HC_THREADS) reinterpret_cast<u32 *>(sm + HC_OFF_HEAD)[i] = 0;
        __syncthreads();
        mbar_wait(bar, parity);
        parity ^= 1u;
        const u32 mflimit = n - 12u, matchlimit = n - 5u;

        // ---- (a) chains: the head table holds position + 1 of the last position of each hash (0: none)
        if (warp == 0) {
            for (u32 base = 0; base <= mflimit; base += 32) {
                const u32 p = base + lane;
                const bool v = p <= mflimit;
                const u32 h = v ? (p2_load32(sm, D + p) * 2654435761u) >> (32 - HC_HASH_LOG) : (1u << HC_HASH_LOG) + lane;
                const u32 grp = __match_any_sync(0xffffffffu, h);
                const u32 below = grp & ((1u << lane) - 1u);
                const u32 ent = HC_OFF_HEAD + 2u * (h & ((1u << HC_HASH_LOG) - 1u));
                u32 q1 = 0;                                         // predecessor + 1
                if (below) q1 = base + (31u - (u32)__clz(below)) + 1u;
                else if (v) q1 = HC_U16(ent);
                __syncwarp();
                if (v && (grp >> lane) == 1u) HC_U16(ent) = (u16)(p + 1u);   // the last position of its group
                if (v) HC_U16(HC_OFF_PREV + 2u * p) = (u16)(q1 ? p + 1u - q1 : 0u);
                __syncwarp();
            }
        }
        __syncthreads();

        // ---- (b) search: the longest match among the first K links, then (length | distance << 16) per position
        const u32 K = pb.pad;
        u32 *rec = hrec + (u64)k * HC_REC_WORDS;
        for (u32 p = threadIdx.x; p <= mflimit; p += HC_THREADS) {
            const u32 lim = matchlimit - p < HC_CMP ? matchlimit - p : HC_CMP;
            const u32 x = p2_load32(sm, D + p);
            u32 best = 0, bd = 0, q = p;
            u32 d = HC_U16(HC_OFF_PREV + 2u * p);
            for (u32 j = 0; d && j < K; ++j) {
                q -= d;
                bool cand = p2_load32(sm, D + q) == x;
                if (cand && best >= 4u) cand = p2_load32(sm, D + q + best - 3u) == p2_load32(sm, D + p + best - 3u);   // can it be longer?
                if (cand) {
                    u32 len = 4;
                    while (len + 4u <= lim) {
                        const u32 y = p2_load32(sm, D + p + len) ^ p2_load32(sm, D + q + len);
                        if (y) { len += (u32)(__ffs(y) - 1) >> 3; break; }
                        len += 4u;
                    }
                    if (len + 4u > lim) while (len < lim && sm[D + p + len] == sm[D + q + len]) ++len;
                    if (len > lim) len = lim;
                    if (len > best) {
                        best = len; bd = p - q;
                        if (best >= lim) break;
                    }
                }
                d = HC_U16(HC_OFF_PREV + 2u * q);
            }
            rec[p] = best >= 4u ? best | (bd << 16) : 0u;
        }
    }
}

__global__ void __launch_bounds__(HC_THREADS, 1)
lz4hc_match_kernel(const u8 *__restrict__ in, const PackBlock *__restrict__ blocks, u32 nblocks, u32 *counter, u32 *hrec) {
    lz4hc_match_body(in, blocks, nblocks, counter, hrec);
}

// One warp per block: the DP over the block's records, then the payload -> scratch + k * 65536, csize[k] (0: store).
ZPB_DEVINL void lz4hc_parse_body(const u8 *__restrict__ in, const PackBlock *__restrict__ blocks, u32 nblocks, u32 *hrec, u8 *scratch,
                                 u32 *csize, u32 k) {
    const u32 lane = threadIdx.x & 31u;
    if (k >= nblocks) return;
    const PackBlock pb = blocks[k];
    const u32 n = pb.len;
    if (n < 13u) {                                                 // lz4.c:883: all literals, one byte more than stored
        if (lane == 0) csize[k] = 0;
        return;
    }
    const u8 *__restrict__ src = in + pb.src_off;
    u32 *rec = hrec + (u64)k * HC_REC_WORDS;
    u32 *cost = rec + 65536u;                                      // bytes from position p to the end of the block
    const u32 mflimit = n - 12u;
    // Every lane runs the same DP and writes the same costs: each lane reads back only what it wrote itself.
    for (u32 p = mflimit + 1u; p < n; ++p) cost[p] = n - p;       // the last 11 bytes: literals
    u32 w[HC_WIN];                                                 // cost[p + 1 .. p + HC_WIN]
#pragma unroll
    for (u32 i = 0; i < HC_WIN; ++i) w[i] = mflimit + 1u + i < n ? n - (mflimit + 1u + i) : 0u;
    u32 tn = 0, dn = 0;                                            // the match at p + 1 (after carrying on)
    u32 fidx = 0xFFFFFFFFu, fval = 0;                              // the last far cost loaded: a run of one distance reuses it
    // positions in chunks of 32, top down: lane l loads the record of position lo + l (one load per chunk, not per step),
    // keeps its decision and writes it back with the chunk
    for (u32 top = mflimit + 1u; top > 0;) {
        const u32 lo = top > 32u ? top - 32u : 0u;
        const u32 rv = lo + lane < top ? rec[lo + lane] : 0u;
        u32 dec = 0;
        for (u32 p = top; p-- > lo;) {
            const u32 r = __shfl_sync(0xffffffffu, rv, (int)(p - lo));
            u32 t = r & 0xFFFFu;
            const u32 d = r >> 16;
            if (t == HC_CMP && d == dn && tn + 1u > t) t = tn + 1u;   // cut at the compare limit: p + 1 continues it
            // (cost << 5 | L) of the literal (L = 0) and of every L = 4 .. min(t, HC_WIN), reduced by a min tree: the
            // cheapest, the shortest among equals
            u32 c[16];
            c[0] = (w[0] + 1u) << 5;
#pragma unroll
            for (u32 l = 4; l <= HC_WIN; ++l) c[l - 3u] = l <= t ? ((w[l - 1u] + 3u) << 5) | l : 0xFFFFFFFFu;
#pragma unroll
            for (u32 h = 8; h; h >>= 1)
#pragma unroll
                for (u32 i = 0; i < h; ++i) c[i] = min(c[i], c[i + h]);
            u32 best = c[0] >> 5, L = c[0] & 31u;
            if (t > HC_WIN) {
                if (p + t != fidx) { fidx = p + t; fval = cost[fidx]; }
                const u32 c = fval + 3u + (t - 19u) / 255u + 1u;
                if (c <= best) { best = c; L = t; }
            }
            cost[p] = best;
            if (lane == p - lo) dec = L ? L | (d << 16) : 0u;
#pragma unroll
            for (u32 i = HC_WIN - 1u; i > 0; --i) w[i] = w[i - 1u];
            w[0] = best;
            tn = t; dn = d;
        }
        if (lo + lane < top) rec[lo + lane] = dec;
        top = lo;
    }
    __syncwarp();
    // ---- forward: the chosen sequences, each checked against the room left (compressed only if smaller).  The decisions
    // of 32 positions are loaded at once; literals are skipped by a ballot.
    u8 *dst = scratch + ((u64)k << 16);
    const u32 cap = n - 1u;
    u32 p = 0, anchor = 0, op = 0, base = 0xFFFFFFFFu, v = 0;
    bool fits = true;
    while (p <= mflimit) {
        if ((p & ~31u) != base) { base = p & ~31u; v = base + lane <= mflimit ? rec[base + lane] : 0u; }
        const u32 m = __ballot_sync(0xffffffffu, v != 0u) & (0xFFFFFFFFu << (p - base));
        if (!m) { p = base + 32u; continue; }
        const u32 j = (u32)__ffs(m) - 1u;
        const u32 x = __shfl_sync(0xffffffffu, v, (int)j), L = x & 0xFFFFu;
        p = base + j;
        const u32 lit = p - anchor;
        if (op + p2_seq_bytes(lit, L) > cap) { fits = false; break; }
        op = p2_emit_coop(dst, op, src, anchor, lit, x >> 16, L, lane);
        p += L;
        anchor = p;
    }
    if (fits) {
        const u32 lit = n - anchor;
        if (op + p2_seq_bytes(lit, 0) > cap) fits = false;
        else op = p2_emit_coop(dst, op, src, anchor, lit, 0, 0, lane);
    }
    __syncwarp();
    if (lane == 0) csize[k] = fits ? op : 0u;
}

#define HC_PARSE_WARPS 4u
__global__ void __launch_bounds__(32 * HC_PARSE_WARPS)
lz4hc_parse_kernel(const u8 *__restrict__ in, const PackBlock *__restrict__ blocks, u32 nblocks, u32 *hrec, u8 *scratch, u32 *csize) {
    lz4hc_parse_body(in, blocks, nblocks, hrec, scratch, csize, (blockIdx.x * blockDim.x + threadIdx.x) >> 5);
}
