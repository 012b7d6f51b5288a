// zstd_decode.cuh — Zstandard frame decoder for one warp per entry (SURVEY.md §8 rows a6-a9).
//
// Replaces the zstd arm of zpack_read_file (/root/reference/lib/zpack_read.c:370-390), i.e.
// ZSTD_decompressDCtx as zstd 1.5.0 runs it:
//   multi-frame loop + skippable frames   externals/zstd/lib/decompress/zstd_decompress.c:907-996
//   frame header                          zstd_decompress.c:419-493
//   block loop                            zstd_decompress.c:819-905, zstd_decompress_block.c:56-70
//   literals section                      zstd_decompress_block.c:79-235
//   Huffman weights / table / decode      common/entropy_common.c:264-329, huf_decompress.c:147-441
//   FSE table description / table build   common/entropy_common.c:64-210, zstd_decompress_block.c:368-485
//   sequence header / decode / execute    zstd_decompress_block.c:577-654, 937-1039, 804-893, 1090-1210
//
// Work split inside the warp (everything an entry needs lives in ~15 KB of shared memory per warp):
//   * entropy tables: table descriptions are short serial bit streams -> lane 0 reads them and lays the
//     FSE cells out; the 2^tableLog Huffman cells are filled by all lanes.
//   * Huffman literals: the format's four independent backward streams are decoded by lanes 0-3, five
//     symbols per 64-bit window refill (aligned 4-byte loads + funnel shifts, never an unaligned load),
//     into a per-warp 128 KB literal buffer in HBM/L2.
//   * sequences: the three interleaved FSE states are one dependency chain -> lane 0 decodes 32
//     sequences at a time into shared memory, resolving repeat offsets and validating sizes as it goes,
//     and classifies each one; then all 32 lanes execute the batch: short literal runs and short
//     matches whose source lies entirely before the batch are copied one-sequence-per-lane, long or
//     dependent ones cooperatively, in order, with the overlap rule of ZSTD_execSequence (a match with
//     offset < length is periodic in `offset`).
//   * the entry digest trails the output front (Xxh3Stream::advance), as in the LZ4 decoders.
//
// Untrusted input: every read is bounded by the entry's compressed range, every write by dst_cap, and
// every table index by the table's size.  A backward bit stream that is read past its beginning is an
// error at once (the library decodes zeros and fails later; the observable class — DECOMPRESS_FAILED —
// is the same; DESIGN.md §2 records the difference).
//
// The file compiles in two modes: CUDA (ZWarp = 32 lanes) and, with -DZPB_HOST_SIM, plain C++ with a
// 1-lane "warp" so that tests/ can run exactly this control logic on a CPU-only box.
// The simulation is a test harness, never a product path: the C-ABI only ever launches the kernel.
#pragma once
#ifdef ZPB_HOST_SIM
#include <cstdint>
#include <cstring>
typedef uint8_t u8;
typedef uint16_t u16;
typedef uint32_t u32;
typedef uint64_t u64;
#define ZPB_DEVINL static inline
#define ZS_CONST static const
static inline u32 ld8(const u8 *p) { return *p; }
static inline u32 ld16u(const u8 *p) { return (u32)p[0] | ((u32)p[1] << 8); }
static inline u32 ld32u(const u8 *p) { return ld16u(p) | (ld16u(p + 2) << 16); }
static inline u64 ld64u(const u8 *p) { return (u64)ld32u(p) | ((u64)ld32u(p + 4) << 32); }
static inline u32 zs_funnel_r(u32 lo, u32 hi, u32 sh) { return (u32)((((u64)hi << 32) | lo) >> (sh & 31)); }
static inline int zs_highbit(u32 v) { return 31 - __builtin_clz(v); }
struct ZWarp {
    static constexpr int W = 1;
    int l = 0;
    void sync() const {}
    template <typename T> T bcast(T v, int) const { return v; }
};
#define ZS_TICK(w, k) do { } while (0)
#else
#include "common.cuh"
#include "xxh3.cuh"
#define ZS_CONST __device__ __constant__
ZPB_DEVINL u32 zs_funnel_r(u32 lo, u32 hi, u32 sh) { return __funnelshift_r(lo, hi, sh); }
ZPB_DEVINL int zs_highbit(u32 v) { return 31 - __clz(v); }
#ifdef ZPB_ZS_PROFILE
// developer build only (tools/zs_profile.sh): cycles per phase, summed over warps (lane 0's clock)
__device__ unsigned long long g_zs_prof[8];
#define ZS_TICK(w, k)                                                                        \
    do {                                                                                     \
        long long now_ = clock64();                                                          \
        if ((w).l == 0) atomicAdd(&g_zs_prof[k], (unsigned long long)(now_ - (w).t_last));   \
        (w).t_last = now_;                                                                   \
    } while (0)
#else
#define ZS_TICK(w, k) do { } while (0)
#endif
struct ZWarp {
    static constexpr int W = 32;
    int l;
    Group<32> g;
#ifdef ZPB_ZS_PROFILE
    mutable long long t_last = 0;
#endif
    ZPB_DEVINL ZWarp() : l(threadIdx.x & 31) {}
    ZPB_DEVINL void sync() const { __syncwarp(); }
    template <typename T> ZPB_DEVINL T bcast(T v, int src) const { return __shfl_sync(0xffffffffu, v, src); }
};
#endif

#define ZS_BLOCK_MAX 131072u
#define ZS_MAGIC 0xFD2FB528u
#define ZS_MAGIC_SKIP 0x184D2A50u
#define ZS_LL 0u
#define ZS_OF 512u
#define ZS_ML 768u
#define ZS_BATCH 32u
#define ZS_LIT_SHORT 16u   // literal runs up to this long are copied by the sequence's own lane
#define ZS_MATCH_SHORT 64u // matches up to this long, source wholly before the batch: own lane
#define ZS_ERR (-1)
#define ZS_LIT_SCRATCH (ZS_BLOCK_MAX + 64u)  // per-warp literal buffer in global memory

// One 4-byte cell per FSE state: next-state base [0,10) | state bits [10,14) | symbol code [14,20) | extra bits [20,25).
// The code's base value comes from the constant tables below (OF: 1 << code).
typedef u32 ZsCell;
#define ZS_CELL(base, nb, code, eb) ((base) | ((nb) << 10) | ((code) << 14) | ((eb) << 20))

// Per-warp decoder state in shared memory.
struct ZstdShared {
    // LL [0,512) | OF [512,768) | ML [768,1280).  One 4-byte cell per state (ZsCell above; the layout idea of
    // ZSTD_seqSymbol, zstd_decompress_block.h, with the base value looked up from the code): 5 KB instead of 10 KB per
    // warp, which is what bounds the number of frames resident on an SM.
    ZsCell fse[1280];
    u32 wfse[64];    // FSE table of the Huffman weights (tableLog <= 6)
    u16 huf[4096];   // sym | nbits << 8, indexed by the next huf_log bits
    u32 seq_ll[ZS_BATCH], seq_ml[ZS_BATCH], seq_off[ZS_BATCH];
    u32 seq_out[ZS_BATCH];  // where the sequence's literals go, relative to the batch's first output byte
    u32 seq_lit[ZS_BATCH];  // where they come from in the literal buffer
    short norm[256];
    u16 next[256];
    u8 wt[256];
    u32 log[3];      // tableLog of LL, OF, ML
    u32 huf_log;
    u32 rep[3];
    u32 huf_valid, seq_valid;
};

ZS_CONST short ZS_LL_DEF[36] = {4, 3, 2, 2, 2, 2, 2, 2, 2, 2, 2, 2, 2, 1, 1, 1, 2, 2,
                                2, 2, 2, 2, 2, 2, 2, 3, 2, 1, 1, 1, 1, 1, -1, -1, -1, -1};
ZS_CONST short ZS_ML_DEF[53] = {1, 4, 3, 2, 2, 2, 2, 2, 2, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1,
                                1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, -1, -1, -1, -1, -1, -1, -1};
ZS_CONST short ZS_OF_DEF[29] = {1, 1, 1, 1, 1, 1, 2, 2, 2, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, -1, -1, -1, -1, -1};
ZS_CONST u32 ZS_LL_BASE[36] = {0, 1, 2, 3, 4, 5, 6, 7, 8, 9, 10, 11, 12, 13, 14, 15, 16, 18, 20, 22, 24, 28, 32, 40,
                               48, 64, 128, 256, 512, 1024, 2048, 4096, 8192, 16384, 32768, 65536};
ZS_CONST u8 ZS_LL_BITS[36] = {0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 1, 1,
                              1, 1, 2, 2, 3, 3, 4, 6, 7, 8, 9, 10, 11, 12, 13, 14, 15, 16};
ZS_CONST u32 ZS_ML_BASE[53] = {3, 4, 5, 6, 7, 8, 9, 10, 11, 12, 13, 14, 15, 16, 17, 18, 19, 20,
                               21, 22, 23, 24, 25, 26, 27, 28, 29, 30, 31, 32, 33, 34, 35, 37, 39, 41,
                               43, 47, 51, 59, 67, 83, 99, 131, 259, 515, 1027, 2051, 4099, 8195, 16387, 32771, 65539};
ZS_CONST u8 ZS_ML_BITS[53] = {0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0,
                              0, 0, 0, 0, 0, 1, 1, 1, 1, 2, 2, 3, 3, 4, 4, 5, 7, 8, 9, 10, 11, 12, 13, 14, 15, 16};

// ------------------------------------------------------------------------------------ bit streams
// forward little-endian bits [pos, pos+n), n <= 25; bits beyond the buffer read as zero
ZPB_DEVINL u32 zs_fwd_bits(const u8 *src, u32 len, u32 pos, u32 n) {
    u32 B = pos >> 3;
    u64 v = 0;
#pragma unroll
    for (u32 k = 0; k < 5; ++k)
        if (B + k < len) v |= (u64)src[B + k] << (8 * k);
    return (u32)(v >> (pos & 7)) & ((1u << n) - 1u);
}

// Backward bit stream (bitstream.h:277-322,425-452): `left` = unread bits below the end marker.
// A 64-bit window holds stream bits [wpos, wpos+64); it is refilled from aligned 32-bit words.
struct ZsRBits {
    const u32 *w;   // the aligned word that holds stream byte 0
    u32 bit0;       // bit offset of stream bit 0 inside w[0]
    u32 last_word;  // index of the last word that holds stream bytes (nothing above it is touched)
    int left;
    u64 win;
    int wpos;
};
ZPB_DEVINL u32 zs_rb_word(const ZsRBits &b, u32 i) {
#ifdef ZPB_HOST_SIM
    return i <= b.last_word ? b.w[i] : 0u;
#else
    return i <= b.last_word ? __ldg(b.w + i) : 0u;  // the archive is read-only for the whole kernel
#endif
}
ZPB_DEVINL void zs_rb_refill(ZsRBits &b) {  // window <- stream bits [left-64, left), zeros below bit 0
    int pos = b.left - 64;
    u32 p = pos < 0 ? 0u : (u32)pos;
    u32 gb = b.bit0 + p, wi = gb >> 5, sh = gb & 31u;
    u32 w0 = zs_rb_word(b, wi), w1 = zs_rb_word(b, wi + 1), w2 = zs_rb_word(b, wi + 2);
    u64 v = ((u64)zs_funnel_r(w1, w2, sh) << 32) | zs_funnel_r(w0, w1, sh);
    if (pos < 0) v = pos <= -64 ? 0ull : v << (u32)(-pos);
    b.win = v;
    b.wpos = pos;
}
ZPB_DEVINL int zs_rb_init(ZsRBits &b, const u8 *src, u32 len) {
    if (len == 0) return ZS_ERR;
    u32 lastb = src[len - 1];
    if (lastb == 0) return ZS_ERR;
    uintptr_t a = (uintptr_t)src;
    b.w = (const u32 *)(a & ~(uintptr_t)3);
    b.bit0 = (u32)(a & 3u) * 8u;
    b.last_word = ((u32)(a & 3u) + len - 1u) >> 2;
    b.left = (int)(len - 1u) * 8 + zs_highbit(lastb);
    b.win = 0;
    b.wpos = b.left;  // empty window: the first read refills
    return 0;
}
ZPB_DEVINL u32 zs_rb_read(ZsRBits &b, u32 n) {  // n <= 32
    if (b.left - b.wpos < (int)n) zs_rb_refill(b);
    b.left -= (int)n;
    return (u32)(b.win >> (u32)(b.left - b.wpos)) & (u32)((1ull << n) - 1ull);
}

// Field of n (<= 32) bits that starts c (< 64) bits below the top of the top-aligned 64-bit value (hi:lo);
// n == 0 gives 0.  All six fields of a sequence are cut from one window with independent shifts.
ZPB_DEVINL u32 zs_field(u32 hi, u32 lo, u32 c, u32 n) {
#ifdef ZPB_HOST_SIM
    u64 v = (((u64)hi << 32) | lo) << c;
    return n ? (u32)(v >> (64 - n)) : 0u;
#else
    u32 top = c < 32 ? __funnelshift_l(lo, hi, c) : lo << (c - 32);  // bits [c, c+32) below the top
    u32 r;
    asm("shr.b32 %0, %1, %2;" : "=r"(r) : "r"(top), "r"(32u - n));   // PTX clamps a shift of 32 to "all out"
    return r;
#endif
}

// ------------------------------------------------------------------------------------ copies
// cooperative forward copy, ranges not overlapping
ZPB_DEVINL void zs_copy(const ZWarp &w, u8 *dst, const u8 *src, u32 n) {
#ifdef ZPB_HOST_SIM
    memcpy(dst, src, n);
#else
    group_copy<32>(w.g, dst, src, n);
#endif
}
ZPB_DEVINL void zs_fill(const ZWarp &w, u8 *dst, u32 v, u64 n) {
    u64 i = 0;
#ifndef ZPB_HOST_SIM
    if (n >= 1024) {
        u32 head = (u32)(-(intptr_t)dst) & 15u;
        for (u32 k = w.l; k < head; k += ZWarp::W) dst[k] = (u8)v;
        u32 v4 = v * 0x01010101u;
        uint4 vv = make_uint4(v4, v4, v4, v4);
        u64 chunks = (n - head) >> 4;
        for (u64 c = w.l; c < chunks; c += ZWarp::W) stg128(dst + head + 16 * c, vv);
        i = head + (chunks << 4);
    }
#endif
    for (u64 k = i + w.l; k < n; k += ZWarp::W) dst[k] = (u8)v;
}
// One lane copies n bytes, ranges not overlapping.  All loads of a 16-byte piece are issued before its
// stores, so a piece costs one memory round trip instead of one per byte.
ZPB_DEVINL void zs_lane_copy(u8 *d, const u8 *s, u32 n) {
    for (u32 base = 0; base < n; base += 16) {
        u32 m = n - base;
        u8 t[16];
#pragma unroll
        for (u32 k = 0; k < 16; ++k) if (k < m) t[k] = s[base + k];
#pragma unroll
        for (u32 k = 0; k < 16; ++k) if (k < m) d[base + k] = t[k];
    }
}
// match copy (ZSTD_execSequence, zstd_decompress_block.c:804-893): source d - off, may overlap
ZPB_DEVINL void zs_match(const ZWarp &w, u8 *d, u32 off, u32 ml) {
    if (off >= ml) {
        zs_copy(w, d, d - off, ml);
    } else if (off == 1) {
        zs_fill(w, d, d[-1], ml);
    } else {  // periodic source: byte i comes from (i mod off) inside the `off` bytes before d
        const u8 *s = d - off;
        u32 r = (u32)w.l % off, step = (u32)ZWarp::W % off;
        for (u32 i = w.l; i < ml; i += ZWarp::W) {
            d[i] = s[r];
            r += step;
            if (r >= off) r -= off;
        }
    }
}

// ------------------------------------------------------------------------------------ FSE
// normalized counts from a table description (entropy_common.c:64-210); serial. Returns bytes used.
ZPB_DEVINL int zs_read_ncount(const u8 *src, u32 len, short *norm, int *max_sym, int *log_out) {
    if (len == 0) return ZS_ERR;
    for (int s = 0; s <= *max_sym; ++s) norm[s] = 0;
    u32 bp = 0;
    int log = (int)zs_fwd_bits(src, len, bp, 4) + 5;
    bp += 4;
    if (log > 15) return ZS_ERR;
    int remaining = (1 << log) + 1, threshold = 1 << log, nbits = log + 1, sym = 0, prev0 = 0;
    while (remaining > 1 && sym <= *max_sym) {
        if (prev0) {
            for (;;) {
                int rep = (int)zs_fwd_bits(src, len, bp, 2);
                bp += 2;
                sym += rep;
                if (rep != 3) break;
                if (bp > 8u * len + 64u) return ZS_ERR;  // ran off the description: only zeros follow
            }
            if (sym > *max_sym) break;
        }
        int max = (2 * threshold - 1) - remaining, count;
        u32 v = zs_fwd_bits(src, len, bp, (u32)nbits);
        if ((int)(v & (u32)(threshold - 1)) < max) {
            count = (int)(v & (u32)(threshold - 1));
            bp += (u32)nbits - 1;
        } else {
            count = (int)(v & (u32)(2 * threshold - 1));
            if (count >= threshold) count -= max;
            bp += (u32)nbits;
        }
        --count;
        remaining -= count < 0 ? -count : count;
        norm[sym++] = (short)count;
        prev0 = !count;
        while (remaining < threshold) { --nbits; threshold >>= 1; }
    }
    if (remaining != 1 || sym > *max_sym + 1) return ZS_ERR;
    u32 used = (bp + 7) >> 3;
    if (used > len) return ZS_ERR;
    for (int s = sym; s <= *max_sym; ++s) norm[s] = 0;
    *max_sym = sym - 1;
    *log_out = log;
    return (int)used;
}

// decode table from normalized counts (zstd_decompress_block.c:368-485); serial
template <typename NormT>
ZPB_DEVINL int zs_fse_build(u32 *cell, u16 *next, const NormT *norm, int max_sym, int log) {
    int size = 1 << log, high = size - 1;
    for (int s = 0; s <= max_sym; ++s) {
        if (norm[s] == -1) { cell[high--] = (u32)s << 16; next[s] = 1; }
        else next[s] = (u16)norm[s];
    }
    int step = (size >> 1) + (size >> 3) + 3, mask = size - 1, pos = 0;
    for (int s = 0; s <= max_sym; ++s)
        for (int i = 0; i < norm[s]; ++i) {
            cell[pos] = (u32)s << 16;
            do pos = (pos + step) & mask; while (pos > high);
        }
    if (pos != 0) return ZS_ERR;
    for (int u = 0; u < size; ++u) {
        u32 s = cell[u] >> 16;
        u32 n = next[s]++;
        u32 nb = (u32)log - (u32)zs_highbit(n);
        cell[u] = (((n << nb) - (u32)size) & 0xFFFFu) | (s << 16) | (nb << 24);
    }
    return 0;
}

// extra bits / base value of a sequence code (which: 0 LL, 1 OF, 2 ML)
ZPB_DEVINL void zs_code_info(u32 which, u32 sym, u32 *eb, u32 *bv) {
    if (which == 0) { *eb = ZS_LL_BITS[sym]; *bv = ZS_LL_BASE[sym]; }
    else if (which == 1) { *eb = sym; *bv = 1u << sym; }
    else { *eb = ZS_ML_BITS[sym]; *bv = ZS_ML_BASE[sym]; }
}

// Sequence decode table from normalized counts; serial.  The symbol spread is staged in the table's own words and
// converted in place.
template <typename NormT>
ZPB_DEVINL int zs_fse_build_seq(ZsCell *cell, u16 *next, const NormT *norm, int max_sym, int log, u32 which) {
    int size = 1 << log, high = size - 1;
    u32 *stage = cell;
    for (int s = 0; s <= max_sym; ++s) {
        if (norm[s] == -1) { stage[high--] = (u32)s; next[s] = 1; }
        else next[s] = (u16)norm[s];
    }
    int step = (size >> 1) + (size >> 3) + 3, mask = size - 1, pos = 0;
    for (int s = 0; s <= max_sym; ++s)
        for (int i = 0; i < norm[s]; ++i) {
            stage[pos] = (u32)s;
            do pos = (pos + step) & mask; while (pos > high);
        }
    if (pos != 0) return ZS_ERR;
    for (int u = 0; u < size; ++u) {
        u32 s = stage[u];
        u32 n = next[s]++;
        u32 nb = (u32)log - (u32)zs_highbit(n);
        u32 eb, bv;
        zs_code_info(which, s, &eb, &bv);
        cell[u] = ZS_CELL(((n << nb) - (u32)size) & 0x3FFu, nb, s, eb);
    }
    return 0;
}

// one of the three sequence tables (zstd_decompress_block.c:529-575); lane 0. Returns bytes used.
ZPB_DEVINL int zs_seq_table(ZstdShared &S, u32 base, u32 which, int mode, const u8 *src, u32 len, int max_sym,
                            int max_log, const short *def, int def_n, int def_log) {
    switch (mode) {
    case 0:
        if (zs_fse_build_seq(S.fse + base, S.next, def, def_n - 1, def_log, which)) return ZS_ERR;
        S.log[which] = (u32)def_log;
        return 0;
    case 1: {
        if (len == 0 || (int)src[0] > max_sym) return ZS_ERR;
        u32 eb, bv;
        zs_code_info(which, src[0], &eb, &bv);
        S.fse[base] = ZS_CELL(0u, 0u, (u32)src[0], eb);
        S.log[which] = 0;
        return 1;
    }
    case 2: {
        int ms = max_sym, log;
        int hs = zs_read_ncount(src, len, S.norm, &ms, &log);
        if (hs < 0 || log > max_log) return ZS_ERR;
        if (zs_fse_build_seq(S.fse + base, S.next, S.norm, ms, log, which)) return ZS_ERR;
        S.log[which] = (u32)log;
        return hs;
    }
    default:
        return S.seq_valid ? 0 : ZS_ERR;
    }
}

// ------------------------------------------------------------------------------------ Huffman
// Tree description (entropy_common.c:264-329) -> S.wt[0..nsym) incl. the implied last weight; lane 0.
// Returns bytes used; *nsym_out gets the symbol count.
ZPB_DEVINL int zs_huf_read_weights(ZstdShared &S, const u8 *src, u32 len, int *nsym_out) {
    if (len == 0) return ZS_ERR;
    int nw;
    u32 used, hb = src[0];
    if (hb >= 128) {
        nw = (int)hb - 127;
        used = 1 + (u32)(nw + 1) / 2;
        if (used > len) return ZS_ERR;
        for (int i = 0; i < nw; ++i) S.wt[i] = (i & 1) ? (src[1 + i / 2] & 15) : (src[1 + i / 2] >> 4);
    } else {
        used = 1 + hb;
        if (used > len) return ZS_ERR;
        int max_sym = 255, log;
        int hs = zs_read_ncount(src + 1, hb, S.norm, &max_sym, &log);
        if (hs < 0 || log > 6) return ZS_ERR;
        if (zs_fse_build(S.wfse, S.next, S.norm, max_sym, log)) return ZS_ERR;
        ZsRBits b;
        if (zs_rb_init(b, src + 1 + hs, hb - (u32)hs)) return ZS_ERR;
        u32 s1 = zs_rb_read(b, (u32)log), s2 = zs_rb_read(b, (u32)log);
        if (b.left < 0) return ZS_ERR;
        nw = 0;
        for (;;) {  // fse_decompress.c tail loop: ends on overflow
            if (nw > 253) return ZS_ERR;
            u32 c = S.wfse[s1];
            S.wt[nw++] = (u8)(c >> 16);
            s1 = (c & 0xFFFFu) + zs_rb_read(b, c >> 24);
            if (b.left < 0) { S.wt[nw++] = (u8)(S.wfse[s2] >> 16); break; }
            if (nw > 253) return ZS_ERR;
            c = S.wfse[s2];
            S.wt[nw++] = (u8)(c >> 16);
            s2 = (c & 0xFFFFu) + zs_rb_read(b, c >> 24);
            if (b.left < 0) { S.wt[nw++] = (u8)(S.wfse[s1] >> 16); break; }
        }
    }
    // weights -> implied last weight, ranks, first cell of every symbol (huf_decompress.c:147-279)
    u32 total = 0;
    for (int i = 0; i < nw; ++i) {
        u32 wv = S.wt[i];
        if (wv > 12) return ZS_ERR;
        if (wv) total += 1u << (wv - 1);
    }
    if (total == 0) return ZS_ERR;
    int log = zs_highbit(total) + 1;
    if (log > 12) return ZS_ERR;
    u32 rest = (1u << log) - total;
    if (rest & (rest - 1)) return ZS_ERR;  // entropy_common.c:307-313
    S.wt[nw] = (u8)(zs_highbit(rest) + 1);
    int nsym = nw + 1;
    u32 rank[16];
    for (int r = 0; r < 16; ++r) rank[r] = 0;
    for (int i = 0; i < nsym; ++i) rank[S.wt[i]]++;
    if (rank[1] < 2 || (rank[1] & 1)) return ZS_ERR;  // entropy_common.c:321
    u32 start[16], acc = 0;
    for (int r = 1; r <= log; ++r) { start[r] = acc; acc += rank[r] << (r - 1); }
    for (int s = 0; s < nsym; ++s) {
        u32 wv = S.wt[s];
        if (!wv) continue;
        S.next[s] = (u16)start[wv];
        start[wv] += 1u << (wv - 1);
    }
    S.huf_log = (u32)log;
    *nsym_out = nsym;
    return (int)used;
}

// all lanes: lay the 2^log cells out from S.wt / S.next
ZPB_DEVINL void zs_huf_fill(const ZWarp &w, ZstdShared &S, int nsym) {
    u32 log = S.huf_log;
    for (int s = 0; s < nsym; ++s) {
        u32 wv = S.wt[s];
        if (!wv) continue;
        u32 n = 1u << (wv - 1), first = S.next[s];
        u16 cell = (u16)((u32)s | ((log + 1 - wv) << 8));
        for (u32 k = w.l; k < n; k += ZWarp::W) S.huf[first + k] = cell;
    }
}

// one backward Huffman stream -> n symbols at dst (huf_decompress.c:350-441 semantics); one lane
ZPB_DEVINL int zs_huf_stream(const ZstdShared &S, const u8 *src, u32 len, u8 *dst, u32 n) {
    ZsRBits b;
    if (zs_rb_init(b, src, len)) return ZS_ERR;
    const u32 log = S.huf_log;
    u32 i = 0;
    while (i < n) {
        zs_rb_refill(b);  // 64 fresh bits: five symbols of <= 12 bits
        u32 used = 0;
#pragma unroll
        for (int k = 0; k < 5; ++k) {
            if (i < n) {
                u32 idx = (u32)((b.win << used) >> (64u - log));
                u32 c = S.huf[idx];
                dst[i++] = (u8)c;
                used += c >> 8;
            }
        }
        b.left -= (int)used;
    }
    return b.left == 0 ? 0 : ZS_ERR;  // BIT_endOfDStream
}

// ------------------------------------------------------------------------------------ literals
// Literals section (zstd_decompress_block.c:79-235).  Returns bytes used; *lit gets a pointer to
// *lit_size literal bytes (inside the compressed block for raw literals, else in `scratch`).
ZPB_DEVINL int zs_literals(const ZWarp &w, ZstdShared &S, const u8 *src, u32 len, u8 *scratch, const u8 **lit,
                           u32 *lit_size) {
    if (len < 3) return ZS_ERR;
    u32 b0 = ld8(src);
    u32 type = b0 & 3, fmt = (b0 >> 2) & 3;
    if (type < 2) {
        u32 lh, ls;
        if (fmt == 0 || fmt == 2) { lh = 1; ls = b0 >> 3; }
        else if (fmt == 1) { lh = 2; ls = ld16u(src) >> 4; }
        else { lh = 3; ls = (ld16u(src) | (ld8(src + 2) << 16)) >> 4; }
        if (type == 0) {
            if (lh + ls > len) return ZS_ERR;
            *lit = src + lh;
            *lit_size = ls;
            return (int)(lh + ls);
        }
        if (fmt == 3 && len < 4) return ZS_ERR;
        if (ls > ZS_BLOCK_MAX) return ZS_ERR;
        zs_fill(w, scratch, ld8(src + lh), ls);
        w.sync();
        *lit = scratch;
        *lit_size = ls;
        return (int)lh + 1;
    }
    if (type == 3 && !S.huf_valid) return ZS_ERR;
    if (len < 5) return ZS_ERR;
    u32 lh, ls, cs;
    bool single = false;
    u32 lhc = ld32u(src);
    if (fmt <= 1) { single = !fmt; lh = 3; ls = (lhc >> 4) & 0x3FFu; cs = (lhc >> 14) & 0x3FFu; }
    else if (fmt == 2) { lh = 4; ls = (lhc >> 4) & 0x3FFFu; cs = lhc >> 18; }
    else { lh = 5; ls = (lhc >> 4) & 0x3FFFFu; cs = (lhc >> 22) + (ld8(src + 4) << 10); }
    if (ls > ZS_BLOCK_MAX || cs + lh > len) return ZS_ERR;
    const u8 *p = src + lh;
    u32 left = cs;
    if (type == 2) {
        int hs = 0, nsym = 0;
        if (w.l == 0) hs = zs_huf_read_weights(S, p, left, &nsym);
        hs = w.bcast(hs, 0);
        nsym = w.bcast(nsym, 0);
        if (hs < 0 || (u32)hs >= left) return ZS_ERR;
        w.sync();
        zs_huf_fill(w, S, nsym);
        if (w.l == 0) S.huf_valid = 1;
        p += hs;
        left -= (u32)hs;
    }
    w.sync();
    int bad = 0;
    if (single) {
        if (w.l == 0) bad = zs_huf_stream(S, p, left, scratch, ls);
    } else {
        if (left < 10) return ZS_ERR;
        u32 s1 = ld16u(p), s2 = ld16u(p + 2), s3 = ld16u(p + 4);
        if (6 + s1 + s2 + s3 > left) return ZS_ERR;
        u32 s4 = left - 6 - s1 - s2 - s3, seg = (ls + 3) / 4;
        if (3 * seg > ls) return ZS_ERR;  // huf_decompress.c:386
        const u8 *q = p + 6;
        for (int k = w.l; k < 4; k += ZWarp::W) {
            const u8 *sp = k == 0 ? q : k == 1 ? q + s1 : k == 2 ? q + s1 + s2 : q + s1 + s2 + s3;
            u32 sl = k == 0 ? s1 : k == 1 ? s2 : k == 2 ? s3 : s4;
            u32 cnt = k == 3 ? ls - 3 * seg : seg;
            if (zs_huf_stream(S, sp, sl, scratch + (u32)k * seg, cnt)) bad = 1;
        }
    }
#ifndef ZPB_HOST_SIM
    bad = __any_sync(0xffffffffu, bad != 0);
#endif
    w.sync();
    if (bad) return ZS_ERR;
    *lit = scratch;
    *lit_size = ls;
    return (int)(lh + cs);
}

// ------------------------------------------------------------------------------------ batch scan
// S.seq_ll/ml/off[0..cnt) -> S.seq_out / S.seq_lit (exclusive prefix sums), bounds checks, and the three
// execution classes.  `room` = output bytes left, `hist` = bytes of this frame already produced.
ZPB_DEVINL int zs_scan_batch(const ZWarp &w, ZstdShared &S, u32 cnt, u32 lit_pos, u32 lit_size, u64 room, u64 hist,
                             u32 *m_long, u32 *m_par, u32 *m_order, u32 *batch_out, u32 *batch_lit) {
#ifdef ZPB_HOST_SIM
    u32 out = 0, lp = 0, ml_ = 0, mp_ = 0, mo_ = 0;
    for (u32 j = 0; j < cnt; ++j) {
        u32 ll = S.seq_ll[j], ml = S.seq_ml[j], off = S.seq_off[j];
        if (ll > lit_size - lit_pos - lp) return ZS_ERR;
        if ((u64)out + ll + ml > room) return ZS_ERR;
        u32 mpos = out + ll;
        if ((u64)off > hist + mpos) return ZS_ERR;
        S.seq_out[j] = out; S.seq_lit[j] = lit_pos + lp;
        if (ll > ZS_LIT_SHORT) ml_ |= 1u << j;
        if (ml <= ZS_MATCH_SHORT && off >= mpos + ml) mp_ |= 1u << j; else mo_ |= 1u << j;
        out = mpos + ml; lp += ll;
    }
    *m_long = ml_; *m_par = mp_; *m_order = mo_; *batch_out = out; *batch_lit = lp;
    return 0;
#else
    const bool live = (u32)w.l < cnt;
    u32 ll = 0, ml = 0, off = 1;
    if (live) { ll = S.seq_ll[w.l]; ml = S.seq_ml[w.l]; off = S.seq_off[w.l]; }
    u32 so = ll + ml, sl = ll;  // inclusive scans; 32 x (131071 + 131074) fits easily
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
        u32 a = __shfl_up_sync(0xffffffffu, so, d), c = __shfl_up_sync(0xffffffffu, sl, d);
        if (w.l >= d) { so += a; sl += c; }
    }
    const u32 out = so - (ll + ml), lp = sl - ll, mpos = out + ll;
    bool bad = live && ((u64)lit_pos + sl > lit_size || (u64)so > room || (u64)off > hist + mpos);
    if (__any_sync(0xffffffffu, bad)) return ZS_ERR;
    const bool par = ml <= ZS_MATCH_SHORT && off >= mpos + ml;
    *m_long = __ballot_sync(0xffffffffu, live && ll > ZS_LIT_SHORT);
    *m_par = __ballot_sync(0xffffffffu, live && par);
    *m_order = __ballot_sync(0xffffffffu, live && !par);
    *batch_out = __shfl_sync(0xffffffffu, so, 31);
    *batch_lit = __shfl_sync(0xffffffffu, sl, 31);
    if (live) { S.seq_out[w.l] = out; S.seq_lit[w.l] = lit_pos + lp; }
    return 0;
#endif
}

// ------------------------------------------------------------------------------------ block
// Compressed block (zstd_decompress_block.c:1456-1525, 1090-1210).  Output goes to dst[op..), bounded by
// cap; matches may reach back to dst[frame_start].  Returns 0 and advances *op_io, or ZS_ERR.
template <class Hasher>
ZPB_DEVINL int zs_block(const ZWarp &w, ZstdShared &S, const u8 *src, u32 len, u8 *dst, u64 frame_start,
                        u64 *op_io, u64 cap, u8 *scratch, Hasher &hs) {
    if (len >= ZS_BLOCK_MAX) return ZS_ERR;
    const u8 *lit = nullptr;
    u32 lit_size = 0;
    ZS_TICK(w, 7);
    int used = zs_literals(w, S, src, len, scratch, &lit, &lit_size);
    ZS_TICK(w, 0);
    if (used < 0) return ZS_ERR;
    src += used;
    len -= (u32)used;
    if (len < 1) return ZS_ERR;
    const u8 *ip = src, *iend = src + len;
    u32 nseq = ld8(ip++);
    u64 op = *op_io;
    u32 lit_pos = 0;
    if (nseq == 0) {
        if (len != 1) return ZS_ERR;
    } else {
        if (nseq > 0x7F) {
            if (nseq == 0xFF) {
                if (ip + 2 > iend) return ZS_ERR;
                nseq = ld16u(ip) + 0x7F00u;
                ip += 2;
            } else {
                if (ip >= iend) return ZS_ERR;
                nseq = ((nseq - 0x80u) << 8) + ld8(ip++);
            }
        }
        if (ip + 1 > iend) return ZS_ERR;
        u32 modes = ld8(ip++);
        // ---- the three tables + bit stream start: lane 0
        int hdr = 0;
        ZsRBits b;
        u32 sl = 0, so = 0, sm = 0;
        if (w.l == 0) {
            const u8 *q = ip;
            int n1 = zs_seq_table(S, ZS_LL, 0, (int)(modes >> 6), q, (u32)(iend - q), 35, 9, ZS_LL_DEF, 36, 6);
            if (n1 >= 0) {
                q += n1;
                int n2 = zs_seq_table(S, ZS_OF, 1, (int)((modes >> 4) & 3), q, (u32)(iend - q), 31, 8, ZS_OF_DEF, 29, 5);
                if (n2 >= 0) {
                    q += n2;
                    int n3 = zs_seq_table(S, ZS_ML, 2, (int)((modes >> 2) & 3), q, (u32)(iend - q), 52, 9, ZS_ML_DEF, 53, 6);
                    if (n3 >= 0) {
                        q += n3;
                        S.seq_valid = 1;
                        if (zs_rb_init(b, q, (u32)(iend - q))) hdr = ZS_ERR;
                        else {
                            sl = zs_rb_read(b, S.log[0]);
                            so = zs_rb_read(b, S.log[1]);
                            sm = zs_rb_read(b, S.log[2]);
                            if (b.left < 0) hdr = ZS_ERR;
                        }
                    } else hdr = ZS_ERR;
                } else hdr = ZS_ERR;
            } else hdr = ZS_ERR;
        }
        hdr = w.bcast(hdr, 0);
        ZS_TICK(w, 1);
        if (hdr < 0) return ZS_ERR;
        // ---- batches of sequences: lane 0 decodes + classifies, the warp executes
        u32 done = 0;
        while (done < nseq) {
            u32 cnt = nseq - done;
            if (cnt > ZS_BATCH) cnt = ZS_BATCH;
            const u64 batch_op = op;
            int err = 0;
            if (w.l == 0) {
                u32 r0 = S.rep[0], r1 = S.rep[1], r2 = S.rep[2];
                for (u32 j = 0; j < cnt; ++j) {
                    const ZsCell cl = S.fse[ZS_LL + sl], co = S.fse[ZS_OF + so], cm = S.fse[ZS_ML + sm];
                    const bool more = done + j + 1 < nseq;
                    // read order (zstd_decompress_block.c:937-1039): OF, ML, LL extra bits, then the LL, ML, OF
                    // state updates (skipped after the last sequence).  All widths are known from the cells,
                    // so the six fields are cut from one 64-bit window at independent offsets.
                    const u32 e_of = co >> 20, e_ml = cm >> 20, e_ll = cl >> 20;
                    const u32 n_ll = more ? (cl >> 10) & 0xFu : 0u, n_ml = more ? (cm >> 10) & 0xFu : 0u,
                              n_of = more ? (co >> 10) & 0xFu : 0u;
                    const u32 v_of = 1u << ((co >> 14) & 0x3Fu), v_ml = ZS_ML_BASE[(cm >> 14) & 0x3Fu],
                              v_ll = ZS_LL_BASE[(cl >> 14) & 0x3Fu];
                    const u32 c1 = e_of, c2 = c1 + e_ml, c3 = c2 + e_ll, c4 = c3 + n_ll, c5 = c4 + n_ml,
                              total = c5 + n_of;
                    u32 ofv, ml, ll;
                    if (total <= 64) {
                        if (b.left - b.wpos < (int)total) zs_rb_refill(b);
                        const u32 avail = (u32)(b.left - b.wpos);        // 1..64 unread bits at the top of the window
                        const u64 v = b.win << (64u - avail);             // top-aligned (avail >= total >= ... > 0 or unused)
                        const u32 hi = (u32)(v >> 32), lo = (u32)v;
                        ofv = v_of + zs_field(hi, lo, 0, e_of);
                        ml = v_ml + zs_field(hi, lo, c1, e_ml);
                        ll = v_ll + zs_field(hi, lo, c2, e_ll);
                        if (more) {
                            sl = (cl & 0x3FFu) + zs_field(hi, lo, c3, n_ll);
                            sm = (cm & 0x3FFu) + zs_field(hi, lo, c4, n_ml);
                            so = (co & 0x3FFu) + zs_field(hi, lo, c5, n_of);
                        }
                        b.left -= (int)total;
                    } else {  // > 64 bits in one sequence (huge offset codes): field by field
                        ofv = v_of + zs_rb_read(b, e_of);
                        ml = v_ml + zs_rb_read(b, e_ml);
                        ll = v_ll + zs_rb_read(b, e_ll);
                        if (more) {
                            sl = (cl & 0x3FFu) + zs_rb_read(b, n_ll);
                            sm = (cm & 0x3FFu) + zs_rb_read(b, n_ml);
                            so = (co & 0x3FFu) + zs_rb_read(b, n_of);
                        }
                    }
                    u32 off;
                    if (ofv > 3) { off = ofv - 3; r2 = r1; r1 = r0; r0 = off; }
                    else {  // repeat offsets (zstd_decompress_block.c:971-987)
                        u32 idx = ofv - 1 + (ll == 0);
                        if (idx == 0) off = r0;
                        else {
                            off = idx == 3 ? r0 - 1 : (idx == 1 ? r1 : r2);
                            if (!off) off = 1;
                            if (idx != 1) r2 = r1;
                            r1 = r0;
                            r0 = off;
                        }
                    }
                    S.seq_ll[j] = ll; S.seq_ml[j] = ml; S.seq_off[j] = off;
                    if (!more) {
                        // the library updates the states once more, then wants every bit consumed (:1195)
                        int tail = (int)(((cl >> 10) & 0xFu) + ((cm >> 10) & 0xFu) + ((co >> 10) & 0xFu));
                        if (b.left > tail) err = 1;
                    }
                }
                if (b.left < 0) err = 1;  // `left` only ever decreases: one check per batch covers every read
                S.rep[0] = r0; S.rep[1] = r1; S.rep[2] = r2;
            }
            err = w.bcast(err, 0);
            ZS_TICK(w, 2);
            if (err) return ZS_ERR;
            w.sync();
            // positions, validation and classification of the whole batch (zstd_decompress_block.c:804-893's
            // checks; any failing sequence fails the entry, so the order of detection does not matter)
            u32 m_long, m_par, m_order, batch_out, batch_lit;
            if (zs_scan_batch(w, S, cnt, lit_pos, lit_size, cap - batch_op, batch_op - frame_start, &m_long, &m_par,
                              &m_order, &batch_out, &batch_lit))
                return ZS_ERR;
            const u64 op_end = batch_op + batch_out;
            const u32 lit_end = lit_pos + batch_lit;
            w.sync();
            u8 *bd = dst + batch_op;
            // phase 1: literal runs — short ones by the sequence's own lane, long ones by the warp
            for (u32 j = w.l; j < cnt; j += ZWarp::W) {
                u32 ll = S.seq_ll[j];
                if (ll <= ZS_LIT_SHORT) zs_lane_copy(bd + S.seq_out[j], lit + S.seq_lit[j], ll);
            }
            for (u32 m = m_long; m; m &= m - 1) {
                u32 j = (u32)zs_highbit(m & (0u - m));
                zs_copy(w, bd + S.seq_out[j], lit + S.seq_lit[j], S.seq_ll[j]);
            }
            ZS_TICK(w, 3);
            // phase 2a: short matches whose source lies wholly before the batch — own lane
            for (u32 j = w.l; j < cnt; j += ZWarp::W) {
                if ((m_par >> j) & 1u) {
                    u8 *d = bd + S.seq_out[j] + S.seq_ll[j];
                    zs_lane_copy(d, d - S.seq_off[j], S.seq_ml[j]);
                }
            }
            ZS_TICK(w, 4);
            // phase 2b: everything else in order, cooperatively
            for (; m_order; m_order &= m_order - 1) {
                u32 j = (u32)zs_highbit(m_order & (0u - m_order));
                w.sync();
                zs_match(w, bd + S.seq_out[j] + S.seq_ll[j], S.seq_off[j], S.seq_ml[j]);
            }
            w.sync();
            op = op_end;
            lit_pos = lit_end;
            done += cnt;
            ZS_TICK(w, 5);
            hs.advance(op, w);
            ZS_TICK(w, 6);
        }
    }
    u32 rest = lit_size - lit_pos;
    if (rest > cap - op) return ZS_ERR;
    zs_copy(w, dst + op, lit + lit_pos, rest);
    op += rest;
    *op_io = op;
    return 0;
}

// XXH64 of the frame content (optional frame checksum; externals/zstd/lib/common/xxhash.c).
// Rare (ZPack's writer never asks for it): evaluated redundantly by every lane.
ZPB_DEVINL u64 zs_rotl64(u64 v, int r) { return (v << r) | (v >> (64 - r)); }
ZPB_DEVINL u64 zs_xxh64(const u8 *p, u64 len) {
    const u64 P1 = 0x9E3779B185EBCA87ull, P2 = 0xC2B2AE3D27D4EB4Full, P3 = 0x165667B19E3779F9ull,
              P4 = 0x85EBCA77C2B2AE63ull, P5 = 0x27D4EB2F165667C5ull;
    const u8 *end = p + len;
    u64 h;
    if (len >= 32) {
        u64 v0 = P1 + P2, v1 = P2, v2 = 0, v3 = 0 - P1;
        do {
            v0 = zs_rotl64(v0 + ld64u(p) * P2, 31) * P1;
            v1 = zs_rotl64(v1 + ld64u(p + 8) * P2, 31) * P1;
            v2 = zs_rotl64(v2 + ld64u(p + 16) * P2, 31) * P1;
            v3 = zs_rotl64(v3 + ld64u(p + 24) * P2, 31) * P1;
            p += 32;
        } while (p + 32 <= end);
        h = zs_rotl64(v0, 1) + zs_rotl64(v1, 7) + zs_rotl64(v2, 12) + zs_rotl64(v3, 18);
        h = (h ^ (zs_rotl64(v0 * P2, 31) * P1)) * P1 + P4;
        h = (h ^ (zs_rotl64(v1 * P2, 31) * P1)) * P1 + P4;
        h = (h ^ (zs_rotl64(v2 * P2, 31) * P1)) * P1 + P4;
        h = (h ^ (zs_rotl64(v3 * P2, 31) * P1)) * P1 + P4;
    } else {
        h = P5;
    }
    h += len;
    for (; p + 8 <= end; p += 8) h = zs_rotl64(h ^ (zs_rotl64(ld64u(p) * P2, 31) * P1), 27) * P1 + P4;
    if (p + 4 <= end) { h = zs_rotl64(h ^ ((u64)ld32u(p) * P1), 23) * P2 + P3; p += 4; }
    for (; p < end; ++p) h = zs_rotl64(h ^ (*p * P5), 11) * P1;
    h ^= h >> 33; h *= P2; h ^= h >> 29; h *= P3; h ^= h >> 32;
    return h;
}

// ------------------------------------------------------------------------------------ entry
// Every frame of one entry (ZSTD_decompressMultiFrame, zstd_decompress.c:907-996).  Returns 0 or ZS_ERR
// (the caller maps any failure to ZPACK_ERROR_DECOMPRESS_FAILED, lib/zpack_read.c:384-388).
template <class Hasher>
ZPB_DEVINL int zstd_decode_entry(const ZWarp &w, ZstdShared &S, u8 *scratch, const u8 *src, u64 n, u8 *dst,
                                 u64 cap, Hasher &hs, u64 *produced) {
    u64 ip = 0, op = 0;
    *produced = 0;
    while (n - ip >= 4) {
        u32 magic = ld32u(src + ip);
        if ((magic & 0xFFFFFFF0u) == ZS_MAGIC_SKIP) {
            if (n - ip < 8) return ZS_ERR;
            u64 skip = (u64)ld32u(src + ip + 4) + 8;
            if (skip > n - ip) return ZS_ERR;
            ip += skip;
            continue;
        }
        if (magic != ZS_MAGIC) return ZS_ERR;
        if (n - ip < 5 + 3) return ZS_ERR;
        u32 fhd = ld8(src + ip + 4);
        u32 did_code = fhd & 3, csum = (fhd >> 2) & 1, single = (fhd >> 5) & 1, fcs_code = fhd >> 6;
        if (fhd & 8) return ZS_ERR;
        u32 did_len = did_code == 3 ? 4u : did_code, fcs_len = fcs_code == 0 ? 0u : (1u << fcs_code);
        u64 hsize = 5 + (single ? 0 : 1) + did_len + fcs_len + ((single && !fcs_code) ? 1 : 0);
        if (n - ip < hsize + 3) return ZS_ERR;
        u64 p = ip + 5;
        if (!single) {
            u32 wd = ld8(src + p++);
            if ((wd >> 3) + 10 > 31) return ZS_ERR;  // ZSTD_WINDOWLOG_MAX (64-bit)
        }
        u32 dict_id = 0;
        for (u32 k = 0; k < did_len; ++k) dict_id |= ld8(src + p++) << (8 * k);
        u64 fcs = 0;
        bool have_fcs = true;
        if (fcs_code == 0) { if (single) fcs = ld8(src + p++); else have_fcs = false; }
        else if (fcs_code == 1) { fcs = ld16u(src + p) + 256; p += 2; }
        else if (fcs_code == 2) { fcs = ld32u(src + p); p += 4; }
        else { fcs = ld64u(src + p); p += 8; }
        if (dict_id) return ZS_ERR;  // no dictionary is ever loaded
        ip += hsize;
        w.sync();
        if (w.l == 0) {
            S.huf_valid = 0; S.seq_valid = 0;
            S.rep[0] = 1; S.rep[1] = 4; S.rep[2] = 8;
        }
        w.sync();
        const u64 frame_start = op;
        for (;;) {  // zstd_decompress.c:850-889
            if (n - ip < 3) return ZS_ERR;
            u32 bh = ld16u(src + ip) | (ld8(src + ip + 2) << 16);
            ip += 3;
            u32 last = bh & 1, type = (bh >> 1) & 3, bsz = bh >> 3;
            if (type == 3) return ZS_ERR;
            u64 csz = type == 1 ? 1 : bsz;
            if (csz > n - ip) return ZS_ERR;
            if (type == 0) {
                if (bsz > cap - op) return ZS_ERR;
                zs_copy(w, dst + op, src + ip, bsz);
                op += bsz;
            } else if (type == 1) {
                if (bsz > cap - op) return ZS_ERR;
                zs_fill(w, dst + op, ld8(src + ip), bsz);
                op += bsz;
            } else {
                if (zs_block(w, S, src + ip, (u32)csz, dst, frame_start, &op, cap, scratch, hs)) return ZS_ERR;
            }
            w.sync();
            hs.advance(op, w);
            ip += csz;
            if (last) break;
        }
        if (have_fcs && op - frame_start != fcs) return ZS_ERR;
        if (csum) {
            if (n - ip < 4) return ZS_ERR;
            w.sync();
            if (ld32u(src + ip) != (u32)zs_xxh64(dst + frame_start, op - frame_start)) return ZS_ERR;
            ip += 4;
        }
    }
    if (ip != n) return ZS_ERR;  // "input not entirely consumed"
    *produced = op;
    return 0;
}

#ifndef ZPB_HOST_SIM
// ------------------------------------------------------------------------------------ kernel
// Persistent warps pull zstd entries from a device-side list (built by the scan kernel / the general
// kernel, which have already applied the guards of zpack_read.c:328-331) and decode + verify them.
#include "../../include/zpack_b200.h"
#define ZS_WARPS 2

// The entry's XXH3-64, streamed as the output front advances; the verdict of zpack_read_file (:466-468).
struct ZsHasher {
    Xxh3Stream<32> s;
    static constexpr int kFailed = ZPB_ST_DECOMPRESS_FAILED;   // lib/zpack_read.c:384-388
    ZPB_DEVINL void init(u8 *dst, const zpb_entry &e, u64 *, const ZWarp &w) { s.init(dst, e.uncomp_size, w.g); }
    ZPB_DEVINL void advance(u64 front, const ZWarp &w) { s.advance(front, w.g); }
    ZPB_DEVINL int finish(const zpb_entry &e, u64, u64 &dg, const ZWarp &w) {
        dg = s.finish(w.g);
        return !(e.flags & ZPB_F_NO_VERIFY) && dg != e.hash ? ZPB_ST_HASH_MISMATCH : ZPB_ST_OK;
    }
};

// One frame of a zstd entry decoded frame-parallel (zpb_unpack_blocks_device, pseudo-entry ZPB_M_ZSTD_FRAME): every
// complete KiB leaves its 16-stripe sums (64 bytes) at partials + (e.reserved + k) * 8, the layout lz4_fast_exec_kernel
// writes for LZ4 blocks; xxh3_chain_kernel runs the scramble chain over them.  No digest, and a frame that fails or
// decodes to another size than its pseudo-entry's declines the shard.
struct ZsPartialHasher {
    Xxh3Stream<32> s;   // base, alignment and the KiB cursor; its accumulators are not used
    u64 *part;
    static constexpr int kFailed = ZPB_ST_NOT_AVAILABLE;
    ZPB_DEVINL void init(u8 *dst, const zpb_entry &e, u64 *partials, const ZWarp &w) {
        s.init(dst, e.uncomp_size, w.g);
        s.full_blocks = e.uncomp_size >> 10;   // every complete KiB: the entry's tail is folded by the chain kernel
        part = partials + e.reserved * 8;
    }
    ZPB_DEVINL void advance(u64 front, const ZWarp &w) {
        if (!(s.next_block < s.full_blocks && ((s.next_block + 1) << 10) <= front)) return;
        w.g.sync();
        while (s.next_block < s.full_blocks && ((s.next_block + 1) << 10) <= front) {
            u64 s0 = 0, s1 = 0;
            s.stripes_sum(s0, s1, s.base + (s.next_block << 10), 16, w.g);
            s.fold(s0, s1, w.g);
            if (w.l < 4) *reinterpret_cast<ulonglong2 *>(part + s.next_block * 8 + 2 * w.l) = make_ulonglong2(s0, s1);
            ++s.next_block;
        }
    }
    ZPB_DEVINL int finish(const zpb_entry &e, u64 produced, u64 &dg, const ZWarp &w) {
        dg = 0;
        if (produced != e.uncomp_size) return kFailed;
        advance(produced, w);
        return ZPB_ST_OK;
    }
};

// `partials` is used by ZsPartialHasher only.
template <class Hasher>
__global__ void __launch_bounds__(ZS_WARPS * 32, 7)
zstd_unpack_kernel(const u8 *__restrict__ archive, u8 *__restrict__ out, const zpb_entry *__restrict__ entries,
                   const u32 *__restrict__ list, const u32 *__restrict__ n_ptr, u32 *counter, u8 *scratch,
                   int *status, u64 *digest, u64 *partials) {
    extern __shared__ __align__(16) u8 zs_smem[];
    ZstdShared &S = reinterpret_cast<ZstdShared *>(zs_smem)[threadIdx.x >> 5];
    ZWarp w;
    u8 *lit_buf = scratch + (u64)(blockIdx.x * ZS_WARPS + (threadIdx.x >> 5)) * ZS_LIT_SCRATCH;
    const u32 n = *n_ptr;
    for (;;) {
        u32 slot = 0;
        if (w.l == 0) slot = atomicAdd(counter, 1u);
        slot = w.bcast(slot, 0);
        if (slot >= n) break;
        const u32 idx = list[slot];
        const zpb_entry e = entries[idx];
        u8 *dst = out + e.dst_off;
        Hasher hs;
        hs.init(dst, e, partials, w);
#ifdef ZPB_ZS_PROFILE
        w.t_last = clock64();
#endif
        u64 produced = 0;
        int rc = zstd_decode_entry(w, S, lit_buf, archive + e.src_off, e.comp_size, dst, e.dst_cap, hs, &produced);
        int st = rc ? Hasher::kFailed : ZPB_ST_OK;
        u64 dg = 0;
        if (st == ZPB_ST_OK) st = hs.finish(e, produced, dg, w);
        if (w.l == 0) {
            status[idx] = st;
            digest[idx] = dg;
        }
        ZS_TICK(w, 7);
        w.sync();
    }
}
#endif
