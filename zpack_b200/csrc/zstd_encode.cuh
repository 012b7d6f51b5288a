// zstd_encode.cuh — zstd Compressed_Blocks from the LZ4 block compressor's matches: one thread per 4 KB window, one set of
// entropy tables per 64 KB block.
//
// The role of ZSTD_compressBlock_internal's back end (/root/reference/externals/zstd/lib/compress/zstd_compress.c,
// zstd_compress_sequences.c:ZSTD_encodeSequences, huf_compress.c, fse_compress.c) for the writer's
// ZPACK_COMPRESSION_ZSTD arm (lib/zpack_write.c:179).  Match finding is NOT zstd's: the sequences are the ones
// lz4_pack_blocks_kernel found for the block (pack_blocks.cuh; greedy, 64 KB window, 4-byte minimum match), read back
// from its LZ4 payload window by window.  Every 4 KB window becomes one zstd Compressed_Block
// (zstd_compression_format.md):
//   * literals: Huffman-coded in four streams with ONE code per 64 KB block, built from the histogram of all the block's
//     literals (lengths limited to 11 bits, direct 4-bit weight description); the block's first window with enough
//     literals carries the tree (Compressed_Literals_Block), the later ones reuse it (Treeless_Literals_Block).  Blocks
//     whose literals use byte values above 128, short sections and sections that would not shrink stay Raw_Literals —
//     unless the context's entropy switch is on (zpb_set_zstd_entropy): then such blocks get a full-alphabet code with
//     FSE-compressed weights when it pays, and a block the LZ4 compressor stored becomes literal-only windows (nbSeq = 0).
//   * sequences: encoded backwards exactly as ZSTD_encodeSequences does (states initialised from the last sequence, extra
//     bits LL / ML / OF, per earlier sequence the OF, ML, LL state transitions, final states ML, OF, LL, end mark), with
//     FSE tables fitted to the block's own LL / OF / ML codes: the block's first window with sequences describes them
//     (FSE_Compressed_Mode, or RLE_Mode for a single code), later windows use Repeat_Mode; small blocks keep the
//     predefined tables.  Repeat-offset codes are used for the part of the offset history a window has built itself.
// The ratio is reported next to ZSTD_compress level 3 by the tests and the bench.  A block that does not shrink stays a
// Raw_Block.
#pragma once
#include "common.cuh"
#include "pack_blocks.cuh"

#ifdef ZPB_SIM
#include <cmath>
#define ZE_CONST static const
#else
#define ZE_CONST __device__ __constant__
#endif

ZE_CONST short ZE_LL_NORM[36] = {4, 3, 2, 2, 2, 2, 2, 2, 2, 2, 2, 2, 2, 1, 1, 1, 2, 2,
                                 2, 2, 2, 2, 2, 2, 2, 3, 2, 1, 1, 1, 1, 1, -1, -1, -1, -1};
ZE_CONST short ZE_ML_NORM[53] = {1, 4, 3, 2, 2, 2, 2, 2, 2, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1,
                                 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, -1, -1, -1, -1, -1, -1, -1};
ZE_CONST short ZE_OF_NORM[29] = {1, 1, 1, 1, 1, 1, 2, 2, 2, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, -1, -1, -1, -1, -1};
ZE_CONST u32 ZE_LL_BASE[36] = {0, 1, 2, 3, 4, 5, 6, 7, 8, 9, 10, 11, 12, 13, 14, 15, 16, 18, 20, 22, 24, 28, 32, 40,
                               48, 64, 128, 256, 512, 1024, 2048, 4096, 8192, 16384, 32768, 65536};
ZE_CONST u8 ZE_LL_BITS[36] = {0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 1, 1,
                              1, 1, 2, 2, 3, 3, 4, 6, 7, 8, 9, 10, 11, 12, 13, 14, 15, 16};
ZE_CONST u32 ZE_ML_BASE[53] = {3, 4, 5, 6, 7, 8, 9, 10, 11, 12, 13, 14, 15, 16, 17, 18, 19, 20,
                               21, 22, 23, 24, 25, 26, 27, 28, 29, 30, 31, 32, 33, 34, 35, 37, 39, 41,
                               43, 47, 51, 59, 67, 83, 99, 131, 259, 515, 1027, 2051, 4099, 8195, 16387, 32771, 65539};
ZE_CONST u8 ZE_ML_BITS[53] = {0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0,
                              0, 0, 0, 0, 0, 1, 1, 1, 1, 2, 2, 3, 3, 4, 4, 5, 7, 8, 9, 10, 11, 12, 13, 14, 15, 16};

// One FSE compression table (FSE_buildCTable_wksp, fse_compress.c:68-180): next-state table + per symbol (deltaNbBits,
// deltaFindState), for a table log up to 9; or an RLE "table" (one symbol, no state bits).
struct ZeSeqTab {
    u16 st[512];
    u32 dnb[53];
    int dfs[53];
    u32 log;        // state bits (0 for RLE)
    u32 rle;        // 1: RLE_Mode, `sym` is the only symbol
    u32 sym;
};
// The three predefined distributions, built once per CTA into shared memory.
struct ZeTables { ZeSeqTab ll, of, ml; };
// One set per 64 KB block (global memory): tables fitted to the block's own sequence codes + their descriptions
// (FSE_writeNCount, or the single byte of RLE_Mode), written by the block's first window that has sequences.
struct ZeBlockTabs {
    ZeSeqTab ll, of, ml;
    u8 desc[3][64];
    u32 desc_len[3];
    u32 valid;      // 0: the block's sequences use the predefined tables
};

#ifdef ZPB_SIM
ZPB_DEVINL int ze_highbit(u32 v) { int r = 0; while (v >>= 1) ++r; return r; }
#else
ZPB_DEVINL int ze_highbit(u32 v) { return 31 - __clz((int)v); }
#endif

ZPB_DEVINL void ze_build(ZeSeqTab &T, const short *norm, int nsym, int log) {
    const int size = 1 << log, mask = size - 1, step = (size >> 1) + (size >> 3) + 3;
    u8 sym_of[512];
    int cumul[54];
    int high = size - 1;
    T.log = (u32)log; T.rle = 0; T.sym = 0;
    cumul[0] = 0;
    for (int s = 0; s < nsym; ++s) {
        if (norm[s] == -1) { cumul[s + 1] = cumul[s] + 1; sym_of[high--] = (u8)s; }
        else cumul[s + 1] = cumul[s] + norm[s];
    }
    int pos = 0;
    for (int s = 0; s < nsym; ++s)
        for (int i = 0; i < norm[s]; ++i) {
            sym_of[pos] = (u8)s;
            do pos = (pos + step) & mask; while (pos > high);
        }
    for (int u = 0; u < size; ++u) { const int s = sym_of[u]; T.st[cumul[s]++] = (u16)(size + u); }
    int total = 0;
    for (int s = 0; s < nsym; ++s) {
        const int n = norm[s];
        if (n == 0) { T.dnb[s] = (u32)(((log + 1) << 16) - size); T.dfs[s] = 0; }
        else if (n == -1 || n == 1) { T.dnb[s] = (u32)((log << 16) - size); T.dfs[s] = total - 1; ++total; }
        else {
            const int mb = log - ze_highbit((u32)(n - 1));
            T.dnb[s] = (u32)((mb << 16) - (n << mb));
            T.dfs[s] = total - n;
            total += n;
        }
    }
}
ZPB_DEVINL void ze_build_tables(ZeTables &T) {
    ze_build(T.ll, ZE_LL_NORM, 36, 6);
    ze_build(T.of, ZE_OF_NORM, 29, 5);
    ze_build(T.ml, ZE_ML_NORM, 53, 6);
}

// Normalised counts for a histogram (the role of FSE_normalizeCount, fse_compress.c:430-490; any distribution that sums to
// the table size and gives every present symbol at least 1 is valid): proportional shares, the rounding error settled
// on the largest shares.  Returns the table log, or 0 when only one symbol occurs (RLE_Mode; *only = that symbol).
ZPB_DEVINL int ze_normalize(const u32 *cnt, int nsym, u32 total, int maxlog, short *norm, int *last, int *only) {
    int present = 0, lastsym = 0;
    for (int s = 0; s < nsym; ++s) if (cnt[s]) { ++present; lastsym = s; }
    *last = lastsym;
    *only = lastsym;
    if (present <= 1) return 0;
    int log = ze_highbit(total) - 2;
    if (log < 5) log = 5;
    if (log > maxlog) log = maxlog;
    while ((1 << log) < present) ++log;
    const int size = 1 << log;
    int sum = 0, big = 0;
    for (int s = 0; s < nsym; ++s) {
        int v = 0;
        if (cnt[s]) {
            v = (int)(((u64)cnt[s] * (u32)size + total / 2) / total);
            if (v < 1) v = 1;
        }
        norm[s] = (short)v;
        sum += v;
        if (v > norm[big]) big = s;
    }
    if (sum < size) norm[big] = (short)(norm[big] + (size - sum));
    while (sum > size) {                               // take the excess from the largest shares, one at a time
        int b = 0;
        for (int s = 1; s < nsym; ++s) if (norm[s] > norm[b]) b = s;
        --norm[b];
        --sum;
    }
    return log;
}
// table description (FSE_writeNCount_generic, fse_compress.c:290-400; read back by FSE_readNCount): returns bytes
ZPB_DEVINL u32 ze_write_ncount(u8 *out, const short *norm, int last, int log) {
    u64 acc = 0;
    u32 n = 0, op = 0;
    const int size = 1 << log;
    int remaining = size + 1, threshold = size, nbits = log + 1, sym = 0;
    bool prev0 = false;
    acc |= (u64)(log - 5) << n; n += 4;
    while (sym <= last && remaining > 1) {
        if (prev0) {
            int start = sym;
            while (sym <= last && norm[sym] == 0) ++sym;
            int run = sym - start;
            while (run >= 3) {
                acc |= (u64)3 << n; n += 2; run -= 3;
                if (n >= 32) { for (int k = 0; k < 4; ++k) out[op++] = (u8)(acc >> (8 * k)); acc >>= 32; n -= 32; }
            }
            acc |= (u64)run << n; n += 2;
        }
        int count = norm[sym++];
        const int max = (2 * threshold - 1) - remaining;
        remaining -= count < 0 ? -count : count;
        ++count;
        if (count >= threshold) count += max;
        acc |= (u64)count << n;
        n += (u32)(count < max ? nbits - 1 : nbits);
        prev0 = count == 1;
        while (remaining < threshold) { --nbits; threshold >>= 1; }
        if (n >= 32) { for (int k = 0; k < 4; ++k) out[op++] = (u8)(acc >> (8 * k)); acc >>= 32; n -= 32; }
    }
    while (n > 0) { out[op++] = (u8)acc; acc >>= 8; n = n > 8 ? n - 8 : 0; }
    return op;
}
// one table fitted to a histogram of codes: RLE or FSE + its description
ZPB_DEVINL void ze_fit(ZeSeqTab &T, u8 *desc, u32 *desc_len, const u32 *cnt, int nsym, u32 total, int maxlog) {
    short norm[53];
    int last = 0, only = 0;
    const int log = ze_normalize(cnt, nsym, total, maxlog, norm, &last, &only);
    if (log == 0) {
        T.log = 0; T.rle = 1; T.sym = (u32)only;
        desc[0] = (u8)only;
        *desc_len = 1;
        return;
    }
    ze_build(T, norm, last + 1, log);
    *desc_len = ze_write_ncount(desc, norm, last, log);
}

// codes (zstd_compress_internal.h: ZSTD_LLcode / ZSTD_MLcode, written as searches over the base tables)
ZPB_DEVINL u32 ze_ll_code(u32 ll) {
    if (ll < 16) return ll;
    if (ll >= 64) return (u32)ze_highbit(ll) + 19u;
    u32 c = 16;
    while (c < 24 && ZE_LL_BASE[c + 1] <= ll) ++c;
    return c;
}
ZPB_DEVINL u32 ze_ml_code(u32 ml) {            // ml = match length (>= 3)
    if (ml < 35) return ml - 3;
    if (ml >= 131) return (u32)ze_highbit(ml - 3) + 36u;
    u32 c = 32;
    while (c < 42 && ZE_ML_BASE[c + 1] <= ml) ++c;
    return c;
}

struct ZeBits {                 // forward little-endian bit writer (bitstream.h: BIT_addBits / BIT_flushBits)
    u64 acc;
    u32 n;
    u8 *p, *end;
    bool ovf;
};
ZPB_DEVINL void ze_add(ZeBits &b, u32 v, u32 nb) { b.acc |= (u64)v << b.n; b.n += nb; }
// The writer only ever stores aligned 32-bit words (one predicated store per flush: lanes of a warp stay converged).
// A stream that starts at an unaligned byte starts at the word below it, the bytes in front taken as `fill` (what is
// already there, or zeros where nothing is yet).
ZPB_DEVINL void ze_open(ZeBits &b, u8 *at, u8 *end, bool keep) {
    const u32 k = (u32)(uintptr_t)at & 3u;
    b.p = at - k;
    b.end = end;
    b.ovf = false;
    b.n = 8u * k;
    b.acc = keep && k ? (u64)(*reinterpret_cast<const u32 *>(b.p) & ((1u << (8u * k)) - 1u)) : 0ull;
}
ZPB_DEVINL void ze_flush(ZeBits &b) {                 // leaves at most 31 bits pending
    if (b.n >= 32) {
        if (b.p + 4 <= b.end) { *reinterpret_cast<u32 *>(b.p) = (u32)b.acc; b.p += 4; } else b.ovf = true;
        b.acc >>= 32;
        b.n -= 32;
    }
}
ZPB_DEVINL void ze_flush_all(ZeBits &b) {             // every whole byte, then the partial one
    while (b.n >= 8) {
        if (b.p < b.end) *b.p++ = (u8)b.acc; else b.ovf = true;
        b.acc >>= 8;
        b.n -= 8;
    }
    if (b.n) { if (b.p < b.end) *b.p++ = (u8)b.acc; else b.ovf = true; b.n = 0; }
}
// sequential reader of the LZ4 payload: eight aligned bytes per load
struct ZeIn {
    const u8 *base;
    u64 w;
    u32 pos;            // next byte to hand out
};
ZPB_DEVINL void ze_in_seek(ZeIn &r, u32 pos) {
    r.pos = pos;
    const u8 *a = r.base + pos;
    r.w = *reinterpret_cast<const u64 *>((uintptr_t)a & ~(uintptr_t)7) >> (8u * ((u32)(uintptr_t)a & 7u));
}
ZPB_DEVINL u32 ze_in_byte(ZeIn &r) {
    const u32 v = (u32)r.w & 0xFFu;
    ++r.pos;
    if ((((uintptr_t)r.base + r.pos) & 7u) == 0) r.w = *reinterpret_cast<const u64 *>(r.base + r.pos);
    else r.w >>= 8;
    return v;
}
ZPB_DEVINL u32 ze_init_state(const ZeSeqTab &T, u32 sym) {      // FSE_initCState2
    if (T.rle) return 0;
    const u32 nbo = (T.dnb[sym] + (1u << 15)) >> 16;
    const u32 value = (nbo << 16) - T.dnb[sym];
    return T.st[(int)(value >> nbo) + T.dfs[sym]];
}
ZPB_DEVINL u32 ze_encode(ZeBits &b, const ZeSeqTab &T, u32 state, u32 sym) {   // FSE_encodeSymbol
    if (T.rle) return 0;
    const u32 nbo = (state + T.dnb[sym]) >> 16;
    ze_add(b, state & ((1u << nbo) - 1u), nbo);
    return T.st[(int)(state >> nbo) + T.dfs[sym]];
}

#define ZE_FAIL 0xFFFFFFFFu
#define ZE_WIN_SEQ 1040u       // records per window: at most 1024 matches start inside 4096 positions
// a block's bodies: window w's at 1.25 x the payload offset of its first sequence + 24 * w (a zstd body can be somewhat
// larger than the LZ4 bytes it restates: 16-bit offsets cost 2 bytes there, code + extra bits here)
#define ZE_SLOT (65536u + 16384u + 512u)
#define ZE_OFF(begin, w) ((begin) + ((begin) >> 2) + 24u * (w))
#define ZE_ZBODY ZE_META       // stride of the per-block words; the first 16: body size of every window's sub-block (0: nothing to emit, ZE_FAIL: store the block raw)
#define ZE_HUF_MIN 64u         // literal sections shorter than this stay raw
#define ZE_HUF_SYMS 129u       // direct (4-bit) weight description: symbols 0..128 (huf_compress.c:HUF_writeCTable, header >= 128)

// ---- stage A: one window's LZ4 sequences lz[begin, end) (+ the block's closing literals-only sequence lz[end, tail_end)
// for its last window) -> literal bytes at `lit_dst` (capacity tail_end - begin), records in `seq`.  false: not what
// pack_blocks.cuh writes.
ZPB_DEVINL bool ze_parse_range(const u8 *lz, u32 begin, u32 end, u32 tail_end, u8 *lit_dst, u64 *seq, u32 seq_cap, u32 *lit_n,
                               u32 *seq_n) {
    u32 lit = 0, nseq = 0;
    ZeIn in;
    in.base = lz;
    ze_in_seek(in, begin);
    ZeBits lw;
    ze_open(lw, lit_dst, lit_dst + (tail_end - begin) + 8u, false);
    bool bad = false;                                 // single-exit loops: the lanes of a warp (one window each) reconverge every iteration
    u32 rp0 = 0, rp1 = 0, rp2 = 0, known = 0;         // the part of the repeat-offset history this window has built itself
    while (in.pos < tail_end && !bad) {
        const u32 token = ze_in_byte(in);
        u32 ll = token >> 4;
        if (ll == 15) {
            u32 x;
            do { x = in.pos < tail_end ? ze_in_byte(in) : 0u; ll += x; } while (x == 255);
        }
        if (in.pos + ll > tail_end) { bad = true; ll = 0; }
        for (u32 i = 0; i < ll; ++i) { ze_add(lw, ze_in_byte(in), 8); ze_flush(lw); }
        lit += ll;
        if (in.pos > end) {                           // the closing sequence of the block: literals only
            bad |= in.pos != tail_end;
        } else if (in.pos + 2 > end) {
            bad = true;
        } else {
            u32 off = ze_in_byte(in);
            off |= ze_in_byte(in) << 8;
            u32 ml = token & 15u;
            if (ml == 15) {
                u32 x;
                do { x = in.pos < end ? ze_in_byte(in) : 0u; ml += x; } while (x == 255);
            }
            ml += 4;
            if (off == 0 || nseq >= seq_cap || ll > 65535u || ml > 65535u) bad = true;
            else {
                // offset VALUE (zstd_compression_format.md, "Repeat offsets"): 1-3 name one of the three most recent offsets,
                // anything else is offset + 3.  The window does not know what the windows before it left in that history,
                // so it only names entries it has pushed itself (`known` of them); the decoder's history evolves the same
                // way whatever the older entries are.
                u32 ofv = off + 3u;
                if (ll) {
                    if (known >= 1 && off == rp0) ofv = 1;
                    else if (known >= 2 && off == rp1) { ofv = 2; rp1 = rp0; rp0 = off; }
                    else if (known >= 3 && off == rp2) { ofv = 3; rp2 = rp1; rp1 = rp0; rp0 = off; }
                } else {                               // literal length 0 shifts the meaning: 1 -> second, 2 -> third, 3 -> first - 1
                    if (known >= 2 && off == rp1) { ofv = 1; rp1 = rp0; rp0 = off; }
                    else if (known >= 3 && off == rp2) { ofv = 2; rp2 = rp1; rp1 = rp0; rp0 = off; }
                    else if (known >= 1 && off == rp0 - 1u && off) { ofv = 3; rp2 = rp1; rp1 = rp0; rp0 = off; if (known < 3) ++known; }
                }
                if (ofv > 3u) { rp2 = rp1; rp1 = rp0; rp0 = off; if (known < 3) ++known; }
                seq[nseq++] = (u64)ll | ((u64)ml << 16) | ((u64)ofv << 32);
            }
        }
    }
    ze_flush_all(lw);
    *lit_n = lit;
    *seq_n = nseq;
    return !bad && !lw.ovf;
}

// ---- stage B: one Huffman code per 64 KB block, from the histogram of all its literals (huf_compress.c:HUF_buildCTable,
// HUF_writeCTable).  Lengths are limited to 11 bits by the overflow rule of deflate's gen_bitlen.  Blocks whose literals
// are bytes 0..128 get the direct description (4-bit weights).  Above that only with `full` (the context's entropy
// switch): the weights are then FSE-compressed, and the caller keeps the table only if ze_huf_settle finds that it pays.
#define ZE_CARRIER_FIRST 0xFFFFFFFFu   // ZeHuf::carrier: the block's first window with ZE_HUF_MIN literals carries the tree (ze_lit_mode)
struct ZeHuf {
    u16 code[256];
    u8 len[256];
    u8 desc[128];         // header byte (>= 128: 4-bit weights of symbols 0 .. last-1, two per byte; < 128: bytes of FSE-compressed weights)
    u32 desc_len;         // 0: no table for this block
    u32 carrier;          // the window that carries the tree, or ZE_CARRIER_FIRST
};

// FSE-compressed weights, as HUF_compressWeights + FSE_compress_usingCTable_generic write them (huf_compress.c,
// fse_compress.c): NCount header with table log <= 6, then two interleaved states over the weights from the last to the
// first.  The decoder counts the weights by where the bitstream ends, so the symbol order, the start of an odd count and
// the final state flushes (state 2, then state 1, then the end mark) follow the reference exactly.  out[0] = size; returns
// 1 + size, or 0 when there is no such description: every weight the same (the reference writes none either), or a
// size of 128 bytes or more, which the header byte cannot express.
ZPB_DEVINL u32 ze_huf_weights_fse(const u8 *wt, int nw, u8 *out) {
    u32 cnt[12];
    for (int s = 0; s < 12; ++s) cnt[s] = 0;
    for (int i = 0; i < nw; ++i) ++cnt[wt[i]];
    short norm[12];
    int last = 0, only = 0;
    const int log = ze_normalize(cnt, 12, (u32)nw, 6, norm, &last, &only);
    if (log == 0 || nw <= 2) return 0;
    u32 buf[32];                                      // the description is built aligned, then copied behind the header byte
    u8 *b8 = reinterpret_cast<u8 *>(buf);
    const u32 hs = ze_write_ncount(b8, norm, last, log);
    ZeSeqTab T;
    ze_build(T, norm, last + 1, log);
    ZeBits b;
    ze_open(b, b8 + hs, b8 + 127, true);
    const u8 *ip = wt + nw;
    u32 s1, s2;
    if (nw & 1) {
        s1 = ze_init_state(T, *--ip);
        s2 = ze_init_state(T, *--ip);
        s1 = ze_encode(b, T, s1, *--ip);
        ze_flush(b);
    } else {
        s2 = ze_init_state(T, *--ip);
        s1 = ze_init_state(T, *--ip);
    }
    while (ip > wt) {                                 // an even number is left: state 2, state 1, ...
        s2 = ze_encode(b, T, s2, *--ip);
        ze_flush(b);
        s1 = ze_encode(b, T, s1, *--ip);
        ze_flush(b);
    }
    ze_add(b, s2 & ((1u << log) - 1u), (u32)log);     // FSE_flushCState: state 2, then state 1
    ze_flush(b);
    ze_add(b, s1 & ((1u << log) - 1u), (u32)log);
    ze_add(b, 1u, 1);                                 // BIT_closeCStream
    ze_flush_all(b);
    if (b.ovf) return 0;
    const u32 size = (u32)(b.p - b8);
    out[0] = (u8)size;
    for (u32 i = 0; i < size; ++i) out[1 + i] = b8[i];
    return 1u + size;
}

// fixed: bytes the block pays for any table besides its description (6 per window of jump table), for the entropy check.
ZPB_DEVINL void ze_huf_build(const u32 *hist, ZeHuf &H, bool full = false, u32 fixed = 0) {
    H.desc_len = 0;
    H.carrier = ZE_CARRIER_FIRST;
    int last = -1, n = 0;
    for (int s = 0; s < 256; ++s) if (hist[s]) { last = s; ++n; }
    if (n < 2 || (last >= (int)ZE_HUF_SYMS && !full)) return;
    if (last >= (int)ZE_HUF_SYMS) {
        // No code beats the order-0 entropy: when even that cannot save the 1/64 ze_huf_settle asks for (near-uniform
        // bytes: random data, most records), skip the build.  The margin keeps the float sum on the safe side, so this
        // refuses only tables that ze_huf_settle would refuse.
        u32 total = 0;
        for (int s = 0; s < 256; ++s) total += hist[s];
        float bits = 0.f;
        const float lt = log2f((float)total);
        for (int s = 0; s < 256; ++s) if (hist[s]) bits += (float)hist[s] * (lt - log2f((float)hist[s]));
        if (bits * (0.999f / 8.f) - 1.f + (float)(fixed + total / 64u) >= (float)total) return;
    }
    // leaves by ascending count (insertion sort), then the two-queue construction
    short order[256];
    u32 cnt[512];
    short parent[512];
    int m = 0;
    for (int s = 0; s <= last; ++s) {
        if (!hist[s]) continue;
        int k = m++;
        while (k > 0 && hist[order[k - 1]] > hist[s]) { order[k] = order[k - 1]; --k; }
        order[k] = (short)s;
    }
    for (int i = 0; i < n; ++i) cnt[i] = hist[order[i]];
    int lf = 0, in0 = n, in1 = n;                       // next leaf, first unused internal node, next free node
    for (int k = 0; k < n - 1; ++k) {
        int a, b;
        if (lf < n && (in0 >= in1 || cnt[lf] <= cnt[in0])) a = lf++; else a = in0++;
        if (lf < n && (in0 >= in1 || cnt[lf] <= cnt[in0])) b = lf++; else b = in0++;
        cnt[in1] = cnt[a] + cnt[b];
        parent[a] = parent[b] = (short)in1;
        ++in1;
    }
    const int root = in1 - 1;
    u8 depth[512];
    depth[root] = 0;
    for (int i = root - 1; i >= 0; --i) depth[i] = (u8)(depth[parent[i]] + 1);     // parents have larger indices
    // length limit 11: leaves deeper than that are lifted, and for every two of them one shallower leaf goes down a level
    int bl[32];
    for (int i = 0; i < 32; ++i) bl[i] = 0;
    int overflow = 0;
    for (int i = 0; i < n; ++i) {
        int d = depth[i];
        if (d > 11) { d = 11; ++overflow; }
        ++bl[d];
    }
    while (overflow > 0) {
        int bits = 10;
        while (bl[bits] == 0) --bits;
        --bl[bits];
        bl[bits + 1] += 2;
        --bl[11];
        overflow -= 2;
    }
    if (last >= (int)ZE_HUF_SYMS) {
        // Full alphabets only (the direct description keeps the rule above as it is): with leaves deeper than 12 the rule
        // leaves the code over-full.  Settle the Kraft sum (in units of 2^-11) exactly: lengthen the longest codes below
        // 11 while it is over, shorten the longest codes that fit the gap while it is under.
        int kraft = 0;
        for (int bits = 1; bits <= 11; ++bits) kraft += bl[bits] << (11 - bits);
        while (kraft > 2048) {
            int bits = 10;
            while (bl[bits] == 0) --bits;
            --bl[bits]; ++bl[bits + 1];
            kraft -= 1 << (10 - bits);
        }
        while (kraft < 2048) {
            int bits = 11;
            while (bl[bits] == 0 || (1 << (11 - bits)) > 2048 - kraft) --bits;
            --bl[bits]; ++bl[bits - 1];
            kraft += 1 << (11 - bits);
        }
    }
    int maxbits = 11;
    while (bl[maxbits] == 0) --maxbits;
    // lengths back to the symbols: the rarest get the longest codes
    for (int s = 0; s < 256; ++s) { H.len[s] = 0; H.code[s] = 0; }
    {
        int i = 0;
        for (int bits = maxbits; bits >= 1; --bits)
            for (int c = 0; c < bl[bits]; ++c) H.len[order[i++]] = (u8)bits;
    }
    // codes as a decoder derives them from the weights (huf_decompress.c:HUF_readDTableX1): weight w = maxbits + 1 - len,
    // table cells of 2^(w-1) in ascending weight, symbols of one weight in ascending order
    u32 start[16], rank[16];
    for (int r = 0; r < 16; ++r) rank[r] = 0;
    for (int s = 0; s <= last; ++s) if (H.len[s]) ++rank[maxbits + 1 - H.len[s]];
    u32 acc = 0;
    for (int r = 1; r <= maxbits; ++r) { start[r] = acc; acc += rank[r] << (r - 1); }
    if (acc != (1u << maxbits)) return;               // not a complete code: cannot happen, but then no table
    for (int s = 0; s <= last; ++s) {
        if (!H.len[s]) continue;
        const int w = maxbits + 1 - H.len[s];
        H.code[s] = (u16)(start[w] >> (w - 1));
        start[w] += 1u << (w - 1);
    }
    // description: 127 + number of weights, then the weights of symbols 0 .. last-1 (the last one is implied); beyond
    // 128 weights the FSE-compressed form, which ze_huf_settle has to accept
    const int nw = last;
    if (last >= (int)ZE_HUF_SYMS) {
        u8 wt[255];
        for (int i = 0; i < nw; ++i) wt[i] = H.len[i] ? (u8)(maxbits + 1 - H.len[i]) : (u8)0;
        H.desc_len = ze_huf_weights_fse(wt, nw, H.desc);
        H.carrier = 16;                              // none yet
        return;
    }
    H.desc[0] = (u8)(127 + nw);
    for (int i = 0; i < nw; i += 2) {
        const u32 w0 = H.len[i] ? (u32)(maxbits + 1 - H.len[i]) : 0u;
        const u32 w1 = i + 1 < nw && H.len[i + 1] ? (u32)(maxbits + 1 - H.len[i + 1]) : 0u;
        H.desc[1 + i / 2] = (u8)((w0 << 4) | w1);
    }
    H.desc_len = 1u + (u32)(nw + 1) / 2u;
}

// which kind of literals section window w writes: 0 raw, 2 Compressed (carries the block's tree), 3 Treeless (uses it).
// The tree rides on the first window with enough literals; windows before it stay raw.
ZPB_DEVINL u32 ze_lit_mode(u32 w, const u32 *lit_n, u32 nwin, bool have_table) {
    if (!have_table || lit_n[w] < ZE_HUF_MIN) return 0;
    for (u32 k = 0; k < w && k < nwin; ++k) if (lit_n[k] >= ZE_HUF_MIN) return 3;
    return 2;
}
// The same for a table that names its carrier (full-alphabet tables, ze_huf_settle).
ZPB_DEVINL u32 ze_lit_mode(u32 w, const u32 *lit_n, u32 nwin, const ZeHuf &H) {
    if (!H.desc_len) return 0;
    if (H.carrier == ZE_CARRIER_FIRST) return ze_lit_mode(w, lit_n, nwin, true);
    if (lit_n[w] < ZE_HUF_MIN || w < H.carrier) return 0;
    return w == H.carrier ? 2u : 3u;
}

// A full-alphabet table (ze_huf_build with `full`, symbols above 128) is kept only if it pays: the block's literals,
// estimated as their coded bits + the description + a 6-byte jump table per window, must save 1/64 against raw
// literals.  Near-uniform literal bytes (random data, records) then keep raw literals at the cost of the histogram.
// The tree rides on the first window with ZE_HUF_MIN literals whose section, tree included, is surely smaller than
// raw (coded bits + one byte per stream + jump table + two bytes of a longer section header): the carrier cannot fall
// back to raw literals, the windows after it can.  bits[w]: window w's literals coded with H.
ZPB_DEVINL void ze_huf_settle(ZeHuf &H, const u32 *lit_n, const u32 *bits, u32 nwin) {
    if (!H.desc_len || H.carrier == ZE_CARRIER_FIRST) return;
    u32 total = 0;
    u64 coded = 0;
    for (u32 w = 0; w < nwin; ++w) { total += lit_n[w]; coded += bits[w]; }
    u32 carrier = 16;
    if (coded / 8u + H.desc_len + 6u * nwin + total / 64u < total)
        for (u32 w = 0; w < nwin && carrier == 16; ++w)
            if (lit_n[w] >= ZE_HUF_MIN && (bits[w] + 7u) / 8u + 4u + 6u + 2u + H.desc_len < lit_n[w]) carrier = w;
    H.carrier = carrier;
    if (carrier == 16) H.desc_len = 0;
}

// which sequence tables window w uses: 0 predefined, 2 the block's own tables, which this window also describes (it is the
// block's first window with sequences), 3 the block's own tables, already described (Repeat_Mode)
ZPB_DEVINL u32 ze_seq_mode(u32 w, const u32 *seq_n, u32 nwin, bool have_tabs) {
    if (!have_tabs || seq_n[w] == 0) return 0;
    for (u32 k = 0; k < w && k < nwin; ++k) if (seq_n[k]) return 3;
    return 2;
}
#define ZE_TABS_MIN 64u        // blocks with fewer sequences keep the predefined tables

// one Huffman stream: symbols lit[0, n) coded last to first (huf_compress.c:HUF_compress1X_usingCTable), end mark; returns bytes
ZPB_DEVINL u32 ze_huf_stream(const u8 *lit, u32 n, u8 *at, u8 *end, const ZeHuf &H, bool *ovf) {
    ZeBits b;
    ze_open(b, at, end, true);
    for (u32 i = n; i-- > 0;) {
        const u32 s = lit[i];
        ze_add(b, H.code[s], H.len[s]);
        ze_flush(b);
    }
    ze_add(b, 1u, 1);
    ze_flush_all(b);
    *ovf |= b.ovf;
    return (u32)(b.p - at);
}

// ---- stage C: one window's sub-block body at `out`: literals section (raw, or Huffman-coded in four streams with the
// block's table), sequences section.  Returns the body size; 0 when the window has nothing to emit; ZE_FAIL when it does
// not fit `cap` (the caller then stores the whole block raw).
// seqmode: 0 predefined tables (T), 2 this window carries the block's own tables (B: descriptions written, FSE_Compressed /
// RLE modes), 3 it reuses them (Repeat_Mode).
ZPB_DEVINL u32 ze_emit_range(const u8 *lit, u32 lit_n, const u64 *seq, u32 nseq, u32 mode, const ZeHuf &H, u8 *out, u32 cap,
                             const ZeTables &T, u32 seqmode, const ZeBlockTabs &B) {
    if (lit_n == 0 && nseq == 0) return 0;
    if (cap < 24) return ZE_FAIL;
    u32 op = 0;
    bool ovf = false;
    if (mode) {
        // Compressed / Treeless literals, four streams (zstd_compression_format.md: Literals_Section_Header, size formats
        // 01 / 10 / 11 by the larger of the two sizes; jump table of three 16-bit stream sizes)
        const u32 fmt = lit_n < 1024 ? 1u : (lit_n < 16384 ? 2u : 3u);
        const u32 hdr = 3u + (fmt - 1u);
        const u32 tree = mode == 2 ? H.desc_len : 0u;
        if (hdr + tree + 6u + 16u >= cap) return ZE_FAIL;
        for (u32 i = 0; i < tree; ++i) out[hdr + i] = H.desc[i];
        u8 *jt = out + hdr + tree;
        u32 pos = hdr + tree + 6u;
        const u32 seg = (lit_n + 3u) / 4u;
        u32 sz[4];
        for (u32 k = 0; k < 4; ++k) {
            const u32 a = k * seg, n = k < 3 ? seg : lit_n - 3u * seg;
            sz[k] = ze_huf_stream(lit + a, n, out + pos, out + cap, H, &ovf);
            pos += sz[k];
        }
        const u32 comp = tree + 6u + sz[0] + sz[1] + sz[2] + sz[3];
        const u32 lim = fmt == 1 ? 1024u : (fmt == 2 ? 16384u : 262144u);
        if (!ovf && comp < lim && comp < lit_n && sz[0] < 65536u && sz[1] < 65536u && sz[2] < 65536u) {
            for (u32 k = 0; k < 3; ++k) { jt[2 * k] = (u8)sz[k]; jt[2 * k + 1] = (u8)(sz[k] >> 8); }
            const u32 bits = 10u + 4u * (fmt - 1u);
            const u64 h = (u64)mode | ((u64)fmt << 2) | ((u64)lit_n << 4) | ((u64)comp << (4 + bits));
            for (u32 i = 0; i < hdr; ++i) out[i] = (u8)(h >> (8 * i));
            op = pos;
        } else if (mode == 2) return ZE_FAIL;         // the tree carrier must not fall back: later windows count on the table
        else mode = 0;
    }
    if (!mode) {
        if (3 + lit_n + 8 >= cap) return ZE_FAIL;
        out[0] = (u8)(0x0Cu | ((lit_n & 0xFu) << 4));  // Raw_Literals_Block, size format 11: 20-bit size
        out[1] = (u8)(lit_n >> 4);
        out[2] = (u8)(lit_n >> 12);
        ZeBits lw;
        ze_open(lw, out + 3, out + cap, true);
        for (u32 i = 0; i < lit_n; ++i) { ze_add(lw, lit[i], 8); ze_flush(lw); }
        ze_flush_all(lw);
        if (lw.ovf) return ZE_FAIL;
        op = 3 + lit_n;
    }
    if (op + 8 >= cap) return ZE_FAIL;
    // ---- sequences section header: count, then symbol compression modes = 0 (all predefined)
    if (nseq == 0) { out[op++] = 0; return op; }
    if (nseq < 128) out[op++] = (u8)nseq;
    else if (nseq < 0x7F00) { out[op++] = (u8)((nseq >> 8) + 0x80); out[op++] = (u8)nseq; }
    else { out[op++] = 0xFF; out[op++] = (u8)(nseq - 0x7F00); out[op++] = (u8)((nseq - 0x7F00) >> 8); }
    const ZeSeqTab &TL = seqmode ? B.ll : T.ll, &TO = seqmode ? B.of : T.of, &TM = seqmode ? B.ml : T.ml;
    if (seqmode == 2) {
        out[op++] = (u8)(((TL.rle ? 1u : 2u) << 6) | ((TO.rle ? 1u : 2u) << 4) | ((TM.rle ? 1u : 2u) << 2));
        if (op + B.desc_len[0] + B.desc_len[1] + B.desc_len[2] + 8 >= cap) return ZE_FAIL;
        for (u32 k = 0; k < 3; ++k)                  // LL, OF, ML (zstd_compression_format.md: Sequences_Section_Header)
            for (u32 i = 0; i < B.desc_len[k]; ++i) out[op++] = B.desc[k][i];
    } else out[op++] = seqmode == 3 ? 0xFCu : 0u;
    // ---- the bitstream, from the last sequence to the first (zstd_compress_sequences.c:ZSTD_encodeSequences_body)
    ZeBits b;
    ze_open(b, out + op, out + cap, true);
    u32 st_ll, st_of, st_ml;
    {
        const u64 r = seq[nseq - 1];
        const u32 ll = (u32)(r & 0xFFFF), ml = (u32)((r >> 16) & 0xFFFF), ob = (u32)(r >> 32);
        const u32 cl = ze_ll_code(ll), cm = ze_ml_code(ml), co = (u32)ze_highbit(ob);
        st_ml = ze_init_state(TM, cm);
        st_of = ze_init_state(TO, co);
        st_ll = ze_init_state(TL, cl);
        ze_add(b, ll - ZE_LL_BASE[cl], ZE_LL_BITS[cl]);
        ze_add(b, ml - ZE_ML_BASE[cm], ZE_ML_BITS[cm]);
        ze_flush(b);
        ze_add(b, ob - (1u << co), co);
        ze_flush(b);
    }
    u64 r_next = nseq > 1 ? seq[nseq - 2] : 0ull;
    for (u32 k = nseq - 1; k-- > 0;) {
        const u64 r = r_next;
        if (k) r_next = seq[k - 1];                  // the record after this one is on its way while this one is encoded
        const u32 ll = (u32)(r & 0xFFFF), ml = (u32)((r >> 16) & 0xFFFF), ob = (u32)(r >> 32);
        const u32 cl = ze_ll_code(ll), cm = ze_ml_code(ml), co = (u32)ze_highbit(ob);
        st_of = ze_encode(b, TO, st_of, co);
        st_ml = ze_encode(b, TM, st_ml, cm);
        st_ll = ze_encode(b, TL, st_ll, cl);
        ze_flush(b);
        ze_add(b, ll - ZE_LL_BASE[cl], ZE_LL_BITS[cl]);
        ze_add(b, ml - ZE_ML_BASE[cm], ZE_ML_BITS[cm]);
        ze_flush(b);
        ze_add(b, ob - (1u << co), co);
        ze_flush(b);
    }
    ze_add(b, st_ml & ((1u << TM.log) - 1u), TM.log);     // FSE_flushCState: ML, OF, LL
    ze_flush(b);
    ze_add(b, st_of & ((1u << TO.log) - 1u), TO.log);
    ze_add(b, st_ll & ((1u << TL.log) - 1u), TL.log);
    ze_flush(b);
    ze_add(b, 1u, 1);                                // BIT_closeCStream: the end mark
    ze_flush_all(b);
    if (b.ovf) return ZE_FAIL;
    return (u32)(b.p - out);
}

#define ZE_LITSLOT (65536u + 256u)                    // a block's staged literals: window w's at ZE_LOFF(payload offset, w)
#define ZE_LOFF(begin, w) ((((begin) + 3u) & ~3u) + 8u * (w))
#define ZE_META 48u                                   // u32 per block: 16 body sizes | 16 literal counts | 16 sequence counts

// Literal-only blocks (the context's entropy switch on, a block of at least 13 bytes that the LZ4 compressor stored):
// the same windows as the framing assumes, window w at input offset 4096 w, the last one taking the rest; each becomes
// a Compressed_Block without sequences whose literals are read in place from the input.  Their bodies sit at
// ZE_OFF(4096 w, w) with room for 1.25 x the window + 20 bytes, like any other window's.
ZPB_DEVINL bool ze_lit_only(int entropy, const PackBlock &pb, u32 cs) { return entropy && pb.pad && !cs && pb.len >= 13u; }
ZPB_DEVINL u32 ze_lit_only_end(u32 len, u32 w, u32 nwin) { return w + 1u == nwin ? len : 4096u * (w + 1u); }
static_assert(15u * 5144u + 4096u + 1024u + 20u <= ZE_SLOT && 14u * 5144u + 4107u + 1026u + 20u <= ZE_SLOT,
              "literal-only window bodies fit the block's zstd slot");

// Stage A for window w of block b (t = 16 b + w): the kernel below runs it one thread per window, the CPU emulation in a loop.
ZPB_DEVINL void ze_stage_parse(u64 t, const u8 *lz_slots, const u32 *csize, const PackBlock *blocks, u32 *winop, u32 *meta, u8 *zlit,
                               u64 *zseq, int entropy) {
    const u32 b = (u32)(t >> 4), w = (u32)(t & 15u);
    const u32 cs = csize[b], len = blocks[b].len;
    u32 *m = meta + (u64)b * ZE_META;
    u32 *wo = winop + (u64)b * 17u;
    u32 lit_n = 0, seq_n = ZE_FAIL;
    if (ze_lit_only(entropy, blocks[b], cs)) {
        const u32 nwin = (len - 12u) / 4096u + 1u;
        seq_n = 0;
        if (w < nwin) {
            wo[w] = 4096u * w;
            lit_n = ze_lit_only_end(len, w, nwin) - 4096u * w;
        }
    } else if (blocks[b].pad && cs) {
        const u32 nwin = (len - 12u) / 4096u + 1u;           // as in pack_blocks.cuh (cs != 0 implies len >= 13)
        seq_n = 0;
        if (w < nwin) {
            const u32 begin = wo[w], end = wo[w + 1u];
            const u32 tail_end = w + 1u == nwin ? cs : end;
            if (!(begin <= end && tail_end <= cs && end <= tail_end) ||
                !ze_parse_range(lz_slots + ((u64)b << 16), begin, end, tail_end, zlit + (u64)b * ZE_LITSLOT + ZE_LOFF(begin, w),
                                zseq + t * ZE_WIN_SEQ, ZE_WIN_SEQ, &lit_n, &seq_n))
                seq_n = ZE_FAIL;
        }
    }
    m[16u + w] = lit_n;
    m[32u + w] = seq_n;
}

// Stage C for window w of block b (t = 16 b + w), likewise.
ZPB_DEVINL void ze_stage_encode(u64 t, const u8 *in, const u32 *csize, const PackBlock *blocks, const u32 *winop, u32 *meta, const u8 *zlit,
                                const u64 *zseq, const ZeHuf *hufs, const ZeBlockTabs *tabs, u8 *zslot, int entropy, const ZeTables &T) {
    const u32 b = (u32)(t >> 4), w = (u32)(t & 15u);
    u32 *m = meta + (u64)b * ZE_META;
    u32 z = 0;
    if (ze_lit_only(entropy, blocks[b], csize[b])) {
        const u32 len = blocks[b].len, nwin = (len - 12u) / 4096u + 1u;
        const ZeHuf &H = hufs[b];
        if (!H.desc_len) z = ZE_FAIL;
        else if (w < nwin) {
            const u32 begin = 4096u * w, n = ze_lit_only_end(len, w, nwin) - begin;
            z = ze_emit_range(in + blocks[b].src_off + begin, n, nullptr, 0, ze_lit_mode(w, m + 16u, nwin, H), H,
                              zslot + (u64)b * ZE_SLOT + ZE_OFF(begin, w), n + (n >> 2) + 20u, T, 0, tabs[b]);
        }
    } else if (blocks[b].pad && csize[b]) {
        const u32 nwin = (blocks[b].len - 12u) / 4096u + 1u;
        if (w < nwin) {
            const u32 begin = winop[(u64)b * 17u + w], end = winop[(u64)b * 17u + w + 1u];
            const u32 tail_end = w + 1u == nwin ? csize[b] : end;
            const u32 seq_n = m[32u + w];
            if (seq_n == ZE_FAIL) z = ZE_FAIL;
            else {
                const ZeHuf &H = hufs[b];
                const ZeBlockTabs &B = tabs[b];
                const u32 mode = ze_lit_mode(w, m + 16u, nwin, H);
                const u32 seqmode = ze_seq_mode(w, m + 32u, nwin, B.valid != 0);
                z = ze_emit_range(zlit + (u64)b * ZE_LITSLOT + ZE_LOFF(begin, w), m[16u + w], zseq + t * ZE_WIN_SEQ, seq_n, mode, H,
                                  zslot + (u64)b * ZE_SLOT + ZE_OFF(begin, w), (tail_end - begin) + ((tail_end - begin) >> 2) + 20u, T,
                                  seqmode, B);
            }
        }
    } else if (w == 0) z = ZE_FAIL;
    m[w] = z;
}

#ifndef ZPB_SIM
// Three launches per round, all over the blocks the host marked (PackBlock::pad != 0: they belong to a
// ZPACK_COMPRESSION_ZSTD file).  meta = ZE_META words per block, winop = 17 window offsets per block.
//
// A: one THREAD per 4 KB window of the block compressor (its payload offsets come from lz4_pack_blocks_kernel: winop):
//    the window's LZ4 sequences -> staged literal bytes + sequence records.  Each walk is serial and latency-bound, so the
//    kernel relies on the number of windows in flight (16 per block, every block of the round at once), not on staging.
//    A literal-only block (entropy switch) needs no walk: its windows' offsets go to winop, their sizes to meta.
__global__ void __launch_bounds__(128)
zstd_parse_windows_kernel(const u8 *__restrict__ lz_slots, const u32 *__restrict__ csize, const PackBlock *__restrict__ blocks,
                          u32 *winop, u32 nblocks, u32 *meta, u8 *zlit, u64 *zseq, int entropy) {
    const u64 nwork = (u64)nblocks * 16u;
    for (u64 t = (u64)blockIdx.x * blockDim.x + threadIdx.x; t < nwork; t += (u64)gridDim.x * blockDim.x)
        ze_stage_parse(t, lz_slots, csize, blocks, winop, meta, zlit, zseq, entropy);
}

// B: one warp per block: histograms of the block's staged literals and of its sequence codes in shared memory; lane 0
// builds the Huffman code and the three FSE tables.  A full-alphabet code (entropy switch, literals above 128) is then
// priced window by window by the whole warp, and ze_huf_settle keeps it or not.
__global__ void __launch_bounds__(128)
zstd_huf_tables_kernel(const u8 *__restrict__ in, const PackBlock *__restrict__ blocks, const u32 *__restrict__ csize,
                       const u32 *__restrict__ winop, u32 nblocks, const u32 *__restrict__ meta, const u8 *__restrict__ zlit,
                       const u64 *__restrict__ zseq, ZeHuf *hufs, ZeBlockTabs *tabs, int entropy) {
    __shared__ u32 hist_all[4][256 + 128];
    __shared__ u32 wbits_all[4][16];
    __shared__ u8 lens_all[4][256];
    const u32 lane = threadIdx.x & 31u, wp = threadIdx.x >> 5;
    u32 *hist = hist_all[wp];
    u32 *hll = hist + 256, *hof = hist + 256 + 36, *hml = hist + 256 + 36 + 32;      // 36 + 32 + 53 code counters
    for (u32 b = blockIdx.x * 4u + wp; b < nblocks; b += gridDim.x * 4u) {
        const u32 *m = meta + (u64)b * ZE_META;
        for (u32 i = lane; i < 256 + 128; i += 32) hist[i] = 0;
        __syncwarp();
        u32 total = 0, nseq = 0;
        const bool lit_only = ze_lit_only(entropy, blocks[b], csize[b]);
        const u32 nwin = (blocks[b].len - 12u) / 4096u + 1u;
        const u8 *blk_in = in + blocks[b].src_off, *blk_lit = zlit + (u64)b * ZE_LITSLOT;
        auto lits = [&](u32 w) { const u32 o = winop[(u64)b * 17u + w]; return lit_only ? blk_in + o : blk_lit + ZE_LOFF(o, w); };
        bool ok = blocks[b].pad && (csize[b] || lit_only);
        if (lit_only) {             // the whole block, contiguous in the input: 16-byte loads between the unaligned ends
            const u32 len = blocks[b].len;
            const u32 head = min((16u - (u32)((uintptr_t)blk_in & 15u)) & 15u, len), nv = (len - head) >> 4;
            const uint4 *v = reinterpret_cast<const uint4 *>(blk_in + head);
            for (u32 i = lane; i < head; i += 32) atomicAdd(&hist[blk_in[i]], 1u);
            for (u32 i = lane; i < nv; i += 32) {
                const uint4 x = v[i];
                const u32 wd[4] = {x.x, x.y, x.z, x.w};
#pragma unroll
                for (int k = 0; k < 16; ++k) atomicAdd(&hist[(wd[k >> 2] >> (8 * (k & 3))) & 0xFFu], 1u);
            }
            for (u32 i = head + (nv << 4) + lane; i < len; i += 32) atomicAdd(&hist[blk_in[i]], 1u);
            total = len;
        } else if (ok) {
            for (u32 w = 0; w < nwin; ++w) {
                if (m[32u + w] == ZE_FAIL) { ok = false; break; }
                const u32 n = m[16u + w];
                const u8 *p = lits(w);
                for (u32 i = lane; i < n; i += 32) atomicAdd(&hist[p[i]], 1u);
                total += n;
                const u32 ns = m[32u + w];
                const u64 *q = zseq + ((u64)b * 16u + w) * ZE_WIN_SEQ;
                for (u32 i = lane; i < ns; i += 32) {
                    const u64 r = q[i];
                    atomicAdd(&hll[ze_ll_code((u32)(r & 0xFFFF))], 1u);
                    atomicAdd(&hml[ze_ml_code((u32)((r >> 16) & 0xFFFF))], 1u);
                    atomicAdd(&hof[ze_highbit((u32)(r >> 32))], 1u);
                }
                nseq += ns;
            }
        }
        __syncwarp();
        // four serial builds on four lanes: the three FSE fits run in lockstep, the Huffman code next to them
        const bool fit = ok && nseq >= ZE_TABS_MIN;
        if (lane < 3) {
            ZeBlockTabs &B = tabs[b];
            if (fit) {
                ZeSeqTab &T = lane == 0 ? B.ll : (lane == 1 ? B.of : B.ml);
                ze_fit(T, B.desc[lane], &B.desc_len[lane], lane == 0 ? hll : (lane == 1 ? hof : hml), lane == 0 ? 36 : (lane == 1 ? 32 : 53),
                       nseq, lane == 1 ? 8 : 9);
            }
            if (lane == 0) B.valid = fit ? 1u : 0u;
        } else if (lane == 3) {
            if (ok && total >= 256u) ze_huf_build(hist, hufs[b], entropy != 0, 6u * nwin);
            else { hufs[b].desc_len = 0; hufs[b].carrier = ZE_CARRIER_FIRST; }
        }
        __syncwarp();
        const int settle = __shfl_sync(0xffffffffu, (int)(lane == 3 && hufs[b].desc_len && hufs[b].carrier != ZE_CARRIER_FIRST), 3);
        if (settle) {
            u32 *wbits = wbits_all[wp];
            u8 *lens = lens_all[wp];
            for (u32 i = lane; i < 256; i += 32) lens[i] = hufs[b].len[i];
            __syncwarp();
            for (u32 w = 0; w < nwin; ++w) {
                const u32 n = m[16u + w];
                const u8 *p = lits(w);
                u32 bits = 0;
                for (u32 i = lane; i < n; i += 32) bits += lens[p[i]];
                for (int d = 16; d; d >>= 1) bits += __shfl_xor_sync(0xffffffffu, bits, d);
                if (lane == 0) wbits[w] = bits;
            }
            __syncwarp();
            if (lane == 0) ze_huf_settle(hufs[b], m + 16u, wbits, nwin);
        }
        __syncwarp();
    }
}

// C: one thread per window again: the window's sub-block body.  meta[w]: body size (0: none, ZE_FAIL: the
// block is stored raw).  A literal-only block without a table is stored without encoding anything.
__global__ void __launch_bounds__(128)
zstd_encode_windows_kernel(const u8 *__restrict__ in, const u32 *__restrict__ csize, const PackBlock *__restrict__ blocks,
                           const u32 *__restrict__ winop, u32 nblocks, u32 *meta, const u8 *__restrict__ zlit, const u64 *__restrict__ zseq,
                           const ZeHuf *__restrict__ hufs, const ZeBlockTabs *__restrict__ tabs, u8 *zslot, int entropy) {
    __shared__ ZeTables T;
    if (threadIdx.x == 0) ze_build_tables(T);
    __syncthreads();
    const u64 nwork = (u64)nblocks * 16u;
    for (u64 t = (u64)blockIdx.x * blockDim.x + threadIdx.x; t < nwork; t += (u64)gridDim.x * blockDim.x)
        ze_stage_encode(t, in, csize, blocks, winop, meta, zlit, zseq, hufs, tabs, zslot, entropy, T);
}
#endif
