// lz4_fast.cuh — the throughput path for LZ4 entries: scan -> parse -> execute (kernels K0/K1/K2).
//
// Same contract as the LZ4 arm of zpack_read_file (/root/reference/lib/zpack_read.c:396-468:
// LZ4F_decompress loop, then XXH3_64bits over uncomp_size bytes), split so that the one
// inherently serial part of LZ4 — finding where each sequence starts — costs a thread, not a warp:
//
//   K0 scan   one thread per entry   frame header (lz4frame.c:1113-1205) + block-header chain
//                                    (lz4frame.c:1503-1531) -> a table of blocks.
//   K1 parse  one thread per block   walks token / length / offset bytes only (the control half of
//                                    LZ4_decompress_generic, lz4.c:1797-2151), validates them, and
//                                    emits one 32-bit descriptor per sequence:
//                                    token position | output position << 16 (both block-relative).
//                                    The compressed stream is staged per lane through shared memory
//                                    with cp.async (LDGSTS), four 64-byte chunks ahead of the cursor,
//                                    so the serial walk never waits on HBM.
//   K2 exec   one warp per entry     32 sequences at a time, one per lane.  The compressed bytes come through a
//                                    per-warp cp.async staging ring; literals and short non-overlapping matches are
//                                    copied one lane per sequence (word-wise, lane_copy), long / periodic ones by the
//                                    whole warp in 16-byte units (coop_match); matches that source an earlier match of
//                                    the same step are redirected through its offset (pointer jumping) so that they
//                                    read final bytes; far matches are fetched from flushed output with cp.async.
//                                    Output is assembled in a 4 KiB shared-memory ring per warp; each finished 1 KiB
//                                    goes out as 16-byte coalesced stores and is folded into XXH3-64 from the same
//                                    registers (the digest never re-reads HBM).
//
// K2 does not wait for K1: K0 sorts blocks into three work lists by weight, K1 (high-priority stream) walks the heavy
// list on its first CTAs and publishes each verdict behind a fence, K2 (three launches over one work queue, see
// zpb_api.cu) starts on the entries that are parsed at once and puts aside what is not parsed yet.
//
// K0/K1 only ACCEPT: anything unusual (checksummed or multi-frame entries, > 64 KB blocks, any
// malformed byte, sizes that do not add up) is handed to the general decoder in lz4_decode.cuh,
// which reproduces the reference's exact error classes.  The fast path therefore only ever
// reports OK or HASH_MISMATCH.
#pragma once
#include "common.cuh"
#include "xxh3.cuh"
#include "lz4_decode.cuh"
#include "ptx.cuh"

#define FAST_RING      4096u
#define FAST_RMASK     4095u
#define FAST_LONG      32u     // lit or match >= this: executed cooperatively by the whole warp
#ifndef FAST_SCR
#define FAST_SCR       80u     // per-lane staging for a far match: 5 x 16 B cover 15 + 64 bytes
#define FAST_ST        64u     // far matches up to this length are staged (cp.async from L2)
#define CR_SIZE        2048u   // per-warp staging ring for the compressed stream
#define CR_ROW         512u    // one fill: 16 bytes per lane
#endif
#define CR_MASK        (CR_SIZE - 1u)
#define FAST_WARP_SMEM (FAST_RING + 32u * FAST_SCR + CR_SIZE + 32u)   // + 32: lane_copy's whole-word over-reads past the staging ring stay inside the warp's own region
#ifndef FAST_EXEC_WARPS
#define FAST_EXEC_WARPS 8u
#endif
#define FAST_EXEC_SMEM (FAST_EXEC_WARPS * FAST_WARP_SMEM + 48u)   // per CTA, plus slack at both ends
// the invariants the copies rely on, whatever the overridable sizes are set to
static_assert(FAST_SCR % 16u == 0 && FAST_SCR >= 15u + FAST_ST + 1u, "a staged far match (<= FAST_ST bytes at any 16-byte phase) fits its scratch");
static_assert((CR_SIZE & (CR_SIZE - 1u)) == 0 && CR_ROW == 32u * 16u && CR_SIZE % CR_ROW == 0, "staging ring: power of two, rows of 16 bytes per lane");
static_assert(FAST_WARP_SMEM - (FAST_RING + 32u * FAST_SCR + CR_SIZE) >= 32u, "lane_copy reads up to four whole words past a range: 32 bytes of padding per warp");
static_assert((FAST_RING & FAST_RMASK) == 0 && FAST_RING % 1024u == 0, "output ring: power of two, flushed in KiB units");

#define FE_DONE    0u   // status already final (guards, unsupported method)
#define FE_FAST    1u   // block table filled, goes through K1/K2
#define FE_GENERAL 2u   // handed to the general kernel
#define FE_ZSTD    3u   // handed to the zstd kernel (zstd_decode.cuh)

#define FAST_DESC_PER_BLOCK 2060ull
#define K1_HEAVY   (24u << 10)   // compressed block bytes: heavy / medium / light parse work lists
#define K1_MEDIUM  (6u << 10)

#define FB_STORED  1u
#define FB_BAD     2u
#define FB_PARSED  4u

// Internal to the library (never in an archive: comp_method is a u8): one raw LZ4 block of a
// block-independent frame, decoded as a pseudo-entry by the block-sharded path (zpb_unpack_blocks_device).
// zpb_entry.reserved = index of the block's first KiB in the per-KiB XXH3 stripe-sum array; such
// "partial" entries emit stripe sums instead of a digest (the chain is run by xxh3_chain_kernel).
#define ZPB_M_LZ4_BLOCK   0x102u
#define ZPB_F_STORED_BLK  0x100u
#define FE_LINK_NONE    0u
#define FE_LINK_WINDOW  1u   // blocks of the frame share the 64 KB window (B.Indep = 0)
#define FE_LINK_PARTIAL 2u   // pseudo-entry of the block-sharded path

struct FastAux {      // host -> device, per entry
    u64 desc_base;    // first descriptor slot of this entry (multiple of 4)
    u32 slot_base;    // first FastBlock slot
    u32 nslots;
};
struct FastEntry {    // K0 -> K2
    u32 first_slot, nblocks, state, linked;
};
struct FastBlock {    // K0 -> K1 -> K2, 32 bytes
    u64 src;          // archive offset of the block payload
    u64 desc_off;     // index of its first descriptor (multiple of 4)
    u32 bsz;          // payload bytes
    u32 flags;        // FB_*
    u32 nseq;         // K1
    u32 out_size;     // K1 (stored: = bsz)
};

// Host: the fast path's scratch of entry e, placed at the running totals `slots` (FastBlock slots) and `ndesc` (descriptor
// words), which grow by what it needs.  An LZ4 frame gets a slot per 64 KB block plus two, and per block FAST_DESC_PER_BLOCK
// words on top of one per 3 payload bytes (fast_scan_lz4 places block b's descriptors there); an entry the fast path
// does not take gets nothing.
inline FastAux fast_entry_layout(const zpb_entry &e, u64 &slots, u64 &ndesc) {
    u32 ns = 0; u64 nd = 0;
    if (e.uncomp_size < 0x7fffffffull && e.comp_size) {
        if (e.method == ZPB_METHOD_NONE) ns = 1;
        else if (e.method == ZPB_M_LZ4_BLOCK) {
            ns = 1;
            nd = ((e.comp_size / 3 + FAST_DESC_PER_BLOCK + 20) + 3) & ~3ull;
        } else if (e.method == ZPB_METHOD_LZ4) {
            ns = (u32)(e.uncomp_size >> 16) + 2;
            nd = ((e.comp_size / 3 + FAST_DESC_PER_BLOCK * ns + 8) + 3) & ~3ull;
        }
    }
    FastAux a;
    a.desc_base = ndesc; a.slot_base = (u32)slots; a.nslots = ns;
    slots += ns; ndesc += nd;
    return a;
}

// ------------------------------------------------------------------------------------------ K0
// Returns true when the entry has the shape the fast path handles and the block table is filled.
__device__ __noinline__ bool fast_scan_lz4(const u8 *src, u64 n, const zpb_entry &e, const FastAux &a,
                                           FastEntry &f, FastBlock *fb) {
    if (n < 11 || e.uncomp_size >= 0x7fffffffull) return false;
    if (ld32u(src) != LZ4F_MAGIC) return false;
    u32 flg = ld8(src + 4);
    if (((flg >> 1) & 1) || ((flg >> 6) & 3) != 1) return false;
    bool indep = (flg >> 5) & 1, bsum = (flg >> 4) & 1, has_size = (flg >> 3) & 1, csum = (flg >> 2) & 1,
         has_dict = flg & 1;
    if (bsum || csum) return false;
    u32 hsize = 7 + (has_size ? 8 : 0) + (has_dict ? 4 : 0);
    if (n < (u64)hsize + 4) return false;
    u32 bd = ld8(src + 5);
    if ((bd >> 7) || ((bd >> 4) & 7) != 4 || (bd & 15)) return false;  // 64 KB blocks only
    if (((xxh32_dev(src + 4, hsize - 5, 0) >> 8) & 0xFF) != ld8(src + hsize - 1)) return false;
    if (has_size && ld64u(src + 6) != e.uncomp_size) return false;
    u64 ip = hsize;
    u32 nb = 0;
    for (;;) {
        if (n - ip < 4) return false;
        u32 bh = ld32u(src + ip);
        ip += 4;
        if (bh == 0) break;
        u32 bsz = bh & 0x7FFFFFFFu;
        if (bsz == 0 || bsz > 65536u || bsz > n - ip || nb == a.nslots) return false;
        FastBlock b;
        b.src = e.src_off + ip;
        b.desc_off = a.desc_base + (((ip / 3) + FAST_DESC_PER_BLOCK * nb + 3ull) & ~3ull);
        b.bsz = bsz;
        b.flags = (bh >> 31) ? FB_STORED : 0u;
        b.nseq = 0;
        b.out_size = (bh >> 31) ? bsz : 0u;
        fb[a.slot_base + nb] = b;
        ip += bsz;
        ++nb;
    }
    if (ip != n) return false;  // trailing bytes: another frame or garbage -> general path decides
    f.nblocks = nb;
    f.linked = indep ? 0u : 1u;
    return true;
}

__global__ void __launch_bounds__(256)
lz4_fast_scan_kernel(const u8 *__restrict__ archive, u64 asz, const zpb_entry *__restrict__ entries,
                     const u32 *__restrict__ order, u32 n, const FastAux *__restrict__ aux, FastEntry *fe,
                     FastBlock *fb, u32 *parse_list, u32 plist_cap, u32 *counters, u32 *general_list, u32 *zstd_list,
                     int *status, u64 *digest) {
    u32 t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= n) return;
    u32 idx = order ? order[t] : t;
    const zpb_entry e = entries[idx];
    const FastAux a = aux[idx];
    FastEntry f;
    f.first_slot = a.slot_base; f.nblocks = 0; f.state = FE_DONE; f.linked = 0;
    int st = ST_OK;
    if (e.comp_size == 0) {
        st = ST_OK;                                            // zpack_read.c:328
    } else if (e.dst_cap < e.uncomp_size) {
        st = ST_TOO_SMALL;                                     // :329
    } else if (e.src_off > asz || e.comp_size > asz - e.src_off) {
        st = ST_OFFSET_INVALID;                                // memory-safety form of :331
    } else if (e.method == ZPB_METHOD_NONE) {                  // :352-368 — one stored "block"
        if (e.uncomp_size > e.comp_size) st = ST_SIZE_INVALID;
        else if (e.uncomp_size >= 0x7fffffffull || a.nslots == 0) f.state = FE_GENERAL;
        else {
            FastBlock b;
            b.src = e.src_off; b.desc_off = a.desc_base; b.bsz = (u32)e.uncomp_size;
            b.flags = FB_STORED; b.nseq = 0; b.out_size = (u32)e.uncomp_size;
            fb[a.slot_base] = b;
            f.nblocks = 1;
            f.state = FE_FAST;
        }
    } else if (e.method == ZPB_METHOD_LZ4) {
        f.state = fast_scan_lz4(archive + e.src_off, e.comp_size, e, a, f, fb) ? FE_FAST : FE_GENERAL;
    } else if (e.method == ZPB_M_LZ4_BLOCK) {                  // one block of an indexed frame (lz4frame.c:1503-1531 done on the host)
        if (e.comp_size > 65536u || e.uncomp_size > 65536u || a.nslots == 0) st = ST_NOT_AVAILABLE;
        else {
            const bool stored = (e.flags & ZPB_F_STORED_BLK) != 0;
            FastBlock b;
            b.src = e.src_off; b.desc_off = a.desc_base; b.bsz = (u32)e.comp_size;
            b.flags = stored ? FB_STORED : 0u; b.nseq = 0; b.out_size = stored ? (u32)e.comp_size : 0u;
            fb[a.slot_base] = b;
            f.nblocks = 1;
            f.linked = FE_LINK_PARTIAL;
            f.state = FE_FAST;
        }
    } else if (e.method == ZPB_METHOD_ZSTD) {
        f.state = FE_ZSTD;                                     // guards passed: the zstd kernel decodes it
    } else {
        f.state = FE_GENERAL;                                  // unknown method: the general kernel answers
    }
    if (f.state == FE_DONE) {
        status[idx] = st;
        digest[idx] = 0;
    } else if (f.state == FE_GENERAL) {
        general_list[atomicAdd(&counters[CNT_GENERAL], 1u)] = idx;
    } else if (f.state == FE_ZSTD) {
        zstd_list[atomicAdd(&counters[CNT_ZSTD], 1u)] = idx;
    } else {
        for (u32 b = 0; b < f.nblocks; ++b)
            if (!(fb[a.slot_base + b].flags & FB_STORED))
            {
                // three work lists by weight (compressed bytes ~ sequences to walk): the parse kernel hands the heavy
                // list to its first CTAs, so that the CTAs holding light blocks retire early and make room for K2
                const u32 bz = fb[a.slot_base + b].bsz;
                const u32 cls = bz >= K1_HEAVY ? 0u : bz >= K1_MEDIUM ? 1u : 2u;
                // one atomic per class and warp, not per block
                const u32 peers = __match_any_sync(__activemask(), cls);
                const int leader = __ffs(peers) - 1;
                u32 base = 0;
                if ((int)(threadIdx.x & 31) == leader) base = atomicAdd(&counters[CNT_PARSE_HEAVY + cls], (u32)__popc(peers));
                base = __shfl_sync(peers, base, leader);
                parse_list[(u64)cls * plist_cap + base + __popc(peers & ((1u << (threadIdx.x & 31)) - 1u))] = a.slot_base + b;
            }
    }
    fe[idx] = f;
}

// Warp-lockstep copy inside shared memory: every lane moves its own n bytes (0 = idle) from s to d, any
// alignment, ranges not overlapping.  Head bytes up to the destination's word boundary, then whole words
// assembled from two aligned source words with a funnel shift, then tail bytes: 4 instructions per word
// instead of 12 per 4 bytes of a byte loop.  The source words may straddle bytes outside [s, s+n) (and the
// last round may read up to four words past it): they are read, never stored.
ZPB_DEVINL void lane_copy(u32 s, u32 d, u32 n) {   // idle lanes: n = 0 (s, d are not dereferenced)
    u32 h = (0u - d) & 3u;
    h = h < n ? h : n;
    const u32 n2 = n - h;
    const u32 nw = n2 >> 2, t = n2 & 3u;
    const u32 s2 = s + h, d2 = d + h;            // d2 is word aligned whenever nw > 0
    const u32 ts = s2 + 4 * nw, td = d2 + 4 * nw;
    // edge bytes (<= 3 before the first whole word, <= 3 after the last): predicated, no branches
#ifdef ZPB_SIM
    copy_edges_ss(h, t, s, d, ts, td);
#else
    asm volatile(
        "{\n\t"
        ".reg .pred p0, p1, p2, q0, q1, q2;\n\t"
        ".reg .b32 a0, a1, a2, b0, b1, b2;\n\t"
        "setp.gt.u32 p0, %0, 0;\n\t"
        "setp.gt.u32 p1, %0, 1;\n\t"
        "setp.gt.u32 p2, %0, 2;\n\t"
        "setp.gt.u32 q0, %1, 0;\n\t"
        "setp.gt.u32 q1, %1, 1;\n\t"
        "setp.gt.u32 q2, %1, 2;\n\t"
        "@p0 ld.shared.u8 a0, [%2];\n\t"
        "@p1 ld.shared.u8 a1, [%2+1];\n\t"
        "@p2 ld.shared.u8 a2, [%2+2];\n\t"
        "@q0 ld.shared.u8 b0, [%4];\n\t"
        "@q1 ld.shared.u8 b1, [%4+1];\n\t"
        "@q2 ld.shared.u8 b2, [%4+2];\n\t"
        "@p0 st.shared.u8 [%3], a0;\n\t"
        "@p1 st.shared.u8 [%3+1], a1;\n\t"
        "@p2 st.shared.u8 [%3+2], a2;\n\t"
        "@q0 st.shared.u8 [%5], b0;\n\t"
        "@q1 st.shared.u8 [%5+1], b1;\n\t"
        "@q2 st.shared.u8 [%5+2], b2;\n\t"
        "}" ::"r"(h), "r"(t), "r"(s), "r"(d), "r"(ts), "r"(td) : "memory");
#endif
    const u32 maxnw = __reduce_max_sync(0xffffffffu, nw);
    const u32 sw = s2 & ~3u, sh = (s2 & 3u) << 3;
    for (u32 kb = 0; kb < maxnw; kb += 4) {      // four whole words per round
        const u32 rem = nw > kb ? nw - kb : 0u;
        const u32 sa = sw + 4 * kb, da = d2 + 4 * kb;
        u32 a0 = 0, a1 = 0, a2 = 0, a3 = 0, a4 = 0;
#ifdef ZPB_SIM
        if (rem > 0) { a0 = lds32_loose(sa); a1 = lds32_loose(sa + 4); a2 = lds32_loose(sa + 8); a3 = lds32_loose(sa + 12); a4 = lds32_loose(sa + 16); }
#else
        asm volatile(
            "{\n\t"
            ".reg .pred p;\n\t"
            "setp.gt.u32 p, %5, 0;\n\t"
            "@p ld.shared.u32 %0, [%6];\n\t"
            "@p ld.shared.u32 %1, [%6+4];\n\t"
            "@p ld.shared.u32 %2, [%6+8];\n\t"
            "@p ld.shared.u32 %3, [%6+12];\n\t"
            "@p ld.shared.u32 %4, [%6+16];\n\t"
            "}" : "+r"(a0), "+r"(a1), "+r"(a2), "+r"(a3), "+r"(a4) : "r"(rem), "r"(sa) : "memory");
#endif
        const u32 w0 = __funnelshift_r(a0, a1, sh), w1 = __funnelshift_r(a1, a2, sh),
                  w2 = __funnelshift_r(a2, a3, sh), w3 = __funnelshift_r(a3, a4, sh);
#ifdef ZPB_SIM
        if (rem > 0) sts32(da, w0);
        if (rem > 1) sts32(da + 4, w1);
        if (rem > 2) sts32(da + 8, w2);
        if (rem > 3) sts32(da + 12, w3);
#else
        asm volatile(
            "{\n\t"
            ".reg .pred p0, p1, p2, p3;\n\t"
            "setp.gt.u32 p0, %0, 0;\n\t"
            "setp.gt.u32 p1, %0, 1;\n\t"
            "setp.gt.u32 p2, %0, 2;\n\t"
            "setp.gt.u32 p3, %0, 3;\n\t"
            "@p0 st.shared.u32 [%1], %2;\n\t"
            "@p1 st.shared.u32 [%1+4], %3;\n\t"
            "@p2 st.shared.u32 [%1+8], %4;\n\t"
            "@p3 st.shared.u32 [%1+12], %5;\n\t"
            "}" ::"r"(rem), "r"(da), "r"(w0), "r"(w1), "r"(w2), "r"(w3) : "memory");
#endif
    }
}

// ------------------------------------------------------------------------------------------ K1
#define K1_THREADS 256
#define K1_ROW     272u   // 256-byte staging ring per lane + 16 bytes of bank skew
#ifndef K1_TOPUP
#define K1_TOPUP   8u     // sequences between two warp-wide top-ups of the staging rings
#endif

// Per-lane view of one block's compressed bytes through a 256-byte staging ring (4 chunks of 64 bytes, cp.async).
// Positions are "ring coordinates" q = block position + skew, so that q & 255 is both the ring slot and the low byte of
// the global address (16-byte alignment of every cp.async piece follows).  The ring is refilled by `topup`, which the
// whole warp executes at once every K1_TOPUP sequences: it first waits for everything requested so far — a group that
// was issued one top-up (hundreds of cycles) earlier, so the wait is normally free — and then requests the chunks up to
// three ahead of the cursor.  In between, a lane may read below `avail` without waiting; a lane that gets ahead of its
// staged data (a long literal run) refills by itself and waits (`need`).
struct LaneStage {
    const u8 *gbase;     // global address of ring coordinate 0 (256-byte aligned; may precede the block)
    const u8 *glo, *ghi; // readable range of the archive
    u32 row_s;           // this lane's ring, shared-window address
    u32 nreq;            // chunks [.., nreq) have been requested
    u32 avail;           // ring coordinates below this are complete (chunks below avail >> 6)
    u32 klo, khi;        // chunks in [klo, khi) lie wholly inside the archive

    ZPB_DEVINL u32 open(const u8 *archive, u64 asz, u64 src, u32 row_shared) {
        const u8 *p = archive + src;
        u32 skew = (u32)((uintptr_t)p & 255u);
        gbase = p - skew;
        glo = archive; ghi = archive + asz;
        row_s = row_shared;
        nreq = 0; avail = 0;
        klo = gbase >= glo ? 0u : (u32)((glo - gbase + 63) >> 6);
        u64 span = (u64)(ghi - gbase) >> 6;
        khi = span > 0x7fffffffull ? 0x7fffffffu : (u32)span;
        return skew;
    }
    ZPB_DEVINL void request(u32 k) {
        const u8 *g = gbase + ((u64)k << 6);
        const u32 s = row_s + ((k << 6) & 255u);
        if (k >= klo && k < khi) { cp_async64_if(true, s, g); return; }
#pragma unroll 1
        for (u32 j = 0; j < 4; ++j) {           // a chunk that straddles an end of the archive
            const u8 *gj = g + 16 * j;
            if (gj + 16 > glo && gj < ghi) {
                if (gj >= glo) {
                    u64 left = (u64)(ghi - gj);
                    cp_async16(s + 16 * j, gj, left < 16 ? (u32)left : 16u);
                } else {
                    for (u32 b = 0; b < 16; ++b) if (gj + b >= glo && gj + b < ghi) sts8(s + 16 * j + b, gj[b]);
                }
            }
        }
    }
    // whole warp, converged; idle lanes pass q with nothing open (act = false)
    ZPB_DEVINL void topup(bool act, u32 q) {
        cp_async_wait_all();
        avail = nreq << 6;
        const u32 c = q >> 6;
        u32 lo = nreq > c ? nreq : c;
        if (!act) lo = 0xfffffff0u;
#pragma unroll
        for (u32 j = 0; j < 4; ++j) {
            const u32 k = lo + j;
            const bool want = act && k < c + 4;
            const bool whole = want && k >= klo && k < khi;
            cp_async64_if(whole, row_s + ((k << 6) & 255u), gbase + ((u64)k << 6));
            if (want && !whole) request(k);
        }
        cp_async_commit();
        if (act && c + 4 > nreq) nreq = c + 4;
    }
    // this lane alone: make ring coordinates [.., hi) readable (hi - (q & ~63) <= 256 is the caller's business)
    ZPB_DEVINL void need(u32 q, u32 hi) {
        if (hi <= avail) return;
        cp_async_wait_all();                     // nothing may be in flight towards a slot that is requested again
        const u32 c = q >> 6;
        u32 lo = nreq > c ? nreq : c;
        for (u32 k = lo; k < c + 4; ++k) request(k);
        cp_async_commit();
        cp_async_wait_all();
        nreq = c + 4;
        avail = nreq << 6;
    }
    ZPB_DEVINL u32 rd(u32 q) const { return lds8(row_s + (q & 255u)); }
};

// One parse kernel, two shapes.  J = 1: a lane walks a whole block (light blocks: nothing to gain from splitting).
// J = 4: the four lanes of a group walk the four quarters of one block at the same time, which cuts the serial walk of
// a heavy block — the floor of this kernel, whatever the batch size — to a quarter.  Lane 0 starts at the block's
// first token; lanes 1-3 start at byte j * bsz / 4, which is almost never a token.  LZ4 token streams re-synchronise:
// a walk that starts on an arbitrary byte lands on a true sequence boundary within a few sequences and stays on the true
// chain from there.  So each lane keeps walking past the start of the next quarter until it stands on a position the
// next lane has also visited (a merge over the next lane's descriptor list, two pointers): from that JOIN on the next
// lane's list is the truth, and everything the next lane emitted before it is discarded.  Output positions of a
// speculative lane are relative to its own start; the join fixes the base (all arithmetic mod 2^16 for the 16-bit
// descriptor field, in full precision for the block's decoded size).  A lane that does not join within K1_MERGE_MAX
// sequences, or a speculative walk that runs off the block, hands the block to the unsplit kernel, which walks it again
// from its first byte.  When the four lanes of a block have finished, the warp moves the valid parts of segments 1-3
// down behind segment 0 (output positions made absolute), so that K2 sees one flat descriptor list per block.
#ifndef K1_MERGE_MAX
#define K1_MERGE_MAX 384u
#endif
#define K1_SEG_SLACK 512u     // descriptor slots per segment beyond (compressed bytes / 3): the overrun until the join (+ a shifted second start)

// where segment j's walk starts (attempt 1 shifts the speculative starts: a second try after a failed join)
ZPB_DEVINL u32 k1_seg_start(u32 bsz, u32 j, u32 J, u32 attempt = 0) {
    return J == 1 || j == 0 ? 0u : (u32)(((u64)bsz * j) / J) + 89u * attempt * j;
}
ZPB_DEVINL u32 k1_seg_desc(u32 bsz, u32 j, u32 J) {   // first descriptor slot of segment j (multiple of 4)
    return J == 1 ? 0u : ((k1_seg_start(bsz, j, J) / 3u + K1_SEG_SLACK * j) + 3u) & ~3u;
}

#ifdef ZPB_SIM
#define K1_WHY(code) do { if (getenv("SIM_K1_WHY")) fprintf(stderr, "sim: k1 slot %u seg %u: %s (q %u qstop %u qend %u nseq %u mptr %u msteps %u)\n", slot, sj, code, q - skew, qstop - skew, qend - skew, nseq, mptr, msteps); } while (0)
#else
#define K1_WHY(code) do { } while (0)
#endif
#define K1M_WALK  0u
#define K1M_MERGE 1u
#define K1M_DONE  2u   // joined (or, last segment, reached the block's end cleanly)
#define K1M_FAIL  3u

template <int J>
ZPB_DEVINL void
lz4_fast_parse_body(const u8 *__restrict__ archive, u64 asz, FastBlock *fb, u32 *parse_list,
                    u32 plist_cap, u32 *counters, u32 *work_counter, u32 *desc, u32 all_lists) {
    // J = 4 walks the heavy list, then the medium one; J = 1 the light one — or, when the batch is so large that even
    // unsplit walks fill the GPU (all_lists bit 0: the host decides), all three, heavy first (K0 sorts blocks by compressed
    // size).  With the split walk the light list is parsed FIRST (bit 2: remember its length in CNT_LIGHT_FIRST) so that the
    // execute kernel has entries to start on, and the blocks the split walk gives back, which it appends to the light
    // list, are walked by a last launch (bit 1: only the items from CNT_LIGHT_FIRST on).
    const u32 n_heavy = (J == 4 || (all_lists & 1u)) ? counters[CNT_PARSE_HEAVY] : 0u;
    const u32 n_medium = (J == 4 || (all_lists & 1u)) ? counters[CNT_PARSE_MEDIUM] : 0u;
    const u32 light_skip = (J == 1 && (all_lists & 2u)) ? counters[CNT_LIGHT_FIRST] : 0u;
    const u32 nitems = J == 4 ? n_heavy + n_medium : n_heavy + n_medium + counters[CNT_PARSE_LIGHT] - light_skip;
    if (J == 1 && (all_lists & 4u) && blockIdx.x == 0 && threadIdx.x == 0) counters[CNT_LIGHT_FIRST] = counters[CNT_PARSE_LIGHT];
    ZPB_DYN_SMEM(k1_smem);
    const u32 lane = threadIdx.x & 31u;
    const u32 sj = lane & (J - 1);                 // this lane's segment
    const u32 row_s = smem_window(k1_smem) + threadIdx.x * K1_ROW;
    const u32 ngroups = gridDim.x * blockDim.x / J;
    const u32 gmask = J == 1 ? (1u << lane) : (0xFu << (lane & ~3u));   // the lanes of this lane's group
    bool active = false, exhausted = false, first = true;
    LaneStage sg;
    sg.gbase = archive; sg.glo = archive; sg.ghi = archive + asz; sg.row_s = row_s; sg.nreq = sg.avail = sg.klo = sg.khi = 0;
    // all positions below are ring coordinates (block position + skew)
    u32 slot = 0, skew = 0, qend = 0, qstop = 0, q = 0, op = 0, nseq = 0, last_ms = 0, mode = K1M_DONE;
    u32 mptr = 0, msteps = 0, jtok = 0, jop = 0, bszv = 0, attempt = 0;
    bool had_match = false;
    u32 b0 = 0, b1 = 0, b2 = 0, b3 = 0;
    u32 *dout = nullptr;     // this segment's descriptor region
    u32 it = 0;

    for (;;) {
        // ---- groups whose lanes are all idle take the next block
        const u32 idle = __ballot_sync(0xffffffffu, !active);
        u32 gidle = idle;                                  // bit g*J set: group g idle
        if (J == 4) { gidle &= gidle >> 1; gidle &= gidle >> 2; gidle &= 0x11111111u; }
        if (gidle) {
            if (!exhausted) {
                // first item: by position in the grid (the heavy end of the list lands on the first CTAs); afterwards
                // from the shared counter, which starts behind the statically dealt items
                const u32 ng = (u32)__popc(gidle);
                u32 base;
                if (first) {
                    base = (blockIdx.x * blockDim.x + (threadIdx.x & ~31u)) / J;
                    first = false;
                } else {
                    base = 0;
                    const int leader = __ffs(gidle) - 1;
                    if ((int)lane == leader) base = atomicAdd(work_counter, ng);
                    base = __shfl_sync(0xffffffffu, base, leader) + ngroups;
                }
                if (base + ng > nitems) exhausted = true;
                if ((gidle >> (lane & ~(J - 1))) & 1u) {
                    const u32 w = base + (u32)__popc(gidle & ((1u << (lane & ~(J - 1))) - 1u));
                    if (w < nitems) {
                        slot = w < n_heavy ? parse_list[w]
                             : w < n_heavy + n_medium ? parse_list[(u64)plist_cap + (w - n_heavy)]
                                                      : parse_list[2ull * plist_cap + (w - n_heavy - n_medium + light_skip)];
                        const FastBlock B = fb[slot];
                        bszv = B.bsz;
                        skew = sg.open(archive, asz, B.src, row_s);
                        qend = B.bsz + skew;
                        q = skew + k1_seg_start(B.bsz, sj, J);
                        qstop = sj + 1 < J ? skew + k1_seg_start(B.bsz, sj + 1, J) : qend;
                        dout = desc + B.desc_off + k1_seg_desc(B.bsz, sj, J);
                        op = 0; nseq = 0; last_ms = 0; had_match = false;
                        mode = K1M_WALK; mptr = 0; msteps = 0; jtok = 0; jop = 0; attempt = 0;
                        active = true;
                        sg.need(q, q + 1);       // the first four chunks, waited for
                    }
                }
            }
            if (__ballot_sync(0xffffffffu, active) == 0) break;
        }
        if ((it++ % K1_TOPUP) == 0) sg.topup(active && mode < K1M_DONE, q);   // warp-uniform

        // ---- a lane that has passed the start of the next quarter looks for its position in the next lane's list
        if (J == 4) {
            const bool merging = active && mode == K1M_MERGE;
            if (__any_sync(0xffffffffu, merging)) {
                __syncwarp();                                                   // the next lane's descriptor stores
                const u32 nx_n = __shfl_down_sync(0xffffffffu, nseq, 1);
                const u32 nx_mode = __shfl_down_sync(0xffffffffu, mode, 1);
                if (merging) {
                    const u32 *nd = desc + fb[slot].desc_off + k1_seg_desc(bszv, sj + 1, J);
                    const u32 avail_n = nx_mode >= K1M_DONE ? nx_n : nx_n & ~3u;   // descriptors of the next lane that are in memory
                    const u32 tq = q - skew;
                    u32 dv = 0xFFFFFFFFu;
                    while (mptr < avail_n && ((dv = __ldcg(nd + mptr)) & 0xFFFFu) < tq) ++mptr;
                    if (mptr < avail_n && (dv & 0xFFFFu) == tq) {
                        mode = K1M_DONE; jtok = tq; jop = dv >> 16;             // joined: the next lane's list is valid from mptr on
                        const u32 r = nseq & 3u;                                // descriptors still in the shift register
                        if (r == 1) dout[nseq - 1] = b3;
                        else if (r == 2) { dout[nseq - 2] = b2; dout[nseq - 1] = b3; }
                        else if (r == 3) { dout[nseq - 3] = b1; dout[nseq - 2] = b2; dout[nseq - 1] = b3; }
                    } else if (nx_mode == K1M_FAIL || (mptr >= avail_n && nx_mode >= K1M_DONE) || ++msteps > K1_MERGE_MAX) {
                        K1_WHY(nx_mode == K1M_FAIL ? "next lane failed" : msteps > K1_MERGE_MAX ? "merge timeout" : "next list exhausted");
                        mode = K1M_FAIL;
                    }
                }
            }
        }
        // ---- block verdict, when every lane of a group has finished (warp-uniform: the shuffles need every lane)
        if (J == 4) {
            const u32 fin_mask = __ballot_sync(0xffffffffu, !active || mode >= K1M_DONE);
            const bool gdone = active && (fin_mask & gmask) == gmask;
            if (__any_sync(0xffffffffu, gdone)) {
                const u32 g0 = lane & ~3u;
                u32 ok = mode == K1M_DONE ? 1u : 0u;
                ok &= __shfl_xor_sync(0xffffffffu, ok, 1);
                ok &= __shfl_xor_sync(0xffffffffu, ok, 2);
                // bases: base_0 = 0, base_{j+1} = (base_j + op_j at the join) - (the next lane's relative position there)
                const u32 delta = op - jop;
                u32 base = 0;
#pragma unroll
                for (u32 kk = 1; kk < 4; ++kk) {
                    const u32 pb_ = __shfl_sync(0xffffffffu, base, g0 + kk - 1), pd = __shfl_sync(0xffffffffu, delta, g0 + kk - 1);
                    if (sj == kk) base = pb_ + pd;
                }
                const u32 pfirst = __shfl_up_sync(0xffffffffu, mptr, 1);      // where the previous lane joined this lane's list
                const u32 firstv = sj == 0 ? 0u : pfirst;
                const u32 cnt = nseq > firstv ? nseq - firstv : 0u;
                u32 total = cnt;
                total += __shfl_xor_sync(0xffffffffu, total, 1);
                total += __shfl_xor_sync(0xffffffffu, total, 2);
                // decoded size = the last lane's end, in full precision: bases are known mod 2^16 only, so it is the previous
                // lane's join (an absolute position below 2^16) plus what the last lane has produced since (below 2^16)
                const u32 abs_join = base + op;
                const u32 pj = __shfl_up_sync(0xffffffffu, abs_join, 1), pjop = __shfl_up_sync(0xffffffffu, jop, 1);
                const u32 out_size = __shfl_sync(0xffffffffu, (pj & 0xFFFFu) + ((op - pjop) & 0xFFFFu), g0 + 3);
                // ---- one flat list per block: the valid part of segments 1..3 moves down behind segment 0 (in place: the
                // destination is always below the source), output positions made absolute on the way.  All 32 lanes copy,
                // one finished group at a time.
                const u32 srcv = k1_seg_desc(bszv, sj, J) + firstv;            // this segment's first valid descriptor, block-relative
                u32 gm = __ballot_sync(0xffffffffu, gdone && sj == 0);
                while (gm) {
                    const int gl = __ffs(gm) - 1;                               // lane 0 of the group being compacted
                    gm &= gm - 1;
                    const u32 okg = __shfl_sync(0xffffffffu, ok, gl), osz = __shfl_sync(0xffffffffu, out_size, gl);
                    u32 *const bd = reinterpret_cast<u32 *>(__shfl_sync(0xffffffffu, (unsigned long long)(uintptr_t)dout, gl));
                    u32 dst = __shfl_sync(0xffffffffu, cnt, gl);                // segment 0 is in place
                    const bool good = okg && osz <= 65536u;
#pragma unroll 1
                    for (int kk = 1; kk < 4 && good; ++kk) {
                        const u32 sv = __shfl_sync(0xffffffffu, srcv, gl + kk), cv = __shfl_sync(0xffffffffu, cnt, gl + kk),
                                  bv = __shfl_sync(0xffffffffu, base, gl + kk);
                        __syncwarp();                                           // the segments' own stores, and the previous move
                        for (u32 i0 = 0; i0 < cv; i0 += 256) {                   // eight loads in flight per lane: the move is latency-bound
                            u32 v[8];
#pragma unroll
                            for (u32 u = 0; u < 8; ++u) {
                                const u32 i = i0 + 32 * u + lane;
                                v[u] = i < cv ? __ldcg(bd + sv + i) : 0u;
                            }
                            __syncwarp();                                       // every load of the batch before any store of it
#pragma unroll
                            for (u32 u = 0; u < 8; ++u) {
                                const u32 i = i0 + 32 * u + lane;
                                if (i < cv) bd[dst + i] = (v[u] & 0xFFFFu) | (((v[u] >> 16) + bv) << 16);
                            }
                        }
                        dst += cv;
                    }
                }
                if (gdone) {
                    const bool failed = !ok || out_size > 65536u;
                    if (failed && attempt == 0) {
                        // No join within reach (a walk started inside a long literal run, or phase-locked on periodic data,
                        // stays off the true chain): once more, the speculative starts shifted by a few bytes.
                        attempt = 1;
                        cp_async_wait_all();
                        skew = sg.open(archive, asz, fb[slot].src, row_s);
                        q = skew + k1_seg_start(bszv, sj, J, 1);
                        qstop = sj + 1 < J ? skew + k1_seg_start(bszv, sj + 1, J, 1) : qend;
                        op = 0; nseq = 0; last_ms = 0; had_match = false;
                        mode = K1M_WALK; mptr = 0; msteps = 0; jtok = 0; jop = 0;
                        sg.need(q, q + 1);
                        if (sj == 3) atomicAdd(&counters[CNT_SPLIT_RETRIES], 1u);   // statistics: second attempts
                    } else {
                        if (sj == 3) {
                            if (failed) {
                                // still no join, or a genuinely bad block: the unsplit kernel, which runs after this one,
                                // walks it again from its first byte and has the verdict
                                parse_list[2ull * plist_cap + atomicAdd(&counters[CNT_PARSE_LIGHT], 1u)] = slot;
                                atomicAdd(&counters[CNT_SPLIT_GIVEN_BACK], 1u);   // statistics: blocks the split walk gave back
                            } else {
                                fb[slot].nseq = total;
                                fb[slot].out_size = out_size;
                                __threadfence();   // K2 may already be running (it polls `flags`): descriptors and sizes first, verdict last
                                *reinterpret_cast<volatile u32 *>(&fb[slot].flags) = FB_PARSED;
                            }
                        }
                        active = false;
                    }
                }
            }
        }
        if (!(active && mode <= K1M_MERGE)) continue;

        // ---- one sequence (control bytes only; mirrors lz4.c:1797-2151 + the spec's end rules)
        bool bad = false, fin = false;
        const u32 token = sg.rd(q);               // q < avail always (need() at open, and below)
        const u32 lim = sg.avail;                 // readable without waiting
        // Common shape first, branch-free: at most one length-extension byte each, offset inside the
        // staged window, not the block's last sequences.  Everything else takes the general walk below.
        bool fast = false;
        {
            const u32 l0 = token >> 4, m0 = token & 15;
            const bool lx = l0 == 15, mx = m0 == 15;
            const u32 e1 = sg.rd(q + 1);                      // stale when q + 1 >= lim: then pq + 3 > lim as well
            const u32 lit = lx ? 15 + e1 : l0;
            const u32 pq = q + (lx ? 2u : 1u) + lit;          // where the offset bytes are
            if (!(lx && e1 == 255) && pq + 3 <= lim && pq + 8 <= qend) {
                const u32 off = sg.rd(pq) | (sg.rd(pq + 1) << 8);
                const u32 e2 = sg.rd(pq + 2);
                if (!(mx && e2 == 255)) {
                    fast = true;
                    const u32 ml = m0 + 4 + (mx ? e2 : 0u);
                    const u32 d = (q - skew) | (op << 16);
                    b0 = b1; b1 = b2; b2 = b3; b3 = d;
                    ++nseq;
                    if ((nseq & 3u) == 0) *reinterpret_cast<uint4 *>(dout + nseq - 4) = make_uint4(b0, b1, b2, b3);
                    op += lit;
                    last_ms = op;
                    had_match = true;
                    op += ml;
                    q = pq + (mx ? 3u : 2u);
                    if ((off == 0 && sj == 0) || (J == 1 && op > 65536u) || q >= qend) bad = true;   // a speculative walk may read anything; K2 checks the offsets it executes
                }
            }
        }
        if (!fast) {
            u32 p = q + 1;
            u32 lit = token >> 4;
            if (lit == 15) {
                u32 b = 0;
                do {
                    if (p >= qend) { bad = true; break; }
                    sg.need(p, p + 1);
                    b = sg.rd(p++);
                    lit += b;
                } while (b == 255 && lit < 0x100000u);
                if (b == 255) bad = true;
            }
            if (lit > qend - p) bad = true;
            if (!bad) {
                const u32 d = (q - skew) | (op << 16);
                b0 = b1; b1 = b2; b2 = b3; b3 = d;
                ++nseq;
                if ((nseq & 3u) == 0) *reinterpret_cast<uint4 *>(dout + nseq - 4) = make_uint4(b0, b1, b2, b3);
                p += lit; op += lit;
                if (J == 1 && op > 65536u) bad = true;
                else if (p == qend) {
                    // final sequence: literals only.  Spec end rules (lz4_Block_format.md:108-137) as
                    // sufficient conditions for the reference's capacity-based checks (lz4.c:2055-2077,2139).
                    if (had_match && (lit < 5 || op - last_ms < 12)) bad = true;
                    if (J == 4 && sj != 3) bad = true;            // a quarter that reaches the block's end without a join
                    fin = true;
                } else if (p + 8 > qend) {
                    bad = true;                                   // lz4.c:2055: must have been the last
                } else {
                    sg.need(p, p + 2);
                    u32 off = sg.rd(p) | (sg.rd(p + 1) << 8);
                    p += 2;
                    u32 ml = token & 15;
                    if (ml == 15) {
                        u32 b = 0;
                        do {
                            if (p >= qend) { bad = true; break; }
                            sg.need(p, p + 1);
                            b = sg.rd(p++);
                            ml += b;
                        } while (b == 255 && ml < 0x100000u);
                        if (b == 255) bad = true;
                    }
                    ml += 4;
                    if (off == 0 && sj == 0) bad = true;
                    last_ms = op;
                    had_match = true;
                    op += ml;
                    if ((J == 1 && op > 65536u) || p >= qend) bad = true;
                    q = p;
                    if (!bad) sg.need(q, q + 1);                  // the next token
                }
            }
        } else if (!bad && q + 1 > sg.avail) {
            sg.need(q, q + 1);
        }
        if (J == 4 && !bad && !fin && mode == K1M_WALK && q >= qstop && sj != 3) mode = K1M_MERGE;
        if (bad || fin) {
            if (!bad) {
                u32 r = nseq & 3u;  // descriptors still in the shift register
                if (r == 1) dout[nseq - 1] = b3;
                else if (r == 2) { dout[nseq - 2] = b2; dout[nseq - 1] = b3; }
                else if (r == 3) { dout[nseq - 3] = b1; dout[nseq - 2] = b2; dout[nseq - 1] = b3; }
            }
            cp_async_wait_all();
            if (J == 1) {
                fb[slot].nseq = nseq;
                fb[slot].out_size = op;
                __threadfence();   // K2 may already be running (it polls `flags`): descriptors and sizes first, verdict last
                *reinterpret_cast<volatile u32 *>(&fb[slot].flags) = bad ? FB_BAD : FB_PARSED;
                active = false;
            } else {
                if (bad) K1_WHY("walk hit an invalid construct");
                mode = bad ? K1M_FAIL : K1M_DONE;
            }
        }
    }
}

__global__ void __launch_bounds__(K1_THREADS)
lz4_fast_parse_kernel(const u8 *__restrict__ archive, u64 asz, FastBlock *fb, u32 *parse_list,
                      u32 plist_cap, u32 *counters, u32 *work_counter, u32 *desc, u32 all_lists) {
    lz4_fast_parse_body<1>(archive, asz, fb, parse_list, plist_cap, counters, work_counter, desc, all_lists);
}
__global__ void __launch_bounds__(K1_THREADS)
lz4_fast_parse4_kernel(const u8 *__restrict__ archive, u64 asz, FastBlock *fb, u32 *parse_list,
                       u32 plist_cap, u32 *counters, u32 *work_counter, u32 *desc) {
    lz4_fast_parse_body<4>(archive, asz, fb, parse_list, plist_cap, counters, work_counter, desc, 0u);
}

// ------------------------------------------------------------------------------------------ K2

// K2 starts while K1 is still walking the heaviest blocks (separate streams): everything K1 produces is read through
// L2 (ld.global.cg / volatile), never through the non-coherent or L1 paths, whose lines could predate K1's stores.
ZPB_DEVINL u32 ldcg32(const u32 *p) { return __ldcg(p); }

#define FAST_LT  16u   // literal runs up to this go one-lane-per-sequence (from global memory); longer ones warp-wide
#ifndef FAST_LTR
#define FAST_LTR 32u   // the same when the source is the staging ring (word copies)
#endif
#ifndef FAST_MT
#define FAST_MT  64u   // matches up to this go one-lane-per-sequence (non-overlapping, linear in shared memory)
#endif

#define DS_FINAL 0u   // source bytes are final (possibly after redirection by `shift`)
#define DS_CHILD 1u   // source wholly inside lane `parent`'s match: being resolved
#define DS_HARD  2u   // source straddles pending matches: executed in lane order

struct FastExec {
    u32 rb;         // this warp's output ring (shared-window address): position p lives at rb + (p & FAST_RMASK)
    u32 scr_s;      // this lane's far-match staging (shared-window address)
    u8 *gout;       // the entry's final place in HBM (16-byte aligned)
    u32 done;       // every byte below is final (in the ring and/or in HBM)
    u32 flushed;    // HBM holds [0, flushed); multiple of 1024 until the very end
    u32 rbase;      // ring content below this position is stale (direct stored path went around it)
    u32 total, full_blocks;
    u64 acc0, acc1; // XXH3 accumulators of pair j = lane & 3
    u64 *part;      // block-sharded path: where this pseudo-entry's per-KiB stripe sums go (else nullptr)
    int lane;

    ZPB_DEVINL u32 ring_lo(u32 hi) const {
        u32 w = hi > FAST_RING ? hi - FAST_RING : 0u;
        return w > rbase ? w : rbase;
    }
    ZPB_DEVINL u32 ra(u32 pos) const { return rb + (pos & FAST_RMASK); }
    ZPB_DEVINL u32 rd(u32 pos, u32 lo) const { return pos >= lo ? lds8(ra(pos)) : ldg8_coherent(gout + pos); }

    ZPB_DEVINL void hash_init() {
        int j = lane & 3;
        acc0 = j == 0 ? (u64)XXH_P32_3 : j == 1 ? XXH_P64_2 : j == 2 ? XXH_P64_4 : XXH_P64_5;
        acc1 = j == 0 ? XXH_P64_1 : j == 1 ? XXH_P64_3 : j == 2 ? (u64)XXH_P32_2 : (u64)XXH_P32_1;
    }
    ZPB_DEVINL void hash_fold_scramble(u64 s0, u64 s1) {
#pragma unroll
        for (int m = 4; m < 32; m <<= 1) {
            s0 += __shfl_xor_sync(0xffffffffu, s0, m);
            s1 += __shfl_xor_sync(0xffffffffu, s1, m);
        }
        int j = lane & 3;
        if (part) {
            // the 16-stripe sums of KiB (flushed >> 10), words 2j and 2j+1: the scramble chain
            // (xxhash.h:3527-3534) over the whole entry is xxh3_chain_kernel's job
            if (lane < 4) *reinterpret_cast<ulonglong2 *>(part + (u64)(flushed >> 10) * 8 + 2 * j) = make_ulonglong2(s0, s1);
            return;
        }
        u64 a0 = acc0 + s0, a1 = acc1 + s1;
        a0 ^= a0 >> 47; a0 ^= c_xxh3_key[16 + 2 * j]; a0 *= XXH_P32_1;
        a1 ^= a1 >> 47; a1 ^= c_xxh3_key[16 + 2 * j + 1]; a1 *= XXH_P32_1;
        acc0 = a0; acc1 = a1;
    }
    // one full 1 KiB block: ring -> HBM (16 B per lane, coalesced) and -> XXH3 from the same registers
    ZPB_DEVINL void flush_kib() {
        u32 a = rb + (flushed & FAST_RMASK) + lane * 16;
        int j = lane & 3;
        u64 s0 = 0, s1 = 0;
        uint4 v0 = lds128(a), v1 = lds128(a + 512);
        stg128(gout + flushed + lane * 16, v0);
        stg128(gout + flushed + 512 + lane * 16, v1);
        u32 s = lane >> 2;
        Xxh3Stream<32>::piece(s0, s1, v0, c_xxh3_key[s + 2 * j], c_xxh3_key[s + 2 * j + 1]);
        Xxh3Stream<32>::piece(s0, s1, v1, c_xxh3_key[s + 8 + 2 * j], c_xxh3_key[s + 8 + 2 * j + 1]);
        hash_fold_scramble(s0, s1);
        flushed += 1024;
    }
    // callers have finished writing [.., done); flushes every hashable full block below done
    ZPB_DEVINL void flush_full() {
        __syncwarp();
        if (flushed + 1024 <= done && (flushed >> 10) < full_blocks) {
            do flush_kib(); while (flushed + 1024 <= done && (flushed >> 10) < full_blocks);
            __syncwarp();
        }
    }
    ZPB_DEVINL u32 room() const { return flushed + FAST_RING - done; }

    // warp-wide: ring[O + i] = sp[i], i < L (inside a segment: no flush)
    ZPB_DEVINL void coop_lit(u32 O, const u8 *__restrict__ sp, u32 L) const {
        for (u32 i = lane; i < L; i += 32) sts8(ra(O + i), sp[i]);
    }
    // warp-wide match: out[MO + i] = out[MO + i - OF], i < ML, everything below MO final
    // 16 source bytes starting at output position p (any alignment), from the ring or from HBM
    ZPB_DEVINL uint4 load16_ring(u32 p) const {
        const u32 b = p & ~3u, sh = (p & 3u) << 3;
        const u32 w0 = lds32_loose(ra(b)), w1 = lds32_loose(ra(b + 4)), w2 = lds32_loose(ra(b + 8)), w3 = lds32_loose(ra(b + 12)),
                  w4 = lds32_loose(ra(b + 16));   // whole words around the source: bytes of neighbouring copies are read, never stored
        return make_uint4(__funnelshift_r(w0, w1, sh), __funnelshift_r(w1, w2, sh), __funnelshift_r(w2, w3, sh),
                          __funnelshift_r(w3, w4, sh));
    }
    ZPB_DEVINL uint4 load16_hbm(u32 p) const {   // plain ld.global: the buffer is written by this kernel
        const u8 *g = gout + (p & ~3u);
        const u32 sh = (p & 3u) << 3;
#ifdef ZPB_SIM
        const u32 w0 = ldg32_coherent(g), w1 = ldg32_coherent(g + 4), w2 = ldg32_coherent(g + 8), w3 = ldg32_coherent(g + 12), w4 = ldg32_coherent(g + 16);
#else
        u32 w0, w1, w2, w3, w4;
        asm volatile("ld.global.u32 %0, [%5];\n\tld.global.u32 %1, [%5+4];\n\tld.global.u32 %2, [%5+8];\n\t"
                     "ld.global.u32 %3, [%5+12];\n\tld.global.u32 %4, [%5+16];"
                     : "=r"(w0), "=r"(w1), "=r"(w2), "=r"(w3), "=r"(w4) : "l"(g) : "memory");
#endif
        return make_uint4(__funnelshift_r(w0, w1, sh), __funnelshift_r(w1, w2, sh), __funnelshift_r(w2, w3, sh),
                          __funnelshift_r(w3, w4, sh));
    }
    // warp-wide match: out[MO + i] = out[MO + i - OF], i < ML, everything below MO final
    ZPB_DEVINL void coop_match(u32 MO, u32 OF, u32 ML, u32 lo) const {
        if (ML >= 32 && (OF == 1 || OF == 2 || OF == 4)) {
            // short period dividing 4 (runs; lz4.c:1917-1921 pattern case): one 32-bit pattern word, 16-byte fills.
            // Byte j of W is the byte that belongs at any output position congruent to j mod 4.
            u32 W = 0;
#pragma unroll
            for (u32 j = 0; j < 4; ++j) W |= rd(MO - OF + ((j - MO) & (OF - 1u)), lo) << (8 * j);
            const u32 head = (0u - MO) & 15u;                    // ML >= 32 > head
            if ((u32)lane < head) sts8(ra(MO + lane), W >> (8 * ((MO + lane) & 3u)));
            const u32 body = MO + head, n16 = (ML - head) >> 4;  // 16-aligned ring positions never straddle the ring end
            for (u32 c = lane; c < n16; c += 32) sts128(ra(body + 16 * c), make_uint4(W, W, W, W));
            const u32 tpos = body + (n16 << 4), tail = MO + ML - tpos;
            if ((u32)lane < tail) sts8(ra(tpos + lane), W >> (8 * (lane & 3u)));
            return;
        }
        if (ML >= 32 && OF >= ML && (MO - OF >= lo || MO - OF + ML + 4 <= lo)) {   // +4: whole-word reads stay below lo
            // long, not self-overlapping, source wholly in the ring or wholly in HBM: 16-byte destination chunks
            // (aligned stores), each lane assembling its 16 source bytes from aligned words
            const bool hbm = MO - OF < lo;
            const u32 head = (0u - MO) & 15u;
            if ((u32)lane < head) sts8(ra(MO + lane), rd(MO - OF + lane, lo));
            const u32 body = MO + head, n16 = (ML - head) >> 4;
            for (u32 c = lane; c < n16; c += 32) {
                const u32 dpos = body + 16 * c;
                const uint4 v = hbm ? load16_hbm(dpos - OF) : load16_ring(dpos - OF);
                sts128(ra(dpos), v);
            }
            const u32 tpos = body + (n16 << 4), tail = MO + ML - tpos;
            if ((u32)lane < tail) sts8(ra(tpos + lane), rd(tpos - OF + lane, lo));
            return;
        }
        if (MO - OF >= lo) {
            // whole source still in the ring (the usual dependent match): no HBM select per byte
            if (OF >= 32) {
                // 32-byte steps never read what they write; later steps may read earlier ones
                for (u32 b = 0; b < ML; b += 32) {
                    const u32 i = b + lane;
                    if (i < ML) sts8(ra(MO + i), lds8(ra(MO - OF + i)));
                    if (OF < ML) __syncwarp();
                }
            } else {  // period OF < 32: byte i is byte (i mod OF) of the OF bytes before MO
                u32 k = (u32)lane < OF ? (u32)lane : (u32)lane % OF;
                const u32 step = 32u % OF;
                for (u32 i = lane; i < ML; i += 32) {
                    sts8(ra(MO + i), lds8(ra(MO - OF + k)));
                    k += step;
                    if (k >= OF) k -= OF;
                }
            }
            return;
        }
        if (OF >= ML) {
            for (u32 i = lane; i < ML; i += 32) sts8(ra(MO + i), rd(MO - OF + i, lo));
        } else {  // periodic with period OF: byte i is byte (i mod OF) of the OF bytes before MO
            u32 k = (u32)lane < OF ? (u32)lane : (u32)lane % OF;
            u32 step = OF > 32 ? 32u : 32u % OF;
            for (u32 i = lane; i < ML; i += 32) {
                sts8(ra(MO + i), rd(MO - OF + k, lo));
                k += step;
                if (k >= OF) k -= OF;
            }
        }
    }
    // the same, for runs too long for the ring: piecewise with flushes in between
    ZPB_DEVINL void stream_lit(const u8 *__restrict__ sp, u32 L) {
        while (L) {
            u32 piece = L < room() ? L : room();
            coop_lit(done, sp, piece);
            sp += piece; L -= piece; done += piece;
            flush_full();
        }
    }
    ZPB_DEVINL void stream_match(u32 OF, u32 ML) {
        while (ML) {
            u32 piece = ML < room() ? ML : room();
            coop_match(done, OF, piece, ring_lo(done + piece));
            ML -= piece; done += piece;
            flush_full();
        }
    }
};

ZPB_DEVINL void cp_async16_cg(u32 smem_addr, const void *gptr) {   // L2 only: coherent with this kernel's own stores
#ifdef ZPB_SIM
    sim::cp_async(smem_addr, gptr, 16, 16);
#else
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(smem_addr), "l"(gptr) : "memory");
#endif
}

// The compressed bytes of the block a warp is executing, staged through a per-warp shared-memory ring:
// rows of CR_ROW bytes (16 per lane, cp.async), requested one row ahead of the step that reads them, so
// the per-lane token / length / offset / literal reads of K2 are shared-memory reads.  Positions are
// "ring coordinates" c = block position + skew, with the global address of coordinate 0 16-byte aligned.
struct CompStage {
    const u8 *gbase;     // global address of ring coordinate 0
    const u8 *glo, *ghi; // readable range (the archive)
    u32 rb;              // the ring (shared-window address)
    u32 skew;
    u32 fill;            // rows below this coordinate have been requested (multiple of CR_ROW)
    u32 pending;         // cp.async groups committed since the last full wait (warp-uniform)
    int lane;

    ZPB_DEVINL void open(const u8 *src) {
        cp_async_wait_all();         // a look-ahead row of the previous block may still be in flight
        __syncwarp();
        skew = (u32)((uintptr_t)src & 15u);
        gbase = src - skew;
        fill = 0;
        pending = 0;
    }
    ZPB_DEVINL void request_row() {
        const u32 c = fill + 16u * lane;
        const u8 *g = gbase + c;
        const u32 sdst = rb + (c & CR_MASK);
        if (16u * lane >= CR_ROW) {
        } else if (g >= glo && g + 16 <= ghi) {
#ifdef ZPB_SIM
            sim::cp_async(sdst, g, 16, 16);
#else
            asm volatile("cp.async.ca.shared.global [%0], [%1], 16;" ::"r"(sdst), "l"(g) : "memory");
#endif
        } else if (g + 16 > glo && g < ghi) {   // straddles an end of the archive: byte by byte
            for (u32 k = 0; k < 16; ++k)
                if (g + k >= glo && g + k < ghi) sts8(sdst + k, g[k]);
        }
        cp_async_commit();
        fill += CR_ROW;
        ++pending;
    }
    // Makes block positions [s_lo, s_hi) readable through the ring; false when the span does not fit
    // (the caller then reads global memory for this step).  Warp-uniform arguments and result.
    ZPB_DEVINL bool prepare(u32 s_lo, u32 s_hi, u32 bsz) {
        const u32 rlo = (s_lo + skew) & ~(CR_ROW - 1u);
        const u32 rhi = (s_hi + skew + CR_ROW - 1u) & ~(CR_ROW - 1u);
        if (rhi - rlo > CR_SIZE) return false;
        if (fill < rlo) {            // rows nobody needs (after a step that went around the ring)
            cp_async_wait_all();
            pending = 0;
            __syncwarp();
            fill = rlo;
        }
        while (fill < rhi) request_row();
        u32 ahead = 0;
        if (fill + CR_ROW - rlo <= CR_SIZE && fill < bsz + skew) { request_row(); ahead = 1; }   // one row of look-ahead
        else if (fill > rhi) ahead = 1;                                                          // requested by the previous step
        if (pending > ahead) {
            if (ahead) cp_async_wait_1(); else cp_async_wait_all();
            pending = ahead;
        }
        __syncwarp();
        return true;
    }
};
struct CompRing {     // byte reader over the staging ring
    u32 rb, skew;
    ZPB_DEVINL u32 operator()(u32 p) const { return lds8(rb + ((p + skew) & CR_MASK)); }
};
struct CompGlobal {   // byte reader over global memory (steps whose span does not fit the ring)
    const u8 *__restrict__ s;
    ZPB_DEVINL u32 operator()(u32 p) const { return s[p]; }
};
// One sequence's control bytes (lz4.c:1797-1822, 1845-1860; K1 has validated them): literal length and
// start, match offset and length (0 for the block's last sequence).
template <class R>
ZPB_DEVINL void fast_decode_seq(const R rd, u32 tok, u32 bsz, u32 &lit, u32 &lsrc, u32 &off, u32 &ml) {
    const u32 t = rd(tok);
    u32 p = tok + 1;
    lit = t >> 4;
    if (lit == 15) { u32 bb; do { bb = rd(p++); lit += bb; } while (bb == 255); }
    lsrc = p;
    p += lit;
    if (p < bsz) {
        off = rd(p) | (rd(p + 1) << 8);
        p += 2;
        ml = t & 15;
        if (ml == 15) { u32 bb; do { bb = rd(p++); ml += bb; } while (bb == 255); }
        ml += 4;
    }
}

// unaligned 16-byte global load assembled from 4-byte-aligned words
ZPB_DEVINL uint4 ldg128_unaligned(const u8 *p) {
    const u32 *s = reinterpret_cast<const u32 *>((uintptr_t)p & ~(uintptr_t)3);
    u32 sh = ((u32)(uintptr_t)p & 3u) * 8u;
    u32 w0 = s[0], w1 = s[1], w2 = s[2], w3 = s[3];
    if (sh == 0) return make_uint4(w0, w1, w2, w3);
    u32 w4 = s[4];
    return make_uint4(__funnelshift_r(w0, w1, sh), __funnelshift_r(w1, w2, sh), __funnelshift_r(w2, w3, sh),
                      __funnelshift_r(w3, w4, sh));
}

#ifdef ZPB_SIM
template <int OFF> ZPB_DEVINL void sts8o(u32 a, u32 v) { sts8(a + OFF, v); }
template <int OFF> ZPB_DEVINL u32 ldg8nc(const u8 *p) { return p[OFF]; }
#else
template <int OFF> ZPB_DEVINL void sts8o(u32 a, u32 v) {
    asm volatile("st.shared.u8 [%0+%2], %1;" ::"r"(a), "r"(v), "n"(OFF) : "memory");
}
template <int OFF> ZPB_DEVINL u32 ldg8nc(const u8 *p) {   // read-only data (the archive), explicit addressing
    u32 v; asm volatile("ld.global.nc.u8 %0, [%1+%2];" : "=r"(v) : "l"(p), "n"(OFF)); return v;
}
#endif
#define FAST_BYTE4(LD, ST, n, i)                                                        \
    {                                                                                   \
        u32 v0_ = 0, v1_ = 0, v2_ = 0, v3_ = 0;                                                       \
        const bool p0_ = (i) + 0 < (n), p1_ = (i) + 1 < (n), p2_ = (i) + 2 < (n), p3_ = (i) + 3 < (n); \
        if (p0_) v0_ = LD(0); if (p1_) v1_ = LD(1); if (p2_) v2_ = LD(2); if (p3_) v3_ = LD(3);       \
        if (p0_) ST(0, v0_); if (p1_) ST(1, v1_); if (p2_) ST(2, v2_); if (p3_) ST(3, v3_);           \
    }

#ifndef FAST_EXEC_CTAS
#define FAST_EXEC_CTAS 3
#endif
// resident CTAs per SM the kernel is compiled for (registers) and launched with

__global__ void __launch_bounds__(32 * FAST_EXEC_WARPS, FAST_EXEC_CTAS)
lz4_fast_exec_kernel(const u8 *__restrict__ archive, u64 asz, u8 *out, const zpb_entry *__restrict__ entries,
                     const u32 *__restrict__ order, u32 n, u32 *counter, const FastEntry *__restrict__ fe,
                     const FastBlock *__restrict__ fb, const u32 *__restrict__ desc, u32 *counters,
                     u32 *general_list, int *status, u64 *digest, u64 *partials, u32 *defer_list, u32 *defer_cnt,
                     const u32 *n_ptr) {
    ZPB_DYN_SMEM(k2_smem);
    if (n_ptr) n = *n_ptr;   // the late pass over the deferred list: its length was only known on the device
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    FastExec x;
    x.lane = lane;
    x.rb = smem_window(k2_smem) + 16u + warp * FAST_WARP_SMEM;   // 16 B of slack in front, 32 behind (lane_copy reads whole words)
    x.scr_s = x.rb + FAST_RING + lane * FAST_SCR;
    const u8 *arch_end = archive + asz;
    CompStage cs;
    cs.lane = lane;
    cs.rb = x.rb + FAST_RING + 32u * FAST_SCR;
    cs.glo = archive;
    cs.ghi = arch_end;
    cs.fill = cs.pending = cs.skew = 0;
    cs.gbase = archive;

    for (;;) {
        u32 wslot = 0;
        if (lane == 0) wslot = atomicAdd(counter, 1u);
        wslot = __shfl_sync(0xffffffffu, wslot, 0);
        if (wslot >= n) break;
        const u32 idx = order ? __ldcg(order + wslot) : wslot;
        const FastEntry f = fe[idx];
        if (f.state != FE_FAST) continue;
        const zpb_entry e = entries[idx];

        // ---- K1 verdicts: every block parsed clean, window reach legal, sizes add up exactly
        bool ok = true, deferred = false;
        {
            u64 before = 0;
            for (u32 b = 0; b < f.nblocks; ++b) {
                const FastBlock *pb = fb + f.first_slot + b;
                // This grid may run while K1 is still walking the heavy blocks.  It never waits for a verdict (a
                // resident CTA that waits could keep K1's own CTAs off the SMs): an entry with a block still in
                // flight goes to the deferred list, which a last launch works off after K1 has finished.
                u32 ready = 1;
                if (lane == 0) {
                    ready = (*reinterpret_cast<const volatile u32 *>(&pb->flags) & (FB_STORED | FB_PARSED | FB_BAD)) != 0;
                    if (ready) __threadfence();
                }
                ready = __shfl_sync(0xffffffffu, ready, 0);
                if (!ready) { deferred = true; break; }
                const u32 bflags = __ldcg(&pb->flags);
                if (!(bflags & FB_STORED)) {
                    if (!(bflags & FB_PARSED) || (bflags & FB_BAD)) ok = false;
                }
                before += __ldcg(&pb->out_size);
            }
            if (before != e.uncomp_size) ok = false;
        }
        if (deferred) {
            if (defer_list) {
                if (lane == 0) defer_list[atomicAdd(defer_cnt, 1u)] = idx;
                continue;
            }
            ok = false;   // launches without a list run after K1, where every verdict is in: never skip an entry silently
        }
        const bool partial = f.linked == FE_LINK_PARTIAL;
        if (!ok) {
            if (lane == 0) {
                // a block of the sharded path that K1 did not accept: the shard call declines (the caller
                // re-reads the entry through zpb_unpack_device, whose general decoder has the exact verdict)
                if (partial) { status[idx] = ST_NOT_AVAILABLE; digest[idx] = 0; }
                else general_list[atomicAdd(&counters[CNT_GENERAL], 1u)] = idx;
            }
            continue;
        }

        x.gout = out + e.dst_off;
        x.done = x.flushed = x.rbase = 0;
        x.total = (u32)e.uncomp_size;
        x.full_blocks = partial ? x.total >> 10 : x.total > 240 ? (x.total - 1) >> 10 : 0;
        x.part = partial ? partials + e.reserved * 8 : nullptr;
        x.hash_init();

        for (u32 b = 0; b < f.nblocks; ++b) {
            const FastBlock *pb = fb + f.first_slot + b;   // fields are read where they are needed, through L2
            const u8 *__restrict__ src = archive + __ldcg(&pb->src);
            if (__ldcg(&pb->flags) & FB_STORED) {
                // ---- stored block / NONE entry (lz4frame.c:1534-1572, zpack_read.c:352-368)
                u32 len = __ldcg(&pb->bsz);
                if (x.done == x.flushed && (x.done & 1023u) == 0) {
                    // direct: HBM -> registers -> XXH3 + HBM, no ring
                    while (len >= 1024 && (x.flushed >> 10) < x.full_blocks && src + 1024 + 16 <= arch_end) {
                        int j = lane & 3;
                        u64 s0 = 0, s1 = 0;
                        uint4 v0 = ldg128_unaligned(src + lane * 16);
                        uint4 v1 = ldg128_unaligned(src + 512 + lane * 16);
                        stg128(x.gout + x.flushed + lane * 16, v0);
                        stg128(x.gout + x.flushed + 512 + lane * 16, v1);
                        u32 s = lane >> 2;
                        Xxh3Stream<32>::piece(s0, s1, v0, c_xxh3_key[s + 2 * j], c_xxh3_key[s + 2 * j + 1]);
                        Xxh3Stream<32>::piece(s0, s1, v1, c_xxh3_key[s + 8 + 2 * j], c_xxh3_key[s + 8 + 2 * j + 1]);
                        x.hash_fold_scramble(s0, s1);
                        x.flushed += 1024; src += 1024; len -= 1024;
                    }
                    x.done = x.flushed;
                    x.rbase = x.done;
                    __syncwarp();
                }
                x.stream_lit(src, len);
                continue;
            }

            // ---- compressed block: 32 sequences per step, one per lane
            const u32 *dp = desc + __ldcg(&pb->desc_off);
            const u32 obase = x.done;
            const u32 bsz = __ldcg(&pb->bsz);
            const u32 nseq = __ldcg(&pb->nseq);
            cs.open(src);
            // two steps of descriptors are kept in flight; the compressed bytes come through the staging ring
            u32 d0 = (u32)lane < nseq ? ldcg32(dp + lane) : 0u;
            u32 d1 = 32u + lane < nseq ? ldcg32(dp + 32 + lane) : 0u;
            for (u32 s0i = 0; s0i < nseq; s0i += 32) {
                const bool have = s0i + lane < nseq;
                const u32 d = d0;
                d0 = d1;
                d1 = s0i + 64 + lane < nseq ? ldcg32(dp + s0i + 64 + lane) : 0u;
                // compressed bytes this step reads: from its first token to the next step's first token
                const u32 s_lo = __shfl_sync(0xffffffffu, d & 0xFFFFu, 0);
                const u32 s_nx = __shfl_sync(0xffffffffu, d0 & 0xFFFFu, 0);
                const bool in_ring = cs.prepare(s_lo, s0i + 32 < nseq ? s_nx : bsz, bsz);   // warp-uniform
                u32 lit = 0, lsrc = 0, off = 0, ml = 0, o = 0;
                if (have) {
                    o = obase + (d >> 16);
                    if (in_ring) fast_decode_seq(CompRing{cs.rb, cs.skew}, d & 0xFFFFu, bsz, lit, lsrc, off, ml);
                    else fast_decode_seq(CompGlobal{src}, d & 0xFFFFu, bsz, lit, lsrc, off, ml);
                }
                const u32 sz = lit + ml;
                const u32 mo = o + lit, msrc = mo - off;
                // a match that reaches below the window (lz4.c:2093: the frame's prefix when the blocks are linked) or has
                // offset 0: not something this path decodes — the entry goes to the general decoder, which has the exact verdict
                if (__any_sync(0xffffffffu, ml > 0 && (off == 0 || off > mo - (f.linked == FE_LINK_WINDOW ? 0u : obase)))) goto bail_entry;
                const u8 *__restrict__ sp = src + lsrc;
                // matches whose whole source is already in HBM: fetch it now, asynchronously, into this lane's
                // scratch (16-byte pieces straight from L2; up to 5 cover any alignment of <= 64 bytes)
                const u32 abase = msrc & ~15u;
                const bool staged = have && ml > 0 && ml <= FAST_ST && msrc + ml <= x.flushed;
                if (staged) {
                    const u32 np = ((msrc - abase) + ml + 15u) >> 4;
                    const u8 *g = x.gout + abase;
                    cp_async16_cg(x.scr_s, g);
                    if (np > 1) cp_async16_cg(x.scr_s + 16, g + 16);
                    if (np > 2) {
                        cp_async16_cg(x.scr_s + 32, g + 32);
                        if (np > 3) cp_async16_cg(x.scr_s + 48, g + 48);
                        if (np > 4) cp_async16_cg(x.scr_s + 64, g + 64);
                    }
                }
                else if (have && ml > 0 && msrc < x.flushed) {
                    // longer match reaching back into flushed output: pull its lines towards L1 now, the
                    // warp-wide copy that needs them runs later in this step
                    u32 pe = msrc + ml < x.flushed ? msrc + ml : x.flushed;
                    if (pe > msrc + 512) pe = msrc + 512;
                    for (u32 a = msrc & ~127u; a < pe; a += 128)
                        prefetch_l1(x.gout + a);
                }
                cp_async_commit();
                // ---- same-step dependencies.  A match whose source lies inside the output of an earlier
                // match of this step would have to wait for it; instead, when the source range is wholly inside
                // that match (the usual case: repeated words, records), it is redirected through the parent's
                // offset (out[x] = out[x - off_k] holds for every x of the parent's match), parents' shifts are
                // composed by pointer jumping, and the match reads bytes that are already final.
                u32 shift = 0, dstate = DS_FINAL;
                {
                    const u32 o_first = __shfl_sync(0xffffffffu, o, 0);
                    const bool has_mm = have && ml > 0;
                    const u32 send_ = msrc + ml < mo ? msrc + ml : mo;
                    const bool inside = has_mm && send_ > o_first && msrc < o;
                    if (__any_sync(0xffffffffu, inside)) {
                        const u32 okey = have ? o : 0xFFFFFFFFu;
                        u32 k = 0;   // largest lane whose sequence starts at or below msrc
#pragma unroll
                        for (u32 st = 16; st; st >>= 1) {
                            const u32 ot = __shfl_sync(0xffffffffu, okey, k + st);
                            if (ot <= msrc) k += st;
                        }
                        const u32 mo_k = __shfl_sync(0xffffffffu, mo, k), e_k = __shfl_sync(0xffffffffu, o + sz, k),
                                  off_k = __shfl_sync(0xffffffffu, off, k);
                        u32 parent = 0;
                        if (inside) {
                            if (msrc < o_first) dstate = DS_HARD;                 // straddles the step start
                            else if (send_ <= mo_k) dstate = DS_FINAL;           // inside lane k's literals
                            else if (msrc >= mo_k && send_ <= e_k && off_k >= e_k - mo_k && off >= ml) {
                                dstate = DS_CHILD; parent = k; shift = off_k;
                            } else dstate = DS_HARD;
                        }
                        while (__any_sync(0xffffffffu, dstate == DS_CHILD)) {
                            const u32 pst = __shfl_sync(0xffffffffu, dstate, parent),
                                      psh = __shfl_sync(0xffffffffu, shift, parent),
                                      pp = __shfl_sync(0xffffffffu, parent, parent);
                            if (dstate == DS_CHILD) {
                                if (pst == DS_HARD) { dstate = DS_HARD; shift = 0; }
                                else { shift += psh; parent = pp; if (pst == DS_FINAL) dstate = DS_FINAL; }
                            }
                        }
                    }
                }
                bool parked = false;
                u32 todo = __ballot_sync(0xffffffffu, have);
                while (todo) {
                    const int first = __ffs(todo) - 1;
                    const bool fits = ((todo >> lane) & 1u) && (o + sz <= x.flushed + FAST_RING);
                    const u32 seg = __ballot_sync(0xffffffffu, fits);   // o + sz is monotone: a prefix of todo
                    if (!((seg >> first) & 1u)) {
                        // ---- one sequence larger than the ring: streamed, whole warp
                        u32 L = __shfl_sync(0xffffffffu, lit, first), S = __shfl_sync(0xffffffffu, lsrc, first);
                        u32 O = __shfl_sync(0xffffffffu, off, first), ML = __shfl_sync(0xffffffffu, ml, first);
                        x.stream_lit(src + S, L);
                        if (ML) x.stream_match(O, ML);
                        todo &= ~(1u << first);
                        continue;
                    }
                    // ---- a run of sequences that fits the ring: literals first (they depend on nothing) ...
                    const bool in = (seg >> lane) & 1u;
                    const int last_lane = 31 - __clz(seg);
                    const u32 seg_end = __shfl_sync(0xffffffffu, o + sz, last_lane);
                    const u32 lo = x.ring_lo(seg_end);
                    {
                        const u32 da = x.ra(o);
                        const u32 cq = (lsrc + cs.skew) & CR_MASK;    // literal source in the staging ring
                        const bool lane_lit = in && (o & FAST_RMASK) + lit <= FAST_RING &&
                                              (in_ring ? lit <= FAST_LTR && cq + lit <= CR_SIZE : lit <= FAST_LT);
                        const u32 mylit = lane_lit ? lit : 0u;
                        if (in_ring) {
                            lane_copy(cs.rb + cq, da, mylit);
                        } else {
                            const u32 maxlit = __reduce_max_sync(0xffffffffu, mylit);
#define STL(u, v) sts8o<u>(dai, v)
#define LDL(u) ldg8nc<u>(spi)
                            for (u32 i = 0; i < maxlit; i += 4) {
                                const u8 *spi = sp + i;
                                const u32 dai = da + i;
                                FAST_BYTE4(LDL, STL, mylit, i)
                            }
#undef LDL
#undef STL
                        }
                        u32 cm = __ballot_sync(0xffffffffu, in && lit > 0 && !lane_lit);
                        while (cm) {
                            int r = __ffs(cm) - 1;
                            cm &= cm - 1;
                            u32 O = __shfl_sync(0xffffffffu, o, r), S = __shfl_sync(0xffffffffu, lsrc, r),
                                L = __shfl_sync(0xffffffffu, lit, r);
                            if (in_ring) {
                                for (u32 i = lane; i < L; i += 32) sts8(x.ra(O + i), lds8(cs.rb + ((S + cs.skew + i) & CR_MASK)));
                            } else {
                                x.coop_lit(O, src + S, L);
                            }
                        }
                    }
                    if (!parked) {   // far-match sources requested at decode time have landed in the scratch
                        cp_async_wait_all();
                        cs.pending = 0;
                        parked = true;
                    }
                    // ... then matches.  Everything whose source bytes are final (before this step, in literal
                    // regions, or redirected there by the dependency pass above) goes first: one lane per short
                    // match, warp-wide for the longer ones, in any order.  What is left (DS_HARD: a source that
                    // straddles pending matches) runs warp-wide in lane order.
                    const bool has_m = in && ml > 0;
                    const u32 esrc = msrc - shift;
                    const bool near_lin = esrc >= lo && (esrc & FAST_RMASK) + ml <= FAST_RING;
                    const bool from_scr = staged && shift == 0;
                    const u32 offe = off + shift;
                    const bool lane_ok = has_m && dstate == DS_FINAL && ml <= FAST_MT && offe >= ml &&
                                         (mo & FAST_RMASK) + ml <= FAST_RING && (from_scr || near_lin);
                    const u32 sa = from_scr ? x.scr_s + (msrc - abase) : x.ra(esrc);
                    const u32 dm = x.ra(mo);
                    __syncwarp();
                    const u32 pend = __ballot_sync(0xffffffffu, has_m);
                    if (pend) {
                        const u32 elmask = __ballot_sync(0xffffffffu, lane_ok);
                        if (elmask) lane_copy(sa, dm, lane_ok ? ml : 0u);
                        u32 rest = pend & ~elmask;
                        const u32 hardmask = __ballot_sync(0xffffffffu, has_m && dstate == DS_HARD);
                        const u32 scr_src = from_scr ? sa : 0u;   // linear copy of the source in the scratch
                        while (rest) {
                            int r = __ffs(rest) - 1;
                            rest &= rest - 1;
                            if ((hardmask >> r) & 1u) __syncwarp();   // needs what earlier lanes have just written
                            const u32 MO = __shfl_sync(0xffffffffu, mo, r), OF = __shfl_sync(0xffffffffu, offe, r),
                                      ML = __shfl_sync(0xffffffffu, ml, r), SS = __shfl_sync(0xffffffffu, scr_src, r);
                            if (SS && OF >= ML) {
                                // far source, fetched at decode time (ML <= FAST_ST = 64)
                                const u32 dd = MO + lane;
                                u32 v0 = 0, v1 = 0;
                                if ((u32)lane < ML) v0 = lds8(SS + lane);
                                if ((u32)lane + 32 < ML) v1 = lds8(SS + lane + 32);
                                if ((u32)lane < ML) sts8(x.ra(dd), v0);
                                if ((u32)lane + 32 < ML) sts8(x.ra(dd + 32), v1);
                            } else if (ML <= 64 && OF >= ML && MO - OF >= lo) {
                                // the common case: short, source still in the ring, no self-overlap
                                const u32 a = MO - OF + lane, dd = MO + lane;
                                u32 v0 = 0, v1 = 0;
                                if ((u32)lane < ML) v0 = lds8(x.ra(a));
                                if ((u32)lane + 32 < ML) v1 = lds8(x.ra(a + 32));
                                if ((u32)lane < ML) sts8(x.ra(dd), v0);
                                if ((u32)lane + 32 < ML) sts8(x.ra(dd + 32), v1);
                            } else {
                                x.coop_match(MO, OF, ML, lo);
                            }
                        }
                    }
                    x.done = seg_end;
                    todo &= ~seg;
                    x.flush_full();
                }
            }
        }

        if (false) {
        bail_entry:
            // nothing of this entry has been reported yet: the general decoder starts it over (a block of the sharded
            // path declines instead: the caller re-reads the entry through zpb_unpack_device)
            __syncwarp();
            cp_async_wait_all();
            if (lane == 0) {
                if (partial) { status[idx] = ST_NOT_AVAILABLE; digest[idx] = 0; }
                else general_list[atomicAdd(&counters[CNT_GENERAL], 1u)] = idx;
            }
            continue;
        }
        // ---- finish: last bytes to HBM, XXH3 tail (xxhash.h:3701-3747) from the ring, verdict
        __syncwarp();
        u64 dg;
        {
            u32 span = x.total - x.flushed;
            for (u32 p = x.flushed + 16 * lane; p + 16 <= x.total; p += 512) stg128(x.gout + p, lds128(x.ra(p)));
            for (u32 p = x.flushed + (span & ~15u) + lane; p < x.total; p += 32) x.gout[p] = (u8)lds8(x.ra(p));
        }
        if (partial) {
            dg = e.hash;   // no digest here: every complete KiB has left its stripe sums in `partials`
        } else if (x.total <= 240) {
            __syncwarp();
            dg = xxh3_small(x.gout, x.total);
        } else {
            const u32 lo = x.ring_lo(x.total);
            const int j = lane & 3;
            const u32 tail_start = x.full_blocks << 10;
            const u32 tail_stripes = ((x.total - 1) - tail_start) >> 6;
            u64 s0 = 0, s1 = 0;
            for (u32 s = lane >> 2; s < tail_stripes; s += 8) {
                u32 p = tail_start + 64 * s + 16 * j;
                uint4 v = p >= lo ? lds128(x.ra(p)) : ldg128_coherent(x.gout + p);
                Xxh3Stream<32>::piece(s0, s1, v, c_xxh3_key[s + 2 * j], c_xxh3_key[s + 2 * j + 1]);
            }
            if (lane < 4) {
                u32 p = x.total - 64 + 16 * j;
                u32 w[4];
#pragma unroll
                for (int k = 0; k < 4; ++k)
                    w[k] = x.rd(p + 4 * k, lo) | (x.rd(p + 4 * k + 1, lo) << 8) | (x.rd(p + 4 * k + 2, lo) << 16) |
                           (x.rd(p + 4 * k + 3, lo) << 24);
                Xxh3Stream<32>::piece(s0, s1, make_uint4(w[0], w[1], w[2], w[3]), c_xxh3_key_last[2 * j],
                                      c_xxh3_key_last[2 * j + 1]);
            }
#pragma unroll
            for (int m = 4; m < 32; m <<= 1) {
                s0 += __shfl_xor_sync(0xffffffffu, s0, m);
                s1 += __shfl_xor_sync(0xffffffffu, s1, m);
            }
            u64 a0 = x.acc0 + s0, a1 = x.acc1 + s1;
            u64 m = xxh_fold128(a0 ^ xxh_sec64(11 + 16 * j), a1 ^ xxh_sec64(19 + 16 * j));
            m += __shfl_xor_sync(0xffffffffu, m, 1);
            m += __shfl_xor_sync(0xffffffffu, m, 2);
            dg = xxh3_avalanche((u64)x.total * XXH_P64_1 + m);
        }
        __syncwarp();
        if (lane == 0) {
            status[idx] = (!(e.flags & ZPB_F_NO_VERIFY) && dg != e.hash) ? ST_HASH_MISMATCH : ST_OK;
            digest[idx] = partial ? 0ull : dg;
        }
    }
}
