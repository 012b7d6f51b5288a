// split_entries.cuh — large entries of a batch decoded block-parallel inside zpb_unpack_device.
//
// A row of a public unpack call is a candidate when it is LZ4 or zstd, decodes to at least ZPB_ZSTD_FRAMED_MIN bytes
// and passes the scan kernel's guards.  The host reserves ceil(uncomp_size / 64 KB) pseudo-rows after the caller's n
// rows (zpb_api.cu); split_index_kernel walks the entry's framing on the device and, when the entry has the shape of
// zpb_lz4_frame_index / zpb_zstd_frame_index, fills them with one ZPB_M_LZ4_BLOCK or ZPB_M_ZSTD_FRAME row per 64 KB,
// the rows zpb_unpack_blocks_device builds on the host.  They go through scan -> parse -> exec / zstd like any row and
// leave per-KiB XXH3 stripe sums; xxh3_chain_batch_kernel (xxh3_chain.cuh) folds them into the parent's digest.
//
// The accepted shape is defined once, by the header checks below, which the host index functions (blocks_api.inl) use
// as well; only the loops that walk the headers differ.
#pragma once
#include "common.cuh"
#include "lz4_fast.cuh"
#include "ptx.cuh"

#define ZPB_HD __host__ __device__ __forceinline__

ZPB_HD u32 split_rd32(const u8 *p) { return (u32)p[0] | ((u32)p[1] << 8) | ((u32)p[2] << 16) | ((u32)p[3] << 24); }

// The header of an LZ4 frame of independent 64 KB blocks without checksums.  h: the frame's first min(comp_size, 19)
// bytes.  Returns the header size (its block headers follow), or 0 when the frame does not have that shape.
// *content = the Content Size field, or ~0 when absent.
ZPB_HD u32 split_lz4_header(const u8 *h, u64 comp_size, u64 *content) {
    *content = ~0ull;
    if (comp_size < 11 || split_rd32(h) != 0x184D2204u) return 0;
    const u32 flg = h[4], bd = h[5];
    // version 01, reserved bits clear, B.Indep = 1, no block / content checksums (their XXH32 chains are not
    // part of this path), 64 KB blocks (the fast kernels' block size)
    if (((flg >> 6) & 3) != 1 || (flg & 2) || !((flg >> 5) & 1) || ((flg >> 4) & 1) || ((flg >> 2) & 1)) return 0;
    if ((bd >> 7) || ((bd >> 4) & 7) != 4 || (bd & 15)) return 0;
    const bool has_size = (flg >> 3) & 1, has_dict = flg & 1;
    const u32 hsize = 7 + (has_size ? 8 : 0) + (has_dict ? 4 : 0);
    if (comp_size < hsize + 4ull) return 0;
    // header checksum byte (lz4frame.c:294-298, 1184-1186): XXH32 of the descriptor, <= 14 bytes
    {
        const u8 *p = h + 4;
        const u32 len = hsize - 5;
        const u32 P1 = 0x9E3779B1u, P2 = 0x85EBCA77u, P3 = 0xC2B2AE3Du, P4 = 0x27D4EB2Fu, P5 = 0x165667B1u;
        u32 x = P5 + len, i = 0;   // len < 16: no stripe loop
        for (; i + 4 <= len; i += 4) {
            x += split_rd32(p + i) * P3;
            x = ((x << 17) | (x >> 15)) * P4;
        }
        for (; i < len; ++i) {
            x += p[i] * P5;
            x = ((x << 11) | (x >> 21)) * P1;
        }
        x ^= x >> 15; x *= P2; x ^= x >> 13; x *= P3; x ^= x >> 16;
        if (((x >> 8) & 0xFF) != h[hsize - 1]) return 0;
    }
    if (has_size) *content = (u64)split_rd32(h + 6) | ((u64)split_rd32(h + 10) << 32);
    return hsize;
}

// An LZ4 block header's size field (end mark excluded) with `left` bytes after the header: whether the block fits.
ZPB_HD bool split_lz4_block_ok(u32 bsz, u64 left) { return bsz != 0 && bsz <= 65536u && bsz <= left; }

// The header of one zstd frame of this library's large layout: Frame_Content_Size present and 1..65536, no checksum, no
// dictionary, not skippable.  h: the frame's first min(left, 14) bytes, `left` = bytes from the frame's start to the end
// of the entry.  Returns the header size, or 0; *fcs = Frame_Content_Size.
ZPB_HD u32 split_zstd_header(const u8 *h, u64 left, u32 *fcs) {
    if (left < 6 || split_rd32(h) != 0xFD2FB528u) return 0;   // skippable frames too
    const u32 fhd = h[4];
    const u32 fcs_code = fhd >> 6, single = (fhd >> 5) & 1;
    if ((fhd & 8) || (fhd & 4) || (fhd & 3) || (!single && !fcs_code)) return 0;   // reserved, checksum, dictionary, no FCS
    const u32 fcs_len = fcs_code ? 1u << fcs_code : 1u;
    const u32 hsize = 5 + (single ? 0 : 1) + fcs_len;
    if (left < hsize) return 0;
    u64 v = 0;
    for (int k = (int)fcs_len - 1; k >= 0; --k) v = (v << 8) | h[hsize - fcs_len + k];
    if (fcs_code == 1) v += 256;
    if (v == 0 || v > 65536) return 0;
    *fcs = (u32)v;
    return hsize;
}

// A 3-byte zstd block header with `left` bytes after it: the bytes the block occupies after its header, or ~0u when
// the block type is reserved or the block does not fit.
ZPB_HD u32 split_zstd_block(u32 bh, u64 left) {
    const u32 type = (bh >> 1) & 3, csz = type == 1 ? 1u : bh >> 3;
    return type == 3 || csz > left ? ~0u : csz;
}

// Internal status of a split parent whose pseudo-rows did not all decode: it is decoded again, unsplit (by the host in
// zpb_unpack_device, after split_retry_kernel in zpb_unpack_device_async).
#define ZPB_ST_SPLIT_RETRY 0x5350u

struct SplitJob {      // host -> pre-pass -> chain kernel -> retry kernel, one per candidate
    u64 kib0;          // its first KiB in the batch's stripe-sum array
    u64 desc_base;     // LZ4: descriptor words reserved for its blocks (fast_scan_lz4's layout)
    u32 parent;        // the caller's row
    u32 row0, nrows;   // its pseudo-rows: [row0, row0 + nrows), nrows = ceil(uncomp_size / 64 KB)
    u32 slot_base;     // LZ4: its FastBlock slots
    u32 method;        // the parent's method (ZPB_METHOD_LZ4 / _ZSTD), which the pre-pass replaces with ZPB_M_SPLIT
};

#define SPLIT_CHUNK 65536u                       // entry bytes per stage; a header starting in a stage is walked there
#define SPLIT_PAD   64u                          // bytes staged past the stage: every header is contiguous (<= 19 bytes)
#define SPLIT_BUF   (SPLIT_CHUNK + SPLIT_PAD + 32u)
#define SPLIT_SMEM  (16u + 2u * SPLIT_BUF)       // two mbarriers, two stages

// One warp per candidate.  The compressed bytes stream through two shared-memory stages (cp.async.bulk, the unaligned
// ends by ordinary loads) while the walk of the previous stage runs; every lane walks the same headers (broadcast
// reads), lane 0 writes the rows.  Every read is inside the entry's compressed range.
__global__ void __launch_bounds__(32)
split_index_kernel(const u8 *__restrict__ archive, zpb_entry *entries, FastAux *aux, const SplitJob *__restrict__ jobs) {
    ZPB_DYN_SMEM(split_smem);
    u8 *sm = reinterpret_cast<u8 *>(split_smem);
    const u32 lane = threadIdx.x & 31u;
    const SplitJob j = jobs[blockIdx.x];
    const zpb_entry pe = entries[j.parent];
    const u8 *src = archive + pe.src_off;
    const u64 n = pe.comp_size;
    const bool zstd = pe.method == ZPB_METHOD_ZSTD;
    const u32 bar0 = smem_window(sm);
    const u32 skew = (u32)(uintptr_t)src & 15u;
    if (lane == 0) { mbar_init(bar0, 1); mbar_init(bar0 + 8, 1); mbar_fence_init(); }
    __syncthreads();
    const u64 nchunks = (n + SPLIT_CHUNK - 1) / SPLIT_CHUNK;
    auto stage = [&](u64 c) {   // entry bytes [c CHUNK, min((c + 1) CHUNK + PAD, n)) -> stage c & 1, at the same offset mod 16
        const u64 p0 = c * SPLIT_CHUNK;
        const u32 len = (u32)((p0 + SPLIT_CHUNK + SPLIT_PAD < n ? p0 + SPLIT_CHUNK + SPLIT_PAD : n) - p0);
        const u32 D = 16u + (u32)(c & 1) * SPLIT_BUF + skew, bar = bar0 + 8u * (u32)(c & 1);
        const u8 *g = src + p0;
        u32 head = (16u - skew) & 15u;
        if (head > len) head = len;
        const u32 al = (len - head) & ~15u;
        if (lane == 0) {
            mbar_arrive_expect_tx(bar, al);
            for (u32 o = 0; o < al; o += 16384u) bulk_g2s(bar0 + D + head + o, g + head + o, al - o < 16384u ? al - o : 16384u, bar);
        }
        for (u32 i = lane; i < head; i += 32) sm[D + i] = g[i];
        for (u32 i = head + al + lane; i < len; i += 32) sm[D + i] = g[i];
    };
    // walk state: ip = the next header; zstd: whether it is a frame header, the frame's start and content size
    u64 ip = 0, f0 = 0, total = 0;
    u32 k = 0, fcs = 0;
    bool in_frame = false, short_seen = false;
    int verdict = 0;   // 0 walking, 1 accepted, -1 declined
    u64 c = 0;
    stage(0);
    for (; c < nchunks && verdict == 0; ++c) {
        if (c + 1 < nchunks) stage(c + 1);
        mbar_wait(bar0 + 8u * (u32)(c & 1), (u32)(c >> 1) & 1u);
        __syncthreads();
        const u8 *base = sm + 16u + (u32)(c & 1) * SPLIT_BUF + skew - c * SPLIT_CHUNK;   // entry byte p is base[p]
        const u64 lim = (c + 1) * SPLIT_CHUNK < n ? (c + 1) * SPLIT_CHUNK : n;
        while (verdict == 0 && ip < lim) {
            if (!zstd) {
                if (ip == 0) {
                    u64 content;
                    const u32 hs = split_lz4_header(base, n, &content);
                    if (!hs || (content != ~0ull && content != pe.uncomp_size)) { verdict = -1; break; }
                    ip = hs;
                    continue;
                }
                if (n - ip < 4) { verdict = -1; break; }
                const u32 bh = split_rd32(base + ip);
                ip += 4;
                if (bh == 0) { verdict = ip == n && k == j.nrows ? 1 : -1; break; }   // trailing bytes: another frame
                const u32 bsz = bh & 0x7FFFFFFFu;
                if (!split_lz4_block_ok(bsz, n - ip) || k == j.nrows) { verdict = -1; break; }
                if (lane == 0) {
                    const u64 usz = k + 1 < j.nrows ? 65536ull : pe.uncomp_size - 65536ull * (j.nrows - 1);
                    zpb_entry r;
                    r.src_off = pe.src_off + ip; r.comp_size = bsz;
                    r.dst_off = pe.dst_off + 65536ull * k; r.dst_cap = usz; r.uncomp_size = usz;
                    r.hash = 0; r.method = ZPB_M_LZ4_BLOCK; r.flags = (bh >> 31) ? ZPB_F_STORED_BLK : 0u;
                    r.reserved = j.kib0 + 64ull * k;
                    entries[j.row0 + k] = r;
                    FastAux a;
                    a.desc_base = j.desc_base + (((ip / 3) + FAST_DESC_PER_BLOCK * k + 3ull) & ~3ull);
                    a.slot_base = j.slot_base + k; a.nslots = 1;
                    aux[j.row0 + k] = a;
                }
                ip += bsz;
                ++k;
            } else if (!in_frame) {
                const u32 hs = short_seen ? 0u : split_zstd_header(base + ip, n - ip, &fcs);
                if (!hs) { verdict = -1; break; }
                short_seen = fcs < 65536u;   // a frame of less than 64 KB ends the entry
                f0 = ip;
                ip += hs;
                in_frame = true;
            } else {
                if (n - ip < 3) { verdict = -1; break; }
                const u32 bh = split_rd32(base + ip) & 0xFFFFFFu;
                ip += 3;
                const u32 csz = split_zstd_block(bh, n - ip);
                if (csz == ~0u) { verdict = -1; break; }
                ip += csz;
                if (!(bh & 1)) continue;
                in_frame = false;
                if (ip - f0 > 0xFFFFFFFFull || k == j.nrows) { verdict = -1; break; }
                if (lane == 0) {
                    zpb_entry r;
                    r.src_off = pe.src_off + f0; r.comp_size = ip - f0;
                    r.dst_off = pe.dst_off + 65536ull * k; r.dst_cap = fcs; r.uncomp_size = fcs;
                    r.hash = 0; r.method = ZPB_M_ZSTD_FRAME; r.flags = 0;
                    r.reserved = j.kib0 + 64ull * k;
                    entries[j.row0 + k] = r;
                }
                total += fcs;
                ++k;
            }
        }
        __syncthreads();   // stage c & 1 is free for chunk c + 2
    }
    if (c < nchunks) mbar_wait(bar0 + 8u * (u32)(c & 1), (u32)(c >> 1) & 1u);   // a stage still in flight lands first
    if (verdict == 0) verdict = zstd && !in_frame && ip == n && k == j.nrows && total == pe.uncomp_size ? 1 : -1;
    if (verdict > 0) {
        if (lane == 0) entries[j.parent].method = ZPB_M_SPLIT;
    } else {
        for (u32 r = lane; r < k; r += 32) entries[j.row0 + r].comp_size = 0;   // inert: the scan kernel reports them OK
    }
}

// One thread per candidate, after xxh3_chain_batch_kernel (zpb_unpack_device_async): a parent marked ZPB_ST_SPLIT_RETRY
// gets its method back and joins the list of the whole-entry decoder it would have reached unsplit, so that its status
// is that path's.  LZ4 -> lz4_list, for the general kernel, which judges every LZ4 entry the fast path declines (a
// fast-path decode of a valid frame and the general kernel's agree); zstd -> zstd_list, for zstd_unpack_kernel<ZsHasher>.
// The lists' lengths are counted at CNT_RETRY_LZ4 and CNT_RETRY_ZSTD.
__global__ void __launch_bounds__(128)
split_retry_kernel(const SplitJob *__restrict__ jobs, u32 njobs, zpb_entry *entries, const int *__restrict__ status,
                   u32 *lz4_list, u32 *zstd_list, u32 *counters) {
    const u32 t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= njobs) return;
    const SplitJob j = jobs[t];
    if (status[j.parent] != (int)ZPB_ST_SPLIT_RETRY) return;
    entries[j.parent].method = j.method;
    if (j.method == ZPB_METHOD_ZSTD) zstd_list[atomicAdd(&counters[CNT_RETRY_ZSTD], 1u)] = j.parent;
    else lz4_list[atomicAdd(&counters[CNT_RETRY_LZ4], 1u)] = j.parent;
}

#ifndef ZPB_SIM   // the chain's inline PTX has no CPU emulation
#include "xxh3_chain.cuh"

// One warp per candidate, after every pseudo-row has decoded: the XXH3 chain over the entry's stripe sums, the tail and
// the merge (xxh3_chain_body), then the parent's status and digest as the one-warp path reports them.  A parent with a
// pseudo-row that did not decode is marked ZPB_ST_SPLIT_RETRY for the unsplit pass.
__global__ void __launch_bounds__(32)
xxh3_chain_batch_kernel(const SplitJob *__restrict__ jobs, const zpb_entry *__restrict__ entries, const u64 *partials,
                        const u8 *out, int *status, u64 *digest) {
    __shared__ ulonglong2 stage[XC_STAGES][XC_BATCH * 4];
    const u32 lane = threadIdx.x & 31u;
    const SplitJob j = jobs[blockIdx.x];
    const zpb_entry e = entries[j.parent];
    if (e.method != ZPB_M_SPLIT) return;   // the pre-pass declined it: the scan kernel took the row as it is
    bool bad = false;
    for (u32 r = lane; r < j.nrows; r += 32) bad |= status[j.row0 + r] != ST_OK;
    if (__any_sync(0xffffffffu, bad)) {
        if (lane == 0) { status[j.parent] = ZPB_ST_SPLIT_RETRY; digest[j.parent] = 0; }
        return;
    }
    const u64 dg = xxh3_chain_body(stage, partials + j.kib0 * 8, (e.uncomp_size - 1) >> 10, nullptr, nullptr, 1,
                                   out + e.dst_off, 0, e.uncomp_size);
    if (lane == 0) {
        status[j.parent] = (!(e.flags & ZPB_F_NO_VERIFY) && dg != e.hash) ? ST_HASH_MISMATCH : ST_OK;
        digest[j.parent] = dg;
    }
}
#endif
