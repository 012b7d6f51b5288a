// pack_kernel.cuh — stage 2 of the pack path: frames + fused XXH3-64 of the input, one warp per file.
//
// Replaces zpack_compress_file's LZ4 arm (/root/reference/lib/zpack_write.c:192-214:
// LZ4F_compressBegin / Update / End, externals/lz4/lib/lz4frame.c:598-1022) and the second pass
// zpack_add_written_file_entry makes for the digest (lib/zpack_write.c:256).  The 64 KB blocks of every LZ4 file of
// the batch were compressed before this kernel runs, one warp per block, by lz4_pack_blocks_kernel (pack_blocks.cuh)
// — or, for the HC levels with the context's switch on, by the kernels of lz4hc_blocks.cuh — into per-block scratch slots; this kernel lays the frame out — header, block headers, payload from the scratch slot
// or the input itself for a block that did not shrink, EndMark — while the same warp streams the file through XXH3.
//
// Frames are written with B.Indep = 1 (FLG 0x60), 64 KB blocks, no checksums, no content size:
// valid for the reference reader (lz4frame.c:1151,1676) and decodable block-parallel.  A block that
// does not shrink is stored (bit 31), as LZ4F_makeBlock does (lz4frame.c:750-754).  Output bytes are
// not identical to the reference's (the format does not require it); the ratio is reported next to
// the reference's in the tests and the bench.
#pragma once
#include "common.cuh"
#include "xxh3.cuh"
#include "lz4_decode.cuh"
#include "pack_blocks.cuh"
#include "lz4hc_blocks.cuh"
#include "zstd_encode.cuh"
#include "../../include/zpack_b200.h"

#define PK_WARPS 4

// zstd: frame header 14 + per 64 KB block a 3-byte header + at most the raw payload; from ZPB_ZSTD_FRAMED_MIN on, one
// frame per 64 KB block: a header of at most 7 bytes + a 3-byte block header + at most the raw payload
__host__ __device__ inline u64 zstd_pack_bound(u64 size) {
    const u64 nb = size ? (size + 65535) >> 16 : 1;
    return size >= ZPB_ZSTD_FRAMED_MIN ? 10 * nb + size : 14 + 3 * nb + size;
}

__global__ void __launch_bounds__(32 * PK_WARPS)
lz4_pack_kernel(const u8 *__restrict__ in, u64 in_size, u8 *out, u64 out_size, const zpb_file *__restrict__ files,
                const u32 *__restrict__ order, u32 n, u32 *counter, u64 *comp_size, u64 *digest, int *status,
                const u32 *__restrict__ blk_base, const u8 *__restrict__ scratch, const u32 *__restrict__ csize,
                const u8 *__restrict__ zslot, const u32 *__restrict__ zbody, const u32 *__restrict__ winop, int lz4hc) {
    const int lane = threadIdx.x & 31;
    Group<32> g;
    for (;;) {
        u32 slot = 0;
        if (lane == 0) slot = atomicAdd(counter, 1u);
        slot = __shfl_sync(0xffffffffu, slot, 0);
        if (slot >= n) break;
        const u32 idx = order ? order[slot] : slot;
        const zpb_file f = files[idx];
        int st = ST_OK;
        u64 csz = 0, dg = 0;
        if (f.src_off > in_size || f.size > in_size - f.src_off || f.dst_off > out_size ||
            f.dst_cap > out_size - f.dst_off) {
            st = ZPB_ST_COMPRESS_FAILED;
        } else if (f.method == ZPB_METHOD_NONE) {              // zpack_write.c:216-219
            if (f.dst_cap < f.size) st = ZPB_ST_COMPRESS_FAILED;
            else {
                const u8 *src = in + f.src_off;
                u8 *dst = out + f.dst_off;
                Xxh3Stream<32> hs;
                hs.init(src, f.size, g);
                for (u64 done = 0; done < f.size;) {
                    u64 chunk = f.size - done;
                    if (chunk > (1u << 20)) chunk = 1u << 20;
                    group_copy<32>(g, dst + done, src + done, (u32)chunk);
                    done += chunk;
                    hs.advance(done, g);
                }
                dg = hs.finish(g);
                csz = f.size;
            }
        } else if (f.method == ZPB_METHOD_LZ4) {
            const u64 nblocks = (f.size + 65535) >> 16;
            if (f.dst_cap < 7 + 4 * nblocks + f.size + 4) st = ZPB_ST_COMPRESS_FAILED;  // LZ4F_compressBound role
            else if (f.level >= 3 && !lz4hc) st = ST_NOT_AVAILABLE;   // lz4frame.c:799-807 selects LZ4 HC from level 3 on: only with the context's HC switch (lz4hc_blocks.cuh); never a silent downgrade
            else {
                const u8 *src = in + f.src_off;
                u8 *dst = out + f.dst_off;
                // frame header: magic, FLG (v01, B.Indep), BD (64 KB), HC (lz4frame.c:669-700)
                if (lane == 0) {
                    dst[0] = 0x04; dst[1] = 0x22; dst[2] = 0x4D; dst[3] = 0x18; dst[4] = 0x60; dst[5] = 0x40;
                }
                __syncwarp();
                u32 hc = (xxh32_dev(dst + 4, 2, 0) >> 8) & 0xFF;
                if (lane == 0) dst[6] = (u8)hc;
                u64 op = 7;
                const u32 b0 = blk_base[idx];                           // this file's first block in the stage-1 list
                Xxh3Stream<32> hs;
                hs.init(src, f.size, g);
                for (u64 b = 0; b < nblocks; ++b) {
                    const u32 blen = (u32)(f.size - (b << 16) < 65536 ? f.size - (b << 16) : 65536);
                    const u8 *bsrc = src + (b << 16);
                    u32 c = csize[b0 + b];
                    u32 hdr = c;
                    if (c) group_copy<32>(g, dst + op + 4, scratch + ((u64)(b0 + b) << 16), c);
                    else {                                              // stored (lz4frame.c:750-754)
                        group_copy<32>(g, dst + op + 4, bsrc, blen);
                        c = blen;
                        hdr = blen | 0x80000000u;
                    }
                    if (lane == 0) {
                        dst[op] = (u8)hdr; dst[op + 1] = (u8)(hdr >> 8); dst[op + 2] = (u8)(hdr >> 16); dst[op + 3] = (u8)(hdr >> 24);
                    }
                    op += 4 + c;
                    hs.advance((b << 16) + blen, g);
                }
                if (lane < 4) dst[op + lane] = 0;                      // EndMark
                op += 4;
                dg = hs.finish(g);
                csz = op;
            }
        } else if (f.method == ZPB_METHOD_ZSTD) {
            // A zstd frame of 64 KB blocks (zstd_compression_format.md:320-404): Compressed_Blocks whose bodies
            // zstd_encode_blocks_kernel built from the block compressor's matches (raw literals + predefined-mode FSE
            // sequences), Raw_Blocks where that did not shrink the block.  From ZPB_ZSTD_FRAMED_MIN on, every 64 KB
            // block is a frame of its own (the same blocks behind a single-segment header): the frames say what the
            // blocks already are — independent — so a reader can decode them in parallel (zpb_zstd_frame_index).
            const u64 nblocks = f.size ? (f.size + 65535) >> 16 : 1;
            const bool framed = f.size >= ZPB_ZSTD_FRAMED_MIN;
            if (f.dst_cap < zstd_pack_bound(f.size)) st = ZPB_ST_COMPRESS_FAILED;
            else {
                const u8 *src = in + f.src_off;
                u8 *dst = out + f.dst_off;
                const u32 b0 = blk_base[idx];
                if (lane == 0 && !framed) {
                    // magic; FHD: 8-byte frame content size, no single-segment, no checksum, no dictionary; window 128 KB
                    dst[0] = 0x28; dst[1] = 0xB5; dst[2] = 0x2F; dst[3] = 0xFD; dst[4] = 0xC0; dst[5] = 0x38;
                    for (int k = 0; k < 8; ++k) dst[6 + k] = (u8)(f.size >> (8 * k));
                }
                u64 op = framed ? 0 : 14;
                Xxh3Stream<32> hs;
                hs.init(src, f.size, g);
                for (u64 b = 0; b < nblocks; ++b) {
                    const u32 blen = (u32)(f.size - (b << 16) < 65536 ? f.size - (b << 16) : 65536);
                    const u64 bb = b0 + b;
                    const bool last_block = framed || b + 1 == nblocks;
                    if (framed) {
                        // magic; FHD: single segment (the window is the content), no checksum, no dictionary, and the
                        // smallest Frame_Content_Size field: 1 byte up to 255, else 2 bytes holding size - 256
                        if (lane == 0) {
                            dst[op] = 0x28; dst[op + 1] = 0xB5; dst[op + 2] = 0x2F; dst[op + 3] = 0xFD;
                            if (blen < 256) { dst[op + 4] = 0x20; dst[op + 5] = (u8)blen; }
                            else { dst[op + 4] = 0x60; dst[op + 5] = (u8)(blen - 256); dst[op + 6] = (u8)((blen - 256) >> 8); }
                        }
                        op += blen < 256 ? 6 : 7;
                    }
                    // the block's windows: lanes 0-15 look at one body size each; any failure, or bodies that are not
                    // smaller than the block, and it is stored raw
                    u32 zw = f.size && lane < 16 ? zbody[bb * ZE_ZBODY + lane] : 0u;
                    const bool zfail = !f.size || __any_sync(0xffffffffu, zw == ZE_FAIL);
                    u32 ztotal = zw && zw != ZE_FAIL ? zw + 3u : 0u;
                    for (int d = 16; d; d >>= 1) ztotal += __shfl_xor_sync(0xffffffffu, ztotal, d);
                    if (!zfail && ztotal && ztotal < blen) {
                        // one Compressed_Block per window of the block compressor that emitted something; the last
                        // window always does (it carries the block's closing literals)
                        const u32 nwin = (blen - 12u) / 4096u + 1u;
                        for (u32 w = 0; w < nwin; ++w) {
                            const u32 z = __shfl_sync(0xffffffffu, zw, (int)w);
                            if (!z) continue;
                            const u32 hdr = ((last_block && w + 1 == nwin) ? 1u : 0u) | (2u << 1) | (z << 3);
                            if (lane == 0) { dst[op] = (u8)hdr; dst[op + 1] = (u8)(hdr >> 8); dst[op + 2] = (u8)(hdr >> 16); }
                            group_copy<32>(g, dst + op + 3, zslot + bb * ZE_SLOT + ZE_OFF(winop[bb * 17u + w], w), z);
                            op += 3 + z;
                        }
                    } else {
                        const u32 hdr = (last_block ? 1u : 0u) | (blen << 3);                      // Raw_Block
                        if (lane == 0) { dst[op] = (u8)hdr; dst[op + 1] = (u8)(hdr >> 8); dst[op + 2] = (u8)(hdr >> 16); }
                        group_copy<32>(g, dst + op + 3, src + (b << 16), blen);
                        op += 3 + blen;
                    }
                    hs.advance((b << 16) + blen, g);
                }
                dg = hs.finish(g);
                csz = op;
            }
        } else {
            st = ST_METHOD_INVALID;
        }
        __syncwarp();
        if (lane == 0) {
            comp_size[idx] = csz;
            digest[idx] = dg;
            status[idx] = st;
        }
    }
}
