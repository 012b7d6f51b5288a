// zpb_api.cu — host side of the C-ABI in include/zpack_b200.h: context, scratch arenas,
// work ordering, launches and CUDA-event timing.  No torch, no CPU codec: every entry is
// (de)compressed and hashed on the device or the call fails.
#include <algorithm>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <chrono>
#include <numeric>
#include <string>
#include <thread>
#include <vector>

#include "../../include/zpack_b200.h"
#include "unpack_kernel.cuh"
#include "lz4_fast.cuh"
#include "pack_kernel.cuh"
#include "zstd_decode.cuh"
#include "xxh3_chain.cuh"
#include "archive_kernels.cuh"

static thread_local std::string g_last_error = "";

struct DevBuf {
    void *p = nullptr;
    size_t cap = 0;
    bool ensure(size_t n) {
        if (n <= cap) return true;
        if (p) cudaFree(p);
        p = nullptr; cap = 0;
        size_t want = std::max(n, (size_t)4096);
        if (cudaMalloc(&p, want) != cudaSuccess) { p = nullptr; return false; }
        cap = want;
        return true;
    }
    void release() { if (p) cudaFree(p); p = nullptr; cap = 0; }
};
struct PinBuf {
    void *p = nullptr;
    size_t cap = 0;
    bool ensure(size_t n) {
        if (n <= cap) return true;
        if (p) cudaFreeHost(p);
        p = nullptr; cap = 0;
        size_t want = std::max(n, (size_t)4096);
        if (cudaMallocHost(&p, want) != cudaSuccess) { p = nullptr; return false; }
        cap = want;
        return true;
    }
    void release() { if (p) cudaFreeHost(p); p = nullptr; cap = 0; }
};

struct zpb_ctx {
    int device = 0;
    int sm_count = 0, cc_major = 0, cc_minor = 0;
    cudaStream_t stream = nullptr;
    cudaEvent_t ev0 = nullptr, ev1 = nullptr;
    std::string err;
    uint64_t launches = 0;
    float unpack_ms = 0.f, pack_ms = 0.f;
    int group = 32;       // lanes per chain in the general kernel (tunable: ZPB_GROUP)
    int ctas_per_sm = 0;  // 0 = occupancy API
    int fast = 1;         // scan/parse/exec pipeline for LZ4 + stored entries (ZPB_FAST=0: general kernel only)
    float stage_ms[4] = {0, 0, 0, 0};
    DevBuf d_aux, d_fe, d_fb, d_plist, d_glist, d_fdesc;
    DevBuf d_zlist, d_zlit;  // zstd work list, per-warp literal buffers
    int zs_grid = 0;         // persistent grid of zstd_unpack_kernel (CTAs)
    float zstd_ms = 0.f;
    cudaEvent_t evs[6] = {nullptr, nullptr, nullptr, nullptr, nullptr, nullptr};
    // the execute kernel runs on its own stream so that it overlaps the tail of the parse kernel
    cudaStream_t stream_p = nullptr, stream_b = nullptr;   // parse (high priority), the late third of the execute grid
    cudaEvent_t ev_scan = nullptr, ev_x0 = nullptr, ev_x1 = nullptr, ev_p0 = nullptr, ev_p1 = nullptr, ev_xb = nullptr;
    DevBuf d_order2, d_defer;
    int overlap = 1;         // ZPB_OVERLAP=0: parse, then execute, on one stream
    // descriptor / result scratch
    DevBuf d_desc, d_order, d_res, d_counter;
    std::vector<uint16_t> h_keys;   // cost key per entry of the batch being prepared
    PinBuf h_stage;
    // staging arenas for the *_host entry points
    DevBuf d_in, d_out;
    DevBuf d_gather, d_goff;   // pack: compacted frames + their sizes / offsets
    PinBuf h_bounce;           // pack: landing zone of the one D2H per chunk
    DevBuf d_pblk, d_pscratch, d_csize;    // pack: block list, one 64 KB payload slot per block of a round, block sizes
    DevBuf d_zslot, d_zseq, d_zmeta;       // pack, zstd files: block bodies, sequence records, window offsets + per-window words of a round
    DevBuf d_zelit, d_zhuf, d_ztabs;       // ... staged literals, one Huffman code and one set of FSE tables per block
    u64 pack_scratch_blocks = 16384;       // slots per round (ZPB_PACK_SCRATCH_MB, default 1 GiB)
    int p2_per_sm = 1, pk_per_sm = 1;      // resident CTAs of the two pack kernels
    std::vector<cudaEvent_t> pack_evs;     // three per round: before the block compressor, between, after the framing kernel
    float pack_blocks_ms = 0.f, pack_frames_ms = 0.f;
    int lz4hc = 0;                         // LZ4 levels >= 3 by the HC compressor (ZPB_LZ4HC=1); off: refused with ZPB_ST_NOT_AVAILABLE
    DevBuf d_hcrec;                        // pack, HC blocks of a round: per-position match records and parse costs
    // pipelined host path: private sub-contexts (own stream + scratch), one per worker thread
    std::vector<zpb_ctx *> workers;
    // block-sharded path (one large block-independent LZ4 entry): per-KiB XXH3 stripe sums of the last shard
    DevBuf d_partials, d_acc;
    u64 *cur_partials = nullptr;       // non-null only while zpb_unpack_blocks_device drives the pipeline
    u64 blk_uncomp = 0;                // decoded bytes of the last shard (0 = none / declined)
    float chain_ms = 0.f;
    int host_workers = 6;              // ZPB_HOST_WORKERS (tools/e2e_sweep.py: profiles/r1_e2e_sweep.jsonl)
    u64 host_chunk_bytes = 256u << 20; // decoded bytes per pipeline chunk (ZPB_HOST_CHUNK_MB)
    // device-resident container operations (archive_api.inl): entry table, record offsets, chunk table, totals, names; CDR walk tables
    DevBuf d_arc_e, d_arc_rec, d_arc_chunk, d_arc_work, d_arc_scan, d_arc_tot, d_arc_names, d_cdr_jump, d_cdr_cnt, d_cdr_j2, d_cdr_anchor;
    int arc_dynamic = 1, arc_head_mask = 127;  // copy kernel: chunks drawn from a counter (ZPB_ARC_DYNAMIC=0: fixed deal), head bytes up to the 128-byte grid (ZPB_ARC_HEAD=15: 16-byte grid)
    int arc_ctas_per_sm = 4;           // copy kernel: CTAs per SM (ZPB_ARC_CTAS)
    float arc_ms[3] = {0, 0, 0};       // layout + directory kernels, copy kernel, open kernels of the last call
};

#define CK(ctx, call)                                                                      \
    do {                                                                                   \
        cudaError_t e_ = (call);                                                           \
        if (e_ != cudaSuccess) {                                                           \
            (ctx)->err = std::string(#call) + ": " + cudaGetErrorString(e_);               \
            g_last_error = (ctx)->err;                                                     \
            return ZPB_E_CUDA;                                                             \
        }                                                                                  \
    } while (0)

static int fail(zpb_ctx *ctx, int code, const char *msg) {
    if (ctx) ctx->err = msg;
    g_last_error = msg;
    return code;
}

extern "C" int zpb_abi_version(void) { return ZPB_ABI_VERSION; }

extern "C" const char *zpb_last_error(const zpb_ctx *ctx) {
    return ctx ? ctx->err.c_str() : g_last_error.c_str();
}

extern "C" zpb_ctx *zpb_create(int device) {
    int count = 0;
    cudaError_t e = cudaGetDeviceCount(&count);
    if (e != cudaSuccess || count == 0) {
        g_last_error = std::string("no CUDA device: ") + cudaGetErrorString(e);
        return nullptr;
    }
    if (device < 0 || device >= count) { g_last_error = "device index out of range"; return nullptr; }
    if (cudaSetDevice(device) != cudaSuccess) { g_last_error = "cudaSetDevice failed"; return nullptr; }
    zpb_ctx *ctx = new zpb_ctx();
    ctx->device = device;
    cudaDeviceProp prop;
    if (cudaGetDeviceProperties(&prop, device) != cudaSuccess) {
        g_last_error = "cudaGetDeviceProperties failed"; delete ctx; return nullptr;
    }
    ctx->sm_count = prop.multiProcessorCount;
    ctx->cc_major = prop.major;
    ctx->cc_minor = prop.minor;
    if (cudaStreamCreateWithFlags(&ctx->stream, cudaStreamNonBlocking) != cudaSuccess ||
        cudaEventCreate(&ctx->ev0) != cudaSuccess || cudaEventCreate(&ctx->ev1) != cudaSuccess ||
        xxh3_upload_tables() != cudaSuccess) {
        g_last_error = std::string("context setup failed: ") + cudaGetErrorString(cudaGetLastError());
        delete ctx; return nullptr;
    }
    if (const char *s = getenv("ZPB_GROUP")) {
        int v = atoi(s);
        if (v == 4 || v == 8 || v == 16 || v == 32) ctx->group = v;
    }
    if (const char *s = getenv("ZPB_CTAS_PER_SM")) ctx->ctas_per_sm = atoi(s);
    if (const char *s = getenv("ZPB_FAST")) ctx->fast = atoi(s);
    if (const char *s = getenv("ZPB_ARC_DYNAMIC")) ctx->arc_dynamic = atoi(s) != 0;
    if (const char *s = getenv("ZPB_ARC_HEAD")) ctx->arc_head_mask = atoi(s) == 127 ? 127 : 15;
    if (const char *s = getenv("ZPB_ARC_CTAS")) ctx->arc_ctas_per_sm = std::max(1, std::min(8, atoi(s)));
    if (const char *s = getenv("ZPB_HOST_WORKERS")) ctx->host_workers = std::max(1, std::min(8, atoi(s)));
    if (const char *s = getenv("ZPB_HOST_CHUNK_MB")) ctx->host_chunk_bytes = (u64)std::max(1, atoi(s)) << 20;
    for (auto &ev : ctx->evs)
        if (cudaEventCreate(&ev) != cudaSuccess) { g_last_error = "event setup failed"; delete ctx; return nullptr; }
    int prio_lo = 0, prio_hi = 0;
    cudaDeviceGetStreamPriorityRange(&prio_lo, &prio_hi);
    if (cudaStreamCreateWithPriority(&ctx->stream_p, cudaStreamNonBlocking, prio_hi) != cudaSuccess ||
        cudaStreamCreateWithPriority(&ctx->stream_b, cudaStreamNonBlocking, prio_lo) != cudaSuccess ||
        cudaEventCreateWithFlags(&ctx->ev_scan, cudaEventDisableTiming) != cudaSuccess ||
        cudaEventCreateWithFlags(&ctx->ev_xb, cudaEventDisableTiming) != cudaSuccess ||
        cudaEventCreate(&ctx->ev_p0) != cudaSuccess || cudaEventCreate(&ctx->ev_p1) != cudaSuccess ||
        cudaEventCreate(&ctx->ev_x0) != cudaSuccess || cudaEventCreate(&ctx->ev_x1) != cudaSuccess) {
        g_last_error = "second stream setup failed"; delete ctx; return nullptr;
    }
    if (const char *e = getenv("ZPB_OVERLAP")) ctx->overlap = atoi(e);
    if (cudaFuncSetAttribute(lz4_fast_parse_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                             (int)(K1_THREADS * K1_ROW)) != cudaSuccess ||
        cudaFuncSetAttribute(lz4_fast_parse4_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                             (int)(K1_THREADS * K1_ROW)) != cudaSuccess ||
        cudaFuncSetAttribute(lz4_fast_exec_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                             (int)(FAST_EXEC_SMEM)) != cudaSuccess) {
        g_last_error = std::string("kernel attribute setup failed: ") + cudaGetErrorString(cudaGetLastError());
        delete ctx; return nullptr;
    }
    {
        int per_sm = 0;
        const int smem = (int)(ZS_WARPS * sizeof(ZstdShared));
        if (cudaFuncSetAttribute(zstd_unpack_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, smem) != cudaSuccess ||
            cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, zstd_unpack_kernel, ZS_WARPS * 32, smem) != cudaSuccess ||
            per_sm < 1) {
            g_last_error = std::string("zstd kernel setup failed: ") + cudaGetErrorString(cudaGetLastError());
            delete ctx; return nullptr;
        }
        ctx->zs_grid = ctx->sm_count * per_sm;
    }
    if (cudaFuncSetAttribute(lz4_pack_blocks_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)P2_SMEM) != cudaSuccess ||
        cudaOccupancyMaxActiveBlocksPerMultiprocessor(&ctx->p2_per_sm, lz4_pack_blocks_kernel, 32 * P2_WARPS, P2_SMEM) != cudaSuccess ||
        cudaOccupancyMaxActiveBlocksPerMultiprocessor(&ctx->pk_per_sm, lz4_pack_kernel, 32 * PK_WARPS, 0) != cudaSuccess ||
        ctx->p2_per_sm < 1 || ctx->pk_per_sm < 1) {
        g_last_error = std::string("pack kernel setup failed: ") + cudaGetErrorString(cudaGetLastError());
        delete ctx; return nullptr;
    }
    if (const char *e = getenv("ZPB_PACK_SCRATCH_MB")) ctx->pack_scratch_blocks = std::max<u64>((u64)atoll(e) * 16, 1);
    if (cudaFuncSetAttribute(lz4hc_match_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)HC_SMEM) != cudaSuccess) {
        g_last_error = std::string("LZ4 HC kernel setup failed: ") + cudaGetErrorString(cudaGetLastError());
        delete ctx; return nullptr;
    }
    if (const char *e = getenv("ZPB_LZ4HC")) ctx->lz4hc = atoi(e) != 0;
    return ctx;
}

extern "C" void zpb_destroy(zpb_ctx *ctx) {
    if (!ctx) return;
    for (zpb_ctx *w : ctx->workers) zpb_destroy(w);
    ctx->workers.clear();
    cudaSetDevice(ctx->device);
    ctx->d_desc.release(); ctx->d_order.release(); ctx->d_res.release(); ctx->d_counter.release();
    ctx->d_in.release(); ctx->d_out.release(); ctx->h_stage.release();
    ctx->d_aux.release(); ctx->d_fe.release(); ctx->d_fb.release(); ctx->d_plist.release();
    ctx->d_glist.release(); ctx->d_fdesc.release(); ctx->d_zlist.release(); ctx->d_zlit.release();
    ctx->d_gather.release(); ctx->d_goff.release(); ctx->h_bounce.release();
    ctx->d_pblk.release(); ctx->d_pscratch.release(); ctx->d_csize.release(); ctx->d_hcrec.release();
    ctx->d_zslot.release(); ctx->d_zseq.release(); ctx->d_zmeta.release(); ctx->d_zelit.release(); ctx->d_zhuf.release(); ctx->d_ztabs.release();
    for (cudaEvent_t e : ctx->pack_evs) cudaEventDestroy(e);
    ctx->d_partials.release(); ctx->d_acc.release();
    ctx->d_arc_e.release(); ctx->d_arc_rec.release(); ctx->d_arc_chunk.release(); ctx->d_arc_work.release(); ctx->d_arc_scan.release(); ctx->d_arc_tot.release(); ctx->d_arc_names.release();
    ctx->d_cdr_jump.release(); ctx->d_cdr_cnt.release(); ctx->d_cdr_j2.release(); ctx->d_cdr_anchor.release();
    for (auto &ev : ctx->evs) if (ev) cudaEventDestroy(ev);
    if (ctx->ev0) cudaEventDestroy(ctx->ev0);
    if (ctx->ev1) cudaEventDestroy(ctx->ev1);
    if (ctx->ev_scan) cudaEventDestroy(ctx->ev_scan);
    if (ctx->ev_x0) cudaEventDestroy(ctx->ev_x0);
    if (ctx->ev_x1) cudaEventDestroy(ctx->ev_x1);
    if (ctx->ev_p0) cudaEventDestroy(ctx->ev_p0);
    if (ctx->ev_p1) cudaEventDestroy(ctx->ev_p1);
    if (ctx->ev_xb) cudaEventDestroy(ctx->ev_xb);
    if (ctx->stream_p) cudaStreamDestroy(ctx->stream_p);
    if (ctx->stream_b) cudaStreamDestroy(ctx->stream_b);
    ctx->d_order2.release(); ctx->d_defer.release();
    if (ctx->stream) cudaStreamDestroy(ctx->stream);
    delete ctx;
}

extern "C" int zpb_device_info(const zpb_ctx *ctx, int *sm_count, int *cc_major, int *cc_minor) {
    if (!ctx) return ZPB_E_ARG;
    if (sm_count) *sm_count = ctx->sm_count;
    if (cc_major) *cc_major = ctx->cc_major;
    if (cc_minor) *cc_minor = ctx->cc_minor;
    return ZPB_OK;
}

extern "C" uint64_t zpb_launch_count(const zpb_ctx *ctx) { return ctx ? ctx->launches : 0; }

extern "C" int zpb_set_tuning(zpb_ctx *ctx, int group_lanes, int ctas_per_sm) {
    if (!ctx) return ZPB_E_ARG;
    if (group_lanes) {
        if (group_lanes != 4 && group_lanes != 8 && group_lanes != 16 && group_lanes != 32)
            return fail(ctx, ZPB_E_ARG, "group_lanes must be 4, 8, 16 or 32");
        ctx->group = group_lanes;
    }
    if (ctas_per_sm >= 0) ctx->ctas_per_sm = ctas_per_sm;
    return ZPB_OK;
}

extern "C" int zpb_last_stage_ms(const zpb_ctx *ctx, float *ms4) {
    if (!ctx || !ms4) return ZPB_E_ARG;
    for (int k = 0; k < 4; ++k) ms4[k] = ctx->stage_ms[k];
    return ZPB_OK;
}

extern "C" int zpb_last_zstd_ms(const zpb_ctx *ctx, float *ms) {
    if (!ctx || !ms) return ZPB_E_ARG;
    *ms = ctx->zstd_ms;
    return ZPB_OK;
}

#ifdef ZPB_ZS_PROFILE
// developer build only: read and clear the per-phase cycle counters of zstd_unpack_kernel
extern "C" int zpb_debug_zstd_profile(unsigned long long *out8) {
    unsigned long long z[8] = {0, 0, 0, 0, 0, 0, 0, 0};
    if (cudaMemcpyFromSymbol(out8, g_zs_prof, sizeof z) != cudaSuccess) return ZPB_E_CUDA;
    return cudaMemcpyToSymbol(g_zs_prof, z, sizeof z) == cudaSuccess ? ZPB_OK : ZPB_E_CUDA;
}
#endif

// developer statistics of the last unpack call: the device-side counters (lz4_fast.cuh: [8..10] parse list lengths,
// [14] blocks the split walk gave back to the unsplit kernel, [1] entries handed to the general decoder)
extern "C" int zpb_debug_counters(zpb_ctx *ctx, unsigned *out16) {
    if (!ctx || !out16 || !ctx->d_counter.p) return ZPB_E_ARG;
    return cudaMemcpy(out16, ctx->d_counter.p, 64, cudaMemcpyDeviceToHost) == cudaSuccess ? ZPB_OK : ZPB_E_CUDA;
}

extern "C" int zpb_set_overlap(zpb_ctx *ctx, int enabled) {
    if (!ctx) return ZPB_E_ARG;
    ctx->overlap = enabled ? 1 : 0;
    return ZPB_OK;
}

extern "C" int zpb_set_fast_path(zpb_ctx *ctx, int enabled) {
    if (!ctx) return ZPB_E_ARG;
    ctx->fast = enabled ? 1 : 0;
    return ZPB_OK;
}

extern "C" int zpb_last_kernel_ms(const zpb_ctx *ctx, float *unpack_ms, float *pack_ms) {
    if (!ctx) return ZPB_E_ARG;
    if (unpack_ms) *unpack_ms = ctx->unpack_ms;
    if (pack_ms) *pack_ms = ctx->pack_ms;
    return ZPB_OK;
}

// ------------------------------------------------------------------------------------ unpack
template <int G>
static cudaError_t launch_unpack(zpb_ctx *ctx, cudaStream_t s, const u8 *arch, u64 asz, u8 *out,
                                 const zpb_entry *d_e, const u32 *d_order, u32 n, u32 *d_counter,
                                 int *d_status, u64 *d_digest) {
    int per_sm = ctx->ctas_per_sm;
    if (per_sm <= 0) {
        cudaError_t e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, unpack_kernel<G>, 256, 0);
        if (e != cudaSuccess) return e;
        if (per_sm < 1) per_sm = 1;
    }
    u64 groups_per_cta = 256 / G;
    u64 want = (n + groups_per_cta - 1) / groups_per_cta;
    u32 grid = (u32)std::min<u64>((u64)ctx->sm_count * per_sm, std::max<u64>(want, 1));
    unpack_kernel<G><<<grid, 256, 0, s>>>(arch, asz, out, d_e, d_order, n, nullptr, d_counter, d_status,
                                          d_digest, nullptr, (u32 *)ctx->d_zlist.p, d_counter + 5);
    return cudaGetLastError();
}

// the general kernel over a device-side list (entries the fast path declined); full persistent grid
template <int G>
static cudaError_t launch_general_list(zpb_ctx *ctx, cudaStream_t s, const u8 *arch, u64 asz, u8 *out,
                                       const zpb_entry *d_e, const u32 *d_list, const u32 *d_count,
                                       u32 *d_counter, int *d_status, u64 *d_digest) {
    int per_sm = 0;
    cudaError_t e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, unpack_kernel<G>, 256, 0);
    if (e != cudaSuccess) return e;
    if (per_sm < 1) per_sm = 1;
    unpack_kernel<G><<<ctx->sm_count * per_sm, 256, 0, s>>>(arch, asz, out, d_e, d_list, 0, d_count, d_counter,
                                                            d_status, d_digest, nullptr, (u32 *)ctx->d_zlist.p,
                                                            (u32 *)ctx->d_counter.p + 5);
    return cudaGetLastError();
}

// zstd entries queued by the scan / general kernel: count at counters[5], work counter at counters[6]
static cudaError_t launch_zstd(zpb_ctx *ctx, cudaStream_t s, const u8 *arch, u8 *out, const zpb_entry *d_e,
                               int *d_status, u64 *d_digest) {
    u32 *cnt = (u32 *)ctx->d_counter.p;
    zstd_unpack_kernel<<<ctx->zs_grid, ZS_WARPS * 32, ZS_WARPS * sizeof(ZstdShared), s>>>(
        arch, out, d_e, (const u32 *)ctx->d_zlist.p, cnt + 5, cnt + 6, (u8 *)ctx->d_zlit.p, d_status, d_digest);
    return cudaGetLastError();
}

static int unpack_device_impl(zpb_ctx *ctx, const u8 *d_archive, u64 archive_size, u8 *d_out,
                              u64 out_size, const zpb_entry *entries, u64 n, int32_t *status,
                              u64 *digest, cudaStream_t s) {
    if (n == 0) return ZPB_OK;
    if (n > 0x7fffffffull) return fail(ctx, ZPB_E_ARG, "too many entries in one batch");
    size_t desc_b = n * sizeof(zpb_entry), ord_b = n * sizeof(u32);
    size_t res_b = n * (sizeof(int) + sizeof(u64));
    if (!ctx->d_desc.ensure(desc_b) || !ctx->d_order.ensure(ord_b) || !ctx->d_res.ensure(res_b + 64) ||
        !ctx->d_counter.ensure(256) || !ctx->d_order2.ensure(ord_b) || !ctx->d_defer.ensure(ord_b) ||
        !ctx->h_stage.ensure(desc_b + 2 * ord_b + res_b + 64 + n * sizeof(FastAux)))
        return fail(ctx, ZPB_E_NOMEM, "scratch allocation failed");

    // ---- one pass over the descriptors (the GPU idles while the host prepares a batch, so this is kept to a single
    // read of the 64-byte records): bounds check, copy into pinned staging, coarse cost key for the work order
    // (expensive entries first: compressed bytes are a good proxy for sequence count; stored-ish entries and raw
    // copies are cheap per byte), and the fast path's scratch layout (block slots + descriptor slots per entry).
    u8 *hs = (u8 *)ctx->h_stage.p;
    zpb_entry *h_desc = (zpb_entry *)hs;
    u32 *h_order = (u32 *)(hs + desc_b);
    FastAux *h_aux = (FastAux *)(hs + desc_b + ord_b + res_b + 64);
    ctx->h_keys.resize(n);
    u16 *keys = ctx->h_keys.data();
    u32 head[1025];
    memset(head, 0, sizeof(head));
    bool any_zstd = false;
    const bool internal = ctx->cur_partials != nullptr;   // method codes above a byte are internal (comp_method is a u8, lib/zpack.h:79)
    u64 slots = 0, ndesc = 0;
    for (u64 i = 0; i < n; ++i) {
        zpb_entry e = entries[i];
        if (e.comp_size != 0 && (e.dst_off > out_size || e.dst_cap > out_size - e.dst_off))
            return fail(ctx, ZPB_E_ARG, "entry output slot exceeds the output buffer");
        // the kernels store 16 bytes at a time into the slot (include/zpack_b200.h: dst_off is 16-byte aligned)
        if (e.comp_size != 0 && (((uintptr_t)d_out + e.dst_off) & 15u))
            return fail(ctx, ZPB_E_ARG, "entry output slot is not 16-byte aligned");
        any_zstd |= e.method == ZPB_METHOD_ZSTD;
        u64 c = (e.method == ZPB_METHOD_NONE || e.comp_size >= e.uncomp_size) ? e.comp_size / 16 : e.comp_size;
        c >>= 9;  // 512-byte cost buckets, descending
        const u32 key = c > 1023 ? 0u : 1023u - (u32)c;
        keys[i] = (u16)key;
        ++head[key + 1];
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
        h_aux[i].desc_base = ndesc; h_aux[i].slot_base = (u32)slots; h_aux[i].nslots = ns;
        slots += ns; ndesc += nd;
        if (!internal && e.method > 0xFFu) e.method = 0xFFu;
        h_desc[i] = e;
    }
    if (slots > 0x7fffffffull) return fail(ctx, ZPB_E_ARG, "too many blocks in one batch");
    for (u32 k = 0; k < 1024; ++k) head[k + 1] += head[k];
    for (u64 i = 0; i < n; ++i) h_order[head[keys[i]]++] = (u32)i;   // counting sort: O(n), stable
    // The execute kernel starts while the heaviest blocks are still being parsed, so ITS order leads with the
    // entries that are parsed (almost) at once — stored and highly compressible ones, the cheap end of the list —
    // and continues with the rest, expensive first as before.
    u32 *h_order2 = (u32 *)(hs + desc_b + ord_b + res_b + 64 + n * sizeof(FastAux));
    {
        u64 ncheap = 0;
        static const u32 front_buckets = [] { const char *e = getenv("ZPB_FRONT_BUCKETS"); int v = e ? atoi(e) : 0; return (u32)(v > 0 && v < 1024 ? v : 32); }();
        while (ncheap < n && keys[h_order[n - 1 - ncheap]] >= 1024u - front_buckets) ++ncheap;   // cost below front_buckets x 512 B (default 16 KB)
        for (u64 k = 0; k < ncheap; ++k) h_order2[k] = h_order[n - 1 - k];
        for (u64 k = ncheap; k < n; ++k) h_order2[k] = h_order[k - ncheap];
    }

    if (any_zstd && (!ctx->d_zlist.ensure(n * 4) ||
                     !ctx->d_zlit.ensure((size_t)ctx->zs_grid * ZS_WARPS * ZS_LIT_SCRATCH)))
        return fail(ctx, ZPB_E_NOMEM, "zstd scratch allocation failed");
    ctx->zstd_ms = 0.f;
    u64 *d_digest = (u64 *)ctx->d_res.p;
    int *d_status = (int *)((u8 *)ctx->d_res.p + n * sizeof(u64));

    CK(ctx, cudaMemcpyAsync(ctx->d_desc.p, h_desc, desc_b, cudaMemcpyHostToDevice, s));
    CK(ctx, cudaMemcpyAsync(ctx->d_order.p, h_order, ord_b, cudaMemcpyHostToDevice, s));
    CK(ctx, cudaMemsetAsync(ctx->d_counter.p, 0, 256, s));
    if (ctx->fast) {
        // ---- scan -> parse -> exec (lz4_fast.cuh), then the general kernel over whatever they declined
        size_t aux_b = n * sizeof(FastAux);
        if (!ctx->d_aux.ensure(aux_b) || !ctx->d_fe.ensure(n * sizeof(FastEntry)) ||
            !ctx->d_fb.ensure((slots + 1) * sizeof(FastBlock)) || !ctx->d_plist.ensure(3 * (slots + 1) * 4) ||
            !ctx->d_glist.ensure(n * 4) || !ctx->d_fdesc.ensure((ndesc + 4) * 4))
            return fail(ctx, ZPB_E_NOMEM, "fast-path scratch allocation failed");
        CK(ctx, cudaMemcpyAsync(ctx->d_aux.p, h_aux, aux_b, cudaMemcpyHostToDevice, s));
        u32 *cnt = (u32 *)ctx->d_counter.p;  // [0] parse items [1] general items [2..4] work counters (zeroed above)
        const zpb_entry *d_e = (const zpb_entry *)ctx->d_desc.p;
        const u32 *d_ord = (const u32 *)ctx->d_order.p;
        CK(ctx, cudaEventRecord(ctx->evs[0], s));
        lz4_fast_scan_kernel<<<(u32)((n + 255) / 256), 256, 0, s>>>(
            d_archive, archive_size, d_e, d_ord, (u32)n, (const FastAux *)ctx->d_aux.p, (FastEntry *)ctx->d_fe.p,
            (FastBlock *)ctx->d_fb.p, (u32 *)ctx->d_plist.p, (u32)(slots + 1), cnt, (u32 *)ctx->d_glist.p, (u32 *)ctx->d_zlist.p,
            d_status, d_digest);
        CK(ctx, cudaGetLastError());
        CK(ctx, cudaEventRecord(ctx->evs[1], s));
        // K2 checks K1's verdict per block (lz4_fast.cuh), so it only needs the scan to have finished.  Parse goes to a
        // high-priority stream and is queued first, so its CTAs (3 per SM) are resident before any of K2's.  K2 runs as
        // three launches sharing the work counters: two CTAs per SM at once (they fill the SMs as parse CTAs retire and
        // never wait: an entry whose blocks are not parsed yet is put aside), the third CTA per SM once the parse kernel
        // has finished, and a last pass over the entries that were put aside.
        const bool overlap = ctx->overlap != 0;
        const int k2_ctas = [] { const char *e = getenv("ZPB_EXEC_CTAS"); int v = e ? atoi(e) : 0; return v > 0 && v <= FAST_EXEC_CTAS ? v : FAST_EXEC_CTAS; }();
        const fast_exec_fn exec_kernel = lz4_fast_exec_kernel;
        const int k1_ctas = ctx->ctas_per_sm > 0 ? ctx->ctas_per_sm : 3;
        cudaStream_t sp = overlap ? ctx->stream_p : s;
        if (overlap) {
            CK(ctx, cudaMemcpyAsync(ctx->d_order2.p, h_order2, ord_b, cudaMemcpyHostToDevice, s));
            CK(ctx, cudaEventRecord(ctx->ev_scan, s));
            CK(ctx, cudaStreamWaitEvent(sp, ctx->ev_scan, 0));
        }
        CK(ctx, cudaEventRecord(ctx->ev_p0, sp));
        // The split walk (four lanes per heavy / medium block: a quarter of the serial floor, then a merge and an in-place
        // compaction; lz4_fast_parse_body<4>) pays when the batch leaves most of the GPU's lanes idle — measured on B200
        // (profiles/r2_summary.md): 8 192 mixed entries 1.83 -> 1.34 ms parse, 2 048 entries 1.76 -> 1.23 ms; from about
        // 16 384 entries on the unsplit walks fill the GPU by themselves and the merge is only extra work (text-only:
        // 2.23 -> 2.95 ms).  ZPB_PARSE_SPLIT=0 / 1 forces either.
        static const int split_env = [] { const char *e = getenv("ZPB_PARSE_SPLIT"); return e ? atoi(e) : -1; }();
        const bool split = split_env >= 0 ? split_env != 0 : slots <= 40000;
        if (split) {
            // The light list first (stored blocks, runs: parsed within microseconds), so that the execute kernel, which
            // starts with the parse kernels, finds entries it can work on while text and record blocks are being walked;
            // then the split walk; then the blocks the split walk gave back (appended to the light list).
            lz4_fast_parse_kernel<<<ctx->sm_count, K1_THREADS, K1_THREADS * K1_ROW, sp>>>(
                d_archive, archive_size, (FastBlock *)ctx->d_fb.p, (u32 *)ctx->d_plist.p, (u32)(slots + 1), cnt, cnt + 13,
                (u32 *)ctx->d_fdesc.p, 4u);
            CK(ctx, cudaGetLastError());
            // Split walks of one batch end at about the same time, so three resident parse CTAs per SM (209 KB of shared
            // memory) would keep every execute CTA out until then.  When two per SM hold all the lanes the batch needs,
            // launch two: the third slot goes to an execute CTA.
            static const int p4_env = [] { const char *e = getenv("ZPB_PARSE4_CTAS"); return e ? atoi(e) : 0; }();
            const int p4_ctas = p4_env > 0 ? p4_env : (overlap && 4ull * slots <= (u64)ctx->sm_count * 2 * K1_THREADS ? 2 : k1_ctas);
            lz4_fast_parse4_kernel<<<ctx->sm_count * p4_ctas, K1_THREADS, K1_THREADS * K1_ROW, sp>>>(
                d_archive, archive_size, (FastBlock *)ctx->d_fb.p, (u32 *)ctx->d_plist.p, (u32)(slots + 1), cnt, cnt + 2,
                (u32 *)ctx->d_fdesc.p);
            CK(ctx, cudaGetLastError());
            lz4_fast_parse_kernel<<<ctx->sm_count, K1_THREADS, K1_THREADS * K1_ROW, sp>>>(
                d_archive, archive_size, (FastBlock *)ctx->d_fb.p, (u32 *)ctx->d_plist.p, (u32)(slots + 1), cnt, cnt + 18,
                (u32 *)ctx->d_fdesc.p, 2u);
            ctx->launches += 2;
        } else {
            lz4_fast_parse_kernel<<<ctx->sm_count * k1_ctas, K1_THREADS, K1_THREADS * K1_ROW, sp>>>(
                d_archive, archive_size, (FastBlock *)ctx->d_fb.p, (u32 *)ctx->d_plist.p, (u32)(slots + 1), cnt, cnt + 13,
                (u32 *)ctx->d_fdesc.p, 1u);
        }
        CK(ctx, cudaGetLastError());
        CK(ctx, cudaEventRecord(ctx->ev_p1, sp));
        CK(ctx, cudaEventRecord(ctx->ev_x0, s));
        const u32 *d_xord = overlap ? (const u32 *)ctx->d_order2.p : d_ord;
        static const int early_env = [] { const char *e = getenv("ZPB_EARLY_CTAS"); return e ? atoi(e) : 0; }();
        const int early = overlap ? (early_env > 0 && early_env <= k2_ctas ? early_env : (k2_ctas > 1 ? k2_ctas - 1 : 1)) : k2_ctas;
        u32 *d_defer = overlap ? (u32 *)ctx->d_defer.p : nullptr;   // cnt[11]: work counter of the last pass, cnt[12]: its length
        exec_kernel<<<ctx->sm_count * early, 32 * FAST_EXEC_WARPS, FAST_EXEC_SMEM, s>>>(
            d_archive, archive_size, d_out, d_e, d_xord, (u32)n, cnt + 3, (const FastEntry *)ctx->d_fe.p,
            (const FastBlock *)ctx->d_fb.p, (const u32 *)ctx->d_fdesc.p, cnt, (u32 *)ctx->d_glist.p, d_status,
            d_digest, ctx->cur_partials, d_defer, cnt + 12, nullptr);
        CK(ctx, cudaGetLastError());
        if (overlap) {
            if (k2_ctas > early) {
                CK(ctx, cudaStreamWaitEvent(ctx->stream_b, ctx->ev_p1, 0));
                exec_kernel<<<ctx->sm_count * (k2_ctas - early), 32 * FAST_EXEC_WARPS, FAST_EXEC_SMEM, ctx->stream_b>>>(
                    d_archive, archive_size, d_out, d_e, d_xord, (u32)n, cnt + 3, (const FastEntry *)ctx->d_fe.p,
                    (const FastBlock *)ctx->d_fb.p, (const u32 *)ctx->d_fdesc.p, cnt, (u32 *)ctx->d_glist.p, d_status,
                    d_digest, ctx->cur_partials, d_defer, cnt + 12, nullptr);
                CK(ctx, cudaGetLastError());
                CK(ctx, cudaEventRecord(ctx->ev_xb, ctx->stream_b));
                CK(ctx, cudaStreamWaitEvent(s, ctx->ev_xb, 0));
                ctx->launches += 1;
            } else {
                CK(ctx, cudaStreamWaitEvent(s, ctx->ev_p1, 0));
            }
            // what the early grids put aside (entries reached before their blocks were parsed): usually nothing
            exec_kernel<<<ctx->sm_count * k2_ctas, 32 * FAST_EXEC_WARPS, FAST_EXEC_SMEM, s>>>(
                d_archive, archive_size, d_out, d_e, d_defer, 0u, cnt + 11, (const FastEntry *)ctx->d_fe.p,
                (const FastBlock *)ctx->d_fb.p, (const u32 *)ctx->d_fdesc.p, cnt, (u32 *)ctx->d_glist.p, d_status,
                d_digest, ctx->cur_partials, nullptr, nullptr, cnt + 12);
            CK(ctx, cudaGetLastError());
            ctx->launches += 1;
        }
        CK(ctx, cudaEventRecord(ctx->ev_x1, s));
        CK(ctx, cudaEventRecord(ctx->evs[2], s));
        CK(ctx, cudaEventRecord(ctx->evs[3], s));
        cudaError_t ge;
        switch (ctx->group) {
        case 4:  ge = launch_general_list<4>(ctx, s, d_archive, archive_size, d_out, d_e, (u32 *)ctx->d_glist.p, cnt + 1, cnt + 4, d_status, d_digest); break;
        case 8:  ge = launch_general_list<8>(ctx, s, d_archive, archive_size, d_out, d_e, (u32 *)ctx->d_glist.p, cnt + 1, cnt + 4, d_status, d_digest); break;
        case 16: ge = launch_general_list<16>(ctx, s, d_archive, archive_size, d_out, d_e, (u32 *)ctx->d_glist.p, cnt + 1, cnt + 4, d_status, d_digest); break;
        default: ge = launch_general_list<32>(ctx, s, d_archive, archive_size, d_out, d_e, (u32 *)ctx->d_glist.p, cnt + 1, cnt + 4, d_status, d_digest); break;
        }
        CK(ctx, ge);
        CK(ctx, cudaEventRecord(ctx->evs[4], s));
        ctx->launches += 4;
        if (any_zstd) {
            CK(ctx, launch_zstd(ctx, s, d_archive, d_out, d_e, d_status, d_digest));
            ctx->launches += 1;
        }
        CK(ctx, cudaEventRecord(ctx->evs[5], s));
        u8 *h_res = hs + desc_b + ord_b;
        CK(ctx, cudaMemcpyAsync(h_res, ctx->d_res.p, res_b, cudaMemcpyDeviceToHost, s));
        CK(ctx, cudaStreamSynchronize(s));
        CK(ctx, cudaEventElapsedTime(&ctx->unpack_ms, ctx->evs[0], ctx->evs[5]));
        for (int k = 0; k < 4; ++k) CK(ctx, cudaEventElapsedTime(&ctx->stage_ms[k], ctx->evs[k], ctx->evs[k + 1]));
        CK(ctx, cudaEventElapsedTime(&ctx->stage_ms[1], ctx->ev_p0, ctx->ev_p1));   // parse, on its own stream when overlapped
        CK(ctx, cudaEventElapsedTime(&ctx->stage_ms[2], ctx->ev_x0, ctx->ev_x1));   // execute: both grids
        CK(ctx, cudaEventElapsedTime(&ctx->zstd_ms, ctx->evs[4], ctx->evs[5]));
        if (digest) memcpy(digest, h_res, n * sizeof(u64));
        if (status) memcpy(status, h_res + n * sizeof(u64), n * sizeof(int));
        return ZPB_OK;
    }
    CK(ctx, cudaEventRecord(ctx->ev0, s));
    cudaError_t le;
    switch (ctx->group) {
    case 4:  le = launch_unpack<4>(ctx, s, d_archive, archive_size, d_out, (zpb_entry *)ctx->d_desc.p, (u32 *)ctx->d_order.p, (u32)n, (u32 *)ctx->d_counter.p, d_status, d_digest); break;
    case 16: le = launch_unpack<16>(ctx, s, d_archive, archive_size, d_out, (zpb_entry *)ctx->d_desc.p, (u32 *)ctx->d_order.p, (u32)n, (u32 *)ctx->d_counter.p, d_status, d_digest); break;
    case 32: le = launch_unpack<32>(ctx, s, d_archive, archive_size, d_out, (zpb_entry *)ctx->d_desc.p, (u32 *)ctx->d_order.p, (u32)n, (u32 *)ctx->d_counter.p, d_status, d_digest); break;
    default: le = launch_unpack<8>(ctx, s, d_archive, archive_size, d_out, (zpb_entry *)ctx->d_desc.p, (u32 *)ctx->d_order.p, (u32)n, (u32 *)ctx->d_counter.p, d_status, d_digest); break;
    }
    CK(ctx, le);
    ctx->launches += 1;
    if (any_zstd) {
        CK(ctx, cudaEventRecord(ctx->evs[4], s));
        CK(ctx, launch_zstd(ctx, s, d_archive, d_out, (const zpb_entry *)ctx->d_desc.p, d_status, d_digest));
        ctx->launches += 1;
        CK(ctx, cudaEventRecord(ctx->evs[5], s));
    }
    CK(ctx, cudaEventRecord(ctx->ev1, s));
    u8 *h_res = hs + desc_b + ord_b;
    CK(ctx, cudaMemcpyAsync(h_res, ctx->d_res.p, res_b, cudaMemcpyDeviceToHost, s));
    CK(ctx, cudaStreamSynchronize(s));
    CK(ctx, cudaEventElapsedTime(&ctx->unpack_ms, ctx->ev0, ctx->ev1));
    if (any_zstd) CK(ctx, cudaEventElapsedTime(&ctx->zstd_ms, ctx->evs[4], ctx->evs[5]));
    if (digest) memcpy(digest, h_res, n * sizeof(u64));
    if (status) memcpy(status, h_res + n * sizeof(u64), n * sizeof(int));
    return ZPB_OK;
}

extern "C" int zpb_unpack_device(zpb_ctx *ctx, const uint8_t *d_archive, uint64_t archive_size,
                                 uint8_t *d_out, uint64_t out_size, const zpb_entry *entries,
                                 uint64_t n, int32_t *status, uint64_t *digest, void *stream) {
    if (!ctx || (!entries && n) || (!d_archive && archive_size) || (!d_out && out_size))
        return fail(ctx, ZPB_E_ARG, "null argument");
    CK(ctx, cudaSetDevice(ctx->device));
    cudaStream_t s = stream ? (cudaStream_t)stream : ctx->stream;
    return unpack_device_impl(ctx, d_archive, archive_size, d_out, out_size, entries, n, status, digest, s);
}

// One chunk, one stream: H2D of the touched archive range -> kernels -> D2H of every entry's output.
static int unpack_host_chunk(zpb_ctx *ctx, const uint8_t *h_archive, uint64_t archive_size,
                             uint8_t *h_out, uint64_t out_size, const zpb_entry *entries,
                             uint64_t n, int32_t *status, uint64_t *digest) {
    if (n == 0) return ZPB_OK;
    CK(ctx, cudaSetDevice(ctx->device));
    cudaStream_t s = ctx->stream;
    // the byte range of the archive the batch touches, and of the output it owns
    u64 lo = ~0ull, hi = 0, olo = ~0ull, ohi = 0;
    for (u64 i = 0; i < n; ++i) {
        const zpb_entry &e = entries[i];
        if (e.comp_size == 0) continue;
        if (e.src_off > archive_size || e.comp_size > archive_size - e.src_off) continue;  // flagged on device
        if (e.dst_off > out_size || e.dst_cap > out_size - e.dst_off)
            return fail(ctx, ZPB_E_ARG, "entry output slot exceeds the output buffer");
        lo = std::min(lo, e.src_off); hi = std::max(hi, e.src_off + e.comp_size);
        olo = std::min(olo, e.dst_off); ohi = std::max(ohi, e.dst_off + e.dst_cap);
    }
    if (hi <= lo) { lo = hi = 0; }
    if (ohi <= olo) { olo = ohi = 0; }
    lo &= ~15ull; olo &= ~15ull;  // keep device layout congruent to the host layout mod 16
    if (!ctx->d_in.ensure(hi - lo + 64) || !ctx->d_out.ensure(ohi - olo + 64))
        return fail(ctx, ZPB_E_NOMEM, "device staging allocation failed");
    std::vector<zpb_entry> rel(entries, entries + n);
    for (auto &e : rel) {
        if (e.comp_size == 0) continue;
        if (e.src_off > archive_size || e.comp_size > archive_size - e.src_off) {
            e.src_off = ~0ull;  // stays invalid after rebasing
            continue;
        }
        e.src_off -= lo;
        e.dst_off -= olo;
    }
    if (hi > lo) CK(ctx, cudaMemcpyAsync(ctx->d_in.p, h_archive + lo, hi - lo, cudaMemcpyHostToDevice, s));
    int rc = unpack_device_impl(ctx, (const u8 *)ctx->d_in.p, hi - lo, (u8 *)ctx->d_out.p, ohi - olo,
                                rel.data(), n, status, digest, s);
    if (rc != ZPB_OK) return rc;
    // copy back maximal runs of adjacent output slots (a slot's whole dst_cap belongs to its entry)
    std::vector<u32> by_dst;
    by_dst.reserve(n);
    for (u64 i = 0; i < n; ++i)
        if (entries[i].comp_size && rel[i].src_off != ~0ull && entries[i].dst_cap >= entries[i].uncomp_size &&
            !(entries[i].flags & ZPB_F_DISCARD))
            by_dst.push_back((u32)i);
    std::sort(by_dst.begin(), by_dst.end(), [&](u32 a, u32 b) { return entries[a].dst_off < entries[b].dst_off; });
    size_t k = 0;
    while (k < by_dst.size()) {
        u64 start = entries[by_dst[k]].dst_off;
        u64 end = start + entries[by_dst[k]].uncomp_size, own = start + entries[by_dst[k]].dst_cap;
        size_t m = k + 1;
        while (m < by_dst.size() && entries[by_dst[m]].dst_off <= own) {
            end = std::max(end, entries[by_dst[m]].dst_off + entries[by_dst[m]].uncomp_size);
            own = std::max(own, entries[by_dst[m]].dst_off + entries[by_dst[m]].dst_cap);
            ++m;
        }
        if (end > start)
            CK(ctx, cudaMemcpyAsync(h_out + start, (u8 *)ctx->d_out.p + (start - olo), end - start,
                                    cudaMemcpyDeviceToHost, s));
        k = m;
    }
    CK(ctx, cudaStreamSynchronize(s));
    return ZPB_OK;
}

// Host buffers in, host buffers out.  Large batches are cut into chunks of ~host_chunk_bytes decoded bytes
// (entries sorted by archive offset, so a chunk's compressed bytes are one contiguous H2D) and dealt to
// `host_workers` threads, each driving a private sub-context: while one chunk's kernels run, the next
// chunk's archive range is on its way in and the previous chunk's output on its way out (PCIe is full
// duplex).  Small batches take the single-shot path.
extern "C" int zpb_unpack_host(zpb_ctx *ctx, const uint8_t *h_archive, uint64_t archive_size,
                               uint8_t *h_out, uint64_t out_size, const zpb_entry *entries,
                               uint64_t n, int32_t *status, uint64_t *digest) {
    if (!ctx || (!entries && n) || (!h_archive && archive_size) || (!h_out && out_size))
        return fail(ctx, ZPB_E_ARG, "null argument");
    if (n == 0) return ZPB_OK;
    u64 total = 0;
    for (u64 i = 0; i < n; ++i) total += entries[i].comp_size ? entries[i].uncomp_size : 0;
    const int W = ctx->host_workers;
    if (W <= 1 || total < 2 * ctx->host_chunk_bytes)
        return unpack_host_chunk(ctx, h_archive, archive_size, h_out, out_size, entries, n, status, digest);

    // ---- chunks over the entries in archive order
    std::vector<u32> by_src(n);
    std::iota(by_src.begin(), by_src.end(), 0u);
    std::sort(by_src.begin(), by_src.end(), [&](u32 a, u32 b) { return entries[a].src_off < entries[b].src_off; });
    std::vector<u64> cuts{0};
    u64 acc = 0;
    for (u64 k = 0; k < n; ++k) {
        acc += entries[by_src[k]].comp_size ? entries[by_src[k]].uncomp_size : 0;
        if (acc >= ctx->host_chunk_bytes && k + 1 < n) { cuts.push_back(k + 1); acc = 0; }
    }
    cuts.push_back(n);
    const size_t nchunks = cuts.size() - 1;
    while ((int)ctx->workers.size() < W) {
        zpb_ctx *w = zpb_create(ctx->device);
        if (!w) return fail(ctx, ZPB_E_CUDA, "pipeline sub-context creation failed");
        w->fast = ctx->fast; w->group = ctx->group; w->ctas_per_sm = ctx->ctas_per_sm; w->overlap = ctx->overlap;
        ctx->workers.push_back(w);
    }
    std::vector<int> rcs(W, ZPB_OK);
    std::vector<std::string> errs(W);
    auto body = [&](int t) {
        zpb_ctx *w = ctx->workers[t];
        w->fast = ctx->fast; w->group = ctx->group; w->ctas_per_sm = ctx->ctas_per_sm; w->overlap = ctx->overlap;
        std::vector<zpb_entry> sub;
        std::vector<int32_t> st;
        std::vector<u64> dg;
        for (size_t c = t; c < nchunks; c += W) {
            const u64 a = cuts[c], b = cuts[c + 1], m = b - a;
            sub.resize(m); st.resize(m); dg.resize(m);
            for (u64 k = 0; k < m; ++k) sub[k] = entries[by_src[a + k]];
            int rc = unpack_host_chunk(w, h_archive, archive_size, h_out, out_size, sub.data(), m, st.data(), dg.data());
            if (rc != ZPB_OK) { rcs[t] = rc; errs[t] = w->err; return; }
            for (u64 k = 0; k < m; ++k) {
                if (status) status[by_src[a + k]] = st[k];
                if (digest) digest[by_src[a + k]] = dg[k];
            }
        }
    };
    std::vector<std::thread> th;
    for (int t = 1; t < W; ++t) th.emplace_back(body, t);
    body(0);
    for (auto &x : th) x.join();
    u64 launches = 0;
    float ms = 0.f;
    for (zpb_ctx *w : ctx->workers) { launches += w->launches; w->launches = 0; ms += w->unpack_ms; }
    ctx->launches += launches;
    ctx->unpack_ms = ms;
    for (int t = 0; t < W; ++t)
        if (rcs[t] != ZPB_OK) return fail(ctx, rcs[t], errs[t].c_str());
    return ZPB_OK;
}

// ------------------------------------------------------------------------------------ block-sharded entry
#include "blocks_api.inl"

// ------------------------------------------------------------------------------------ xxh3
extern "C" int zpb_xxh3_device(zpb_ctx *ctx, const uint8_t *d_data, const uint64_t *offsets,
                               const uint64_t *lengths, uint64_t n, uint64_t *digest, void *stream) {
    if (!ctx || !offsets || !lengths || !digest) return fail(ctx, ZPB_E_ARG, "null argument");
    if (n == 0) return ZPB_OK;
    if (n > 0x7fffffffull) return fail(ctx, ZPB_E_ARG, "too many ranges");
    CK(ctx, cudaSetDevice(ctx->device));
    cudaStream_t s = stream ? (cudaStream_t)stream : ctx->stream;
    size_t b = n * sizeof(u64);
    if (!ctx->d_desc.ensure(2 * b) || !ctx->d_res.ensure(b) || !ctx->d_counter.ensure(256) ||
        !ctx->h_stage.ensure(3 * b))
        return fail(ctx, ZPB_E_NOMEM, "scratch allocation failed");
    u64 *h = (u64 *)ctx->h_stage.p;
    memcpy(h, offsets, b);
    memcpy(h + n, lengths, b);
    CK(ctx, cudaMemcpyAsync(ctx->d_desc.p, h, 2 * b, cudaMemcpyHostToDevice, s));
    CK(ctx, cudaMemsetAsync(ctx->d_counter.p, 0, 256, s));
    u32 grid = (u32)std::min<u64>((u64)ctx->sm_count * 8, (n + 7) / 8);
    xxh3_kernel<32><<<grid, 256, 0, s>>>(d_data, (u64 *)ctx->d_desc.p, (u64 *)ctx->d_desc.p + n, (u32)n,
                                         (u32 *)ctx->d_counter.p, (u64 *)ctx->d_res.p);
    CK(ctx, cudaGetLastError());
    ctx->launches += 1;
    CK(ctx, cudaMemcpyAsync(h + 2 * n, ctx->d_res.p, b, cudaMemcpyDeviceToHost, s));
    CK(ctx, cudaStreamSynchronize(s));
    memcpy(digest, h + 2 * n, b);
    return ZPB_OK;
}

extern "C" int zpb_xxh3_host(zpb_ctx *ctx, const uint8_t *h_data, uint64_t length, uint64_t *digest) {
    if (!ctx || (!h_data && length) || !digest) return fail(ctx, ZPB_E_ARG, "null argument");
    CK(ctx, cudaSetDevice(ctx->device));
    if (!ctx->d_in.ensure(length + 64)) return fail(ctx, ZPB_E_NOMEM, "device staging allocation failed");
    if (length) CK(ctx, cudaMemcpyAsync(ctx->d_in.p, h_data, length, cudaMemcpyHostToDevice, ctx->stream));
    u64 off = 0;
    return zpb_xxh3_device(ctx, (const u8 *)ctx->d_in.p, &off, &length, 1, digest, ctx->stream);
}

// ------------------------------------------------------------------------------------ pack
#include "pack_api.inl"

// ------------------------------------------------------------------------------------ several GPUs, one call
#include "group_api.inl"

// ------------------------------------------------------------------------------------ the container level on the device
#include "archive_api.inl"
