// zpb_api.cu — host side of the C-ABI in include/zpack_b200.h: context, scratch arenas,
// work ordering, launches and CUDA-event timing.  No torch, no CPU codec: every entry is
// (de)compressed and hashed on the device or the call fails.
#include <algorithm>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <chrono>
#include <memory>
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

// Scratch that only grows: ensure(n) leaves room for at least n bytes (4 KiB or more), without keeping the contents.
// Device memory, or pinned host memory when Pinned.  Freed by its owner's destructor.
template <bool Pinned>
struct Scratch {
    void *p = nullptr;
    size_t cap = 0;
    Scratch() = default;
    Scratch(const Scratch &) = delete;
    Scratch &operator=(const Scratch &) = delete;
    ~Scratch() { release(); }
    bool ensure(size_t n) {
        if (n <= cap) return true;
        release();
        size_t want = std::max(n, (size_t)4096);
        if ((Pinned ? cudaMallocHost(&p, want) : cudaMalloc(&p, want)) != cudaSuccess) { p = nullptr; return false; }
        cap = want;
        return true;
    }
    void release() {
        if (p) (Pinned ? cudaFreeHost(p) : cudaFree(p));
        p = nullptr; cap = 0;
    }
};
typedef Scratch<false> DevBuf;
typedef Scratch<true> PinBuf;

// One CUDA stream or event (created through &h), destroyed by its owner's destructor.
template <typename T, cudaError_t (*Destroy)(T)>
struct Handle {
    T h = nullptr;
    Handle() = default;
    Handle(Handle &&o) noexcept : h(o.h) { o.h = nullptr; }
    Handle(const Handle &) = delete;
    Handle &operator=(const Handle &) = delete;
    ~Handle() { if (h) Destroy(h); }
    operator T() const { return h; }
};
typedef Handle<cudaStream_t, cudaStreamDestroy> Stream;
typedef Handle<cudaEvent_t, cudaEventDestroy> Event;

// Every knob of a context.  settings_from_env() fills it when the context is created, the zpb_set_* calls change it, and
// the pipelined host calls give each worker sub-context a copy at the start of every call.
struct Settings {
    int group = 32;                    // lanes per chain in the general kernel (ZPB_GROUP)
    int ctas_per_sm = 0;               // 0 = occupancy API (ZPB_CTAS_PER_SM)
    int fast = 1;                      // scan/parse/exec pipeline for LZ4 + stored entries (ZPB_FAST=0: general kernel only)
    int overlap = 1;                   // ZPB_OVERLAP=0: parse, then execute, on one stream
    int lz4hc = 0;                     // LZ4 levels >= 3 by the HC compressor (ZPB_LZ4HC=1); off: refused with ZPB_ST_NOT_AVAILABLE
    u64 pack_scratch_blocks = 16384;   // pack: 64 KB slots per round (ZPB_PACK_SCRATCH_MB, default 1 GiB)
    int arc_dynamic = 1, arc_head_mask = 127;  // copy kernel: chunks drawn from a counter (ZPB_ARC_DYNAMIC=0: fixed deal), head bytes up to the 128-byte grid (ZPB_ARC_HEAD=15: 16-byte grid)
    int arc_ctas_per_sm = 4;           // copy kernel: CTAs per SM (ZPB_ARC_CTAS)
    int host_workers = 6;              // ZPB_HOST_WORKERS (tools/e2e_sweep.py: profiles/r1_e2e_sweep.jsonl)
    u64 host_chunk_bytes = 256u << 20; // decoded bytes per pipeline chunk (ZPB_HOST_CHUNK_MB)
    // developer knobs of the LZ4 fast path (unpack_device_impl)
    u32 front_buckets = 32;            // cost buckets the execute order starts with (ZPB_FRONT_BUCKETS)
    int parse_split = -1;              // split parse walk: -1 by batch size, 0 never, 1 always (ZPB_PARSE_SPLIT)
    int parse4_ctas = 0;               // CTAs per SM of the split walk, 0 = by batch size (ZPB_PARSE4_CTAS)
    int exec_ctas = FAST_EXEC_CTAS;    // CTAs per SM of the execute kernel (ZPB_EXEC_CTAS)
    int early_ctas = 0;                // of them launched at once, 0 = all but one (ZPB_EARLY_CTAS)
};

static Settings settings_from_env() {
    Settings st;
    if (const char *s = getenv("ZPB_GROUP")) {
        int v = atoi(s);
        if (v == 4 || v == 8 || v == 16 || v == 32) st.group = v;
    }
    if (const char *s = getenv("ZPB_CTAS_PER_SM")) st.ctas_per_sm = atoi(s);
    if (const char *s = getenv("ZPB_FAST")) st.fast = atoi(s);
    if (const char *s = getenv("ZPB_OVERLAP")) st.overlap = atoi(s);
    if (const char *s = getenv("ZPB_LZ4HC")) st.lz4hc = atoi(s) != 0;
    if (const char *s = getenv("ZPB_PACK_SCRATCH_MB")) st.pack_scratch_blocks = std::max<u64>((u64)atoll(s) * 16, 1);
    if (const char *s = getenv("ZPB_ARC_DYNAMIC")) st.arc_dynamic = atoi(s) != 0;
    if (const char *s = getenv("ZPB_ARC_HEAD")) st.arc_head_mask = atoi(s) == 127 ? 127 : 15;
    if (const char *s = getenv("ZPB_ARC_CTAS")) st.arc_ctas_per_sm = std::max(1, std::min(8, atoi(s)));
    if (const char *s = getenv("ZPB_HOST_WORKERS")) st.host_workers = std::max(1, std::min(8, atoi(s)));
    if (const char *s = getenv("ZPB_HOST_CHUNK_MB")) st.host_chunk_bytes = (u64)std::max(1, atoi(s)) << 20;
    if (const char *s = getenv("ZPB_FRONT_BUCKETS")) {
        int v = atoi(s);
        if (v > 0 && v < 1024) st.front_buckets = (u32)v;
    }
    if (const char *s = getenv("ZPB_PARSE_SPLIT")) st.parse_split = atoi(s);
    if (const char *s = getenv("ZPB_PARSE4_CTAS")) st.parse4_ctas = atoi(s);
    if (const char *s = getenv("ZPB_EXEC_CTAS")) {
        int v = atoi(s);
        if (v > 0 && v <= FAST_EXEC_CTAS) st.exec_ctas = v;
    }
    if (const char *s = getenv("ZPB_EARLY_CTAS")) st.early_ctas = atoi(s);
    return st;
}

struct zpb_ctx {
    int device = 0;
    int sm_count = 0, cc_major = 0, cc_minor = 0;
    Settings set;
    Stream stream;
    Event ev0, ev1;
    std::string err;
    uint64_t launches = 0;
    float unpack_ms = 0.f, pack_ms = 0.f;
    float stage_ms[4] = {0, 0, 0, 0};
    DevBuf d_aux, d_fe, d_fb, d_plist, d_glist, d_fdesc;
    DevBuf d_zlist, d_zlit;  // zstd work list, per-warp literal buffers
    int zs_grid = 0;         // persistent grid of zstd_unpack_kernel (CTAs)
    float zstd_ms = 0.f;
    Event evs[6];
    // the execute kernel runs on its own stream so that it overlaps the tail of the parse kernel
    Stream stream_p, stream_b;   // parse (high priority), the late third of the execute grid
    Event ev_scan, ev_x0, ev_x1, ev_p0, ev_p1, ev_xb;
    DevBuf d_order2, d_defer;
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
    int p2_per_sm = 1, pk_per_sm = 1;      // resident CTAs of the two pack kernels
    std::vector<Event> pack_evs;           // three per round: before the block compressor, between, after the framing kernel
    float pack_blocks_ms = 0.f, pack_frames_ms = 0.f;
    DevBuf d_hcrec;                        // pack, HC blocks of a round: per-position match records and parse costs
    // pipelined host path: private sub-contexts (own stream + scratch), one per worker thread
    std::vector<std::unique_ptr<zpb_ctx>> workers;
    // block-sharded path (one large block-independent LZ4 entry): per-KiB XXH3 stripe sums of the last shard
    DevBuf d_partials, d_acc;
    u64 *cur_partials = nullptr;       // non-null only while zpb_unpack_blocks_device drives the pipeline
    u64 blk_uncomp = 0;                // decoded bytes of the last shard (0 = none / declined)
    float chain_ms = 0.f;
    // device-resident container operations (archive_api.inl): entry table, record offsets, chunk table, totals, names; CDR walk tables
    DevBuf d_arc_e, d_arc_rec, d_arc_chunk, d_arc_work, d_arc_scan, d_arc_tot, d_arc_names, d_cdr_jump, d_cdr_cnt, d_cdr_j2, d_cdr_anchor;
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
    std::unique_ptr<zpb_ctx> ctx(new zpb_ctx());   // a failure below releases whatever was created before it
    ctx->device = device;
    ctx->set = settings_from_env();
    cudaDeviceProp prop;
    if (cudaGetDeviceProperties(&prop, device) != cudaSuccess) {
        g_last_error = "cudaGetDeviceProperties failed"; return nullptr;
    }
    ctx->sm_count = prop.multiProcessorCount;
    ctx->cc_major = prop.major;
    ctx->cc_minor = prop.minor;
    if (cudaStreamCreateWithFlags(&ctx->stream.h, cudaStreamNonBlocking) != cudaSuccess ||
        cudaEventCreate(&ctx->ev0.h) != cudaSuccess || cudaEventCreate(&ctx->ev1.h) != cudaSuccess ||
        xxh3_upload_tables() != cudaSuccess) {
        g_last_error = std::string("context setup failed: ") + cudaGetErrorString(cudaGetLastError());
        return nullptr;
    }
    for (Event &ev : ctx->evs)
        if (cudaEventCreate(&ev.h) != cudaSuccess) { g_last_error = "event setup failed"; return nullptr; }
    int prio_lo = 0, prio_hi = 0;
    cudaDeviceGetStreamPriorityRange(&prio_lo, &prio_hi);
    if (cudaStreamCreateWithPriority(&ctx->stream_p.h, cudaStreamNonBlocking, prio_hi) != cudaSuccess ||
        cudaStreamCreateWithPriority(&ctx->stream_b.h, cudaStreamNonBlocking, prio_lo) != cudaSuccess ||
        cudaEventCreateWithFlags(&ctx->ev_scan.h, cudaEventDisableTiming) != cudaSuccess ||
        cudaEventCreateWithFlags(&ctx->ev_xb.h, cudaEventDisableTiming) != cudaSuccess ||
        cudaEventCreate(&ctx->ev_p0.h) != cudaSuccess || cudaEventCreate(&ctx->ev_p1.h) != cudaSuccess ||
        cudaEventCreate(&ctx->ev_x0.h) != cudaSuccess || cudaEventCreate(&ctx->ev_x1.h) != cudaSuccess) {
        g_last_error = "second stream setup failed"; return nullptr;
    }
    if (cudaFuncSetAttribute(lz4_fast_parse_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                             (int)(K1_THREADS * K1_ROW)) != cudaSuccess ||
        cudaFuncSetAttribute(lz4_fast_parse4_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                             (int)(K1_THREADS * K1_ROW)) != cudaSuccess ||
        cudaFuncSetAttribute(lz4_fast_exec_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                             (int)(FAST_EXEC_SMEM)) != cudaSuccess) {
        g_last_error = std::string("kernel attribute setup failed: ") + cudaGetErrorString(cudaGetLastError());
        return nullptr;
    }
    {
        int per_sm = 0;
        const int smem = (int)(ZS_WARPS * sizeof(ZstdShared));
        if (cudaFuncSetAttribute(zstd_unpack_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, smem) != cudaSuccess ||
            cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, zstd_unpack_kernel, ZS_WARPS * 32, smem) != cudaSuccess ||
            per_sm < 1) {
            g_last_error = std::string("zstd kernel setup failed: ") + cudaGetErrorString(cudaGetLastError());
            return nullptr;
        }
        ctx->zs_grid = ctx->sm_count * per_sm;
    }
    if (cudaFuncSetAttribute(lz4_pack_blocks_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)P2_SMEM) != cudaSuccess ||
        cudaOccupancyMaxActiveBlocksPerMultiprocessor(&ctx->p2_per_sm, lz4_pack_blocks_kernel, 32 * P2_WARPS, P2_SMEM) != cudaSuccess ||
        cudaOccupancyMaxActiveBlocksPerMultiprocessor(&ctx->pk_per_sm, lz4_pack_kernel, 32 * PK_WARPS, 0) != cudaSuccess ||
        ctx->p2_per_sm < 1 || ctx->pk_per_sm < 1) {
        g_last_error = std::string("pack kernel setup failed: ") + cudaGetErrorString(cudaGetLastError());
        return nullptr;
    }
    if (cudaFuncSetAttribute(lz4hc_match_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)HC_SMEM) != cudaSuccess) {
        g_last_error = std::string("LZ4 HC kernel setup failed: ") + cudaGetErrorString(cudaGetLastError());
        return nullptr;
    }
    return ctx.release();
}

extern "C" void zpb_destroy(zpb_ctx *ctx) {
    if (!ctx) return;
    cudaSetDevice(ctx->device);
    ctx->workers.clear();
    delete ctx;   // its scratch, streams and events release themselves
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
        ctx->set.group = group_lanes;
    }
    if (ctas_per_sm >= 0) ctx->set.ctas_per_sm = ctas_per_sm;
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

// developer statistics of the last unpack call: the first 16 slots of the counter block (common.cuh), among them
// CNT_PARSE_HEAVY / _MEDIUM / _LIGHT (parse list lengths), CNT_SPLIT_GIVEN_BACK (blocks the split walk gave back to the
// unsplit kernel), CNT_SPLIT_RETRIES and CNT_GENERAL (entries handed to the general decoder)
extern "C" int zpb_debug_counters(zpb_ctx *ctx, unsigned *out16) {
    if (!ctx || !out16 || !ctx->d_counter.p) return ZPB_E_ARG;
    return cudaMemcpy(out16, ctx->d_counter.p, 16 * sizeof(u32), cudaMemcpyDeviceToHost) == cudaSuccess ? ZPB_OK : ZPB_E_CUDA;
}

extern "C" int zpb_set_overlap(zpb_ctx *ctx, int enabled) {
    if (!ctx) return ZPB_E_ARG;
    ctx->set.overlap = enabled ? 1 : 0;
    return ZPB_OK;
}

extern "C" int zpb_set_fast_path(zpb_ctx *ctx, int enabled) {
    if (!ctx) return ZPB_E_ARG;
    ctx->set.fast = enabled ? 1 : 0;
    return ZPB_OK;
}

extern "C" int zpb_last_kernel_ms(const zpb_ctx *ctx, float *unpack_ms, float *pack_ms) {
    if (!ctx) return ZPB_E_ARG;
    if (unpack_ms) *unpack_ms = ctx->unpack_ms;
    if (pack_ms) *pack_ms = ctx->pack_ms;
    return ZPB_OK;
}

// ------------------------------------------------------------------------------------ unpack
// The general kernel over d_list[0, n) (the host's order), or over a list the fast path wrote on the device, whose
// length is *n_ptr: the first grid is capped by the batch and ctas_per_sm, the second is the full persistent grid.
static cudaError_t launch_general(zpb_ctx *ctx, cudaStream_t s, const u8 *arch, u64 asz, u8 *out, const zpb_entry *d_e,
                                  const u32 *d_list, u32 n, const u32 *n_ptr, u32 *work, int *d_status, u64 *d_digest) {
    auto launch = [&](auto kernel, int G) {
        int per_sm = n_ptr ? 0 : ctx->set.ctas_per_sm;
        if (per_sm <= 0) {
            cudaError_t e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kernel, 256, 0);
            if (e != cudaSuccess) return e;
            if (per_sm < 1) per_sm = 1;
        }
        u64 grid = (u64)ctx->sm_count * per_sm;
        if (!n_ptr) grid = std::min<u64>(grid, std::max<u64>((n + 256 / G - 1) / (256 / G), 1));
        kernel<<<(u32)grid, 256, 0, s>>>(arch, asz, out, d_e, d_list, n, n_ptr, work, d_status, d_digest, nullptr,
                                         (u32 *)ctx->d_zlist.p, (u32 *)ctx->d_counter.p + CNT_ZSTD);
        return cudaGetLastError();
    };
    switch (ctx->set.group) {   // zpb_set_tuning and ZPB_GROUP admit these four
    case 4:  return launch(unpack_kernel<4>, 4);
    case 8:  return launch(unpack_kernel<8>, 8);
    case 16: return launch(unpack_kernel<16>, 16);
    default: return launch(unpack_kernel<32>, 32);
    }
}

// zstd entries queued by the scan / general kernel: count at CNT_ZSTD, work counter at CNT_ZSTD_WORK
static cudaError_t launch_zstd(zpb_ctx *ctx, cudaStream_t s, const u8 *arch, u8 *out, const zpb_entry *d_e,
                               int *d_status, u64 *d_digest) {
    u32 *cnt = (u32 *)ctx->d_counter.p;
    zstd_unpack_kernel<<<ctx->zs_grid, ZS_WARPS * 32, ZS_WARPS * sizeof(ZstdShared), s>>>(
        arch, out, d_e, (const u32 *)ctx->d_zlist.p, cnt + CNT_ZSTD, cnt + CNT_ZSTD_WORK, (u8 *)ctx->d_zlit.p, d_status, d_digest);
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
        !ctx->d_counter.ensure(CNT_SLOTS * sizeof(u32)) || !ctx->d_order2.ensure(ord_b) || !ctx->d_defer.ensure(ord_b) ||
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
        h_aux[i] = fast_entry_layout(e, slots, ndesc);
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
        const u32 front_buckets = ctx->set.front_buckets;
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
    const zpb_entry *d_e = (const zpb_entry *)ctx->d_desc.p;
    const u32 *d_ord = (const u32 *)ctx->d_order.p;
    u32 *cnt = (u32 *)ctx->d_counter.p;   // slots: CounterSlot (common.cuh)

    CK(ctx, cudaMemcpyAsync(ctx->d_desc.p, h_desc, desc_b, cudaMemcpyHostToDevice, s));
    CK(ctx, cudaMemcpyAsync(ctx->d_order.p, h_order, ord_b, cudaMemcpyHostToDevice, s));
    CK(ctx, cudaMemsetAsync(ctx->d_counter.p, 0, CNT_SLOTS * sizeof(u32), s));
    const Settings &set = ctx->set;
    if (set.fast) {
        // ---- scan -> parse -> exec (lz4_fast.cuh), then the general kernel over whatever they declined
        size_t aux_b = n * sizeof(FastAux);
        if (!ctx->d_aux.ensure(aux_b) || !ctx->d_fe.ensure(n * sizeof(FastEntry)) ||
            !ctx->d_fb.ensure((slots + 1) * sizeof(FastBlock)) || !ctx->d_plist.ensure(3 * (slots + 1) * 4) ||
            !ctx->d_glist.ensure(n * 4) || !ctx->d_fdesc.ensure((ndesc + 4) * 4))
            return fail(ctx, ZPB_E_NOMEM, "fast-path scratch allocation failed");
        CK(ctx, cudaMemcpyAsync(ctx->d_aux.p, h_aux, aux_b, cudaMemcpyHostToDevice, s));
        const FastEntry *d_fe = (const FastEntry *)ctx->d_fe.p;
        FastBlock *d_fb = (FastBlock *)ctx->d_fb.p;
        u32 *d_plist = (u32 *)ctx->d_plist.p, *d_glist = (u32 *)ctx->d_glist.p, *d_fdesc = (u32 *)ctx->d_fdesc.p;
        CK(ctx, cudaEventRecord(ctx->evs[0], s));
        lz4_fast_scan_kernel<<<(u32)((n + 255) / 256), 256, 0, s>>>(
            d_archive, archive_size, d_e, d_ord, (u32)n, (const FastAux *)ctx->d_aux.p, (FastEntry *)ctx->d_fe.p,
            d_fb, d_plist, (u32)(slots + 1), cnt, d_glist, (u32 *)ctx->d_zlist.p, d_status, d_digest);
        CK(ctx, cudaGetLastError());
        CK(ctx, cudaEventRecord(ctx->evs[1], s));
        // K2 checks K1's verdict per block (lz4_fast.cuh), so it only needs the scan to have finished.  Parse goes to a
        // high-priority stream and is queued first, so its CTAs (3 per SM) are resident before any of K2's.  K2 runs as
        // three launches sharing the work counters: two CTAs per SM at once (they fill the SMs as parse CTAs retire and
        // never wait: an entry whose blocks are not parsed yet is put aside), the third CTA per SM once the parse kernel
        // has finished, and a last pass over the entries that were put aside.
        const bool overlap = set.overlap != 0;
        const int k2_ctas = set.exec_ctas;
        const int k1_ctas = set.ctas_per_sm > 0 ? set.ctas_per_sm : 3;
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
        const bool split = set.parse_split >= 0 ? set.parse_split != 0 : slots <= 40000;
        if (split) {
            // The light list first (stored blocks, runs: parsed within microseconds), so that the execute kernel, which
            // starts with the parse kernels, finds entries it can work on while text and record blocks are being walked;
            // then the split walk; then the blocks the split walk gave back (appended to the light list).
            lz4_fast_parse_kernel<<<ctx->sm_count, K1_THREADS, K1_THREADS * K1_ROW, sp>>>(
                d_archive, archive_size, d_fb, d_plist, (u32)(slots + 1), cnt, cnt + CNT_PARSE_WORK, d_fdesc, 4u);
            CK(ctx, cudaGetLastError());
            // Split walks of one batch end at about the same time, so three resident parse CTAs per SM (209 KB of shared
            // memory) would keep every execute CTA out until then.  When two per SM hold all the lanes the batch needs,
            // launch two: the third slot goes to an execute CTA.
            const int p4_ctas = set.parse4_ctas > 0 ? set.parse4_ctas
                                                    : (overlap && 4ull * slots <= (u64)ctx->sm_count * 2 * K1_THREADS ? 2 : k1_ctas);
            lz4_fast_parse4_kernel<<<ctx->sm_count * p4_ctas, K1_THREADS, K1_THREADS * K1_ROW, sp>>>(
                d_archive, archive_size, d_fb, d_plist, (u32)(slots + 1), cnt, cnt + CNT_PARSE4_WORK, d_fdesc);
            CK(ctx, cudaGetLastError());
            lz4_fast_parse_kernel<<<ctx->sm_count, K1_THREADS, K1_THREADS * K1_ROW, sp>>>(
                d_archive, archive_size, d_fb, d_plist, (u32)(slots + 1), cnt, cnt + CNT_PARSE_LAST_WORK, d_fdesc, 2u);
            ctx->launches += 2;
        } else {
            lz4_fast_parse_kernel<<<ctx->sm_count * k1_ctas, K1_THREADS, K1_THREADS * K1_ROW, sp>>>(
                d_archive, archive_size, d_fb, d_plist, (u32)(slots + 1), cnt, cnt + CNT_PARSE_WORK, d_fdesc, 1u);
        }
        CK(ctx, cudaGetLastError());
        CK(ctx, cudaEventRecord(ctx->ev_p1, sp));
        CK(ctx, cudaEventRecord(ctx->ev_x0, s));
        // K2 with `ctas` CTAs per SM over list[0, nl), or [0, *n_ptr) when the device wrote the length
        auto exec = [&](int ctas, cudaStream_t st, const u32 *list, u32 nl, u32 *work, u32 *defer, u32 *defer_len,
                        const u32 *n_ptr) {
            lz4_fast_exec_kernel<<<ctx->sm_count * ctas, 32 * FAST_EXEC_WARPS, FAST_EXEC_SMEM, st>>>(
                d_archive, archive_size, d_out, d_e, list, nl, work, d_fe, d_fb, d_fdesc, cnt, d_glist, d_status, d_digest,
                ctx->cur_partials, defer, defer_len, n_ptr);
            return cudaGetLastError();
        };
        const u32 *d_xord = overlap ? (const u32 *)ctx->d_order2.p : d_ord;
        const int early = overlap ? (set.early_ctas > 0 && set.early_ctas <= k2_ctas ? set.early_ctas : (k2_ctas > 1 ? k2_ctas - 1 : 1))
                                  : k2_ctas;
        u32 *d_defer = overlap ? (u32 *)ctx->d_defer.p : nullptr;
        CK(ctx, exec(early, s, d_xord, (u32)n, cnt + CNT_EXEC_WORK, d_defer, cnt + CNT_DEFER, nullptr));
        if (overlap) {
            if (k2_ctas > early) {
                CK(ctx, cudaStreamWaitEvent(ctx->stream_b, ctx->ev_p1, 0));
                CK(ctx, exec(k2_ctas - early, ctx->stream_b, d_xord, (u32)n, cnt + CNT_EXEC_WORK, d_defer, cnt + CNT_DEFER, nullptr));
                CK(ctx, cudaEventRecord(ctx->ev_xb, ctx->stream_b));
                CK(ctx, cudaStreamWaitEvent(s, ctx->ev_xb, 0));
                ctx->launches += 1;
            } else {
                CK(ctx, cudaStreamWaitEvent(s, ctx->ev_p1, 0));
            }
            // what the early grids put aside (entries reached before their blocks were parsed): usually nothing
            CK(ctx, exec(k2_ctas, s, d_defer, 0u, cnt + CNT_DEFER_WORK, nullptr, nullptr, cnt + CNT_DEFER));
            ctx->launches += 1;
        }
        CK(ctx, cudaEventRecord(ctx->ev_x1, s));
        CK(ctx, cudaEventRecord(ctx->evs[2], s));
        CK(ctx, cudaEventRecord(ctx->evs[3], s));
        CK(ctx, launch_general(ctx, s, d_archive, archive_size, d_out, d_e, d_glist, 0u, cnt + CNT_GENERAL,
                               cnt + CNT_GENERAL_WORK, d_status, d_digest));
        ctx->launches += 4;
    } else {
        CK(ctx, cudaEventRecord(ctx->evs[0], s));
        CK(ctx, launch_general(ctx, s, d_archive, archive_size, d_out, d_e, d_ord, (u32)n, nullptr, cnt + CNT_WORK,
                               d_status, d_digest));
        ctx->launches += 1;
    }
    CK(ctx, cudaEventRecord(ctx->evs[4], s));
    if (any_zstd) {
        CK(ctx, launch_zstd(ctx, s, d_archive, d_out, d_e, d_status, d_digest));
        ctx->launches += 1;
    }
    CK(ctx, cudaEventRecord(ctx->evs[5], s));
    u8 *h_res = hs + desc_b + ord_b;
    CK(ctx, cudaMemcpyAsync(h_res, ctx->d_res.p, res_b, cudaMemcpyDeviceToHost, s));
    CK(ctx, cudaStreamSynchronize(s));
    CK(ctx, cudaEventElapsedTime(&ctx->unpack_ms, ctx->evs[0], ctx->evs[5]));
    if (set.fast) {
        for (int k = 0; k < 4; ++k) CK(ctx, cudaEventElapsedTime(&ctx->stage_ms[k], ctx->evs[k], ctx->evs[k + 1]));
        CK(ctx, cudaEventElapsedTime(&ctx->stage_ms[1], ctx->ev_p0, ctx->ev_p1));   // parse, on its own stream when overlapped
        CK(ctx, cudaEventElapsedTime(&ctx->stage_ms[2], ctx->ev_x0, ctx->ev_x1));   // execute: every grid
    }
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

// Runs fn(t) for t in [0, W): on W - 1 threads and the caller's, which is t = 0.  Returns when every call has returned.
template <typename Fn>
static void run_parallel(int W, const Fn &fn) {
    std::vector<std::thread> th;
    for (int t = 1; t < W; ++t) th.emplace_back([&fn, t] { fn(t); });
    fn(0);
    for (auto &x : th) x.join();
}

// The pipelined host calls: items (entries or files) in source order, so that a chunk's input is one contiguous H2D,
// cut after every ~chunk_bytes of weight(item).  Returns that order; chunk c is order[cuts[c] .. cuts[c + 1]).
template <typename Item, typename Weight>
static std::vector<u32> cut_by_source(const Item *items, u64 n, u64 chunk_bytes, Weight weight, std::vector<u64> &cuts) {
    std::vector<u32> order(n);
    std::iota(order.begin(), order.end(), 0u);
    std::sort(order.begin(), order.end(), [&](u32 a, u32 b) { return items[a].src_off < items[b].src_off; });
    cuts.assign(1, 0);
    u64 acc = 0;
    for (u64 k = 0; k < n; ++k) {
        acc += weight(items[order[k]]);
        if (acc >= chunk_bytes && k + 1 < n) { cuts.push_back(k + 1); acc = 0; }
    }
    cuts.push_back(n);
    return order;
}

// Deals chunks 0 .. nchunks-1 to W = min(host_workers, nchunks) worker sub-contexts (own streams and scratch, created on
// first use): worker t runs chunk(w, c) for c = t, t + W, ... with the caller's settings, so that one chunk's H2D, the
// previous one's kernels and the one before's D2H overlap.  A worker stops at its first failing chunk; the first failing
// worker's code and message are returned.  The workers' launches count as the caller's.
template <typename Chunk>
static int run_workers(zpb_ctx *ctx, size_t nchunks, const Chunk &chunk) {
    const int W = (int)std::min<size_t>((size_t)ctx->set.host_workers, nchunks);
    while ((int)ctx->workers.size() < W) {
        zpb_ctx *w = zpb_create(ctx->device);
        if (!w) return fail(ctx, ZPB_E_CUDA, "pipeline sub-context creation failed");
        ctx->workers.emplace_back(w);
    }
    std::vector<int> rcs(W, ZPB_OK);
    run_parallel(W, [&](int t) {
        zpb_ctx *w = ctx->workers[t].get();
        w->set = ctx->set;
        for (size_t c = t; c < nchunks && rcs[t] == ZPB_OK; c += W) rcs[t] = chunk(w, c);
    });
    for (int t = 0; t < W; ++t) { ctx->launches += ctx->workers[t]->launches; ctx->workers[t]->launches = 0; }
    for (int t = 0; t < W; ++t)
        if (rcs[t] != ZPB_OK) return fail(ctx, rcs[t], ctx->workers[t]->err.c_str());
    return ZPB_OK;
}

// Host buffers in, host buffers out.  Large batches are cut into chunks of ~host_chunk_bytes decoded bytes and
// pipelined over the worker sub-contexts (run_workers; PCIe is full duplex).  Small batches take the single-shot path.
extern "C" int zpb_unpack_host(zpb_ctx *ctx, const uint8_t *h_archive, uint64_t archive_size,
                               uint8_t *h_out, uint64_t out_size, const zpb_entry *entries,
                               uint64_t n, int32_t *status, uint64_t *digest) {
    if (!ctx || (!entries && n) || (!h_archive && archive_size) || (!h_out && out_size))
        return fail(ctx, ZPB_E_ARG, "null argument");
    if (n == 0) return ZPB_OK;
    auto decoded = [](const zpb_entry &e) -> u64 { return e.comp_size ? e.uncomp_size : 0; };
    u64 total = 0;
    for (u64 i = 0; i < n; ++i) total += decoded(entries[i]);
    if (ctx->set.host_workers <= 1 || total < 2 * ctx->set.host_chunk_bytes)
        return unpack_host_chunk(ctx, h_archive, archive_size, h_out, out_size, entries, n, status, digest);

    std::vector<u64> cuts;
    const std::vector<u32> by_src = cut_by_source(entries, n, ctx->set.host_chunk_bytes, decoded, cuts);
    const int rc = run_workers(ctx, cuts.size() - 1, [&](zpb_ctx *w, size_t c) {
        const u64 a = cuts[c], m = cuts[c + 1] - a;
        std::vector<zpb_entry> sub(m);
        std::vector<int32_t> st(m);
        std::vector<u64> dg(m);
        for (u64 k = 0; k < m; ++k) sub[k] = entries[by_src[a + k]];
        const int r = unpack_host_chunk(w, h_archive, archive_size, h_out, out_size, sub.data(), m, st.data(), dg.data());
        if (r == ZPB_OK)
            for (u64 k = 0; k < m; ++k) {
                if (status) status[by_src[a + k]] = st[k];
                if (digest) digest[by_src[a + k]] = dg[k];
            }
        return r;
    });
    ctx->unpack_ms = 0.f;
    for (const auto &w : ctx->workers) ctx->unpack_ms += w->unpack_ms;
    return rc;
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
    if (!ctx->d_desc.ensure(2 * b) || !ctx->d_res.ensure(b) || !ctx->d_counter.ensure(CNT_SLOTS * sizeof(u32)) ||
        !ctx->h_stage.ensure(3 * b))
        return fail(ctx, ZPB_E_NOMEM, "scratch allocation failed");
    u64 *h = (u64 *)ctx->h_stage.p;
    memcpy(h, offsets, b);
    memcpy(h + n, lengths, b);
    CK(ctx, cudaMemcpyAsync(ctx->d_desc.p, h, 2 * b, cudaMemcpyHostToDevice, s));
    CK(ctx, cudaMemsetAsync(ctx->d_counter.p, 0, CNT_SLOTS * sizeof(u32), s));
    u32 grid = (u32)std::min<u64>((u64)ctx->sm_count * 8, (n + 7) / 8);
    xxh3_kernel<32><<<grid, 256, 0, s>>>(d_data, (u64 *)ctx->d_desc.p, (u64 *)ctx->d_desc.p + n, (u32)n,
                                         (u32 *)ctx->d_counter.p + CNT_WORK, (u64 *)ctx->d_res.p);
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
