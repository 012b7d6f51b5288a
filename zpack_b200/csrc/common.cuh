// common.cuh — lane-group primitives shared by every kernel in this library.
//
// A "group" is G consecutive lanes of a warp (G = 4..32, power of two) that cooperate on ONE
// dependency chain (one entry, or one independent block).  Control state (ip, op, lengths) is
// kept replicated in every lane of the group and derived from broadcast loads, so the group
// never needs a shuffle to agree on what to do next; lanes differ only in which bytes they move.
#pragma once
#include <cstdint>
#ifdef ZPB_SIM
#include "../../tests/sim/sim_cuda.h"   // CPU emulation of the CUDA names (test infrastructure, see tests/sim/sim_rt.h)
#else
#include <cuda_runtime.h>
#endif

typedef uint8_t u8;
typedef uint16_t u16;
typedef uint32_t u32;
typedef uint64_t u64;

#define ZPB_DEVINL __device__ __forceinline__

// Slots of a context's counter block (zpb_ctx::d_counter), zeroed before every unpack batch, xxh3 batch and pack round.
// A "work counter" is the next item a persistent kernel takes; a "length" is a list's size as the kernels appended to it.
enum CounterSlot : u32 {
    CNT_WORK = 0,              // work counter of the one-kernel launches: the general kernel, xxh3_kernel, lz4_pack_kernel
    CNT_GENERAL = 1,           // length of the list the fast path hands to the general kernel
    CNT_PARSE4_WORK = 2,       // work counter of the split parse walk (lz4_fast_parse4_kernel)
    CNT_EXEC_WORK = 3,         // work counter of the execute grids over the host's order
    CNT_GENERAL_WORK = 4,      // work counter of the general kernel over the fast path's list
    CNT_ZSTD = 5,              // length of the zstd list
    CNT_ZSTD_WORK = 6,         // work counter of zstd_unpack_kernel
    CNT_PARSE_HEAVY = 8,       // lengths of the parse lists by weight: heavy, medium (+1), light (+2)
    CNT_PARSE_MEDIUM = 9,
    CNT_PARSE_LIGHT = 10,
    CNT_DEFER_WORK = 11,       // work counter of the execute pass over the entries the early grids put aside
    CNT_DEFER = 12,            // length of that put-aside list
    CNT_PARSE_WORK = 13,       // work counter of the first unsplit parse launch
    CNT_SPLIT_GIVEN_BACK = 14, // statistics: blocks the split walk gave back to the unsplit walk
    CNT_SPLIT_RETRIES = 15,    // statistics: second attempts of the split walk
    CNT_LIGHT_FIRST = 17,      // light-list length the first parse launch walked (the last launch walks the rest)
    CNT_PARSE_LAST_WORK = 18,  // work counter of the last parse launch
    CNT_PACK_BLOCKS_WORK = 32, // work counter of lz4_pack_blocks_kernel
    CNT_HC_MATCH_WORK = 48,    // work counter of lz4hc_match_kernel
    CNT_SLOTS = 64             // size of the block in u32 words
};

template <int G>
struct Group {
    static_assert(G >= 4 && G <= 32 && (G & (G - 1)) == 0, "group size");
    u32 mask;  // participating lanes of this warp
    int l;     // lane index inside the group
    ZPB_DEVINL Group() {
        int lane = threadIdx.x & 31;
        l = lane & (G - 1);
        mask = (G == 32) ? 0xffffffffu : (((1u << G) - 1u) << (lane & ~(G - 1)));
    }
    ZPB_DEVINL void sync() const { __syncwarp(mask); }
    template <typename T>
    ZPB_DEVINL T bcast(T v, int src) const { return __shfl_sync(mask, v, src, G); }
    template <typename T>
    ZPB_DEVINL T xor_(T v, int m) const { return __shfl_xor_sync(mask, v, m, G); }
    ZPB_DEVINL u32 ballot(bool p) const { return __ballot_sync(mask, p); }
};

ZPB_DEVINL u32 ld8(const u8 *p) { return *p; }
ZPB_DEVINL u32 ld16u(const u8 *p) { return (u32)p[0] | ((u32)p[1] << 8); }
ZPB_DEVINL u32 ld32u(const u8 *p) {
    return (u32)p[0] | ((u32)p[1] << 8) | ((u32)p[2] << 16) | ((u32)p[3] << 24);
}
ZPB_DEVINL u64 ld64u(const u8 *p) { return (u64)ld32u(p) | ((u64)ld32u(p + 4) << 32); }

// streaming 16-byte accesses (data touched once: keep it out of L1)
ZPB_DEVINL uint4 ldg128_stream(const void *p) {
#ifdef ZPB_SIM
    return *reinterpret_cast<const uint4 *>(p);
#else
    uint4 r;
    asm volatile("ld.global.L1::no_allocate.v4.u32 {%0,%1,%2,%3}, [%4];"
                 : "=r"(r.x), "=r"(r.y), "=r"(r.z), "=r"(r.w) : "l"(p));
    return r;
#endif
}
ZPB_DEVINL uint4 ldg128(const void *p) { return *reinterpret_cast<const uint4 *>(p); }
ZPB_DEVINL void stg128(void *p, uint4 v) { *reinterpret_cast<uint4 *>(p) = v; }

// Cooperative forward copy of n bytes, src and dst NOT overlapping within the copy
// (or src entirely before dst by >= n).  Short runs go byte-per-lane; long runs switch to
// aligned 16-byte stores fed by 4-byte-aligned loads and a funnel shift.
template <int G>
ZPB_DEVINL void group_copy(const Group<G> &g, u8 *dst, const u8 *src, u32 n) {
    if (n >= 16u * G + 32u) {
        u32 head = (u32)(-(intptr_t)dst) & 15u;
        for (u32 i = g.l; i < head; i += G) dst[i] = src[i];
        dst += head; src += head; n -= head;
        u32 chunks = (n - 4) >> 4;  // leave >= 4 bytes for the byte loop: the funnel's 5th word stays inside src[0..n)
        const u32 *s4 = reinterpret_cast<const u32 *>((uintptr_t)src & ~(uintptr_t)3);
        u32 sh = ((u32)(uintptr_t)src & 3u) * 8u;
        if (sh == 0) {
            for (u32 c = g.l; c < chunks; c += G) {
                const u32 *s = s4 + 4 * c;
                uint4 v = make_uint4(s[0], s[1], s[2], s[3]);
                stg128(dst + 16 * c, v);
            }
        } else {
            for (u32 c = g.l; c < chunks; c += G) {
                const u32 *s = s4 + 4 * c;
                u32 w0 = s[0], w1 = s[1], w2 = s[2], w3 = s[3], w4 = s[4];
                uint4 v = make_uint4(__funnelshift_r(w0, w1, sh), __funnelshift_r(w1, w2, sh),
                                     __funnelshift_r(w2, w3, sh), __funnelshift_r(w3, w4, sh));
                stg128(dst + 16 * c, v);
            }
        }
        u32 done = chunks << 4;
        dst += done; src += done; n -= done;
    }
    for (u32 i = g.l; i < n; i += G) dst[i] = src[i];
}
