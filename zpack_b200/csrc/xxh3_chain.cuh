// xxh3_chain.cuh — the serial half of XXH3-64 for ONE entry whose blocks were decoded in parallel.
//
// XXH3's long-input loop (externals/xxHash/xxhash.h:3682-3711) is, per 1 KiB block n,
//     acc = scramble(acc + S_n)          S_n = the 16 stripe sums of block n (xxhash.h:3502-3518)
// where S_n depends on the data only (pure adds) and scramble is the non-linear per-lane step
// (xxhash.h:3527-3534).  The block-sharded decode (lz4_fast_exec_kernel in partial mode) leaves
// S_n for every complete KiB in HBM (64 bytes each); this kernel runs the chain.  Nothing about
// it is parallel beyond the 8 independent accumulator lanes (SURVEY.md F5): one warp, lanes 0-7
// each carrying one accumulator, the other lanes only help to stage S_n.
//
// Multi-GPU (BASELINE config C5): shard k's chain starts from the 64-byte accumulator state shard
// k-1 ended with (acc_in / acc_out); the last shard also folds the tail (xxhash.h:3701-3711) from
// the decoded bytes and merges (xxhash.h:3714-3747).
#pragma once
#include "common.cuh"
#include "xxh3.cuh"

#define XC_BATCH  64u   // KiB steps per batch: 64 x 64 B = 4 KiB of shared memory
#define XC_STAGES 8u    // batches in flight (cp.async ring, 32 KiB)

// The chain of one warp (all 32 lanes), shared by xxh3_chain_kernel and xxh3_chain_batch_kernel (split_entries.cuh).
// acc[8] in xxHash order.  nscr = how many leading S_n are followed by a scramble (all of the shard's
// complete KiBs, except that the entry's very last KiB is never scrambled: it belongs to the tail).
// When `final`: tail_ptr = decoded bytes starting at entry position tail_pos (<= both the tail start
// and total - 64), total = the entry's uncomp_size; returns the digest (0 when not final).
ZPB_DEVINL u64 xxh3_chain_body(ulonglong2 (*stage)[XC_BATCH * 4], const u64 *__restrict__ partials, u64 nscr,
                               const u64 *__restrict__ acc_in, u64 *acc_out, int final, const u8 *tail_ptr, u64 tail_pos,
                               u64 total) {
    const int lane = threadIdx.x & 31;
    const int j = lane & 3;
    const int i8 = lane & 7;      // the chain runs one accumulator per lane on lanes 0-7: every instruction of a
                                  // step then serves all 8 chains (a warp instruction costs the same for 1 or 32 lanes)
    u64 a;
    if (acc_in) a = acc_in[i8];
    else {
        const u64 init[8] = {XXH_P32_3, XXH_P64_1, XXH_P64_2, XXH_P64_3, XXH_P64_4, XXH_P32_2, XXH_P64_5, XXH_P32_1};
        a = init[i8];
    }
    // One chain step is acc' = ((x ^ (x >> 47)) ^ key) * PRIME32_1 with x = acc + S_n.  Carrying x instead of
    // acc (x' = acc' + S_{n+1}) puts the next add INSIDE the multiply-add: with y = (x ^ (x >> 47)) ^ key,
    //     x' = (y_lo * P + S') + (y_hi * P << 32)
    // so the loop-carried path is shift -> xor3 -> multiply-add (wide) -> multiply-add (high word) instead of
    // add.cc -> addc -> shift -> xor3 -> mad.wide -> mad.  The stream consumed is S shifted by one with a
    // trailing zero, so after the last step x is the accumulator itself.
    // How the step is written decides what NVVM / ptxas make of it (SASS checked with cuobjdump, timed on B200).  An
    // inline `mad.wide.u32` with a 64-bit addend, or the plain 64-bit C expression (NVVM reassociates it so that S' is
    // added last) come out as IMAD.WIDE, IADD3, IADD3.X: five dependent instructions, 33 cycles per step.  Leaving only
    // the additions in C makes ptxas fold y_hi * P + S'_hi into the addend's high half — behind a register-pair copy it
    // spells `IMAD.WIDE R, RZ, x, R`, which puts two wide multiplies on the path: still 33 cycles.  With the product and
    // the high-word multiply-add both opaque (asm) and S' added in C, the step is
    //     IMAD.WIDE R, y_lo, P, S' (the pair LDS.64 delivered) -> IMAD hi -> SHF -> LOP3 -> next IMAD.WIDE.
    const u64 kk = c_xxh3_key[16 + i8];
    const u32 kl = (u32)kk, kh = (u32)(kk >> 32);
    const ulonglong2 *src = reinterpret_cast<const ulonglong2 *>(partials);   // 4 x 16 B per KiB
    if (nscr) a += partials[i8];
    auto step = [&](u64 x, u64 vnext) -> u64 {
        const u32 xl = (u32)x, xh = (u32)(x >> 32);
        const u32 yl = xl ^ (xh >> 15) ^ kl;
        u64 m;
        asm("mul.wide.u32 %0, %1, %2;" : "=l"(m) : "r"(yl), "r"(XXH_P32_1));
        m += vnext;                                                      // fused by ptxas: IMAD.WIDE R, y_lo, P, S'
        u32 ml, mh, hi;
        asm("mov.b64 {%0, %1}, %2;" : "=r"(ml), "=r"(mh) : "l"(m));
        asm("mad.lo.u32 %0, %1, %2, %3;" : "=r"(hi) : "r"(xh ^ kh), "r"(XXH_P32_1), "r"(mh));   // IMAD on the high word
        u64 r;
        asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "r"(ml), "r"(hi));
        return r;
    };
    const u64 nbatch = (nscr + XC_BATCH - 1) / XC_BATCH;
    // XC_STAGES-deep cp.async ring: a batch is 64 chain steps (~0.7 us of dependent arithmetic), an HBM round trip
    // is about as long, so several batches must be in flight for the walk never to wait on memory
    const u32 stage_s = (u32)__cvta_generic_to_shared(&stage[0][0]);
    auto issue = [&](u64 b) {
        if (b < nbatch) {
            const u64 lo = b * XC_BATCH * 4 + 4, hi = nscr * 4;   // + 4: the stream is S shifted by one KiB
            const u32 dst = stage_s + (u32)(b % XC_STAGES) * (XC_BATCH * 64u);
#pragma unroll
            for (int k = 0; k < 8; ++k) {
                const u64 i = lo + (u64)k * 32 + lane;
                const bool in = i < hi;                           // beyond the shard: zero-filled (src-size 0)
                asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"(dst + (u32)(k * 32 + lane) * 16u),
                             "l"(src + (in ? i : 0)), "r"(in ? 16u : 0u) : "memory");
            }
        }
        asm volatile("cp.async.commit_group;" ::: "memory");
    };
    for (u64 b = 0; b + 1 < XC_STAGES; ++b) issue(b);
    for (u64 b = 0; b < nbatch; ++b) {
        issue(b + XC_STAGES - 1);
        asm volatile("cp.async.wait_group %0;" ::"n"(XC_STAGES - 1) : "memory");
        __syncwarp();
        const u64 *st = reinterpret_cast<const u64 *>(stage[b % XC_STAGES]);
        if (lane < 8) {
            const u32 steps = (u32)(nscr - b * XC_BATCH < XC_BATCH ? nscr - b * XC_BATCH : XC_BATCH);
            u32 s = 0;
            for (; s + 16 <= steps; s += 16) {
                u64 v[16];
#pragma unroll
                for (int k = 0; k < 16; ++k) v[k] = st[(s + k) * 8 + i8];
#pragma unroll
                for (int k = 0; k < 16; ++k) a = step(a, v[k]);
            }
            for (; s < steps; ++s) a = step(a, st[s * 8 + i8]);
        }
        __syncwarp();
    }
    if (acc_out && lane < 8) acc_out[i8] = a;
    if (!final) return 0;

    // ---- tail (xxhash.h:3701-3711) + merge (:3714-3747): pairwise layout again (lane l works for pair l & 3)
    const u64 a0 = __shfl_sync(0xffffffffu, a, 2 * j);
    const u64 a1 = __shfl_sync(0xffffffffu, a, 2 * j + 1);
    u64 dg;
    if (total <= 240) {
        dg = xxh3_small(tail_ptr, (u32)total);   // tail_pos == 0
    } else {
        const u64 full_blocks = (total - 1) >> 10;
        const u64 tail_start = full_blocks << 10;
        const u32 tail_stripes = (u32)(((total - 1) - tail_start) >> 6);
        u64 s0 = 0, s1 = 0;
        for (u32 s = lane >> 2; s < tail_stripes; s += 8) {
            const u8 *q = tail_ptr + (tail_start - tail_pos) + 64 * s + 16 * j;
            uint4 v = make_uint4(ld32u(q), ld32u(q + 4), ld32u(q + 8), ld32u(q + 12));
            Xxh3Stream<32>::piece(s0, s1, v, c_xxh3_key[s + 2 * j], c_xxh3_key[s + 2 * j + 1]);
        }
        if (lane < 4) {
            const u8 *q = tail_ptr + (total - 64 - tail_pos) + 16 * j;
            uint4 v = make_uint4(ld32u(q), ld32u(q + 4), ld32u(q + 8), ld32u(q + 12));
            Xxh3Stream<32>::piece(s0, s1, v, c_xxh3_key_last[2 * j], c_xxh3_key_last[2 * j + 1]);
        }
#pragma unroll
        for (int m = 4; m < 32; m <<= 1) {
            s0 += __shfl_xor_sync(0xffffffffu, s0, m);
            s1 += __shfl_xor_sync(0xffffffffu, s1, m);
        }
        u64 b0 = a0 + s0, b1 = a1 + s1;
        u64 m = xxh_fold128(b0 ^ xxh_sec64(11 + 16 * j), b1 ^ xxh_sec64(19 + 16 * j));
        m += __shfl_xor_sync(0xffffffffu, m, 1);
        m += __shfl_xor_sync(0xffffffffu, m, 2);
        dg = xxh3_avalanche(total * XXH_P64_1 + m);
    }
    return dg;
}

__global__ void __launch_bounds__(32)
xxh3_chain_kernel(const u64 *__restrict__ partials, u64 nscr, const u64 *__restrict__ acc_in, u64 *acc_out,
                  int final, const u8 *tail_ptr, u64 tail_pos, u64 total, u64 *digest_out) {
    __shared__ ulonglong2 stage[XC_STAGES][XC_BATCH * 4];
    const u64 dg = xxh3_chain_body(stage, partials, nscr, acc_in, acc_out, final, tail_ptr, tail_pos, total);
    if (final && threadIdx.x == 0 && digest_out) *digest_out = dg;
}
