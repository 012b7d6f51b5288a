// zstd_entropy_sim.cpp — TEST INFRASTRUCTURE: the zstd writer's block stages on the CPU emulation (sim_rt.h), with the
// context's entropy switch as a parameter, so that tests/test_zstd_entropy_sim.py can decode what they write without a GPU.
// The block compressor (pack_blocks.cuh) runs on the fiber emulation; stages A and C run the kernels' own per-window
// functions (ze_stage_parse, ze_stage_encode) window by window; stage B restates the warp's histogram and pricing
// serially around the same serial builds (ze_fit, ze_huf_build, ze_huf_settle).
// Built by tests/test_zstd_entropy_sim.py:  g++ -O1 -g -DZPB_SIM -shared -fPIC zstd_entropy_sim.cpp -o libzstd_entropy_sim.so
#include <cstring>
#include <vector>

#include "../../include/zpack_b200.h"
#include "../../zpack_b200/csrc/pack_blocks.cuh"
#include "../../zpack_b200/csrc/zstd_encode.cuh"

static void stage_tables(const u8 *in, const PackBlock *blocks, const u32 *csize, const u32 *winop, u32 b, const u32 *meta, const u8 *zlit,
                         const u64 *zseq, ZeHuf *hufs, ZeBlockTabs *tabs, int entropy) {
    const u32 *m = meta + (u64)b * ZE_META;
    u32 hist[256] = {0}, hll[36] = {0}, hof[32] = {0}, hml[53] = {0};
    u32 total = 0, nseq = 0;
    const bool lit_only = ze_lit_only(entropy, blocks[b], csize[b]);
    const u32 nwin = (blocks[b].len - 12u) / 4096u + 1u;
    auto lits = [&](u32 w) {
        const u32 o = winop[(u64)b * 17u + w];
        return lit_only ? in + blocks[b].src_off + o : zlit + (u64)b * ZE_LITSLOT + ZE_LOFF(o, w);
    };
    bool ok = blocks[b].pad && (csize[b] || lit_only);
    if (ok) {
        for (u32 w = 0; w < nwin; ++w) {
            if (m[32u + w] == ZE_FAIL) { ok = false; break; }
            const u32 n = m[16u + w];
            const u8 *p = lits(w);
            for (u32 i = 0; i < n; ++i) ++hist[p[i]];
            total += n;
            const u64 *q = zseq + ((u64)b * 16u + w) * ZE_WIN_SEQ;
            for (u32 i = 0; i < m[32u + w]; ++i) {
                ++hll[ze_ll_code((u32)(q[i] & 0xFFFF))]; ++hml[ze_ml_code((u32)((q[i] >> 16) & 0xFFFF))]; ++hof[ze_highbit((u32)(q[i] >> 32))];
            }
            nseq += m[32u + w];
        }
    }
    ZeBlockTabs &B = tabs[b];
    const bool fit = ok && nseq >= ZE_TABS_MIN;
    if (fit) {
        ze_fit(B.ll, B.desc[0], &B.desc_len[0], hll, 36, nseq, 9);
        ze_fit(B.of, B.desc[1], &B.desc_len[1], hof, 32, nseq, 8);
        ze_fit(B.ml, B.desc[2], &B.desc_len[2], hml, 53, nseq, 9);
    }
    B.valid = fit ? 1u : 0u;
    ZeHuf &H = hufs[b];
    if (ok && total >= 256u) ze_huf_build(hist, H, entropy != 0, 6u * nwin);
    else { H.desc_len = 0; H.carrier = ZE_CARRIER_FIRST; }
    if (H.desc_len && H.carrier != ZE_CARRIER_FIRST) {
        u32 bits[16] = {0};
        for (u32 w = 0; w < nwin; ++w) {
            const u8 *p = lits(w);
            for (u32 i = 0; i < m[16u + w]; ++i) bits[w] += H.len[p[i]];
        }
        ze_huf_settle(H, m + 16u, bits, nwin);
    }
}

// One round of zstd blocks: (src_off, len) per block, every block marked as a zstd file's.  Outputs per block: csize (the
// LZ4 compressor's size, 0 = stored), winop[17], zbody[16] (body sizes; ZE_FAIL anywhere: the block is written raw),
// zslot (ZE_SLOT bytes, window w's body at ZE_OFF(winop[w], w)), modes[16] (literals section kind of each window:
// 0 raw, 2 with the tree, 3 treeless), huf[2] (description bytes, carrier).
extern "C" int sim_zstd_pack_blocks(const uint8_t *in, const uint64_t *src_off, const uint32_t *len, uint32_t nblocks, int entropy,
                                    int grid, uint64_t seed, uint32_t *csize, uint32_t *winop, uint32_t *zbody, uint8_t *zslot,
                                    uint32_t *modes, uint32_t *huf) {
    std::vector<PackBlock> pb(nblocks);
    for (u32 i = 0; i < nblocks; ++i) { pb[i].src_off = src_off[i]; pb[i].len = len[i]; pb[i].pad = 1; }
    std::vector<u8> scratch((size_t)nblocks * 65536 + 64, 0);
    u32 counter = 0;
    const PackBlock *dpb = pb.data();
    u32 *cnt = &counter;
    u8 *scr = scratch.data();
    sim::launch(sim::Dim3((unsigned)grid), sim::Dim3(32 * P2_WARPS), P2_SMEM, [&] {
        lz4_pack_blocks_body(in, dpb, nblocks, cnt, scr, csize, winop);
    }, seed);

    std::vector<u32> meta((size_t)nblocks * ZE_META, 0);
    std::vector<u8> zlit((size_t)nblocks * ZE_LITSLOT + 64, 0);
    std::vector<u64> zseq((size_t)nblocks * 16 * ZE_WIN_SEQ);
    std::vector<ZeHuf> hufs(nblocks);
    std::vector<ZeBlockTabs> tabs(nblocks);
    ZeTables T;
    ze_build_tables(T);
    for (u64 t = 0; t < (u64)nblocks * 16; ++t)
        ze_stage_parse(t, scratch.data(), csize, pb.data(), winop, meta.data(), zlit.data(), zseq.data(), entropy);
    for (u32 b = 0; b < nblocks; ++b)
        stage_tables(in, pb.data(), csize, winop, b, meta.data(), zlit.data(), zseq.data(), hufs.data(), tabs.data(), entropy);
    for (u64 t = 0; t < (u64)nblocks * 16; ++t)
        ze_stage_encode(t, in, csize, pb.data(), winop, meta.data(), zlit.data(), zseq.data(), hufs.data(), tabs.data(), zslot, entropy, T);
    for (u32 b = 0; b < nblocks; ++b) {
        const u32 *m = meta.data() + (u64)b * ZE_META;
        const u32 nwin = len[b] >= 13 ? (len[b] - 12u) / 4096u + 1u : 0u;
        for (u32 w = 0; w < 16; ++w) {
            zbody[b * 16 + w] = m[w];
            modes[b * 16 + w] = w < nwin && m[32u + w] != ZE_FAIL ? ze_lit_mode(w, m + 16u, nwin, hufs[b]) : 0u;
        }
        huf[2 * b] = hufs[b].desc_len;
        huf[2 * b + 1] = hufs[b].carrier;
    }
    return 0;
}

// ze_huf_build on a histogram: the description (desc_len bytes) and the code lengths (256).  Returns desc_len.
extern "C" uint32_t sim_huf_build(const uint32_t *hist, int full, uint8_t *desc, uint8_t *lens) {
    static ZeHuf H;
    ze_huf_build(hist, H, full != 0);
    memcpy(desc, H.desc, H.desc_len);
    memcpy(lens, H.len, 256);
    return H.desc_len;
}

// ze_huf_weights_fse on an arbitrary weight array: out[0..returned) (0: no description).
extern "C" uint32_t sim_huf_weights_fse(const uint8_t *wt, int nw, uint8_t *out) { return ze_huf_weights_fse(wt, nw, out); }
