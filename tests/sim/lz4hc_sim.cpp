// lz4hc_sim.cpp — TEST INFRASTRUCTURE: runs the LZ4 HC block compressor of zpack_b200/csrc/lz4hc_blocks.cuh (the match
// kernel, then the parse kernel) on the CPU emulation (sim_rt.h), so that tests/test_lz4hc_sim.py can check its output
// with the oracle without a GPU.
// Built by tests/test_lz4hc_sim.py:  g++ -O1 -g -DZPB_SIM -shared -fPIC lz4hc_sim.cpp -o liblz4hc_sim.so
#include <cstring>
#include <vector>

#include "../../include/zpack_b200.h"
#include "../../zpack_b200/csrc/lz4hc_blocks.cuh"

// blocks: (src_off, len, chain links) triples; scratch: nblocks * 65536 bytes; csize: nblocks
extern "C" int sim_lz4hc_pack_blocks(const uint8_t *in, const uint64_t *src_off, const uint32_t *len, const uint32_t *links,
                                     uint32_t nblocks, uint8_t *scratch, uint32_t *csize, int grid, uint64_t seed) {
    std::vector<PackBlock> pb(nblocks);
    for (u32 i = 0; i < nblocks; ++i) { pb[i].src_off = src_off[i]; pb[i].len = len[i]; pb[i].pad = links[i]; }
    std::vector<u32> hrec((size_t)nblocks * HC_REC_WORDS + 1, 0xA5A5A5A5u);
    u32 counter = 0;
    const PackBlock *dpb = pb.data();
    u32 *cnt = &counter, *rec = hrec.data();
    sim::launch(sim::Dim3((unsigned)grid), sim::Dim3(HC_THREADS), HC_SMEM, [&] {
        lz4hc_match_body(in, dpb, nblocks, cnt, rec);
    }, seed);
    sim::launch(sim::Dim3((nblocks + HC_PARSE_WARPS - 1) / HC_PARSE_WARPS), sim::Dim3(32 * HC_PARSE_WARPS), 0, [&] {
        lz4hc_parse_body(in, dpb, nblocks, rec, scratch, csize, (blockIdx.x * blockDim.x + threadIdx.x) >> 5);
    }, seed + 1);
    return 0;
}
