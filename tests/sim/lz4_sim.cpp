// lz4_sim.cpp — TEST INFRASTRUCTURE: runs the LZ4 scan / parse / execute kernels of zpack_b200/csrc/lz4_fast.cuh on the
// CPU emulation (sim_rt.h) so that tests/test_lz4_sim.py can compare their output with the oracle without a GPU.
// Built by tests/test_lz4_sim.py:  g++ -O1 -g -DZPB_SIM -shared -fPIC lz4_sim.cpp -o liblz4_sim.so
#include <algorithm>
#include <cstring>
#include <vector>

#include "../../include/zpack_b200.h"
#include "../../zpack_b200/csrc/lz4_fast.cuh"

// Mirrors the fast-path half of unpack_device_impl (zpack_b200/csrc/zpb_api.cu): the same scratch layout
// (fast_entry_layout), the scan, parse and execute launches.
// Entries the fast path hands to the general decoder come back with status -1000 (the GPU tests cover that kernel).
// grid_parse / grid_exec: CTAs of the persistent kernels (small here: the emulation runs one CTA at a time).
extern "C" int sim_lz4_unpack(const uint8_t *archive, uint64_t asz, uint8_t *out, uint64_t out_size,
                              const zpb_entry *entries, uint64_t n, int32_t *status, uint64_t *digest,
                              int grid_parse, int grid_exec, uint64_t seed, uint64_t *races, uint64_t *partials) {
    (void)out_size;
    sim::S().races = 0;
    xxh3_upload_tables();
    std::vector<FastAux> aux(n);
    u64 slots = 0, ndesc = 0;
    for (u64 i = 0; i < n; ++i) aux[i] = fast_entry_layout(entries[i], slots, ndesc);
    std::vector<FastEntry> fe(n);
    std::vector<FastBlock> fb(slots + 1);
    std::vector<u32> plist(3 * (slots + 1)), glist(n + 1), zlist(n + 1), fdesc(ndesc + 8, 0xDEADBEEFu), counters(CNT_SLOTS, 0), defer(n + 1);
    for (u64 i = 0; i < n; ++i) { status[i] = -1000; digest[i] = 0; }
    const u8 *a = archive; u8 *o = out;
    const zpb_entry *de = entries;
    FastAux *dax = aux.data(); FastEntry *dfe = fe.data(); FastBlock *dfb = fb.data();
    u32 *dpl = plist.data(), *dgl = glist.data(), *dzl = zlist.data(), *dfd = fdesc.data(), *cnt = counters.data();
    const u32 pcap = (u32)(slots + 1);
    sim::launch(sim::Dim3((unsigned)((n + 255) / 256)), sim::Dim3(256), 0, [&] {
        lz4_fast_scan_kernel(a, asz, de, nullptr, (u32)n, dax, dfe, dfb, dpl, pcap, cnt, dgl, dzl, status, digest);
    }, seed);
    sim::launch(sim::Dim3((unsigned)grid_parse), sim::Dim3(K1_THREADS), K1_THREADS * K1_ROW, [&] {
        if (!getenv("SIM_NOSPLIT")) lz4_fast_parse_body<4>(a, asz, dfb, dpl, pcap, cnt, cnt + CNT_PARSE4_WORK, dfd, 0u);
    }, seed + 1);
    sim::launch(sim::Dim3((unsigned)grid_parse), sim::Dim3(K1_THREADS), K1_THREADS * K1_ROW, [&] {
        lz4_fast_parse_body<1>(a, asz, dfb, dpl, pcap, cnt, cnt + CNT_PARSE_WORK, dfd, getenv("SIM_NOSPLIT") ? 1u : 0u);
    }, seed + 3);
    sim::launch(sim::Dim3((unsigned)grid_exec), sim::Dim3(32 * FAST_EXEC_WARPS), FAST_EXEC_SMEM, [&] {
        lz4_fast_exec_kernel(a, asz, o, de, nullptr, (u32)n, cnt + CNT_EXEC_WORK, dfe, dfb, dfd, cnt, dgl, status, digest, partials, nullptr,
                           nullptr, nullptr);
    }, seed + 2);
    if (races) *races = sim::S().races;
    if (getenv("SIM_STATS")) fprintf(stderr, "sim: split list %u + %u, light %u, split retries %u\n", counters[CNT_PARSE_HEAVY], counters[CNT_PARSE_MEDIUM],
                                 counters[CNT_PARSE_LIGHT], counters[CNT_SPLIT_GIVEN_BACK]);
    return (int)counters[CNT_GENERAL];   // entries handed to the general decoder
}

// K0 + the split parse only (statistics: which blocks the split walk gives back, and why: SIM_K1_WHY=1)
extern "C" int sim_lz4_parse_only(const uint8_t *archive, uint64_t asz, const zpb_entry *entries, uint64_t n, uint64_t seed) {
    sim::S().race_check = false;
    xxh3_upload_tables();
    std::vector<FastAux> aux(n);
    u64 slots = 0, ndesc = 0;
    for (u64 i = 0; i < n; ++i) aux[i] = fast_entry_layout(entries[i], slots, ndesc);
    std::vector<FastEntry> fe(n);
    std::vector<FastBlock> fb(slots + 1);
    std::vector<u32> plist(3 * (slots + 1)), glist(n + 1), zlist(n + 1), fdesc(ndesc + 8), counters(CNT_SLOTS, 0);
    std::vector<int> status(n); std::vector<u64> digest(n);
    const u32 pcap = (u32)(slots + 1);
    sim::launch(sim::Dim3((unsigned)((n + 255) / 256)), sim::Dim3(256), 0, [&] {
        lz4_fast_scan_kernel(archive, asz, entries, nullptr, (u32)n, aux.data(), fe.data(), fb.data(), plist.data(), pcap, counters.data(),
                             glist.data(), zlist.data(), status.data(), digest.data());
    }, seed);
    sim::launch(sim::Dim3(4), sim::Dim3(K1_THREADS), K1_THREADS * K1_ROW, [&] {
        lz4_fast_parse_body<4>(archive, asz, fb.data(), plist.data(), pcap, counters.data(), counters.data() + CNT_PARSE4_WORK, fdesc.data(), 0u);
    }, seed + 1);
    sim::S().race_check = true;
    fprintf(stderr, "sim: split list %u + %u, split retries %u\n", counters[CNT_PARSE_HEAVY], counters[CNT_PARSE_MEDIUM],
            counters[CNT_SPLIT_GIVEN_BACK]);
    return (int)counters[CNT_SPLIT_GIVEN_BACK];
}

extern "C" void sim_set_race_check(int on) { sim::S().race_check = on != 0; }
