// split_retry_sim.cpp — TEST INFRASTRUCTURE: runs split_retry_kernel (zpack_b200/csrc/split_entries.cuh) on the CPU
// emulation (sim_rt.h) so that tests/test_split_retry_sim.py can check the lists it builds for the device-side retry of
// zpb_unpack_device_async.
// Built by tests/test_split_retry_sim.py:  g++ -O1 -g -DZPB_SIM -shared -fPIC split_retry_sim.cpp -o libsplit_retry_sim.so
#include "../../include/zpack_b200.h"
#include "../../zpack_b200/csrc/split_entries.cuh"

extern "C" uint32_t sim_split_job_size(void) { return (uint32_t)sizeof(SplitJob); }

// One launch as unpack_enqueue makes it (128 threads per CTA), over jobs[0, njobs); a grid of one CTA when njobs is 0.
extern "C" void sim_split_retry(const SplitJob *jobs, uint32_t njobs, zpb_entry *entries, const int32_t *status,
                                uint32_t *lz4_list, uint32_t *zstd_list, uint32_t *counters, uint64_t seed) {
    const unsigned grid = njobs ? (njobs + 127) / 128 : 1;
    sim::launch(sim::Dim3(grid), sim::Dim3(128), 0,
                [&] { split_retry_kernel(jobs, njobs, entries, status, lz4_list, zstd_list, counters); }, seed);
}
