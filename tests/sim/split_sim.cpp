// split_sim.cpp — TEST INFRASTRUCTURE: runs split_index_kernel (zpack_b200/csrc/split_entries.cuh) on the CPU emulation
// (sim_rt.h) so that tests/test_split_sim.py can compare the pseudo-rows it writes with the host index functions.
// Built by tests/test_split_sim.py:  g++ -O1 -g -DZPB_SIM -shared -fPIC split_sim.cpp -o libsplit_sim.so
#include <cstring>
#include <vector>

#include "../../include/zpack_b200.h"
#include "../../zpack_b200/csrc/split_entries.cuh"

// One candidate `parent` with its pseudo-rows as unpack_device_impl reserves them (row 0 = the parent, rows 1..nrows
// inert), through the pre-pass.  rows_out: nrows + 1 entries afterwards, aux_out: nrows + 1.  Returns 1 when the
// pre-pass accepted the entry (the parent's method became ZPB_M_SPLIT), 0 when it declined.
extern "C" int sim_split_index(const uint8_t *archive, const zpb_entry *parent, uint64_t kib0, uint64_t desc_base,
                               uint32_t slot_base, zpb_entry *rows_out, FastAux *aux_out, uint64_t seed) {
    SplitJob j;
    j.parent = 0; j.row0 = 1;
    j.nrows = (u32)((parent->uncomp_size + 65535) >> 16);
    j.kib0 = kib0; j.desc_base = desc_base; j.slot_base = slot_base;
    std::vector<zpb_entry> rows(j.nrows + 1);
    std::vector<FastAux> aux(j.nrows + 1);
    memset(rows.data(), 0, rows.size() * sizeof(zpb_entry));
    memset(aux.data(), 0, aux.size() * sizeof(FastAux));
    rows[0] = *parent;
    zpb_entry *de = rows.data(); FastAux *da = aux.data(); const SplitJob *dj = &j;
    sim::launch(sim::Dim3(1), sim::Dim3(32), SPLIT_SMEM, [&] { split_index_kernel(archive, de, da, dj); }, seed);
    memcpy(rows_out, rows.data(), rows.size() * sizeof(zpb_entry));
    memcpy(aux_out, aux.data(), aux.size() * sizeof(FastAux));
    return rows[0].method == ZPB_M_SPLIT ? 1 : 0;
}
