// pf_sim_count_f64.cu -- f64 event-loop instantiations (DPOMP_SIM_F64) for the count observation families: draw-for-draw
// parity with the oracle.  Generic rate-table shapes only.
#include "pf_sim.cuh"
namespace dpomp {
int sim_count_f64(const ModelHost& m, int items, const SimLaunch& a, cudaStream_t stream, int mode) {
    return sim_count_typed<double>(m, items, a, stream, mode);
}
}  // namespace dpomp
