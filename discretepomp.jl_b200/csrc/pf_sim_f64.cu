// pf_sim_f64.cu -- f64 event-loop instantiations (DPOMP_SIM_F64): the reference's expressions bit for bit, used for
// draw-for-draw parity against the oracle.
#include "pf_sim.cuh"
namespace dpomp {
int sim_f64(int model_id, const ModelHost& m, int items, const SimLaunch& a, cudaStream_t stream, int mode) {
    return sim_typed<double>(model_id, m, items, a, stream, mode);
}
}  // namespace dpomp
