// pf_sim_f32.cu -- f32 event-loop instantiations of the simulate+weight kernel (DPOMP_SIM_F32, the fast default).
#include "pf_sim.cuh"
namespace dpomp {
int sim_f32(int model_id, const ModelHost& m, int items, const SimLaunch& a, cudaStream_t stream, int mode) {
    return sim_typed<float>(model_id, m, items, a, stream, mode);
}
}  // namespace dpomp

#ifdef DPOMP_PHASE_TIMERS
extern "C" int dpomp_debug_phases_sim(unsigned long long* out /* [2][4096][8] */) {
    return (int)cudaMemcpyFromSymbol(out, dpomp::g_dpomp_phase, sizeof(unsigned long long) * 2 * 4096 * 8);
}
#endif
