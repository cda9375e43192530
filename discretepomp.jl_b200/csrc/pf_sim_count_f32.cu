// pf_sim_count_f32.cu -- f32 event-loop instantiations of the simulate+weight kernel for the count observation families
// (Poisson, binomial, negative binomial: dpomp_model_set_obs_model).  Generic rate-table shapes only; a translation unit of
// its own so that it compiles in parallel with the Gaussian instantiations.
#include "pf_sim.cuh"
namespace dpomp {
int sim_count_f32(const ModelHost& m, int items, const SimLaunch& a, cudaStream_t stream, int mode) {
    return sim_count_typed<float>(m, items, a, stream, mode);
}
}  // namespace dpomp
