// dpomp_models.cuh -- the predefined density-dependent models of the reference with compile-time rate structure, shared by
// the particle-filter event loop (pf_sim.cuh) and the trajectory walks of the MBP and DA layers (mbp.cu, da.cu).
#pragma once

namespace dpomp {

// ---- predefined models with compile-time rate structure (src/hmm_examples.jl:103-208, density dependent) ----------
// rate[e] = theta[e] * x[A[e]] * (B[e] >= 0 ? x[B[e]] : 1), evaluated as (theta * x_a) * x_b like the reference; the
// compiler folds the zero coefficients away (12 FFMA + 4 FMUL of the generic table become 3 FMUL + 1 FADD for SIR).
enum : int { kModelGeneric = 0, kModelSI, kModelSIR, kModelSIS, kModelSEI, kModelSEIR, kModelSEIS, kModelLOTKA, kNumModels };
template <int MODEL> struct Builtin;
#define DPOMP_BUILTIN(ID, CC, EE, AL, BL, TL)                                                                        \
    template <> struct Builtin<ID> {                                                                                 \
        static constexpr int C = CC, E = EE;                                                                         \
        __host__ __device__ static constexpr int A(int e) { constexpr int v[EE] = AL; return v[e]; }                 \
        __host__ __device__ static constexpr int B(int e) { constexpr int v[EE] = BL; return v[e]; }                 \
        __host__ __device__ static constexpr int T(int e, int c) { constexpr int v[EE][CC] = TL; return v[e][c]; }   \
    };
#define DPOMP_L(...) {__VA_ARGS__}
DPOMP_BUILTIN(kModelSI, 2, 1, DPOMP_L(0), DPOMP_L(1), DPOMP_L({-1, 1}))
DPOMP_BUILTIN(kModelSIR, 3, 2, DPOMP_L(0, 1), DPOMP_L(1, -1), DPOMP_L({-1, 1, 0}, {0, -1, 1}))
DPOMP_BUILTIN(kModelSIS, 2, 2, DPOMP_L(0, 1), DPOMP_L(1, -1), DPOMP_L({-1, 1}, {1, -1}))
DPOMP_BUILTIN(kModelSEI, 3, 2, DPOMP_L(0, 1), DPOMP_L(2, -1), DPOMP_L({-1, 1, 0}, {0, -1, 1}))
DPOMP_BUILTIN(kModelSEIR, 4, 3, DPOMP_L(0, 1, 2), DPOMP_L(2, -1, -1), DPOMP_L({-1, 1, 0, 0}, {0, -1, 1, 0}, {0, 0, -1, 1}))
DPOMP_BUILTIN(kModelSEIS, 3, 3, DPOMP_L(0, 1, 2), DPOMP_L(2, -1, -1), DPOMP_L({-1, 1, 0}, {0, -1, 1}, {1, 0, -1}))
DPOMP_BUILTIN(kModelLOTKA, 2, 3, DPOMP_L(1, 0, 0), DPOMP_L(-1, 1, -1), DPOMP_L({0, 1}, {1, -1}, {-1, 0}))
#undef DPOMP_L
#undef DPOMP_BUILTIN
// the predefined models above: the filter, the MBP walks and the DA walks are instantiated for each of them, and
// kernel_model_id (pf_kernels.cu) recognises a model's rate table as one of them
#define DPOMP_BUILTIN_MODELS(X) X(kModelSI) X(kModelSIR) X(kModelSIS) X(kModelSEI) X(kModelSEIR) X(kModelSEIS) X(kModelLOTKA)

// the generic rate table with a count observation family (obs_count.cuh): the kernels of every model with a count family
constexpr int kModelCountObs = -1;

}  // namespace dpomp
