// dpomp_internal.cuh -- host-side handle layouts and the launcher interface between capi.cu and the kernel TUs.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include <atomic>
#include <string>
#include <vector>

#include "../../include/dpomp.h"
#include "dpomp_dev.cuh"
#include "dpomp_models.cuh"
#include "obs_count.cuh"

namespace dpomp {

// Rate / observation table in the arithmetic of the event loop (Real = float or double), padded to the
// instantiated (C, E).  Passed to kernels by value (constant bank).
template <typename Real, int C, int E>
struct DevModel {
    int par[E];       // parameter index or -1
    Real f1[E][C], k1[E];
    Real f2[E][C], k2[E];
    Real dn[E][C], kd[E];
    int has_den[E];
    int any_den;
    Real trans[E][C];
    int xmask_i[C];
    int ic[C];
    double obs_inv_tmp2;
    int obs_tmp2_pow2;
    double obs_tmp1, obs_tmp2;  // log(1/(sqrt(2 pi) sigma)), 2 sigma^2 (src/hmm_examples.jl:61-62)
    int t0_index;
    int n_params;
};

// Everything one launch of the simulate+weight kernel needs besides the model.
struct SimLaunch {
    int32_t* pop;            // [B][C][n_pad] current populations (read unless fresh, written)
    double* logw;            // [B][n_pad] log weights (diagnostics; written only when record_logw)
    double* wtile;           // [B][n_pad] tile-local inclusive scan of exp(logw - tile max) (deterministic tree)
    int record_logw;
    const double* theta;     // [B][n_params] device
    const double* obs_time;  // [T]
    const double* obs_ysum;  // [T]  sum_v ymask[v] * y.val[v]
    double* tile_m;          // [B][ntiles]
    double* tile_s;          // [B][ntiles]
    double* tile_f;          // [B][ntiles]  f_{b|g} = exp(m_b - m_g): tile scale inside its group of kGroupTiles tiles
    double* tile_off;        // [B][ntiles]  o_{b|g}: exclusive offset of the tile inside its group (group scale)
    double* grp_m;           // [B][ngroups] group maxima / sums / scales F_g = exp(m_g - M) / exclusive offsets O_g
    double* grp_s;
    double* grp_f;
    double* grp_off;
    unsigned int* grp_counter;  // [B][ngroups] tickets of the tiles of a group
    int ngroups;
    double* filt_m;          // [B]
    double* filt_s;          // [B]
    double* ll_acc;          // [B]
    unsigned int* tile_counter;      // [B]
    unsigned long long* grp_ev;      // [B][ngroups] Gillespie events of the call, one counter per (filter, group of tiles)
    unsigned long long* ev_count;    // [1]
    unsigned long long* ovf_count;   // [1]
    long long n;             // particles per filter
    long long n_pad;         // ntiles * tile
    int ntiles;
    int n_filters;           // filters in this launch
    int n_comp;              // real C (<= instantiated C)
    int t;                   // 0-based observation index
    int fresh;               // 1: start from the initial condition at t_prev = 0 / theta[t0_index]
    int has_lik;             // obs_id[t] > 0
    // fused step (simulate + resample in ONE launch; all tiles of a filter must be co-resident): see pf_sim.cuh
    int two_per_lane;        // plain kernel, 1024-particle tiles of a predefined model: the two-particles-per-lane loop (pf_sim.cuh)
    int defer_l2;            // plain kernel followed by the resample kernel, ngroups <= kDeferGroups: level 2 of the combine
                             // (and the log-likelihood increment) is left to the resample kernel, no second ticket level
    int do_resample;         // fused kernel only: resample after the combine
    int rs_type;
    int32_t* pop_dst;        // [B][C][n_pad] offspring populations
    int32_t* anc;            // [B][n_pad] 0-based ancestors or nullptr
    ChunkPerm perm;          // offspring placement (identity or chunk-interleaved)
    unsigned long long* work_counter;  // dynamic logical CTA index (arrival order) = atomicAdd(work_counter) - work_base
    unsigned long long work_base;
    unsigned int* filt_gen;  // [B] set to `gen` by the CTA that finished the filter's combine
    unsigned int gen;
    // persistent kernel (one cooperative launch for observations t .. t_last of the call): see pf_sim.cuh
    int t_last;                  // last 0-based observation index of the call
    int n_obs_total;             // T: resampling after observation t iff obs_haslik[t] and t + 1 < T
    const int* obs_haslik;       // [T] obs_id[t] > 0
    unsigned int* rows_done;     // [B][ntiles] offspring rows written into the tile by the resample phase (consumer resets)
    unsigned int* gen_flags;     // [B][ngroups][32] generation of the last finished combine, one 128-byte line per group
    uint64_t key;
    uint32_t filter0;        // global id of local filter 0
    const uint32_t* filter_ids;  // optional explicit global ids [n_filters] (overrides filter0 + b)
    long long max_events;
    CountObs cobs;           // count observation family (read only by the kModelCountObs instantiations, pf_sim_count_*.cu)
};

struct ResampleLaunch {
    const int32_t* pop_src;  // [B][C][n_pad]
    int32_t* pop_dst;
    const double* wtile;     // [B][n_pad] tile-local inclusive scans written by the simulate kernel
    const double* tile_m;
    const double* tile_f;
    const double* tile_off;
    const double* grp_f;
    const double* grp_off;
    int ngroups;
    const double* filt_s;
    // deferred level 2 (defer_l2): the group partials of the simulate kernel, and where the filter totals / the group scales
    // and offsets go (written by the tile-0 CTA of every filter for later consumers; every CTA combines for itself)
    int defer_l2, has_lik;
    const double* grp_m;
    const double* grp_s;
    double* grp_f_w;
    double* grp_off_w;
    double* filt_s_w;
    double* filt_m_w;
    double* ll_acc;
    int32_t* anc;            // [B][n_pad] 0-based ancestors, or nullptr
    double* cw;              // [B][n_pad] cumulative weights (multinomial only), or nullptr
    long long n, n_pad;
    int ntiles, n_filters, n_comp;
    int t, rs_type;
    ChunkPerm perm;          // offspring placement (identity or chunk-interleaved)
    uint64_t key;
    uint32_t filter0;
    const uint32_t* filter_ids;
};

struct ModelHost {
    dpomp_model_desc desc;  // pointers re-targeted to the vectors below
    std::vector<double> obs_time;
    std::vector<int32_t> obs_id;
    std::vector<int64_t> obs_val;
    std::vector<double> obs_ysum;
    // observation family (dpomp_model_set_obs_model); obs_lgy / obs_lgk are the host constants lgamma(Y+1) and, for a fixed k,
    // lgamma(Y+k) - lgamma(k), empty for the Gaussian
    int obs_family = DPOMP_OBS_GAUSSIAN;
    int obs_par_index[2] = {-1, -1};
    double obs_par_value[2] = {0.0, 0.0};
    std::vector<double> obs_lgy, obs_lgk;
};

}  // namespace dpomp

// ---- the opaque handles of include/dpomp.h (host-side state; shared by capi.cu and comm.cu) -------------------------
struct dpomp_model {
    dpomp::ModelHost h;
    mutable std::atomic<bool> frozen{false};  // set when a filter or MBP handle is created from the model
};

struct dpomp_pf {
    const dpomp_model* model = nullptr;
    int device = 0;
    cudaStream_t stream = nullptr;
    cudaEvent_t ev0 = nullptr, ev1 = nullptr;
    long long n = 0, n_pad = 0;
    int n_batch = 0, ntiles = 0, items = 4, tile = 1024;
    int rs_type = DPOMP_RS_SYSTEMATIC, sim_precision = DPOMP_SIM_F32;
    long long max_events = 1ll << 20;
    uint64_t seed = 0, call_index = 0, forced_key = 0;
    bool key_forced = false;
    long long batch_offset = 0;
    int n_comp = 0, n_params = 0, n_obs = 0;
    int32_t* pop[2] = {nullptr, nullptr};
    int cur = 0;
    double* logw = nullptr;
    double* wtile = nullptr;
    double* cw = nullptr;
    int32_t* anc = nullptr;
    bool record_anc = false, initialised = false, last_resampled = false;
    double *theta_dev = nullptr, *tile_m = nullptr, *tile_s = nullptr, *tile_f = nullptr, *tile_off = nullptr;
    double *filt_m = nullptr, *filt_s = nullptr, *ll_acc = nullptr;
    double *grp_m = nullptr, *grp_s = nullptr, *grp_f = nullptr, *grp_off = nullptr;
    unsigned int* grp_counter = nullptr;
    unsigned long long* grp_ev = nullptr;        // [n_batch][ngroups] event counters of the current call
    int ngroups = 0;
    unsigned int* tile_counter = nullptr;
    unsigned long long* counters = nullptr;  // [0] events of the last call, [1] sticky overflow count
    double *obs_time_dev = nullptr, *obs_ysum_dev = nullptr;
    double *obs_lgy_dev = nullptr, *obs_lgk_dev = nullptr;  // count observation constants [T] (count families only)
    int64_t* slots_dev = nullptr;            // 2 * n_batch
    unsigned long long* work_counter = nullptr;  // fused step kernel: arrival-order CTA tickets (monotone)
    unsigned long long work_base = 0;
    unsigned int* filt_gen = nullptr;            // [n_batch] generation of the last finished combine
    unsigned int gen = 0;
    int scatter_mode = DPOMP_SCATTER_DEFAULT;    // offspring placement: 0 reference order, 1 chunk-interleaved over the tiles
    int persist_mode = DPOMP_PERSIST_DEFAULT;   // one cooperative launch per call: 0 never, 1 for calls over several observations, 2 always
    int persist_capacity = -1;                   // co-resident CTAs of the persistent kernel (lazy; 0 = unavailable)
    unsigned int* rows_done = nullptr;           // [n_batch][ntiles]
    unsigned int* gen_flags = nullptr;           // [n_batch][ngroups][32]
    int* obs_haslik_dev = nullptr;               // [T]
    bool fused_enabled = true;
    int fused_mode = 1;                          // 1: automatic (one tile per filter), 2: whenever the tiles fit
    int sm_count = 148;
    bool defer_l2_enabled = true;                // two-kernel chain: level 2 of the combine in the resample kernel (DPOMP_DEFER_L2=0: off)
    int fused_capacity[2] = {-1, -1};            // co-resident CTAs of the fused kernel per sim precision (lazy)
    uint32_t* filter_ids_dev = nullptr;      // n_batch, valid when use_filter_ids
    bool use_filter_ids = false;
    double* h_theta = nullptr;               // pinned staging
    double* h_ll = nullptr;
    int64_t* h_slots = nullptr;
    unsigned long long* h_cnt = nullptr;     // pinned: event count of the last call
    float last_ms = 0.f;
    int last_launches = 0;
    long long last_events = 0;
    long long enqueued_steps = 0;                // particle-observation steps of the call in flight
    long long last_steps = 0;                    // particle-observation steps of the last call (event intensity = last_events / last_steps)
    int two_per_lane_mode = -1;                  // -1 automatic, 0 never, 1 always (DPOMP_TWO_PER_LANE: A/B and test knob)
    // optional per-kernel timing (bench.py roofline): events around every launch of the last call
    bool kernel_timing = false;
    std::vector<cudaEvent_t> kev;      // 2 events per launch slot
    std::vector<int> kev_kind;         // 0 = simulate+weight, 1 = resample
    float kernel_ms[2] = {0.f, 0.f};
    int kernel_launches[2] = {0, 0};
    // hidden-state history (dpomp_pf_set_history, pf_history.cu)
    int hist_flags = 0;
    int32_t* hist_states = nullptr;    // PATHS:   [T][n_batch][C][n_pad] simulated states before resampling
    int32_t* hist_anc = nullptr;       // PATHS:   [T][n_batch][n_pad] 0-based ancestors of the resampling after observation t
    double* hist_part = nullptr;       // MOMENTS: [T][n_batch][ntiles][history_partials_stride(C)] tile partials
    double* hist_mom = nullptr;        // MOMENTS: [n_batch][T][2 C + 1] output of the moments combine
    int* hist_haslik = nullptr;        // [T] obs_id[t] > 0
    int hist_upto = 0;                 // observations 1..hist_upto are recorded for the first hist_nb filters
    int hist_nb = 0;
    int hist_weights_t = 0;            // observation whose weights are still on the device (last of the last call), 0 = none
    const int32_t* anc_last = nullptr; // where the last resampling wrote its ancestors when that was not `anc` (history on)
};


int dpomp_set_error(int code, const std::string& msg);  // sets the thread-local message of dpomp_last_error()
// partial_log_likelihood! launch sequence split in two so that callers can append work on the handle's stream before the
// single synchronisation: enqueue (out_mode 0: host `out`, 1: device `out`, 2: leave the increments in pf->ll_acc) + finish
extern "C" int dpomp_run_partial_enqueue(dpomp_pf* pf, const double* theta, bool theta_on_device, int nb, int ymin, int ymax,
                                         double* out, int out_mode);
extern "C" int dpomp_run_partial_finish(dpomp_pf* pf, double* out, int nb, int out_mode);

struct dpomp_comm;
namespace dpomp {

// ---- multi-GPU helpers implemented in comm.cu (used by the MBP store in mbp.cu) ---------------------------------------
struct MigrationPlan {  // 1-based LOCAL slots; send / recv lists ordered by peer rank, then by destination index
    std::vector<int64_t> local_src, send_slots, recv_slots;
    std::vector<int> send_counts, recv_counts;
};
void migration_plan(const int64_t* nidx, int64_t n_total, int world, int rank, MigrationPlan& out);
int comm_alltoallv_bytes(dpomp_comm* c, const void* send, const size_t* send_bytes, void* recv, const size_t* recv_bytes,
                         cudaStream_t stream);
int comm_allgather_rows_device(dpomp_comm* c, const double* send, long long n_total, int width, double* out, cudaStream_t stream);
void comm_bounds(const dpomp_comm* c, long long n_total, long long* lo, long long* hi);
int comm_rank(const dpomp_comm* c);
int comm_world(const dpomp_comm* c);
struct CommScratch {
    int64_t *h_slots, *d_slots;
    unsigned char *d_send, *d_recv;
    int *h_int, *d_int;
};
int comm_scratch(dpomp_comm* c, size_t slots, size_t send_bytes, size_t recv_bytes, size_t ints, CommScratch* out);

// launchers implemented in the kernel TUs; all asynchronous on `stream`; return cudaGetLastError()
cudaError_t launch_sim_weight(const ModelHost& m, int sim_precision, int items, int fused, const SimLaunch& a, cudaStream_t stream);
// fused: 0 plain, 1 fused step, 3 persistent (cooperative)
// co-resident CTAs of the persistent kernel (0 = not instantiated for this model / precision / geometry)
int sim_persist_capacity(const ModelHost& m, int sim_precision, int items);
// co-resident CTAs of the fused step kernel for this model / geometry on the current device (0 = unavailable)
int sim_fused_capacity(const ModelHost& m, int sim_precision, int items);
// the kernel family a model runs on (dpomp_models.cuh): kModelCountObs for a count observation family, else the id of the
// predefined model its rate table equals, else kModelGeneric
int kernel_model_id(const ModelHost& m);
cudaError_t launch_resample(int items, const ResampleLaunch& a, cudaStream_t stream);
cudaError_t launch_sum_events(const unsigned long long* grp_ev_dev, long long n, unsigned long long* out_dev, cudaStream_t stream);
cudaError_t launch_gather_filters(int32_t* dst, const int32_t* src, const int64_t* dst_slots_dev,
                                  const int64_t* src_slots_dev, int n, long long filter_stride_words, cudaStream_t stream);
cudaError_t launch_pack_filters(int32_t* dst_packed, const int32_t* pop, const int64_t* slots_dev, int n,
                                long long filter_stride_words, int unpack, cudaStream_t stream);
cudaError_t launch_search_hook(int rs_type, const double* cw_dev, long long n, const double* u_dev, long long n_out,
                               int64_t* out_dev, cudaStream_t stream);
int sim_kernel_supported(int n_comp, int n_events);

// ---- hidden-state history (pf_history.cu) -----------------------------------------------------------------------------
// tile partials of one (observation, filter, tile): m, sum w, sum w^2, then per compartment sum w d_c, sum w d_c^2 and the
// shift x0_c, with w = exp(logw - m) and d_c = x_c - x0_c (x0 = particle 0 of the filter: no cancellation in the variance)
__host__ __device__ inline int history_partials_stride(int n_comp) { return 3 + 3 * n_comp; }
struct HistoryLaunch {
    const int32_t* pop;      // [B][C][n_pad] simulated states of observation t
    const double* logw;      // [B][n_pad] their log weights (-inf: padding or event cap)
    int32_t* states;         // [B][C][n_pad] slice t of the state history, or nullptr
    double* part;            // [B][ntiles][stride] slice t of the tile partials, or nullptr
    long long n, n_pad;
    int ntiles, n_filters, n_comp, has_lik;
};
cudaError_t launch_history(int items, const HistoryLaunch& a, cudaStream_t stream);
// mean, variance and ESS of observations 1..t_last of the first nb filters: out [nb][t_last][2 C + 1]
cudaError_t launch_history_moments(const double* part, int t_last, int n_batch, int nb, int ntiles, int n_comp, double* out,
                                   cudaStream_t stream);
struct PathLaunch {
    const int32_t* states;   // [T][B][C][n_pad]
    const int32_t* anc;      // [T][B][n_pad]
    const int* haslik;       // [T]
    // the filter's scan tree at observation t_last (as the resample kernel reads it)
    const double* wtile; const double* tile_f; const double* tile_off; const double* grp_f; const double* grp_off;
    const double* filt_s;
    int64_t* out;            // [nb][n_paths][t_last][C]
    long long n, n_pad;
    int ntiles, ngroups, tile, n_batch, nb, n_paths, n_comp, t_last, n_obs;
    uint64_t key;
    uint32_t filter0;
    const uint32_t* filter_ids;
};
cudaError_t launch_paths(const PathLaunch& a, cudaStream_t stream);
// count observation law of a model with its device arrays (obs_lgy / obs_lgk uploaded by the caller)
CountObs count_obs_of(const ModelHost& m, const double* lgy_dev, const double* lgk_dev);

}  // namespace dpomp
