/*
 * dpomp.h -- C ABI of libdpomp: the B200 (sm_100a) particle-filter hot path of DiscretePOMP.jl.
 *
 * Every entry point below replaces a plain Julia function value of the reference (there is no FFI in the
 * reference; the Julia shim in discretepomp.jl_b200/julia/ binds these with `ccall`, the Python host in
 * discretepomp.jl_b200/ binds them with ctypes).  Citations are path:line under the reference repository.
 *
 * Conventions
 *   - every function returns DPOMP_OK (0) or a negative dpomp_status; nothing throws across the ABI;
 *     dpomp_last_error() returns a thread-local message for the last failure.
 *   - the caller owns all host buffers; the library owns device memory behind opaque handles.
 *   - a handle is bound to one device and one stream and is NOT thread-safe; distinct handles are.
 *   - all index arrays crossing the ABI are 1-based int64 (Julia convention); observation indices
 *     ymin/ymax are 1-based inclusive exactly as in partial_log_likelihood! (src/hmm_particle_filter.jl:39).
 *   - every call is synchronous on return unless its name ends in _async.
 *   - there is no CPU fallback: without a CUDA device every compute entry point fails with DPOMP_ERR_CUDA.
 */
#ifndef DPOMP_H
#define DPOMP_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define DPOMP_MAX_COMPARTMENTS 8
#define DPOMP_MAX_EVENTS 8
#define DPOMP_MAX_PARAMS 16
#define DPOMP_MAX_OBS_VALS 8

typedef enum dpomp_status {
    DPOMP_OK = 0,
    DPOMP_ERR_ARG = -1,      /* bad argument (null pointer, out-of-range size, unknown enum)        */
    DPOMP_ERR_CUDA = -2,     /* CUDA runtime failure / no device (message has the CUDA error string) */
    DPOMP_ERR_MODEL = -3,    /* model descriptor not representable as a device rate table             */
    DPOMP_ERR_STATE = -4,    /* call sequence error (e.g. partial with ymin>1 on a never-run filter)  */
    DPOMP_ERR_OVERFLOW = -5, /* reserved; event-cap overflow is reported by dpomp_pf_overflow_count    */
    DPOMP_ERR_COMM = -6      /* NCCL failure or NCCL library not loadable (multi-GPU entry points only) */
} dpomp_status;

/* rs_type as in get_log_pdf_fn (src/hmm_particle_filter.jl:87-94): 1 systematic, 2 stratified, 3 multinomial */
#define DPOMP_RS_SYSTEMATIC 1
#define DPOMP_RS_STRATIFIED 2
#define DPOMP_RS_MULTINOMIAL 3

/* arithmetic of the Gillespie event loop.  Weights, cumulative weights and log-likelihoods are always f64. */
#define DPOMP_SIM_F32 0 /* rates/time in f32, lg2.approx + rcp on the XU pipe (default, fast)          */
#define DPOMP_SIM_F64 1 /* rates/time in f64 with the reference's expressions: draw-for-draw oracle parity */

/*
 * Device rate table: what the reference's closures rate_function / fn_transition / obs_model
 * (src/hmm_structs.jl:119-130; predefined models src/hmm_examples.jl:103-208) are compiled to.
 *
 *   rate[e](x, theta) = P * L1 * L2 / D
 *       P  = rate_par[e] >= 0 ? theta[rate_par[e]] : 1          (0-based parameter index)
 *       L1 = rate_k1[e] + sum_c rate_f1[e][c] * x[c]
 *       L2 = rate_k2[e] + sum_c rate_f2[e][c] * x[c]
 *       D  = rate_has_den[e] ? rate_kd[e] + sum_c rate_dn[e][c] * x[c] : 1   (D == 0  =>  rate 0)
 *   evaluated as ((P*L1)*L2)/D, the association of the reference's mass-action expressions
 *   (src/hmm_examples.jl:107-121,126-144,149-154).
 *
 *   transition: x += trans[e][:]  (row = event; Julia's m_transition is column-major E x C, the shim transposes)
 *
 *   observation model (Gaussian, partial_gaussian_obs_model src/hmm_examples.jl:59-67):
 *       log g = log(1/(sqrt(2 pi) sigma)) - (sum_v obs_ymask[v]*y.val[v] - sum_c obs_xmask[c]*x[c])^2 / (2 sigma^2)
 *   or one of the count families selected by dpomp_model_set_obs_model (below), on the same masks.
 */
typedef struct dpomp_model_desc {
    int32_t n_compartments;                                   /* C, 1..DPOMP_MAX_COMPARTMENTS */
    int32_t n_events;                                         /* E, 1..DPOMP_MAX_EVENTS       */
    int32_t n_params;                                         /* length of theta              */
    int32_t t0_index;                                         /* 1-based index into theta of the initial time, 0 = fixed 0.0 (src/hmm_structs.jl:129) */
    int32_t rate_par[DPOMP_MAX_EVENTS];
    int32_t rate_f1[DPOMP_MAX_EVENTS][DPOMP_MAX_COMPARTMENTS];
    int32_t rate_k1[DPOMP_MAX_EVENTS];
    int32_t rate_f2[DPOMP_MAX_EVENTS][DPOMP_MAX_COMPARTMENTS];
    int32_t rate_k2[DPOMP_MAX_EVENTS];
    int32_t rate_has_den[DPOMP_MAX_EVENTS];
    int32_t rate_dn[DPOMP_MAX_EVENTS][DPOMP_MAX_COMPARTMENTS];
    int32_t rate_kd[DPOMP_MAX_EVENTS];
    int32_t trans[DPOMP_MAX_EVENTS][DPOMP_MAX_COMPARTMENTS];
    int64_t initial_condition[DPOMP_MAX_COMPARTMENTS];       /* fn_initial_condition() (src/DiscretePOMP.jl:96-99) */
    double obs_sigma;
    int32_t obs_xmask[DPOMP_MAX_COMPARTMENTS];
    int32_t n_obs_vals;                                       /* V = length(y.val), 1..DPOMP_MAX_OBS_VALS */
    int32_t obs_ymask[DPOMP_MAX_OBS_VALS];
    /* observations (struct Observation, src/hmm_structs.jl:30-35), sorted by time */
    int32_t n_obs;                                            /* T */
    const double* obs_time;                                   /* [T]   */
    const int32_t* obs_id;                                    /* [T]   <1: not a likelihood/resampling step */
    const int64_t* obs_val;                                   /* [T*V] row t = y[t].val */
} dpomp_model_desc;

typedef struct dpomp_model dpomp_model;
typedef struct dpomp_pf dpomp_pf;
typedef struct dpomp_comm dpomp_comm; /* multi-GPU communicator, see below */

const char* dpomp_last_error(void);
/* library/ABI version and the geometry of the deterministic scan tree (needed by the parity oracle) */
int dpomp_version(void);
int dpomp_device_count(int* out_count);

/* replaces get_private_model (src/DiscretePOMP.jl:96-99): validates the descriptor, copies observations */
int dpomp_model_create(const dpomp_model_desc* desc, dpomp_model** out_model);
int dpomp_model_destroy(dpomp_model* model);

/*
 * Observation family of a model (the reference's arbitrary obs_model closure restricted to the laws epidemic counts are
 * modelled with).  Write Y = sum_v obs_ymask[v] * y.val[v] and X = sum_c obs_xmask[c] * x[c]; for the count families both
 * masks must have 0/1 entries.  Every log g is evaluated in f64 on the device, by both event loops.
 *
 *   DPOMP_OBS_GAUSSIAN  the desc's obs_sigma and masks (the law above the descriptor): the default of dpomp_model_create
 *   DPOMP_OBS_POISSON   Y ~ Poisson(rho X):          log g = Y log(rho X) - rho X - lgamma(Y+1)                         rho > 0
 *   DPOMP_OBS_BINOMIAL  Y ~ Binomial(X, p):          log g = lgamma(X+1) - lgamma(Y+1) - lgamma(X-Y+1)
 *                                                            + Y log p + (X-Y) log1p(-p)                            0 <= p <= 1
 *   DPOMP_OBS_NEGBIN    mean mu = rho X, size k:     log g = lgamma(Y+k) - lgamma(k) - lgamma(Y+1)
 *                                                            + k log(k/(k+mu)) + Y log(mu/(k+mu))                rho > 0, k > 0
 * Parameters: Poisson (rho, unused), binomial (p, unused), negative binomial (rho, k).  par_index[i] >= 0 takes parameter i
 * from theta[par_index[i]] (0-based) of each filter / trajectory, so pMCMC, SMC^2 and ARQ can infer it; par_index[i] = -1
 * takes the fixed par_value[i].
 * Boundary cases: 0 log 0 = 0; rho X = 0 (or mu = 0) gives log g = 0 when Y = 0 and -Inf otherwise; Y > X in the binomial
 * gives -Inf; p = 0 and p = 1 are exact (log g = 0 for Y = 0, resp. Y = X, else -Inf); Y < 0 gives -Inf.  A theta-indexed
 * value outside its range (p outside [0, 1], rho or k not positive and finite) gives -Inf for every particle: the filter
 * then returns what it returns when every weight is zero, and an MH step rejects the proposal.
 * obs_sigma keeps its validation in dpomp_model_create and is ignored by the count families.  The per-observation constants
 * lgamma(Y+1) and, for a fixed k, lgamma(Y+k) - lgamma(k) are computed on the host.
 * Returns DPOMP_ERR_ARG for an unknown family or a null pointer, DPOMP_ERR_MODEL for an index >= n_params, a fixed value out of
 * range or a mask entry other than 0 / 1, and DPOMP_ERR_STATE once a filter or MBP handle has been created from the model
 * (handles read the model when they launch, so it is frozen from then on).
 */
#define DPOMP_OBS_GAUSSIAN 0 /* the desc's sigma / masks: the default */
#define DPOMP_OBS_POISSON 1
#define DPOMP_OBS_BINOMIAL 2
#define DPOMP_OBS_NEGBIN 3
int dpomp_model_set_obs_model(dpomp_model* model, int32_t family, const int32_t* par_index /*[2], -1 = fixed*/,
                              const double* par_value /*[2]*/);

/*
 * Which kernels the model runs on (read-only, no device needed).  *out_id = 1..7 (SI, SIR, SIS, SEI, SEIR, SEIS, LOTKA) when
 * the rate table is exactly that predefined density-dependent model -- same compartments, events, parameter order, factors
 * and transition rows -- and the filter, the MBP walks and the DA walks use its compile-time instantiations; 0 for every other
 * table, which runs the generic rate-table kernels on the smallest instantiated (compartments, events) shape covering it.
 * A count observation family (dpomp_model_set_obs_model) always gives 0: those kernels evaluate the generic table.
 */
int dpomp_model_builtin_id(const dpomp_model* model, int32_t* out_id);

/*
 * A batch of n_batch independent bootstrap filters of n_particles each on one device
 * (the `pop::Array{Int64,2}` workspaces of estimate_likelihood src/hmm_particle_filter.jl:79-84 and of
 * run_pibis src/hmm_ibis.jl:26-35, resident in HBM as int32 SoA [batch][compartment][particle]).
 * seed selects the Philox4x32-10 key stream; device < 0 = current device.
 */
int dpomp_pf_create(const dpomp_model* model, int64_t n_particles, int32_t n_batch, int32_t rs_type,
                    uint64_t seed, int32_t device, dpomp_pf** out_pf);
int dpomp_pf_destroy(dpomp_pf* pf);

/* options (all optional; defaults in parentheses) */
int dpomp_pf_set_sim_precision(dpomp_pf* pf, int32_t sim_precision);  /* (DPOMP_SIM_F32) */
int dpomp_pf_set_max_events(dpomp_pf* pf, int64_t max_events);        /* per particle per interval (1<<20); the
                                                                         reference PF has no cap (src/hmm_particle_filter.jl:19-27) */
int dpomp_pf_set_batch_offset(dpomp_pf* pf, int64_t batch_offset);    /* global id of local filter 0 (0): makes the
                                                                         random streams independent of the sharding  */
int dpomp_pf_set_fused(dpomp_pf* pf, int32_t on);                     /* fused simulate+resample launch per observation: 0 never, (1) for
                                                                         filters of one tile, 2 whenever all tiles of a filter are co-resident.
                                                                         Mode 2 spin-waits inside the kernel for the other tiles of the filter and
                                                                         therefore REQUIRES AN EXCLUSIVE DEVICE: with another handle, stream or
                                                                         process (MPS) holding SM slots the wait can hang; modes 0 and 1 never wait */
/* Persistent launch: all observations of a call in ONE cooperative kernel launch; a tile starts the next observation as soon as
 * its own rows have been written by the resample phase (no kernel boundaries, no grid-wide barrier besides the weight
 * combine).  Used when every CTA of the call is co-resident (n_batch_used x tiles <= device capacity), the event loop is
 * f32, the resampler systematic or stratified and the row order the reference's; otherwise the per-observation launch chain
 * runs.  0 never, 1 for calls over more than one observation, 2 also for single-observation calls.  Results are bit-identical
 * to the launch chain. */
#ifndef DPOMP_PERSIST_DEFAULT
#define DPOMP_PERSIST_DEFAULT 0
#endif
int dpomp_pf_set_persistent(dpomp_pf* pf, int32_t mode);
/* Row order of the offspring after a resampling step.  The ancestors chosen for offspring i = 1..N are always those of the
 * reference's walk (src/hmm_pf_resample.jl:34-40); the mode only says where offspring i is stored:
 *   DPOMP_SCATTER_REFERENCE    row i, as `pop[i,:] = old_p[j,:]` (src/hmm_pf_resample.jl:38)
 *   DPOMP_SCATTER_INTERLEAVED  32-row chunk k goes to chunk sigma(k), sigma = rank of k ordered by (k mod tiles, k div tiles)
 *                              over the floor(N/32) full chunks, the trailing partial chunk stays: every tile of the next
 *                              simulation step holds a uniform sample of the lineages (load balance).  Particle order is
 *                              arbitrary in a bootstrap filter; the estimate has the same law. */
#define DPOMP_SCATTER_REFERENCE 0
#define DPOMP_SCATTER_INTERLEAVED 1
#ifndef DPOMP_SCATTER_DEFAULT
#define DPOMP_SCATTER_DEFAULT DPOMP_SCATTER_REFERENCE
#endif
int dpomp_pf_set_scatter(dpomp_pf* pf, int32_t mode);
int dpomp_pf_set_filter_ids(dpomp_pf* pf, const int64_t* ids, int32_t n); /* explicit 0-based GLOBAL ids of the first n
                                                                         filters for the random streams; NULL = batch_offset + b */
int dpomp_pf_set_stream_key(dpomp_pf* pf, uint64_t key);              /* force the Philox key of the NEXT call (tests) */
int dpomp_pf_get_stream_key(dpomp_pf* pf, uint64_t* out_key);         /* key the next fresh call will use            */
int dpomp_pf_geometry(const dpomp_pf* pf, int32_t* out_tile, int32_t* out_items_per_thread);

/*
 * estimate_likelihood (src/hmm_particle_filter.jl:79-84), batched: theta is n_params x n_batch_used
 * column-major (one theta vector per filter, contiguous), out_ll[n_batch_used].
 */
int dpomp_pf_loglik(dpomp_pf* pf, const double* theta, int32_t n_batch_used, double* out_ll);

/*
 * partial_log_likelihood! (src/hmm_particle_filter.jl:39-76), batched over filters with device-resident
 * populations: runs observations ymin..ymax (1-based, inclusive).  ymin == 1 re-initialises the populations
 * from the initial condition (t_prev = 0 or theta[t0_index]); otherwise continues from the stored state.
 * Resampling after observation i happens iff obs_id[i] > 0 and i < T (global last), as in the reference.
 * out_gx[n_batch_used] receives the log-likelihood increments.
 */
int dpomp_pf_partial(dpomp_pf* pf, const double* theta, int32_t n_batch_used, int32_t ymin, int32_t ymax,
                     double* out_gx);

/* outer-layer resample gather (src/hmm_ibis.jl:71-79): filter p <- filter nidx[p] (1-based), p = 1..n */
int dpomp_pf_permute(dpomp_pf* pf, const int64_t* nidx, int32_t n);
/* accepted mutation proposals (src/hmm_ibis.jl:105-108): dst filter dst_slots[k] <- src filter src_slots[k] (1-based) */
int dpomp_pf_copy_filters(dpomp_pf* dst, const dpomp_pf* src, const int64_t* dst_slots,
                          const int64_t* src_slots, int32_t n);
/* read back one population as the reference's Matrix{Int64} (n_particles x C, column-major) */
int dpomp_pf_get_pop(dpomp_pf* pf, int32_t b /*1-based*/, int64_t* out);
int dpomp_pf_set_pop(dpomp_pf* pf, int32_t b /*1-based*/, const int64_t* in);
/* diagnostics of the LAST partial/loglik call: per-particle log weights and ancestors (1-based) of the last
 * observation processed, for filter b; out_anc may be NULL.  Ancestors are valid only if that observation resampled. */
int dpomp_pf_get_last_logw(dpomp_pf* pf, int32_t b, double* out_logw);
int dpomp_pf_get_last_ancestors(dpomp_pf* pf, int32_t b, int64_t* out_anc);
int dpomp_pf_set_record_ancestors(dpomp_pf* pf, int32_t on);  /* switches the diagnostics (log weights AND ancestors) on/off */
/*
 * Hidden-state history of the filters (the filtering distributions that partial_log_likelihood!,
 * src/hmm_particle_filter.jl:39-76, forms at every observation and then discards).
 *
 * dpomp_pf_set_history: flags = 0 (default, off) or an OR of
 *   DPOMP_HISTORY_MOMENTS  per-observation partial sums of the weighted states, for dpomp_pf_get_filtered_moments
 *   DPOMP_HISTORY_PATHS    per-observation states and resampling ancestors, for dpomp_pf_sample_paths
 * The buffers are allocated here, for n_batch filters and all T observations: PATHS needs T * n_batch * n_pad * (4 C + 4)
 * bytes (n_pad = n_particles rounded up to the tile), MOMENTS T * n_batch * (tiles * (3 + 3 C) + 2 C + 1) * 8 bytes.  On an allocation
 * failure the call returns DPOMP_ERR_CUDA and the history is off.  Changing the flags discards the recorded history;
 * setting the current flags again does nothing.  With the history on, partial / loglik run the per-observation launch chain (never the fused or
 * persistent launch), record the log weights (as dpomp_pf_set_record_ancestors does) and run one more kernel per observation;
 * log-likelihoods, populations, event counts and the last-call diagnostics are bit-identical to the history off.
 *
 * The history belongs to the current lineages of the filters.  It covers observations 1..t when every call since the last
 * call with ymin == 1 ran with the history on, each call continuing at the observation after the previous one.
 * dpomp_pf_permute, dpomp_pf_copy_filters (its destination), dpomp_pf_set_pop, dpomp_pf_import_filters and
 * dpomp_pf_resample_migrate discard it.  Both getters return DPOMP_ERR_STATE when the history is off or does not cover
 * 1..t_last for the first n_batch_used filters, and DPOMP_ERR_ARG for other arguments out of range.
 */
#define DPOMP_HISTORY_MOMENTS 1
#define DPOMP_HISTORY_PATHS 2
int dpomp_pf_set_history(dpomp_pf* pf, int32_t flags);
/* Filtering moments at observations 1..t_last: the particles are the simulated states before resampling, weighted by
 * exp(log g) normalised (particles at the event cap weigh 0, as in the filter); an observation with obs_id <= 0 has no
 * likelihood and weighs the n particles equally.  out_mean / out_var [b][t][c] (weighted mean and biased second central
 * moment), out_ess [b][t] = (sum w)^2 / sum w^2 as compute_ess (src/hmm_particle_filter.jl:4-6).  Needs MOMENTS. */
int dpomp_pf_get_filtered_moments(dpomp_pf* pf, int32_t n_batch_used, int32_t t_last, double* out_mean, double* out_var,
                                  double* out_ess);
/* State paths x_1..x_{t_last} by the genealogy of the particles (Kitagawa's filter-smoother; in particle marginal
 * Metropolis-Hastings one such path per step gives samples of (theta, x_1..x_T), Andrieu, Doucet & Holenstein 2010).
 * For each filter, n_paths lineage ends are drawn independently from the weights of observation t_last with the rule of
 * rs_multinomial (src/hmm_resample.jl:9-16): the first particle q with u S < cw_q, cw the filter's own cumulative weights;
 * u = u53 of Philox(key; path, global filter id, t_last - 1, resample tag, block 2).  When observation t_last has obs_id <= 0
 * the end is floor(u n).  Then k_{t-1} = ancestor_{t-1}[k_t] where observation t-1 resampled (k unchanged where it did not)
 * and x_t = state_t[k_t].  out [b][path][t][c] int64, t = 1..t_last (the Julia array C x t_last x n_paths x n_batch_used).
 * The weights of t_last must still be on the device: t_last is the last observation of the last call, and no other filter
 * call may come between (DPOMP_ERR_STATE otherwise).  Needs PATHS. */
int dpomp_pf_sample_paths(dpomp_pf* pf, int32_t n_batch_used, int32_t n_paths, int32_t t_last, uint64_t key, int64_t* out);

/* number of (filter, particle, interval) simulations that hit the event cap since creation (sticky) */
int dpomp_pf_overflow_count(dpomp_pf* pf, int64_t* out_count);
/* total Gillespie events simulated by the last call (all filters) -- for events/s reporting */
int dpomp_pf_last_event_count(dpomp_pf* pf, int64_t* out_events);
/* device time (ms, CUDA events on the handle's stream) and kernel launches of the last call */
int dpomp_pf_last_timing(dpomp_pf* pf, float* out_ms, int32_t* out_launches);

/* per-kernel device time of the last call, measured with CUDA events around every launch when switched on:
 * out_ms2 / out_launches2 = {simulate+weight kernel, resample kernel(s)} summed over the call */
int dpomp_pf_set_kernel_timing(dpomp_pf* pf, int32_t on);
int dpomp_pf_last_kernel_timing(dpomp_pf* pf, float* out_ms2, int32_t* out_launches2);

/* migration of whole filters between devices (multi-GPU SMC^2, SURVEY 8e): pack / unpack the int32 SoA state of the
 * listed filters (1-based) to / from a caller-provided DEVICE buffer of n * C * n_particles int32 */
int dpomp_pf_export_filters(dpomp_pf* pf, const int64_t* slots, int32_t n, void* device_dst);
int dpomp_pf_import_filters(dpomp_pf* pf, const int64_t* slots, int32_t n, const void* device_src);

/* device-resident variant used by bench.py's kernel-only arm: theta and out_ll are DEVICE pointers,
 * nothing crosses PCIe inside the call; synchronises the handle's stream before returning */
int dpomp_pf_loglik_device(dpomp_pf* pf, const double* theta_dev, int32_t n_batch_used, double* out_ll_dev);

/*
 * MBP-IBIS layer (run_mbp_ibis src/hmm_ibis.jl:140-244): n_particles theta-particles, each ONE trajectory with its event
 * list (struct Particle src/hmm_structs.jl:51-58) resident in HBM; max_traj plays MAX_TRAJ (src/DiscretePOMP.jl:40).
 */
typedef struct dpomp_mbp dpomp_mbp;
/* max_traj is the HARD limit of events per trajectory (MAX_TRAJ = 196000 in the reference): reaching it gives log-likelihood
 * -Inf exactly like src/hmm_sim.jl:17-20 / src/hmm_mbp.jl:98-101.  The stores reserve far less (a stride of 1024 events per
 * trajectory at creation) and grow on demand: a walk that reaches the stride is not committed, the stride doubles and the
 * call is repeated for the uncommitted particles with the same random streams, so results never depend on the stride. */
int dpomp_mbp_create(const dpomp_model* model, int32_t n_particles, int32_t max_traj, uint64_t seed, int32_t device,
                     dpomp_mbp** out_mbp);
int dpomp_mbp_destroy(dpomp_mbp* mbp);
int dpomp_mbp_set_batch_offset(dpomp_mbp* mbp, int64_t batch_offset);  /* global id of local particle 0 */
int dpomp_mbp_set_stream_key(dpomp_mbp* mbp, uint64_t key);            /* Philox key of the NEXT call */
int dpomp_mbp_set_mode(dpomp_mbp* mbp, int32_t mode);                  /* trajectory walks: (0) automatic, 1 one thread per trajectory
                                                                         (throughput, many trajectories), 2 one warp per trajectory (latency,
                                                                         up to a few thousand); identical results */
int dpomp_mbp_reset(dpomp_mbp* mbp);  /* every particle back to the initial condition, empty trajectory, log_like = 0 */
/* iterate_particle! (src/hmm_sim.jl:6-25) for particles 1..n up to observation obs_i (1-based); theta is n_params x n
 * column-major; fresh != 0 starts at t = 0 / theta[t0_index], else at the previous observation time.
 * out_logg[n] = observation log-likelihood (-Inf after a trajectory overflow). */
int dpomp_mbp_iterate(dpomp_mbp* mbp, const double* theta, int32_t n, int32_t obs_i, int32_t fresh, double* out_logg);
/* partial_model_based_proposal (src/hmm_mbp.jl:83-108) for particles 1..n: proposal trajectories under theta_f conditional
 * on the current ones (theta_i); valid[p] == 0 marks a proposal outside the prior (log_like = -Inf, nothing simulated).
 * out_loglike[n][2] = Particle.log_like of the proposals.  The proposals stay in the handle until dpomp_mbp_accept. */
int dpomp_mbp_propose(dpomp_mbp* mbp, const double* theta_i, const double* theta_f, const uint8_t* valid, int32_t n,
                      int32_t ymax, double* out_loglike);
int dpomp_mbp_accept(dpomp_mbp* mbp, const int64_t* slots, int32_t n);    /* ptcls[p] = xf (src/hmm_ibis.jl:214), 1-based */
int dpomp_mbp_permute(dpomp_mbp* mbp, const int64_t* nidx, int32_t n);    /* ptcls2[p] = deepcopy(ptcls[nidx[p]]) (:196-199) */
/* migration of particles between ranks (SURVEY.md 8e: lengths first, then one packed payload).  dpomp_mbp_get_lengths
 * returns the event counts of the listed particles (1-based); offsets[k] = position of particle k's events in the packed
 * DEVICE buffers dev_times (f64) / dev_types (u8); dev_fixed holds 16 int32 words per particle (length, final state,
 * log_like[2]).  Import writes into the CURRENT store. */
int dpomp_mbp_get_lengths(dpomp_mbp* mbp, const int64_t* slots, int32_t n, int32_t* out_len);
int dpomp_mbp_export(dpomp_mbp* mbp, const int64_t* slots, const int64_t* offsets, int32_t n, void* dev_fixed,
                     void* dev_times, void* dev_types);
int dpomp_mbp_import(dpomp_mbp* mbp, const int64_t* slots, const int64_t* offsets, int32_t n, const void* dev_fixed,
                     const void* dev_times, const void* dev_types);
/*
 * Device-resident outer layer of run_mbp_ibis (src/hmm_ibis.jl:140-244).  theta, log prior, log-likelihood, weights and the
 * marginal increments of ALL n_total theta-particles live on the device, replicated on every rank of `comm` (a world-size-1
 * communicator for one GPU); the host keeps only scalars (lml, ESS, the proposal scale tj, mu / covariance for the Cholesky
 * factor, the evidence).  The prior must be a product of uniforms (prior_lo / prior_hi), as generate_weak_prior
 * (src/hmm_examples.jl:33-35) and the reference's tests use; other priors take the host-driven entry points above.
 * Proposal and accept draws are Philox streams keyed by the GLOBAL particle id, so results do not depend on the rank count.
 *   begin    theta_all is n_params x n_total column-major; every particle back to the initial condition, w = 1
 *   iterate  iterate_particle! of the rank's block + all-gather + reweight (:176-185);
 *            out5 = { sum w_old, sum w_old gx, sum w_new, sum w_new^2, sum w_new gx }
 *   moments  compute_is_mu_covar! (src/cmn.jl:91-99)
 *   resample rs_systematic / rs_stratified with the given rand() draws, gather, trajectory migration, w = 1 (:194-201);
 *            out2[0] = mean(gx[nidx])
 *   sweep    one mutation sweep over all particles (:203-219): theta_f = (ind_prop ? mu : theta) + scale * chol * z,
 *            partial_model_based_proposal, accept test, accepted trajectories replace the current ones;
 *            out2 = { accepted proposals, mean(mtd_gx) }
 */
int dpomp_mbp_outer_begin(dpomp_mbp* mbp, dpomp_comm* comm, int64_t n_total, const double* theta_all, const double* prior_lo,
                          const double* prior_hi);
int dpomp_mbp_outer_iterate(dpomp_mbp* mbp, int32_t obs_i, int32_t fresh, double* out5);
int dpomp_mbp_outer_moments(dpomp_mbp* mbp, double* out_mu, double* out_cv);
int dpomp_mbp_outer_resample(dpomp_mbp* mbp, int32_t rs_type, const double* u, int64_t n_u, double* out2);
int dpomp_mbp_outer_sweep(dpomp_mbp* mbp, const double* mu, const double* chol, double scale, int32_t ind_prop, int32_t obs_i,
                          double* out2);
int dpomp_mbp_outer_get(dpomp_mbp* mbp, double* out_theta, double* out_w);
int dpomp_mbp_outer_end(dpomp_mbp* mbp);
/* current stride of the stores and the hard limit; dpomp_mbp_reserve widens the stride ahead of time (e.g. before importing
 * trajectories that grew elsewhere) */
int dpomp_mbp_capacity(dpomp_mbp* mbp, int32_t* out_stride, int32_t* out_max_traj);
int dpomp_mbp_reserve(dpomp_mbp* mbp, int32_t stride);
/* final states of particles 1..n, row-major n x C */
int dpomp_mbp_get_states(dpomp_mbp* mbp, int32_t n, int64_t* out);
/* read back one particle (which: 0 current, 1 proposal): final state, event list (types 1-based), log_like[2] */
int dpomp_mbp_get_particle(dpomp_mbp* mbp, int32_t p, int32_t which, int64_t* fc, int64_t* len, double* times,
                           int32_t* types, int64_t cap_out, double* loglike2);

/*
 * Data-augmented MCMC (run_std_mcmc, src/hmm_mcmc.jl; the sampler of run_mcmc_analysis(...; mbp = false)) over the
 * trajectory store of an MBP handle: chain p is trajectory p, theta is n_params x n column-major.
 *
 * Full log-likelihood (compute_full_log_like!, src/hmm_mcmc.jl:78), f64.  From t = t0 (0 or theta[t0_index]) and the initial
 * condition, events and observations are walked in time order (an event at an observation time belongs to the interval that
 * ends there): an event (t_k, e_k) adds log rate[e_k] - (sum of rates) (t_k - t), then its transition applies; an observation
 * subtracts (sum of rates) (t_obs - t) and, if obs_id > 0, adds log g(y | x, theta).  -Inf for a zero-rate event, a negative
 * compartment, an event at or before t0, or an event after the last observation.  out_ll2[p] = {full, observation part}.
 */
int dpomp_da_loglike(dpomp_mbp* mbp, const double* theta, int32_t n, double* out_ll2);  /* writes nothing to the store */
/*
 * One Gibbs step (gibbs_mh_alg!, src/hmm_mcmc.jl:138) for chains 1..n in one launch; kind[p] selects what chain p does:
 *   0  evaluates its trajectory under theta_f (a theta proposal; the host takes the decision): out_ll2[p], store unchanged
 *   1  runs traj_props proposals (src/hmm_std.jl) one after another under theta_cur: kind k uniform on 1..mvp,
 *        1 insert  a type uniform on 1..E at a time uniform on (t0, T]     ratio E (T - t0) / (n + 1)
 *        2 delete  an event uniform on 1..n                                ratio n / (E (T - t0))
 *       >2 move    an event uniform on 1..n to a time uniform on (t0, T]   ratio 1
 *      accepted with probability min(1, ratio exp(l_f - l)); a delete or move of an empty trajectory and an insert into a
 *      trajectory of max_traj events are rejected.  l is the full log-likelihood of the current trajectory under theta_cur.
 *      Accepted edits are written to the store (events, length, final state, log_like = out_ll2[p] under theta_cur);
 *      out_acc[p][3] = accepted inserts, deletes, moves
 *   2  nothing (a theta proposal outside the prior): out_ll2[p] = -Inf
 * T is the last observation time.  The stride grows before the launch to hold traj_props more events than the longest
 * trajectory.  Draws are Philox streams keyed by the call key and the GLOBAL chain id (dpomp_mbp_set_batch_offset), so results
 * do not depend on the number of ranks; the mapping of the words is documented in da.cu.
 */
int dpomp_da_step(dpomp_mbp* mbp, const double* theta_cur, const double* theta_f, const uint8_t* kind, int32_t n,
                  int32_t traj_props, int32_t mvp, double* out_ll2, int32_t* out_acc);

/*
 * Bit-exactness hook for the resampling searches (host buffers).
 *   on_cumulative = 1: `w` is already cumulative  -> rsp_* semantics (src/hmm_pf_resample.jl:24-42, and the
 *                      intended semantics of the broken rsp_stratified/rsp_multinomial :46-63, :5-20)
 *   on_cumulative = 0: `w` are raw weights, cumulated sequentially in f64 on the host exactly as
 *                      cumsum/cumsum! -> rs_* semantics (src/hmm_resample.jl:4-20,44-62,66-83)
 *   u: the raw rand() draws the reference would consume: 1 (systematic), n_out (stratified, n_out == n), n_out (multinomial)
 *   out_idx[n_out]: 1-based ancestors.  The search itself runs on the GPU.
 */
int dpomp_resample_indices(int32_t rs_type, int32_t on_cumulative, const double* w, int64_t n, const double* u,
                           int64_t n_u, int64_t n_out, int64_t* out_idx, int32_t device);

/*
 * Multi-GPU (SURVEY.md 8e): one process per GPU, theta-particles / chains partitioned contiguously over the ranks
 * (dpomp_partition_bounds), NCCL over NVLink inside the library, every collective enqueued on the stream of the handle
 * whose data it moves.  The reference is single-process; these entry points are what a sharded host (Julia with
 * Distributed / MPI.jl, or the Python host of this repository) calls around run_pibis / run_mbp_ibis:
 *   rank 0: dpomp_comm_unique_id -> host-side broadcast of the DPOMP_UNIQUE_ID_BYTES bytes -> every rank: dpomp_comm_create.
 * world == 1 communicators need no id and make every entry point below a local operation.  Like the other handles a
 * communicator is not thread-safe, and its staging buffers are shared by the calls that take it: one call at a time.
 */
#define DPOMP_UNIQUE_ID_BYTES 128
int dpomp_comm_unique_id(void* out_id, int32_t nbytes);
int dpomp_comm_create(const void* id, int32_t nbytes, int32_t rank, int32_t world, int32_t device, dpomp_comm** out_comm);
int dpomp_comm_destroy(dpomp_comm* comm);
int dpomp_comm_info(const dpomp_comm* comm, int32_t* out_rank, int32_t* out_world);
int dpomp_comm_barrier(dpomp_comm* comm);
/* rank's contiguous block [lo, hi) (0-based) of n items; block sizes differ by at most one */
int dpomp_partition_bounds(int64_t n, int32_t world, int32_t rank, int64_t* out_lo, int64_t* out_hi);
/* all-gather of per-item rows of `width` doubles (host buffers): local = this rank's block of the n_total items,
 * out = all n_total rows.  The theta-weight exchange of run_pibis (src/hmm_ibis.jl:57-62) for host-computed values. */
int dpomp_comm_allgather_f64(dpomp_comm* comm, const double* local, int64_t n_total, int32_t width, double* out);
/* dpomp_pf_partial for this rank's block of the n_total filters (n_batch_used must equal the block size) + all-gather of
 * the increments of ALL ranks into out_all[n_total] (src/hmm_ibis.jl:53-62): kernels -> ncclAllGather -> one copy to the
 * host, all on the filter's stream, one synchronisation. */
int dpomp_pf_partial_allgather(dpomp_pf* pf, dpomp_comm* comm, const double* theta_local, int32_t n_batch_used,
                               int32_t ymin, int32_t ymax, int64_t n_total, double* out_all);
/* outer resample across ranks, pop2[p] .= pop[nidx[p]] (src/hmm_ibis.jl:71-79): nidx[n_total] are GLOBAL 1-based ancestors,
 * identical on every rank; remote ancestors arrive as packed int32 populations over NVLink (grouped ncclSend/ncclRecv) */
int dpomp_pf_resample_migrate(dpomp_pf* pf, dpomp_comm* comm, const int64_t* nidx, int64_t n_total);
/* the same for the MBP-IBIS trajectory store, ptcls2[p] = deepcopy(ptcls[nidx[p]]) (src/hmm_ibis.jl:194-201): two-phase
 * exchange (event counts, then fixed records + event times + event types) */
int dpomp_mbp_resample_migrate(dpomp_mbp* mbp, dpomp_comm* comm, const int64_t* nidx, int64_t n_total);

/* diagnostics: the f32 uniform conversions of the event loop evaluated on the device for the given 32-bit Philox words:
 * out_wait in (0, 1] (waiting time), out_event in [0, 1) (choose_event, src/hmm_cmn.jl:5) */
int dpomp_debug_uniforms_f32(const uint32_t* words, int32_t n, float* out_wait, float* out_event);

#ifdef __cplusplus
}
#endif
#endif /* DPOMP_H */
