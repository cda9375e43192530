// capi.cu -- the C ABI of libdpomp (include/dpomp.h): opaque handles, device memory ownership, launch sequencing.
// Host logic only; every numeric step of the path runs in the kernels of pf_sim.cuh / pf_kernels.cu.
#include <math.h>
#include <stdlib.h>
#include <string.h>

#include <new>
#include <string>
#include <vector>

#include "dpomp_dev.cuh"
#include "dpomp_internal.cuh"

using namespace dpomp;

static thread_local std::string g_err;

static int fail(int code, const std::string& msg) {
    g_err = msg;
    return code;
}
int dpomp_set_error(int code, const std::string& msg) { return fail(code, msg); }  // for the other C-ABI TUs
#define CK(expr)                                                                                     \
    do {                                                                                             \
        cudaError_t _e = (expr);                                                                     \
        if (_e != cudaSuccess)                                                                       \
            return fail(DPOMP_ERR_CUDA, std::string(#expr) + ": " + cudaGetErrorString(_e));         \
    } while (0)

static uint64_t splitmix64(uint64_t x) {
    x += 0x9E3779B97F4A7C15ull;
    x = (x ^ (x >> 30)) * 0xBF58476D1CE4E5B9ull;
    x = (x ^ (x >> 27)) * 0x94D049BB133111EBull;
    return x ^ (x >> 31);
}
static uint64_t call_key(const dpomp_pf* pf) {
    return pf->key_forced ? pf->forced_key : splitmix64(pf->seed ^ splitmix64(pf->call_index));
}

extern "C" {

const char* dpomp_last_error(void) { return g_err.c_str(); }
int dpomp_version(void) { return 101; }

int dpomp_device_count(int* out_count) {
    if (!out_count) return fail(DPOMP_ERR_ARG, "out_count is null");
    int n = 0;
    cudaError_t e = cudaGetDeviceCount(&n);
    if (e != cudaSuccess) {
        *out_count = 0;
        return fail(DPOMP_ERR_CUDA, std::string("cudaGetDeviceCount: ") + cudaGetErrorString(e));
    }
    *out_count = n;
    return DPOMP_OK;
}

int dpomp_model_create(const dpomp_model_desc* d, dpomp_model** out_model) {
    if (!d || !out_model) return fail(DPOMP_ERR_ARG, "null argument");
    if (d->n_compartments < 1 || d->n_compartments > DPOMP_MAX_COMPARTMENTS || d->n_events < 1 ||
        d->n_events > DPOMP_MAX_EVENTS || d->n_params < 1 || d->n_params > DPOMP_MAX_PARAMS)
        return fail(DPOMP_ERR_MODEL, "model dimensions outside the device table limits");
    if (d->t0_index < 0 || d->t0_index > d->n_params) return fail(DPOMP_ERR_MODEL, "t0_index out of range");
    if (d->n_obs < 1 || !d->obs_time || !d->obs_id || !d->obs_val) return fail(DPOMP_ERR_MODEL, "no observations");
    if (d->n_obs_vals < 1 || d->n_obs_vals > DPOMP_MAX_OBS_VALS) return fail(DPOMP_ERR_MODEL, "n_obs_vals out of range");
    if (!(d->obs_sigma > 0.0)) return fail(DPOMP_ERR_MODEL, "obs_sigma must be positive");
    for (int e = 0; e < d->n_events; ++e)
        if (d->rate_par[e] >= d->n_params) return fail(DPOMP_ERR_MODEL, "rate_par out of range");
    for (int c = 0; c < d->n_compartments; ++c)
        if (d->initial_condition[c] < 0 || d->initial_condition[c] > 0x7fffffffll)
            return fail(DPOMP_ERR_MODEL, "initial condition outside int32 range");
    for (int t = 1; t < d->n_obs; ++t)
        if (d->obs_time[t] < d->obs_time[t - 1]) return fail(DPOMP_ERR_MODEL, "observations are not sorted by time");
    dpomp_model* m = new (std::nothrow) dpomp_model();
    if (!m) return fail(DPOMP_ERR_ARG, "out of host memory");
    m->h.desc = *d;
    m->h.obs_time.assign(d->obs_time, d->obs_time + d->n_obs);
    m->h.obs_id.assign(d->obs_id, d->obs_id + d->n_obs);
    m->h.obs_val.assign(d->obs_val, d->obs_val + (size_t)d->n_obs * d->n_obs_vals);
    m->h.obs_ysum.resize(d->n_obs);
    for (int t = 0; t < d->n_obs; ++t) {
        int64_t s = 0;
        for (int v = 0; v < d->n_obs_vals; ++v) s += (int64_t)d->obs_ymask[v] * d->obs_val[(size_t)t * d->n_obs_vals + v];
        m->h.obs_ysum[t] = (double)s;
    }
    m->h.desc.obs_time = m->h.obs_time.data();
    m->h.desc.obs_id = m->h.obs_id.data();
    m->h.desc.obs_val = m->h.obs_val.data();
    *out_model = m;
    return DPOMP_OK;
}

// lgamma(Y+1) and, for a fixed negative-binomial size k, lgamma(Y+k) - lgamma(k) of every observation (glibc, as the oracle)
static void count_obs_constants(ModelHost& h) {
    h.obs_lgy.assign(h.obs_ysum.size(), 0.0);
    h.obs_lgk.assign(h.obs_ysum.size(), 0.0);
    const bool fixed_k = h.obs_family == DPOMP_OBS_NEGBIN && h.obs_par_index[1] < 0;
    for (size_t t = 0; t < h.obs_ysum.size(); ++t) {
        const double y = h.obs_ysum[t];
        if (!(y >= 0.0)) continue;  // Y < 0: log g = -Inf, the constants are not read
        h.obs_lgy[t] = lgamma(y + 1.0);
        if (fixed_k) h.obs_lgk[t] = lgamma(y + h.obs_par_value[1]) - lgamma(h.obs_par_value[1]);
    }
}

int dpomp_model_set_obs_model(dpomp_model* model, int32_t family, const int32_t* par_index, const double* par_value) {
    if (!model || !par_index || !par_value) return fail(DPOMP_ERR_ARG, "null argument");
    if (family < DPOMP_OBS_GAUSSIAN || family > DPOMP_OBS_NEGBIN) return fail(DPOMP_ERR_ARG, "unknown observation family");
    if (model->frozen.load()) return fail(DPOMP_ERR_STATE, "the model already has a filter or MBP handle; it is frozen");
    ModelHost& h = model->h;
    const dpomp_model_desc& d = h.desc;
    if (family != DPOMP_OBS_GAUSSIAN) {
        const int n_par = family == DPOMP_OBS_NEGBIN ? 2 : 1;
        for (int i = 0; i < n_par; ++i) {
            if (par_index[i] >= d.n_params || par_index[i] < -1)
                return fail(DPOMP_ERR_MODEL, "observation parameter index out of range");
            if (par_index[i] >= 0) continue;
            const double v = par_value[i];
            const bool ok = family == DPOMP_OBS_BINOMIAL ? (v >= 0.0 && v <= 1.0) : (v > 0.0 && v < INFINITY);
            if (!ok) return fail(DPOMP_ERR_MODEL, family == DPOMP_OBS_BINOMIAL ? "binomial p outside [0, 1]"
                                                                               : "rate / size must be positive and finite");
        }
        for (int c = 0; c < d.n_compartments; ++c)
            if (d.obs_xmask[c] != 0 && d.obs_xmask[c] != 1) return fail(DPOMP_ERR_MODEL, "count families need a 0/1 obs_xmask");
        for (int v = 0; v < d.n_obs_vals; ++v)
            if (d.obs_ymask[v] != 0 && d.obs_ymask[v] != 1) return fail(DPOMP_ERR_MODEL, "count families need a 0/1 obs_ymask");
    }
    h.obs_family = family;
    for (int i = 0; i < 2; ++i) {
        const bool used = family != DPOMP_OBS_GAUSSIAN && (i == 0 || family == DPOMP_OBS_NEGBIN);
        h.obs_par_index[i] = used ? par_index[i] : -1;
        h.obs_par_value[i] = used && par_index[i] < 0 ? par_value[i] : 0.0;
    }
    if (family == DPOMP_OBS_GAUSSIAN) {
        h.obs_lgy.clear();
        h.obs_lgk.clear();
    } else {
        count_obs_constants(h);
    }
    return DPOMP_OK;
}

int dpomp_model_destroy(dpomp_model* model) {
    delete model;
    return DPOMP_OK;
}

static void pf_free(dpomp_pf* pf) {
    if (!pf) return;
    cudaSetDevice(pf->device);
    cudaFree(pf->pop[0]); cudaFree(pf->pop[1]); cudaFree(pf->logw); cudaFree(pf->wtile); cudaFree(pf->cw); cudaFree(pf->anc);
    cudaFree(pf->theta_dev); cudaFree(pf->tile_m); cudaFree(pf->tile_s); cudaFree(pf->tile_f); cudaFree(pf->tile_off);
    cudaFree(pf->grp_m); cudaFree(pf->grp_s); cudaFree(pf->grp_f); cudaFree(pf->grp_off); cudaFree(pf->grp_counter); cudaFree(pf->grp_ev);
    cudaFree(pf->filt_m); cudaFree(pf->filt_s); cudaFree(pf->ll_acc); cudaFree(pf->tile_counter); cudaFree(pf->counters);
    cudaFree(pf->obs_time_dev); cudaFree(pf->obs_ysum_dev); cudaFree(pf->slots_dev); cudaFree(pf->filter_ids_dev); cudaFree(pf->work_counter); cudaFree(pf->filt_gen);
    cudaFree(pf->rows_done); cudaFree(pf->gen_flags); cudaFree(pf->obs_haslik_dev);
    cudaFree(pf->obs_lgy_dev); cudaFree(pf->obs_lgk_dev);
    cudaFreeHost(pf->h_theta); cudaFreeHost(pf->h_ll); cudaFreeHost(pf->h_slots); cudaFreeHost(pf->h_cnt);
    for (cudaEvent_t e : pf->kev) cudaEventDestroy(e);
    if (pf->ev0) cudaEventDestroy(pf->ev0);
    if (pf->ev1) cudaEventDestroy(pf->ev1);
    if (pf->stream) cudaStreamDestroy(pf->stream);
    delete pf;
}

int dpomp_pf_create(const dpomp_model* model, int64_t n_particles, int32_t n_batch, int32_t rs_type, uint64_t seed,
                    int32_t device, dpomp_pf** out_pf) {
    if (!model || !out_pf) return fail(DPOMP_ERR_ARG, "null argument");
    if (n_particles < 1 || n_particles > 0x7fffffffll) return fail(DPOMP_ERR_ARG, "n_particles out of range");
    if (n_batch < 1) return fail(DPOMP_ERR_ARG, "n_batch must be >= 1");
    if (rs_type < 1 || rs_type > 3) return fail(DPOMP_ERR_ARG, "rs_type must be 1, 2 or 3");
    int ndev = 0;
    cudaError_t e = cudaGetDeviceCount(&ndev);
    if (e != cudaSuccess || ndev < 1)
        return fail(DPOMP_ERR_CUDA, std::string("no CUDA device (there is no CPU fallback): ") + cudaGetErrorString(e));
    if (device < 0) CK(cudaGetDevice(&device));
    if (device >= ndev) return fail(DPOMP_ERR_ARG, "device index out of range");
    CK(cudaSetDevice(device));
    const dpomp_model_desc& d = model->h.desc;
    if (!sim_kernel_supported(d.n_compartments, d.n_events)) return fail(DPOMP_ERR_MODEL, "no kernel instantiation covers the model");

    dpomp_pf* pf = new (std::nothrow) dpomp_pf();
    if (!pf) return fail(DPOMP_ERR_ARG, "out of host memory");
    pf->model = model;
    pf->device = device;
    pf->n = n_particles;
    pf->n_batch = n_batch;
    pf->rs_type = rs_type;
    pf->seed = seed;
    pf->items = n_particles <= 256 ? kItemsSmall : kItemsLarge;  // scan-tree geometry: 256-particle tiles for tiny filters, 1024 otherwise
    pf->tile = kBlockThreads * pf->items;
    pf->ntiles = (int)((n_particles + pf->tile - 1) / pf->tile);
    pf->n_pad = (long long)pf->ntiles * pf->tile;
    pf->n_comp = d.n_compartments;
    pf->n_params = d.n_params;
    pf->n_obs = d.n_obs;
    if (const char* ev = getenv("DPOMP_DEFER_L2")) pf->defer_l2_enabled = atoi(ev) != 0;  // A/B knob (scripts/): 0 = two ticket levels
    if (const char* ev = getenv("DPOMP_TWO_PER_LANE")) pf->two_per_lane_mode = atoi(ev);   // A/B and test knob: 0 never, 1 always
    if (cudaDeviceGetAttribute(&pf->sm_count, cudaDevAttrMultiProcessorCount, device) != cudaSuccess) pf->sm_count = 148;
    if ((long long)n_batch * pf->ntiles > 0x7fffffffll) { delete pf; return fail(DPOMP_ERR_ARG, "n_batch * tiles exceeds the grid limit"); }

    const size_t B = (size_t)n_batch, NP = (size_t)pf->n_pad, NT = (size_t)pf->ntiles;
#define ALLOC(ptr, bytes)                                                                                     \
    do {                                                                                                      \
        cudaError_t _e = cudaMalloc((void**)&(ptr), (bytes));                                                 \
        if (_e != cudaSuccess) {                                                                              \
            pf_free(pf);                                                                                      \
            return fail(DPOMP_ERR_CUDA, std::string("cudaMalloc " #ptr ": ") + cudaGetErrorString(_e));       \
        }                                                                                                     \
    } while (0)
    ALLOC(pf->pop[0], B * pf->n_comp * NP * sizeof(int32_t));
    ALLOC(pf->pop[1], B * pf->n_comp * NP * sizeof(int32_t));
    ALLOC(pf->logw, B * NP * sizeof(double));
    ALLOC(pf->wtile, B * NP * sizeof(double));
    if (rs_type == DPOMP_RS_MULTINOMIAL) ALLOC(pf->cw, B * NP * sizeof(double));
    ALLOC(pf->theta_dev, B * pf->n_params * sizeof(double));
    ALLOC(pf->tile_m, B * NT * sizeof(double));
    ALLOC(pf->tile_s, B * NT * sizeof(double));
    ALLOC(pf->tile_f, B * NT * sizeof(double));
    ALLOC(pf->tile_off, B * (NT + 1) * sizeof(double));
    pf->ngroups = (pf->ntiles + kGroupTiles - 1) / kGroupTiles;
    const size_t NG = (size_t)pf->ngroups;
    ALLOC(pf->grp_m, B * NG * sizeof(double));
    ALLOC(pf->grp_s, B * NG * sizeof(double));
    ALLOC(pf->grp_f, B * NG * sizeof(double));
    ALLOC(pf->grp_off, B * NG * sizeof(double));
    ALLOC(pf->grp_counter, B * NG * sizeof(unsigned int));
    ALLOC(pf->grp_ev, B * NG * sizeof(unsigned long long));
    ALLOC(pf->filt_m, B * sizeof(double));
    ALLOC(pf->filt_s, B * sizeof(double));
    ALLOC(pf->ll_acc, B * sizeof(double));
    ALLOC(pf->tile_counter, B * sizeof(unsigned int));
    ALLOC(pf->counters, 2 * sizeof(unsigned long long));
    ALLOC(pf->obs_time_dev, (size_t)d.n_obs * sizeof(double));
    ALLOC(pf->obs_ysum_dev, (size_t)d.n_obs * sizeof(double));
    ALLOC(pf->slots_dev, 2 * B * sizeof(int64_t));
    ALLOC(pf->filter_ids_dev, B * sizeof(uint32_t));
    ALLOC(pf->work_counter, sizeof(unsigned long long));
    ALLOC(pf->filt_gen, B * sizeof(unsigned int));
    const bool count_obs = model->h.obs_family != DPOMP_OBS_GAUSSIAN;
    if (count_obs) {
        ALLOC(pf->obs_lgy_dev, (size_t)d.n_obs * sizeof(double));
        ALLOC(pf->obs_lgk_dev, (size_t)d.n_obs * sizeof(double));
    }
#undef ALLOC
    bool ok = cudaMallocHost((void**)&pf->h_theta, B * pf->n_params * sizeof(double)) == cudaSuccess &&
              cudaMallocHost((void**)&pf->h_ll, B * sizeof(double)) == cudaSuccess &&
              cudaMallocHost((void**)&pf->h_slots, 2 * B * sizeof(int64_t)) == cudaSuccess &&
              cudaMallocHost((void**)&pf->h_cnt, sizeof(unsigned long long)) == cudaSuccess &&
              cudaStreamCreateWithFlags(&pf->stream, cudaStreamNonBlocking) == cudaSuccess &&
              cudaEventCreate(&pf->ev0) == cudaSuccess && cudaEventCreate(&pf->ev1) == cudaSuccess &&
              cudaMemsetAsync(pf->pop[0], 0, B * pf->n_comp * NP * sizeof(int32_t), pf->stream) == cudaSuccess &&
              cudaMemsetAsync(pf->pop[1], 0, B * pf->n_comp * NP * sizeof(int32_t), pf->stream) == cudaSuccess &&
              cudaMemsetAsync(pf->tile_counter, 0, B * sizeof(unsigned int), pf->stream) == cudaSuccess &&
              cudaMemsetAsync(pf->grp_counter, 0, B * (size_t)pf->ngroups * sizeof(unsigned int), pf->stream) == cudaSuccess &&
              cudaMemsetAsync(pf->counters, 0, 2 * sizeof(unsigned long long), pf->stream) == cudaSuccess &&
              cudaMemsetAsync(pf->work_counter, 0, sizeof(unsigned long long), pf->stream) == cudaSuccess &&
              cudaMemsetAsync(pf->filt_gen, 0, B * sizeof(unsigned int), pf->stream) == cudaSuccess &&
              cudaMemcpyAsync(pf->obs_time_dev, model->h.obs_time.data(), (size_t)d.n_obs * sizeof(double),
                              cudaMemcpyHostToDevice, pf->stream) == cudaSuccess &&
              cudaMemcpyAsync(pf->obs_ysum_dev, model->h.obs_ysum.data(), (size_t)d.n_obs * sizeof(double),
                              cudaMemcpyHostToDevice, pf->stream) == cudaSuccess &&
              (!count_obs ||
               (cudaMemcpyAsync(pf->obs_lgy_dev, model->h.obs_lgy.data(), (size_t)d.n_obs * sizeof(double),
                                cudaMemcpyHostToDevice, pf->stream) == cudaSuccess &&
                cudaMemcpyAsync(pf->obs_lgk_dev, model->h.obs_lgk.data(), (size_t)d.n_obs * sizeof(double),
                                cudaMemcpyHostToDevice, pf->stream) == cudaSuccess)) &&
              cudaStreamSynchronize(pf->stream) == cudaSuccess;
    if (!ok) {
        std::string msg = std::string("pf setup: ") + cudaGetErrorString(cudaGetLastError());
        pf_free(pf);
        return fail(DPOMP_ERR_CUDA, msg);
    }
    model->frozen.store(true);
    *out_pf = pf;
    return DPOMP_OK;
}

int dpomp_pf_destroy(dpomp_pf* pf) {
    pf_free(pf);
    return DPOMP_OK;
}

int dpomp_pf_set_sim_precision(dpomp_pf* pf, int32_t p) {
    if (!pf || (p != DPOMP_SIM_F32 && p != DPOMP_SIM_F64)) return fail(DPOMP_ERR_ARG, "bad sim precision");
    pf->sim_precision = p;
    return DPOMP_OK;
}
int dpomp_pf_set_max_events(dpomp_pf* pf, int64_t m) {
    if (!pf || m < 1 || m > 0x7fffffffll) return fail(DPOMP_ERR_ARG, "max_events out of range");
    pf->max_events = m;
    return DPOMP_OK;
}
int dpomp_pf_set_batch_offset(dpomp_pf* pf, int64_t off) {
    if (!pf || off < 0 || off + pf->n_batch > 0xffffffffll) return fail(DPOMP_ERR_ARG, "batch_offset out of range");
    pf->batch_offset = off;
    return DPOMP_OK;
}
int dpomp_pf_set_fused(dpomp_pf* pf, int32_t on) {
    if (!pf) return fail(DPOMP_ERR_ARG, "null handle");
    pf->fused_enabled = on != 0;
    pf->fused_mode = on >= 2 ? 2 : 1;
    return DPOMP_OK;
}
int dpomp_pf_set_persistent(dpomp_pf* pf, int32_t mode) {
    if (!pf || mode < 0 || mode > 2) return fail(DPOMP_ERR_ARG, "persistent mode must be 0, 1 or 2");
    pf->persist_mode = mode;
    return DPOMP_OK;
}
int dpomp_pf_set_scatter(dpomp_pf* pf, int32_t mode) {
    if (!pf || (mode != DPOMP_SCATTER_REFERENCE && mode != DPOMP_SCATTER_INTERLEAVED)) return fail(DPOMP_ERR_ARG, "bad scatter mode");
    pf->scatter_mode = mode;
    return DPOMP_OK;
}
int dpomp_pf_set_filter_ids(dpomp_pf* pf, const int64_t* ids, int32_t n) {
    if (!pf) return fail(DPOMP_ERR_ARG, "null handle");
    if (!ids) { pf->use_filter_ids = false; return DPOMP_OK; }
    if (n < 1 || n > pf->n_batch) return fail(DPOMP_ERR_ARG, "n out of range");
    CK(cudaSetDevice(pf->device));
    std::vector<uint32_t> tmp((size_t)n);
    for (int i = 0; i < n; ++i) {
        if (ids[i] < 0 || ids[i] > 0xffffffffll) return fail(DPOMP_ERR_ARG, "filter id out of range");
        tmp[(size_t)i] = (uint32_t)ids[i];
    }
    CK(cudaMemcpyAsync(pf->filter_ids_dev, tmp.data(), (size_t)n * sizeof(uint32_t), cudaMemcpyHostToDevice, pf->stream));
    CK(cudaStreamSynchronize(pf->stream));
    pf->use_filter_ids = true;
    return DPOMP_OK;
}
int dpomp_pf_set_stream_key(dpomp_pf* pf, uint64_t key) {
    if (!pf) return fail(DPOMP_ERR_ARG, "null handle");
    pf->forced_key = key;
    pf->key_forced = true;
    return DPOMP_OK;
}
int dpomp_pf_get_stream_key(dpomp_pf* pf, uint64_t* out_key) {
    if (!pf || !out_key) return fail(DPOMP_ERR_ARG, "null argument");
    *out_key = call_key(pf);
    return DPOMP_OK;
}
int dpomp_pf_geometry(const dpomp_pf* pf, int32_t* out_tile, int32_t* out_items) {
    if (!pf || !out_tile || !out_items) return fail(DPOMP_ERR_ARG, "null argument");
    *out_tile = pf->tile;
    *out_items = pf->items;
    return DPOMP_OK;
}
int dpomp_pf_set_record_ancestors(dpomp_pf* pf, int32_t on) {
    if (!pf) return fail(DPOMP_ERR_ARG, "null handle");
    CK(cudaSetDevice(pf->device));
    if (on && !pf->anc) CK(cudaMalloc((void**)&pf->anc, (size_t)pf->n_batch * pf->n_pad * sizeof(int32_t)));
    pf->record_anc = on != 0;
    return DPOMP_OK;
}

// kind >= 0 opens a timed launch slot, kind < 0 closes the open one
static cudaError_t kernel_event(dpomp_pf* pf, int kind, cudaStream_t st) {
    if (kind >= 0) {
        const size_t slot = pf->kev_kind.size();
        while (pf->kev.size() < 2 * (slot + 1)) {
            cudaEvent_t e;
            cudaError_t err = cudaEventCreate(&e);
            if (err != cudaSuccess) return err;
            pf->kev.push_back(e);
        }
        pf->kev_kind.push_back(kind);
        return cudaEventRecord(pf->kev[2 * slot], st);
    }
    return cudaEventRecord(pf->kev[2 * (pf->kev_kind.size() - 1) + 1], st);
}

// the launch sequence of partial_log_likelihood! (src/hmm_particle_filter.jl:39-76), batched over filters
int dpomp_run_partial_enqueue(dpomp_pf* pf, const double* theta, bool theta_on_device, int nb, int ymin, int ymax, double* out,
                              int out_mode) {
    if (!pf || !theta || (!out && out_mode != 2)) return fail(DPOMP_ERR_ARG, "null argument");
    if (nb < 1 || nb > pf->n_batch) return fail(DPOMP_ERR_ARG, "n_batch_used out of range");
    if (ymin < 1 || ymax < ymin || ymax > pf->n_obs) return fail(DPOMP_ERR_ARG, "observation range out of bounds");
    if (ymin > 1 && !pf->initialised) return fail(DPOMP_ERR_STATE, "ymin > 1 on a filter that has never been run from ymin == 1");
    CK(cudaSetDevice(pf->device));
    const ModelHost& mh = pf->model->h;
    const uint64_t key = call_key(pf);
    pf->key_forced = false;
    pf->call_index += 1;
    cudaStream_t st = pf->stream;
    CK(cudaEventRecord(pf->ev0, st));
    const size_t th_bytes = (size_t)nb * pf->n_params * sizeof(double);
    if (theta_on_device) {
        CK(cudaMemcpyAsync(pf->theta_dev, theta, th_bytes, cudaMemcpyDeviceToDevice, st));
    } else {
        memcpy(pf->h_theta, theta, th_bytes);
        CK(cudaMemcpyAsync(pf->theta_dev, pf->h_theta, th_bytes, cudaMemcpyHostToDevice, st));
    }
    CK(cudaMemsetAsync(pf->ll_acc, 0, (size_t)nb * sizeof(double), st));
    CK(cudaMemsetAsync(pf->counters, 0, sizeof(unsigned long long), st));
    CK(cudaMemsetAsync(pf->grp_ev, 0, (size_t)nb * pf->ngroups * sizeof(unsigned long long), st));
    int launches = 0;
    pf->kev_kind.clear();
    bool fused_ok = false;
    if (pf->fused_enabled && pf->rs_type != DPOMP_RS_MULTINOMIAL) {
        int& cap = pf->fused_capacity[pf->sim_precision == DPOMP_SIM_F64 ? 1 : 0];
        if (cap < 0) cap = sim_fused_capacity(mh, pf->sim_precision, pf->items);
        // measured on B200: with several tiles per filter the CTAs that wait for the combine hold SM slots and the fused
        // launch loses to the two-kernel PDL chain (C2 4.25 vs 4.10 ms, SEIR 64 x 65536 18.8 vs 16.9 ms); with one tile per
        // filter nothing waits and it wins slightly (1024 x 1024: 4.02 vs 4.10 ms).  fused_mode 2 forces it when it fits.
        fused_ok = cap >= pf->ntiles && (pf->ntiles == 1 || pf->fused_mode == 2);
    }
    // persistent path: ONE cooperative launch for all observations of the call (pf_sim.cuh, MODE 2) when every CTA of the
    // launch is co-resident; otherwise the per-observation launch chain below
    bool persist_ok = false;
    if (pf->persist_mode != 0 && pf->rs_type != DPOMP_RS_MULTINOMIAL && pf->sim_precision == DPOMP_SIM_F32 && !pf->kernel_timing &&
        make_chunk_perm(pf->scatter_mode, pf->n, pf->ntiles).ncf == 0 && (pf->persist_mode == 2 || ymax > ymin)) {
        if (pf->persist_capacity < 0) pf->persist_capacity = sim_persist_capacity(mh, pf->sim_precision, pf->items);
        persist_ok = (long long)nb * pf->ntiles <= pf->persist_capacity;
    }
    if (persist_ok) {
        const size_t B = (size_t)pf->n_batch;
        if (!pf->rows_done) {
            std::vector<int> hl((size_t)pf->n_obs);
            for (int t = 0; t < pf->n_obs; ++t) hl[(size_t)t] = mh.obs_id[(size_t)t] > 0;
            CK(cudaMalloc((void**)&pf->rows_done, B * pf->ntiles * sizeof(unsigned int)));
            if (!pf->gen_flags) {
                CK(cudaMalloc((void**)&pf->gen_flags, B * pf->ngroups * 32 * sizeof(unsigned int)));
                CK(cudaMemsetAsync(pf->gen_flags, 0, B * pf->ngroups * 32 * sizeof(unsigned int), st));
            }
            CK(cudaMalloc((void**)&pf->obs_haslik_dev, (size_t)pf->n_obs * sizeof(int)));
            CK(cudaMemcpyAsync(pf->obs_haslik_dev, hl.data(), (size_t)pf->n_obs * sizeof(int), cudaMemcpyHostToDevice, st));
            CK(cudaStreamSynchronize(st));  // hl is a stack vector
        }
        CK(cudaMemsetAsync(pf->rows_done, 0, (size_t)nb * pf->ntiles * sizeof(unsigned int), st));
        SimLaunch a{};
        a.pop = pf->pop[pf->cur]; a.pop_dst = pf->pop[pf->cur ^ 1];
        a.logw = pf->logw; a.wtile = pf->wtile; a.record_logw = pf->record_anc ? 1 : 0;
        a.theta = pf->theta_dev; a.obs_time = pf->obs_time_dev; a.obs_ysum = pf->obs_ysum_dev;
        a.tile_m = pf->tile_m; a.tile_s = pf->tile_s; a.tile_f = pf->tile_f; a.tile_off = pf->tile_off;
        a.filt_m = pf->filt_m; a.filt_s = pf->filt_s; a.ll_acc = pf->ll_acc;
        a.grp_m = pf->grp_m; a.grp_s = pf->grp_s; a.grp_f = pf->grp_f; a.grp_off = pf->grp_off;
        a.grp_counter = pf->grp_counter; a.ngroups = pf->ngroups; a.tile_counter = pf->tile_counter;
        a.ev_count = pf->counters; a.ovf_count = pf->counters + 1; a.grp_ev = pf->grp_ev;
        a.n = pf->n; a.n_pad = pf->n_pad; a.ntiles = pf->ntiles; a.n_filters = nb; a.n_comp = pf->n_comp;
        a.t = ymin - 1; a.t_last = ymax - 1; a.n_obs_total = pf->n_obs; a.obs_haslik = pf->obs_haslik_dev;
        a.fresh = (ymin == 1); a.has_lik = 0; a.do_resample = 0;
        a.rs_type = pf->rs_type; a.anc = pf->record_anc ? pf->anc : nullptr;
        a.perm = make_chunk_perm(0, pf->n, pf->ntiles);
        a.rows_done = pf->rows_done; a.gen_flags = pf->gen_flags; a.gen = pf->gen + 1;
        a.key = key; a.filter0 = (uint32_t)pf->batch_offset; a.max_events = pf->max_events;
        a.filter_ids = pf->use_filter_ids ? pf->filter_ids_dev : nullptr;
        cudaError_t le = launch_sim_weight(mh, pf->sim_precision, pf->items, 3, a, st);
        if (le == cudaSuccess) {
            int flips = 0, last_rs = 0;
            for (int oi = ymin; oi <= ymax; ++oi) {
                last_rs = (mh.obs_id[(size_t)oi - 1] > 0) && oi < pf->n_obs;
                flips += last_rs;
            }
            pf->gen += (unsigned int)(ymax - ymin + 1);
            pf->cur ^= (flips & 1);
            pf->last_resampled = last_rs != 0;
            launches = 1;
        } else if (le == cudaErrorCooperativeLaunchTooLarge || le == cudaErrorLaunchOutOfResources) {
            (void)cudaGetLastError();  // not co-resident after all (another context holds SMs): per-observation chain
            pf->persist_capacity = 0;
            persist_ok = false;
        } else {
            return fail(DPOMP_ERR_CUDA, std::string("persistent launch: ") + cudaGetErrorString(le));
        }
    }
    for (int oi = ymin; oi <= ymax && !persist_ok; ++oi) {
        const int t = oi - 1;
        const int has_lik = mh.obs_id[t] > 0;
        const int do_rs = has_lik && oi < pf->n_obs;  // src/hmm_particle_filter.jl:58,62
        SimLaunch a{};
        a.pop = pf->pop[pf->cur];
        a.logw = pf->logw;
        a.wtile = pf->wtile;
        a.record_logw = pf->record_anc ? 1 : 0;
        a.theta = pf->theta_dev;
        a.obs_time = pf->obs_time_dev;
        a.obs_ysum = pf->obs_ysum_dev;
        a.tile_m = pf->tile_m; a.tile_s = pf->tile_s; a.tile_f = pf->tile_f; a.tile_off = pf->tile_off;
        a.filt_m = pf->filt_m; a.filt_s = pf->filt_s; a.ll_acc = pf->ll_acc;
        a.grp_m = pf->grp_m; a.grp_s = pf->grp_s; a.grp_f = pf->grp_f; a.grp_off = pf->grp_off;
        a.grp_counter = pf->grp_counter; a.ngroups = pf->ngroups;
        a.tile_counter = pf->tile_counter;
        a.ev_count = pf->counters; a.ovf_count = pf->counters + 1; a.grp_ev = pf->grp_ev;
        a.n = pf->n; a.n_pad = pf->n_pad; a.ntiles = pf->ntiles; a.n_filters = nb; a.n_comp = pf->n_comp;
        a.t = t; a.fresh = (oi == 1); a.has_lik = has_lik;
        a.key = key; a.filter0 = (uint32_t)pf->batch_offset; a.max_events = pf->max_events;
        a.filter_ids = pf->use_filter_ids ? pf->filter_ids_dev : nullptr;
        a.cobs = count_obs_of(mh, pf->obs_lgy_dev, pf->obs_lgk_dev);
        // one fused launch (simulate + resample) when every tile of a filter can be resident at once
        const bool fused = do_rs && fused_ok;
        bool fused_tickets = false;
        // two-kernel chain: level 2 of the combine runs in the resample kernel (no second ticket level in the simulate kernel)
        // -- in the latency regime only (the launch is at most one wave of CTAs): measured on B200, C2 3.39 -> 3.26 ms and 8 x 65536
        // SEIR 2.88 -> 2.76 ms, but 64 x 65536 SEIR 13.06 -> 13.55 ms (every CTA of a multi-wave launch repeats level 2, and the
        // serial tail it removes is amortised over the waves anyway)
        const bool defer_l2 = do_rs && !fused && pf->ngroups <= kDeferGroups && pf->defer_l2_enabled &&
                              (long long)nb * pf->ntiles <= 8ll * pf->sm_count;
        a.defer_l2 = defer_l2 ? 1 : 0;
        // two particles per lane on 1024-particle tiles: event-heavy model (>= 16 events per particle-step in the previous call of
        // this handle) in a launch of at most one wave of CTAs (pf_sim.cuh, sim_plain_two_per_lane; measured: 256 CTAs -22 %,
        // 512 -6.6 %, 768 / 1024 -5.4 %, 4096 +0.7 %)
        a.two_per_lane = pf->two_per_lane_mode >= 0 ? pf->two_per_lane_mode
                         : ((long long)nb * pf->ntiles <= 8ll * pf->sm_count && pf->last_steps > 0 &&
                            pf->last_events >= 16 * pf->last_steps);
        if (fused) {
            a.do_resample = 1;
            a.rs_type = pf->rs_type;
            a.pop_dst = pf->pop[pf->cur ^ 1];
            a.anc = pf->record_anc ? pf->anc : nullptr;
            a.perm = make_chunk_perm(pf->scatter_mode, pf->n, pf->ntiles);
            // arrival-order tickets only when the launch has more CTAs than the device holds at once
            fused_tickets = (long long)nb * pf->ntiles > pf->fused_capacity[pf->sim_precision == DPOMP_SIM_F64 ? 1 : 0];
            a.work_counter = fused_tickets ? pf->work_counter : nullptr;
            a.work_base = pf->work_base;
            a.filt_gen = pf->filt_gen;
            if (!pf->gen_flags) {
                const size_t fb = (size_t)pf->n_batch * pf->ngroups * 32 * sizeof(unsigned int);
                CK(cudaMalloc((void**)&pf->gen_flags, fb));
                CK(cudaMemsetAsync(pf->gen_flags, 0, fb, st));
            }
            a.gen_flags = pf->gen_flags;
            a.gen = pf->gen + 1;
        }
        if (pf->kernel_timing) CK(kernel_event(pf, 0, st));
        CK(launch_sim_weight(mh, pf->sim_precision, pf->items, fused ? 1 : 0, a, st));
        if (pf->kernel_timing) CK(kernel_event(pf, -1, st));
        ++launches;
        if (fused) {
            // the host mirrors of the device ticket counter / generation advance only once the launch is enqueued: a failed
            // launch leaves the handle consistent (the device counter has not moved either)
            pf->gen += 1;
            if (fused_tickets) pf->work_base += (unsigned long long)nb * pf->ntiles;
            pf->cur ^= 1;
        } else if (do_rs) {
            ResampleLaunch r{};
            r.pop_src = pf->pop[pf->cur]; r.pop_dst = pf->pop[pf->cur ^ 1];
            r.wtile = pf->wtile; r.tile_m = pf->tile_m; r.tile_f = pf->tile_f; r.tile_off = pf->tile_off; r.filt_s = pf->filt_s;
            r.grp_f = pf->grp_f; r.grp_off = pf->grp_off; r.ngroups = pf->ngroups;
            r.defer_l2 = defer_l2 ? 1 : 0; r.has_lik = has_lik;
            r.grp_m = pf->grp_m; r.grp_s = pf->grp_s; r.grp_f_w = pf->grp_f; r.grp_off_w = pf->grp_off;
            r.filt_s_w = pf->filt_s; r.filt_m_w = pf->filt_m; r.ll_acc = pf->ll_acc;
            r.anc = pf->record_anc ? pf->anc : nullptr;
            r.cw = pf->cw;
            r.n = pf->n; r.n_pad = pf->n_pad; r.ntiles = pf->ntiles; r.n_filters = nb; r.n_comp = pf->n_comp;
            r.t = t; r.rs_type = pf->rs_type; r.key = key; r.filter0 = (uint32_t)pf->batch_offset;
            r.perm = make_chunk_perm(pf->scatter_mode, pf->n, pf->ntiles);
            r.filter_ids = pf->use_filter_ids ? pf->filter_ids_dev : nullptr;
            if (pf->kernel_timing) CK(kernel_event(pf, 1, st));
            CK(launch_resample(pf->items, r, st));
            if (pf->kernel_timing) CK(kernel_event(pf, -1, st));
            launches += (pf->rs_type == DPOMP_RS_MULTINOMIAL) ? 2 : 1;
            pf->cur ^= 1;
        }
        pf->last_resampled = do_rs != 0;
    }
    if (out_mode == 1) {
        CK(cudaMemcpyAsync(out, pf->ll_acc, (size_t)nb * sizeof(double), cudaMemcpyDeviceToDevice, st));
    } else if (out_mode == 0) {
        CK(cudaMemcpyAsync(pf->h_ll, pf->ll_acc, (size_t)nb * sizeof(double), cudaMemcpyDeviceToHost, st));
    }
    CK(launch_sum_events(pf->grp_ev, (long long)nb * pf->ngroups, pf->counters, st));
    CK(cudaMemcpyAsync(pf->h_cnt, pf->counters, sizeof(unsigned long long), cudaMemcpyDeviceToHost, st));
    CK(cudaEventRecord(pf->ev1, st));
    pf->last_launches = launches;
    pf->enqueued_steps = (long long)nb * pf->n * (ymax - ymin + 1);
    return DPOMP_OK;
}

int dpomp_run_partial_finish(dpomp_pf* pf, double* out, int nb, int out_mode) {
    CK(cudaStreamSynchronize(pf->stream));
    if (out_mode == 0) memcpy(out, pf->h_ll, (size_t)nb * sizeof(double));
    CK(cudaEventElapsedTime(&pf->last_ms, pf->ev0, pf->ev1));
    pf->last_events = (long long)*pf->h_cnt;
    pf->last_steps = pf->enqueued_steps;
    pf->kernel_ms[0] = pf->kernel_ms[1] = 0.f;
    pf->kernel_launches[0] = pf->kernel_launches[1] = 0;
    for (size_t i = 0; i < pf->kev_kind.size(); ++i) {
        float ms = 0.f;
        CK(cudaEventElapsedTime(&ms, pf->kev[2 * i], pf->kev[2 * i + 1]));
        pf->kernel_ms[pf->kev_kind[i]] += ms;
        pf->kernel_launches[pf->kev_kind[i]] += 1;
    }
    pf->initialised = true;
    return DPOMP_OK;
}

static int run_partial(dpomp_pf* pf, const double* theta, bool theta_on_device, int nb, int ymin, int ymax, double* out,
                       bool out_on_device) {
    const int mode = out_on_device ? 1 : 0;
    int rc = dpomp_run_partial_enqueue(pf, theta, theta_on_device, nb, ymin, ymax, out, mode);
    return rc ? rc : dpomp_run_partial_finish(pf, out, nb, mode);
}

int dpomp_pf_loglik(dpomp_pf* pf, const double* theta, int32_t nb, double* out_ll) {
    if (!pf) return fail(DPOMP_ERR_ARG, "null handle");
    return run_partial(pf, theta, false, nb, 1, pf->n_obs, out_ll, false);
}
int dpomp_pf_loglik_device(dpomp_pf* pf, const double* theta_dev, int32_t nb, double* out_ll_dev) {
    if (!pf) return fail(DPOMP_ERR_ARG, "null handle");
    return run_partial(pf, theta_dev, true, nb, 1, pf->n_obs, out_ll_dev, true);
}
int dpomp_pf_partial(dpomp_pf* pf, const double* theta, int32_t nb, int32_t ymin, int32_t ymax, double* out_gx) {
    return run_partial(pf, theta, false, nb, ymin, ymax, out_gx, false);
}

static int upload_slots(dpomp_pf* pf, const int64_t* a, const int64_t* b, int n, int limit_a, int limit_b) {
    for (int i = 0; i < n; ++i) {
        if (a && (a[i] < 1 || a[i] > limit_a)) return fail(DPOMP_ERR_ARG, "filter index out of range");
        if (b && (b[i] < 1 || b[i] > limit_b)) return fail(DPOMP_ERR_ARG, "filter index out of range");
        if (a) pf->h_slots[i] = a[i];
        if (b) pf->h_slots[pf->n_batch + i] = b[i];
    }
    CK(cudaMemcpyAsync(pf->slots_dev, pf->h_slots, 2 * (size_t)pf->n_batch * sizeof(int64_t), cudaMemcpyHostToDevice, pf->stream));
    return DPOMP_OK;
}

int dpomp_pf_permute(dpomp_pf* pf, const int64_t* nidx, int32_t n) {
    if (!pf || !nidx) return fail(DPOMP_ERR_ARG, "null argument");
    if (n < 1 || n > pf->n_batch) return fail(DPOMP_ERR_ARG, "n out of range");
    CK(cudaSetDevice(pf->device));
    int rc = upload_slots(pf, nullptr, nidx, n, 0, pf->n_batch);
    if (rc) return rc;
    const long long stride = (long long)pf->n_comp * pf->n_pad;
    CK(launch_gather_filters(pf->pop[pf->cur ^ 1], pf->pop[pf->cur], nullptr, pf->slots_dev + pf->n_batch, n, stride, pf->stream));
    if (n < pf->n_batch)  // filters beyond n keep their state
        CK(cudaMemcpyAsync(pf->pop[pf->cur ^ 1] + (size_t)n * stride, pf->pop[pf->cur] + (size_t)n * stride,
                           (size_t)(pf->n_batch - n) * stride * sizeof(int32_t), cudaMemcpyDeviceToDevice, pf->stream));
    CK(cudaStreamSynchronize(pf->stream));
    pf->cur ^= 1;
    return DPOMP_OK;
}

int dpomp_pf_copy_filters(dpomp_pf* dst, const dpomp_pf* src, const int64_t* dst_slots, const int64_t* src_slots, int32_t n) {
    if (!dst || !src || !dst_slots || !src_slots) return fail(DPOMP_ERR_ARG, "null argument");
    if (n == 0) return DPOMP_OK;
    if (n < 0 || n > dst->n_batch) return fail(DPOMP_ERR_ARG, "n out of range");
    if (dst->n_pad != src->n_pad || dst->n_comp != src->n_comp || dst->device != src->device)
        return fail(DPOMP_ERR_ARG, "filters have different geometry or device");
    CK(cudaSetDevice(dst->device));
    int rc = upload_slots(dst, dst_slots, src_slots, n, dst->n_batch, src->n_batch);
    if (rc) return rc;
    const long long stride = (long long)dst->n_comp * dst->n_pad;
    CK(launch_gather_filters(dst->pop[dst->cur], src->pop[src->cur], dst->slots_dev, dst->slots_dev + dst->n_batch, n, stride, dst->stream));
    CK(cudaStreamSynchronize(dst->stream));
    dst->initialised = true;
    return DPOMP_OK;
}

int dpomp_pf_get_pop(dpomp_pf* pf, int32_t b, int64_t* out) {
    if (!pf || !out) return fail(DPOMP_ERR_ARG, "null argument");
    if (b < 1 || b > pf->n_batch) return fail(DPOMP_ERR_ARG, "filter index out of range");
    CK(cudaSetDevice(pf->device));
    const size_t words = (size_t)pf->n_comp * pf->n_pad;
    std::vector<int32_t> tmp(words);
    CK(cudaMemcpyAsync(tmp.data(), pf->pop[pf->cur] + (size_t)(b - 1) * words, words * sizeof(int32_t), cudaMemcpyDeviceToHost, pf->stream));
    CK(cudaStreamSynchronize(pf->stream));
    for (int c = 0; c < pf->n_comp; ++c)
        for (long long p = 0; p < pf->n; ++p) out[(size_t)c * pf->n + p] = tmp[(size_t)c * pf->n_pad + p];
    return DPOMP_OK;
}

int dpomp_pf_set_pop(dpomp_pf* pf, int32_t b, const int64_t* in) {
    if (!pf || !in) return fail(DPOMP_ERR_ARG, "null argument");
    if (b < 1 || b > pf->n_batch) return fail(DPOMP_ERR_ARG, "filter index out of range");
    CK(cudaSetDevice(pf->device));
    const size_t words = (size_t)pf->n_comp * pf->n_pad;
    std::vector<int32_t> tmp(words, 0);
    for (int c = 0; c < pf->n_comp; ++c)
        for (long long p = 0; p < pf->n; ++p) tmp[(size_t)c * pf->n_pad + p] = (int32_t)in[(size_t)c * pf->n + p];
    CK(cudaMemcpyAsync(pf->pop[pf->cur] + (size_t)(b - 1) * words, tmp.data(), words * sizeof(int32_t), cudaMemcpyHostToDevice, pf->stream));
    CK(cudaStreamSynchronize(pf->stream));
    pf->initialised = true;
    return DPOMP_OK;
}

int dpomp_pf_get_last_logw(dpomp_pf* pf, int32_t b, double* out) {
    if (!pf || !out) return fail(DPOMP_ERR_ARG, "null argument");
    if (b < 1 || b > pf->n_batch) return fail(DPOMP_ERR_ARG, "filter index out of range");
    if (!pf->record_anc) return fail(DPOMP_ERR_STATE, "diagnostics recording is off (dpomp_pf_set_record_ancestors)");
    CK(cudaSetDevice(pf->device));
    CK(cudaMemcpyAsync(out, pf->logw + (size_t)(b - 1) * pf->n_pad, (size_t)pf->n * sizeof(double), cudaMemcpyDeviceToHost, pf->stream));
    CK(cudaStreamSynchronize(pf->stream));
    return DPOMP_OK;
}

int dpomp_pf_get_last_ancestors(dpomp_pf* pf, int32_t b, int64_t* out) {
    if (!pf || !out) return fail(DPOMP_ERR_ARG, "null argument");
    if (b < 1 || b > pf->n_batch) return fail(DPOMP_ERR_ARG, "filter index out of range");
    if (!pf->record_anc || !pf->anc) return fail(DPOMP_ERR_STATE, "ancestor recording is off");
    CK(cudaSetDevice(pf->device));
    std::vector<int32_t> tmp((size_t)pf->n);
    CK(cudaMemcpyAsync(tmp.data(), pf->anc + (size_t)(b - 1) * pf->n_pad, (size_t)pf->n * sizeof(int32_t), cudaMemcpyDeviceToHost, pf->stream));
    CK(cudaStreamSynchronize(pf->stream));
    for (long long p = 0; p < pf->n; ++p) out[p] = (int64_t)tmp[(size_t)p] + 1;
    return DPOMP_OK;
}

int dpomp_pf_overflow_count(dpomp_pf* pf, int64_t* out) {
    if (!pf || !out) return fail(DPOMP_ERR_ARG, "null argument");
    CK(cudaSetDevice(pf->device));
    unsigned long long v = 0;
    CK(cudaMemcpyAsync(&v, pf->counters + 1, sizeof(v), cudaMemcpyDeviceToHost, pf->stream));
    CK(cudaStreamSynchronize(pf->stream));
    *out = (int64_t)v;
    return DPOMP_OK;
}
int dpomp_pf_last_event_count(dpomp_pf* pf, int64_t* out) {
    if (!pf || !out) return fail(DPOMP_ERR_ARG, "null argument");
    *out = pf->last_events;
    return DPOMP_OK;
}
int dpomp_pf_last_timing(dpomp_pf* pf, float* out_ms, int32_t* out_launches) {
    if (!pf) return fail(DPOMP_ERR_ARG, "null handle");
    if (out_ms) *out_ms = pf->last_ms;
    if (out_launches) *out_launches = pf->last_launches;
    return DPOMP_OK;
}

int dpomp_pf_set_kernel_timing(dpomp_pf* pf, int32_t on) {
    if (!pf) return fail(DPOMP_ERR_ARG, "null handle");
    pf->kernel_timing = on != 0;
    return DPOMP_OK;
}
int dpomp_pf_last_kernel_timing(dpomp_pf* pf, float* out_ms2, int32_t* out_launches2) {
    if (!pf || !out_ms2 || !out_launches2) return fail(DPOMP_ERR_ARG, "null argument");
    out_ms2[0] = pf->kernel_ms[0]; out_ms2[1] = pf->kernel_ms[1];
    out_launches2[0] = pf->kernel_launches[0]; out_launches2[1] = pf->kernel_launches[1];
    return DPOMP_OK;
}

int dpomp_pf_export_filters(dpomp_pf* pf, const int64_t* slots, int32_t n, void* device_dst) {
    if (!pf || !slots || !device_dst) return fail(DPOMP_ERR_ARG, "null argument");
    if (n < 1 || n > pf->n_batch) return fail(DPOMP_ERR_ARG, "n out of range");
    CK(cudaSetDevice(pf->device));
    int rc = upload_slots(pf, slots, nullptr, n, pf->n_batch, 0);
    if (rc) return rc;
    CK(launch_pack_filters((int32_t*)device_dst, pf->pop[pf->cur], pf->slots_dev, n, (long long)pf->n_comp * pf->n_pad, 0, pf->stream));
    CK(cudaStreamSynchronize(pf->stream));
    return DPOMP_OK;
}
int dpomp_pf_import_filters(dpomp_pf* pf, const int64_t* slots, int32_t n, const void* device_src) {
    if (!pf || !slots || !device_src) return fail(DPOMP_ERR_ARG, "null argument");
    if (n < 1 || n > pf->n_batch) return fail(DPOMP_ERR_ARG, "n out of range");
    CK(cudaSetDevice(pf->device));
    int rc = upload_slots(pf, slots, nullptr, n, pf->n_batch, 0);
    if (rc) return rc;
    CK(launch_pack_filters((int32_t*)device_src, pf->pop[pf->cur], pf->slots_dev, n, (long long)pf->n_comp * pf->n_pad, 1, pf->stream));
    CK(cudaStreamSynchronize(pf->stream));
    pf->initialised = true;
    return DPOMP_OK;
}

int dpomp_resample_indices(int32_t rs_type, int32_t on_cumulative, const double* w, int64_t n, const double* u, int64_t n_u,
                           int64_t n_out, int64_t* out_idx, int32_t device) {
    if (!w || !u || !out_idx) return fail(DPOMP_ERR_ARG, "null argument");
    if (rs_type < 1 || rs_type > 3) return fail(DPOMP_ERR_ARG, "rs_type must be 1, 2 or 3");
    if (n < 1 || n_out < 1) return fail(DPOMP_ERR_ARG, "empty input");
    if (rs_type != DPOMP_RS_MULTINOMIAL && n_out != n) return fail(DPOMP_ERR_ARG, "systematic/stratified produce n offspring");
    const int64_t need_u = rs_type == DPOMP_RS_SYSTEMATIC ? 1 : n_out;
    if (n_u < need_u) return fail(DPOMP_ERR_ARG, "not enough uniforms");
    int ndev = 0;
    cudaError_t e = cudaGetDeviceCount(&ndev);
    if (e != cudaSuccess || ndev < 1) return fail(DPOMP_ERR_CUDA, std::string("no CUDA device: ") + cudaGetErrorString(e));
    if (device >= 0) CK(cudaSetDevice(device));
    std::vector<double> cw(w, w + n);
    if (!on_cumulative)  // cumsum / cumsum! (src/hmm_resample.jl:5,45,67): sequential f64, bit-exact by construction
        for (int64_t i = 1; i < n; ++i) cw[(size_t)i] = cw[(size_t)i - 1] + cw[(size_t)i];
    // persistent per-device workspace (grown on demand): the outer layers call this once per resampling step
    struct HookWs {
        double* cw = nullptr; double* u = nullptr; int64_t* out = nullptr;
        size_t cap_cw = 0, cap_u = 0, cap_out = 0;
        cudaStream_t stream = nullptr;
    };
    static thread_local HookWs ws_all[64];
    int dev = device;
    if (dev < 0) CK(cudaGetDevice(&dev));
    if (dev >= 64) return fail(DPOMP_ERR_ARG, "device index out of range");
    HookWs& ws = ws_all[dev];
    if (!ws.stream) CK(cudaStreamCreateWithFlags(&ws.stream, cudaStreamNonBlocking));
    auto grow = [](void** ptr, size_t* cap, size_t need, size_t elem) -> cudaError_t {
        if (need <= *cap) return cudaSuccess;
        if (*ptr) cudaFree(*ptr);
        *ptr = nullptr; *cap = 0;
        const size_t want = need + need / 2 + 1024;
        cudaError_t e2 = cudaMalloc(ptr, want * elem);
        if (e2 == cudaSuccess) *cap = want;
        return e2;
    };
    CK(grow((void**)&ws.cw, &ws.cap_cw, (size_t)n, sizeof(double)));
    CK(grow((void**)&ws.u, &ws.cap_u, (size_t)need_u, sizeof(double)));
    CK(grow((void**)&ws.out, &ws.cap_out, (size_t)n_out, sizeof(int64_t)));
    CK(cudaMemcpyAsync(ws.cw, cw.data(), (size_t)n * sizeof(double), cudaMemcpyHostToDevice, ws.stream));
    CK(cudaMemcpyAsync(ws.u, u, (size_t)need_u * sizeof(double), cudaMemcpyHostToDevice, ws.stream));
    CK(launch_search_hook(rs_type, ws.cw, n, ws.u, n_out, ws.out, ws.stream));
    CK(cudaMemcpyAsync(out_idx, ws.out, (size_t)n_out * sizeof(int64_t), cudaMemcpyDeviceToHost, ws.stream));
    CK(cudaStreamSynchronize(ws.stream));
    return DPOMP_OK;
}

}  // extern "C"
