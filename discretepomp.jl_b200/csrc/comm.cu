// comm.cu -- the multi-GPU exchange steps of the path behind the C ABI (include/dpomp.h, "multi-GPU"): one process per
// GPU, NCCL over NVLink / NVSwitch, every collective enqueued on the stream of the handle whose data it moves, so that a
// filter step + all-gather or a pack + all-to-all + unpack is ONE stream-ordered sequence with a single synchronisation.
//
// The reference is single-process (SURVEY.md F2); these entry points replace what a sharded Julia host would otherwise
// have to do itself around run_pibis / run_mbp_ibis (src/hmm_ibis.jl:53-62 weights, :71-79 and :194-201 resampling copies).
//
// NCCL is loaded at run time (dlopen of libnccl.so.2: in a process that imported torch this resolves to the copy torch
// already loaded), so libdpomp.so has no link-time dependency on it and single-GPU users never touch it.
#include <dlfcn.h>
#include <nccl.h>  // types and enums only
#include <string.h>

#include <string>
#include <vector>

#include "dpomp_internal.cuh"

using namespace dpomp;

namespace {

struct NcclApi {
    void* lib = nullptr;
    ncclResult_t (*GetUniqueId)(ncclUniqueId*) = nullptr;
    ncclResult_t (*CommInitRank)(ncclComm_t*, int, ncclUniqueId, int) = nullptr;
    ncclResult_t (*CommDestroy)(ncclComm_t) = nullptr;
    ncclResult_t (*AllGather)(const void*, void*, size_t, ncclDataType_t, ncclComm_t, cudaStream_t) = nullptr;
    ncclResult_t (*AllReduce)(const void*, void*, size_t, ncclDataType_t, ncclRedOp_t, ncclComm_t, cudaStream_t) = nullptr;
    ncclResult_t (*Send)(const void*, size_t, ncclDataType_t, int, ncclComm_t, cudaStream_t) = nullptr;
    ncclResult_t (*Recv)(void*, size_t, ncclDataType_t, int, ncclComm_t, cudaStream_t) = nullptr;
    ncclResult_t (*GroupStart)() = nullptr;
    ncclResult_t (*GroupEnd)() = nullptr;
    const char* (*GetErrorString)(ncclResult_t) = nullptr;
    std::string error;
};

NcclApi* nccl_api() {
    static NcclApi api;
    static bool tried = false;
    if (tried) return api.lib ? &api : nullptr;
    tried = true;
    const char* names[] = {"libnccl.so.2", "libnccl.so"};
    for (const char* nm : names) {
        api.lib = dlopen(nm, RTLD_NOW | RTLD_GLOBAL);
        if (api.lib) break;
    }
    if (!api.lib) {
        api.error = std::string("cannot load NCCL (libnccl.so.2): ") + dlerror();
        return nullptr;
    }
    bool ok = true;
#define LOAD(field, sym)                                              \
    do {                                                              \
        *(void**)(&api.field) = dlsym(api.lib, sym);                  \
        if (!api.field) { ok = false; api.error = std::string("NCCL symbol missing: ") + sym; } \
    } while (0)
    LOAD(GetUniqueId, "ncclGetUniqueId");
    LOAD(CommInitRank, "ncclCommInitRank");
    LOAD(CommDestroy, "ncclCommDestroy");
    LOAD(AllGather, "ncclAllGather");
    LOAD(AllReduce, "ncclAllReduce");
    LOAD(Send, "ncclSend");
    LOAD(Recv, "ncclRecv");
    LOAD(GroupStart, "ncclGroupStart");
    LOAD(GroupEnd, "ncclGroupEnd");
    LOAD(GetErrorString, "ncclGetErrorString");
#undef LOAD
    if (!ok) {
        dlclose(api.lib);
        api.lib = nullptr;
        return nullptr;
    }
    return &api;
}

}  // namespace

struct dpomp_comm {
    int rank = 0, world = 1, device = 0;
    ncclComm_t nccl = nullptr;
    cudaStream_t stream = nullptr;  // for collectives that belong to no handle (dpomp_comm_allgather_f64, barrier)
    // staging, grown on demand
    double *d_send = nullptr, *d_recv = nullptr, *h_send = nullptr, *h_recv = nullptr;
    size_t cap_f64 = 0;  // doubles per rank block
    int64_t *h_slots = nullptr, *d_slots = nullptr;
    size_t cap_slots = 0;
    unsigned char *d_pack_send = nullptr, *d_pack_recv = nullptr;
    size_t cap_pack_send = 0, cap_pack_recv = 0;
    int *d_int = nullptr, *h_int = nullptr;
    size_t cap_int = 0;
};

#define CCK(expr)                                                                                              \
    do {                                                                                                       \
        cudaError_t _e = (expr);                                                                               \
        if (_e != cudaSuccess) return dpomp_set_error(DPOMP_ERR_CUDA, std::string(#expr) + ": " + cudaGetErrorString(_e)); \
    } while (0)
#define NCK(expr)                                                                                              \
    do {                                                                                                       \
        ncclResult_t _r = (expr);                                                                              \
        if (_r != ncclSuccess)                                                                                 \
            return dpomp_set_error(DPOMP_ERR_COMM, std::string(#expr) + ": " + nccl_api()->GetErrorString(_r)); \
    } while (0)

namespace {

void bounds(int64_t n, int world, int rank, int64_t* lo, int64_t* hi) {
    const int64_t base = n / world, extra = n % world;
    *lo = rank * base + (rank < extra ? rank : extra);
    *hi = *lo + base + (rank < extra ? 1 : 0);
}
int owner_of(int64_t n, int world, int64_t idx) {
    const int64_t base = n / world, extra = n % world, cut = extra * (base + 1);
    return (int)(idx < cut ? idx / (base + 1) : extra + (idx - cut) / (base > 0 ? base : 1));
}
int64_t max_block(int64_t n, int world) { return n / world + (n % world ? 1 : 0); }

int grow_f64(dpomp_comm* c, size_t per_rank) {
    if (per_rank <= c->cap_f64) return DPOMP_OK;
    cudaFree(c->d_send); cudaFree(c->d_recv); cudaFreeHost(c->h_send); cudaFreeHost(c->h_recv);
    c->d_send = c->d_recv = c->h_send = c->h_recv = nullptr;
    c->cap_f64 = 0;
    const size_t want = per_rank + per_rank / 2 + 64;
    CCK(cudaMalloc((void**)&c->d_send, want * sizeof(double)));
    CCK(cudaMalloc((void**)&c->d_recv, want * c->world * sizeof(double)));
    CCK(cudaMallocHost((void**)&c->h_send, want * sizeof(double)));
    CCK(cudaMallocHost((void**)&c->h_recv, want * c->world * sizeof(double)));
    c->cap_f64 = want;
    return DPOMP_OK;
}
int grow_slots(dpomp_comm* c, size_t n) {
    if (n <= c->cap_slots) return DPOMP_OK;
    cudaFree(c->d_slots); cudaFreeHost(c->h_slots);
    c->d_slots = c->h_slots = nullptr;
    c->cap_slots = 0;
    const size_t want = n + n / 2 + 64;
    CCK(cudaMalloc((void**)&c->d_slots, want * sizeof(int64_t)));
    CCK(cudaMallocHost((void**)&c->h_slots, want * sizeof(int64_t)));
    c->cap_slots = want;
    return DPOMP_OK;
}
int grow_bytes(unsigned char** p, size_t* cap, size_t need) {
    if (need <= *cap) return DPOMP_OK;
    cudaFree(*p);
    *p = nullptr;
    *cap = 0;
    const size_t want = need + need / 4 + 4096;
    CCK(cudaMalloc((void**)p, want));
    *cap = want;
    return DPOMP_OK;
}
int grow_int(dpomp_comm* c, size_t n) {
    if (n <= c->cap_int) return DPOMP_OK;
    cudaFree(c->d_int); cudaFreeHost(c->h_int);
    c->d_int = c->h_int = nullptr;
    c->cap_int = 0;
    const size_t want = n + n / 2 + 64;
    CCK(cudaMalloc((void**)&c->d_int, want * sizeof(int)));
    CCK(cudaMallocHost((void**)&c->h_int, want * sizeof(int)));
    c->cap_int = want;
    return DPOMP_OK;
}

// the rows of an all-gathered [world][maxn][width] block -> contiguous [n_total][width]
void compact(const double* gathered, int64_t n_total, int world, int64_t maxn, int width, double* out) {
    for (int r = 0; r < world; ++r) {
        int64_t lo, hi;
        bounds(n_total, world, r, &lo, &hi);
        memcpy(out + lo * width, gathered + (size_t)r * maxn * width, (size_t)(hi - lo) * width * sizeof(double));
    }
}

}  // namespace

namespace dpomp {

// Who sends what after the outer resample new[p] <- old[nidx[p]] (nidx 1-based global, contiguous partition).
void migration_plan(const int64_t* nidx, int64_t n_total, int world, int rank, MigrationPlan& pl) {
    int64_t lo, hi;
    bounds(n_total, world, rank, &lo, &hi);
    const int64_t n_loc = hi - lo;
    pl.local_src.resize((size_t)n_loc);
    pl.send_counts.assign((size_t)world, 0);
    pl.recv_counts.assign((size_t)world, 0);
    std::vector<std::vector<int64_t>> send((size_t)world), recv((size_t)world);
    for (int64_t p = 0; p < n_total; ++p) {
        const int64_t src = nidx[p] - 1;
        const int so = owner_of(n_total, world, src), dn = owner_of(n_total, world, p);
        if (dn == rank) {
            if (so == rank) pl.local_src[(size_t)(p - lo)] = src - lo + 1;
            else {
                pl.local_src[(size_t)(p - lo)] = p - lo + 1;  // placeholder: overwritten by the received block
                recv[(size_t)so].push_back(p - lo + 1);
            }
        } else if (so == rank) {
            send[(size_t)dn].push_back(src - lo + 1);
        }
    }
    pl.send_slots.clear();
    pl.recv_slots.clear();
    for (int r = 0; r < world; ++r) {  // ordered by peer rank, then by destination index (both sides enumerate p ascending)
        pl.send_counts[(size_t)r] = (int)send[(size_t)r].size();
        pl.recv_counts[(size_t)r] = (int)recv[(size_t)r].size();
        pl.send_slots.insert(pl.send_slots.end(), send[(size_t)r].begin(), send[(size_t)r].end());
        pl.recv_slots.insert(pl.recv_slots.end(), recv[(size_t)r].begin(), recv[(size_t)r].end());
    }
}

// all-to-all-v of raw bytes between device buffers (grouped ncclSend / ncclRecv), enqueued on `stream`
int comm_alltoallv_bytes(dpomp_comm* c, const void* send, const size_t* send_bytes, void* recv, const size_t* recv_bytes,
                         cudaStream_t stream) {
    NcclApi* api = nccl_api();
    size_t so = 0, ro = 0;
    if (c->world == 1) return DPOMP_OK;
    NCK(api->GroupStart());
    for (int r = 0; r < c->world; ++r) {
        if (r != c->rank) {
            if (send_bytes[r]) NCK(api->Send((const char*)send + so, send_bytes[r], ncclUint8, r, c->nccl, stream));
            if (recv_bytes[r]) NCK(api->Recv((char*)recv + ro, recv_bytes[r], ncclUint8, r, c->nccl, stream));
        }
        so += send_bytes[r];
        ro += recv_bytes[r];
    }
    NCK(api->GroupEnd());
    return DPOMP_OK;
}

// rows of an all-gathered [world][maxn][width] block -> contiguous [n_total][width] (device)
__global__ void compact_rows_kernel(const double* gathered, double* out, long long n_total, int world, long long maxn, int width) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n_total * width) return;
    const long long row = i / width;
    const int col = (int)(i % width);
    const long long base = n_total / world, extra = n_total % world, cut = extra * (base + 1);
    const long long r = row < cut ? row / (base + 1) : extra + (row - cut) / (base > 0 ? base : 1);
    const long long lo = r * base + (r < extra ? r : extra);
    out[i] = gathered[((size_t)r * maxn + (row - lo)) * width + col];
}

// all-gather of per-item rows between DEVICE buffers on `stream`: send = this rank's block [n_loc][width], out = all
// [n_total][width] rows in global order on every rank (ncclAllGather of the padded blocks + a compaction kernel)
int comm_allgather_rows_device(dpomp_comm* c, const double* send, long long n_total, int width, double* out, cudaStream_t stream) {
    int64_t lo, hi;
    bounds(n_total, c->world, c->rank, &lo, &hi);
    const size_t nloc = (size_t)(hi - lo) * width;
    if (c->world == 1) {
        if (nloc) CCK(cudaMemcpyAsync(out, send, nloc * sizeof(double), cudaMemcpyDeviceToDevice, stream));
        return DPOMP_OK;
    }
    const int64_t maxn = max_block(n_total, c->world);
    const size_t per = (size_t)maxn * width;
    int rc = grow_f64(c, per);
    if (rc) return rc;
    if (nloc) CCK(cudaMemcpyAsync(c->d_send, send, nloc * sizeof(double), cudaMemcpyDeviceToDevice, stream));
    NCK(nccl_api()->AllGather(c->d_send, c->d_recv, per, ncclFloat64, c->nccl, stream));
    const long long total = n_total * width;
    compact_rows_kernel<<<(unsigned)((total + 255) / 256), 256, 0, stream>>>(c->d_recv, out, n_total, c->world, maxn, width);
    CCK(cudaGetLastError());
    return DPOMP_OK;
}
void comm_bounds(const dpomp_comm* c, long long n_total, long long* lo, long long* hi) {
    int64_t l, h;
    bounds(n_total, c->world, c->rank, &l, &h);
    *lo = l; *hi = h;
}

int comm_rank(const dpomp_comm* c) { return c->rank; }
int comm_world(const dpomp_comm* c) { return c->world; }
int comm_scratch(dpomp_comm* c, size_t slots, size_t send_bytes, size_t recv_bytes, size_t ints, CommScratch* out) {
    int rc = grow_slots(c, slots);
    if (!rc) rc = grow_bytes(&c->d_pack_send, &c->cap_pack_send, send_bytes);
    if (!rc) rc = grow_bytes(&c->d_pack_recv, &c->cap_pack_recv, recv_bytes);
    if (!rc) rc = grow_int(c, ints);
    if (rc) return rc;
    *out = CommScratch{c->h_slots, c->d_slots, c->d_pack_send, c->d_pack_recv, c->h_int, c->d_int};
    return DPOMP_OK;
}

}  // namespace dpomp

extern "C" {

int dpomp_comm_unique_id(void* out_id, int32_t nbytes) {
    if (!out_id || nbytes < (int32_t)sizeof(ncclUniqueId)) return dpomp_set_error(DPOMP_ERR_ARG, "unique id buffer must hold DPOMP_UNIQUE_ID_BYTES");
    NcclApi* api = nccl_api();
    if (!api) return dpomp_set_error(DPOMP_ERR_COMM, "NCCL unavailable");
    ncclUniqueId id;
    NCK(api->GetUniqueId(&id));
    memset(out_id, 0, (size_t)nbytes);
    memcpy(out_id, &id, sizeof(id));
    return DPOMP_OK;
}

int dpomp_comm_create(const void* id, int32_t nbytes, int32_t rank, int32_t world, int32_t device, dpomp_comm** out) {
    if (!out) return dpomp_set_error(DPOMP_ERR_ARG, "null argument");
    if (world < 1 || rank < 0 || rank >= world) return dpomp_set_error(DPOMP_ERR_ARG, "rank / world out of range");
    int ndev = 0;
    cudaError_t e = cudaGetDeviceCount(&ndev);
    if (e != cudaSuccess || ndev < 1)
        return dpomp_set_error(DPOMP_ERR_CUDA, std::string("no CUDA device (there is no CPU fallback): ") + cudaGetErrorString(e));
    if (device < 0) CCK(cudaGetDevice(&device));
    if (device >= ndev) return dpomp_set_error(DPOMP_ERR_ARG, "device index out of range");
    CCK(cudaSetDevice(device));
    dpomp_comm* c = new (std::nothrow) dpomp_comm();
    if (!c) return dpomp_set_error(DPOMP_ERR_ARG, "out of host memory");
    c->rank = rank; c->world = world; c->device = device;
    if (cudaStreamCreateWithFlags(&c->stream, cudaStreamNonBlocking) != cudaSuccess) {
        delete c;
        return dpomp_set_error(DPOMP_ERR_CUDA, "cudaStreamCreate failed");
    }
    if (world > 1) {
        NcclApi* api = nccl_api();
        if (!api || !id || nbytes < (int32_t)sizeof(ncclUniqueId)) {
            cudaStreamDestroy(c->stream);
            delete c;
            return dpomp_set_error(api ? DPOMP_ERR_ARG : DPOMP_ERR_COMM, api ? "unique id missing" : "NCCL unavailable");
        }
        ncclUniqueId uid;
        memcpy(&uid, id, sizeof(uid));
        ncclResult_t r = api->CommInitRank(&c->nccl, world, uid, rank);
        if (r != ncclSuccess) {
            cudaStreamDestroy(c->stream);
            delete c;
            return dpomp_set_error(DPOMP_ERR_COMM, std::string("ncclCommInitRank: ") + api->GetErrorString(r));
        }
    }
    *out = c;
    return DPOMP_OK;
}

int dpomp_comm_destroy(dpomp_comm* c) {
    if (!c) return DPOMP_OK;
    cudaSetDevice(c->device);
    if (c->nccl) nccl_api()->CommDestroy(c->nccl);
    cudaFree(c->d_send); cudaFree(c->d_recv); cudaFreeHost(c->h_send); cudaFreeHost(c->h_recv);
    cudaFree(c->d_slots); cudaFreeHost(c->h_slots); cudaFree(c->d_pack_send); cudaFree(c->d_pack_recv);
    cudaFree(c->d_int); cudaFreeHost(c->h_int);
    if (c->stream) cudaStreamDestroy(c->stream);
    delete c;
    return DPOMP_OK;
}

int dpomp_comm_info(const dpomp_comm* c, int32_t* out_rank, int32_t* out_world) {
    if (!c) return dpomp_set_error(DPOMP_ERR_ARG, "null handle");
    if (out_rank) *out_rank = c->rank;
    if (out_world) *out_world = c->world;
    return DPOMP_OK;
}

int dpomp_partition_bounds(int64_t n, int32_t world, int32_t rank, int64_t* out_lo, int64_t* out_hi) {
    if (!out_lo || !out_hi || world < 1 || rank < 0 || rank >= world || n < 0) return dpomp_set_error(DPOMP_ERR_ARG, "bad argument");
    bounds(n, world, rank, out_lo, out_hi);
    return DPOMP_OK;
}

int dpomp_comm_barrier(dpomp_comm* c) {
    if (!c) return dpomp_set_error(DPOMP_ERR_ARG, "null handle");
    if (c->world == 1) return DPOMP_OK;
    CCK(cudaSetDevice(c->device));
    int rc = grow_f64(c, 1);
    if (rc) return rc;
    NCK(nccl_api()->AllReduce(c->d_send, c->d_recv, 1, ncclFloat64, ncclSum, c->nccl, c->stream));
    CCK(cudaStreamSynchronize(c->stream));
    return DPOMP_OK;
}

int dpomp_comm_allgather_f64(dpomp_comm* c, const double* local, int64_t n_total, int32_t width, double* out) {
    if (!c || !out || width < 1 || n_total < 0) return dpomp_set_error(DPOMP_ERR_ARG, "bad argument");
    int64_t lo, hi;
    bounds(n_total, c->world, c->rank, &lo, &hi);
    const size_t nloc = (size_t)(hi - lo) * width;
    if (nloc && !local) return dpomp_set_error(DPOMP_ERR_ARG, "null argument");
    if (c->world == 1) {
        if (nloc) memcpy(out, local, nloc * sizeof(double));
        return DPOMP_OK;
    }
    CCK(cudaSetDevice(c->device));
    const int64_t maxn = max_block(n_total, c->world);
    const size_t per = (size_t)maxn * width;
    int rc = grow_f64(c, per);
    if (rc) return rc;
    if (nloc) memcpy(c->h_send, local, nloc * sizeof(double));
    CCK(cudaMemcpyAsync(c->d_send, c->h_send, per * sizeof(double), cudaMemcpyHostToDevice, c->stream));
    NCK(nccl_api()->AllGather(c->d_send, c->d_recv, per, ncclFloat64, c->nccl, c->stream));
    CCK(cudaMemcpyAsync(c->h_recv, c->d_recv, per * c->world * sizeof(double), cudaMemcpyDeviceToHost, c->stream));
    CCK(cudaStreamSynchronize(c->stream));
    compact(c->h_recv, n_total, c->world, maxn, width, out);
    return DPOMP_OK;
}

// partial_log_likelihood! of this rank's block of filters + all-gather of the increments of ALL ranks (run_pibis
// src/hmm_ibis.jl:53-56 followed by the theta-weight exchange): one stream-ordered sequence on the filter's stream
// (kernels -> ncclAllGather -> one device-to-host copy), one synchronisation.
int dpomp_pf_partial_allgather(dpomp_pf* pf, dpomp_comm* c, const double* theta_local, int32_t nb, int32_t ymin, int32_t ymax,
                               int64_t n_total, double* out_all) {
    if (!pf || !c || !out_all) return dpomp_set_error(DPOMP_ERR_ARG, "null argument");
    int64_t lo, hi;
    bounds(n_total, c->world, c->rank, &lo, &hi);
    if (nb != (int32_t)(hi - lo)) return dpomp_set_error(DPOMP_ERR_ARG, "n_batch_used must equal this rank's block of n_total");
    if (pf->device != c->device) return dpomp_set_error(DPOMP_ERR_ARG, "filter and communicator live on different devices");
    if (c->world == 1) return nb ? dpomp_pf_partial(pf, theta_local, nb, ymin, ymax, out_all) : DPOMP_OK;
    CCK(cudaSetDevice(c->device));
    const int64_t maxn = max_block(n_total, c->world);
    int rc = grow_f64(c, (size_t)maxn);
    if (rc) return rc;
    cudaStream_t st = pf->stream;
    if (nb) {
        rc = dpomp_run_partial_enqueue(pf, theta_local, false, nb, ymin, ymax, nullptr, 2);
        if (rc) return rc;
        CCK(cudaMemcpyAsync(c->d_send, pf->ll_acc, (size_t)nb * sizeof(double), cudaMemcpyDeviceToDevice, st));
    }
    NCK(nccl_api()->AllGather(c->d_send, c->d_recv, (size_t)maxn, ncclFloat64, c->nccl, st));
    CCK(cudaMemcpyAsync(c->h_recv, c->d_recv, (size_t)maxn * c->world * sizeof(double), cudaMemcpyDeviceToHost, st));
    if (nb) {
        rc = dpomp_run_partial_finish(pf, nullptr, nb, 2);
        if (rc) return rc;
    } else {
        CCK(cudaStreamSynchronize(st));
    }
    compact(c->h_recv, n_total, c->world, maxn, 1, out_all);
    return DPOMP_OK;
}

// pop2[p] .= pop[nidx[p]] (src/hmm_ibis.jl:74) across ranks: nidx is the GLOBAL 1-based ancestor vector of all n_total
// theta-particles (identical on every rank).  Filters whose ancestor lives on another rank arrive over NVLink (grouped
// ncclSend / ncclRecv of the packed int32 populations); the local ones are gathered on the device.
int dpomp_pf_resample_migrate(dpomp_pf* pf, dpomp_comm* c, const int64_t* nidx, int64_t n_total) {
    if (!pf || !c || !nidx) return dpomp_set_error(DPOMP_ERR_ARG, "null argument");
    int64_t lo, hi;
    bounds(n_total, c->world, c->rank, &lo, &hi);
    const int n_loc = (int)(hi - lo);
    if (n_loc > pf->n_batch) return dpomp_set_error(DPOMP_ERR_ARG, "this rank's block exceeds the handle's n_batch");
    for (int64_t p = 0; p < n_total; ++p)
        if (nidx[p] < 1 || nidx[p] > n_total) return dpomp_set_error(DPOMP_ERR_ARG, "ancestor index out of range");
    if (c->world == 1) return dpomp_pf_permute(pf, nidx, (int32_t)n_total);
    if (pf->device != c->device) return dpomp_set_error(DPOMP_ERR_ARG, "filter and communicator live on different devices");
    CCK(cudaSetDevice(c->device));
    MigrationPlan pl;
    migration_plan(nidx, n_total, c->world, c->rank, pl);
    const size_t n_send = pl.send_slots.size(), n_recv = pl.recv_slots.size();
    const long long stride = (long long)pf->n_comp * pf->n_pad;  // int32 words of one filter
    const size_t fbytes = (size_t)stride * sizeof(int32_t);
    int rc = grow_slots(c, n_send + (size_t)n_loc + n_recv);
    if (!rc) rc = grow_bytes(&c->d_pack_send, &c->cap_pack_send, n_send * fbytes);
    if (!rc) rc = grow_bytes(&c->d_pack_recv, &c->cap_pack_recv, n_recv * fbytes);
    if (rc) return rc;
    cudaStream_t st = pf->stream;
    int64_t* hs = c->h_slots;
    if (n_send) memcpy(hs, pl.send_slots.data(), n_send * sizeof(int64_t));
    if (n_loc) memcpy(hs + n_send, pl.local_src.data(), (size_t)n_loc * sizeof(int64_t));
    if (n_recv) memcpy(hs + n_send + n_loc, pl.recv_slots.data(), n_recv * sizeof(int64_t));
    CCK(cudaMemcpyAsync(c->d_slots, hs, (n_send + n_loc + n_recv) * sizeof(int64_t), cudaMemcpyHostToDevice, st));
    if (n_send) CCK(launch_pack_filters((int32_t*)c->d_pack_send, pf->pop[pf->cur], c->d_slots, (int)n_send, stride, 0, st));
    std::vector<size_t> sb((size_t)c->world), rb((size_t)c->world);
    for (int r = 0; r < c->world; ++r) {
        sb[(size_t)r] = (size_t)pl.send_counts[(size_t)r] * fbytes;
        rb[(size_t)r] = (size_t)pl.recv_counts[(size_t)r] * fbytes;
    }
    rc = comm_alltoallv_bytes(c, c->d_pack_send, sb.data(), c->d_pack_recv, rb.data(), st);
    if (rc) return rc;
    if (n_loc) {
        CCK(launch_gather_filters(pf->pop[pf->cur ^ 1], pf->pop[pf->cur], nullptr, c->d_slots + n_send, n_loc, stride, st));
        if (n_loc < pf->n_batch)
            CCK(cudaMemcpyAsync(pf->pop[pf->cur ^ 1] + (size_t)n_loc * stride, pf->pop[pf->cur] + (size_t)n_loc * stride,
                                (size_t)(pf->n_batch - n_loc) * fbytes, cudaMemcpyDeviceToDevice, st));
        pf->cur ^= 1;
    }
    if (n_recv) CCK(launch_pack_filters((int32_t*)c->d_pack_recv, pf->pop[pf->cur], c->d_slots + n_send + n_loc, (int)n_recv, stride, 1, st));
    CCK(cudaStreamSynchronize(st));
    pf->initialised = true;
    pf->hist_upto = 0;  // the filters have new lineages: their history is gone (include/dpomp.h)
    pf->hist_weights_t = 0;
    return DPOMP_OK;
}

}  // extern "C"
