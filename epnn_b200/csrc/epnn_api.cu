// C-ABI of libepnn_b200.so: context, weight upload, workspace management and the launch sequence.
// See include/epnn_b200.h for the contract of every entry point and the reference code it replaces.
#include <dlfcn.h>
#include <math.h>
#include <stdarg.h>
#include <stdlib.h>

#include <algorithm>
#include <mutex>
#include <new>
#include <string>
#include <vector>

#include "epnn_elst.cuh"
#include "epnn_internal.cuh"
#include "epnn_pack.h"
#include "epnn_plan.h"

#define EPNN_VERSION_STR "epnn_b200 0.1.0 sm_100a"

// ------------------------------------------------------------------------------------------------
struct DevBuf {
    void* p = nullptr;
    size_t cap = 0;
};

// ------------------------------------------------------------------------------------------------
// NCCL, bound at run time (dlopen of libnccl.so.2: the copy the process already holds -- e.g. torch's -- or the system one).
// Only four entry points are used; all exchanges are in-place all-gathers of equal slices on the ctx stream.
typedef struct ncclComm* ncclComm_t;
struct NcclApi {
    void* handle = nullptr;
    int (*GetUniqueId)(void*) = nullptr;
    int (*CommInitRank)(ncclComm_t*, int, /* ncclUniqueId by value: 128 bytes */ struct NcclId, int) = nullptr;
    int (*AllGather)(const void*, void*, size_t, int, ncclComm_t, cudaStream_t) = nullptr;
    int (*CommDestroy)(ncclComm_t) = nullptr;
    const char* (*GetErrorString)(int) = nullptr;
};
struct NcclId { char bytes[128]; };
static NcclApi g_nccl;
static std::mutex g_nccl_mu;
static const char* load_nccl() {
    std::lock_guard<std::mutex> lk(g_nccl_mu);
    if (g_nccl.handle) return nullptr;
    void* h = dlopen("libnccl.so.2", RTLD_NOW | RTLD_GLOBAL);
    if (!h) h = dlopen("libnccl.so", RTLD_NOW | RTLD_GLOBAL);
    if (!h) return "libnccl.so.2 not found (needed for epnn_shard_init with world > 1)";
    NcclApi a;
    a.GetUniqueId = (int (*)(void*))dlsym(h, "ncclGetUniqueId");
    a.CommInitRank = (int (*)(ncclComm_t*, int, NcclId, int))dlsym(h, "ncclCommInitRank");
    a.AllGather = (int (*)(const void*, void*, size_t, int, ncclComm_t, cudaStream_t))dlsym(h, "ncclAllGather");
    a.CommDestroy = (int (*)(ncclComm_t))dlsym(h, "ncclCommDestroy");
    a.GetErrorString = (const char* (*)(int))dlsym(h, "ncclGetErrorString");
    if (!a.GetUniqueId || !a.CommInitRank || !a.AllGather || !a.CommDestroy) { dlclose(h); return "libnccl.so.2 lacks a required symbol"; }
    a.handle = h;
    g_nccl = a;
    return nullptr;
}

struct epnn_ctx {
    int device = 0, T = 0, n_x = 0, n_species = 0, sm_count = 0;
    cudaStream_t stream = nullptr;           // the stream every kernel / copy of the ctx is enqueued on (own_stream, or the caller's: epnn_set_stream)
    cudaStream_t own_stream = nullptr;
    // multi-chunk calls keep two chunks in flight: even chunks on `stream`, odd chunks on `stream2`, each with its own set of
    // workspaces (bufs[slot * B_COUNT + ...]) and flags -- the list building of one chunk runs beside the pair kernels of the other
    cudaStream_t stream2 = nullptr;
    cudaEvent_t ev_fork = nullptr, ev_join = nullptr;
    int chunk_streams = 1;       // option "chunk_streams": 2 = two chunks in flight (+2 % throughput at 1 M molecules; default 1: one chunk at a time,
                                 // so that the per-phase CUDA-event times of epnn_stats stay additive)
    // host-buffer calls: chunk k + 1 is uploaded and chunk k - 1 downloaded while chunk k computes (two staging slots)
    cudaStream_t h2d_stream = nullptr, d2h_stream = nullptr;
    cudaEvent_t ev_h2d[2] = {nullptr, nullptr}, ev_done[2] = {nullptr, nullptr}, ev_d2h[2] = {nullptr, nullptr};
    int precision = 32, timing = 0, keep_hidden = 0;      // precision: 32, 48 (mixed), 64, 0 (auto: probe on the first call)
    int auto_choice = 0;         // precision chosen by the probe (0 = not probed yet)
    double auto_tol = 2.5e-6;    // a cheaper precision is accepted if its probe charges are within this of the FP64 kernels
    double probe_err32 = -1, probe_err48 = -1;
    KernelOptions kopt;          // options "pair_const", "pair_tensor", "gnn_far_tensor", "gnn_far_tensor_min", "gnn_far_tensor_impl" (resolve_kernels)
    int dedup_far = 1;           // option "dedup_far": collapse species-equivalent far columns (exact)
    int fused_prep = 1;          // option "fused_prep": chunks of small systems only build their lists with the two bundle kernels of epnn_bundle_prep.cu
    int atom_tensor = 1;         // option "atom_tensor": FP32 per-atom kernel on mma.sync 3xTF32 (epnn_atom_mma.cu); 0 = the FP32 SIMT warp-tile kernel
    int auto_atom_tensor = 1;    // precision 0 (auto): what the probe decided for the FP32 per-atom kernel
    std::vector<float> wf_host;  // host mirror of wf (pair_const passes a step's weights as kernel parameters)
    float* w2split = nullptr;    // [T][2][32][32]: hi / lo parts of W2^T of every message MLP (tensor-core far kernel)
    int shard_rank = 0, shard_world = 1;      // large systems of a call are split over shard_world ranks (epnn_shard_init)
    ncclComm_t comm = nullptr;
    int64_t xchg_calls = 0, xchg_bytes = 0;   // all-gathers issued / bytes received by this rank since epnn_shard_init
    int64_t chunk_atoms = 4 * 1024 * 1024;
    PackedOffsets po;
    float* wf = nullptr;         // packed weights, float
    double* wd = nullptr;        // packed weights, double
    std::vector<DevBuf> bufs;    // grow-only workspaces, indexed by enum below
    ChunkPlan plan;              // plan of the current chunk (host staging of its bundle, cell and row-block tables)
    int* d_flags = nullptr;      // [0] error bits, [1..4] totals (nnz, P, n_far, n_rg_large)
    int* h_flags = nullptr;      // pinned mirror
    int64_t hidden_atoms = 0;    // atoms covered by the retained hidden state
    int hidden_precision = 32;
    std::string err;
};

static thread_local std::string g_create_err;

enum {
    B_XYZ, B_SPECIES, B_OFF, B_Q, B_NPAD, B_ATOMSYS, B_DEG, B_DEGU, B_ROWPTR, B_USTART, B_COL, B_PID, B_PI, B_PJ, B_PD,
    B_E, B_NEAR, B_BUNDLE, B_RGL, B_FARCNT, B_FAROFF, B_FARLIST, B_FAR0CNT, B_FAR0OFF, B_FAR0LIST, B_FAR0W, B_REP, B_ATOMB0, B_BNAT, B_PERM, B_LARGESYS, B_GRID, B_CELLCNT, B_CELLSTART, B_CELLATOMS, B_DTMP, B_H, B_L2, B_S, B_U, B_V, B_DELTA, B_QD, B_SCANTMP, B_CNTL, B_RGLOFF,
    B_OUT32, B_OUT64, B_MISC, B_OFFIN, B_SPTAB, B_SPSTAMP, B_ROWBLK, B_ROWL, B_ARGS, B_DEGALL, B_ACTIVE, B_XYZ_1, B_SPECIES_1, B_Q_1, B_OUT32_1, B_OUT64_1, B_OFFIN_1, B_BPMASK, B_BPTOT, B_BPOFF,
    B_EL_OFF, B_EL_XYZ, B_EL_Q, B_EL_FRAG, B_EL_E, B_EL_MU, B_EL_PHI, B_EL_PLAN, B_EL_PART,
    B_PT_XYZ, B_PT_Q, B_PT_PTS, B_PT_PHI, B_PT_FIELD, B_PT_PLAN, B_PT_PART, B_COUNT
};

static int fail(epnn_ctx* c, int code, const char* fmt, ...) {
    char buf[512];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(buf, sizeof buf, fmt, ap);
    va_end(ap);
    if (c) c->err = buf; else g_create_err = buf;
    return code;
}

#define CU(c, call)                                                                                   \
    do {                                                                                              \
        cudaError_t _e = (call);                                                                      \
        if (_e != cudaSuccess)                                                                        \
            return fail((c), _e == cudaErrorMemoryAllocation ? EPNN_E_NOMEM : EPNN_E_CUDA, "%s failed: %s (%s:%d)", #call, \
                        cudaGetErrorString(_e), __FILE__, __LINE__);                                  \
    } while (0)

static int ensure(epnn_ctx* c, int which, size_t bytes, void** out) {
    DevBuf& b = c->bufs[which];
    if (bytes > b.cap) {
        if (b.p) { CU(c, cudaStreamSynchronize(c->stream)); CU(c, cudaStreamSynchronize(c->stream2)); CU(c, cudaFree(b.p)); b.p = nullptr; b.cap = 0; }
        size_t want = bytes + bytes / 8 + 256;
        CU(c, cudaMalloc(&b.p, want));
        b.cap = want;
    }
    *out = b.p;
    return EPNN_OK;
}

extern "C" int epnn_rbf_centers(double* mu) {
    if (!mu) return EPNN_E_INVALID;
    rbf_centers_impl(mu);
    return EPNN_OK;
}

extern "C" int epnn_rbf_basis(double* B) {
    if (!B) return EPNN_E_INVALID;
    static std::once_flag once;
    static double cached[ED * EDR];
    std::call_once(once, [] { compute_rbf_basis(cached); });
    memcpy(B, cached, sizeof(cached));
    return EPNN_OK;
}

extern "C" const char* epnn_version(void) { return EPNN_VERSION_STR; }

extern "C" const char* epnn_last_error(const epnn_ctx* ctx) { return ctx ? ctx->err.c_str() : g_create_err.c_str(); }

extern "C" int epnn_create(int device, int T, int n_x, const float* w, size_t n_floats, epnn_ctx** out) {
    if (!out) return fail(nullptr, EPNN_E_INVALID, "epnn_create: out is NULL");
    *out = nullptr;
    if (!w) return fail(nullptr, EPNN_E_INVALID, "epnn_create: packed_weights is NULL");
    if (T < 1 || T > 64) return fail(nullptr, EPNN_E_INVALID, "epnn_create: T=%d out of range", T);
    if (n_x != 9 && n_x != 10) return fail(nullptr, EPNN_E_INVALID, "epnn_create: n_x must be 9 or 10 (got %d)", n_x);
    if (n_floats != expected_floats(T, n_x))
        return fail(nullptr, EPNN_E_INVALID, "epnn_create: expected %zu packed floats for T=%d n_x=%d, got %zu",
                    expected_floats(T, n_x), T, n_x, n_floats);
    int ndev = 0;
    cudaError_t ce = cudaGetDeviceCount(&ndev);
    if (ce != cudaSuccess || ndev == 0)
        return fail(nullptr, EPNN_E_CUDA, "epnn_create: no usable CUDA device (%s); this library has no CPU fallback",
                    ce == cudaSuccess ? "device count is 0" : cudaGetErrorString(ce));
    if (device < 0 || device >= ndev) return fail(nullptr, EPNN_E_INVALID, "epnn_create: device %d not in [0,%d)", device, ndev);

    epnn_ctx* c = new (std::nothrow) epnn_ctx();
    if (!c) return fail(nullptr, EPNN_E_NOMEM, "epnn_create: out of host memory");
    c->device = device; c->T = T; c->n_x = n_x; c->n_species = n_x - 1;
    c->bufs.resize(2 * B_COUNT);
#define CUC(call)                                                                                               \
    do {                                                                                                        \
        cudaError_t _e = (call);                                                                                \
        if (_e != cudaSuccess) {                                                                                \
            int rc = fail(nullptr, EPNN_E_CUDA, "%s failed: %s", #call, cudaGetErrorString(_e));               \
            epnn_destroy(c);                                                                                    \
            return rc;                                                                                          \
        }                                                                                                       \
    } while (0)
    CUC(cudaSetDevice(device));
    CUC(cudaDeviceGetAttribute(&c->sm_count, cudaDevAttrMultiProcessorCount, device));
    CUC(cudaStreamCreateWithFlags(&c->own_stream, cudaStreamNonBlocking));
    c->stream = c->own_stream;
    CUC(cudaStreamCreateWithFlags(&c->stream2, cudaStreamNonBlocking));
    CUC(cudaEventCreateWithFlags(&c->ev_fork, cudaEventDisableTiming));
    CUC(cudaEventCreateWithFlags(&c->ev_join, cudaEventDisableTiming));
    CUC(cudaStreamCreateWithFlags(&c->h2d_stream, cudaStreamNonBlocking));
    CUC(cudaStreamCreateWithFlags(&c->d2h_stream, cudaStreamNonBlocking));
    for (int k = 0; k < 2; ++k) {
        CUC(cudaEventCreateWithFlags(&c->ev_h2d[k], cudaEventDisableTiming));
        CUC(cudaEventCreateWithFlags(&c->ev_done[k], cudaEventDisableTiming));
        CUC(cudaEventCreateWithFlags(&c->ev_d2h[k], cudaEventDisableTiming));
    }
    CUC(cudaMalloc(&c->d_flags, 16 * sizeof(int)));          // 8 per workspace slot
    CUC(cudaMallocHost(&c->h_flags, 16 * sizeof(int)));
    double mu[48];
    epnn_rbf_centers(mu);
    CUC(upload_rbf_centers(mu));
    std::vector<double> basis(ED * EDR);
    epnn_rbf_basis(basis.data());
    CUC(upload_rbf_basis(basis.data()));

    // ---- pack + fold (epnn_pack.h)
    PackedOffsets& po = c->po;
    std::vector<double> P;
    pack_all(T, n_x, c->n_species, w, basis.data(), po, P);
    {   // 3xTF32 split of W2^T for the tensor-core far kernel: hi = W with the low 13 mantissa bits cleared, lo = W - hi
        std::vector<float> ws((size_t)T * 2 * 32 * 32);
        for (int t = 0; t < T; ++t)
            for (int n = 0; n < 32; ++n)
                for (int k = 0; k < 32; ++k) {
                    const float wv = (float)P[po.msg[t].W2 + (size_t)k * 32 + n];
                    uint32_t bits; memcpy(&bits, &wv, 4); bits &= 0xFFFFE000u;
                    float hi; memcpy(&hi, &bits, 4);
                    ws[((size_t)t * 2 + 0) * 1024 + n * 32 + k] = hi;
                    ws[((size_t)t * 2 + 1) * 1024 + n * 32 + k] = wv - hi;
                }
        CUC(cudaMalloc(&c->w2split, ws.size() * sizeof(float)));
        CUC(cudaMemcpy(c->w2split, ws.data(), ws.size() * sizeof(float), cudaMemcpyHostToDevice));
    }
    std::vector<float> Pf(po.total);
    for (size_t i = 0; i < po.total; ++i) Pf[i] = (float)P[i];
    CUC(cudaMalloc(&c->wf, po.total * sizeof(float)));
    CUC(cudaMalloc(&c->wd, po.total * sizeof(double)));
    CUC(cudaMemcpy(c->wf, Pf.data(), po.total * sizeof(float), cudaMemcpyHostToDevice));
    c->wf_host = Pf;
    CUC(cudaMemcpy(c->wd, P.data(), po.total * sizeof(double), cudaMemcpyHostToDevice));
#undef CUC
    *out = c;
    return EPNN_OK;
}

extern "C" void epnn_destroy(epnn_ctx* c) {
    if (!c) return;
    cudaSetDevice(c->device);
    if (c->stream) cudaStreamSynchronize(c->stream);
    if (c->stream2) { cudaStreamSynchronize(c->stream2); cudaStreamDestroy(c->stream2); }
    if (c->ev_fork) cudaEventDestroy(c->ev_fork);
    if (c->ev_join) cudaEventDestroy(c->ev_join);
    if (c->comm) { g_nccl.CommDestroy(c->comm); c->comm = nullptr; }
    for (DevBuf& b : c->bufs) if (b.p) cudaFree(b.p);
    if (c->wf) cudaFree(c->wf);
    if (c->wd) cudaFree(c->wd);
    if (c->w2split) cudaFree(c->w2split);
    if (c->d_flags) cudaFree(c->d_flags);
    if (c->h_flags) cudaFreeHost(c->h_flags);
    for (int k = 0; k < 2; ++k) {
        if (c->ev_h2d[k]) cudaEventDestroy(c->ev_h2d[k]);
        if (c->ev_done[k]) cudaEventDestroy(c->ev_done[k]);
        if (c->ev_d2h[k]) cudaEventDestroy(c->ev_d2h[k]);
    }
    if (c->h2d_stream) cudaStreamDestroy(c->h2d_stream);
    if (c->d2h_stream) cudaStreamDestroy(c->d2h_stream);
    if (c->own_stream) cudaStreamDestroy(c->own_stream);
    delete c;
}

extern "C" int epnn_set_option(epnn_ctx* c, const char* key, double value) {
    if (!c || !key) return EPNN_E_INVALID;
    const std::string k(key);
    if (k == "precision") {
        if (value != 32 && value != 64 && value != 48 && value != 0)
            return fail(c, EPNN_E_INVALID, "precision must be 32, 48 (mixed), 64 or 0 (auto)");
        c->precision = (int)value;
        c->auto_choice = 0;
    } else if (k == "auto_tol") {
        if (!(value > 0)) return fail(c, EPNN_E_INVALID, "auto_tol must be positive");
        c->auto_tol = value; c->auto_choice = 0;
    } else if (k == "timing") c->timing = value != 0;
    else if (k == "keep_hidden") c->keep_hidden = value != 0;
    else if (k == "gnn_far_tensor") {
        if (value != 0 && value != 1 && value != 2) return fail(c, EPNN_E_INVALID, "gnn_far_tensor must be 0 (off), 1 (on) or 2 (auto)");
        c->kopt.far_tensor = (int)value;
    } else if (k == "gnn_far_tensor_impl") {
        if (value != 1 && value != 2) return fail(c, EPNN_E_INVALID, "gnn_far_tensor_impl must be 1 or 2");
        c->kopt.far_tensor_impl = (int)value;
    } else if (k == "gnn_far_tensor_min") {
        if (value < SMALL_MAX + 1) return fail(c, EPNN_E_INVALID, "gnn_far_tensor_min must exceed %d", SMALL_MAX);
        c->kopt.far_tensor_min = (int)value;
    }
    else if (k == "dedup_far") c->dedup_far = value != 0;
    else if (k == "pair_tensor") c->kopt.pair_tensor = value != 0;
    else if (k == "atom_tensor") c->atom_tensor = value != 0;
    else if (k == "fused_prep") c->fused_prep = value != 0;
    else if (k == "chunk_streams") {
        if (value != 1 && value != 2) return fail(c, EPNN_E_INVALID, "chunk_streams must be 1 or 2");
        c->chunk_streams = (int)value;
    }
    else if (k == "pair_const") {
        if (value != 0 && value != 1 && value != 2) return fail(c, EPNN_E_INVALID, "pair_const must be 0, 1 or 2");
        c->kopt.pair_const = (int)value;
    }
    else if (k == "chunk_atoms") {
        if (value < 64) return fail(c, EPNN_E_INVALID, "chunk_atoms must be >= 64");
        c->chunk_atoms = (int64_t)value;
    } else return fail(c, EPNN_E_INVALID, "unknown option '%s'", key);
    return EPNN_OK;
}

extern "C" int epnn_host_alloc(void** ptr, size_t bytes) {
    if (!ptr) return EPNN_E_INVALID;
    return cudaMallocHost(ptr, bytes ? bytes : 1) == cudaSuccess ? EPNN_OK : EPNN_E_NOMEM;
}
extern "C" int epnn_host_free(void* ptr) { return cudaFreeHost(ptr) == cudaSuccess ? EPNN_OK : EPNN_E_CUDA; }

// ------------------------------------------------------------------------------------------------
// Per-system prep: rebased offsets, default npad, validation, row-group counts.
__global__ void sys_prep_kernel(int n_sys, const int* __restrict__ off_in, int base, int* __restrict__ off_out,
                                const int* __restrict__ npad_in, int* __restrict__ npad_out,
                                int* __restrict__ cnt_large, int* __restrict__ flags) {
    const int s = blockIdx.x * blockDim.x + threadIdx.x;
    if (s > n_sys) return;
    const int o = off_in[s] - base;
    off_out[s] = o;
    if (s == n_sys) return;
    const int n = off_in[s + 1] - off_in[s];
    int np = npad_in ? npad_in[s] : n;
    if (np < n || n <= 0) { atomicOr(flags, n <= 0 ? 2 : 1); np = n; }
    npad_out[s] = np;
    cnt_large[s] = n <= SMALL_MAX ? 0 : (n + 3) >> 2;      // 4-row groups of the large systems
}

__global__ void rg_fill_kernel(int n_sys, const int* __restrict__ off, const int* __restrict__ rgl_off, int* __restrict__ rg_large) {
    const int s = blockIdx.x * blockDim.x + threadIdx.x;
    if (s >= n_sys) return;
    const int a0 = off[s], a1 = off[s + 1];
    if (a1 - a0 <= SMALL_MAX) return;
    int* dst = rg_large + rgl_off[s];
    int k = 0;
    for (int i = a0; i < a1; i += 4) dst[k++] = i;
}

__global__ void species_check_kernel(int n, const int* __restrict__ species, int n_species, int* __restrict__ flags) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n && (species[i] < 0 || species[i] >= n_species)) atomicOr(flags, 4);
}

__global__ void collect_totals_kernel(const int* rowptr, const int* ustart, const int* far_off, int n_atoms,
                                      const int* rgl_off, int n_sys, int* flags) {
    flags[1] = rowptr[n_atoms]; flags[2] = ustart[n_atoms]; flags[3] = far_off[n_atoms]; flags[4] = rgl_off[n_sys];
}

// Sharded calls: active[i] = 1 for the rows of this rank's slice (PASS 0) and for every column of one of those rows (PASS 1).
template <int PASS>
__global__ void active_mark_kernel(int n_atoms, int row_lo, int row_hi, const int* __restrict__ rowptr, const int* __restrict__ col,
                                   unsigned char* __restrict__ active) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n_atoms) return;
    const bool mine = i >= row_lo && i < row_hi;
    if (PASS == 0) { active[i] = mine ? 1 : 0; return; }
    if (mine) for (int k = rowptr[i]; k < rowptr[i + 1]; ++k) active[col[k]] = 1;
}

struct Timer {
    bool on; cudaStream_t st; std::vector<cudaEvent_t> ev; std::vector<int> tag;
    ~Timer() { for (cudaEvent_t e : ev) cudaEventDestroy(e); }      // early returns (errors) must not leak the events
    void mark(int t) { if (!on) return; cudaEvent_t e; cudaEventCreate(&e); cudaEventRecord(e, st); ev.push_back(e); tag.push_back(t); }
    void finish(epnn_stats* s) {
        if (!on) return;
        if (s && !ev.empty()) {
            cudaEventSynchronize(ev.back());
            for (size_t i = 1; i < ev.size(); ++i) {
                float ms = 0; cudaEventElapsedTime(&ms, ev[i - 1], ev[i]);
                switch (tag[i]) {
                    case 1: s->ms_h2d += ms; break; case 2: s->ms_neighbor += ms; break; case 3: s->ms_gnn_pair += ms; break;
                    case 4: s->ms_gnn_atom += ms; break; case 5: s->ms_epn_pair += ms; break; case 6: s->ms_epn_atom += ms; break;
                    case 7: s->ms_d2h += ms; break; default: break;
                }
                s->ms_total += ms;
            }
        }
        for (cudaEvent_t e : ev) cudaEventDestroy(e);
        ev.clear(); tag.clear();
    }
};

// In-place all-gather of an array of pl.rows_pad rows of a sharded chunk: every rank contributes its slice (NCCL on `st`).
static int gather_rows(epnn_ctx* c, const ChunkPlan& pl, void* buf, size_t row_bytes, cudaStream_t st) {
    const int rcn = g_nccl.AllGather((char*)buf + (size_t)pl.slice * c->shard_rank * row_bytes, buf, (size_t)pl.slice * row_bytes, /* ncclInt8 */ 0, c->comm, st);
    if (rcn != 0) return fail(c, EPNN_E_CUDA, "ncclAllGather failed: %s", g_nccl.GetErrorString ? g_nccl.GetErrorString(rcn) : "?");
    ++c->xchg_calls; c->xchg_bytes += (int64_t)pl.slice * (c->shard_world - 1) * (int64_t)row_bytes;
    return EPNN_OK;
}

// Lists of one chunk (plan pl), device-resident inputs: d_off_in = slice of the caller's GLOBAL offsets (n_sys+1), h_off = the
// same offsets on the host.  Allocates the chunk's list workspaces, launches the list building, synchronises the stream once
// (totals and error flags) and fills w.  dedup: also build the species tables of the far-column de-duplication.
static int build_lists(epnn_ctx* c, const KernelChoice& kc, const ChunkPlan& pl, int n_sys, const int32_t* h_off, const int* d_off_in,
                       const float* d_xyz, const int* d_species, const float* d_Q, const int* d_npad_in, bool dedup,
                       epnn_stats* stats, Timer& tm, int* n_launch, int slot, Workspace& w) {
    cudaStream_t st = slot ? c->stream2 : c->stream;      // workspace slot 1 belongs to the second chunk stream
    const int sb = slot * B_COUNT;
    int* d_flags = c->d_flags + 8 * slot;
    int* h_flags = c->h_flags + 8 * slot;
    const int base = h_off[0], n_atoms = h_off[n_sys] - h_off[0];
    memset(&w, 0, sizeof(w));
    w.n_atoms = n_atoms; w.n_sys = n_sys; w.sm_count = c->sm_count;
    // sharded call (epnn_shard_init, world > 1): the rows of the chunk's LARGE systems are split into equal slices of the
    // atom index space, one per rank (pl.row_lo, pl.row_hi); small systems are replicated
    w.row_lo = pl.row_lo; w.row_hi = pl.row_hi;
    w.ek = kc.precision == 64 ? ED : EDR;
    w.n_species = c->n_species;
    w.kc = kc;
    w.wf_host = c->wf_host.data(); w.wf_dev = c->wf;
    w.work_counter = d_flags + 7;
    w.near_counter = stats && c->bufs[B_MISC].p ? (unsigned long long*)c->bufs[B_MISC].p : nullptr;
    w.slot_counter = stats && c->bufs[B_MISC].p ? (unsigned long long*)c->bufs[B_MISC].p + 2 : nullptr;
    { void* pa; int rca = ensure(c, sb + B_ARGS, 1024, &pa); if (rca != EPNN_OK) return rca; w.args_dev = pa; }
    w.xyz = d_xyz; w.species = d_species; w.Qsys = d_Q;
    void* p;
    int rc;
#define ENS(which, bytes, field, type) do { if ((rc = ensure(c, sb + (which), (bytes), &p)) != EPNN_OK) return rc; field = (type)p; } while (0)
    int *off_local, *npad_local, *cnt_l, *rgl_off, *scantmp, *far_cnt, *atom_b0;
    ENS(B_OFF, sizeof(int) * ((size_t)n_sys + 1), off_local, int*);
    ENS(B_NPAD, sizeof(int) * ((size_t)n_sys + 1), npad_local, int*);
    ENS(B_CNTL, sizeof(int) * ((size_t)n_sys + 1), cnt_l, int*);
    ENS(B_RGLOFF, sizeof(int) * ((size_t)n_sys + 1), rgl_off, int*);
    const size_t nmax = (size_t)(n_atoms > n_sys ? n_atoms : n_sys);
    ENS(B_SCANTMP, sizeof(int) * (nmax / 1024 + 2), scantmp, int*);
    ENS(B_ATOMSYS, sizeof(int) * (size_t)n_atoms, w.atom_sys, int*);
    ENS(B_DEG, sizeof(int) * (size_t)n_atoms, w.deg, int*);
    ENS(B_DEGU, sizeof(int) * (size_t)n_atoms, w.degU, int*);
    ENS(B_ROWPTR, sizeof(int) * ((size_t)n_atoms + 1), w.rowptr, int*);
    ENS(B_USTART, sizeof(int) * ((size_t)n_atoms + 1), w.ustart, int*);
    ENS(B_FARCNT, sizeof(int) * ((size_t)n_atoms + 1), far_cnt, int*);
    ENS(B_FAROFF, sizeof(int) * ((size_t)n_atoms + 1), w.far_off, int*);
    int* far0_cnt;
    ENS(B_FAR0CNT, sizeof(int) * ((size_t)n_atoms + 1), far0_cnt, int*);
    ENS(B_FAR0OFF, sizeof(int) * ((size_t)n_atoms + 1), w.far0_off, int*);
    ENS(B_REP, sizeof(int) * ((size_t)n_atoms + 1), w.rep, int*);
    w.dedup_far = dedup;
    ENS(B_ATOMB0, sizeof(int) * ((size_t)n_atoms + 1), atom_b0, int*);
    ENS(B_BNAT, sizeof(int) * ((size_t)n_atoms + 1), w.bundle_nat, int*);
    ENS(B_QD, sizeof(double) * (size_t)pl.rows_pad, w.q, double*);
    w.sys_off = off_local; w.npad = npad_local;

    w.n_bundles = (int)pl.bundles.size();
    ENS(B_BUNDLE, sizeof(int2) * (pl.bundles.size() + 1), w.bundle, int2*);
    if (!pl.bundles.empty()) CU(c, cudaMemcpyAsync(w.bundle, pl.bundles.data(), sizeof(int2) * pl.bundles.size(), cudaMemcpyHostToDevice, st));

    // ---- cell lists for the big systems of the chunk (the plan's budgets give the cell bases without a sync)
    CellWork cw;
    memset(&cw, 0, sizeof(cw));
    cw.n_large = pl.n_large; cw.n_cells = (int)pl.n_cells;
    if (cw.n_large) {
        int* dl;
        ENS(B_LARGESYS, sizeof(int) * pl.cell_tab.size(), dl, int*);
        CU(c, cudaMemcpyAsync(dl, pl.cell_tab.data(), sizeof(int) * pl.cell_tab.size(), cudaMemcpyHostToDevice, st));
        cw.large_sys = dl; cw.large_base = dl + cw.n_large;
        ENS(B_GRID, sizeof(CellGrid) * ((size_t)n_sys + 1), cw.grid, CellGrid*);
        ENS(B_CELLCNT, sizeof(int) * ((size_t)pl.n_cells + 2), cw.cell_cnt, int*);
        ENS(B_CELLSTART, sizeof(int) * ((size_t)pl.n_cells + 2), cw.cell_start, int*);
        ENS(B_CELLATOMS, sizeof(int) * ((size_t)pl.big_atoms + 1), cw.cell_atoms, int*);
        int* st2;
        ENS(B_SCANTMP, sizeof(int) * (((size_t)pl.n_cells > nmax ? (size_t)pl.n_cells : nmax) / 1024 + 2), st2, int*);
        scantmp = st2;
    }

    CU(c, cudaMemsetAsync(d_flags, 0, 8 * sizeof(int), st));
    sys_prep_kernel<<<div_up(n_sys + 1, 256), 256, 0, st>>>(n_sys, d_off_in, base, off_local, d_npad_in, npad_local, cnt_l, d_flags);
    species_check_kernel<<<div_up(n_atoms, 256), 256, 0, st>>>(n_atoms, d_species, c->n_species, d_flags);
    *n_launch += 2;
    CU(c, cudaGetLastError());
    CU(c, launch_scan_i32(cnt_l, rgl_off, n_sys, scantmp, st, n_launch));
    CU(c, launch_prep(w, st, n_launch));
    // Chunks of small systems only (the batched-molecule path): one warp per bundle builds every list from a 48-bit neighbour
    // mask per row (epnn_bundle_prep.cu); chunks with a larger system take the general thread-per-atom kernels.
    const bool fused = c->fused_prep && !pl.has_large && w.n_bundles > 0;
    BundlePrepWork bw;
    memset(&bw, 0, sizeof(bw));
    if (fused) {
        ENS(B_BPMASK, sizeof(unsigned long long) * (size_t)n_atoms, bw.mask, unsigned long long*);
        ENS(B_BPTOT, sizeof(int) * 4 * (size_t)w.n_bundles, bw.btot, int*);
        ENS(B_BPOFF, sizeof(int) * 4 * ((size_t)w.n_bundles + 1), bw.boff, int*);
        bw.atom_b0 = atom_b0;
        CU(c, launch_bundle_prep_count(w, bw, scantmp, d_flags, st, n_launch));
    } else {
        CU(c, launch_cell_build(w, cw, scantmp, st, n_launch));
        CU(c, launch_nbr_count(w, cw, st, n_launch));
        CU(c, launch_scan_i32(w.deg, w.rowptr, n_atoms, scantmp, st, n_launch));
        CU(c, launch_scan_i32(w.degU, w.ustart, n_atoms, scantmp, st, n_launch));
        CU(c, launch_far_count(w, far_cnt, atom_b0, st, n_launch));
        CU(c, launch_scan_i32(far_cnt, w.far_off, n_atoms, scantmp, st, n_launch));
        collect_totals_kernel<<<1, 1, 0, st>>>(w.rowptr, w.ustart, w.far_off, n_atoms, rgl_off, n_sys, d_flags);
        ++*n_launch;
    }
    CU(c, cudaMemcpyAsync(h_flags, d_flags, 8 * sizeof(int), cudaMemcpyDeviceToHost, st));
    CU(c, cudaStreamSynchronize(st));
    if (h_flags[0] & 1) return fail(c, EPNN_E_INVALID, "npad smaller than the number of atoms for at least one system");
    if (h_flags[0] & 2) return fail(c, EPNN_E_INVALID, "a system with zero (or negative) atoms was passed");
    if (h_flags[0] & 4) return fail(c, EPNN_E_INVALID, "species index outside the element table (n_x=%d has %d species)", c->n_x, c->n_species);
    w.nnz = h_flags[1]; w.P = h_flags[2]; w.n_far = h_flags[3];
    w.n_far0 = (int64_t)(MAX_SPECIES + 1) * n_atoms;      // capacity: at most one slot per species + the pad slot per row
    if (w.nnz < 0 || w.P < 0 || w.n_far < 0) return fail(c, EPNN_E_UNSUPPORTED, "pair lists of one chunk exceed 2^31 entries; lower chunk_atoms");
    w.n_rg_large = pl.n_rg_large; w.rg_begin = pl.rg_begin; w.rg_end = pl.rg_end;
    w.far_kernel = pl.far; w.nsplit = pl.nsplit;
    if (pl.far == FAR_CONST) {      // row-per-thread far kernel: warp units = 32-row block x column range
        w.n_rowblk = (int)pl.rowblk.size();
        w.blk_begin = pl.blk_begin; w.blk_end = pl.blk_end;
        int2* d_blk;
        ENS(B_ROWBLK, sizeof(int2) * (pl.rowblk.size() + 1), d_blk, int2*);
        CU(c, cudaMemcpyAsync(d_blk, pl.rowblk.data(), sizeof(int2) * pl.rowblk.size(), cudaMemcpyHostToDevice, st));
        CU(c, cudaStreamSynchronize(st));
        w.rowblk = d_blk;
    }

    ENS(B_COL, sizeof(int) * (size_t)(w.nnz + 1), w.col, int*);
    ENS(B_PID, sizeof(int) * (size_t)(w.nnz + 1), w.pid, int*);
    ENS(B_ROWL, (size_t)(w.nnz + 16), w.rowl, unsigned char*);
    ENS(B_PI, sizeof(int) * (size_t)(w.P + 1), w.pair_i, int*);
    ENS(B_PJ, sizeof(int) * (size_t)(w.P + 1), w.pair_j, int*);
    ENS(B_PD, sizeof(double) * (size_t)(w.P + 1), w.pair_D, double*);
    ENS(B_E, sizeof(float) * ED * (size_t)(w.P + 1), w.e, float*);
    ENS(B_NEAR, (size_t)(w.P + 16), w.near, unsigned char*);
    ENS(B_PERM, (size_t)(w.P + 16), w.perm_j, unsigned char*);
    ENS(B_FARLIST, sizeof(unsigned short) * (size_t)(w.n_far + 2), w.far_list, unsigned short*);
    ENS(B_FAR0LIST, sizeof(unsigned short) * (size_t)(w.n_far0 + 2), w.far0_list, unsigned short*);
    ENS(B_FAR0W, (size_t)(w.n_far0 + 16), w.far0_w, unsigned char*);
    ENS(B_RGL, sizeof(int) * (size_t)(w.n_rg_large + 1), w.rg_large, int*);
    rg_fill_kernel<<<div_up(n_sys, 256), 256, 0, st>>>(n_sys, off_local, rgl_off, w.rg_large);
    ++*n_launch;
    CU(c, cudaGetLastError());
    w.rgl_off = rgl_off;
    if (w.n_rg_large > 0 && dedup) {      // species tables of the large systems (far-column de-duplication)
        w.n_sp_tab = w.n_rg_large / 8 + 2;
        ENS(B_SPTAB, sizeof(int) * 32 * (size_t)w.n_sp_tab, w.sp_tab, int*);
        ENS(B_SPSTAMP, sizeof(int) * 2 * (size_t)w.n_sp_tab, w.sp_stamp, int*);
        if (pl.sharded) {      // the tables' "a row has more than 255 neighbours" flag must come out the same on every rank: full degrees
            int* dall;
            ENS(B_DEGALL, sizeof(int) * (size_t)pl.rows_pad, dall, int*);
            CU(c, cudaMemcpyAsync(dall, w.deg, sizeof(int) * (size_t)n_atoms, cudaMemcpyDeviceToDevice, st));
            if ((rc = gather_rows(c, pl, dall, sizeof(int), st)) != EPNN_OK) return rc;
            w.deg_all = dall;
        }
        CU(c, launch_sp_tab_build(w, st, n_launch));
        w.dedup_rows = stats ? (unsigned long long*)c->bufs[B_MISC].p + 1 : nullptr;
    }
    if (fused) {
        CU(c, launch_bundle_prep_fill(w, bw, st, n_launch));
        CU(c, launch_edge_desc(w, st, n_launch, true));
        CU(c, launch_tile_perm(w, atom_b0, st, n_launch));
    } else {
        if (cw.n_large) ENS(B_DTMP, sizeof(double) * (size_t)(w.nnz + 1), cw.Dtmp, double*);
        CU(c, launch_nbr_fill(w, cw, st, n_launch));
        CU(c, launch_far_fill(w, atom_b0, st, n_launch));
        if (kc.csr_rowl) CU(c, launch_csr_rowl(w, atom_b0, st, n_launch));
        // species-compressed far list (needs the filled CSR): counts -> offsets -> slots; its size is bounded, no host sync
        CU(c, launch_far0_count(w, far0_cnt, st, n_launch));
        CU(c, launch_scan_i32(far0_cnt, w.far0_off, n_atoms, scantmp, st, n_launch));
        CU(c, launch_far0_fill(w, atom_b0, st, n_launch));
    }
#undef ENS
    tm.mark(2);
    if (stats) {
        stats->n_pairs_e += w.P;
        stats->n_row_groups += w.n_bundles + w.n_rg_large;
    }
    return EPNN_OK;
}

// The T message-passing steps and T electron-passing passes of one chunk whose lists build_lists made (R = float: precision
// 32 and 48, double: 64).  Enqueued without a host sync.
template <typename R>
static int run_layers(epnn_ctx* c, const KernelChoice& kc, const ChunkPlan& pl, Workspace& w, float* d_out32, double* d_out64,
                      Timer& tm, int* n_launch, int slot) {
    cudaStream_t st = slot ? c->stream2 : c->stream;
    const int sb = slot * B_COUNT;
    const int n_atoms = w.n_atoms;
    // mixed precision (48): FP32 pair kernels around an FP64 per-atom kernel (state l2 / h in FP64, S / u / v / delta in FP32)
    const bool mixed = kc.precision == 48;
    const bool sharded = pl.sharded;
    void* p;
    int rc;
#define ENS(which, bytes, field, type) do { if ((rc = ensure(c, sb + (which), (bytes), &p)) != EPNN_OK) return rc; field = (type)p; } while (0)
    const size_t state_sz = mixed ? sizeof(double) : sizeof(R);
    ENS(B_H, state_sz * HD * (size_t)pl.rows_pad, w.h, void*);
    ENS(B_L2, state_sz * HID * (size_t)pl.rows_pad, w.l2, void*);
    ENS(B_S, sizeof(R) * HID * (size_t)n_atoms * w.nsplit, w.S, void*);
    ENS(B_U, sizeof(R) * HID * (size_t)n_atoms, w.u, void*);
    ENS(B_V, sizeof(R) * HID * (size_t)pl.rows_pad, w.v, void*);
    ENS(B_DELTA, sizeof(R) * (size_t)(w.P + 1), w.delta, void*);
#undef ENS
    CU(c, cudaMemsetAsync(w.h, 0, state_sz * HD * (size_t)n_atoms, st));

    const R* wb = sizeof(R) == 4 ? (const R*)c->wf : (const R*)c->wd;
    const UpdW<R> upd = upd_view<R>(wb, c->po);
    std::vector<StepW<R>> msg(c->T), pas(c->T);
    for (int t = 0; t < c->T; ++t) { msg[t] = step_view<R>(wb, c->po.msg[t]); pas[t] = step_view<R>(wb, c->po.pas[t]); }
    const UpdW<double> updd = upd_view<double>(c->wd, c->po);
    std::vector<StepW<double>> msgd(mixed ? c->T : 0), pasd(mixed ? c->T : 0);
    for (int t = 0; t < (int)msgd.size(); ++t) { msgd[t] = step_view<double>(c->wd, c->po.msg[t]); pasd[t] = step_view<double>(c->wd, c->po.pas[t]); }
    // per-atom kernel in the precision of the call; prev / next index the message (0 .. T-1) and pass (T .. 2T-1) MLPs, -1 = none
    auto atom = [&](int mode, int prev, int next, int h_is_zero, float* o32, double* o64, int scope) -> cudaError_t {
        auto pick = [&](auto& ms, auto& ps, int i) { return i < 0 ? nullptr : (i < c->T ? &ms[i] : &ps[i - c->T]); };
        if (mixed) return launch_atom_mixed(w, mode, pick(msgd, pasd, prev), &updd, pick(msgd, pasd, next), h_is_zero, o32, o64, st, n_launch, scope);
        return launch_atom<R>(w, mode, pick(msg, pas, prev), &upd, pick(msg, pas, next), h_is_zero, o32, o64, st, n_launch, scope);
    };

    // Sharded call: rows of large systems outside [row_lo, row_hi) belong to other ranks.  Per-atom work runs on the owned rows
    // (scope 1); the electron-passing projections also on the near neighbours of owned rows ("active", scope 2), because the
    // pair kernel needs u / v of both members of a cut pair.  Exchanges (in-place all-gathers of equal slices, NCCL on the ctx
    // stream): v after every message-passing step but the last (128 B/atom; the all-pairs sum reads every column), the update
    // MLP's last hidden layer once after the last step (128 B/atom), the charges after every pass (8 B/atom).  Cut pairs are
    // evaluated on both owners in the same canonical orientation, so no transfer is exchanged, and every row is computed by
    // exactly the arithmetic of the single-GPU run: results are bit-identical.
    const int own = sharded ? 1 : 0, act = sharded ? 2 : 0;
    if (sharded) {
        unsigned char* am;
        if ((rc = ensure(c, sb + B_ACTIVE, (size_t)n_atoms + 16, &p)) != EPNN_OK) return rc;
        am = (unsigned char*)p;
        active_mark_kernel<0><<<div_up(n_atoms, 256), 256, 0, st>>>(n_atoms, w.row_lo, w.row_hi, w.rowptr, w.col, am);
        active_mark_kernel<1><<<div_up(n_atoms, 256), 256, 0, st>>>(n_atoms, w.row_lo, w.row_hi, w.rowptr, w.col, am);
        *n_launch += 2;
        CU(c, cudaGetLastError());
        w.active = am;
    }
    const size_t state_row = (mixed ? sizeof(double) : sizeof(R)) * HID;
    // ---- GNN layer: T message-passing steps (charge_gn.py:60-74)
    CU(c, atom(ATOM_PROJECT, -1, 0, 1, nullptr, nullptr, 0));        // h = 0: u, v follow from species and q alone -- every rank, every atom
    tm.mark(4);
    for (int t = 0; t < c->T; ++t) {
        CU(c, launch_gnn_bundle<R>(w, msg[t], st, n_launch));
        w.stamp = w.sp_tab ? t + 1 : 0;             // large systems: are this step's v rows equal species by species?
        CU(c, launch_sp_check<R>(w, st, n_launch));
        if (w.far_kernel == FAR_TC || w.far_kernel == FAR_TC2) {
            if (w.far_kernel == FAR_TC2)
                CU(c, launch_gnn_far_tc2(w, c->w2split + (size_t)t * 2048, c->w2split + (size_t)t * 2048 + 1024, (const float*)msg[t].b2,
                                         w.nsplit - 1, st, n_launch));
            else
                CU(c, launch_gnn_far_tc(w, c->w2split + (size_t)t * 2048, c->w2split + (size_t)t * 2048 + 1024, (const float*)msg[t].b2,
                                        w.nsplit - 1, st, n_launch));
        }
        if constexpr (sizeof(R) == 4) {
            if (w.far_kernel == FAR_CONST) CU(c, launch_gnn_far_const(w, msg[t], w.nsplit - 1, st, n_launch));
        }
        CU(c, launch_gnn_pair<R>(w, msg[t], st, n_launch));
        tm.mark(3);
        const bool last = t + 1 == c->T;
        if (!sharded) {
            CU(c, atom(ATOM_UPDATE | ATOM_PROJECT | (t == 0 ? ATOM_FIRST : 0) | (last ? ATOM_WRITE_H : 0), t, t + 1, 0, nullptr, nullptr, 0));
        } else if (!last) {
            CU(c, atom(ATOM_UPDATE | ATOM_PROJECT | (t == 0 ? ATOM_FIRST : 0), t, t + 1, 0, nullptr, nullptr, own));
            if ((rc = gather_rows(c, pl, w.v, sizeof(R) * HID, st)) != EPNN_OK) return rc;
        } else {
            CU(c, atom(ATOM_UPDATE | ATOM_WRITE_H | (t == 0 ? ATOM_FIRST : 0), t, -1, 0, nullptr, nullptr, own));
            if ((rc = gather_rows(c, pl, w.l2, state_row, st)) != EPNN_OK) return rc;
            if (c->keep_hidden && (rc = gather_rows(c, pl, w.h, state_row / HID * HD, st)) != EPNN_OK) return rc;
            CU(c, atom(ATOM_PROJECT, -1, c->T, 0, nullptr, nullptr, act));
        }
        tm.mark(!last ? 4 : 6);
    }
    // ---- EPN layer: T electron-passing passes (charge_gn.py:98-118)
    for (int t = 0; t < c->T; ++t) {
        CU(c, launch_epn_bundle<R>(w, pas[t], st, n_launch));
        CU(c, launch_epn_pair<R>(w, pas[t], st, n_launch));
        tm.mark(5);
        const bool last = t + 1 == c->T;
        if (!sharded) {
            if (!last) CU(c, atom(ATOM_QUPDATE | ATOM_PROJECT, -1, c->T + t + 1, 0, nullptr, nullptr, 0));
            else CU(c, atom(ATOM_QUPDATE | ATOM_OUTPUT, -1, -1, 0, d_out32, d_out64, 0));
        } else {
            CU(c, atom(ATOM_QUPDATE, -1, -1, 0, nullptr, nullptr, own));
            if ((rc = gather_rows(c, pl, w.q, sizeof(double), st)) != EPNN_OK) return rc;
            if (!last) CU(c, atom(ATOM_PROJECT, -1, c->T + t + 1, 0, nullptr, nullptr, act));
            else CU(c, atom(ATOM_OUTPUT, -1, -1, 0, d_out32, d_out64, 0));
        }
        tm.mark(6);
    }
    c->hidden_atoms = n_atoms;
    c->hidden_precision = kc.precision == 32 ? 32 : 64;
    return EPNN_OK;
}

static int validate_offsets(epnn_ctx* c, int64_t n_sys, const int32_t* off) {
    if (n_sys < 0) return fail(c, EPNN_E_INVALID, "n_sys is negative");
    if (n_sys > 0 && !off) return fail(c, EPNN_E_INVALID, "atom_offsets is NULL");
    if (n_sys > 0 && off[0] != 0) return fail(c, EPNN_E_INVALID, "atom_offsets[0] must be 0");
    for (int64_t s = 0; s < n_sys; ++s)
        if (off[s + 1] <= off[s]) return fail(c, EPNN_E_INVALID, "system %lld has no atoms (offsets must be strictly increasing)", (long long)s);
    return EPNN_OK;
}


static int infer_impl(epnn_ctx* c, int precision, int atom_tensor, int64_t n_sys, const int32_t* off, bool host_io, const float* xyz,
                      const int32_t* species, const float* Q, const int32_t* npad_host, float* q_out, double* q_out64, epnn_stats* stats);

// "precision" 0 (auto): run a bounded prefix of the first call through the FP32, mixed and FP64 kernels and keep the cheapest
// precision whose charges stay within auto_tol of the FP64 kernels (which agree with the float64 oracle to 1e-9).  The
// conditioning of the model is a property of checkpoint AND data (|h| reaches 150 for model_weights on QM9), so it is
// measured on the caller's own systems, not assumed.  Sticky for the ctx until "precision" / "auto_tol" is set again.
static int probe_precision(epnn_ctx* c, int64_t n_sys, const int32_t* off, bool host_io, const float* xyz, const int32_t* species,
                           const float* Q, const int32_t* npad_host) {
    int64_t ns = n_sys < 64 ? n_sys : 64;
    while (ns > 1 && off[ns] > 8192) --ns;
    // a first system of more than 8192 atoms: the probe runs on a contiguous cut of its first 8192 atoms, taken as a system
    // of its own (same Q and npad), so that the choice still rests on the caller's data
    const int32_t cut_off[2] = {0, 8192};
    if (off[ns] > 8192) off = cut_off;
    const int64_t na = off[ns];
    c->probe_err32 = c->probe_err48 = -1;
    std::vector<float> hx, hQ, tmp((size_t)na);
    std::vector<int32_t> hs;
    const float* px = xyz; const int32_t* ps = species; const float* pq = Q;
    if (!host_io) {
        // the caller's inputs are ordered on the ctx stream (a caller stream after epnn_set_stream, typically non-blocking):
        // copy them there, not on the legacy default stream, which would not wait for the kernels that produce them
        hx.resize(3 * (size_t)na); hs.resize((size_t)na); hQ.resize((size_t)ns);
        CU(c, cudaSetDevice(c->device));
        CU(c, cudaMemcpyAsync(hx.data(), xyz, sizeof(float) * 3 * (size_t)na, cudaMemcpyDeviceToHost, c->stream));
        CU(c, cudaMemcpyAsync(hs.data(), species, sizeof(int32_t) * (size_t)na, cudaMemcpyDeviceToHost, c->stream));
        CU(c, cudaMemcpyAsync(hQ.data(), Q, sizeof(float) * (size_t)ns, cudaMemcpyDeviceToHost, c->stream));
        CU(c, cudaStreamSynchronize(c->stream));
        px = hx.data(); ps = hs.data(); pq = hQ.data();
    }
    // candidates, cheapest first: FP32 with the per-atom kernel on the tensor path (if the option allows it), plain FP32 SIMT,
    // mixed -- each measured against the FP64 kernels
    std::vector<double> q[2];
    const int64_t hidden_atoms = c->hidden_atoms;
    const int atom_tensor = c->atom_tensor;
    auto run = [&](int prec, int tensor, std::vector<double>& out) {
        out.resize((size_t)na);
        return infer_impl(c, prec, tensor, ns, off, true, px, ps, pq, npad_host, tmp.data(), out.data(), nullptr);
    };
    auto dist = [&]() { double e = 0; for (int64_t i = 0; i < na; ++i) e = fmax(e, fabs(q[1][i] - q[0][i])); return e; };
    int rc = run(64, 0, q[0]);
    int choice = 64, tensor = atom_tensor;
    if (rc == EPNN_OK && atom_tensor) {
        if ((rc = run(32, 1, q[1])) == EPNN_OK) { c->probe_err32 = dist(); if (c->probe_err32 <= c->auto_tol) choice = 32; }
    }
    if (rc == EPNN_OK && choice == 64) {
        if ((rc = run(32, 0, q[1])) == EPNN_OK) { c->probe_err32 = dist(); if (c->probe_err32 <= c->auto_tol) { choice = 32; tensor = 0; } }
    }
    if (rc == EPNN_OK && choice == 64) {
        if ((rc = run(48, 0, q[1])) == EPNN_OK) { c->probe_err48 = dist(); if (c->probe_err48 <= c->auto_tol) choice = 48; }
    }
    c->hidden_atoms = hidden_atoms;
    if (rc != EPNN_OK) return rc;
    c->auto_choice = choice; c->auto_atom_tensor = tensor;
    return EPNN_OK;
}

// precision 32 / 48 / 64 with the FP32 per-atom kernel on the tensor path or not (atom_tensor), or 0: the ctx's auto choice
// (probed on first use)
static int infer_impl(epnn_ctx* c, int precision, int atom_tensor, int64_t n_sys, const int32_t* off, bool host_io, const float* xyz,
                      const int32_t* species, const float* Q, const int32_t* npad_host, float* q_out, double* q_out64, epnn_stats* stats) {
    int rc = validate_offsets(c, n_sys, off);
    if (rc != EPNN_OK) return rc;
    if (stats) memset(stats, 0, sizeof(*stats));
    if (n_sys == 0) return EPNN_OK;
    if (!xyz || !species || !Q || (!q_out && !q_out64)) return fail(c, EPNN_E_INVALID, "NULL input/output pointer");
    if (precision == 0) {
        if (c->auto_choice == 0 && (rc = probe_precision(c, n_sys, off, host_io, xyz, species, Q, npad_host)) != EPNN_OK) return rc;
        precision = c->auto_choice; atom_tensor = c->auto_atom_tensor;
    }
    const KernelChoice kc = resolve_kernels(precision, atom_tensor, c->kopt);
    CU(c, cudaSetDevice(c->device));
    cudaStream_t st = c->stream;
    std::vector<int64_t> bounds;
    plan_chunks(off, n_sys, c->chunk_atoms, bounds);
    Timer tm{c->timing != 0, st, {}, {}};
    int n_launch = 0;
    unsigned long long* d_near_count = nullptr;
    void* p;
    if ((rc = ensure(c, B_MISC, 64, &p)) != EPNN_OK) return rc;
    d_near_count = (unsigned long long*)p;
    CU(c, cudaMemsetAsync(d_near_count, 0, 4 * sizeof(unsigned long long), st));      // [0] near pairs, [1] de-duplicated rows, [2] near / [3] far slots run by the bundle GNN kernel
    tm.mark(0);
    // ---- staging: two slots, sized once for the largest chunk (no regrow while copies are in flight).  Host-buffer calls
    // pipeline the chunks: upload(k + 1) and download(k - 1) run on their own streams while chunk k computes.
    const size_t n_chunks = bounds.size() - 1;
    int64_t max_na = 0, max_ns = 0;
    for (size_t ci = 0; ci < n_chunks; ++ci) {
        max_na = std::max<int64_t>(max_na, off[bounds[ci + 1]] - off[bounds[ci]]);
        max_ns = std::max<int64_t>(max_ns, bounds[ci + 1] - bounds[ci]);
    }
    struct Slot { int* off = nullptr; float* xyz = nullptr; int* sp = nullptr; float* Q = nullptr; float* o32 = nullptr; double* o64 = nullptr; } slot[2];
    const int n_slots = host_io && n_chunks > 1 ? 2 : 1;
    for (int k = 0; k < n_slots; ++k) {
        if ((rc = ensure(c, k ? B_OFFIN_1 : B_OFFIN, sizeof(int) * ((size_t)max_ns + 1) * 2 + 64, &p)) != EPNN_OK) return rc; slot[k].off = (int*)p;
        if (!host_io) continue;
        if ((rc = ensure(c, k ? B_XYZ_1 : B_XYZ, sizeof(float) * 3 * (size_t)max_na, &p)) != EPNN_OK) return rc; slot[k].xyz = (float*)p;
        if ((rc = ensure(c, k ? B_SPECIES_1 : B_SPECIES, sizeof(int) * (size_t)max_na, &p)) != EPNN_OK) return rc; slot[k].sp = (int*)p;
        if ((rc = ensure(c, k ? B_Q_1 : B_Q, sizeof(float) * (size_t)max_ns, &p)) != EPNN_OK) return rc; slot[k].Q = (float*)p;
        if (q_out) { if ((rc = ensure(c, k ? B_OUT32_1 : B_OUT32, sizeof(float) * (size_t)max_na, &p)) != EPNN_OK) return rc; slot[k].o32 = (float*)p; }
        if (q_out64) { if ((rc = ensure(c, k ? B_OUT64_1 : B_OUT64, sizeof(double) * (size_t)max_na, &p)) != EPNN_OK) return rc; slot[k].o64 = (double*)p; }
    }
    const bool piped = n_slots == 2;
    // two chunks in flight (even chunks: ctx stream + workspace slot 0, odd chunks: second stream + slot 1): the list building
    // of chunk k + 1 -- latency-bound, and followed by the call's one host sync per chunk -- runs beside the pair kernels of
    // chunk k.  Not for sharded contexts (their collectives share one communicator).
    const bool two = c->chunk_streams == 2 && n_chunks > 1 && c->shard_world <= 1;
    Timer tm2{c->timing != 0, c->stream2, {}, {}};
    if (two) {
        CU(c, cudaEventRecord(c->ev_fork, st));      // the second stream starts after whatever precedes this call on the ctx stream
        CU(c, cudaStreamWaitEvent(c->stream2, c->ev_fork, 0));
    }
    cudaStream_t down = piped ? c->d2h_stream : st;
    auto upload = [&](size_t ci, int k) -> int {      // offsets / npad always come from the host: they drive launch geometry
        cudaStream_t up = piped ? c->h2d_stream : (two && (ci & 1) ? c->stream2 : st);
        const int64_t s0 = bounds[ci], s1 = bounds[ci + 1];
        const int ns = (int)(s1 - s0), a0 = off[s0], na = off[s1] - off[s0];
        CU(c, cudaMemcpyAsync(slot[k].off, off + s0, sizeof(int) * ((size_t)ns + 1), cudaMemcpyHostToDevice, up));
        if (npad_host) CU(c, cudaMemcpyAsync(slot[k].off + ns + 1, npad_host + s0, sizeof(int) * (size_t)ns, cudaMemcpyHostToDevice, up));
        if (host_io) {
            CU(c, cudaMemcpyAsync(slot[k].xyz, xyz + 3 * (size_t)a0, sizeof(float) * 3 * (size_t)na, cudaMemcpyHostToDevice, up));
            CU(c, cudaMemcpyAsync(slot[k].sp, species + a0, sizeof(int) * (size_t)na, cudaMemcpyHostToDevice, up));
            CU(c, cudaMemcpyAsync(slot[k].Q, Q + s0, sizeof(float) * (size_t)ns, cudaMemcpyHostToDevice, up));
        }
        if (piped) CU(c, cudaEventRecord(c->ev_h2d[k], up));
        return EPNN_OK;
    };
    if ((rc = upload(0, 0)) != EPNN_OK) return rc;
    for (size_t ci = 0; ci < n_chunks; ++ci) {
        const int k = piped ? (int)(ci & 1) : 0;
        const int64_t s0 = bounds[ci], s1 = bounds[ci + 1];
        const int ns = (int)(s1 - s0);
        const int a0 = off[s0], a1 = off[s1];
        const int na = a1 - a0;
        const int ws = two ? (int)(ci & 1) : 0;
        cudaStream_t cs = ws ? c->stream2 : st;
        Timer& tmc = ws ? tm2 : tm;
        if (!piped && ci > 0 && (rc = upload(ci, 0)) != EPNN_OK) return rc;
        if (piped) CU(c, cudaStreamWaitEvent(cs, c->ev_h2d[k], 0));
        int* d_off = slot[k].off;
        int* d_npad_in = npad_host ? d_off + ns + 1 : nullptr;
        const float* d_xyz; const int* d_species; const float* d_Q; float* d_o32 = nullptr; double* d_o64 = nullptr;
        if (host_io) {
            d_xyz = slot[k].xyz; d_species = slot[k].sp; d_Q = slot[k].Q; d_o32 = slot[k].o32; d_o64 = slot[k].o64;
        } else {
            d_xyz = xyz + 3 * (size_t)a0; d_species = species + a0; d_Q = Q + s0;
            d_o32 = q_out ? q_out + a0 : nullptr; d_o64 = q_out64 ? q_out64 + a0 : nullptr;
        }
        tmc.mark(1);
        Workspace w;
        ChunkPlan& pl = c->plan;
        if (!plan_chunk(off + s0, ns, c->sm_count, c->shard_rank, c->comm ? c->shard_world : 1, kc, pl))
            rc = fail(c, EPNN_E_UNSUPPORTED, "cell grid exceeds 2^31 cells; lower chunk_atoms");
        else
            rc = build_lists(c, kc, pl, ns, off + s0, d_off, d_xyz, d_species, d_Q, d_npad_in, c->dedup_far, stats, tmc, &n_launch, ws, w);
        if (rc == EPNN_OK)
            rc = kc.precision == 64 ? run_layers<double>(c, kc, pl, w, d_o32, d_o64, tmc, &n_launch, ws)
                                    : run_layers<float>(c, kc, pl, w, d_o32, d_o64, tmc, &n_launch, ws);
        if (rc != EPNN_OK) { cudaStreamSynchronize(c->h2d_stream); cudaStreamSynchronize(down); cudaStreamSynchronize(c->stream2); cudaStreamSynchronize(st); return rc; }
        if (piped) {
            // build_lists made the chunk's one host sync (neighbour count): chunk ci - 1 is complete, the bulk of chunk ci is
            // queued.  Its results go down on their own stream; the other slot is free for chunk ci + 1 once ITS download is done.
            CU(c, cudaEventRecord(c->ev_done[k], cs));
            CU(c, cudaStreamWaitEvent(down, c->ev_done[k], 0));
        }
        if (host_io) {
            if (q_out) CU(c, cudaMemcpyAsync(q_out + a0, d_o32, sizeof(float) * (size_t)na, cudaMemcpyDeviceToHost, down));
            if (q_out64) CU(c, cudaMemcpyAsync(q_out64 + a0, d_o64, sizeof(double) * (size_t)na, cudaMemcpyDeviceToHost, down));
        }
        if (piped) {
            CU(c, cudaEventRecord(c->ev_d2h[k], down));
            if (ci + 1 < n_chunks) {
                if (ci >= 1) CU(c, cudaEventSynchronize(c->ev_d2h[k ^ 1]));       // chunk ci - 1 has left slot k ^ 1
                if ((rc = upload(ci + 1, k ^ 1)) != EPNN_OK) return rc;
            }
        } else if (host_io) {
            CU(c, cudaStreamSynchronize(cs));      // the single staging slot is reused by the next chunk
        }
        tmc.mark(7);
    }
    if (piped) { CU(c, cudaStreamSynchronize(c->h2d_stream)); CU(c, cudaStreamSynchronize(down)); }
    if (two) {
        CU(c, cudaEventRecord(c->ev_join, c->stream2));      // later work on the ctx stream is ordered after the odd chunks too
        CU(c, cudaStreamWaitEvent(st, c->ev_join, 0));
    }
    CU(c, cudaStreamSynchronize(st));
    if (stats) {
        unsigned long long nn[4] = {0, 0, 0, 0};
        CU(c, cudaMemcpy(nn, d_near_count, sizeof(nn), cudaMemcpyDeviceToHost));
        stats->n_pairs_near = (int64_t)nn[0];
        stats->n_far_dedup_rows = (int64_t)nn[1];
        stats->n_gnn_near_slots = (int64_t)nn[2]; stats->n_gnn_far_slots = (int64_t)nn[3];
        stats->n_systems = n_sys; stats->n_atoms = off[n_sys]; stats->n_chunks = (int64_t)bounds.size() - 1;
        stats->n_launches = n_launch;
        stats->precision_used = kc.precision;
        stats->probe_err32 = (float)c->probe_err32; stats->probe_err48 = (float)c->probe_err48;
        stats->atom_tensor_used = kc.precision == 32 ? atom_tensor : 0;
    }
    tm.finish(stats);
    tm2.finish(stats);          // (two chunk streams: the phase times of both are added up; they overlap in wall-clock time)
    if (bounds.size() != 2) c->hidden_atoms = 0;       // hidden state only meaningful for single-chunk calls
    return EPNN_OK;
}

extern "C" int epnn_infer_batch(epnn_ctx* c, int64_t n_sys, const int32_t* off, const float* xyz, const int32_t* species,
                                const float* Q, const int32_t* npad, float* q_out, double* q_out64, epnn_stats* stats) {
    if (!c) return EPNN_E_INVALID;
    return infer_impl(c, c->precision, c->atom_tensor, n_sys, off, true, xyz, species, Q, npad, q_out, q_out64, stats);
}

extern "C" int epnn_infer_batch_dev(epnn_ctx* c, int64_t n_sys, const int32_t* off_host, const float* xyz_dev,
                                    const int32_t* species_dev, const float* Q_dev, const int32_t* npad_host,
                                    float* q_out_dev, double* q_out64_dev, epnn_stats* stats) {
    if (!c) return EPNN_E_INVALID;
    return infer_impl(c, c->precision, c->atom_tensor, n_sys, off_host, false, xyz_dev, species_dev, Q_dev, npad_host, q_out_dev, q_out64_dev, stats);
}

// ------------------------------------------------------------------------------------------------
// Electrostatics of given charges (epnn_elst.cu).  Chunks of plan_chunks (whole systems) run one after the other on the ctx
// stream; the stream orders the reuse of every workspace, so the call synchronises once, at the end.
static int elst_impl(epnn_ctx* c, int64_t n_sys, const int32_t* off, bool host_io, const float* xyz, const double* q,
                     const int32_t* frag, double* energy, double* dipole, double* phi) {
    if (!c) return EPNN_E_INVALID;
    int rc = validate_offsets(c, n_sys, off);
    if (rc != EPNN_OK) return rc;
    if (n_sys == 0) return EPNN_OK;
    if (!xyz || !q) return fail(c, EPNN_E_INVALID, "NULL input pointer (xyz or q)");
    if (!energy && !dipole && !phi) return fail(c, EPNN_E_INVALID, "every output pointer is NULL (energy_out, dipole_out, phi_out)");
    CU(c, cudaSetDevice(c->device));
    cudaStream_t st = c->stream;
    std::vector<int64_t> bounds;
    plan_chunks(off, n_sys, c->chunk_atoms, bounds);
    std::vector<ElstItem> items;
    std::vector<ElstSys> sys;
    void* p;
    for (size_t ci = 0; ci + 1 < bounds.size(); ++ci) {
        const int64_t s0 = bounds[ci], s1 = bounds[ci + 1];
        const int ns = (int)(s1 - s0), a0 = off[s0], na = off[s1] - off[s0];
        const long long plen = elst_plan(off + s0, ns, (int64_t)c->sm_count * ELST_CTAS_PER_SM, items, sys);
        ElstArgs a;
        a.n_sys = ns; a.base = a0;
        if ((rc = ensure(c, B_EL_OFF, sizeof(int) * ((size_t)ns + 1), &p)) != EPNN_OK) return rc;
        a.off = (const int*)p;
        CU(c, cudaMemcpyAsync(p, off + s0, sizeof(int) * ((size_t)ns + 1), cudaMemcpyHostToDevice, st));
        const size_t items_bytes = sizeof(ElstItem) * items.size(), sys_bytes = sizeof(ElstSys) * sys.size();
        a.items = nullptr; a.sys = nullptr; a.partial = nullptr;
        if (!items.empty()) {
            if ((rc = ensure(c, B_EL_PLAN, items_bytes + sys_bytes, &p)) != EPNN_OK) return rc;
            CU(c, cudaMemcpyAsync(p, items.data(), items_bytes, cudaMemcpyHostToDevice, st));
            CU(c, cudaMemcpyAsync((char*)p + items_bytes, sys.data(), sys_bytes, cudaMemcpyHostToDevice, st));
            a.items = (const ElstItem*)p; a.sys = (const ElstSys*)((char*)p + items_bytes);
            if ((rc = ensure(c, B_EL_PART, sizeof(double) * (size_t)plen, &p)) != EPNN_OK) return rc;
            a.partial = (double*)p;
        }
        if (host_io) {
            if ((rc = ensure(c, B_EL_XYZ, sizeof(float) * 3 * (size_t)na, &p)) != EPNN_OK) return rc;
            a.xyz = (const float*)p;
            CU(c, cudaMemcpyAsync(p, xyz + 3 * (size_t)a0, sizeof(float) * 3 * (size_t)na, cudaMemcpyHostToDevice, st));
            if ((rc = ensure(c, B_EL_Q, sizeof(double) * (size_t)na, &p)) != EPNN_OK) return rc;
            a.q = (const double*)p;
            CU(c, cudaMemcpyAsync(p, q + a0, sizeof(double) * (size_t)na, cudaMemcpyHostToDevice, st));
            a.frag = nullptr;
            if (frag) {
                if ((rc = ensure(c, B_EL_FRAG, sizeof(int) * (size_t)na, &p)) != EPNN_OK) return rc;
                a.frag = (const int*)p;
                CU(c, cudaMemcpyAsync(p, frag + a0, sizeof(int) * (size_t)na, cudaMemcpyHostToDevice, st));
            }
            a.energy = a.dipole = a.phi = nullptr;
            if (energy) { if ((rc = ensure(c, B_EL_E, sizeof(double) * (size_t)ns, &p)) != EPNN_OK) return rc; a.energy = (double*)p; }
            if (dipole) { if ((rc = ensure(c, B_EL_MU, sizeof(double) * 3 * (size_t)ns, &p)) != EPNN_OK) return rc; a.dipole = (double*)p; }
            if (phi) { if ((rc = ensure(c, B_EL_PHI, sizeof(double) * (size_t)na, &p)) != EPNN_OK) return rc; a.phi = (double*)p; }
        } else {
            a.xyz = xyz + 3 * (size_t)a0; a.q = q + a0; a.frag = frag ? frag + a0 : nullptr;
            a.energy = energy ? energy + s0 : nullptr; a.dipole = dipole ? dipole + 3 * s0 : nullptr; a.phi = phi ? phi + a0 : nullptr;
        }
        CU(c, launch_elst(a, (int)items.size(), (int)sys.size(), st));
        if (host_io) {
            if (energy) CU(c, cudaMemcpyAsync(energy + s0, a.energy, sizeof(double) * (size_t)ns, cudaMemcpyDeviceToHost, st));
            if (dipole) CU(c, cudaMemcpyAsync(dipole + 3 * s0, a.dipole, sizeof(double) * 3 * (size_t)ns, cudaMemcpyDeviceToHost, st));
            if (phi) CU(c, cudaMemcpyAsync(phi + a0, a.phi, sizeof(double) * (size_t)na, cudaMemcpyDeviceToHost, st));
        }
    }
    CU(c, cudaStreamSynchronize(st));
    return EPNN_OK;
}

extern "C" int epnn_electrostatics(epnn_ctx* c, int64_t n_sys, const int32_t* off, const float* xyz, const double* q,
                                   const int32_t* fragment, double* energy_out, double* dipole_out, double* phi_out) {
    return elst_impl(c, n_sys, off, true, xyz, q, fragment, energy_out, dipole_out, phi_out);
}

extern "C" int epnn_electrostatics_dev(epnn_ctx* c, int64_t n_sys, const int32_t* off_host, const float* xyz_dev,
                                       const double* q_dev, const int32_t* fragment_dev, double* energy_out_dev,
                                       double* dipole_out_dev, double* phi_out_dev) {
    return elst_impl(c, n_sys, off_host, false, xyz_dev, q_dev, fragment_dev, energy_out_dev, dipole_out_dev, phi_out_dev);
}

// ------------------------------------------------------------------------------------------------
// Potential and field of given charges at given points (epnn_elst.cu).  Chunks of elst_pt_chunks run one after the other
// on the ctx stream, which orders the reuse of every workspace, so the call synchronises once, at the end.
static int points_impl(epnn_ctx* c, int64_t n_sys, const int32_t* off, bool host_io, const float* xyz, const double* q,
                       const int64_t* poff, const double* pts, double* phi, double* field) {
    if (!c) return EPNN_E_INVALID;
    int rc = validate_offsets(c, n_sys, off);
    if (rc != EPNN_OK) return rc;
    if (n_sys > 0 && !poff) return fail(c, EPNN_E_INVALID, "point_offsets is NULL");
    if (n_sys > 0 && poff[0] != 0) return fail(c, EPNN_E_INVALID, "point_offsets[0] must be 0");
    for (int64_t s = 0; s < n_sys; ++s)
        if (poff[s + 1] < poff[s]) return fail(c, EPNN_E_INVALID, "point_offsets decrease at system %lld", (long long)s);
    if (n_sys == 0) return EPNN_OK;
    if (!xyz || !q) return fail(c, EPNN_E_INVALID, "NULL input pointer (xyz or q)");
    if (!phi && !field) return fail(c, EPNN_E_INVALID, "every output pointer is NULL (phi_out, field_out)");
    if (poff[n_sys] > 0 && !pts) return fail(c, EPNN_E_INVALID, "points is NULL");
    CU(c, cudaSetDevice(c->device));
    cudaStream_t st = c->stream;
    std::vector<ElstPtChunk> chunks;
    elst_pt_chunks(off, poff, n_sys, c->chunk_atoms, ELST_PT_CHUNK, chunks);
    std::vector<ElstPtItem> items;
    std::vector<ElstPtRed> red;
    void* p;
    for (const ElstPtChunk& ch : chunks) {
        const int a0 = off[ch.s0], na = off[ch.s1] - off[ch.s0];
        const int64_t np = ch.p1 - ch.p0;
        const long long rows = elst_pt_plan(off, poff, ch, items, red);
        ElstPtArgs a;
        const size_t items_bytes = sizeof(ElstPtItem) * items.size(), red_bytes = sizeof(ElstPtRed) * red.size();
        if ((rc = ensure(c, B_PT_PLAN, items_bytes + red_bytes, &p)) != EPNN_OK) return rc;
        CU(c, cudaMemcpyAsync(p, items.data(), items_bytes, cudaMemcpyHostToDevice, st));
        if (!red.empty()) CU(c, cudaMemcpyAsync((char*)p + items_bytes, red.data(), red_bytes, cudaMemcpyHostToDevice, st));
        a.items = (const ElstPtItem*)p; a.red = (const ElstPtRed*)((char*)p + items_bytes);
        a.partial = nullptr;
        if (rows > 0) {
            if ((rc = ensure(c, B_PT_PART, sizeof(double) * (field ? 4 : 1) * (size_t)rows, &p)) != EPNN_OK) return rc;
            a.partial = (double*)p;
        }
        if (host_io) {
            if ((rc = ensure(c, B_PT_XYZ, sizeof(float) * 3 * (size_t)na, &p)) != EPNN_OK) return rc;
            a.xyz = (const float*)p;
            CU(c, cudaMemcpyAsync(p, xyz + 3 * (size_t)a0, sizeof(float) * 3 * (size_t)na, cudaMemcpyHostToDevice, st));
            if ((rc = ensure(c, B_PT_Q, sizeof(double) * (size_t)na, &p)) != EPNN_OK) return rc;
            a.q = (const double*)p;
            CU(c, cudaMemcpyAsync(p, q + a0, sizeof(double) * (size_t)na, cudaMemcpyHostToDevice, st));
            if ((rc = ensure(c, B_PT_PTS, sizeof(double) * 3 * (size_t)np, &p)) != EPNN_OK) return rc;
            a.pts = (const double*)p;
            CU(c, cudaMemcpyAsync(p, pts + 3 * ch.p0, sizeof(double) * 3 * (size_t)np, cudaMemcpyHostToDevice, st));
            a.phi = a.field = nullptr;
            if (phi) { if ((rc = ensure(c, B_PT_PHI, sizeof(double) * (size_t)np, &p)) != EPNN_OK) return rc; a.phi = (double*)p; }
            if (field) { if ((rc = ensure(c, B_PT_FIELD, sizeof(double) * 3 * (size_t)np, &p)) != EPNN_OK) return rc; a.field = (double*)p; }
        } else {
            a.xyz = xyz + 3 * (size_t)a0; a.q = q + a0; a.pts = pts + 3 * ch.p0;
            a.phi = phi ? phi + ch.p0 : nullptr; a.field = field ? field + 3 * ch.p0 : nullptr;
        }
        CU(c, launch_elst_points(a, (int)items.size(), (int)red.size(), st));
        if (host_io) {
            if (phi) CU(c, cudaMemcpyAsync(phi + ch.p0, a.phi, sizeof(double) * (size_t)np, cudaMemcpyDeviceToHost, st));
            if (field) CU(c, cudaMemcpyAsync(field + 3 * ch.p0, a.field, sizeof(double) * 3 * (size_t)np, cudaMemcpyDeviceToHost, st));
        }
    }
    CU(c, cudaStreamSynchronize(st));
    return EPNN_OK;
}

extern "C" int epnn_potential_points(epnn_ctx* c, int64_t n_sys, const int32_t* off, const float* xyz, const double* q,
                                     const int64_t* point_offsets, const double* points, double* phi_out, double* field_out) {
    return points_impl(c, n_sys, off, true, xyz, q, point_offsets, points, phi_out, field_out);
}

extern "C" int epnn_potential_points_dev(epnn_ctx* c, int64_t n_sys, const int32_t* off_host, const float* xyz_dev,
                                         const double* q_dev, const int64_t* point_offsets_host, const double* points_dev,
                                         double* phi_out_dev, double* field_out_dev) {
    return points_impl(c, n_sys, off_host, false, xyz_dev, q_dev, point_offsets_host, points_dev, phi_out_dev, field_out_dev);
}

// ------------------------------------------------------------------------------------------------
extern "C" int epnn_neighbors(epnn_ctx* c, int64_t n_sys, const int32_t* off, const float* xyz, int which,
                              int32_t* rowptr, int32_t* col, int64_t col_capacity, int64_t* nnz_out) {
    if (!c) return EPNN_E_INVALID;
    int rc = validate_offsets(c, n_sys, off);
    if (rc != EPNN_OK) return rc;
    if (!rowptr || !nnz_out || (which != 0 && which != 1)) return fail(c, EPNN_E_INVALID, "bad argument to epnn_neighbors");
    *nnz_out = 0;
    rowptr[0] = 0;
    if (n_sys == 0) return EPNN_OK;
    if (!xyz) return fail(c, EPNN_E_INVALID, "xyz is NULL");
    CU(c, cudaSetDevice(c->device));
    cudaStream_t st = c->stream;
    std::vector<int64_t> bounds;
    plan_chunks(off, n_sys, c->chunk_atoms, bounds);
    Timer tm{false, st, {}, {}};
    int n_launch = 0;
    const KernelChoice kc = resolve_kernels(32, c->atom_tensor, c->kopt);
    int64_t written = 0;
    bool overflow = false;
    std::vector<int> h_rowptr, h_col, h_pid;
    std::vector<unsigned char> h_near;
    for (size_t ci = 0; ci + 1 < bounds.size(); ++ci) {
        const int64_t s0 = bounds[ci], s1 = bounds[ci + 1];
        const int ns = (int)(s1 - s0), a0 = off[s0], na = off[s1] - off[s0];
        void* p;
        if ((rc = ensure(c, B_OFFIN, sizeof(int) * ((size_t)ns + 1) * 2 + 64, &p)) != EPNN_OK) return rc;
        int* d_off = (int*)p;
        CU(c, cudaMemcpyAsync(d_off, off + s0, sizeof(int) * ((size_t)ns + 1), cudaMemcpyHostToDevice, st));
        float* bx; int* bs; float* bq;
        if ((rc = ensure(c, B_XYZ, sizeof(float) * 3 * (size_t)na, &p)) != EPNN_OK) return rc; bx = (float*)p;
        if ((rc = ensure(c, B_SPECIES, sizeof(int) * (size_t)na, &p)) != EPNN_OK) return rc; bs = (int*)p;
        if ((rc = ensure(c, B_Q, sizeof(float) * (size_t)ns, &p)) != EPNN_OK) return rc; bq = (float*)p;
        CU(c, cudaMemcpyAsync(bx, xyz + 3 * (size_t)a0, sizeof(float) * 3 * (size_t)na, cudaMemcpyHostToDevice, st));
        CU(c, cudaMemsetAsync(bs, 0, sizeof(int) * (size_t)na, st));
        CU(c, cudaMemsetAsync(bq, 0, sizeof(float) * (size_t)ns, st));
        Workspace w;
        if (!plan_chunk(off + s0, ns, c->sm_count, 0, 1, kc, c->plan)) return fail(c, EPNN_E_UNSUPPORTED, "cell grid exceeds 2^31 cells; lower chunk_atoms");
        rc = build_lists(c, kc, c->plan, ns, off + s0, d_off, bx, bs, bq, nullptr, false, nullptr, tm, &n_launch, 0, w);
        if (rc != EPNN_OK) return rc;
        h_rowptr.resize((size_t)na + 1); h_col.resize((size_t)w.nnz + 1); h_pid.resize((size_t)w.nnz + 1); h_near.resize((size_t)w.P + 1);
        CU(c, cudaMemcpyAsync(h_rowptr.data(), w.rowptr, sizeof(int) * ((size_t)na + 1), cudaMemcpyDeviceToHost, st));
        if (w.nnz) {
            CU(c, cudaMemcpyAsync(h_col.data(), w.col, sizeof(int) * (size_t)w.nnz, cudaMemcpyDeviceToHost, st));
            CU(c, cudaMemcpyAsync(h_pid.data(), w.pid, sizeof(int) * (size_t)w.nnz, cudaMemcpyDeviceToHost, st));
            CU(c, cudaMemcpyAsync(h_near.data(), w.near, (size_t)w.P, cudaMemcpyDeviceToHost, st));
        }
        CU(c, cudaStreamSynchronize(st));
        for (int i = 0; i < na; ++i) {
            for (int k = h_rowptr[i]; k < h_rowptr[i + 1]; ++k) {
                if (which == 0 && !h_near[h_pid[k]]) continue;
                if (written < col_capacity && col) col[written] = h_col[k] + a0; else overflow = true;
                ++written;
            }
            rowptr[(size_t)a0 + i + 1] = (int32_t)written;
        }
    }
    *nnz_out = written;
    if (overflow) return fail(c, EPNN_E_CAPACITY, "col_capacity %lld too small for %lld entries", (long long)col_capacity, (long long)written);
    return EPNN_OK;
}

extern "C" int epnn_init_edges(epnn_ctx* c, int32_t n, const float* xyz, float* e_out) {
    if (!c) return EPNN_E_INVALID;
    if (n < 0 || (n > 0 && (!xyz || !e_out))) return fail(c, EPNN_E_INVALID, "bad argument to epnn_init_edges");
    if (n == 0) return EPNN_OK;
    CU(c, cudaSetDevice(c->device));
    void* p; int rc;
    if ((rc = ensure(c, B_XYZ, sizeof(float) * 3 * (size_t)n, &p)) != EPNN_OK) return rc;
    float* dx = (float*)p;
    const size_t tot = (size_t)n * n * ED;
    if ((rc = ensure(c, B_E, sizeof(float) * tot, &p)) != EPNN_OK) return rc;
    float* de = (float*)p;
    CU(c, cudaMemcpyAsync(dx, xyz, sizeof(float) * 3 * (size_t)n, cudaMemcpyHostToDevice, c->stream));
    CU(c, launch_edges_dense(n, dx, de, c->stream));
    CU(c, cudaMemcpyAsync(e_out, de, sizeof(float) * tot, cudaMemcpyDeviceToHost, c->stream));
    CU(c, cudaStreamSynchronize(c->stream));
    return EPNN_OK;
}

__global__ void d2f_kernel(const double* in, float* out, int64_t n) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) out[i] = (float)in[i];
}

extern "C" int epnn_get_hidden(epnn_ctx* c, float* h_out, int64_t n_floats) {
    if (!c || !h_out) return EPNN_E_INVALID;
    if (c->hidden_atoms == 0) return fail(c, EPNN_E_INVALID, "no hidden state retained (needs a preceding single-chunk epnn_infer_batch)");
    if (n_floats != c->hidden_atoms * HD) return fail(c, EPNN_E_INVALID, "expected %lld floats", (long long)(c->hidden_atoms * HD));
    CU(c, cudaSetDevice(c->device));
    if (c->hidden_precision == 32) {
        CU(c, cudaMemcpy(h_out, c->bufs[B_H].p, sizeof(float) * (size_t)n_floats, cudaMemcpyDeviceToHost));
    } else {
        void* p; int rc;
        if ((rc = ensure(c, B_OUT32, sizeof(float) * (size_t)n_floats, &p)) != EPNN_OK) return rc;
        d2f_kernel<<<div_up(n_floats, 256), 256, 0, c->stream>>>((const double*)c->bufs[B_H].p, (float*)p, n_floats);
        CU(c, cudaGetLastError());
        CU(c, cudaMemcpyAsync(h_out, p, sizeof(float) * (size_t)n_floats, cudaMemcpyDeviceToHost, c->stream));
        CU(c, cudaStreamSynchronize(c->stream));
    }
    return EPNN_OK;
}

template <typename R>
static int dense_impl(epnn_ctx* c, int B, int N, const float* h, const float* e, const float* x, const float* q,
                      const float* mask, float* q_out) {
    cudaStream_t st = c->stream;
    const size_t rows = (size_t)B * N, pairs = rows * N;
    const int F = c->n_x + HD + 1;
    void* p; int rc;
    float *dh, *de, *dx, *dq, *dm, *dout;
    R *da, *dnm, *duv, *dmsg;
#define ENS(which, bytes, var, type) do { if ((rc = ensure(c, which, (bytes), &p)) != EPNN_OK) return rc; var = (type)p; } while (0)
    ENS(B_H, sizeof(float) * pairs * HD, dh, float*);
    ENS(B_E, sizeof(float) * pairs * ED, de, float*);
    ENS(B_XYZ, sizeof(float) * pairs * c->n_x, dx, float*);
    ENS(B_Q, sizeof(float) * pairs, dq, float*);
    ENS(B_DELTA, sizeof(float) * pairs, dm, float*);
    ENS(B_OUT32, sizeof(float) * rows, dout, float*);
    ENS(B_S, sizeof(R) * rows * F, da, R*);
    ENS(B_QD, sizeof(R) * rows, dnm, R*);
    ENS(B_U, sizeof(R) * rows * 64, duv, R*);
    ENS(B_V, sizeof(R) * rows * HID, dmsg, R*);
#undef ENS
    CU(c, cudaMemcpyAsync(dh, h, sizeof(float) * pairs * HD, cudaMemcpyHostToDevice, st));
    CU(c, cudaMemcpyAsync(de, e, sizeof(float) * pairs * ED, cudaMemcpyHostToDevice, st));
    CU(c, cudaMemcpyAsync(dx, x, sizeof(float) * pairs * c->n_x, cudaMemcpyHostToDevice, st));
    CU(c, cudaMemcpyAsync(dq, q, sizeof(float) * pairs, cudaMemcpyHostToDevice, st));
    CU(c, cudaMemcpyAsync(dm, mask, sizeof(float) * pairs, cudaMemcpyHostToDevice, st));
    const R* wb = sizeof(R) == 4 ? (const R*)c->wf : (const R*)c->wd;
    std::vector<DenseW<R>> msg(c->T), pas(c->T);
    for (int t = 0; t < c->T; ++t) { msg[t] = dense_view<R>(wb, c->po.msg[t]); pas[t] = dense_view<R>(wb, c->po.pas[t]); }
    const UpdW<R> upd = upd_view<R>(wb, c->po);
    CU(c, launch_dense_forward<R>(B, N, c->n_x, c->T, dh, de, dx, dq, dm, msg.data(), upd, pas.data(), da, dnm, duv, dmsg, dout, st));
    CU(c, cudaMemcpyAsync(q_out, dout, sizeof(float) * rows, cudaMemcpyDeviceToHost, st));
    CU(c, cudaStreamSynchronize(st));
    c->hidden_atoms = 0;
    return EPNN_OK;
}

extern "C" int epnn_infer_dense(epnn_ctx* c, int32_t B, int32_t N, const float* h, const float* e, const float* x,
                                const float* q, const float* mask, float* q_out) {
    if (!c) return EPNN_E_INVALID;
    if (B < 0 || N < 0) return fail(c, EPNN_E_INVALID, "epnn_infer_dense: negative shape");
    if (B == 0 || N == 0) return EPNN_OK;
    if (!h || !e || !x || !q || !mask || !q_out) return fail(c, EPNN_E_INVALID, "epnn_infer_dense: NULL pointer");
    CU(c, cudaSetDevice(c->device));
    return c->precision == 64 ? dense_impl<double>(c, B, N, h, e, x, q, mask, q_out)
                              : dense_impl<float>(c, B, N, h, e, x, q, mask, q_out);
}

// ------------------------------------------------------------------------------------------------
extern "C" int epnn_shard_unique_id(void* id128) {
    if (!id128) return EPNN_E_INVALID;
    if (const char* e = load_nccl()) return fail(nullptr, EPNN_E_UNSUPPORTED, "%s", e);
    const int rc = g_nccl.GetUniqueId(id128);
    return rc == 0 ? EPNN_OK : fail(nullptr, EPNN_E_CUDA, "ncclGetUniqueId failed: %s", g_nccl.GetErrorString ? g_nccl.GetErrorString(rc) : "?");
}


extern "C" int epnn_shard_slice(int64_t n_atoms, int rank, int world, int64_t* begin, int64_t* end) {
    if (n_atoms < 0 || world < 1 || rank < 0 || rank >= world || !begin || !end) return EPNN_E_INVALID;
    const int64_t s = shard_slice_rows(n_atoms, world);
    *begin = s * rank < n_atoms ? s * rank : n_atoms;
    *end = s * (rank + 1) < n_atoms ? s * (rank + 1) : n_atoms;
    return EPNN_OK;
}

extern "C" int epnn_shard_init(epnn_ctx* c, int rank, int world, const void* id128) {
    if (!c) return EPNN_E_INVALID;
    if (world < 1 || rank < 0 || rank >= world) return fail(c, EPNN_E_INVALID, "epnn_shard_init: rank %d not in [0,%d)", rank, world);
    CU(c, cudaSetDevice(c->device));
    if (c->comm) {
        CU(c, cudaStreamSynchronize(c->stream));
        g_nccl.CommDestroy(c->comm);
        c->comm = nullptr;
    }
    c->shard_rank = 0; c->shard_world = 1; c->xchg_calls = 0; c->xchg_bytes = 0;
    if (world == 1) return EPNN_OK;
    if (!id128) return fail(c, EPNN_E_INVALID, "epnn_shard_init: the NCCL unique id (epnn_shard_unique_id on rank 0, shared with every rank) is required for world > 1");
    if (const char* e = load_nccl()) return fail(c, EPNN_E_UNSUPPORTED, "%s", e);
    NcclId id;
    memcpy(id.bytes, id128, sizeof(id.bytes));
    const int rc = g_nccl.CommInitRank(&c->comm, world, id, rank);
    if (rc != 0) { c->comm = nullptr; return fail(c, EPNN_E_CUDA, "ncclCommInitRank failed: %s", g_nccl.GetErrorString ? g_nccl.GetErrorString(rc) : "?"); }
    c->shard_rank = rank; c->shard_world = world;
    return EPNN_OK;
}

extern "C" int epnn_shard_stats(epnn_ctx* c, int64_t* calls, int64_t* bytes) {
    if (!c) return EPNN_E_INVALID;
    if (calls) *calls = c->xchg_calls;
    if (bytes) *bytes = c->xchg_bytes;
    return EPNN_OK;
}

extern "C" int epnn_set_stream(epnn_ctx* c, void* stream) {
    if (!c) return EPNN_E_INVALID;
    CU(c, cudaSetDevice(c->device));
    CU(c, cudaStreamSynchronize(c->stream));          // nothing of the ctx is in flight on the old stream when it switches
    c->stream = stream ? (cudaStream_t)stream : c->own_stream;
    return EPNN_OK;
}

extern "C" int epnn_get_stream(epnn_ctx* c, void** stream_out) {
    if (!c || !stream_out) return EPNN_E_INVALID;
    *stream_out = (void*)c->stream;
    return EPNN_OK;
}

// FP32 FMA micro-benchmark: 8 independent accumulator chains per thread, ITER x 8 FMAs, nothing else in the loop.
#define FMA_ITERS 4096
__global__ void __launch_bounds__(256) fma_peak_kernel(float* out, float a, float b) {
    float x0 = threadIdx.x, x1 = x0 + 1, x2 = x0 + 2, x3 = x0 + 3, x4 = x0 + 4, x5 = x0 + 5, x6 = x0 + 6, x7 = x0 + 7;
#pragma unroll 16
    for (int i = 0; i < FMA_ITERS; ++i) {
        x0 = fmaf(x0, a, b); x1 = fmaf(x1, a, b); x2 = fmaf(x2, a, b); x3 = fmaf(x3, a, b);
        x4 = fmaf(x4, a, b); x5 = fmaf(x5, a, b); x6 = fmaf(x6, a, b); x7 = fmaf(x7, a, b);
    }
    const float s = ((x0 + x1) + (x2 + x3)) + ((x4 + x5) + (x6 + x7));
    if (s == 123.456f) out[0] = s;            // never true in practice; keeps the chains alive
}

extern "C" int epnn_measure_fp32_peak(epnn_ctx* c, int repeats, double* tflops_out) {
    if (!c || !tflops_out || repeats < 1) return EPNN_E_INVALID;
    CU(c, cudaSetDevice(c->device));
    void* p; int rc;
    if ((rc = ensure(c, B_MISC, 64, &p)) != EPNN_OK) return rc;
    const int blocks = c->sm_count * 32, threads = 256;
    cudaEvent_t e0, e1;
    CU(c, cudaEventCreate(&e0)); CU(c, cudaEventCreate(&e1));
    double best = 0.0;
    for (int r = 0; r < repeats + 1; ++r) {            // first launch is the warm-up
        cudaEventRecord(e0, c->stream);
        fma_peak_kernel<<<blocks, threads, 0, c->stream>>>((float*)p + 8, 0.999f, 0.001f);
        cudaEventRecord(e1, c->stream);
        cudaError_t e = cudaEventSynchronize(e1);
        if (e != cudaSuccess) { cudaEventDestroy(e0); cudaEventDestroy(e1); CU(c, e); }
        float ms = 0; cudaEventElapsedTime(&ms, e0, e1);
        const double tf = 2.0 * 8.0 * FMA_ITERS * (double)blocks * threads / (ms * 1e-3) * 1e-12;
        if (r > 0 && tf > best) best = tf;
    }
    cudaEventDestroy(e0); cudaEventDestroy(e1);
    *tflops_out = best;
    return EPNN_OK;
}
