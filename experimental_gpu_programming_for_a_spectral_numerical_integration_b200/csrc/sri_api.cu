// sri_api.cu -- C ABI (include/sri.h) over the sm_100a kernels.  No torch types, no CPU fallback.
#include "../../include/sri.h"

#include <cuda_runtime.h>
#include <dlfcn.h>
#include <nvtx3/nvToolsExt.h>  // header-only NVTX v3: ranges are no-ops unless a profiler is attached

#include <algorithm>
#include <atomic>
#include <cmath>
#include <condition_variable>
#include <cstdio>
#include <cstdlib>
#include <cstdint>
#include <cstring>
#include <map>
#include <mutex>
#include <string>
#include <thread>
#include <tuple>
#include <utility>
#include <vector>

#include "sri_fused16.cuh"
#include "sri_fused16_dmma.cuh"
#include "sri_generic.cuh"
#include "sri_jacobian_dmma.cuh"
#include "sri_stage_dmma.cuh"
#include "sri_stage_generic.cuh"
#include "sri_stage_generic_tma.cuh"
#include "sri_stage_tma.cuh"
#include "sri_tiled.cuh"
#include "sri_tiled_dmma.cuh"
#include "sri_vjp16.cuh"
#include "sri_vjp_tiled.cuh"
#include "sri_wrench_generic.cuh"
#include "sri_wrench_gj.cuh"
#include "sri_wrench_gj_multi.cuh"
#include "sri_wrench_gj_static.cuh"
#include "sri_wrench_solve.cuh"
#include "sri_host_math.hpp"

namespace {

thread_local std::string g_last_error;
std::atomic<long long> g_launches{0};

int fail(int code, const std::string& msg) {
    g_last_error = msg;
    return code;
}

#define SRI_CUDA(expr)                                                                               \
    do {                                                                                             \
        cudaError_t e__ = (expr);                                                                    \
        if (e__ != cudaSuccess)                                                                      \
            return fail(SRI_ERR_CUDA, std::string(#expr) + ": " + cudaGetErrorString(e__));          \
    } while (0)

}  // namespace

struct sri_context {
    int N = 0, M = 0, device = 0;
    cudaStream_t stream = nullptr;
    cudaStream_t own_stream = nullptr;
    int sm_count = 0;
    sri_host::OperatorSet ops;
    double* d_ops16 = nullptr;   // OpsLayout16 tables (N <= 16) or OpsLayoutGeneric tables (N > 16)
    int R = 0;                   // generic kernel: row lanes (32 or 64); 0 for the N <= 16 kernel
    double* d_ops2 = nullptr;    // N > 16: tables of the DMMA kernel (Stx | AS | AT, TiledDmmaCfg)
    double* d_dtt = nullptr;     // D_TT (M x M, column-major), D_TI (M), D_TT^-1 (M x M): operator of the local-frame statics solve and its preconditioner
    double* d_tnodes = nullptr;  // 2 x_i - 1, i = 0..N-1
    double* d_reduce = nullptr;  // 2 doubles: sum rho^2, max |rho|
    double* d_ccw = nullptr;     // Clenshaw-Curtis weights of the nodes, [N]
    double* d_ptab = nullptr;    // Legendre polynomials at the nodes, P_k(2 x_i - 1), [8][N]
    double* d_jac = nullptr;     // S = Dn_NN^-1 and S_T = D_TT^-1, row-major [M][M] each (sri_shape_jacobian, sri_integrate_all_vjp), built on first use
    double* d_dnn = nullptr;     // Dn_NN, column-major [M][M] (sri_assemble_A), built on first use
    double* d_dnin = nullptr;    // Dn_IN [M] (sri_integrate_all_vjp), built on first use
    double* d_wrench_scratch = nullptr;  // 58 <= N <= 64: per-CTA operator of sri_integrate_wrench_local (L2-resident)
    size_t wrench_scratch_cap = 0;
    int wrench_impl = 0;         // SRI_WRENCH_IMPL: 0 = default (register-resident rolled Gauss-Jordan, N <= 33: one row per lane over 1-3 warps, two rows per lane for 12 <= N <= 16), 1 = blocked (N <= 16: shared-memory blocked LU with DMMA), 2 = generic (N > 16: CTA-wide LU), 3 = multi (one row per lane also for 12 <= N <= 16), 4 = warp (two rows per lane for every N <= 16)
    int jac_impl = 0;            // 0: DMMA kernel for N <= 16 (default), 1: SRI_JACOBIAN_IMPL=scalar everywhere (A/B measurements)
    const int* skip = nullptr;   // Newton loop with the device-side convergence flag: kernels launched while this is set take
                                 // it as their "already converged, do nothing" flag (NULL everywhere else)
    void* nccl_comm = nullptr;   // ncclComm_t attached by sri_nccl_init
    int nccl_nranks = 1, nccl_rank = 0;
    double* d_gather = nullptr;  // [2 * nccl_nranks] all-gathered norms
    double dmma_growth = sri::kDmmaGrowthDefault;
    bool use_dmma = false;       // DMMA elimination first, row-pivoting kernel for the rods it hands back (SRI_FUSED16_IMPL)
    struct NewtonWorkspace {  // buffers of sri_newton_static_shape, kept for the next call of the same shape
        int64_t B = -1; int ne = 0; unsigned present = 0; bool analytic = false;   // present: bits K0, q0, Gamma, fbar, lbar
        double* block = nullptr;
        double *K, *Q, *m, *nn, *g0, *J, *delta, *qe, *red, *F, *Mt, *K0, *qw, *Kw, *Qw, *mw, *gw, *Fw, *Mtw, *K0w;
        double *q0, *G, *fb, *lb, *q0w, *Gw, *fbw, *lbw;   // optional inputs of the problem and their forward-difference replicas
        int* sinfo = nullptr;            // [B] zero-pivot report of the per-rod Newton solve
        sri::NewtonState* state = nullptr;       // device: convergence flag, singular count, norm history
        sri::NewtonState* host_state = nullptr;  // two pinned mirrors: test t is copied to mirror t & 1 (followed by event t & 1)
        cudaEvent_t ev[2] = {nullptr, nullptr};
        // one Newton iteration + its device-side convergence test as a CUDA graph (lagged mode), replayed from iteration 2 on
        struct GraphKey { double H[3], tol, dof, fd_step; const void* block; const void* list; void* comm; cudaStream_t stream; };  // (no padding: compared bytewise)
        cudaGraphExec_t graph = nullptr;
        GraphKey graph_key{};
        long long graph_kernels = 0;     // kernel nodes per replay (for sri_kernel_launch_count)
        bool graph_off = false;          // SRI_NEWTON_GRAPH=0, or a capture failed on this handle
    } newton;
    struct AdjointWorkspace {  // buffers of sri_static_shape_vjp, kept for the next call of the same shape
        int64_t B = -1; int ne = 0;
        double* block = nullptr;
        double *K, *Q, *n, *m, *J, *rhs, *delta, *gKd, *gKi, *gQ, *gm, *gMd, *gMi, *gFi, *gHw, *lam, *gq0d, *gq0i;
        int *sinfo, *vinfo;      // [B] pivot reports of the J_a^T solve and of the transposed stage-1 solve
    } adjoint;
    double* d_partial = nullptr;  // block partials of galerkin_residual_kernel's norms, and its ticket counter
    size_t partial_cap = 0;
    unsigned* d_counter = nullptr;
    cudaEvent_t pipe_event = nullptr;  // orders the host-buffer pipeline after the work already queued on `stream`
    // tracing: every API call is an NVTX range; with sri_set_timing a CUDA-event pair brackets its work on `stream`
    bool timing = false;
    int call_depth = 0;                // nested entry points (e.g. sri_integrate_quaternions -> sri_integrate_all) time once
    cudaEvent_t t0 = nullptr, t1 = nullptr;
    const char* timed_call = nullptr;
    int stage_impl = 0;          // N <= 16 separate-stage entry points: 0 = measured best per stage (position, couple: TMA-staged;
                                 // stress: direct loads), 1 = SRI_STAGE_IMPL=tma everywhere, 2 = SRI_STAGE_IMPL=ldg everywhere
    // rods handed back by the DMMA kernel: [0] = count, entries from [4]; one list per pipeline slot + the handle stream
    int* d_list[5] = {nullptr, nullptr, nullptr, nullptr, nullptr};   // hand-back lists: pipeline slots 0-2, handle stream 3, local-frame statics 4
    size_t list_cap[5] = {0, 0, 0, 0, 0};
    int last_handback_slot = 3;  // list of the most recent two-pass call on the handle's stream (sri_get_handback_count)
    // host-buffer pipeline: chunks of rods flow H2D -> kernel -> D2H on rotating streams with persistent staging
    static constexpr int kPipeSlots = 3;
    static constexpr int kPipeArrays = 13;
    cudaStream_t pipe_stream[kPipeSlots] = {nullptr, nullptr, nullptr};
    void* pipe_buf[kPipeSlots][kPipeArrays] = {};
    size_t pipe_cap[kPipeSlots][kPipeArrays] = {};
};

namespace {

// ---- device/host buffer staging ----------------------------------------------------------------------------

bool is_device_pointer(const void* p) {
    if (!p) return false;
    cudaPointerAttributes a;
    if (cudaPointerGetAttributes(&a, p) != cudaSuccess) {
        cudaGetLastError();
        return false;
    }
    return a.type == cudaMemoryTypeDevice || a.type == cudaMemoryTypeManaged;
}

// Stages host buffers of one API call through stream-ordered device allocations.
class Staging {
public:
    explicit Staging(sri_context* h) : h_(h) {}
    ~Staging() {
        for (void* p : allocs_) cudaFreeAsync(p, h_->stream);
    }
    // read-only input: returns a device pointer (nullptr stays nullptr)
    template <typename T>
    int in(const T* p, size_t count, const T** out) {
        *out = nullptr;
        if (!p || count == 0) return SRI_OK;
        if (is_device_pointer(p)) { *out = p; return SRI_OK; }
        void* d = nullptr;
        SRI_CUDA(cudaMallocAsync(&d, count * sizeof(T), h_->stream));
        allocs_.push_back(d);
        SRI_CUDA(cudaMemcpyAsync(d, p, count * sizeof(T), cudaMemcpyHostToDevice, h_->stream));
        *out = static_cast<const T*>(d);
        used_host_ = true;
        return SRI_OK;
    }
    // output: returns a device pointer; host outputs are copied back by finish()
    template <typename T>
    int out(T* p, size_t count, T** outp) {
        *outp = nullptr;
        if (!p || count == 0) return SRI_OK;
        if (is_device_pointer(p)) { *outp = p; return SRI_OK; }
        void* d = nullptr;
        SRI_CUDA(cudaMallocAsync(&d, count * sizeof(T), h_->stream));
        allocs_.push_back(d);
        backs_.push_back({p, d, count * sizeof(T)});
        *outp = static_cast<T*>(d);
        used_host_ = true;
        return SRI_OK;
    }
    // an in-out host array that went in through in(): copy the staged device buffer back at finish()
    void copy_back(void* host, void* dev, size_t bytes) { backs_.push_back({host, dev, bytes}); }
    int finish() {
        for (auto& b : backs_) SRI_CUDA(cudaMemcpyAsync(b.host, b.dev, b.bytes, cudaMemcpyDeviceToHost, h_->stream));
        if (used_host_) SRI_CUDA(cudaStreamSynchronize(h_->stream));
        return SRI_OK;
    }

private:
    struct Back { void* host; void* dev; size_t bytes; };
    sri_context* h_;
    std::vector<void*> allocs_;
    std::vector<Back> backs_;
    bool used_host_ = false;
};

#define SRI_TRY(expr)              \
    do {                           \
        int rc__ = (expr);         \
        if (rc__ != SRI_OK) return rc__; \
    } while (0)

// cudaFuncAttributeMaxDynamicSharedMemorySize is a property of (kernel, device), not of a handle: keep one process-wide
// high-water mark per (kernel, device) that only grows, so that handles with different N / optional inputs on the same GPU
// cannot lower the limit under each other.
template <typename Kernel>
int ensure_dynamic_smem(Kernel kernel, int device, size_t bytes) {
    static std::mutex mu;
    static std::map<std::pair<const void*, int>, size_t> high;
    if (bytes <= 48 * 1024) return SRI_OK;
    std::lock_guard<std::mutex> lock(mu);
    size_t& cur = high[{reinterpret_cast<const void*>(kernel), device}];
    if (bytes > cur) {
        SRI_CUDA(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes));
        cur = bytes;
    }
    return SRI_OK;
}

// Resident CTAs per SM of `kernel` at this block size and dynamic shared memory (0: it does not fit), with the kernel's
// shared-memory limit raised first.  Like that limit, the answer belongs to (kernel, device), so it is cached process-wide.
template <typename Kernel>
int resident_ctas(const sri_context* h, Kernel kernel, int threads, size_t smem, int* occ) {
    SRI_TRY(ensure_dynamic_smem(kernel, h->device, smem));
    static std::mutex mu;
    static std::map<std::tuple<const void*, int, int, size_t>, int> cache;
    std::lock_guard<std::mutex> lock(mu);
    const auto key = std::make_tuple(reinterpret_cast<const void*>(kernel), h->device, threads, smem);
    auto it = cache.find(key);
    if (it == cache.end()) {
        int n = 0;
        SRI_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&n, kernel, threads, smem));
        it = cache.emplace(key, n).first;
    }
    *occ = it->second;
    return SRI_OK;
}

// Every kernel launch that sri_kernel_launch_count counts goes through here.
template <typename... Params, typename... Args>
int launch(void (*kernel)(Params...), dim3 grid, int threads, size_t smem, cudaStream_t stream, Args&&... args) {
    kernel<<<grid, threads, smem, stream>>>(std::forward<Args>(args)...);
    g_launches.fetch_add(1);
    SRI_CUDA(cudaGetLastError());
    return SRI_OK;
}

// the diagonal stiffness H_diag (3 doubles) from a host or device pointer
int read_H(const double* H_diag, double* H) {
    if (is_device_pointer(H_diag)) SRI_CUDA(cudaMemcpy(H, H_diag, 3 * sizeof(double), cudaMemcpyDeviceToHost));
    else std::memcpy(H, H_diag, 3 * sizeof(double));
    return SRI_OK;
}

// Makes the handle's device current for the duration of one API call and restores the caller's device afterwards.
class DeviceGuard {
public:
    DeviceGuard() = default;
    DeviceGuard(const DeviceGuard&) = delete;
    DeviceGuard& operator=(const DeviceGuard&) = delete;
    int enter(sri_context* h) {
        if (!h) return fail(SRI_ERR_INVALID_ARGUMENT, "null handle");
        if (cudaGetDevice(&prev_) != cudaSuccess) { cudaGetLastError(); prev_ = -1; }
        if (prev_ != h->device) {
            cudaError_t e = cudaSetDevice(h->device);
            if (e != cudaSuccess) return fail(SRI_ERR_CUDA, std::string("cudaSetDevice: ") + cudaGetErrorString(e));
            restore_ = prev_ >= 0;
        }
        return SRI_OK;
    }
    ~DeviceGuard() { if (restore_) cudaSetDevice(prev_); }

private:
    int prev_ = -1;
    bool restore_ = false;
};
// One API call on a handle: device guard + NVTX range named after the entry point + (optional) CUDA-event timer.
class CallScope {
public:
    explicit CallScope(const char* name) : name_(name) { nvtxRangePushA(name); }
    CallScope(const CallScope&) = delete;
    CallScope& operator=(const CallScope&) = delete;
    int enter(sri_context* h) {
        SRI_TRY(guard_.enter(h));
        h_ = h;
        if (h->call_depth++ == 0 && h->timing && h->t0) {
            timed_ = cudaEventRecord(h->t0, h->stream) == cudaSuccess;
            if (timed_) h->timed_call = nullptr;
        }
        return SRI_OK;
    }
    ~CallScope() {
        if (h_) {
            if (--h_->call_depth == 0 && timed_ && cudaEventRecord(h_->t1, h_->stream) == cudaSuccess) h_->timed_call = name_;
        }
        nvtxRangePop();
    }

private:
    const char* name_;
    DeviceGuard guard_;
    sri_context* h_ = nullptr;
    bool timed_ = false;
};
#define SRI_ENTER(h)               \
    CallScope scope__(__func__);   \
    SRI_TRY(scope__.enter(h))

}  // namespace

#include "sri_small_kernels.cuh"  // strain / residual / projection / Newton helper / peak kernels

namespace {

// ---- launch helpers --------------------------------------------------------------------------------------------

constexpr size_t kFusedSmem = (sri::OpsLayout16::total + (sri::kFusedThreads / 32) * sri::kWarpScratch16) * sizeof(double);

int list_reserve(sri_context* h, int slot, long long batch) {
    size_t need = (size_t)batch + 4;
    if (h->list_cap[slot] < need) {
        // grow generously (>= 2^20 entries, then doubling): a reallocation synchronises the device
        need = std::max(need, std::max((size_t)1 << 20, 2 * h->list_cap[slot]));
        if (h->d_list[slot]) SRI_CUDA(cudaFree(h->d_list[slot]));
        h->d_list[slot] = nullptr;
        h->list_cap[slot] = 0;
        SRI_CUDA(cudaMalloc(&h->d_list[slot], need * sizeof(int)));
        h->list_cap[slot] = need;
    }
    return SRI_OK;
}

// Points p.rod_count / p.rod_list at the emptied hand-back list `slot` (pipeline slots 0-2, handle stream 3, local-frame
// statics 4) for a first pass over `batch` rods; sri_get_handback_count reports the last list used on the handle's stream.
template <typename Params>
int handback_list(sri_context* h, int slot, long long batch, cudaStream_t stream, Params& p) {
    if (batch > 0x7fffffffLL) return fail(SRI_ERR_INVALID_ARGUMENT, "batch too large for one call (2^31 rods)");
    SRI_TRY(list_reserve(h, slot, batch));
    p.rod_count = h->d_list[slot];
    p.rod_list = h->d_list[slot] + 4;
    SRI_CUDA(cudaMemsetAsync(p.rod_count, 0, sizeof(int), stream));
    if (slot >= 3) h->last_handback_slot = slot;
    return SRI_OK;
}

// The fused four-stage integration runs in two passes: static-order elimination on the FP64 tensor cores, then the
// row-pivoting kernel over the rods that the first pass hands back (over every rod with SRI_FUSED16_IMPL=scalar).
// Kernel, block size, dynamic shared memory and rods per CTA of each pass for this handle's N:
struct FusedPass {
    void (*kernel)(sri::FusedParams);
    int threads;
    size_t smem;
    int rods_per_cta;
};
FusedPass fused_first_pass(const sri_context* h) {
    using C32 = sri::TiledDmmaCfg<4, 4, 4>;   // <row tiles per warp, column tiles, warps> for N <= 32
    using C64 = sri::TiledDmmaCfg<2, 8, 16>;  // and for N <= 64
    if (h->R == 0)  // one rod per warp
        return {h->M == 15 ? sri::fused16_dmma_kernel<15> : sri::fused16_dmma_kernel<0>, sri::kDmmaThreads, sri::kDmmaSmem, sri::kDmmaThreads / 32};
    if (h->R == 32) return {sri::tiled_dmma_kernel<4, 4, 4>, C32::threads, C32::smem_bytes, 1};
    return {sri::tiled_dmma_kernel<2, 8, 16>, C64::threads, C64::smem_bytes, 1};
}
FusedPass fused_second_pass(const sri_context* h) {
    if (h->R == 0)  // two rods per warp
        return {h->M == 15 ? sri::fused16_kernel<15> : sri::fused16_kernel<0>, sri::kFusedThreads, kFusedSmem, 2 * (sri::kFusedThreads / 32)};
    if (h->R == 32) return {sri::tiled_kernel<16, 4>, 128, sri::TiledSmem<16, 4>::total() * sizeof(double), 2};
    return {sri::tiled_kernel<32, 8>, 256, sri::TiledSmem<32, 8>::total() * sizeof(double), 1};
}

// list_slot: which hand-back list to use (pipeline slot, or 3 for the handle stream)
int launch_fused(sri_context* h, const sri::FusedParams& p_in, cudaStream_t stream = nullptr, bool use_handle_stream = true,
                 int list_slot = 3) {
    if (p_in.batch <= 0) return SRI_OK;
    sri::FusedParams p = p_in;
    if (use_handle_stream) { stream = h->stream; p.skip = h->skip; }
    // grid: one CTA per rods_per_cta rods, at most as many as are resident at once
    auto run = [&](const FusedPass& k) -> int {
        int occ = 0;
        SRI_TRY(resident_ctas(h, k.kernel, k.threads, k.smem, &occ));
        const long long want = (p.batch + k.rods_per_cta - 1) / k.rods_per_cta;
        return launch(k.kernel, (int)std::min(want, (long long)h->sm_count * occ), k.threads, k.smem, stream, p);
    };
    if (h->use_dmma) {
        SRI_TRY(handback_list(h, list_slot, p.batch, stream, p));
        const double g2 = h->dmma_growth * h->dmma_growth;
        const double lg = (g2 > 0.0) ? std::log2(g2) * 1048576.0 : -2.0e9;
        p.growth_log = (int)std::lround(std::max(-2.0e9, std::min(2.0e9, lg)));
        p.ops2 = h->d_ops2;
        SRI_TRY(run(fused_first_pass(h)));
        // second pass (row pivoting) over the rods handed back; CTAs without work exit at once
    }
    return run(fused_second_pass(h));
}

// ---- host-buffer pipeline --------------------------------------------------------------------------------------

// Host-buffer calls with an info array: every output has landed; report SRI_ERR_SINGULAR when any rod met a zero or
// non-finite pivot (info[b] != 0).  The other rods' results are valid.
int singular_status(const int* info_host, int64_t batch, const char* where) {
    if (!info_host) return SRI_OK;
    int64_t bad = 0, first = -1;
    for (int64_t b = 0; b < batch; ++b)
        if (info_host[b] != 0) { if (!bad) first = b; ++bad; }
    if (!bad) return SRI_OK;
    return fail(SRI_ERR_SINGULAR, std::string(where) + ": " + std::to_string(bad) + " rod(s) met a zero or non-finite pivot (first: rod " +
                                      std::to_string(first) + ", info = " + std::to_string(info_host[first]) + "); see the info array");
}

bool all_host_pointers(const sri_rod_batch* r) {
    const void* ptrs[] = {r->K, r->q0, r->r0, r->Gamma, r->fbar, r->lbar, r->F_tip, r->M_tip, r->Q, r->r, r->n, r->m, r->info};
    for (const void* p : ptrs)
        if (p && is_device_pointer(p)) return false;
    return true;
}

int pipe_reserve(sri_context* h, int slot, int arr, size_t bytes, void** out) {
    if (h->pipe_cap[slot][arr] < bytes) {
        if (h->pipe_buf[slot][arr]) SRI_CUDA(cudaFree(h->pipe_buf[slot][arr]));
        h->pipe_buf[slot][arr] = nullptr;
        h->pipe_cap[slot][arr] = 0;
        SRI_CUDA(cudaMalloc(&h->pipe_buf[slot][arr], bytes));
        h->pipe_cap[slot][arr] = bytes;
    }
    *out = h->pipe_buf[slot][arr];
    return SRI_OK;
}

// All buffers live on the host: split the batch into chunks and overlap the H2D copy of chunk c+1, the kernel of
// chunk c and the D2H copy of chunk c-1 on three streams (pinned host memory makes the copies truly asynchronous;
// pageable memory still works, serialised by the driver).  Returns after every result has landed.  The pipeline is ordered
// after whatever the caller has already queued on the handle's stream (e.g. an asynchronous copy that fills a pinned input
// buffer), and when a step fails it drains the copies already in flight before the error is returned.
int integrate_all_host_pipeline_body(sri_context* h, const sri_rod_batch* r);
int integrate_all_host_pipeline(sri_context* h, const sri_rod_batch* r) {
    for (int sl = 0; sl < sri_context::kPipeSlots; ++sl)
        if (!h->pipe_stream[sl]) SRI_CUDA(cudaStreamCreateWithFlags(&h->pipe_stream[sl], cudaStreamNonBlocking));
    if (!h->pipe_event) SRI_CUDA(cudaEventCreateWithFlags(&h->pipe_event, cudaEventDisableTiming));
    SRI_CUDA(cudaEventRecord(h->pipe_event, h->stream));
    for (int sl = 0; sl < sri_context::kPipeSlots; ++sl) SRI_CUDA(cudaStreamWaitEvent(h->pipe_stream[sl], h->pipe_event, 0));
    const int rc = integrate_all_host_pipeline_body(h, r);
    if (rc != SRI_OK) {
        const std::string keep = g_last_error;
        for (int sl = 0; sl < sri_context::kPipeSlots; ++sl) cudaStreamSynchronize(h->pipe_stream[sl]);
        cudaGetLastError();
        g_last_error = keep;
    }
    return rc;
}
int integrate_all_host_pipeline_body(sri_context* h, const sri_rod_batch* r) {
    const int N = h->N, M = h->M;
    const int64_t B = r->batch;
    // chunk schedule: a short first chunk fills the pipeline quickly (its H2D copy and kernel are the only work that is
    // not hidden behind the D2H stream, which bounds the call), the following ones are long enough that the per-transfer
    // set-up of the copy engines does not show
    const int64_t chunk = (N <= 16) ? 65536 : (N <= 32 ? 16384 : 4096);
    const int64_t first_chunk = chunk / 8;
    struct Arr { const void* src; void* dst; size_t per_rod; };
    int c = 0;
    for (int64_t first = 0, step = first_chunk; first < B; first += step, step = chunk, ++c) {
        const int slot = c % sri_context::kPipeSlots;
        cudaStream_t st = h->pipe_stream[slot];
        const int64_t nb = (B - first < step) ? (B - first) : step;
        const Arr ins[8] = {{r->K, nullptr, (size_t)3 * N * 8}, {r->q0, nullptr, 32}, {r->r0, nullptr, 24},
                            {r->Gamma, nullptr, (size_t)3 * N * 8}, {r->fbar, nullptr, (size_t)3 * N * 8},
                            {r->lbar, nullptr, (size_t)3 * N * 8}, {r->F_tip, nullptr, 24}, {r->M_tip, nullptr, 24}};
        const Arr outs[5] = {{nullptr, r->Q, (size_t)4 * M * 8}, {nullptr, r->r, (size_t)3 * M * 8}, {nullptr, r->n, (size_t)3 * M * 8},
                             {nullptr, r->m, (size_t)3 * M * 8}, {nullptr, r->info, 4}};
        void* din[8] = {};
        void* dout[5] = {};
        for (int a = 0; a < 8; ++a) {
            if (!ins[a].src) continue;
            SRI_TRY(pipe_reserve(h, slot, a, (size_t)chunk * ins[a].per_rod, &din[a]));
            SRI_CUDA(cudaMemcpyAsync(din[a], static_cast<const char*>(ins[a].src) + (size_t)first * ins[a].per_rod,
                                     (size_t)nb * ins[a].per_rod, cudaMemcpyHostToDevice, st));
        }
        for (int a = 0; a < 5; ++a) {
            if (!outs[a].dst) continue;
            SRI_TRY(pipe_reserve(h, slot, 8 + a, (size_t)chunk * outs[a].per_rod, &dout[a]));
        }
        sri::FusedParams p{};
        p.batch = nb; p.N = N; p.M = M; p.ops = h->d_ops16;
        p.K = static_cast<const double*>(din[0]); p.q0 = static_cast<const double*>(din[1]);
        p.r0 = static_cast<const double*>(din[2]); p.Gamma = static_cast<const double*>(din[3]);
        p.fbar = static_cast<const double*>(din[4]); p.lbar = static_cast<const double*>(din[5]);
        p.F_tip = static_cast<const double*>(din[6]); p.M_tip = static_cast<const double*>(din[7]);
        p.Q = static_cast<double*>(dout[0]); p.r = static_cast<double*>(dout[1]); p.n = static_cast<double*>(dout[2]);
        p.m = static_cast<double*>(dout[3]); p.info = static_cast<int*>(dout[4]);
        SRI_TRY(launch_fused(h, p, st, false, slot));
        for (int a = 0; a < 5; ++a) {
            if (!outs[a].dst) continue;
            SRI_CUDA(cudaMemcpyAsync(static_cast<char*>(outs[a].dst) + (size_t)first * outs[a].per_rod, dout[a],
                                     (size_t)nb * outs[a].per_rod, cudaMemcpyDeviceToHost, st));
        }
    }
    for (int sl = 0; sl < sri_context::kPipeSlots; ++sl) SRI_CUDA(cudaStreamSynchronize(h->pipe_stream[sl]));
    return singular_status(r->info, B, "sri_integrate_all");
}

template <int STAGE>
int launch_stage_dmma(sri_context* h, const sri::FusedParams& p) {
    if (p.batch <= 0) return SRI_OK;
    const long long tiles = (p.batch + 7) / 8;
    const long long want = (tiles + 3) / 4;
    return launch(sri::stage_dmma_kernel<STAGE>, (int)std::min(want, (long long)h->sm_count * 8), 128, 0, h->stream, p);
}

// the rods [done, batch) of a separate-stage call
sri::FusedParams stage_tail(const sri::FusedParams& p, long long done) {
    const int M = p.M, N = p.N;
    sri::FusedParams t = p;
    t.batch = p.batch - done;
    if (t.Qin) t.Qin += done * 4 * M;
    if (t.nin) t.nin += done * 3 * M;
    if (t.Gamma) t.Gamma += done * 3 * N;
    if (t.fbar) t.fbar += done * 3 * N;
    if (t.lbar) t.lbar += done * 3 * N;
    if (t.F_tip) t.F_tip += done * 3;
    if (t.M_tip) t.M_tip += done * 3;
    if (t.q0) t.q0 += done * 4;
    if (t.r0) t.r0 += done * 3;
    if (t.r) t.r += done * 3 * M;
    if (t.n) t.n += done * 3 * M;
    if (t.m) t.m += done * 3 * M;
    return t;
}

template <int STAGE>
bool stage_pointers_aligned(const sri::FusedParams& p) {
    auto al = [](const void* q) { return (reinterpret_cast<uintptr_t>(q) & 15u) == 0; };
    const double* load = (STAGE == sri::kStageStress) ? p.fbar : p.lbar;
    const double* tip = (STAGE == sri::kStageStress) ? p.F_tip : p.M_tip;
    double* out = (STAGE == sri::kStagePosition) ? p.r : (STAGE == sri::kStageStress ? p.n : p.m);
    return al(p.Qin) && al(p.nin) && al(p.Gamma) && al(load) && al(tip) && al(p.q0) && al(p.r0) && al(out);
}

// Separate-stage entry points for N <= 16: whole tiles of 8 rods through the TMA-staged kernel when every pointer is
// 16-byte aligned, the ragged tail (and unaligned calls) through the direct-load kernel.
template <int STAGE>
int launch_stage(sri_context* h, const sri::FusedParams& p_in) {
    if (p_in.batch <= 0) return SRI_OK;
    sri::FusedParams p = p_in;
    const int M = p.M, N = p.N;
    const long long tiles = p.batch / 8;
    const double* load = (STAGE == sri::kStageStress) ? p.fbar : p.lbar;
    const bool aligned = stage_pointers_aligned<STAGE>(p);
    // stress reads [3][16] stacks whose rows are 128-byte aligned: direct loads are already sector-exact there (92 % of HBM
    // against 83 % through shared memory); position / couple read 15-double rows and gain 5 % / 37 % from the staging
    const bool want_tma = h->stage_impl == 1 || (h->stage_impl == 0 && STAGE != sri::kStageStress);
    if (!want_tma || tiles == 0 || !aligned) return launch_stage_dmma<STAGE>(h, p);
    sri::StageTmaLayout L{};
    int off = 0;
    auto put = [&](bool present, int bytes) { if (!present) return -1; const int o = off; off += bytes; return o; };
    L.q = put(STAGE != sri::kStageStress, 8 * 4 * M * 8);
    L.nin = put(STAGE == sri::kStageCouple, 8 * 3 * M * 8);
    L.gam = put(STAGE != sri::kStageStress && p.Gamma, 8 * 3 * N * 8);
    L.load = put(STAGE != sri::kStagePosition && load, 8 * 3 * N * 8);
    L.tip = put(STAGE != sri::kStagePosition, 192);
    L.q0 = put(STAGE == sri::kStageCouple && p.q0, 256);
    L.r0 = put(STAGE == sri::kStagePosition && p.r0, 192);
    L.in_bytes = off;
    L.out = 2 * off;
    L.warp_bytes = 2 * off + 8 * 3 * M * 8;
    const size_t smem = (size_t)sri::kStageTmaWarps * L.warp_bytes;
    constexpr int threads = 32 * sri::kStageTmaWarps;
    int occ = 0;
    SRI_TRY(resident_ctas(h, sri::stage_tma_kernel<STAGE>, threads, smem, &occ));
    if (occ < 1) return launch_stage_dmma<STAGE>(h, p);
    const long long want = (tiles + sri::kStageTmaWarps - 1) / sri::kStageTmaWarps;
    SRI_TRY(launch(sri::stage_tma_kernel<STAGE>, (int)std::min(want, (long long)h->sm_count * occ), threads, smem, h->stream, p, L, tiles));
    if (tiles * 8 < p.batch) return launch_stage_dmma<STAGE>(h, stage_tail(p, tiles * 8));
    return SRI_OK;
}

// Separate-stage entry points for 17 <= N <= 64: streaming DMMA contraction against the fragment-ordered operator tables;
// whole tiles of 8 rods with TMA-staged inputs when the pointers are 16-byte aligned, the rest with direct loads.
template <int STAGE>
int launch_stage_generic_direct(sri_context* h, const sri::FusedParams& p) {
    if (p.batch <= 0) return SRI_OK;
    const long long tiles = (p.batch + 7) / 8;
    const long long want = (tiles + 3) / 4;
    const size_t smem = (size_t)h->R * h->R * sizeof(double);
    auto* kernel = h->R == 32 ? sri::stage_generic_kernel<STAGE, 32> : sri::stage_generic_kernel<STAGE, 64>;
    int occ = 0;
    SRI_TRY(resident_ctas(h, kernel, 128, smem, &occ));
    if (occ < 1) return fail(SRI_ERR_CUDA, "stage kernel does not fit on this device");
    return launch(kernel, (int)std::min(want, (long long)h->sm_count * occ), 128, smem, h->stream, p);
}

template <int STAGE>
int launch_stage_generic(sri_context* h, const sri::FusedParams& p_in) {
    if (p_in.batch <= 0) return SRI_OK;
    sri::FusedParams p = p_in;
    p.ops2 = h->d_ops2;
    const int M = p.M, N = p.N;
    const long long tiles = p.batch / 8;
    // as for N <= 16: the force stage reads 128-byte aligned [3][N] rows and is faster with direct loads (N = 32: 72 % of HBM
    // against 62 % staged), position and couple gain from the staging (N = 32: 64 -> 75 %, 59 -> 91 %; N = 64: +47 %, +20 %)
    const bool want_tma = h->stage_impl == 1 || (h->stage_impl == 0 && STAGE != sri::kStageStress);
    if (!want_tma || tiles == 0 || !stage_pointers_aligned<STAGE>(p)) return launch_stage_generic_direct<STAGE>(h, p);
    const double* load = (STAGE == sri::kStageStress) ? p.fbar : p.lbar;
    const double* tip = (STAGE == sri::kStagePosition) ? p.r0 : (STAGE == sri::kStageStress ? p.F_tip : p.M_tip);
    sri::StageTmaLayout L{};
    int off = 0;
    auto put = [&](bool present, int bytes) { if (!present) return -1; const int o = off; off += bytes; return o; };
    L.q = put(STAGE != sri::kStageStress, 8 * 4 * M * 8);
    L.nin = put(STAGE == sri::kStageCouple, 8 * 3 * M * 8);
    L.gam = put(STAGE != sri::kStageStress && p.Gamma, 8 * 3 * N * 8);
    L.load = put(STAGE != sri::kStagePosition && load, 8 * 3 * N * 8);
    L.tip = put(tip != nullptr, 192);
    L.q0 = put(STAGE == sri::kStageCouple && p.q0, 256);
    L.r0 = -1;
    L.in_bytes = off;
    L.out = 0;
    L.warp_bytes = off;
    if (off == 0) return launch_stage_generic_direct<STAGE>(h, p);  // nothing to stage (force stage without inputs)
    const size_t smem = (size_t)h->R * h->R * sizeof(double) + (size_t)4 * off;
    if (smem > 220 * 1024) return launch_stage_generic_direct<STAGE>(h, p);
    auto* kernel = h->R == 32 ? sri::stage_generic_tma_kernel<STAGE, 32> : sri::stage_generic_tma_kernel<STAGE, 64>;
    int occ = 0;
    SRI_TRY(resident_ctas(h, kernel, 128, smem, &occ));
    if (occ < 1) return launch_stage_generic_direct<STAGE>(h, p);
    const long long want = (tiles + 3) / 4;
    SRI_TRY(launch(kernel, (int)std::min(want, (long long)h->sm_count * occ), 128, smem, h->stream, p, L, tiles));
    if (tiles * 8 < p.batch) return launch_stage_generic_direct<STAGE>(h, stage_tail(p, tiles * 8));
    return SRI_OK;
}

// Tables of the DMMA kernels for row capacity R (16, 32 or 64; zero-filled by the caller): Stx [R][R] row-major =
// -1/2 S with g in the last column, and the stage operators S and -S_T as A fragments [R/8][R/4][32] with the boundary
// terms g and g_T as the last k index.
void dmma_tables(const sri_host::OperatorSet& ops, int M, int R, double* Stx, double* AS, double* AT) {
    const int KT = R / 4;
    for (int i = 0; i < M; ++i) {
        for (int j = 0; j < M; ++j) Stx[(size_t)i * R + j] = -0.5 * ops.S[j * M + i];
        Stx[(size_t)i * R + R - 1] = ops.g[i];
    }
    for (int mt = 0; mt < R / 8; ++mt)
        for (int kt = 0; kt < KT; ++kt)
            for (int lane = 0; lane < 32; ++lane) {
                const int i = 8 * mt + lane / 4, j = 4 * kt + lane % 4;
                double s = 0.0, t = 0.0;
                if (i < M && j < M) { s = ops.S[j * M + i]; t = -ops.ST[j * M + i]; }
                if (i < M && j == R - 1) { s = ops.g[i]; t = ops.gT[i]; }
                AS[(mt * KT + kt) * 32 + lane] = s;
                AT[(mt * KT + kt) * 32 + lane] = t;
            }
}

}  // namespace

// =================================================================================================================
//  C ABI
// =================================================================================================================

extern "C" {

const char* sri_last_error_string(void) { return g_last_error.c_str(); }
int64_t sri_kernel_launch_count(void) { return g_launches.load(); }

int sri_chebyshev_points(int N, double L, double* x) {
    if (N < 2 || !x) return fail(SRI_ERR_INVALID_ARGUMENT, "sri_chebyshev_points: need N >= 2 and x != NULL");
    sri_host::chebyshev_points(N, L, x);
    return SRI_OK;
}

int sri_chebyshev_coefficients(int N, double* c) {
    if (N < 2 || !c) return fail(SRI_ERR_INVALID_ARGUMENT, "sri_chebyshev_coefficients: need N >= 2 and c != NULL");
    sri_host::chebyshev_coefficients(N, c);
    return SRI_OK;
}

int sri_chebyshev_dn(int N, double* Dn) {
    if (N < 2 || !Dn) return fail(SRI_ERR_INVALID_ARGUMENT, "sri_chebyshev_dn: need N >= 2 and Dn != NULL");
    sri_host::chebyshev_dn(N, Dn);
    return SRI_OK;
}

int sri_phi(int na, int ne, double X, double begin, double end, double* out) {
    if (na < 1 || ne < 1 || !out || end == begin) return fail(SRI_ERR_INVALID_ARGUMENT, "sri_phi: bad arguments");
    const double x = (2 * X - (end + begin)) / (end - begin);
    const int cols = na * ne;
    std::memset(out, 0, sizeof(double) * na * cols);
    for (int k = 0; k < ne; ++k) {
        const double pk = sri_host::legendre(k, x);
        for (int a = 0; a < na; ++a) out[(a * ne + k) * na + a] = pk;
    }
    return SRI_OK;
}

int sri_create(int N, int device, sri_handle* out) {
    if (!out) return fail(SRI_ERR_INVALID_ARGUMENT, "sri_create: out == NULL");
    *out = nullptr;
    if (N < 2 || N > 64) return fail(SRI_ERR_UNSUPPORTED_N, "sri_create: N must be in [2, 64]");
    int ndev = 0;
    SRI_CUDA(cudaGetDeviceCount(&ndev));
    if (device < 0 || device >= ndev) return fail(SRI_ERR_CUDA, "sri_create: no such CUDA device (there is no CPU fallback)");
    sri_context* h = new (std::nothrow) sri_context();
    if (!h) return fail(SRI_ERR_ALLOC, "sri_create: out of host memory");
    h->N = N; h->M = N - 1; h->device = device;
    DeviceGuard guard;  // restores the caller's current device on every path out of this function
    const int rc = [&]() -> int {
    SRI_TRY(guard.enter(h));
    if (!h->ops.build(N)) return fail(SRI_ERR_INVALID_ARGUMENT, "sri_create: singular differentiation block");
    cudaDeviceProp prop;
    SRI_CUDA(cudaGetDeviceProperties(&prop, device));
    h->sm_count = prop.multiProcessorCount;
    SRI_CUDA(cudaStreamCreateWithFlags(&h->own_stream, cudaStreamNonBlocking));
    h->stream = h->own_stream;

    const int M = h->M;
    if (N <= 16) {
        using L = sri::OpsLayout16;
        std::vector<double> t(sri::StageTables::total, 0.0);
        for (int i = 0; i < M; ++i)
            for (int j = 0; j < M; ++j) {
                t[sri::StageTables::Srm + i * 16 + j] = h->ops.S[j * M + i];
                t[sri::StageTables::STrm + i * 16 + j] = h->ops.ST[j * M + i];
                t[sri::StageTables::STsh + i * 16 + j + 1] = h->ops.ST[j * M + i];
            }
        for (int j = 0; j < M; ++j) t[sri::StageTables::DTIsh + j + 1] = h->ops.D_TI[j];
        for (int j = 0; j < M; ++j)
            for (int i = 0; i < M; ++i) {
                t[L::St + j * sri::MP16 + i] = -0.5 * h->ops.S[j * M + i];
                t[L::Sp + j * sri::MP16 + i] = h->ops.S[j * M + i];
                t[L::STt + j * sri::MP16 + i] = h->ops.ST[j * M + i];
            }
        for (int i = 0; i < M; ++i) {
            t[L::g + i] = h->ops.g[i];
            t[L::gT + i] = h->ops.gT[i];
            t[L::DTI + i] = h->ops.D_TI[i];
            t[L::DnIN + i] = h->ops.Dn_IN[i];
        }
        t.resize(sri::DmmaTables::total, 0.0);
        dmma_tables(h->ops, M, 16, t.data() + sri::DmmaTables::Stx, t.data() + sri::DmmaTables::AS, t.data() + sri::DmmaTables::AT);
        SRI_CUDA(cudaMalloc(&h->d_ops16, sizeof(double) * sri::DmmaTables::total));
        SRI_CUDA(cudaMemcpy(h->d_ops16, t.data(), sizeof(double) * sri::DmmaTables::total, cudaMemcpyHostToDevice));
    } else {
        h->R = (M <= 31) ? 32 : 64;  // row capacity / table stride of the tiled kernel
        const sri::OpsLayoutGeneric L{h->R};
        std::vector<double> t(L.total(), 0.0);
        for (int j = 0; j < M; ++j)
            for (int i = 0; i < M; ++i) {
                t[L.Sp() + j * h->R + i] = h->ops.S[j * M + i];
                t[L.STt() + j * h->R + i] = h->ops.ST[j * M + i];
            }
        for (int i = 0; i < M; ++i) {
            t[L.g() + i] = h->ops.g[i];
            t[L.gT() + i] = h->ops.gT[i];
            t[L.DTI() + i] = h->ops.D_TI[i];
        }
        SRI_CUDA(cudaMalloc(&h->d_ops16, sizeof(double) * L.total()));
        SRI_CUDA(cudaMemcpy(h->d_ops16, t.data(), sizeof(double) * L.total(), cudaMemcpyHostToDevice));
        const int R = h->R;
        std::vector<double> t2((size_t)3 * R * R, 0.0);  // tables of the DMMA kernel
        dmma_tables(h->ops, M, R, t2.data(), t2.data() + (size_t)R * R, t2.data() + (size_t)2 * R * R);
        SRI_CUDA(cudaMalloc(&h->d_ops2, sizeof(double) * t2.size()));
        SRI_CUDA(cudaMemcpy(h->d_ops2, t2.data(), sizeof(double) * t2.size(), cudaMemcpyHostToDevice));
    }
    for (const FusedPass& k : {fused_first_pass(h), fused_second_pass(h)}) {
        int occ = 0;
        SRI_TRY(resident_ctas(h, k.kernel, k.threads, k.smem, &occ));
        if (occ < 1) return fail(SRI_ERR_CUDA, "sri_create: kernel does not fit on this device");
    }
    {
        std::vector<double> t(N);
        for (int i = 0; i < N; ++i) t[i] = 2 * h->ops.x[i] - 1;
        SRI_CUDA(cudaMalloc(&h->d_tnodes, sizeof(double) * N));
        SRI_CUDA(cudaMemcpy(h->d_tnodes, t.data(), sizeof(double) * N, cudaMemcpyHostToDevice));
        SRI_CUDA(cudaMalloc(&h->d_ptab, sizeof(double) * 8 * N));
        legendre_table_kernel<<<1, 64>>>(N, h->d_tnodes, h->d_ptab);
        SRI_CUDA(cudaGetLastError());
        SRI_CUDA(cudaDeviceSynchronize());
    }
    {
        std::vector<double> t((size_t)2 * M * M + M);   // D_TT, D_TI, D_TT^-1
        std::copy(h->ops.D_TT.begin(), h->ops.D_TT.end(), t.begin());
        std::copy(h->ops.D_TI.begin(), h->ops.D_TI.end(), t.begin() + (size_t)M * M);
        std::copy(h->ops.ST.begin(), h->ops.ST.end(), t.begin() + (size_t)M * M + M);
        SRI_CUDA(cudaMalloc(&h->d_dtt, sizeof(double) * t.size()));
        SRI_CUDA(cudaMemcpy(h->d_dtt, t.data(), sizeof(double) * t.size(), cudaMemcpyHostToDevice));
    }
    SRI_CUDA(cudaMalloc(&h->d_reduce, sizeof(double) * 2));
    {
        std::vector<double> w(N);
        sri_host::clenshaw_curtis_weights(N, w.data());
        SRI_CUDA(cudaMalloc(&h->d_ccw, sizeof(double) * N));
        SRI_CUDA(cudaMemcpy(h->d_ccw, w.data(), sizeof(double) * N, cudaMemcpyHostToDevice));
    }
    {
        const char* impl = std::getenv("SRI_FUSED16_IMPL");
        h->use_dmma = !(impl && std::strcmp(impl, "scalar") == 0);
        if (const char* si = std::getenv("SRI_STAGE_IMPL")) h->stage_impl = std::strcmp(si, "tma") == 0 ? 1 : (std::strcmp(si, "ldg") == 0 ? 2 : 0);
        if (const char* wi = std::getenv("SRI_WRENCH_IMPL")) h->wrench_impl = std::strcmp(wi, "blocked") == 0 ? 1 : (std::strcmp(wi, "generic") == 0 ? 2 : (std::strcmp(wi, "multi") == 0 ? 3 : (std::strcmp(wi, "warp") == 0 ? 4 : 0)));
        if (const char* ji = std::getenv("SRI_JACOBIAN_IMPL")) h->jac_impl = std::strcmp(ji, "scalar") == 0 ? 1 : 0;
        if (const char* gs = std::getenv("SRI_DMMA_GROWTH")) { const double gv = std::atof(gs); if (gv >= 0.0) h->dmma_growth = gv; }
    }
    return SRI_OK;
    }();
    if (rc != SRI_OK) {  // nothing allocated so far may leak: the context, its stream, the tables already uploaded
        const std::string keep = g_last_error;
        sri_destroy(h);
        g_last_error = keep;
        return rc;
    }
    *out = h;
    return SRI_OK;
}

int sri_destroy(sri_handle h) {
    if (!h) return SRI_OK;
    DeviceGuard guard;
    if (guard.enter(h) != SRI_OK) { delete h; return SRI_ERR_CUDA; }
    if (h->nccl_comm) sri_nccl_finalize(h);
    if (h->d_dnn) cudaFree(h->d_dnn);
    if (h->d_wrench_scratch) cudaFree(h->d_wrench_scratch);
    if (h->d_gather) cudaFree(h->d_gather);
    if (h->pipe_event) cudaEventDestroy(h->pipe_event);
    if (h->t0) cudaEventDestroy(h->t0);
    if (h->t1) cudaEventDestroy(h->t1);
    if (h->newton.host_state) cudaFreeHost(h->newton.host_state);
    for (cudaEvent_t e : h->newton.ev) if (e) cudaEventDestroy(e);
    if (h->d_ops16) cudaFree(h->d_ops16);
    if (h->d_ops2) cudaFree(h->d_ops2);
    if (h->d_tnodes) cudaFree(h->d_tnodes);
    if (h->d_dtt) cudaFree(h->d_dtt);
    if (h->d_reduce) cudaFree(h->d_reduce);
    if (h->d_ccw) cudaFree(h->d_ccw);
    if (h->d_ptab) cudaFree(h->d_ptab);
    if (h->d_jac) cudaFree(h->d_jac);
    if (h->d_dnin) cudaFree(h->d_dnin);
    if (h->d_partial) cudaFree(h->d_partial);
    if (h->d_counter) cudaFree(h->d_counter);
    if (h->newton.graph) cudaGraphExecDestroy(h->newton.graph);
    if (h->newton.block) cudaFree(h->newton.block);
    if (h->adjoint.block) cudaFree(h->adjoint.block);
    for (int sl = 0; sl < 5; ++sl)
        if (h->d_list[sl]) cudaFree(h->d_list[sl]);
    for (int sl = 0; sl < sri_context::kPipeSlots; ++sl) {
        for (int a = 0; a < sri_context::kPipeArrays; ++a)
            if (h->pipe_buf[sl][a]) cudaFree(h->pipe_buf[sl][a]);
        if (h->pipe_stream[sl]) cudaStreamDestroy(h->pipe_stream[sl]);
    }
    if (h->own_stream) cudaStreamDestroy(h->own_stream);
    delete h;
    return SRI_OK;
}

int sri_set_stream(sri_handle h, void* cuda_stream) {
    SRI_ENTER(h);
    h->stream = static_cast<cudaStream_t>(cuda_stream);
    return SRI_OK;
}

int sri_reset_stream(sri_handle h) {
    SRI_ENTER(h);
    h->stream = h->own_stream;
    return SRI_OK;
}

int sri_set_timing(sri_handle h, int enabled) {
    SRI_ENTER(h);
    if (enabled && !h->t0) {
        SRI_CUDA(cudaEventCreate(&h->t0));
        SRI_CUDA(cudaEventCreate(&h->t1));
    }
    h->timing = enabled != 0;
    h->timed_call = nullptr;
    return SRI_OK;
}

int sri_get_last_timing(sri_handle h, float* ms, const char** entry_point) {
    if (!h || !ms) return fail(SRI_ERR_INVALID_ARGUMENT, "sri_get_last_timing: null argument");
    DeviceGuard guard;
    SRI_TRY(guard.enter(h));
    if (!h->timing || !h->timed_call) return fail(SRI_ERR_INVALID_ARGUMENT, "sri_get_last_timing: no timed call yet (sri_set_timing(h, 1) first)");
    SRI_CUDA(cudaEventSynchronize(h->t1));
    SRI_CUDA(cudaEventElapsedTime(ms, h->t0, h->t1));
    if (entry_point) *entry_point = h->timed_call;
    return SRI_OK;
}

int sri_synchronize(sri_handle h) {
    SRI_ENTER(h);
    SRI_CUDA(cudaStreamSynchronize(h->stream));
    return SRI_OK;
}

int sri_get_N(sri_handle h, int* N) {
    if (!h || !N) return fail(SRI_ERR_INVALID_ARGUMENT, "sri_get_N: null argument");
    *N = h->N;
    return SRI_OK;
}

int sri_get_operator(sri_handle h, int which, double* out) {
    if (!h || !out) return fail(SRI_ERR_INVALID_ARGUMENT, "sri_get_operator: null argument");
    const std::vector<double>* src = nullptr;
    switch (which) {
        case 0: src = &h->ops.Dn; break;
        case 1: src = &h->ops.Dn_NN; break;
        case 2: src = &h->ops.Dn_IN; break;
        case 3: src = &h->ops.S; break;
        case 4: src = &h->ops.D_TT; break;
        case 5: src = &h->ops.D_TI; break;
        case 6: src = &h->ops.ST; break;
        default: return fail(SRI_ERR_INVALID_ARGUMENT, "sri_get_operator: which must be 0..6");
    }
    std::memcpy(out, src->data(), sizeof(double) * src->size());
    return SRI_OK;
}

// device pointers, handle's device current
static int strain_from_modes_dev(sri_context* h, int64_t batch, int ne, const double* dqe, double* dK) {
    if (ne <= 8) {
        const long long rows = (long long)batch * 3;
        const int per_cta = h->N <= 16 ? 16 : (h->N <= 32 ? 8 : 4);  // rows per CTA of 256 threads
        auto* kernel = h->N <= 16 ? strain_from_modes_table_kernel<16> : (h->N <= 32 ? strain_from_modes_table_kernel<32> : strain_from_modes_table_kernel<64>);
        return launch(kernel, (unsigned)((rows + per_cta - 1) / per_cta), 256, 0, h->stream, rows, h->N, ne, h->d_ptab, dqe, dK, h->skip);
    }
    const long long total = (long long)batch * 3 * h->N;
    return launch(strain_from_modes_kernel, (unsigned)((total + 255) / 256), 256, 0, h->stream, batch, h->N, ne, h->d_tnodes, dqe, dK, h->skip);
}

int sri_strain_from_modes(sri_handle h, int64_t batch, int ne, const double* qe, double* K) {
    SRI_ENTER(h);
    if (batch < 0 || ne < 1 || (batch > 0 && (!qe || !K))) return fail(SRI_ERR_INVALID_ARGUMENT, "sri_strain_from_modes: bad arguments");
    if (batch == 0) return SRI_OK;
    Staging st(h);
    const double* dqe; double* dK;
    SRI_TRY(st.in(qe, (size_t)batch * 3 * ne, &dqe));
    SRI_TRY(st.out(K, (size_t)batch * 3 * h->N, &dK));
    SRI_TRY(strain_from_modes_dev(h, batch, ne, dqe, dK));
    return st.finish();
}

int sri_scale_for_length(sri_handle h, int64_t batch, const double* length, double uniform_length, double* K, double* Gamma,
                         double* fbar, double* lbar) {
    SRI_ENTER(h);
    if (batch < 0) return fail(SRI_ERR_INVALID_ARGUMENT, "sri_scale_for_length: negative batch");
    if (batch == 0) return SRI_OK;
    const int per_rod = 3 * h->N;
    Staging st(h);
    const double* dl = nullptr;
    SRI_TRY(st.in(length, (size_t)batch, &dl));
    double* arr[4] = {K, Gamma, fbar, lbar};
    double* dev[4] = {nullptr, nullptr, nullptr, nullptr};
    for (int i = 0; i < 4; ++i) {
        if (!arr[i]) continue;
        if (is_device_pointer(arr[i])) { dev[i] = arr[i]; continue; }
        const double* in = nullptr;   // host array: in-out through a staged copy
        SRI_TRY(st.in(arr[i], (size_t)batch * per_rod, &in));
        dev[i] = const_cast<double*>(in);
        st.copy_back(arr[i], dev[i], (size_t)batch * per_rod * sizeof(double));
    }
    const long long total = (long long)batch * per_rod;
    SRI_TRY(launch(scale_for_length_kernel, (unsigned)std::min<long long>((total + 255) / 256, (long long)h->sm_count * 16), 256, 0,
                   h->stream, batch, per_rod, dl, uniform_length, dev[0], dev[1], dev[2], dev[3]));
    return st.finish();
}

int sri_assemble_A(sri_handle h, int64_t batch, const double* K, double* A_NN) {
    SRI_ENTER(h);
    if (batch < 0 || (batch > 0 && (!K || !A_NN))) return fail(SRI_ERR_INVALID_ARGUMENT, "sri_assemble_A: bad arguments");
    if (batch == 0) return SRI_OK;
    const int N = h->N, M = h->M, n = 4 * M;
    if (!h->d_dnn) {
        SRI_CUDA(cudaMalloc(&h->d_dnn, sizeof(double) * M * M));
        SRI_CUDA(cudaMemcpy(h->d_dnn, h->ops.Dn_NN.data(), sizeof(double) * M * M, cudaMemcpyHostToDevice));
    }
    Staging st(h);
    const double* dK; double* dA;
    SRI_TRY(st.in(K, (size_t)batch * 3 * N, &dK));
    SRI_TRY(st.out(A_NN, (size_t)batch * n * n, &dA));
    SRI_TRY(launch(assemble_A_kernel, (unsigned)std::min<long long>(batch, (long long)h->sm_count * 8), 256, 0, h->stream, batch, N, h->d_dnn, dK, dA));
    return st.finish();
}

int sri_integrate_all(sri_handle h, const sri_rod_batch* rods) {
    SRI_ENTER(h);
    if (!rods) return fail(SRI_ERR_INVALID_ARGUMENT, "sri_integrate_all: rods == NULL");
    const int64_t B = rods->batch;
    if (B < 0) return fail(SRI_ERR_INVALID_ARGUMENT, "sri_integrate_all: negative batch");
    if (B == 0) return SRI_OK;
    if (!rods->K) return fail(SRI_ERR_INVALID_ARGUMENT, "sri_integrate_all: K is required");
    if ((rods->n || rods->m) && !rods->F_tip) return fail(SRI_ERR_INVALID_ARGUMENT, "sri_integrate_all: F_tip is required for n/m");
    if (rods->m && !rods->M_tip) return fail(SRI_ERR_INVALID_ARGUMENT, "sri_integrate_all: M_tip is required for m");
    const int N = h->N, M = h->M;
    if (all_host_pointers(rods)) return integrate_all_host_pipeline(h, rods);
    Staging st(h);
    sri::FusedParams p{};
    p.batch = B; p.N = N; p.M = M; p.ops = h->d_ops16;
    SRI_TRY(st.in(rods->K, (size_t)B * 3 * N, &p.K));
    SRI_TRY(st.in(rods->q0, (size_t)B * 4, &p.q0));
    SRI_TRY(st.in(rods->r0, (size_t)B * 3, &p.r0));
    SRI_TRY(st.in(rods->Gamma, (size_t)B * 3 * N, &p.Gamma));
    SRI_TRY(st.in(rods->fbar, (size_t)B * 3 * N, &p.fbar));
    SRI_TRY(st.in(rods->lbar, (size_t)B * 3 * N, &p.lbar));
    SRI_TRY(st.in(rods->F_tip, (size_t)B * 3, &p.F_tip));
    SRI_TRY(st.in(rods->M_tip, (size_t)B * 3, &p.M_tip));
    SRI_TRY(st.out(rods->Q, (size_t)B * 4 * M, &p.Q));
    SRI_TRY(st.out(rods->r, (size_t)B * 3 * M, &p.r));
    SRI_TRY(st.out(rods->n, (size_t)B * 3 * M, &p.n));
    SRI_TRY(st.out(rods->m, (size_t)B * 3 * M, &p.m));
    SRI_TRY(st.out(rods->info, (size_t)B, &p.info));
    SRI_TRY(launch_fused(h, p));
    SRI_TRY(st.finish());
    if (rods->info && !is_device_pointer(rods->info)) return singular_status(rods->info, B, "sri_integrate_all");
    return SRI_OK;
}

int sri_integrate_quaternions(sri_handle h, int64_t batch, const double* K, const double* q0, double* Q, int* info) {
    SRI_ENTER(h);  // (its own NVTX range and timer; the nested sri_integrate_all does not time again)
    if (batch > 0 && !Q) return fail(SRI_ERR_INVALID_ARGUMENT, "sri_integrate_quaternions: Q == NULL");
    sri_rod_batch rb{};
    rb.batch = batch; rb.K = K; rb.q0 = q0; rb.Q = Q; rb.info = info;
    return sri_integrate_all(h, &rb);
}

int sri_integrate_position(sri_handle h, int64_t batch, const double* Q, const double* Gamma, const double* r0, double* r) {
    SRI_ENTER(h);
    if (batch < 0 || (batch > 0 && (!Q || !r))) return fail(SRI_ERR_INVALID_ARGUMENT, "sri_integrate_position: bad arguments");
    if (batch == 0) return SRI_OK;
    const int N = h->N, M = h->M;
    Staging st(h);
    sri::FusedParams p{};
    p.batch = batch; p.N = N; p.M = M; p.ops = h->d_ops16;
    SRI_TRY(st.in(Q, (size_t)batch * 4 * M, &p.Qin));
    SRI_TRY(st.in(Gamma, (size_t)batch * 3 * N, &p.Gamma));
    SRI_TRY(st.in(r0, (size_t)batch * 3, &p.r0));
    SRI_TRY(st.out(r, (size_t)batch * 3 * M, &p.r));
    if (h->R == 0) SRI_TRY(launch_stage<sri::kStagePosition>(h, p));
    else SRI_TRY(launch_stage_generic<sri::kStagePosition>(h, p));
    return st.finish();
}

int sri_integrate_stress(sri_handle h, int64_t batch, const double* fbar, const double* F_tip, double* n) {
    SRI_ENTER(h);
    if (batch < 0 || (batch > 0 && (!F_tip || !n))) return fail(SRI_ERR_INVALID_ARGUMENT, "sri_integrate_stress: bad arguments");
    if (batch == 0) return SRI_OK;
    const int N = h->N, M = h->M;
    Staging st(h);
    sri::FusedParams p{};
    p.batch = batch; p.N = N; p.M = M; p.ops = h->d_ops16;
    SRI_TRY(st.in(fbar, (size_t)batch * 3 * N, &p.fbar));
    SRI_TRY(st.in(F_tip, (size_t)batch * 3, &p.F_tip));
    SRI_TRY(st.out(n, (size_t)batch * 3 * M, &p.n));
    if (!p.fbar) {
        // no distributed load: n_i = gT_i F_tip, a pure streaming write (one 2 KB tile per warp and pass, 128-bit streaming stores)
        const long long total = (long long)batch * 3 * M, chunks = (total + 255) / 256 * 32;  // 32 lanes per 2 KB tile
        const double* gT = h->d_ops16 + (h->R == 0 ? sri::OpsLayout16::gT : sri::OpsLayoutGeneric{h->R}.gT());
        const bool aligned = (reinterpret_cast<uintptr_t>(p.n) & 15u) == 0;
        SRI_TRY(launch(sri::stress_noload_kernel, (unsigned)std::min<long long>((chunks + 255) / 256, (long long)h->sm_count * 8), 256, 0,
                       h->stream, total, M, gT, p.F_tip, p.n, aligned ? 1 : 0));
    } else if (h->R == 0) {
        SRI_TRY(launch_stage<sri::kStageStress>(h, p));
    } else {
        SRI_TRY(launch_stage_generic<sri::kStageStress>(h, p));
    }
    return st.finish();
}

int sri_integrate_couple(sri_handle h, int64_t batch, const double* Q, const double* q0, const double* Gamma,
                         const double* n, const double* lbar, const double* M_tip, double* m) {
    SRI_ENTER(h);
    if (batch < 0 || (batch > 0 && (!Q || !n || !M_tip || !m))) return fail(SRI_ERR_INVALID_ARGUMENT, "sri_integrate_couple: bad arguments");
    if (batch == 0) return SRI_OK;
    const int N = h->N, M = h->M;
    Staging st(h);
    sri::FusedParams p{};
    p.batch = batch; p.N = N; p.M = M; p.ops = h->d_ops16;
    SRI_TRY(st.in(Q, (size_t)batch * 4 * M, &p.Qin));
    SRI_TRY(st.in(q0, (size_t)batch * 4, &p.q0));
    SRI_TRY(st.in(Gamma, (size_t)batch * 3 * N, &p.Gamma));
    SRI_TRY(st.in(n, (size_t)batch * 3 * M, &p.nin));
    SRI_TRY(st.in(lbar, (size_t)batch * 3 * N, &p.lbar));
    SRI_TRY(st.in(M_tip, (size_t)batch * 3, &p.M_tip));
    p.F_tip = p.M_tip;  // unused when nin is given; keeps the pointer valid
    SRI_TRY(st.out(m, (size_t)batch * 3 * M, &p.m));
    if (h->R == 0) SRI_TRY(launch_stage<sri::kStageCouple>(h, p));
    else SRI_TRY(launch_stage_generic<sri::kStageCouple>(h, p));
    return st.finish();
}

int sri_shape_residual(sri_handle h, int64_t batch, const double* K, const double* K0, const double* H_diag,
                       const double* Q, const double* q0, const double* m, const double* M_tip, double* rho,
                       double* norm2_and_max) {
    SRI_ENTER(h);
    if (batch < 0 || (batch > 0 && (!K || !H_diag || !Q || !m || !M_tip))) return fail(SRI_ERR_INVALID_ARGUMENT, "sri_shape_residual: bad arguments");
    if (batch == 0) return SRI_OK;
    const int N = h->N, M = h->M;
    double H[3];
    SRI_TRY(read_H(H_diag, H));
    Staging st(h);
    const double *dK, *dK0, *dQ, *dq0, *dm, *dMt; double* drho; double* dred = nullptr;
    SRI_TRY(st.in(K, (size_t)batch * 3 * N, &dK));
    SRI_TRY(st.in(K0, (size_t)batch * 3 * N, &dK0));
    SRI_TRY(st.in(Q, (size_t)batch * 4 * M, &dQ));
    SRI_TRY(st.in(q0, (size_t)batch * 4, &dq0));
    SRI_TRY(st.in(m, (size_t)batch * 3 * M, &dm));
    SRI_TRY(st.in(M_tip, (size_t)batch * 3, &dMt));
    SRI_TRY(st.out(rho, (size_t)batch * 3 * N, &drho));
    if (norm2_and_max) {
        SRI_TRY(st.out(norm2_and_max, 2, &dred));
        SRI_CUDA(cudaMemsetAsync(dred, 0, 2 * sizeof(double), h->stream));
    }
    const long long total = (long long)batch * N;
    SRI_TRY(launch(shape_residual_kernel, (unsigned)((total + 255) / 256), 256, 0, h->stream, batch, N, dK, dK0, H[0], H[1], H[2], dQ, dq0,
                   dm, dMt, drho, dred));
    return st.finish();
}

int sri_wrench_local(sri_handle h, int64_t batch, const double* Q, const double* q0, const double* n, const double* m,
                     const double* F_tip, const double* M_tip, double* Lambda) {
    SRI_ENTER(h);
    if (batch < 0 || (batch > 0 && (!Q || !n || !m || !F_tip || !M_tip || !Lambda))) return fail(SRI_ERR_INVALID_ARGUMENT, "sri_wrench_local: bad arguments");
    if (batch == 0) return SRI_OK;
    const int N = h->N, M = h->M;
    Staging st(h);
    const double *dQ, *dq0, *dn, *dm, *dF, *dMt; double* dL;
    SRI_TRY(st.in(Q, (size_t)batch * 4 * M, &dQ));
    SRI_TRY(st.in(q0, (size_t)batch * 4, &dq0));
    SRI_TRY(st.in(n, (size_t)batch * 3 * M, &dn));
    SRI_TRY(st.in(m, (size_t)batch * 3 * M, &dm));
    SRI_TRY(st.in(F_tip, (size_t)batch * 3, &dF));
    SRI_TRY(st.in(M_tip, (size_t)batch * 3, &dMt));
    SRI_TRY(st.out(Lambda, (size_t)batch * 6 * N, &dL));
    const long long total = (long long)batch * N;
    SRI_TRY(launch(wrench_local_kernel, (unsigned)((total + 255) / 256), 256, 0, h->stream, batch, N, dQ, dq0, dn, dm, dF, dMt, dL));
    return st.finish();
}

// one rod per CTA of NW warps (csrc/sri_wrench_gj_multi.cuh); grid = min(batch, resident CTAs)
extern "C++" {
namespace {
template <int NW, int WMAX, int MINB>
int launch_wrench_gjm(sri_context* h, const sri::WrenchParams& p, int64_t batch) {
    using C = sri::WrenchGjMultiCfg<NW, WMAX>;
    static_assert(C::NODES <= 33, "node capacity");
    auto* kern = sri::wrench_local_solve_gj_multi_kernel<NW, WMAX, MINB>;
    int occ = 0;
    SRI_TRY(resident_ctas(h, kern, 32 * NW, C::smem_bytes, &occ));
    if (occ < 1) return fail(SRI_ERR_CUDA, "sri_integrate_wrench_local: kernel does not fit on this device");
    return launch(kern, (int)std::min<long long>(batch, (long long)h->sm_count * occ), 32 * NW, C::smem_bytes, h->stream, p);
}
template <int NW, int WMAX, int MINB>
int launch_wrench_gjs(sri_context* h, const sri::WrenchParams& p, int64_t batch) {
    using C = sri::WrenchGjStaticCfg<NW, WMAX>;
    auto* kern = sri::wrench_local_solve_gj_static_kernel<NW, WMAX, MINB>;
    int occ = 0;
    SRI_TRY(resident_ctas(h, kern, 32 * NW, C::smem_bytes, &occ));
    if (occ < 1) return fail(SRI_ERR_CUDA, "sri_integrate_wrench_local: kernel does not fit on this device");
    return launch(kern, (int)std::min<long long>(batch, (long long)h->sm_count * occ), 32 * NW, C::smem_bytes, h->stream, p);
}
}  // namespace
}  // extern "C++"

int sri_integrate_wrench_local(sri_handle h, int64_t batch, const double* K, const double* Q, const double* q0,
                               const double* Gamma, const double* fbar, const double* lbar, const double* F_tip,
                               const double* M_tip, double* Lambda, int* info) {
    SRI_ENTER(h);
    if (batch < 0 || (batch > 0 && (!K || !Q || !F_tip || !M_tip || !Lambda))) return fail(SRI_ERR_INVALID_ARGUMENT, "sri_integrate_wrench_local: bad arguments");
    if (batch == 0) return SRI_OK;
    const int N = h->N, M = h->M;
    Staging st(h);
    sri::WrenchParams p{};
    p.batch = batch; p.N = N; p.M = M; p.D_TT = h->d_dtt; p.D_TI = h->d_dtt + (size_t)M * M;
    SRI_TRY(st.in(K, (size_t)batch * 3 * N, &p.K));
    SRI_TRY(st.in(Q, (size_t)batch * 4 * M, &p.Q));
    SRI_TRY(st.in(q0, (size_t)batch * 4, &p.q0));
    SRI_TRY(st.in(Gamma, (size_t)batch * 3 * N, &p.Gamma));
    SRI_TRY(st.in(fbar, (size_t)batch * 3 * N, &p.fbar));
    SRI_TRY(st.in(lbar, (size_t)batch * 3 * N, &p.lbar));
    SRI_TRY(st.in(F_tip, (size_t)batch * 3, &p.F_tip));
    SRI_TRY(st.in(M_tip, (size_t)batch * 3, &p.M_tip));
    SRI_TRY(st.out(Lambda, (size_t)batch * 6 * N, &p.Lambda));
    SRI_TRY(st.out(info, (size_t)batch, &p.info));
    // N = 17 and 23 <= N <= 33 (where it is measured faster: DESIGN 2.4), default: static-order Gauss-Jordan on the operator
    // preconditioned by the cached D_TT^-1 (one row per lane, one rod per CTA of 2-3 warps), growth-checked; the rods it hands
    // back are re-solved with partial pivoting by the second pass
    const bool two_pass = h->wrench_impl == 0 && (N == 17 || (N >= 23 && N <= 33));
    if (two_pass) {
        SRI_TRY(handback_list(h, 4, batch, h->stream, p));
        p.S = h->d_dtt + (size_t)M * M + M;
        {
            const double g = h->dmma_growth;
            long long bits; std::memcpy(&bits, &g, sizeof bits);
            p.growth_hi = g > 0.0 ? (int)(bits >> 32) : -1;   // (bound 0: every rod goes to the row-pivoting pass)
        }
        if (N == 17) SRI_TRY((launch_wrench_gjs<2, 48, 6>(h, p, batch)));
        else SRI_TRY((launch_wrench_gjs<3, 96, 1>(h, p, batch)));
        p.from_list = 1;   // second pass: CTAs without work exit at once
    }
    // row-pivoting kernels: register-resident rolled Gauss-Jordan, one row per lane over 1-3 warps, or (12 <= N <= 16, where it
    // is faster) two rows per lane in one warp
    if ((h->wrench_impl == 0 || h->wrench_impl == 3) && N <= 11) {
        SRI_TRY((launch_wrench_gjm<1, 32, 16>(h, p, batch)));
    } else if ((h->wrench_impl == 3 && N <= 17) || (h->wrench_impl == 0 && N == 17)) {
        SRI_TRY((launch_wrench_gjm<2, 48, 6>(h, p, batch)));
    } else if (N > 16 && N <= 33 && h->wrench_impl != 2) {
        if (N <= 22) SRI_TRY((launch_wrench_gjm<2, 64, 5>(h, p, batch)));
        else SRI_TRY((launch_wrench_gjm<3, 96, 1>(h, p, batch)));
    } else if (N > 16) {
        // one rod per CTA, dense 3M x 3M operator in shared memory while it fits (N <= 55), else in an L2-resident scratch
        const int n = 3 * M, ld = n | 1;
        sri::WrenchGenLayout L{n, ld, N, true};
        bool in_smem = (size_t)L.total() * sizeof(double) <= 227 * 1024;
        if (!in_smem) L.in_smem = false;
        const size_t smem = (size_t)L.total() * sizeof(double);
        int occ = 0;
        SRI_TRY(resident_ctas(h, sri::wrench_local_solve_generic_kernel, sri::kWrenchGenThreads, smem, &occ));
        if (occ < 1) return fail(SRI_ERR_CUDA, "sri_integrate_wrench_local: kernel does not fit on this device");
        const long long capg = (long long)h->sm_count * occ;
        const int grid = (int)(batch < capg ? batch : capg);
        if (!in_smem) {
            const size_t need = (size_t)grid * n * ld * sizeof(double);
            if (h->wrench_scratch_cap < need) {
                SRI_CUDA(cudaStreamSynchronize(h->stream));
                if (h->d_wrench_scratch) SRI_CUDA(cudaFree(h->d_wrench_scratch));
                h->d_wrench_scratch = nullptr; h->wrench_scratch_cap = 0;
                SRI_CUDA(cudaMalloc(&h->d_wrench_scratch, (size_t)capg * n * ld * sizeof(double)));
                h->wrench_scratch_cap = (size_t)capg * n * ld * sizeof(double);
            }
        }
        SRI_TRY(launch(sri::wrench_local_solve_generic_kernel, grid, sri::kWrenchGenThreads, smem, h->stream, p, h->d_wrench_scratch, in_smem ? 1 : 0));
    } else if (h->wrench_impl != 1) {
        // one rod per warp, the whole operator in registers: rolled Gauss-Jordan with implicit partial pivoting
        int occ = 0;
        SRI_TRY(resident_ctas(h, sri::wrench_local_solve_gj_kernel, 32 * sri::kWrenchGjWarps, sri::kWrenchGjSmem, &occ));
        if (occ < 1) return fail(SRI_ERR_CUDA, "sri_integrate_wrench_local: kernel does not fit on this device");
        const long long want = (batch + sri::kWrenchGjWarps - 1) / sri::kWrenchGjWarps;
        SRI_TRY(launch(sri::wrench_local_solve_gj_kernel, (int)std::min(want, (long long)h->sm_count * occ), 32 * sri::kWrenchGjWarps,
                       sri::kWrenchGjSmem, h->stream, p));
    } else {
        SRI_TRY(ensure_dynamic_smem(sri::wrench_local_solve_kernel, h->device, sri::kWrenchSmem));
        const long long want = (batch + sri::kWrenchWarps - 1) / sri::kWrenchWarps;
        // one CTA of 8 warps per SM (24 KB of shared memory per rod)
        SRI_TRY(launch(sri::wrench_local_solve_kernel, (int)std::min(want, (long long)h->sm_count), 32 * sri::kWrenchWarps, sri::kWrenchSmem, h->stream, p));
    }
    SRI_TRY(st.finish());
    if (info && !is_device_pointer(info)) return singular_status(info, batch, "sri_integrate_wrench_local");
    return SRI_OK;
}

// device pointers, H on the host, handle's device current
static int galerkin_residual_dev(sri_context* h, int64_t batch, int ne, const double* dK, const double* dK0, const double* H,
                                 const double* dQ, const double* dq0, const double* dm, const double* dMt, double* dg,
                                 double* dred) {
    const int N = h->N;
    const int G = N <= 16 ? 16 : 32;
    const long long chunks = ((long long)batch * G + 255) / 256;
    const long long blocks = std::min<long long>(chunks, (long long)h->sm_count * 4);  // persistent: 4 resident blocks per SM
    if (dred) {
        if (!h->d_counter) {
            SRI_CUDA(cudaMalloc(&h->d_counter, sizeof(unsigned)));
            SRI_CUDA(cudaMemset(h->d_counter, 0, sizeof(unsigned)));
        }
        if ((size_t)blocks > h->partial_cap) {  // (grows outside stream capture: the first, eager call of a shape sizes it)
            size_t cap = h->partial_cap ? h->partial_cap : 4096;
            while (cap < (size_t)blocks) cap *= 2;
            SRI_CUDA(cudaStreamSynchronize(h->stream));
            if (h->d_partial) SRI_CUDA(cudaFree(h->d_partial));
            h->d_partial = nullptr; h->partial_cap = 0;
            SRI_CUDA(cudaMalloc(&h->d_partial, cap * 2 * sizeof(double)));
            h->partial_cap = cap;
        }
    }
    auto* kernel = G == 16 ? galerkin_residual_kernel<16, 8> : galerkin_residual_kernel<32, 8>;
    switch (ne) {
#define SRI_GALERKIN(NE_) case NE_: kernel = G == 16 ? galerkin_residual_kernel<16, NE_> : galerkin_residual_kernel<32, NE_>; break;
        SRI_GALERKIN(1) SRI_GALERKIN(2) SRI_GALERKIN(3) SRI_GALERKIN(4) SRI_GALERKIN(5) SRI_GALERKIN(6) SRI_GALERKIN(7)
#undef SRI_GALERKIN
    }
    return launch(kernel, (unsigned)blocks, 256, 0, h->stream, batch, N, h->d_ptab, h->d_ccw, dK, dK0, H[0], H[1], H[2], dQ, dq0, dm,
                  dMt, dg, h->d_partial, h->d_counter, dred, h->skip);
}

int sri_galerkin_residual(sri_handle h, int64_t batch, int ne, const double* K, const double* K0, const double* H_diag,
                          const double* Q, const double* q0, const double* m, const double* M_tip, double* g,
                          double* norm2_and_max) {
    SRI_ENTER(h);
    if (batch < 0 || ne < 1 || ne > 8 || (batch > 0 && (!K || !H_diag || !Q || !m || !M_tip || !g)))
        return fail(SRI_ERR_INVALID_ARGUMENT, "sri_galerkin_residual: bad arguments (1 <= ne <= 8)");
    if (batch == 0) return SRI_OK;
    const int N = h->N, M = h->M;
    double H[3];
    SRI_TRY(read_H(H_diag, H));
    Staging st(h);
    const double *dK, *dK0, *dQ, *dq0, *dm, *dMt; double* dg; double* dred = nullptr;
    SRI_TRY(st.in(K, (size_t)batch * 3 * N, &dK));
    SRI_TRY(st.in(K0, (size_t)batch * 3 * N, &dK0));
    SRI_TRY(st.in(Q, (size_t)batch * 4 * M, &dQ));
    SRI_TRY(st.in(q0, (size_t)batch * 4, &dq0));
    SRI_TRY(st.in(m, (size_t)batch * 3 * M, &dm));
    SRI_TRY(st.in(M_tip, (size_t)batch * 3, &dMt));
    SRI_TRY(st.out(g, (size_t)batch * 3 * ne, &dg));
    if (norm2_and_max) SRI_TRY(st.out(norm2_and_max, 2, &dred));
    SRI_TRY(galerkin_residual_dev(h, batch, ne, dK, dK0, H, dQ, dq0, dm, dMt, dg, dred));
    return st.finish();
}

extern "C++" {
namespace {
// the instantiation <G, ne> (1 <= ne <= 8) of one of the per-rod lane-group kernels, G = 16 for N <= 16, else 32
template <template <int, int> class Pick>
auto pick_lanes_ne(int N, int ne) {
    const bool g16 = N <= 16;
    switch (ne) {
#define SRI_PICK(NE_) case NE_: return g16 ? Pick<16, NE_>::get() : Pick<32, NE_>::get();
        SRI_PICK(1) SRI_PICK(2) SRI_PICK(3) SRI_PICK(4) SRI_PICK(5) SRI_PICK(6) SRI_PICK(7)
#undef SRI_PICK
        default: return g16 ? Pick<16, 8>::get() : Pick<32, 8>::get();
    }
}
template <int G, int NE> struct PickResidualVjp { static auto get() { return galerkin_residual_vjp_kernel<G, NE>; } };
template <int G, int NE> struct PickAdjointRefine { static auto get() { return static_adjoint_refine_kernel<G, NE>; } };
}  // namespace
}  // extern "C++"

// persistent grid of the lane-group kernels: 256 threads, at most 4 resident blocks per SM
static unsigned lane_group_blocks(const sri_context* h, int64_t batch) {
    const int G = h->N <= 16 ? 16 : 32;
    const long long chunks = ((long long)batch * G + 255) / 256;
    return (unsigned)std::min<long long>(chunks, (long long)h->sm_count * 4);
}

// device pointers, H on the host, handle's device current
static int galerkin_residual_vjp_dev(sri_context* h, int64_t batch, int ne, const double* dK, const double* dK0, const double* H,
                                     const double* dQ, const double* dq0, const double* dm, const double* dMt, const double* dgg,
                                     double* gK, double* gK0, double* gH, double* gQ, double* gq0, double* gm, double* gMt) {
    return launch(pick_lanes_ne<PickResidualVjp>(h->N, ne), lane_group_blocks(h, batch), 256, 0, h->stream, batch, h->N, h->d_ptab,
                  h->d_ccw, dK, dK0, H[0], H[1], H[2], dQ, dq0, dm, dMt, dgg, gK, gK0, gH, gQ, gq0, gm, gMt);
}

int sri_galerkin_residual_vjp(sri_handle h, int64_t batch, int ne, const double* K, const double* K0, const double* H_diag,
                              const double* Q, const double* q0, const double* m, const double* M_tip, const double* gg,
                              double* gK, double* gK0, double* gH, double* gQ, double* gq0, double* gm, double* gM_tip) {
    SRI_ENTER(h);
    if (batch < 0 || ne < 1 || ne > 8 || !H_diag || (batch > 0 && (!K || !Q || !m || !M_tip || !gg)))
        return fail(SRI_ERR_INVALID_ARGUMENT, "sri_galerkin_residual_vjp: bad arguments (1 <= ne <= 8)");
    if (batch == 0) return SRI_OK;
    const int N = h->N, M = h->M;
    double H[3];
    SRI_TRY(read_H(H_diag, H));
    Staging st(h);
    const double *dK, *dK0, *dQ, *dq0, *dm, *dMt, *dgg;
    double *dgK, *dgK0, *dgH, *dgQ, *dgq0, *dgm, *dgMt;
    SRI_TRY(st.in(K, (size_t)batch * 3 * N, &dK));
    SRI_TRY(st.in(K0, (size_t)batch * 3 * N, &dK0));
    SRI_TRY(st.in(Q, (size_t)batch * 4 * M, &dQ));
    SRI_TRY(st.in(q0, (size_t)batch * 4, &dq0));
    SRI_TRY(st.in(m, (size_t)batch * 3 * M, &dm));
    SRI_TRY(st.in(M_tip, (size_t)batch * 3, &dMt));
    SRI_TRY(st.in(gg, (size_t)batch * 3 * ne, &dgg));
    SRI_TRY(st.out(gK, (size_t)batch * 3 * N, &dgK));
    SRI_TRY(st.out(gK0, (size_t)batch * 3 * N, &dgK0));
    SRI_TRY(st.out(gH, (size_t)batch * 3, &dgH));
    SRI_TRY(st.out(gQ, (size_t)batch * 4 * M, &dgQ));
    SRI_TRY(st.out(gq0, (size_t)batch * 4, &dgq0));
    SRI_TRY(st.out(gm, (size_t)batch * 3 * M, &dgm));
    SRI_TRY(st.out(gM_tip, (size_t)batch * 3, &dgMt));
    SRI_TRY(galerkin_residual_vjp_dev(h, batch, ne, dK, dK0, H, dQ, dq0, dm, dMt, dgg, dgK, dgK0, dgH, dgQ, dgq0, dgm, dgMt));
    return st.finish();
}

int sri_project_onto_modes(sri_handle h, int64_t batch, int ne, const double* f, double* out) {
    SRI_ENTER(h);
    if (batch < 0 || ne < 1 || ne > 8 || (batch > 0 && (!f || !out))) return fail(SRI_ERR_INVALID_ARGUMENT, "sri_project_onto_modes: bad arguments (1 <= ne <= 8)");
    if (batch == 0) return SRI_OK;
    Staging st(h);
    const double* df; double* dout;
    SRI_TRY(st.in(f, (size_t)batch * 3 * h->N, &df));
    SRI_TRY(st.out(out, (size_t)batch * 3 * ne, &dout));
    const long long total = (long long)batch * 3;
    SRI_TRY(launch(project_onto_modes_kernel, (unsigned)((total + 127) / 128), 128, 0, h->stream, batch, h->N, ne, 3LL * h->N, 1.0,
                   h->d_ptab, h->d_ccw, df, dout));
    return st.finish();
}

int sri_generalised_forces(sri_handle h, int64_t batch, int ne, const double* Lambda, double* Qad) {
    SRI_ENTER(h);
    if (batch < 0 || ne < 1 || ne > 8 || (batch > 0 && (!Lambda || !Qad))) return fail(SRI_ERR_INVALID_ARGUMENT, "sri_generalised_forces: bad arguments (1 <= ne <= 8)");
    if (batch == 0) return SRI_OK;
    Staging st(h);
    const double* dL; double* dout;
    SRI_TRY(st.in(Lambda, (size_t)batch * 6 * h->N, &dL));
    SRI_TRY(st.out(Qad, (size_t)batch * 3 * ne, &dout));
    const long long total = (long long)batch * 3;
    SRI_TRY(launch(project_onto_modes_kernel, (unsigned)((total + 127) / 128), 128, 0, h->stream, batch, h->N, ne, 6LL * h->N, -1.0,
                   h->d_ptab, h->d_ccw, dL, dout));
    return st.finish();
}

// S = Dn_NN^-1 and S_T = D_TT^-1, row-major [M][M] each (h->d_jac: the scalar kernel of sri_shape_jacobian and the
// reverse-mode kernels), built on first use
static int ensure_rowmajor_ops(sri_context* h) {
    if (h->d_jac) return SRI_OK;
    const int M = h->M;
    std::vector<double> t((size_t)2 * M * M);
    for (int i = 0; i < M; ++i)
        for (int j = 0; j < M; ++j) {
            t[(size_t)i * M + j] = h->ops.S[(size_t)j * M + i];
            t[(size_t)M * M + (size_t)i * M + j] = h->ops.ST[(size_t)j * M + i];
        }
    SRI_CUDA(cudaMalloc(&h->d_jac, t.size() * sizeof(double)));
    SRI_CUDA(cudaMemcpy(h->d_jac, t.data(), t.size() * sizeof(double), cudaMemcpyHostToDevice));
    return SRI_OK;
}

// VjpParams with the handle's operator tables (built on first use) and the batch shape; every data pointer NULL
static int vjp_params(sri_context* h, int64_t batch, sri::VjpParams* p) {
    const int M = h->M;
    SRI_TRY(ensure_rowmajor_ops(h));
    if (!h->d_dnin) {
        SRI_CUDA(cudaMalloc(&h->d_dnin, sizeof(double) * M));
        SRI_CUDA(cudaMemcpy(h->d_dnin, h->ops.Dn_IN.data(), sizeof(double) * M, cudaMemcpyHostToDevice));
    }
    *p = sri::VjpParams{};
    p->batch = batch; p->N = h->N; p->M = M;
    p->S_rm = h->d_jac; p->ST_rm = h->d_jac + (size_t)M * M; p->DTI = h->d_dtt + (size_t)M * M; p->DnIN = h->d_dnin;
    return SRI_OK;
}

// device pointers, handle's device current: N <= 16 two rods per warp (sri_vjp16.cuh), else one rod per CTA
static int launch_vjp(sri_context* h, const sri::VjpParams& p) {
    const bool small = h->N <= 16;  // two rods per warp, else one rod per CTA
    auto* kernel = !small ? sri::vjp_tiled_kernel : (h->M == 15 ? sri::vjp16_kernel<15> : sri::vjp16_kernel<0>);
    const int threads = small ? sri::kFusedThreads : sri::kVjpTiledThreads;
    const size_t smem = small ? (sri::VjpTables16::total + (size_t)(sri::kFusedThreads / 32) * 2 * sri::VjpScratch16::total) * sizeof(double)
                              : sri::VjpTiledSmem{h->M}.bytes();
    const long long rods_per_cta = small ? 2 * (sri::kFusedThreads / 32) : 1;
    int occ = 0;
    SRI_TRY(resident_ctas(h, kernel, threads, smem, &occ));
    if (occ < 1) return fail(SRI_ERR_CUDA, "sri_integrate_all_vjp: kernel does not fit on this device");
    const long long want = (p.batch + rods_per_cta - 1) / rods_per_cta;
    return launch(kernel, (int)std::min(want, (long long)h->sm_count * occ), threads, smem, h->stream, p);
}

int sri_integrate_all_vjp(sri_handle h, const sri_rod_batch* rods, const sri_rod_batch_grad* grads) {
    SRI_ENTER(h);
    if (!rods || !grads) return fail(SRI_ERR_INVALID_ARGUMENT, "sri_integrate_all_vjp: rods and grads are required");
    const int64_t B = rods->batch;
    if (B < 0) return fail(SRI_ERR_INVALID_ARGUMENT, "sri_integrate_all_vjp: negative batch");
    if (B == 0) return SRI_OK;
    if (!rods->K) return fail(SRI_ERR_INVALID_ARGUMENT, "sri_integrate_all_vjp: K is required");
    if (!rods->Q) return fail(SRI_ERR_INVALID_ARGUMENT, "sri_integrate_all_vjp: Q (the forward's output) is required");
    if (grads->gm && !rods->n) return fail(SRI_ERR_INVALID_ARGUMENT, "sri_integrate_all_vjp: n (the forward's output) is required with gm");
    const int N = h->N, M = h->M;
    Staging st(h);
    sri::VjpParams p{};
    SRI_TRY(vjp_params(h, B, &p));
    SRI_TRY(st.in(rods->K, (size_t)B * 3 * N, &p.K));
    SRI_TRY(st.in(rods->q0, (size_t)B * 4, &p.q0));
    SRI_TRY(st.in(rods->Gamma, (size_t)B * 3 * N, &p.Gamma));
    SRI_TRY(st.in<double>(rods->Q, (size_t)B * 4 * M, &p.Q));
    if (grads->gm) SRI_TRY(st.in<double>(rods->n, (size_t)B * 3 * M, &p.n));
    SRI_TRY(st.in(grads->gQ, (size_t)B * 4 * M, &p.gQ));
    SRI_TRY(st.in(grads->gr, (size_t)B * 3 * M, &p.gr));
    SRI_TRY(st.in(grads->gn, (size_t)B * 3 * M, &p.gn));
    SRI_TRY(st.in(grads->gm, (size_t)B * 3 * M, &p.gm));
    SRI_TRY(st.out(grads->gK, (size_t)B * 3 * N, &p.gK));
    SRI_TRY(st.out(grads->gq0, (size_t)B * 4, &p.gq0));
    SRI_TRY(st.out(grads->gr0, (size_t)B * 3, &p.gr0));
    SRI_TRY(st.out(grads->gGamma, (size_t)B * 3 * N, &p.gGamma));
    SRI_TRY(st.out(grads->gfbar, (size_t)B * 3 * N, &p.gfbar));
    SRI_TRY(st.out(grads->glbar, (size_t)B * 3 * N, &p.glbar));
    SRI_TRY(st.out(grads->gF_tip, (size_t)B * 3, &p.gF_tip));
    SRI_TRY(st.out(grads->gM_tip, (size_t)B * 3, &p.gM_tip));
    SRI_TRY(st.out(rods->info, (size_t)B, &p.info));
    SRI_TRY(launch_vjp(h, p));
    SRI_TRY(st.finish());
    if (rods->info && !is_device_pointer(rods->info)) return singular_status(rods->info, B, "sri_integrate_all_vjp");
    return SRI_OK;
}

int sri_strain_from_modes_transpose(sri_handle h, int64_t batch, int ne, const double* gK, double* gqe) {
    SRI_ENTER(h);
    if (batch < 0 || ne < 1 || ne > 8 || (batch > 0 && (!gK || !gqe)))
        return fail(SRI_ERR_INVALID_ARGUMENT, "sri_strain_from_modes_transpose: bad arguments (1 <= ne <= 8)");
    if (batch == 0) return SRI_OK;
    Staging st(h);
    const double* dgK; double* dgqe;
    SRI_TRY(st.in(gK, (size_t)batch * 3 * h->N, &dgK));
    SRI_TRY(st.out(gqe, (size_t)batch * 3 * ne, &dgqe));
    const long long total = (long long)batch * 3;
    // the projection kernel without quadrature weights: gqe[b][c*ne+k] = sum_i P_k(t_i) gK[b][c][i]
    SRI_TRY(launch(project_onto_modes_kernel, (unsigned)((total + 127) / 128), 128, 0, h->stream, batch, h->N, ne, 3LL * h->N, 1.0,
                   h->d_ptab, nullptr, dgK, dgqe));
    return st.finish();
}

// device pointers, H on the host, handle's device current
static int shape_jacobian_dev(sri_context* h, int64_t batch, int ne, const double* H, const double* dQ, const double* dq0,
                              const double* dG, const double* dn, const double* dm, const double* dMt, double* dJ) {
    const int N = h->N, M = h->M;
    if (N <= 16 && h->jac_impl == 0) {
        // two [16 x 16] x [16 x 9 ne] contractions + the projection on the FP64 tensor cores, one rod per warp
        auto* kernel = sri::shape_jacobian_dmma_kernel<8>;
        size_t scratch = sri::JacDmmaScratch<8>::total;
        switch (ne) {
#define SRI_JAC(NE_) case NE_: kernel = sri::shape_jacobian_dmma_kernel<NE_>; scratch = sri::JacDmmaScratch<NE_>::total; break;
            SRI_JAC(1) SRI_JAC(2) SRI_JAC(3) SRI_JAC(4) SRI_JAC(5) SRI_JAC(6) SRI_JAC(7)
#undef SRI_JAC
        }
        const size_t smem = (256 + sri::kJacWarps * scratch) * sizeof(double);
        int occ = 0;
        SRI_TRY(resident_ctas(h, kernel, 32 * sri::kJacWarps, smem, &occ));
        if (occ < 1) return fail(SRI_ERR_CUDA, "sri_shape_jacobian: kernel does not fit on this device");
        const long long want = (batch + sri::kJacWarps - 1) / sri::kJacWarps;
        return launch(kernel, (unsigned)std::min(want, (long long)h->sm_count * occ), 32 * sri::kJacWarps, smem, h->stream,
                      batch, N, h->d_ops16, h->d_ptab, h->d_ccw, H[0], H[1], H[2], dQ, dq0, dG, dn, dm, dMt, dJ, h->skip);
    }
    SRI_TRY(ensure_rowmajor_ops(h));
    constexpr int kWarps = 4;
    const size_t smem = ((size_t)2 * M * M + (size_t)9 * N + (size_t)kWarps * JacobianScratch::total(N)) * sizeof(double);
    SRI_TRY(ensure_dynamic_smem(shape_jacobian_kernel, h->device, smem));
    const long long want = (batch + kWarps - 1) / kWarps;
    return launch(shape_jacobian_kernel, (unsigned)std::min(want, (long long)h->sm_count * 8), 32 * kWarps, smem, h->stream,
                  batch, N, ne, h->d_jac, h->d_jac + (size_t)M * M, h->d_ptab, h->d_ccw, H[0], H[1], H[2], dQ, dq0, dG, dn, dm, dMt, dJ, h->skip);
}

int sri_shape_jacobian(sri_handle h, int64_t batch, int ne, const double* H_diag, const double* Q, const double* q0,
                       const double* Gamma, const double* n, const double* m, const double* M_tip, double* J) {
    SRI_ENTER(h);
    if (batch < 0 || ne < 1 || ne > 8 || !H_diag || (batch > 0 && (!Q || !n || !m || !M_tip || !J)))
        return fail(SRI_ERR_INVALID_ARGUMENT, "sri_shape_jacobian: bad arguments (1 <= ne <= 8)");
    if (batch == 0) return SRI_OK;
    const int N = h->N, M = h->M, nq = 3 * ne;
    double H[3];
    SRI_TRY(read_H(H_diag, H));
    Staging st(h);
    const double *dQ, *dq0, *dG, *dn, *dm, *dMt; double* dJ;
    SRI_TRY(st.in(Q, (size_t)batch * 4 * M, &dQ));
    SRI_TRY(st.in(q0, (size_t)batch * 4, &dq0));
    SRI_TRY(st.in(Gamma, (size_t)batch * 3 * N, &dG));
    SRI_TRY(st.in(n, (size_t)batch * 3 * M, &dn));
    SRI_TRY(st.in(m, (size_t)batch * 3 * M, &dm));
    SRI_TRY(st.in(M_tip, (size_t)batch * 3, &dMt));
    SRI_TRY(st.out(J, (size_t)batch * nq * nq, &dJ));
    SRI_TRY(shape_jacobian_dev(h, batch, ne, H, dQ, dq0, dG, dn, dm, dMt, dJ));
    return st.finish();
}

// trans: solve A^T x = b instead (A read transposed, not copied)
static int solve_small_dev(sri_context* h, int64_t batch, int n, double* A, const double* b, double* x, int* info, bool trans = false) {
    if (n == 3 || n == 6 || n == 9) {  // ne <= 3: the whole system lives in the thread's registers
        auto* kernel = trans ? (n == 3 ? solve_small_reg_kernel<3, true> : (n == 6 ? solve_small_reg_kernel<6, true> : solve_small_reg_kernel<9, true>))
                             : (n == 3 ? solve_small_reg_kernel<3, false> : (n == 6 ? solve_small_reg_kernel<6, false> : solve_small_reg_kernel<9, false>));
        return launch(kernel, (unsigned)((batch + 63) / 64), 64, 0, h->stream, batch, A, b, x, info, h->skip);
    }
    const int T = n <= 13 ? 128 : (n <= 19 ? 64 : 32);
    const size_t smem = (size_t)(n * n + n) * (T + 1) * sizeof(double);
    auto* kernel = trans ? solve_small_kernel<true> : solve_small_kernel<false>;
    SRI_TRY(ensure_dynamic_smem(kernel, h->device, smem));
    return launch(kernel, (unsigned)((batch + T - 1) / T), T, smem, h->stream, batch, n, A, b, x, info, h->skip);
}

int sri_solve_small_batched(sri_handle h, int64_t batch, int n, double* A, const double* b, double* x, int* info) {
    SRI_ENTER(h);
    if (batch < 0 || n < 1 || n > 24 || (batch > 0 && (!A || !b || !x))) return fail(SRI_ERR_INVALID_ARGUMENT, "sri_solve_small_batched: bad arguments (1 <= n <= 24)");
    if (batch == 0) return SRI_OK;
    for (const void* p : {(const void*)A, (const void*)b, (const void*)x, (const void*)info})
        if (p && !is_device_pointer(p)) return fail(SRI_ERR_INVALID_ARGUMENT, "sri_solve_small_batched: device pointers only");
    return solve_small_dev(h, batch, n, A, b, x, info);
}

// Implicit adjoint of the static shape solve (DESIGN section 5e).  At the caller's qe (one integration and one analytic
// Jacobian J_a), solve J_d^T lam = gqe by iterative refinement preconditioned with J_a^T:
//     lam_0 = J_a^-T gqe,   lam_{k+1} = lam_k + J_a^-T (gqe - J_d^T lam_k)   (refine_steps times),
// where J_d^T lam = Phi^T (gK_dir + gK_int) comes from chain(lam): the residual's VJP (cotangent lam) followed by the
// integration's VJP of its (gQ, gm).  A final chain(lam) gives the parameter gradients -(dg/dtheta)^T lam and the residual.
// `who` names the entry point in error messages.
static int static_problem_vjp(sri_context* h, const sri_static_problem& P, const double* qe, const double* gqe, int refine_steps,
                              const sri_static_problem_grad& G, const char* who) {
    const int64_t B = P.batch;
    const int ne = P.ne;
    if (B < 0 || ne < 1 || ne > 8 || !P.H_diag || refine_steps < 0 || refine_steps > 1000 ||
        (B > 0 && (!P.F_tip || !P.M_tip || !qe || !gqe)))
        return fail(SRI_ERR_INVALID_ARGUMENT, std::string(who) + ": bad arguments (1 <= ne <= 8, 0 <= refine_steps <= 1000)");
    if (B == 0) return SRI_OK;
    const int N = h->N, M = h->M, n = 3 * ne;
    double H[3];
    SRI_TRY(read_H(P.H_diag, H));
    auto& ws = h->adjoint;
    if (ws.B != B || ws.ne != ne || !ws.block) {
        SRI_CUDA(cudaStreamSynchronize(h->stream));
        if (ws.block) SRI_CUDA(cudaFree(ws.block));
        ws.block = nullptr; ws.B = -1;
        auto up = [](size_t v) { return (v + 1) & ~(size_t)1; };  // 16-byte aligned pieces
        const size_t sz[] = {up((size_t)3 * N * B), up((size_t)4 * M * B), up((size_t)3 * M * B), up((size_t)3 * M * B),
                             up((size_t)n * n * B), up((size_t)n * B), up((size_t)n * B), up((size_t)3 * N * B), up((size_t)3 * N * B),
                             up((size_t)4 * M * B), up((size_t)3 * M * B), up((size_t)3 * B), up((size_t)3 * B), up((size_t)3 * B),
                             up((size_t)3 * B), up((size_t)n * B), up((size_t)4 * B), up((size_t)4 * B)};
        double** fields[] = {&ws.K, &ws.Q, &ws.n, &ws.m, &ws.J, &ws.rhs, &ws.delta, &ws.gKd, &ws.gKi, &ws.gQ, &ws.gm, &ws.gMd,
                             &ws.gMi, &ws.gFi, &ws.gHw, &ws.lam, &ws.gq0d, &ws.gq0i};
        static_assert(sizeof(sz) / sizeof(sz[0]) == sizeof(fields) / sizeof(fields[0]), "one size per workspace field");
        size_t total = 2 * up(((size_t)B + 1) / 2);
        for (size_t v : sz) total += v;
        SRI_CUDA(cudaMalloc(&ws.block, total * sizeof(double)));
        size_t off = 0;
        for (size_t i = 0; i < sizeof(sz) / sizeof(sz[0]); ++i) { *fields[i] = ws.block + off; off += sz[i]; }
        ws.sinfo = reinterpret_cast<int*>(ws.block + off);
        ws.vinfo = ws.sinfo + 2 * up(((size_t)B + 1) / 2);
        ws.B = B; ws.ne = ne;
    }
    Staging st(h);
    const double *dF, *dMt, *dK0, *dq0, *dG, *dfb, *dlb, *dqe, *dgqe;
    double *dgF, *dgMt, *dgK0, *dgH, *dgq0, *dgG, *dgfb, *dglb, *dlam, *dres;
    int* dinfo;
    SRI_TRY(st.in(P.F_tip, (size_t)B * 3, &dF));
    SRI_TRY(st.in(P.M_tip, (size_t)B * 3, &dMt));
    SRI_TRY(st.in(P.K0, (size_t)B * 3 * N, &dK0));
    SRI_TRY(st.in(P.q0, (size_t)B * 4, &dq0));
    SRI_TRY(st.in(P.Gamma, (size_t)B * 3 * N, &dG));
    SRI_TRY(st.in(P.fbar, (size_t)B * 3 * N, &dfb));
    SRI_TRY(st.in(P.lbar, (size_t)B * 3 * N, &dlb));
    SRI_TRY(st.in(qe, (size_t)B * n, &dqe));
    SRI_TRY(st.in(gqe, (size_t)B * n, &dgqe));
    SRI_TRY(st.out(G.gF_tip, (size_t)B * 3, &dgF));
    SRI_TRY(st.out(G.gM_tip, (size_t)B * 3, &dgMt));
    SRI_TRY(st.out(G.gK0, (size_t)B * 3 * N, &dgK0));
    SRI_TRY(st.out(G.gH, (size_t)B * 3, &dgH));
    SRI_TRY(st.out(G.gq0, (size_t)B * 4, &dgq0));
    SRI_TRY(st.out(G.gGamma, (size_t)B * 3 * N, &dgG));
    SRI_TRY(st.out(G.gfbar, (size_t)B * 3 * N, &dgfb));
    SRI_TRY(st.out(G.glbar, (size_t)B * 3 * N, &dglb));
    SRI_TRY(st.out(G.lambda, (size_t)B * n, &dlam));
    SRI_TRY(st.out(G.resid, (size_t)B, &dres));
    SRI_TRY(st.out(G.info, (size_t)B, &dinfo));
    double* lam = dlam ? dlam : ws.lam;

    // forward state at qe: K = Phi qe, the four stages (Q, n, m), the analytic Jacobian J_a
    SRI_TRY(strain_from_modes_dev(h, B, ne, dqe, ws.K));
    {
        sri::FusedParams p{};
        p.batch = B; p.N = N; p.M = M; p.ops = h->d_ops16;
        p.K = ws.K; p.q0 = dq0; p.Gamma = dG; p.fbar = dfb; p.lbar = dlb; p.F_tip = dF; p.M_tip = dMt;
        p.Q = ws.Q; p.n = ws.n; p.m = ws.m;
        SRI_TRY(launch_fused(h, p));
    }
    SRI_TRY(shape_jacobian_dev(h, B, ne, H, ws.Q, dq0, dG, ws.n, ws.m, dMt, ws.J));
    SRI_TRY(solve_small_dev(h, B, n, ws.J, dgqe, lam, ws.sinfo, true));

    sri::VjpParams vp{};
    SRI_TRY(vjp_params(h, B, &vp));
    vp.K = ws.K; vp.q0 = dq0; vp.Gamma = dG; vp.Q = ws.Q; vp.n = ws.n; vp.gQ = ws.gQ; vp.gm = ws.gm; vp.gK = ws.gKi;
    vp.info = ws.vinfo;
    auto refine_kernel = pick_lanes_ne<PickAdjointRefine>(N, ne);
    const unsigned blocks = lane_group_blocks(h, B);
    const long long tu = (long long)n * B;
    const bool finals = dres || dgF || dgMt || dgH || dgq0 || dgG || dgfb || dglb || dinfo;
    for (int step = 0; step <= refine_steps; ++step) {
        const bool last = step == refine_steps;
        // chain(lam): K0-gradient = H rho_bar = gK_dir, so the last chain writes gK_dir straight into that output
        double* gKd = last && dgK0 ? dgK0 : ws.gKd;
        SRI_TRY(galerkin_residual_vjp_dev(h, B, ne, ws.K, dK0, H, ws.Q, dq0, ws.m, dMt, lam, gKd, nullptr,
                                          last && dgH ? ws.gHw : nullptr, ws.gQ, last && dgq0 ? ws.gq0d : nullptr, ws.gm,
                                          last && dgMt ? ws.gMd : nullptr));
        vp.gF_tip = last && dgF ? ws.gFi : nullptr;
        vp.gM_tip = last && dgMt ? ws.gMi : nullptr;
        vp.gq0 = last && dgq0 ? ws.gq0i : nullptr;
        // the last VJP writes the Gamma / fbar / lbar gradients into the outputs; the refine kernel negates them there
        vp.gGamma = last ? dgG : nullptr;
        vp.gfbar = last ? dgfb : nullptr;
        vp.glbar = last ? dglb : nullptr;
        SRI_TRY(launch_vjp(h, vp));
        AdjointRefineParams rp{};
        rp.batch = B; rp.N = N; rp.ptab = h->d_ptab; rp.gqe = dgqe; rp.gKd = gKd; rp.gKi = ws.gKi;
        if (!last) {
            rp.rhs = ws.rhs;
        } else {
            rp.resid = dres;
            rp.gFi = ws.gFi; rp.gMd = ws.gMd; rp.gMi = ws.gMi; rp.gHw = ws.gHw;
            rp.gF = dgF; rp.gM = dgMt; rp.gH = dgH;
            rp.gq0d = ws.gq0d; rp.gq0i = ws.gq0i; rp.gq0 = dgq0;
            rp.gGamma = dgG; rp.gfbar = dgfb; rp.glbar = dglb;
            rp.sinfo = ws.sinfo; rp.vinfo = ws.vinfo; rp.info = dinfo;
        }
        if (!last || finals) SRI_TRY(launch(refine_kernel, blocks, 256, 0, h->stream, rp));
        if (!last) {
            // lam -= J_a^-T (J_d^T lam - gqe), skipped for rods whose J_a^T is singular
            SRI_TRY(solve_small_dev(h, B, n, ws.J, ws.rhs, ws.delta, ws.sinfo, true));
            SRI_TRY(launch(newton_update_kernel, (unsigned)((tu + 255) / 256), 256, 0, h->stream, (long long)B, n, lam, ws.delta,
                           ws.sinfo, (sri::NewtonState*)nullptr, (const int*)nullptr));
        }
    }
    SRI_TRY(st.finish());
    if (G.info && !is_device_pointer(G.info)) return singular_status(G.info, B, who);
    return SRI_OK;
}

int sri_static_shape_vjp(sri_handle h, int64_t batch, int ne, const double* H_diag, const double* F_tip, const double* M_tip,
                         const double* K0, const double* qe, const double* gqe, int refine_steps, double* gF_tip,
                         double* gM_tip, double* gK0, double* gH, double* lambda, double* resid, int* info) {
    SRI_ENTER(h);
    sri_static_problem P{};
    P.batch = batch; P.ne = ne; P.H_diag = H_diag; P.F_tip = F_tip; P.M_tip = M_tip; P.K0 = K0;
    sri_static_problem_grad G{};
    G.gF_tip = gF_tip; G.gM_tip = gM_tip; G.gK0 = gK0; G.gH = gH; G.lambda = lambda; G.resid = resid; G.info = info;
    return static_problem_vjp(h, P, qe, gqe, refine_steps, G, "sri_static_shape_vjp");
}

int sri_static_problem_vjp(sri_handle h, const sri_static_problem* problem, const double* qe, const double* gqe, int refine_steps,
                           const sri_static_problem_grad* grads) {
    SRI_ENTER(h);
    if (!problem || !grads) return fail(SRI_ERR_INVALID_ARGUMENT, "sri_static_problem_vjp: problem and grads are required");
    return static_problem_vjp(h, *problem, qe, gqe, refine_steps, *grads, "sri_static_problem_vjp");
}

// ---- NCCL, bound at run time --------------------------------------------------------------------------------------
// The library does not link against NCCL: libnccl.so.2 is opened with dlopen when sri_nccl_* is first called (inside a
// PyTorch process that resolves to the copy torch has already loaded).  Only the five entry points below are used.
namespace {
struct NcclUniqueId { char internal[128]; };  // ncclUniqueId (nccl.h: NCCL_UNIQUE_ID_BYTES = 128)
struct NcclApi {
    void* lib = nullptr;
    int (*GetUniqueId)(NcclUniqueId*) = nullptr;
    int (*CommInitRank)(void**, int, NcclUniqueId, int) = nullptr;
    int (*CommDestroy)(void*) = nullptr;
    int (*AllGather)(const void*, void*, size_t, int, void*, cudaStream_t) = nullptr;
    const char* (*GetErrorString)(int) = nullptr;
};
constexpr int kNcclDouble = 8;  // ncclFloat64

int nccl_api(NcclApi** out) {
    static std::mutex mu;
    static NcclApi api;
    std::lock_guard<std::mutex> lock(mu);
    if (!api.lib) {
        void* lib = nullptr;
        if (const char* path = std::getenv("SRI_NCCL_LIB")) lib = dlopen(path, RTLD_NOW | RTLD_GLOBAL);
        if (!lib) lib = dlopen("libnccl.so.2", RTLD_NOW | RTLD_GLOBAL);
        if (!lib) lib = dlopen("libnccl.so", RTLD_NOW | RTLD_GLOBAL);
        if (!lib) return fail(SRI_ERR_CUDA, std::string("NCCL is not available: ") + (dlerror() ? dlerror() : "dlopen(libnccl.so.2) failed"));
        NcclApi a;
        a.GetUniqueId = reinterpret_cast<decltype(a.GetUniqueId)>(dlsym(lib, "ncclGetUniqueId"));
        a.CommInitRank = reinterpret_cast<decltype(a.CommInitRank)>(dlsym(lib, "ncclCommInitRank"));
        a.CommDestroy = reinterpret_cast<decltype(a.CommDestroy)>(dlsym(lib, "ncclCommDestroy"));
        a.AllGather = reinterpret_cast<decltype(a.AllGather)>(dlsym(lib, "ncclAllGather"));
        a.GetErrorString = reinterpret_cast<decltype(a.GetErrorString)>(dlsym(lib, "ncclGetErrorString"));
        if (!a.GetUniqueId || !a.CommInitRank || !a.CommDestroy || !a.AllGather || !a.GetErrorString) {
            dlclose(lib);
            return fail(SRI_ERR_CUDA, "NCCL library lacks an expected symbol");
        }
        a.lib = lib;
        api = a;
    }
    *out = &api;
    return SRI_OK;
}
#define SRI_NCCL(api, expr)                                                                                   \
    do {                                                                                                      \
        const int r__ = (expr);                                                                               \
        if (r__ != 0) return fail(SRI_ERR_CUDA, std::string(#expr) + ": " + (api)->GetErrorString(r__));      \
    } while (0)

// all-gathers the 2 doubles at `red` of every rank into h->d_gather (rank-major) on the handle's stream; without a
// communicator the "gather" is a 16-byte device copy
int gather_norms(sri_context* h, const double* red) {
    if (!h->d_gather) SRI_CUDA(cudaMalloc(&h->d_gather, sizeof(double) * 2 * std::max(1, h->nccl_nranks)));
    if (h->nccl_comm) {
        NcclApi* api = nullptr;
        SRI_TRY(nccl_api(&api));
        SRI_NCCL(api, api->AllGather(red, h->d_gather, 2, kNcclDouble, h->nccl_comm, h->stream));
    } else {
        SRI_CUDA(cudaMemcpyAsync(h->d_gather, red, 2 * sizeof(double), cudaMemcpyDeviceToDevice, h->stream));
    }
    return SRI_OK;
}
}  // namespace

int sri_nccl_unique_id(void* id128) {
    if (!id128) return fail(SRI_ERR_INVALID_ARGUMENT, "sri_nccl_unique_id: null argument");
    NcclApi* api = nullptr;
    SRI_TRY(nccl_api(&api));
    NcclUniqueId id;
    SRI_NCCL(api, api->GetUniqueId(&id));
    std::memcpy(id128, id.internal, sizeof(id.internal));
    return SRI_OK;
}

int sri_nccl_init(sri_handle h, int nranks, int rank, const void* id128) {
    SRI_ENTER(h);
    if (!id128 || nranks < 1 || rank < 0 || rank >= nranks) return fail(SRI_ERR_INVALID_ARGUMENT, "sri_nccl_init: bad arguments");
    if (h->nccl_comm) SRI_TRY(sri_nccl_finalize(h));
    NcclApi* api = nullptr;
    SRI_TRY(nccl_api(&api));
    NcclUniqueId id;
    std::memcpy(id.internal, id128, sizeof(id.internal));
    void* comm = nullptr;
    SRI_NCCL(api, api->CommInitRank(&comm, nranks, id, rank));
    h->nccl_comm = comm; h->nccl_nranks = nranks; h->nccl_rank = rank;
    if (h->d_gather) { SRI_CUDA(cudaFree(h->d_gather)); h->d_gather = nullptr; }
    return SRI_OK;
}

int sri_nccl_finalize(sri_handle h) {
    SRI_ENTER(h);
    if (!h->nccl_comm) return SRI_OK;
    NcclApi* api = nullptr;
    SRI_TRY(nccl_api(&api));
    SRI_CUDA(cudaStreamSynchronize(h->stream));
    void* comm = h->nccl_comm;
    h->nccl_comm = nullptr; h->nccl_nranks = 1; h->nccl_rank = 0;
    if (h->d_gather) { cudaFree(h->d_gather); h->d_gather = nullptr; }
    SRI_NCCL(api, api->CommDestroy(comm));
    return SRI_OK;
}

int sri_nccl_allreduce_norms(sri_handle h, double* norm2_and_max) {
    SRI_ENTER(h);
    if (!norm2_and_max || !is_device_pointer(norm2_and_max)) return fail(SRI_ERR_INVALID_ARGUMENT, "sri_nccl_allreduce_norms: device pointer required");
    SRI_TRY(gather_norms(h, norm2_and_max));
    return launch(fold_norms_kernel, 1, 32, 0, h->stream, h->d_gather, std::max(1, h->nccl_nranks), norm2_and_max);
}

// Newton iteration of the static shape problem, host loop in this library (no torch, no Python in the loop).  Per
// iteration: Jacobian (analytic: one kernel; forward differences: ONE hot-path call on the 3 ne perturbed copies of the
// batch), per-rod solve, update, re-evaluation (modal adapter, fused four-stage integration, Galerkin residual + norms),
// then the convergence test.  rod_modeling.pdf section 2.2; BASELINE configs[4].
//
// reduce == NULL (device-side reduction): the norms are all-gathered over the handle's NCCL communicator on its stream
// (or copied, single rank), newton_check_kernel turns them into a device-side `done` flag, and the host enqueues
// iteration k+1 BEFORE it waits for the 16 bytes of iteration k (pinned mirror + event): the test lags by one iteration
// and the GPU never idles on the host.  Kernels enqueued after convergence see the flag and exit, so qe, the iteration
// count and the history are exactly those of the unlagged loop.  From the second iteration on, one iteration + its test
// (8-12 stream operations) is ONE CUDA graph launch, captured once per workspace / H / tol (SRI_NEWTON_GRAPH=0 keeps eager
// launches; so does a communicator of more than one rank, see below): worth 1 % at 10^5 rods and 5-8 % at 3 000-12 500.
// reduce != NULL: the caller's host callback reduces the norms; the loop synchronises once per iteration.
// `who` names the entry point in error messages.
static int newton_static_problem(sri_context* h, const sri_static_problem& P, double* qe, double tol, int max_iter, double fd_step,
                                 int64_t total_dof, sri_allreduce_fn reduce, void* reduce_ctx, sri_newton_report* report,
                                 const char* who) {
    const int64_t batch = P.batch;
    const int ne = P.ne;
    if (batch < 0 || ne < 1 || ne > 8 || !P.H_diag || max_iter < 0 || max_iter > 62 || !(fd_step >= 0.0) ||
        (batch > 0 && (!P.F_tip || !P.M_tip || !qe)))
        return fail(SRI_ERR_INVALID_ARGUMENT, std::string(who) + ": bad arguments (1 <= ne <= 8, 0 <= max_iter <= 62, fd_step >= 0)");
    const bool analytic = fd_step == 0.0;  // Jacobian from sri_shape_jacobian instead of forward differences
    const bool lagged = reduce == nullptr;
    const int N = h->N, M = h->M, n = 3 * ne;
    const int64_t B = batch, W = analytic ? 0 : (int64_t)n * B;
    double H[3];
    SRI_TRY(read_H(P.H_diag, H));
    auto& ws = h->newton;
    // which optional arrays the problem has is part of the workspace key: a captured graph never points at a missing copy
    const unsigned present = (P.K0 ? 1u : 0u) | (P.q0 ? 2u : 0u) | (P.Gamma ? 4u : 0u) | (P.fbar ? 8u : 0u) | (P.lbar ? 16u : 0u);
    if (ws.B != B || ws.ne != ne || ws.present != present || ws.analytic != analytic || !ws.block) {
        SRI_CUDA(cudaStreamSynchronize(h->stream));
        if (ws.graph) { cudaGraphExecDestroy(ws.graph); ws.graph = nullptr; }
        if (ws.block) SRI_CUDA(cudaFree(ws.block));
        ws.block = nullptr; ws.B = -1;
        auto up = [](size_t v) { return (v + 1) & ~(size_t)1; };  // 16-byte aligned pieces
        // an optional array of `per_rod` doubles for `rods` rods, or nothing when the problem does not have it
        auto opt = [&](unsigned bit, size_t per_rod, int64_t rods) { return (present & bit) ? up(per_rod * (size_t)rods) : (size_t)0; };
        const size_t state_doubles = up((sizeof(NewtonState) + 7) / 8);
        const size_t sz[] = {up((size_t)3 * N * B), up((size_t)4 * M * B), up((size_t)3 * M * B), up((size_t)3 * M * B), up((size_t)n * B), up((size_t)n * n * B),
                             up((size_t)n * B), up((size_t)n * B), 8, up((size_t)3 * B), up((size_t)3 * B), opt(1, 3 * N, B),
                             up((size_t)n * W), up((size_t)3 * N * W), up((size_t)4 * M * W), up((size_t)3 * M * W), up((size_t)n * W),
                             up((size_t)3 * W), up((size_t)3 * W), opt(1, 3 * N, W),
                             opt(2, 4, B), opt(4, 3 * N, B), opt(8, 3 * N, B), opt(16, 3 * N, B),
                             opt(2, 4, W), opt(4, 3 * N, W), opt(8, 3 * N, W), opt(16, 3 * N, W)};
        size_t total = state_doubles + up(((size_t)B + 1) / 2);
        for (size_t v : sz) total += v;
        SRI_CUDA(cudaMalloc(&ws.block, total * sizeof(double)));
        double** fields[] = {&ws.K, &ws.Q, &ws.m, &ws.nn, &ws.g0, &ws.J, &ws.delta, &ws.qe, &ws.red, &ws.F, &ws.Mt, &ws.K0,
                             &ws.qw, &ws.Kw, &ws.Qw, &ws.mw, &ws.gw, &ws.Fw, &ws.Mtw, &ws.K0w,
                             &ws.q0, &ws.G, &ws.fb, &ws.lb, &ws.q0w, &ws.Gw, &ws.fbw, &ws.lbw};
        static_assert(sizeof(sz) / sizeof(sz[0]) == sizeof(fields) / sizeof(fields[0]), "one size per workspace field");
        size_t off = 0;
        for (size_t i = 0; i < sizeof(sz) / sizeof(sz[0]); ++i) { *fields[i] = sz[i] ? ws.block + off : nullptr; off += sz[i]; }
        ws.state = reinterpret_cast<NewtonState*>(ws.block + off); off += state_doubles;
        ws.sinfo = reinterpret_cast<int*>(ws.block + off);
        ws.B = B; ws.ne = ne; ws.present = present; ws.analytic = analytic;
    }
    if (!ws.host_state) {
        SRI_CUDA(cudaMallocHost(reinterpret_cast<void**>(&ws.host_state), 2 * sizeof(NewtonState)));
        if (const char* g = std::getenv("SRI_NEWTON_GRAPH")) ws.graph_off = std::atoi(g) == 0;
    }
    for (cudaEvent_t& e : ws.ev)
        if (!e) SRI_CUDA(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
    // The legacy default stream cannot be captured.  This call is synchronous for the host anyway (it returns after qe has
    // been copied back), so in that case the loop runs on the handle's own stream, ordered after the work already queued on
    // the caller's stream, and the handle's stream is restored on the way out.
    struct StreamSwap { sri_context* h; cudaStream_t saved; bool on = false; ~StreamSwap() { if (on) h->stream = saved; } } swap{h, h->stream};
    // (Several ranks: the iteration is NOT captured.  An ncclAllGather recorded into the graph on two ranks hung in this
    // build's test run; with a communicator of more than one rank the loop keeps the eager launches it was verified with.)
    const bool use_graph = lagged && !ws.graph_off && !(h->nccl_comm && h->nccl_nranks > 1);
    if (use_graph && (h->stream == nullptr || h->stream == cudaStreamLegacy) && h->own_stream) {
        if (!h->pipe_event) SRI_CUDA(cudaEventCreateWithFlags(&h->pipe_event, cudaEventDisableTiming));
        SRI_CUDA(cudaEventRecord(h->pipe_event, h->stream));
        SRI_CUDA(cudaStreamWaitEvent(h->own_stream, h->pipe_event, 0));
        h->stream = h->own_stream;
        swap.on = true;
    }
    cudaStream_t st = h->stream;
    SRI_CUDA(cudaMemsetAsync(ws.state, 0, sizeof(NewtonState), st));
    SRI_CUDA(cudaMemsetAsync(ws.red, 0, 2 * sizeof(double), st));  // a rank without rods contributes (0, 0)
    if (B > 0) {
        SRI_CUDA(cudaMemcpyAsync(ws.qe, qe, sizeof(double) * n * B, cudaMemcpyDefault, st));
        // the problem's inputs, and their replicas in each of the n forward-difference copies of the batch
        struct Input { const double* src; double* dst; double* rep; size_t per_rod; };
        const Input inputs[] = {{P.F_tip, ws.F, ws.Fw, 3}, {P.M_tip, ws.Mt, ws.Mtw, 3}, {P.K0, ws.K0, ws.K0w, (size_t)3 * N},
                                {P.q0, ws.q0, ws.q0w, 4}, {P.Gamma, ws.G, ws.Gw, (size_t)3 * N}, {P.fbar, ws.fb, ws.fbw, (size_t)3 * N},
                                {P.lbar, ws.lb, ws.lbw, (size_t)3 * N}};
        for (const Input& in : inputs)
            if (in.src) SRI_CUDA(cudaMemcpyAsync(in.dst, in.src, sizeof(double) * in.per_rod * B, cudaMemcpyDefault, st));
        for (int d = 0; d < n && !analytic; ++d)
            for (const Input& in : inputs)
                if (in.src)
                    SRI_CUDA(cudaMemcpyAsync(in.rep + (size_t)d * in.per_rod * B, in.dst, sizeof(double) * in.per_rod * B,
                                             cudaMemcpyDeviceToDevice, st));
    }
    // every kernel launched from here on takes the device-side flag (lagged mode only); cleared on every way out
    struct SkipScope { sri_context* h; ~SkipScope() { h->skip = nullptr; } } skip_scope{h};
    h->skip = lagged ? &ws.state->done : nullptr;

    // the loads of the batch (base) and of its forward-difference copies (w): workspace copies, NULL when absent
    struct Loads { const double *F, *Mt, *K0, *q0, *G, *fb, *lb; };
    const Loads base{ws.F, ws.Mt, ws.K0, ws.q0, ws.G, ws.fb, ws.lb}, w{ws.Fw, ws.Mtw, ws.K0w, ws.q0w, ws.Gw, ws.fbw, ws.lbw};
    auto evaluate = [&](int64_t rods, const double* q, double* K, double* Q, double* m, const Loads& L, double* g, double* red,
                        double* nout = nullptr) -> int {
        SRI_TRY(strain_from_modes_dev(h, rods, ne, q, K));
        sri::FusedParams p{};
        p.batch = rods; p.N = N; p.M = M; p.ops = h->d_ops16;
        p.K = K; p.q0 = L.q0; p.Gamma = L.G; p.fbar = L.fb; p.lbar = L.lb; p.F_tip = L.F; p.M_tip = L.Mt;
        p.Q = Q; p.m = m; p.n = nout;
        SRI_TRY(launch_fused(h, p));
        return galerkin_residual_dev(h, rods, ne, K, L.K0, H, Q, L.q0, m, L.Mt, g, red);
    };
    // one Newton update + re-evaluation of the base point, all asynchronous on the handle's stream
    auto iterate = [&]() -> int {
        if (B == 0) return SRI_OK;
        const long long tq = (long long)n * W, tj = (long long)B * n * n, tu = (long long)n * B;
        if (analytic) {
            SRI_TRY(shape_jacobian_dev(h, B, ne, H, ws.Q, ws.q0, ws.G, ws.nn, ws.m, ws.Mt, ws.J));
        } else {
            SRI_TRY(launch(fd_perturb_kernel, (unsigned)((tq + 255) / 256), 256, 0, st, B, n, fd_step, ws.qe, ws.qw, h->skip));
            SRI_TRY(evaluate(W, ws.qw, ws.Kw, ws.Qw, ws.mw, w, ws.gw, nullptr));
            SRI_TRY(launch(fd_jacobian_kernel, (unsigned)((tj + 255) / 256), 256, 0, st, B, n, fd_step, ws.gw, ws.g0, ws.J, h->skip));
        }
        SRI_TRY(solve_small_dev(h, B, n, ws.J, ws.g0, ws.delta, ws.sinfo));
        SRI_TRY(launch(newton_update_kernel, (unsigned)((tu + 255) / 256), 256, 0, st, B, n, ws.qe, ws.delta, ws.sinfo, ws.state, h->skip));
        return evaluate(B, ws.qe, ws.K, ws.Q, ws.m, base, ws.g0, ws.red, analytic ? ws.nn : nullptr);
    };
    const double dof = (double)(total_dof > 0 ? total_dof : (int64_t)n * B);
    const int nranks = std::max(1, h->nccl_nranks);
    // device-side convergence test number `t` and the asynchronous copy of its outcome to the pinned mirror
    auto test_device = [&]() -> int {
        SRI_TRY(gather_norms(h, ws.red));
        return launch(newton_check_kernel, 1, 32, 0, st, h->d_gather, nranks, dof, tol, ws.state);
    };
    auto test_mirror = [&](int t) -> int {
        SRI_CUDA(cudaMemcpyAsync(ws.host_state + (t & 1), ws.state, sizeof(NewtonState), cudaMemcpyDeviceToHost, st));
        SRI_CUDA(cudaEventRecord(ws.ev[t & 1], st));
        return SRI_OK;
    };
    auto test = [&](int t) -> int {
        SRI_TRY(test_device());
        return test_mirror(t);
    };
    // iterate() + test_device() as one graph launch.  Every argument of every node is fixed for the lifetime of the workspace
    // (pointers into ws.block, handle tables) or part of the key below; the first iteration of a call always runs eagerly, so
    // every lazy allocation and attribute of the kernels involved exists before a capture starts.
    auto iterate_and_test_graph = [&]() -> int {
        sri_context::NewtonWorkspace::GraphKey key{};
        key.H[0] = H[0]; key.H[1] = H[1]; key.H[2] = H[2]; key.tol = tol; key.dof = dof; key.fd_step = fd_step;
        key.block = ws.block; key.list = h->d_list[3]; key.comm = h->nccl_comm; key.stream = st;   // (the hand-back list may be re-allocated by a larger call in between)
        if (ws.graph && std::memcmp(&key, &ws.graph_key, sizeof key) != 0) { cudaGraphExecDestroy(ws.graph); ws.graph = nullptr; }
        if (!ws.graph) {
            const long long before = g_launches.load();
            cudaGraph_t graph = nullptr;
            if (cudaStreamBeginCapture(st, cudaStreamCaptureModeThreadLocal) != cudaSuccess) {   // (a stream that cannot be captured)
                cudaGetLastError();
                ws.graph_off = true;
                SRI_TRY(iterate());
                return test_device();
            }
            int rc = iterate();
            if (rc == SRI_OK) rc = test_device();
            const cudaError_t ce = cudaStreamEndCapture(st, &graph);
            const long long captured = g_launches.load() - before;
            g_launches.fetch_sub(captured);   // (recorded, not run)
            if (rc != SRI_OK || ce != cudaSuccess || !graph) {
                if (graph) cudaGraphDestroy(graph);
                cudaGetLastError();
                ws.graph_off = true;   // this handle falls back to eager launches
                if (rc != SRI_OK) return rc;
                SRI_TRY(iterate());
                return test_device();
            }
            const cudaError_t ie = cudaGraphInstantiate(&ws.graph, graph, 0);
            cudaGraphDestroy(graph);
            if (ie != cudaSuccess) {
                cudaGetLastError();
                ws.graph = nullptr; ws.graph_off = true;
                SRI_TRY(iterate());
                return test_device();
            }
            ws.graph_key = key;
            ws.graph_kernels = captured;
        }
        SRI_CUDA(cudaGraphLaunch(ws.graph, st));
        g_launches.fetch_add(ws.graph_kernels);
        return SRI_OK;
    };

    sri_newton_report rep{};
    if (B > 0) SRI_TRY(evaluate(B, ws.qe, ws.K, ws.Q, ws.m, base, ws.g0, ws.red, analytic ? ws.nn : nullptr));
    rep.integrations = 1;
    unsigned long long singular = 0;
    int last_mirror = 0;
    if (lagged) {
        SRI_TRY(test(0));
        for (int it = 0;; ++it) {
            // enqueue iteration it+1 and its test before looking at test `it` (no-ops on the device if `it` converged)
            if (it < max_iter) {
                if (it >= 1 && B > 0 && use_graph && !ws.graph_off) {
                    SRI_TRY(iterate_and_test_graph());
                    SRI_TRY(test_mirror(it + 1));
                } else {
                    SRI_TRY(iterate());
                    SRI_TRY(test(it + 1));
                }
                last_mirror = (it + 1) & 1;
            }
            // test `it` was copied to mirror it & 1; the next copy into that mirror (test it + 2) is only enqueued in the next
            // pass of this loop, after the read below
            SRI_CUDA(cudaEventSynchronize(ws.ev[it & 1]));
            const NewtonState* hs = ws.host_state + (it & 1);
            const double s2 = hs->hist[it][0], mx = hs->hist[it][1];
            rep.rms = dof > 0 ? std::sqrt(s2 / dof) : 0.0;
            rep.max_abs = mx;
            rep.rms_history[rep.history_len++] = rep.rms;
            if (rep.rms < tol) { rep.converged = 1; break; }
            if (it == max_iter) break;
            rep.iterations += 1;
            rep.integrations += analytic ? 1 : n + 1;
        }
        SRI_CUDA(cudaStreamSynchronize(st));
        // every copy has landed; the newest state is in the mirror of the last test that was enqueued
        singular = ws.host_state[last_mirror].singular;
    } else {
        for (int it = 0;; ++it) {
            double red[2] = {0.0, 0.0};
            SRI_CUDA(cudaMemcpyAsync(red, ws.red, sizeof(red), cudaMemcpyDeviceToHost, st));
            SRI_CUDA(cudaStreamSynchronize(st));
            if (reduce(red, reduce_ctx) != 0) return fail(SRI_ERR_INVALID_ARGUMENT, std::string(who) + ": the reduction callback failed");
            rep.rms = dof > 0 ? std::sqrt(red[0] / dof) : 0.0;
            rep.max_abs = red[1];
            rep.rms_history[rep.history_len++] = rep.rms;
            if (rep.rms < tol) { rep.converged = 1; break; }
            if (it == max_iter) break;
            SRI_TRY(iterate());
            rep.iterations += 1;
            rep.integrations += analytic ? 1 : n + 1;
        }
        SRI_CUDA(cudaMemcpyAsync(ws.host_state, ws.state, sizeof(NewtonState), cudaMemcpyDeviceToHost, st));
        SRI_CUDA(cudaStreamSynchronize(st));
        singular = ws.host_state->singular;
    }
    rep.singular_solves = (int64_t)singular;
    if (B > 0) {
        SRI_CUDA(cudaMemcpyAsync(qe, ws.qe, sizeof(double) * n * B, cudaMemcpyDefault, st));
        SRI_CUDA(cudaStreamSynchronize(st));
    }
    if (report) *report = rep;
    return SRI_OK;
}

int sri_newton_static_shape(sri_handle h, int64_t batch, int ne, const double* H_diag, const double* F_tip,
                            const double* M_tip, const double* K0, double* qe, double tol, int max_iter, double fd_step,
                            int64_t total_dof, sri_allreduce_fn reduce, void* reduce_ctx, sri_newton_report* report) {
    SRI_ENTER(h);
    sri_static_problem P{};
    P.batch = batch; P.ne = ne; P.H_diag = H_diag; P.F_tip = F_tip; P.M_tip = M_tip; P.K0 = K0;
    return newton_static_problem(h, P, qe, tol, max_iter, fd_step, total_dof, reduce, reduce_ctx, report, "sri_newton_static_shape");
}

int sri_newton_static_problem(sri_handle h, const sri_static_problem* problem, double* qe, double tol, int max_iter,
                              double fd_step, int64_t total_dof, sri_allreduce_fn reduce, void* reduce_ctx,
                              sri_newton_report* report) {
    SRI_ENTER(h);
    if (!problem) return fail(SRI_ERR_INVALID_ARGUMENT, "sri_newton_static_problem: problem is required");
    return newton_static_problem(h, *problem, qe, tol, max_iter, fd_step, total_dof, reduce, reduce_ctx, report,
                                 "sri_newton_static_problem");
}

// ---- several devices in one process ------------------------------------------------------------------------------------

}  // extern "C"

struct sri_multi_context {
    int N = 0;
    std::vector<int> devices;
    std::vector<sri_handle> handles;
};

namespace {

// the rods [first, first + count) of a whole-batch description with HOST pointers
sri_rod_batch shard_of(const sri_rod_batch& r, int N, int64_t first, int64_t count) {
    const int M = N - 1;
    sri_rod_batch s = r;
    s.batch = count;
    auto adv = [first](const double* p, size_t per_rod) { return p ? p + (size_t)first * per_rod : nullptr; };
    auto advw = [first](double* p, size_t per_rod) { return p ? p + (size_t)first * per_rod : nullptr; };
    s.K = adv(r.K, 3 * N); s.q0 = adv(r.q0, 4); s.r0 = adv(r.r0, 3); s.Gamma = adv(r.Gamma, 3 * N);
    s.fbar = adv(r.fbar, 3 * N); s.lbar = adv(r.lbar, 3 * N); s.F_tip = adv(r.F_tip, 3); s.M_tip = adv(r.M_tip, 3);
    s.Q = advw(r.Q, 4 * M); s.r = advw(r.r, 3 * M); s.n = advw(r.n, 3 * M); s.m = advw(r.m, 3 * M);
    s.info = r.info ? r.info + first : nullptr;
    return s;
}

// Runs fn(g) on one host thread per device and returns the first failure (its message becomes this thread's
// sri_last_error_string; g_last_error is thread-local).
template <typename Fn>
int for_each_device(sri_multi_context* mh, Fn fn) {
    const int G = (int)mh->handles.size();
    std::vector<int> rc(G, SRI_OK);
    std::vector<std::string> msg(G);
    std::vector<std::thread> threads;
    threads.reserve(G);
    for (int g = 0; g < G; ++g)
        threads.emplace_back([&, g]() {
            rc[g] = fn(g);
            if (rc[g] != SRI_OK) msg[g] = g_last_error;
        });
    for (auto& t : threads) t.join();
    int worst = SRI_OK;
    for (int g = 0; g < G; ++g)
        if (rc[g] != SRI_OK && (worst == SRI_OK || worst == SRI_ERR_SINGULAR)) {  // a hard error outranks "some rod was singular"
            worst = rc[g];
            g_last_error = "device " + std::to_string(mh->devices[g]) + ": " + msg[g];
        }
    return worst;
}

// sum / max of the per-thread norms between the device threads of one process, added in shard order
struct ThreadReduce {
    std::mutex mu;
    std::condition_variable cv;
    int n = 0, arrived = 0;
    long generation = 0;
    bool failed = false;
    std::vector<double> parts;
    double out[2] = {0.0, 0.0};
};
struct ThreadReduceCtx { ThreadReduce* red; int rank; };
int thread_reduce_callback(double* v, void* ctx_) {
    auto* ctx = static_cast<ThreadReduceCtx*>(ctx_);
    ThreadReduce& R = *ctx->red;
    std::unique_lock<std::mutex> lock(R.mu);
    if (R.failed) return 1;
    R.parts[2 * ctx->rank] = v[0];
    R.parts[2 * ctx->rank + 1] = v[1];
    if (++R.arrived == R.n) {
        double s = 0.0, m = 0.0;
        for (int r = 0; r < R.n; ++r) { s += R.parts[2 * r]; m = std::max(m, R.parts[2 * r + 1]); }
        R.out[0] = s; R.out[1] = m;
        R.arrived = 0;
        ++R.generation;
        R.cv.notify_all();
    } else {
        const long gen = R.generation;
        R.cv.wait(lock, [&] { return R.generation != gen || R.failed; });
        if (R.generation == gen) return 1;  // another shard failed
    }
    v[0] = R.out[0]; v[1] = R.out[1];
    return 0;
}

}  // namespace

extern "C" {

int sri_shard_range(int64_t total, int rank, int world, int64_t* first, int64_t* last) {
    if (total < 0 || world < 1 || rank < 0 || rank >= world || !first || !last) return fail(SRI_ERR_INVALID_ARGUMENT, "sri_shard_range: bad arguments");
    // floor(rank * total / world) without overflow for any int64 total
    auto cut = [&](int64_t r) { return (int64_t)(((__int128)r * (__int128)total) / world); };
    *first = cut(rank);
    *last = cut(rank + 1);
    return SRI_OK;
}

int sri_device_count(int* ndev) {
    if (!ndev) return fail(SRI_ERR_INVALID_ARGUMENT, "sri_device_count: null argument");
    *ndev = 0;
    SRI_CUDA(cudaGetDeviceCount(ndev));
    return SRI_OK;
}

int sri_create_multi(int N, const int* devices, int ndev, sri_multi_handle* out) {
    if (!out) return fail(SRI_ERR_INVALID_ARGUMENT, "sri_create_multi: out == NULL");
    *out = nullptr;
    if (ndev < 1) return fail(SRI_ERR_INVALID_ARGUMENT, "sri_create_multi: ndev must be >= 1");
    sri_multi_context* mh = new (std::nothrow) sri_multi_context();
    if (!mh) return fail(SRI_ERR_ALLOC, "sri_create_multi: out of host memory");
    mh->N = N;
    for (int g = 0; g < ndev; ++g) {
        const int dev = devices ? devices[g] : g;
        sri_handle h = nullptr;
        const int rc = sri_create(N, dev, &h);
        if (rc != SRI_OK) {
            const std::string keep = g_last_error;
            sri_destroy_multi(mh);
            g_last_error = keep;
            return rc;
        }
        mh->devices.push_back(dev);
        mh->handles.push_back(h);
    }
    *out = mh;
    return SRI_OK;
}

int sri_destroy_multi(sri_multi_handle mh) {
    if (!mh) return SRI_OK;
    for (sri_handle h : mh->handles) sri_destroy(h);
    delete mh;
    return SRI_OK;
}

int sri_multi_device_count(sri_multi_handle mh, int* ndev) {
    if (!mh || !ndev) return fail(SRI_ERR_INVALID_ARGUMENT, "sri_multi_device_count: null argument");
    *ndev = (int)mh->handles.size();
    return SRI_OK;
}

int sri_multi_get_handle(sri_multi_handle mh, int index, sri_handle* h) {
    if (!mh || !h || index < 0 || index >= (int)mh->handles.size()) return fail(SRI_ERR_INVALID_ARGUMENT, "sri_multi_get_handle: bad arguments");
    *h = mh->handles[index];
    return SRI_OK;
}

int sri_integrate_all_sharded(sri_multi_handle mh, const sri_rod_batch* rods) {
    if (!mh || !rods) return fail(SRI_ERR_INVALID_ARGUMENT, "sri_integrate_all_sharded: null argument");
    if (rods->batch < 0) return fail(SRI_ERR_INVALID_ARGUMENT, "sri_integrate_all_sharded: negative batch");
    if (rods->batch == 0) return SRI_OK;
    if (!all_host_pointers(rods)) return fail(SRI_ERR_INVALID_ARGUMENT, "sri_integrate_all_sharded: host pointers only (use sri_integrate_all_per_device for resident data)");
    const int G = (int)mh->handles.size();
    return for_each_device(mh, [&](int g) -> int {
        int64_t first = 0, last = 0;
        SRI_TRY(sri_shard_range(rods->batch, g, G, &first, &last));
        if (last == first) return SRI_OK;
        const sri_rod_batch mine = shard_of(*rods, mh->N, first, last - first);
        return sri_integrate_all(mh->handles[g], &mine);
    });
}

int sri_integrate_all_per_device(sri_multi_handle mh, const sri_rod_batch* per_device) {
    if (!mh || !per_device) return fail(SRI_ERR_INVALID_ARGUMENT, "sri_integrate_all_per_device: null argument");
    const int G = (int)mh->handles.size();
    for (int g = 0; g < G; ++g)  // device buffers: every call returns as soon as its kernels are queued
        if (per_device[g].batch > 0) SRI_TRY(sri_integrate_all(mh->handles[g], &per_device[g]));
    for (int g = 0; g < G; ++g) SRI_TRY(sri_synchronize(mh->handles[g]));
    return SRI_OK;
}

}  // extern "C"

// `who` names the entry point in error messages.
static int newton_static_problem_sharded(sri_multi_handle mh, const sri_static_problem& P, double* qe, double tol, int max_iter,
                                         double fd_step, sri_newton_report* report, const char* who) {
    if (!mh) return fail(SRI_ERR_INVALID_ARGUMENT, std::string(who) + ": null handle");
    const int64_t batch = P.batch;
    const int ne = P.ne;
    if (batch < 0 || ne < 1 || ne > 8 || !P.H_diag || (batch > 0 && (!P.F_tip || !P.M_tip || !qe)))
        return fail(SRI_ERR_INVALID_ARGUMENT, std::string(who) + ": bad arguments");
    for (const void* p : {(const void*)P.H_diag, (const void*)P.F_tip, (const void*)P.M_tip, (const void*)P.K0, (const void*)P.q0,
                          (const void*)P.Gamma, (const void*)P.fbar, (const void*)P.lbar, (const void*)qe})
        if (p && is_device_pointer(p)) return fail(SRI_ERR_INVALID_ARGUMENT, std::string(who) + ": host pointers only");
    const int G = (int)mh->handles.size(), N = mh->N, n = 3 * ne;
    ThreadReduce red;
    red.n = G;
    red.parts.assign(2 * (size_t)G, 0.0);
    std::vector<sri_newton_report> reps(G);
    const int rc = for_each_device(mh, [&](int g) -> int {
        int64_t first = 0, last = 0;
        int r = sri_shard_range(batch, g, G, &first, &last);
        ThreadReduceCtx ctx{&red, g};
        auto adv = [first](const double* p, size_t per_rod) { return p ? p + (size_t)first * per_rod : nullptr; };
        sri_static_problem mine = P;
        mine.batch = last - first;
        mine.F_tip = adv(P.F_tip, 3); mine.M_tip = adv(P.M_tip, 3); mine.K0 = adv(P.K0, (size_t)3 * N);
        mine.q0 = adv(P.q0, 4); mine.Gamma = adv(P.Gamma, (size_t)3 * N); mine.fbar = adv(P.fbar, (size_t)3 * N);
        mine.lbar = adv(P.lbar, (size_t)3 * N);
        if (r == SRI_OK)
            r = sri_newton_static_problem(mh->handles[g], &mine, qe ? qe + (size_t)n * first : nullptr, tol, max_iter, fd_step,
                                          (int64_t)n * batch, thread_reduce_callback, &ctx, &reps[g]);
        if (r != SRI_OK) {  // release the shards waiting in the reduction
            std::lock_guard<std::mutex> lock(red.mu);
            red.failed = true;
            red.cv.notify_all();
        }
        return r;
    });
    if (rc != SRI_OK) return rc;
    if (report) {
        *report = reps[0];
        for (int g = 1; g < G; ++g) report->singular_solves += reps[g].singular_solves;
    }
    return SRI_OK;
}

extern "C" {

int sri_newton_static_shape_sharded(sri_multi_handle mh, int64_t batch, int ne, const double* H_diag, const double* F_tip,
                                    const double* M_tip, const double* K0, double* qe, double tol, int max_iter,
                                    double fd_step, sri_newton_report* report) {
    sri_static_problem P{};
    P.batch = batch; P.ne = ne; P.H_diag = H_diag; P.F_tip = F_tip; P.M_tip = M_tip; P.K0 = K0;
    return newton_static_problem_sharded(mh, P, qe, tol, max_iter, fd_step, report, "sri_newton_static_shape_sharded");
}

int sri_newton_static_problem_sharded(sri_multi_handle mh, const sri_static_problem* problem, double* qe, double tol,
                                      int max_iter, double fd_step, sri_newton_report* report) {
    if (!problem) return fail(SRI_ERR_INVALID_ARGUMENT, "sri_newton_static_problem_sharded: problem is required");
    return newton_static_problem_sharded(mh, *problem, qe, tol, max_iter, fd_step, report, "sri_newton_static_problem_sharded");
}

int sri_generate_rods(sri_handle h, uint64_t seed, int64_t first_rod, int64_t batch, double* K, double* F_tip,
                      double* M_tip, double* fbar) {
    SRI_ENTER(h);
    if (batch < 0 || first_rod < 0) return fail(SRI_ERR_INVALID_ARGUMENT, "sri_generate_rods: bad arguments");
    if (batch == 0) return SRI_OK;
    for (const void* p : {(const void*)K, (const void*)F_tip, (const void*)M_tip, (const void*)fbar})
        if (p && !is_device_pointer(p)) return fail(SRI_ERR_INVALID_ARGUMENT, "sri_generate_rods: device pointers only");
    return launch(generate_rods_kernel, (unsigned)((batch + 127) / 128), 128, 0, h->stream, seed, first_rod, batch, h->N, h->d_tnodes, K,
                  F_tip, M_tip, fbar);
}

int sri_get_handback_count(sri_handle h, int64_t* count) {
    SRI_ENTER(h);
    if (!count) return fail(SRI_ERR_INVALID_ARGUMENT, "sri_get_handback_count: null argument");
    *count = 0;
    const int slot = h->last_handback_slot;
    if ((slot == 3 && !h->use_dmma) || !h->d_list[slot]) return SRI_OK;
    int c = 0;
    SRI_CUDA(cudaMemcpyAsync(&c, h->d_list[slot], sizeof(int), cudaMemcpyDeviceToHost, h->stream));
    SRI_CUDA(cudaStreamSynchronize(h->stream));
    *count = c;
    return SRI_OK;
}

static int measure_peak(sri_handle h, bool tensor, double* tflops) {
    double* d = nullptr;
    SRI_CUDA(cudaMalloc(&d, 8));
    const int iters = tensor ? 2048 : 8192, threads = 512, blocks = h->sm_count * 2;
    cudaEvent_t e0, e1;
    SRI_CUDA(cudaEventCreate(&e0));
    SRI_CUDA(cudaEventCreate(&e1));
    float best = 1e30f;
    for (int rep = 0; rep < 6; ++rep) {
        SRI_CUDA(cudaEventRecord(e0, h->stream));
        SRI_TRY(launch(tensor ? dmma_peak_kernel : fp64_peak_kernel, blocks, threads, 0, h->stream, d, iters, 0.5));
        SRI_CUDA(cudaEventRecord(e1, h->stream));
        SRI_CUDA(cudaEventSynchronize(e1));
        float ms = 0;
        SRI_CUDA(cudaEventElapsedTime(&ms, e0, e1));
        if (rep > 0 && ms < best) best = ms;
    }
    cudaEventDestroy(e0);
    cudaEventDestroy(e1);
    cudaFree(d);
    // per thread and iteration: 16 FMA (scalar) or 16 DMMA x 256 FMA / 32 lanes = 128 FMA (tensor)
    *tflops = 2.0 * (tensor ? 128.0 : 16.0) * iters * (double)blocks * threads / (best * 1e-3) * 1e-12;
    return SRI_OK;
}

int sri_measure_fp64_peak(sri_handle h, double* tflops) {
    SRI_ENTER(h);
    if (!tflops) return fail(SRI_ERR_INVALID_ARGUMENT, "sri_measure_fp64_peak: null argument");
    return measure_peak(h, false, tflops);
}

int sri_measure_dmma_peak(sri_handle h, double* tflops) {
    SRI_ENTER(h);
    if (!tflops) return fail(SRI_ERR_INVALID_ARGUMENT, "sri_measure_dmma_peak: null argument");
    return measure_peak(h, true, tflops);
}

}  // extern "C"
