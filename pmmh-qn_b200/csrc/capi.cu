// capi.cu -- extern "C" boundary of libpmmh_qn_b200.so (declared in include/pmmh_qn.h).
// Plain pointers and sizes in, status codes out; no torch types, no CPU fallback.
#include <cuda_runtime.h>
#include <stdint.h>
#include <math.h>
#include <stdio.h>
#include <string.h>

#include <mutex>
#include <string>
#include <vector>

#include "../../include/pmmh_qn.h"
#include "aux_kernels.cuh"
#include "pf_model.cuh"
#include "sv_filter.cuh"
#include "sv_grid.cuh"
#include "sv_split.cuh"

namespace {

thread_local std::string g_last_error;

int fail(int code, const char* what) {
    g_last_error = what;
    return code;
}
int fail_cuda(cudaError_t err, const char* where) {
    char buf[512];
    snprintf(buf, sizeof(buf), "%s: %s", where, cudaGetErrorString(err));
    g_last_error = buf;
    return PMMH_ERR_CUDA;
}
#define PMMH_CUDA(call)                                       \
    do {                                                      \
        cudaError_t e__ = (call);                             \
        if (e__ != cudaSuccess) return fail_cuda(e__, #call); \
    } while (0)

}  // namespace

namespace pmmh {
// error plumbing for the other translation units (sv_split.cu)
int set_error(int code, const char* what) { return fail(code, what); }
int set_cuda_error(cudaError_t err, const char* where) { return fail_cuda(err, where); }
}  // namespace pmmh

namespace {

struct DeviceInfo {
    int sm = 0, major = 0, minor = 0, coop = 0;
    bool ok = false;
};

int get_device_info(DeviceInfo* out) {
    static thread_local DeviceInfo cache[64];
    int dev = 0;
    cudaError_t err = cudaGetDevice(&dev);
    if (err != cudaSuccess) return fail_cuda(err, "cudaGetDevice");
    if (dev < 0 || dev >= 64) return fail(PMMH_ERR_NO_DEVICE, "device ordinal out of range");
    DeviceInfo& d = cache[dev];
    if (!d.ok) {
        PMMH_CUDA(cudaDeviceGetAttribute(&d.sm, cudaDevAttrMultiProcessorCount, dev));
        PMMH_CUDA(cudaDeviceGetAttribute(&d.major, cudaDevAttrComputeCapabilityMajor, dev));
        PMMH_CUDA(cudaDeviceGetAttribute(&d.minor, cudaDevAttrComputeCapabilityMinor, dev));
        PMMH_CUDA(cudaDeviceGetAttribute(&d.coop, cudaDevAttrCooperativeLaunch, dev));
        d.ok = true;
    }
    *out = d;
    return PMMH_OK;
}

// an sm_100 device and, for the kernels that need it, cooperative launch
int check_device(const DeviceInfo& di, bool coop) {
    if (di.major < 10) return fail(PMMH_ERR_NO_DEVICE, "an sm_100 (B200) device is required");
    if (coop && !di.coop) return fail(PMMH_ERR_NO_DEVICE, "device lacks cooperative launch");
    return PMMH_OK;
}

// The SV smoother's kernels (diag[PMMH_DIAG_KERNEL] in brackets)
enum class SvKernel {
    None,            // host-streamed entry: no kernel takes the sizes (the call is refused)
    General,         // sv_filter.cu, any problem (diag 1)
    Chain,           // sv_chain.cu, one CTA per problem (diag 3)
    Grid,            // sv_grid.cu, one problem, one tile per CTA (diag 5)
    StreamRecords,   // sv_split.cu, one problem, genealogy records (diag 4)
    StreamPath,      // sv_split.cu, one problem, path storage (diag 4)
    Exchange,        // sv_fast.cu, teams of CTAs (diag 2)
};
// pmmh_flps_sv_corr / pmmh_bpf_sv_corr (u in device memory) or pmmh_flps_sv_corr_streamed (u in host memory)
enum class SvEntry { Resident, HostStreamed };

struct SvShape {
    int nobs, n, lag, batch, hess, mode, hist, ctas;
};

struct SvChoice {
    SvKernel kernel;
    bool fallback;   // the general kernel re-runs the problems `kernel` abandoned (diag status 1)
    int G;           // general kernel: CTAs per problem (its summation order depends on it); exchange kernel too
    int grid_G;      // grid kernel: CTAs (tiles)
    int NSUB, CP;    // exchange kernel
};

struct SvPlan {
    SvChoice c;
    // general kernel
    int G, n_teams, grid, NB, RING, SQ, SQW;
    size_t stamp_bytes, sync_bytes, team_stride;
    // chain / exchange kernel
    size_t chain_stride, fast_sync_bytes, fast_team_stride;
    size_t total;   // the chosen kernel's workspace; on the resident entry at least the general kernel's
};

// pmmh_sv_set_algorithm (0 = automatic; how each value selects the kernel: sv_choose).
// The selection is per host thread (thread_local): a thread that calls pmmh_sv_set_algorithm changes the
// sizing and the kernel choice of its own later calls only, so a toggle on one thread cannot land between
// another thread's workspace query and its run call.
thread_local int g_sv_algorithm = 0;
constexpr int kSplitMinParticles = 1 << 20;       // automatic selection of the streaming kernels from this N on
constexpr int kSplitPathMaxParticles = 1 << 23;   // ... with path storage below this N, with records from it on
constexpr int kGridMinParticles = 1 << 14;        // automatic selection of the grid kernel from this N on (while a tile fits one CTA)
constexpr int kGridHessMinParticles = 1 << 14;    // ... with the Hessian branch (T = 1000: 51.8 ms against 101.8 ms on the general kernel at 2^14)
long long* g_sv_prof = nullptr;   // development: per-CTA phase clocks of the exchange kernel
constexpr int kMaxDynSmem = 227 * 1024;

// Does the exchange kernel take N particles on G CTAs per problem?
bool exchange_fits(int n, int G, int* nsub, int* cp) {
    if (!pmmh::sv_fast_eligible(n, G)) return false;
    *nsub = pmmh::sv_fast_nsub(n, G);
    *cp = pmmh::sv_fast_pair_cap(n, G);
    const long long nv = (long long)G * G * (pmmh::kFastThreads / 32) * *cp;
    return nv < (1ll << 31) && pmmh::sv_fast_smem_bytes(n, G, *nsub) <= kMaxDynSmem &&
           2 * *nsub + 10 <= pmmh::kMaxAllgatherHost;
}

// The kernel that evaluates shape `s` under algorithm A on `sm` SMs.  In order:
//  1. chain: flps, A in {0, 3}, ctas <= 1, N <= 4096, lag <= 10 and its shared memory fits (resident entry
//     only; where the rule holds but the kernel cannot run, G = 1 keeps the exchange kernel out as well);
//  2. grid: flps, one problem, A = 6 or automatically (A = 0, ctas = 0) from N = 2^14 on, while a tile of
//     N / G particles fits one CTA; the host-streamed entry takes it only with ctas = 0;
//  3. streaming (resident entry): flps without Hessian or history, one problem, ctas = 0, A in {4, 5} or
//     automatically from N = 2^20 on: there they are as fast as the exchange kernel or faster (174.7 vs
//     181.0 ms at N = 2^20, T = 1000) and have no size limit (the exchange kernel stops at ~1.16 M
//     particles; the general kernel is ~4x slower).  Path storage for A = 5 or, automatically, while its
//     jump tables stay (mostly) L2 resident (7.2e9 vs 6.4e9 particle-steps/s at N = 2^22); records from
//     N = 2^23 on (6.45e9 vs 6.24e9 at 2^23, 5.8e9 vs 4.9e9 at 2^24: random 4-byte reads from HBM);
//  4. exchange: flps without Hessian, A = 2 or automatically for teams of CTAs (G > 1: one CTA per problem
//     has no exchange to save, the general kernel is faster there: 8.8e9 vs 7.0e9 particle-steps/s at
//     1024 x N = 4096).  The host-streamed entry tries it before the streaming kernels (at N = 2^20: 206 ms
//     per call against 242 ms, whose strided reads of the particle-major slots cost more than they save)
//     and takes those (path storage only) for A in {0, 5} from N = 2^20 on;
//  5. the general kernel on the resident entry; the host-streamed entry has none left and refuses.
// With A = 0 the general kernel follows a special kernel as the fallback pass; A = 2 .. 6 run theirs alone.
SvChoice sv_choose(const SvShape& s, int A, SvEntry entry, int sm) {
    const bool resident = entry == SvEntry::Resident;
    const bool flps = s.mode == pmmh::kSvFlps;
    SvChoice c = {};
    const bool chain_rule = flps && (A == 0 || A == 3) && s.ctas <= 1 && pmmh::sv_chain_eligible(s.n, s.lag);
    int G;
    if (s.ctas > 0) G = s.ctas;
    else if (chain_rule) G = 1;
    else if (s.batch > 1) G = (s.n + 4095) / 4096;
    else G = (s.n + 1023) / 1024;
    if (G < 1) G = 1;
    if (G > sm) G = sm;
    c.G = G;
    c.grid_G = pmmh::sv_grid_ctas(s.n, sm, s.ctas);
    auto pick = [&](SvKernel k) {
        c.kernel = k;
        c.fallback = resident && A == 0 && k != SvKernel::General;
        return c;
    };
    if (resident && chain_rule && pmmh::sv_chain_smem_bytes(s.n) <= kMaxDynSmem) return pick(SvKernel::Chain);
    const int grid_min = s.hess ? kGridHessMinParticles : kGridMinParticles;
    if (flps && s.batch == 1 && (resident || s.ctas == 0) &&
        (A == 6 || (A == 0 && s.ctas == 0 && s.n >= grid_min)) &&
        pmmh::sv_grid_eligible(s.nobs, s.n, s.lag, c.grid_G))
        return pick(SvKernel::Grid);
    const bool stream_wanted = resident ? (A == 4 || A == 5 || (A == 0 && s.n >= kSplitMinParticles))
                                        : ((A == 0 || A == 5) && s.n >= kSplitMinParticles);
    const bool stream = flps && !s.hess && s.batch == 1 && !s.hist && s.ctas == 0 && stream_wanted &&
                        pmmh::sv_split_single_eligible(s.nobs, s.n, s.lag);
    const bool path = !resident || A == 5 || (A == 0 && s.n < kSplitPathMaxParticles);
    const SvKernel streaming = path ? SvKernel::StreamPath : SvKernel::StreamRecords;
    if (resident && stream) return pick(streaming);
    if (flps && !s.hess && (A == 2 || (A == 0 && G > 1)) && exchange_fits(s.n, G, &c.NSUB, &c.CP))
        return pick(SvKernel::Exchange);
    if (stream) return pick(streaming);
    return pick(resident ? SvKernel::General : SvKernel::None);
}

int sv_make_plan(SvShape s, SvEntry entry, SvPlan* p) {
    if (s.nobs < 2 || s.n < 1 || s.batch < 1) return fail(PMMH_ERR_INVALID, "sizes must be positive");
    if (s.mode == pmmh::kSvFlps) {
        if (s.lag < 2 || s.lag >= 64) return fail(PMMH_ERR_INVALID, "lag must be in [2, 63]");
        if (s.nobs < s.lag + 1) return fail(PMMH_ERR_INVALID, "n_obs must be at least lag + 1");
    } else {
        s.lag = 2;
    }
    if ((long long)s.n + s.nobs >= (1ll << 31)) return fail(PMMH_ERR_INVALID, "n_particles too large");
    DeviceInfo di;
    int rc = get_device_info(&di);
    if (rc == PMMH_OK) rc = check_device(di, true);
    if (rc != PMMH_OK) return rc;
    memset(p, 0, sizeof(*p));
    p->c = sv_choose(s, g_sv_algorithm, entry, di.sm);
    const int G = p->c.G, n = s.n, nobs = s.nobs;
    int n_teams = di.sm / G;
    if (n_teams > s.batch) n_teams = s.batch;
    if (n_teams < 1) n_teams = 1;
    p->G = G;
    p->n_teams = n_teams;
    p->grid = G * n_teams;
    p->NB = ((n + 31) / 32) * 32;
    if (p->NB < 64) p->NB = 64;
    p->RING = s.lag + 1;
    p->SQ = s.hess ? (nobs + n - 2) / nobs + 1 : 1;
    p->SQW = (s.mode != pmmh::kSvFlps) ? (n + nobs - 1) / nobs : 0;
    p->stamp_bytes = pmmh::sv_align((size_t)p->grid * sizeof(unsigned));
    p->sync_bytes = p->stamp_bytes +
                    pmmh::sv_align((size_t)n_teams * 2 * G * pmmh::kMaxAllgatherHost * sizeof(double));
    p->team_stride = pmmh::sv_ws_layout(n, nobs, s.lag, p->NB, p->RING, s.hess, s.mode, p->SQ, p->SQW,
                                        s.hist, nullptr, nullptr);
    // the general kernel (the fallback pass) uses the head of the chosen kernel's workspace
    if (entry == SvEntry::Resident) p->total = p->sync_bytes + (size_t)n_teams * p->team_stride;
    size_t kernel_bytes = 0;
    switch (p->c.kernel) {
    case SvKernel::Chain:
        p->chain_stride = pmmh::sv_chain_ws_bytes(n, s.lag, nobs, s.hess, 0);
        kernel_bytes = (size_t)p->grid * p->chain_stride;
        break;
    case SvKernel::Grid:
        kernel_bytes = pmmh::sv_grid_ws_bytes(nobs, n, s.lag, p->c.grid_G, s.hist, s.hess);
        break;
    case SvKernel::StreamRecords: kernel_bytes = pmmh::sv_split_single_ws_bytes(nobs, n, s.lag); break;
    case SvKernel::StreamPath: kernel_bytes = pmmh::sv_split_path_ws_bytes(nobs, n, s.lag); break;
    case SvKernel::Exchange:
        p->fast_sync_bytes = pmmh::sv_fast_sync_bytes(G, n_teams);
        p->fast_team_stride = pmmh::sv_fast_ws_bytes(n, G, p->c.NSUB, p->c.CP, s.lag, s.hist);
        kernel_bytes = p->fast_sync_bytes + (size_t)n_teams * p->fast_team_stride;
        break;
    default: break;
    }
    if (kernel_bytes > p->total) p->total = kernel_bytes;
    return PMMH_OK;
}

// Arguments of the general, chain and exchange kernels (the ws_* fields are per kernel)
pmmh::SvArgs sv_args(const SvPlan& p, const SvShape& s, const pmmh::SvCall& c) {
    pmmh::SvArgs a;
    memset(&a, 0, sizeof(a));
    a.N = s.n;
    a.NOBS = s.nobs;
    a.LAG = (s.mode == pmmh::kSvFlps) ? s.lag : 2;
    a.B = s.batch;
    a.G = p.G;
    a.n_teams = p.n_teams;
    a.NB = p.NB;
    a.RING = p.RING;
    a.mode = s.mode;
    a.hess = s.hess;
    a.model_id = c.model;
    a.SQ = p.SQ;
    a.SQW = p.SQW;
    a.obs = c.obs;
    a.obs_stride = c.obs_stride;
    a.params = c.params;
    a.rvr = c.rvr;
    a.U = c.u;
    a.u_chunk = c.slot;
    a.u_ready = c.u_flag;
    a.filt = c.filt;
    a.smo = c.smo;
    a.loglike = c.ll;
    a.grad = c.grad;
    a.traj = c.traj;
    a.hess1 = c.hess1;
    a.hess2 = c.hess2;
    a.diag = c.diag;
    a.Xhist = c.x_hist;
    a.Ahist = c.a_hist;
    a.prof = c.prof;
    a.ws = (char*)c.ws;
    return a;
}

cudaError_t exchange_launch(const SvPlan& p, pmmh::SvArgs& a, cudaStream_t st) {
    a.NSUB = p.c.NSUB;
    a.CP = p.c.CP;
    a.ws_sync_bytes = p.fast_sync_bytes;
    a.ws_team_stride = p.fast_team_stride;
    cudaError_t err = cudaMemsetAsync(a.ws, 0, p.fast_sync_bytes, st);
    return err != cudaSuccess ? err : pmmh::sv_fast_launch(a, p.grid, st);
}

// Runs the plan's kernel on call `c`, then the general kernel where it is the plan's kernel or its fallback pass
// (in the same stream, reusing the workspace).  The grid kernel without its Hessian branch and the streaming
// kernels write no Hessian: where the entry has Hessian outputs they are zeroed.
int sv_launch_plan(const SvPlan& p, const SvShape& s, const pmmh::SvCall& c) {
    pmmh::SvArgs a = sv_args(p, s, c);
    int rc = PMMH_OK;
    bool zero_hess = false;
    switch (p.c.kernel) {
    case SvKernel::Chain:
        a.ws_team_stride = p.chain_stride;
        PMMH_CUDA(pmmh::sv_chain_launch(a, p.grid, c.filter, c.stream));
        break;
    case SvKernel::Grid:
        rc = pmmh::sv_grid_run(c, 1, s.nobs, s.n, s.lag, p.c.grid_G, 1, s.hess);
        zero_hess = !s.hess;
        break;
    case SvKernel::StreamRecords:
        rc = pmmh::sv_split_single_run(c, s.nobs, s.n, s.lag);
        zero_hess = true;
        break;
    case SvKernel::StreamPath:
        rc = pmmh::sv_split_path_run(c, s.nobs, s.n, s.lag);
        zero_hess = true;
        break;
    case SvKernel::Exchange:
        PMMH_CUDA(exchange_launch(p, a, c.stream));
        break;
    default: break;
    }
    if (rc != PMMH_OK) return rc;
    if (zero_hess && c.hess1) {
        PMMH_CUDA(cudaMemsetAsync(c.hess1, 0, 16 * sizeof(double), c.stream));
        PMMH_CUDA(cudaMemsetAsync(c.hess2, 0, 16 * sizeof(double), c.stream));
    }
    if (p.c.kernel != SvKernel::General) {
        if (!p.c.fallback) return PMMH_OK;
        a.only_failed = 1;
    }
    a.ws_sync_bytes = p.sync_bytes;
    a.ws_team_stride = p.team_stride;
    PMMH_CUDA(cudaMemsetAsync(c.ws, 0, p.stamp_bytes, c.stream));
    PMMH_CUDA(pmmh::sv_launch(a, p.grid, c.stream));
    return PMMH_OK;
}

int sv_run(int mode, const double* d_obs, long long obs_stride, const double* d_params,
           const double* d_rvr, const double* d_u, int nobs, int n, int lag, int batch, int hess,
           double* d_filt, double* d_smo, double* d_ll, double* d_grad, double* d_traj, double* d_h1,
           double* d_h2, long long* d_diag, double* d_xh, int* d_ah, void* d_ws, size_t ws_bytes,
           int ctas, void* stream) {
    if (!d_obs || !d_params || !d_rvr || !d_u || !d_filt || !d_ll || !d_traj || !d_diag || !d_ws)
        return fail(PMMH_ERR_INVALID, "null pointer argument");
    if (mode == pmmh::kSvFlps && (!d_smo || !d_grad || !d_h1 || !d_h2))
        return fail(PMMH_ERR_INVALID, "null output pointer");
    if ((d_xh == nullptr) != (d_ah == nullptr))
        return fail(PMMH_ERR_INVALID, "d_x_hist and d_a_hist must be given together");
    const SvShape s = {nobs, n, lag, batch, hess, mode, d_xh != nullptr, ctas};
    SvPlan p;
    int rc = sv_make_plan(s, SvEntry::Resident, &p);
    if (rc != PMMH_OK) return rc;
    if (ws_bytes < p.total) return fail(PMMH_ERR_WORKSPACE, "workspace too small");
    pmmh::SvCall c = {};
    c.obs = d_obs; c.obs_stride = obs_stride; c.params = d_params; c.rvr = d_rvr; c.u = d_u;
    c.filt = d_filt; c.smo = d_smo; c.ll = d_ll; c.grad = d_grad; c.traj = d_traj; c.hess1 = d_h1; c.hess2 = d_h2;
    c.diag = d_diag; c.x_hist = d_xh; c.a_hist = d_ah; c.prof = g_sv_prof;
    c.ws = d_ws; c.ws_bytes = ws_bytes; c.stream = (cudaStream_t)stream;
    return sv_launch_plan(p, s, c);
}

struct DevBuf {
    void* p = nullptr;
    ~DevBuf() {
        if (p) cudaFree(p);
    }
    cudaError_t alloc(size_t bytes) { return cudaMalloc(&p, bytes ? bytes : 1); }
    template <typename T>
    T* as() {
        return (T*)p;
    }
};

}  // namespace

extern "C" {

int pmmh_version(void) { return 100; }

const char* pmmh_last_error(void) { return g_last_error.c_str(); }

int pmmh_device_info(int* sm_count, int* cc_major, int* cc_minor) {
    DeviceInfo di;
    int rc = get_device_info(&di);
    if (rc != PMMH_OK) return rc;
    if (sm_count) *sm_count = di.sm;
    if (cc_major) *cc_major = di.major;
    if (cc_minor) *cc_minor = di.minor;
    return PMMH_OK;
}

int pmmh_sv_set_algorithm(int algorithm) {
    if (algorithm < 0 || algorithm > 6) return fail(PMMH_ERR_INVALID, "algorithm must be 0 .. 6");
    g_sv_algorithm = algorithm;
    return PMMH_OK;
}

int pmmh_sv_debug_profile(long long* d_clocks) {
    g_sv_prof = d_clocks;
    return PMMH_OK;
}

int pmmh_sv_workspace_bytes(int n_obs, int n_particles, int lag, int batch, int compute_hessian,
                            int mode, int have_history, int ctas_per_problem, size_t* bytes) {
    if (!bytes) return fail(PMMH_ERR_INVALID, "bytes is null");
    SvPlan p;
    int rc = sv_make_plan({n_obs, n_particles, lag, batch, compute_hessian,
                           mode == 0 ? pmmh::kSvFlps : pmmh::kSvBpfParity, have_history, ctas_per_problem},
                          SvEntry::Resident, &p);
    if (rc != PMMH_OK) return rc;
    *bytes = p.total;
    return PMMH_OK;
}

int pmmh_flps_sv_corr(const double* d_obs, long long obs_stride, const double* d_params,
                      const double* d_rvr, const double* d_u, int n_obs, int n_particles, int lag,
                      int batch, int compute_hessian, double* d_filt, double* d_smo,
                      double* d_log_like, double* d_gradient, double* d_traj, double* d_hess1,
                      double* d_hess2, long long* d_diag, double* d_x_hist, int* d_a_hist,
                      void* d_workspace, size_t workspace_bytes, int ctas_per_problem, void* stream) {
    return sv_run(pmmh::kSvFlps, d_obs, obs_stride, d_params, d_rvr, d_u, n_obs, n_particles, lag, batch,
                  compute_hessian ? 1 : 0, d_filt, d_smo, d_log_like, d_gradient, d_traj, d_hess1,
                  d_hess2, d_diag, d_x_hist, d_a_hist, d_workspace, workspace_bytes, ctas_per_problem,
                  stream);
}

// ---- auxiliary variables defined by a Philox stream (never stored) --------------------------
int pmmh_flps_sv_corr_philox(const double* d_obs, const double* d_params, const double* d_rvr,
                             unsigned long long seed, unsigned long long philox_offset, int n_obs,
                             int n_particles, int lag, double* d_filt, double* d_smo, double* d_log_like,
                             double* d_gradient, double* d_traj, long long* d_diag, void* d_workspace,
                             size_t workspace_bytes, void* stream) {
    if (!d_obs || !d_params || !d_rvr || !d_filt || !d_smo || !d_log_like || !d_gradient || !d_traj || !d_diag ||
        !d_workspace)
        return fail(PMMH_ERR_INVALID, "pmmh_flps_sv_corr_philox: null pointer argument");
    DeviceInfo di;
    int rc = get_device_info(&di);
    if (rc == PMMH_OK) rc = check_device(di, false);
    if (rc != PMMH_OK) return rc;
    if (!pmmh::sv_split_single_eligible(n_obs, n_particles, lag))
        return fail(PMMH_ERR_INVALID, "pmmh_flps_sv_corr_philox: needs lag in [2, 63] and n_obs >= 2 * lag");
    if (workspace_bytes < pmmh::sv_split_path_ws_bytes(n_obs, n_particles, lag))
        return fail(PMMH_ERR_WORKSPACE, "workspace too small");
    SvPlan p = {};
    p.c.kernel = SvKernel::StreamPath;
    const SvShape s = {n_obs, n_particles, lag, 1, 0, pmmh::kSvFlps, 0, 0};
    pmmh::SvCall c = {};
    c.obs = d_obs; c.params = d_params; c.rvr = d_rvr; c.seed = seed; c.philox_offset = philox_offset;
    c.filt = d_filt; c.smo = d_smo; c.ll = d_log_like; c.grad = d_gradient; c.traj = d_traj; c.diag = d_diag;
    c.prof = g_sv_prof;
    c.ws = d_workspace; c.ws_bytes = workspace_bytes; c.stream = (cudaStream_t)stream;
    return sv_launch_plan(p, s, c);
}

int pmmh_flps_sv_corr_philox_workspace_bytes(int n_obs, int n_particles, int lag, size_t* bytes) {
    if (!bytes || !pmmh::sv_split_single_eligible(n_obs, n_particles, lag))
        return fail(PMMH_ERR_INVALID, "pmmh_flps_sv_corr_philox_workspace_bytes: bad arguments");
    *bytes = pmmh::sv_split_path_ws_bytes(n_obs, n_particles, lag);
    return PMMH_OK;
}

// ---- host-resident auxiliary variables, copied while the kernel runs ----------------------
namespace {
// The copy engine lays the reference's particle-major host array down in slots of time steps: slot c holds
// steps [c W, (c + 1) W) of every particle as rows of W doubles.
constexpr int kUSlot = 64;        // exchange and streaming kernels (512-byte rows)
constexpr int kGridUSlot = 256;   // grid kernel (2 KB rows)
constexpr int kGridUTaperMin = 48;   // smallest copy of the grid kernel's tapered schedule, in time steps

size_t staged_bytes(int n_obs, int n, int slot) {
    return (size_t)((n_obs + slot - 1) / slot) * (size_t)n * slot * sizeof(double);
}

// Next piece of a copy schedule: time steps [t0, t0 + return value).  It never crosses a slot of `ch` steps
// and ends on a multiple of 4 steps unless it ends the series (32-byte sectors of the staged rows, ch % 4 == 0).
// taper_min = 0: whole slots.  Otherwise the pieces get shorter towards the end of the series.  The kernel
// needs ~0.11 ms per time step, the host link ~0.157 ms (2 KB rows: 53.5 GB/s; 1 KB: 51.7; 512 B: 48.4; and
// ~8 ns per row whatever its width, i.e. 8.4 ms for any piece of fewer than ~52 steps at N = 2^20).  The kernel
// can only start a piece when all of it has landed, so after the last copy it still has to work off what it was
// behind: a piece of p steps that starts with `rem` steps to go delays the end unless
// 0.157 p <= (0.157 - 0.11) rem + 0.11 p_last, i.e. p <= 0.3 rem + 0.7 p_last.  Hence: whole slots (widest rows)
// while that holds, then pieces of ~0.3 x what remains, the last one ~taper_min steps.  Measured at T = 1000,
// N = 2^20: one copy per slot 157.7 ms of copies + 26.3 ms of kernel after the last one; this schedule: see
// DESIGN 3.
int grid_u_next_piece(int t0, int n_obs, int ch, int taper_min) {
    const int c = t0 / ch, in = t0 - c * ch;
    const int rem = n_obs - t0;
    int wsteps = (rem < ch - in) ? rem : ch - in;            // what is left of this slot
    if (taper_min > 0 && rem >= 2 * taper_min) {
        int w = (3 * rem) / 10 + (7 * taper_min) / 10;
        if (w < taper_min) w = taper_min;
        if (w < wsteps) wsteps = w;
    }
    if (t0 + wsteps < n_obs) wsteps = (wsteps + 3) & ~3;   // pieces end on 32-byte sectors of the staged rows (ch % 4 == 0)
    const int whole = (rem < ch - in) ? rem : ch - in;
    // no sliver at the end of a slot (what is left over at the end of the series may be half as short: it is the last piece)
    if (wsteps > whole || (taper_min > 0 && whole - wsteps < (whole == rem ? taper_min / 2 : taper_min))) wsteps = whole;
    return wsteps;
}

// immutable pinned table tab[i] = i: the copy engine writes &tab[rows landed] to the device flag, so
// no call ever rewrites a host value that a queued copy may still read
const int* step_table(int need) {
    static std::mutex mu;
    static int* tab = nullptr;
    static int cap = 0;
    std::lock_guard<std::mutex> lk(mu);
    if (cap < need + 1) {
        int ncap = need + 1 > 65536 ? need + 1 : 65536;
        int* t = nullptr;
        if (cudaHostAlloc((void**)&t, (size_t)ncap * sizeof(int), cudaHostAllocPortable) != cudaSuccess) return nullptr;
        for (int i = 0; i < ncap; ++i) t[i] = i;
        tab = t;   // an older, smaller table stays allocated: copies queued earlier may still read it
        cap = ncap;
    }
    return tab;
}

// the copy stream and events of the current device and host thread
struct StreamedState {
    cudaStream_t copy_stream = nullptr;
    cudaEvent_t ev_start = nullptr, ev_reset = nullptr, ev_done = nullptr;
    std::vector<cudaEvent_t> ev_slot;   // signal by event: one per slot
};

int streamed_state(StreamedState** out) {
    static thread_local StreamedState states[64];
    int dev = 0;
    PMMH_CUDA(cudaGetDevice(&dev));
    if (dev < 0 || dev >= 64) return fail(PMMH_ERR_NO_DEVICE, "device ordinal out of range");
    StreamedState& s = states[dev];
    if (!s.copy_stream) PMMH_CUDA(cudaStreamCreateWithFlags(&s.copy_stream, cudaStreamNonBlocking));
    for (cudaEvent_t* e : {&s.ev_start, &s.ev_reset, &s.ev_done})
        if (!*e) PMMH_CUDA(cudaEventCreateWithFlags(e, cudaEventDisableTiming));
    *out = &s;
    return PMMH_OK;
}

// Enqueues the copies of u from the reference's (n_obs, N + 1) host array into the slots of `slot` steps of
// d_stage, on the copy stream, once everything queued so far on `st` has finished (the previous evaluation may
// still be reading the staging buffer).  Pieces follow grid_u_next_piece(.., taper_min).  Each piece is
// signalled either through the device flag d_flag (steps landed so far; `st` then waits until the flag has
// been reset) or, with d_flag == NULL, by the event of its slot, ss.ev_slot[c].  ss.ev_done follows the last copy.
int enqueue_u_copies(const double* h_rvs, int n_obs, int n, char* d_stage, int slot, int taper_min, int* d_flag,
                     StreamedState& ss, cudaStream_t st) {
    const int* tab = nullptr;
    if (d_flag) {
        tab = step_table(n_obs);
        if (!tab) return fail(PMMH_ERR_CUDA, "pinned step table allocation failed");
    }
    while (!d_flag && (int)ss.ev_slot.size() < (n_obs + slot - 1) / slot) {
        cudaEvent_t e;
        PMMH_CUDA(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
        ss.ev_slot.push_back(e);
    }
    PMMH_CUDA(cudaEventRecord(ss.ev_start, st));
    PMMH_CUDA(cudaStreamWaitEvent(ss.copy_stream, ss.ev_start, 0));
    if (d_flag) {
        PMMH_CUDA(cudaMemsetAsync(d_flag, 0, sizeof(int), ss.copy_stream));
        PMMH_CUDA(cudaEventRecord(ss.ev_reset, ss.copy_stream));
    }
    for (int t0 = 0; t0 < n_obs;) {
        const int c = t0 / slot, in = t0 - c * slot;
        const int w = grid_u_next_piece(t0, n_obs, slot, taper_min);
        const double* src = h_rvs + (size_t)n_obs + (size_t)t0;   // rvp[i + j * n_obs], cython.py:89-91
        char* dst = d_stage + ((size_t)c * (size_t)n * slot + (size_t)in) * sizeof(double);
        PMMH_CUDA(cudaMemcpy2DAsync(dst, (size_t)slot * sizeof(double), src, (size_t)n_obs * sizeof(double),
                                    (size_t)w * sizeof(double), (size_t)n, cudaMemcpyHostToDevice, ss.copy_stream));
        if (d_flag)
            PMMH_CUDA(cudaMemcpyAsync(d_flag, &tab[t0 + w], sizeof(int), cudaMemcpyHostToDevice, ss.copy_stream));
        else
            PMMH_CUDA(cudaEventRecord(ss.ev_slot[c], ss.copy_stream));
        t0 += w;
    }
    PMMH_CUDA(cudaEventRecord(ss.ev_done, ss.copy_stream));
    if (d_flag) PMMH_CUDA(cudaStreamWaitEvent(st, ss.ev_reset, 0));   // the kernel must not start before the flag is reset
    return PMMH_OK;
}

SvShape streamed_shape(int n_obs, int n, int lag, int ctas) { return {n_obs, n, lag, 1, 0, pmmh::kSvFlps, 0, ctas}; }
}  // namespace

int pmmh_sv_stream_schedule(int n_obs, int* pieces, int max_pieces) {
    if (n_obs < 1 || (max_pieces > 0 && !pieces)) return -1;
    int t0 = 0, k = 0;
    while (t0 < n_obs) {
        const int w = grid_u_next_piece(t0, n_obs, kGridUSlot, kGridUTaperMin);
        if (k < max_pieces) pieces[k] = w;
        ++k;
        t0 += w;
    }
    return k;
}

int pmmh_sv_stage_bytes(int n_obs, int n_particles, size_t* bytes) {
    if (!bytes || n_obs < 2 || n_particles < 1) return fail(PMMH_ERR_INVALID, "pmmh_sv_stage_bytes: bad arguments");
    const size_t b = staged_bytes(n_obs, n_particles, kUSlot), bg = staged_bytes(n_obs, n_particles, kGridUSlot);
    *bytes = (bg > b ? bg : b) + 256;   // + the device flag
    return PMMH_OK;
}

int pmmh_sv_streamed_workspace_bytes(int n_obs, int n_particles, int lag, int ctas_per_problem, size_t* bytes) {
    if (!bytes) return fail(PMMH_ERR_INVALID, "bytes is null");
    SvPlan p;
    int rc = sv_make_plan(streamed_shape(n_obs, n_particles, lag, ctas_per_problem), SvEntry::HostStreamed, &p);
    if (rc != PMMH_OK) return rc;
    *bytes = p.total;
    return PMMH_OK;
}

int pmmh_sv_streamed_eligible(int n_obs, int n_particles, int lag, int ctas_per_problem) {
    SvPlan p;
    return sv_make_plan(streamed_shape(n_obs, n_particles, lag, ctas_per_problem), SvEntry::HostStreamed, &p) == PMMH_OK &&
           p.c.kernel != SvKernel::None;
}

int pmmh_flps_sv_corr_streamed(const double* h_rvs, const double* d_obs, const double* d_params,
                               const double* d_rvr, int n_obs, int n_particles, int lag, void* d_stage,
                               size_t stage_bytes, double* d_filt, double* d_smo, double* d_log_like,
                               double* d_gradient, double* d_traj, double* d_hess1, double* d_hess2,
                               long long* d_diag, void* d_workspace, size_t workspace_bytes,
                               int ctas_per_problem, void* stream) {
    if (!h_rvs || !d_obs || !d_params || !d_rvr || !d_stage || !d_filt || !d_smo || !d_log_like || !d_gradient ||
        !d_traj || !d_hess1 || !d_hess2 || !d_diag || !d_workspace)
        return fail(PMMH_ERR_INVALID, "pmmh_flps_sv_corr_streamed: null pointer argument");
    const SvShape s = streamed_shape(n_obs, n_particles, lag, ctas_per_problem);
    SvPlan p;
    int rc = sv_make_plan(s, SvEntry::HostStreamed, &p);
    if (rc != PMMH_OK) return rc;
    const SvKernel k = p.c.kernel;
    if (k == SvKernel::None)
        return fail(PMMH_ERR_INVALID, "pmmh_flps_sv_corr_streamed: no kernel takes these sizes (pmmh_sv_streamed_eligible)");
    if (workspace_bytes < p.total) return fail(PMMH_ERR_WORKSPACE, "workspace too small (pmmh_sv_streamed_workspace_bytes)");
    // The grid kernel reads its column of a slot with a stride and polls one flag per time step; the call is
    // bound by the host link, not by the kernel.  The exchange kernel polls the flag as well; the host-driven
    // step loop of the streaming kernels waits for a slot's event when it enters it.
    const int slot = k == SvKernel::Grid ? kGridUSlot : kUSlot;
    const size_t data_bytes = staged_bytes(n_obs, n_particles, slot);
    if (stage_bytes < data_bytes + 256) return fail(PMMH_ERR_WORKSPACE, "staging buffer too small");
    if (k == SvKernel::Grid && ((uintptr_t)d_stage & 31) != 0)
        return fail(PMMH_ERR_INVALID, "d_stage must be 32-byte aligned (the kernel reads 32-byte sectors of the staged rows)");
    StreamedState* ss = nullptr;
    rc = streamed_state(&ss);
    if (rc != PMMH_OK) return rc;
    cudaStream_t st = (cudaStream_t)stream;
    const double* d_u = (const double*)d_stage;
    int* d_flag = k == SvKernel::StreamPath ? nullptr : (int*)((char*)d_stage + data_bytes);
    rc = enqueue_u_copies(h_rvs, n_obs, n_particles, (char*)d_stage, slot, k == SvKernel::Grid ? kGridUTaperMin : 0,
                          d_flag, *ss, st);
    if (rc != PMMH_OK) return rc;
    pmmh::SvCall c = {};
    c.obs = d_obs; c.params = d_params; c.rvr = d_rvr;
    c.u = d_u; c.slot = slot; c.u_flag = d_flag; c.slot_ready = ss->ev_slot.data();
    c.filt = d_filt; c.smo = d_smo; c.ll = d_log_like; c.grad = d_gradient; c.traj = d_traj;
    c.hess1 = d_hess1; c.hess2 = d_hess2; c.diag = d_diag; c.prof = g_sv_prof;
    c.ws = d_workspace; c.ws_bytes = workspace_bytes; c.stream = st;
    rc = sv_launch_plan(p, s, c);
    if (rc != PMMH_OK) return rc;
    // an evaluation that is abandoned early leaves copies behind: the caller's stream ends after them
    PMMH_CUDA(cudaStreamWaitEvent(st, ss->ev_done, 0));
    return PMMH_OK;
}

// ---- model-generic entry points: the chain or the grid kernel instantiated for a model of pf_model.cuh ----------
namespace {
// The workspace queries take no model id: any model takes their shapes, the Hessian a model that has it.
constexpr int kQueryModel = PMMH_MODEL_SV_LEVERAGE;

// the four entries: one problem or a batch (`batched`), the smoother or the filter alone (`filter`, lag 2: no lag
// condition); their names (pmmh_<name>_corr, pmmh_<name>_workspace_bytes) and the shapes they take, for the refusals
std::string model_entry_name(bool batched, int filter) {
    return std::string(filter ? "pmmh_filter_model" : "pmmh_flps_model") + (batched ? "_batch" : "");
}
const char* model_entry_shapes(bool batched, int filter) {
    if (batched)
        return filter ? "pmmh_filter_model_batch_corr: batch >= 1, n_obs >= 2, a tile of n_particles / "
                        "ceil(n_particles / 2048) particles fits one CTA and a known model id"
                      : "pmmh_flps_model_batch_corr: batch >= 1, 2 <= lag <= 10, n_obs >= 2 lag, a tile of n_particles / "
                        "ceil(n_particles / 2048) particles fits one CTA, a known model id, compute_hessian only for the "
                        "SV models (0, 8) and the fully adapted linear Gaussian model with a Hessian (6)";
    return filter ? "pmmh_filter_model_corr: a known model id, n_obs >= 2 and 2 <= n_particles <= 4096 (any batch), "
                    "or batch == 1 and n_particles up to 7168 per SM (1,060,864 on 148 SMs)"
                  : "pmmh_flps_model_corr: a known model id, 2 <= lag <= 10 and 2 <= n_particles <= 4096 (any batch), "
                    "or batch == 1, n_obs >= 2 lag and n_particles up to 7168 per SM (1,060,864 on 148 SMs)";
}

// The plan of a model entry: its kernel (c.kernel), CTAs per problem on the grid kernel (c.grid_G), teams (n_teams)
// and workspace (total: the chosen kernel's alone, there is no fallback pass; with history on the grid kernel).
// One problem: the chain kernel wherever it applies (any batch; one CTA per problem, at most one problem per SM at a
// time), else the grid kernel for one problem on sv_grid_ctas(N, SMs, 0) CTAs.  A batch: the grid kernel, one team of
// that many CTAs per problem.  Anything else is refused.
int model_plan(bool batched, int filter, int model_id, int n_obs, int n, int lag, int batch, int hess, DeviceInfo* di,
               SvPlan* p) {
    const char* shapes = model_entry_shapes(batched, filter);
    if (!pmmh::model_known(model_id) || (hess && (filter || !pmmh::model_has_hessian(model_id))))
        return fail(PMMH_ERR_INVALID, shapes);
    if (batch < 1 || n_obs < 2 || (hess != 0 && hess != 1)) return fail(PMMH_ERR_INVALID, shapes);
    int rc = get_device_info(di);
    if (rc != PMMH_OK) return rc;
    memset(p, 0, sizeof(*p));
    const int G = p->c.grid_G = pmmh::sv_grid_ctas(n, di->sm, 0);
    if (!batched && pmmh::sv_chain_eligible(n, lag) && pmmh::sv_chain_smem_bytes(n) <= kMaxDynSmem) {
        p->c.kernel = SvKernel::Chain;
        p->G = 1;
        p->n_teams = p->grid = batch < di->sm ? batch : di->sm;
        p->chain_stride = pmmh::sv_chain_ws_bytes(n, lag, n_obs, 0, filter);
        p->total = (size_t)p->grid * p->chain_stride;
    } else if ((batched || batch == 1) && (filter ? pmmh::sv_grid_filter_eligible(n_obs, n, G)
                                                  : pmmh::sv_grid_eligible(n_obs, n, lag, G))) {
        p->c.kernel = SvKernel::Grid;
        p->n_teams = pmmh::sv_grid_teams(batch, di->sm, G);
        p->total = (size_t)p->n_teams * pmmh::sv_grid_ws_bytes(n_obs, n, lag, G, 1, hess, filter);
    } else {
        return fail(PMMH_ERR_INVALID, shapes);
    }
    return PMMH_OK;
}

int model_query(bool batched, int filter, int n_obs, int n, int lag, int batch, int hess, size_t* bytes) {
    if (!bytes)
        return fail(PMMH_ERR_INVALID, (model_entry_name(batched, filter) + "_workspace_bytes: bytes is null").c_str());
    DeviceInfo di;
    SvPlan p;
    int rc = model_plan(batched, filter, kQueryModel, n_obs, n, lag, batch, hess, &di, &p);
    if (rc == PMMH_OK) *bytes = p.total;
    return rc;
}

// Checks and runs one model entry (the filter: d_smo, d_grad unused; the Hessian outputs: batched smoother only).
// No fallback pass: an abandoned evaluation is reported in d_diag[PMMH_DIAG_STATUS].
int model_run(bool batched, int filter, int model_id, const double* d_obs, long long obs_stride, const double* d_params,
              const double* d_rvr, const double* d_u, int n_obs, int n, int lag, int batch, int hess, double* d_filt,
              double* d_smo, double* d_ll, double* d_grad, double* d_traj, double* d_h1, double* d_h2,
              long long* d_diag, double* d_xh, int* d_ah, void* d_ws, size_t ws_bytes, void* stream) {
    const std::string name = model_entry_name(batched, filter) + "_corr";
    if (!d_obs || !d_params || !d_rvr || !d_u || !d_filt || !d_ll || !d_traj || !d_diag ||
        (!filter && (!d_smo || !d_grad)) || (!d_ws && (batched || !filter)) || (hess && (!d_h1 || !d_h2)))
        return fail(PMMH_ERR_INVALID, (name + ": null pointer argument").c_str());
    if ((d_xh == nullptr) != (d_ah == nullptr))
        return fail(PMMH_ERR_INVALID, "d_x_hist and d_a_hist must be given together");
    if (!batched && !filter && n_obs < lag + 1) return fail(PMMH_ERR_INVALID, "n_obs must be at least lag + 1");
    DeviceInfo di;
    SvPlan p;
    int rc = model_plan(batched, filter, model_id, n_obs, n, lag, batch, hess, &di, &p);
    if (rc != PMMH_OK) return rc;
    if (ws_bytes < p.total) return fail(PMMH_ERR_WORKSPACE, (name + ": workspace too small").c_str());
    if (p.total && !d_ws) return fail(PMMH_ERR_INVALID, (name + ": null workspace").c_str());
    rc = check_device(di, p.c.kernel == SvKernel::Grid);
    if (rc != PMMH_OK) return rc;
    pmmh::SvCall c = {};
    c.obs = d_obs; c.obs_stride = obs_stride; c.params = d_params; c.rvr = d_rvr; c.u = d_u;
    c.filt = d_filt; c.smo = d_smo; c.ll = d_ll; c.grad = d_grad; c.traj = d_traj; c.diag = d_diag;
    if (hess) { c.hess1 = d_h1; c.hess2 = d_h2; }
    c.x_hist = d_xh; c.a_hist = d_ah; c.model = model_id; c.filter = filter;
    c.prof = batched ? nullptr : g_sv_prof;   // (phase clocks: one problem only)
    c.ws = d_ws; c.ws_bytes = ws_bytes; c.stream = (cudaStream_t)stream;
    if (p.c.kernel == SvKernel::Grid) return pmmh::sv_grid_run(c, batch, n_obs, n, lag, p.c.grid_G, p.n_teams, hess);
    return sv_launch_plan(p, {n_obs, n, lag, batch, 0, pmmh::kSvFlps, d_xh != nullptr, 0}, c);
}
}  // namespace

int pmmh_flps_model_workspace_bytes(int n_obs, int n_particles, int lag, int batch, size_t* bytes) {
    return model_query(false, 0, n_obs, n_particles, lag, batch, 0, bytes);
}

int pmmh_flps_model_corr(int model_id, const double* d_obs, long long obs_stride, const double* d_params,
                         const double* d_rvr, const double* d_u, int n_obs, int n_particles, int lag, int batch,
                         double* d_filt, double* d_smo, double* d_log_like, double* d_gradient, double* d_traj,
                         long long* d_diag, double* d_x_hist, int* d_a_hist, void* d_workspace,
                         size_t workspace_bytes, void* stream) {
    return model_run(false, 0, model_id, d_obs, obs_stride, d_params, d_rvr, d_u, n_obs, n_particles, lag, batch, 0,
                     d_filt, d_smo, d_log_like, d_gradient, d_traj, nullptr, nullptr, d_diag, d_x_hist, d_a_hist,
                     d_workspace, workspace_bytes, stream);
}

int pmmh_filter_model_workspace_bytes(int n_obs, int n_particles, int batch, size_t* bytes) {
    return model_query(false, 1, n_obs, n_particles, 2, batch, 0, bytes);
}

int pmmh_filter_model_corr(int model_id, const double* d_obs, long long obs_stride, const double* d_params,
                           const double* d_rvr, const double* d_u, int n_obs, int n_particles, int batch,
                           double* d_filt, double* d_log_like, double* d_traj, long long* d_diag,
                           double* d_x_hist, int* d_a_hist, void* d_workspace, size_t workspace_bytes,
                           void* stream) {
    return model_run(false, 1, model_id, d_obs, obs_stride, d_params, d_rvr, d_u, n_obs, n_particles, 2, batch, 0,
                     d_filt, nullptr, d_log_like, nullptr, d_traj, nullptr, nullptr, d_diag, d_x_hist, d_a_hist,
                     d_workspace, workspace_bytes, stream);
}

int pmmh_flps_model_batch_workspace_bytes(int n_obs, int n_particles, int lag, int batch, int compute_hessian,
                                          size_t* bytes) {
    return model_query(true, 0, n_obs, n_particles, lag, batch, compute_hessian, bytes);
}

int pmmh_flps_model_batch_corr(int model_id, const double* d_obs, long long obs_stride, const double* d_params,
                               const double* d_rvr, const double* d_u, int n_obs, int n_particles, int lag, int batch,
                               int compute_hessian, double* d_filt, double* d_smo, double* d_log_like,
                               double* d_gradient, double* d_traj, double* d_hess1, double* d_hess2, long long* d_diag,
                               double* d_x_hist, int* d_a_hist, void* d_workspace, size_t workspace_bytes,
                               void* stream) {
    return model_run(true, 0, model_id, d_obs, obs_stride, d_params, d_rvr, d_u, n_obs, n_particles, lag, batch,
                     compute_hessian, d_filt, d_smo, d_log_like, d_gradient, d_traj, d_hess1, d_hess2, d_diag, d_x_hist,
                     d_a_hist, d_workspace, workspace_bytes, stream);
}

int pmmh_filter_model_batch_workspace_bytes(int n_obs, int n_particles, int batch, size_t* bytes) {
    return model_query(true, 1, n_obs, n_particles, 2, batch, 0, bytes);
}

int pmmh_filter_model_batch_corr(int model_id, const double* d_obs, long long obs_stride, const double* d_params,
                                 const double* d_rvr, const double* d_u, int n_obs, int n_particles, int batch,
                                 double* d_filt, double* d_log_like, double* d_traj, long long* d_diag,
                                 double* d_x_hist, int* d_a_hist, void* d_workspace, size_t workspace_bytes,
                                 void* stream) {
    return model_run(true, 1, model_id, d_obs, obs_stride, d_params, d_rvr, d_u, n_obs, n_particles, 2, batch, 0,
                     d_filt, nullptr, d_log_like, nullptr, d_traj, nullptr, nullptr, d_diag, d_x_hist, d_a_hist,
                     d_workspace, workspace_bytes, stream);
}

int pmmh_bpf_sv_corr(const double* d_obs, long long obs_stride, const double* d_params,
                     const double* d_rvr, const double* d_u, int n_obs, int n_particles, int batch,
                     int read_mode, double* d_filt, double* d_log_like, double* d_traj,
                     long long* d_diag, double* d_x_hist, int* d_a_hist, void* d_workspace,
                     size_t workspace_bytes, int ctas_per_problem, void* stream) {
    const int mode = (read_mode == PMMH_BPF_INTENDED) ? pmmh::kSvBpfIntended : pmmh::kSvBpfParity;
    return sv_run(mode, d_obs, obs_stride, d_params, d_rvr, d_u, n_obs, n_particles, 2, batch, 0, d_filt,
                  nullptr, d_log_like, nullptr, d_traj, nullptr, nullptr, d_diag, d_x_hist, d_a_hist,
                  d_workspace, workspace_bytes, ctas_per_problem, stream);
}

int pmmh_split_rvs(const double* d_rvs, int n_obs, int n_particles, int batch, double* d_r_raw,
                   double* d_u, void* stream) {
    if (!d_rvs || !d_r_raw || !d_u || n_obs < 1 || n_particles < 1 || batch < 1)
        return fail(PMMH_ERR_INVALID, "pmmh_split_rvs: bad arguments");
    cudaStream_t st = (cudaStream_t)stream;
    const long long per = (long long)n_obs * ((long long)n_particles + 1);
    PMMH_CUDA(pmmh::launch_copy_head(d_rvs, d_r_raw, n_obs, batch, per, n_obs, st));
    // flat remainder viewed as [n_particles][n_obs] -> [n_obs][n_particles]
    PMMH_CUDA(pmmh::launch_transpose(d_rvs + n_obs, d_u, n_particles, n_obs, batch, per,
                                     (long long)n_obs * n_particles, st));
    return PMMH_OK;
}

int pmmh_norm_cdf(const double* d_in, double* d_out, long long n, void* stream) {
    if (!d_in || !d_out || n < 0) return fail(PMMH_ERR_INVALID, "pmmh_norm_cdf: bad arguments");
    PMMH_CUDA(pmmh::launch_norm_cdf(d_in, d_out, n, (cudaStream_t)stream));
    return PMMH_OK;
}

int pmmh_importance_discrete(const double* d_obs, long long obs_stride, const double* d_params,
                             const double* d_rvr, const double* d_rvp, int n_obs, int n_particles,
                             int batch, double* d_filt, double* d_log_like, double* d_traj,
                             double* d_gradient, int* d_traj_idx, void* stream) {
    if (!d_obs || !d_params || !d_rvr || !d_rvp || !d_filt || !d_log_like || !d_traj || !d_gradient ||
        !d_traj_idx || n_obs < 1 || n_particles < 1 || batch < 1)
        return fail(PMMH_ERR_INVALID, "pmmh_importance_discrete: bad arguments");
    if ((size_t)3 * n_particles * sizeof(double) > 200 * 1024)
        return fail(PMMH_ERR_INVALID, "pmmh_importance_discrete: n_particles above 8533 unsupported");
    PMMH_CUDA(pmmh::launch_importance_discrete(d_obs, obs_stride, d_params, d_rvr, d_rvp, n_obs,
                                               n_particles, batch, d_filt, d_log_like, d_traj,
                                               d_gradient, d_traj_idx, (cudaStream_t)stream));
    return PMMH_OK;
}

int pmmh_crank_nicolson(const double* d_u, const double* d_xi, double* d_out, long long n,
                        double sigma_u, unsigned long long seed, unsigned long long philox_offset,
                        void* stream) {
    if (!d_u || !d_out || n < 0) return fail(PMMH_ERR_INVALID, "pmmh_crank_nicolson: bad arguments");
    const double a = sqrt(1.0 - sigma_u * sigma_u);
    PMMH_CUDA(pmmh::launch_crank_nicolson(d_u, d_xi, d_out, n, a, sigma_u, seed, philox_offset,
                                          (cudaStream_t)stream));
    return PMMH_OK;
}

int pmmh_subsample_workspace_bytes(int m, size_t* bytes) {
    if (!bytes || m < 1) return fail(PMMH_ERR_INVALID, "pmmh_subsample_workspace_bytes: bad arguments");
    *bytes = pmmh::subsample_ws_bytes(m);
    return PMMH_OK;
}

int pmmh_subsample_indices(const double* d_u, int m, int n_data, int apply_cdf, int* d_idx,
                           double* d_sorted, void* d_workspace, size_t workspace_bytes, void* stream) {
    if (!d_u || !d_idx || !d_workspace || m < 1 || n_data < 1)
        return fail(PMMH_ERR_INVALID, "pmmh_subsample_indices: bad arguments");
    if (workspace_bytes < pmmh::subsample_ws_bytes(m)) return fail(PMMH_ERR_WORKSPACE, "workspace too small");
    PMMH_CUDA(pmmh::launch_subsample_indices(d_u, m, n_data, apply_cdf, d_idx, d_sorted, d_workspace,
                                             (cudaStream_t)stream));
    return PMMH_OK;
}

int pmmh_logistic_workspace_bytes(int m, int d, int compute_hessian, size_t* bytes) {
    if (!bytes || m < 1 || d < 1) return fail(PMMH_ERR_INVALID, "pmmh_logistic_workspace_bytes: bad arguments");
    *bytes = pmmh::logistic_ws_bytes(m, d, compute_hessian);
    return PMMH_OK;
}

int pmmh_logistic_loglike(const double* d_x, const double* d_y, const int* d_idx, int m, int d,
                          long long row_begin, long long row_end, const double* d_beta,
                          int compute_hessian, double* d_out, void* d_workspace,
                          size_t workspace_bytes, void* stream) {
    if (!d_x || !d_y || !d_idx || !d_beta || !d_out || !d_workspace || m < 1 || d < 1)
        return fail(PMMH_ERR_INVALID, "pmmh_logistic_loglike: bad arguments");
    if (d > 32) return fail(PMMH_ERR_INVALID, "pmmh_logistic_loglike: d > 32 not supported yet");
    if (workspace_bytes < pmmh::logistic_ws_bytes(m, d, compute_hessian))
        return fail(PMMH_ERR_WORKSPACE, "workspace too small");
    PMMH_CUDA(pmmh::launch_logistic(d_x, d_y, d_idx, m, d, row_begin, row_end, d_beta,
                                    compute_hessian ? 1 : 0, d_out, d_workspace, (cudaStream_t)stream));
    return PMMH_OK;
}

// ------------------------------------------------------------------ host-buffer wrappers

static int sv_host(int mode, const double* obs, const double* params, const double* rvr,
                   const double* rvp, int n_obs, int n, int lag, int hess, int read_mode, double* filt,
                   double* smo, double* log_like, double* gradient, double* traj, double* hess1,
                   double* hess2, long long* diag) {
    if (!obs || !params || !rvr || !rvp || !filt || !log_like || !traj)
        return fail(PMMH_ERR_INVALID, "null host pointer");
    const size_t nt = (size_t)n_obs * n;
    size_t ws_bytes = 0;
    int rc = pmmh_sv_workspace_bytes(n_obs, n, lag, 1, hess, mode, 0, 0, &ws_bytes);
    if (rc != PMMH_OK) return rc;
    DevBuf b_obs, b_par, b_rvr, b_rvp, b_u, b_out, b_diag, b_ws;
    const size_t n_out = (size_t)n_obs * 7 + 1 + 32;   // filt smo traj grad[4] ll h1 h2
    PMMH_CUDA(b_obs.alloc(n_obs * sizeof(double)));
    PMMH_CUDA(b_par.alloc(4 * sizeof(double)));
    PMMH_CUDA(b_rvr.alloc(n_obs * sizeof(double)));
    PMMH_CUDA(b_rvp.alloc(nt * sizeof(double)));
    PMMH_CUDA(b_u.alloc(nt * sizeof(double)));
    PMMH_CUDA(b_out.alloc(n_out * sizeof(double)));
    PMMH_CUDA(b_diag.alloc(PMMH_DIAG_COUNT * sizeof(long long)));
    PMMH_CUDA(b_ws.alloc(ws_bytes));
    PMMH_CUDA(cudaMemcpy(b_obs.p, obs, n_obs * sizeof(double), cudaMemcpyHostToDevice));
    PMMH_CUDA(cudaMemcpy(b_par.p, params, 4 * sizeof(double), cudaMemcpyHostToDevice));
    PMMH_CUDA(cudaMemcpy(b_rvr.p, rvr, n_obs * sizeof(double), cudaMemcpyHostToDevice));
    PMMH_CUDA(cudaMemcpy(b_rvp.p, rvp, nt * sizeof(double), cudaMemcpyHostToDevice));
    PMMH_CUDA(cudaMemset(b_out.p, 0, n_out * sizeof(double)));
    PMMH_CUDA(cudaMemset(b_diag.p, 0, PMMH_DIAG_COUNT * sizeof(long long)));
    PMMH_CUDA(pmmh::launch_transpose(b_rvp.as<double>(), b_u.as<double>(), n, n_obs, 1, 0, 0, 0));
    double* o = b_out.as<double>();
    double* d_filt = o;
    double* d_smo = o + n_obs;
    double* d_traj = o + 2 * (size_t)n_obs;
    double* d_grad = o + 3 * (size_t)n_obs;
    double* d_ll = o + 7 * (size_t)n_obs;
    double* d_h1 = d_ll + 1;
    double* d_h2 = d_h1 + 16;
    if (mode == 0)
        rc = pmmh_flps_sv_corr(b_obs.as<double>(), 0, b_par.as<double>(), b_rvr.as<double>(),
                               b_u.as<double>(), n_obs, n, lag, 1, hess, d_filt, d_smo, d_ll, d_grad,
                               d_traj, d_h1, d_h2, b_diag.as<long long>(), nullptr, nullptr, b_ws.p,
                               ws_bytes, 0, nullptr);
    else
        rc = pmmh_bpf_sv_corr(b_obs.as<double>(), 0, b_par.as<double>(), b_rvr.as<double>(),
                              b_u.as<double>(), n_obs, n, 1, read_mode, d_filt, d_ll, d_traj,
                              b_diag.as<long long>(), nullptr, nullptr, b_ws.p, ws_bytes, 0, nullptr);
    if (rc != PMMH_OK) return rc;
    PMMH_CUDA(cudaDeviceSynchronize());
    std::vector<double> h(n_out);
    PMMH_CUDA(cudaMemcpy(h.data(), o, n_out * sizeof(double), cudaMemcpyDeviceToHost));
    memcpy(filt, h.data(), n_obs * sizeof(double));
    if (smo) memcpy(smo, h.data() + n_obs, n_obs * sizeof(double));
    memcpy(traj, h.data() + 2 * (size_t)n_obs, n_obs * sizeof(double));
    if (gradient) memcpy(gradient, h.data() + 3 * (size_t)n_obs, 4 * (size_t)n_obs * sizeof(double));
    *log_like = h[7 * (size_t)n_obs];
    if (hess1) memcpy(hess1, h.data() + 7 * (size_t)n_obs + 1, 16 * sizeof(double));
    if (hess2) memcpy(hess2, h.data() + 7 * (size_t)n_obs + 17, 16 * sizeof(double));
    if (diag)
        PMMH_CUDA(cudaMemcpy(diag, b_diag.p, PMMH_DIAG_COUNT * sizeof(long long), cudaMemcpyDeviceToHost));
    return PMMH_OK;
}

int pmmh_flps_sv_corr_host(const double* obs, const double* params, const double* rvr,
                           const double* rvp, int n_obs, int n_particles, int lag,
                           int compute_hessian, double* filt, double* smo, double* log_like,
                           double* gradient, double* traj, double* hess1, double* hess2,
                           long long* diag) {
    if (!smo || !gradient || !hess1 || !hess2) return fail(PMMH_ERR_INVALID, "null host pointer");
    return sv_host(0, obs, params, rvr, rvp, n_obs, n_particles, lag, compute_hessian ? 1 : 0, 0, filt,
                   smo, log_like, gradient, traj, hess1, hess2, diag);
}

int pmmh_bpf_sv_corr_host(const double* obs, const double* params, const double* rvr,
                          const double* rvp, int n_obs, int n_particles, int read_mode,
                          double* filt, double* log_like, double* traj, long long* diag) {
    return sv_host(1, obs, params, rvr, rvp, n_obs, n_particles, 2, 0, read_mode, filt, nullptr,
                   log_like, nullptr, traj, nullptr, nullptr, diag);
}

int pmmh_importance_discrete_host(const double* obs, const double* params, double rvr,
                                  const double* rvp, int n_obs, int n_particles, double* filt,
                                  double* log_like, double* traj, double* gradient) {
    if (!obs || !params || !rvp || !filt || !log_like || !traj || !gradient)
        return fail(PMMH_ERR_INVALID, "null host pointer");
    const size_t nt = (size_t)n_obs * n_particles;
    DevBuf b_obs, b_par, b_rvr, b_rvp, b_out, b_idx;
    const size_t n_out = (size_t)2 * n_obs + 3;
    PMMH_CUDA(b_obs.alloc(n_obs * sizeof(double)));
    PMMH_CUDA(b_par.alloc(2 * sizeof(double)));
    PMMH_CUDA(b_rvr.alloc(sizeof(double)));
    PMMH_CUDA(b_rvp.alloc(nt * sizeof(double)));
    PMMH_CUDA(b_out.alloc(n_out * sizeof(double)));
    PMMH_CUDA(b_idx.alloc(sizeof(int)));
    PMMH_CUDA(cudaMemcpy(b_obs.p, obs, n_obs * sizeof(double), cudaMemcpyHostToDevice));
    PMMH_CUDA(cudaMemcpy(b_par.p, params, 2 * sizeof(double), cudaMemcpyHostToDevice));
    PMMH_CUDA(cudaMemcpy(b_rvr.p, &rvr, sizeof(double), cudaMemcpyHostToDevice));
    PMMH_CUDA(cudaMemcpy(b_rvp.p, rvp, nt * sizeof(double), cudaMemcpyHostToDevice));
    double* o = b_out.as<double>();
    int rc = pmmh_importance_discrete(b_obs.as<double>(), 0, b_par.as<double>(), b_rvr.as<double>(),
                                      b_rvp.as<double>(), n_obs, n_particles, 1, o, o + 2 * (size_t)n_obs,
                                      o + n_obs, o + 2 * (size_t)n_obs + 1, b_idx.as<int>(), nullptr);
    if (rc != PMMH_OK) return rc;
    PMMH_CUDA(cudaDeviceSynchronize());
    std::vector<double> h(n_out);
    PMMH_CUDA(cudaMemcpy(h.data(), o, n_out * sizeof(double), cudaMemcpyDeviceToHost));
    memcpy(filt, h.data(), n_obs * sizeof(double));
    memcpy(traj, h.data() + n_obs, n_obs * sizeof(double));
    *log_like = h[2 * (size_t)n_obs];
    gradient[0] = h[2 * (size_t)n_obs + 1];
    gradient[1] = h[2 * (size_t)n_obs + 2];
    return PMMH_OK;
}

int pmmh_stratified_host(const double* rnd_sorted, int m, int n_data, int* indices) {
    if (!rnd_sorted || !indices || m < 1 || n_data < 1) return fail(PMMH_ERR_INVALID, "bad arguments");
    size_t ws_bytes = pmmh::subsample_ws_bytes(m);
    DevBuf b_u, b_idx, b_ws;
    PMMH_CUDA(b_u.alloc(m * sizeof(double)));
    PMMH_CUDA(b_idx.alloc(m * sizeof(int)));
    PMMH_CUDA(b_ws.alloc(ws_bytes));
    PMMH_CUDA(cudaMemcpy(b_u.p, rnd_sorted, m * sizeof(double), cudaMemcpyHostToDevice));
    int rc = pmmh_subsample_indices(b_u.as<double>(), m, n_data, 0, b_idx.as<int>(), nullptr, b_ws.p,
                                    ws_bytes, nullptr);
    if (rc != PMMH_OK) return rc;
    PMMH_CUDA(cudaDeviceSynchronize());
    PMMH_CUDA(cudaMemcpy(indices, b_idx.p, m * sizeof(int), cudaMemcpyDeviceToHost));
    return PMMH_OK;
}

}  // extern "C"
