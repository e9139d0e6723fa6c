// sv_filter.cuh -- argument block and workspace layout of the persistent SV particle-filter
// kernel (shared between the kernel and the C-ABI host code).
#pragma once
#include <cuda_runtime.h>
#include <stddef.h>
#include <stdint.h>

namespace pmmh {

constexpr int kSvThreads = 1024;         // threads per CTA (1 CTA per SM)
constexpr int kStageDoubles = 12288;     // smem staging window for the cumulative weights
constexpr int kBinCap = 4096;            // max occupancy of one sort bin before we give up
constexpr int kMaxAllgatherHost = 48;    // must equal kMaxAllgather (common.cuh)
constexpr int kFastThreads = 512;        // exchange kernel: threads per CTA (128 registers each)
constexpr int kFastCap = 10240;          // exchange kernel: arrivals per CTA and generation (smem capacity)
constexpr int kFastMaxSub = 8;           // exchange kernel: at most this many chunks per CTA

constexpr int kChainThreads = 1024;      // chain kernel: threads per CTA (one CTA per problem)
constexpr int kChainMaxN = 4096;         // chain kernel: particles per problem (all in shared memory)

constexpr int kProfSlots = 16;

enum SvMode { kSvFlps = 0, kSvBpfParity = 1, kSvBpfIntended = 2 };

// diag[] slots (per problem, int64)
enum SvDiag {
    kDiagNearTies = 0,     // ancestor decisions within 64 ulp of a cumulative-weight tie
    kDiagMaxBin = 1,       // largest sort-bin occupancy seen
    kDiagStatus = 2,       // 0 ok, 1 degenerate cloud (bin overflow), 2 non-finite range
    kDiagKeyTies = 3,      // equal adjacent keys after sorting
    kDiagWavefront = 4,    // bpf parity mode: max dependency-chain depth
    kDiagTrajIdx = 5,      // bpf: sampled trajectory index (Q10)
    kDiagKernel = 6,       // which kernel produced the outputs: 1 general, 2 exchange, 3 chain
    kDiagFastInfo = 7,     // exchange kernel: reason (1 run, 2 CTA overflow, 3 weights) | step << 8 | most arrivals << 32
    kDiagCount = 8
};

struct SvArgs {
    int N, NOBS, LAG, B;
    int G, n_teams;
    int NB;          // sort bins (general kernel)
    int NSUB;        // exchange kernel: chunks per CTA
    int CP;          // exchange kernel: capacity of one (destination, source CTA, source warp) run
    int only_failed; // general kernel: only run problems whose diag status is 1 (fallback pass)
    int RING;        // ring depth of the X / A / R histories (LAG + 1), or NOBS with full history
    int mode, hess;
    int model_id;    // chain kernel: the model id (the table Models in pf_model.cuh)
    int SQ;          // low slots of X kept for all times (Q7 / Q11)
    int SQW;         // low slots of W kept for all times (Q10, bpf only)
    const double* obs;
    long long obs_stride;     // 0: shared observations
    const double* params;     // [B][4]
    const double* rvr;        // [B][NOBS]  (already Phi-transformed)
    const double* U;          // [B][NOBS][N] time-major, or (u_chunk > 0, exchange kernel, B = 1)
                              // [chunks][N][u_chunk]: particle-major chunks of u_chunk time steps
    int u_chunk;              // 0 = time-major
    const int* u_ready;       // streamed u: number of time steps that have landed (written by the copy stream)
    double *filt, *smo, *loglike, *grad, *traj, *hess1, *hess2;
    long long* diag;          // [B][kDiagCount]
    double* Xhist;            // optional [B][NOBS][N]
    int* Ahist;               // optional [B][NOBS][N]
    long long* prof;          // optional [grid][kProfSlots] per-CTA phase clocks (development)
    char* ws;                 // workspace base
    size_t ws_sync_bytes;     // leading region: stamps + slots for all CTAs
    size_t ws_team_stride;
};

struct SvWs {
    double *cum, *xnew, *tkey, *sh0, *sh1, *shtail, *Xring, *Rring, *Xlow, *Wlow, *X0;
    int *aun, *rnk, *tpay, *tidx, *hist, *binstart, *Aring, *root0, *root1;
};

__host__ __device__ inline size_t sv_align(size_t x) { return (x + 255) & ~(size_t)255; }

// Bump-allocates the per-team workspace; returns its size.  `have_hist` = caller supplied
// Xhist/Ahist (then no rings are carved).
__host__ __device__ inline size_t sv_ws_layout(int N, int NOBS, int LAG, int NB, int RING, int hess,
                                               int mode, int SQ, int SQW, int have_hist, char* base,
                                               SvWs* w) {
    size_t off = 0;
    size_t n = (size_t)N;
#define PMMH_CARVE(field, type, count)                         \
    do {                                                       \
        if (w) w->field = (type*)(base + off);                 \
        off += sv_align((size_t)(count) * sizeof(type));       \
    } while (0)
    PMMH_CARVE(hist, int, NB);
    PMMH_CARVE(binstart, int, NB + 1);
    PMMH_CARVE(cum, double, n);
    PMMH_CARVE(xnew, double, n);
    PMMH_CARVE(tkey, double, n);
    PMMH_CARVE(sh0, double, n);
    PMMH_CARVE(sh1, double, n);
    PMMH_CARVE(shtail, double, (size_t)LAG * n);
    PMMH_CARVE(aun, int, n);
    PMMH_CARVE(rnk, int, n);
    PMMH_CARVE(tpay, int, n);
    PMMH_CARVE(tidx, int, n);
    PMMH_CARVE(Xlow, double, (size_t)NOBS * SQ);
    PMMH_CARVE(Wlow, double, (size_t)NOBS * (SQW > 0 ? SQW : 1));
    if (!have_hist) {
        PMMH_CARVE(Xring, double, (size_t)RING * n);
        PMMH_CARVE(Aring, int, (size_t)RING * n);
    } else if (w) {
        w->Xring = nullptr;
        w->Aring = nullptr;
    }
    if (hess) PMMH_CARVE(Rring, double, (size_t)RING * 4 * n);
    else if (w) w->Rring = nullptr;
    if (mode != kSvFlps) {
        PMMH_CARVE(root0, int, n);
        PMMH_CARVE(root1, int, n);
        PMMH_CARVE(X0, double, n);
    } else if (w) {
        w->root0 = w->root1 = nullptr;
        w->X0 = nullptr;
    }
#undef PMMH_CARVE
    return off;
}

// Host-side launcher (sv_filter.cu)
cudaError_t sv_launch(const SvArgs& a, int grid, cudaStream_t stream);
int sv_dynamic_smem_bytes(int G);

// chain kernel (sv_chain.cu): one CTA per problem, N <= kChainMaxN; filter = 1: the particle filter alone
// (no fixed-lag smoother, no workspace)
int sv_chain_eligible(int N, int LAG);
size_t sv_chain_ws_bytes(int N, int LAG, int NOBS, int hess, int filter);
int sv_chain_smem_bytes(int N);
cudaError_t sv_chain_launch(const SvArgs& a, int grid, int filter, cudaStream_t stream);

// exchange kernel (sv_fast.cu)
int sv_fast_nsub(int N, int G);
int sv_fast_pair_cap(int N, int G);
int sv_fast_eligible(int N, int G);
size_t sv_fast_ws_bytes(int N, int G, int S, int CW, int LAG, int hist);
size_t sv_fast_sync_bytes(int G, int n_teams);
int sv_fast_smem_bytes(int N, int G, int S);
cudaError_t sv_fast_launch(const SvArgs& a, int grid, cudaStream_t stream);

}  // namespace pmmh
