// sv_chain.cu -- "chain" kernel for the SV fixed-lag particle smoother: one CTA per problem,
// the whole particle generation in shared memory (N <= 4096).  This is the shape of BASELINE
// config 4 (1024 independent CPMH-QN chains / proposals x N = 4096, T = 1000) and of small single
// evaluations: log-likelihood + fixed-lag gradient (flps_sv_corr with compute_hessian = 0,
// stochastic_volatility.pyx:205-655; mh_quasi_newton.py:333,378 makes this call twice per
// iteration) and, as a second instantiation, the Hessian branch (compute_hessian = 1,
// :361-390 alpha recursion with Q7 / Q8, :472-534, :564-626: what mh_second_order.py asks for).
// The kernel is a template over the MODEL (pf_model.cuh: propagation, log-weight, score terms);
// its Hessian branch exists for the reference's SV model only.
//
// One persistent launch, CTAs loop over the problems of the batch; nothing is exchanged between
// CTAs.  Per time step (all in shared memory unless noted):
//   * correlated systematic resampling (:694-715): every child binary-searches the cumulative
//     weights (normalised at look-up), 4 children per thread, u read coalesced from HBM;
//   * propagation (:354-358);
//   * sort (:392-424): counting sort over N bins spanning the exact range of the propagation
//     mean +- 6.5 innovation standard deviations, all-pairs rank inside a bin;
//   * log-weights (:427-437), block scan in sorted order -> cumulative weights, likelihood term;
//   * fixed-lag score terms (:445-470): every particle carries the sorted positions of its
//     ancestors 1..4 steps back (16-bit), a ring of the "4 steps back" columns reaches the
//     ancestor LAG-2 steps back in two shared-memory look-ups; its (value, parent value) pair
//     comes from a ring in global memory (L2 resident: 64 KB per generation and problem).
// The tail (:540-562, Q6) chases one-step ancestors through global rings of the last LAG
// generations.  Quirks reproduced: Q1, Q3 (as in the other kernels: cumulative weights are
// normalised at look-up), Q5 and Q6 for the SV model (M::kPairing; the other models pair the fixed-lag terms
// exactly, pf_model.cuh), Q11.  Sums over particles are fixed-order tree sums.
// Hessian branch: the cumulative alpha of a particle (4 doubles) lives in a global ring by sorted
// position next to the (value, parent value) ring; the child adds its own term to its parent's
// (one 32-byte gather), the score phase gathers the lagged ancestor's; Q7's flat-layout read needs
// the first few sorted values of every past generation (a [NOBS][SQ] table) and of the unsorted new
// one; the 20 sums of hessian1 / hessian2 stay thread-local over the whole series (normalised
// weights, as the reference) and are reduced once.  1024 chains x N = 4096, T = 1000: 0.87 s
// against 1.50 s on the general kernel (0.27 s without the Hessian).
// A degenerate cloud (a sort bin with more than 1024 keys) abandons the problem with status 1;
// the host re-runs the general kernel for it.
// SMO = false is the particle filter alone (pmmh_filter_model_corr): the same resampling, sort, weights and
// sums, without the carried ancestor positions, the (value, parent value) ring, the fixed-lag terms and the
// tail; it needs no workspace.
#include <math.h>

#include "common.cuh"
#include "sv_filter.cuh"
#include "pf_model.cuh"
#include "sv_math.cuh"

namespace pmmh {

namespace {

constexpr int kCT = kChainThreads;
constexpr int kCNW = kCT / 32;
constexpr int kP = kChainMaxN / kCT;   // particles per thread
constexpr int kMaxLagC = 64;
constexpr int kB4Ring = 5;
constexpr int kChainBinMax = 1024;

static_assert(kChainMaxN % kCT == 0, "particles per thread");
static_assert(kCNW == 32, "the block scans assume 32 warps");
static_assert(kChainMaxN <= 65536, "positions are 16 bit");

struct ChainWs {
    double2* xp;   // [LAG + 1][N]  (value, parent value) by sorted position, ring over generations
    int* b1;       // [LAG][N]      one-step ancestor position, last LAG generations (tail)
    double* sh;    // [LAG][N]      shifted weights, last LAG generations (tail)
    // Hessian branch (:361-390, :472-534, :564-626) only:
    double4* al;   // [LAG + 1][N]  cumulative alpha of a particle (4 parameters) by sorted position, ring
    double* xlow;  // [NOBS][SQ]    the first SQ sorted values of every generation (Q7 reads them)
    double* xnf;   // [SQ]          the first SQ UNSORTED values of the generation being built (Q7)
};

__host__ __device__ inline size_t chain_ws_carve(int N, int LAG, int NOBS, int SQ, int hess, char* base, ChainWs* w) {
    size_t off = 0;
#define PMMH_CARVE(field, type, count)                   \
    do {                                                 \
        if (w) w->field = (type*)(base + off);           \
        off += sv_align((size_t)(count) * sizeof(type)); \
    } while (0)
    PMMH_CARVE(xp, double2, (size_t)(LAG + 1) * N);
    PMMH_CARVE(b1, int, (size_t)LAG * N);
    PMMH_CARVE(sh, double, (size_t)LAG * N);
    if (hess) {
        PMMH_CARVE(al, double4, (size_t)(LAG + 1) * N);
        PMMH_CARVE(xlow, double, (size_t)NOBS * SQ);
        PMMH_CARVE(xnf, double, (size_t)SQ);
    } else if (w) {
        w->al = nullptr;
        w->xlow = w->xnf = nullptr;
    }
#undef PMMH_CARVE
    return off;
}

// exclusive block scans over kCT threads (fixed order)
__device__ __forceinline__ double chain_scan_d(double v, double* s_w, double* total) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const double incl = warp_incl_scan(v, lane);
    __syncthreads();
    if (lane == 31) s_w[warp] = incl;
    __syncthreads();
    if (warp == 0) {
        const double tv = s_w[lane];
        const double ti = warp_incl_scan(tv, lane);
        __syncwarp();
        s_w[lane] = ti - tv;
        if (lane == 31) s_w[32] = ti;
    }
    __syncthreads();
    const double r = s_w[warp] + (incl - v);
    *total = s_w[32];
    return r;
}
__device__ __forceinline__ int chain_scan_i(int v, int* s_w, int* total) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int incl = warp_incl_scan(v, lane);
    __syncthreads();
    if (lane == 31) s_w[warp] = incl;
    __syncthreads();
    if (warp == 0) {
        const int tv = s_w[lane];
        const int ti = warp_incl_scan(tv, lane);
        __syncwarp();
        s_w[lane] = ti - tv;
        if (lane == 31) s_w[32] = ti;
    }
    __syncthreads();
    const int r = s_w[warp] + (incl - v);
    *total = s_w[32];
    return r;
}

__device__ __forceinline__ double4 chain_ld_d4(const double4* p) {
    const double2 lo = __ldcg((const double2*)p), hi = __ldcg((const double2*)p + 1);
    return make_double4(lo.x, lo.y, hi.x, hi.y);
}

// development instrumentation: cycles per phase, accumulated by thread 0 of every CTA
#define CPROF(slot)                                                              \
    do {                                                                         \
        if (a.prof && threadIdx.x == 0) {                                        \
            const long long now__ = clock64();                                   \
            a.prof[(size_t)blockIdx.x * kProfSlots + (slot)] += now__ - prof_t;  \
            prof_t = now__;                                                      \
        }                                                                        \
    } while (0)

// M = the model (pf_model.cuh): propagation, log-weight, score terms
// HESS (SvLeverageModel only): the Hessian branch of the reference with its quirks Q7 / Q8
// SMO: the fixed-lag smoother (smo, gradient); false: the filter alone (log-likelihood, filt, traj, diag, history)
template <class M, bool HESS, bool SMO>
__global__ void __launch_bounds__(kCT, 1) sv_chain_kernel(SvArgs a) {
    static_assert(SMO || !HESS, "the Hessian branch needs the smoother");
    long long prof_t = clock64();
    extern __shared__ __align__(16) unsigned char dsm_raw[];
    const int N = a.N, NOBS = a.NOBS, LAG = a.LAG;
    const int K = LAG - 2, RXP = LAG + 1;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int NP = (N + 1) & ~1;   // keeps the 8-byte arrays aligned

    double* s_x = (double*)dsm_raw;                              // [N] sorted values of the current generation
    double* s_cum = s_x + NP;                                    // [N] inclusive cumulative shifted weights
    double* s_key = s_cum + NP;                                  // [N] children in bin order
    int* s_hist = (int*)(s_key + NP);                            // [N + 2] bin counts / starts
    unsigned short* s_b = (unsigned short*)(s_hist + NP + 2);    // [4][N] positions of the ancestors 1..4 steps back
    unsigned short* s_B4 = s_b + 4 * (size_t)NP;                 // [kB4Ring][N] ring of the "4 steps back" column
    unsigned short* s_pay = s_B4 + kB4Ring * (size_t)NP;         // [N] bin order: ancestor of the child

    __shared__ double s_w[33];
    __shared__ int s_iw[33];
    __shared__ double s_red[20 * 32];
    __shared__ double s_hacc[20];        // running hessian1 / hessian2 (upper triangles)
    __shared__ double s_S[kMaxLagC];
    __shared__ double s_bin[4];
    __shared__ int s_flag;

    char* wsbase = a.ws + (size_t)blockIdx.x * a.ws_team_stride;
    ChainWs w;
    const int SQ = HESS ? a.SQ : 1;
    if constexpr (SMO) chain_ws_carve(N, LAG, NOBS, SQ, HESS ? 1 : 0, wsbase, &w);
#define XPG(t) (w.xp + (size_t)((t) % RXP) * N)
#define B1G(t) (w.b1 + (size_t)((t) - (NOBS - LAG)) * N)
#define SHG(t) (w.sh + (size_t)((t) - (NOBS - LAG)) * N)
#define ALG(t) (w.al + (size_t)((t) % RXP) * N)

    for (int prob = blockIdx.x; prob < a.B; prob += gridDim.x) {
        if (a.only_failed && a.diag[(size_t)prob * kDiagCount + kDiagStatus] != 1) continue;
        const double* obs = a.obs + (size_t)prob * a.obs_stride;
        const double* rvr = a.rvr + (size_t)prob * NOBS;
        const double* U = a.U + (size_t)prob * NOBS * N;
        double* o_filt = a.filt + (size_t)prob * NOBS;
        double* o_smo = a.smo + (size_t)prob * NOBS;
        double* o_grad = a.grad + (size_t)prob * 4 * NOBS;
        double* o_traj = a.traj + (size_t)prob * NOBS;
        long long* o_diag = a.diag + (size_t)prob * kDiagCount;
        double* Xh = a.Xhist ? a.Xhist + (size_t)prob * NOBS * N : nullptr;
        int* Ah = a.Ahist ? a.Ahist + (size_t)prob * NOBS * N : nullptr;

        typename M::Const c;
        M::init(c, a.params + (size_t)prob * 4);
        const double logN = log((double)N);

        // ---------------- time 0 (:306-323, Q1): every particle starts at the same point
        const double x0 = M::initial_state(c);
        __syncthreads();
        for (int p = tid; p < N; p += kCT) {
            s_x[p] = x0;
            s_cum[p] = (double)(p + 1);
            s_hist[p] = 0;
            if constexpr (SMO) {
                s_b[p] = s_b[NP + p] = s_b[2 * NP + p] = s_b[3 * NP + p] = 0;
                for (int q = 0; q < kB4Ring; ++q) s_B4[q * (size_t)NP + p] = 0;
                XPG(0)[p] = make_double2(x0, x0);
            }
            if (HESS) {
                ALG(0)[p] = make_double4(0.0, 0.0, 0.0, 0.0);
                if (p < SQ) w.xlow[p] = x0;
            }
            if (Xh) {
                Xh[p] = x0;
                Ah[p] = p;
            }
        }
        for (int t = tid; SMO && t < NOBS; t += kCT) {
            o_smo[t] = 0.0;
            o_grad[t] = 0.0;
            o_grad[NOBS + t] = 0.0;
            o_grad[2 * NOBS + t] = 0.0;
            o_grad[3 * NOBS + t] = 0.0;
        }
        if (tid == 0) {
            o_filt[0] = x0;
            o_traj[0] = x0;
            s_S[0] = (double)N;
            s_flag = 0;
        }
        double hacc[HESS ? 20 : 1];   // thread-local hessian1 / hessian2 sums (upper triangles)
#pragma unroll
        for (int q = 0; q < (HESS ? 20 : 1); ++q) hacc[q] = 0.0;
        double loglike = 0.0;
        double S_prev = (double)N;
        long long near_ties = 0, key_ties2 = 0;
        int max_occ = 0, status = 0;
        __syncthreads();

        // u of my children is fetched one time step ahead (HBM latency off the critical path)
        double un_next[kP];
#pragma unroll
        for (int m = 0; m < kP; ++m) {
            const int j = tid + m * kCT;
            un_next[m] = (j < N) ? ld_stream_f64(&U[(size_t)N + j]) : 0.0;
        }
        for (int inext = 1; inext < NOBS; ++inext) {
            const double y1 = obs[inext - 1], yi = obs[inext];
            const double u = rvr[inext];
            double un[kP];
#pragma unroll
            for (int m = 0; m < kP; ++m) {
                const int j = tid + m * kCT;
                un[m] = un_next[m];
                if (inext + 1 < NOBS) un_next[m] = (j < N) ? ld_stream_f64(&U[(size_t)(inext + 1) * N + j]) : 0.0;
            }
            // bin range predicted from the sorted parents: exact range of the propagation mean
            // over [x_min, x_max], widened by 6.5 sd (outliers clamp into the end bins)
            if (tid == 0) {
                double lo, hi;
                M::child_range(c, s_x[0], s_x[N - 1], y1, 6.5, lo, hi);
                double scale = (double)N / (hi - lo);
                if (!(hi > lo) || !isfinite(scale) || !isfinite(lo)) scale = 0.0;
                s_bin[0] = isfinite(lo) ? lo : 0.0;
                s_bin[1] = scale;
                s_bin[2] = hi;
            }
            __syncthreads();
            const double bin_lo = s_bin[0], bin_scale = s_bin[1], bin_hi = s_bin[2];
            // shift: maximum of the (concave) log-weight over the predicted range (the
            // reference's my_max, Q4, picks another element; the shift cancels analytically)
            const double shift = M::logw_max(c, bin_lo, bin_hi, yi);

            // =========== resample (:694-715) + propagate (:354-358) + bin histogram
            double xn[kP];
            int an[kP], bn[kP], rk[kP];
#pragma unroll
            for (int m = 0; m < kP; ++m) {
                const int j = tid + m * kCT;
                an[m] = bn[m] = rk[m] = 0;
                xn[m] = 0.0;
                if (j < N) {
                    const double cp = (u + (double)j) / (double)N;
                    // lower bound of cp among cum / S: searched with one multiplication per probe,
                    // then settled with the exact predicate (cum[m] / S < cp) on the neighbours
                    const double cps = cp * S_prev;
                    int l = 0, h = N - 1;
                    while (l < h) {
                        const int mid = (l + h) >> 1;
                        if (s_cum[mid] < cps) l = mid + 1;
                        else h = mid;
                    }
                    double cv_hi = s_cum[l] / S_prev;
                    double cv_lo = (l > 0) ? s_cum[l - 1] / S_prev : -1.0;
                    while (l > 0 && !(cv_lo < cp)) {   // (rare: the two quotients settle the probe result)
                        --l;
                        cv_hi = cv_lo;
                        cv_lo = (l > 0) ? s_cum[l - 1] / S_prev : -1.0;
                    }
                    while (l < N - 1 && (cv_hi < cp)) {
                        ++l;
                        cv_lo = cv_hi;
                        cv_hi = s_cum[l] / S_prev;
                    }
                    {   // diagnostics: decisions within 64 ulp of a cumulative-weight tie
                        const double tol = 64.0 * 2.220446049250313e-16 * cp;
                        if (fabs(cv_hi - cp) <= tol || (cv_lo >= 0.0 && fabs(cp - cv_lo) <= tol)) near_ties++;
                    }
                    xn[m] = M::propagate(c, s_x[l], y1, un[m]);
                    an[m] = l;
                    bn[m] = sv_bin(xn[m], bin_lo, bin_scale, N);
                    rk[m] = atomicAdd(&s_hist[bn[m]], 1);
                    if (HESS && j < SQ) w.xnf[j] = xn[m];
                }
            }
            __syncthreads();
            CPROF(0);   // resample + propagate + histogram
            // =========== bin starts (exclusive scan over N bins, kP consecutive bins per thread)
            {
                int v[kP], tsum = 0, occ = 0;
#pragma unroll
                for (int q = 0; q < kP; ++q) {
                    const int b = tid * kP + q;
                    v[q] = (b < N) ? s_hist[b] : 0;
                    tsum += v[q];
                    occ = max(occ, v[q]);
                }
                int total;
                int run = chain_scan_i(tsum, s_iw, &total);
#pragma unroll
                for (int q = 0; q < kP; ++q) {
                    const int b = tid * kP + q;
                    if (b < N) s_hist[b] = run;
                    run += v[q];
                }
                if (tid == 0) s_hist[N] = N;
                max_occ = max(max_occ, occ);
                if (occ > kChainBinMax) s_flag = 1;
            }
            __syncthreads();
            if (s_flag) {   // degenerate particle cloud: give up on this problem (uniform)
                status = 1;
                break;
            }
            CPROF(1);   // bin scan
            // =========== scatter into bin order
#pragma unroll
            for (int m = 0; m < kP; ++m) {
                const int j = tid + m * kCT;
                if (j < N) {
                    const int slot = s_hist[bn[m]] + rk[m];
                    s_key[slot] = xn[m];
                    int payv = an[m];
                    if (HESS) {
                        // Q7 reads xnew[slot'] only when slot' <= j: remember that in the spare bit
                        const long long qq = (long long)inext - 1 + an[m];
                        if ((int)(qq / NOBS) <= j) payv |= 0x8000;
                    }
                    s_pay[slot] = (unsigned short)payv;
                }
            }
            __syncthreads();
            // =========== order each bin (all pairs), fetch what the children inherit
            double xs[kP], xpar[kP];
            int pos[kP], anc[kP], ib1[kP], ib2[kP], ib3[kP];
            bool q7ok[kP];
#pragma unroll
            for (int m = 0; m < kP; ++m) {
                const int s = tid + m * kCT;
                pos[m] = -1;
                xs[m] = xpar[m] = 0.0;
                anc[m] = ib1[m] = ib2[m] = ib3[m] = 0;
                q7ok[m] = false;
                if (s < N) {
                    const double key = s_key[s];
                    const int payf = s_pay[s];
                    const int pay = payf & 0x7fff;
                    q7ok[m] = (payf & 0x8000) != 0;
                    const int b = sv_bin(key, bin_lo, bin_scale, N);
                    const int start = s_hist[b], end = s_hist[b + 1];
                    int rank = 0;
                    for (int q = start; q < end; ++q) {
                        if (q == s) continue;
                        const double k2 = s_key[q];
                        if (k2 < key) rank++;
                        else if (k2 == key) {
                            key_ties2++;
                            const int p2 = s_pay[q] & 0x7fff;
                            if ((p2 < pay) || (p2 == pay && q < s)) rank++;
                        }
                    }
                    pos[m] = start + rank;
                    xs[m] = key;
                    anc[m] = pay;
                    if constexpr (SMO) {
                        xpar[m] = s_x[pay];
                        ib1[m] = s_b[pay];
                        ib2[m] = s_b[NP + pay];
                        ib3[m] = s_b[2 * NP + pay];
                    }
                }
            }
            __syncthreads();   // every read of the parent generation is done
            CPROF(2);   // scatter + rank
            // =========== the new generation: values, carried positions, weights (:427-437), tables
            {
                double2* xpn = XPG(inext);
                unsigned short* b4n = s_B4 + (size_t)(inext % kB4Ring) * NP;
                const bool keep_tail = inext >= NOBS - LAG;
#pragma unroll
                for (int m = 0; m < kP; ++m) {
                    const int p = pos[m];
                    if (p >= 0) {
                        s_x[p] = xs[m];
                        if constexpr (SMO) {
                            s_b[p] = (unsigned short)anc[m];
                            s_b[NP + p] = (unsigned short)ib1[m];
                            s_b[2 * NP + p] = (unsigned short)ib2[m];
                            s_b[3 * NP + p] = (unsigned short)ib3[m];
                            b4n[p] = (unsigned short)ib3[m];
                        }
                        double sh = exp(M::logw(c, xs[m], yi) - shift);
                        if (!isfinite(sh)) sh = 0.0;
                        s_cum[p] = sh;
                        if constexpr (SMO) xpn[p] = make_double2(xs[m], xpar[m]);
                        if constexpr (HESS) {
                            // alpha recursion (:361-390).  Q7: particles[i - 1 + ancestors[j]] read through the flat
                            // layout = sorted value `sl` of time tq, or the unsorted new value `sl`, or 0
                            const long long qq = (long long)inext - 1 + anc[m];
                            const int tq = (int)(qq % NOBS), sl = (int)(qq / NOBS);
                            double curr;
                            if (tq < inext) curr = __ldcg(&w.xlow[(size_t)tq * SQ + sl]);
                            else if (tq == inext) curr = q7ok[m] ? __ldcg(&w.xnf[sl]) : 0.0;
                            else curr = 0.0;
                            const double ylag = obs_wrap(obs, inext - LAG, NOBS);   // Q8
                            double sq = xs[m] - c.mu - c.phi * (curr - c.mu);
                            const double ec = exp(-0.5 * curr);
                            sq -= c.sr * ec * ylag;
                            const double a0 = c.q * sq * c.one_m_phi;
                            const double a1 = c.q * sq * (curr - c.mu) * c.one_m_phi2;
                            double a2 = sq;
                            a2 += c.sr * ec * yi;
                            a2 *= c.q * sq;
                            a2 -= 1.0;
                            double a3 = c.rho - c.q * c.rho * sq * sq;
                            a3 += c.inv_sv * sq * ec * yi;
                            const double4 pa = chain_ld_d4(&ALG(inext - 1)[anc[m]]);
                            ALG(inext)[p] = make_double4(a0 + pa.x, a1 + pa.y, a2 + pa.z, a3 + pa.w);
                            if (p < SQ) w.xlow[(size_t)inext * SQ + p] = xs[m];
                        }
                        if (SMO && keep_tail) {
                            B1G(inext)[p] = anc[m];
                            SHG(inext)[p] = sh;
                        }
                        if (Xh) {
                            Xh[(size_t)inext * N + p] = xs[m];
                            Ah[(size_t)inext * N + p] = anc[m];
                        }
                    }
                }
                for (int b = tid; b < N; b += kCT) s_hist[b] = 0;
            }
            __syncthreads();
            CPROF(3);   // new generation: weights, tables
            // =========== position order: cumulative weights, sums, fixed-lag terms (:445-470)
            constexpr int NACC = SMO ? 6 : 1;   // sh x; sh x_lagged, sh g[0..3]
            double acc[NACC];
#pragma unroll
            for (int q = 0; q < NACC; ++q) acc[q] = 0.0;
            double S_i;
            {
                double v[kP], tsum = 0.0;
#pragma unroll
                for (int q = 0; q < kP; ++q) {
                    const int p = tid * kP + q;
                    v[q] = (p < N) ? s_cum[p] : 0.0;
                    tsum += v[q];
                }
                double run = chain_scan_d(tsum, s_w, &S_i);
                // pairing of the fixed-lag terms (pf_model.cuh): the reference's (Q5 / Q6) or the exact one, whose main
                // loop starts one step earlier (the pair (x_0, x_1) at step LAG - 1) and whose tail starts one step later
                const bool lagged = SMO && inext >= pair_first_step(M::kPairing, LAG);
                // the pair (x_tt, x_tt+1), tt = inext - LAG + 1: y = obs[tt - 1] (Q5), obs[tt + 1], or obs[tt] (predictive)
                const double yl = lagged ? obs[pair_obs(M::kPairing, inext - LAG + 1)] : 0.0;
                const int hop0 = (K >= 1) ? ((K - 1) & 3) : 0;
                const int nh = (K >= 1) ? ((K - 1) >> 2) : 0;        // 0 or 1 (LAG <= 10)
                const int g1 = inext - (hop0 + 1);
                const double2* xpk = SMO ? XPG(inext - K) : nullptr;
                int idl[kP];
#pragma unroll
                for (int q = 0; q < kP; ++q) {
                    const int p = tid * kP + q;
                    idl[q] = 0;
                    if (p < N && lagged) {
                        int id = p;
                        if (K >= 1) {
                            id = s_b[(size_t)hop0 * NP + p];
                            if (nh) id = s_B4[(size_t)(g1 % kB4Ring) * NP + id];
                        }
                        idl[q] = id;
                    }
                }
                double2 pv[kP];
#pragma unroll
                for (int q = 0; q < kP; ++q) pv[q] = lagged ? __ldcg(&xpk[idl[q]]) : make_double2(0.0, 0.0);
#pragma unroll
                for (int q = 0; q < kP; ++q) {
                    const int p = tid * kP + q;
                    if (p < N) {
                        run += v[q];
                        s_cum[p] = run;
                        const double sx = v[q] * s_x[p];
                        if (isfinite(sx)) acc[0] += sx;
                        if constexpr (SMO) if (lagged) {
                            double g[4];
                            if constexpr (HESS) {
                                double sq;
                                const double ec = exp(-0.5 * pv[q].y);
                                sv_score_main_e(c, pv[q].y, ec, pv[q].x, yl, sq, g);
                                const double4 a4 = chain_ld_d4(&ALG(inext - K)[idl[q]]);
                                const double al[4] = {a4.x, a4.y, a4.z, a4.w};
                                // (normalised weight, as the reference; the 20 sums stay thread-local over the
                                // whole series and are reduced once at the end)
                                sv_hessian_terms_e(c, pv[q].y, ec, ec * ec, sq, yl, g, al, v[q] / S_i, hacc);
                            } else {
                                pair_score<M>(c, inext == LAG - 1, pv[q].y, pv[q].x, yl, g);
                            }
                            acc[1] += v[q] * pv[q].y;
                            acc[2] += g[0] * v[q];
                            acc[3] += g[1] * v[q];
                            acc[4] += g[2] * v[q];
                            acc[5] += g[3] * v[q];
                        }
                    }
                }
                block_sum<NACC>(acc, s_red);
            }
            if (!(S_i > 0.0) || !isfinite(S_i)) {   // uniform
                status = 1;
                break;
            }
            loglike += shift + log(S_i) - logN;   // :537
            if (tid == 0) {
                s_S[inext % kMaxLagC] = S_i;
                o_filt[inext] = acc[0] / S_i;
                o_traj[inext] = s_x[0];   // Q11: traj[i] = X_i[0]
                if constexpr (SMO) if (inext >= pair_first_step(M::kPairing, LAG)) {
                    const int tt = inext - LAG + 1;
                    const int gs = pair_slot(M::kPairing, tt);
                    o_smo[tt] = acc[1] / S_i;
                    o_grad[gs] = acc[2] / S_i;
                    o_grad[NOBS + gs] = acc[3] / S_i;
                    o_grad[2 * NOBS + gs] = acc[4] / S_i;
                    o_grad[3 * NOBS + gs] = acc[5] / S_i;
                }
            }
            S_prev = S_i;
            __syncthreads();
            CPROF(4);   // cumulative weights, sums, fixed-lag terms, outputs
        }   // time loop

        // ---------------- tail (:540-562, Q6; exact pairing: slots NOBS-LAG+1 .. NOBS-1, pairs under the final weights;
        // predictive: the same slots, k = 0 adds the final generation's term into slot T).  n_obs >= LAG + 1, so the
        // tail's pairs start at x_2 and the pair (x_0, x_1) is the main loop's)
        if (SMO && status == 0) {
            const int T = NOBS - 1;
            const double S_T = s_S[T % kMaxLagC];
            const double* shT = SHG(T);
            constexpr Pairing PR = M::kPairing;
            for (int k = 0; k < (PR == Pairing::Reference ? LAG : LAG - 1); ++k) {
                const int ip = T - k;
                constexpr int NT = 5;
                double tacc[NT];
#pragma unroll
                for (int q = 0; q < NT; ++q) tacc[q] = 0.0;
                const double ylag = obs_wrap(obs, ip - LAG, NOBS);
                const double S_ip = s_S[ip % kMaxLagC];
                const double y1 = PR == Pairing::Reference ? obs_wrap(obs, pair_obs(PR, ip), NOBS)
                                  : (k >= 1 || PR == Pairing::Predictive ? obs[pair_obs(PR, ip)] : 0.0);
                const double* shI = SHG(ip);
                for (int j = tid; j < N; j += kCT) {
                    int b = j, bprev = j;
                    for (int h = 0; h < k; ++h) {
                        bprev = b;
                        b = __ldcg(&B1G(T - h)[b]);
                    }
                    const double curr = __ldcg(&XPG(ip)[b]).x;
                    double sT = __ldcg(&shT[j]);
                    if (!isfinite(sT)) sT = 0.0;
                    tacc[0] += (sT / S_T) * curr;
                    if (k >= 1) {
                        const double next = __ldcg(&XPG(ip + 1)[bprev]).x;
                        double g[4];
                        double wi;
                        if constexpr (PR == Pairing::Reference) {
                            double si = __ldcg(&shI[j]);
                            if (!isfinite(si)) si = 0.0;
                            wi = si / S_ip;
                        } else {
                            wi = sT / S_T;
                        }
                        if constexpr (HESS) {
                            double sq;
                            sv_score_tail(c, curr, next, y1, sq, g);
                            int b_l2 = j;   // index at lag LAG-2 (for alpha)
                            for (int h = 0; h < LAG - 2; ++h) b_l2 = __ldcg(&B1G(T - h)[b_l2]);
                            const double4 a4 = chain_ld_d4(&ALG(T - LAG + 2)[b_l2]);
                            const double al[4] = {a4.x, a4.y, a4.z, a4.w};
                            sv_hessian_terms(c, curr, sq, ylag, g, al, wi, hacc);
                        } else {
                            M::score_tail(c, curr, next, y1, g);
                        }
                        tacc[1] += g[0] * wi;
                        tacc[2] += g[1] * wi;
                        tacc[3] += g[2] * wi;
                        tacc[4] += g[3] * wi;
                    } else if constexpr (PR == Pairing::Predictive) {   // the final generation's term
                        const double wi = sT / S_T;
                        double g[4];
                        M::score_last(c, curr, y1, g);
                        tacc[1] += g[0] * wi;
                        tacc[2] += g[1] * wi;
                        tacc[3] += g[2] * wi;
                        tacc[4] += g[3] * wi;
                    }
                }
                block_sum<NT>(tacc, s_red);
                if (tid == 0) {
                    o_smo[ip] += tacc[0];
                    if (k >= 1 || PR == Pairing::Predictive) {
                        const int tt = PR == Pairing::Reference ? ip - LAG + 1 : pair_slot(PR, ip);
                        if (tt >= 0) {
                            o_grad[tt] += tacc[1];
                            o_grad[NOBS + tt] += tacc[2];
                            o_grad[2 * NOBS + tt] += tacc[3];
                            o_grad[3 * NOBS + tt] += tacc[4];
                        }
                    }
                }
                __syncthreads();
            }
        }

        // ---------------- outputs
        if constexpr (HESS) {
            block_sum<20>(hacc, s_red);
            if (tid < 20) s_hacc[tid] = hacc[tid];
            __syncthreads();
        }
        {
            double nt[2] = {(double)near_ties, (double)key_ties2};
            block_sum<2>(nt, s_red);
            int mo = warp_max(max_occ);
            if (lane == 0) s_iw[warp] = mo;
            __syncthreads();
            if (tid == 0) {
                for (int q = 0; q < kCNW; ++q) mo = max(mo, s_iw[q]);
                a.loglike[prob] = (status == 0) ? loglike : NAN;
                o_diag[kDiagNearTies] = (long long)nt[0];
                o_diag[kDiagKeyTies] = (long long)(nt[1] * 0.5);
                o_diag[kDiagMaxBin] = mo;
                o_diag[kDiagStatus] = status;
                o_diag[kDiagWavefront] = 0;
                o_diag[kDiagTrajIdx] = 0;
                o_diag[kDiagKernel] = 3;
                o_diag[kDiagFastInfo] = 0;
            }
            if (tid < 16 && status == 0 && a.hess1) {
                // expand the upper triangles into the symmetric 4x4 outputs
                const int r = tid >> 2, cidx = tid & 3;
                const int k = min(r, cidx), l = max(r, cidx);
                const int tri = k * 4 - (k * (k - 1)) / 2 + (l - k);
                a.hess1[(size_t)prob * 16 + tid] = HESS ? s_hacc[tri] : 0.0;
                a.hess2[(size_t)prob * 16 + tid] = HESS ? s_hacc[10 + tri] : 0.0;
            }
            __syncthreads();
        }
    }   // problem loop
#undef XPG
#undef B1G
#undef SHG
#undef ALG
}

}  // namespace

int sv_chain_eligible(int N, int LAG) { return N >= 2 && N <= kChainMaxN && LAG >= 2 && LAG <= 10; }

size_t sv_chain_ws_bytes(int N, int LAG, int NOBS, int hess, int filter) {
    if (filter) return 0;
    const int SQ = hess ? (NOBS + N - 2) / NOBS + 1 : 1;
    return chain_ws_carve(N, LAG, NOBS, SQ, hess, nullptr, nullptr);
}

int sv_chain_smem_bytes(int N) {
    const size_t NP = (size_t)((N + 1) & ~1);
    return (int)(NP * 8 * 3 + (NP + 2) * 4 + NP * 2 * (4 + kB4Ring + 1) + 64);
}

template <class M, bool HESS, bool SMO>
static cudaError_t chain_launch_one(const SvArgs& a, int grid, int smem, cudaStream_t stream) {
    cudaError_t err = cudaFuncSetAttribute(sv_chain_kernel<M, HESS, SMO>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem);
    if (err != cudaSuccess) return err;
    sv_chain_kernel<M, HESS, SMO><<<grid, kCT, smem, stream>>>(a);
    return cudaGetLastError();
}

// the filter runs the instantiation of M::Filter, the smoother without the Hessian that of M::Gradient; this kernel has
// the SV model's Hessian branch only (the generic one is the grid kernel's)
cudaError_t sv_chain_launch(const SvArgs& a, int grid, int filter, cudaStream_t stream) {
    const int smem = sv_chain_smem_bytes(a.N);
    cudaError_t err = cudaErrorInvalidValue;
    Models::with(a.model_id, [&](auto m) {
        typedef typename decltype(m)::type M;
        if (filter) {
            if (!a.hess) err = chain_launch_one<typename M::Filter, false, false>(a, grid, smem, stream);
        } else if (!a.hess) {
            err = chain_launch_one<typename M::Gradient, false, true>(a, grid, smem, stream);
        } else if constexpr (M::kHessian && M::kPairing == Pairing::Reference) {
            err = chain_launch_one<M, true, true>(a, grid, smem, stream);
        }
    });
    return err;
}

}  // namespace pmmh
