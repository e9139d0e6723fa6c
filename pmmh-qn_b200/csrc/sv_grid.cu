// sv_grid.cu -- the "grid kernel": ONE stochastic-volatility fixed-lag smoother evaluation
// (log-likelihood + gradient) as ONE persistent cooperative launch over all SMs.
//
// Restates flps_sv_corr (/root/reference/python/state/particle_methods/stochastic_volatility.pyx
// :205-655: correlated systematic resampling :694-715, propagation :354-358, argsort :392-424 /
// :23-52, weights :427-442, fixed-lag score terms :445-470, tail :540-562, log-likelihood :537,
// trajectory :630-633 with quirks Q10/Q11).  B200 design, 148 CTAs, one CTA per SM:
//
//   * the sorted generation is cut into G TILES of ~N/G particles (7 085 at N = 2^20, G = 148);
//     CTA c owns tile c while it is sorted and weighted (shared memory) and owns the CHILDREN
//     [c*Wc, (c+1)*Wc) while they are generated (equal work for every CTA whatever the weights
//     look like);
//   * four grid barriers per time step (one atomic counter, arrive / wait split so that work that
//     only feeds outputs sits between the two):
//       C  owner of a tile: cumulative weights -> PARENT-side child ranges in closed form
//          ub(p) = #{j : (u + j)/N <= cum(p)} (exact predicate re-checked), ancestor of every
//          child written to H (coalesced fill)                                     | barrier 4
//       A1 owner of a child range: parent (x, exp(-x/2), birth row), propagation, 8192-bin value
//          histogram (shared-memory atomics, merged into the global one), payload of the child
//          for the fixed-lag terms 8 steps later                                   | barrier 1
//          (after the arrive: genealogy records)
//       A2 scan of the global histogram -> tile boundaries on bin edges (every tile gets N/G
//          particles +- one bin), slot reservation per (CTA, tile), entries written to the
//          mailbox of their tile in runs (value, birth row, lagged ancestor row)  | barrier 2
//       B  owner of a tile: counting sort over 4096 sub-bins of the tile's value range + exact
//          in-bin ranking by (value, birth row) = the reference's argsort; weights, sorted
//          generation written out, block scan of the weights, moments             | barrier 3
//          (after the arrive: fixed-lag score terms, one random 32-byte sector per particle)
//   * genealogy: a generation is stored ONCE in birth order as P[t][j] = (parent value, residual
//     of the transition, exp(-parent/2) obs, value) and R[t][j] = birth rows of the ancestors 1..8
//     steps back (one 32-byte sector each).  The fixed-lag terms of step t need one random sector
//     of P[t-lag+2]; a child copies its parent's R with one random sector read.  No history is
//     ever moved.
//   * two exp per particle and step: exp(-x/2) is shared by the weight, the propagation mean of
//     the children and the payload; the score terms need none.
//   * L2 eviction hints on every access (createpolicy): data that is dead after its read (previous record
//     table, mailbox entries, H, the parents' (x, e) / perm entries, lagged payloads, u) is read
//     evict_first, what the next phase reads is stored evict_last: 114 -> 103 us per step.
//   * tried and measured slower (git history): descendant weights by integer atomics + sequential
//     payload pass (132 us per step), genealogy and score terms on dedicated helper warps (122 -
//     150 us: the helper's traffic slows the main warps as much as it saves them), pointer-jumping
//     tables instead of records, bulk L2 prefetch of the lagged generation, L2 prefetch of the record / payload
//     sectors a phase ahead, 16-byte payloads with an exp in the score terms, pointer-jumping tables by all
//     threads (DRAM traffic 189 -> 138 MB per step, but the three dependent 4-byte gathers still miss L2:
//     27 us against 14 us for the records, 118 us per step).  With the hints: 100 us; with the fence-free barrier
//     (release / acquire on the counter, abandon flag in its bit 31): 94 - 96 us.
//   * per-thread state off the stack (1024 threads at 64 registers, and 208 KB of shared memory leave ~28 KB of L1:
//     a stack slot is an L2 round trip): the records pass selects the lagged ancestor by compare-and-select (pick8),
//     phase C's rare exact search runs after its unrolled loop, the tie counters of phase C are shared-memory
//     atomics, and the children's values, ancestor rows and mailbox slots of phase A sit in shared memory regions
//     that are dead from phase C's ancestor fill to phase B (ChildSlots).  ptxas (-Xptxas -v): stack frame / spill
//     stores / loads of the SV gradient instantiation 144 / 516 / 556 -> 32 / 96 / 112 bytes, team 152 / 544 / 568
//     -> 80 / 316 / 492 (tools/grid_local_memory.py counts the STL / LDL sites per phase).  Measured (B200, 1000 W):
//     94 -> 82 us per step, bit-identical outputs.
//   * second instantiation HESS = true: the Hessian branch (:361-390, :472-534, :564-626), cumulative alpha in the second
//     sector of 64-byte record / payload entries; 162 us per step (DESIGN 4.0).
//   * host-resident u: particle-major slots filled by the copy engine, one 32-byte sector (4 steps) per particle re-laid
//     time-major every fourth step (DESIGN 3).
//   * template over the model (pf_model.cuh): SvLeverageModel is everything above; another model runs the generic path
//     in the same body (XE = (x, propagation mean of the children), payload = (parent value, -, -, value), score terms
//     M::score_main / M::score_tail), gradient only (DESIGN 4.0).
//   * TEAM = true (pmmh_flps_model_batch_corr / pmmh_filter_model_batch_corr): a batch of problems, one team of G CTAs
//     per problem -- CTA b runs tile b % G of problem b / G on that team's own slice of the workspace (the one-problem
//     layout: own barrier counter, abandon bit and status word), so every problem is bit-identical to its one-problem
//     run and an abandoned problem stops its team only; waves of floor(SMs / G) teams, one cooperative launch each.
//     A wave of one problem (and a one-problem call, a batch of one) runs TEAM = false.
//   * SMO = false: the particle filter alone (pmmh_filter_model_corr) -- no payloads, no genealogy records, no score
//     terms, no tail; the workspace has no R / P tables and no weight ring.  The birth rows stay: the in-bin ranking
//     breaks ties on them.
//
// Deviations from the reference's operation order: parallel sums / scans, log(exp(x/2)) = x/2 and
// 1/exp(x/2)^2 = exp(-x/2)^2 in the log-weight, cumulative weights multiplied by 1/S; any
// log-weight shift cancels (Q4).  Resampling decisions within 64 ulp of a cumulative-weight tie
// are counted in diag[0]; decisions closer than the sequential-vs-tree summation bound are
// counted separately (ctrl->soft_ties, reported by pmmh_sv_grid_last_info).
// fp64, -fmad=false.  Bound: L2 / HBM streaming and gathers; no tensor cores (no contraction).
#include <cuda_runtime.h>
#include <math.h>
#include <stdint.h>
#include <string.h>

#include <type_traits>

#include "../../include/pmmh_qn.h"
#include "common.cuh"
#include "pf_model.cuh"
#include "sv_grid.cuh"
#include "sv_math.cuh"

namespace pmmh {

int set_error(int code, const char* what);           // capi.cu
int set_cuda_error(cudaError_t err, const char* where);

namespace {

constexpr int kCap = 8192;         // entries of one tile (shared-memory capacity)
constexpr int kNF = 8192;          // bins of the global value histogram
constexpr int kNSB = 4096;         // sub-bins of the in-tile counting sort
constexpr int kMaxSub = 1024;      // a sub-bin larger than this abandons the evaluation
constexpr int kMaxTiles = 160;     // >= SM count
constexpr int kCntStride = 32;     // ints between two slot counters (one 128-byte line each)
constexpr double kZ = 6.5;         // histogram range: predicted mean +- 6.5 predicted sd
constexpr int kDynSmem = 208 * 1024;
constexpr int kProf = 32;

struct __align__(16) MailEntry {   // aliases one (x, exp(-x/2)) pair of the sorted generation
    double x;
    int j, a;
};
// Payload of a particle for the fixed-lag terms (one 32-byte sector, birth order): parent value c,
// residual sq of the transition (:452-453), ey = exp(-c/2) * obs[i - LAG], own value x (tail)
struct __align__(32) PEntry {
    double c, sq, ey, x;
};
struct __align__(32) REntry {
    int a[8];              // birth rows of the ancestors 1 .. 8 steps back
};

struct GridCtrl {
    unsigned bar;                  // arrival counter of the grid barrier (monotone)
    int status;                    // 0, or (reason << 24) | first barrier index at which everybody stops
    int max_bin;
    int pad0;
    unsigned long long near_ties, soft_ties, key_ties;
};

struct GridArgs {
    int N, NOBS, LAG, G, Wc, RP, hist;
    // always 0 (grid_args).  The kernel's tests of it are dead, but deleting them changes register allocation and
    // measured slower (B200, 1000 W: 94.1 -> 96.9 ms per evaluation at N = 2^20, T = 1000, lag 10)
    int dbg;
    const double *obs, *params, *rvr, *U;
    // U[t][j] = U[(t / u_cs) * u_cstride + (t % u_cs) * u_tstride + j * u_jstride]: time-major resident array
    // (u_cs = 2^30, u_tstride = N, u_jstride = 1) or particle-major chunks of u_cs time steps as the copy
    // engine lays them down from the reference's host array (u_tstride = 1, u_jstride = u_cs)
    long long u_cstride, u_tstride, u_jstride;
    int u_cs;
    const int* u_flag;   // host-streamed u: number of time rows that have landed (written by the copy engine)
    double* ustash;      // [4][N] host-streamed u: the four time steps of one 32-byte sector per particle, time-major
    GridCtrl* ctrl;
    int* ghist;        // [2][kNF]
    int* tilecnt;      // [2][kMaxTiles * kCntStride]
    double* tinfo;     // [kMaxTiles][4]  tot, n, sum sh m, sum sh m^2
    int* H;            // [N] ancestor (sorted position) of every child
    double2* XE;       // [N] sorted generation: (x, exp(-x/2)); the mailbox of the next generation aliases it
    int* perm;         // [N] sorted position -> birth row
    REntry* R;         // [2][N]
    PEntry* P;         // [RP][N] payloads of generation t % RP
    double* psum;      // [NOBS][G][8]
    // Hessian branch (:361-390, :472-534, :564-626) only: the entries of R and P are 64 bytes (RS = 2 sectors), the
    // second sector is the cumulative alpha (4 parameters) of the particle -- next to its record for the children
    // (who gather both with one 64-byte access) and next to its payload for the descendants LAG-2 steps later
    int RS;            // 32-byte sectors per entry of R and P (1, Hessian branch 2)
    double* xlow;      // [SQ][NOBS] the first SQ sorted values of every generation, slot-major: consecutive parents read
                       // consecutive times (Q7), so the reads of a warp coalesce
    double* psumH;     // [NOBS][G][20] per-step sums: [0..3] monomials of hessian1, [10..19] hessian2 (upper triangle)
    int SQ;
    double *shiftv, *xminv;   // [NOBS]
    double* shring;    // [LAG][N] sh of the last LAG generations (sorted order)
    int* parentpos;    // [N] (history dump only)
    double* Xhist;
    int* Ahist;
    long long* prof;
};

struct StepScalars {
    double S, invS, mhat, shat, inv_shat, shift, lo, scale, tot, offk;
    double tol_soft, tol_near;   // resampling ties: sequential-vs-tree summation bound, 64 ulp of N
    int carry, abort_now, binlo, binhi;
};

// ---- small device helpers ---------------------------------------------------------------------
// the SV model's constants, which the SV code of the kernel reads; another model has none (zeros, never used)
__device__ __forceinline__ const SvConst& sv_of(const SvConst& k) { return k; }
template <class C>
__device__ __forceinline__ SvConst sv_of(const C&) {
    return SvConst();
}
__device__ __forceinline__ void red_release_add(unsigned* p, unsigned v) {
    asm volatile("red.release.gpu.global.add.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}
__device__ __forceinline__ void prefetch_l2_bulk(const void* p, unsigned bytes) {
    asm volatile("cp.async.bulk.prefetch.L2.global [%0], %1;" ::"l"(p), "r"(bytes) : "memory");
}
// [p0, p1) -> L2 in 16 KB pieces (sequential HBM reads issued by the copy unit, no SM cycles);
// the pieces are dealt to the callers round-robin: piece k goes to caller k % nlanes == lane
__device__ __forceinline__ void prefetch_range(const void* b0, const void* b1, int lane, int nlanes) {
    const char* q0 = (const char*)(((uintptr_t)b0 + 15) & ~(uintptr_t)15);
    const char* q1 = (const char*)((uintptr_t)b1 & ~(uintptr_t)15);
    for (const char* q = q0 + (size_t)lane * 16384; q < q1; q += (size_t)nlanes * 16384)
        prefetch_l2_bulk(q, (unsigned)min((long long)16384, (long long)(q1 - q)));
}
__device__ __forceinline__ unsigned long long policy_evict_first() {
    unsigned long long pol;
    asm volatile("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(pol));
    return pol;
}
__device__ __forceinline__ unsigned long long policy_evict_normal() {
    unsigned long long pol;
    asm volatile("createpolicy.fractional.L2::evict_normal.b64 %0, 1.0;" : "=l"(pol));
    return pol;
}
__device__ __forceinline__ unsigned long long policy_evict_last() {
    unsigned long long pol;
    asm volatile("createpolicy.fractional.L2::evict_last.b64 %0, 1.0;" : "=l"(pol));
    return pol;
}
// 32-byte genealogy records: one 256-bit access with an L2 eviction hint (no persisting L2 set-aside: see
// grid_set_attributes)
__device__ __forceinline__ void ld_rec(const REntry* p, unsigned long long pol, int (&r)[8]) {
    asm volatile("ld.global.cg.L2::cache_hint.v8.s32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8], %9;"
                 : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7])
                 : "l"(p), "l"(pol));
}
__device__ __forceinline__ void st_rec(REntry* p, unsigned long long pol, int a0, int a1, int a2, int a3, int a4,
                                       int a5, int a6, int a7) {
    asm volatile("st.global.cg.L2::cache_hint.v8.s32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8}, %9;" ::"l"(p), "r"(a0),
                 "r"(a1), "r"(a2), "r"(a3), "r"(a4), "r"(a5), "r"(a6), "r"(a7), "l"(pol)
                 : "memory");
}
// streaming 32-byte store that should leave L2 first (written once, read lag - 2 steps later)
__device__ __forceinline__ void st_stream_f64x4(void* p, unsigned long long pol, double a, double b, double c, double d) {
    asm volatile("st.global.cs.L2::cache_hint.v4.f64 [%0], {%1,%2,%3,%4}, %5;" ::"l"(p), "d"(a), "d"(b), "d"(c), "d"(d),
                 "l"(pol)
                 : "memory");
}
__device__ __forceinline__ double ld_stream_hint_f64(const double* p, unsigned long long pol) {
    double v;
    asm volatile("ld.global.nc.L1::no_allocate.L2::cache_hint.f64 %0, [%1], %2;" : "=d"(v) : "l"(p), "l"(pol));
    return v;
}
// L2 residency plan: what the next phase or the next step reads again -- the
// sorted (x, e) pairs / the mailbox that aliases them, perm, H, the genealogy records being written -- is
// stored evict_last (56 MB at N = 2^20); what is dead after its read -- the previous record table, the
// mailbox entries, H, u -- and what is not read for 8 steps -- the payloads -- goes evict_first
__device__ __forceinline__ void st_hint_b128(void* p, unsigned long long pol, int4 v) {
    asm volatile("st.global.cg.L2::cache_hint.v4.s32 [%0], {%1,%2,%3,%4}, %5;" ::"l"(p), "r"(v.x), "r"(v.y), "r"(v.z),
                 "r"(v.w), "l"(pol)
                 : "memory");
}
__device__ __forceinline__ int4 ld_hint_b128(const void* p, unsigned long long pol) {
    int4 v;
    asm volatile("ld.global.cg.L2::cache_hint.v4.s32 {%0,%1,%2,%3}, [%4], %5;"
                 : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w)
                 : "l"(p), "l"(pol));
    return v;
}
__device__ __forceinline__ void st_hint_b32(void* p, unsigned long long pol, int v) {
    asm volatile("st.global.cg.L2::cache_hint.s32 [%0], %1, %2;" ::"l"(p), "r"(v), "l"(pol) : "memory");
}
__device__ __forceinline__ int ld_hint_b32(const void* p, unsigned long long pol) {
    int v;
    asm volatile("ld.global.cg.L2::cache_hint.s32 %0, [%1], %2;" : "=r"(v) : "l"(p), "l"(pol));
    return v;
}
__device__ __forceinline__ void ld_f64x4(const void* p, unsigned long long pol, double& a, double& b, double& c, double& d) {
    asm volatile("ld.global.cg.L2::cache_hint.v4.f64 {%0,%1,%2,%3}, [%4], %5;"
                 : "=d"(a), "=d"(b), "=d"(c), "=d"(d)
                 : "l"(p), "l"(pol));
}
__device__ __forceinline__ void st_keep_f64x4(void* p, unsigned long long pol, double a, double b, double c, double d) {
    asm volatile("st.global.cg.L2::cache_hint.v4.f64 [%0], {%1,%2,%3,%4}, %5;" ::"l"(p), "d"(a), "d"(b), "d"(c), "d"(d),
                 "l"(pol)
                 : "memory");
}
__device__ __forceinline__ int warp_incl_max(int v, int lane) {
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
        const int o = __shfl_up_sync(kFullMask, v, d);
        if (lane >= d) v = max(v, o);
    }
    return v;
}
// r[min(idx, 7)] for idx >= 0 by compare-and-select over the static indices: a runtime index into r would put the
// records of the records pass on the stack
__device__ __forceinline__ int pick8(const int (&r)[8], int idx) {
    int v = r[0];
#pragma unroll
    for (int z = 1; z < 8; ++z) v = idx >= z ? r[z] : v;
    return v;
}

// the resampling point of child j, (u + j) / N as the reference computes it (:703)
__device__ __forceinline__ double cpoint(double u, int j, double dn, double inv_n, bool pow2) {
    const double s = u + (double)j;
    return pow2 ? s * inv_n : s / dn;
}
__device__ __forceinline__ int count_le_slow(int est, double c, double u, int N, double dn, double inv_n, bool pow2) {
    while (est > 0 && cpoint(u, est - 1, dn, inv_n, pow2) > c) --est;
    while (est < N && cpoint(u, est, dn, inv_n, pow2) <= c) ++est;
    return est;
}
// #{ j in [0, N) : (u + j) / N <= c }: closed form, then the exact predicate of :703-711 on both
// neighbours.  false: the closed form missed (a tie within rounding, or the ends of the range: rare), `est` is where
// the exact search count_le_slow starts.  frac_out = distance of c*N - u to the nearest integer (how close to a tie).
__device__ __forceinline__ bool count_le_fast(double c, double u, int N, double dn, double inv_n, bool pow2, int& est,
                                              double& frac_out) {
    const double e = c * dn - u;
    if (!(e >= 0.0) || e >= dn - 1.0) {
        frac_out = 1.0;
        est = e >= 0.0 ? N : 0;
        return false;
    }
    const int fi = (int)e;               // floor(e), 0 <= fi <= N - 2
    const double fl = (double)fi;
    const double fr = e - fl;
    frac_out = fmin(fr, 1.0 - fr);
    const double slo = u + fl, shi = u + (fl + 1.0);   // u + j for j = fi, fi + 1 (both exact conversions)
    est = fi + 1;
    return pow2 ? (slo * inv_n <= c && !(shi * inv_n <= c)) : (slo / dn <= c && !(shi / dn <= c));
}
__device__ __forceinline__ int count_le(double c, double u, int N, double dn, double inv_n, bool pow2,
                                        double& frac_out) {
    int est;
    return count_le_fast(c, u, N, dn, inv_n, pow2, est, frac_out) ? est : count_le_slow(est, c, u, N, dn, inv_n, pow2);
}

__device__ __forceinline__ int fine_bin(double x, double mhat, double inv_shat) {
    const double t = ((x - mhat) * inv_shat + kZ) * ((double)kNF / (2.0 * kZ));
    if (!(t >= 0.0)) return 0;
    if (t >= (double)kNF) return kNF - 1;
    return (int)t;
}
__device__ __forceinline__ int sub_bin(double x, double lo, double scale) {
    const double t = (x - lo) * scale;
    if (!(t >= 0.0)) return 0;
    if (t >= (double)kNSB) return kNSB - 1;
    return (int)t;
}

// Block-wide exclusive scans over one value per thread.  s_w: shared [32].  Every warp scans the
// warp totals itself (shuffles), so there are two barriers and no serial loop; the order of the
// additions is fixed (deterministic).  s_w may be reused right after the call.
template <int GT>
__device__ __forceinline__ int block_excl_scan_int(int v, int* s_w, int& total, int lane, int warp) {
    constexpr int NW = GT / 32;
    const int incl = warp_incl_scan(v, lane);
    __syncthreads();
    if (lane == 31) s_w[warp] = incl;
    __syncthreads();
    const int wt = (lane < NW) ? s_w[lane] : 0;
    const int wincl = warp_incl_scan(wt, lane);
    total = __shfl_sync(kFullMask, wincl, 31);
    const int woff = __shfl_sync(kFullMask, wincl - wt, warp);
    return woff + incl - v;
}
template <int GT>
__device__ __forceinline__ int block_excl_max_int(int v, int init, int* s_w, int lane, int warp) {
    constexpr int NW = GT / 32;
    const int incl = warp_incl_max(v, lane);
    __syncthreads();
    if (lane == 31) s_w[warp] = incl;
    __syncthreads();
    const int wt = (lane < NW) ? s_w[lane] : init;
    const int wincl = warp_incl_max(wt, lane);
    int wex = __shfl_up_sync(kFullMask, wincl, 1);
    if (lane == 0) wex = init;
    const int woff = max(init, __shfl_sync(kFullMask, wex, warp));
    int ex = __shfl_up_sync(kFullMask, incl, 1);
    if (lane == 0) ex = init;
    return max(woff, ex);
}

// Hessian branch: the alpha terms whose Q7 read falls into the generation being built (listed by the records pass),
// one thread per entry
__device__ __forceinline__ void deferred_alpha_pass(const GridArgs& a, const SvConst& k, const int2* list, int nd, int t,
                                                    int jb, int tid, int nthreads, unsigned long long pol_rld,
                                                    unsigned long long pol_rst, unsigned long long pol_stream) {
    const int N = a.N, NOBS = a.NOBS, RS = a.RS;
    const double yi = a.obs[t], ylagH = obs_wrap(a.obs, t - a.LAG, NOBS);
    const REntry* Rp = a.R + (size_t)((t - 1) & 1) * N * RS;
    REntry* Rc = a.R + (size_t)(t & 1) * N * RS;
    PEntry* Pt = a.P + (size_t)(t % a.RP) * N * RS;
    for (int d = tid; d < nd; d += nthreads) {
        const int2 e = list[d];
        const int j = jb + e.x;
        const int b = min(max(e.y, 0), N - 1);
        const int ppos = min(max(__ldcg(&a.H[j]), 0), N - 1);
        const int sl = (int)(((unsigned)(t - 1) + (unsigned)ppos) / (unsigned)NOBS);
        const double x = __ldcg(&Pt[(size_t)j * RS].x);
        const double curr = (sl <= j && sl < N) ? __ldcg(&Pt[(size_t)sl * RS].x) : 0.0;
        double p0, p1, p2, p3;
        ld_f64x4(&Rp[(size_t)b * RS + 1], pol_rld, p0, p1, p2, p3);
        double al[4];
        sv_alpha_terms(k, x, curr, yi, ylagH, al);
        const double c0 = al[0] + p0, c1 = al[1] + p1, c2 = al[2] + p2, c3 = al[3] + p3;
        st_keep_f64x4(&Rc[(size_t)j * RS + 1], pol_rst, c0, c1, c2, c3);
        st_stream_f64x4((REntry*)&Pt[(size_t)j * RS] + 1, pol_stream, c0, c1, c2, c3);
    }
}

// generic Hessian branch (pf_model.cuh): h1 += w H and h2 += w (g g' + al g' + g al') over the upper triangles (row by
// row, as M::hess_main writes H)
__device__ __forceinline__ void louis_add(const double (&hh)[10], const double (&g)[4], const double* al, double w,
                                          double* h1, double* h2) {
    int z = 0;
#pragma unroll
    for (int r = 0; r < 4; ++r)
#pragma unroll
        for (int c = r; c < 4; ++c, ++z) {
            h1[z] = fma(w, hh[z], h1[z]);
            h2[z] = fma(w, g[r] * g[c] + al[r] * g[c] + g[r] * al[c], h2[z]);
        }
}

// Teams: CTA b runs tile b % G of problem (team) b / G.  a_in addresses team 0; team k's workspace slice starts
// ws_stride bytes after team k-1's (the one-problem layout, so every team has its own barrier counter, abandon bit
// and status word), its inputs and history one problem further on (obs by obs_stride doubles)
struct GridTeam {
    long long ws_stride;
    long long obs_stride;
};
template <class T>
__device__ __forceinline__ T* team_ptr(T* p, long long bytes) {
    return (T*)((char*)p + bytes);
}
__device__ __forceinline__ GridArgs team_args(const GridArgs& a0, const GridTeam& tm) {
    const int team = blockIdx.x / a0.G;
    const long long w = tm.ws_stride * team, nu = (long long)a0.NOBS * a0.N * team;
    GridArgs a = a0;
    a.obs += tm.obs_stride * team;
    a.params += 4 * team;
    a.rvr += (long long)a0.NOBS * team;
    a.U += nu;
    a.ctrl = team_ptr(a0.ctrl, w);
    a.ghist = team_ptr(a0.ghist, w);
    a.tilecnt = team_ptr(a0.tilecnt, w);
    a.tinfo = team_ptr(a0.tinfo, w);
    a.H = team_ptr(a0.H, w);
    a.XE = team_ptr(a0.XE, w);
    a.perm = team_ptr(a0.perm, w);
    a.R = team_ptr(a0.R, w);
    a.P = team_ptr(a0.P, w);
    a.psum = team_ptr(a0.psum, w);
    a.xlow = team_ptr(a0.xlow, w);
    a.psumH = team_ptr(a0.psumH, w);
    a.shiftv = team_ptr(a0.shiftv, w);
    a.xminv = team_ptr(a0.xminv, w);
    a.shring = team_ptr(a0.shring, w);
    a.parentpos = team_ptr(a0.parentpos, w);
    if (a0.hist) {
        a.Xhist += nu;
        a.Ahist += nu;
    }
    return a;
}

// K values per thread, entry kk of thread tid for child kk * GT + tid: in shared memory from `base` on (SH; every
// slot is read back only by the thread that wrote it, so no synchronisation), or in registers
template <class T, int K, int GT, bool SH>
struct ChildSlots {
    T* p;
    __device__ __forceinline__ explicit ChildSlots(unsigned char* base) : p((T*)base + threadIdx.x) {}
    __device__ __forceinline__ T& operator[](int kk) { return p[kk * GT]; }
};
template <class T, int K, int GT>
struct ChildSlots<T, K, GT, false> {
    T v[K];
    __device__ __forceinline__ explicit ChildSlots(unsigned char*) {}
    __device__ __forceinline__ T& operator[](int kk) { return v[kk]; }
};

// ---------------------------------------------------------------------------------------------
// the kernel
// ---------------------------------------------------------------------------------------------
// HESS: the Hessian branch of the reference with its quirks Q7 / Q8 (second instantiation, SV only).
// M: the model (pf_model.cuh).  SvLeverageModel runs the SV code with its shared exp(-x/2); any other model
// runs the generic path: the second double of XE is the propagation mean prop_mean(x, obs[t]) of the
// children, a payload is (parent value, -, -, own value) and the score terms are M::score_main of the pair.
// SMO: the fixed-lag smoother; false: the filter alone, whose outputs are bit-identical to the smoother's.
// TEAM: teams of a_in.G CTAs, one per problem (GridTeam below); false: one problem on a_in.G CTAs.
template <int GT, bool HESS, class M, bool SMO, bool TEAM>
__global__ void __launch_bounds__(GT, 1) sv_grid_kernel(const GridArgs a_in, const GridTeam tm) {
    GridArgs a_team;
    if constexpr (TEAM) a_team = team_args(a_in, tm);
    const GridArgs& a = TEAM ? a_team : a_in;   // this CTA's problem
    constexpr bool GEN = !std::is_same<M, SvLeverageModel>::value;
    // (static: a plain constexpr local changes the register allocation of the SV instantiations)
    static constexpr bool SVH = HESS && !GEN;   // the SV model's Hessian branch (the reference's, Q7 / Q8)
    static constexpr bool GENH = HESS && GEN;   // the generic Hessian branch (pf_model.cuh), predictive pairing
    static_assert(!GENH || M::kPairing == Pairing::Predictive, "the generic Hessian branch pairs the terms predictively");
    static_assert(SMO || !HESS, "the Hessian branch needs the smoother");
    constexpr int KPT = kCap / GT;          // entries per thread (strided assignment)
    constexpr int KCH = KPT | 1;            // longest chunk of the thread-contiguous passes (odd)
    constexpr int BPT = kNF / GT;           // histogram bins per thread
    constexpr int SPT = kNSB / GT;          // sub-bins per thread
    constexpr int NW = GT / 32;
    constexpr int CH = KPT >= 16 ? 8 : 4;   // independent loads in flight per thread in the gather loops
    constexpr int RB = KPT >= 16 ? 4 : 2;   // genealogy records in flight per thread
    constexpr int RS = HESS ? 2 : 1;        // 32-byte sectors per entry of R and P
    static_assert(SPT % 4 == 0 && BPT % 4 == 0, "vector loads of the counters");
    extern __shared__ __align__(16) unsigned char smem[];
    // phase B / C view
    double* s_xb = (double*)smem;                      // [kCap] values in sub-bin order
    int* s_jb = (int*)(smem + 65536);                  // [kCap] birth rows in sub-bin order
    int* s_ab = (int*)(smem + 98304);                  // [kCap] lagged ancestor rows in sub-bin order
    double* s_sh = (double*)(smem + 131072);           // [kCap] unnormalised weights, sorted order
    int* s_sub = (int*)(smem + 196608);                // [kNSB] sub-bin counters, then first positions
    int* s_ub = s_jb;                                  // [kCap] child range ends (phase C)
    // phase A1 -> A2: the children's values, parent / lagged ancestor rows and mailbox slots (xn, bp, kr below) in the
    // s_jb / s_ab / s_sh regions, dead from the end of phase C's ancestor fill to phase B; the SV Hessian branch's
    // s_deflist holds s_jb / s_ab then, so there they stay in registers; so they do in the generic filter, whose
    // phase A holds them there with less stack and spilling than through shared memory (ptxas -v)
    constexpr bool SLOTS_SMEM = !SVH && (SMO || !GEN);
    // phase A view (Hessian branch: list of deferred alpha terms = (child, parent row) pairs in the s_jb / s_ab region)
    int2* s_deflist = (int2*)(smem + 65536);         // [kCap]
    int* s_fhist = (int*)smem;                         // [kNF] histogram of this CTA's children
    unsigned short* s_tileof = (unsigned short*)(smem + 32768);   // [kNF] tile of a histogram bin

    __shared__ typename M::Const s_k;
    __shared__ StepScalars s_sc;
    __shared__ double s_tot[kMaxTiles], s_off[kMaxTiles + 1];
    __shared__ int s_tstart[kMaxTiles + 1], s_tbin[kMaxTiles + 1], s_tcnt[kMaxTiles], s_tbase[kMaxTiles];
    __shared__ double s_red[9 * 32];
    __shared__ double s_redH[HESS ? 20 * 32 : 1];   // Hessian branch: warp sums of the 20 hessian1 / hessian2 terms
    __shared__ int s_wi[32];
    __shared__ long long s_prof[kProf];
    __shared__ int s_ndef;   // Hessian branch: length of the list of deferred alpha terms
    __shared__ unsigned s_ties[2];   // resampling decisions near a tie (diag: near, soft) of this CTA

    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int c = TEAM ? (int)(blockIdx.x % (unsigned)a.G) : blockIdx.x, G = a.G, N = a.N, NOBS = a.NOBS, L = a.LAG, Wc = a.Wc, RP = a.RP;
    GridCtrl* ctrl = a.ctrl;
    const double dn = (double)N, inv_n = 1.0 / dn;
    const bool pow2 = (N & (N - 1)) == 0;
    const unsigned long long pol_stream = policy_evict_first();
    const unsigned long long pol_keep = (a.dbg & 64) ? policy_evict_normal() : policy_evict_last();
    const unsigned long long pol_dead = (a.dbg & 64) ? policy_evict_normal() : policy_evict_first();
    // (measured one by one, N = 2^20: the previous record table, the lagged payloads and the parents' (x, e)
    // / perm entries read as evict_first are worth 8 + 3 us per step; evict_last on the stores alone is not)
    const unsigned long long pol_rld = pol_dead, pol_pld = pol_dead, pol_xld = pol_dead, pol_rst = pol_keep;
    constexpr double kBinW = 2.0 * kZ / (double)kNF;    // width of a histogram bin in predicted sd
    unsigned epoch = 0;                 // arrives done so far
    unsigned cnt_key = 0;
    int my_max_bin = 0;
    long long pclk = 0;
    const bool prof = a.prof != nullptr;

// The arrive is bar.sync + red.release.gpu by one thread, the wait ld.acquire.gpu by one thread + bar.sync: release /
// acquire at gpu scope are cumulative over what bar.sync ordered before / after them, so no separate __threadfence is
// needed (measured: 99.5 -> 96.8 ms per evaluation)
// Abandoning: the reason goes to ctrl->status (first one wins), and bit 31 of the barrier counter is set, so that the
// load every CTA polls the barrier with also tells it to stop -- at its next wait, whichever barrier that is (nothing
// after the time loop needs the grid); a second load of the status word after every barrier costs an L2 round trip
#define GRID_FLAG(reason)                                                                        \
    do {                                                                                         \
        atomicCAS(&ctrl->status, 0, (int)((epoch + 1u) | ((unsigned)(reason) << 24)));           \
        atomicOr(&ctrl->bar, 0x80000000u);                                                       \
    } while (0)
#define GRID_POLL(tgt)                                                                \
    do {                                                                              \
        unsigned v__;                                                                 \
        do {                                                                          \
            v__ = ld_acquire_u32(&ctrl->bar);                                         \
        } while ((v__ & 0x7fffffffu) < (tgt) && !(v__ & 0x80000000u));                \
        s_sc.abort_now = (int)(v__ >> 31);                                            \
    } while (0)
#define GRID_ARRIVE()                                    \
    do {                                                 \
        __syncthreads();                                 \
        if (tid == 0) red_release_add(&ctrl->bar, 1u);   \
        ++epoch;                                         \
    } while (0)
#define GRID_WAIT()                                                                   \
    do {                                                                              \
        if (tid == 0) {                                                               \
            const unsigned tgt = epoch * (unsigned)G;                                 \
            GRID_POLL(tgt);                                                           \
        }                                                                             \
        __syncthreads();                                                              \
    } while (0)
#define PROF_MARK(slot)                              \
    do {                                             \
        if (prof && tid == 0) {                      \
            const long long now__ = clock64();       \
            s_prof[slot] += now__ - pclk;            \
            pclk = now__;                            \
        }                                            \
    } while (0)

    if (tid == 0) {
        M::init(s_k, a.params);
        s_sc.abort_now = 0;
        s_sc.tol_soft = 2.220446049250313e-16 * dn * (4.0 + 2.0 * sqrt(dn));
        s_sc.tol_near = 64.0 * 2.220446049250313e-16 * dn;
        s_ties[0] = s_ties[1] = 0;
        for (int i = 0; i < kProf; ++i) s_prof[i] = 0;
    }
    for (int i = tid; i < kMaxTiles; i += GT) s_tcnt[i] = 0;
    __syncthreads();

    // ------------------------------------------------------------------------------------------
    // generation 0 (:306-323, Q1): every particle = mu (M::initial_state), uniform weights, identity order
    // ------------------------------------------------------------------------------------------
    const int jb = min(N, c * Wc), je = min(N, jb + Wc), nc = je - jb;   // this CTA's children
    int pstart = jb, n = nc;                                             // this CTA's tile
    double toff;                                                          // cumulative weight in front of this thread's chunk
    {
        double mu, e0, m0;   // value, second double of XE, propagation mean
        if constexpr (GEN) {
            mu = M::initial_state(s_k);
            m0 = M::prop_mean(s_k, mu, a.obs[0]);
            e0 = m0;
        } else {
            mu = s_k.mu;
            e0 = exp(-0.5 * mu);
            m0 = s_k.mu + s_k.phi * (mu - s_k.mu);
            m0 += (s_k.sr * e0) * a.obs[0];
        }
        for (int q = tid; q < n; q += GT) {
            __stcg(&a.XE[pstart + q], make_double2(mu, e0));
            __stcg(&a.perm[pstart + q], pstart + q);
            s_sh[q] = 1.0;
            if constexpr (SMO) st_rec(&a.R[(size_t)(pstart + q) * RS], pol_keep, 0, 0, 0, 0, 0, 0, 0, 0);
            if constexpr (HESS) {
                st_rec(&a.R[(size_t)(pstart + q) * RS + 1], pol_keep, 0, 0, 0, 0, 0, 0, 0, 0);   // alpha = 0
                if constexpr (SVH) {
                    if (pstart + q < a.SQ) a.xlow[(size_t)(pstart + q) * NOBS] = mu;
                }
            }
            if (a.hist) {
                a.Xhist[pstart + q] = mu;
                a.Ahist[pstart + q] = pstart + q;
            }
        }
        const int Lc = ((n + GT - 1) / GT) | 1;
        toff = (double)min(tid * Lc, n);
        if (tid == 0) {
            const double dnk = (double)n;
            __stcg((double2*)&a.tinfo[c * 4], make_double2(dnk, dnk));
            __stcg((double2*)&a.tinfo[c * 4 + 2], make_double2(dnk * m0, dnk * (m0 * m0)));
            double* ps = a.psum + ((size_t)0 * G + c) * 8;
            ps[0] = dnk;
            ps[1] = dnk * mu;
            for (int i = 2; i < 8; ++i) ps[i] = 0.0;
            if (c == 0) {
                a.shiftv[0] = 0.0;
                a.xminv[0] = mu;
            }
        }
    }
    GRID_ARRIVE();
    GRID_WAIT();
    if (prof && tid == 0) pclk = clock64();

    for (int t = 1; t < NOBS; ++t) {
        const int par = t & 1;
        // --------------------------------------------------------------------------------------
        // phase C: totals of all tiles -> offsets; child ranges of this tile's parents (:694-715)
        // --------------------------------------------------------------------------------------
        const double ur = a.rvr[t];
        double mom1 = 0.0, mom2 = 0.0;   // warp 0: weighted moments of the propagation mean
        if (warp == 0) {
            constexpr int kPer = kMaxTiles / 32;
            double tv[kPer], m1v[kPer], m2v[kPer];
#pragma unroll
            for (int i = 0; i < kPer; ++i) {
                const int k = lane * kPer + i;
                tv[i] = m1v[i] = m2v[i] = 0.0;
                if (k < G) {
                    const double2 t0 = __ldcg((const double2*)&a.tinfo[k * 4]);
                    const double2 t1 = __ldcg((const double2*)&a.tinfo[k * 4 + 2]);
                    tv[i] = t0.x;
                    m1v[i] = t1.x;
                    m2v[i] = t1.y;
                }
            }
            double loc = 0.0, l1 = 0.0, l2 = 0.0;
#pragma unroll
            for (int i = 0; i < kPer; ++i) {
                loc = loc + tv[i];
                l1 = l1 + m1v[i];
                l2 = l2 + m2v[i];
            }
            const double incl = warp_incl_scan(loc, lane);
            double run = __shfl_up_sync(kFullMask, incl, 1);
            if (lane == 0) run = 0.0;
#pragma unroll
            for (int i = 0; i < kPer; ++i) {
                const int k = lane * kPer + i;
                if (k < G) {
                    s_off[k] = run;
                    s_tot[k] = tv[i];
                    run = run + tv[i];
                }
            }
            const double S = __shfl_sync(kFullMask, incl, 31);
            const double invS = 1.0 / S;
            __syncwarp();
            if (lane == 0) {
                s_sc.S = S;
                s_sc.invS = invS;
                s_sc.offk = s_off[c];
                if (!(S > 0.0) || !isfinite(S)) GRID_FLAG(2);
            }
            // child range end of the tiles in front of this one (running maximum, see below)
            {
                int carry = 0;
                const int k = c - 1 - lane;
                if (lane < 2 && k >= 0) {
                    double fr;
                    carry = count_le((s_off[k] + s_tot[k]) * invS, ur, N, dn, inv_n, pow2, fr);
                }
                carry = max(carry, __shfl_down_sync(kFullMask, carry, 1));
                if (lane == 0) s_sc.carry = carry;
            }
            mom1 = warp_sum(l1);
            mom2 = warp_sum(l2);
        }
        __syncthreads();
        PROF_MARK(16);   // C: totals -> offsets (warp 0)
        {
            const double invS = s_sc.invS, offk = s_sc.offk;
            const int Lc = ((n + GT - 1) / GT) | 1, q0 = tid * Lc;
            const double tol_soft = s_sc.tol_soft, tol_near = s_sc.tol_near;
            unsigned nsoft = 0, nnear = 0;
            int ubv[KCH];
            unsigned slow = 0;   // bit kk: the closed form missed for parent q0 + kk, exact search below
            double run = 0.0;
#pragma unroll
            for (int kk = 0; kk < KCH; ++kk) {
                const int q = q0 + kk;
                ubv[kk] = 0;
                if (kk < Lc && q < n) {
                    run = run + s_sh[q];
                    const double cN = (offk + (toff + run)) * invS;
                    int ub;
                    if (pstart + q == N - 1) {
                        ub = N;
                    } else {
                        double fr;
                        if (!count_le_fast(cN, ur, N, dn, inv_n, pow2, ub, fr)) {
                            slow |= 1u << kk;
                            s_ub[q] = ub;
                        }
                        if (fr < tol_soft) {
                            ++nsoft;
                            if (fr < tol_near * fmax(cN, inv_n)) ++nnear;
                        }
                    }
                    ubv[kk] = ub;
                }
            }
            if (nsoft) {
                atomicAdd(&s_ties[1], nsoft);
                if (nnear) atomicAdd(&s_ties[0], nnear);
            }
            if (slow) {
                // the exact search, kept out of the unrolled loop (its live registers would go to the stack): the
                // same running sum again, the result through this thread's own s_ub slots
                double rs = 0.0;
#pragma unroll 1
                for (int kk = 0; kk < Lc && q0 + kk < n; ++kk) {
                    const int q = q0 + kk;
                    rs = rs + s_sh[q];
                    if ((slow >> kk) & 1u) s_ub[q] = count_le_slow(s_ub[q], (offk + (toff + rs)) * invS, ur, N, dn, inv_n, pow2);
                }
#pragma unroll
                for (int kk = 0; kk < KCH; ++kk)
                    if ((slow >> kk) & 1u) ubv[kk] = s_ub[q0 + kk];
            }
            int rmax = 0;
#pragma unroll
            for (int kk = 0; kk < KCH; ++kk) {
                if (kk < Lc && q0 + kk < n) {
                    rmax = max(rmax, ubv[kk]);
                    ubv[kk] = rmax;
                }
            }
            // parallel scans are monotone only up to an ulp: a running maximum over all parents
            PROF_MARK(17);   // C: cumulative weights + child counts
            // (and over the tiles in front) keeps the child ranges disjoint
            int prev = block_excl_max_int<GT>(rmax, s_sc.carry, s_wi, lane, warp);
#pragma unroll
            for (int kk = 0; kk < KCH; ++kk) {
                const int q = q0 + kk;
                if (kk < Lc && q < n) {
                    prev = max(ubv[kk], prev);
                    s_ub[q] = prev;
                }
            }
        }
        __syncthreads();
        PROF_MARK(18);   // C: running maximum
        {
            // ancestor of every child: parent q owns the children [ub(q-1), ub(q)); consecutive
            // lanes hold consecutive parents, so the stores of a warp fall into a few lines
            const int carry = s_sc.carry;
#pragma unroll 1
            for (int kk = 0; kk < KPT; ++kk) {
                const int q = kk * GT + tid;
                if (kk * GT >= n) break;
                int lo = 0, hi = 0;
                if (q < n) {
                    hi = s_ub[q];
                    lo = q ? s_ub[q - 1] : carry;
                }
                const int P = pstart + q;
                const bool longr = hi - lo > 8;
                if (!longr)
                    for (int k = lo; k < hi; ++k) st_hint_b32(&a.H[k], pol_keep, P);
                unsigned m = __ballot_sync(kFullMask, longr);
                while (m) {
                    const int src = __ffs(m) - 1;
                    m &= m - 1;
                    const int l0 = __shfl_sync(kFullMask, lo, src), h0 = __shfl_sync(kFullMask, hi, src);
                    const int P0 = __shfl_sync(kFullMask, P, src);
                    for (int k = l0 + lane; k < h0; k += 32) st_hint_b32(&a.H[k], pol_keep, P0);
                }
            }
        }
        if (tid == 0) {
            // predicted mean / sd of the children: histogram range of phase A
            const double S = s_sc.S;
            const double mhat = mom1 / S;
            double var = mom2 / S - mhat * mhat;
            if (!(var > 0.0)) var = 0.0;
            if constexpr (GEN) {
                const double psd = M::prop_sd(s_k);
                var = var + psd * psd;
            } else {
                var = var + s_k.sd * s_k.sd;
            }
            const double shat = sqrt(var);
            s_sc.mhat = mhat;
            s_sc.shat = shat;
            s_sc.inv_shat = 1.0 / shat;
            if (!isfinite(mhat) || !(shat > 0.0) || !isfinite(shat)) GRID_FLAG(2);
        }
        PROF_MARK(0);   // C ranges+fill
        GRID_ARRIVE();   // ---- barrier 4: ancestors complete
        for (int b = tid; b < kNF; b += GT) s_fhist[b] = 0;
        PROF_MARK(1);   // zero hist
        if (a.u_flag && tid == 0) {
            // host-streamed u: row t has to have landed (the flag is written by the copy engine); at the first of
            // the four steps that share a 32-byte sector, all four (see the stash below)
            const int need = (((t % a.u_cs) & 3) == 0 || t == 1) ? min(t | 3, NOBS - 1) : t;
            while (ld_acquire_sys_s32(a.u_flag) <= need) {
            }
        }
        GRID_WAIT();
        PROF_MARK(2);   // wait 4
        if (s_sc.abort_now) break;

        // --------------------------------------------------------------------------------------
        // phase A1: parents of this CTA's children, propagation (:354-358), value histogram
        // --------------------------------------------------------------------------------------
        ChildSlots<double, KPT, GT, SLOTS_SMEM> xn(smem + 131072);   // value
        ChildSlots<int, KPT, GT, SLOTS_SMEM> bp(smem + 65536);       // birth row of the parent, then lagged ancestor row
        {
            int hp[KPT];   // sorted position of the parent
#pragma unroll
            for (int kk = 0; kk < KPT; ++kk) {
                const int i = kk * GT + tid;
                hp[kk] = 0;
                if (i < nc) hp[kk] = ld_hint_b32(&a.H[jb + i], pol_dead);
            }
            const double y1 = a.obs[t - 1];
            const double ylag = a.obs[t >= 2 ? t - 2 : 0];   // Q5: the score terms of step i use obs[i - LAG]; i = t + LAG - 2
            const double mhat = s_sc.mhat, inv_shat = s_sc.inv_shat;
            const double mu = sv_of(s_k).mu, phi = sv_of(s_k).phi, sr = sv_of(s_k).sr, sd = M::prop_sd(s_k);
            const double* Ut = a.U + (size_t)(t / a.u_cs) * a.u_cstride + (size_t)(t % a.u_cs) * a.u_tstride;
            long long ujs = a.u_jstride;
            if (a.u_flag) {
                // host-streamed u lies particle-major (rows of u_cs steps): a strided 8-byte read per particle and step
                // fetches a 64-byte DRAM burst for 8 bytes and costs the LSU one sector per lane (measured: 142 instead
                // of 94 us per step).  Every fourth step each thread reads the whole 32-byte sector of its particles once
                // and lays the four steps down time-major in a small stash (coalesced stores); all steps then read the
                // stash coalesced.  A thread reads back only what it wrote itself: no synchronisation.
                const int tin = t % a.u_cs;
                if ((tin & 3) == 0 || t == 1) {   // (the time loop starts at t = 1: that step fills the first sector)
                    const double* Ug = Ut - (tin & 3);
#pragma unroll
                    for (int kk = 0; kk < KPT; ++kk) {
                        const int i = kk * GT + tid;
                        if (i < nc) {
                            double v0, v1, v2, v3;
                            asm volatile("ld.global.nc.L1::no_allocate.L2::cache_hint.v4.f64 {%0,%1,%2,%3}, [%4], %5;"
                                         : "=d"(v0), "=d"(v1), "=d"(v2), "=d"(v3)
                                         : "l"(Ug + (size_t)(jb + i) * ujs), "l"(pol_stream));
                            double* sp = a.ustash + jb + i;
                            __stcg(sp, v0);
                            __stcg(sp + N, v1);
                            __stcg(sp + 2 * (size_t)N, v2);
                            __stcg(sp + 3 * (size_t)N, v3);
                        }
                    }
                }
                Ut = a.ustash + (size_t)(tin & 3) * N;
                ujs = 1;
            }
            PEntry* Pt = a.P + (size_t)(t % RP) * N * RS;
            bool bad = false, orphan = false;
#pragma unroll
            for (int k0 = 0; k0 < KPT; k0 += CH) {
                // all loads of CH children are in flight before the first one is used
                double2 xe[CH];
                double uu[CH];
#pragma unroll
                for (int u = 0; u < CH; ++u) {
                    const int i = (k0 + u) * GT + tid;
                    xe[u] = make_double2(0.0, 0.0);
                    uu[u] = 0.0;
                    if (i < nc) {
                        int p = hp[k0 + u];
                        if ((unsigned)p >= (unsigned)N) {
                            orphan = true;
                            p = 0;
                        }
                        {
                            const int4 xr = ld_hint_b128(&a.XE[p], pol_xld);
                            xe[u].x = __longlong_as_double(((long long)xr.y << 32) | (long long)(unsigned)xr.x);
                            xe[u].y = __longlong_as_double(((long long)xr.w << 32) | (long long)(unsigned)xr.z);
                        }
                        bp[k0 + u] = ld_hint_b32(&a.perm[p], pol_xld);
                        // (the stash is rewritten every four steps: coherent load, not the read-only path)
                        uu[u] = a.u_flag ? __ldcg(Ut + (size_t)(jb + i) * ujs) : ld_stream_hint_f64(Ut + (size_t)(jb + i) * ujs, pol_stream);
                        if (a.hist) a.parentpos[jb + i] = p;
                    }
                }
#pragma unroll
                for (int u = 0; u < CH; ++u) {
                    const int i = (k0 + u) * GT + tid;
                    xn[k0 + u] = 0.0;
                    if (i < nc) {
                        double x;
                        if constexpr (GEN) {
                            x = xe[u].y + sd * uu[u];                 // M::propagate, the mean stored with the parent
                        } else {
                            double mean = mu + phi * (xe[u].x - mu);     // :355
                            mean += (sr * xe[u].y) * y1;                  // :356
                            x = mean + sd * uu[u];                        // :357-358
                        }
                        if (!isfinite(x)) bad = true;
                        xn[k0 + u] = x;
                        atomicAdd(&s_fhist[fine_bin(x, mhat, inv_shat)], 1);
                        if constexpr (SMO) {
                            if constexpr (GEN) {
                                if (!(a.dbg & 2)) st_stream_f64x4(&Pt[(size_t)(jb + i) * RS], pol_stream, xe[u].x, 0.0, 0.0, x);
                            } else if (!(a.dbg & 2)) {
                                // residual of the transition parent -> child as the score terms use it (:452-453)
                                double sq = x - mu - phi * (xe[u].x - mu);
                                sq -= sr * xe[u].y * ylag;
                                st_stream_f64x4(&Pt[(size_t)(jb + i) * RS], pol_stream, xe[u].x, sq, xe[u].y * ylag, x);
                            }
                        }
                    }
                }
            }
            if (bad) GRID_FLAG(2);
            if (orphan) GRID_FLAG(4);
        }
        PROF_MARK(19);   // A1: gathers + propagation + histogram
        if (SVH && tid == 0) s_ndef = 0;
        __syncthreads();
        {
            int* gh = a.ghist + (size_t)par * kNF;
#pragma unroll
            for (int kk = 0; kk < BPT; ++kk) {
                const int b = kk * GT + tid;
                const int cnt = s_fhist[b];
                if (cnt) atomicAdd(&gh[b], cnt);
            }
        }
        PROF_MARK(3);   // A1 children+hist
        GRID_ARRIVE();   // ---- barrier 1: global histogram complete
        if (SMO && !(a.dbg & 1)) {
            // genealogy records (only feed outputs): child = (parent row, parent's ancestors 1..7)
            const REntry* Rp = a.R + (size_t)((t - 1) & 1) * N * RS;
            REntry* Rc = a.R + (size_t)(t & 1) * N * RS;
            // Hessian branch: alpha recursion (:361-390) in the same pass -- the parent's cumulative alpha is the
            // second sector of its record entry.  cumulative alpha of the child = its own term + its parent's.
            // Q7: the "current" state is particles[t - 1 + ancestor] read through the flat layout = sorted value
            // `sl` of time tq (table of the first SQ sorted values of every generation), or the unsorted new value
            // `sl` of this generation (complete only after barrier 1: deferred), or 0.  Q8: obs[t - LAG] wraps.
            // Generic Hessian branch: the child's term is pair_score of its own pair (parent value from the payload
            // this thread wrote in phase A1, y = obs[t - 1]); the record's second sector takes the child's cumulative
            // alpha, the payload's second sector the parent's (alpha_k of the pair (x_k, x_k+1) the payload holds).
            const double yi = a.obs[t], ylagH = SVH ? obs_wrap(a.obs, t - L, NOBS) : 0.0;
            const double ypair = GENH ? a.obs[pair_obs(M::kPairing, t - 1)] : 0.0;
            REntry* Pc = (REntry*)(a.P + (size_t)(t % RP) * N * RS);
#pragma unroll
            for (int k0 = 0; k0 < KPT; k0 += RB) {
                int r[RB][8];
                double2 pa0[HESS ? RB : 1], pa1[HESS ? RB : 1];
                double cur[SVH ? RB : 1];
#pragma unroll
                for (int u = 0; u < RB; ++u) {
                    const int i = (k0 + u) * GT + tid;
#pragma unroll
                    for (int z = 0; z < 8; ++z) r[u][z] = 0;
                    if constexpr (HESS) pa0[u] = pa1[u] = make_double2(0.0, 0.0);
                    if constexpr (SVH) cur[u] = 0.0;
                    if (i < nc) {
                        const REntry* src = &Rp[(size_t)((a.dbg & 8) ? jb + i : bp[k0 + u]) * RS];
                        ld_rec(src, pol_rld, r[u]);
                        if constexpr (HESS) ld_f64x4(src + 1, pol_rld, pa0[u].x, pa0[u].y, pa1[u].x, pa1[u].y);
                        if constexpr (SVH) {
                            const unsigned qq = (unsigned)(t - 1) + (unsigned)__ldcg(&a.H[jb + i]);
                            const unsigned sl = qq / (unsigned)NOBS, tq = qq - sl * (unsigned)NOBS;
                            if ((int)tq < t) cur[u] = ((int)sl < a.SQ) ? __ldcg(&a.xlow[(size_t)sl * NOBS + tq]) : 0.0;
                            else if ((int)tq == t) s_deflist[atomicAdd(&s_ndef, 1)] = make_int2(i, bp[k0 + u]);
                        }
                    }
                }
#pragma unroll
                for (int u = 0; u < RB; ++u) {
                    const int i = (k0 + u) * GT + tid;
                    if (i < nc) {
                        const int j = jb + i;
                        const int b = bp[k0 + u];
                        st_rec(&Rc[(size_t)j * RS], pol_rst, b, r[u][0], r[u][1], r[u][2], r[u][3], r[u][4], r[u][5], r[u][6]);
                        // row of the ancestor L-2 steps back (new record = (b, r[0..6]))
                        int anc = j;
                        if (L == 3) anc = b;
                        else if (L > 3) anc = pick8(r[u], L - 4);
                        bp[k0 + u] = anc;
                        if constexpr (SVH) {
                            double al[4];
                            sv_alpha_terms(s_k, xn[k0 + u], cur[u], yi, ylagH, al);
                            const double c0 = al[0] + pa0[u].x, c1 = al[1] + pa0[u].y;
                            const double c2 = al[2] + pa1[u].x, c3 = al[3] + pa1[u].y;
                            st_keep_f64x4(&Rc[(size_t)j * RS + 1], pol_rst, c0, c1, c2, c3);
                            st_stream_f64x4(&Pc[(size_t)j * RS + 1], pol_stream, c0, c1, c2, c3);
                        } else if constexpr (GENH) {
                            double g[4];
                            pair_score<M>(s_k, t == 1, __ldcg(&((const PEntry*)Pc)[(size_t)j * RS].c), xn[k0 + u],
                                          ypair, g);
                            st_keep_f64x4(&Rc[(size_t)j * RS + 1], pol_rst, pa0[u].x + g[0], pa0[u].y + g[1],
                                          pa1[u].x + g[2], pa1[u].y + g[3]);
                            st_stream_f64x4(&Pc[(size_t)j * RS + 1], pol_stream, pa0[u].x, pa0[u].y, pa1[u].x, pa1[u].y);
                        }
                    }
                }
            }
        }
        {
            // housekeeping for the next step
            const int zper = (kNF + G - 1) / G;
            int* ghn = a.ghist + (size_t)(par ^ 1) * kNF;
            for (int b = c * zper + tid; b < min(kNF, (c + 1) * zper); b += GT) __stcg(&ghn[b], 0);
            if (tid == 0) __stcg(&a.tilecnt[((par ^ 1) * kMaxTiles + c) * kCntStride], 0);
        }
        PROF_MARK(4);   // A1 records
        GRID_WAIT();
        PROF_MARK(5);   // wait 1
        if (s_sc.abort_now) break;
        // Hessian branch, Q7 reads that fall into this generation (ancestor position = 1 mod NOBS: one child in NOBS):
        // the unsorted new value `sl` (complete since barrier 1) if sl <= j, else 0.  The records pass listed these
        // children; one thread per entry redoes the term after the arrive of barrier 2 (outputs only: read by the
        // children of the next step and by the score terms LAG-2 steps later; LAG = 2: before the arrive)
        if constexpr (SVH) {
            if (L == 2) {
                __syncthreads();
                deferred_alpha_pass(a, s_k, s_deflist, min(s_ndef, kCap), t, jb, tid, GT, pol_rld, pol_rst, pol_stream);
            }
        }

        // --------------------------------------------------------------------------------------
        // phase A2: scan of the global histogram: tile boundaries on bin edges, tile of every bin;
        // entries ordered by tile in shared memory, copied to the mailboxes in runs
        // --------------------------------------------------------------------------------------
        {
            const int* gh = a.ghist + (size_t)par * kNF;
            int cnt[BPT];
#pragma unroll
            for (int i = 0; i < BPT; ++i) cnt[i] = 0;
#pragma unroll
            for (int i = 0; i < BPT; i += 4) {
                const int4 v = __ldcg((const int4*)(gh + BPT * tid + i));
                cnt[i] += v.x;
                cnt[i + 1] += v.y;
                cnt[i + 2] += v.z;
                cnt[i + 3] += v.w;
            }
            int prevcnt = 0;
            if (tid > 0) prevcnt += __ldcg(gh + BPT * tid - 1);
            int loc = 0, mxb = 0;
#pragma unroll
            for (int i = 0; i < BPT; ++i) {
                loc += cnt[i];
                mxb = max(mxb, cnt[i]);
            }
            my_max_bin = max(my_max_bin, mxb);
            int total;
            int start = block_excl_scan_int<GT>(loc, s_wi, total, lane, warp);
            int tprev = (tid == 0) ? -1 : min(G - 1, (start - prevcnt) / Wc);
            int tl = min(G - 1, start / Wc);
#pragma unroll
            for (int i = 0; i < BPT; ++i) {
                while (tl < G - 1 && start >= (tl + 1) * Wc) ++tl;
                s_tileof[BPT * tid + i] = (unsigned short)tl;
                for (int k = tprev + 1; k <= tl; ++k) {
                    s_tstart[k] = start;
                    s_tbin[k] = BPT * tid + i;
                }
                tprev = tl;
                if (cnt[i] > 0) {
                    if (start == 0) s_sc.binlo = BPT * tid + i;
                    if (start + cnt[i] == total) s_sc.binhi = BPT * tid + i;
                }
                start += cnt[i];
            }
            if (tid == GT - 1) {
                for (int k = tprev + 1; k <= G; ++k) {
                    s_tstart[k] = N;
                    s_tbin[k] = kNF;
                }
                if (total != N) GRID_FLAG(5);
            }
        }
        __syncthreads();
        PROF_MARK(20);   // A2: histogram scan + tile map
        ChildSlots<int, KPT, GT, SLOTS_SMEM> kr(smem + 98304);   // (tile << 16) | rank in the tile's run
        {
            const double mhat = s_sc.mhat, inv_shat = s_sc.inv_shat;
#pragma unroll
            for (int kk = 0; kk < KPT; ++kk) {
                const int i = kk * GT + tid;
                kr[kk] = 0;
                // (the children of a warp spread over ~25 tiles -- the innovation is wide against a tile -- so the plain
                // atomics hardly conflict: one atomic per (warp, tile) through __match_any_sync costs 13.8 -> 17.5 us for
                // this phase, through a ballot loop over the distinct tiles 2 -> 52 us for the counting alone)
                if (i < nc) {
                    const int tl = s_tileof[fine_bin(xn[kk], mhat, inv_shat)];
                    const int r = atomicAdd(&s_tcnt[tl], 1);
                    kr[kk] = (tl << 16) | r;
                }
            }
        }
        __syncthreads();
        PROF_MARK(21);   // A2: slot counting
        if (tid < G) {
            // slots of this CTA's run in every mailbox
            const int cnt = s_tcnt[tid];
            int base = s_tstart[tid];
            if (cnt) base += atomicAdd(&a.tilecnt[(par * kMaxTiles + tid) * kCntStride], cnt);
            s_tbase[tid] = base;
            s_tcnt[tid] = 0;
        }
        __syncthreads();
        PROF_MARK(22);   // A2: global reservation
        {
            MailEntry* mail = (MailEntry*)a.XE;
#pragma unroll
            for (int kk = 0; kk < KPT; ++kk) {
                const int i = kk * GT + tid;
                if (i < nc) {
                    const int pos = s_tbase[kr[kk] >> 16] + (kr[kk] & 0xffff);
                    const long long xb = __double_as_longlong(xn[kk]);
                    const int4 ent = make_int4((int)(xb & 0xffffffffll), (int)(xb >> 32), jb + i, SMO ? bp[kk] : 0);
                    if (pos >= 0 && pos < N) st_hint_b128(&mail[pos], pol_keep, ent);
                }
            }
        }
        pstart = s_tstart[c];
        n = s_tstart[c + 1] - pstart;
        if (n > kCap || n < 0) {
            if (tid == 0) GRID_FLAG(1);
            n = n < 0 ? 0 : kCap;
        }
        if (tid == 0) {
            // sub-bins of this tile: its histogram bins cover [lo, hi)
            const double mhat = s_sc.mhat, shat = s_sc.shat;
            const double lo = mhat + shat * ((double)s_tbin[c] * kBinW - kZ);
            const double hi = mhat + shat * ((double)s_tbin[c + 1] * kBinW - kZ);
            s_sc.lo = lo;
            s_sc.scale = (hi > lo) ? (double)kNSB / (hi - lo) : 0.0;
            // shift = largest log-weight over the occupied bins (any shift cancels, Q4)
            const double y = a.obs[t];
            const double xmin = mhat + shat * ((double)s_sc.binlo * kBinW - kZ);
            const double xmax = mhat + shat * ((double)(s_sc.binhi + 1) * kBinW - kZ);
            if constexpr (GEN) {
                s_sc.shift = M::logw_max(s_k, xmin, xmax, y);
            } else {
                double xs_ = (y != 0.0) ? 2.0 * log(fabs(y)) : xmin;
                xs_ = fmin(fmax(xs_, xmin), xmax);
                const double es_ = exp(-0.5 * xs_);
                s_sc.shift = (-0.91893853320467267 - 0.5 * xs_) - (0.5 * y * y) * (es_ * es_);
            }
            if (c == 0) a.shiftv[t] = s_sc.shift;
        }
        PROF_MARK(6);   // A2 scan+scatter
        GRID_ARRIVE();   // ---- barrier 2: mailboxes complete
        if constexpr (SVH) {
            if (L != 2) deferred_alpha_pass(a, s_k, s_deflist, min(s_ndef, kCap), t, jb, tid, GT, pol_rld, pol_rst, pol_stream);
            PROF_MARK(14);   // deferred alpha terms (Hessian branch)
        }
        for (int b = tid; b < kNSB; b += GT) s_sub[b] = 0;
        if (warp == 0 && nc > 0) {
            // the generation the fixed-lag terms of this step gather from, and the next step's slice of u -> L2
            if (t + 1 < NOBS && !a.u_flag) {
                const double* Un = a.U + (size_t)(t + 1) * N;
                prefetch_range(Un + jb, Un + je, lane, 32);
            }
            if (SMO && t >= L && (a.dbg & 8)) {   // (measured: the bulk prefetch of the lagged generation costs more than it saves)
                const PEntry* Pg = a.P + (size_t)((t - (L - 2)) % RP) * N;
                prefetch_range(Pg + jb, Pg + je, lane, 32);
            }
        }
        PROF_MARK(7);   // zero+prefetch
        GRID_WAIT();
        PROF_MARK(8);   // wait 2
        if (s_sc.abort_now) break;

        // --------------------------------------------------------------------------------------
        // phase B: sort this tile (:392-424 / :23-52), weights (:427-442), fixed-lag score terms
        // (:445-470), block scan
        // --------------------------------------------------------------------------------------
        double acc[3] = {0.0, 0.0, 0.0};   // sh * {x, m, m^2}
        {
            const MailEntry* mb = (const MailEntry*)a.XE + pstart;
            const double lo = s_sc.lo, scale = s_sc.scale;
            double bx[KPT];
            int bj[KPT], bae[KPT];
#pragma unroll
            for (int k0 = 0; k0 < KPT; k0 += CH) {
                int4 raw[CH];
#pragma unroll
                for (int u = 0; u < CH; ++u) {
                    const int e = (k0 + u) * GT + tid;
                    raw[u] = make_int4(0, 0, 0, 0);
                    if (e < n) raw[u] = ld_hint_b128(mb + e, pol_dead);
                }
#pragma unroll
                for (int u = 0; u < CH; ++u) {
                    const int e = (k0 + u) * GT + tid;
                    const double x = __longlong_as_double(((long long)raw[u].y << 32) | (long long)(unsigned)raw[u].x);
                    bx[k0 + u] = x;
                    bj[k0 + u] = raw[u].z;
                    bae[k0 + u] = raw[u].w & 0x1fffff;
                    if (e < n) {
                        const int er = atomicAdd(&s_sub[sub_bin(x, lo, scale)], 1);
                        bae[k0 + u] |= min(er, 2047) << 21;
                    }
                }
            }
            __syncthreads();
            PROF_MARK(23);   // B: mailbox load + sub-bin count
            {
                // exclusive scan of the sub-bin counters in place (SPT consecutive bins per thread)
                int cnt[SPT];
#pragma unroll
                for (int i = 0; i < SPT; i += 4) {
                    const int4 v = *(const int4*)(s_sub + SPT * tid + i);
                    cnt[i] = v.x;
                    cnt[i + 1] = v.y;
                    cnt[i + 2] = v.z;
                    cnt[i + 3] = v.w;
                }
                int loc = 0, mxb = 0;
#pragma unroll
                for (int i = 0; i < SPT; ++i) {
                    loc += cnt[i];
                    mxb = max(mxb, cnt[i]);
                }
                if (mxb > kMaxSub) GRID_FLAG(3);
                int total;
                int start = block_excl_scan_int<GT>(loc, s_wi, total, lane, warp);
#pragma unroll
                for (int i = 0; i < SPT; ++i) {
                    const int cn = cnt[i];
                    cnt[i] = start;
                    start += cn;
                }
#pragma unroll
                for (int i = 0; i < SPT; i += 4)
                    *(int4*)(s_sub + SPT * tid + i) = make_int4(cnt[i], cnt[i + 1], cnt[i + 2], cnt[i + 3]);
            }
            __syncthreads();
            PROF_MARK(24);   // B: sub-bin scan
#pragma unroll
            for (int kk = 0; kk < KPT; ++kk) {
                const int e = kk * GT + tid;
                if (e < n) {
                    const int pos = min(s_sub[sub_bin(bx[kk], lo, scale)] + (int)((unsigned)bae[kk] >> 21), kCap - 1);
                    s_xb[pos] = bx[kk];
                    s_jb[pos] = bj[kk];
                    if constexpr (SMO) s_ab[pos] = bae[kk] & 0x1fffff;
                }
            }
            __syncthreads();
        }
        PROF_MARK(9);   // B bin sort
        {
            // sub-bin order -> exact order (by value, then by birth row: :32-35 never returns 0), in place
            const double lo = s_sc.lo, scale = s_sc.scale;
            double bx[KPT];
            int bj[KPT], ba[KPT], np[KPT];
#pragma unroll
            for (int kk = 0; kk < KPT; ++kk) {
                const int q = kk * GT + tid;
                bx[kk] = 0.0;
                bj[kk] = ba[kk] = 0;
                np[kk] = q;
                if (q < n) {
                    const double x = s_xb[q];
                    const int j = s_jb[q];
                    bx[kk] = x;
                    bj[kk] = j;
                    if constexpr (SMO) ba[kk] = s_ab[q];
                    const int kb = sub_bin(x, lo, scale);
                    const int b0 = s_sub[kb];
                    const int b1 = (kb + 1 < kNSB) ? s_sub[kb + 1] : n;
                    if (b1 - b0 > 1 && b1 - b0 <= kMaxSub) {
                        int rank = 0;
                        for (int m = b0; m < b1; ++m) {
                            const double xm = s_xb[m];
                            if (xm < x) ++rank;
                            else if (xm == x && m != q) {
                                ++cnt_key;
                                if (s_jb[m] < j) ++rank;
                            }
                        }
                        np[kk] = b0 + rank;
                    }
                }
            }
            __syncthreads();
            PROF_MARK(25);   // B: exact ranks
#pragma unroll
            for (int kk = 0; kk < KPT; ++kk) {
                const int q = kk * GT + tid;
                if (q < n && np[kk] != q) {
                    s_xb[np[kk]] = bx[kk];
                    s_jb[np[kk]] = bj[kk];
                    if constexpr (SMO) s_ab[np[kk]] = ba[kk];
                }
            }
            __syncthreads();
            PROF_MARK(26);   // B: reorder
        }
        {
            // weights (:427-437): lw = -0.9189 - x/2 - y^2 exp(-x) / 2 (M::logw), sh = exp(lw - shift);
            // fixed-lag score terms (:445-470): ancestor pair (time t-L+1, t-L+2) from one half sector
            const double y = a.obs[t], hy2 = 0.5 * y * y, shift = s_sc.shift;
            const double mu = sv_of(s_k).mu, phi = sv_of(s_k).phi, sr = sv_of(s_k).sr;
            bool bad = false;
#pragma unroll
            for (int kk = 0; kk < KPT; ++kk) {
                const int q = kk * GT + tid;
                if (q < n) {
                    const double x = s_xb[q];
                    const int j = s_jb[q];
                    // e: the second double of XE (SV exp(-x/2), else the children's propagation mean)
                    const double e = GEN ? M::prop_mean(s_k, x, y) : exp(-0.5 * x);
                    const double lw = GEN ? M::logw(s_k, x, y) : (-0.91893853320467267 - 0.5 * x) - hy2 * (e * e);
                    double sh = exp(lw - shift);
                    if (!isfinite(sh)) {
                        bad = true;
                        sh = 0.0;
                    }
                    {
                        const long long xb = __double_as_longlong(x), eb = __double_as_longlong(e);
                        st_hint_b128(&a.XE[pstart + q], pol_keep,
                                     make_int4((int)(xb & 0xffffffffll), (int)(xb >> 32), (int)(eb & 0xffffffffll), (int)(eb >> 32)));
                    }
                    st_hint_b32(&a.perm[pstart + q], pol_keep, j);
                    if constexpr (SVH) {
                        if (pstart + q < a.SQ) a.xlow[(size_t)(pstart + q) * NOBS + t] = x;
                    }
                    s_sh[q] = sh;
                    if (pstart + q == 0) a.xminv[t] = x;   // Q10/Q11: traj[t] = X_t[0]
                    if (a.hist) {
                        a.Xhist[(size_t)t * N + pstart + q] = x;
                        a.Ahist[(size_t)t * N + pstart + q] = __ldcg(&a.parentpos[j]);
                    }
                    acc[0] = fma(sh, x, acc[0]);
                    double m = GEN ? e : mu + phi * (x - mu);
                    if (!GEN) m += (sr * e) * y;
                    const double shm = sh * m;
                    acc[1] += shm;
                    acc[2] = fma(shm, m, acc[2]);
                }
            }
            if (bad) GRID_FLAG(2);
        }
        __syncthreads();
        PROF_MARK(10);   // B rank+weights+score
        {
            // cumulative weights: thread = Lc consecutive sorted particles, sequential running sum;
            // one block-wide pass gives the offsets of the chunks and the eight weighted sums
            const int Lc = ((n + GT - 1) / GT) | 1, q0 = tid * Lc;
            double run = 0.0;
#pragma unroll
            for (int kk = 0; kk < KCH; ++kk) {
                const int q = q0 + kk;
                if (kk < Lc && q < n) run = run + s_sh[q];
            }
            const double incl = warp_incl_scan(run, lane);
#pragma unroll
            for (int i = 0; i < 3; ++i) acc[i] = warp_sum(acc[i]);
            if (lane == 31) s_red[warp] = incl;
            if (lane == 0) {
#pragma unroll
                for (int i = 0; i < 3; ++i) s_red[32 * (1 + i) + warp] = acc[i];
            }
            __syncthreads();
            const double wt = (lane < NW) ? s_red[lane] : 0.0;
            const double wincl = warp_incl_scan(wt, lane);
            double wex = __shfl_up_sync(kFullMask, wincl, 1);
            if (lane == 0) wex = 0.0;
            const double woff = __shfl_sync(kFullMask, wex, warp);
            double ex = __shfl_up_sync(kFullMask, incl, 1);
            if (lane == 0) ex = 0.0;
            toff = woff + ex;
            double* ps = a.psum + ((size_t)t * G + c) * 8;
            if ((n > 0 && tid == (n - 1) / Lc) || (n == 0 && tid == 0)) {
                const double tot = (n > 0) ? toff + run : 0.0;   // cumulative weight of the tile's last particle
                __stcg(&a.tinfo[c * 4], tot);
                ps[0] = tot;
            }
            if (warp == 0) {
                double v[3];
#pragma unroll
                for (int i = 0; i < 3; ++i) v[i] = warp_sum((lane < NW) ? s_red[32 * (1 + i) + lane] : 0.0);
                if (lane == 0) {
                    __stcg(&a.tinfo[c * 4 + 1], (double)n);
                    __stcg((double2*)&a.tinfo[c * 4 + 2], make_double2(v[1], v[2]));
                    ps[1] = v[0];
                    ps[7] = 0.0;
                    // later steps: the score terms below write ps[2..6]
                    if (!SMO || t < pair_first_step(M::kPairing, L) || (a.dbg & 4)) {
#pragma unroll
                        for (int i = 2; i < 7; ++i) ps[i] = 0.0;
                    }
                }
            }
            if (SMO && t >= NOBS - L) {
#pragma unroll
                for (int kk = 0; kk < KPT; ++kk) {
                    const int q = kk * GT + tid;
                    if (q < n) a.shring[(size_t)(t % L) * N + pstart + q] = s_sh[q];
                }
            }
        }
        PROF_MARK(11);   // B scan+publish
        GRID_ARRIVE();   // ---- barrier 3: tile totals published
        if (SMO && t >= pair_first_step(M::kPairing, L) && !(a.dbg & 4)) {
            // fixed-lag score terms (:445-470): weight x monomials of the payload of the ancestor
            // LAG-2 generations back (one random sector each), fixed summation order
            const PEntry* Pg = a.P + (size_t)((t - (L - 2)) % RP) * N * RS;
            double sc[5] = {0.0, 0.0, 0.0, 0.0, 0.0};
            // Hessian branch (:472-534): hessian1 is a polynomial in (curr - mu, sq, ey) with constant coefficients, so
            // four more weighted monomials (ey, curr^2, curr ey, ey^2 -> hacc[0..3]) next to the five of the gradient
            // give its ten entries afterwards (grid_hess_finish_kernel); hessian2 needs the cumulative alpha of the
            // same ancestor (the second sector of its payload entry) and is accumulated entry by entry in a second
            // pass (hacc[10..19]; the payloads come from L2 there).  Weights are the unnormalised ones (divided by S
            // afterwards).  The isfinite guards of :521-534 are kept for hessian2; a non-finite particle value
            // abandons the evaluation (phase A1), so hessian1 needs none.
            double hm[SVH ? 4 : 1];
            if constexpr (SVH) {
#pragma unroll
                for (int i = 0; i < 4; ++i) hm[i] = 0.0;
            }
            if constexpr (GEN) {
                // generic path: sc[0] = sum sh curr (smoother), sc[1 + k] = sum sh g[k] of pair_score on the pair
                // (curr, next) = (parent value, own value) of the ancestor = (x_tt, x_tt+1), tt = t - LAG + 1;
                // y = obs[t - LAG] (Q5), obs[tt + 1], or obs[tt] (predictive)
                const double yl = a.obs[pair_obs(M::kPairing, t - L + 1)];
#pragma unroll
                for (int k0 = 0; k0 < KPT; k0 += 4) {
                    double pc[4], px[4];
#pragma unroll
                    for (int u = 0; u < 4; ++u) {
                        const int q = (k0 + u) * GT + tid;
                        pc[u] = px[u] = 0.0;
                        if (q < n) {
                            const PEntry* pp = &Pg[(size_t)min(max(s_ab[q], 0), N - 1) * RS];
                            double d1, d2;
                            asm volatile("ld.global.cg.L2::cache_hint.v4.f64 {%0,%1,%2,%3}, [%4], %5;"
                                         : "=d"(pc[u]), "=d"(d1), "=d"(d2), "=d"(px[u])
                                         : "l"(pp), "l"(HESS ? pol_keep : pol_pld));
                        }
                    }
#pragma unroll
                    for (int u = 0; u < 4; ++u) {
                        const int q = (k0 + u) * GT + tid;
                        if (q < n) {
                            const double wd = s_sh[q];
                            sc[0] = fma(wd, pc[u], sc[0]);
                            if constexpr (!M::kScoreIsZero) {
                                double g[4];
                                pair_score<M>(s_k, t == L - 1, pc[u], px[u], yl, g);
#pragma unroll
                                for (int i = 0; i < 4; ++i) sc[1 + i] = fma(wd, g[i], sc[1 + i]);
                            }
                        }
                    }
                }
            } else {
#pragma unroll
                for (int k0 = 0; k0 < KPT; k0 += 4) {
                    double pc[4], psq[4], pey[4];
#pragma unroll
                    for (int u = 0; u < 4; ++u) {
                        const int q = (k0 + u) * GT + tid;
                        pc[u] = psq[u] = pey[u] = 0.0;
                        if (q < n) {
                            const PEntry* pp = &Pg[(size_t)min(max(s_ab[q], 0), N - 1) * RS];
                            double d3;
                            asm volatile("ld.global.cg.L2::cache_hint.v4.f64 {%0,%1,%2,%3}, [%4], %5;"
                                         : "=d"(pc[u]), "=d"(psq[u]), "=d"(pey[u]), "=d"(d3)
                                         : "l"(pp), "l"(HESS ? pol_keep : pol_pld));
                        }
                    }
#pragma unroll
                    for (int u = 0; u < 4; ++u) {
                        const int q = (k0 + u) * GT + tid;
                        if (q < n) {
                            const double wd = s_sh[q];
                            const double ws = wd * psq[u];
                            sc[0] = fma(wd, pc[u], sc[0]);
                            sc[1] += ws;
                            sc[2] = fma(ws, pc[u], sc[2]);
                            sc[3] = fma(ws, psq[u], sc[3]);
                            sc[4] = fma(ws, pey[u], sc[4]);
                            if constexpr (HESS) {
                                const double we = wd * pey[u], wc = wd * pc[u];
                                hm[0] += we;
                                hm[1] = fma(wc, pc[u], hm[1]);
                                hm[2] = fma(wc, pey[u], hm[2]);
                                hm[3] = fma(we, pey[u], hm[3]);
                            }
                        }
                    }
                }
            }
#pragma unroll
            for (int i = 0; i < 5; ++i) sc[i] = warp_sum(sc[i]);
            __syncthreads();
            if constexpr (SVH) {
#pragma unroll
                for (int i = 0; i < 4; ++i) hm[i] = warp_sum(hm[i]);
            }
            if (lane == 0) {
#pragma unroll
                for (int i = 0; i < 5; ++i) s_red[32 * i + warp] = sc[i];
                if constexpr (SVH) {
#pragma unroll
                    for (int i = 0; i < 4; ++i) s_redH[32 * i + warp] = hm[i];
                }
            }
            if constexpr (SVH) {
                constexpr int SB = 1;   // 64-byte entries in flight per thread
                double h2[10];
#pragma unroll
                for (int i = 0; i < 10; ++i) h2[i] = 0.0;
#pragma unroll
                for (int k0 = 0; k0 < KPT; k0 += SB) {
                    double pc[SB], psq[SB], pey[SB];
                    double2 al0[SB], al1[SB];
#pragma unroll
                    for (int u = 0; u < SB; ++u) {
                        const int q = (k0 + u) * GT + tid;
                        pc[u] = psq[u] = pey[u] = 0.0;
                        al0[u] = al1[u] = make_double2(0.0, 0.0);
                        if (q < n) {
                            const PEntry* pp = &Pg[(size_t)min(max(s_ab[q], 0), N - 1) * RS];
                            double d3;
                            asm volatile("ld.global.cg.L2::cache_hint.v4.f64 {%0,%1,%2,%3}, [%4], %5;"
                                         : "=d"(pc[u]), "=d"(psq[u]), "=d"(pey[u]), "=d"(d3)
                                         : "l"(pp), "l"(pol_pld));
                            asm volatile("ld.global.cg.L2::cache_hint.v4.f64 {%0,%1,%2,%3}, [%4], %5;"
                                         : "=d"(al0[u].x), "=d"(al0[u].y), "=d"(al1[u].x), "=d"(al1[u].y)
                                         : "l"(pp + 1), "l"(pol_pld));
                        }
                    }
#pragma unroll
                    for (int u = 0; u < SB; ++u) {
                        const int q = (k0 + u) * GT + tid;
                        if (q < n) {
                            const double wd = s_sh[q];
                            const double sq = psq[u], ey = pey[u];
                            // g of :454-465 from (curr, sq, ey)
                            const double g0 = s_k.q * sq * s_k.one_m_phi;
                            const double g1 = s_k.q * sq * (pc[u] - s_k.mu) * s_k.one_m_phi2;
                            double g2 = sq;
                            g2 += s_k.sr * ey;
                            g2 *= s_k.q * sq;
                            g2 -= 1.0;
                            double g3 = s_k.rho - s_k.q * s_k.rho * sq * sq;
                            g3 += s_k.inv_sv * sq * ey;
                            const double a0 = al0[u].x, a1 = al0[u].y, a2 = al1[u].x, a3 = al1[u].y;
                            double h;   // :505-519 (the '*' typos of :513,514,517 kept)
#define HESS2_ADD(slot, expr)                           \
    h = (expr);                                         \
    if (isfinite(h)) h2[slot - 10] += h * wd;
                            HESS2_ADD(10, g0 * g0 + 2.0 * a0 * g0)
                            HESS2_ADD(11, g0 * g1 + a0 * g1 + a1 * g0)
                            HESS2_ADD(12, g0 * g2 + a0 * g2 + a2 * g0)
                            HESS2_ADD(13, g0 * g3 + a0 * g3 + a3 * g0)
                            HESS2_ADD(14, g1 * g1 + 2.0 * a1 * g1)
                            HESS2_ADD(15, g1 * g2 + a1 * g2 * a2 * g1)
                            HESS2_ADD(16, g1 * g3 + a1 * g3 * a3 * g1)
                            HESS2_ADD(17, g2 * g2 + 2.0 * a2 * g2)
                            HESS2_ADD(18, g2 * g3 + a2 * g3 * a3 * g2)
                            HESS2_ADD(19, g3 * g3 + 2.0 * a3 * g3)
#undef HESS2_ADD
                        }
                    }
                }
#pragma unroll
                for (int i = 0; i < 10; ++i) h2[i] = warp_sum(h2[i]);
                if (lane == 0) {
#pragma unroll
                    for (int i = 0; i < 10; ++i) s_redH[32 * (10 + i) + warp] = h2[i];
                }
            } else if constexpr (GENH) {
                // generic Hessian branch: a second pass over the same payloads (from L2) with their second sector,
                // alpha_k; the ten entries of hessian1 and of hessian2 under the unnormalised weights (divided by S
                // afterwards)
                double h1[10], h2[10];
#pragma unroll
                for (int i = 0; i < 10; ++i) h1[i] = h2[i] = 0.0;
                const double yl = a.obs[pair_obs(M::kPairing, t - L + 1)];
#pragma unroll 1
                for (int kk = 0; kk < KPT; ++kk) {
                    const int q = kk * GT + tid;
                    if (q < n) {
                        const PEntry* pp = &Pg[(size_t)min(max(s_ab[q], 0), N - 1) * RS];
                        double pc, d1, d2, px, al[4];
                        ld_f64x4(pp, pol_pld, pc, d1, d2, px);
                        ld_f64x4(pp + 1, pol_pld, al[0], al[1], al[2], al[3]);
                        double g[4], hh[10];
                        pair_score<M>(s_k, t == L - 1, pc, px, yl, g);
                        pair_hess<M>(s_k, t == L - 1, pc, px, yl, hh);
                        louis_add(hh, g, al, s_sh[q], h1, h2);
                    }
                }
#pragma unroll
                for (int i = 0; i < 10; ++i) {
                    h1[i] = warp_sum(h1[i]);
                    h2[i] = warp_sum(h2[i]);
                }
                if (lane == 0) {
#pragma unroll
                    for (int i = 0; i < 10; ++i) {
                        s_redH[32 * i + warp] = h1[i];
                        s_redH[32 * (10 + i) + warp] = h2[i];
                    }
                }
            }
            __syncthreads();
            if constexpr (HESS) {
                for (int k = warp; k < 20; k += NW) {   // a warp sums component k over the warps (fixed order)
                    const double v = (GEN || k < 4 || k >= 10) ? warp_sum((lane < NW) ? s_redH[32 * k + lane] : 0.0) : 0.0;
                    if (lane == 0) a.psumH[((size_t)t * G + c) * 20 + k] = v;
                }
            }
            if (warp == 0) {
                double* ps = a.psum + ((size_t)t * G + c) * 8;
#pragma unroll
                for (int i = 0; i < 5; ++i) {
                    const double v = warp_sum((lane < NW) ? s_red[32 * i + lane] : 0.0);
                    if (lane == 0) ps[2 + i] = v;
                }
            }
        }
        PROF_MARK(13);   // score terms
        GRID_WAIT();
        PROF_MARK(12);   // wait 3
        if (s_sc.abort_now) break;
    }

    // diagnostics (every exit from the time loop follows a __syncthreads: s_ties is complete)
    if (tid == 0) {
        if (s_ties[0]) atomicAdd(&ctrl->near_ties, (unsigned long long)s_ties[0]);
        if (s_ties[1]) atomicAdd(&ctrl->soft_ties, (unsigned long long)s_ties[1]);
    }
    cnt_key = __reduce_add_sync(kFullMask, cnt_key);
    my_max_bin = __reduce_max_sync(kFullMask, my_max_bin);
    if (lane == 0) {
        if (cnt_key) atomicAdd(&ctrl->key_ties, (unsigned long long)(cnt_key / 2));
        atomicMax(&ctrl->max_bin, my_max_bin);
    }
    if (prof && tid == 0)
        for (int i = 0; i < kProf; ++i) a.prof[(size_t)c * kProf + i] += s_prof[i];
#undef GRID_FLAG
#undef GRID_POLL
#undef GRID_ARRIVE
#undef GRID_WAIT
#undef PROF_MARK
}

// ---------------------------------------------------------------------------------------------
// after the persistent kernel: O(T G) reductions, the tail (:540-562, Q6), output assembly
// ---------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) grid_reduce_kernel(const double* __restrict__ psum, int G,
                                                          double* __restrict__ sums) {
    const int t = blockIdx.x, k = threadIdx.x >> 5, lane = threadIdx.x & 31;   // 8 warps = 8 components
    double s = 0.0;
    for (int c = lane; c < G; c += 32) s = s + psum[((size_t)t * G + c) * 8 + k];
    s = warp_sum(s);
    if (lane == 0) sums[(size_t)t * 8 + k] = s;
}

// part[irel][block][0] = sum_p W_T[p] hist_idx[p];  [1..4] = sum_p W_i[p] g(hist_idx, hist_idx-1)
// with i = NOBS - L + irel, idx = L - 1 - irel; hist_k[p] = value of the ancestor k steps back of
// the particle at sorted position p of the final generation.  Exact pairing (pf_model.cuh, Pairing::Exact):
// irel = 0 is 0 (the main loop has that slot), the pair is weighted by W_T and takes y = obs[i + 1]; predictive pairing
// (Pairing::Predictive): y = obs[i], and irel = L - 1 (idx = 0, i = T) adds M::score_last of the final particle.
// HESS: partH[irel][block][0..19] = the hessian1 / hessian2 terms of :564-626 (alpha of the ancestor LAG-2 steps
// back of the final particle, weights W_i, obs[i - LAG] with wrap-around, Q8); for a generic model the upper triangles
// of hessian1 / hessian2 of the same pairs as the gradient (M::hess_main, and M::hess_last with the final particle's own
// alpha for irel = L - 1).  M: the model (g = M::score_tail).  n_obs >= 2 LAG, so the pairs start at x_LAG+1 here: the
// pair (x_0, x_1) (pair_score) is the persistent kernel's.
template <bool HESS, class M>
__global__ void __launch_bounds__(256) grid_tail_kernel(GridArgs a, const double* __restrict__ sums,
                                                        double* __restrict__ part, double* __restrict__ partH,
                                                        int nblk) {
    __shared__ double red[(HESS ? 20 : 5) * 32];
    const int tid = threadIdx.x;
    const int L = a.LAG, N = a.N, T = a.NOBS - 1, RP = a.RP;
    const int irel = blockIdx.y, i = a.NOBS - L + irel, idx = L - 1 - irel;
    typename M::Const k;
    M::init(k, a.params);
    constexpr bool REF = M::kPairing == Pairing::Reference;
    const double y1 = REF ? obs_wrap(a.obs, pair_obs(M::kPairing, i), a.NOBS)
                          : a.obs[M::kPairing == Pairing::Predictive ? i : min(i + 1, T)];
    const double ST = sums[(size_t)T * 8], Si = sums[(size_t)i * 8];
    const double* shT = a.shring + (size_t)(T % L) * N;
    const double* shi = a.shring + (size_t)(i % L) * N;
    const int RS = a.RS;
    const REntry* Rt = a.R + (size_t)(T & 1) * N * RS;
    double acc[5] = {0.0, 0.0, 0.0, 0.0, 0.0};
    double hacc[HESS ? 20 : 1];
    if constexpr (HESS) {
#pragma unroll
        for (int q = 0; q < 20; ++q) hacc[q] = 0.0;
    }
    const double ylagH = obs_wrap(a.obs, i - L, a.NOBS);
    const bool live = a.ctrl->status == 0 && (REF || irel >= 1);   // an abandoned evaluation leaves stale rows behind
    for (int p = blockIdx.x * 256 + tid; live && p < N; p += nblk * 256) {
        const int b = min(max(a.perm[p], 0), N - 1);
        const double wT = shT[p] / ST;
        double curr;
        if (idx == 0) {
            curr = a.XE[p].x;
            acc[0] += wT * curr;
            if constexpr (M::kPairing == Pairing::Predictive) {
                double g[4];
                M::score_last(k, curr, y1, g);
#pragma unroll
                for (int q = 0; q < 4; ++q) acc[1 + q] += g[q] * wT;
                if constexpr (HESS) {
                    double hh[10];
                    M::hess_last(k, curr, y1, hh);
                    louis_add(hh, g, (const double*)&Rt[(size_t)b * RS + 1], wT, hacc, hacc + 10);
                }
            }
        } else {
            // entry of the ancestor idx-1 steps back holds (next = its value, curr = its parent's value)
            const int m = idx - 1;
            const int row = (m == 0) ? b : min(max(Rt[(size_t)b * RS].a[m - 1], 0), N - 1);
            const PEntry pe = a.P[((size_t)((T - m) % RP) * N + row) * RS];
            curr = pe.c;
            const double pe_n = pe.x;
            acc[0] += wT * curr;
            const double wi = REF ? shi[p] / Si : wT;
            double sq, g[4], ec;
            if constexpr (std::is_same<M, SvLeverageModel>::value) {
                ec = exp(-0.5 * curr);
                sv_score_tail_e(k, curr, ec, pe_n, y1, sq, g);   // the tail uses obs[i - 1] (Q6)
            } else {
                M::score_tail(k, curr, pe_n, y1, g);
            }
#pragma unroll
            for (int q = 0; q < 4; ++q) acc[1 + q] += g[q] * wi;
            if constexpr (HESS && !REF) {
                double hh[10];
                M::hess_main(k, curr, pe_n, y1, hh);
                louis_add(hh, g, (const double*)&a.P[((size_t)((T - m) % RP) * N + row) * RS + 1], wT, hacc, hacc + 10);
            } else if constexpr (HESS) {
                const int m2 = L - 2;
                const int row2 = (m2 == 0) ? b : min(max(Rt[(size_t)b * RS].a[m2 - 1], 0), N - 1);
                const double* a4 = (const double*)&a.P[((size_t)((T - m2) % RP) * N + row2) * RS + 1];
                const double al[4] = {a4[0], a4[1], a4[2], a4[3]};
                sv_hessian_terms_e(k, curr, ec, exp(-curr), sq, ylagH, g, al, wi, hacc);
            }
        }
    }
    block_sum<5>(acc, red);
    if (tid < 5) part[((size_t)irel * nblk + blockIdx.x) * 8 + tid] = acc[tid];
    if constexpr (HESS) {
        __syncthreads();
        block_sum<20>(hacc, red);
        if (tid < 20) partH[((size_t)irel * nblk + blockIdx.x) * 20 + tid] = hacc[tid];
    }
}

// Hessian branch: sumsH[t][k] = sum over the tiles of psumH[t][.][k] (t >= first, the first step with fixed-lag terms;
// 0 before)
__global__ void __launch_bounds__(640) grid_reduceH_kernel(const double* __restrict__ psumH, int G, int first,
                                                           double* __restrict__ sumsH) {
    const int t = blockIdx.x, k = threadIdx.x >> 5, lane = threadIdx.x & 31;   // 20 warps = 20 components
    double s = 0.0;
    if (t >= first)
        for (int c = lane; c < G; c += 32) s = s + psumH[((size_t)t * G + c) * 20 + k];
    s = warp_sum(s);
    if (lane == 0) sumsH[(size_t)t * 20 + k] = s;
}

// hessian1 / hessian2 (:521-534, :613-626): main-loop terms divided by the weight sum of their step + tail terms,
// upper triangles expanded into the symmetric 4 x 4 outputs
__global__ void __launch_bounds__(32) grid_hess_finish_kernel(const GridCtrl* __restrict__ ctrl,
                                                              const double* __restrict__ sums,
                                                              const double* __restrict__ sumsH,
                                                              const double* __restrict__ partH,
                                                              const double* __restrict__ params, int nblk, int nobs,
                                                              int lag, double* __restrict__ hess1,
                                                              double* __restrict__ hess2) {
    __shared__ double tri[20];
    const int k = threadIdx.x;
    if (ctrl->status != 0) return;   // abandoned: the general kernel writes the outputs
    if (k < 20) {
        SvConst c;
        sv_const_init(c, params);
        double h = 0.0;
        for (int t = lag; t < nobs; ++t) {
            const double* sm = sums + (size_t)t * 8;
            const double* sh = sumsH + (size_t)t * 20;
            const double S = sm[0];
            double v;
            if (k >= 10) {
                v = sh[k];
            } else {
                // weighted monomials in cm = curr - mu, sq, ey (sums[t][2..6] = c, sq, sq c, sq^2, sq ey; sumsH[t][0..3] =
                // ey, c^2, c ey, ey^2)
                const double A = c.one_m_phi2, B = c.one_m_phi;
                const double Mc = sm[2] - c.mu * S, Ms = sm[3], Me = sh[0];
                const double Mcc = sh[1] - 2.0 * c.mu * sm[2] + c.mu * c.mu * S;
                const double Mcs = sm[4] - c.mu * sm[3], Mce = sh[2] - c.mu * sh[0];
                const double Mss = sm[5], Mse = sm[6], Mee = sh[3];
                switch (k) {
                    case 0: v = -c.q * (B * B) * S; break;                                              // (0,0)
                    case 1: v = -c.q * A * (B * Mc + Ms); break;                                        // (0,1)
                    case 2: v = -2.0 * B * Ms - c.q * B * c.sr * Mse; break;                            // (0,2)
                    case 3: v = 2.0 * c.q * c.rho * B * Ms - c.inv_sv2 * B * c.sigmav * Me; break;      // (0,3)
                    case 4: v = -c.q * A * (2.0 * c.phi * Mcs + A * Mcc); break;                        // (1,1)
                    case 5: v = -c.q * A * (2.0 * Mcs + c.sr * Mce); break;                             // (1,2)
                    case 6: v = c.q * A * (2.0 * c.rho * Mcs - c.sigmav * c.rho_term * Mce); break;     // (1,3)
                    case 7: v = -2.0 * c.q * Mss - c.q * c.sr * Mse - c.q * (c.sr * c.sr) * Mee; break; // (2,2)
                    case 8:                                                                              // (2,3)
                        v = 2.0 * c.q * c.rho * Mss + (2.0 * (c.rho * c.rho) * c.q * c.sigmav + c.inv_sv) * Mse - c.rho * Mee;
                        break;
                    default:                                                                             // (3,3), "sigmav*(-2)" typo kept
                        v = c.rho_term * S - 2.0 * c.q * (c.rho * c.rho) * Mss + 2.0 * c.sigmav * Mss +
                            2.0 * c.inv_sv * c.rho * Mse - c.rho_term * Mee;
                        break;
                }
            }
            h += v / S;
        }
        for (int irel = 0; irel < lag - 1; ++irel)
            for (int q = 0; q < nblk; ++q) h += partH[((size_t)irel * nblk + q) * 20 + k];
        tri[k] = h;
    }
    __syncwarp();
    if (k < 16) {
        const int r = k >> 2, cidx = k & 3;
        const int lo = min(r, cidx), hi = max(r, cidx);
        const int ti = lo * 4 - (lo * (lo - 1)) / 2 + (hi - lo);
        hess1[k] = tri[ti];
        hess2[k] = tri[10 + ti];
    }
}

// generic Hessian branch: hessian1 / hessian2 = the main-loop sums of steps first .. nobs-1 divided by the weight sum
// of their step, plus the tail blocks irel = 1 .. lag-1, in that order; upper triangles expanded into the symmetric
// 4 x 4 outputs
__global__ void __launch_bounds__(32) grid_hess_finish_gen_kernel(const GridCtrl* __restrict__ ctrl,
                                                                  const double* __restrict__ sums,
                                                                  const double* __restrict__ sumsH,
                                                                  const double* __restrict__ partH, int nblk, int nobs,
                                                                  int first, int lag, double* __restrict__ hess1,
                                                                  double* __restrict__ hess2) {
    __shared__ double tri[20];
    const int k = threadIdx.x;
    if (ctrl->status != 0) return;   // abandoned: diag reports it
    if (k < 20) {
        double h = 0.0;
        for (int t = first; t < nobs; ++t) h += sumsH[(size_t)t * 20 + k] / sums[(size_t)t * 8];
        for (int irel = 1; irel < lag; ++irel)
            for (int q = 0; q < nblk; ++q) h += partH[((size_t)irel * nblk + q) * 20 + k];
        tri[k] = h;
    }
    __syncwarp();
    if (k < 16) {
        const int r = k >> 2, cidx = k & 3;
        const int lo = min(r, cidx), hi = max(r, cidx);
        const int ti = lo * 4 - (lo * (lo - 1)) / 2 + (hi - lo);
        hess1[k] = tri[ti];
        hess2[k] = tri[10 + ti];
    }
}

__global__ void __launch_bounds__(256) grid_tail_reduce_kernel(const double* __restrict__ part, int nblk,
                                                               double* __restrict__ out) {
    __shared__ double red[5 * 32];
    const int irel = blockIdx.x, tid = threadIdx.x;
    double acc[5] = {0.0, 0.0, 0.0, 0.0, 0.0};
    for (int q = tid; q < nblk; q += 256)
#pragma unroll
        for (int k = 0; k < 5; ++k) acc[k] += part[((size_t)irel * nblk + q) * 8 + k];
    block_sum<5>(acc, red);
    if (tid < 5) out[irel * 8 + tid] = acc[tid];
}

// sums[t][0] = sum sh, [1] = sum sh x, [2] = sum sh c, [3] = sum sh sq, [4] = sum sh sq c, [5] = sum sh sq^2,
// [6] = sum sh sq ey (c = lagged ancestor value, sq / ey as stored in P);  tail[irel][0..4].
// GEN (the generic path of a model other than SV): [3..6] = sum sh g[0..3], traj[0] = the initial state, exact pairing of
// the fixed-lag terms (pf_model.cuh).  PRED: the predictive pairing.  Both derive from the model in grid_finish_for.
// SMO = false (the filter alone): no smo / grad, tail unused.
template <bool GEN, bool SMO, bool PRED = false>
__global__ void grid_finish_kernel(const GridCtrl* __restrict__ ctrl, const double* __restrict__ sums,
                                   const double* __restrict__ shift, const double* __restrict__ xmin,
                                   const double* __restrict__ tail, const double* __restrict__ params,
                                   int nobs, int L, double n_total, double* __restrict__ log_like,
                                   double* __restrict__ filt, double* __restrict__ smo,
                                   double* __restrict__ grad, double* __restrict__ traj,
                                   long long* __restrict__ diag, long long* __restrict__ info) {
    const int tid = blockIdx.x * blockDim.x + threadIdx.x;
    // log-likelihood (:537): the terms are computed by the whole first block (the loads and logs of a single thread took
    // 0.29 ms at T = 1000), added up by thread 0 in time order -- the reference's summation order
    __shared__ double s_term[256];
    __shared__ double s_ll;
    if (blockIdx.x == 0) {
        const double logn = log(n_total);
        if (threadIdx.x == 0) s_ll = 0.0;
        for (int base = 1; base < nobs; base += (int)blockDim.x) {
            const int t = base + (int)threadIdx.x;
            if (t < nobs && threadIdx.x < 256) s_term[threadIdx.x] = shift[t] + log(sums[(size_t)t * 8]) - logn;
            __syncthreads();
            if (threadIdx.x == 0) {
                double ll = s_ll;
                const int cnt = min((int)blockDim.x, nobs - base);
                for (int k = 0; k < cnt; ++k) ll += s_term[k];
                s_ll = ll;
            }
            __syncthreads();
        }
    }
    if (tid == 0) {
        log_like[0] = s_ll;
        for (int k = 0; k < PMMH_DIAG_COUNT; ++k) diag[k] = 0;
        diag[PMMH_DIAG_NEAR_TIES] = (long long)ctrl->near_ties;
        diag[PMMH_DIAG_MAX_BIN] = ctrl->max_bin;
        diag[PMMH_DIAG_STATUS] = ctrl->status ? 1 : 0;
        diag[PMMH_DIAG_KEY_TIES] = (long long)ctrl->key_ties;
        diag[PMMH_DIAG_SOFT_TIES] = (long long)ctrl->soft_ties;
        diag[PMMH_DIAG_KERNEL] = 5;
        diag[PMMH_DIAG_FAST_INFO] = ctrl->status;
        if (info) {
            info[0] = (long long)ctrl->soft_ties;
            info[1] = ctrl->status;
        }
    }
    for (int t = tid; t < nobs; t += gridDim.x * blockDim.x) {
        filt[t] = sums[(size_t)t * 8 + 1] / sums[(size_t)t * 8];
        traj[t] = (t == 0 && !GEN) ? params[0] : xmin[t];   // Q10/Q11: traj[t] = X_t[0] for t >= 1, X_0 == mu
        if constexpr (!SMO) continue;
        double s = 0.0, g[4] = {0.0, 0.0, 0.0, 0.0};
        if constexpr (PRED) {
            // predictive pairing (pf_model.cuh): smo[t] and gradient slot t (the pair (x_t, x_t+1) with obs[t]) from step
            // t + L - 1; every tail block irel >= 1 adds smo[nobs-L+irel] and gradient[.][nobs-L+irel] (irel = L - 1: the
            // final generation's term); irel = 0 is empty
            const int ss = t + L - 1;
            if (ss < nobs) {
                const double* sm = sums + (size_t)ss * 8;
                s = sm[2] / sm[0];
                for (int q = 0; q < 4; ++q) g[q] = sm[3 + q] / sm[0];
            }
            const int irel = t - (nobs - L);
            if (irel >= 1 && irel < L) {
                s += tail[irel * 8];
                for (int q = 0; q < 4; ++q) g[q] += tail[irel * 8 + 1 + q];
            }
        } else if constexpr (GEN) {
            // exact pairing (pf_model.cuh): smo[t] from step t + L - 1 (t >= 0), gradient slot t = the pair (x_t-1, x_t)
            // from step t + L - 2; the tail (irel >= 1) adds smo[nobs-L+irel] and gradient[.][nobs-L+irel+1]
            const int ss = t + L - 1, sg = t + L - 2;
            if (ss < nobs) s = sums[(size_t)ss * 8 + 2] / sums[(size_t)ss * 8];
            if (t >= 1 && sg < nobs) {
                const double* sm = sums + (size_t)sg * 8;
                for (int q = 0; q < 4; ++q) g[q] = sm[3 + q] / sm[0];
            }
            const int irel_s = t - (nobs - L);
            if (irel_s >= 1 && irel_s < L) s += tail[irel_s * 8];
            const int irel_g = t - 1 - (nobs - L);
            if (irel_g >= 1 && irel_g < L - 1)
                for (int q = 0; q < 4; ++q) g[q] += tail[irel_g * 8 + 1 + q];
        } else {
            const int src = t + L - 1;   // main-loop terms land at tt = i - L + 1 (:445-470)
            if (t >= 1 && src < nobs) {
                const double* sm = sums + (size_t)src * 8;
                const double S = sm[0];
                s = sm[2] / S;
                SvConst k;
                sv_const_init(k, params);
                // weighted means of g[0..3] of :454-465 written in the monomials sq, sq c, sq^2, sq ey
                g[0] = k.q * k.one_m_phi * sm[3] / S;
                g[1] = k.q * k.one_m_phi2 * (sm[4] - k.mu * sm[3]) / S;
                g[2] = (k.q * sm[5] + k.q * k.sr * sm[6] - S) / S;
                g[3] = (k.rho * S - k.q * k.rho * sm[5] + k.inv_sv * sm[6]) / S;
            }
            const int irel_s = t - (nobs - L);   // tail: i = nobs-L+irel adds smo[i], gradient[.][i-L+1]
            if (irel_s >= 0 && irel_s < L) s += tail[irel_s * 8];
            const int irel_g = t + L - 1 - (nobs - L);
            if (irel_g >= 0 && irel_g < L - 1)
                for (int q = 0; q < 4; ++q) g[q] += tail[irel_g * 8 + 1 + q];
        }
        smo[t] = s;
        for (int q = 0; q < 4; ++q) grad[(size_t)q * nobs + t] = g[q];
    }
}

// the finish kernel of model M: GEN is the grid kernel's (the layout of its sums), which pairs the terms as the
// reference does on the SV path alone
template <class M, bool SMO>
auto grid_finish_for() {
    constexpr bool GEN = !std::is_same<M, SvLeverageModel>::value;
    static_assert(GEN == (M::kPairing != Pairing::Reference), "the SV path alone pairs the terms as the reference does");
    return grid_finish_kernel<GEN, SMO, SMO && M::kPairing == Pairing::Predictive>;
}

struct GridLayout {
    size_t ctrl, ghist, tilecnt, tinfo, H, XE, perm, R, P, psum, shiftv, xminv, shring, parentpos, sums,
        tailpart, tail, info, ustash, xlow, psumH, sumsH, tailpartH, total;
    int RP, nblk, SQ;
};

size_t al256(size_t x) { return (x + 255) & ~(size_t)255; }

// filter: the filter alone -- no genealogy records (R), payloads (P), weight ring or tail sums
GridLayout grid_layout(int nobs, int n, int lag, int G, int hist, int hess, int filter) {
    GridLayout L = GridLayout();
    // ring depth of the payloads: step t writes generation t and gathers from generation t-(lag-2)
    L.RP = lag < 2 ? 2 : lag;
    L.nblk = 296;
    size_t o = 0;
    const size_t N = (size_t)n;
    L.ctrl = o;      o += al256(sizeof(GridCtrl));
    L.ghist = o;     o += al256((size_t)2 * kNF * 4);
    L.tilecnt = o;   o += al256((size_t)2 * kMaxTiles * kCntStride * 4);
    L.tinfo = o;     o += al256((size_t)kMaxTiles * 4 * 8);
    L.H = o;         o += al256(N * 4);
    L.XE = o;        o += al256(N * 16);
    L.perm = o;      o += al256(N * 4);
    const size_t RS = hess ? 2 : 1;   // Hessian branch: 64-byte entries (record | alpha, payload | alpha)
    const size_t smo = filter ? 0 : 1;
    L.R = o;         o += al256(smo * 2 * N * 32 * RS);
    L.P = o;         o += al256(smo * L.RP * N * 32 * RS);
    L.psum = o;      o += al256((size_t)nobs * G * 8 * 8);
    L.shiftv = o;    o += al256((size_t)nobs * 8);
    L.xminv = o;     o += al256((size_t)nobs * 8);
    L.shring = o;    o += al256(smo * lag * N * 8);
    L.parentpos = o; o += al256(hist ? N * 4 : 256);
    L.sums = o;      o += al256((size_t)nobs * 8 * 8);
    L.tailpart = o;  o += al256(smo * lag * L.nblk * 8 * 8);
    L.tail = o;      o += al256(smo * lag * 8 * 8);
    L.info = o;      o += al256(8 * 8);
    L.ustash = o;    o += al256(4 * N * 8);   // host-streamed u: four time steps, time-major
    // Hessian branch: the first SQ sorted values of every generation (Q7: particles[i - 1 + ancestor] read through
    // the flat layout), per-tile / per-step sums
    L.SQ = hess ? (nobs + n - 2) / nobs + 1 : 1;
    L.xlow = o;      o += al256(hess ? (size_t)nobs * L.SQ * 8 : 0);
    L.psumH = o;     o += al256(hess ? (size_t)nobs * G * 20 * 8 : 0);
    L.sumsH = o;     o += al256(hess ? (size_t)nobs * 20 * 8 : 0);
    L.tailpartH = o; o += al256(hess ? (size_t)lag * L.nblk * 20 * 8 : 0);
    L.total = o;
    return L;
}

#define GRID_CUDA(call)                                                  \
    do {                                                                 \
        cudaError_t e__ = (call);                                        \
        if (e__ != cudaSuccess) return pmmh::set_cuda_error(e__, #call); \
    } while (0)

template <bool HESS, class M, bool SMO>
const void* grid_kernel_of(bool team) {
    return team ? (const void*)sv_grid_kernel<1024, HESS, M, SMO, true> : (const void*)sv_grid_kernel<1024, HESS, M, SMO, false>;
}
// the persistent kernel of (model, hess, filter): one problem, or teams of CTAs; the filter runs the model's Filter,
// the smoother without the Hessian its Gradient; nullptr for an unknown model id or a Hessian the model does not have
const void* grid_kernel_for(int model, int hess, int filter, bool team) {
    const void* k = nullptr;
    Models::with(model, [&](auto m) {
        typedef typename decltype(m)::type M;
        if (filter) {
            k = grid_kernel_of<false, typename M::Filter, false>(team);
        } else if (!hess) {
            k = grid_kernel_of<false, typename M::Gradient, true>(team);
        } else if constexpr (M::kHessian) {
            k = grid_kernel_of<true, M, true>(team);
        }
    });
    return k;
}

int grid_check(const SvCall& c, int nobs, int n, int lag, int G, int hess) {
    if (c.filter ? (hess || !sv_grid_filter_eligible(nobs, n, G)) : !sv_grid_eligible(nobs, n, lag, G))
        return set_error(PMMH_ERR_INVALID, "grid kernel: sizes not eligible");
    if (!model_known(c.model)) return set_error(PMMH_ERR_INVALID, "grid kernel: unknown model id");
    if (hess && !model_has_hessian(c.model))
        return set_error(PMMH_ERR_INVALID, "grid kernel: compute_hessian for a model without a Hessian branch");
    return PMMH_OK;
}

// dynamic shared memory of every persistent kernel, once per device and host thread
int grid_set_attributes() {
    static thread_local bool attr_set[64] = {false};
    int dev = 0;
    GRID_CUDA(cudaGetDevice(&dev));
    if (dev >= 0 && dev < 64 && !attr_set[dev]) {
        // no persisting L2 set-aside for the kernel's evict_last accesses: with one every phase is slower
        // (DESIGN 4.0), and left unset the evaluation at N = 2^20 is ~6 % slower
        GRID_CUDA(cudaDeviceSetLimit(cudaLimitPersistingL2CacheSize, 0));
        cudaError_t err = cudaSuccess;
        Models::each([&](auto m) {
            for (int team = 0; team < 2; ++team)
                for (int v = 0; v < 3; ++v)   // smoother, smoother with Hessian (where the model has one), filter
                    if (const void* k = grid_kernel_for(decltype(m)::type::kId, v == 1, v == 2, team != 0))
                        if (err == cudaSuccess)
                            err = cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, kDynSmem);
        });
        GRID_CUDA(err);
        attr_set[dev] = true;
    }
    return PMMH_OK;
}

// arguments of the problem `c` describes, its workspace slice (layout L) at ws
GridArgs grid_args(const SvCall& c, const GridLayout& L, char* ws, int nobs, int n, int lag, int G, int hess) {
    GridArgs a;
    memset(&a, 0, sizeof(a));
    a.N = n;
    a.NOBS = nobs;
    a.LAG = lag;
    a.G = G;
    a.Wc = (n + G - 1) / G;
    a.RP = L.RP;
    a.hist = c.x_hist != nullptr;
    a.obs = c.obs;
    a.params = c.params;
    a.rvr = c.rvr;
    a.U = c.u;
    if (c.slot > 0) {   // particle-major slots of c.slot time steps (host-streamed)
        a.u_cs = c.slot;
        a.u_cstride = (long long)n * c.slot;
        a.u_tstride = 1;
        a.u_jstride = c.slot;
        a.u_flag = c.u_flag;
        a.ustash = (double*)(ws + L.ustash);
    } else {
        a.u_cs = 1 << 30;
        a.u_cstride = 0;
        a.u_tstride = n;
        a.u_jstride = 1;
        a.u_flag = nullptr;
    }
    a.ctrl = (GridCtrl*)(ws + L.ctrl);
    a.ghist = (int*)(ws + L.ghist);
    a.tilecnt = (int*)(ws + L.tilecnt);
    a.tinfo = (double*)(ws + L.tinfo);
    a.H = (int*)(ws + L.H);
    a.XE = (double2*)(ws + L.XE);
    a.perm = (int*)(ws + L.perm);
    a.R = (REntry*)(ws + L.R);
    a.P = (PEntry*)(ws + L.P);
    a.psum = (double*)(ws + L.psum);
    a.shiftv = (double*)(ws + L.shiftv);
    a.xminv = (double*)(ws + L.xminv);
    a.shring = (double*)(ws + L.shring);
    a.parentpos = (int*)(ws + L.parentpos);
    a.xlow = (double*)(ws + L.xlow);
    a.psumH = (double*)(ws + L.psumH);
    a.SQ = L.SQ;
    a.RS = hess ? 2 : 1;
    a.Xhist = c.x_hist;
    a.Ahist = c.a_hist;
    a.prof = c.prof;
    return a;
}

// the kernels after the persistent one (reductions, tail, output assembly) for the problem `c` / `a` describe:
// 2 launches (filter), 4 (smoother), 6 (smoother with the Hessian branch)
int grid_after(const SvCall& c, const GridArgs& a, const GridLayout& L, char* ws, int nobs, int n, int lag, int G,
               int hess) {
    const cudaStream_t st = c.stream;
    double* sums = (double*)(ws + L.sums);
    double* tailpart = (double*)(ws + L.tailpart);
    double* tail = (double*)(ws + L.tail);
    grid_reduce_kernel<<<nobs, 256, 0, st>>>(a.psum, G, sums);
    Models::with(c.model, [&](auto m) {   // (grid_check has refused an unknown id and a Hessian the model lacks)
        typedef typename decltype(m)::type M;
        const auto finish = c.filter ? grid_finish_for<typename M::Filter, false>() : grid_finish_for<M, true>();
        if (!c.filter) {
            if (!hess) {
                grid_tail_kernel<false, typename M::Gradient><<<dim3(L.nblk, lag), 256, 0, st>>>(a, sums, tailpart,
                                                                                                nullptr, L.nblk);
            } else if constexpr (M::kHessian) {
                double* sumsH = (double*)(ws + L.sumsH);
                double* tailpartH = (double*)(ws + L.tailpartH);
                grid_reduceH_kernel<<<nobs, 640, 0, st>>>(a.psumH, G, pair_first_step(M::kPairing, lag), sumsH);
                grid_tail_kernel<true, M><<<dim3(L.nblk, lag), 256, 0, st>>>(a, sums, tailpart, tailpartH, L.nblk);
                if constexpr (M::kPairing == Pairing::Reference)
                    grid_hess_finish_kernel<<<1, 32, 0, st>>>(a.ctrl, sums, sumsH, tailpartH, c.params, L.nblk, nobs,
                                                              lag, c.hess1, c.hess2);
                else
                    grid_hess_finish_gen_kernel<<<1, 32, 0, st>>>(a.ctrl, sums, sumsH, tailpartH, L.nblk, nobs,
                                                                  pair_first_step(M::kPairing, lag), lag, c.hess1,
                                                                  c.hess2);
            }
            grid_tail_reduce_kernel<<<lag, 256, 0, st>>>(tailpart, L.nblk, tail);
        }
        finish<<<(nobs + 255) / 256, 256, 0, st>>>(a.ctrl, sums, a.shiftv, a.xminv, c.filter ? nullptr : tail, c.params,
                                                   nobs, lag, (double)n, c.ll, c.filt, c.smo, c.grad, c.traj, c.diag,
                                                   (long long*)(ws + L.info));
    });
    GRID_CUDA(cudaGetLastError());
    return PMMH_OK;
}

// problem b of a batch call: its inputs, outputs and history
SvCall grid_problem(const SvCall& c, int b, int nobs, int n) {
    SvCall p = c;
    const size_t bn = (size_t)b * nobs;
    p.obs = c.obs + b * c.obs_stride;
    p.params = c.params + 4 * (size_t)b;
    p.rvr = c.rvr + bn;
    p.u = c.u + bn * n;
    p.filt = c.filt + bn;
    if (c.smo) p.smo = c.smo + bn;
    p.ll = c.ll + b;
    if (c.grad) p.grad = c.grad + 4 * bn;
    p.traj = c.traj + bn;
    if (c.hess1) p.hess1 = c.hess1 + 16 * (size_t)b;
    if (c.hess2) p.hess2 = c.hess2 + 16 * (size_t)b;
    p.diag = c.diag + (size_t)b * PMMH_DIAG_COUNT;
    if (c.x_hist) p.x_hist = c.x_hist + bn * n;
    if (c.a_hist) p.a_hist = c.a_hist + bn * n;
    return p;
}

}  // namespace

int sv_grid_ctas(int n, int sm_count, int ctas) {
    int G = ctas > 0 ? ctas : (n + 2047) / 2048;
    if (G > sm_count) G = sm_count;
    if (G > kMaxTiles) G = kMaxTiles;
    if (G < 1) G = 1;
    return G;
}

// a tile holds N/G particles +- one histogram bin; 12 % head room below the shared-memory capacity
static bool grid_tile_fits(int n, int G) {
    if (G < 1 || G > kMaxTiles || n < 32 || n > (1 << 21)) return false;
    const int Wc = (n + G - 1) / G;
    return Wc <= kCap - kCap / 8;
}

bool sv_grid_eligible(int nobs, int n, int lag, int G) {
    return lag >= 2 && lag <= 10 && nobs >= 2 * lag && grid_tile_fits(n, G);
}

bool sv_grid_filter_eligible(int nobs, int n, int G) { return nobs >= 2 && grid_tile_fits(n, G); }

size_t sv_grid_ws_bytes(int nobs, int n, int lag, int G, int hist, int hess, int filter) {
    return grid_layout(nobs, n, lag, G, hist, hess, filter).total;
}

int sv_grid_teams(int batch, int sm_count, int G) {
    int t = G > 0 ? sm_count / G : 0;
    if (t > batch) t = batch;
    return t < 1 ? 1 : t;
}

int sv_grid_run(const SvCall& c, int batch, int nobs, int n, int lag, int G, int nteams, int hess) {
    int rc = grid_check(c, nobs, n, lag, G, hess);
    if (rc != PMMH_OK) return rc;
    if (batch < 1 || nteams < 1) return set_error(PMMH_ERR_INVALID, "grid kernel: bad team count");
    if (batch > 1 && (c.slot > 0 || c.prof)) return set_error(PMMH_ERR_INVALID, "grid kernel: teams take device-resident u only");
    const GridLayout L = grid_layout(nobs, n, lag, G, c.x_hist != nullptr, hess, c.filter);
    const int slices = batch < nteams ? batch : nteams;
    if (c.ws_bytes < (size_t)slices * L.total) return set_error(PMMH_ERR_WORKSPACE, "grid kernel: workspace too small");
    char* ws = (char*)c.ws;
    const cudaStream_t st = c.stream;
    rc = grid_set_attributes();
    if (rc != PMMH_OK) return rc;
    GridTeam tm;
    tm.ws_stride = (long long)L.total;
    tm.obs_stride = c.obs_stride;
    for (int b0 = 0; b0 < batch; b0 += nteams) {
        const int nw = batch - b0 < nteams ? batch - b0 : nteams;   // problems (teams) of this wave
        // control block, histograms, reservation counters, tile info of every team: zero
        for (int k = 0; k < nw; ++k)
            GRID_CUDA(cudaMemsetAsync(ws + (size_t)k * L.total + L.ctrl, 0, L.H - L.ctrl, st));
        GridArgs a = grid_args(grid_problem(c, b0, nobs, n), L, ws, nobs, n, lag, G, hess);
        void* kargs[] = {(void*)&a, (void*)&tm};
        // a wave of one problem runs the one-problem instantiation
        GRID_CUDA(cudaLaunchCooperativeKernel(grid_kernel_for(c.model, hess, c.filter, nw > 1), dim3(nw * G), dim3(1024),
                                              kargs, kDynSmem, st));
        for (int k = 0; k < nw; ++k) {
            char* wk = ws + (size_t)k * L.total;
            const SvCall pc = grid_problem(c, b0 + k, nobs, n);
            rc = grid_after(pc, grid_args(pc, L, wk, nobs, n, lag, G, hess), L, wk, nobs, n, lag, G, hess);
            if (rc != PMMH_OK) return rc;
        }
    }
    return PMMH_OK;
}

}  // namespace pmmh
