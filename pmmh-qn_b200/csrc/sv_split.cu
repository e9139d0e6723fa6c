// sv_split.cu -- ONE stochastic-volatility particle filter / fixed-lag smoother whose particles
// are split over the GPUs of a box (BASELINE.json configs[4], SURVEY.md 8e "single large PF").
//
// Same algorithm as flps_sv_corr (/root/reference/python/state/particle_methods/
// stochastic_volatility.pyx:205-655: sort -> correlated systematic resampling -> propagate ->
// weights -> fixed-lag score terms); what is new is the partition.  Rank r of `world` owns a
// contiguous VALUE range of the sorted generation (n_r particles, every value on rank r <= every
// value on rank r+1).  One time step is a sequence of device phases with three exchanges between
// them; the exchanges themselves are issued by the host layer (torch.distributed / NCCL):
//
//   weights    log-weights, sh_j = exp(lw_j - shift), tiled inclusive scan of sh over the local
//              generation, local sums for the outputs              -> 4 doubles per rank
//   [all-gather of (sum sh, n_r, min x, max x)]   <- the "per-shard weight totals"
//   children   global offset of this rank's cumulative weights; the children of LOCAL parents
//              form a contiguous range [jlo, jhi) of the N resampling points (:694-715 evaluated
//              parent-side, so no parent is ever fetched from another GPU); vectorised binary
//              search of every child in the local cumulative weights, propagation (:354-358),
//              coarse value histogram (4096 bins)                  -> 4096 ints per rank
//   [all-gather of the histograms]
//   plan       splitters on histogram-bin boundaries that give every rank ~N/world arrivals,
//              send / receive counts, fine sort bins for the local value range
//   pack       records (value + lagged ancestor values) grouped by destination rank
//   [all-to-all-v of the records]
//   sort       counting sort of the arrivals into fine bins (~8 per bin) + exact in-bin ranking
//              = the reference's argsort (:392-424, :23-52) restricted to this value range
//
// On ONE device the same phases are driven from C++ without any host synchronisation
// (sv_split_single_run: records as above; sv_split_path_run: "path storage" -- a generation is
// stored once in birth order as (value, parent row), nothing is copied when a particle has
// children, jump tables reach the lagged ancestors); pmmh_flps_sv_corr selects the latter for
// problems larger than the persistent exchange kernel takes (N > 2^20).
//
// Deviations from the reference's operation order are confined to summation order (parallel
// scans / reductions instead of one sequential loop) and the choice of the log-weight shift
// (any shift cancels analytically; Q4).  Resampling decisions that fall within 64 ulp of a
// cumulative-weight tie are counted (diag[0]).  fp64, -fmad=false.  HBM/L2-bound streaming and
// gather work: no tensor cores.
#include <cuda_runtime.h>
#include <math.h>
#include <stdint.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include "../../include/pmmh_qn.h"
#include "common.cuh"
#include "philox.cuh"
#include "sv_math.cuh"
#include "sv_split.cuh"

namespace pmmh {

int set_error(int code, const char* what);           // capi.cu
int set_cuda_error(cudaError_t err, const char* where);

namespace {

constexpr int kBins = 4096;         // coarse value bins of the routing histogram
constexpr int kTile = 1024;         // particles per scan tile (128 threads x 8)
constexpr int kTileThreads = kTile / 8;
constexpr int kFine = 8;            // target occupancy of a fine sort bin
constexpr int kMaxWorld = 16;
constexpr int kStage = 4096;        // cumulative weights staged in shared memory per child tile
constexpr int kChildTile = 1024;    // children per tile (256 threads x 4)
constexpr int kMaxRounds = 64;      // child tiles whose boundaries one block resolves at once
constexpr int kMaxBinRank = 8192;   // a fine bin larger than this abandons the evaluation
constexpr int kLineageGrid = 148 * 4;   // blocks of the lineage kernel (one partial-sum row each)
constexpr double kChildNsd = 6.5;   // histogram range: extreme propagation means +- 6.5 sd

struct SplitState {
    long long N;
    int world, rank, LR, nobs;
    long long cap, capc;
    // step scalars (children kernel)
    long long jlo, jhi;
    int nc;
    double S, off, lo, scale, shift;
    // plan
    int n_arrivals, NF;
    int send_cnt[kMaxWorld], send_off[kMaxWorld], recv_cnt[kMaxWorld], cursor[kMaxWorld];
    // diagnostics
    unsigned long long near_ties, key_ties;
    int max_bin, status;
    unsigned int ticket_c;   // last-block-done counter of the children kernel (fused plan)
};

__global__ void split_set_state_kernel(SplitState* dst, const SplitState h) { *dst = h; }

struct Layout {
    size_t state, cumblk, boff, btot, tlast, bpart, gpart, cstart, xc, pa, cb, dest, nfc, fstart, counts, fcnt, fst,
        rnk, fb, tkey, tidx, tfb, total;
    long long ntiles_max, nf_max;
};

size_t al(size_t x) { return (x + 255) & ~(size_t)255; }

Layout make_layout(long long cap, long long capc) {
    Layout L = Layout();
    L.ntiles_max = (cap + kTile - 1) / kTile + 1;
    L.nf_max = cap / kFine + kBins + 64;
    size_t o = 0;
    L.state = o;   o += al(sizeof(SplitState));
    L.cumblk = o;  o += al((size_t)cap * 8);
    L.boff = o;    o += al((size_t)(L.ntiles_max + 1) * 8);
    L.btot = o;    o += al((size_t)L.ntiles_max * 8);
    L.tlast = o;   o += al((size_t)L.ntiles_max * 8);
    L.bpart = o;   o += al((size_t)L.ntiles_max * 8 * 8);
    L.gpart = o;   o += 2 * al((size_t)kLineageGrid * 8 * 8);   // two generations in flight
    L.cstart = o;  o += al((size_t)kBins * 4);
    L.xc = o;      o += al((size_t)capc * 8);
    L.pa = o;      o += al((size_t)capc * 4);
    L.cb = o;      o += al((size_t)capc * 2);
    L.dest = o;    o += al((size_t)kBins * 4);
    L.nfc = o;     o += al((size_t)kBins * 4);
    L.fstart = o;  o += al((size_t)(kBins + 1) * 4);
    L.counts = o;  o += al((size_t)(2 * kMaxWorld + 4) * 4);
    L.fcnt = o;    o += al((size_t)(L.nf_max + 1) * 4);
    L.fst = o;     o += al((size_t)(L.nf_max + 1) * 4);
    L.rnk = o;     o += al((size_t)cap * 4);
    L.fb = o;      o += al((size_t)cap * 4);
    L.tkey = o;    o += al((size_t)cap * 16);   // SortEntry[cap]
    L.tidx = o;    o += al((size_t)cap * 4);
    L.tfb = o;     o += al((size_t)cap * 4);
    L.total = o;
    return L;
}

// ---------------------------------------------------------------------------------------------
// generation 0: every particle = mu (Q1, :306-323), identity order, history rows (mu, 0, ...)
// ---------------------------------------------------------------------------------------------
__global__ void split_init_kernel(double* __restrict__ xs, int* __restrict__ perm,
                                  double* __restrict__ rec, int n, int LR,
                                  const double* __restrict__ params) {
    const double mu = params[0];
    for (int p = blockIdx.x * blockDim.x + threadIdx.x; p < n; p += gridDim.x * blockDim.x) {
        xs[p] = mu;
        perm[p] = p;
        rec[(size_t)p * LR] = mu;
        for (int m = 1; m < LR; ++m) rec[(size_t)p * LR + m] = 0.0;
    }
}

// ---------------------------------------------------------------------------------------------
// weights: one block per tile of 2048 sorted particles (thread = 8 consecutive particles)
//   sh_j = exp(norm_logpdf(y_t; 0, exp(x_j / 2)) - shift)          (:427-437, :659-664)
//   cumblk[p] = inclusive sum of sh inside the tile, btot[tile] = tile total
//   bpart[tile][0..6] = sum sh x | sum sh curr | sum sh g_0..3     (:439-470, unnormalised)
// ---------------------------------------------------------------------------------------------
template <bool GRAD>
__global__ void __launch_bounds__(kTileThreads) split_weights_kernel(
    SplitState* __restrict__ st, const double* __restrict__ xs, const int* __restrict__ perm,
    const double* __restrict__ rec, int n, int LR, const double* __restrict__ obs, int t, int lag,
    const double* __restrict__ params, int uniform, double* __restrict__ cumblk,
    double* __restrict__ btot, double* __restrict__ tlast, double* __restrict__ bpart,
    double* __restrict__ shsave) {
    __shared__ double red[7 * 32];
    __shared__ double s_wtot[kTileThreads / 32];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    SvConst c;
    sv_const_init(c, params);
    const double shift = uniform ? 0.0 : st->shift;
    const double y = obs[t], ylag = GRAD ? obs[t - lag] : 0.0;   // Q5: obs[i - LAG]
    const int base = blockIdx.x * kTile + tid * 8;
    double loc[8];
    double acc[7] = {0.0, 0.0, 0.0, 0.0, 0.0, 0.0, 0.0};
    double run = 0.0;
    bool bad = false;
#pragma unroll
    for (int k = 0; k < 8; ++k) {
        const int p = base + k;
        if (p < n) {
            const double x = xs[p];
            double s = uniform ? 1.0 : exp(sv_logw(x, y) - shift);
            if (!isfinite(s)) {
                bad = true;
                s = 0.0;
            }
            if (shsave) shsave[p] = s;
            run = run + s;
            acc[0] += s * x;
            if (GRAD) {
                const size_t row = (size_t)perm[p] * LR;
                const double curr = rec[row + LR - 1], next = rec[row + LR - 2];
                double sq, g[4];
                sv_score_main(c, curr, next, ylag, sq, g);
                acc[1] += s * curr;
#pragma unroll
                for (int q = 0; q < 4; ++q) acc[2 + q] += g[q] * s;
            }
        }
        loc[k] = run;
    }
    if (bad) atomicOr(&st->status, 2);
    const double incl = warp_incl_scan(run, lane);
    double excl = __shfl_up_sync(kFullMask, incl, 1);
    if (lane == 0) excl = 0.0;
    if (lane == 31) s_wtot[warp] = incl;
    __syncthreads();
    double woff = 0.0;
    for (int w = 0; w < warp; ++w) woff = woff + s_wtot[w];
    const double toff = woff + excl;
#pragma unroll
    for (int k = 0; k < 8; ++k) {
        const int p = base + k;
        if (p < n) {
            const double v = toff + loc[k];
            cumblk[p] = v;
            if (p == n - 1 || p == (int)(blockIdx.x + 1) * kTile - 1) tlast[blockIdx.x] = v;
        }
    }
    if (tid == 0) {
        double tot = 0.0;
        for (int w = 0; w < kTileThreads / 32; ++w) tot = tot + s_wtot[w];
        btot[blockIdx.x] = tot;
    }
    if (GRAD) {
        block_sum<7>(acc, red);
        if (tid < 7) bpart[(size_t)blockIdx.x * 8 + tid] = acc[tid];
    } else {   // only sum sh x is non-zero
        double a1[1] = {acc[0]};
        block_sum<1>(a1, red);
        if (tid == 0) bpart[(size_t)blockIdx.x * 8] = a1[0];
    }
}

// one block: sequential-in-chunks exclusive scan of the tile totals, fixed-order sums of the
// tile partials, the 4 doubles this rank contributes to the all-gather
__global__ void __launch_bounds__(1024) split_weights_finalize_kernel(
    SplitState* __restrict__ st, const double* __restrict__ xs, int n, int ntiles,
    const double* __restrict__ btot, const double* __restrict__ bpart, const double* __restrict__ gpart,
    double* __restrict__ sums_prev, double* __restrict__ boff, double* __restrict__ sums_t,
    double* __restrict__ gather_send, int nval) {
    __shared__ double red[7 * 32];
    __shared__ double s_lane[33];
    __shared__ double s_part[1024], s_off[1024];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, nthr = blockDim.x;
    // exclusive scan of the tile totals in a fixed order: every thread sums a short run of tiles
    // (independent loads), warp 0 scans the 1024 partial sums in shared memory, every thread
    // writes the offsets of its run
    const int per = (ntiles + nthr - 1) / nthr;
    const int qb = min(ntiles, tid * per), qe = min(ntiles, qb + per);
    {
        double sp = 0.0;
        for (int q = qb; q < qe; ++q) sp = sp + btot[q];
        s_part[tid] = sp;
    }
    __syncthreads();
    if (warp == 0) {
        const int chunk = (nthr + 31) / 32;
        const int cb0 = min(nthr, lane * chunk), ce0 = min(nthr, cb0 + chunk);
        double sl = 0.0;
        for (int q = cb0; q < ce0; ++q) sl = sl + s_part[q];
        s_lane[lane + 1] = sl;
        __syncwarp();
        if (lane == 0) {
            s_lane[0] = 0.0;
            for (int q = 1; q <= 32; ++q) s_lane[q] = s_lane[q - 1] + s_lane[q];
        }
        __syncwarp();
        double r = s_lane[lane];
        for (int q = cb0; q < ce0; ++q) {
            s_off[q] = r;
            r = r + s_part[q];
        }
    }
    __syncthreads();
    {
        double r = s_off[tid];
        for (int q = qb; q < qe; ++q) {
            boff[q] = r;
            r = r + btot[q];
        }
        if (tid == 0) boff[ntiles] = s_lane[32];
    }
    // (the two ends of the sorted generation, needed at the very end: loads issued early)
    const double x_first = (tid == 0 && n > 0) ? xs[0] : 0.0, x_last = (tid == 0 && n > 0) ? xs[n - 1] : 0.0;
    double acc[7] = {0.0, 0.0, 0.0, 0.0, 0.0, 0.0, 0.0};
    if (nval == 1) {   // no gather variant: only sum sh x is live
        double a1[1] = {0.0};
        for (int q = tid; q < ntiles; q += blockDim.x) a1[0] += bpart[(size_t)q * 8];
        block_sum<1>(a1, red);
        acc[0] = a1[0];
    } else {
        for (int q = tid; q < ntiles; q += blockDim.x)
#pragma unroll
            for (int k = 0; k < 7; ++k) acc[k] += bpart[(size_t)q * 8 + k];
        block_sum<7>(acc, red);
    }
    // path storage: sum sh curr, sum sh g_0..3 of the PREVIOUS generation come from the lineage
    // kernel, which runs one step behind on the second stream (these sums only feed outputs)
    double late[5] = {0.0, 0.0, 0.0, 0.0, 0.0};
    if (gpart) {
        for (int q = tid; q < kLineageGrid; q += blockDim.x)
#pragma unroll
            for (int k = 0; k < 5; ++k) late[k] += gpart[(size_t)q * 8 + k];
        block_sum<5>(late, red);
    }
    __syncthreads();
    if (tid == 0) {
        if (gpart)
            for (int k = 0; k < 5; ++k) sums_prev[2 + k] = late[k];
        const double tot = s_lane[32];
        sums_t[0] = tot;
        for (int k = 0; k < 7; ++k) sums_t[1 + k] = acc[k];
        gather_send[0] = tot;
        gather_send[1] = (double)n;
        gather_send[2] = n > 0 ? x_first : INFINITY;
        gather_send[3] = n > 0 ? x_last : -INFINITY;
    }
}

// ---------------------------------------------------------------------------------------------
// children
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ double cum_at(int p, double off, double S, const double* __restrict__ boff,
                                         const double* __restrict__ cumblk) {
    return ((off + boff[p / kTile]) + cumblk[p]) / S;
}

// first p in [lo, hi) with cum(p) >= cp, hi if none
__device__ __forceinline__ int cum_search(double cp, int lo, int hi, double off, double S,
                                          const double* __restrict__ boff,
                                          const double* __restrict__ cumblk) {
    while (lo < hi) {
        const int mid = (lo + hi) >> 1;
        if (cum_at(mid, off, S, boff, cumblk) < cp) lo = mid + 1;
        else hi = mid;
    }
    return lo;
}

// Warp-cooperative search: every round the 32 lanes probe 32 evenly spaced positions of
// [lo, hi) and a ballot narrows the range 32-fold -- 2 + 2 dependent rounds of loads for 1024
// tiles x 1024 particles instead of ~20 dependent probes by one thread.  pred must be
// monotone (false ... false true ... true); returns the first true position, hi if none.
template <typename Pred>
__device__ __forceinline__ int warp_first_true(int lo, int hi, int lane, Pred pred) {
    while (hi > lo) {
        const int span = hi - lo, step = (span + 31) >> 5;
        const int pos = lo + lane * step;
        const bool ge = (pos < hi) ? pred(pos) : true;
        const unsigned m = __ballot_sync(kFullMask, ge);
        if (m == 0) {                      // all 32 probes false: the answer lies behind the last one
            lo = lo + 31 * step + 1;
            continue;
        }
        const int f = __ffs(m) - 1;
        if (f == 0) return lo;
        hi = min(hi, lo + f * step);       // first probed true position (or the old end)
        lo = lo + (f - 1) * step + 1;      // one behind the last probed false position
    }
    return lo;
}

__device__ __forceinline__ int cum_search_warp(double cp, int n, double off, double S,
                                               const double* __restrict__ boff,
                                               const double* __restrict__ tlast,
                                               const double* __restrict__ cumblk, int lane) {
    const int ntiles = (n + kTile - 1) / kTile;
    const int tl = warp_first_true(0, ntiles, lane, [&](int q) {
        return !(((off + boff[q]) + tlast[q]) / S < cp);
    });
    if (tl >= ntiles) return n;
    return warp_first_true(tl * kTile, min(n, (tl + 1) * kTile), lane, [&](int q) {
        return !(cum_at(q, off, S, boff, cumblk) < cp);
    });
}

// #{ j in [0, N) : (u + j) / N <= c }, the exact predicate of :703-711 re-checked
__device__ long long count_le(double c, double u, long long N) {
    const double dn = (double)N;
    const double e = c * dn - u;
    long long est = (e < 0.0) ? 0 : (e >= dn ? N : (long long)floor(e) + 1);
    if (est < 0) est = 0;
    if (est > N) est = N;
    while (est > 0 && (u + (double)(est - 1)) / dn > c) --est;
    while (est < N && (u + (double)est) / dn <= c) ++est;
    return est;
}

struct ChildScalars {
    long long jlo, jhi;
    double S, off, lo, scale, cprev;
    int nc;
};

__global__ void __launch_bounds__(256, 4) split_children_kernel(
    SplitState* __restrict__ st, int t, int n, const double* __restrict__ obs,
    const double* __restrict__ params, const double* __restrict__ rvr, const double* __restrict__ u,
    unsigned long long seed, unsigned long long philox_offset, const double* __restrict__ gather,
    const double* __restrict__ xs, const double* __restrict__ cumblk, const double* __restrict__ boff,
    const double* __restrict__ tlast, double* __restrict__ xc, int* __restrict__ pa, unsigned short* __restrict__ cb,
    int* __restrict__ hist_out, double* __restrict__ shift_out, double* __restrict__ xmin_out,
    const int* __restrict__ perm, int* __restrict__ par_out, int fuse_plan, int* __restrict__ nfc,
    int* __restrict__ fstart, int* __restrict__ cstart, int u_pm_chunk) {
    extern __shared__ unsigned char smem_raw[];
    double* s_cum = (double*)smem_raw;                       // [kStage]
    int* s_hist = (int*)(smem_raw + (size_t)kStage * 8);     // [kBins]
    __shared__ ChildScalars sc;
    __shared__ int s_tp[2 * kMaxRounds];
    __shared__ int s_near[8];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    SvConst c;
    sv_const_init(c, params);
    const long long N = st->N;
    const double uu = rvr[t], y1 = obs[t - 1];
    for (int b = tid; b < kBins; b += 256) s_hist[b] = 0;
    if (tid == 0) {
        const int G = st->world, r = st->rank;
        double S = 0.0, off = 0.0, xmin = INFINITY, xmax = -INFINITY, tot_r = 0.0;
        int last_nonempty = -1, prev_nonempty = -1;
        for (int q = 0; q < G; ++q) {
            const double tot = gather[q * 4];
            const int nq = (int)gather[q * 4 + 1];
            if (q == r) {
                off = S;
                tot_r = tot;
            }
            S = S + tot;
            if (nq > 0) {
                xmin = fmin(xmin, gather[q * 4 + 2]);
                xmax = fmax(xmax, gather[q * 4 + 3]);
                last_nonempty = q;
                if (q < r) prev_nonempty = q;
            }
        }
        long long jlo = 0, jhi = 0;
        if (n > 0) {
            jlo = (prev_nonempty < 0) ? 0 : count_le(off / S, uu, N);
            jhi = (r == last_nonempty) ? N : count_le((off + tot_r) / S, uu, N);
            if (jhi < jlo) jhi = jlo;
        }
        long long nc = jhi - jlo;
        double lo, hi;
        sv_child_range(c, xmin, xmax, y1, kChildNsd, lo, hi);
        const double scale = (double)kBins / (hi - lo);
        const double y = obs[t];
        double xstar = (y != 0.0) ? log(y * y) : lo;
        xstar = fmin(fmax(xstar, lo), hi);
        const double shift = sv_logw(xstar, y);
        int bad = 0;
        if (!(S > 0.0) || !isfinite(S) || !isfinite(scale) || !(scale > 0.0) || !isfinite(shift)) bad = 1;
        if (nc > st->capc) {
            bad = 4;
            nc = st->capc;
        }
        sc.jlo = jlo;
        sc.jhi = jhi;
        sc.S = S;
        sc.off = off;
        sc.lo = lo;
        sc.scale = scale;
        sc.cprev = off / S;
        sc.nc = (int)nc;
        if (bad) sc.nc = (bad == 4) ? sc.nc : 0;
        if (blockIdx.x == 0) {
            st->jlo = jlo;
            st->jhi = jhi;
            st->nc = sc.nc;
            st->S = S;
            st->off = off;
            st->lo = lo;
            st->scale = scale;
            st->shift = shift;
            if (bad) atomicOr(&st->status, bad == 4 ? 4 : 1);
            shift_out[t] = shift;
            xmin_out[t - 1] = xmin;
        }
    }
    __syncthreads();
    const int nc = sc.nc;
    const double S = sc.S, off = sc.off, lo = sc.lo, scale = sc.scale;
    const long long jlo = sc.jlo;
    const double dn = (double)N;
    // tile size chosen so that every block handles the same number of (equal) tiles
    const int per_blk = (nc + (int)gridDim.x - 1) / (int)gridDim.x;
    const int rounds_blk = max(1, (per_blk + kChildTile - 1) / kChildTile);
    const int ctile = max(1, (per_blk + rounds_blk - 1) / rounds_blk);
    const int ntl = (nc + ctile - 1) / ctile;
    int near = 0;
    for (int r0 = 0; blockIdx.x + (long long)r0 * gridDim.x < ntl; r0 += kMaxRounds) {
        // boundaries (first and last parent) of up to kMaxRounds of this block's tiles at once
        // (one warp per boundary)
        for (int bq = warp; bq < 2 * kMaxRounds; bq += 8) {
            const long long tile = blockIdx.x + (long long)(r0 + (bq >> 1)) * gridDim.x;
            if (tile >= ntl) break;
            long long k = tile * ctile;
            if (bq & 1) k = min((long long)nc, k + ctile) - 1;
            const double cp = (uu + (double)(jlo + k)) / dn;
            const int pos = cum_search_warp(cp, n, off, S, boff, tlast, cumblk, lane);
            if (lane == 0) s_tp[bq] = min(n - 1, pos);
        }
        __syncthreads();
        for (int rr = 0; rr < kMaxRounds; ++rr) {
            const long long tile = blockIdx.x + (long long)(r0 + rr) * gridDim.x;
            if (tile >= ntl) break;
            const int pf = s_tp[2 * rr], pl = max(pf, s_tp[2 * rr + 1]);
            const int cnt = pl - pf + 1;
            const bool staged = cnt <= kStage;
            // u comes from DRAM and is read exactly once: its loads are issued before the staging
            double uvp[4];
#pragma unroll
            for (int m = 0; m < 4; ++m) {
                const long long k = tile * ctile + tid + 256 * m;
                // time-major u[t][j], or (host-streamed) particle-major chunks u[j][t % chunk] whose
                // 32-byte sectors serve four consecutive time steps out of L2
                uvp[m] = (u && tid + 256 * m < ctile && k < nc)
                             ? (u_pm_chunk ? __ldg(u + (size_t)(jlo + k) * u_pm_chunk + (t % u_pm_chunk))
                                           : ld_stream_f64(u + (size_t)t * (size_t)N + (size_t)(jlo + k)))
                             : 0.0;
            }
            if (staged)
                for (int q = tid; q < cnt; q += 256) s_cum[q] = cum_at(pf + q, off, S, boff, cumblk);
            __syncthreads();
#pragma unroll
            for (int m = 0; m < 4; ++m) {
                const long long k = tile * ctile + tid + 256 * m;
                if (tid + 256 * m < ctile && k < nc) {
                    const long long j = jlo + k;
                    const double cp = (uu + (double)j) / dn;
                    int a;
                    double ca;
                    if (staged) {
                        int l = 0, h = cnt;
                        while (l < h) {
                            const int mid = (l + h) >> 1;
                            if (s_cum[mid] < cp) l = mid + 1;
                            else h = mid;
                        }
                        l = min(l, cnt - 1);
                        a = pf + l;
                        ca = s_cum[l];
                    } else {
                        a = min(pl, cum_search(cp, pf, pl + 1, off, S, boff, cumblk));
                        ca = cum_at(a, off, S, boff, cumblk);
                    }
                    const double cprev = (a > 0) ? ((staged && a > pf) ? s_cum[a - pf - 1]
                                                                        : cum_at(a - 1, off, S, boff, cumblk))
                                                 : sc.cprev;
                    const double tol = 1.4210854715202004e-14 * cp;   // 64 ulp
                    if (fabs(ca - cp) <= tol || fabs(cprev - cp) <= tol) ++near;
                    const double x = xs[a];
                    double mean = c.mu + c.phi * (x - c.mu);
                    mean += c.sr * exp(-0.5 * x) * y1;
                    const double uv = u ? uvp[m]
                                        : philox_normal(seed, philox_offset,
                                                        (unsigned long long)t * (unsigned long long)N +
                                                            (unsigned long long)j);
                    const double xn = mean + c.sd * uv;
                    const int bin = sv_bin(xn, lo, scale, kBins);
                    atomicAdd(&s_hist[bin], 1);
                    xc[k] = xn;
                    pa[k] = a;
                    if (par_out) par_out[k] = perm[a];   // path storage: birth row of the parent
                    cb[k] = (unsigned short)bin;
                }
            }
            __syncthreads();
        }
        __syncthreads();
    }
    __syncthreads();
    for (int b = tid; b < kBins; b += 256) {
        const int v = s_hist[b];
        if (v) atomicAdd(&hist_out[b], v);
    }
    near = near + __shfl_xor_sync(kFullMask, near, 16);
    near = near + __shfl_xor_sync(kFullMask, near, 8);
    near = near + __shfl_xor_sync(kFullMask, near, 4);
    near = near + __shfl_xor_sync(kFullMask, near, 2);
    near = near + __shfl_xor_sync(kFullMask, near, 1);
    if (lane == 0) s_near[warp] = near;
    __syncthreads();
    if (tid == 0) {
        int tot = 0;
        for (int w = 0; w < 8; ++w) tot += s_near[w];
        if (tot) atomicAdd(&st->near_ties, (unsigned long long)tot);
    }
    if (!fuse_plan) return;
    // One rank: every child stays here, so the plan is two exclusive scans over the 4096 bins
    // (arrivals before a bin, fine bins before a bin).  The last block to finish does it
    // instead of a launch of its own (split_plan_kernel).
    __shared__ int s_lastc;
    __threadfence();
    __syncthreads();
    if (tid == 0) {
        const unsigned int tk = atomicAdd(&st->ticket_c, 1u);
        s_lastc = (tk == gridDim.x - 1) ? 1 : 0;
        if (s_lastc) st->ticket_c = 0;
    }
    __syncthreads();
    if (!s_lastc) return;
    __threadfence();
    constexpr int BPT = kBins / 256;
    // the global histogram into shared memory with coalesced, independent loads (the block's own
    // histogram has been flushed), then every thread takes BPT consecutive bins
    for (int b = tid; b < kBins; b += 256) s_hist[b] = __ldcg(&hist_out[b]);
    __shared__ int s_wa[8], s_wb[8];
    __syncthreads();
    int run = 0, nfrun = 0;
    const int b0 = tid * BPT;
    for (int k = 0; k < BPT; ++k) {
        const int g = s_hist[b0 + k];
        run += g;
        nfrun += max(1, (g + kFine - 1) / kFine);
    }
    const int incl = warp_incl_scan(run, lane), fincl = warp_incl_scan(nfrun, lane);
    if (lane == 31) {
        s_wa[warp] = incl;
        s_wb[warp] = fincl;
    }
    __syncthreads();
    int before = incl - run, fbefore = fincl - nfrun, total = 0, ftotal = 0;
    for (int w = 0; w < 8; ++w) {
        if (w < warp) {
            before += s_wa[w];
            fbefore += s_wb[w];
        }
        total += s_wa[w];
        ftotal += s_wb[w];
    }
    for (int k = 0; k < BPT; ++k) {
        const int g = s_hist[b0 + k];
        const int nf = max(1, (g + kFine - 1) / kFine);
        cstart[b0 + k] = before;
        nfc[b0 + k] = nf;
        fstart[b0 + k] = fbefore;
        before += g;
        fbefore += nf;
    }
    if (tid == 0) {
        fstart[kBins] = ftotal;
        st->send_cnt[0] = total;
        st->send_off[0] = 0;
        st->recv_cnt[0] = total;
        st->cursor[0] = 0;
        if (total > st->cap) atomicOr(&st->status, 8);
        st->n_arrivals = total;
        st->NF = ftotal;
    }
}

// ---------------------------------------------------------------------------------------------
// plan: one block of 1024 threads over the 4096 coarse bins (thread = 4 consecutive bins)
// ---------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(1024) split_plan_kernel(SplitState* __restrict__ st,
                                                          const int* __restrict__ H,
                                                          int* __restrict__ dest, int* __restrict__ nfc,
                                                          int* __restrict__ fstart,
                                                          int* __restrict__ cstart,
                                                          int* __restrict__ counts) {
    __shared__ unsigned long long s_first;
    __shared__ long long s_w[32];
    __shared__ int s_wi[32];
    __shared__ int s_send[kMaxWorld], s_recv[kMaxWorld];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int G = st->world, me = st->rank;
    if (tid < kMaxWorld) {
        s_send[tid] = 0;
        s_recv[tid] = 0;
    }
    if (tid == 0) s_first = ~0ull;
    long long gc[4], bef[4], run = 0;
#pragma unroll
    for (int k = 0; k < 4; ++k) {
        const int b = tid * 4 + k;
        long long s = 0;
        for (int r = 0; r < G; ++r) s += H[r * kBins + b];
        gc[k] = s;
        run += s;
    }
    // block-wide exclusive scan of `run`
    long long incl = run;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
        const long long o = __shfl_up_sync(kFullMask, incl, d);
        if (lane >= d) incl += o;
    }
    if (lane == 31) s_w[warp] = incl;
    __syncthreads();
    long long woff = 0, total = 0;
    for (int w = 0; w < 32; ++w) {
        if (w < warp) woff += s_w[w];
        total += s_w[w];
    }
    long long before = woff + incl - run;
    int mydest[4], mynf[4], nfrun = 0;
#pragma unroll
    for (int k = 0; k < 4; ++k) {
        const int b = tid * 4 + k;
        long long d = (total > 0) ? (before * G) / total : 0;
        if (d > G - 1) d = G - 1;
        mydest[k] = (int)d;
        dest[b] = (int)d;
        bef[k] = before;
        if ((int)d == me) atomicMin(&s_first, (unsigned long long)before);
        const int hs = H[me * kBins + b];
        if (hs) atomicAdd(&s_send[d], hs);
        int nf = 0;
        if ((int)d == me) {
            for (int r = 0; r < G; ++r) {
                const int h = H[r * kBins + b];
                if (h) atomicAdd(&s_recv[r], h);
            }
            nf = (int)((gc[k] + kFine - 1) / kFine);
            if (nf < 1) nf = 1;
        }
        mynf[k] = nf;
        nfrun += nf;
        before += gc[k];
    }
    __syncthreads();
    int iincl = warp_incl_scan(nfrun, lane);
    if (lane == 31) s_wi[warp] = iincl;
    __syncthreads();
    int iwoff = 0, nftot = 0;
    for (int w = 0; w < 32; ++w) {
        if (w < warp) iwoff += s_wi[w];
        nftot += s_wi[w];
    }
    int fbefore = iwoff + iincl - nfrun;
#pragma unroll
    for (int k = 0; k < 4; ++k) {
        const int b = tid * 4 + k;
        nfc[b] = mynf[k];
        fstart[b] = fbefore;
        cstart[b] = (mydest[k] == me) ? (int)(bef[k] - (long long)s_first) : 0;
        fbefore += mynf[k];
    }
    if (tid == 0) {
        fstart[kBins] = nftot;
        int so = 0, narr = 0;
        for (int d = 0; d < G; ++d) {
            st->send_cnt[d] = s_send[d];
            st->send_off[d] = so;
            st->recv_cnt[d] = s_recv[d];
            st->cursor[d] = 0;
            counts[d] = s_send[d];
            counts[G + d] = s_recv[d];
            so += s_send[d];
            narr += s_recv[d];
        }
        if (narr > st->cap) atomicOr(&st->status, 8);
        st->n_arrivals = narr;
        st->NF = nftot;
        counts[2 * G] = narr;
        counts[2 * G + 1] = st->nc;
        counts[2 * G + 2] = nftot;
        counts[2 * G + 3] = st->status;
    }
}

// ---------------------------------------------------------------------------------------------
// pack: children grouped by destination rank; record = (value, parent's value, parent's lagged
// ancestors ...) -- the particle_history shift of :334-341 carried with the particle
// ---------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) split_pack_kernel(
    SplitState* __restrict__ st, const double* __restrict__ xc, const int* __restrict__ pa,
    const unsigned short* __restrict__ cb, const int* __restrict__ dest, const int* __restrict__ perm,
    const double* __restrict__ rec, double* __restrict__ send, double* __restrict__ send_keys,
    double* __restrict__ self_rec, double* __restrict__ self_keys) {
    __shared__ int s_cnt[kMaxWorld], s_base[kMaxWorld];
    const int tid = threadIdx.x, lane = tid & 31;
    const int nc = st->nc, G = st->world, LR = st->LR;
    // self_rec / self_keys (optional): the receive buffers of THIS rank.  Children that stay on this rank are
    // written straight to their arrival slots (behind the arrivals from the ranks in front), so the exchange
    // moves only what crosses ranks.  Slots of such children are encoded as -2 - arrival slot.
    long long self_off = 0;
    if (self_rec)
        for (int r = 0; r < st->rank; ++r) self_off += st->recv_cnt[r];
    const int me = self_rec ? st->rank : -1;
    for (long long base = (long long)blockIdx.x * 256; base < nc; base += (long long)gridDim.x * 256) {
        const long long k = base + tid;
        const bool valid = k < nc;
        long long slot = -1;
        if (G == 1) {
            slot = valid ? k : -1;                  // one rank: birth order is arrival order
        } else {
            if (tid < G) s_cnt[tid] = 0;
            __syncthreads();
            int d = 0, r = 0;
            if (valid) {
                d = dest[cb[k]];
                r = atomicAdd(&s_cnt[d], 1);
            }
            __syncthreads();
            if (tid < G && s_cnt[tid] > 0) s_base[tid] = atomicAdd(&st->cursor[tid], s_cnt[tid]);
            __syncthreads();
            if (valid) slot = (d == me) ? -2 - (self_off + s_base[d] + r) : st->send_off[d] + s_base[d] + r;
            __syncthreads();
        }
        const double xv = valid ? xc[k] : 0.0;
        if (send_keys && valid) {   // values alone, for the receiver's sort
            if (slot >= 0) send_keys[slot] = xv;
            else if (self_keys) self_keys[-2 - slot] = xv;
        }
        if (LR == 1) {
            if (valid) {
                if (slot >= 0) send[slot] = xv;
                else self_rec[-2 - slot] = xv;
            }
            continue;
        }
        // the warp copies its 32 records together: consecutive lanes move consecutive doubles of
        // a record, so both the parent-row reads and the record writes are 72 / 80-byte runs
        const long long row = valid ? (long long)perm[pa[k]] : 0;
        for (int idx = lane; idx < 32 * LR; idx += 32) {
            const int cc = idx / LR, m = idx - cc * LR;
            const long long sc = __shfl_sync(kFullMask, slot, cc);
            const long long rc = __shfl_sync(kFullMask, row, cc);
            const double xvc = __shfl_sync(kFullMask, xv, cc);
            if (sc >= 0) send[(size_t)sc * LR + m] = (m == 0) ? xvc : rec[(size_t)rc * LR + m - 1];
            else if (sc <= -2) self_rec[(size_t)(-2 - sc) * LR + m] = (m == 0) ? xvc : rec[(size_t)rc * LR + m - 1];
        }
    }
}

// ---------------------------------------------------------------------------------------------
// sort of the arrivals
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ int fine_bin(double x, double lo, double scale, const int* __restrict__ nfc,
                                        const int* __restrict__ fstart) {
    const int cbin = sv_bin(x, lo, scale, kBins);
    const double tt = (x - lo) * scale;
    double frac = tt - (double)cbin;
    const int nf = nfc[cbin];
    int sub = (!(frac > 0.0)) ? 0 : (int)(frac * (double)nf);
    if (sub > nf - 1) sub = nf - 1;
    if (sub < 0) sub = 0;
    return fstart[cbin] + sub;
}

__global__ void split_fine_hist_kernel(const SplitState* __restrict__ st, const double* __restrict__ recn,
                                       const double* __restrict__ keys, int n, int LR,
                                       const int* __restrict__ nfc,
                                       const int* __restrict__ fstart, int* __restrict__ fcnt,
                                       int* __restrict__ rnk, int* __restrict__ fb) {
    const double lo = st->lo, scale = st->scale;
    for (int e = blockIdx.x * blockDim.x + threadIdx.x; e < n; e += gridDim.x * blockDim.x) {
        const double x = keys ? keys[e] : recn[(size_t)e * LR];
        const int f = fine_bin(x, lo, scale, nfc, fstart);
        rnk[e] = atomicAdd(&fcnt[f], 1);
        fb[e] = f;
    }
}

// start slot of every fine bin: arrivals before its coarse bin (known exactly from the gathered
// histograms) + a warp scan over the fine bins of that coarse bin.  One warp per coarse bin.
__global__ void __launch_bounds__(256) split_fine_offsets_kernel(const int* __restrict__ nfc,
                                                                 const int* __restrict__ fstart,
                                                                 const int* __restrict__ cstart,
                                                                 const int* __restrict__ fcnt,
                                                                 int* __restrict__ fst) {
    const int cbin = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
    if (cbin >= kBins) return;
    const int nf = nfc[cbin];
    if (nf == 0) return;
    const int f0 = fstart[cbin];
    int carry = cstart[cbin];
    for (int i0 = 0; i0 < nf; i0 += 32) {
        const int i = i0 + lane;
        const int v = (i < nf) ? fcnt[f0 + i] : 0;
        const int incl = warp_incl_scan(v, lane);
        if (i < nf) fst[f0 + i] = carry + incl - v;
        carry += __shfl_sync(kFullMask, incl, 31);
    }
    if (lane == 0) fst[f0 + nf] = carry;   // == first slot of the next coarse bin (same value)
}

struct __align__(16) SortEntry {
    double key;
    int idx, fb;
};

__global__ void split_scatter_kernel(const double* __restrict__ recn, const double* __restrict__ keys,
                                     int n, int LR, const int* __restrict__ fst,
                                     const int* __restrict__ rnk, const int* __restrict__ fb,
                                     SortEntry* __restrict__ ent) {
    for (int e = blockIdx.x * blockDim.x + threadIdx.x; e < n; e += gridDim.x * blockDim.x) {
        const int f = fb[e];
        SortEntry v;
        v.key = keys ? keys[e] : recn[(size_t)e * LR];
        v.idx = e;
        v.fb = f;
        ent[fst[f] + rnk[e]] = v;   // one 16-byte store: one sector per particle
    }
}

// exact order inside each fine bin: (value, arrival index); any correct sort reproduces the
// reference's qsort order when values are distinct (SURVEY 7 "hard parts"); equal values counted
__global__ void split_rank_kernel(SplitState* __restrict__ st, const SortEntry* __restrict__ ent,
                                  const int* __restrict__ fst, int* __restrict__ fcnt, int n,
                                  double* __restrict__ xs, int* __restrict__ perm) {
    int mx = 0, ties = 0;
    for (int s = blockIdx.x * blockDim.x + threadIdx.x; s < n; s += gridDim.x * blockDim.x) {
        const SortEntry me = ent[s];
        const int f = me.fb;
        const int b = fst[f], e = fst[f + 1];
        const double v = me.key;
        const int oi = me.idx;
        int rank = 0;
        if (e - b <= kMaxBinRank) {
            for (int q = b; q < e; ++q) {
                const SortEntry o = ent[q];
                if (o.key < v) ++rank;
                else if (o.key == v && q != s) {
                    ++ties;
                    if (o.idx < oi) ++rank;
                }
            }
        } else {
            rank = s - b;
            atomicOr(&st->status, 16);
        }
        xs[b + rank] = v;
        perm[b + rank] = oi;
        mx = max(mx, e - b);
        fcnt[f] = 0;   // every counter that was touched is reset for the next step (no memset)
    }
    mx = warp_max(mx);
    if ((threadIdx.x & 31) == 0 && mx > 0) atomicMax(&st->max_bin, mx);
    if (ties) atomicAdd(&st->key_ties, (unsigned long long)ties);
}

// ---------------------------------------------------------------------------------------------
// path storage (one device): a generation is stored ONCE, in birth order, as value X[g][k] and
// parent row J[0][g][k]; nothing is copied when a particle has children.  Jump tables
// J[q][g][k] = row (in generation g - 2^q) of the ancestor 2^q steps back are extended by one
// random 4-byte read per table per particle-step.  The fixed-lag terms (:445-470) reach the
// ancestors lag-2 / lag-1 steps back through them.  Rings of depth R over the generations.
// ---------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) split_lineage_kernel(
    const SplitState* __restrict__ st, int t, int n, int lag, int R, int Q, const double* __restrict__ X,
    int* __restrict__ J, const double* __restrict__ obs, const double* __restrict__ params,
    const double* __restrict__ shift_arr, double* __restrict__ gpart) {
    __shared__ double red[5 * 32];
    const int tid = threadIdx.x;
    const size_t N = (size_t)n;
    SvConst c;
    sv_const_init(c, params);
    const bool grad = t >= lag;
    // (the shift of step t from the per-step array: the state's copy is overwritten by the
    // children kernel of step t + 1, which may already have run)
    const double shift = shift_arr[t], y = obs[t], ylag = grad ? obs[t - lag] : 0.0;   // Q5: obs[i - LAG]
    const int m = lag - 2;
    double acc[5] = {0.0, 0.0, 0.0, 0.0, 0.0};
    bool bad = false;
    for (int k = blockIdx.x * 256 + tid; k < n; k += gridDim.x * 256) {
        // extend the jump tables of generation t
        int jq[6];
        jq[0] = J[((size_t)0 * R + (t % R)) * N + k];
        for (int q = 1; q <= Q; ++q) {
            const int b = 1 << q, h = b >> 1;
            if (t >= b) {
                jq[q] = J[((size_t)(q - 1) * R + ((t - h) % R)) * N + jq[q - 1]];
                J[((size_t)q * R + (t % R)) * N + k] = jq[q];
            } else {
                jq[q] = 0;
            }
        }
        if (!grad) continue;
        // ancestor m = lag - 2 steps back: binary decomposition of m over the tables
        int r = k, g = t;
        for (int q = Q; q >= 0; --q) {
            const int b = 1 << q;
            if (m & b) {
                r = (g == t) ? jq[q] : J[((size_t)q * R + (g % R)) * N + r];
                g -= b;
            }
        }
        const double next = X[(size_t)(g % R) * N + r];
        const int rp = (g == t) ? jq[0] : J[((size_t)0 * R + (g % R)) * N + r];
        const double curr = X[(size_t)((g - 1) % R) * N + rp];
        double sh = exp(sv_logw(X[(size_t)(t % R) * N + k], y) - shift);
        if (!isfinite(sh)) {
            bad = true;
            sh = 0.0;
        }
        double sq, gg[4];
        sv_score_main(c, curr, next, ylag, sq, gg);
        acc[0] += sh * curr;
#pragma unroll
        for (int q = 0; q < 4; ++q) acc[1 + q] += gg[q] * sh;
    }
    if (bad) atomicOr(&((SplitState*)st)->status, 2);
    block_sum<5>(acc, red);
    if (tid < 5) gpart[(size_t)blockIdx.x * 8 + tid] = acc[tid];
}

// the last generation's lineage sums (no later weights phase picks them up)
__global__ void __launch_bounds__(256) split_lineage_reduce_kernel(const double* __restrict__ gpart,
                                                                   double* __restrict__ sums_row) {
    __shared__ double red[5 * 32];
    double late[5] = {0.0, 0.0, 0.0, 0.0, 0.0};
    for (int q = threadIdx.x; q < kLineageGrid; q += 256)
#pragma unroll
        for (int k = 0; k < 5; ++k) late[k] += gpart[(size_t)q * 8 + k];
    block_sum<5>(late, red);
    if (threadIdx.x < 5) sums_row[2 + threadIdx.x] = late[threadIdx.x];
}

// records [n][lag] of the FINAL generation (row = birth row): rec[k][idx] = value of the ancestor
// idx steps back -- what the tail terms (:540-562) read; built once by walking the parent rows
__global__ void split_build_records_kernel(int T, int n, int lag, int R, const double* __restrict__ X,
                                           const int* __restrict__ J, double* __restrict__ rec) {
    const size_t N = (size_t)n;
    for (int k = blockIdx.x * blockDim.x + threadIdx.x; k < n; k += gridDim.x * blockDim.x) {
        int r = k, g = T;
        for (int idx = 0; idx < lag; ++idx) {
            rec[(size_t)k * lag + idx] = X[(size_t)(g % R) * N + r];
            if (idx + 1 < lag) {
                r = J[(size_t)(g % R) * N + r];
                --g;
            }
        }
    }
}

// ---------------------------------------------------------------------------------------------
// tail (:540-562, Q6) on the final generation: wt[k][p] = normalised weight at global position
// (gstart + p) of generation nobs-1-k... see pmmh_svsplit_tail
//   part[i_rel][0] = sum_j W_T[j] ph[idx][j];  part[i_rel][1..4] = sum_j g_p W_i[j]
// one block per (i_rel, tile)
// ---------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) split_tail_kernel(
    const int* __restrict__ perm, const double* __restrict__ rec, int n, int LR, int nobs,
    const double* __restrict__ obs, const double* __restrict__ params, const double* __restrict__ wfinal,
    const double* __restrict__ wlag, long long wlag_stride, double* __restrict__ part, int ntiles) {
    __shared__ double red[5 * 32];
    const int tid = threadIdx.x;
    const int irel = blockIdx.y;                 // i = nobs - LR + irel, idx = LR - 1 - irel
    const int i = nobs - LR + irel, idx = LR - 1 - irel;
    SvConst c;
    sv_const_init(c, params);
    const double y1 = obs_wrap(obs, i - 1, nobs);
    double acc[5] = {0.0, 0.0, 0.0, 0.0, 0.0};
    const int base = blockIdx.x * kTile;
    for (int p = base + tid; p < min(n, base + kTile); p += blockDim.x) {
        const size_t row = (size_t)perm[p] * LR;
        const double curr = rec[row + idx];
        acc[0] += wfinal[p] * curr;
        if (idx >= 1) {
            const double next = rec[row + idx - 1];
            const double wi = wlag[(size_t)irel * wlag_stride + p];
            double sq, g[4];
            sv_score_tail(c, curr, next, y1, sq, g);
#pragma unroll
            for (int q = 0; q < 4; ++q) acc[1 + q] += g[q] * wi;
        }
    }
    block_sum<5>(acc, red);
    if (tid < 5) part[((size_t)irel * ntiles + blockIdx.x) * 8 + tid] = acc[tid];
}

__global__ void __launch_bounds__(256) split_tail_reduce_kernel(const double* __restrict__ part,
                                                                int ntiles, double* __restrict__ out) {
    __shared__ double red[5 * 32];
    const int irel = blockIdx.x, tid = threadIdx.x;
    double acc[5] = {0.0, 0.0, 0.0, 0.0, 0.0};
    for (int q = tid; q < ntiles; q += 256)
#pragma unroll
        for (int k = 0; k < 5; ++k) acc[k] += part[((size_t)irel * ntiles + q) * 8 + k];
    block_sum<5>(acc, red);
    if (tid < 5) out[irel * 8 + tid] = acc[tid];
}

// normalised weights of the local generation (for the tail): w[p] = sh[p] / S
__global__ void split_normalise_kernel(const double* __restrict__ sh, int n,
                                       const double* __restrict__ S_ptr, double* __restrict__ w) {
    const double S = *S_ptr;
    for (int p = blockIdx.x * blockDim.x + threadIdx.x; p < n; p += gridDim.x * blockDim.x)
        w[p] = sh[p] / S;
}

// ---------------------------------------------------------------------------------------------
// finish: O(T) assembly of the outputs from the rank-summed per-step sums
//   sums[t][0] = sum sh, [1] = sum sh x, [2] = sum sh curr, [3..6] = sum sh g
//   tail[irel][0] = smo term, [1..4] = gradient terms (already normalised weights)
// ---------------------------------------------------------------------------------------------
__global__ void split_finish_kernel(const double* __restrict__ sums, const double* __restrict__ shift,
                                    const double* __restrict__ xmin, const double* __restrict__ tail,
                                    const double* __restrict__ gather_last, int world,
                                    const double* __restrict__ params, int nobs, int LR, double n_total,
                                    double* __restrict__ log_like, double* __restrict__ filt,
                                    double* __restrict__ smo, double* __restrict__ grad,
                                    double* __restrict__ traj) {
    const int tid = blockIdx.x * blockDim.x + threadIdx.x;
    if (tid == 0) {
        double ll = 0.0;
        const double logn = log(n_total);
        for (int t = 1; t < nobs; ++t) ll += shift[t] + log(sums[t * 8]) - logn;   // :537
        log_like[0] = ll;
    }
    for (int t = tid; t < nobs; t += gridDim.x * blockDim.x) {
        filt[t] = sums[t * 8 + 1] / sums[t * 8];
        // Q10/Q11: traj[t] = X_t[0] for t >= 1, X_0 == mu
        double tr = (t == 0) ? params[0] : xmin[t];
        if (t == nobs - 1) {
            tr = INFINITY;
            for (int q = 0; q < world; ++q)
                if (gather_last[q * 4 + 1] > 0.0) tr = fmin(tr, gather_last[q * 4 + 2]);
        }
        traj[t] = tr;
        if (LR > 1) {
            // main loop terms land at tt = t - LR + 1 (:445-470); the tail adds to the same slots
            double s = 0.0, g[4] = {0.0, 0.0, 0.0, 0.0};
            const int src = t + LR - 1;   // time step whose weights produced slot t
            if (t >= 1 && src < nobs) {
                const double S = sums[src * 8];
                s = sums[src * 8 + 2] / S;
                for (int q = 0; q < 4; ++q) g[q] = sums[src * 8 + 3 + q] / S;
            }
            // tail (:540-562): i = nobs-LR+irel adds smo[i] and gradient[.][i-LR+1]
            if (tail) {
                const int irel_s = t - (nobs - LR);
                if (irel_s >= 0 && irel_s < LR) s += tail[irel_s * 8];
                const int irel_g = t + LR - 1 - (nobs - LR);
                if (irel_g >= 0 && irel_g < LR - 1)
                    for (int q = 0; q < 4; ++q) g[q] += tail[irel_g * 8 + 1 + q];
            }
            smo[t] = s;
            for (int q = 0; q < 4; ++q) grad[(size_t)q * nobs + t] = g[q];
        }
    }
}

// diag[] of a one-rank evaluation without a host round trip
__global__ void split_diag_kernel(const SplitState* __restrict__ st, long long* __restrict__ diag) {
    if (threadIdx.x == 0 && blockIdx.x == 0) {
        for (int k = 0; k < PMMH_DIAG_COUNT; ++k) diag[k] = 0;
        diag[PMMH_DIAG_NEAR_TIES] = (long long)st->near_ties;
        diag[PMMH_DIAG_MAX_BIN] = st->max_bin;
        diag[PMMH_DIAG_STATUS] = st->status ? 1 : 0;
        diag[PMMH_DIAG_KEY_TIES] = (long long)st->key_ties;
        diag[PMMH_DIAG_KERNEL] = 4;
        diag[PMMH_DIAG_FAST_INFO] = st->status;
    }
}

int check_ws(void* ws, size_t bytes, long long cap, long long capc, Layout* L) {
    if (!ws) return set_error(PMMH_ERR_INVALID, "svsplit: null workspace");
    *L = make_layout(cap, capc);
    if (bytes < L->total) return set_error(PMMH_ERR_WORKSPACE, "svsplit: workspace too small");
    return PMMH_OK;
}

#define SPLIT_CUDA(call)                                                \
    do {                                                                \
        cudaError_t e__ = (call);                                       \
        if (e__ != cudaSuccess) return pmmh::set_cuda_error(e__, #call); \
    } while (0)

int grid_for(long long n, int per_block) {
    long long g = (n + per_block - 1) / per_block;
    if (g < 1) g = 1;
    if (g > 148 * 8) g = 148 * 8;
    return (int)g;
}

struct SingleLayout {
    size_t split, xs, perm, xs2, perm2, recA, recB, sums, shift, xmin, gather, hist, keep, tail, total;
    size_t split_bytes;
};

SingleLayout make_single_layout(int nobs, long long n, int lag) {
    SingleLayout S;
    const size_t LR = lag;
    size_t o = 0;
    S.split_bytes = make_layout(n, n).total;
    S.split = o;   o += al(S.split_bytes);
    S.xs = o;      o += al((size_t)n * 8);
    S.perm = o;    o += al((size_t)n * 4);
    S.xs2 = o;     o += al((size_t)n * 8);
    S.perm2 = o;   o += al((size_t)n * 4);
    S.recA = o;    o += al((size_t)n * LR * 8);
    S.recB = o;    o += al((size_t)n * LR * 8);
    S.sums = o;    o += al((size_t)nobs * 8 * 8);
    S.shift = o;   o += al((size_t)nobs * 8);
    S.xmin = o;    o += al((size_t)nobs * 8);
    S.gather = o;  o += al(4 * 8);
    S.hist = o;    o += al((size_t)kBins * 4);
    S.keep = o;    o += al((size_t)n * LR * 8);
    S.tail = o;    o += al((size_t)LR * 8 * 8);
    S.total = o;
    return S;
}

}  // namespace

size_t sv_split_single_ws_bytes(int nobs, int n, int lag) { return make_single_layout(nobs, n, lag).total; }
bool sv_split_single_eligible(int nobs, int n, int lag) {
    return lag >= 2 && lag <= 63 && nobs >= 2 * lag && n >= 1;
}

}  // namespace pmmh

using namespace pmmh;

extern "C" {

int pmmh_svsplit_workspace_bytes(long long cap_particles, long long cap_children, size_t* bytes) {
    if (cap_particles < 1 || cap_children < 1 || cap_particles >= (1ll << 31) - 4096 ||
        cap_children >= (1ll << 31) - 4096 || !bytes)
        return set_error(PMMH_ERR_INVALID, "svsplit: capacities must be in [1, 2^31)");
    *bytes = make_layout(cap_particles, cap_children).total;
    return PMMH_OK;
}

int pmmh_svsplit_init(void* d_ws, size_t ws_bytes, long long n_total, int n_obs, int world, int rank,
                      int lag, long long cap_particles, long long cap_children, int n_local,
                      const double* d_params, double* d_xs, int* d_perm, double* d_rec, void* stream) {
    Layout L = Layout();
    if (int rc = check_ws(d_ws, ws_bytes, cap_particles, cap_children, &L)) return rc;
    if (world < 1 || world > kMaxWorld || rank < 0 || rank >= world || n_total < 1 || n_obs < 2 ||
        (lag != 0 && (lag < 2 || lag > 63)) || n_local < 0 || n_local > cap_particles)
        return set_error(PMMH_ERR_INVALID, "svsplit_init: bad sizes");
    cudaStream_t st = (cudaStream_t)stream;
    SplitState h;
    memset(&h, 0, sizeof(h));
    h.N = n_total;
    h.world = world;
    h.rank = rank;
    h.LR = lag == 0 ? 1 : lag;
    h.nobs = n_obs;
    h.cap = cap_particles;
    h.capc = cap_children;
    // the state travels as a kernel argument (copied at launch): no host buffer to keep alive, no
    // synchronisation -- the call is asynchronous on the stream like every other entry point
    split_set_state_kernel<<<1, 1, 0, st>>>((SplitState*)((char*)d_ws + L.state), h);
    SPLIT_CUDA(cudaMemsetAsync((char*)d_ws + L.fcnt, 0, (size_t)(L.nf_max + 1) * 4, st));
    if (n_local > 0)
        split_init_kernel<<<grid_for(n_local, 256), 256, 0, st>>>(d_xs, d_perm, d_rec, n_local, h.LR,
                                                                   d_params);
    SPLIT_CUDA(cudaGetLastError());
    return PMMH_OK;
}

static int weights_impl(void* d_ws, size_t ws_bytes, long long cap_particles, long long cap_children,
                        int t, int n_local, int lag, int n_obs, const double* d_obs,
                        const double* d_params, const double* d_xs, const int* d_perm,
                        const double* d_rec, double* d_sums, double* d_gather_send, double* d_sh_save,
                        void* stream, int path_storage) {
    Layout L = Layout();
    if (int rc = check_ws(d_ws, ws_bytes, cap_particles, cap_children, &L)) return rc;
    if (t < 0 || t >= n_obs || n_local < 0 || n_local > cap_particles)
        return set_error(PMMH_ERR_INVALID, "svsplit_weights: bad sizes");
    cudaStream_t st = (cudaStream_t)stream;
    char* ws = (char*)d_ws;
    SplitState* state = (SplitState*)(ws + L.state);
    const int LR = lag == 0 ? 1 : lag;
    const int ntiles = (n_local + kTile - 1) / kTile;
    const bool grad_t = lag > 0 && t >= lag;
    const bool grad = grad_t && !path_storage;   // gather variant; path storage: sums from the lineage kernel
    double* cumblk = (double*)(ws + L.cumblk);
    double* btot = (double*)(ws + L.btot);
    double* bpart = (double*)(ws + L.bpart);
    double* boff = (double*)(ws + L.boff);
    double* tlast = (double*)(ws + L.tlast);
    if (ntiles > 0) {
        if (grad)
            split_weights_kernel<true><<<ntiles, kTileThreads, 0, st>>>(state, d_xs, d_perm, d_rec, n_local, LR, d_obs,
                                                               t, lag, d_params, t == 0, cumblk, btot,
                                                               tlast, bpart, d_sh_save);
        else
            split_weights_kernel<false><<<ntiles, kTileThreads, 0, st>>>(state, d_xs, d_perm, d_rec, n_local, LR,
                                                                d_obs, t, lag, d_params, t == 0, cumblk, btot,
                                                                tlast, bpart, d_sh_save);
    }
    const bool late = path_storage && lag > 0 && t - 1 >= lag;
    const size_t gstride = al((size_t)kLineageGrid * 8 * 8);
    split_weights_finalize_kernel<<<1, 1024, 0, st>>>(
        state, d_xs, n_local, ntiles, btot, bpart,
        late ? (const double*)(ws + L.gpart + (size_t)((t - 1) & 1) * gstride) : nullptr,
        late ? d_sums + (size_t)(t - 1) * 8 : nullptr, boff, d_sums + (size_t)t * 8, d_gather_send,
        grad ? 7 : 1);
    (void)grad_t;
    SPLIT_CUDA(cudaGetLastError());
    return PMMH_OK;
}

int pmmh_svsplit_weights(void* d_ws, size_t ws_bytes, long long cap_particles, long long cap_children,
                         int t, int n_local, int lag, int n_obs, const double* d_obs,
                         const double* d_params, const double* d_xs, const int* d_perm,
                         const double* d_rec, double* d_sums, double* d_gather_send, double* d_sh_save,
                         void* stream) {
    return weights_impl(d_ws, ws_bytes, cap_particles, cap_children, t, n_local, lag, n_obs, d_obs, d_params,
                        d_xs, d_perm, d_rec, d_sums, d_gather_send, d_sh_save, stream, 0);
}

static int children_impl(void* d_ws, size_t ws_bytes, long long cap_particles, long long cap_children,
                         int t, int n_local, const double* d_obs, const double* d_params,
                         const double* d_rvr, const double* d_u, unsigned long long seed,
                         unsigned long long philox_offset, const double* d_gather, const double* d_xs,
                         int* d_hist_send, double* d_shift, double* d_xmin, void* stream,
                         double* xc_override, const int* perm, int* par_out, int fuse_plan = 0,
                         int u_pm_chunk = 0) {
    Layout L = Layout();
    if (int rc = check_ws(d_ws, ws_bytes, cap_particles, cap_children, &L)) return rc;
    if (t < 1 || n_local < 0) return set_error(PMMH_ERR_INVALID, "svsplit_children: bad sizes");
    cudaStream_t st = (cudaStream_t)stream;
    char* ws = (char*)d_ws;
    SplitState* state = (SplitState*)(ws + L.state);
    static thread_local bool attr_set[64] = {false};
    int dev = 0;
    SPLIT_CUDA(cudaGetDevice(&dev));
    const int smem = kStage * 8 + kBins * 4;
    if (dev >= 0 && dev < 64 && !attr_set[dev]) {
        SPLIT_CUDA(cudaFuncSetAttribute(split_children_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                        smem));
        attr_set[dev] = true;
    }
    SPLIT_CUDA(cudaMemsetAsync(d_hist_send, 0, (size_t)kBins * 4, st));
    split_children_kernel<<<148 * 4, 256, smem, st>>>(
        state, t, n_local, d_obs, d_params, d_rvr, d_u, seed, philox_offset, d_gather, d_xs,
        (const double*)(ws + L.cumblk), (const double*)(ws + L.boff), (const double*)(ws + L.tlast),
        xc_override ? xc_override : (double*)(ws + L.xc),
        (int*)(ws + L.pa), (unsigned short*)(ws + L.cb), d_hist_send, d_shift, d_xmin, perm, par_out,
        fuse_plan, (int*)(ws + L.nfc), (int*)(ws + L.fstart), (int*)(ws + L.cstart), u_pm_chunk);
    SPLIT_CUDA(cudaGetLastError());
    return PMMH_OK;
}

int pmmh_svsplit_children(void* d_ws, size_t ws_bytes, long long cap_particles, long long cap_children,
                          int t, int n_local, const double* d_obs, const double* d_params,
                          const double* d_rvr, const double* d_u, unsigned long long seed,
                          unsigned long long philox_offset, const double* d_gather, const double* d_xs,
                          int* d_hist_send, double* d_shift, double* d_xmin, void* stream) {
    return children_impl(d_ws, ws_bytes, cap_particles, cap_children, t, n_local, d_obs, d_params, d_rvr, d_u,
                         seed, philox_offset, d_gather, d_xs, d_hist_send, d_shift, d_xmin, stream, nullptr,
                         nullptr, nullptr);
}

int pmmh_svsplit_plan(void* d_ws, size_t ws_bytes, long long cap_particles, long long cap_children,
                      int world, const int* d_hist, int* h_counts, void* stream) {
    Layout L = Layout();
    if (int rc = check_ws(d_ws, ws_bytes, cap_particles, cap_children, &L)) return rc;
    cudaStream_t st = (cudaStream_t)stream;
    char* ws = (char*)d_ws;
    SplitState* state = (SplitState*)(ws + L.state);
    split_plan_kernel<<<1, 1024, 0, st>>>(state, d_hist, (int*)(ws + L.dest), (int*)(ws + L.nfc),
                                          (int*)(ws + L.fstart), (int*)(ws + L.cstart),
                                          (int*)(ws + L.counts));
    SPLIT_CUDA(cudaGetLastError());
    if (h_counts)
        SPLIT_CUDA(cudaMemcpyAsync(h_counts, ws + L.counts, (size_t)(2 * world + 4) * 4,
                                   cudaMemcpyDeviceToHost, st));
    return PMMH_OK;
}

int pmmh_svsplit_pack(void* d_ws, size_t ws_bytes, long long cap_particles, long long cap_children,
                      const int* d_perm, const double* d_rec, double* d_send, double* d_send_keys,
                      void* stream) {
    Layout L = Layout();
    if (int rc = check_ws(d_ws, ws_bytes, cap_particles, cap_children, &L)) return rc;
    cudaStream_t st = (cudaStream_t)stream;
    char* ws = (char*)d_ws;
    SplitState* state = (SplitState*)(ws + L.state);
    split_pack_kernel<<<148 * 8, 256, 0, st>>>(state, (const double*)(ws + L.xc), (const int*)(ws + L.pa),
                                               (const unsigned short*)(ws + L.cb),
                                               (const int*)(ws + L.dest), d_perm, d_rec, d_send,
                                               d_send_keys, nullptr, nullptr);
    SPLIT_CUDA(cudaGetLastError());
    return PMMH_OK;
}

// pmmh_svsplit_pack with the children that stay on this rank written straight into this rank's receive buffers
// (d_self_rec = the d_rec_new the sort will read, d_self_keys = its d_keys or NULL) at their arrival slots; the
// exchange that follows skips the self part (send / receive offsets of the other ranks are unchanged)
int pmmh_svsplit_pack_direct(void* d_ws, size_t ws_bytes, long long cap_particles, long long cap_children,
                             const int* d_perm, const double* d_rec, double* d_send, double* d_send_keys,
                             double* d_self_rec, double* d_self_keys, void* stream) {
    Layout L = Layout();
    if (int rc = check_ws(d_ws, ws_bytes, cap_particles, cap_children, &L)) return rc;
    if (!d_self_rec) return pmmh::set_error(PMMH_ERR_INVALID, "pmmh_svsplit_pack_direct: d_self_rec is required");
    if (d_send_keys && !d_self_keys) return pmmh::set_error(PMMH_ERR_INVALID, "pmmh_svsplit_pack_direct: d_self_keys is required with d_send_keys");
    cudaStream_t st = (cudaStream_t)stream;
    char* ws = (char*)d_ws;
    SplitState* state = (SplitState*)(ws + L.state);
    split_pack_kernel<<<148 * 8, 256, 0, st>>>(state, (const double*)(ws + L.xc), (const int*)(ws + L.pa),
                                               (const unsigned short*)(ws + L.cb),
                                               (const int*)(ws + L.dest), d_perm, d_rec, d_send,
                                               d_send_keys, d_self_rec, d_self_keys);
    SPLIT_CUDA(cudaGetLastError());
    return PMMH_OK;
}

int pmmh_svsplit_sort(void* d_ws, size_t ws_bytes, long long cap_particles, long long cap_children,
                      int n_arrivals, int n_fine, int lag, const double* d_rec_new, const double* d_keys,
                      int keys_are_children, double* d_xs, int* d_perm, void* stream) {
    Layout L = Layout();
    if (int rc = check_ws(d_ws, ws_bytes, cap_particles, cap_children, &L)) return rc;
    if (n_arrivals < 0 || n_arrivals > cap_particles || n_fine < 0 || n_fine > L.nf_max)
        return set_error(PMMH_ERR_INVALID, "svsplit_sort: bad sizes");
    if (n_arrivals == 0) return PMMH_OK;
    cudaStream_t st = (cudaStream_t)stream;
    char* ws = (char*)d_ws;
    SplitState* state = (SplitState*)(ws + L.state);
    const int LR = lag == 0 ? 1 : lag;
    int* fcnt = (int*)(ws + L.fcnt);
    int* fst = (int*)(ws + L.fst);
    int* rnk = (int*)(ws + L.rnk);
    int* fb = (int*)(ws + L.fb);
    SortEntry* ent = (SortEntry*)(ws + L.tkey);
    const int g = grid_for(n_arrivals, 256);
    // one rank: the arrivals ARE the children in birth order, their values are a dense array
    const double* keys = keys_are_children ? (const double*)(ws + L.xc) : d_keys;
    split_fine_hist_kernel<<<g, 256, 0, st>>>(state, d_rec_new, keys, n_arrivals, LR, (const int*)(ws + L.nfc),
                                              (const int*)(ws + L.fstart), fcnt, rnk, fb);
    split_fine_offsets_kernel<<<kBins * 32 / 256, 256, 0, st>>>((const int*)(ws + L.nfc),
                                                                (const int*)(ws + L.fstart),
                                                                (const int*)(ws + L.cstart), fcnt, fst);
    split_scatter_kernel<<<g, 256, 0, st>>>(d_rec_new, keys, n_arrivals, LR, fst, rnk, fb, ent);
    split_rank_kernel<<<g, 256, 0, st>>>(state, ent, fst, fcnt, n_arrivals, d_xs, d_perm);
    SPLIT_CUDA(cudaGetLastError());
    return PMMH_OK;
}

int pmmh_svsplit_normalise(const double* d_sh, int n_local, const double* d_total, double* d_w,
                           void* stream) {
    if (n_local <= 0) return PMMH_OK;
    split_normalise_kernel<<<grid_for(n_local, 256), 256, 0, (cudaStream_t)stream>>>(d_sh, n_local, d_total,
                                                                                      d_w);
    SPLIT_CUDA(cudaGetLastError());
    return PMMH_OK;
}

int pmmh_svsplit_tail(void* d_ws, size_t ws_bytes, long long cap_particles, long long cap_children,
                      int n_local, int lag, int n_obs, const double* d_obs, const double* d_params,
                      const int* d_perm, const double* d_rec, const double* d_w_final,
                      const double* d_w_lagged, long long w_lagged_stride, double* d_tail,
                      void* stream) {
    Layout L = Layout();
    if (int rc = check_ws(d_ws, ws_bytes, cap_particles, cap_children, &L)) return rc;
    if (lag < 2 || n_local < 0) return set_error(PMMH_ERR_INVALID, "svsplit_tail: bad sizes");
    cudaStream_t st = (cudaStream_t)stream;
    char* ws = (char*)d_ws;
    const int ntiles = (n_local + kTile - 1) / kTile;
    // scratch: tkey is free after the last sort (needs lag * ntiles * 8 doubles)
    double* part = (double*)(ws + L.tkey);
    if ((size_t)lag * (size_t)max(ntiles, 1) * 8 > (size_t)cap_particles)
        return set_error(PMMH_ERR_WORKSPACE, "svsplit_tail: scratch too small");
    SPLIT_CUDA(cudaMemsetAsync(d_tail, 0, (size_t)lag * 8 * 8, st));
    if (ntiles > 0) {
        dim3 grid(ntiles, lag);
        split_tail_kernel<<<grid, 256, 0, st>>>(d_perm, d_rec, n_local, lag, n_obs, d_obs, d_params,
                                                d_w_final, d_w_lagged, w_lagged_stride, part, ntiles);
        split_tail_reduce_kernel<<<lag, 256, 0, st>>>(part, ntiles, d_tail);
    }
    SPLIT_CUDA(cudaGetLastError());
    return PMMH_OK;
}

int pmmh_svsplit_finish(const double* d_sums, const double* d_shift, const double* d_xmin,
                        const double* d_tail, const double* d_gather_last, int world,
                        const double* d_params, int n_obs, int lag,
                        long long n_total, double* d_log_like, double* d_filt, double* d_smo,
                        double* d_gradient, double* d_traj, void* stream) {
    const int LR = lag == 0 ? 1 : lag;
    split_finish_kernel<<<grid_for(n_obs, 256), 256, 0, (cudaStream_t)stream>>>(
        d_sums, d_shift, d_xmin, d_tail, d_gather_last, world, d_params, n_obs, LR, (double)n_total,
        d_log_like, d_filt, d_smo, d_gradient, d_traj);
    SPLIT_CUDA(cudaGetLastError());
    return PMMH_OK;
}

int pmmh_svsplit_diag(void* d_ws, size_t ws_bytes, long long cap_particles, long long cap_children,
                      long long* h_diag) {
    Layout L = Layout();
    if (int rc = check_ws(d_ws, ws_bytes, cap_particles, cap_children, &L)) return rc;
    SplitState h;
    SPLIT_CUDA(cudaMemcpy(&h, (char*)d_ws + L.state, sizeof(h), cudaMemcpyDeviceToHost));
    for (int k = 0; k < PMMH_DIAG_COUNT; ++k) h_diag[k] = 0;
    h_diag[PMMH_DIAG_NEAR_TIES] = (long long)h.near_ties;
    h_diag[PMMH_DIAG_MAX_BIN] = h.max_bin;
    h_diag[PMMH_DIAG_STATUS] = h.status;
    h_diag[PMMH_DIAG_KEY_TIES] = (long long)h.key_ties;
    h_diag[PMMH_DIAG_KERNEL] = 4;
    return PMMH_OK;
}

}  // extern "C"

namespace pmmh {

namespace {
// The second stream of the current device and host thread, beside the caller's: a fork event and two join events
// (the records driver joins through join[0], the path driver alternates between both)
struct SideStream {
    cudaStream_t s = nullptr;
    cudaEvent_t fork = nullptr, join[2] = {nullptr, nullptr};
};

int side_stream(SideStream** out) {
    static thread_local SideStream sides[64];
    int dev = 0;
    SPLIT_CUDA(cudaGetDevice(&dev));
    if (dev < 0 || dev >= 64) return set_error(PMMH_ERR_NO_DEVICE, "device ordinal out of range");
    SideStream& side = sides[dev];
    if (!side.s) {
        SPLIT_CUDA(cudaStreamCreateWithFlags(&side.s, cudaStreamNonBlocking));
        for (cudaEvent_t* e : {&side.fork, &side.join[0], &side.join[1]})
            SPLIT_CUDA(cudaEventCreateWithFlags(e, cudaEventDisableTiming));
    }
    *out = &side;
    return PMMH_OK;
}

// The end of a one-device evaluation (layout WsLayout: SingleLayout or PathLayout): the weights kept for the last
// `lag` generations are normalised in place; then before_tail() enqueues what else the tail needs; then the tail,
// finish and diag kernels.  The tail kernel takes the lagged weights as one base and stride, [irel][p]: generation
// nobs - lag + irel sits in slot (r0 + irel) % lag, r0 = (nobs - lag) % lag, so unless r0 == 0 they are rotated into
// `scratch` (lag x n doubles, free by then).
template <class WsLayout, class BeforeTail>
int split_end(const SvCall& c, int nobs, int n, int lag, const WsLayout& S, const int* perm, const double* rec,
              double* scratch, BeforeTail before_tail) {
    char* ws = (char*)c.ws;
    void* sws = ws + S.split;
    double* sums = (double*)(ws + S.sums);
    double* keep = (double*)(ws + S.keep);
    double* tail = (double*)(ws + S.tail);
    int rc;
    for (int irel = 0; irel < lag; ++irel) {
        const int i = nobs - lag + irel;
        double* kp = keep + (size_t)(i % lag) * n;
        if ((rc = pmmh_svsplit_normalise(kp, n, sums + (size_t)i * 8, kp, c.stream))) return rc;
    }
    rc = before_tail();
    if (rc != PMMH_OK) return rc;
    const int r0 = (nobs - lag) % lag;
    double* wl = keep;
    if (r0 != 0) {
        wl = scratch;
        for (int irel = 0; irel < lag; ++irel)
            SPLIT_CUDA(cudaMemcpyAsync(wl + (size_t)irel * n, keep + (size_t)((r0 + irel) % lag) * n,
                                       (size_t)n * 8, cudaMemcpyDeviceToDevice, c.stream));
    }
    if ((rc = pmmh_svsplit_tail(sws, S.split_bytes, n, n, n, lag, nobs, c.obs, c.params, perm, rec,
                                wl + (size_t)(lag - 1) * n, wl, n, tail, c.stream)))
        return rc;
    if ((rc = pmmh_svsplit_finish(sums, (double*)(ws + S.shift), (double*)(ws + S.xmin), tail,
                                  (double*)(ws + S.gather), 1, c.params, nobs, lag, n, c.ll, c.filt, c.smo, c.grad,
                                  c.traj, c.stream)))
        return rc;
    split_diag_kernel<<<1, 32, 0, c.stream>>>((const SplitState*)((char*)sws + make_layout(n, n).state), c.diag);
    SPLIT_CUDA(cudaGetLastError());
    return PMMH_OK;
}

// ---- path storage on one device (algorithm 5) ------------------------------------------------
struct PathLayout {
    size_t split, xs, perm, X, J, sums, shift, xmin, gather, hist, keep, tail, rec, total, split_bytes;
    int R, Q;
};

PathLayout make_path_layout(int nobs, long long n, int lag) {
    PathLayout P;
    P.R = lag + 1;
    P.Q = 0;
    while ((2 << P.Q) <= lag - 2) ++P.Q;      // largest q with 2^q <= lag - 2 (0 when lag <= 3)
    size_t o = 0;
    P.split_bytes = make_layout(n, n).total;
    P.split = o;   o += al(P.split_bytes);
    P.xs = o;      o += al((size_t)n * 8);
    P.perm = o;    o += al((size_t)n * 4);
    P.X = o;       o += al((size_t)P.R * n * 8);
    P.J = o;       o += al((size_t)(P.Q + 1) * P.R * n * 4);
    P.sums = o;    o += al((size_t)nobs * 8 * 8);
    P.shift = o;   o += al((size_t)nobs * 8);
    P.xmin = o;    o += al((size_t)nobs * 8);
    P.gather = o;  o += al(4 * 8);
    P.hist = o;    o += al((size_t)kBins * 4);
    P.keep = o;    o += al((size_t)n * lag * 8);
    P.tail = o;    o += al((size_t)lag * 8 * 8);
    P.rec = o;     o += al((size_t)n * lag * 8);
    P.total = o;
    return P;
}
}  // namespace

size_t sv_split_path_ws_bytes(int nobs, int n, int lag) { return make_path_layout(nobs, n, lag).total; }

// The whole evaluation on ONE device (world = 1): the same phases, no exchange, no host
// synchronisation -- T x 11 kernel launches on c.stream.  Returns a PMMH_* status.
int sv_split_single_run(const SvCall& c, int nobs, int n, int lag) {
    if (!sv_split_single_eligible(nobs, n, lag)) return set_error(PMMH_ERR_INVALID, "split kernels: sizes not eligible");
    const SingleLayout S = make_single_layout(nobs, n, lag);
    if (c.ws_bytes < S.total) return set_error(PMMH_ERR_WORKSPACE, "split kernels: workspace too small");
    const double *d_obs = c.obs, *d_params = c.params, *d_rvr = c.rvr, *d_u = c.u;
    const cudaStream_t st = c.stream;
    char* ws = (char*)c.ws;
    void* sws = ws + S.split;
    const size_t sb = S.split_bytes;
    double* xs = (double*)(ws + S.xs);
    int* perm = (int*)(ws + S.perm);
    double* xs_next = (double*)(ws + S.xs2);
    int* perm_next = (int*)(ws + S.perm2);
    double* rec = (double*)(ws + S.recA);
    double* rec_next = (double*)(ws + S.recB);
    double* sums = (double*)(ws + S.sums);
    double* shift = (double*)(ws + S.shift);
    double* xmin = (double*)(ws + S.xmin);
    double* gather = (double*)(ws + S.gather);
    int* hist = (int*)(ws + S.hist);
    double* keep = (double*)(ws + S.keep);
    const int nf_bound = (int)(n / kFine + kBins);
    int rc;
    // pack (record traffic, DRAM bound) and the sort (latency / L2 bound) both depend only on
    // the plan: they run side by side on two streams
    SideStream* side = nullptr;
    if ((rc = side_stream(&side))) return rc;
    SPLIT_CUDA(cudaMemsetAsync(sums, 0, (size_t)nobs * 8 * 8, st));
    if ((rc = pmmh_svsplit_init(sws, sb, n, nobs, 1, 0, lag, n, n, n, d_params, xs, perm, rec, st))) return rc;
    if ((rc = pmmh_svsplit_weights(sws, sb, n, n, 0, n, lag, nobs, d_obs, d_params, xs, perm, rec, sums, gather,
                                   nullptr, st)))
        return rc;
    for (int t = 1; t < nobs; ++t) {
        if ((rc = pmmh_svsplit_children(sws, sb, n, n, t, n, d_obs, d_params, d_rvr, d_u, 0, 0, gather, xs, hist,
                                        shift, xmin, st)))
            return rc;
        if ((rc = pmmh_svsplit_plan(sws, sb, n, n, 1, hist, nullptr, st))) return rc;
        SPLIT_CUDA(cudaEventRecord(side->fork, st));
        SPLIT_CUDA(cudaStreamWaitEvent(side->s, side->fork, 0));
        if ((rc = pmmh_svsplit_pack(sws, sb, n, n, perm, rec, rec_next, nullptr, side->s))) return rc;
        SPLIT_CUDA(cudaEventRecord(side->join[0], side->s));
        double* tmp = rec;
        rec = rec_next;
        rec_next = tmp;
        // the sort reads the dense child values and writes xs / perm of the NEW generation: pack
        // still reads perm of the OLD one, so the new order goes to the alternate buffers
        if ((rc = pmmh_svsplit_sort(sws, sb, n, n, n, nf_bound, lag, rec, nullptr, 1, xs_next, perm_next, st))) return rc;
        SPLIT_CUDA(cudaStreamWaitEvent(st, side->join[0], 0));
        { double* tx = xs; xs = xs_next; xs_next = tx; int* tp = perm; perm = perm_next; perm_next = tp; }
        double* kp = (t >= nobs - lag) ? keep + (size_t)(t % lag) * n : nullptr;
        if ((rc = pmmh_svsplit_weights(sws, sb, n, n, t, n, lag, nobs, d_obs, d_params, xs, perm, rec, sums,
                                       gather, kp, st)))
            return rc;
    }
    // the alternate record buffer is free now
    return split_end(c, nobs, n, lag, S, perm, rec, rec_next, [] { return (int)PMMH_OK; });
}

int sv_split_path_run(const SvCall& c, int nobs, int n, int lag) {
    if (!sv_split_single_eligible(nobs, n, lag)) return set_error(PMMH_ERR_INVALID, "split kernels: sizes not eligible");
    const PathLayout P = make_path_layout(nobs, n, lag);
    if (c.ws_bytes < P.total) return set_error(PMMH_ERR_WORKSPACE, "split kernels: workspace too small");
    const double *d_obs = c.obs, *d_params = c.params, *d_rvr = c.rvr, *d_u = c.u;
    const int u_pm_chunk = c.slot;
    const cudaStream_t st = c.stream;
    char* ws = (char*)c.ws;
    void* sws = ws + P.split;
    const size_t sb = P.split_bytes;
    const int R = P.R, Q = P.Q;
    double* xs = (double*)(ws + P.xs);
    int* perm = (int*)(ws + P.perm);
    double* X = (double*)(ws + P.X);
    int* J = (int*)(ws + P.J);
    double* sums = (double*)(ws + P.sums);
    double* shift = (double*)(ws + P.shift);
    double* xmin = (double*)(ws + P.xmin);
    double* gather = (double*)(ws + P.gather);
    int* hist = (int*)(ws + P.hist);
    double* keep = (double*)(ws + P.keep);
    double* rec = (double*)(ws + P.rec);
    const Layout L = make_layout(n, n);
    SplitState* state = (SplitState*)((char*)sws + L.state);
    const int nf_bound = (int)(n / kFine + kBins);
    int rc;
    SideStream* side = nullptr;
    if ((rc = side_stream(&side))) return rc;
    const size_t gstride = al((size_t)kLineageGrid * 8 * 8);
    SPLIT_CUDA(cudaMemsetAsync(sums, 0, (size_t)nobs * 8 * 8, st));
    // generation 0: xs = mu, perm = identity, X[0] = mu (the LR = 1 "records" of init are X[0])
    if ((rc = pmmh_svsplit_init(sws, sb, n, nobs, 1, 0, 0, n, n, n, d_params, xs, perm, X, st))) return rc;
    if ((rc = weights_impl(sws, sb, n, n, 0, n, lag, nobs, d_obs, d_params, xs, perm, nullptr, sums, gather,
                           nullptr, st, 1)))
        return rc;
    for (int t = 1; t < nobs; ++t) {
        double* Xt = X + (size_t)(t % R) * n;
        int* J1t = J + (size_t)(t % R) * n;
        // host-streamed u: d_u holds particle-major chunks of u_pm_chunk time steps that the copy
        // engine is still filling; wait for the chunk of this step when it is entered
        const double* ut = d_u;
        if (u_pm_chunk) {
            if (t == 1 || t % u_pm_chunk == 0) SPLIT_CUDA(cudaStreamWaitEvent(st, c.slot_ready[t / u_pm_chunk], 0));
            ut = d_u + (size_t)(t / u_pm_chunk) * (size_t)n * (size_t)u_pm_chunk;
        }
        if ((rc = children_impl(sws, sb, n, n, t, n, d_obs, d_params, d_rvr, ut, c.seed, c.philox_offset, gather, xs, hist, shift,
                                xmin, st, Xt, perm, J1t, 1, u_pm_chunk)))
            return rc;
        // jump tables + fixed-lag sums (birth order) on the second stream.  They depend only on the
        // children and feed only outputs, so they get a whole step of slack: the weights phase of
        // step t picks up the sums of generation t - 1 (its ring slots stay untouched until t + lag)
        SPLIT_CUDA(cudaEventRecord(side->fork, st));
        SPLIT_CUDA(cudaStreamWaitEvent(side->s, side->fork, 0));
        split_lineage_kernel<<<kLineageGrid, 256, 0, side->s>>>(
            state, t, n, lag, R, Q, X, J, d_obs, d_params, shift,
            (double*)((char*)sws + L.gpart + (size_t)(t & 1) * gstride));
        SPLIT_CUDA(cudaEventRecord(side->join[t & 1], side->s));
        if ((rc = pmmh_svsplit_sort(sws, sb, n, n, n, nf_bound, 0, Xt, Xt, 0, xs, perm, st))) return rc;
        if (t > 1) SPLIT_CUDA(cudaStreamWaitEvent(st, side->join[(t - 1) & 1], 0));
        double* kp = (t >= nobs - lag) ? keep + (size_t)(t % lag) * n : nullptr;
        if ((rc = weights_impl(sws, sb, n, n, t, n, lag, nobs, d_obs, d_params, xs, perm, nullptr, sums, gather,
                               kp, st, 1)))
            return rc;
    }
    // the tail waits for the sums of the last generation's lineage kernel and reads records of the final
    // generation, built once from the stored paths; X is free by then and large enough (R > lag rows)
    return split_end(c, nobs, n, lag, P, perm, rec, X, [&]() -> int {
        SPLIT_CUDA(cudaStreamWaitEvent(st, side->join[(nobs - 1) & 1], 0));
        if (nobs - 1 >= lag)
            split_lineage_reduce_kernel<<<1, 256, 0, st>>>(
                (const double*)((char*)sws + L.gpart + (size_t)((nobs - 1) & 1) * gstride),
                sums + (size_t)(nobs - 1) * 8);
        split_build_records_kernel<<<grid_for(n, 256), 256, 0, st>>>(nobs - 1, n, lag, R, X, J, rec);
        return PMMH_OK;
    });
}
}  // namespace pmmh
