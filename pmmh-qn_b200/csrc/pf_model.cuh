// pf_model.cuh -- the device-function interface a scalar-state model implements to run on the
// chain kernel (sv_chain.cu) and the grid kernel (sv_grid.cu): the three things the reference tells a user to change when porting
// its Cython particle smoother to another model (/root/reference/python/README.md:73-76:
// "how the propagation and weighting of particles is carried out as well as the gradients of the
// log joint distribution of states and measurements").  Everything else -- sorted correlated
// systematic resampling, the counting sort, cumulative weights, fixed-lag bookkeeping, the tail --
// is model independent and lives in the kernel; kPairing picks how the kernel pairs the fixed-lag score terms.
//
// A model M provides (all __device__, fp64, no contraction):
//   M::kId                               its model id (PMMH_MODEL_*, include/pmmh_qn.h)
//   M::Filter                            the model whose filter instantiation the filter entries run (itself, or
//                                        the model it adds a gradient to)
//   M::Gradient                          the model whose smoother instantiation a call without the Hessian runs
//                                        (itself, or the model it adds a Hessian to)
//   M::kHessian                          constexpr: the kernels have its Hessian branch (the SV model: the
//                                        reference's, Pairing::Reference; models 6 and 8: the generic one, grid kernel)
//   struct M::Const                      constants derived from the parameter vector (<= 4 doubles)
//   M::init(Const&, const double* par)
//   M::initial_state(c)                  value of every particle of generation 0 (the reference's
//                                        flps starts all particles at one point, Q1)
//   M::propagate(c, x_parent, y_prev, u) child value; u = the particle's standard normal
//                                        (SV: stochastic_volatility.pyx:354-358)
//   M::prop_mean(c, x_parent, y_prev)    the same split as mean + sd * u: propagate(c, xp, y, u) ==
//   M::prop_sd(c)                        prop_mean(c, xp, y) + prop_sd(c) * u bit for bit (the grid
//                                        kernel stores the mean with the parent and predicts the
//                                        children's value range from its weighted moments)
//   M::child_range(c, xmin, xmax, y_prev, nsd, lo, hi)
//                                        an interval holding the children of parents in
//                                        [xmin, xmax] up to nsd innovation sd (sort-bin range)
//   M::logw(c, x, y)                     log observation density up to the reference's constant
//                                        (SV: :427-437)
//   M::logw_max(c, lo, hi, y)            an upper bound of logw on [lo, hi] that is attained or
//                                        nearly so (the shift of the weights; any value cancels)
//   M::score_main(c, curr, next, y, g)   the 4 score terms of the pair (curr, next) in the main loop
//   M::score_tail(c, curr, next, y, g)   the same in the tail loop
//   M::kScoreIsZero                      constexpr: score_main / score_tail are identically 0 (the
//                                        grid kernel then skips the calls; the smoother still runs)
//   M::kPairing                          constexpr: how the fixed-lag terms are paired (below)
//   M::score_last(c, x, y_next, g)       (Pairing::Predictive only) the final generation's term
//   M::hess_main(c, curr, next, y, h)    (generic Hessian branch only) the second derivatives of score_main's term:
//   M::hess_last(c, x, y_next, h)        10 entries, the upper triangle of the 4 x 4 matrix row by row ((0,0), (0,1),
//                                        (0,2), (0,3), (1,1), .. (3,3)); and of score_last's term
//   M::score_first(c, x1, y0, g)         (optional, Pairing::Predictive) the term of the pair (x_0, x_1) in place of
//   M::hess_first(c, x1, y0, h)          score_main / hess_main: for a model whose initial state depends on the
//                                        parameters, the total derivative through x_0 = initial_state (pair_score)
// A new model is such a struct plus its entry in Models at the end of this file, and its id in include/pmmh_qn.h.
//
// Pairing::Reference (the SV model, parity with the reference): the reference's quirks Q5 / Q6.  The main loop
// at step i >= LAG adds the pair (x_tt, x_tt+1), tt = i - LAG + 1, with y = obs[tt - 1] (score_main, Q5) into slot tt;
// the tail i = NOBS-LAG .. NOBS-1 adds smo[i] under the final weights and the pair (x_i, x_i+1) with y = obs[i - 1]
// wrapped (score_tail, Q6, :548-557, another operation order) under the weights of generation i into slot i - LAG + 1.
// Pairing::Exact (models of no reference): the pair (x_t, x_t+1), t = 0 .. NOBS-2,
// contributes d/dtheta log p(x_t+1 | x_t) + d/dtheta log p(y_t+1 | x_t+1) once, with y = obs[t + 1], weighted by the
// generation at which it is read: W_{t+LAG-1} in the main loop (steps i >= LAG - 1; the pair t = 0 has curr =
// initial_state for every particle, Q1), W_{NOBS-1} in the tail (t = NOBS-LAG+1 .. NOBS-2).  Gradient slot s holds
// step s's contribution (the pair (x_s-1, x_s)); slot 0 is 0.  smo[t] = the weighted mean of x_t under the same
// weights, every slot written once: the tail starts one step after the last main-loop slot.
// Pairing::Predictive: the same pairs, read under the same weights, but the pair (x_t, x_t+1) reads y = obs[t] and
// fills slot t; the final generation adds score_last(x_NOBS-1, obs[NOBS-1]) under W_{NOBS-1} into slot NOBS-1.  obs[t]
// is the observation the transition x_t -> x_t+1 is conditioned on: the leverage observation of a bootstrap filter
// whose propagation reads obs[t] (model 8, score_last = 0: its observation density has no parameters), or, on the
// shifted series of a fully adapted filter (model 4), y_t+1, with score_last the pair (x_NOBS-1, x_NOBS) with x_NOBS
// integrated out.  Either way the slots sum to an estimate of the score of the whole series.
// Unused gradient slots stay 0.  Model ids are part of the C ABI (include/pmmh_qn.h).
//
// The generic Hessian branch (Pairing::Predictive, grid kernel): Louis' identity on the gradient's pairs and weights.
// s_k is gradient slot k's term and H_k = hess_main / hess_last of the same pair; alpha is the score accumulated along
// a lineage, alpha(x_0) = 0, alpha(child) = alpha(parent) + score_main(parent, child, obs[t - 1]) at the child's birth
// (generation t).  hess1 = sum_k E[H_k] and hess2 = sum_k E[s_k s_k' + alpha_k s_k' + s_k alpha_k'] under the weights
// that read slot k, alpha_k = alpha of x_k on the lineage read (the pair's first state).  The estimate of the
// log-likelihood's Hessian is hess1 + hess2 - g g' with g = the sum of the gradient slots.  alpha runs along the whole
// genealogy, so its variance grows with T / N as the genealogy degenerates (the reference's estimator for the SV model).
#pragma once
#include <math.h>

#include "../../include/pmmh_qn.h"
#include "sv_math.cuh"

namespace pmmh {

enum class Pairing { Reference, Exact, Predictive };

// The offsets of the pairings above; the main loop reads the pair (x_t, x_t+1) at step t + LAG - 1.
// The first step of the main loop that adds a fixed-lag term:
__host__ __device__ constexpr int pair_first_step(Pairing p, int lag) {
    return p == Pairing::Reference ? lag : lag - 1;
}
// the observation index of the pair (x_t, x_t+1) (Reference: t - 1, wrapped in the tail):
__host__ __device__ constexpr int pair_obs(Pairing p, int t) {
    return p == Pairing::Reference ? t - 1 : (p == Pairing::Predictive ? t : t + 1);
}
// the gradient slot of the pair (x_t, x_t+1) (Reference: in the main loop; its tail puts it into t - LAG + 1, Q6):
__host__ __device__ constexpr int pair_slot(Pairing p, int t) { return p == Pairing::Exact ? t + 1 : t; }

// ---- 0: stochastic volatility with leverage (the reference's model; models/stochastic_volatility.py)
struct SvLeverageModel {
    static constexpr int kId = PMMH_MODEL_SV_LEVERAGE;
    typedef SvLeverageModel Filter;
    typedef SvLeverageModel Gradient;
    static constexpr bool kHessian = true;
    typedef SvConst Const;
    static __device__ __forceinline__ void init(Const& c, const double* par) { sv_const_init(c, par); }
    static __device__ __forceinline__ double initial_state(const Const& c) {
        const double stdev0 = c.sigmav / sqrt(1.0 - (c.phi * c.phi));
        return c.mu + stdev0 * 0.0;   // :309 (Q1)
    }
    static constexpr bool kScoreIsZero = false;
    static constexpr Pairing kPairing = Pairing::Reference;
    static __device__ __forceinline__ double propagate(const Const& c, double xp, double y1, double u) {
        double mean = c.mu + c.phi * (xp - c.mu);
        mean += c.sr * exp(-0.5 * xp) * y1;
        return mean + c.sd * u;
    }
    static __device__ __forceinline__ double prop_mean(const Const& c, double xp, double y1) {
        double mean = c.mu + c.phi * (xp - c.mu);
        mean += c.sr * exp(-0.5 * xp) * y1;
        return mean;
    }
    static __device__ __forceinline__ double prop_sd(const Const& c) { return c.sd; }
    static __device__ __forceinline__ void child_range(const Const& c, double xmin, double xmax, double y1, double nsd,
                                                       double& lo, double& hi) {
        sv_child_range(c, xmin, xmax, y1, nsd, lo, hi);
    }
    static __device__ __forceinline__ double logw(const Const&, double x, double y) {
        const double e = exp(-0.5 * x);
        return (-0.91893853320467267 - 0.5 * x) - (0.5 * (y * y)) * (e * e);
    }
    static __device__ __forceinline__ double logw_max(const Const& c, double lo, double hi, double y) {
        double xs = log(y * y);   // the log-weight is concave in x with its maximum at log y^2
        if (!(xs >= lo)) xs = lo;
        if (xs > hi) xs = hi;
        if (!isfinite(xs)) xs = 0.0;
        return logw(c, xs, y);
    }
    static __device__ __forceinline__ void score_main(const Const& c, double curr, double next, double y, double g[4]) {
        double sq;
        sv_score_main(c, curr, next, y, sq, g);
    }
    static __device__ __forceinline__ void score_tail(const Const& c, double curr, double next, double y, double g[4]) {
        double sq;
        sv_score_tail(c, curr, next, y, sq, g);
    }
};

// ---- 8: the SV model with the exact fixed-lag score and a Hessian.  Its particle system is model 0's (inherited:
// initial state, propagation, weights, shift, child range), so filt, log_like, traj, diag and the history are model 0's
// bit for bit and the filter entries run model 0's filter (Filter).  The fixed-lag terms pair the states predictively
// (Pairing::Predictive): the pair (x_t, x_t+1) is scored with its own leverage observation obs[t] -- the one the
// propagation x_t -> x_t+1 read -- into slot t (model 0 gives it obs[t - 1], Q5, and re-adds tail pairs, Q6).  Free
// parameters as the reference's: theta = (mu, atanh phi, log sigma_v, atanh rho).  One id for the gradient and the
// Hessian: a call without the Hessian runs this instantiation (Gradient), the Hessian the generic branch of the grid
// kernel.  The transition density is N(x'; m, sigma_v^2 (1 - rho^2)), m = mu + phi (x - mu) + sigma_v rho e^{-x/2} y;
// with s = x' - m and q = 1 / (sigma_v^2 (1 - rho^2)), log p = 1/2 log q - q s^2 / 2 + const, so
//   d log p = 1/2 dlog q (1 - q s^2) - q s ds,
//   d2 log p = 1/2 d2log q (1 - q s^2) - 1/2 q s^2 dlog q dlog q' - q s (dlog q ds' + ds dlog q') - q ds ds' - q s d2s,
// with dlog q = (0, 0, -2, 2 rho), d2log q nonzero only at (3,3): 2 (1 - rho^2).  The pair (x_0, x_1) has x_0 = mu
// (Q1), so its s depends on mu through x_0 too (score_first / hess_first).  The observation density has no parameters.
struct SvLeverageExact : SvLeverageModel {
    static constexpr int kId = PMMH_MODEL_SV_LEVERAGE_EXACT;
    typedef SvLeverageExact Gradient;
    static constexpr Pairing kPairing = Pairing::Predictive;
    // score_main: model 0's (sv_score_main, the derivative of log N(next; m, sigma_v^2 (1 - rho^2)) in theta)
    static __device__ __forceinline__ void score_tail(const Const& c, double curr, double next, double y, double g[4]) {
        score_main(c, curr, next, y, g);
    }
    static __device__ __forceinline__ void score_last(const Const&, double, double, double g[4]) {
        g[0] = g[1] = g[2] = g[3] = 0.0;
    }
    // the pair (x_0 = mu, x_1): ds/dmu = -(1 - sigma_v rho e^{-mu/2} y0 / 2), ds/d atanh phi = 0
    static __device__ __forceinline__ void score_first(const Const& c, double x1, double y0, double g[4]) {
        double sq;
        sv_score_main(c, c.mu, x1, y0, sq, g);
        g[0] = c.q * sq * (1.0 - 0.5 * c.sr * exp(-0.5 * c.mu) * y0);
        g[1] = 0.0;
    }
    static __device__ __forceinline__ void hess_main(const Const& c, double curr, double next, double y, double h[10]) {
        const double d = curr - c.mu, ey = exp(-0.5 * curr) * y;
        const double s = (next - c.mu - c.phi * d) - c.sr * ey;
        // ds and the second derivatives of s: (mu, a) entries from m's mu + phi (x - mu), (b, c) from sigma_v rho ey
        const double ds[4] = {-c.one_m_phi, -d * c.one_m_phi2, -c.sr * ey, -c.sigmav * ey * c.rho_term};
        const double d2s[10] = {0.0, c.one_m_phi2, 0.0, 0.0, 2.0 * c.phi * c.one_m_phi2 * d, 0.0, 0.0, -c.sr * ey,
                                -c.sigmav * ey * c.rho_term, 2.0 * c.sr * ey * c.rho_term};
        sv_exact_hess(c, s, ds, d2s, h);
    }
    // the pair (x_0 = mu, x_1): s = x1 - mu - sigma_v rho e^{-mu/2} y0
    static __device__ __forceinline__ void hess_first(const Const& c, double x1, double y0, double h[10]) {
        const double ey = exp(-0.5 * c.mu) * y0;
        const double s = (x1 - c.mu) - c.sr * ey;
        const double ds[4] = {-(1.0 - 0.5 * c.sr * ey), 0.0, -c.sr * ey, -c.sigmav * ey * c.rho_term};
        const double d2s[10] = {-0.25 * c.sr * ey, 0.0, 0.5 * c.sr * ey, 0.5 * c.sigmav * ey * c.rho_term, 0.0, 0.0, 0.0,
                                -c.sr * ey, -c.sigmav * ey * c.rho_term, 2.0 * c.sr * ey * c.rho_term};
        sv_exact_hess(c, s, ds, d2s, h);
    }
    static __device__ __forceinline__ void hess_last(const Const&, double, double, double h[10]) {
#pragma unroll
        for (int i = 0; i < 10; ++i) h[i] = 0.0;
    }

  private:
    // the second derivatives of 1/2 log q - q s^2 / 2 (the formula above) from s, ds and d2s (upper triangle)
    static __device__ __forceinline__ void sv_exact_hess(const Const& c, double s, const double ds[4],
                                                         const double d2s[10], double h[10]) {
        const double dlq[4] = {0.0, 0.0, -2.0, 2.0 * c.rho};
        const double qs = c.q * s, hq = 0.5 * c.q * (s * s);
        int z = 0;
#pragma unroll
        for (int i = 0; i < 4; ++i)
#pragma unroll
            for (int j = i; j < 4; ++j, ++z) {
                double v = -hq * (dlq[i] * dlq[j]) - qs * (dlq[i] * ds[j] + ds[i] * dlq[j]) - c.q * (ds[i] * ds[j]) -
                           qs * d2s[z];
                if (i == 3 && j == 3) v += c.rho_term * (1.0 - 2.0 * hq);
                h[z] = v;
            }
    }
};

// the score (pair_score) and second derivatives (pair_hess) of the pair (x_t, x_t+1), first = (t == 0): M::score_first /
// M::hess_first for the first pair where the model has them, M::score_main / M::hess_main otherwise
template <class M, class = void>
struct HasFirstPair {
    static constexpr bool value = false;
};
template <class M>
struct HasFirstPair<M, decltype((void)&M::score_first)> {
    static constexpr bool value = true;
};
template <class M>
__device__ __forceinline__ void pair_score(const typename M::Const& c, bool first, double curr, double next, double y,
                                           double g[4]) {
    if constexpr (HasFirstPair<M>::value) {
        if (first) {
            M::score_first(c, next, y, g);
            return;
        }
    }
    M::score_main(c, curr, next, y, g);
}
template <class M>
__device__ __forceinline__ void pair_hess(const typename M::Const& c, bool first, double curr, double next, double y,
                                          double h[10]) {
    if constexpr (HasFirstPair<M>::value) {
        if (first) {
            M::hess_first(c, next, y, h);
            return;
        }
    }
    M::hess_main(c, curr, next, y, h);
}

// ---- 1: linear Gaussian state space model  x_t = phi x_{t-1} + sigma_v v_t,  y_t = x_t + sigma_e e_t
// (parameters phi, sigma_v, sigma_e; the fourth slot is unused).  Not a model of the reference: it is
// here to show that a second model plugs into the same kernel, and because its exact likelihood is
// known (Kalman filter), which the tests use.
struct LinearGaussianModel {
    static constexpr int kId = PMMH_MODEL_LINEAR_GAUSSIAN;
    typedef LinearGaussianModel Filter;
    typedef LinearGaussianModel Gradient;
    static constexpr bool kHessian = false;
    struct Const {
        double phi, sv, se, inv_sv2, inv_se2, log_se;
    };
    static __device__ __forceinline__ void init(Const& c, const double* par) {
        c.phi = par[0];
        c.sv = par[1];
        c.se = par[2];
        c.inv_sv2 = 1.0 / (c.sv * c.sv);
        c.inv_se2 = 1.0 / (c.se * c.se);
        c.log_se = log(c.se);
    }
    static __device__ __forceinline__ double initial_state(const Const&) { return 0.0; }
    static constexpr bool kScoreIsZero = false;
    static constexpr Pairing kPairing = Pairing::Exact;
    static __device__ __forceinline__ double propagate(const Const& c, double xp, double, double u) {
        return c.phi * xp + c.sv * u;
    }
    static __device__ __forceinline__ double prop_mean(const Const& c, double xp, double) { return c.phi * xp; }
    static __device__ __forceinline__ double prop_sd(const Const& c) { return c.sv; }
    static __device__ __forceinline__ void child_range(const Const& c, double xmin, double xmax, double, double nsd,
                                                       double& lo, double& hi) {
        const double a = c.phi * xmin, b = c.phi * xmax;
        lo = fmin(a, b) - nsd * c.sv;
        hi = fmax(a, b) + nsd * c.sv;
    }
    static __device__ __forceinline__ double logw(const Const& c, double x, double y) {
        const double r = y - x;
        return (-0.91893853320467267 - c.log_se) - (0.5 * (r * r)) * c.inv_se2;
    }
    static __device__ __forceinline__ double logw_max(const Const& c, double lo, double hi, double y) {
        double xs = y;
        if (!(xs >= lo)) xs = lo;
        if (xs > hi) xs = hi;
        if (!isfinite(xs)) xs = 0.0;
        return logw(c, xs, y);
    }
    // d/d(phi, sigma_v, sigma_e) of log N(next; phi curr, sigma_v^2) + log N(y; next, sigma_e^2), y = obs[time(next)]
    static __device__ __forceinline__ void score_main(const Const& c, double curr, double next, double y, double g[4]) {
        const double r = next - c.phi * curr;
        const double ry = y - next;
        g[0] = (r * curr) * c.inv_sv2;
        g[1] = ((r * r) * c.inv_sv2 - 1.0) / c.sv;
        g[2] = ((ry * ry) * c.inv_se2 - 1.0) / c.se;
        g[3] = 0.0;
    }
    static __device__ __forceinline__ void score_tail(const Const& c, double curr, double next, double y, double g[4]) {
        score_main(c, curr, next, y, g);
    }
};

// ---- 2: the same linear Gaussian model run as a FULLY ADAPTED particle filter (Pitt & Shephard): particles are
// drawn from p(x_t | x_{t-1}, y_t) and weighted with the predictive density p(y_{t+1} | x_t), both in closed form
// for this model.  The kernel's algorithm is untouched: the caller hands over the observations shifted by one
// (obs'[t] = obs[t + 1]), so `propagate` sees y_t where the SV model sees y_{t-1} (leverage) and `logw` sees
// y_{t+1}.  The reference has no fully adapted filter (SURVEY 8a note), so parity is unpinned with respect to it; the
// kernels are pinned to the NumPy restatement oracle/generic_pf.py LinearGaussianFullyAdapted (ancestors exact),
// which is checked against the conditional moments and the exact Kalman likelihood.  Outputs: log-likelihood of
// y_2 .. y_T given y_1 (the caller adds log p(y_1)), and E[x_t | y_1 .. y_{t+1}] in `filt`; the score terms are not
// defined for this variant (gradient rows 0).
struct LinearGaussianFullyAdapted {
    static constexpr int kId = PMMH_MODEL_LINEAR_GAUSSIAN_FA;
    typedef LinearGaussianFullyAdapted Filter;
    typedef LinearGaussianFullyAdapted Gradient;
    static constexpr bool kHessian = false;
    struct Const {
        double phi, sv, se, k, sdp, inv_s2, log_s;   // gain, proposal sd, predictive variance
    };
    static __device__ __forceinline__ void init(Const& c, const double* par) {
        c.phi = par[0];
        c.sv = par[1];
        c.se = par[2];
        const double s2 = c.sv * c.sv + c.se * c.se;
        c.k = (c.sv * c.sv) / s2;
        c.sdp = sqrt((c.sv * c.sv) * (c.se * c.se) / s2);
        c.inv_s2 = 1.0 / s2;
        c.log_s = 0.5 * log(s2);
    }
    static __device__ __forceinline__ double initial_state(const Const&) { return 0.0; }
    // x_t | x_{t-1}, y_t ~ N(phi x + k (y_t - phi x), sv^2 se^2 / (sv^2 + se^2))
    static constexpr bool kScoreIsZero = true;
    static constexpr Pairing kPairing = Pairing::Exact;   // smo: x_t under W_{t+LAG-1}, i.e. given y_1 .. y_{t+LAG}
    static __device__ __forceinline__ double propagate(const Const& c, double xp, double y_now, double u) {
        const double m = c.phi * xp;
        return (m + c.k * (y_now - m)) + c.sdp * u;
    }
    static __device__ __forceinline__ double prop_mean(const Const& c, double xp, double y_now) {
        const double m = c.phi * xp;
        return m + c.k * (y_now - m);
    }
    static __device__ __forceinline__ double prop_sd(const Const& c) { return c.sdp; }
    static __device__ __forceinline__ void child_range(const Const& c, double xmin, double xmax, double y_now, double nsd,
                                                       double& lo, double& hi) {
        const double a = c.phi * xmin, b = c.phi * xmax;
        const double ma = a + c.k * (y_now - a), mb = b + c.k * (y_now - b);
        lo = fmin(ma, mb) - nsd * c.sdp;
        hi = fmax(ma, mb) + nsd * c.sdp;
    }
    // log p(y_{t+1} | x_t) = log N(y; phi x, sv^2 + se^2)
    static __device__ __forceinline__ double logw(const Const& c, double x, double y_next) {
        const double r = y_next - c.phi * x;
        return (-0.91893853320467267 - c.log_s) - (0.5 * (r * r)) * c.inv_s2;
    }
    static __device__ __forceinline__ double logw_max(const Const& c, double lo, double hi, double y_next) {
        double xs = (c.phi != 0.0) ? y_next / c.phi : lo;
        const double l2 = fmin(lo, hi), h2 = fmax(lo, hi);
        if (!(xs >= l2)) xs = l2;
        if (xs > h2) xs = h2;
        if (!isfinite(xs)) xs = 0.0;
        return logw(c, xs, y_next);
    }
    static __device__ __forceinline__ void score_main(const Const&, double, double, double, double g[4]) {
        g[0] = g[1] = g[2] = g[3] = 0.0;
    }
    static __device__ __forceinline__ void score_tail(const Const&, double, double, double, double g[4]) {
        g[0] = g[1] = g[2] = g[3] = 0.0;
    }
};

// ---- 4: model 2's fully adapted filter with a fixed-lag gradient.  Propagation, weights, shift and child range are
// model 2's (inherited), so every output model 2 has -- filt, smo, log-likelihood, traj, diag, history -- is
// bit-identical to it, and the filter entries run model 2's instantiation (Filter).  The gradient pairs the terms
// predictively (Pairing::Predictive above): slot t holds the
// contribution of obs'[t] = y_t+1, and the slots sum to an estimate of the score of log p(y_1 .. y_T), the first
// observation's term included (the log-likelihood still lacks log p(y_1)).  Checked against the restatement
// oracle/generic_pf.py LinearGaussianFullyAdaptedGrad and the exact fixed-lag Kalman targets of oracle/kalman.py.
struct LinearGaussianFullyAdaptedGrad : LinearGaussianFullyAdapted {
    static constexpr int kId = PMMH_MODEL_LINEAR_GAUSSIAN_FA_GRAD;
    typedef LinearGaussianFullyAdaptedGrad Gradient;
    struct Const : LinearGaussianFullyAdapted::Const {
        double inv_sv2, inv_sv, inv_se2, inv_se;
    };
    static __device__ __forceinline__ void init(Const& c, const double* par) {
        LinearGaussianFullyAdapted::init(c, par);
        c.inv_sv2 = 1.0 / (c.sv * c.sv);
        c.inv_sv = 1.0 / c.sv;
        c.inv_se2 = 1.0 / (c.se * c.se);
        c.inv_se = 1.0 / c.se;
    }
    static constexpr bool kScoreIsZero = false;
    static constexpr Pairing kPairing = Pairing::Predictive;
    // d/d(phi, sigma_v, sigma_e) of log N(next; phi curr, sigma_v^2) + log N(y; next, sigma_e^2), y = obs'[time(curr)]
    static __device__ __forceinline__ void score_main(const Const& c, double curr, double next, double y, double g[4]) {
        const double r = next - c.phi * curr;
        const double ry = y - next;
        g[0] = (r * curr) * c.inv_sv2;
        g[1] = ((r * r) * c.inv_sv2 - 1.0) * c.inv_sv;
        g[2] = ((ry * ry) * c.inv_se2 - 1.0) * c.inv_se;
        g[3] = 0.0;
    }
    static __device__ __forceinline__ void score_tail(const Const& c, double curr, double next, double y, double g[4]) {
        score_main(c, curr, next, y, g);
    }
    // d/d(phi, sigma_v, sigma_e) of log N(y_next; phi x, sigma_v^2 + sigma_e^2): the last pair with its second state
    // integrated out (the conditional score of that state has mean 0)
    static __device__ __forceinline__ void score_last(const Const& c, double x, double y_next, double g[4]) {
        const double r = y_next - c.phi * x;
        const double a = (r * r) * c.inv_s2 - 1.0;
        g[0] = (r * x) * c.inv_s2;
        g[1] = (a * c.sv) * c.inv_s2;
        g[2] = (a * c.se) * c.inv_s2;
        g[3] = 0.0;
    }
};

// ---- 6: model 4 with the generic Hessian branch (grid kernel; the header comment above).  Every output model 4 has is
// bit-identical to it: a call without the Hessian runs model 4's instantiation (Gradient), the filter entries model 2's.
// The Hessian hooks are the second derivatives over (phi, sigma_v, sigma_e) of score_main's and score_last's terms; row
// and column 3 stay 0.
struct LinearGaussianFullyAdaptedHess : LinearGaussianFullyAdaptedGrad {
    static constexpr int kId = PMMH_MODEL_LINEAR_GAUSSIAN_FA_HESS;
    static constexpr bool kHessian = true;
    static __device__ __forceinline__ void hess_main(const Const& c, double curr, double next, double y, double h[10]) {
        const double r = next - c.phi * curr;
        const double ry = y - next;
        h[0] = -(curr * curr) * c.inv_sv2;
        h[1] = -2.0 * (r * curr) * (c.inv_sv2 * c.inv_sv);
        h[4] = (1.0 - 3.0 * (r * r) * c.inv_sv2) * c.inv_sv2;
        h[7] = (1.0 - 3.0 * (ry * ry) * c.inv_se2) * c.inv_se2;
        h[2] = h[3] = h[5] = h[6] = h[8] = h[9] = 0.0;
    }
    // s2 = sigma_v^2 + sigma_e^2, r = y_next - phi x, a = r^2 / s2 - 1, b = 2 r^2 / s2 - 1
    static __device__ __forceinline__ void hess_last(const Const& c, double x, double y_next, double h[10]) {
        const double r = y_next - c.phi * x;
        const double a = (r * r) * c.inv_s2 - 1.0, b = 2.0 * (r * r) * c.inv_s2 - 1.0;
        const double i4 = c.inv_s2 * c.inv_s2;
        h[0] = -(x * x) * c.inv_s2;
        h[1] = -2.0 * (r * x) * c.sv * i4;
        h[2] = -2.0 * (r * x) * c.se * i4;
        h[4] = (a - 2.0 * (c.sv * c.sv) * c.inv_s2 * b) * c.inv_s2;
        h[5] = -2.0 * (c.sv * c.se) * i4 * b;
        h[7] = (a - 2.0 * (c.se * c.se) * c.inv_s2 * b) * c.inv_s2;
        h[3] = h[6] = h[8] = h[9] = 0.0;
    }
};

// ---- the model table: every model the kernels are instantiated for.  Models::with(id, f) calls f(ModelTag<M>()) for
// the model M of that id (false, and no call, for an unknown id); Models::each(f) calls it for every model.
template <class M>
struct ModelTag {
    typedef M type;
};
template <class... Ms>
struct ModelList {
    template <class F>
    static bool with(int id, F&& f) { return ((Ms::kId == id ? (f(ModelTag<Ms>()), true) : false) || ...); }
    template <class F>
    static void each(F&& f) { (f(ModelTag<Ms>()), ...); }
    static constexpr bool ids_distinct() {   // (a derived model inherits its base's id unless it states its own)
        int same = 0;
        for (int a : {Ms::kId...}) for (int b : {Ms::kId...}) same += a == b;
        return same == (int)sizeof...(Ms);
    }
};
typedef ModelList<SvLeverageModel, LinearGaussianModel, LinearGaussianFullyAdapted, LinearGaussianFullyAdaptedGrad,
                  LinearGaussianFullyAdaptedHess, SvLeverageExact>
    Models;
static_assert(Models::ids_distinct(), "every model states its own id");

inline bool model_known(int id) { return Models::with(id, [](auto) {}); }
inline bool model_has_hessian(int id) {
    bool h = false;
    Models::with(id, [&](auto m) { h = decltype(m)::type::kHessian; });
    return h;
}

}  // namespace pmmh
