/*
 * pmmh_oracle.c -- CPU restatement of the pmmh-qn likelihood-estimation hot path.
 *
 * TEST INFRASTRUCTURE ONLY.  This file is the parity oracle for the CUDA path.
 * Only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline / --impl
 * reference legs may load it.  The product path (pmmh-qn_b200/) never does.
 *
 * Parity status: PINNED.  Every function here is checked bit-for-bit against the
 * reference's own Cython kernels compiled unmodified from /root/reference
 * (oracle/build_ref.py -> oracle/_ref/ modules), and against golden vectors generated
 * from those kernels (tests/golden/make_golden.py -> tests/golden/ npz files).
 *
 * What is restated (reference file:line, relative to /root/reference/python):
 *   oracle_argsort            state/particle_methods/stochastic_volatility.pyx:23-52
 *   oracle_systematic_corr    ...stochastic_volatility.pyx:694-715
 *   oracle_my_max             ...stochastic_volatility.pyx:738-746
 *   oracle_sample_particle    ...stochastic_volatility.pyx:785-806
 *   oracle_flps_sv_corr       ...stochastic_volatility.pyx:205-655
 *   oracle_bpf_sv_corr        ...stochastic_volatility.pyx:61-201
 *   oracle_importance_discrete  state/importance_sampling/random_effects.pyx:21-104
 *   oracle_stratified         state/direct/subsampling.pyx:34-51
 *
 * The arithmetic keeps the reference's operation order (IEEE fp64, libm exp/log/pow,
 * glibc qsort with the reference's never-zero comparator) and all of its quirks
 * (SURVEY.md appendix Q1-Q10).  The ONLY structural change is the genealogy: the
 * reference copies the whole i x N ancestry matrix twice per step (O(T^2 N),
 * :344-351,:404-406,:423-424); here the composed one-step ancestor
 * A[t][j] = ancestors[new_idx[j]] is stored per step and traced back once, which
 * yields the same trajectory in O(T N).  Sizes are runtime arguments.
 *
 * Layouts: rvp is the reference's flat layout rvp[i + j*NOBS] (time fastest).
 * Internally particles/weights are kept time-major X[t*N + j]; the reference's
 * flat reads particles[q] / weights[q] (Q7, Q10) are emulated through
 * time = q % NOBS, slot = q / NOBS.
 */
#include <math.h>
#include <stdlib.h>
#include <string.h>
#include <stdint.h>

#define NPARAMS 4

typedef struct {
    int index;
    double value;
} sorter_t;

/* stochastic_volatility.pyx:32-35 -- never returns 0 for ordered values */
static int compare_sorter(const void *a, const void *b)
{
    double v = ((const sorter_t *)a)->value - ((const sorter_t *)b)->value;
    if (v < 0) return -1;
    if (v >= 0) return 1;
    return 0; /* NaN: Cython's implicit return value */
}

/* stochastic_volatility.pyx:37-52 */
void oracle_argsort(const double *data, int *order, int n)
{
    sorter_t *s = (sorter_t *)malloc((size_t)n * sizeof(sorter_t));
    for (int i = 0; i < n; i++) {
        s[i].index = i;
        s[i].value = data[i];
    }
    qsort(s, (size_t)n, sizeof(sorter_t), compare_sorter);
    for (int i = 0; i < n; i++) order[i] = s[i].index;
    free(s);
}

/* stochastic_volatility.pyx:659-664 */
static double norm_logpdf(double x, double m, double s)
{
    double part1 = -0.91893853320467267;
    double part2 = -log(s);
    double part3 = -0.5 * (x - m) * (x - m) / (s * s);
    return part1 + part2 + part3;
}

/* stochastic_volatility.pyx:738-746 (Q4: last element greater than element 0) */
double oracle_my_max(const double *w, int n)
{
    int idx = 0;
    double current_largest = w[0];
    for (int i = 1; i < n; i++)
        if (w[i] > current_largest && isfinite(w[i])) idx = i;
    return w[idx];
}

/* stochastic_volatility.pyx:694-715 (Q3: cum[0] is not normalised) */
void oracle_systematic_corr(int *ancestors, const double *weights, double rnd, int n,
                            double *cum_scratch)
{
    double *cum = cum_scratch ? cum_scratch : (double *)malloc((size_t)n * sizeof(double));
    double sum = weights[0];
    cum[0] = weights[0];
    for (int j = 1; j < n; j++) {
        cum[j] = cum[j - 1] + weights[j];
        sum += weights[j];
    }
    for (int j = 1; j < n; j++) cum[j] /= sum;
    int cur = 0;
    for (int j = 0; j < n; j++) {
        double cpoint = (rnd + j) / n;
        while (cum[cur] < cpoint && cur < n - 1) cur++;
        ancestors[j] = cur;
    }
    if (!cum_scratch) free(cum);
}

/* stochastic_volatility.pyx:785-806 on a weight vector of length n.
 * Returns cur in [0, n]; n means the reference would read out of bounds. */
int oracle_sample_particle(const double *weights, double rnd, int n)
{
    double *cum = (double *)malloc((size_t)n * sizeof(double));
    double sum = weights[0];
    cum[0] = weights[0];
    for (int j = 1; j < n; j++) {
        cum[j] = cum[j - 1] + weights[j];
        sum += weights[j];
    }
    for (int j = 1; j < n; j++) cum[j] /= sum;
    int cur = 0;
    for (int j = 0; j < n; j++) {
        if (cum[cur] < rnd) cur++;
        else break;
    }
    free(cum);
    return cur;
}

static inline double obs_wrap(const double *obs, int k, int nobs)
{
    /* Cython memoryview wraparound (Q8) */
    return obs[k < 0 ? k + nobs : k];
}

/* The 4 score terms of the main smoother loop, stochastic_volatility.pyx:452-465 */
static inline void score_main(double curr, double next, double y, double mu, double phi,
                              double sigmav, double rho, double q_matrix,
                              double *sq_out, double g[NPARAMS])
{
    double sq = next - mu - phi * (curr - mu);
    sq -= sigmav * rho * exp(-0.5 * curr) * y;
    g[0] = q_matrix * sq * (1.0 - phi);
    g[1] = q_matrix * sq * (curr - mu) * (1.0 - pow(phi, 2.0));
    g[2] = sq;
    g[2] += sigmav * rho * exp(-0.5 * curr) * y;
    g[2] *= q_matrix * sq;
    g[2] -= 1.0;
    g[3] = rho - q_matrix * rho * sq * sq;
    g[3] += pow(sigmav, -1.0) * sq * exp(-0.5 * curr) * y;
    *sq_out = sq;
}

/* sub_hessian1 / sub_hessian2 and their accumulation,
 * stochastic_volatility.pyx:473-534 (identical text at :565-626).
 * yl = obs[i - LAG] as used there; al[c] = alpha_history_c[LAG-2][j]. */
static void hessian_terms(double curr, double sq, double yl, const double g[NPARAMS],
                          const double al[NPARAMS], double w, double mu, double phi,
                          double sigmav, double rho, double q_matrix, double rho_term,
                          double hessian1[NPARAMS][NPARAMS], double hessian2[NPARAMS][NPARAMS])
{
    double h1[NPARAMS][NPARAMS];
    double h2[NPARAMS][NPARAMS];
    memset(h1, 0, sizeof(h1));
    memset(h2, 0, sizeof(h2));

    h1[0][0] = -q_matrix * pow((1.0 - phi), 2.0);
    h1[1][1] = 2.0 * phi * sq + (curr - mu) * (1.0 - pow(phi, 2.0));
    h1[1][1] *= -q_matrix * (curr - mu) * (1.0 - pow(phi, 2.0));
    h1[2][2] = -2.0 * q_matrix * sq * sq;
    h1[2][2] -= 2.0 * q_matrix * sq * rho * sigmav * exp(-0.5 * curr) * yl;
    h1[2][2] -= q_matrix * pow(rho * sigmav * exp(-0.5 * curr) * yl, 2.0);
    h1[2][2] += q_matrix * sq * rho * sigmav * exp(-0.5 * curr) * yl;
    h1[3][3] = rho_term - 2.0 * q_matrix * pow(rho, 2.0) * pow(sq, 2.0) - sigmav * (-2.0) * pow(sq, 2.0);
    h1[3][3] += 2.0 * pow(sigmav, -1.0) * rho * sq * exp(-0.5 * curr) * yl;
    h1[3][3] -= exp(-curr) * pow(yl, 2.0) * rho_term;

    h1[0][1] = -q_matrix * (curr - mu) * (1.0 - phi) - q_matrix * sq;
    h1[0][1] *= (1.0 - pow(phi, 2.0));
    h1[0][2] = -2.0 * sq * (1.0 - phi);
    h1[0][2] -= q_matrix * (1.0 - phi) * sigmav * rho * sq * exp(-0.5 * curr) * yl;
    h1[0][3] = 2.0 * q_matrix * rho * sq * (1.0 - phi);
    h1[0][3] -= pow(sigmav, -2.0) * (1.0 - phi) * sigmav * exp(-0.5 * curr) * yl;

    h1[1][2] = -2.0 * sq - rho * sigmav * exp(-0.5 * curr) * yl;
    h1[1][2] *= q_matrix * (curr - mu) * (1.0 - pow(phi, 2.0));
    h1[1][3] = 2.0 * rho * sq - sigmav * exp(-0.5 * curr) * yl * rho_term;
    h1[1][3] *= q_matrix * (curr - mu) * (1.0 - pow(phi, 2.0));

    h1[2][3] = 2.0 * q_matrix * pow(sq, 2.0) * rho;
    h1[2][3] += 2.0 * pow(rho, 2.0) * q_matrix * sq * sigmav * exp(-0.5 * curr) * yl;
    h1[2][3] -= rho * exp(-curr) * pow(yl, 2.0);
    h1[2][3] += pow(sigmav, -1.0) * sq * exp(-0.5 * curr) * yl;

    h2[0][0] = pow(g[0], 2.0) + 2.0 * al[0] * g[0];
    h2[0][1] = g[0] * g[1] + al[0] * g[1] + al[1] * g[0];
    h2[0][2] = g[0] * g[2] + al[0] * g[2] + al[2] * g[0];
    h2[0][3] = g[0] * g[3] + al[0] * g[3] + al[3] * g[0];
    h2[1][1] = pow(g[1], 2.0) + 2.0 * al[1] * g[1];
    h2[1][2] = g[1] * g[2] + al[1] * g[2] * al[2] * g[1];
    h2[1][3] = g[1] * g[3] + al[1] * g[3] * al[3] * g[1];
    h2[2][2] = pow(g[2], 2.0) + 2.0 * al[2] * g[2];
    h2[2][3] = g[2] * g[3] + al[2] * g[3] * al[3] * g[2];
    h2[3][3] = pow(g[3], 2.0) + 2.0 * al[3] * g[3];

    for (int k = 0; k < NPARAMS; k++) {
        if (isfinite(h1[k][k])) hessian1[k][k] += h1[k][k] * w;
        if (isfinite(h2[k][k])) hessian2[k][k] += h2[k][k] * w;
        for (int l = k + 1; l < NPARAMS; l++) {
            if (isfinite(h1[k][l])) {
                hessian1[k][l] += h1[k][l] * w;
                hessian1[l][k] += h1[k][l] * w;
            }
            if (isfinite(h2[k][l])) {
                hessian2[k][l] += h2[k][l] * w;
                hessian2[l][k] += h2[k][l] * w;
            }
        }
    }
}

/*
 * Fixed-lag particle smoother, stochastic_volatility.pyx:205-655.
 *
 * Outputs (caller-allocated): filt[NOBS], smo[NOBS], log_like[1],
 * gradient[4*NOBS] (row-major [p][t]), traj[NOBS], hess1[16], hess2[16].
 * Optional dumps (may be NULL): X_out[NOBS*N] sorted particles per time,
 * A_out[NOBS*N] composed one-step ancestors (A_out[0][j] = j),
 * W_out[NOBS*N] normalised weights per time, info[4] =
 * {trajectory index, trajectory-oob flag, 0, 0}.
 * Returns 0 on success, non-zero on allocation failure.
 */
int oracle_flps_sv_corr(const double *obs, const double *params, const double *rvr,
                        const double *rvp, int N, int NOBS, int LAG, int compute_hessian,
                        double *filt, double *smo, double *log_like_out, double *gradient,
                        double *traj, double *hess1_out, double *hess2_out, double *X_out,
                        int *A_out, double *W_out, int *info)
{
    const size_t NT = (size_t)N * (size_t)NOBS;
    double *X = X_out ? X_out : (double *)malloc(NT * sizeof(double));
    double *W = W_out ? W_out : (double *)malloc(NT * sizeof(double));
    int *A = A_out ? A_out : (int *)malloc(NT * sizeof(int));
    int *ancestors = (int *)malloc((size_t)N * sizeof(int));
    int *new_idx = (int *)malloc((size_t)N * sizeof(int));
    double *xnew = (double *)malloc((size_t)N * sizeof(double));
    double *lw = (double *)malloc((size_t)N * sizeof(double));
    double *sh = (double *)malloc((size_t)N * sizeof(double));
    double *cum = (double *)malloc((size_t)N * sizeof(double));
    /* history buffers, lag-major: ph[k*N + j] == particle_history[k + j*LAG] */
    const size_t LN = (size_t)LAG * (size_t)N;
    double *ph = (double *)calloc(LN, sizeof(double));
    double *oph = (double *)calloc(LN, sizeof(double));
    double *ah[NPARAMS] = {0, 0, 0, 0}, *oah[NPARAMS] = {0, 0, 0, 0};
    if (!X || !W || !A || !ancestors || !new_idx || !xnew || !lw || !sh || !cum || !ph || !oph)
        return 1;
    if (compute_hessian == 1) {
        for (int c = 0; c < NPARAMS; c++) {
            ah[c] = (double *)calloc(LN, sizeof(double));
            oah[c] = (double *)calloc(LN, sizeof(double));
            if (!ah[c] || !oah[c]) return 1;
        }
    }
    memset(X, 0, NT * sizeof(double));
    memset(W, 0, NT * sizeof(double));
    memset(A, 0, NT * sizeof(int));

    double hessian1[NPARAMS][NPARAMS], hessian2[NPARAMS][NPARAMS];
    memset(hessian1, 0, sizeof(hessian1));
    memset(hessian2, 0, sizeof(hessian2));
    for (int i = 0; i < NOBS; i++) {
        filt[i] = 0.0;
        smo[i] = 0.0;
        traj[i] = 0.0;
    }
    for (int p = 0; p < NPARAMS; p++)
        for (int t = 0; t < NOBS; t++) gradient[(size_t)p * NOBS + t] = 0.0;

    const double mu = params[0], phi = params[1], sigmav = params[2], rho = params[3];
    double log_like = 0.0;
    double mean, stDev, max_weight = 0.0, norm_factor, foo_double;
    const double q_matrix = 1.0 / (sigmav * sigmav * (1.0 - rho * rho));
    const double rho_term = 1.0 - rho * rho;
    double g[NPARAMS], sq;

    /* :306-323 initial state.  Q1: particles were just zeroed, so x0 = mu + stDev*0.0 */
    stDev = sigmav / sqrt(1.0 - (phi * phi));
    for (int j = 0; j < N; j++) {
        double x0 = mu + stDev * 0.0;
        xnew[j] = x0;
        W[j] = 1.0 / N;
        ph[j] = x0;
        A[j] = j;
    }
    filt[0] = 0.0;
    for (int j = 0; j < N; j++) filt[0] += W[j] * xnew[j];
    oracle_argsort(xnew, new_idx, N);
    for (int j = 0; j < N; j++) X[j] = xnew[new_idx[j]];

    for (int i = 1; i < NOBS; i++) {
        double *Xi = X + (size_t)i * N;
        const double *Xp = X + (size_t)(i - 1) * N;
        double *Wi = W + (size_t)i * N;

        /* :329-331 */
        oracle_systematic_corr(ancestors, W + (size_t)(i - 1) * N, rvr[i], N, cum);

        /* :334-341 */
        memcpy(oph, ph, LN * sizeof(double));
        if (compute_hessian == 1)
            for (int c = 0; c < NPARAMS; c++) memcpy(oah[c], ah[c], LN * sizeof(double));

        /* :354-390 propagate (+ alpha recursion) */
        for (int j = 0; j < N; j++) {
            int a = ancestors[j];
            mean = mu + phi * (Xp[a] - mu);
            mean += sigmav * rho * exp(-0.5 * Xp[a]) * obs[i - 1];
            stDev = sqrt(rho_term) * sigmav;
            xnew[j] = mean + stDev * rvp[(size_t)i + (size_t)j * NOBS];

            if (compute_hessian == 1) {
                /* Q7: particles[i - 1 + ancestors[j]] (missing *NOBS) read through the
                 * flat layout: time = q % NOBS, slot = q / NOBS */
                long q = (long)i - 1 + a;
                int tq = (int)(q % NOBS);
                int sq_slot = (int)(q / NOBS);
                double curr;
                if (tq < i) curr = X[(size_t)tq * N + sq_slot];
                else if (tq == i) curr = (sq_slot <= j) ? xnew[sq_slot] : 0.0;
                else curr = 0.0;
                double next = xnew[j];
                double yl = obs_wrap(obs, i - LAG, NOBS); /* Q8 */
                double s = next - mu - phi * (curr - mu);
                s -= sigmav * rho * exp(-0.5 * curr) * yl;

                double a0 = q_matrix * s * (1.0 - phi);
                double a1 = q_matrix * s * (curr - mu) * (1.0 - pow(phi, 2.0));
                double a2 = s;
                a2 += sigmav * rho * exp(-0.5 * curr) * obs[i];
                a2 *= q_matrix * s;
                a2 -= 1.0;
                double a3 = rho - q_matrix * rho * s * s;
                a3 += pow(sigmav, -1.0) * s * exp(-0.5 * curr) * obs[i];
                double av[NPARAMS] = {a0, a1, a2, a3};
                for (int c = 0; c < NPARAMS; c++) {
                    for (int k = 1; k < LAG; k++)
                        ah[c][(size_t)k * N + j] = oah[c][(size_t)(k - 1) * N + a];
                    ah[c][j] = av[c] + oah[c][a];
                }
            }
        }

        /* :392-424 sort and permute */
        if (compute_hessian == 1)
            for (int c = 0; c < NPARAMS; c++) memcpy(oah[c], ah[c], LN * sizeof(double));
        oracle_argsort(xnew, new_idx, N);
        for (int j = 0; j < N; j++) {
            int src = new_idx[j];
            Xi[j] = xnew[src];
            ph[j] = xnew[src];
            for (int k = 1; k < LAG; k++)
                ph[(size_t)k * N + j] = oph[(size_t)(k - 1) * N + ancestors[src]];
            if (compute_hessian == 1)
                for (int c = 0; c < NPARAMS; c++)
                    for (int k = 0; k < LAG; k++)
                        ah[c][(size_t)k * N + j] = oah[c][(size_t)k * N + src];
            A[(size_t)i * N + j] = ancestors[src];
        }

        /* :427-437 weights */
        for (int j = 0; j < N; j++) lw[j] = norm_logpdf(obs[i], 0.0, exp(0.5 * Xi[j]));
        max_weight = oracle_my_max(lw, N);
        norm_factor = 0.0;
        for (int j = 0; j < N; j++) {
            sh[j] = exp(lw[j] - max_weight);
            foo_double = norm_factor + sh[j];
            if (isfinite(foo_double) != 0) norm_factor = foo_double;
        }
        /* :439-442 */
        for (int j = 0; j < N; j++) {
            Wi[j] = sh[j] / norm_factor;
            if (isfinite(Wi[j] * Xi[j]) != 0) filt[i] += Wi[j] * Xi[j];
        }

        /* :445-534 fixed-lag smoother */
        if (i >= LAG) {
            const double yl = obs[i - LAG]; /* Q5 */
            double *gr = gradient;
            const int tt = i - LAG + 1;
            for (int j = 0; j < N; j++) {
                double curr = ph[(size_t)(LAG - 1) * N + j];
                double next = ph[(size_t)(LAG - 2) * N + j];
                smo[tt] += Wi[j] * curr;
                score_main(curr, next, yl, mu, phi, sigmav, rho, q_matrix, &sq, g);
                gr[0 * (size_t)NOBS + tt] += g[0] * Wi[j];
                gr[1 * (size_t)NOBS + tt] += g[1] * Wi[j];
                gr[2 * (size_t)NOBS + tt] += g[2] * Wi[j];
                gr[3 * (size_t)NOBS + tt] += g[3] * Wi[j];
                if (compute_hessian == 1) {
                    double al[NPARAMS];
                    for (int c = 0; c < NPARAMS; c++) al[c] = ah[c][(size_t)(LAG - 2) * N + j];
                    hessian_terms(curr, sq, yl, g, al, Wi[j], mu, phi, sigmav, rho, q_matrix,
                                  rho_term, hessian1, hessian2);
                }
            }
        }

        /* :537 */
        log_like += max_weight + log(norm_factor) - log((double)N);
    }

    /* :540-626 tail (Q6) */
    for (int i = NOBS - LAG; i < NOBS; i++) {
        int idx = NOBS - i - 1;
        const double *WT = W + (size_t)(NOBS - 1) * N;
        const double *Wi = W + (size_t)i * N;
        for (int j = 0; j < N; j++) {
            double curr = ph[(size_t)idx * N + j];
            smo[i] += WT[j] * curr;
            if ((idx - 1) >= 0) {
                double next = ph[(size_t)(idx - 1) * N + j];
                double y1 = obs_wrap(obs, i - 1, NOBS);
                sq = next - mu - phi * (curr - mu);
                sq -= sigmav * rho * exp(-0.5 * curr) * y1;
                g[0] = q_matrix * sq * (1.0 - phi);
                g[1] = q_matrix * sq * (curr - mu) * (1.0 - pow(phi, 2.0));
                g[2] = q_matrix * sq * sq - 1.0;
                g[2] += q_matrix * sq * sigmav * rho * exp(-0.5 * curr) * y1;
                g[3] = rho;
                g[3] -= q_matrix * rho * sq * sq;
                g[3] += q_matrix * sq * sigmav * exp(-0.5 * curr) * y1 * rho_term;
                /* Short series (DESIGN.md §2): for NOBS <= 2 LAG - 2 the first tail steps index slot tt < 0,
                 * outside the reference's C array (undefined there).  Rule: that gradient term is dropped, as
                 * every kernel drops it; the Hessian sums, which have no slot, keep it. */
                const int tt = i - LAG + 1;
                if (tt >= 0) {
                    gradient[0 * (size_t)NOBS + tt] += g[0] * Wi[j];
                    gradient[1 * (size_t)NOBS + tt] += g[1] * Wi[j];
                    gradient[2 * (size_t)NOBS + tt] += g[2] * Wi[j];
                    gradient[3 * (size_t)NOBS + tt] += g[3] * Wi[j];
                }
                if (compute_hessian == 1) {
                    double al[NPARAMS];
                    for (int c = 0; c < NPARAMS; c++) al[c] = ah[c][(size_t)(LAG - 2) * N + j];
                    hessian_terms(curr, sq, obs_wrap(obs, i - LAG, NOBS), g, al, Wi[j], mu, phi,
                                  sigmav, rho, q_matrix, rho_term, hessian1, hessian2);
                }
            }
        }
    }

    /* :630-633 trajectory.  Q10: sampleParticle_corr gets the whole flat weights
     * buffer and uses weights[0..N-1] = (time k % NOBS, slot k / NOBS). */
    {
        double *wflat = (double *)malloc((size_t)N * sizeof(double));
        for (int k = 0; k < N; k++) wflat[k] = W[(size_t)(k % NOBS) * N + (k / NOBS)];
        int idx = oracle_sample_particle(wflat, rvr[0], N);
        free(wflat);
        int oob = 0;
        if (idx >= N) {
            oob = 1; /* reference reads out of bounds here; out of contract */
            idx = N - 1;
        }
        if (info) {
            info[0] = idx;
            info[1] = oob;
            info[2] = 0;
            info[3] = 0;
        }
        /* Q11: the sort step copies rows k < i into old_ancestry (:404-406) but then
         * reads rows k <= i back (:423-424), so row i is refilled from the never-
         * written (zero) row of old_ancestry: ancestry[i][.] == 0 for every i >= 1.
         * Hence traj[i] = particles[i, 0] = X_i[0] for i >= 1; only row 0 carries a
         * real genealogy, traj[0] = X_0[b_0] with b_0 the time-0 ancestor of idx. */
        int b = idx;
        for (int t = NOBS - 1; t >= 1; t--) {
            b = A[(size_t)t * N + b];
            traj[t] = X[(size_t)t * N + 0];
        }
        traj[0] = X[b];
        if (info) info[2] = b;
    }

    *log_like_out = log_like;
    for (int k = 0; k < NPARAMS; k++)
        for (int l = 0; l < NPARAMS; l++) {
            hess1_out[k * NPARAMS + l] = hessian1[k][l];
            hess2_out[k * NPARAMS + l] = hessian2[k][l];
        }

    if (!X_out) free(X);
    if (!W_out) free(W);
    if (!A_out) free(A);
    free(ancestors);
    free(new_idx);
    free(xnew);
    free(lw);
    free(sh);
    free(cum);
    free(ph);
    free(oph);
    for (int c = 0; c < NPARAMS; c++) {
        free(ah[c]);
        free(oah[c]);
    }
    return 0;
}

/*
 * Bootstrap particle filter, stochastic_volatility.pyx:61-201.
 * Q2: the leverage term reads particles[i + ancestors[j]*NOBS] -- the column of
 * time i that is being written in this very loop -- so
 *     z_j = x_new[a_j] if a_j < j else 0.0
 * (zero-initialised, not yet written).  intended_read != 0 switches to the
 * evidently intended time i-1 read (a labelled deviation, not reference parity).
 */
int oracle_bpf_sv_corr(const double *obs, const double *params, const double *rvr,
                       const double *rvp, int N, int NOBS, int intended_read, double *filt,
                       double *log_like_out, double *traj, double *X_out, int *A_out,
                       double *W_out, int *info)
{
    const size_t NT = (size_t)N * (size_t)NOBS;
    double *X = X_out ? X_out : (double *)malloc(NT * sizeof(double));
    double *W = W_out ? W_out : (double *)malloc(NT * sizeof(double));
    int *A = A_out ? A_out : (int *)malloc(NT * sizeof(int));
    int *ancestors = (int *)malloc((size_t)N * sizeof(int));
    int *new_idx = (int *)malloc((size_t)N * sizeof(int));
    double *xnew = (double *)malloc((size_t)N * sizeof(double));
    double *lw = (double *)malloc((size_t)N * sizeof(double));
    double *sh = (double *)malloc((size_t)N * sizeof(double));
    double *cum = (double *)malloc((size_t)N * sizeof(double));
    if (!X || !W || !A || !ancestors || !new_idx || !xnew || !lw || !sh || !cum) return 1;
    memset(X, 0, NT * sizeof(double));
    memset(W, 0, NT * sizeof(double));
    memset(A, 0, NT * sizeof(int));
    for (int i = 0; i < NOBS; i++) {
        filt[i] = 0.0;
        traj[i] = 0.0;
    }
    const double mu = params[0], phi = params[1], sigmav = params[2], rho = params[3];
    double log_like = 0.0, mean, stDev, max_weight, norm_factor;

    /* :110-122 */
    stDev = sigmav / sqrt(1.0 - (phi * phi));
    for (int j = 0; j < N; j++) {
        xnew[j] = mu + stDev * rvp[(size_t)0 + (size_t)j * NOBS];
        W[j] = 1.0 / N;
        A[j] = j;
        filt[0] += W[j] * xnew[j];
    }
    oracle_argsort(xnew, new_idx, N);
    for (int j = 0; j < N; j++) X[j] = xnew[new_idx[j]];

    for (int i = 1; i < NOBS; i++) {
        double *Xi = X + (size_t)i * N;
        const double *Xp = X + (size_t)(i - 1) * N;
        double *Wi = W + (size_t)i * N;
        oracle_systematic_corr(ancestors, W + (size_t)(i - 1) * N, rvr[i], N, cum);

        /* :142-146 */
        for (int j = 0; j < N; j++) {
            int a = ancestors[j];
            double z;
            if (intended_read) z = Xp[a];
            else z = (a < j) ? xnew[a] : 0.0; /* Q2 */
            mean = mu + phi * (Xp[a] - mu);
            mean += sigmav * rho * exp(-0.5 * z) * obs[i - 1];
            stDev = sqrt(1.0 - rho * rho) * sigmav;
            xnew[j] = mean + stDev * rvp[(size_t)i + (size_t)j * NOBS];
        }
        /* :149-163 */
        oracle_argsort(xnew, new_idx, N);
        for (int j = 0; j < N; j++) {
            Xi[j] = xnew[new_idx[j]];
            A[(size_t)i * N + j] = ancestors[new_idx[j]];
        }
        /* :166-176 */
        for (int j = 0; j < N; j++) lw[j] = norm_logpdf(obs[i], 0.0, exp(0.5 * Xi[j]));
        max_weight = oracle_my_max(lw, N);
        norm_factor = 0.0;
        for (int j = 0; j < N; j++) {
            sh[j] = exp(lw[j] - max_weight);
            if (isfinite(sh[j])) norm_factor += sh[j];
            else sh[j] = 0.0;
        }
        /* :179-183 */
        filt[i] = 0.0;
        for (int j = 0; j < N; j++) {
            Wi[j] = sh[j] / norm_factor;
            if (isfinite(Wi[j] * Xi[j]) != 0) filt[i] += Wi[j] * Xi[j];
        }
        /* :186 */
        log_like += max_weight + log(norm_factor) - log((double)N);
    }

    /* :189-192 (Q10 as in flps) */
    {
        double *wflat = (double *)malloc((size_t)N * sizeof(double));
        for (int k = 0; k < N; k++) wflat[k] = W[(size_t)(k % NOBS) * N + (k / NOBS)];
        int idx = oracle_sample_particle(wflat, rvr[0], N);
        free(wflat);
        int oob = 0;
        if (idx >= N) {
            oob = 1;
            idx = N - 1;
        }
        if (info) {
            info[0] = idx;
            info[1] = oob;
            info[2] = 0;
            info[3] = 0;
        }
        /* Q11: the sort step copies rows k < i into old_ancestry (:404-406) but then
         * reads rows k <= i back (:423-424), so row i is refilled from the never-
         * written (zero) row of old_ancestry: ancestry[i][.] == 0 for every i >= 1.
         * Hence traj[i] = particles[i, 0] = X_i[0] for i >= 1; only row 0 carries a
         * real genealogy, traj[0] = X_0[b_0] with b_0 the time-0 ancestor of idx. */
        int b = idx;
        for (int t = NOBS - 1; t >= 1; t--) {
            b = A[(size_t)t * N + b];
            traj[t] = X[(size_t)t * N + 0];
        }
        traj[0] = X[b];
        if (info) info[2] = b;
    }
    *log_like_out = log_like;
    if (!X_out) free(X);
    if (!W_out) free(W);
    if (!A_out) free(A);
    free(ancestors);
    free(new_idx);
    free(xnew);
    free(lw);
    free(sh);
    free(cum);
    return 0;
}

/*
 * Correlated importance sampler for the random-effects model,
 * random_effects.pyx:21-104.  rvp flat layout rvp[i + j*NOBS].
 * Outputs: filt[NOBS], log_like[1], traj[NOBS], gradient[2], info[2] = {idx, oob}.
 */
int oracle_importance_discrete(const double *obs, const double *params, double rvr,
                               const double *rvp, int N, int NOBS, double *filt,
                               double *log_like_out, double *traj, double *gradient, int *info)
{
    double *particles = (double *)malloc((size_t)N * NOBS * sizeof(double));
    double *weights = (double *)calloc((size_t)N, sizeof(double));
    double *unw = (double *)calloc((size_t)N, sizeof(double));
    double *shw = (double *)calloc((size_t)N, sizeof(double));
    if (!particles || !weights || !unw || !shw) return 1;
    for (int i = 0; i < NOBS; i++) {
        filt[i] = 0.0;
        traj[i] = 0.0;
    }
    gradient[0] = 0.0;
    gradient[1] = 0.0;
    const double mu = params[0], sigma = params[1];

    /* :54-56 */
    for (int i = 0; i < NOBS; i++)
        for (int j = 0; j < N; j++)
            particles[(size_t)i + (size_t)j * NOBS] = mu + sigma * rvp[(size_t)i + (size_t)j * NOBS];
    /* :63-67 */
    for (int i = 0; i < NOBS; i++)
        for (int j = 0; j < N; j++) {
            double gw = norm_logpdf(obs[i], particles[(size_t)i + (size_t)j * NOBS], 1.0);
            if (isfinite(gw)) unw[j] += gw;
        }
    /* :69-76 */
    double max_weight = oracle_my_max(unw, N);
    double norm_factor = 0.0;
    for (int j = 0; j < N; j++) {
        shw[j] = exp(unw[j] - max_weight);
        if (isfinite(shw[j])) norm_factor += shw[j];
        else shw[j] = 0.0;
    }
    /* :79 (note the NOBS factor) */
    double log_like = max_weight + log(norm_factor) - NOBS * log((double)N);
    /* :82-85 */
    for (int j = 0; j < N; j++) {
        weights[j] = shw[j] / norm_factor;
        for (int i = 0; i < NOBS; i++)
            filt[i] += weights[j] * particles[(size_t)i + (size_t)j * NOBS];
    }
    /* :88-90 */
    int idx = oracle_sample_particle(weights, rvr, N);
    int oob = 0;
    if (idx >= N) {
        oob = 1;
        idx = N - 1;
    }
    if (info) {
        info[0] = idx;
        info[1] = oob;
    }
    for (int i = 0; i < NOBS; i++) traj[i] = particles[(size_t)i + (size_t)idx * NOBS];
    /* :93-99 */
    for (int j = 0; j < N; j++)
        for (int i = 0; i < NOBS; i++) {
            double p = particles[(size_t)i + (size_t)j * NOBS];
            double g_mu = pow(sigma, -2.0) * (p - mu);
            gradient[0] += weights[j] * g_mu;
            double g_sigma = pow(sigma, -2.0) * pow(p - mu, 2.0) - 1.0;
            gradient[1] += weights[j] * g_sigma;
        }
    *log_like_out = log_like;
    free(particles);
    free(weights);
    free(unw);
    free(shw);
    return 0;
}

/* subsampling.pyx:34-51: m sorted uniforms -> m data indices in [0, n) */
int oracle_stratified(const double *rnd, int m, int n, int *indices)
{
    double *cum = (double *)malloc((size_t)n * sizeof(double));
    if (!cum) return 1;
    for (int i = 0; i < n; i++) cum[i] = (i + 1.0) / n;
    int cur = 0;
    for (int j = 0; j < m; j++) {
        double cpoint = (rnd[j] + j) / m;
        while (cum[cur] < cpoint && cur < n - 1) cur++;
        indices[j] = cur;
    }
    free(cum);
    return 0;
}
