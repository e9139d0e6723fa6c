/*
 * pmmh_qn.h -- C ABI of libpmmh_qn_b200.so, the B200 (sm_100a) implementation of the
 * likelihood-estimation hot path of compops/pmmh-qn.
 *
 * Every entry point replaces one native call the reference's Python estimator classes make
 * into its Cython extensions (paths relative to /root/reference/python):
 *
 *   pmmh_flps_sv_corr            flps_sv_corr(obs, params, rvr, rvp, compute_hessian)
 *                                state/particle_methods/stochastic_volatility.pyx:205,
 *                                called at state/particle_methods/cython.py:97
 *   pmmh_bpf_sv_corr             bpf_sv_corr(obs, params, rvr, rvp)
 *                                ...stochastic_volatility.pyx:61, called at cython.py:57,63
 *   pmmh_sv_workspace_bytes      (new) the reference malloc()s scratch inside each call
 *                                (:208-238); here the caller owns one reusable workspace
 *   pmmh_flps_sv_corr_streamed   the same call fed straight from the sampler's host array
 *                                (copies overlap the kernel)
 *   pmmh_split_rvs               rvs.flatten() / rvs[NOBS:] of cython.py:54-56,89-91 plus
 *                                the change to the device's time-major layout
 *   pmmh_norm_cdf                scipy.stats.norm.cdf of cython.py:55,90 / standard.py:52,75
 *   pmmh_importance_discrete     importance_discrete(obs, params, rvr, rvp)
 *                                state/importance_sampling/random_effects.pyx:21,
 *                                called at state/importance_sampling/cython.py:59,89
 *   pmmh_crank_nicolson          _propose_rvs, parameter/mcmc/base_class.py:221-241
 *   pmmh_subsample_indices       np.sort(norm.cdf(u)) + stratified(rnd)
 *                                state/direct/standard.py:52-53,75-76, subsampling.pyx:34-51
 *   pmmh_logistic_loglike        LogisticRegressionModel.get_loglike_gradient
 *                                models/logistic_regression.py:108-176
 *   pmmh_svsplit_*               (new) the same smoother with its particles split over the GPUs of
 *                                one box; phases of one time step, see below
 *   pmmh_*_host                  the same calls with HOST buffers in the reference's own
 *                                layouts (what a cgo/ctypes/Cython stub would bind 1:1)
 *
 * Conventions: plain pointers and sizes; `d_` = device memory, no prefix = host memory;
 * all reals are IEEE fp64; `stream` is a cudaStream_t passed as void* (NULL = default
 * stream); functions are asynchronous on `stream` unless named *_host; return value 0 on
 * success, non-zero otherwise (pmmh_last_error() gives the text).  The reference's estimator
 * contract maps non-zero / non-finite results to `return False`
 * (state/particle_methods/cython.py:71-75,133-137).  No function allocates device memory
 * except the *_host convenience wrappers.  There is no CPU fallback.
 */
#ifndef PMMH_QN_H
#define PMMH_QN_H

#include <stddef.h>

#ifdef __cplusplus
extern "C" {
#endif

#define PMMH_OK 0
#define PMMH_ERR_INVALID 1      /* bad sizes / null pointers */
#define PMMH_ERR_WORKSPACE 2    /* workspace too small */
#define PMMH_ERR_CUDA 3         /* CUDA runtime error */
#define PMMH_ERR_NO_DEVICE 4    /* no sm_100 device */

/* pmmh_bpf_sv_corr leverage-term read (SURVEY.md Q2) */
#define PMMH_BPF_PARITY 0       /* reference behaviour: reads the time-i column (serial chain) */
#define PMMH_BPF_INTENDED 1     /* the evidently intended time i-1 read; NOT reference parity */

/* diag[] layout (int64 per problem) written by the SV kernels */
#define PMMH_DIAG_NEAR_TIES 0   /* ancestor decisions within 64 ulp of a cumulative-weight tie */
#define PMMH_DIAG_MAX_BIN 1     /* largest sort-bin occupancy */
#define PMMH_DIAG_STATUS 2      /* 0 ok, 1 degenerate particle cloud (evaluation abandoned) */
#define PMMH_DIAG_KEY_TIES 3    /* equal keys met while sorting */
#define PMMH_DIAG_WAVEFRONT 4   /* bpf parity mode: deepest dependency chain */
#define PMMH_DIAG_SOFT_TIES 4   /* flps, grid kernel: ancestor decisions whose margin is below the bound on the
                                   difference between the reference's sequential cumulative sums and parallel ones
                                   (eps N (4 + 2 sqrt N) child-index units): only these can differ from the reference */
#define PMMH_DIAG_TRAJ_IDX 5    /* bpf: sampled trajectory index */
#define PMMH_DIAG_KERNEL 6      /* kernel that produced the outputs: 1 general, 2 exchange, 3 chain, 4 split (streaming), 5 grid */
#define PMMH_DIAG_FAST_INFO 7   /* exchange kernel: abandon reason (1 run / 2 chunk overflow) |
                                   step << 8 | longest mailbox run << 32 */
#define PMMH_DIAG_COUNT 8

int pmmh_version(void);
const char* pmmh_last_error(void);
/* sm count / compute capability of the current device */
int pmmh_device_info(int* sm_count, int* cc_major, int* cc_minor);

/* ---------------------------------------------------------------- SV particle methods -- */

/* Kernel selection for pmmh_flps_sv_corr and pmmh_flps_sv_corr_streamed (per host thread; default 0).
 *   0  automatic, tried in this order:
 *      chain kernel (one CTA per problem, everything in shared memory): n_particles <= 4096, lag <= 10,
 *        ctas_per_problem <= 1 (device-resident u only);
 *      grid kernel (one persistent launch, one tile of the sorted generation per CTA): one problem,
 *        ctas_per_problem == 0, N >= 2^14 while a tile of N / #SMs fits one CTA (N <= ~1.06 M);
 *      streaming kernels: one problem without Hessian or history, ctas_per_problem == 0, N >= 2^20 (no
 *        size limit; with device-resident u: variant 5 below N = 2^23, variant 4 from there on; host-streamed:
 *        variant 5, and only where the exchange kernel does not take the size);
 *      exchange kernel (two exchanges per step between the CTAs of a team): without Hessian, for more than
 *        one CTA per problem (N > 1024 alone, N > 4096 in a batch, or ctas_per_problem > 1), up to ~1.16 M
 *        particles;
 *      general kernel: everything else (the host-streamed entry refuses instead), and after each of the
 *        kernels above the fallback pass for problems they abandon (degenerate clouds)
 *   1  general kernel only
 *   2  exchange kernel where eligible, without the fallback pass (else the general kernel)
 *   3  chain kernel where eligible, without the fallback pass (else the general kernel)
 *   4  streaming kernels (sv_split.cu driven on one device: ~11 launches per time step, no
 *      persistent kernel) for one problem with compute_hessian == 0, no history output and
 *      ctas_per_problem == 0, without the fallback pass (else the general kernel)
 *   5  the same with path storage: a generation is stored once in birth order (value + parent
 *      row), no records are copied; the lagged ancestors are reached through jump tables
 *   6  grid kernel for one problem (also with compute_hessian) where a tile fits one CTA, without the
 *      fallback pass (else the general kernel)
 * pmmh_flps_sv_corr_streamed has no fallback pass: 0 as above, 2 the exchange kernel, 5 the streaming
 * kernels from N = 2^20 on, 6 the grid kernel with ctas_per_problem == 0; sizes no kernel takes and the other
 * algorithms are refused (pmmh_sv_streamed_eligible).
 * Call before pmmh_sv_workspace_bytes: the workspace size depends on it. */
int pmmh_sv_set_algorithm(int algorithm);

/* Development hook: d_clocks = device buffer of [n_ctas][16] int64 (or NULL to switch off);
 * the exchange kernel adds the SM clock cycles each CTA spent per phase. */
int pmmh_sv_debug_profile(long long* d_clocks);

/* Bytes of device workspace pmmh_flps_sv_corr / pmmh_bpf_sv_corr need for these sizes.
 * mode: 0 = flps, 1 = bpf.  have_history: caller passes d_x_hist / d_a_hist.
 * ctas_per_problem: 0 = choose automatically. */
int pmmh_sv_workspace_bytes(int n_obs, int n_particles, int lag, int batch, int compute_hessian,
                            int mode, int have_history, int ctas_per_problem, size_t* bytes);

/* Fixed-lag particle smoother for `batch` independent (params, u) problems.
 *   d_obs      [n_obs] (obs_stride = 0) or [batch][obs_stride]
 *   d_params   [batch][4]  = mu, phi, sigma_v, rho
 *   d_rvr      [batch][n_obs]  uniforms for the resampler (Phi already applied)
 *   d_u        [batch][n_obs][n_particles]  time-major: d_u[t][j] == rvp[t + j*n_obs]
 * outputs (per problem): d_filt[n_obs], d_smo[n_obs], d_log_like[1], d_gradient[4][n_obs],
 *   d_traj[n_obs], d_hess1[4][4], d_hess2[4][4], d_diag[PMMH_DIAG_COUNT];
 *   optional d_x_hist / d_a_hist [n_obs][n_particles]: sorted particles and composed
 *   one-step ancestors of every time step (both NULL: only a ring of depth lag+1 is kept). */
int pmmh_flps_sv_corr(const double* d_obs, long long obs_stride, const double* d_params,
                      const double* d_rvr, const double* d_u, int n_obs, int n_particles, int lag,
                      int batch, int compute_hessian, double* d_filt, double* d_smo,
                      double* d_log_like, double* d_gradient, double* d_traj, double* d_hess1,
                      double* d_hess2, long long* d_diag, double* d_x_hist, int* d_a_hist,
                      void* d_workspace, size_t workspace_bytes, int ctas_per_problem, void* stream);

/* The same evaluation (log-likelihood + gradient, one problem) with the auxiliary variables still
 * in HOST memory -- what the samplers hand to estimator.smoother(model, rvs={'rvs': ndarray})
 * (mh_quasi_newton.py:333, state/particle_methods/cython.py:89-91).  h_rvs is the reference's
 * (n_obs, N+1) row-major array (pinned memory makes the copies asynchronous).  The copy engine
 * moves it in chunks of time steps on an internal stream into d_stage (particle-major chunks, no
 * layout kernel) while the persistent kernel is already running; the kernel waits for a chunk only
 * when it reaches it, and the caller's stream ends after the last copy.  d_rvr = Phi of the first
 * n_obs flat entries (computed by the caller as in cython.py:90).  Kernel by size: the grid kernel
 * where a tile fits one SM (2^14 <= N <= ~1.06 M; slots of 256 time steps filled by copies that get
 * shorter towards the end of the series, so that the kernel ends a few ms after the last copy), else the exchange
 * kernel where it is eligible (chunks of 64), else the streaming kernels, whose host-driven step
 * loop waits for a chunk's event when it enters it (pmmh_sv_streamed_eligible tells whether a size
 * is taken at all).  There is no fallback inside: if d_diag[PMMH_DIAG_STATUS] == 1 afterwards,
 * upload the array and call pmmh_flps_sv_corr.  d_stage needs pmmh_sv_stage_bytes() bytes and must
 * stay untouched until the stream has been synchronised; the workspace needs
 * pmmh_sv_streamed_workspace_bytes() bytes.  Not re-entrant per device and host thread: the internal
 * copy stream and its events are per (thread, device) state. */
int pmmh_sv_streamed_workspace_bytes(int n_obs, int n_particles, int lag, int ctas_per_problem, size_t* bytes);
int pmmh_sv_stage_bytes(int n_obs, int n_particles, size_t* bytes);
/* the copy schedule of the host-streamed grid path for a series of n_obs steps (no device needed): the number of
 * pieces (negative: bad arguments); the first max_pieces lengths, in time steps, are written to pieces */
int pmmh_sv_stream_schedule(int n_obs, int* pieces, int max_pieces);
int pmmh_sv_streamed_eligible(int n_obs, int n_particles, int lag, int ctas_per_problem);
int pmmh_flps_sv_corr_streamed(const double* h_rvs, const double* d_obs, const double* d_params,
                               const double* d_rvr, int n_obs, int n_particles, int lag, void* d_stage,
                               size_t stage_bytes, double* d_filt, double* d_smo, double* d_log_like,
                               double* d_gradient, double* d_traj, double* d_hess1, double* d_hess2,
                               long long* d_diag, void* d_workspace, size_t workspace_bytes,
                               int ctas_per_problem, void* stream);

/* The same evaluation (log-likelihood + gradient, one problem, any N) with the auxiliary variables
 * defined by a Philox4x32-10 stream instead of an array: u[t][j] = standard normal number t*N + j of
 * stream (seed, philox_offset), exactly what pmmh_crank_nicolson draws with d_xi == NULL.  At
 * N = 2^26, T = 1000 the array of flps_sv_corr's rvp argument would be 537 GB.  d_rvr as above.
 * Runs on the streaming kernels with path storage. */
int pmmh_flps_sv_corr_philox_workspace_bytes(int n_obs, int n_particles, int lag, size_t* bytes);
int pmmh_flps_sv_corr_philox(const double* d_obs, const double* d_params, const double* d_rvr,
                             unsigned long long seed, unsigned long long philox_offset, int n_obs,
                             int n_particles, int lag, double* d_filt, double* d_smo, double* d_log_like,
                             double* d_gradient, double* d_traj, long long* d_diag, void* d_workspace,
                             size_t workspace_bytes, void* stream);

/* Model-generic fixed-lag smoother (log-likelihood + gradient): the same algorithm as pmmh_flps_sv_corr
 * (sorted correlated systematic resampling, fixed-lag score terms, tail, quirk Q1) with the
 * model's propagation, log-weight and score formulas plugged in through the device-function interface
 * of csrc/pf_model.cuh -- the three things python/README.md:73-76 tells a user to change in the Cython
 * smoother for another scalar-state model.  2 <= lag <= 10.  The reference's pairing quirks Q5 / Q6 apply to
 * PMMH_MODEL_SV_LEVERAGE only (parity).  Model 4 pairs them predictively (PMMH_MODEL_LINEAR_GAUSSIAN_FA_GRAD
 * below).  Models 1 and 2 pair the fixed-lag terms exactly: gradient[k][s] holds the
 * expectation of d/dtheta_k [log p(x_s | x_{s-1}) + log p(y_s | x_s)] (y_s = obs[s]) under the weights of generation
 * min(s + lag - 2, n_obs - 1), gradient[k][0] = 0, and the sum over s estimates the score of the log-likelihood;
 * smo[t] is the mean of x_t under the weights of generation min(t + lag - 1, n_obs - 1).  For model 1 these are
 * E[. | y_1 .. y_c] of that generation c; model 2's weights condition on one more observation.  The kernel (d_diag[PMMH_DIAG_KERNEL]):
 *   3  chain kernel, one CTA per problem: 2 <= n_particles <= 4096, any batch;
 *   5  grid kernel, one persistent launch over the GPU: batch == 1, n_obs >= 2 lag and a tile of
 *      n_particles / min(SMs, ceil(n_particles / 2048)) particles fits one CTA (<= 7168: up to 1,060,864
 *      particles on 148 SMs); d_x_hist / d_a_hist as on pmmh_flps_sv_corr's grid kernel;
 * other sizes are refused (PMMH_ERR_INVALID; also by pmmh_flps_model_workspace_bytes, which returns the size
 * with history for the kernel the call runs).  d_params [batch][4] (unused slots ignored), gradient [4][n_obs]
 * (unused rows 0).  PMMH_MODEL_SV_LEVERAGE gives bit-identical results to pmmh_flps_sv_corr run on the same
 * kernel: the chain kernel (algorithm 3) up to 4096 particles, the grid kernel (algorithm 6, or 0 from 2^14 on)
 * above.  No fallback inside: d_diag[PMMH_DIAG_STATUS] == 1 reports an abandoned problem (chain kernel:
 * log-likelihood NaN). */
#define PMMH_MODEL_SV_LEVERAGE 0      /* mu, phi, sigma_v, rho   (models/stochastic_volatility.py) */
#define PMMH_MODEL_LINEAR_GAUSSIAN 1  /* phi, sigma_v, sigma_e: x' = phi x + sigma_v v, y = x + sigma_e e */
#define PMMH_MODEL_LINEAR_GAUSSIAN_FA 2 /* the same model as a FULLY ADAPTED particle filter: pass the observations shifted by
                                         one (obs'[t] = obs[t + 1], n_obs - 1 entries); log-likelihood of y_2..y_T given y_1 */
/* PMMH_MODEL_LINEAR_GAUSSIAN_FA_GRAD: model 2's fully adapted filter with a fixed-lag gradient.  Same inputs as model 2
 * (the shifted series obs' = obs[1:], x_0 = 0, y_t = obs[t]); d_filt, d_smo, d_log_like, d_traj, d_diag and the history
 * are bit-identical to model 2's.  Gradient rows 0..2 are d/d(phi, sigma_v, sigma_e), row 3 is 0, and slot k holds the
 * contribution of obs'[k] = y_{k+1}: for k <= n_obs - 2 the expectation of
 * d/dtheta [log p(x_{k+1} | x_k) + log p(obs'[k] | x_{k+1})] under the weights of generation c(k) = min(k + lag - 1,
 * n_obs - 1), and for k = n_obs - 1 that of d/dtheta log N(obs'[n_obs - 1]; phi x_{n_obs - 1}, sigma_v^2 + sigma_e^2)
 * under the final weights.  The slots sum to an estimate of the score of the FULL log-likelihood log p(y_1 .. y_T), so the
 * gradient needs no correction, while d_log_like still lacks log p(y_1) as for model 2.  pmmh_flps_model_corr and
 * pmmh_flps_model_batch_corr take it on the sizes of model 2 (compute_hessian == 1 is refused); the filter entries run
 * model 2's filter for it. */
#define PMMH_MODEL_LINEAR_GAUSSIAN_FA_GRAD 4   /* id 3 is unassigned: every entry refuses it as an unknown id */
/* PMMH_MODEL_LINEAR_GAUSSIAN_FA_HESS: model 4 with a fixed-lag Hessian.  Every output model 4 has is bit-identical to
 * model 4's on every entry and shape (with compute_hessian 0 or 1); the filter entries run model 2's filter for it.
 * pmmh_flps_model_batch_corr with compute_hessian == 1 (on the grid kernel: batch 1 and small n_particles included)
 * writes d_hess1 / d_hess2 [4][4] (rows and columns 0..2 = phi, sigma_v, sigma_e; row and column 3 are 0) by Louis'
 * identity on the gradient's pairs and weights: with s_k the term of gradient slot k and H_k its matrix of second
 * derivatives, hess1 = sum_k E[H_k] and hess2 = sum_k E[s_k s_k' + alpha_k s_k' + s_k alpha_k'], where alpha_k is the
 * sum of the slot terms 0 .. k-1 along the lineage of the particle read (the score accumulated along its genealogy),
 * each expectation under the weights that read slot k.  hess1 + hess2 - g g', g = the sum of the gradient slots,
 * estimates the Hessian of the full log-likelihood log p(y_1 .. y_T).  alpha runs along the whole genealogy, so the
 * estimate's variance grows with n_obs / n_particles. */
#define PMMH_MODEL_LINEAR_GAUSSIAN_FA_HESS 6   /* id 5 is unassigned */
/* PMMH_MODEL_SV_LEVERAGE_EXACT: the SV model with the exact fixed-lag score and a fixed-lag Hessian.  Same inputs as
 * PMMH_MODEL_SV_LEVERAGE (the unshifted series, params mu, phi, sigma_v, rho); d_filt, d_log_like, d_traj, d_diag and the
 * history are bit-identical to model 0's on the same kernel, and the filter entries run model 0's filter for it.  The
 * gradient is over the reference's free parameters (mu, atanh phi, log sigma_v, atanh rho), and slot k holds the
 * expectation of d/dtheta log p(x_{k+1} | x_k, obs[k]) -- the transition scored with the leverage observation its
 * propagation read -- under the weights of generation c(k) = min(k + lag - 1, n_obs - 1); slot n_obs - 1 is 0.  The
 * pair (x_0, x_1) takes the total derivative through x_0 = mu.  The slots sum to an estimate of the score of log_like
 * (model 0 pairs the terms as the reference does, obs[k - 1] and tail pairs re-added: a biased estimate when rho != 0).
 * d_smo[k] is the mean of x_k under the same weights.  pmmh_flps_model_batch_corr with compute_hessian == 1 (grid kernel)
 * writes d_hess1 / d_hess2 [4][4] over the same parameters by Louis' identity as for
 * PMMH_MODEL_LINEAR_GAUSSIAN_FA_HESS; hess1 + hess2 - g g' estimates the Hessian of log_like.  Sizes as for model 0 on
 * the model entries. */
#define PMMH_MODEL_SV_LEVERAGE_EXACT 8   /* id 7 is unassigned: every entry refuses it as an unknown id */
int pmmh_flps_model_workspace_bytes(int n_obs, int n_particles, int lag, int batch, size_t* bytes);
int pmmh_flps_model_corr(int model_id, const double* d_obs, long long obs_stride, const double* d_params,
                         const double* d_rvr, const double* d_u, int n_obs, int n_particles, int lag, int batch,
                         double* d_filt, double* d_smo, double* d_log_like, double* d_gradient, double* d_traj,
                         long long* d_diag, double* d_x_hist, int* d_a_hist, void* d_workspace,
                         size_t workspace_bytes, void* stream);

/* Model-generic particle filter: the log-likelihood without the fixed-lag smoother.  The filter half of
 * pmmh_flps_model_corr, unchanged (Q1 initial state, sorted correlated systematic resampling, the model's
 * propagation and log-weight, Q10 / Q11 trajectory); no genealogy, score terms or tail, and no lag.  On every
 * shape both entries take, d_log_like, d_filt, d_traj, d_diag and the history d_x_hist / d_a_hist are
 * bit-identical to pmmh_flps_model_corr's for any lag.  The kernel (d_diag[PMMH_DIAG_KERNEL]):
 *   3  chain kernel: n_obs >= 2, 2 <= n_particles <= 4096, any batch (no workspace: 0 bytes, d_workspace may be NULL);
 *   5  grid kernel: n_obs >= 2, batch == 1 and a tile of n_particles / min(SMs, ceil(n_particles / 2048))
 *      particles fits one CTA (<= 7168: up to 1,060,864 particles on 148 SMs), on the same tiles as
 *      pmmh_flps_model_corr; its workspace has no genealogy records or payloads;
 * other sizes are refused (PMMH_ERR_INVALID; also by pmmh_filter_model_workspace_bytes, which returns the size
 * with history for the kernel the call runs).  No fallback inside: d_diag[PMMH_DIAG_STATUS] == 1 reports an
 * abandoned problem. */
int pmmh_filter_model_workspace_bytes(int n_obs, int n_particles, int batch, size_t* bytes);
int pmmh_filter_model_corr(int model_id, const double* d_obs, long long obs_stride, const double* d_params,
                           const double* d_rvr, const double* d_u, int n_obs, int n_particles, int batch,
                           double* d_filt, double* d_log_like, double* d_traj, long long* d_diag,
                           double* d_x_hist, int* d_a_hist, void* d_workspace, size_t workspace_bytes,
                           void* stream);

/* Batches on the grid kernel: `batch` problems of one shape, each on its own team of G = ceil(n_particles / 2048)
 * CTAs (capped at the SM count: the one-problem grid run's G, hence its tiles and its summation order), so that
 * every output of problem b -- d_log_like, d_filt, d_smo, d_gradient, d_traj, d_hess1 / d_hess2, d_diag and the
 * history -- is bit-identical to the grid kernel run on that problem alone (pmmh_flps_model_corr /
 * pmmh_filter_model_corr with batch 1, and for PMMH_MODEL_SV_LEVERAGE pmmh_flps_sv_corr at algorithm 6).  The
 * problems run in waves of nteams = min(batch, floor(SMs / G)) teams, one cooperative launch per wave, followed by
 * the reduction and output kernels of each problem (per problem: 2 launches for the filter, 4 for the smoother, 6
 * with the Hessian).  Each team has its own workspace slice, barrier and status word: a problem whose particle
 * cloud degenerates is abandoned alone (d_diag[b][PMMH_DIAG_STATUS] == 1; there is no fallback pass), the others
 * finish.  d_diag[b][PMMH_DIAG_KERNEL] == 5.
 *   Layouts: those of pmmh_flps_model_corr / pmmh_filter_model_corr -- d_obs [n_obs] (obs_stride 0) or
 * [batch][obs_stride], d_params [batch][4], d_rvr [batch][n_obs], d_u [batch][n_obs][n_particles]; outputs per
 * problem d_filt, d_smo, d_traj [n_obs], d_log_like [1], d_gradient [4][n_obs], d_hess1 / d_hess2 [4][4],
 * d_diag [PMMH_DIAG_COUNT]; optional d_x_hist / d_a_hist [batch][n_obs][n_particles], given together.
 *   Shapes: any batch >= 1 with a tile of n_particles / G particles that fits one CTA (up to 7168 particles per
 * CTA); the smoother needs 2 <= lag <= 10 and n_obs >= 2 lag, the filter n_obs >= 2.  compute_hessian == 1 (the
 * Hessian branch; d_hess1 / d_hess2 required) is taken for PMMH_MODEL_SV_LEVERAGE,
 * PMMH_MODEL_LINEAR_GAUSSIAN_FA_HESS and PMMH_MODEL_SV_LEVERAGE_EXACT only; with 0 the
 * Hessian outputs may be NULL and are not written.  Anything else is refused with PMMH_ERR_INVALID, by the
 * workspace queries too; a workspace below the query's size gives PMMH_ERR_WORKSPACE.
 *   Workspace: min(batch, nteams) slices of the one-problem grid workspace with history (per slice:
 * pmmh_flps_model_workspace_bytes / pmmh_filter_model_workspace_bytes at batch 1 and the same sizes; the Hessian
 * slice is larger).
 *   Speed (B200, T = 1000, lag 10; profiles/r6_grid_batch_T1000.jsonl): see INTEGRATION.md. */
int pmmh_flps_model_batch_workspace_bytes(int n_obs, int n_particles, int lag, int batch, int compute_hessian,
                                          size_t* bytes);
int pmmh_flps_model_batch_corr(int model_id, const double* d_obs, long long obs_stride, const double* d_params,
                               const double* d_rvr, const double* d_u, int n_obs, int n_particles, int lag, int batch,
                               int compute_hessian, double* d_filt, double* d_smo, double* d_log_like,
                               double* d_gradient, double* d_traj, double* d_hess1, double* d_hess2, long long* d_diag,
                               double* d_x_hist, int* d_a_hist, void* d_workspace, size_t workspace_bytes,
                               void* stream);
int pmmh_filter_model_batch_workspace_bytes(int n_obs, int n_particles, int batch, size_t* bytes);
int pmmh_filter_model_batch_corr(int model_id, const double* d_obs, long long obs_stride, const double* d_params,
                                 const double* d_rvr, const double* d_u, int n_obs, int n_particles, int batch,
                                 double* d_filt, double* d_log_like, double* d_traj, long long* d_diag,
                                 double* d_x_hist, int* d_a_hist, void* d_workspace, size_t workspace_bytes,
                                 void* stream);

/* Bootstrap particle filter (filter only).  read_mode: PMMH_BPF_PARITY / PMMH_BPF_INTENDED. */
int pmmh_bpf_sv_corr(const double* d_obs, long long obs_stride, const double* d_params,
                     const double* d_rvr, const double* d_u, int n_obs, int n_particles, int batch,
                     int read_mode, double* d_filt, double* d_log_like, double* d_traj,
                     long long* d_diag, double* d_x_hist, int* d_a_hist, void* d_workspace,
                     size_t workspace_bytes, int ctas_per_problem, void* stream);

/* rvs [batch][n_obs][n_particles + 1] row-major (the reference's dim_rvs) ->
 *   d_r_raw [batch][n_obs]   the first n_obs FLAT entries (not yet Phi-transformed)
 *   d_u     [batch][n_obs][n_particles] time-major view of the flat remainder */
int pmmh_split_rvs(const double* d_rvs, int n_obs, int n_particles, int batch, double* d_r_raw,
                   double* d_u, void* stream);

/* out[k] = Phi(in[k]) (standard normal cdf), in place allowed */
int pmmh_norm_cdf(const double* d_in, double* d_out, long long n, void* stream);

/* ------------------------------------------------------ random-effects importance sampler -- */

/*   d_obs [n_obs] (obs_stride 0) or [batch][obs_stride]; d_params [batch][2] = mu, sigma;
 *   d_rvr [batch] uniforms; d_rvp [batch][n_obs * n_particles] in the reference's flat layout
 *   rvp[i + j*n_obs].  outputs per problem: d_filt[n_obs], d_log_like[1], d_traj[n_obs],
 *   d_gradient[2], d_traj_idx[1]. */
int pmmh_importance_discrete(const double* d_obs, long long obs_stride, const double* d_params,
                             const double* d_rvr, const double* d_rvp, int n_obs, int n_particles,
                             int batch, double* d_filt, double* d_log_like, double* d_traj,
                             double* d_gradient, int* d_traj_idx, void* stream);

/* ------------------------------------------------------------------ Crank-Nicolson on u -- */

/* d_out[k] = sqrt(1 - sigma_u^2) * d_u[k] + sigma_u * xi[k].  If d_xi is NULL, xi is drawn on
 * the device (Philox4x32-10 + Box-Muller, counter = philox_offset + k/2, key = seed). */
int pmmh_crank_nicolson(const double* d_u, const double* d_xi, double* d_out, long long n,
                        double sigma_u, unsigned long long seed, unsigned long long philox_offset,
                        void* stream);

/* ------------------------------------------------------------- data-subsampling estimator -- */

/* Workspace bytes for pmmh_subsample_indices. */
int pmmh_subsample_workspace_bytes(int m, size_t* bytes);

/* d_u [m] standard normals -> d_idx [m] data indices in [0, n_data):
 * sort(Phi(u)) then the stratified merge walk in closed form.  If apply_cdf == 0, d_u is
 * taken as already-transformed uniforms.  d_sorted (optional, [m]) receives the sorted
 * uniforms. */
int pmmh_subsample_indices(const double* d_u, int m, int n_data, int apply_cdf, int* d_idx,
                           double* d_sorted, void* d_workspace, size_t workspace_bytes,
                           void* stream);

/* Subsampled logistic log-likelihood, gradient and (optionally) Hessian over the rows
 * d_idx[0..m) that fall inside [row_begin, row_end) (the shard this device owns; pass 0 and
 * n_data for all).  d_x is [*][d] row-major and holds rows row_begin..row_end-1.
 * d_out [1 + d + d*d]: log_like, gradient[d], hessian[d][d] (Hessian = -sum s_i x_i x_i^T as
 * in logistic_regression.py:155-165; zero-filled when compute_hessian == 0).
 * The sums are reductions (atomic-free, fixed order); d_out is overwritten. */
int pmmh_logistic_workspace_bytes(int m, int d, int compute_hessian, size_t* bytes);
int pmmh_logistic_loglike(const double* d_x, const double* d_y, const int* d_idx, int m, int d,
                          long long row_begin, long long row_end, const double* d_beta,
                          int compute_hessian, double* d_out, void* d_workspace,
                          size_t workspace_bytes, void* stream);

/* ------------------------------------------- one SV particle filter split over several GPUs -- */

/* BASELINE.json configs[4] / SURVEY.md 8e: a single flps_sv_corr evaluation
 * (state/particle_methods/stochastic_volatility.pyx:205-655; called at
 * state/particle_methods/cython.py:97) whose N particles do not fit, or are not wanted, on one
 * GPU.  NEW API -- the reference has no multi-device call.  Rank r of `world` owns a contiguous
 * value range of the sorted generation.  The library provides the device phases of one time step;
 * the three exchanges between them are issued by the host layer on the same stream (NCCL through
 * torch.distributed in pmmh-qn_b200/state/particle_methods/split.py):
 *
 *   weights(t) -> all-gather [world][4] -> children(t+1) -> all-gather [world][4096] int ->
 *   plan (+ counts to pinned host memory) -> pack -> all-to-all-v of records -> sort -> weights(t+1)
 *
 * Buffers the caller owns (per rank): d_xs [cap] sorted values, d_perm [cap] sorted position ->
 * arrival row, two record buffers [cap][LR] (current / next generation, LR = lag, or 1 when
 * lag == 0 = log-likelihood and filter means only), d_send [cap_children][LR], d_sums [n_obs][8],
 * d_shift [n_obs], d_xmin [n_obs], and the workspace.  cap_particles / cap_children bound the
 * arrivals and the children of one rank; exceeding them sets diag[PMMH_DIAG_STATUS] (4 = children,
 * 8 = arrivals, 16 = degenerate sort bin, 1/2 = non-finite weights) and the evaluation must be
 * abandoned (the estimator returns False, as state/particle_methods/cython.py:71-75 does).
 * u: d_u = [n_obs][N] time-major on every rank, or NULL = Philox stream (seed, philox_offset),
 * element t*N + j as pmmh_crank_nicolson draws it. */
int pmmh_svsplit_workspace_bytes(long long cap_particles, long long cap_children, size_t* bytes);
/* generation 0 (Q1: every particle = mu); n_local = particles this rank starts with */
int pmmh_svsplit_init(void* d_ws, size_t ws_bytes, long long n_total, int n_obs, int world, int rank,
                      int lag, long long cap_particles, long long cap_children, int n_local,
                      const double* d_params, double* d_xs, int* d_perm, double* d_rec, void* stream);
/* weights of generation t (:427-470): d_sums[t][0..6] = local sums of sh, sh x, sh curr, sh g_0..3;
 * d_gather_send[4] = (sum sh, n_local, min x, max x); d_sh_save (optional, [n_local]) keeps sh */
int pmmh_svsplit_weights(void* d_ws, size_t ws_bytes, long long cap_particles, long long cap_children,
                         int t, int n_local, int lag, int n_obs, const double* d_obs,
                         const double* d_params, const double* d_xs, const int* d_perm,
                         const double* d_rec, double* d_sums, double* d_gather_send, double* d_sh_save,
                         void* stream);
/* resampling + propagation of the children of the local parents for time t (:694-715, :354-358);
 * d_gather = all-gathered [world][4]; d_hist_send [4096] = local value histogram of the children */
int pmmh_svsplit_children(void* d_ws, size_t ws_bytes, long long cap_particles, long long cap_children,
                          int t, int n_local, const double* d_obs, const double* d_params,
                          const double* d_rvr, const double* d_u, unsigned long long seed,
                          unsigned long long philox_offset, const double* d_gather, const double* d_xs,
                          int* d_hist_send, double* d_shift, double* d_xmin, void* stream);
/* splitters and counts from the all-gathered histograms [world][4096]; h_counts (pinned host,
 * 2*world + 4 ints, valid after the stream is synchronised; may be NULL when world == 1) = send counts per destination, receive
 * counts per source, arrivals, children, fine sort bins, status */
int pmmh_svsplit_plan(void* d_ws, size_t ws_bytes, long long cap_particles, long long cap_children,
                      int world, const int* d_hist, int* h_counts, void* stream);
/* records of the children grouped by destination rank -> d_send (rows of LR doubles); d_send_keys
 * (optional, [cap_children]) receives the values alone in the same order, so that they can be
 * exchanged first and sorted while the records are still in flight */
int pmmh_svsplit_pack(void* d_ws, size_t ws_bytes, long long cap_particles, long long cap_children,
                      const int* d_perm, const double* d_rec, double* d_send, double* d_send_keys,
                      void* stream);
/* the same with the children that stay on this rank written straight into this rank's receive buffers
 * (d_self_rec = the d_rec_new pmmh_svsplit_sort will read, d_self_keys = its d_keys, NULL without
 * d_send_keys) at their arrival slots [sum of the receive counts of the ranks in front, ...): the exchange
 * that follows moves only what crosses ranks; all other send / receive offsets are unchanged */
int pmmh_svsplit_pack_direct(void* d_ws, size_t ws_bytes, long long cap_particles, long long cap_children,
                             const int* d_perm, const double* d_rec, double* d_send, double* d_send_keys,
                             double* d_self_rec, double* d_self_keys, void* stream);
/* argsort of the arrivals (:392-424): d_xs / d_perm of the new generation.  The values come from
 * d_keys [n_arrivals] if given, else from column 0 of d_rec_new; keys_are_children = 1 (world == 1
 * only): arrival e is child e, its value is read from the dense child array in the workspace */
int pmmh_svsplit_sort(void* d_ws, size_t ws_bytes, long long cap_particles, long long cap_children,
                      int n_arrivals, int n_fine, int lag, const double* d_rec_new, const double* d_keys,
                      int keys_are_children, double* d_xs, int* d_perm, void* stream);
/* d_w[p] = d_sh[p] / *d_total (normalised weights of a kept generation, for the tail) */
int pmmh_svsplit_normalise(const double* d_sh, int n_local, const double* d_total, double* d_w,
                           void* stream);
/* tail terms (:540-562, Q6) of the final generation.  d_w_lagged[irel][p] = normalised weight of
 * generation n_obs - lag + irel at the GLOBAL sorted position of local particle p (redistributed
 * by the host layer), irel < lag - 1.  d_tail [lag][8]: [irel][0] = smo term of time
 * n_obs - lag + irel, [irel][1..4] = gradient terms of slot n_obs - 2 lag + 1 + irel (local sums) */
int pmmh_svsplit_tail(void* d_ws, size_t ws_bytes, long long cap_particles, long long cap_children,
                      int n_local, int lag, int n_obs, const double* d_obs, const double* d_params,
                      const int* d_perm, const double* d_rec, const double* d_w_final,
                      const double* d_w_lagged, long long w_lagged_stride, double* d_tail,
                      void* stream);
/* O(T) assembly from the rank-summed d_sums / d_tail: log-likelihood (:537), filter and smoother
 * means, gradient [4][n_obs], trajectory (Q10/Q11) */
int pmmh_svsplit_finish(const double* d_sums, const double* d_shift, const double* d_xmin,
                        const double* d_tail, const double* d_gather_last, int world,
                        const double* d_params, int n_obs, int lag, long long n_total,
                        double* d_log_like, double* d_filt, double* d_smo, double* d_gradient,
                        double* d_traj, void* stream);
/* h_diag[PMMH_DIAG_COUNT] of this rank (synchronises) */
int pmmh_svsplit_diag(void* d_ws, size_t ws_bytes, long long cap_particles, long long cap_children,
                      long long* h_diag);

/* ------------------------------------------------------------------- host-buffer wrappers -- */

/* Same signature shape as the reference's Cython entry point: host arrays in the reference's
 * own layouts (rvp[i + j*n_obs]); copies in, runs on the current device, copies out,
 * synchronises.  gradient is [4][n_obs]. */
int pmmh_flps_sv_corr_host(const double* obs, const double* params, const double* rvr,
                           const double* rvp, int n_obs, int n_particles, int lag,
                           int compute_hessian, double* filt, double* smo, double* log_like,
                           double* gradient, double* traj, double* hess1, double* hess2,
                           long long* diag);
int pmmh_bpf_sv_corr_host(const double* obs, const double* params, const double* rvr,
                          const double* rvp, int n_obs, int n_particles, int read_mode,
                          double* filt, double* log_like, double* traj, long long* diag);
int pmmh_importance_discrete_host(const double* obs, const double* params, double rvr,
                                  const double* rvp, int n_obs, int n_particles, double* filt,
                                  double* log_like, double* traj, double* gradient);
int pmmh_stratified_host(const double* rnd_sorted, int m, int n_data, int* indices);

#ifdef __cplusplus
}
#endif
#endif /* PMMH_QN_H */
