// sv_grid.cuh -- the grid kernel (sv_grid.cu): one smoother evaluation (the SV model or another model of
// pf_model.cuh) as one persistent cooperative launch, one tile of the sorted generation per CTA
#pragma once
#include <cuda_runtime.h>
#include <stddef.h>

namespace pmmh {
int sv_grid_ctas(int n, int sm_count, int ctas);
bool sv_grid_eligible(int nobs, int n, int lag, int G);
size_t sv_grid_ws_bytes(int nobs, int n, int lag, int G, int hist, int hess = 0);
int sv_grid_run(const double* d_obs, const double* d_params, const double* d_rvr, const double* d_u, int nobs,
                int n, int lag, int G, double* d_filt, double* d_smo, double* d_ll, double* d_grad, double* d_traj,
                long long* d_diag, double* d_xh, int* d_ah, void* d_ws, size_t ws_bytes, long long* d_prof,
                cudaStream_t st, int u_chunk_steps = 0, const int* d_u_flag = nullptr,
                double* d_hess1 = nullptr, double* d_hess2 = nullptr,   // both given: the Hessian branch (SV only)
                int model = 0);   // PMMH_MODEL_* (pf_model.cuh): the grid kernel instantiated for that model
int sv_grid_read_info(const void* d_ws, int nobs, int n, int lag, int G, int hist, long long* h_info);
}  // namespace pmmh
