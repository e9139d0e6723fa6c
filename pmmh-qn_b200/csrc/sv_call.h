// sv_call.h -- one evaluation as the C entries of capi.cu receive it: inputs, the source of u, outputs, history,
// workspace and stream.  Host only: the kernels receive SvArgs (sv_filter.cuh) or the grid kernel's GridArgs.
#pragma once
#include <cuda_runtime.h>
#include <stddef.h>

namespace pmmh {
struct SvCall {
    const double* obs;
    long long obs_stride;   // 0: one series shared by the batch
    const double* params;   // [B][4]
    const double* rvr;      // [B][NOBS]
    // u: time-major [B][NOBS][N] (slot == 0), or particle-major slots of `slot` time steps that the copy engine is
    // still filling (host-streamed, B = 1), signalled by the device flag u_flag (steps landed so far: grid and
    // exchange kernels) or by the event slot_ready[c] of each slot (streaming kernels); u == NULL: the Philox stream
    // (seed, philox_offset) (streaming kernel with path storage)
    const double* u;
    int slot;
    const int* u_flag;
    const cudaEvent_t* slot_ready;
    unsigned long long seed, philox_offset;
    double *filt, *smo, *ll, *grad, *traj;
    double *hess1, *hess2;   // NULL where the entry has no Hessian outputs
    long long* diag;
    double* x_hist;          // optional, together with a_hist
    int* a_hist;
    int model;               // model id (the table Models in pf_model.cuh)
    int filter;              // 1: the particle filter alone (chain and grid kernels): smo / grad are not written
    long long* prof;         // optional per-CTA phase clocks (pmmh_sv_debug_profile)
    void* ws;
    size_t ws_bytes;
    cudaStream_t stream;
};
}  // namespace pmmh
