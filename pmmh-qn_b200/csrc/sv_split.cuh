// sv_split.cuh -- the streaming ("split") SV kernels driven on one device (sv_split.cu)
#pragma once
#include <cuda_runtime.h>
#include <stddef.h>

#include "sv_call.h"

namespace pmmh {
size_t sv_split_single_ws_bytes(int nobs, int n, int lag);
bool sv_split_single_eligible(int nobs, int n, int lag);
int sv_split_single_run(const SvCall& c, int nobs, int n, int lag);
// path storage variant (algorithm 5): generations stored once in birth order, jump tables.  Also reads u as
// particle-major slots signalled by c.slot_ready, or, with c.u == NULL, as the Philox stream (c.seed, c.philox_offset)
size_t sv_split_path_ws_bytes(int nobs, int n, int lag);
int sv_split_path_run(const SvCall& c, int nobs, int n, int lag);
}  // namespace pmmh
