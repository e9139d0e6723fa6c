// sv_grid.cuh -- the grid kernel (sv_grid.cu): one smoother evaluation (the SV model or another model of
// pf_model.cuh) as one persistent cooperative launch, one tile of the sorted generation per CTA
#pragma once
#include <cuda_runtime.h>
#include <stddef.h>

#include "sv_call.h"

namespace pmmh {
int sv_grid_ctas(int n, int sm_count, int ctas);
bool sv_grid_eligible(int nobs, int n, int lag, int G);
// the filter alone (no lag): n_obs >= 2 and a tile fits one CTA
bool sv_grid_filter_eligible(int nobs, int n, int G);
size_t sv_grid_ws_bytes(int nobs, int n, int lag, int G, int hist, int hess = 0, int filter = 0);
// `batch` problems of one shape (problem b's inputs and outputs one problem further on), each on its own G CTAs, in
// waves of nteams = sv_grid_teams(batch, SMs, G) problems: one cooperative launch of (problems in the wave) x G CTAs per
// wave.  Every problem's outputs are bit-identical to its run alone (batch = nteams = 1).  The workspace is
// min(batch, nteams) slices of sv_grid_ws_bytes (hist: c.x_hist given).  c.model selects the instantiation (the table
// Models in pf_model.cuh; the filter runs the model's Filter); hess: the Hessian branch (SV only); c.filter: the filter
// alone (lag unused).  Host-streamed u (c.slot > 0) and the phase clocks (c.prof) take batch = 1 only.
int sv_grid_teams(int batch, int sm_count, int G);
int sv_grid_run(const SvCall& c, int batch, int nobs, int n, int lag, int G, int nteams, int hess);
}  // namespace pmmh
