"""Kernel selection of the SV smoother (pmmh_sv_set_algorithm): which kernel produces the outputs
(diag[PMMH_DIAG_KERNEL]) for each algorithm, size, batch, Hessian, history and CTA count, on the
device-resident entry point (pmmh_flps_sv_corr / pmmh_bpf_sv_corr) and on the host-streamed one
(pmmh_flps_sv_corr_streamed, which refuses the sizes no kernel of it takes).

Both streaming variants report 4; which one ran is pinned by bit-equality with an explicit
algorithm 5 (path storage) or 4 (records) run on the same inputs.
"""
import numpy as np
import pytest

import golden_inputs as gi

pytestmark = pytest.mark.gpu

DIAG_STATUS, DIAG_KERNEL = 2, 6
GENERAL, EXCHANGE, CHAIN, STREAMING, GRID = 1, 2, 3, 4, 5
PATH, RECORDS = "path", "records"   # streaming kernels with path storage (algorithm 5) / records (algorithm 4)
REFUSED = None
PARAMS = (0.2, 0.9, 0.4, -0.5)
LAG = 10
M = 1 << 20


def _with_algorithm(K, alg, fn):
    K.set_sv_algorithm(alg)
    try:
        return fn()
    finally:
        K.set_sv_algorithm(0)


def _resident_inputs(dev, n, nobs, batch):
    import torch
    g = torch.Generator(device=dev)
    g.manual_seed(n + nobs)
    obs = torch.from_numpy(gi.sv_obs(nobs)).to(dev)
    params = torch.tensor([PARAMS] * batch, dtype=torch.float64, device=dev)
    u = torch.randn((batch, nobs, n), dtype=torch.float64, device=dev, generator=g)
    rvr = torch.rand((batch, nobs), dtype=torch.float64, device=dev, generator=g)
    return obs, params, rvr, u


# (algorithm, N, batch, Hessian, history, ctas per problem, n_obs, expected kernel)
RESIDENT = [
    (0, 1024, 1, False, False, 0, 24, CHAIN),
    (0, 1024, 3, True, True, 1, 24, CHAIN),
    (0, 8192, 1, False, False, 0, 24, EXCHANGE),
    (0, 8192, 2, False, True, 0, 24, EXCHANGE),
    (0, 8192, 1, True, False, 0, 24, GENERAL),
    (0, 1 << 14, 1, False, False, 0, 24, GRID),
    (0, 1 << 14, 1, True, False, 0, 24, GRID),
    (0, 1 << 14, 2, False, False, 0, 24, EXCHANGE),
    (0, 1 << 15, 1, False, False, 16, 24, EXCHANGE),
    (0, 1 << 15, 1, True, False, 16, 24, GENERAL),
    (0, M, 1, False, False, 0, 24, GRID),
    (0, M, 1, True, False, 0, 24, GRID),
    (0, M, 1, False, True, 0, 24, GRID),
    (0, 1500000, 1, False, False, 0, 24, PATH),
    (0, 1500000, 1, True, False, 0, 24, GENERAL),
    (0, 1500000, 1, False, True, 0, 24, GENERAL),
    (0, 1 << 23, 1, False, False, 0, 24, RECORDS),
    (1, 1024, 1, False, False, 0, 24, GENERAL),
    (1, 1 << 16, 1, False, False, 0, 24, GENERAL),
    (2, 8192, 1, False, False, 0, 24, EXCHANGE),
    (2, 1 << 16, 1, False, False, 16, 24, EXCHANGE),
    (2, 1 << 16, 1, True, False, 0, 24, GENERAL),
    (2, 1500000, 1, False, False, 0, 24, GENERAL),
    (3, 1024, 1, True, False, 0, 24, CHAIN),
    (3, 8192, 1, False, False, 0, 24, GENERAL),
    (4, 1 << 16, 1, False, False, 0, 40, RECORDS),
    (4, 1 << 16, 1, True, False, 0, 40, GENERAL),
    (4, 1 << 16, 1, False, False, 4, 40, GENERAL),
    (5, 1 << 16, 1, False, False, 0, 40, PATH),
    (5, 1 << 16, 2, False, False, 0, 40, GENERAL),
    (5, 1 << 16, 1, False, True, 0, 40, GENERAL),
    (6, 4096, 1, False, False, 0, 32, GRID),
    (6, 1 << 16, 1, True, True, 16, 32, GRID),
    (6, 1 << 16, 2, False, False, 0, 32, GENERAL),
    (6, 1500000, 1, False, False, 0, 32, GENERAL),
]


@pytest.mark.parametrize("alg,n,batch,hess,hist,ctas,nobs,expect", RESIDENT)
def test_resident_entry_selects(cuda_dev, alg, n, batch, hess, hist, ctas, nobs, expect):
    import torch
    from pmmh_qn_b200 import kernels as K
    obs, params, rvr, u = _resident_inputs(cuda_dev, n, nobs, batch)

    def run(a):
        out = _with_algorithm(K, a, lambda: K.flps_sv_corr(obs, params, rvr, u, lag=LAG, compute_hessian=hess,
                                                            store_history=hist, ctas_per_problem=ctas))
        torch.cuda.synchronize()
        return out

    out = run(alg)
    diag = out["diag"].cpu().numpy()
    assert (diag[:, DIAG_STATUS] == 0).all(), diag
    got = diag[:, DIAG_KERNEL].tolist()
    if expect in (PATH, RECORDS):
        assert got == [STREAMING] * batch, got
        ref = run(5 if expect == PATH else 4)
        for k in ("log_like", "filt", "smo", "gradient", "traj"):
            assert torch.equal(out[k], ref[k]), k
    else:
        assert got == [expect] * batch, got


@pytest.mark.parametrize("alg,ctas", [(0, 0), (0, 16), (5, 0), (6, 0)])
def test_bpf_runs_on_the_general_kernel(cuda_dev, alg, ctas):
    import torch
    from pmmh_qn_b200 import kernels as K
    obs, params, rvr, u = _resident_inputs(cuda_dev, 1 << 15, 24, 1)
    out = _with_algorithm(K, alg, lambda: K.bpf_sv_corr(obs, params, rvr, u, ctas_per_problem=ctas))
    torch.cuda.synchronize()
    assert int(out["diag"][0, DIAG_STATUS]) == 0
    assert int(out["diag"][0, DIAG_KERNEL]) == GENERAL


# (algorithm, N, ctas per problem, n_obs, expected kernel or REFUSED)
STREAMED = [
    (0, 1024, 0, 24, REFUSED),
    (0, 8192, 0, 24, EXCHANGE),
    (0, 1 << 15, 16, 24, EXCHANGE),
    (0, 1 << 16, 0, 24, GRID),
    (0, M, 0, 24, GRID),
    (0, 1500000, 0, 24, STREAMING),
    (0, 1500000, 16, 24, REFUSED),
    (1, 1 << 16, 0, 24, REFUSED),
    (2, 8192, 0, 24, EXCHANGE),
    (2, 1 << 16, 16, 24, EXCHANGE),
    (2, 1500000, 0, 24, REFUSED),
    (3, 1024, 0, 24, REFUSED),
    (3, 1 << 16, 0, 24, REFUSED),
    (4, 1 << 16, 0, 24, REFUSED),
    (4, 1500000, 0, 24, REFUSED),
    (5, 1 << 16, 0, 24, REFUSED),
    (5, 1500000, 0, 24, STREAMING),
    (6, 4096, 0, 32, GRID),
    (6, 1 << 16, 8, 32, REFUSED),
    (6, 1500000, 0, 32, REFUSED),
]


@pytest.mark.parametrize("alg,n,ctas,nobs,expect", STREAMED)
def test_host_streamed_entry_selects(cuda_dev, alg, n, ctas, nobs, expect):
    import torch
    from pmmh_qn_b200 import _lib
    from pmmh_qn_b200 import kernels as K
    eligible = _with_algorithm(K, alg, lambda: K.sv_streamed_eligible(nobs, n, LAG, ctas))
    assert eligible == (expect is not REFUSED)
    rvs = np.random.default_rng(n + nobs).standard_normal((nobs, n + 1))
    obs = torch.from_numpy(gi.sv_obs(nobs)).to(cuda_dev)
    params = torch.tensor([PARAMS], dtype=torch.float64, device=cuda_dev)
    rvr = torch.from_numpy(gi.split_particle(rvs, nobs)[0]).to(cuda_dev)

    def run():
        return K.flps_sv_corr_streamed(rvs, obs, params, rvr, nobs, n, lag=LAG, ctas_per_problem=ctas)

    if expect is REFUSED:
        with pytest.raises(_lib.PmmhError):
            _with_algorithm(K, alg, run)
        return
    out = _with_algorithm(K, alg, run)
    torch.cuda.synchronize()
    assert int(out["diag"][0, DIAG_STATUS]) == 0
    assert int(out["diag"][0, DIAG_KERNEL]) == expect
