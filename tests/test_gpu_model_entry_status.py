"""Status and workspace answers of the eight model functions of the C ABI: pmmh_flps_model_corr,
pmmh_filter_model_corr, pmmh_flps_model_batch_corr, pmmh_filter_model_batch_corr and their workspace queries.

One table (tests/golden/model_entry_status.json) holds, for every case, the query's status and bytes and the entry's
status.  The cases cover model ids -1 .. 5 (3 is unassigned), the Hessian flag where the entry takes it, a chain size,
a grid size, a size one particle above the grid kernel's capacity and a batch above 4096 particles, lag 1, 2, 10 and
11 with n_obs at its limits, missing history halves, a workspace one byte short and a null workspace.  Accepted calls
run on small random inputs.  Workspace sizes depend on the SM count: they are compared where the device has the SM
count the table was recorded with (statuses always).

Regenerate the table on a GPU with ``python tests/test_gpu_model_entry_status.py [out.json]``.
"""
import ctypes
import json
import os
import sys

import pytest

pytestmark = pytest.mark.gpu

HERE = os.path.dirname(os.path.abspath(__file__))
TABLE = os.path.join(HERE, "golden", "model_entry_status.json")
TILE_MAX = 7168   # particles of one grid-kernel tile (one CTA per SM)

ENTRIES = ("flps", "filter", "flps_batch", "filter_batch")
MODELS = (-1, 0, 1, 2, 3, 4, 5)
SIZES = ("chain", "grid", "big", "batch")   # (N, B): (256, 2), (8192, 1), (SMs x TILE_MAX + 1, 1), (8192, 2)


def _cases():
    out = []
    for entry in ENTRIES:
        smoother = entry.startswith("flps")
        hs = (0, 1, 2) if entry == "flps_batch" else (0,)
        base_lag = 4 if smoother else 2
        for size in SIZES:
            for model in MODELS:
                for hess in hs:
                    out.append((entry, model, hess, size, base_lag, 12, "both", "exact"))
            if smoother:
                shapes = sorted({(lag, nobs) for lag in (1, 2, 10, 11)
                                 for nobs in (1, 2, lag, lag + 1, 2 * lag - 1, 2 * lag) if nobs >= 1})
            else:
                shapes = [(2, 1), (2, 2), (2, 3)]
            for lag, nobs in shapes:
                out.append((entry, 1, 0, size, lag, nobs, "both", "exact"))
            for hist in ("none", "x_only", "a_only"):
                out.append((entry, 1, 0, size, base_lag, 12, hist, "exact"))
            for ws in ("short", "null"):
                out.append((entry, 1, 0, size, base_lag, 12, "both", ws))
    return out


def _case_id(case):
    entry, model, hess, size, lag, nobs, hist, ws = case
    return "%s-m%d-h%d-%s-lag%d-nobs%d-%s-%s" % (entry, model, hess, size, lag, nobs, hist, ws)


CASES = _cases()


def _shape(size, sm):
    return {"chain": (256, 2), "grid": (8192, 1), "big": (sm * TILE_MAX + 1, 1), "batch": (8192, 2)}[size]


def _query(lib, entry, nobs, n, lag, batch, hess):
    out = ctypes.c_size_t()
    if entry == "flps":
        rc = lib.pmmh_flps_model_workspace_bytes(nobs, n, lag, batch, ctypes.byref(out))
    elif entry == "filter":
        rc = lib.pmmh_filter_model_workspace_bytes(nobs, n, batch, ctypes.byref(out))
    elif entry == "flps_batch":
        rc = lib.pmmh_flps_model_batch_workspace_bytes(nobs, n, lag, batch, hess, ctypes.byref(out))
    else:
        rc = lib.pmmh_filter_model_batch_workspace_bytes(nobs, n, batch, ctypes.byref(out))
    return rc, (out.value if rc == 0 else None)


def _run(case, dev, sm):
    """[query status, query bytes or None, entry status] of one case"""
    import torch
    from pmmh_qn_b200 import _lib
    lib = _lib.load()
    entry, model, hess, size, lag, nobs, hist, ws_kind = case
    n, batch = _shape(size, sm)
    qrc, qbytes = _query(lib, entry, nobs, n, lag, batch, hess)
    g = torch.Generator(device=dev)
    g.manual_seed(1234)
    f64 = lambda *s: torch.zeros(s, dtype=torch.float64, device=dev)   # noqa: E731
    obs = 0.5 * torch.randn((nobs,), dtype=torch.float64, device=dev, generator=g)
    params = torch.tensor([(0.2, 0.9, 0.4, -0.5) if model == 0 else (0.8, 0.5, 0.3, 0.0)] * batch,
                          dtype=torch.float64, device=dev)
    rvr = torch.rand((batch, nobs), dtype=torch.float64, device=dev, generator=g)
    u = torch.randn((batch, nobs, n), dtype=torch.float64, device=dev, generator=g)
    filt, smo, traj, ll, grad = f64(batch, nobs), f64(batch, nobs), f64(batch, nobs), f64(batch), f64(batch, 4, nobs)
    h1, h2 = f64(batch, 16), f64(batch, 16)
    diag = torch.zeros((batch, _lib.DIAG_COUNT), dtype=torch.int64, device=dev)
    xh = f64(batch, nobs, n) if hist in ("both", "x_only") else None
    ah = torch.zeros((batch, nobs, n), dtype=torch.int32, device=dev) if hist in ("both", "a_only") else None
    nb = qbytes if qbytes is not None else 256
    if ws_kind == "short":
        nb -= 1
    elif ws_kind == "null":
        nb = 0
    ws = None if ws_kind == "null" else torch.empty(max(nb, 1), dtype=torch.uint8, device=dev)
    p = lambda t: None if t is None else ctypes.c_void_p(t.data_ptr())   # noqa: E731
    st = ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)
    if entry == "flps":
        rc = lib.pmmh_flps_model_corr(model, p(obs), 0, p(params), p(rvr), p(u), nobs, n, lag, batch, p(filt), p(smo),
                                      p(ll), p(grad), p(traj), p(diag), p(xh), p(ah), p(ws), nb, st)
    elif entry == "filter":
        rc = lib.pmmh_filter_model_corr(model, p(obs), 0, p(params), p(rvr), p(u), nobs, n, batch, p(filt), p(ll),
                                        p(traj), p(diag), p(xh), p(ah), p(ws), nb, st)
    elif entry == "flps_batch":
        rc = lib.pmmh_flps_model_batch_corr(model, p(obs), 0, p(params), p(rvr), p(u), nobs, n, lag, batch, hess,
                                            p(filt), p(smo), p(ll), p(grad), p(traj), p(h1), p(h2), p(diag), p(xh),
                                            p(ah), p(ws), nb, st)
    else:
        rc = lib.pmmh_filter_model_batch_corr(model, p(obs), 0, p(params), p(rvr), p(u), nobs, n, batch, p(filt),
                                              p(ll), p(traj), p(diag), p(xh), p(ah), p(ws), nb, st)
    torch.cuda.synchronize()
    return [qrc, qbytes, rc]


@pytest.fixture(scope="module")
def table():
    with open(TABLE) as fh:
        return json.load(fh)


@pytest.mark.parametrize("case", CASES, ids=_case_id)
def test_status_matrix(cuda_dev, table, case):
    from pmmh_qn_b200 import kernels as K
    sm = K.device_info()[0]
    want = table["cases"][_case_id(case)]
    got = _run(case, cuda_dev, sm)
    if sm != table["sm"]:
        want, got = [want[0], want[2]], [got[0], got[2]]
    assert got == want


def test_table_covers_every_case(table):
    assert sorted(table["cases"]) == sorted(_case_id(c) for c in CASES)


if __name__ == "__main__":
    sys.path.insert(0, os.path.dirname(HERE))
    import torch
    from pmmh_qn_b200 import kernels as K
    dev = torch.device("cuda:0")
    sm = K.device_info()[0]
    rows = sorted((_case_id(c), _run(c, dev, sm)) for c in CASES)
    with open(sys.argv[1] if len(sys.argv) > 1 else TABLE, "w") as fh:
        fh.write('{"sm": %d, "cases": {\n%s\n}}\n' % (sm, ",\n".join("%s: %s" % (json.dumps(k), json.dumps(v))
                                                                    for k, v in rows)))
    print("%d cases, sm %d" % (len(CASES), sm))
