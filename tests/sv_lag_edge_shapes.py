"""(lag, n_obs) shapes of tests/test_gpu_sv_lag_edges.py, built from each SV smoother kernel's own eligibility rule.

The entry (sv_make_plan, capi.cu) takes 2 <= lag <= 63 and n_obs >= lag + 1.  Inside that region each kernel has its
rule on (lag, n_obs) (its rule on N is the test's choice of N and CTAs):

- chain (sv_chain_eligible): lag <= 10;
- general and exchange: the entry's region;
- grid (sv_grid_eligible): lag <= 10 and n_obs >= 2 lag;
- streaming, records and path storage (sv_split_single_eligible): n_obs >= 2 lag.

Each kernel's list takes its lags and, per lag, the shortest series its rule accepts, the next one, and 2 lag - 2,
2 lag - 1, 2 lag where those are accepted: the reference's tail drops gradient terms up to n_obs = 2 lag - 2 (DESIGN.md
section 2), so the lists straddle that boundary wherever a kernel reaches it.  The streaming lags cover every size of
the path-storage jump tables (Q = the largest q with 2^q <= lag - 2, 0 for lag <= 3), at lag - 2 = 2^q and beside it.
tests/test_sv_lag_edge_shapes.py checks that each list reaches the corners of its kernel's region.
"""
MIN_LAG, MAX_LAG = 2, 63


def entry_accepts(lag, nobs):
    return MIN_LAG <= lag <= MAX_LAG and nobs >= lag + 1


RULES = {
    "chain": lambda lag, nobs: entry_accepts(lag, nobs) and lag <= 10,
    "general": entry_accepts,
    "exchange": entry_accepts,
    "grid": lambda lag, nobs: entry_accepts(lag, nobs) and lag <= 10 and nobs >= 2 * lag,
    "streaming": lambda lag, nobs: entry_accepts(lag, nobs) and nobs >= 2 * lag,
}

LAGS = {
    "chain": (2, 3, 4, 9, 10),
    "general": (2, 10, 11, 14, 31, 32, 33, 62, 63),
    "exchange": (2, 10, 11, 14, 31, 63),
    "grid": (2, 3, 9, 10),
    "streaming": (2, 3, 4, 5, 6, 10, 11, 17, 18, 34, 35, 63),
}


def min_nobs(kernel, lag):
    """the shortest series the kernel's rule accepts at this lag"""
    return next(m for m in range(lag + 1, 2 * lag + 2) if RULES[kernel](lag, m))


def nobs_list(kernel, lag):
    m0 = min_nobs(kernel, lag)
    return sorted(m for m in {m0, m0 + 1, 2 * lag - 2, 2 * lag - 1, 2 * lag} if m >= m0 and RULES[kernel](lag, m))


def shapes(kernel):
    return [(lag, m) for lag in LAGS[kernel] for m in nobs_list(kernel, lag)]


def jump_levels(lag):
    """Q of the path-storage jump tables (sv_split.cu make_path_layout)"""
    q = 0
    while (2 << q) <= lag - 2:
        q += 1
    return q


def drops_terms(lag, nobs):
    """the reference's tail indexes gradient slots < 0 here (the terms are dropped)"""
    return nobs <= 2 * lag - 2
