"""not-gpu: the float64 restatement of the posterior summary (tests/mcmc_summary_reference.py) against sampling theory, and
the C ABI of psgla_mcmc_summary (csrc/mcmc_summary.cu): declared and bound, and every bad argument rejected on the host
before any CUDA call."""
import os
import re

import numpy as np
import pytest
from scipy import stats

import mcmc_summary_reference as SR


@pytest.fixture(scope="module")
def built():
    import __graft_entry__ as g
    g.build()
    import psgla_b200
    return psgla_b200


def test_iid_normal_ess_and_mcse():
    """i.i.d. N(0, 1): ess_mean ~ S, mcse_mean ~ sd / sqrt(S), mcse_quantiles ~ sqrt(p (1 - p) / S) / phi(z_p), within 10 %
    (averaged over 20 elements for the quantiles, whose single-element MCSE is itself a noisy order statistic)."""
    N, M, E = 1000, 4, 20
    x = np.random.default_rng(0).standard_normal((N, M, E))
    probs = (0.05, 0.5, 0.95)
    r = SR.summary(x, probs)
    S = 2 * M * (N // 2)
    assert np.all(np.abs(r["ess_mean"] / S - 1) < 0.1), r["ess_mean"] / S
    assert np.all(np.abs(r["mcse_mean"] / (r["sd"] / np.sqrt(S)) - 1) < 0.1)
    for j, p in enumerate(probs):
        want = np.sqrt(p * (1 - p) / S) / stats.norm.pdf(stats.norm.ppf(p))
        got = r["mcse_quantiles"][j].mean()
        assert abs(got / want - 1) < 0.1, (p, got, want)


def test_ar1_ess_mean():
    """AR(1), rho = 0.5: ess_mean ~ S (1 - rho) / (1 + rho) within 10 %."""
    rho, N, M = 0.5, 5000, 16
    rng = np.random.default_rng(1)
    x = np.empty((N, M, 3))
    x[0] = rng.standard_normal((M, 3)) / np.sqrt(1 - rho ** 2)
    for n in range(1, N):
        x[n] = rho * x[n - 1] + rng.standard_normal((M, 3))
    r = SR.summary(x)
    want = 2 * M * (N // 2) * (1 - rho) / (1 + rho)
    assert np.all(np.abs(r["ess_mean"] / want - 1) < 0.1), r["ess_mean"] / want


def test_hdi_of_symmetric_unimodal_is_central():
    a = np.sort(np.random.default_rng(2).standard_normal(200000))
    lo, hi, _ = SR.hdi(a, 0.9)
    q = np.quantile(a, [0.05, 0.95])
    assert abs(lo - q[0]) < 0.02 and abs(hi - q[1]) < 0.02, (lo, hi, q)


def test_hdi_of_bimodal_is_the_shortest_window_ties_to_the_lowest():
    # two separated clusters of 40 and 60 equally spaced draws: 50 % of 100 draws is a window of 51 draws, found only in the
    # larger cluster (spacing 0.1) -> width 5.0; the smaller one cannot hold it
    a = np.sort(np.concatenate([np.arange(40) * 0.1, 100 + np.arange(60) * 0.1]))
    lo, hi, i = SR.hdi(a, 0.5)
    k = 50
    widths = a[k:] - a[:-k]
    assert np.isclose(hi - lo, widths.min()) and i == int(np.flatnonzero(widths == widths.min())[0])
    assert lo >= 100 and i == 40  # the windows 40..49 all have width 5.0: the lowest index wins
    assert np.sum(widths == widths.min()) > 1


def test_nan_and_constant_elements():
    x = np.random.default_rng(3).standard_normal((40, 2, 3))
    x[:, :, 1] = 0.25
    x[5, 1, 2] = np.nan
    r = SR.summary(x)
    assert r["sd"][1] == 0 and np.isnan(r["ess_mean"][1]) and np.isnan(r["mcse_mean"][1])
    assert np.all(np.isnan(r["mcse_quantiles"][:, 1])) and r["hdi_low"][1] == r["hdi_high"][1] == 0.25
    for k in SR.KEYS:
        assert np.isnan(r[k][2]), k
    for k in SR.PKEYS:
        assert np.all(np.isnan(r[k][:, 2])), k


def test_header_declares_the_summary(built):
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    with open(os.path.join(root, "include", "psgla_b200.h")) as f:
        header = f.read()
    for name in ("psgla_mcmc_summary_workspace_bytes", "psgla_mcmc_summary"):
        assert re.search(r"\b%s\(" % name, header) and name in built._lib.SIGNATURES
    assert re.search(r"#define PSGLA_MCMC_MAX_PROBS %d\b" % built.diagnostics.MAX_PROBS, header)
    assert callable(built.mcmc_summary)


def test_workspace(built):
    f = built._lib.lib().psgla_mcmc_summary_workspace_bytes
    large = built._lib.lib().psgla_mcmc_diag_large_workspace_bytes
    for N, M, E in ((1000, 8, 196608), (1001, 8, 300), (800, 1000000, 2), (5, 4097, 7)):
        assert f(N, M, E, 3) > large(N, M, E) > 0
        assert f(N, M, E, 8) >= f(N, M, E, 1)
    assert f(1000, 8, 196608, 8) > f(1000, 8, 196608, 1)  # per-p slots of a group of 32 768 elements
    # odd N keeps the merged sorted draws: 4 B more per draw of a group
    assert f(1001, 8, 300, 3) - f(1000, 8, 300, 3) >= 4 * 300 * 8 * 1001 - 4 * 300 * 8 * 1000
    for N, M, E, P in ((3, 8, 1, 3), (4, 2 ** 29, 1, 3), (100, 0, 1, 3), (100, 4, 0, 3), (100, 4, 1, 0), (100, 4, 1, 9),
                       (100, 4, 1, -1)):
        assert f(N, M, E, P) == 0, (N, M, E, P)


def test_argument_errors_without_gpu(built):
    """psgla_mcmc_summary rejects each bad argument on the host before any CUDA call (fake pointers are never
    dereferenced)."""
    import ctypes as C
    lib = built._lib.lib()
    fake = 0x1000

    def call(draws=fake, N=100, M=4, E=10, probs=(0.05, 0.5, 0.95), n_probs=None, hdi=0.94, ws=fake, ws_bytes=None,
             outs=None):
        P = len(probs) if n_probs is None else n_probs
        arr = None if probs is None else (C.c_double * max(1, len(probs)))(*probs)
        if ws_bytes is None:
            ws_bytes = lib.psgla_mcmc_summary_workspace_bytes(N, M, E, P) or 1 << 20
        outs = outs or [fake] * 9
        return lib.psgla_mcmc_summary(draws, N, M, E, arr, P, hdi, ws, ws_bytes, *outs, None)

    for kw in [dict(draws=None), dict(ws=None), dict(probs=None, n_probs=3)] + \
              [dict(outs=[None if j == i else fake for j in range(9)]) for i in range(9)]:
        assert call(**kw) == -1 and b"null" in lib.psgla_last_error(), kw
    for kw, word in ((dict(N=3), b"n_draws"), (dict(N=-1), b"n_draws"), (dict(M=0), b"n_chains"), (dict(M=-3), b"n_chains"),
                     (dict(E=0), b"n_elem"), (dict(E=1 << 40), b"n_elem"), (dict(n_probs=0), b"n_probs"),
                     (dict(probs=(0.1,) * 9), b"n_probs"), (dict(n_probs=-2), b"n_probs")):
        assert call(**kw) == -1 and word in lib.psgla_last_error(), kw
    for probs in ((0.0,), (1.0,), (0.5, -0.1), (0.5, float("nan")), (float("inf"),), (0.2, 0.3, 1.5)):
        assert call(probs=probs) == -1 and b"probs[" in lib.psgla_last_error(), probs
    for h in (0.0, 1.0, -0.5, 2.0, float("nan"), float("inf")):
        assert call(hdi=h) == -1 and b"hdi_prob" in lib.psgla_last_error(), h
    for N, M in ((2 ** 31 + 1, 1), (4, 2 ** 29), (1 << 40, 2)):
        assert call(N=N, M=M) == -1 and b"2^31 - 1" in lib.psgla_last_error(), (N, M)
    need = lib.psgla_mcmc_summary_workspace_bytes(100, 4, 10, 3)
    assert call(ws_bytes=need - 1) == -4 and b"workspace" in lib.psgla_last_error()
    assert call(ws=fake + 16) == -1 and b"aligned" in lib.psgla_last_error()
