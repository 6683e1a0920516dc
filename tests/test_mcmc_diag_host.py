"""not-gpu: the float64 restatement of split-R-hat / bulk and tail ESS (tests/mcmc_reference.py) behaves as sampling theory says it
must, and the C ABI of the on-device diagnostics rejects bad arguments on the host before any CUDA call."""
import os
import re

import numpy as np
import pytest

import mcmc_reference as R


@pytest.fixture(scope="module")
def built():
    import __graft_entry__ as g
    g.build()
    import psgla_b200
    return psgla_b200


def _ar1(rng, rho, N, M, E):
    """Stationary AR(1) chains [N, M, E] with unit innovations."""
    x = np.empty((N, M, E))
    x[0] = rng.standard_normal((M, E)) / np.sqrt(1 - rho ** 2)
    for n in range(1, N):
        x[n] = rho * x[n - 1] + rng.standard_normal((M, E))
    return x


def test_iid_draws_rhat_near_one_and_ess_near_s():
    """4 chains x 1 000 iid N(0, 1) draws, 20 elements: R-hat - 1 is O(1 / N') (max 2e-3 over the elements, bound 1e-2); bulk
    ESS averages to S within 5 % (its per-element spread is a few %); tail ESS is of the order of S."""
    x = np.random.default_rng(0).standard_normal((1000, 4, 20))
    rhat, bulk, tail = R.diag(x)
    S = 4000
    assert np.all(np.abs(rhat - 1) < 1e-2), rhat
    assert abs(bulk.mean() / S - 1) < 0.05, bulk.mean()
    assert np.all((tail > 0.5 * S) & (tail < 1.5 * S)), tail


def test_ar1_ess_matches_the_integrated_autocorrelation():
    """AR(1) with rho = 0.9: ESS = S (1 - rho) / (1 + rho) = S / 19.  4 chains x 4 000 draws, 10 elements: the mean bulk ESS is
    within 10 % of it (the Geyer estimate's relative spread is ~7 % per element at this length, ~2 % for the mean)."""
    x = _ar1(np.random.default_rng(1), 0.9, 4000, 4, 10)
    _, bulk, _ = R.diag(x)
    want = 16000 * 0.1 / 1.9
    assert abs(bulk.mean() / want - 1) < 0.10, (bulk.mean(), want)


def test_shifted_chain_means_give_large_rhat():
    """One of 4 chains shifted by 3 sd: R-hat far above the usual 1.01 threshold (rank normalisation bounds it: 1.45 .. 1.49
    measured here)."""
    x = np.random.default_rng(2).standard_normal((400, 4, 5))
    x[:, 3] += 3.0
    rhat, _, _ = R.diag(x)
    assert np.all(rhat > 1.3), rhat


def test_rank_statistics_are_invariant_under_increasing_maps():
    """Bulk R-hat and bulk ESS use ranks only: exp() leaves them exactly as they are.  The full R-hat also folds the draws
    around their median, so it is invariant under maps that keep the order of |x - median| too: an odd map about the median
    (sinh around it; the draw count is odd, so the median is a draw)."""
    x = _ar1(np.random.default_rng(3), 0.5, 401, 3, 6)
    for e in range(x.shape[2]):
        a, b = x[:, :, e], np.exp(x[:, :, e])
        za, zb = R.z_scale(R.split_chains(a)), R.z_scale(R.split_chains(b))
        assert np.array_equal(za, zb)
        assert R.rhat_split(za) == R.rhat_split(zb) and R.ess_split(za) == R.ess_split(zb)
    med = np.median(x, axis=(0, 1))
    y = med + np.sinh(x - med)
    (ra, ba, _), (rb, bb, _) = R.diag(x), R.diag(y)
    np.testing.assert_allclose(rb, ra, rtol=1e-12)
    np.testing.assert_array_equal(bb, ba)


def test_odd_n_drops_the_middle_draw():
    x = np.random.default_rng(4).standard_normal((9, 2))
    s = R.split_chains(x)
    np.testing.assert_array_equal(s, np.vstack((x[:4].T, x[5:].T)))
    # the middle draws enter the median and the quantiles only: the bulk statistics do not see them
    y = x.copy()
    y[4] = [100.0, -100.0]
    zx, zy = R.z_scale(R.split_chains(x)), R.z_scale(R.split_chains(y))
    assert np.array_equal(zx, zy)


def test_constant_element_is_nan():
    x = np.random.default_rng(5).standard_normal((20, 3, 2))
    x[:, :, 1] = 0.25
    rhat, bulk, tail = R.diag(x)
    assert np.all(np.isfinite([rhat[0], bulk[0], tail[0]]))
    assert np.isnan(rhat[1]) and np.isnan(bulk[1]) and np.isnan(tail[1])


def test_header_declares_the_diagnostics(built):
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    with open(os.path.join(root, "include", "psgla_b200.h")) as f:
        header = f.read()
    assert re.search(r"#define PSGLA_MCMC_MAX_DRAWS 16384\b", header)
    for name in ("psgla_mcmc_diag_workspace_bytes", "psgla_mcmc_diag"):
        assert re.search(r"\b%s\(" % name, header) and name in built._lib.SIGNATURES
    assert built.diagnostics.MAX_DRAWS == 16384


def test_workspace_bytes(built):
    lib = built._lib.lib()
    assert lib.psgla_mcmc_diag_workspace_bytes(1000, 8) == 256 + ((2 * 8000 + 1) * 4 + 255) // 256 * 256
    assert lib.psgla_mcmc_diag_workspace_bytes(2048, 8) > 0 and lib.psgla_mcmc_diag_workspace_bytes(2049, 8) > 0
    for n, m in ((2050, 8), (3, 8), (1000, 0), (4, 1 << 40), (1 << 62, 1)):
        assert lib.psgla_mcmc_diag_workspace_bytes(n, m) == 0, (n, m)


def test_argument_errors_without_gpu(built):
    """psgla_mcmc_diag rejects each bad argument on the host before any CUDA call (fake pointers are never dereferenced)."""
    lib = built._lib.lib()
    fake = 0x1000

    def call(draws=fake, N=100, M=4, E=10, ws=fake, ws_bytes=None, r=fake, b=fake, t=fake):
        if ws_bytes is None:
            ws_bytes = lib.psgla_mcmc_diag_workspace_bytes(N, M) or 1 << 20
        return lib.psgla_mcmc_diag(draws, N, M, E, ws, ws_bytes, r, b, t, None)

    for kw in (dict(draws=None), dict(ws=None), dict(r=None), dict(b=None), dict(t=None)):
        assert call(**kw) == -1 and b"null" in lib.psgla_last_error(), kw
    for kw, word in ((dict(N=3), b"n_draws"), (dict(N=-1), b"n_draws"), (dict(M=0), b"n_chains"), (dict(E=0), b"n_elem"),
                     (dict(E=1 << 40), b"n_elem")):
        assert call(**kw) == -1 and word in lib.psgla_last_error(), kw
    for N, M in ((2050, 8), (16386, 1), (4, 4097), (1 << 40, 2)):
        assert call(N=N, M=M) == -1, (N, M)
        assert b"n_inter" in lib.psgla_last_error() and b"16384" in lib.psgla_last_error()
    need = lib.psgla_mcmc_diag_workspace_bytes(100, 4)
    assert call(ws_bytes=need - 1) == -4 and b"workspace" in lib.psgla_last_error()
