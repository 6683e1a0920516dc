"""-m gpu: the posterior summary (csrc/mcmc_summary.cu, ``psgla_b200.mcmc_summary``) against its float64 restatement
(tests/mcmc_summary_reference.py, PARITY UNPINNED against arviz itself).

Stated tolerances
  * quantiles, hdi_low, hdi_high, mcse_quantiles: equal to the restatement rounded to fp32 (they are draws, or half the
    difference of two draws).  mcse_quantiles excludes elements whose unrounded Beta position ppf K - 1 lies within 1e-6 of a
    rounding boundary (counted; the seeds here give none) and elements whose quantile ESS truncates at a different lag.
  * mean, sd: relative error <= 1e-6.
  * ess_mean, ess_quantiles, mcse_mean: the rule of tests/test_mcmc_diag_gpu.py -- ESS relative error <= 1e-3 (mcse_mean
    5e-4: a square root), except where Geyer's truncation meets a pair sum within rounding of 0: at most 0.1 % of the
    elements, each with a reference pair sum below 1e-4.
Bit-exact: two calls; an element alone, inside a batch and across two groups of elements; the quantile ESS at 0.05 / 0.95
against mcmc_diagnostics_large's tail ESS."""
import numpy as np
import pytest
import torch

import mcmc_summary_reference as SR
import psgla_b200 as P
from conftest import observed
from test_mcmc_diag_gpu import _draws, _psgla_run

pytestmark = pytest.mark.gpu

ESS_RTOL, MOMENT_RTOL = 1e-3, 1e-6
ALL_KEYS = SR.KEYS + SR.PKEYS


def _np(t):
    return t.double().cpu().numpy()


def _compare(x, s, what, probs=(0.05, 0.5, 0.95), hdi_prob=0.94):
    """s: mcmc_summary's dict on x (float32 [N, M, E])."""
    pos, traces = [], []
    want = SR.summary(x.astype(np.float64), probs, hdi_prob, pos, traces)
    got = {k: _np(s[k]).reshape(want[k].shape) for k in ALL_KEYS}
    E = x.shape[2]
    for k in ALL_KEYS:
        np.testing.assert_array_equal(np.isnan(got[k]), np.isnan(want[k]), err_msg="%s %s NaN pattern" % (what, k))
    for k in ("quantiles", "hdi_low", "hdi_high"):
        w = want[k].astype(np.float32).astype(np.float64)
        np.testing.assert_array_equal(got[k], w, err_msg="%s %s" % (what, k))
    for k in ("mean", "sd"):
        ok = ~np.isnan(want[k])
        err = np.abs(got[k][ok] - want[k][ok]) / np.maximum(np.abs(want[k][ok]), 1e-30)
        err[want[k][ok] == got[k][ok]] = 0
        observed("%s: %s rel err" % (what, k), err.max() if err.size else 0.0, MOMENT_RTOL)
    # ESS rule; an element flagged in any series is a Geyer flip
    flip = np.zeros(E, bool)
    worst = {}
    for k, rows in (("ess_mean", [(got["ess_mean"], want["ess_mean"], ESS_RTOL)]),
                    ("mcse_mean", [(got["mcse_mean"], want["mcse_mean"], ESS_RTOL / 2)]),
                    ("ess_quantiles", [(got["ess_quantiles"][j], want["ess_quantiles"][j], ESS_RTOL) for j in range(len(probs))])):
        for g, w, tol in rows:
            ok = ~np.isnan(w)
            err = np.zeros(E)
            err[ok] = np.abs(g[ok] / w[ok] - 1)
            flip |= err > tol
            worst[k] = max(worst.get(k, 0.0), err[err <= tol].max() if (err <= tol).any() else 0.0)
    for e in np.flatnonzero(flip):
        assert traces[e]["min_pair"] < 1e-4, (what, e, traces[e])
    observed("%s: Geyer truncation flips" % what, flip.sum() / E, 1e-3 + 1e-12)
    for k, v in worst.items():
        observed("%s: %s rel err" % (what, k), v, ESS_RTOL / 2 if k == "mcse_mean" else ESS_RTOL)
    # mcse_quantiles: exact, away from rounding boundaries of the Beta positions
    K = x.shape[0] * x.shape[1]
    near = 0
    for j in range(len(probs)):
        w = want["mcse_quantiles"][j].astype(np.float32).astype(np.float64)
        for e in range(E):
            s1, s2 = pos[e][j]
            if np.isnan(s1) or flip[e]:
                continue
            v = np.array([max(s1, 0.0), min(s2, K - 1.0)])
            if np.any(np.abs(v - np.floor(v) - 0.5) < 1e-6):
                near += 1
                continue
            assert got["mcse_quantiles"][j][e] == w[e], (what, j, e, got["mcse_quantiles"][j][e], w[e])
    assert near == 0, (what, near)


def _summary(x, **kw):
    return P.mcmc_summary(torch.from_numpy(x).cuda() if isinstance(x, np.ndarray) else x, **kw)


@pytest.mark.parametrize("M,N,E,quantise", [(1, 400, 23, False), (2, 301, 29, False), (8, 200, 31, True),
                                            (8, 201, 17, False), (2, 1001, 40, True), (4, 5, 37, False),
                                            (64, 401, 3, False)])
def test_against_reference(M, N, E, quantise):
    """odd and even N; M = 1, 2, 4, 8, 64; S from 16 to 25 600 (above the small path's 16 384); 8-bit draws with long tie
    runs; a constant element and a NaN element."""
    x = _draws(M * 1000 + N + 7, N, M, E, quantise, constant=(1,))
    x[N // 2, M - 1, E - 1] = np.nan
    s = _summary(x)
    assert s["mean"].shape == (E,) and s["quantiles"].shape == (3, E) and s["n_draws"] == N and s["n_chains"] == M
    assert s["probs"] == (0.05, 0.5, 0.95) and s["hdi_prob"] == 0.94
    assert s["sd"][1].item() == 0 and np.isnan(s["ess_mean"][1].item()) and np.isnan(s["mcse_quantiles"][1, 1].item())
    assert all(np.isnan(s[k].reshape(-1, E)[:, E - 1].cpu().numpy()).all() for k in ALL_KEYS)
    _compare(x, s, "summary M=%d N=%d E=%d q=%d" % (M, N, E, quantise))


def test_other_probabilities():
    x = _draws(17, 300, 4, 19)
    probs = (0.01, 0.25, 0.3, 0.5, 0.6, 0.75, 0.9, 0.99)
    _compare(x, _summary(x, probs=probs, hdi_prob=0.5), "summary 8 probs hdi 0.5", probs, 0.5)


@pytest.mark.parametrize("M,N,E,quantise", [(8, 201, 29, True), (2, 1000, 60, False), (64, 400, 3, False)])
def test_tail_ess_is_the_large_paths(M, N, E, quantise):
    x = torch.from_numpy(_draws(N + M, N, M, E, quantise, constant=(2,))).cuda()
    s = P.mcmc_summary(x, probs=(0.05, 0.95))
    d = P.mcmc_diagnostics_large(x)
    tail = torch.minimum(s["ess_quantiles"][0], s["ess_quantiles"][1])
    assert torch.equal(tail.nan_to_num(-1), d["ess_tail"].nan_to_num(-1))


def test_infinite_draws_hdi_follows_argmin():
    """Infinite draws (a chain that overflowed) make window widths +inf, or NaN where both ends are the same infinity: the
    HDI follows np.argmin (the first NaN, else the first smallest width, all +inf giving window 0), never faults, and leaves
    the other elements alone."""
    N, M, E = 201, 4, 8
    x = _draws(5, N, M, E)
    rng = np.random.default_rng(1)

    def put(e, frac, v):
        f = x[:, :, e].reshape(-1)
        f[rng.choice(N * M, int(frac * N * M), replace=False)] = v
        x[:, :, e] = f.reshape(N, M)

    put(2, 0.1, np.inf)          # 10 % +inf: every window's upper end is +inf -> window 0
    put(3, 0.1, -np.inf)         # 10 % -inf: every lower end -inf -> window 0
    put(4, 0.05, np.inf)
    put(4, 0.05, -np.inf)
    x[:, :, 5] = np.inf          # 97 % +inf: the windows inside the +inf run have NaN widths -> the first of them
    put(5, 0.03, 0.5)
    x[:, :, 6] = np.inf          # all +inf: all widths NaN -> window 0
    s = _summary(x)
    with np.errstate(invalid="ignore"):
        want = SR.summary(x.astype(np.float64))
    for k in ("hdi_low", "hdi_high"):
        np.testing.assert_array_equal(_np(s[k]), want[k].astype(np.float32).astype(np.float64), err_msg=k)
    assert s["hdi_low"][3].item() == -np.inf and s["hdi_low"][5].item() == np.inf
    fin = [0, 1, 7]
    alone = _summary(np.ascontiguousarray(x[:, :, fin]))
    for k in ALL_KEYS:
        assert torch.equal(alone[k].nan_to_num(-1), s[k][..., fin].nan_to_num(-1)), k
    _compare(np.ascontiguousarray(x[:, :, fin]), alone, "summary finite elements beside infinite ones")


def test_mcse_quantile_upper_index_wraps_like_numpy():
    """N = 4, 4 096 chains: S = 16 384 and the indicator series of p = 1e-6 (one draw) has Geyer's ESS at its S log10 S floor,
    4.2 K, so the upper Beta position hi K - 1 rounds to -1, which arviz's sorted_ary[-1] reads as the largest draw."""
    x = _draws(41, 4, 4096, 5)
    probs = (1e-6, 0.5)
    s = _summary(x, probs=probs)
    pos = []
    SR.summary(x.astype(np.float64), probs, 0.94, pos)
    assert all(np.rint(min(p[0][1], x.shape[0] * x.shape[1] - 1.0)) == -1 for p in pos)
    _compare(x, s, "summary mcse index -1", probs)


def test_bit_identical_and_independent_of_the_group():
    """S = 2^20, E = 300: groups of 2^28 / S = 256 elements, so the batch spans two groups."""
    g = torch.Generator(device="cuda").manual_seed(0)
    N, M, E = 1 << 17, 8, 300
    x = torch.randn((N, M, E), generator=g, device="cuda")
    x += torch.randn((1, M, E), generator=g, device="cuda") * 0.05
    x[:, :, 7] = 0.5
    a, b = P.mcmc_summary(x), P.mcmc_summary(x)
    for k in ALL_KEYS:
        assert torch.equal(a[k].nan_to_num(-1), b[k].nan_to_num(-1)), k
    for e0, e1 in ((0, 1), (7, 8), (255, 256), (256, 257), (299, 300), (250, 262)):
        part = P.mcmc_summary(x[:, :, e0:e1].contiguous())
        for k in ALL_KEYS:
            assert torch.equal(part[k].nan_to_num(-1), a[k][..., e0:e1].nan_to_num(-1)), (k, e0)


def test_sampler_run_in_place(monkeypatch):
    """a DnCNN PSGLA run of 2 chains, store='all', read in place; against the stacked Xlist and the restatement"""
    run = _psgla_run(n_chains=2)
    stacked = P.mcmc_summary(torch.stack(run.Xlist))
    seen = []
    real_ptr = P._lib.ptr
    monkeypatch.setattr(P._lib, "ptr", lambda t: seen.append(t.data_ptr() if t is not None else None) or real_ptr(t))
    s = P.mcmc_summary(run, burn_in=4)
    assert seen[0] == run.samples[4].data_ptr()
    monkeypatch.undo()
    assert s["mean"].shape == (3, 24, 32) and s["quantiles"].shape == (3, 3, 24, 32) and s["n_draws"] == 16
    ref = P.mcmc_summary(torch.stack(run.Xlist[4:]))
    for k in ALL_KEYS:
        assert torch.equal(ref[k].nan_to_num(-1), s[k].nan_to_num(-1)), k
    _compare(torch.stack(run.Xlist).reshape(20, 2, -1).cpu().numpy(), stacked, "PSGLA DnCNN 2 chains")


def test_padded_drunet_run_is_cropped():
    torch.manual_seed(5)
    im = torch.rand(1, 3, 37, 50, device="cuda")
    dg, init, _, _ = P.make_inpainting(im, prop=0.5, sigma=1.0, seed_ip=0)
    den = P.DRUNet(pretrained=P.random_drunet_state_dict(0))
    run = P.psgla_run(init, dg, den, alpha=0.8, lambd=25.0, sig_float=5 / 255, delta=(2 / 255) ** 2, n_iter=16, n_inter=2,
                      n_inter_mmse=4, seed=1, n_chains=2, store="all")
    for i in range(16):
        run.step(i)
    run.finish()
    assert run.crop == (37, 50)
    s = P.mcmc_summary(run)
    full = P.mcmc_summary(run.samples[:len(run.Xlist)].contiguous())
    assert s["mean"].shape == (3, 37, 50) and s["quantiles"].shape == (3, 3, 37, 50)
    assert full["mean"].shape == (3, 40, 56)
    for k in ALL_KEYS:
        assert torch.equal(s[k].nan_to_num(-1), full[k][..., :37, :50].nan_to_num(-1)), k


def test_gmm2d_trajectory_against_reference():
    """10^5 chains of a 2D PSGLA cell, 400 steps thinned by 4: [100, 10^5, 2], S = 10^7 per element"""
    mu, Sig, pi = P.gaussian_mixt_example("symetric_gaussians")
    y = np.array((0.0, -2.0))
    n = 100000
    x0 = torch.tensor(y, dtype=torch.float32, device="cuda").repeat(n, 1).contiguous()
    ch = P.GMMChains("psgla", y, 0.3, np.eye(2), 1.0, P.Theorical_MMSE(mu, Sig, pi), 2.0 / 3.0, 1.0, n_chains=n, x0=x0,
                     seed=3, dtype="float32", device="cuda")
    traj = ch.run(400, thin=4)
    assert traj.shape == (100, n, 2)
    s = P.mcmc_summary(traj, burn_in=10)
    assert s["mean"].shape == (2,) and s["n_chains"] == n and s["n_draws"] == 90
    _compare(traj[10:].cpu().numpy(), s, "2D PSGLA 10^5 chains x 90 draws")


def test_truth_coverage_and_calibration():
    run = _psgla_run(n_chains=2)
    truth = torch.rand(3, 24, 32, device="cuda")
    probs = (0.1, 0.5, 0.9)
    s = P.mcmc_summary(run, probs=probs, truth=truth)
    lo, hi = s["hdi_low"], s["hdi_high"]
    ok = ~torch.isnan(lo)
    assert s["coverage_hdi"] == ((lo <= truth) & (truth <= hi) & ok).sum().item() / ok.sum().item()
    assert len(s["frac_truth_below"]) == 3
    for j in range(3):
        q = s["quantiles"][j]
        okq = ~torch.isnan(q)
        assert s["frac_truth_below"][j] == ((truth <= q) & okq).sum().item() / okq.sum().item()
    m = s["mcse_mean"][~torch.isnan(s["mcse_mean"])]
    assert s["mcse_mean_max"] == m.max().item() and len(s["mcse_quantiles_max"]) == 3
    # the median map as the truth lies at or below every median
    mid = P.mcmc_summary(run, truth=s["quantiles"][1])
    assert mid["frac_truth_below"][1] == 1.0


def test_python_rejections():
    run = _psgla_run(store="stats", n_chains=2, n_iter=10)
    with pytest.raises(ValueError, match="store='all'"):
        P.mcmc_summary(run)
    with pytest.raises(RuntimeError, match="CPU"):
        P.mcmc_summary(torch.zeros(8, 2, 5))
    with pytest.raises(TypeError, match="float32"):
        P.mcmc_summary(torch.zeros(8, 2, 5, dtype=torch.float64, device="cuda"))
    x = torch.rand(8, 2, 5, device="cuda")
    for b in (-1, 8, 5):
        with pytest.raises(ValueError, match="burn_in|4 draws"):
            P.mcmc_summary(x, burn_in=b)
    for probs in ((), (0.0,), (0.5, 1.0), (float("nan"),), tuple([0.5] * 9), (-0.2, 0.5)):
        with pytest.raises(ValueError, match="probs"):
            P.mcmc_summary(x, probs=probs)
    for h in (0.0, 1.0, float("nan"), 1.5):
        with pytest.raises(ValueError, match="hdi_prob"):
            P.mcmc_summary(x, hdi_prob=h)
    with pytest.raises(ValueError, match="shape"):
        P.mcmc_summary(x, truth=torch.zeros(4, device="cuda"))
