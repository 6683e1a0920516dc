"""-m gpu: the on-device convergence diagnostics (csrc/mcmc_diag.cu, ``psgla_b200.mcmc_diagnostics``) against the float64
restatement of arviz's rank-normalised split-R-hat and bulk / tail ESS (tests/mcmc_reference.py, PARITY UNPINNED against arviz
itself).

Stated tolerances (observed values are printed by ``observed``)
  * R-hat: |kernel - reference| <= 1e-4; ESS: relative error <= 1e-3.  The kernel's normal scores are fp32 (the reference's
    fp64) and its autocovariances sum fp32 centred values: both are ~1e-7 relative.
  * Except where Geyer's truncation rule meets a pair sum rho_2k + rho_2k+1 within rounding of 0: the two sides may then stop at
    different lags.  Such elements are counted; they must be below 0.1 % and each must show a pair sum below 1e-4 in the
    reference.
Bit-exact: two calls; an element alone and inside a larger batch; the in-place run path and the stacked Xlist."""
import numpy as np
import pytest
import torch

import mcmc_reference as R
import psgla_b200 as P
from conftest import observed

pytestmark = pytest.mark.gpu

RHAT_TOL, ESS_RTOL = 1e-4, 1e-3


def _draws(seed, N, M, E, quantise=False, constant=()):
    """AR(1) chains with a per-element correlation in [0, 0.95) and per-chain offsets (some elements far from mixed)."""
    rng = np.random.default_rng(seed)
    rho = rng.uniform(0, 0.95, E)
    off = rng.standard_normal((M, E)) * rng.choice([0.0, 0.05, 1.0], E)
    x = np.empty((N, M, E))
    x[0] = rng.standard_normal((M, E)) / np.sqrt(1 - rho ** 2)
    for n in range(1, N):
        x[n] = rho * x[n - 1] + rng.standard_normal((M, E))
    x = 0.5 + 0.1 * (x + off)
    if quantise:  # 8-bit images: many ties, so the average ranks matter
        x = np.round(np.clip(x, 0, 1) * 255) / 255
    for e in constant:
        x[:, :, e] = 0.25
    return x.astype(np.float32)


def _compare(x, got, what):
    """got: (rhat, ess_bulk, ess_tail) CUDA tensors; x: float32 draws [N, M, E]."""
    traces = []
    want = R.diag(x.astype(np.float64), traces)
    got = [g.double().cpu().numpy() for g in got]
    E = x.shape[2]
    for name, w, g in zip(("rhat", "ess_bulk", "ess_tail"), want, got):
        np.testing.assert_array_equal(np.isnan(g), np.isnan(w), err_msg="%s %s NaN pattern" % (what, name))
    ok = ~np.isnan(want[0])
    err_r = np.abs(got[0] - want[0])[ok]
    err_b = np.abs(got[1] / want[1] - 1)[~np.isnan(want[1])]
    err_t = np.abs(got[2] / want[2] - 1)[~np.isnan(want[2])]
    bad = np.zeros(E, bool)
    bad[~np.isnan(want[1])] |= err_b > ESS_RTOL
    bad[~np.isnan(want[2])] |= err_t > ESS_RTOL
    for e in np.flatnonzero(bad):
        assert traces[e]["min_pair"] < 1e-4, (what, e, got[1][e], want[1][e], got[2][e], want[2][e], traces[e])
    observed("%s: Geyer truncation flips" % what, bad.sum() / E, 1e-3 + 1e-12)
    observed("%s: R-hat |err|" % what, err_r.max() if err_r.size else 0.0, RHAT_TOL)
    ok_b, ok_t = err_b[err_b <= ESS_RTOL], err_t[err_t <= ESS_RTOL]
    observed("%s: bulk ESS rel err" % what, ok_b.max() if ok_b.size else 0.0, ESS_RTOL)
    observed("%s: tail ESS rel err" % what, ok_t.max() if ok_t.size else 0.0, ESS_RTOL)


@pytest.mark.parametrize("M,N,E,quantise", [(1, 400, 37, False), (2, 301, 53, False), (8, 200, 41, False),
                                            (8, 201, 29, True), (2, 1000, 1100, True), (4, 5, 67, False)])
def test_kernel_against_reference(M, N, E, quantise):
    x = _draws(M * 1000 + N, N, M, E, quantise, constant=(3, E - 1))
    d = P.mcmc_diagnostics(torch.from_numpy(x).cuda())
    assert d["n_draws"] == N and d["n_chains"] == M and d["rhat"].shape == (E,)
    assert np.isnan(d["rhat"][3].item()) and np.isnan(d["ess_bulk"][E - 1].item()) and np.isnan(d["ess_tail"][3].item())
    _compare(x, (d["rhat"], d["ess_bulk"], d["ess_tail"]), "M=%d N=%d E=%d q=%d" % (M, N, E, quantise))


@pytest.mark.parametrize("M,N", [(8, 2048), (8, 2049), (1, 16384)])
def test_size_limit_is_accepted(M, N):
    x = _draws(N, N, M, 3)
    d = P.mcmc_diagnostics(torch.from_numpy(x).cuda())
    _compare(x, (d["rhat"], d["ess_bulk"], d["ess_tail"]), "limit M=%d N=%d" % (M, N))


@pytest.mark.parametrize("M,N", [(8, 2050), (1, 16386), (4097, 4)])
def test_above_the_limit_is_rejected_on_the_host(M, N):
    x = torch.zeros((N, M, 1), device="cuda")
    with pytest.raises(ValueError, match="n_inter"):
        P.mcmc_diagnostics(x)
    lib = P._lib.lib()
    assert lib.psgla_mcmc_diag(x.data_ptr(), N, M, 1, x.data_ptr(), 1 << 20, x.data_ptr(), x.data_ptr(), x.data_ptr(),
                               None) == -1
    assert b"n_inter" in lib.psgla_last_error()


def test_deterministic_and_batch_invariant():
    x = torch.from_numpy(_draws(7, 300, 4, 500, True)).cuda()
    a, b = P.mcmc_diagnostics(x), P.mcmc_diagnostics(x)
    for k in ("rhat", "ess_bulk", "ess_tail"):
        assert torch.equal(a[k].nan_to_num(-1), b[k].nan_to_num(-1)), k
    for e in (0, 17, 499):
        one = P.mcmc_diagnostics(x[:, :, e:e + 1].contiguous())
        for k in ("rhat", "ess_bulk", "ess_tail"):
            assert torch.equal(one[k].nan_to_num(-1), a[k][e:e + 1].nan_to_num(-1)), (k, e)
    part = P.mcmc_diagnostics(x[:, :, 100:229].contiguous())
    for k in ("rhat", "ess_bulk", "ess_tail"):
        assert torch.equal(part[k].nan_to_num(-1), a[k][100:229].nan_to_num(-1)), k


def _psgla_run(store="all", n_chains=4, n_iter=40):
    torch.manual_seed(0)
    im = torch.rand(1, 3, 24, 32, device="cuda")
    dg, init, _, _ = P.make_inpainting(im, prop=0.5, sigma=1.0, seed_ip=0)
    den = P.DnCNN(pretrained=P.random_dncnn_state_dict(0))
    run = P.psgla_run(init, dg, den, alpha=1.0, lambd=5.0, sig_float=2 / 255, delta=(2 / 255) ** 2, n_iter=n_iter, n_inter=2,
                      n_inter_mmse=5, seed=1, n_chains=n_chains, store=store)
    for i in range(n_iter):
        run.step(i)
    run.finish()
    return run


def _same(a, b):
    for k in ("rhat", "ess_bulk", "ess_tail"):
        assert a[k].shape == b[k].shape and torch.equal(a[k].nan_to_num(-1), b[k].nan_to_num(-1)), k
    for k in ("rhat_max", "frac_rhat_above_1_01", "ess_bulk_min", "ess_bulk_median", "ess_tail_min", "n_draws", "n_chains"):
        assert a[k] == b[k] or (a[k] != a[k] and b[k] != b[k]), k


def test_sampler_run_in_place(monkeypatch):
    run = _psgla_run()
    assert len(run.Xlist) == 20
    stacked = P.mcmc_diagnostics(torch.stack(run.Xlist))
    seen = []
    real_ptr = P._lib.ptr
    monkeypatch.setattr(P._lib, "ptr", lambda t: seen.append(t.data_ptr() if t is not None else None) or real_ptr(t))
    in_place = P.mcmc_diagnostics(run)
    assert seen[0] == run.samples.data_ptr()  # the kernel reads the run's own buffer: no copy
    _same(in_place, stacked)
    assert in_place["rhat"].shape == (3, 24, 32) and in_place["n_chains"] == 4 and in_place["n_draws"] == 20
    seen.clear()
    burnt = P.mcmc_diagnostics(run, burn_in=6)
    assert seen[0] == run.samples[6].data_ptr()
    _same(burnt, P.mcmc_diagnostics(torch.stack(run.Xlist[6:])))
    assert burnt["n_draws"] == 14
    # a sampler's Xlist is accepted as it is
    _same(P.mcmc_diagnostics(run.Xlist), stacked)
    x = torch.stack(run.Xlist).reshape(20, 4, -1)
    _compare(x.cpu().numpy(), (stacked["rhat"].reshape(-1), stacked["ess_bulk"].reshape(-1), stacked["ess_tail"].reshape(-1)),
             "PSGLA DnCNN 4 chains")


def test_single_chain_xlist_forms():
    run = _psgla_run(n_chains=1, n_iter=16)
    xs = [t[0] for t in run.Xlist]  # [3, H, W], as psgla() returns for one chain
    d = P.mcmc_diagnostics(xs)
    assert d["n_chains"] == 1 and d["rhat"].shape == (3, 24, 32)
    _same(d, P.mcmc_diagnostics(run))
    g = P.mcmc_diagnostics([t[0, 0] for t in run.Xlist])  # [H, W], a grayscale chain's form
    assert g["rhat"].shape == (1, 24, 32)
    assert torch.equal(g["ess_bulk"][0].nan_to_num(-1), d["ess_bulk"][0].nan_to_num(-1))


def test_python_rejections():
    run = _psgla_run(store="stats", n_chains=2, n_iter=10)
    with pytest.raises(ValueError, match="store='all'"):
        P.mcmc_diagnostics(run)
    with pytest.raises(ValueError, match="store='all'"):
        P.mcmc_diagnostics(run.Xlist)
    with pytest.raises(RuntimeError, match="CPU"):
        P.mcmc_diagnostics(torch.zeros(8, 2, 3, 4, 4))
    with pytest.raises(ValueError, match="shapes"):
        P.mcmc_diagnostics([torch.zeros(2, 3, 4, 4, device="cuda")] * 5 + [torch.zeros(2, 3, 4, 5, device="cuda")])
    with pytest.raises(ValueError, match="burn_in"):
        P.mcmc_diagnostics(torch.zeros(8, 2, 5, device="cuda"), burn_in=8)
    with pytest.raises(ValueError, match="4 draws"):
        P.mcmc_diagnostics(torch.zeros(8, 2, 5, device="cuda"), burn_in=5)
