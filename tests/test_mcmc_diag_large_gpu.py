"""-m gpu: the device-wide convergence diagnostics for any S (csrc/mcmc_diag_large.cu, ``psgla_b200.mcmc_diagnostics_large``)
against the float64 restatement of arviz's rank-normalised split-R-hat and bulk / tail ESS (tests/mcmc_reference.py), with the
tolerances and the Geyer-flip rule of tests/test_mcmc_diag_gpu.py: R-hat |err| <= 1e-4, ESS relative error <= 1e-3, at most
0.1 % of elements truncating at a different lag, each with a reference pair sum below 1e-4.
Bit-exact: two calls; an element alone and inside a batch that spans two groups of elements."""
import numpy as np
import pytest
import torch

import psgla_b200 as P
from test_mcmc_diag_gpu import _compare, _draws

pytestmark = pytest.mark.gpu

KEYS = ("rhat", "ess_bulk", "ess_tail")


def _large(x, **kw):
    d = P.mcmc_diagnostics_large(torch.from_numpy(x).cuda() if isinstance(x, np.ndarray) else x, **kw)
    return d, (d["rhat"].reshape(-1), d["ess_bulk"].reshape(-1), d["ess_tail"].reshape(-1))


def _ar1(seed, rho, N, M, E):
    """Stationary AR(1) chains [N, M, E] (float64), unit innovations."""
    rng = np.random.default_rng(seed)
    x = np.empty((N, M, E))
    x[0] = rng.standard_normal((M, E)) / np.sqrt(1 - rho ** 2)
    for n in range(1, N):
        x[n] = rho * x[n - 1] + rng.standard_normal((M, E))
    return x


@pytest.mark.parametrize("M,N", [(8, 2050), (1, 16386), (4097, 4)])
def test_shapes_the_small_path_rejects(M, N):
    x = _draws(N + M, N, M, 3)
    d, got = _large(x)
    assert d["n_draws"] == N and d["n_chains"] == M
    _compare(x, got, "large M=%d N=%d" % (M, N))


def test_many_chains_few_draws():
    """The 2D shape: 20 000 chains x 400 draws x 2 elements, S = 8 x 10^6."""
    x = _draws(11, 400, 20000, 2)
    _compare(x, _large(x)[1], "large 20000 chains x 400 draws")


def test_few_chains_long_draws_slow_mixing():
    """rho = 0.95 (a long lag loop: several lag rounds), 2 chains, odd N = 20 001."""
    x = (0.5 + 0.1 * _ar1(3, 0.95, 20001, 2, 3)).astype(np.float32)
    _compare(x, _large(x)[1], "large rho 0.95 M=2 N=20001")


def test_quantised_draws_long_tie_runs():
    """8-bit values: 64 000 split draws on 256 levels, tie runs of hundreds to thousands; odd N; a constant and a NaN
    element."""
    x = _draws(5, 4001, 16, 6, quantise=True, constant=(2,))
    x[1000, 3, 4] = np.nan
    d, got = _large(x)
    assert np.isnan(d["rhat"][2].item()) and np.isnan(d["ess_bulk"][2].item()) and np.isnan(d["ess_tail"][2].item())
    assert np.isnan(d["rhat"][4].item()) and np.isnan(d["ess_bulk"][4].item()) and np.isnan(d["ess_tail"][4].item())
    _compare(x, got, "large quantised 16 chains x 4001 draws")


@pytest.mark.parametrize("M,N,E,quantise", [(1, 400, 37, False), (2, 301, 53, False), (8, 200, 41, False),
                                            (8, 201, 29, True), (2, 1000, 1100, True), (4, 5, 67, False)])
def test_small_shapes_against_reference(M, N, E, quantise):
    x = _draws(M * 1000 + N, N, M, E, quantise, constant=(3, E - 1))
    d, got = _large(x)
    assert d["rhat"].shape == (E,)
    assert np.isnan(d["rhat"][3].item()) and np.isnan(d["ess_bulk"][E - 1].item()) and np.isnan(d["ess_tail"][3].item())
    _compare(x, got, "large M=%d N=%d E=%d q=%d" % (M, N, E, quantise))


def test_bit_identical_and_independent_of_the_group():
    """S = 2^20, E = 300: groups of 2^28 / S = 256 elements, so the batch spans two groups."""
    g = torch.Generator(device="cuda").manual_seed(0)
    N, M, E = 1 << 17, 8, 300
    x = torch.randn((N, M, E), generator=g, device="cuda")
    x += torch.randn((1, M, E), generator=g, device="cuda") * 0.05  # chain offsets
    x[:, :, 7] = 0.5  # a constant element
    a = P.mcmc_diagnostics_large(x)
    b = P.mcmc_diagnostics_large(x)
    for k in KEYS:
        assert torch.equal(a[k].nan_to_num(-1), b[k].nan_to_num(-1)), k
    for e in (0, 7, 255, 256, 299):
        one = P.mcmc_diagnostics_large(x[:, :, e:e + 1].contiguous())
        for k in KEYS:
            assert torch.equal(one[k].nan_to_num(-1), a[k][e:e + 1].nan_to_num(-1)), (k, e)
    part = P.mcmc_diagnostics_large(x[:, :, 250:262].contiguous())
    for k in KEYS:
        assert torch.equal(part[k].nan_to_num(-1), a[k][250:262].nan_to_num(-1)), k


@pytest.mark.parametrize("alg", ["psgla", "pnp_ula"])
def test_gmm2d_trajectory_end_to_end(alg):
    """A 2D cell as bench.py sets it up (symmetric Gaussians, y = (0, -2)), 4 000 chains, 2 000 steps thinned by 4, diagnosed
    on the device from GMMChains.run's own trajectory and by the reference on its host copy."""
    prm = {"psgla": dict(delta=0.3, alpha=2.0 / 3.0, epsilon=1.0), "pnp_ula": dict(delta=0.1, alpha=1.5, epsilon=0.5)}[alg]
    mu, Sig, pi = P.gaussian_mixt_example("symetric_gaussians")
    y = np.array((0.0, -2.0))
    n = 4000
    x0 = torch.tensor(y, dtype=torch.float32, device="cuda").repeat(n, 1).contiguous()
    ch = P.GMMChains(alg, y, prm["delta"], np.eye(2), 1.0, P.Theorical_MMSE(mu, Sig, pi), prm["alpha"], prm["epsilon"],
                     n_chains=n, x0=x0, seed=3, dtype="float32", device="cuda")
    traj = ch.run(2000, thin=4)
    assert traj.shape == (500, n, 2) and traj.dtype == torch.float32
    d, got = _large(traj, burn_in=50)
    assert d["rhat"].shape == (2,) and d["n_draws"] == 450 and d["n_chains"] == n
    _compare(traj[50:].cpu().numpy(), got, "2D %s 4000 chains x 450 draws" % alg)


@pytest.mark.parametrize("seed", [1, 2])
def test_ar1_bulk_ess(seed):
    """Stationary AR(1), rho = 0.5, 2 000 chains x 1 000 draws: bulk ESS within 5 % of S (1 - rho) / (1 + rho) (the reference
    gives 1.014 and 1.016 times it for these seeds)."""
    x = _ar1(seed, 0.5, 1000, 2000, 1).astype(np.float32)
    d, _ = _large(x)
    want = 2000 * 1000 * 0.5 / 1.5
    assert abs(d["ess_bulk"].item() / want - 1) < 0.05, (d["ess_bulk"].item(), want)


def test_python_rejections():
    with pytest.raises(TypeError, match="float32"):
        P.mcmc_diagnostics_large(torch.zeros(8, 2, 5, dtype=torch.float64, device="cuda"))
    with pytest.raises(RuntimeError, match="CPU"):
        P.mcmc_diagnostics_large(torch.zeros(8, 2, 5))
    with pytest.raises(ValueError, match="4 draws"):
        P.mcmc_diagnostics_large(torch.zeros(8, 2, 5, device="cuda"), burn_in=5)
    with pytest.raises(ValueError, match="mcmc_diagnostics_large"):
        P.mcmc_diagnostics(torch.zeros(2050, 8, 1, device="cuda"))
