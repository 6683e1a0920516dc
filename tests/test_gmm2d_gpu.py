"""-m gpu: the 2D chain kernel through the drop-in API / C ABI against the CPU oracle, the golden vectors generated
from the unmodified reference, and the closed-form posterior.

Stated tolerances: fp64 kernel vs float64 reference <= 1e-9 abs per iterate (observed ~1e-14); fp32 kernel <= 1e-3 abs
per iterate under replayed noise (observed ~3e-6; SURVEY 7 "hard parts")."""
import json
import os

import numpy as np
import pytest
import torch

import psgla_b200 as P
from oracle import gmm2d_oracle as o

pytestmark = pytest.mark.gpu
GOLD = json.load(open(os.path.join(os.path.dirname(__file__), "golden", "gmm2d_golden.json")))
TOL64, TOL32 = 1e-9, 1e-3


def test_denoiser_golden_points():
    for name in o.PRIOR_NAMES:
        D = P.Theorical_MMSE(*P.gaussian_mixt_example(name))
        for eps in (0.3, 0.5, 0.05):
            rows = [g for g in GOLD["denoiser"] if g["prior"] == name and g["eps"] == eps]
            got = D(np.array([g["x"] for g in rows]), eps)
            assert np.allclose(got, np.array([g["D"] for g in rows]), rtol=1e-11, atol=1e-11)
        assert D(np.array([1.0, 2.0]), 0.3).shape == (2,)


def test_denoiser_far_from_modes_is_finite_where_reference_is_nan():
    D = P.Theorical_MMSE(*P.gaussian_mixt_example("symetric_gaussians"))
    x = np.array([60.0, -60.0])
    with np.errstate(all="ignore"):
        ref = o.theorical_mmse(*o.gaussian_mixt_example("symetric_gaussians"))(x, 0.3)
    assert not np.all(np.isfinite(ref))  # plain exp underflows to 0/0 (utils_2D.py:223-232)
    assert np.all(np.isfinite(D(x, 0.3)))  # log-sum-exp form


@pytest.mark.parametrize("idx", range(len(GOLD["trajectories"])))
def test_golden_trajectories_replay(idx):
    g = GOLD["trajectories"][idx]
    D = P.Theorical_MMSE(*P.gaussian_mixt_example(g["prior"]))
    y = np.array(g["y"], dtype=float)
    A = np.array(g.get("A", np.eye(2)))
    sigma = g.get("sigma", 1)
    noise = np.array(g["noise"])
    want = np.array(g["X"])
    for dtype, tol in (("float64", TOL64), ("float32", TOL32)):
        if g["alg"] == "psgla":
            delta, alpha = g.get("params", [o.PSGLA_DELTA, o.PSGLA_ALPHA])
            X = P.SnoPnP_ULA(g["N"], y, y, delta, A, sigma, D, alpha, noise=noise, dtype=dtype)
        else:
            delta, eps, alpha = g.get("params", [o.ULA_DELTA, o.ULA_EPSILON, o.ULA_ALPHA])
            X = P.PnP_ULA(g["N"], y, y, delta, A, sigma, D, eps, alpha, noise=noise, dtype=dtype)
        assert X.shape == want.shape and X.dtype == np.float64
        assert np.abs(X - want).max() <= tol, (dtype, np.abs(X - want).max())


def test_global_numpy_stream_drop_in():
    """np.random.seed(k) + call == the reference's trajectory: the default rng replays the global NumPy stream."""
    g = next(t for t in GOLD["trajectories"] if t["prior"] == "symetric_gaussians" and t["y"] == [0, -2] and t["alg"] == "psgla")
    D = P.Theorical_MMSE(*P.gaussian_mixt_example("symetric_gaussians"))
    np.random.seed(0)
    X = P.SnoPnP_ULA(g["N"], np.array([0, -2]), np.array([0, -2]), 0.3, np.eye(2), 1, D, 2 / 3)
    assert np.abs(X - np.array(g["X"])).max() <= TOL64
    assert np.allclose(X[1], [-0.4973529172, -2.4721697964], atol=1e-9)  # SURVEY 8c


def test_long_replay_all_cells_fp32_tolerance():
    rng = np.random.default_rng(7)
    worst = 0.0
    for name in o.PRIOR_NAMES:
        mu, Sig, pi = o.gaussian_mixt_example(name)
        D, Do = P.Theorical_MMSE(mu, Sig, pi), o.theorical_mmse(mu, Sig, pi)
        for y in o.OBSERVATIONS:
            y = y.astype(float)
            noise = rng.standard_normal((1999, 2))
            want = o.snopnp_ula(2000, y, y, 0.3, np.eye(2), 1, Do, 2 / 3, noise=noise)
            got = P.SnoPnP_ULA(2000, y, y, 0.3, np.eye(2), 1, D, 2 / 3, noise=noise, dtype="float32")
            worst = max(worst, np.abs(got - want).max())
            got64 = P.SnoPnP_ULA(2000, y, y, 0.3, np.eye(2), 1, D, 2 / 3, noise=noise)
            assert np.abs(got64 - want).max() <= TOL64
    assert worst <= TOL32, worst


def test_many_chains_replay_matches_batched_oracle():
    rng = np.random.default_rng(3)
    mu, Sig, pi = o.gaussian_mixt_example("cross")
    D = P.Theorical_MMSE(mu, Sig, pi)
    C, n = 3000, 64  # not a multiple of the block size: ragged tail
    noise = rng.standard_normal((n, C, 2))
    x0 = rng.uniform(-3, 3, size=(C, 2))
    y = np.array([0.5, -1.0])
    for alg, kw in (("psgla", dict(delta=0.3, alpha=2 / 3)), ("pnp_ula", dict(delta=0.1, alpha=1.5, epsilon=0.5))):
        want, want_traj = o.run_chains(alg, n, x0, y, A=np.eye(2), sigma=1, mu_list=mu, sigma_list=Sig, pi_list=pi,
                                       noise=noise, thin=16, **kw)
        for dtype, tol in (("float64", TOL64), ("float32", TOL32)):
            fin, traj = P.run_chains(alg, n, y, A=np.eye(2), sigma=1, denoiser=D, n_chains=C, x0=x0, noise=noise, thin=16,
                                     dtype=dtype, **kw)
            assert np.abs(fin.cpu().numpy() - want).max() <= tol
            assert traj.shape == (4, C, 2) and np.abs(traj.cpu().numpy() - want_traj).max() <= tol


def test_general_r_path_three_components():
    rng = np.random.default_rng(4)
    mu = [np.array([2.0, 0.0]), np.array([-2.0, 1.0]), np.array([0.0, -3.0])]
    Sig = [np.eye(2), np.array([[1.0, 0.3], [0.3, 0.5]]), np.eye(2) * 0.4]
    pi = [0.2, 0.5, 0.3]
    D = P.Theorical_MMSE(mu, Sig, pi)
    Do = o.theorical_mmse(mu, Sig, pi)
    x = rng.uniform(-5, 5, size=(200, 2))
    assert np.allclose(D(x, 0.3), np.array([Do(xi, 0.3) for xi in x]), atol=1e-11)
    y = np.array([0.0, 0.0])
    noise = rng.standard_normal((99, 2))
    want = o.snopnp_ula(100, y, y, 0.3, np.eye(2), 1, Do, 2 / 3, noise=noise)
    assert np.abs(P.SnoPnP_ULA(100, y, y, 0.3, np.eye(2), 1, D, 2 / 3, noise=noise) - want).max() <= TOL64
    assert np.abs(P.SnoPnP_ULA(100, y, y, 0.3, np.eye(2), 1, D, 2 / 3, noise=noise, dtype="float32") - want).max() <= TOL32


def test_philox_noise_is_standard_normal_and_replayable():
    lib = P._lib.lib()
    C, n = 50000, 8
    z = torch.empty(n, C, 2, device="cuda")
    P._lib.check(lib.psgla_gmm2d_noise(z.data_ptr(), C, 17, n, 3, 1234, None), "noise")
    torch.cuda.synchronize()
    zz = z.double().cpu().numpy().reshape(-1)
    assert abs(zz.mean()) < 5e-3 and abs(zz.var() - 1) < 1e-2
    assert abs((zz ** 3).mean()) < 2e-2 and abs((zz ** 4).mean() - 3) < 5e-2
    assert abs(np.corrcoef(zz[0::2], zz[1::2])[0, 1]) < 5e-3
    # the kernel consumes exactly these draws: Philox run == replay of the dumped stream
    mu, Sig, pi = P.gaussian_mixt_example("disymmetric_gaussians")
    D = P.Theorical_MMSE(mu, Sig, pi)
    y = np.array([0.0, -2.0])
    a, _ = P.run_chains("psgla", n, y, 0.3, np.eye(2), 1, D, 2 / 3, n_chains=C, seed=1234, chain_id0=17, philox_offset=3)
    b, _ = P.run_chains("psgla", n, y, 0.3, np.eye(2), 1, D, 2 / 3, n_chains=C, noise=z)
    assert torch.equal(a, b)


@pytest.mark.parametrize("alg", ["psgla", "pnp_ula"])
@pytest.mark.parametrize("name,A", [("symetric_gaussians", np.eye(2)), ("disymmetric_gaussians", np.eye(2)), ("cross", np.eye(2)),
                                    ("symetric_gaussians", np.array([[1.0, 0.3], [-0.2, 0.8]]))])
def test_lean_kernel_and_every_launch_geometry_equal_the_replayed_stream(name, A, alg):
    """Each launch path of csrc/gmm2d.cu must consume exactly the library's Philox stream and do the general kernel's
    arithmetic: a Philox run == the replay of the dumped draws, bit for bit, in the number of launches its policy makes.
      fp32, no trajectory: the register-lean one-chain-per-thread kernel with 4 Philox blocks per round and its
        constants-structure specialisation (STRUCT 2 on the diagonal priors, 1 on `cross`, 0 with a non-diagonal A); 45 steps
        from the odd global step 3 = 1 lead step + 5 lean rounds of 8 + 4 tail steps, 3 launches;
      fp32 with a trajectory: one launch of the general kernel in 1-warp blocks (final state and trajectory rows);
      fp64: occupancy-sized waves of the general kernel.  2 * 10^6 chains are more than 4 per resident thread at any
        occupancy of its 128-thread blocks (at most 16 per SM), so full waves of 4 chains per thread and a remainder wave run."""
    lib = P._lib.lib()
    C, n, off, thin = 2_000_003, 45, 3, 16
    z = torch.empty(n, C, 2, device="cuda")
    P._lib.check(lib.psgla_gmm2d_noise(z.data_ptr(), C, 5, n, off, 77, None), "noise")
    D = P.Theorical_MMSE(*P.gaussian_mixt_example(name))
    y = np.array([0.0, -2.0])
    prm = dict(delta=0.3, alpha=2 / 3, epsilon=1.0) if alg == "psgla" else dict(delta=0.1, alpha=1.5, epsilon=0.5)
    kw = dict(y=y, A=A, sigma=1, denoiser=D, n_chains=C, **prm)
    philox = dict(seed=77, chain_id0=5, philox_offset=off)
    want, want_traj = P.run_chains(alg, n, noise=z, thin=thin, **kw)
    got, _ = P.run_chains(alg, n, **philox, **kw)
    assert torch.equal(got, want) and lib.psgla_gmm2d_last_launches() == 3
    got, traj = P.run_chains(alg, n, thin=thin, **philox, **kw)
    assert torch.equal(got, want) and torch.equal(traj, want_traj) and lib.psgla_gmm2d_last_launches() == 1
    want, _ = P.run_chains(alg, n, noise=z, dtype="float64", **kw)
    got, _ = P.run_chains(alg, n, dtype="float64", **philox, **kw)
    assert torch.equal(got, want) and lib.psgla_gmm2d_last_launches() >= 2  # every launch but the last is a full wave


def test_sharding_and_segmentation_invariance():
    """Chain i's result depends only on (seed, global id, step index): not on the shard or on how steps are split."""
    mu, Sig, pi = P.gaussian_mixt_example("cross")
    D = P.Theorical_MMSE(mu, Sig, pi)
    y = np.array([0.0, -2.0])
    kw = dict(y=y, delta=0.1, A=np.eye(2), sigma=1, denoiser=D, alpha=1.5, epsilon=0.5)
    full, _ = P.run_chains("pnp_ula", 101, n_chains=5000, seed=9, **kw)
    lo, _ = P.run_chains("pnp_ula", 101, n_chains=1999, seed=9, chain_id0=0, **kw)
    hi, _ = P.run_chains("pnp_ula", 101, n_chains=3001, seed=9, chain_id0=1999, **kw)
    assert torch.equal(full, torch.cat([lo, hi]))
    ch = P.GMMChains("pnp_ula", n_chains=5000, seed=9, **kw)
    ch.run(37)
    ch.run(64)
    assert torch.equal(full, ch.state)


@pytest.mark.parametrize("alg", ["psgla", "pnp_ula"])
@pytest.mark.parametrize("name", o.PRIOR_NAMES)
def test_statistical_parity_with_oracle_population(name, alg):
    """In-kernel Philox chains against an oracle population driven by NumPy noise: the two empirical laws after 600
    steps must agree (means within 6 standard errors, covariances within 10 %), and both must sit near the closed-form
    posterior (utils_2D.py:139-162) up to the discretisation bias of the scheme (the reference's figure reports W2^2
    up to ~0.8 for PSGLA and ~24 for PnP-ULA at these step sizes)."""
    mu, Sig, pi = P.gaussian_mixt_example(name)
    D = P.Theorical_MMSE(mu, Sig, pi)
    y = np.array([0.0, -2.0])
    prm = dict(psgla=dict(delta=0.3, alpha=2 / 3, epsilon=1.0), pnp_ula=dict(delta=0.1, alpha=1.5, epsilon=0.5))[alg]
    n_steps, n_gpu, n_cpu = 600, 400000, 20000
    fin, _ = P.run_chains(alg, n_steps, y, prm["delta"], np.eye(2), 1, D, prm["alpha"], prm["epsilon"], n_chains=n_gpu, seed=0)
    X = fin.double().cpu().numpy()
    assert np.all(np.isfinite(X))
    Xo = o.run_chains(alg, n_steps, np.tile(y, (n_cpu, 1)), y, prm["delta"], np.eye(2), 1, mu, Sig, pi, prm["alpha"],
                      epsilon=prm["epsilon"], rng=np.random.default_rng(11))
    se = np.sqrt(Xo.var(0) / n_cpu + X.var(0) / n_gpu)
    assert np.all(np.abs(X.mean(0) - Xo.mean(0)) < 6 * se + 1e-3), (X.mean(0), Xo.mean(0), se)
    cg, co = np.cov(X.T), np.cov(Xo.T)
    assert np.abs(cg - co).max() < 0.1 * np.abs(co).max() + 0.02, (cg, co)
    # sliced W2 between the two populations is at the Monte-Carlo floor of two 20 000-point clouds of one law
    assert P.sliced_wasserstein_distance(X[:n_cpu], Xo, seed=0) < 0.08
    # and both sit as close to the exact posterior as the scheme's bias allows (W2^2 averaged over 6 subsamples)
    rng = np.random.default_rng(0)
    post = P.sample_posterior(np.eye(2), y, 1, 200000, mu, Sig, pi, rng=rng)
    w_gpu = np.mean([P.Wasserstein_distance(X, post, rng=rng) for _ in range(6)])
    w_cpu = np.mean([P.Wasserstein_distance(Xo, post, rng=rng) for _ in range(6)])
    assert abs(w_gpu - w_cpu) < 0.5 * max(w_cpu, 0.2) + 0.15, (w_gpu, w_cpu)


def test_metric_each_step_interleaving():
    mu, Sig, pi = P.gaussian_mixt_example("symetric_gaussians")
    D = P.Theorical_MMSE(mu, Sig, pi)
    y = np.array([0.0, -2.0])
    np.random.seed(0)
    post = P.sample_posterior(np.eye(2), y, 1, 300, mu, Sig, pi)
    X, W = P.SnoPnP_ULA(250, y, y, 0.3, np.eye(2), 1, D, 2 / 3, Sample_posterior=post, compute_metric_each_step=True)
    assert X.shape == (250, 2) and len(W) == 3 and all(np.isfinite(W))  # i = 0, 100, 200 (sampling_2D.py:65)


def test_bad_arguments_raise():
    D = P.Theorical_MMSE(*P.gaussian_mixt_example("cross"))
    with pytest.raises(RuntimeError, match="must be > 0"):
        P.run_chains("psgla", 4, np.zeros(2), -1.0, np.eye(2), 1, D, 2 / 3)
    with pytest.raises(ValueError):
        P.Theorical_MMSE([np.zeros(2)] * 17, [np.eye(2)] * 17, [1 / 17] * 17)
