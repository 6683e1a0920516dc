"""Convergence diagnostics of multi-chain image runs, on the device: rank-normalised split-R-hat and bulk / tail ESS per pixel
(Vehtari, Gelman, Simpson, Carpenter, Buerkner 2021; arviz's rhat(method="rank"), ess(method="bulk"), ess(method="tail")).

    d = psgla_b200.mcmc_diagnostics(run, burn_in=100)      # run = psgla_run(...) / pnpula_run(...) after its steps
    d["rhat"], d["ess_bulk"], d["ess_tail"]                  # [C, H, W] maps
    d["rhat_max"], d["frac_rhat_above_1_01"], d["ess_bulk_min"], d["ess_bulk_median"], d["ess_tail_min"]

    d = psgla_b200.mcmc_diagnostics_large(traj, burn_in=b)  # traj = GMMChains.run(n, thin=k): [N, M, 2]

and the posterior summary with its Monte Carlo standard errors (arviz's _mcse_mean, _mcse_quantile, _ess_mean,
_ess_quantile, _hdi), with the calibration check against a ground truth:

    s = psgla_b200.mcmc_summary(run, burn_in=100, probs=(0.05, 0.5, 0.95), hdi_prob=0.94, truth=x_true)
    s["mean"], s["sd"], s["mcse_mean"], s["ess_mean"], s["hdi_low"], s["hdi_high"]   # [C, H, W] maps
    s["quantiles"], s["mcse_quantiles"], s["ess_quantiles"]                          # [P, C, H, W]
    s["coverage_hdi"], s["frac_truth_below"]                                        # with truth=

The kernels (csrc/mcmc_diag.cu, csrc/mcmc_diag_large.cu, csrc/mcmc_summary.cu) read the draws where the sampler stored them, [N][M][C][H][W]: a run
object is diagnosed in place, with no copy.  mcmc_diagnostics sorts one element in shared memory: S = 2 M floor(N / 2) <=
PSGLA_MCMC_MAX_DRAWS = 16 384 split draws per element.  mcmc_diagnostics_large computes the same statistics device-wide for
S up to 2^31 - 1 (a 2D population of 10^6 chains x 2 000 draws, an image run with the reference's own thinning), with a
workspace of about 16 bytes per split draw of a group of elements.  mcmc_summary runs on the engine of
mcmc_diagnostics_large, with the same inputs and limits.
"""
from __future__ import annotations

import ctypes as C

import torch

from . import _lib

__all__ = ["mcmc_diagnostics", "mcmc_diagnostics_large", "mcmc_summary", "MAX_DRAWS", "MAX_DRAWS_LARGE", "MAX_PROBS"]

MAX_DRAWS = 16384  # PSGLA_MCMC_MAX_DRAWS
MAX_DRAWS_LARGE = 2 ** 31 - 1  # psgla_mcmc_diag_large
MAX_PROBS = 8  # PSGLA_MCMC_MAX_PROBS


def _as_draws(draws):
    """-> (contiguous CUDA fp32 [N, M, E] tensor, map shape [C, H, W], crop (h, w) or None)."""
    from .restoration_algorithms import _Run
    if isinstance(draws, _Run):
        if draws.samples is None:
            raise ValueError("mcmc_diagnostics needs stored draws: this run has store='stats', which keeps none (run it "
                             "with store='all')")
        n = len(draws.Xlist)  # slots written so far
        x = draws.samples[:n]  # [n, B, C, Hp, Wp], a contiguous view of the run's own buffer
        return x, tuple(x.shape[2:]), draws.crop
    if isinstance(draws, (list, tuple)):
        if len(draws) == 0:
            raise ValueError("mcmc_diagnostics needs stored draws: Xlist is empty (a store='stats' run keeps none; run it "
                             "with store='all')")
        shapes = {tuple(t.shape) for t in draws}
        if len(shapes) != 1:
            raise ValueError("the draws of the list have different shapes: %s" % sorted(shapes))
        for t in draws:
            _check_tensor(t)
        x = torch.stack(list(draws))
        if x.dim() == 3:    # squeezed single grayscale chain [H, W]
            x = x[:, None, None]
        elif x.dim() == 4:  # squeezed single chain [C, H, W]
            x = x[:, None]
        if x.dim() != 5:
            raise ValueError("Xlist entries must be [M, C, H, W], [C, H, W] or [H, W], got %s" % (tuple(draws[0].shape),))
        return x, tuple(x.shape[2:]), None
    if isinstance(draws, torch.Tensor):
        _check_tensor(draws)
        if draws.dim() not in (3, 5):
            raise ValueError("draws must be [N, M, C, H, W] or [N, M, E], got %s" % (tuple(draws.shape),))
        return draws, tuple(draws.shape[2:]), None
    raise TypeError("draws must be a CUDA tensor, a sampler's Xlist or a psgla_run / pnpula_run object")


def _check_tensor(t):
    if not isinstance(t, torch.Tensor):
        raise TypeError("expected torch tensors, got %s" % type(t).__name__)
    if not t.is_cuda:
        raise RuntimeError("mcmc_diagnostics needs CUDA tensors: there is no CPU path")
    if t.dtype != torch.float32:
        raise TypeError("draws must be float32 (the samplers' dtype), got %s" % t.dtype)


def _prepare(draws, burn_in):
    """-> (contiguous fp32 [N, M, ...] CUDA tensor after burn-in, N, M, E, map shape, crop); the checks both paths share."""
    x, map_shape, crop = _as_draws(draws)
    burn_in = int(burn_in)
    if burn_in < 0 or burn_in >= x.shape[0]:
        raise ValueError("burn_in = %d must be in [0, %d) (the number of stored draws)" % (burn_in, x.shape[0]))
    x = x[burn_in:]
    if not x.is_contiguous():
        x = x.contiguous()
    N, M = int(x.shape[0]), int(x.shape[1])
    if N < 4:
        raise ValueError("split chains need at least 4 draws after burn-in, got %d" % N)
    return x, N, M, x[0, 0].numel(), map_shape, crop


def _check_large(N, M):
    S = 2 * M * (N // 2)
    if S > MAX_DRAWS_LARGE:
        raise ValueError("%d chains x %d draws give S = %d split draws per element, above the limit of 2^31 - 1: thin more, "
                         "raise burn_in or diagnose fewer chains" % (M, N, S))


def _run(fn, ws_bytes, x, N, M, E, map_shape, crop, name):
    """Calls the C-ABI diagnostics ``fn`` and builds the result dict from its [3, E] output."""
    with torch.cuda.device(x.device):
        ws = torch.empty(ws_bytes, dtype=torch.uint8, device=x.device)
        out = torch.empty((3, E), dtype=torch.float32, device=x.device)
        _lib.check(fn(_lib.ptr(x), N, M, E, _lib.ptr(ws), C.c_size_t(ws_bytes), out[0].data_ptr(), out[1].data_ptr(),
                      out[2].data_ptr(), _lib.stream_ptr(x.device)), name)
    maps = out.reshape((3,) + map_shape)
    if crop is not None:
        maps = maps[..., :crop[0], :crop[1]]
    rhat, ess_bulk, ess_tail = maps[0], maps[1], maps[2]

    def finite(t):
        t = t.reshape(-1)
        return t[~torch.isnan(t)]

    r, b, t = finite(rhat), finite(ess_bulk), finite(ess_tail)
    nan = float("nan")
    return {
        "rhat": rhat, "ess_bulk": ess_bulk, "ess_tail": ess_tail,
        "rhat_max": float(r.max()) if r.numel() else nan,
        "frac_rhat_above_1_01": float((rhat > 1.01).sum()) / rhat.numel(),
        "ess_bulk_min": float(b.min()) if b.numel() else nan,
        "ess_bulk_median": float(b.median()) if b.numel() else nan,
        "ess_tail_min": float(t.min()) if t.numel() else nan,
        "n_draws": N, "n_chains": M,
    }


def mcmc_diagnostics(draws, *, burn_in: int = 0) -> dict:
    """Rank-normalised split-R-hat and bulk / tail ESS of every element of a multi-chain run.

    draws: a CUDA fp32 tensor [N, M, C, H, W] or [N, M, E] (N stored draws of M chains); a sampler's ``Xlist`` (entries
    [M, C, H, W], or the squeezed single-chain [C, H, W] / [H, W], taken as M = 1); or a ``psgla_run`` / ``pnpula_run`` object,
    read in place from its sample buffer (the slots written so far).  A DRUNet run padded to multiples of 8 is diagnosed at the
    padded size and the maps are cropped like its outputs.  burn_in: the first ``burn_in`` draws are dropped.

    Returns a dict: ``rhat``, ``ess_bulk``, ``ess_tail`` -- CUDA fp32 maps [C, H, W] (an [N, M, E] tensor gives [E]) --, and
    the floats ``rhat_max``, ``frac_rhat_above_1_01``, ``ess_bulk_min``, ``ess_bulk_median``, ``ess_tail_min`` over the
    elements whose statistic is not NaN (NaN: NaN draws, or an element constant within every split chain; the fraction counts
    NaN as not above; the median is torch's, the lower middle value for an even count), and the ints ``n_draws``,
    ``n_chains``.  Stream-ordered on the current stream; reading the scalars synchronises it.  Up to 16 384 split draws per
    element; mcmc_diagnostics_large takes more."""
    x, N, M, E, map_shape, crop = _prepare(draws, burn_in)
    S = 2 * M * (N // 2)
    if S > MAX_DRAWS:
        raise ValueError("%d chains x %d draws give S = %d split draws per element, above the limit of %d: store fewer draws "
                         "(thin more with a larger n_inter), raise burn_in, diagnose fewer chains, or use "
                         "mcmc_diagnostics_large" % (M, N, S, MAX_DRAWS))
    lib = _lib.lib()
    return _run(lib.psgla_mcmc_diag, lib.psgla_mcmc_diag_workspace_bytes(N, M), x, N, M, E, map_shape, crop,
                "psgla_mcmc_diag")


def mcmc_diagnostics_large(draws, *, burn_in: int = 0) -> dict:
    """mcmc_diagnostics for up to 2^31 - 1 split draws per element (csrc/mcmc_diag_large.cu): the same inputs, definitions and
    result dict, computed device-wide (radix sort, tie runs, autocovariances in rounds of lags) instead of in one CTA's shared
    memory.  The 2D trajectory of ``GMMChains.run(n, thin=k)`` ([N, M, 2] fp32) is taken as it is:

        d = psgla_b200.mcmc_diagnostics_large(chains.run(n_steps, thin=k), burn_in=b)   # rhat, ess_bulk, ess_tail: [2]

    The workspace is allocated per call: about 16 bytes per split draw of a group of min(E, 2^28 / S) elements."""
    x, N, M, E, map_shape, crop = _prepare(draws, burn_in)
    _check_large(N, M)
    lib = _lib.lib()
    return _run(lib.psgla_mcmc_diag_large, lib.psgla_mcmc_diag_large_workspace_bytes(N, M, E), x, N, M, E, map_shape, crop,
                "psgla_mcmc_diag_large")


def _open_unit(v, name):
    v = float(v)
    if not 0.0 < v < 1.0:  # NaN fails too
        raise ValueError("%s = %r must be in the open interval (0, 1)" % (name, v))
    return v


def mcmc_summary(draws, *, burn_in: int = 0, probs=(0.05, 0.5, 0.95), hdi_prob: float = 0.94, truth=None) -> dict:
    """Posterior summary of every element of a multi-chain run with its Monte Carlo standard errors, on the device
    (csrc/mcmc_summary.cu, on the engine of mcmc_diagnostics_large), as arviz's published functions define it.  With A the
    N M draws of an element after burn-in (the middle draws of odd N included) and split chains as in mcmc_diagnostics:

      mean, sd          fp64 mean and sd (ddof 1) of A
      ess_mean          Geyer ESS of the raw draws in split-chain order (arviz's _ess_mean: not rank-normalised)
      mcse_mean         sd / sqrt(ess_mean): the Monte Carlo error of the MMSE estimate
      quantiles[i]      np.quantile(A, probs[i]) (method "linear")
      ess_quantiles[i]  Geyer ESS of the indicator x <= quantiles[i] (_ess_quantile; at 0.05 / 0.95 the tail ESS's series)
      mcse_quantiles[i] _mcse_quantile: half the distance between the sorted draws at the Beta(ess p + 1, ess (1 - p) + 1)
                        quantiles 0.1586553 / 0.8413447 of the draw ranks
      hdi_low, hdi_high the narrowest interval holding floor(hdi_prob N M) + 1 sorted draws (_hdi; ties: the lowest)

    draws: as mcmc_diagnostics_large (a run object read in place, an Xlist, [N, M, C, H, W] or [N, M, E]); a padded DRUNet
    run's maps are cropped like its outputs.  probs: 1 to 8 probabilities in (0, 1); hdi_prob in (0, 1).

    Returns a dict of CUDA fp32 maps ``mean``, ``sd``, ``mcse_mean``, ``ess_mean``, ``hdi_low``, ``hdi_high`` (the map shape)
    and ``quantiles``, ``mcse_quantiles``, ``ess_quantiles`` ([P, *map]); ``probs``, ``hdi_prob``, ``n_draws``, ``n_chains``;
    the floats ``mcse_mean_max`` and ``mcse_quantiles_max`` (a list, one per p) over the elements where they are not NaN.
    NaN draws make every output of their element NaN; a series constant within every split chain gives NaN for its ESS and
    MCSE.  ``truth`` (the ground truth at the map shape) adds ``coverage_hdi``, the fraction of the elements with an HDI
    (not NaN) that hold it, and ``frac_truth_below`` (one per p), the fraction of the elements with a quantile that it does not
    exceed: for calibrated intervals these approach hdi_prob and p.  Stream-ordered on the current stream; the scalars
    synchronise it."""
    x, N, M, E, map_shape, crop = _prepare(draws, burn_in)
    _check_large(N, M)
    probs = tuple(_open_unit(p, "probs[%d]" % i) for i, p in enumerate(probs))
    if not 1 <= len(probs) <= MAX_PROBS:
        raise ValueError("probs must hold 1 to %d probabilities, got %d" % (MAX_PROBS, len(probs)))
    hdi_prob = _open_unit(hdi_prob, "hdi_prob")
    P = len(probs)
    lib = _lib.lib()
    ws_bytes = lib.psgla_mcmc_summary_workspace_bytes(N, M, E, P)
    with torch.cuda.device(x.device):
        ws = torch.empty(ws_bytes, dtype=torch.uint8, device=x.device)
        out = torch.empty((6 + 3 * P, E), dtype=torch.float32, device=x.device)
        maps6, per_p = out[:6], out[6:].reshape(3, P, E)
        _lib.check(lib.psgla_mcmc_summary(
            _lib.ptr(x), N, M, E, (C.c_double * P)(*probs), P, hdi_prob, _lib.ptr(ws), C.c_size_t(ws_bytes),
            *[maps6[i].data_ptr() for i in range(4)], *[per_p[i].data_ptr() for i in range(3)], maps6[4].data_ptr(),
            maps6[5].data_ptr(), _lib.stream_ptr(x.device)), "psgla_mcmc_summary")
    maps6 = maps6.reshape((6,) + map_shape)
    per_p = per_p.reshape((3, P) + map_shape)
    if crop is not None:
        maps6, per_p = maps6[..., :crop[0], :crop[1]], per_p[..., :crop[0], :crop[1]]
    mean, sd, mcse_mean, ess_mean, hdi_low, hdi_high = maps6
    quantiles, mcse_quantiles, ess_quantiles = per_p

    def finite_max(t):
        t = t.reshape(-1)
        t = t[~torch.isnan(t)]
        return float(t.max()) if t.numel() else float("nan")

    res = {
        "mean": mean, "sd": sd, "mcse_mean": mcse_mean, "ess_mean": ess_mean, "hdi_low": hdi_low, "hdi_high": hdi_high,
        "quantiles": quantiles, "mcse_quantiles": mcse_quantiles, "ess_quantiles": ess_quantiles,
        "probs": probs, "hdi_prob": hdi_prob, "n_draws": N, "n_chains": M,
        "mcse_mean_max": finite_max(mcse_mean), "mcse_quantiles_max": [finite_max(t) for t in mcse_quantiles],
    }
    if truth is not None:
        if not isinstance(truth, torch.Tensor):
            raise TypeError("truth must be a torch tensor, got %s" % type(truth).__name__)
        if tuple(truth.shape) != tuple(mean.shape):
            raise ValueError("truth has shape %s; the summary maps have shape %s" % (tuple(truth.shape), tuple(mean.shape)))
        t = truth.to(device=mean.device, dtype=torch.float32)
        ok = ~torch.isnan(hdi_low)
        n_ok = int(ok.sum())
        res["coverage_hdi"] = (float(((hdi_low <= t) & (t <= hdi_high) & ok).sum()) / n_ok) if n_ok else float("nan")
        below = []
        for q in quantiles:
            okq = ~torch.isnan(q)
            n_q = int(okq.sum())
            below.append(float(((t <= q) & okq).sum()) / n_q if n_q else float("nan"))
        res["frac_truth_below"] = below
    return res
