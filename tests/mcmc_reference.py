"""float64 numpy / scipy restatement of rank-normalised split-R-hat and bulk / tail ESS (Vehtari, Gelman, Simpson, Carpenter,
Buerkner 2021), following arviz's ``_split_chains``, ``_z_scale``, ``_rhat``, ``_rhat_rank``, ``_ess``, ``_ess_bulk`` and
``_ess_tail`` as published.  arviz is not installed here, so this is parity *unpinned*: it restates the published functions
and is checked by the sampling-theory sanity tests of tests/test_mcmc_diag_host.py, not against arviz itself.

Where it departs from arviz, on purpose (psgla_b200.mcmc_diagnostics follows these definitions):
  - a series whose within-chain variance W is 0 gives NaN for every statistic built from it.  arviz returns S for an ESS
    series whose values are all equal (a max - min shortcut in ``_ess``) and 0 / 0 = NaN for R-hat;
  - a single chain (M = 1) is split into two and R-hat is computed from the halves, as the definitions state; arviz's
    ``rhat`` asks for two chains before it splits.

draws: array [N, M] (one element) or [N, M, E] -- N stored draws, M chains -- the layout of the library's sample buffer.
"""
import numpy as np
from scipy import fft, stats


def split_chains(x):
    """[N, M] -> [2M, N // 2]: first halves of every chain, then second halves; for odd N the middle draw is dropped."""
    x = np.asarray(x, dtype=np.float64).T  # [M, N], arviz's (chain, draw)
    half = x.shape[1] // 2
    return np.vstack((x[:, :half], x[:, -half:]))


def z_scale(x):
    """Average ranks over all draws, back-transformed with c = 3/8 (Blom) and mapped through the normal quantile."""
    r = stats.rankdata(x, method="average", axis=None).reshape(x.shape)
    return stats.norm.ppf((r - 3 / 8) / (x.size - 2 * 3 / 8 + 1))


def _moments(x):
    """Split-chain series [M', N'] -> (W, var+, n') or None when W == 0."""
    _, n = x.shape
    w = np.mean(np.var(x, axis=1, ddof=1))
    if not w > 0:
        return None
    b = n * np.var(np.mean(x, axis=1), ddof=1)
    return w, (n - 1) / n * w + b / n, n


def rhat_split(x):
    m = _moments(x)
    return np.nan if m is None else float(np.sqrt(m[1] / m[0]))


def autocov(x):
    """Per-chain autocovariance at every lag, divisor N' (arviz's ``_autocov``: zero-padded FFT)."""
    n = x.shape[1]
    m = fft.next_fast_len(2 * n)
    f = np.fft.rfft(x - x.mean(axis=1, keepdims=True), n=m, axis=1)
    return np.fft.irfft(f * np.conjugate(f), n=m, axis=1)[:, :n] / n


def ess_split(x, trace=None):
    """arviz's ``_ess`` on a split series [M', N'], Geyer's initial positive then monotone sequence.  ``trace``: a dict that
    receives ``min_pair`` = the smallest |rho_2k + rho_2k+1| the truncation rule tested (how close the cut-off was to
    flipping)."""
    mo = _moments(x)
    if mo is None:
        return np.nan
    mean_var, var_plus, n_draw = mo
    n_chain = x.shape[0]
    acov = autocov(x)
    rho = np.zeros(n_draw)
    rho_even = 1.0
    rho[0] = rho_even
    rho_odd = 1.0 - (mean_var - np.mean(acov[:, 1])) / var_plus
    rho[1] = rho_odd
    min_pair = abs(rho_even + rho_odd)
    t = 1
    while t < (n_draw - 3) and (rho_even + rho_odd) > 0.0:
        rho_even = 1.0 - (mean_var - np.mean(acov[:, t + 1])) / var_plus
        rho_odd = 1.0 - (mean_var - np.mean(acov[:, t + 2])) / var_plus
        min_pair = min(min_pair, abs(rho_even + rho_odd))
        if (rho_even + rho_odd) >= 0:
            rho[t + 1] = rho_even
            rho[t + 2] = rho_odd
        t += 2
    max_t = t - 2
    if rho_even > 0:
        rho[max_t + 1] = rho_even
    t = 1
    while t <= max_t - 2:
        if (rho[t + 1] + rho[t + 2]) > (rho[t - 1] + rho[t]):
            rho[t + 1] = (rho[t - 1] + rho[t]) / 2.0
            rho[t + 2] = rho[t + 1]
        t += 2
    s = n_chain * n_draw
    tau = -1.0 + 2.0 * np.sum(rho[: max_t + 1]) + np.sum(rho[max_t + 1: max_t + 2])
    tau = max(tau, 1 / np.log10(s))
    if trace is not None:
        trace["min_pair"] = min(trace.get("min_pair", np.inf), min_pair)
    return np.nan if np.isnan(rho).any() else s / tau


def diag_one(x, trace=None):
    """(rhat, ess_bulk, ess_tail) of one element's draws [N, M] (N >= 4)."""
    x = np.asarray(x, dtype=np.float64)
    if np.isnan(x).any():
        return np.nan, np.nan, np.nan
    sx = split_chains(x)
    z = z_scale(sx)
    folded = np.abs(x - np.median(x))  # median of all N M draws, the middle ones of odd N included
    rb, rt = rhat_split(z), rhat_split(z_scale(split_chains(folded)))
    rhat = np.nan if np.isnan(rb) or np.isnan(rt) else max(rb, rt)
    ess_bulk = ess_split(z, trace)
    q05, q95 = np.quantile(x, [0.05, 0.95])  # all N M draws, linear interpolation (numpy's default, R's type 7)
    lo = ess_split(split_chains((x <= q05).astype(np.float64)), trace)
    hi = ess_split(split_chains((x <= q95).astype(np.float64)), trace)
    return rhat, ess_bulk, (np.nan if np.isnan(lo) or np.isnan(hi) else min(lo, hi))


def diag(draws, traces=None):
    """draws [N, M, E] -> three float64 arrays [E]; ``traces``: a list that receives one trace dict per element."""
    d = np.asarray(draws, dtype=np.float64)
    out = np.empty((3, d.shape[2]))
    for e in range(d.shape[2]):
        tr = {} if traces is not None else None
        out[:, e] = diag_one(d[:, :, e], tr)
        if traces is not None:
            traces.append(tr)
    return out[0], out[1], out[2]
