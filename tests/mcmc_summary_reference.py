"""float64 numpy / scipy restatement of the posterior summary of psgla_b200.mcmc_summary, following arviz's ``_ess_mean``,
``_mcse_mean``, ``_ess_quantile``, ``_mcse_quantile`` and ``_hdi`` as published.  Parity *unpinned*, as tests/mcmc_reference.py
is: arviz is not installed here; tests/test_mcmc_summary_host.py checks this restatement against sampling theory.

The details of ``_mcse_quantile`` are recalled, not checked against arviz's source: the Beta(ess p + 1, ess (1 - p) + 1)
quantiles at 0.1586553 / 0.8413447 (the normal's +-1 sd), the indices rint(max(lo K - 1, 0)) and rint(min(hi K - 1, K - 1))
rounded half to even (np.rint) into the sorted draws, and half the distance between the two draws.  The upper index has no
lower clamp: when hi K - 1 < -0.5 (a tiny p at an ESS above about 3.7 K, reachable since Geyer's ESS goes up to S log10 S)
it is -1, which numpy reads as the largest draw; the device mirrors that.

``hdi`` follows np.argmin over the widths: with infinite draws a width can be +inf, or NaN where both ends are the same
infinity, and argmin returns the first NaN if there is one, else the first smallest width.

Deviation from arviz, on purpose and shared with tests/mcmc_reference.py: a series whose within-chain variance W is 0 gives
NaN for its ESS and for the MCSE built from it (arviz returns S for the ESS).  NaN draws give NaN for every output.

draws: array [N, M] (one element) or [N, M, E] -- N draws, M chains -- the layout of the library's sample buffer.
"""
import numpy as np
from scipy import stats

from mcmc_reference import ess_split, split_chains

BETA_P = (0.1586553, 0.8413447)
KEYS = ("mean", "sd", "mcse_mean", "ess_mean", "hdi_low", "hdi_high")
PKEYS = ("quantiles", "mcse_quantiles", "ess_quantiles")


def hdi(a, hdi_prob):
    """_hdi on sorted a: (low, high, index) of the narrowest window of floor(hdi_prob K) + 1 draws; np.argmin takes the first
    of equal widths."""
    k = int(np.floor(hdi_prob * a.size))
    width = np.subtract(a[k:], a[:a.size - k], dtype=np.float64)
    i = int(np.argmin(width))
    return a[i], a[i + k], i


def mcse_quantile_index(ess, p, K):
    """The unrounded positions ppf K - 1 of _mcse_quantile (before the clamps and np.rint)."""
    lo, hi = stats.beta.ppf(BETA_P, ess * p + 1, ess * (1 - p) + 1)
    return lo * K - 1, hi * K - 1


def summary_one(x, probs, hdi_prob, ppf_pos=None, trace=None):
    """dict of the outputs for one element's draws [N, M]; ``ppf_pos``: a list that receives, per p, the two unrounded
    positions of mcse_quantile_index (NaN when the ESS is); ``trace``: a dict that receives the smallest Geyer pair sum of
    its ESS series (tests/mcmc_reference.py's ``min_pair``)."""
    x = np.asarray(x, dtype=np.float64)
    P = len(probs)
    nan = {k: np.nan for k in KEYS}
    nan.update({k: np.full(P, np.nan) for k in PKEYS})
    if np.isnan(x).any():
        if ppf_pos is not None:
            ppf_pos.extend([(np.nan, np.nan)] * P)
        return nan
    a = np.sort(x.ravel())
    K = a.size
    mean = np.mean(a)
    sd = np.sqrt(np.sum((a - mean) ** 2) / (K - 1))
    ess_mean = ess_split(split_chains(x), trace)
    lo, hi, _ = hdi(a, hdi_prob)
    out = {"mean": mean, "sd": sd, "ess_mean": ess_mean, "mcse_mean": sd / np.sqrt(ess_mean), "hdi_low": lo, "hdi_high": hi,
           "quantiles": np.empty(P), "mcse_quantiles": np.empty(P), "ess_quantiles": np.empty(P)}
    for j, p in enumerate(probs):
        q = np.quantile(a, p)
        e = ess_split(split_chains((x <= q).astype(np.float64)), trace)
        out["quantiles"][j], out["ess_quantiles"][j] = q, e
        if np.isnan(e):
            out["mcse_quantiles"][j] = np.nan
            if ppf_pos is not None:
                ppf_pos.append((np.nan, np.nan))
            continue
        s1, s2 = mcse_quantile_index(e, p, K)
        if ppf_pos is not None:
            ppf_pos.append((s1, s2))
        i1, i2 = int(np.rint(max(s1, 0))), int(np.rint(min(s2, K - 1)))
        out["mcse_quantiles"][j] = (a[i2] - a[i1]) / 2
    return out


def summary(draws, probs=(0.05, 0.5, 0.95), hdi_prob=0.94, ppf_pos=None, traces=None):
    """draws [N, M, E] -> dict of float64 arrays: [E] for KEYS, [P, E] for PKEYS.  ``ppf_pos``, ``traces``: lists that
    receive per element its list of per-p position pairs and its trace dict."""
    d = np.asarray(draws, dtype=np.float64)
    E, P = d.shape[2], len(probs)
    res = {k: np.empty(E) for k in KEYS}
    res.update({k: np.empty((P, E)) for k in PKEYS})
    for e in range(E):
        pos = [] if ppf_pos is not None else None
        tr = {} if traces is not None else None
        o = summary_one(d[:, :, e], probs, hdi_prob, pos, tr)
        if traces is not None:
            traces.append(tr)
        for k in KEYS:
            res[k][e] = o[k]
        for k in PKEYS:
            res[k][:, e] = o[k]
        if ppf_pos is not None:
            ppf_pos.append(pos)
    return res
