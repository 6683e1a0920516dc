"""Posterior summary on one GPU: the time of psgla_mcmc_summary (csrc/mcmc_summary.cu) at the sizes runs produce, beside
psgla_mcmc_diag_large on the same draws, and the calibration of one real prior's credible intervals.  Prints one JSON
document (and writes it to --out, default profiles/summary_bench.json).

    python scripts/summary_bench.py [--reps 3] [--out FILE]

Per case, CUDA events around the C-ABI call (median of --reps after one warm-up call), probs (0.05, 0.5, 0.95), hdi_prob 0.94:
  ms, stage_fraction  the call, and its own GPU-timer split (workspace head): gather / sort (with the odd-N merge and the
                      quantiles) / series building / chain and element moments (with mean and sd) / lag rounds / HDI scan /
                      Beta quantiles and outputs / merge of odd N; stage_ms the same in ms (the last timed call);
                      lag_rounds_run / launched over the 1 + P series
  beta_evals, cf_terms, cf_terms_max_pair   the Beta quantiles of _mcse_quantile, counted by the kernel: incomplete-beta
                      evaluations (Newton steps) and continued-fraction terms in all, and the most terms one (element, p)
                      pair ran (the finishing stage's critical path); finish_ns_per_term = the finish stage over that
                      maximum, an upper bound on the time of one dependent term
  sort_gb             bytes the radix sort moves per split draw, as diag_bench.py counts them (gather 12, 4 passes x 20, key
                      conversion 8), plus 8 for the merge of odd N
  series_gb           (1 + P) series x 24 B per split draw (build: 4 + 4 read, 4 written; moments: 4 + 4 read, 4 written), plus
                      8 B per split draw per lag round run (an upper bound: every element of a group counted unfinished)
  hdi_gb              8 B per draw (both window ends read)
  hbm_fraction        (sort_gb + series_gb + hdi_gb) over the copy bandwidth measured in the same run, divided by ms
  diag_large          psgla_mcmc_diag_large on the same draws (diag_bench.py's timing)
Cases: (a) synthetic AR(1) draws (rho 0.5), 8 chains x 1 000 draws x 256 x 256 x 3; (b) a PSGLA cell of BASELINE.json
configs[1] as diag_bench.py sets it up (symetric_gaussians, y = (0, 0)), 10^6 chains, 10^4 steps thinned by 10, the first 200
stored draws dropped: 800 draws x 10^6 chains x 2; (c) PSGLA-TV inpainting of set3c/butterfly.png (50 % observed,
sigma = 1/255) with tv_bench.py's lambda = 100 and s = 10/255, 8 chains (philox), 2 000 iterations stored every 2nd
(store="all"), the first 100 stored draws dropped; coverage_hdi and frac_truth_below against the clean image.  These
describe the TV prior at that lambda and s, not the reference's trained networks; (d) case (a) with an odd N = 1 001, so the
middle draws are merged into the sorted union: the merge's share of the call."""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "scripts"))

import psgla_b200 as P  # noqa: E402
from diag_bench import ar1, copy_bandwidth_gbs, time_diag_large  # noqa: E402

PROBS = (0.05, 0.5, 0.95)
HDI_PROB = 0.94
STAGES = (("gather", 0), ("sort", 1), ("series", 2), ("moments", 3), ("lag_rounds", 4), ("hdi", 9), ("finish", 10), ("merge", 11))


def card():
    res = dict(device=torch.cuda.get_device_name(0), power_limit_w=None, sm_clock_mhz=None, sm_clock_max_mhz=None)
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.sm,clocks.max.sm", "--format=csv,noheader,nounits",
                              "-i", "0"], capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
        p, c, cm = (float(v) for v in out.split(","))
        res.update(power_limit_w=p, sm_clock_mhz=c, sm_clock_max_mhz=cm)
    except Exception:  # noqa: BLE001 -- the card's settings are reported when the query tool is present
        pass
    return res


def time_summary(x, reps, copy_gbs):
    """x: CUDA fp32 [N, M, E] (contiguous).  psgla_mcmc_summary, timed with CUDA events."""
    N, M, E = x.shape
    Pn = len(PROBS)
    lib = P._lib.lib()
    ws_bytes = lib.psgla_mcmc_summary_workspace_bytes(N, M, E, Pn)
    ws = torch.empty(ws_bytes, dtype=torch.uint8, device=x.device)
    out = torch.empty((6 + 3 * Pn, E), dtype=torch.float32, device=x.device)  # mean, sd, mcse, ess, hdi lo / hi; [3][P]
    st = P._lib.stream_ptr(x.device)
    probs = (C.c_double * Pn)(*PROBS)

    def call():
        P._lib.check(lib.psgla_mcmc_summary(x.data_ptr(), N, M, E, probs, Pn, HDI_PROB, ws.data_ptr(), C.c_size_t(ws_bytes),
                                            *[out[i].data_ptr() for i in (0, 1, 2, 3, 6, 6 + Pn, 6 + 2 * Pn, 4, 5)], st),
                     "psgla_mcmc_summary")

    call()
    ms = []
    for _ in range(reps):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        call()
        e1.record()
        e1.synchronize()
        ms.append(e0.elapsed_time(e1))
    head = ws[:128].cpu().view(torch.int64).tolist()
    stage_ns = {k: head[i] for k, i in STAGES}
    total_ns = sum(stage_ns.values())
    t = sorted(ms)[len(ms) // 2]
    S, K = 2 * M * (N // 2), N * M
    groups = -(-E // max(1, min(E, max(1, (1 << 28) // S), 65535)))
    sort_b = S * E * (12 + 4 * 20 + 8) + (K * E * 8 if N % 2 else 0)
    series_b = S * E * (1 + Pn) * 24 + head[5] * 8 * S * E / groups
    hdi_b = K * E * 8
    fin = lambda v: v[~v.isnan()]  # noqa: E731
    return dict(n_draws=N, n_chains=M, n_elem=E, S=S, workspace_gb=ws_bytes / 1e9, ms=t, ms_all=ms,
                stage_fraction={k: v / total_ns for k, v in stage_ns.items()},
                stage_ms={k: v * 1e-6 for k, v in stage_ns.items()},  # the last call's: each call resets the head
                lag_rounds_run=head[5], lag_rounds_launched=head[6],
                beta_evals=head[12], cf_terms=head[13], cf_terms_max_pair=head[14],
                finish_ns_per_term=head[10] / head[14] if head[14] else None,
                sort_gb=sort_b / 1e9, series_gb=series_b / 1e9, hdi_gb=hdi_b / 1e9,
                hbm_fraction=(sort_b + series_b + hdi_b) / (copy_gbs * 1e9) / (t * 1e-3),
                ess_mean_median=float(fin(out[3]).median()) if fin(out[3]).numel() else None,
                ess_quantiles_min=[float(fin(out[12 + j]).min()) if fin(out[12 + j]).numel() else None for j in range(Pn)],
                mcse_mean_max=float(fin(out[2]).max()) if fin(out[2]).numel() else None)


def both(case, x, reps, copy_gbs, **extra):
    s = time_summary(x, reps, copy_gbs)
    d, _ = time_diag_large(x, reps, copy_gbs)
    res = dict(case=case, summary=s, diag_large=dict(ms=d["ms"], ms_all=d["ms_all"], stage_fraction=d["stage_fraction"]),
               **extra)
    print(json.dumps(res), flush=True)
    return res


def gmm_cell(dev, n_chains=10 ** 6, n_steps=10 ** 4, thin=10, burn=200):
    mu, Sig, pi = P.gaussian_mixt_example("symetric_gaussians")
    y = (0.0, 0.0)
    x0 = torch.tensor(y, dtype=torch.float32, device=dev).repeat(n_chains, 1).contiguous()
    ch = P.GMMChains("psgla", np.array(y), 0.3, np.eye(2), 1.0, P.Theorical_MMSE(mu, Sig, pi), 2.0 / 3.0, 1.0,
                     n_chains=n_chains, x0=x0, seed=0, dtype="float32", device=dev)
    return ch.run(n_steps, thin=thin)[burn:].contiguous()


def tv_run(dev, n_iter=2000, n_inter=2, burn=100):
    im = P.load_image(os.path.join(ROOT, "tests", "golden", "set3c", "butterfly.png"), device=dev)
    dg, init, _, _ = P.make_inpainting(im, prop=0.5, sigma=1.0, seed_ip=0)
    s = 10.0 / 255.0
    run = P.psgla_run(init, dg, P.TVDenoiser(), alpha=1.0, lambd=100.0, sig_float=s, delta=s * s, n_iter=n_iter,
                      n_inter=n_inter, n_inter_mmse=n_iter, seed=0, n_chains=8, rng="philox", store="all")
    for i in range(n_iter):
        run.step(i)
    run.finish()
    summ = P.mcmc_summary(run, burn_in=burn, probs=PROBS, hdi_prob=HDI_PROB, truth=im[0])
    diag = P.mcmc_diagnostics_large(run, burn_in=burn)
    n = len(run.Xlist)
    x = run.samples[burn:n]
    x = x.reshape(x.shape[0], x.shape[1], -1)
    calib = dict(stored_draws=n, burn_in=burn, coverage_hdi=summ["coverage_hdi"], frac_truth_below=summ["frac_truth_below"],
                 mcse_mean_max=summ["mcse_mean_max"], mcse_quantiles_max=summ["mcse_quantiles_max"],
                 mcse_mean_median=float(summ["mcse_mean"].nanmedian()), sd_median=float(summ["sd"].nanmedian()),
                 rhat_max=diag["rhat_max"], ess_bulk_median=diag["ess_bulk_median"])
    return run, x, calib


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "summary_bench.json"))
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("summary_bench.py needs a CUDA device")
    dev = torch.device("cuda:0")
    torch.cuda.set_device(dev)
    copy_gbs = copy_bandwidth_gbs(dev)
    res = dict(kind="mcmc_summary", **card(), copy_bandwidth_gbs=copy_gbs, probs=PROBS, hdi_prob=HDI_PROB, cases=[])
    x = ar1(1000, 8, 256 * 256 * 3, 0.5, dev, 0)
    res["cases"].append(both("(a) 8 chains x 1000 draws x 256x256x3, synthetic AR(1) rho 0.5", x, args.reps, copy_gbs))
    del x
    torch.cuda.empty_cache()
    x = gmm_cell(dev)
    res["cases"].append(both("(b) 2D PSGLA cell of configs[1], 10^6 chains x 10^4 steps thin 10, burn-in 200 stored draws",
                             x, args.reps, copy_gbs))
    del x
    torch.cuda.empty_cache()
    x = ar1(1001, 8, 256 * 256 * 3, 0.5, dev, 0)
    res["cases"].append(both("(d) 8 chains x 1001 draws x 256x256x3, synthetic AR(1) rho 0.5 (odd N: merged union)", x,
                             args.reps, copy_gbs))
    del x
    torch.cuda.empty_cache()
    run, x, calib = tv_run(dev)
    res["cases"].append(both("(c) PSGLA-TV inpainting of butterfly.png (lambda 100, s 10/255), 8 chains, 2000 iterations "
                             "stored every 2nd, burn-in 100 stored draws; the TV prior, not the reference's networks",
                             x, args.reps, copy_gbs, calibration=calib))
    del run, x
    torch.cuda.empty_cache()
    res.update(card_after=card())
    line = json.dumps(res, indent=1)
    print(line)
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as fh:
        fh.write(line + "\n")


if __name__ == "__main__":
    main()
