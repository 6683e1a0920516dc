"""Convergence diagnostics on one GPU: the time of psgla_mcmc_diag (csrc/mcmc_diag.cu) at the sizes runs produce, and the
effective sample size per second of sampling that PSGLA and PnP-ULA reach on the same problem.  Prints one JSON document (and
writes it to --out when given).

    python scripts/diag_bench.py [--reps 3] [--out FILE]

Diagnostic timing, CUDA events around the C-ABI call (median of --reps after one warm-up call), per case:
  ms                  the call (z table + one CTA per element)
  hbm_fraction        N M E x 4 bytes (reading the draws once) over the measured copy bandwidth, divided by ms: the share of
                      the HBM bound.  The copy bandwidth is measured here: a 2 GiB device-to-device copy, read + write bytes
                      over its CUDA-event time (best of 5)
  stage_fraction      the kernel's own clock64 accounting, SM cycles summed over CTAs: load / sort (with median and
                      quantiles) / ranks and normal scores / chain moments and autocovariances (the lag loop)
Cases: 8 chains x 1 000 draws x 256 x 256 x 3 (synthetic AR(1) draws, rho = 0.5, and the PSGLA run's own draws below) and
64 chains x 256 draws x 480 x 320 x 3 (synthetic AR(1), rho = 0.5).

Samplers: DnCNN PSGLA (N = 10^4) and PnP-ULA (N = 10^5) with the sampler_params table, inpainting set3c/butterfly.png (50 %
observed, sigma = 1/255), 8 chains (philox noise), thinned to 1 000 stored draws per chain (n_inter = 10 resp. 100; the table's
own PnP-ULA thinning would store 10 000, above the diagnostic's limit).  Window means every 1 000 iterations (n_inter_mmse;
they are not measured and the table's 10 would hold 9 090 windows of PnP-ULA's 8 chains).  The DnCNN weights are the
library's seeded Lipschitz stand-in (lipschitz_dncnn_state_dict(0)), not the reference's checkpoint: the ESS figures
describe that network's chains.  Reported: sampling wall clock (host clock around the loop, ending in a synchronise), the
diagnostics after dropping the first 100 stored draws (10 %), and min / median bulk ESS per second of sampling.

The device-wide path for any S (psgla_mcmc_diag_large, csrc/mcmc_diag_large.cu), under "large":
  ms, stage_fraction  CUDA events around the call; the call's own GPU-timer split (workspace head): gather / sort (with median
                      and quantiles) / ranks, normal scores and indicators / chain moments / lag rounds; lag_rounds_run (rounds
                      with an unfinished element, summed over the three ESS series and the element groups) and launched
  sort_gb             bytes the radix sort moves: gather (4 read + 8 written), 4 passes x (4 histogram + 8 read + 8 written),
                      the in-place key conversion (8), per split draw
  series_gb           bytes the series passes move: 4 series x (ranks or indicators: 4 + 4 read, 4 written; moments: 4 + 4
                      read, 4 written) per split draw, plus 8 per split draw per lag round run (the series and its lagged
                      copy), counting every element of a group as unfinished (an upper bound)
  hbm_fraction        (sort_gb + series_gb) over the measured copy bandwidth, divided by ms
Cases: (a) one PSGLA and one PnP-ULA cell of BASELINE.json configs[1] (prior symetric_gaussians, y = (0, 0), the GMM_ALGS
constants of bench.py), 10^6 chains, fp32, Philox noise, 10^4 steps thinned by 10 (1 000 stored draws), the first 200 stored
draws (2 000 steps) dropped as burn-in: R-hat and bulk / tail ESS per coordinate, and ESS per second against the device time
of the same 10^4 steps on the throughput path (no trajectory) and of the trajectory-writing run; (b) image PnP-ULA with the
table's own thinning, n_inter = 10: 10^4 stored draws x 8 chains x 256 x 256 x 3 (a 63 GB sample buffer), S = 72 000 after
dropping 1 000 stored draws; (c) the synthetic 8 chains x 1 000 draws x 256 x 256 x 3 case through both paths.

    python scripts/diag_bench.py --large-only   # cases (a) - (c) only"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import psgla_b200 as P  # noqa: E402

BURN_IN = 100


def power_limit():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader,nounits", "-i", "0"],
                             capture_output=True, text=True, timeout=30)
        return float(out.stdout.strip().splitlines()[0])
    except Exception:  # noqa: BLE001 -- the power limit is reported when the query tool is present
        return None


def copy_bandwidth_gbs(dev):
    a = torch.empty(1 << 29, dtype=torch.float32, device=dev)  # 2 GiB
    b = torch.empty_like(a)
    b.copy_(a)
    best = float("inf")
    for _ in range(5):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        b.copy_(a)
        e1.record()
        e1.synchronize()
        best = min(best, e0.elapsed_time(e1))
    return 2 * a.numel() * 4 / (best * 1e-3) / 1e9


def ar1(N, M, E, rho, dev, seed):
    g = torch.Generator(device=dev).manual_seed(seed)
    x = torch.empty((N, M, E), dtype=torch.float32, device=dev)
    x[0] = torch.randn((M, E), generator=g, device=dev) / (1 - rho * rho) ** 0.5
    for n in range(1, N):
        torch.add(x[n - 1].mul(rho), torch.randn((M, E), generator=g, device=dev), out=x[n])
    return x


def time_diag(x, reps, copy_gbs):
    """x: CUDA fp32 [N, M, E] (contiguous).  The raw C-ABI call, timed with CUDA events."""
    N, M, E = x.shape
    lib = P._lib.lib()
    ws_bytes = lib.psgla_mcmc_diag_workspace_bytes(N, M)
    ws = torch.empty(ws_bytes, dtype=torch.uint8, device=x.device)
    out = torch.empty((3, E), dtype=torch.float32, device=x.device)
    st = P._lib.stream_ptr(x.device)

    def call():
        P._lib.check(lib.psgla_mcmc_diag(x.data_ptr(), N, M, E, ws.data_ptr(), C.c_size_t(ws_bytes), out[0].data_ptr(),
                                         out[1].data_ptr(), out[2].data_ptr(), st), "psgla_mcmc_diag")

    call()
    ms = []
    for _ in range(reps):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        call()
        e1.record()
        e1.synchronize()
        ms.append(e0.elapsed_time(e1))
    cycles = ws[:32].cpu().view(torch.int64).double()
    frac = (cycles / cycles.sum()).tolist()
    t = sorted(ms)[len(ms) // 2]
    bytes_read = N * M * E * 4
    return dict(n_draws=N, n_chains=M, n_elem=E, S=2 * M * (N // 2), ms=t, ms_all=ms, gb_read=bytes_read / 1e9,
                hbm_fraction=bytes_read / (copy_gbs * 1e9) / (t * 1e-3),
                stage_fraction=dict(load=frac[0], sort=frac[1], rank=frac[2], moments_autocov=frac[3]),
                rhat_max=float(out[0][~out[0].isnan()].max()), ess_bulk_median=float(out[1][~out[1].isnan()].median()))


def time_diag_large(x, reps, copy_gbs):
    """x: CUDA fp32 [N, M, E] (contiguous).  psgla_mcmc_diag_large, timed with CUDA events."""
    N, M, E = x.shape
    lib = P._lib.lib()
    ws_bytes = lib.psgla_mcmc_diag_large_workspace_bytes(N, M, E)
    ws = torch.empty(ws_bytes, dtype=torch.uint8, device=x.device)
    out = torch.empty((3, E), dtype=torch.float32, device=x.device)
    st = P._lib.stream_ptr(x.device)

    def call():
        P._lib.check(lib.psgla_mcmc_diag_large(x.data_ptr(), N, M, E, ws.data_ptr(), C.c_size_t(ws_bytes), out[0].data_ptr(),
                                               out[1].data_ptr(), out[2].data_ptr(), st), "psgla_mcmc_diag_large")

    call()
    ms = []
    for _ in range(reps):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        call()
        e1.record()
        e1.synchronize()
        ms.append(e0.elapsed_time(e1))
    head = ws[:64].cpu().view(torch.int64).tolist()
    stage = head[:5]
    t = sorted(ms)[len(ms) // 2]
    S = 2 * M * (N // 2)
    groups = -(-E // max(1, min(E, max(1, (1 << 28) // S), 65535)))
    draws = S * E
    sort_b = draws * (12 + 4 * 20 + 8)
    series_b = draws * 4 * 24 + head[5] * 8 * draws / groups
    r, b, tl = out[0], out[1], out[2]
    fin = lambda v: v[~v.isnan()]  # noqa: E731
    return dict(n_draws=N, n_chains=M, n_elem=E, S=S, workspace_gb=ws_bytes / 1e9, ms=t, ms_all=ms,
                sort_gb=sort_b / 1e9, series_gb=series_b / 1e9,
                hbm_fraction=(sort_b + series_b) / (copy_gbs * 1e9) / (t * 1e-3),
                stage_fraction=dict(zip(("gather", "sort", "rank", "moments", "lag_rounds"), (v / sum(stage) for v in stage))),
                lag_rounds_run=head[5], lag_rounds_launched=head[6],
                rhat_max=float(fin(r).max()) if fin(r).numel() else None,
                ess_bulk_median=float(fin(b).median()) if fin(b).numel() else None,
                ess_tail_min=float(fin(tl).min()) if fin(tl).numel() else None), out


def gmm_cell(alg, dev, reps, copy_gbs, n_chains=10 ** 6, n_steps=10 ** 4, thin=10, burn=200):
    """Case (a): one cell of configs[1] as bench.py sets it up; trajectory diagnosed with psgla_mcmc_diag_large."""
    import numpy as np
    prm = dict(psgla=dict(delta=0.3, alpha=2.0 / 3.0, epsilon=1.0), pnp_ula=dict(delta=0.1, alpha=1.5, epsilon=0.5))[alg]
    mu, Sig, pi = P.gaussian_mixt_example("symetric_gaussians")
    y = (0.0, 0.0)
    x0 = torch.tensor(y, dtype=torch.float32, device=dev).repeat(n_chains, 1).contiguous()
    ch = P.GMMChains(alg, np.array(y), prm["delta"], np.eye(2), 1.0, P.Theorical_MMSE(mu, Sig, pi), prm["alpha"],
                     prm["epsilon"], n_chains=n_chains, x0=x0, seed=0, dtype="float32", device=dev)

    def timed(thin_):
        ch.state.copy_(x0)
        ch.step = 0
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        tr = ch.run(n_steps, thin=thin_)
        e1.record()
        e1.synchronize()
        return e0.elapsed_time(e1) * 1e-3, tr

    timed(0)  # warm-up
    s_plain = min(timed(0)[0] for _ in range(3))
    s_traj, traj = timed(thin)
    timing, out = time_diag_large(traj[burn:].contiguous(), reps, copy_gbs)
    ess_b, ess_t = out[1].tolist(), out[2].tolist()
    return dict(case="(a) 2D %s cell, %d chains x %d steps, thin %d, burn-in %d stored draws" % (alg, n_chains, n_steps, thin, burn),
                alg=alg, steps_s_throughput_path=s_plain, steps_s_trajectory_run=s_traj, rhat=out[0].tolist(), ess_bulk=ess_b,
                ess_tail=ess_t, ess_bulk_per_s_throughput=[v / s_plain for v in ess_b],
                ess_bulk_per_s_trajectory=[v / s_traj for v in ess_b], ess_tail_per_s_throughput=[v / s_plain for v in ess_t],
                **timing)


def pnpula_table_thinning(dev, reps, copy_gbs):
    """Case (b): image PnP-ULA with the table's n_inter = 10 (10^4 stored draws x 8 chains)."""
    im = P.load_image(os.path.join(ROOT, "tests", "golden", "set3c", "butterfly.png"), device=dev)
    dg, init, _, _ = P.make_inpainting(im, prop=0.5, sigma=1.0, seed_ip=0)
    den = P.DnCNN(pretrained=P.lipschitz_dncnn_state_dict(0), device=dev)
    prm = P.sampler_params("pnp_ula", den="DnCNN")
    run = P.pnpula_run(init, dg, P.PriorGrad(den, prm["alpha"], prm["s1"], prm["s2"]),
                       **dict(P.as_pnpula_kwargs(prm, seed=0), n_inter=10, n_inter_mmse=1000), n_chains=8)
    run.step(0)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for i in range(1, run.n_iter):
        run.step(i)
    torch.cuda.synchronize()
    wall = (time.perf_counter() - t0) * run.n_iter / (run.n_iter - 1)
    run.finish()
    n = len(run.Xlist)
    burn = n // 10
    s = run.samples[burn:n]
    timing, _ = time_diag_large(s.reshape(s.shape[0], s.shape[1], -1), reps, copy_gbs)
    d = P.mcmc_diagnostics_large(run, burn_in=burn)
    del run, s
    return dict(case="(b) image PnP-ULA, n_inter = 10: %d stored draws x 8 chains x 256x256x3, burn-in %d" % (n, burn),
                n_iter=prm["N"], sampling_s=wall,
                **{k: d[k] for k in ("rhat_max", "frac_rhat_above_1_01", "ess_bulk_min", "ess_bulk_median", "ess_tail_min")},
                ess_bulk_min_per_s=d["ess_bulk_min"] / wall, ess_bulk_median_per_s=d["ess_bulk_median"] / wall,
                timing=timing)


def run_sampler(alg, dev):
    im = P.load_image(os.path.join(ROOT, "tests", "golden", "set3c", "butterfly.png"), device=dev)
    dg, init, _, _ = P.make_inpainting(im, prop=0.5, sigma=1.0, seed_ip=0)
    den = P.DnCNN(pretrained=P.lipschitz_dncnn_state_dict(0), device=dev)
    prm = P.sampler_params(alg, den="DnCNN")
    n_inter = prm["N"] // 1000
    if alg == "psgla":
        run = P.psgla_run(init, dg, den, **dict(P.as_psgla_kwargs(prm, seed=0), n_inter=n_inter, n_inter_mmse=1000),
                          n_chains=8)
    else:
        run = P.pnpula_run(init, dg, P.PriorGrad(den, prm["alpha"], prm["s1"], prm["s2"]),
                           **dict(P.as_pnpula_kwargs(prm, seed=0), n_inter=n_inter, n_inter_mmse=1000), n_chains=8)
    run.step(0)  # first launches load the modules
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for i in range(1, run.n_iter):
        run.step(i)
    torch.cuda.synchronize()
    wall = (time.perf_counter() - t0) * run.n_iter / (run.n_iter - 1)
    run.finish()
    d = P.mcmc_diagnostics(run, burn_in=BURN_IN)
    res = dict(alg=alg, n_iter=run.n_iter, n_inter=n_inter, n_chains=8, stored_draws=len(run.Xlist), burn_in=BURN_IN,
               sampling_s=wall,
               **{k: d[k] for k in ("rhat_max", "frac_rhat_above_1_01", "ess_bulk_min", "ess_bulk_median", "ess_tail_min")})
    res["ess_bulk_min_per_s"] = d["ess_bulk_min"] / wall
    res["ess_bulk_median_per_s"] = d["ess_bulk_median"] / wall
    return res, run


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--out", default=None)
    ap.add_argument("--large-only", action="store_true", help="cases (a) - (c) of the large-S path only")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("diag_bench.py needs a CUDA device")
    dev = torch.device("cuda:0")
    torch.cuda.set_device(dev)
    copy_gbs = copy_bandwidth_gbs(dev)
    res = dict(kind="mcmc_diag", device=torch.cuda.get_device_name(dev), power_limit_w=power_limit(),
               copy_bandwidth_gbs=copy_gbs, weights="lipschitz_dncnn_state_dict(0) (seeded stand-in, not the reference's "
               "checkpoint)", diag=[], samplers=[], large=[])
    x = ar1(1000, 8, 256 * 256 * 3, 0.5, dev, 0)
    case = "(c) 8 chains x 1000 draws x 256x256x3, synthetic AR(1) rho 0.5"
    small = time_diag(x, args.reps, copy_gbs)
    large, out = time_diag_large(x, args.reps, copy_gbs)
    ref = P.mcmc_diagnostics(x)
    large["max_abs_diff_vs_small_path"] = {k: float((out[i] - ref[k]).abs().nan_to_num(0).max())
                                           for i, k in enumerate(("rhat", "ess_bulk", "ess_tail"))}
    res["large"].append(dict(case=case, small_path=small, **large))
    print(json.dumps(res["large"][-1]), flush=True)
    del x, out, ref
    torch.cuda.empty_cache()
    for alg in ("psgla", "pnp_ula"):
        res["large"].append(gmm_cell(alg, dev, args.reps, copy_gbs))
        print(json.dumps(res["large"][-1]), flush=True)
        torch.cuda.empty_cache()
    res["large"].append(pnpula_table_thinning(dev, args.reps, copy_gbs))
    print(json.dumps(res["large"][-1]), flush=True)
    torch.cuda.empty_cache()
    if args.large_only:
        return finish(res, args)
    x = ar1(1000, 8, 256 * 256 * 3, 0.5, dev, 0)
    res["diag"].append(dict(case="8 chains x 1000 draws x 256x256x3, synthetic AR(1) rho 0.5", **time_diag(x, args.reps, copy_gbs)))
    del x
    x = ar1(256, 64, 480 * 320 * 3, 0.5, dev, 1)
    res["diag"].append(dict(case="64 chains x 256 draws x 480x320x3, synthetic AR(1) rho 0.5", **time_diag(x, args.reps, copy_gbs)))
    del x
    torch.cuda.empty_cache()
    for alg in ("psgla", "pnp_ula"):
        r, run = run_sampler(alg, dev)
        res["samplers"].append(r)
        print(json.dumps(r), flush=True)
        s = run.samples[:len(run.Xlist)]
        res["diag"].append(dict(case="8 chains x 1000 draws x 256x256x3, the %s run's own draws" % alg,
                                **time_diag(s.reshape(s.shape[0], s.shape[1], -1), args.reps, copy_gbs)))
        del run, s
        torch.cuda.empty_cache()
    finish(res, args)


def finish(res, args):
    line = json.dumps(res, indent=1)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as fh:
            fh.write(line + "\n")


if __name__ == "__main__":
    main()
