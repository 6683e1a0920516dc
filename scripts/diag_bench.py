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
diagnostics after dropping the first 100 stored draws (10 %), and min / median bulk ESS per second of sampling."""
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
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("diag_bench.py needs a CUDA device")
    dev = torch.device("cuda:0")
    torch.cuda.set_device(dev)
    copy_gbs = copy_bandwidth_gbs(dev)
    res = dict(kind="mcmc_diag", device=torch.cuda.get_device_name(dev), power_limit_w=power_limit(),
               copy_bandwidth_gbs=copy_gbs, weights="lipschitz_dncnn_state_dict(0) (seeded stand-in, not the reference's "
               "checkpoint)", diag=[], samplers=[])
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
    line = json.dumps(res, indent=1)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as fh:
            fh.write(line + "\n")


if __name__ == "__main__":
    main()
