"""PSGLA-TV throughput on one GPU: the TV prox (csrc/tv_prox.cu) inside the PSGLA inpainting loop, and the reference's eager loop
shape for comparison.  Prints one JSON line (and writes it to --out when given).

    python scripts/tv_bench.py [--steps 20] [--warmup 5] [--eager-steps 3] [--out FILE]

Problem: inpainting (50 % of the pixels observed, sigma = 1/255) of butterfly.png (256 x 256) or castle.png (321 x 481), the
table's TV step s = 10/255 with alpha = 1 and lambda = 100, i.e. a data-step gain (delta / lambda) / sigma^2 = 1: the table's
lambda = 10 (gain 10) diverges with this prox.  B chains per image (philox noise, statistics-only storage), warm-started prox
as in the reference.  Per configuration:
  psgla_it_per_s          PSGLA iterations per second (each: one "pre" launch + one prox launch), all chains
  cp_iters_mean           CP iterations per prox call and chain;  cp_iters_max_mean: the slowest chain's, per call (the
                          kernel runs until every chain has stopped, plus one iteration)
  prox_us, us_per_cp_iter prox call time (CUDA events around the launch) and that over (cp_iters_max_mean + 1) barriers
  hbm_*                   the algorithmic 28 B per element and CP iteration (read y, x2, u2; write x2, u2) over prox time,
                          against the data-sheet 7.7 TB/s; working_set_mb = 28 B per element (y, state, ping-pong copy) and
                          whether it fits the 126 MB L2
eager: the restated deepinv loop (tests/tv_reference.py's algorithm with deepinv's whole-batch stopping test: one host
synchronisation per CP iteration) inside the reference's PSGLA step, B = 1, timed over a few iterations on the same GPU."""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

import psgla_b200 as P  # noqa: E402
import tv_reference as TV  # noqa: E402

S = 10.0 / 255.0
LAMBD = 100.0
CONFIGS = [(1, "set3c/butterfly.png"), (8, "set3c/butterfly.png"), (32, "set3c/butterfly.png"), (1, "set1c/castle.png"),
           (8, "set1c/castle.png")]
HBM_TBPS = 7.7
L2_MB = 126


def card():
    name = torch.cuda.get_device_name(0)
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader,nounits", "-i", "0"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
        power = float(out.splitlines()[0])
    except Exception:  # noqa: BLE001 -- the power limit is reported when the query tool is present
        power = None
    return name, power


def problem(path):
    im = P.load_image(os.path.join(ROOT, "tests", "golden", path), device="cuda")
    dg, init, y, _ = P.make_inpainting(im, prop=0.5, sigma=1.0, seed_ip=0)
    return im, dg, init


def bench_cuda(B, path, steps, warmup):
    im, dg, init = problem(path)
    den = P.TVDenoiser()
    n_iter = warmup + steps
    run = P.psgla_run(init, dg, den, alpha=1.0, lambd=LAMBD, sig_float=S, delta=S * S, n_iter=n_iter, n_inter=n_iter,
                      n_inter_mmse=n_iter, seed=0, n_chains=B, rng="philox", store="stats")
    cp = torch.zeros((steps, B), dtype=torch.int32, device="cuda")
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
    for i in range(warmup):
        run.step(i)
    t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    t0.record()
    for j in range(steps):  # run.step(i) for the TV prox: the pre launch, then the prox launch with the post
        i = warmup + j
        run.pre(i, run.pre_params)
        ev[j][0].record()
        run.post(i, run.gain)
        ev[j][1].record()
        cp[j].copy_(den.last_iterations)
    t1.record()
    torch.cuda.synchronize()
    total_ms = t0.elapsed_time(t1)
    prox_ms = sum(a.elapsed_time(b) for a, b in ev)
    cpf = cp.double()
    n_el = B * 3 * im.shape[2] * im.shape[3]
    cp_sum = float(cpf.sum())  # chain-iterations
    bytes_alg = 28.0 * cp_sum * 3 * im.shape[2] * im.shape[3]
    max_mean = float(cpf.max(1).values.mean())
    ws_mb = 28.0 * n_el / 1e6
    assert torch.isfinite(run.X).all()
    return dict(B=B, H=int(im.shape[2]), W=int(im.shape[3]), lambd=LAMBD, s=S, alpha=1.0, steps=steps, warmup=warmup,
                psgla_it_per_s=steps / (total_ms / 1e3), psgla_iter_ms=total_ms / steps,
                cp_iters_mean=cp_sum / (steps * B), cp_iters_max_mean=max_mean,
                prox_us=prox_ms * 1e3 / steps, us_per_cp_iter=prox_ms * 1e3 / steps / (max_mean + 1),
                hbm_bytes_per_call=bytes_alg / steps, hbm_tb_per_s=bytes_alg / (prox_ms / 1e3) / 1e12,
                hbm_fraction_of_datasheet=bytes_alg / (prox_ms / 1e3) / 1e12 / HBM_TBPS,
                working_set_mb=ws_mb, fits_l2=ws_mb < L2_MB)


def eager_tv(y, ths, state, tau=0.01, rho=1.99, n_it_max=1000, crit=1e-5):
    """deepinv's TVDenoiser.forward loop shape: whole-batch norms, a host synchronisation per CP iteration (the `if`)."""
    sigma = 1 / tau / 8
    if state.get("x2") is None or state["x2"].shape != y.shape:
        state["x2"], state["u2"] = y.clone(), torch.zeros(tuple(y.shape) + (2,), device=y.device)
    x2, u2 = state["x2"], state["u2"]
    for k in range(n_it_max):
        x_prev = x2
        x = (x2 - tau * TV.nabla_adjoint(u2) + tau * y) / (1 + tau)
        u = u2 + sigma * TV.nabla(2 * x - x2)
        u = u / torch.clamp(torch.sqrt((u ** 2).sum(-1)) / ths, min=1.0).unsqueeze(-1)
        x2 = x2 + rho * (x - x2)
        u2 = u2 + rho * (u - u2)
        c = torch.linalg.norm(x_prev.flatten() - x2.flatten()) / torch.linalg.norm(x2.flatten() + 1e-12)
        if k > 1 and c < crit:
            break
    state["x2"], state["u2"] = x2, u2
    state["cp"] = state.get("cp", 0) + k + 1
    return x2


def bench_eager(path, steps, warmup=2):
    """The reference's PSGLA step (restoration_algorithms.py:232-238) with the eager TV prox, one chain."""
    im, dg, init = problem(path)
    X = init.clone()
    g = torch.Generator(device="cuda").manual_seed(0)
    sig = torch.tensor(S, device="cuda")
    delta = torch.tensor(S * S, device="cuda")
    state = {}

    def step():
        nonlocal X
        Z = torch.randn(X.shape, generator=g, device="cuda")
        Y = X + (delta / LAMBD) * dg(X) + torch.tensor(np.sqrt(2), device="cuda") * sig * Z
        X = eager_tv(Y, sig, state)

    for _ in range(warmup):
        step()
    torch.cuda.synchronize()
    state["cp"] = 0
    t = time.perf_counter()
    for _ in range(steps):
        step()
    torch.cuda.synchronize()
    dt = time.perf_counter() - t
    return dict(B=1, H=int(im.shape[2]), W=int(im.shape[3]), steps=steps, psgla_iter_ms=dt * 1e3 / steps,
                cp_iters_mean=state["cp"] / steps, us_per_cp_iter=dt * 1e6 / state["cp"])


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--eager-steps", type=int, default=3)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("tv_bench.py needs a CUDA device")
    torch.cuda.set_device(0)
    name, power = card()
    res = dict(kind="psgla_tv", device=name, power_limit_w=power, hbm_datasheet_tb_per_s=HBM_TBPS, configs=[], eager=[])
    for B, path in CONFIGS:
        res["configs"].append(bench_cuda(B, path, a.steps, a.warmup))
    for path in ("set3c/butterfly.png", "set1c/castle.png"):
        e = bench_eager(path, a.eager_steps)
        mine = next(c for c in res["configs"] if c["B"] == 1 and (c["H"], c["W"]) == (e["H"], e["W"]))
        e["speedup_cuda_over_eager"] = e["psgla_iter_ms"] / mine["psgla_iter_ms"]
        res["eager"].append(e)
    line = json.dumps(res)
    print(line)
    if a.out:
        with open(a.out, "w") as fh:
            fh.write(line + "\n")


if __name__ == "__main__":
    main()
