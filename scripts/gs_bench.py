"""GS-PSGLA throughput on one GPU: PSGLA inpainting with the gradient-step DRUNet (csrc/gsdrunet.cu), its forward / backward
split, and the reference's loop shape (the fp32 eager restatement with autograd) for comparison.  Prints one JSON line and
writes it to --out (default profiles/gs_bench.json).

    python scripts/gs_bench.py [--steps 20] [--warmup 5] [--eager-steps 3] [--out FILE]

Configurations: 1 chain of 256 x 256 (butterfly.png) and 64 chains of 480 x 320 (castle.png cropped), seeded random weights,
s = 5/255, lambda = 25, alpha = 1, philox noise, statistics-only storage, the fused next-iteration pre.  Per configuration:
  image_it_per_s      chains x PSGLA iterations per second (host clock around n steps ending in a device synchronise)
  fwd_ms / bwd_ms     sums over the 36 forward and the 36 backward layers, each timed alone with CUDA events
                      (psgla_gsdrunet_layer, same kernels as a denoiser call, random operands)
  tflops              4.34 MFLOP per pixel (2.17 forward + 2.17 backward) over the iteration time, and that over the sustained
                      bf16 figure bench.py uses (MEASURED_PEAKS.json, else its 1 400 TFLOP/s fallback)
eager: one PSGLA iteration of the reference's shape (tests/gs_reference.py's torch restatement in fp32, autograd for J^T v),
min(chains, 8) chains, on the same GPU."""
import argparse
import json
import os
import subprocess
import sys
import time

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

import psgla_b200 as P  # noqa: E402
import gs_reference as GS  # noqa: E402

MFLOP_PER_PX = 4.34
S, LAMBD = 5.0 / 255.0, 25.0
CONFIGS = [(1, "set3c/butterfly.png", 256, 256), (64, "set1c/castle.png", 480, 320)]  # castle.png is 481 x 321, cropped
EAGER_CHAINS = 8  # the autograd restatement keeps every activation: 8 chains of 480 x 320 hold tens of GB


def card():
    name = torch.cuda.get_device_name(0)
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader,nounits", "-i", "0"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
        power = float(out.splitlines()[0])
    except Exception:  # noqa: BLE001 -- the power limit is reported when the query tool is present
        power = None
    return name, power


def sustained_tflops():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as fh:
            d = json.load(fh)
        return d.get("bf16_tflops_sustained", d["bf16_tflops"]), "measured"
    return 1400.0, "fallback"


def problem(path, H, W):
    im = P.load_image(os.path.join(ROOT, "tests", "golden", path), device="cuda")
    im = im[:, :, :H, :W].contiguous()
    assert tuple(im.shape[2:]) == (H, W)
    dg, init, y, _ = P.make_inpainting(im, prop=0.5, sigma=1.0, seed_ip=0)
    return dg, init


def layer_split(den, B, H, W, reps=5):
    """(forward ms, backward ms): each of the 72 layers timed alone over `reps` launches."""
    lib = P._lib.lib()
    shape = P._lib.ImgShape(B, 3, H, W)
    keys = P.GSDRUNET_KEYS
    big = torch.randn(B * H * W * 64 + 1024, device="cuda").to(torch.bfloat16)  # inputs / residuals / gates: any bf16 data
    out = torch.empty(B * H * W * 64 * 4 + 1024, dtype=torch.uint8, device="cuda")
    gate = big.clone()
    res1, res2 = big.clone(), big.clone()
    tot = [0.0, 0.0]
    for backward in (0, 1):
        for idx in range(36):
            fl = 35 - idx if backward else idx
            k = keys[fl]
            first = ".res.0." in k
            if backward:
                r1 = res1 if first else None
                r2 = res2 if first and (k.startswith("m_body.0.") or (k.startswith("m_down") and ".0.res." in k)) else None
                gt = gate if ".res.2." in k else None
            else:
                r1 = res1 if ".res.2." in k else None
                r2 = res2 if (".res.2." in k and (k.startswith("m_body.1.") or (k.startswith("m_up") and ".2.res." in k))) else None
                gt = None
            ptr = lambda t: t.data_ptr() if t is not None else None  # noqa: E731

            def call():
                P._lib.check(lib.psgla_gsdrunet_layer(den.packed.data_ptr(), shape, backward, idx, big.data_ptr(), ptr(r1),
                                                      ptr(r2), ptr(gt), out.data_ptr(), None), "psgla_gsdrunet_layer")
            call()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(reps):
                call()
            e1.record()
            torch.cuda.synchronize()
            tot[backward] += e0.elapsed_time(e1) / reps
    return tot


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--eager-steps", type=int, default=3)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "gs_bench.json"))
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("gs_bench.py needs a CUDA device")
    name, power = card()
    peak, peak_src = sustained_tflops()
    sd = P.random_gsdrunet_state_dict(0)
    den = P.GSDRUNet(pretrained=sd)
    ref = GS.GSDRUNet({k: v.cuda() for k, v in sd.items()})
    res = dict(card=name, power_limit_w=power, sustained_bf16_tflops=peak, peak_source=peak_src, mflop_per_pixel=MFLOP_PER_PX,
               configs=[])
    for B, path, H, W in CONFIGS:
        dg, init = problem(path, H, W)
        n = a.warmup + a.steps
        run = P.psgla_run(init, dg, den, 1.0, LAMBD, sig_float=S, delta=S * S, n_iter=n, n_inter=n, n_inter_mmse=n, seed=0,
                          n_chains=B, rng="philox", store="stats")
        for i in range(a.warmup):
            run.step(i)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        for i in range(a.warmup, n):
            run.step(i)
        torch.cuda.synchronize()
        dt = (time.perf_counter() - t0) / a.steps
        assert torch.isfinite(run.X).all()
        fwd, bwd = layer_split(den, B, H, W)
        tflops = MFLOP_PER_PX * 1e6 * B * H * W / dt / 1e12
        # the reference's loop shape: Y = X + data step + noise; X = D(Y) with autograd (restoration_algorithms.py:232-238)
        Be = min(B, EAGER_CHAINS)
        X = init.expand(Be, -1, -1, -1).contiguous()
        gen = torch.Generator(device="cuda").manual_seed(0)

        def eager_step(X):
            Y = X + (S * S / LAMBD) * dg(X) + (2 ** 0.5) * S * torch.randn(X.shape, generator=gen, device="cuda")
            return ref.forward(Y, S)
        X = eager_step(X)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        for _ in range(a.eager_steps):
            X = eager_step(X)
        torch.cuda.synchronize()
        dte = (time.perf_counter() - t0) / a.eager_steps
        res["configs"].append(dict(chains=B, H=H, W=W, image_it_per_s=B / dt, ms_per_iteration=dt * 1e3, fwd_ms=fwd, bwd_ms=bwd,
                                   tflops=tflops, frac_of_sustained=tflops / peak, eager_chains=Be, eager_image_it_per_s=Be / dte,
                                   speedup_vs_eager=(B / dt) / (Be / dte)))
        del run, X
        torch.cuda.empty_cache()
    line = json.dumps(res)
    print(line)
    if a.out:
        os.makedirs(os.path.dirname(a.out), exist_ok=True)
        with open(a.out, "w") as fh:
            fh.write(line + "\n")


if __name__ == "__main__":
    main()
