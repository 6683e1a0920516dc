"""Grayscale against colour on one GPU: the same sampler configurations with one-channel and three-channel DnCNN / DRUNet,
timed alternately in one process.  Prints one JSON line and writes it to --out (default profiles/gray_bench.json).

    python scripts/gray_bench.py [--steps 20] [--warmup 5] [--rounds 3] [--out FILE]

Configurations (seeded random weights and images, philox noise, statistics-only storage, the fused next pre where it applies):
  dncnn_psgla_inpaint_32x256   DnCNN-PSGLA inpainting, 32 chains of 256 x 256
  dncnn_psgla_inpaint_1x256    the same, one chain
  dncnn_pnpula_deblur_32x256   DnCNN PnP-ULA deblurring (l = 4, the A^T A pre kernel), 32 chains of 256 x 256
  drunet_psgla_inpaint_64x480  DRUNet-PSGLA inpainting, 64 chains of 480 x 320 (W x H)
and two kernels alone with CUDA events at 32 chains of 256 x 256: the last DnCNN layer with the fused post and next pre
(psgla_dncnn_last_layer_post_next) and the A^T A deblurring pre (psgla_img_pre_deblur_ata).  Each sampler figure is
image-iterations per second (chains x iterations over a host clock around `steps` iterations ending in a device synchronise),
the best of `rounds` alternating gray / colour rounds; kernel figures are microseconds per launch.  The conv layers do the same
tensor-core work at C = 1 and C = 3 (first-layer K and last-layer N are padded to 16): only the fp32 streams around the
network shrink."""
import argparse
import ctypes
import json
import os
import subprocess
import sys
import time

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import psgla_b200 as P  # noqa: E402

L = P._lib
S = 5.0 / 255.0


def card():
    name = torch.cuda.get_device_name(0)
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader,nounits", "-i", "0"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
        power = float(out.splitlines()[0])
    except Exception:  # noqa: BLE001 -- the power limit is reported when the query tool is present
        power = None
    return name, power


def make_run(family, alg, problem, C, B, H, W, dens):
    g = torch.Generator(device="cuda").manual_seed(0)
    im = torch.rand((1, C, H, W), generator=g, device="cuda")
    if problem == "inpainting":
        dg, init, _, _ = P.make_inpainting(im, prop=0.5, sigma=1.0, seed_ip=0)
    else:
        dg, init, _ = P.make_deblurring(im, l=4, sigma=1.0, seed_ip=0)
    den = dens[(family, C)]
    kw = dict(n_iter=10 ** 6, n_inter=10 ** 6, n_inter_mmse=10 ** 6, seed=0, rng="philox", n_chains=B, store="stats")
    if alg == "psgla":
        return P.psgla_run(init, dg, den, 1.0, 25.0 if family == "drunet" else 5.0, sig_float=S, delta=S ** 2, **kw)
    return P.pnpula_run(init, dg, P.PriorGrad(den, 1.0, S, S ** 2), 1e-5, 2e-5, **kw)


def time_run(run, steps, warmup, start):
    for i in range(start, start + warmup):
        run.step(i)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for i in range(start + warmup, start + warmup + steps):
        run.step(i)
    torch.cuda.synchronize()
    return (time.perf_counter() - t0) / steps


def kernel_times(dens, reps=50):
    """us per launch of the last DnCNN layer (post + next pre) and the A^T A deblurring pre, at C = 1 and C = 3."""
    lib = L.lib()
    B, H, W = 32, 256, 256
    out = {}
    taps = (ctypes.c_float * 9)(*([1.0 / 9] * 9))
    for C in (1, 3, 1, 3):
        den = dens[("dncnn", C)]
        sh = L.ImgShape(B, C, H, W)
        hidden = torch.randn(B * H * W * 64, device="cuda").relu_().to(torch.bfloat16)
        x = torch.rand(B, C, H, W, device="cuda")
        base, xo, m1, m2 = (torch.rand_like(x) for _ in range(4))
        mask, y = torch.ones(1, C, H, W, device="cuda"), torch.rand(1, C, H, W, device="cuda")
        den_in = torch.empty(B * H * W * 16, dtype=torch.bfloat16, device="cuda")
        pre = L.PreParams()
        pre.alg, pre.gain_data, pre.noise_scale, pre.den_in_c3 = L.ALG_PSGLA, 1.0, 0.01, 0.0
        nxt = L.NextPre(ctypes.pointer(pre), mask.data_ptr(), y.data_ptr(), 1, 1, base.data_ptr(), den_in.data_ptr())
        post = L.PostParams(1.0, 1.0, 0.5, 0.5)
        ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]

        def last():
            L.check(lib.psgla_dncnn_last_layer_post_next(den.depth, den.packed.data_ptr(), sh, hidden.data_ptr(), base.data_ptr(),
                                                         ctypes.byref(post), xo.data_ptr(), None, m1.data_ptr(), m2.data_ptr(),
                                                         ctypes.byref(nxt), None), "last layer")

        def ata():
            L.check(lib.psgla_img_pre_deblur_ata(ctypes.byref(pre), sh, x.data_ptr(), taps, 4, y.data_ptr(), 1, None, base.data_ptr(),
                                                 den_in.data_ptr(), None), "ata")

        for name, fn in (("last_layer_post_next", last), ("deblur_ata_pre", ata)):
            for _ in range(5):
                fn()
            ev[0].record()
            for _ in range(reps):
                fn()
            ev[1].record()
            torch.cuda.synchronize()
            us = ev[0].elapsed_time(ev[1]) * 1e3 / reps
            key = "%s_C%d_us" % (name, C)
            out[key] = min(out.get(key, us), us)
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "gray_bench.json"))
    a = ap.parse_args()
    torch.cuda.set_device(0)
    name, power = card()
    dens = {}
    for C in (1, 3):
        dens[("dncnn", C)] = P.DnCNN(C, C, pretrained=P.lipschitz_dncnn_state_dict(0, channels=C))
        dens[("drunet", C)] = P.DRUNet(C, C, pretrained=P.random_drunet_state_dict(0, channels=C))
    configs = [("dncnn_psgla_inpaint_32x256", "dncnn", "psgla", "inpainting", 32, 256, 256),
               ("dncnn_psgla_inpaint_1x256", "dncnn", "psgla", "inpainting", 1, 256, 256),
               ("dncnn_pnpula_deblur_32x256", "dncnn", "pnpula", "deblurring", 32, 256, 256),
               ("drunet_psgla_inpaint_64x480", "drunet", "psgla", "inpainting", 64, 320, 480)]
    res = {"card": name, "power_limit_w": power, "steps": a.steps, "warmup": a.warmup, "rounds": a.rounds}
    for key, fam, alg, prob, B, H, W in configs:
        runs = {C: make_run(fam, alg, prob, C, B, H, W, dens) for C in (1, 3)}
        best = {1: float("inf"), 3: float("inf")}
        it = 0
        for _ in range(a.rounds):
            for C in (1, 3):  # alternating
                best[C] = min(best[C], time_run(runs[C], a.steps, a.warmup, it))
            it += a.steps + a.warmup
        res[key] = {"gray_image_it_per_s": B / best[1], "colour_image_it_per_s": B / best[3], "gray_over_colour": best[3] / best[1]}
        del runs
        torch.cuda.empty_cache()
    res["kernels_32x256"] = kernel_times(dens)
    line = json.dumps(res)
    print(line)
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as fh:
        fh.write(line + "\n")


if __name__ == "__main__":
    main()
