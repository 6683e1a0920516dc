#!/usr/bin/env python
"""bench.py -- throughput of the PSGLA / PnP-ULA hot path on B200, next to the reference's CPU path.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port P \
        bench.py --gpus N --steps K --warmup W

Headline (BASELINE.json configs[1]): 2D Gaussian-mixture posterior sampling, the 18 cells
(3 priors x 3 observations x {PSGLA, PnP-ULA}), 10^6 chains x 10^4 Langevin steps per cell and per GPU.
A "step" of this bench is ONE cell = 10^10 chain-steps per GPU, one launch of the persistent chain kernel;
the K timed steps cycle through the cells.  Chains shard over GPUs with no per-step communication (weak scaling:
10^6 chains per GPU, global chain ids keep every chain's Philox stream independent of the GPU count).
The same line carries `strong` (the config AS WRITTEN: 10^6 chains per cell in total, sharded over the GPUs, all 18 cells),
`config0_single_chain` (configs[0]: the one-chain SnoPnP_ULA(1000) call's latency), `image` / `image_deblur` / `image_drunet` /
`image_set` (configs[2..4]) and, as its last key, `image_summary`.

The same JSON line carries, under "image", the second half of BASELINE.json's metric: PSGLA image
iterations/s at 256x256 with the DnCNN denoiser (configs[2]: random inpainting 50 %, sigma = 1/255, s = 2/255,
lambda = 5, delta = s^2, alpha = 1), a batch of independent chains per GPU; there a "step" is one PSGLA iteration
of the whole batch (1 fused Langevin kernel + 20 tcgen05 conv launches).

Timing: CUDA events on the launching stream around every step, an L2 flush (256 MiB memset, not timed) between
steps, W warm-up steps, barrier + synchronize on both sides, max over ranks.  `value` has its inputs resident in
HBM; `e2e` goes through the public Python API with pinned-host inputs and outputs (copies inside the timed region).
`--impl reference` times the reference's own CPU algorithm (the unmodified reference when /root/reference exists,
else the oracle port) on all host cores.

`--dump-outputs DIR` writes, after the timed steps, what the last timed step of four blocks computed for rank 0's chains:
the 2D headline block's chain states (`gmm2d_state`, after step --steps; --only-image forces --steps to 1) and, for the
three image blocks, the iterate and the running first and second moments (`image_X`, `image_mean`, `image_mean2`, the
same for `image_deblur_*` and `image_drunet_*`, after the --image-steps / --drunet-steps steps of those blocks).  The
strong-scaling, config0, e2e, image-set and GPU-reference timings are not dumped.  Files are DIR/<name>.npy in the array's
own float32 / float64.  An array of more than 2^20 elements is written as the flattened array at a fixed set of 2^20
indices (seeded, sorted; for `gmm2d_state` these are single coordinates, not whole chains), so the ten arrays stay under
64 MB.  Every input is seeded: two builds run with the same arguments can be compared output for output.
"""
from __future__ import annotations

import argparse
import contextlib
import ctypes as C
import json
import os
import statistics
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

PRIORS = ("symetric_gaussians", "cross", "disymmetric_gaussians")  # utils_2D.py:23-33
OBSERVATIONS = ((0.0, 0.0), (0.0, -2.0), (-6.0, 6.0))  # sampling_2D.py:91
GMM_ALGS = {  # sampling_2D.py:83-90,130-131
    "psgla": dict(delta=0.3, alpha=2.0 / 3.0, epsilon=1.0),
    "pnp_ula": dict(delta=0.1, alpha=1.5, epsilon=0.5),
}
CELLS = [(p, y, a) for a in ("psgla", "pnp_ula") for p in PRIORS for y in OBSERVATIONS]
# SURVEY.md section 8(d): algorithmic FP32 flop per chain-step (r = 2, FMA = 2 flop, constants folded on the host)
FLOP_PER_CHAIN_STEP = {"psgla": 82, "pnp_ula": 88}
MUFU_PER_CHAIN_STEP = 7
FP32_PEAK_TFLOPS_NOMINAL = 148 * 128 * 2 * 1.965e9 / 1e12  # 74.5; the denominator used is MEASURED here (measure_fp32_peak)
# What the fp32, r = 2 loop of the shipped kernel issues per chain-step (SASS of gmm2d_lean_kernel, general-structure PSGLA):
# 28 FP32 (FFMA / FMUL / FADD), 9 IMAD.WIDE.U32 + 10 LOP3 (Philox), 6 MUFU, 2 I2FP.  On the FMA pipe an FP32 instruction costs a
# warp 1 cycle and an IMAD.WIDE.U32 4 (scripts/pipe_rates.py, profiles/r02_pipe_rates.txt), so the pipe needs 28 + 4 * 9 = 64 cycles
# per warp-step (55 for cells whose constants are diagonal): the kernel's real bound.
FMA_PIPE_CYCLES_PER_WARP_STEP = {0: 28 + 36, 1: 26 + 36, 2: 19 + 36}
DNCNN_FLOP_PER_PIXEL = 2 * 9 * (3 * 64 + 18 * 64 * 64 + 64 * 3)  # 1 334 016
CONV64_FLOP_PER_PIXEL = 2 * 9 * 64 * 64  # 73 728, one hidden layer
DRUNET_FLOP_PER_PIXEL = 4235136  # head 4 608 + 3 x 16 x 73 728 + 8 x 73 728 + 6 x 16 384 (down / up) + tail 3 456
IMG_BYTES_PER_PIXEL_CHANNEL = 32  # SURVEY.md section 8(d): X r/w, y, mask, E[X], E[X^2] r/w (fp32, Philox mode)


def log(*a):
    print(*a, file=sys.stderr, flush=True)


# The contract is ONE JSON line on stdout.  Libraries (NCCL's version banner, the samplers' reference-style prints)
# write to file descriptor 1 too, so fd 1 is pointed at stderr for the whole run and the line goes to the saved fd.
_REAL_STDOUT = None


def capture_stdout():
    global _REAL_STDOUT
    if _REAL_STDOUT is None:
        sys.stdout.flush()
        _REAL_STDOUT = os.fdopen(os.dup(1), "w")
        os.dup2(2, 1)
        sys.stdout = sys.stderr


def emit(line):
    out = _REAL_STDOUT if _REAL_STDOUT is not None else sys.__stdout__
    out.write(json.dumps(line) + "\n")
    out.flush()


def measured_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as fh:
            d = json.load(fh)
        return dict(hbm_gbs=d["hbm_gbs"], bf16_tflops=d["bf16_tflops"],
                    bf16_tflops_sustained=d.get("bf16_tflops_sustained", d["bf16_tflops"]), source="measured")
    return dict(hbm_gbs=6650.0, bf16_tflops=1590.0, bf16_tflops_sustained=1400.0, source="fallback")


# ------------------------------------------------------------------------------------------------ clocks
class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled every 200 ms while the timed regions run."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.idx = gpu_index
        self.proc = None
        self.path = None

    def start(self):
        try:
            fd, self.path = tempfile.mkstemp(prefix="clocks_", suffix=".csv")
            os.close(fd)
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.idx), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "200"],
                                         stdout=open(self.path, "w"), stderr=subprocess.DEVNULL)
        except Exception as exc:  # noqa: BLE001 -- clocks are evidence, not a dependency
            log("clock sampler unavailable:", exc)
            self.proc = None

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.25)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except subprocess.TimeoutExpired:
            self.proc.kill()
        sm, mx, pw, reasons = [], [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        with open(self.path) as fh:
            for line in fh:
                f = [t.strip() for t in line.split(",")]
                if len(f) < 8:
                    continue
                try:
                    sm.append(float(f[1]))
                    mx.append(float(f[2]))
                    pw.append(float(f[3]))
                except ValueError:
                    continue
                for n, v in zip(names, f[4:8]):
                    if v.lower().startswith("active"):
                        reasons.add(n)
        try:
            os.unlink(self.path)
        except OSError:
            pass
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no samples"]}
        busy = [s for s, p in zip(sm, pw) if p >= 0.5 * max(pw)] or sm
        return {"sm_mhz": statistics.median(busy), "sm_max_mhz": max(mx), "power_w_max": max(pw), "samples": len(sm),
                "reasons": sorted(reasons)}


# ------------------------------------------------------------------------------------------------ helpers
class Timer:
    """Per-step CUDA events on the current stream; the L2 flush between steps is outside the event pairs."""

    def __init__(self, torch, dev):
        self.torch = torch
        self.flush_buf = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
        self.pairs = []

    def flush(self):
        self.flush_buf.zero_()

    def step(self, fn):
        self.flush()
        e0 = self.torch.cuda.Event(enable_timing=True)
        e1 = self.torch.cuda.Event(enable_timing=True)
        e0.record()
        fn()
        e1.record()
        self.pairs.append((e0, e1))

    def total_ms(self):
        self.torch.cuda.synchronize()
        ms = [a.elapsed_time(b) for a, b in self.pairs]
        self.pairs = []
        return sum(ms), ms


DUMP_MAX_ELEMENTS = 1 << 20
_OUTPUTS = {}


def keep_output(args, name, t):
    """Copies (a fixed seeded sample of) a timed block's result to the host for --dump-outputs; a no-op without it."""
    if not args.dump_outputs:
        return
    import numpy as np
    import torch
    a = t.detach()
    if a.numel() > DUMP_MAX_ELEMENTS:
        idx = np.sort(np.random.default_rng(0).choice(a.numel(), DUMP_MAX_ELEMENTS, replace=False))
        a = a.reshape(-1)[torch.from_numpy(idx).to(a.device)]
    _OUTPUTS[name] = (a if a.dtype == torch.float64 else a.float()).cpu().numpy()


def keep_run_outputs(args, block, run):
    """An image sampler's state after its last timed iteration: the iterate and the running moments its windows return."""
    for field in ("X", "mean", "mean2"):
        keep_output(args, "%s_%s" % (block, field), getattr(run, field))


def write_outputs(path):
    import numpy as np
    os.makedirs(path, exist_ok=True)
    for name, a in _OUTPUTS.items():
        np.save(os.path.join(path, name + ".npy"), a)
    log("--dump-outputs: %s written to %s" % (", ".join(sorted(_OUTPUTS)), path))


def barrier(torch, dist_mod):
    torch.cuda.synchronize()
    if dist_mod.world()[1] > 1:
        import torch.distributed as dist
        dist.barrier()
    torch.cuda.synchronize()


def measure_fp32_peak(P, torch, dev):
    """Measured FP32 issue peak of this GPU (csrc/selftest.cu: nothing but dependent FFMA chains, 8 per thread), TFLOP/s.
    Burst figure: best of 4 launches of ~25 ms, CUDA events."""
    lib = P._lib.lib()
    scratch = torch.empty(148 * 8 * 256 * 2, dtype=torch.float32, device=dev)
    best = {}
    for mode, name in ((0, "ffma"), (1, "ffma2")):
        flop = C.c_double()
        for _ in range(4):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            P._lib.check(lib.psgla_selftest_fp32_rate(mode, 150000, 8, scratch.data_ptr(), C.byref(flop), P._lib.stream_ptr(dev)), "fp32_rate")
            e1.record()
            torch.cuda.synchronize()
            best[name] = max(best.get(name, 0.0), flop.value / (e0.elapsed_time(e1) * 1e-3) / 1e12)
    return best


# FP32 pipe slots per chain-step of gmm2d_lean_kernel<ALG, STRUCT, 4, 64, 16, 1> (SASS of the loop, scalar FP32 + 2 x packed):
# the NF of the matching instruction-mix probe (psgla_selftest_pipe_rate mode 100 + NF)
MIX_NF = {("psgla", 2): 21, ("pnp_ula", 2): 23, ("psgla", 1): 26, ("pnp_ula", 1): 28, ("psgla", 0): 28, ("pnp_ula", 0): 30}


def measure_mix_ceiling(P, torch, dev):
    """Chain-steps/s this GPU sustains for the chain kernel's per-step INSTRUCTION MIX (6 MUFU, 9 IMAD.WIDE.U32, NF FP32, 10 LOP3,
    2 I2FP) when the instructions are independent (csrc/selftest.cu, pipe_rate_kernel<11, NF>): the measured roofline of a kernel
    that is bound by neither memory nor a single pipe but by how the SM issues this mix.  One figure per NF."""
    lib = P._lib.lib()
    scratch = torch.empty(148 * 8 * 256 * 2, dtype=torch.float32, device=dev)
    out = {}
    for nf in sorted(set(MIX_NF.values())):
        ops = C.c_double()
        best = 0.0
        for _ in range(3):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            P._lib.check(lib.psgla_selftest_pipe_rate(100 + nf, 20000, 8, scratch.data_ptr(), C.byref(ops), P._lib.stream_ptr(dev)), "pipe_rate")
            e1.record()
            torch.cuda.synchronize()
            best = max(best, ops.value / (e0.elapsed_time(e1) * 1e-3))
        out[nf] = best
    return out


def gmm_structure(P, prior):
    """Which specialisation of the chain kernel a cell takes (csrc/gmm2d.cu constants_structure): 2 = all matrices diagonal
    (isotropic / axis-aligned covariances), 1 = only the data term (A = I), 0 = general."""
    import numpy as np
    _, Sig, _ = P.gaussian_mixt_example(prior)
    return 2 if all(abs(np.asarray(S)[0][1]) == 0 and abs(np.asarray(S)[1][0]) == 0 for S in Sig) else 1


# ------------------------------------------------------------------------------------------------ 2D GMM (product)
def bench_gmm2d_strong(args, P, torch, rank, ws, dev):
    """BASELINE.json configs[1] AS WRITTEN: 10^6 chains in total per cell, sharded over the GPUs (contiguous blocks of global
    chain ids, dist.shard_range), all 18 cells once.  Cells are independent sampling problems, so a rank keeps up to
    --strong-streams cells in flight on separate CUDA streams: with 125 000 chains per GPU one cell fills 0.8 of a wave and
    the second cell's blocks take the slots the first leaves free."""
    import numpy as np
    total = args.strong_chains
    world = args.emulate_world if (ws == 1 and args.emulate_world > 1) else ws
    me = 0 if world != ws else rank
    lo, hi = P.dist.shard_range(total, me, world)
    n_local = hi - lo
    pops = []
    for prior, y, alg in CELLS:
        mu, Sig, pi = P.gaussian_mixt_example(prior)
        prm = GMM_ALGS[alg]
        x0 = torch.tensor(y, dtype=torch.float32, device=dev).repeat(n_local, 1).contiguous()
        pops.append((P.GMMChains(alg, np.array(y), prm["delta"], np.eye(2), 1.0, P.Theorical_MMSE(mu, Sig, pi), prm["alpha"],
                                 prm["epsilon"], n_chains=n_local, x0=x0, seed=args.seed, chain_id0=lo, dtype="float32",
                                 device=dev), x0))
    streams = [torch.cuda.Stream(device=dev) for _ in range(max(1, args.strong_streams))]

    def all_cells():
        cur = torch.cuda.current_stream(dev)
        for st in streams:
            st.wait_stream(cur)
        for i, (ch, x0) in enumerate(pops):
            with torch.cuda.stream(streams[i % len(streams)]):
                ch.state.copy_(x0)
                ch.step = 0
                ch.run(args.chain_steps)
        for st in streams:
            cur.wait_stream(st)

    all_cells()  # warm-up pass (all 18 cells)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    flush.zero_()
    barrier(torch, P.dist)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    all_cells()
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1)
    barrier(torch, P.dist)
    ms = P.dist.max_over_ranks(ms, dev)
    units = float(total) * args.chain_steps * len(CELLS)
    out = {"scaling": "strong", "value": units / (ms * 1e-3), "unit": "chain-steps/s",
           "total_chains_per_cell": total, "chains_per_gpu": n_local, "cells": len(CELLS), "ms_all_cells": ms,
           "streams": len(streams), "n_gpus": ws,
           "note": "10^6 chains per cell in total, sharded over the GPUs; value = 18 x 10^6 x 10^4 chain-steps / max-over-ranks device time"}
    if world != ws:
        out["emulated_world"] = world
        out["note"] = ("rank 0's shard of an emulated %d-GPU split on one GPU: value = this GPU's chain-steps/s at %d chains per cell"
                       % (world, n_local))
        out["value"] = float(n_local) * args.chain_steps * len(CELLS) / (ms * 1e-3)
    return out


def bench_gmm2d_config0(args, P, torch, dev):
    """BASELINE.json configs[0]: `sampling_2D.py --N 1000 --name symetric_gaussians` -- ONE chain, 999 steps, through the drop-in
    SnoPnP_ULA exactly as the script calls it (float64, the global NumPy stream replayed).  Latency, not throughput: one thread
    of one warp walks 999 dependent steps."""
    import numpy as np
    mu, Sig, pi = P.gaussian_mixt_example("symetric_gaussians")
    D = P.Theorical_MMSE(mu, Sig, pi)
    y = np.array([0.0, -2.0])
    times = []
    for rep in range(6):
        np.random.seed(rep)
        t0 = time.perf_counter()
        X = P.SnoPnP_ULA(1000, y, y, 0.3, np.eye(2), 1, D, 2.0 / 3.0)
        dt = time.perf_counter() - t0
        if rep:
            times.append(dt)
    assert X.shape == (1000, 2)
    # the kernel alone (device time of the 999-step launch, replay mode, fp64)
    ch = P.GMMChains("psgla", y, 0.3, np.eye(2), 1.0, D, 2.0 / 3.0, n_chains=1, dtype="float64", device=dev)
    z = torch.randn(999, 1, 2, dtype=torch.float64, device=dev)
    ch.run(999, noise=z)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    ch.run(999, noise=z)
    e1.record()
    torch.cuda.synchronize()
    best = min(times)
    return {"workload": "SnoPnP_ULA(1000, x0 = y = (0,-2), delta 0.3, alpha 2/3, symetric_gaussians), one chain, float64, NumPy stream replayed",
            "call_ms": best * 1e3, "us_per_step": best * 1e6 / 999, "steps_per_s": 999 / best,
            "kernel_ms": e0.elapsed_time(e1), "kernel_us_per_step": e0.elapsed_time(e1) * 1e3 / 999,
            "reference_us_per_step_here": None}


def bench_gmm2d(args, P, torch, rank, ws, dev):
    import numpy as np
    n_chains, n_steps = args.chains, args.chain_steps
    K, W = args.steps, args.warmup
    chain_id0 = rank * n_chains
    used = sorted({k % len(CELLS) for k in range(W + K)})
    pops, x0s = {}, {}
    for ci in used:
        prior, y, alg = CELLS[ci]
        mu, Sig, pi = P.gaussian_mixt_example(prior)
        D = P.Theorical_MMSE(mu, Sig, pi)
        prm = GMM_ALGS[alg]
        x0 = torch.tensor(y, dtype=torch.float32, device=dev).repeat(n_chains, 1).contiguous()
        pops[ci] = P.GMMChains(alg, np.array(y), prm["delta"], np.eye(2), 1.0, D, prm["alpha"], prm["epsilon"],
                               n_chains=n_chains, x0=x0, seed=args.seed, chain_id0=chain_id0, dtype="float32", device=dev)
        x0s[ci] = x0

    def one(k):
        ch = pops[k % len(CELLS)]
        ch.state.copy_(x0s[k % len(CELLS)])
        ch.step = 0
        return ch

    for k in range(W):
        one(k).run(n_steps)
    timer = Timer(torch, dev)
    barrier(torch, P.dist)
    flop = 0.0
    for k in range(W, W + K):
        ch = one(k)
        timer.step(lambda: ch.run(n_steps))
        flop += FLOP_PER_CHAIN_STEP[CELLS[k % len(CELLS)][2]] * float(n_chains) * n_steps
    total_ms, per_step = timer.total_ms()
    keep_output(args, "gmm2d_state", ch.state)
    launches_per_step = int(P._lib.lib().psgla_gmm2d_last_launches())
    barrier(torch, P.dist)
    total_ms = P.dist.max_over_ranks(total_ms, dev)

    # ---- e2e: the public API with pinned-host initial states and pinned-host results, copies inside the timed region
    x0_host = {ci: torch.tensor(CELLS[ci][1], dtype=torch.float32).repeat(n_chains, 1).pin_memory() for ci in used}
    out_host = torch.empty((n_chains, 2), dtype=torch.float32).pin_memory()

    def e2e_step(k):
        ci = k % len(CELLS)
        prior, y, alg = CELLS[ci]
        prm = GMM_ALGS[alg]
        mu, Sig, pi = P.gaussian_mixt_example(prior)
        ch = P.GMMChains(alg, np.array(y), prm["delta"], np.eye(2), 1.0, P.Theorical_MMSE(mu, Sig, pi), prm["alpha"],
                         prm["epsilon"], n_chains=n_chains, x0=x0_host[ci], seed=args.seed, chain_id0=chain_id0,
                         dtype="float32", device=dev)
        ch.run(n_steps)
        out_host.copy_(ch.state, non_blocking=True)

    for k in range(min(W, 3)):
        e2e_step(k)
    barrier(torch, P.dist)
    t0 = time.perf_counter()
    for k in range(W, W + K):
        e2e_step(k)
    torch.cuda.synchronize()
    e2e_ms = (time.perf_counter() - t0) * 1e3
    barrier(torch, P.dist)
    e2e_ms = P.dist.max_over_ranks(e2e_ms, dev)

    # ---- quality next to the speed: W2^2 to the true posterior per cell (utils_2D.py:235-244), all ranks' chains
    w2 = {}
    for ci in used:
        prior, y, alg = CELLS[ci]
        finals = P.dist.gather_to_rank0(pops[ci].state)
        if rank == 0:
            mu, Sig, pi = P.gaussian_mixt_example(prior)
            rng = np.random.default_rng(1234)
            ref = P.sample_posterior(np.eye(2), np.array(y), 1.0, 10000, mu, Sig, pi, rng=rng)
            sub = finals[torch.randperm(finals.shape[0], device=finals.device)[:10000]].double().cpu().numpy()
            w2["%s|%s|y=(%g,%g)" % (alg, prior, y[0], y[1])] = round(P.Wasserstein_distance(sub, ref, rng=rng), 4)
    units = float(n_chains) * n_steps * K * ws
    pipe_cycles = sum(FMA_PIPE_CYCLES_PER_WARP_STEP[gmm_structure(P, CELLS[k % len(CELLS)][0])] for k in range(W, W + K)) / K
    cells_nf = [MIX_NF[(CELLS[k % len(CELLS)][2], gmm_structure(P, CELLS[k % len(CELLS)][0]))] for k in range(W, W + K)]
    return dict(cells_nf=cells_nf, pipe_cycles=pipe_cycles, value=units / (total_ms * 1e-3), total_ms=total_ms, per_step_ms=per_step, flop=flop,
                e2e_value=units / (e2e_ms * 1e-3), e2e_ms=e2e_ms, h2d=n_chains * 2 * 4, d2h=n_chains * 2 * 4, w2=w2,
                launches_per_step=launches_per_step)


# ------------------------------------------------------------------------------------------------ image PSGLA (product)
def synthetic_image(torch, H, W, seed, dev):
    """Smooth synthetic colour image in [0,1] (no dataset travels to the GPU box)."""
    g = torch.Generator().manual_seed(seed)
    low = torch.rand((1, 3, H // 16 + 2, W // 16 + 2), generator=g)
    im = torch.nn.functional.interpolate(low, size=(H, W), mode="bicubic", align_corners=False).clamp(0, 1)
    return im.to(dev).contiguous()


def bench_image(args, P, torch, rank, ws, dev, peaks):
    from importlib import import_module
    _lib = import_module("psgla_b200._lib")
    B, H, Wd = args.image_chains, args.image_size, args.image_size
    K, W = args.image_steps, max(args.warmup, 3)
    s = 2.0 / 255.0  # sampling_images.py:170-198: DnCNN => s = 2/255, lambda = 5, delta = s^2
    kw = dict(alpha=1.0, lambd=5.0, sig_float=s, delta=s * s, n_inter=10, n_inter_mmse=10, seed=args.seed)
    im = synthetic_image(torch, H, Wd, 0, dev)
    den = P.DnCNN(pretrained=P.lipschitz_dncnn_state_dict(0), device=dev)
    dg, init, y, mask = P.make_inpainting(im, prop=0.5, sigma=1.0, seed_ip=0)
    run = P.psgla_run(init, dg, den, n_iter=W + K, n_chains=B, chain_id0=rank * B, **kw)
    for i in range(W):
        run.step(i)
    timer = Timer(torch, dev)
    barrier(torch, P.dist)
    for i in range(W, W + K):
        timer.step(lambda: run.step(i))
    total_ms, per_step = timer.total_ms()
    keep_run_outputs(args, "image", run)
    barrier(torch, P.dist)
    total_ms = P.dist.max_over_ranks(total_ms, dev)
    finite = bool(torch.isfinite(run.X).all().item())
    x_absmax = float(run.X.abs().max().item())

    # ---- the dominant kernel alone: the 18 hidden 64->64 conv layers, CUDA events around back-to-back launches
    shape = _lib.ImgShape(B, 3, H, Wd)
    wsbuf, _ = den.buffers(shape)
    half = (B * H * Wd * 64 * 2 + 1023) // 1024 * 1024
    bufs = [wsbuf.data_ptr(), wsbuf.data_ptr() + half]
    lib = _lib.lib()
    st = _lib.stream_ptr(dev)

    def hidden_layers():
        for l in range(1, 19):
            rc = lib.psgla_conv3x3_layer(den.packed.data_ptr(), den.depth, l, shape, bufs[l & 1], bufs[(l + 1) & 1], 1, st)
            if rc:
                _lib.check(rc, "psgla_conv3x3_layer")

    hidden_layers()
    reps = 5
    for _ in range(9):
        timer.step(hidden_layers)
    _, conv_reps = timer.total_ms()
    conv_launch_ms = sorted(conv_reps)[len(conv_reps) // 2] / 18  # median repetition: the block sits at the power cap

    # ---- the reference's own shape of run: ONE chain (launch-latency bound: 20 launches of ~8 us per iteration)
    # Two hidden layers per launch here (csrc/conv_fused2.cu): 11 launches per iteration.  The loop is latency-bound, so it is
    # timed in ITS OWN steady state: ~0.2 s of iterations first -- the power-capped 32-chain blocks above leave the SM clock
    # low for tens of milliseconds (134 us per iteration right after them, 125 us once the clock is back, same box).
    run1 = P.psgla_run(init, dg, den, n_iter=2000, n_chains=1, chain_id0=rank, **kw)
    for i in range(1500):
        run1.step(i)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for i in range(1500, 1800):
        run1.step(i)
    e1.record()
    torch.cuda.synchronize()
    single_chain_its = 300.0 / (e0.elapsed_time(e1) * 1e-3)
    del run1
    os.environ["PSGLA_CONV_FUSE2"] = "0"  # the same loop with one layer per launch (the switch is read per call)
    try:
        run1 = P.psgla_run(init, dg, den, n_iter=800, n_chains=1, chain_id0=rank, **kw)
        for i in range(300):
            run1.step(i)
        torch.cuda.synchronize()
        e0.record()
        for i in range(300, 600):
            run1.step(i)
        e1.record()
        torch.cuda.synchronize()
        single_chain_unfused_its = 300.0 / (e0.elapsed_time(e1) * 1e-3)
        del run1
    finally:
        os.environ.pop("PSGLA_CONV_FUSE2", None)

    # ---- the fused Langevin "pre" kernel alone (HBM-bound stage)
    def pre_only():
        run.pre(W + K - 1, run.pre_params)
    pre_only()
    for _ in range(reps):
        timer.step(pre_only)
    pre_ms, _ = timer.total_ms()
    pre_launch_ms = pre_ms / reps

    # ---- the last layer alone: 64 -> 3 conv + Langevin post (X+, thinning every 10th, moments) + the next iteration's pre
    nxt_params = _lib.PreParams()
    C.memmove(C.byref(nxt_params), C.byref(run.pre_params), C.sizeof(_lib.PreParams))
    run._stamp(nxt_params, W + K)
    nxt = _lib.NextPre(C.pointer(nxt_params), _lib.ptr(run.mask), _lib.ptr(run.y), int(run.mask.shape[0]), int(run.y.shape[0]),
                       _lib.ptr(run.base), _lib.ptr(run.den_in))
    post = _lib.PostParams(1.0, 1.0, 0.5, 0.5)
    x_scratch = torch.empty_like(run.X)

    def last_only():
        rc = lib.psgla_dncnn_last_layer_post_next(den.depth, den.packed.data_ptr(), shape, bufs[0], _lib.ptr(run.base), C.byref(post),
                                                  _lib.ptr(x_scratch), None, _lib.ptr(run.mean), _lib.ptr(run.mean2), C.byref(nxt), st)
        if rc:
            _lib.check(rc, "psgla_dncnn_last_layer_post_next")

    last_only()
    for _ in range(reps):
        timer.step(last_only)
    last_ms, _ = timer.total_ms()
    last_launch_ms = last_ms / reps
    # algorithmic bytes per pixel: 128 (bf16 hidden in) + fp32 x 3 channels x (base in, X out, E[X] in/out, E[X^2] in/out, mask, y,
    # next base out) = 9 x 12 + 32 (bf16 NHWC16 next denoiser input) = 268; thinned sample (+12 every n_inter-th iteration) not counted
    last_bytes_px = 128 + 9 * 12 + 32

    # ---- e2e: psgla() itself, pinned-host image / mask / observation in, pinned-host posterior mean out
    n_e2e = max(K, 100)  # one psgla() call of 100 iterations (the reference runs 10^4 per image); set-up amortised as in use
    host = dict(init=init.cpu().pin_memory(), mask=mask.cpu().pin_memory(), y=y.cpu().pin_memory())
    out_host = torch.empty((B, 3, H, Wd), dtype=torch.float32).pin_memory()

    def e2e_call():
        with contextlib.redirect_stdout(sys.stderr):
            dg2 = P.InpaintingDataGrad(host["mask"].to(dev, non_blocking=True), host["y"].to(dev, non_blocking=True),
                                       dg.sigma2)
            Xl, Mm, _ = P.psgla(host["init"].to(dev, non_blocking=True), dg2, den, n_iter=n_e2e, n_chains=B,
                                chain_id0=rank * B, **kw)
            out_host.copy_(Mm[-1], non_blocking=True)
        torch.cuda.synchronize()

    e2e_call()
    barrier(torch, P.dist)
    t0 = time.perf_counter()
    e2e_call()
    e2e_ms = (time.perf_counter() - t0) * 1e3
    barrier(torch, P.dist)
    e2e_ms = P.dist.max_over_ranks(e2e_ms, dev)

    px = B * H * Wd
    conv_tflops = CONV64_FLOP_PER_PIXEL * px / (conv_launch_ms * 1e-3) / 1e12
    step_tflops = DNCNN_FLOP_PER_PIXEL * px * K / (total_ms * 1e-3) / 1e12
    pre_gbs = (IMG_BYTES_PER_PIXEL_CHANNEL - 16) * 3 * px / (pre_launch_ms * 1e-3) / 1e9  # pre touches X, y, mask, base
    return {
        "metric": "psgla_image_iterations_per_sec_256x256_dncnn", "unit": "image-iterations/s",
        "value": B * K * ws / (total_ms * 1e-3), "ms_per_step": total_ms / K, "steps": K, "warmup": W,
        "config": {"workload": "random inpainting 50%%, sigma=1/255, PSGLA s=2/255 lambda=5 delta=s^2 alpha=1, DnCNN depth 20 "
                               "(seeded random-init, Lipschitz 0.9), %d chains/GPU of %dx%dx3, in-kernel Philox" % (B, H, Wd),
                   "chains_per_gpu": B, "l2": "256 MiB flush between timed iterations"},
        "dtype": "bf16 activations / fp32 accumulate, fp32 state",
        "gpu_launches": 20 * K,  # 20 conv launches; the Langevin pre / post steps live in the last layer's epilogue
        "e2e": {"value": B * n_e2e * ws / (e2e_ms * 1e-3), "unit": "image-iterations/s", "iterations": n_e2e,
                "h2d_bytes_per_step": int(3 * 3 * H * Wd * 4 / n_e2e), "d2h_bytes_per_step": int(B * 3 * H * Wd * 4 / n_e2e)},
        "roofline": {"kernel": "conv3x3_ts2_kernel<64,false> (CTA-pair tcgen05 implicit GEMM; 18 of the 20 launches per iteration)", "bound": "tensor",
                     # the kernel is timed ALONE here (18 launches back to back, ~2 ms per repetition): the burst cuBLAS figure is its
                     # denominator; the sustained one (cuBLAS's own rate after seconds at the power cap) is the whole iteration's
                     "achieved": conv_tflops, "peak": peaks["bf16_tflops"], "unit": "TFLOP/s",
                     "frac": conv_tflops / peaks["bf16_tflops"], "frac_of_sustained_peak": conv_tflops / peaks["bf16_tflops_sustained"],
                     "peak_source": peaks["source"] + " (cuBLAS bf16, burst; frac_of_sustained_peak can read above 1: this block is "
                                                      "too short to heat the box the way the 4 s sustained measurement does)",
                     "launch_ms": conv_launch_ms,
                     # ncu --set full, one launch at 32 chains of 256 x 256 (profiles/r02_conv3x3_ts2_full.txt): 274.8 MB read +
                     # 218.6 MB written against 536.9 MB algorithmic (bf16 in + out); part of the output is still in L2.
                     # Same capture: 101.2 us for the launch alone (1 527 TFLOP/s), tensor pipe active 88.1 % of the active and
                     # 80.8 % of the elapsed cycles (round 1: 75.2 %; single-CTA TS kernel: 62.4 %).  Timed here back to back at the
                     # power cap, the kernel sits at what cuBLAS sustains there.
                     "traffic": 493.3e6 if (B == 32 and H == 256) else None,
                     "traffic_source": "profiles/r02_conv3x3_ts2_full.txt",
                     "ncu_tensor_pipe_active_pct": 88.1, "ncu_launch_us_alone": 101.2},
        "whole_iteration_tensor_tflops": step_tflops,
        "whole_iteration_frac": step_tflops / peaks["bf16_tflops_sustained"],
        "pre_kernel": {"bound": "hbm", "achieved": pre_gbs, "peak": peaks["hbm_gbs"], "unit": "GB/s",
                       "frac": pre_gbs / peaks["hbm_gbs"], "launch_ms": pre_launch_ms,
                       # the kernel also writes the padded bf16 NHWC16 denoiser input (32 B per pixel), which the algorithmic
                       # 16 B per pixel-channel above does not count
                       "moved_gbs_incl_den_in": (16 * 3 + 32) * px / (pre_launch_ms * 1e-3) / 1e9},
        "last_layer_kernel": {"kernel": "conv3x3_ts_kernel<16,POST> (64 -> 3 conv + fused Langevin post + next-iteration pre)",
                              "bound": "hbm", "achieved": last_bytes_px * px / (last_launch_ms * 1e-3) / 1e9, "peak": peaks["hbm_gbs"],
                              "unit": "GB/s", "frac": last_bytes_px * px / (last_launch_ms * 1e-3) / 1e9 / peaks["hbm_gbs"],
                              "launch_ms": last_launch_ms, "algorithmic_bytes_per_pixel": last_bytes_px},
        "single_chain_iterations_per_sec": single_chain_its,
        "single_chain": {"iterations_per_sec": single_chain_its, "us_per_iteration": 1e6 / single_chain_its,
                         "tensor_tflops": DNCNN_FLOP_PER_PIXEL * H * Wd * single_chain_its / 1e12,
                         "frac_of_burst_peak": DNCNN_FLOP_PER_PIXEL * H * Wd * single_chain_its / 1e12 / peaks["bf16_tflops"],
                         "us_per_iteration_one_layer_per_launch": 1e6 / single_chain_unfused_its,
                         "note": "the reference's own run shape (configs[2]: one chain of one 256 x 256 image): 11 launches per "
                                 "iteration, two hidden layers per launch (conv_fused2.cu, bit-identical to the 20-launch form)"},
        "state_finite": finite, "state_absmax": x_absmax,
        "per_step_ms": [round(v, 3) for v in per_step],
    }


def bench_image_deblur(args, P, torch, rank, ws, dev, peaks):
    """BASELINE.json configs[3]: uniform 9x9 blur (l = 4), PnP-ULA with DnCNN, a batch of independent chains of one 256 x 256
    image; hyper-parameters as the script resolves them (sampling_images.py:147-168 via P.sampler_params)."""
    B, H, Wd = args.image_chains, args.image_size, args.image_size
    K, W = args.image_steps, max(args.warmup, 3)
    prm = P.sampler_params("pnp_ula", den="DnCNN")
    im = synthetic_image(torch, H, Wd, 1, dev)
    den = P.DnCNN(pretrained=P.lipschitz_dncnn_state_dict(0), device=dev)
    dg, init, y = P.make_deblurring(im, l=4, blur_type="uniform", sigma=1.0, seed_ip=0)
    pg = P.PriorGrad(den, prm["alpha"], prm["s1"], prm["s2"])
    run = P.pnpula_run(init, dg, pg, prm["delta"], prm["lambd"], n_iter=W + K, n_inter=prm["n_inter"],
                       n_inter_mmse=prm["n_inter_mmse"], seed=args.seed, n_chains=B, chain_id0=rank * B)
    for i in range(W):
        run.step(i)
    timer = Timer(torch, dev)
    barrier(torch, P.dist)
    for i in range(W, W + K):
        timer.step(lambda: run.step(i))
    total_ms, per_step = timer.total_ms()
    keep_run_outputs(args, "image_deblur", run)
    barrier(torch, P.dist)
    total_ms = P.dist.max_over_ranks(total_ms, dev)
    finite = bool(torch.isfinite(run.X).all().item())

    def pre_only():
        run.pre(W + K - 1, run.pre_params)
    pre_only()
    reps = 5
    for _ in range(reps):
        timer.step(pre_only)
    pre_ms, _ = timer.total_ms()
    pre_launch_ms = pre_ms / reps
    px = B * H * Wd
    # deblur_ata_kernel<8>: reads X and A^T y, writes base (fp32, 12 B per pixel-channel) + the bf16 NHWC16 denoiser input (32 B/px)
    pre_bytes = (12 * 3 + 32) * px
    step_tflops = DNCNN_FLOP_PER_PIXEL * px * K / (total_ms * 1e-3) / 1e12
    return {
        "metric": "pnpula_image_iterations_per_sec_256x256_dncnn_deblur", "unit": "image-iterations/s",
        "value": B * K * ws / (total_ms * 1e-3), "ms_per_step": total_ms / K, "steps": K, "warmup": W,
        "config": {"workload": "uniform 9x9 blur (l=4), sigma=1/255, PnP-ULA delta=%.3g lambda=%.3g s1=%.3g (sampling_images.py:147-168), "
                               "DnCNN depth 20 (seeded random-init, Lipschitz 0.9), %d chains/GPU of %dx%dx3, in-kernel Philox"
                               % (prm["delta"], prm["lambd"], prm["s1"], B, H, Wd),
                   "chains_per_gpu": B, "l2": "256 MiB flush between timed iterations"},
        "dtype": "bf16 activations / fp32 accumulate, fp32 state", "gpu_launches": 21 * K,
        "whole_iteration_tensor_tflops": step_tflops,
        "whole_iteration_frac": step_tflops / peaks["bf16_tflops_sustained"],
        "pre_kernel": {"kernel": ("blur_kernel_t<true,4> (four 9-tap passes, PSGLA_BLUR_4PASS=1)" if run.aty is None else
                                  "deblur_ata_kernel<8> ((A^T A) x - A^T y: row-streaming separable 17-tap stencil, A^T y precomputed, "
                                  "+ projection + noise)"), "bound": "hbm", "achieved": pre_bytes / (pre_launch_ms * 1e-3) / 1e9,
                       "peak": peaks["hbm_gbs"], "unit": "GB/s",
                       "frac": pre_bytes / (pre_launch_ms * 1e-3) / 1e9 / peaks["hbm_gbs"], "launch_ms": pre_launch_ms,
                       "algorithmic_bytes_per_pixel": 12 * 3 + 32},
        "state_finite": finite, "per_step_ms": [round(v, 3) for v in per_step],
    }


def bench_image_drunet(args, P, torch, rank, ws, dev, peaks):
    """BASELINE.json configs[4]: inpainting PSGLA with the DRUNet-architecture denoiser (seeded random init), a batch of
    independent chains of one 320 x 480 image (a CBSD68 image cropped to multiples of 8) per GPU."""
    B, H, Wd = args.drunet_chains, args.drunet_h, args.drunet_w
    K, W = args.drunet_steps, max(args.warmup, 3)
    s = 5.0 / 255.0  # sampling_images.py:194-198: non-DnCNN denoisers => s = 5/255, delta = s^2; lambda = 25 keeps the
    lambd = 25.0     # data-term gain (delta/lambda)/sigma^2 at 1 (the script's default lambda = 1 gives 25 and diverges)
    kw = dict(alpha=1.0, lambd=lambd, sig_float=s, delta=s * s, n_inter=10, n_inter_mmse=10, seed=args.seed)
    im = synthetic_image(torch, H, Wd, 1, dev)
    den = P.DRUNet(pretrained=P.random_drunet_state_dict(0), device=dev)
    dg, init, y, mask = P.make_inpainting(im, prop=0.5, sigma=1.0, seed_ip=0)
    run = P.psgla_run(init, dg, den, n_iter=W + K, n_chains=B, chain_id0=rank * B, **kw)
    for i in range(W):
        run.step(i)
    timer = Timer(torch, dev)
    barrier(torch, P.dist)
    for i in range(W, W + K):
        timer.step(lambda: run.step(i))
    total_ms, per_step = timer.total_ms()
    keep_run_outputs(args, "image_drunet", run)
    barrier(torch, P.dist)
    total_ms = P.dist.max_over_ranks(total_ms, dev)
    finite = bool(torch.isfinite(run.X).all().item())
    del run

    # ---- e2e: psgla() itself, pinned-host image / mask / observation in, pinned-host posterior mean out
    n_e2e = 33
    host = dict(init=init.cpu().pin_memory(), mask=mask.cpu().pin_memory(), y=y.cpu().pin_memory())
    out_host = torch.empty((B, 3, H, Wd), dtype=torch.float32).pin_memory()

    def e2e_call():
        with contextlib.redirect_stdout(sys.stderr):
            dg2 = P.InpaintingDataGrad(host["mask"].to(dev, non_blocking=True), host["y"].to(dev, non_blocking=True), dg.sigma2)
            Xl, Mm, _ = P.psgla(host["init"].to(dev, non_blocking=True), dg2, den, n_iter=n_e2e, n_chains=B, chain_id0=rank * B, **kw)
            out_host.copy_(Mm[-1], non_blocking=True)
        torch.cuda.synchronize()

    e2e_call()
    barrier(torch, P.dist)
    t0 = time.perf_counter()
    e2e_call()
    e2e_ms = (time.perf_counter() - t0) * 1e3
    barrier(torch, P.dist)
    e2e_ms = P.dist.max_over_ranks(e2e_ms, dev)

    px = B * H * Wd
    tflops = DRUNET_FLOP_PER_PIXEL * px * K / (total_ms * 1e-3) / 1e12
    return {
        "metric": "psgla_image_iterations_per_sec_drunet", "unit": "image-iterations/s",
        "value": B * K * ws / (total_ms * 1e-3), "ms_per_step": total_ms / K, "steps": K, "warmup": W,
        "config": {"workload": "random inpainting 50%%, sigma=1/255, PSGLA s=5/255 lambda=25 delta=s^2 alpha=1, DRUNet "
                               "(KAIR UNetRes 64/128/256/512, seeded random-init), %d chains/GPU of %dx%dx3" % (B, H, Wd),
                   "chains_per_gpu": B, "l2": "256 MiB flush between timed iterations"},
        "dtype": "bf16 activations / fp32 accumulate, fp32 state", "gpu_launches": 68 * K,
        "e2e": {"value": B * n_e2e * ws / (e2e_ms * 1e-3), "unit": "image-iterations/s", "iterations": n_e2e,
                "h2d_bytes_per_step": int(3 * 3 * H * Wd * 4 / n_e2e), "d2h_bytes_per_step": int(B * 3 * H * Wd * 4 / n_e2e)},
        "roofline": {"kernel": "whole iteration: 68 conv launches, the Langevin step in the last one (CTA-pair kernels conv_gemm2_kernel<128|256> and "
                               "conv3x3_ts2_kernel<64>; conv_gemm_kernel<64> for the 64-channel up-conv)",
                     "bound": "tensor", "achieved": tflops, "peak": peaks["bf16_tflops_sustained"], "unit": "TFLOP/s",
                     "frac": tflops / peaks["bf16_tflops_sustained"], "frac_of_burst_peak": tflops / peaks["bf16_tflops"],
                     "peak_source": peaks["source"] + " (cuBLAS bf16, sustained)", "traffic": None,
                     # one ncu --set full capture of this workload's 256-channel 3x3 layer (64 chains, 80 x 120 pixels):
                     # 466 us = 1 555 TFLOP/s useful, tensor pipe active 97.9 % of the active cycles at 1.50 GHz
                     "dominant_kernel_ncu": {"kernel": "conv_gemm2_kernel<256,false>", "tensor_pipe_active_pct": 97.9,
                                             "launch_us": 466.5, "dram_bytes": 588.5e6,
                                             "source": "profiles/r01f_conv_gemm2_full.txt"}},
        "state_finite": finite, "per_step_ms": [round(v, 3) for v in per_step],
    }


def gpu_reference_image(args, torch, dev):
    """The fair GPU comparator (SURVEY.md 2.1, BASELINE.md 3): the reference's OWN PyTorch loop run unchanged on the same B200 --
    restoration_algorithms.psgla (the unmodified reference when it is loadable, else the oracle's restatement) on device cuda,
    eager ops + cuDNN convolutions of the torch DnCNN (torch's default flags: TF32 convolutions allowed), same problem, same
    weights.  B = 1 is the reference's run shape; B = --image-chains is the same code on a batch (its ops broadcast)."""
    import psgla_b200 as P
    from oracle import image_oracle as io_
    H = args.image_size
    im = synthetic_image(torch, H, H, 0, dev)
    net = io_.DnCNN().to(dev)
    net.load_state_dict(P.lipschitz_dncnn_state_dict(0))
    net.eval()
    prob = io_.make_inpainting(im, prop=0.5, sigma=1.0, seed_ip=0, device=dev)
    s = 2.0 / 255.0
    kw = dict(alpha=torch.tensor(1.0, device=dev), lambd=torch.tensor(5.0, device=dev), sig_float=s, delta=s * s, n_inter=10,
              n_inter_mmse=10, seed=0)
    kind = "port"
    fn = lambda *a, **k: io_.psgla(*a, device=dev, **k)  # noqa: E731
    if _reference_available():
        from oracle import ref_loader
        ra = ref_loader.load_restoration_algorithms()
        fn, kind = (lambda *a, **k: ra.psgla(*a, device=dev, **k)), "reference"
    out = {"kind": kind, "flags": "torch defaults (cudnn.allow_tf32 = %s), eager, fp32 tensors" % torch.backends.cudnn.allow_tf32}
    for B, n_iter in ((1, 60), (args.image_chains, 20)):
        init = prob["init"].expand(B, -1, -1, -1).contiguous()
        with contextlib.redirect_stdout(sys.stderr), contextlib.redirect_stderr(open(os.devnull, "w")), torch.no_grad():
            fn(init, prob["data_grad"], net, n_iter=10, **kw)
            torch.cuda.synchronize()
            dt = float("inf")
            for _ in range(3):  # its eager loop is bound by the host's launch rate: best of three calls
                t0 = time.perf_counter()
                fn(init, prob["data_grad"], net, n_iter=n_iter, **kw)
                torch.cuda.synchronize()
                dt = min(dt, time.perf_counter() - t0)
        out["B%d" % B] = {"value": B * n_iter / dt, "unit": "image-iterations/s", "ms_per_iteration": dt / n_iter * 1e3,
                          "iterations": n_iter}
    return out


def bench_image_set(args, P, torch, rank, ws, dev):
    """BASELINE.json configs[4] as a whole job: a SET of CBSD-sized images (320 x 480), --set-chains chains per image, images dealt
    round-robin over the GPUs (psgla_b200.run_image_set), PSGLA with the DRUNet-architecture denoiser in statistics-only mode,
    per-image PSNR / SSIM / std reduced on the device and gathered on rank 0 -- the only communication of the job."""
    n_img, B, n_iter = args.set_images, args.set_chains, args.set_iters
    images = [synthetic_image(torch, args.drunet_h, args.drunet_w, 100 + i, "cpu")[0] for i in range(n_img)]
    den = P.DRUNet(pretrained=P.random_drunet_state_dict(0), device=dev)
    s = 5.0 / 255.0
    prm = dict(P.sampler_params("psgla", den="DRUNet", lambd=25.0, N=max(n_iter, 1000)), N=n_iter, n_inter=10, n_inter_mmse=10)

    def job():
        with contextlib.redirect_stdout(sys.stderr):
            return P.run_image_set(images, den, problem="inpainting", alg="psgla", n_chains=B, params=prm, seed=args.seed)

    small = dict(prm, N=11)
    with contextlib.redirect_stdout(sys.stderr):
        P.run_image_set(images[:ws], den, problem="inpainting", alg="psgla", n_chains=B, params=small, seed=args.seed)  # warm-up
    barrier(torch, P.dist)
    t0 = time.perf_counter()
    res = job()
    torch.cuda.synchronize()
    dt = time.perf_counter() - t0
    barrier(torch, P.dist)
    dt = P.dist.max_over_ranks(dt, dev)
    out = {"metric": "psgla_image_iterations_per_sec_drunet_image_set", "unit": "image-iterations/s",
           "value": n_img * B * n_iter / dt, "seconds": dt, "images": n_img, "chains_per_image": B, "iterations": n_iter,
           "config": {"workload": "%d synthetic %dx%d images x %d chains x %d PSGLA iterations, DRUNet, statistics-only mode, images "
                                  "round-robin over %d GPU(s), per-image metrics gathered on rank 0; wall clock incl. problem set-up"
                                  % (n_img, args.drunet_h, args.drunet_w, B, n_iter, ws)},
           "s": s}
    if rank == 0 and res:
        out["per_image"] = [{k: (round(v, 4) if isinstance(v, float) else v) for k, v in d.items()
                             if k in ("index", "psnr_mmse", "ssim_mmse", "psnr_chain_mean", "psnr_observation", "std_mean")} for d in res]
    return out


# ------------------------------------------------------------------------------------------------ CPU legs (oracle)
def _cpu_chain_worker(job):
    """One host core: the reference's single-chain Python loop (sampling_2D.py:48-72 / :21-45)."""
    alg, prior, y, n, seed, use_ref = job
    import numpy as np
    from oracle import gmm2d_oracle as o
    fn = None
    if use_ref:
        from oracle import ref_loader
        ns = ref_loader.load_sampling_2D()
        u2 = ref_loader.load_utils_2D()
        mu, Sig, pi = u2.gaussian_mixt_example(prior)
        D = u2.Theorical_MMSE(mu, Sig, pi)
        np.random.seed(seed)
        prm = GMM_ALGS[alg]
        t0 = time.perf_counter()
        if alg == "psgla":
            ns.SnoPnP_ULA(n + 1, np.array(y), np.array(y), prm["delta"], np.eye(2), 1, D, prm["alpha"])
        else:
            ns.PnP_ULA(n + 1, np.array(y), np.array(y), prm["delta"], np.eye(2), 1, D, prm["epsilon"], prm["alpha"])
        return time.perf_counter() - t0
    mu, Sig, pi = o.gaussian_mixt_example(prior)
    D = o.theorical_mmse(mu, Sig, pi)
    prm = GMM_ALGS[alg]
    noise = np.random.default_rng(seed).standard_normal((n, 2))
    t0 = time.perf_counter()
    if alg == "psgla":
        fn = o.snopnp_ula(n + 1, np.array(y), np.array(y), prm["delta"], np.eye(2), 1, D, prm["alpha"], noise=noise)
    else:
        fn = o.pnp_ula(n + 1, np.array(y), np.array(y), prm["delta"], np.eye(2), 1, D, prm["epsilon"], prm["alpha"], noise=noise)
    assert fn.shape == (n + 1, 2)
    return time.perf_counter() - t0


def _reference_available():
    from oracle import ref_loader
    return ref_loader.reference_available()


def cpu_baseline_gmm2d(n_steps):
    use_ref = _reference_available()
    dt = _cpu_chain_worker(("psgla", "symetric_gaussians", (0.0, -2.0), n_steps, 0, use_ref))
    out = {"value": n_steps / dt, "unit": "chain-steps/s", "cores": 1, "kind": "reference" if use_ref else "port",
           "sample": "1 chain x %d PSGLA steps, symetric_gaussians prior, y=(0,-2), float64 Python loop "
                     "(the reference is single-threaded; independent chains scale with cores)" % n_steps}
    # the same algorithm as compiled C (oracle/gmm2d_oracle.c, float64, operation for operation): what one host core can do
    # once the interpreter is out of the way -- the fairer yardstick for the kernel, reported beside the reference's own speed
    try:
        import numpy as np
        from oracle import c_oracle, gmm2d_oracle as o
        prior = o.gaussian_mixt_example("symetric_gaussians")
        y = np.array([0.0, -2.0])
        n_c = 4000000
        c_oracle.run_chain("psgla", 1000, y, y, o.PSGLA_DELTA, np.eye(2), 1, prior, 1.0, o.PSGLA_ALPHA, seed=1)
        t0 = time.perf_counter()
        c_oracle.run_chain("psgla", n_c, y, y, o.PSGLA_DELTA, np.eye(2), 1, prior, 1.0, o.PSGLA_ALPHA, seed=0)
        dt_c = time.perf_counter() - t0
        out["c_port"] = {"value": n_c / dt_c, "unit": "chain-steps/s", "cores": 1, "kind": "port",
                         "sample": "1 chain x %d PSGLA steps, oracle/gmm2d_oracle.c (gcc -O2, float64, own Box-Muller stream)" % n_c}
    except Exception as exc:  # noqa: BLE001
        out["c_port"] = {"error": repr(exc)[:200]}
    return out


def cpu_baseline_image(args, n_iter=12):
    """The reference's psgla loop on the host cores with the fp32 torch DnCNN of the oracle (same weights, same problem)."""
    import torch
    import psgla_b200 as P
    from oracle import image_oracle as io_
    H = args.image_size
    im = synthetic_image(torch, H, H, 0, "cpu")
    net = io_.DnCNN()
    net.load_state_dict(P.lipschitz_dncnn_state_dict(0))
    net.eval()
    prob = io_.make_inpainting(im, prop=0.5, sigma=1.0, seed_ip=0, device="cpu")
    s = 2.0 / 255.0
    kw = dict(alpha=torch.tensor(1.0), lambd=torch.tensor(5.0), sig_float=s, delta=s * s, n_inter=10, n_inter_mmse=10, seed=0)
    fn, kind = io_.psgla, "port"
    if _reference_available():
        from oracle import ref_loader
        ra = ref_loader.load_restoration_algorithms()
        fn, kind = (lambda *a, **k: ra.psgla(*a, device="cpu", **k)), "reference"
    else:
        fn = lambda *a, **k: io_.psgla(*a, device="cpu", **k)  # noqa: E731
    with contextlib.redirect_stdout(sys.stderr), contextlib.redirect_stderr(open(os.devnull, "w")):
        fn(prob["init"], prob["data_grad"], net, n_iter=10, **kw)  # warm-up (n_iter >= 10: restoration_algorithms.py:246)
        t0 = time.perf_counter()
        fn(prob["init"], prob["data_grad"], net, n_iter=n_iter, **kw)
        dt = time.perf_counter() - t0
    return {"value": n_iter / dt, "unit": "image-iterations/s", "cores": torch.get_num_threads(), "kind": kind,
            "sample": "%d PSGLA iterations, 1 chain, %dx%dx3, fp32 torch DnCNN on the host" % (n_iter, H, H)}


def cpu_baseline_drunet(args, n_iter=10):
    """The reference's psgla loop on the host cores with the fp32 torch DRUNet of the oracle (same weights, same problem)."""
    import torch
    import psgla_b200 as P
    from oracle import image_oracle as io_
    H, Wd = args.drunet_h, args.drunet_w
    im = synthetic_image(torch, H, Wd, 1, "cpu")
    net = io_.DRUNet()
    net.load_state_dict(P.random_drunet_state_dict(0))
    net.eval()
    prob = io_.make_inpainting(im, prop=0.5, sigma=1.0, seed_ip=0, device="cpu")
    s = 5.0 / 255.0
    kw = dict(alpha=torch.tensor(1.0), lambd=torch.tensor(25.0), sig_float=s, delta=s * s, n_inter=10, n_inter_mmse=10, seed=0)
    kind = "port"
    if _reference_available():
        from oracle import ref_loader
        ra = ref_loader.load_restoration_algorithms()
        fn, kind = (lambda *a, **k: ra.psgla(*a, device="cpu", **k)), "reference"
    else:
        fn = lambda *a, **k: io_.psgla(*a, device="cpu", **k)  # noqa: E731
    with contextlib.redirect_stdout(sys.stderr), contextlib.redirect_stderr(open(os.devnull, "w")):
        t0 = time.perf_counter()
        fn(prob["init"], prob["data_grad"], net, n_iter=n_iter, **kw)
        dt = time.perf_counter() - t0
    return {"value": n_iter / dt, "unit": "image-iterations/s", "cores": torch.get_num_threads(), "kind": kind,
            "sample": "%d PSGLA iterations, 1 chain, %dx%dx3, fp32 torch DRUNet on the host" % (n_iter, H, Wd)}


def run_reference(args):
    """--impl reference: the reference's CPU algorithm for the headline workload on every host core."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    import multiprocessing as mp
    cores = os.cpu_count() or 1
    use_ref = _reference_available()
    n = args.ref_chain_steps
    K, W = args.steps, args.warmup
    ctx = mp.get_context("spawn")
    times = []
    with ctx.Pool(cores) as pool:
        for k in range(W + K):
            prior, y, alg = CELLS[k % len(CELLS)]
            jobs = [(alg, prior, y, n, 1000 * k + c, use_ref) for c in range(cores)]
            dt = max(pool.map(_cpu_chain_worker, jobs))  # slowest core's loop time; process start-up is not counted
            if k >= W:
                times.append(dt)
    total = sum(times)
    value = cores * n * K / total
    kind = "reference" if use_ref else "port"
    sample = "%d independent chains (one per host core) x %d steps per bench step, cells cycled as in the GPU arm" % (cores, n)
    line = {
        "impl": "reference", "metric": "langevin_chain_steps_per_sec_2d_gmm", "value": value, "unit": "chain-steps/s",
        "n_gpus": args.gpus, "steps": K, "warmup": W, "ms_per_step": total / K * 1e3, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": config_block(args),
        "cpu_baseline": {"value": value, "unit": "chain-steps/s", "cores": cores, "kind": kind, "sample": sample},
        "e2e": {"value": value, "unit": "chain-steps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    if not args.skip_image:
        try:
            line["image"] = {"impl": "reference", "metric": "psgla_image_iterations_per_sec_256x256_dncnn",
                             **cpu_baseline_image(args, n_iter=12)}
        except Exception as exc:  # noqa: BLE001
            line["image"] = {"impl": "reference", "error": repr(exc)[:200]}
    emit(line)


def config_block(args):
    return {"workload": "2D GMM posterior sampling, 18 cells = 3 priors x 3 observations x {PSGLA, PnP-ULA} "
                        "(sampling_2D.py:83-91,130-131), %d chains x %d steps per cell per GPU, one cell per bench step"
                        % (args.chains, args.chain_steps),
            "chains_per_gpu": args.chains, "steps_per_chain": args.chain_steps, "cells": len(CELLS),
            "rng": "in-kernel Philox4x32-10 + Box-Muller, subsequence = global chain id",
            "sharding": "chains split over GPUs, no per-step communication; NCCL gather of finals for W2; the `strong` block of the "
                        "line runs the same 18 cells with 10^6 chains per cell IN TOTAL, sharded",
            "l2": "256 MiB flush between timed steps (state lives in registers; HBM sees 16 B per chain per step of the bench)"}


# ------------------------------------------------------------------------------------------------ main
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=18)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--chains", type=int, default=1000000, help="2D chains per GPU")
    ap.add_argument("--chain-steps", type=int, default=10000, help="Langevin steps per chain per cell")
    ap.add_argument("--image-chains", type=int, default=32, help="independent PSGLA chains per GPU")
    ap.add_argument("--image-size", type=int, default=256)
    ap.add_argument("--image-steps", type=int, default=20)
    ap.add_argument("--drunet-chains", type=int, default=64, help="independent DRUNet-PSGLA chains per GPU (configs[4])")
    ap.add_argument("--drunet-h", type=int, default=320)
    ap.add_argument("--drunet-w", type=int, default=480)
    ap.add_argument("--drunet-steps", type=int, default=6)
    ap.add_argument("--skip-drunet", action="store_true")
    ap.add_argument("--strong-chains", type=int, default=1000000, help="2D chains per cell IN TOTAL for the strong-scaling block")
    ap.add_argument("--strong-streams", type=int, default=3, help="cells a rank keeps in flight in the strong-scaling block")
    ap.add_argument("--emulate-world", type=int, default=0, help="1 GPU only: time rank 0's shard of an N-way strong split")
    ap.add_argument("--skip-strong", action="store_true")
    ap.add_argument("--set-images", type=int, default=8, help="image-set block: number of 320x480 images")
    ap.add_argument("--set-chains", type=int, default=64)
    ap.add_argument("--set-iters", type=int, default=24)
    ap.add_argument("--skip-set", action="store_true")
    ap.add_argument("--skip-gpu-reference", action="store_true")
    ap.add_argument("--ref-chain-steps", type=int, default=20000, help="--impl reference: steps per core per bench step")
    ap.add_argument("--cpu-sample-steps", type=int, default=100000, help="cpu_baseline sample: steps of one CPU chain")
    ap.add_argument("--skip-image", action="store_true")
    ap.add_argument("--only-image", action="store_true", help="profiling aid: shrink the 2D part to a token run")
    ap.add_argument("--skip-cpu", action="store_true")
    ap.add_argument("--seed", type=int, default=0)
    ap.add_argument("--dump-outputs", metavar="DIR", help="write what the last timed step of the 2D block and of the image blocks computed to "
                                                        "DIR/<name>.npy (see the module docstring)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs applies to the GPU path, not to --impl reference")
    args.warmup = max(args.warmup, 0)
    capture_stdout()
    if args.only_image:
        args.chains, args.chain_steps, args.steps, args.skip_cpu, args.skip_strong = 4096, 16, 1, True, True

    if args.impl == "reference":
        run_reference(args)
        return

    import torch
    import psgla_b200 as P
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the product has no CPU path (use --impl reference for the CPU arm)")
    rank, ws, local = P.dist.init_from_env("nccl")
    if rank != 0:
        args.dump_outputs = None  # only rank 0 writes its chains' outputs, so the other ranks keep none
    if ws != max(args.gpus, 1):
        log("warning: --gpus %d but WORLD_SIZE %d; using WORLD_SIZE" % (args.gpus, ws))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    arch = P._lib.lib().psgla_device_arch()
    if arch < 100:
        raise SystemExit("libpsgla_b200 targets sm_100a; device reports sm_%d" % arch)
    peaks = measured_peaks()
    W = max(args.warmup, 3)
    if W != args.warmup:
        log("warm-up raised to 3 steps (timing rule)")
        args.warmup = W

    fp32_peak = measure_fp32_peak(P, torch, dev)
    mix = measure_mix_ceiling(P, torch, dev)
    sampler = ClockSampler(local)  # clocks during the headline (2D) timed regions ...
    if rank == 0:
        sampler.start()
    g = bench_gmm2d(args, P, torch, rank, ws, dev)
    strong = None if args.skip_strong else bench_gmm2d_strong(args, P, torch, rank, ws, dev)
    clocks = sampler.stop() if rank == 0 else None
    cfg0 = bench_gmm2d_config0(args, P, torch, dev) if (rank == 0 and not args.only_image) else None
    sampler = ClockSampler(local)  # ... and during the image blocks (tensor-core work under the power cap: lower clocks)
    if rank == 0:
        sampler.start()
    img = dru = deb = iset = None
    if not args.skip_image:
        img = bench_image(args, P, torch, rank, ws, dev, peaks)
        deb = bench_image_deblur(args, P, torch, rank, ws, dev, peaks)
        if not args.skip_drunet:
            dru = bench_image_drunet(args, P, torch, rank, ws, dev, peaks)
            if not args.skip_set:
                iset = bench_image_set(args, P, torch, rank, ws, dev)
    clocks_image = sampler.stop() if rank == 0 else None

    if rank != 0:
        if ws > 1:
            import torch.distributed as dist
            dist.destroy_process_group()
        return
    K = args.steps
    achieved_tflops = g["flop"] * ws / (g["total_ms"] * 1e-3) / 1e12
    line = {
        "metric": "langevin_chain_steps_per_sec_2d_gmm", "value": g["value"], "unit": "chain-steps/s", "n_gpus": ws,
        "steps": K, "warmup": args.warmup, "ms_per_step": g["total_ms"] / K, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic", "config": config_block(args),
        "clocks": clocks, "clocks_image_blocks": clocks_image,
        "e2e": {"value": g["e2e_value"], "unit": "chain-steps/s", "h2d_bytes_per_step": g["h2d"],
                "d2h_bytes_per_step": g["d2h"]},
        "gpu_launches": K * g["launches_per_step"],
        "roofline": {"kernel": "gmm2d_lean_kernel<ALG,STRUCT,4,64,16,true> (one chain per thread, 4 Philox blocks = 8 steps per round; "
                               "%d launch(es) per step)" % g["launches_per_step"],
                     "bound": "fp32",
                     "achieved": achieved_tflops / ws, "peak": fp32_peak["ffma"], "unit": "TFLOP/s",
                     "frac": achieved_tflops / ws / fp32_peak["ffma"],
                     "peak_source": "measured on this GPU in this run: FFMA-only probe (psgla_selftest_fp32_rate), burst; FFMA2 probe %.1f, "
                                    "nominal %.1f.  Algorithmic 82/88 flop + 7 MUFU per chain-step (SURVEY 8d), Philox INT work not counted"
                                    % (fp32_peak["ffma2"], FP32_PEAK_TFLOPS_NOMINAL),
                     "frac_of_nominal_peak": achieved_tflops / ws / FP32_PEAK_TFLOPS_NOMINAL,
                     "mufu_gops": g["value"] / ws * MUFU_PER_CHAIN_STEP / 1e9,
                     # the bound that actually binds: FMA-pipe cycles the issued mix needs (FP32 1 cycle, IMAD.WIDE.U32 4 cycles per
                     # warp instruction, measured by scripts/pipe_rates.py) over the SM-cycles the step took at the sampled clock
                     "fma_pipe": {"cycles_needed_per_warp_step": g["pipe_cycles"],
                                  "cycles_taken_per_warp_step": (clocks or {}).get("sm_mhz") and
                                  (clocks["sm_mhz"] * 1e6 * 148 * 4 * 32) / (g["value"] / ws),
                                  "note": "taken = sm_clock x 592 SM sub-partitions x 32 lanes / (chain-steps/s); needed / taken = FMA-pipe utilisation"},
                     # the bound that binds: the issue ceiling of the kernel's own instruction mix, measured by a dependency-free probe
                     # of the same mix on this GPU; a timed step = one cell, so the ceiling of the run is the harmonic mean over its cells
                     "instruction_mix": {"ceiling": len(g["cells_nf"]) / sum(1.0 / mix[nf] for nf in g["cells_nf"]),
                                         "unit": "chain-steps/s per GPU",
                                         "frac": (g["value"] / ws) / (len(g["cells_nf"]) / sum(1.0 / mix[nf] for nf in g["cells_nf"])),
                                         "per_fp32_count": {str(k): v for k, v in mix.items()},
                                         "note": "6 MUFU + 9 IMAD.WIDE.U32 + NF FP32 + 10 LOP3 + 2 I2FP per chain-step as independent chains "
                                                 "(psgla_selftest_pipe_rate 100 + NF), NF = 21 / 23 (diagonal cells, PSGLA / PnP-ULA), 26 / 28 (cross prior); "
                                                 "the probe's own loop issues ~8 % more LOP3 / IADD than the kernel, so it estimates the ceiling "
                                                 "slightly from below and frac can read a little above 1"},
                     "launch_ms": g["total_ms"] / K / g["launches_per_step"],
                     # dram__bytes_read.sum + dram__bytes_write.sum of one launch, ncu --set full (profiles/r02_gmm2d_lean_full.txt)
                     "traffic": 8.03e6 if args.chains == 1000000 else None,
                     "traffic_source": "profiles/r02_gmm2d_lean_full.txt (8.06 / 8.01 MB read, 0 written back to DRAM within the launch: "
                                       "8 B per chain in, the 8 B per chain out stay in L2)"},
        "w2_squared_to_true_posterior": g["w2"],
    }
    if strong is not None:
        strong["value_over_weak_value"] = strong["value"] / g["value"] if not strong.get("emulated_world") else None
        line["strong"] = strong
    if cfg0 is not None:
        line["config0_single_chain"] = cfg0
    if img is not None:
        line["image"] = img
    if deb is not None:
        line["image_deblur"] = deb
    if dru is not None:
        line["image_drunet"] = dru
    if iset is not None:
        line["image_set"] = iset
    if ws == 1 and not args.skip_cpu:
        line["cpu_baseline"] = cpu_baseline_gmm2d(args.cpu_sample_steps)
        if img is not None:
            try:
                img["cpu_baseline"] = cpu_baseline_image(args)
            except Exception as exc:  # noqa: BLE001
                img["cpu_baseline"] = {"error": repr(exc)[:200]}
        if dru is not None:
            try:
                dru["cpu_baseline"] = cpu_baseline_drunet(args)
            except Exception as exc:  # noqa: BLE001
                dru["cpu_baseline"] = {"error": repr(exc)[:200]}
        if cfg0 is not None and "value" in line["cpu_baseline"]:
            cfg0["reference_us_per_step_here"] = 1e6 / line["cpu_baseline"]["value"]
        if img is not None and not args.skip_gpu_reference:
            try:
                img["gpu_reference"] = gpu_reference_image(args, torch, dev)
            except Exception as exc:  # noqa: BLE001
                img["gpu_reference"] = {"error": repr(exc)[:200]}
    # the image half of BASELINE.json's metric, compact, as the LAST key of the line (the nested blocks above hold the detail)
    if img is not None:
        summ = {"dncnn_psgla_image_iterations_per_sec": img["value"], "dncnn_psgla_e2e": img["e2e"]["value"],
                "dncnn_chains_per_gpu": args.image_chains, "dncnn_hidden_conv_frac_of_burst_bf16_peak": img["roofline"]["frac"],
                "dncnn_whole_iteration_frac_of_sustained_bf16_peak": img["whole_iteration_frac"],
                "dncnn_single_chain_iterations_per_sec": img["single_chain_iterations_per_sec"], "n_gpus": ws}
        if deb is not None:
            summ["dncnn_pnpula_deblur_image_iterations_per_sec"] = deb["value"]
        if dru is not None:
            summ["drunet_psgla_image_iterations_per_sec"] = dru["value"]
            summ["drunet_whole_iteration_frac_of_sustained_bf16_peak"] = dru["roofline"]["frac"]
        if iset is not None:
            summ["drunet_image_set_image_iterations_per_sec"] = iset["value"]
        if "cpu_baseline" in img and "value" in img["cpu_baseline"]:
            summ["cpu_reference_image_iterations_per_sec"] = img["cpu_baseline"]["value"]
        if "gpu_reference" in img and "B1" in img["gpu_reference"]:
            summ["gpu_reference_B1_image_iterations_per_sec"] = img["gpu_reference"]["B1"]["value"]
        line["image_summary"] = summ
    if args.dump_outputs:
        write_outputs(args.dump_outputs)
    emit(line)
    if ws > 1:
        import torch.distributed as dist
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
