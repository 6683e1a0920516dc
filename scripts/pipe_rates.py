#!/usr/bin/env python
"""Measured per-SM issue rates of the instruction classes the 2D chain kernel mixes (development aid).
    python scripts/pipe_rates.py > gpurun_out/pipe_rates.txt"""
import ctypes as C
import os
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch  # noqa: E402
import psgla_b200 as P  # noqa: E402

NAMES = ["IMAD.WIDE.U32", "IMAD.HI.U32", "IMAD (lo)", "LOP3", "MUFU.EX2", "I2FP.F32.U32", "FFMA", "MUFU.SIN (+FMUL.RZ)",
         "IMAD.WIDE + FFMA 1:1", "MUFU.EX2 + IMAD.WIDE 1:1", "MUFU.EX2 + 4 FFMA", "chain-step mix (6M 9W 19F 10L 2C)",
         "DFMA.RM", "IMAD + DFMA.RM + LOP3", "DFMA.RM + FFMA 1:1"]
# the chain-step mix with the integer Philox multiply (100 + NF) and with the FP64-pipe one (200 + NF), NF = FP32 slots per step
MIXES = [(100 + nf, "mix, IMAD.WIDE form, NF = %d" % nf) for nf in (21, 23, 26, 28, 30)] + \
        [(200 + nf, "mix, FP64-pipe form, NF = %d" % nf) for nf in (21, 23, 26, 28, 30)]
lib = P._lib.lib()
scratch = torch.empty(148 * 8 * 256, dtype=torch.float32, device="cuda")
sms = torch.cuda.get_device_properties(0).multi_processor_count
print("# %s, %d SMs; %s" % (torch.cuda.get_device_name(0), sms, subprocess.run(
    ["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm,clocks.sm", "--format=csv,noheader", "-i", "0"],
    capture_output=True, text=True).stdout.strip() or "nvidia-smi unavailable"))
try:
    clk = torch.cuda.clock_rate() * 1e6  # current SM clock (needs pynvml)
except Exception:
    clk = 1.965e9  # the B200's boost clock
for mode, name in list(enumerate(NAMES)) + MIXES:
    ops = C.c_double()
    best = None
    for rep in range(3):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        P._lib.check(lib.psgla_selftest_pipe_rate(mode, 20000, 8, scratch.data_ptr(), C.byref(ops), None), "pipe_rate")
        e1.record()
        torch.cuda.synchronize()
        t = e0.elapsed_time(e1) * 1e-3
        best = t if best is None else min(best, t)
    per_s = ops.value / best
    mix = mode == 11 or mode >= 100
    print("%-36s %8.2f Gop/s/SM  = %6.2f thread-instr/clk/SM at %.2f GHz%s"
          % (name, per_s / sms / 1e9, per_s / sms / clk, clk / 1e9,
             "  -> %.1f SM-sub-partition cycles per warp-step" % (clk * 4 * 32 / (per_s / sms)) if mix else ""), flush=True)
