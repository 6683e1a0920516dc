#!/usr/bin/env python
"""Same-box A/B of two builds of libpsgla_b200.so (boxes differ by a few per cent, so two gpurun calls cannot be compared):
   python scripts/ab_lib.py libA.so libB.so [rounds] -- scripts/probe.py [args]
runs the probe alternately with each library (A B A B ...), one process per run, and prints each run's last stdout line."""
import os, runpy, subprocess, sys

if sys.argv[1] == "--run":
    sys.path.insert(0, os.getcwd())
    from importlib import import_module
    import psgla_b200  # noqa: F401
    import_module("psgla_b200._lib").LIB_PATH = os.path.abspath(sys.argv[2])
    sys.argv = sys.argv[3:]
    runpy.run_path(sys.argv[0], run_name="__main__")
else:
    sep = sys.argv.index("--")
    libs = sys.argv[1:3]
    rounds = int(sys.argv[3]) if sep > 3 else 2
    for r in range(rounds):
        for name, lib in zip("AB", libs):
            out = subprocess.run([sys.executable, __file__, "--run", lib] + sys.argv[sep + 1:], capture_output=True, text=True)
            # the probe's result is its last stdout line (bench.py logs to stderr); a run that printed nothing there shows its
            # last stderr line instead
            lines = [l for l in out.stdout.splitlines() if l.strip()] or [l for l in out.stderr.splitlines() if l.strip()]
            print("%s %s: %s" % (name, os.path.basename(lib), lines[-1] if lines else "(no output, rc %d)" % out.returncode), flush=True)
