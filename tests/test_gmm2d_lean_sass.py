"""not-gpu: what ptxas made of the 2D throughput kernel, read back from the built object.  gmm2d_lean_kernel is bound by the
rate at which the SM issues its instruction mix, and each Philox IMAD.WIDE.U32 costs about 4 issue slots against 1 for the
other instructions.  With Philox's launch-uniform round-2 words read from the kernel's parameters, the loop of every
instantiation issues the 16 products per counter block that rounds 3-10 need and no more: 8 per chain-step."""
import collections
import os
import re
import shutil
import subprocess

import pytest


@pytest.fixture(scope="module")
def gmm2d_obj():
    import __graft_entry__ as g
    g.build()
    import psgla_b200
    return os.path.join(os.path.dirname(psgla_b200._lib.LIB_PATH), "build", "gmm2d.o")


def _cuobjdump(*args):
    tool = shutil.which("cuobjdump") or "/usr/local/cuda/bin/cuobjdump"
    if not os.path.exists(tool):
        pytest.skip("cuobjdump not available")
    return subprocess.run([tool, *args], capture_output=True, text=True, check=True).stdout


def _loop_opcodes(body):
    """Opcode counts of the kernel's longest backward-branch loop (the rounds loop)."""
    ins = [(int(a, 16), t) for a, t in re.findall(r"/\*([0-9a-f]{4,})\*/\s+([^;]*);", body)]
    loops = [(int(m.group(1), 16), a) for a, t in ins for m in [re.search(r"\bBRA\S*\s.*?(0x[0-9a-f]+)", t)]
             if m and int(m.group(1), 16) < a]
    lo, hi = max(loops, key=lambda l: l[1] - l[0])
    return collections.Counter(re.sub(r"^@!?U?P\w+\s+", "", t).split()[0] for a, t in ins if lo <= a <= hi)


def test_lean_loop_issues_eight_philox_products_per_step(gmm2d_obj):
    sass = _cuobjdump("-sass", gmm2d_obj)
    kernels = re.findall(r"Function : (\S*gmm2d_lean_kernel\S*)\n(.*?)(?=\n\s*Function : |\Z)", sass, flags=re.S)
    assert len(kernels) == 6  # PSGLA / PnP-ULA x constants structure 0 / 1 / 2
    for fn, body in kernels:
        ops = _loop_opcodes(body)
        steps = ops["MUFU.SIN"]  # one Box-Muller pair, i.e. one chain-step, per sine
        assert steps > 0, fn
        assert ops["IMAD.WIDE.U32"] <= 8 * steps, (fn, ops["IMAD.WIDE.U32"] / steps)
        assert ops["UIMAD.WIDE.U32"] == 0, fn
    usage = re.findall(r"Function (\S*gmm2d_lean_kernel\S*):\s*\n?\s*REG:(\d+) STACK:(\d+) SHARED:\d+ LOCAL:(\d+)",
                       _cuobjdump("-res-usage", gmm2d_obj))
    assert len(usage) == 6
    for fn, reg, stack, local in usage:
        assert int(reg) <= 64 and int(stack) == 0 and int(local) == 0, (fn, reg, stack, local)
