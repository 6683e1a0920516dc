"""not-gpu: the C ABI of the device-wide convergence diagnostics (csrc/mcmc_diag_large.cu): declared and bound, its workspace
formula, and every bad argument rejected on the host before any CUDA call."""
import os
import re

import pytest

GROUP_DRAWS, MAX_S, MAX_SEGMENTS, MAX_LAGS = 1 << 28, 2 ** 31 - 1, 65535, 1 << 22
ELEM_BYTES = 152  # sizeof(LgElem)


@pytest.fixture(scope="module")
def built():
    import __graft_entry__ as g
    g.build()
    import psgla_b200
    return psgla_b200


def _al(b):
    return (b + 255) // 256 * 256


def _workspace(N, M, E):
    """The layout of mcmc_diag_large.cu, restated: head; keys and payloads, ping-pong; radix histograms; odd N: the middle
    draws, ping-pong; per-element state; per-chain moments; one round's autocovariances; the largest round's lag partials."""
    n = N // 2
    S, Mp, odd = 2 * M * n, 2 * M, N & 1
    G = min(E, max(1, GROUP_DRAWS // S), MAX_SEGMENTS)
    rounds, nxt, t = [], 1, 1
    for r in range(512):
        B = min(32 << min(r, 20), MAX_LAGS, n - nxt)
        if B < 1:
            break
        rounds.append((B, max(4096, 16 * B)))
        end = nxt + B - 1
        while t < n - 3 and t + 2 <= end:
            t += 2
        if not t < n - 3:
            break
        nxt = t + 1
    part = max([-(-S // tile) * B for B, tile in rounds], default=0)
    lags = max([B for B, _ in rounds], default=1)
    nb = -(-S // 4096)
    total = 256 + 4 * _al(G * S * 4) + _al(G * 256 * nb * 4)
    total += 2 * _al(G * M * 4) if odd else 0
    total += _al(G * ELEM_BYTES) + _al(G * Mp * 16) + _al(G * lags * 8) + _al(G * part * 8)
    return total


def test_header_declares_the_large_diagnostics(built):
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    with open(os.path.join(root, "include", "psgla_b200.h")) as f:
        header = f.read()
    for name in ("psgla_mcmc_diag_large_workspace_bytes", "psgla_mcmc_diag_large"):
        assert re.search(r"\b%s\(" % name, header) and name in built._lib.SIGNATURES
    assert callable(built.mcmc_diagnostics_large) and built.diagnostics.MAX_DRAWS_LARGE == MAX_S


@pytest.mark.parametrize("N,M,E", [(1000, 8, 196608), (10000, 8, 196608), (2050, 8, 1), (16386, 1, 3), (4, 4097, 3),
                                   (5, 4097, 70000), (400, 20000, 2), (1001, 1000000, 2), (20001, 2, 3), (1 << 17, 8, 300)])
def test_workspace_formula(built, N, M, E):
    assert built._lib.lib().psgla_mcmc_diag_large_workspace_bytes(N, M, E) == _workspace(N, M, E)


def test_workspace_is_bounded(built):
    f = built._lib.lib().psgla_mcmc_diag_large_workspace_bytes
    # groups of 2^28 split draws: about 17 bytes per draw, whatever E is
    assert f(1000, 8, 196608) == f(1000, 8, 10 ** 9 // 3) < 18 * GROUP_DRAWS
    assert f(2 ** 31 - 1, 1, 1) < 40e9  # one element of S = 2^31 - 2


def test_workspace_zero_out_of_range(built):
    f = built._lib.lib().psgla_mcmc_diag_large_workspace_bytes
    assert f(2 ** 31 - 1, 1, 1) > 0 and f(2, 2 ** 30 - 1, 1) == 0 and f(4, (2 ** 31 - 1) // 4, 1) > 0
    for N, M, E in ((2 ** 31 + 1, 1, 1), (4, 2 ** 29, 1), (1 << 62, 1, 1), (4, 1 << 40, 1), (3, 8, 1), (-4, 8, 1),
                    (100, 0, 1), (100, 4, 0), (100, 4, 1 << 40)):
        assert f(N, M, E) == 0, (N, M, E)


def test_argument_errors_without_gpu(built):
    """psgla_mcmc_diag_large rejects each bad argument on the host before any CUDA call (fake pointers are never
    dereferenced)."""
    lib = built._lib.lib()
    fake = 0x1000

    def call(draws=fake, N=100, M=4, E=10, ws=fake, ws_bytes=None, r=fake, b=fake, t=fake):
        if ws_bytes is None:
            ws_bytes = lib.psgla_mcmc_diag_large_workspace_bytes(N, M, E) or 1 << 20
        return lib.psgla_mcmc_diag_large(draws, N, M, E, ws, ws_bytes, r, b, t, None)

    for kw in (dict(draws=None), dict(ws=None), dict(r=None), dict(b=None), dict(t=None)):
        assert call(**kw) == -1 and b"null" in lib.psgla_last_error(), kw
    for kw, word in ((dict(N=3), b"n_draws"), (dict(N=-1), b"n_draws"), (dict(M=0), b"n_chains"), (dict(M=-3), b"n_chains"),
                     (dict(E=0), b"n_elem"), (dict(E=1 << 40), b"n_elem")):
        assert call(**kw) == -1 and word in lib.psgla_last_error(), kw
    for N, M in ((2 ** 31 + 1, 1), (4, 2 ** 29), (1 << 40, 2), (1 << 62, 1 << 40)):
        assert call(N=N, M=M) == -1, (N, M)
        assert b"2^31 - 1" in lib.psgla_last_error() and b"n_draws" in lib.psgla_last_error()
    need = lib.psgla_mcmc_diag_large_workspace_bytes(100, 4, 10)
    assert call(ws_bytes=need - 1) == -4 and b"workspace" in lib.psgla_last_error()
    assert call(ws=fake + 16) == -1 and b"aligned" in lib.psgla_last_error()
