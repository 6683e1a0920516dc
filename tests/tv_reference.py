"""TEST INFRASTRUCTURE ONLY -- plain-PyTorch restatement of deepinv's ``TVDenoiser``, the fourth denoiser of the reference's
image driver (sampling_images.py:139-140).

Parity status: deepinv 0.2.1 is neither vendored nor installed, so the algorithm is restated from its published definition
and is PARITY UNPINNED against deepinv itself.  ``tests/test_tv_host.py`` checks that the restatement solves the problem it
claims to (adjoint, primal-dual gap).  One deliberate difference: the stopping test runs per chain (per batch entry), and a
chain that meets it keeps that iteration's state while the others go on; for one chain -- every run the reference makes --
this is deepinv's rule.

Dtype-generic: the state follows y's dtype, so tests run it in fp64 as well as in the fp32 of the reference.  It plugs into
``oracle.image_oracle.psgla`` / ``pnp`` like the other oracle denoisers (``forward(y, ths)``).
"""
from __future__ import annotations

import torch


def nabla(x):
    """Forward differences of [B,C,H,W] -> [B,C,H,W,2]: component 0 along H, 1 along W, 0 on the last row / column."""
    u = torch.zeros(tuple(x.shape) + (2,), dtype=x.dtype, device=x.device)
    u[:, :, :-1, :, 0] = x[:, :, 1:] - x[:, :, :-1]
    u[:, :, :, :-1, 1] = x[..., 1:] - x[..., :-1]
    return u


def nabla_adjoint(u):
    """The exact adjoint of ``nabla``."""
    x = torch.zeros(tuple(u.shape[:-1]), dtype=u.dtype, device=u.device)
    x[:, :, :-1] -= u[:, :, :-1, :, 0]
    x[:, :, 1:] += u[:, :, :-1, :, 0]
    x[..., :-1] -= u[..., :-1, 1]
    x[..., 1:] += u[..., :-1, 1]
    return x


def tv(x):
    """Isotropic TV per channel and pixel: sum ||nabla x||_2 over the last axis."""
    return torch.sqrt((nabla(x) ** 2).sum(-1)).sum()


class TVDenoiser:
    """deepinv's ``TVDenoiser(verbose=False, tau=0.01, rho=1.99, n_it_max=1000, crit=1e-5)``: over-relaxed Chambolle-Pock for
    argmin_x 1/2 ||x - y||^2 + ths TV(x), sigma = 1 / (8 tau), warm-started from the previous call's (x2, u2)."""

    def __init__(self, verbose=False, tau=0.01, rho=1.99, n_it_max=1000, crit=1e-5):
        self.verbose, self.tau, self.rho, self.n_it_max, self.crit = verbose, tau, rho, n_it_max, crit
        self.sigma = 1 / tau / 8
        self.restart = True
        self.x2 = self.u2 = None
        self.last_iterations = None  # per chain, of the last call
        self.calls = []              # last_iterations of every call

    def reset(self):
        self.restart = True

    def forward(self, y, ths):
        if self.restart or self.x2 is None or self.x2.shape != y.shape:
            self.x2 = y.clone()
            self.u2 = torch.zeros(tuple(y.shape) + (2,), dtype=y.dtype, device=y.device)
            self.restart = False
        x2, u2 = self.x2, self.u2
        B = y.shape[0]
        active = torch.ones(B, dtype=torch.bool, device=y.device)
        iters = torch.full((B,), self.n_it_max, dtype=torch.int64)
        for k in range(self.n_it_max):
            x_prev = x2
            x = (x2 - self.tau * nabla_adjoint(u2) + self.tau * y) / (1 + self.tau)
            u = u2 + self.sigma * nabla(2 * x - x2)
            u = u / torch.clamp(torch.sqrt((u ** 2).sum(-1)) / ths, min=1.0).unsqueeze(-1)
            a4 = active[:, None, None, None]
            x2 = torch.where(a4, x2 + self.rho * (x - x2), x2)
            u2 = torch.where(a4[..., None], u2 + self.rho * (u - u2), u2)
            crit = torch.linalg.vector_norm((x_prev - x2).reshape(B, -1), dim=1) / \
                torch.linalg.vector_norm((x2 + 1e-12).reshape(B, -1), dim=1)
            if k > 1:
                stop = active & (crit < self.crit)
                iters[stop.cpu()] = k + 1
                active = active & ~stop
                if not bool(active.any()):
                    break
        self.x2, self.u2 = x2, u2
        self.last_iterations = iters
        self.calls.append(iters.tolist())
        if self.verbose:
            print("TV prox: %s Chambolle-Pock iterations" % iters.tolist())
        return x2

    __call__ = forward


def primal_dual_gap(y, x, u, ths):
    """(P(x) - D(u_feasible)) / P(x) for P(x) = 1/2 ||x - y||^2 + ths TV(x) and its dual D(u) = 1/2 ||y||^2 - 1/2 ||y - nabla^T u||^2
    over ||u_p|| <= ths; u is projected onto that set first."""
    P = 0.5 * ((x - y) ** 2).sum() + ths * tv(x)
    u = u / torch.clamp(torch.sqrt((u ** 2).sum(-1)) / ths, min=1.0).unsqueeze(-1)
    D = 0.5 * (y ** 2).sum() - 0.5 * ((y - nabla_adjoint(u)) ** 2).sum()
    return float((P - D) / P)
