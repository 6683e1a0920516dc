"""Structured forward operators / data-fidelity gradients for the image samplers.

The reference builds ``data_grad``, ``A``, ``AT`` and ``prior_grad`` as opaque lambdas inside its script
(sampling_images.py:283-341,156-157).  A fused CUDA kernel cannot call a lambda, so the drop-in boundary uses
*structured callables*: objects that can still be called exactly like the reference closures (so the reference's
own ``psgla`` / ``pnpula`` accept them in parity tests) but that expose the mask / observation / blur taps /
noise level the kernels read.  ``psgla`` / ``pnpula`` here reject anything else with a ``TypeError``.
"""
from __future__ import annotations

import ctypes as C

import numpy as np
import torch

from . import _lib
from .denoisers import TVDenoiser

__all__ = ["InpaintingDataGrad", "DeblurDataGrad", "PriorGrad", "make_inpainting", "make_deblurring", "blur_taps"]


def _shape_of(x) -> "_lib.ImgShape":
    if x.dim() != 4 or x.shape[1] not in (1, 3):
        raise ValueError("expected a [B,3,H,W] (colour) or [B,1,H,W] (grayscale) tensor, got %s" % (tuple(x.shape),))
    return _lib.ImgShape(int(x.shape[0]), int(x.shape[1]), int(x.shape[2]), int(x.shape[3]))


class InpaintingDataGrad:
    """``data_grad(x) = -mask * (x - y) / sigma2`` (sampling_images.py:295).

    mask, y: tensors broadcastable to [B,C,H,W] (the reference uses [1,C,H,W]; C = 3, or 1 for grayscale); sigma2: float."""

    kind = "inpainting"

    def __init__(self, mask, y, sigma2):
        self.mask = mask.to(torch.float32).contiguous()
        self.y = y.to(torch.float32).contiguous()
        self.sigma2 = float(sigma2)

    def __call__(self, x):  # the reference's closure, for interoperability with the reference's samplers
        return -self.mask * (x - self.y) / torch.tensor(self.sigma2, dtype=torch.float32, device=x.device)


def blur_taps(l=4, blur_type="uniform", si=1.0):
    """Normalised 1 x (2l+1) taps as sampling_images.py:306-312 builds them (float64 row vector)."""
    if blur_type == "uniform":
        h = np.ones((1, 2 * l + 1))
    elif blur_type == "gaussian":
        h = np.array([[np.exp(-i ** 2 / (2 * si ** 2)) for i in range(-l, l + 1)]])
    else:
        raise ValueError("blur_type must be 'uniform' or 'gaussian'")
    return h / np.sum(h)


class DeblurDataGrad:
    """``data_grad(x) = -AT(A(x) - y) / sigma2`` with A = AT = circular separable blur (sampling_images.py:313-338).

    h1d: the 2l+1 taps of the separable kernel (``h_ = h^T h`` in the reference; ``flip(h_) == h_`` for the uniform
    and Gaussian taps it supports, so A and AT coincide)."""

    kind = "deblurring"

    def __init__(self, h1d, l, y, sigma2):
        self.h1d = np.asarray(h1d, dtype=np.float64).reshape(-1)
        self.l = int(l)
        if self.h1d.shape[0] != 2 * self.l + 1:
            raise ValueError("h1d must have 2l+1 taps")
        if not np.allclose(self.h1d, self.h1d[::-1], rtol=0, atol=0):
            raise ValueError("only symmetric taps are supported (the reference's uniform / gaussian kernels are)")
        self.y = y.to(torch.float32).contiguous()
        self.sigma2 = float(sigma2)
        self._taps_c = (C.c_float * (2 * self.l + 1))(*[float(np.float32(v)) for v in self.h1d])

    def A(self, x):
        """The blur itself: the library's circular separable stencil kernel (CUDA tensors only -- there is no CPU path; the
        reference's pad-circular + depthwise ``conv2d`` formulation is restated in the test infrastructure, not here)."""
        if not x.is_cuda:
            raise RuntimeError("DeblurDataGrad needs CUDA tensors: there is no CPU path")
        x = x.to(torch.float32).contiguous()
        out = torch.empty_like(x)
        with torch.cuda.device(x.device):
            _lib.check(_lib.lib().psgla_img_blur(_shape_of(x), _lib.ptr(x), self._taps_c, self.l, _lib.ptr(out),
                                                 _lib.stream_ptr(x.device)), "psgla_img_blur")
        return out

    AT = A

    def __call__(self, x):
        return -self.AT(self.A(x) - self.y) / torch.tensor(self.sigma2, dtype=torch.float32, device=x.device)


class PriorGrad:
    """``prior_grad(x) = alpha * (D(x; s1) - x) / s2`` (sampling_images.py:156-157)."""

    def __init__(self, denoiser, alpha, s1, s2):
        if isinstance(denoiser, TVDenoiser):
            raise TypeError("PriorGrad supports a psgla_b200.DnCNN, DRUNet or GSDRUNet denoiser, not the TV prox")
        self.denoiser, self.alpha, self.s1, self.s2 = denoiser, float(alpha), float(s1), float(s2)

    def __call__(self, x):
        return torch.tensor(self.alpha, dtype=torch.float32, device=x.device) * (self.denoiser.forward(x, self.s1) - x) \
            / torch.tensor(self.s2, dtype=torch.float32, device=x.device)


def make_inpainting(im_t, prop=0.5, sigma=1.0, seed_ip=0):
    """Observation, data-fidelity and chain initialisation for random inpainting, following
    sampling_images.py:283-302 on ``im_t``'s device.  Returns (data_grad, init, y, mask)."""
    device = im_t.device
    sigma1 = sigma / 255.0
    gen = torch.Generator(device=device)
    gen.manual_seed(seed_ip)
    u = torch.rand((im_t.shape[2], im_t.shape[3]), generator=gen, device=device)
    mask = (u > prop).to(torch.float32)[None, None].expand(1, im_t.shape[1], -1, -1).contiguous()
    noise = torch.normal(torch.zeros(*im_t.size(), device=device), std=sigma1 * torch.ones(*im_t.size(), device=device),
                         generator=gen)
    y = mask * im_t + noise
    init = mask * y + (1 - mask) * 0.5
    return InpaintingDataGrad(mask, y, sigma1 ** 2), init, y, mask


def make_deblurring(im_t, l=4, blur_type="uniform", si=1.0, sigma=1.0, seed_ip=0):
    """Observation, data-fidelity and initialisation for deblurring (sampling_images.py:304-341).
    Returns (data_grad, init, y)."""
    device = im_t.device
    sigma1 = sigma / 255.0
    h = blur_taps(l, blur_type, si).reshape(-1)
    op = DeblurDataGrad(h, l, torch.zeros_like(im_t), sigma1 ** 2)
    gen = torch.Generator(device=device)
    gen.manual_seed(seed_ip)
    noise = torch.normal(torch.zeros(*im_t.size(), device=device), std=sigma1 * torch.ones(*im_t.size(), device=device),
                         generator=gen)
    y = op.A(im_t.to(torch.float32)) + noise
    op.y = y.contiguous()
    return op, y.clone(), y
