"""Restatement of deepinv 0.2.1's gradient-step DRUNet (``deepinv.models.GSDRUNet``, the fourth denoiser of the reference's
image driver, sampling_images.py:129-140), dtype-generic, for the tests.  PARITY UNPINNED: deepinv is not installed, and what
follows is recalled from its source, not checked against it:

  N(x; sigma)  KAIR UNetRes(in_nc = 4, out_nc = 3, nc = [64, 128, 256, 512], nb = 2, act_mode = "E", no biases): the image with
               a constant sigma map as fourth channel, residual blocks x + conv(elu(conv(x))), 2x2 stride-2 convs down, 2x2
               stride-2 transposed convs up, U-Net skips added before each up stage and the tail.
  g(x)         1/2 ||x - N(x)||^2
  grad g(x)    v - J^T v,  v = x - N(x),  J^T v = torch.autograd.grad(N, x, grad_outputs=v)  (sigma's gradient dropped)
  D(x; sigma)  x - alpha grad g(x)

``network`` with ``act = F.relu`` and ``nb = 4`` is oracle.image_oracle.DRUNet (tests/test_gsdrunet_host.py checks it).
"""
import torch
import torch.nn.functional as F


def _conv3(x, w):
    return F.conv2d(x, w.to(x.dtype), padding=1)


def network(sd, x, sigma, nb=2, act=F.elu):
    """N(x; sigma) for a state dict with KAIR keys (``psgla_b200.denoisers._drunet_keys(nb)``), in x's dtype."""
    w = lambda k: sd[k].to(x.device, x.dtype)  # noqa: E731

    def blocks(prefix, h, first):
        for i in range(first, first + nb):
            h = h + _conv3(act(_conv3(h, w("%s.%d.res.0.weight" % (prefix, i)))), w("%s.%d.res.2.weight" % (prefix, i)))
        return h

    noise_map = torch.full((x.shape[0], 1, x.shape[2], x.shape[3]), float(sigma), dtype=x.dtype, device=x.device)
    x1 = _conv3(torch.cat((x, noise_map), 1), w("m_head.weight"))
    xs = [x1]
    for s in (1, 2, 3):
        h = blocks("m_down%d" % s, xs[-1], 0)
        xs.append(F.conv2d(h, w("m_down%d.%d.weight" % (s, nb)), stride=2))
    h = blocks("m_body", xs[3], 0)
    for s in (3, 2, 1):
        h = F.conv_transpose2d(h + xs[s], w("m_up%d.0.weight" % s), stride=2)
        h = blocks("m_up%d" % s, h, 1)
    return _conv3(h + xs[0], w("m_tail.weight"))


def grad_g(sd, x, sigma, create_graph=False):
    """(grad g(x), N(x), J^T v) in x's dtype."""
    with torch.enable_grad():
        xr = x.detach().requires_grad_(True)
        n = network(sd, xr, sigma)
        v = xr - n
        jtv = torch.autograd.grad(n, xr, grad_outputs=v, create_graph=create_graph)[0]
        return v - jtv, n, jtv


class GSDRUNet:
    """``forward(x, sigma)`` = D(x; sigma) in x's dtype (autograd), the denoiser the oracle samplers call."""

    def __init__(self, sd, alpha=1.0):
        self.sd, self.alpha = sd, float(alpha)

    def forward(self, x, sigma):
        if isinstance(sigma, torch.Tensor):
            sigma = float(sigma.reshape(-1)[0])
        g, _, _ = grad_g(self.sd, x, sigma)
        return (x - self.alpha * g).detach()

    __call__ = forward
