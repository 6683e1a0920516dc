"""The image denoisers: DnCNN, DRUNet and the gradient-step DRUNet (its network and the network's vector-Jacobian product,
csrc/gsdrunet.cu) as tcgen05 implicit-GEMM convolutions (csrc/conv_tc.cu, csrc/conv_gemm.cu), and the TV proximal operator
(csrc/tv_prox.cu).

``DnCNN`` mirrors ``deepinv.models.DnCNN(in_channels=3, out_channels=3, pretrained=..., device=...)`` as the reference constructs
it (sampling_images.py:130), and its one-channel form ``in_channels=out_channels=1`` for grayscale images and calls it (``denoiser.forward(x, sigma)``, restoration_algorithms.py:238): depth 20,
64 features, 3x3, bias, ReLU, residual output, ``sigma`` ignored.  Weights come from a deepinv-style state dict
(keys ``in_conv``, ``conv_list.i``, ``out_conv``) -- a checkpoint path, a dict, or ``None`` for seeded random init.
Activations are bf16 with fp32 accumulation; the input / output images stay fp32.
"""
from __future__ import annotations

import ctypes as C
import math

import torch

from . import _lib

__all__ = ["DnCNN", "DRUNet", "GSDRUNet", "TVDenoiser", "random_dncnn_state_dict", "lipschitz_dncnn_state_dict",
           "smoothing_dncnn_state_dict", "random_drunet_state_dict", "random_gsdrunet_state_dict", "DRUNET_KEYS", "GSDRUNET_KEYS"]


def random_dncnn_state_dict(seed=0, depth=20, nf=64, scale=1.0, channels=3):
    """Deterministic random-init DnCNN state dict (uniform +-1/sqrt(fan_in) like nn.Conv2d's default), on the CPU.
    ``channels``: image channels, 3 (colour) or 1 (grayscale)."""
    g = torch.Generator().manual_seed(seed)
    sd = {}

    def conv(name, cout, cin):
        bound = scale / math.sqrt(cin * 9)
        sd[name + ".weight"] = (torch.rand((cout, cin, 3, 3), generator=g) * 2 - 1) * bound
        sd[name + ".bias"] = (torch.rand((cout,), generator=g) * 2 - 1) * 0.01

    conv("in_conv", nf, channels)
    for i in range(depth - 2):
        conv("conv_list.%d" % i, nf, nf)
    conv("out_conv", channels, nf)
    return sd


def _conv_operator_norm(w, spatial=16, n_power_iter=40):
    """Spectral norm of the circular 3x3 convolution with weight ``w`` [O,I,3,3] on a spatial x spatial grid: the
    operator is block-diagonalised by the 2-D DFT, so the norm is the largest singular value over frequencies."""
    k = torch.zeros((w.shape[0], w.shape[1], spatial, spatial), dtype=torch.float64)
    k[:, :, :3, :3] = w.double()
    kf = torch.fft.fft2(k).permute(2, 3, 0, 1).reshape(-1, w.shape[0], w.shape[1])
    gram = kf.conj().transpose(1, 2) @ kf  # per-frequency Hermitian [I, I]
    v = torch.ones((gram.shape[0], gram.shape[1], 1), dtype=gram.dtype)
    lam = torch.ones(gram.shape[0], dtype=torch.float64)
    for _ in range(n_power_iter):  # batched power iteration; a norm estimate from below, within 1e-3 after 40 rounds
        v = gram @ v
        lam = torch.linalg.vector_norm(v, dim=(1, 2))
        v = v / lam.clamp_min(1e-300)[:, None, None]
    return float(lam.max().sqrt())


def lipschitz_dncnn_state_dict(seed=0, depth=20, nf=64, lipschitz=0.9, spatial=16, channels=3):
    """Seeded random-init DnCNN whose residual branch has Lipschitz bound ``lipschitz`` < 1 (the stand-in BASELINE.json
    prescribes for the unavailable ``dncnn_sigma2_lipschitz_color.pth``, README.md:28-29): every conv is divided by
    its exact circular operator norm and the layers share the bound evenly.  Set-up code, runs once on the CPU.
    ``channels``: image channels, 3 (colour) or 1 (grayscale)."""
    sd = random_dncnn_state_dict(seed, depth, nf, channels=channels)
    per_layer = lipschitz ** (1.0 / depth)
    for name in ["in_conv"] + ["conv_list.%d" % i for i in range(depth - 2)] + ["out_conv"]:
        w = sd[name + ".weight"]
        sd[name + ".weight"] = (w * (per_layer / _conv_operator_norm(w, spatial))).float()
    return sd


def smoothing_dncnn_state_dict(eps=0.5, n_smooth=6, depth=20, nf=64, channels=3):
    """A DnCNN-architecture state dict, written down by hand, that IS a (weak) denoiser: its residual is
    ``R(x) = eps * (G x - x)`` with G = ``n_smooth`` passes of the 3 x 3 binomial kernel [1 2 1]^T [1 2 1] / 16.  The checkpoint the
    reference uses cannot be fetched offline and a random-init network restores nothing (unobserved pixels random-walk), so
    this is the stand-in for runs whose PSNR should MEAN something: PSGLA with it is diffusion inpainting / smoothing-regularised
    deblurring, stable at any length, and ||R||_Lip <= eps < 1.  Construction (ReLU networks compute linear maps on
    x = relu(x) - relu(-x)): features 0-2 / 3-5 carry relu(+-x) and are smoothed by layers 1..n_smooth, features 6-8 / 9-11
    carry relu(+-x) unchanged, every other feature is zero; the last layer forms eps ((f0-2 - f3-5) - (f6-8 - f9-11)).
    ``channels``: image channels, 3 (colour) or 1 (grayscale: features 0, 3, 6, 9 carry the one channel)."""
    if depth < n_smooth + 2 or nf < 12:
        raise ValueError("needs depth >= n_smooth + 2 and nf >= 12")
    g1 = torch.tensor([1.0, 2.0, 1.0]) / 4.0
    G = torch.outer(g1, g1)
    ident = torch.zeros(3, 3)
    ident[1, 1] = 1.0
    sd = {}
    w = torch.zeros(nf, channels, 3, 3)
    for c in range(channels):
        for base, sign in ((0, 1.0), (3, -1.0), (6, 1.0), (9, -1.0)):
            w[base + c, c, 1, 1] = sign
    sd["in_conv.weight"], sd["in_conv.bias"] = w, torch.zeros(nf)
    for i in range(depth - 2):
        w = torch.zeros(nf, nf, 3, 3)
        for f in range(12):
            w[f, f] = G if (f < 6 and i < n_smooth) else ident
        sd["conv_list.%d.weight" % i], sd["conv_list.%d.bias" % i] = w, torch.zeros(nf)
    w = torch.zeros(channels, nf, 3, 3)
    for c in range(channels):
        w[c, c, 1, 1], w[c, 3 + c, 1, 1], w[c, 6 + c, 1, 1], w[c, 9 + c, 1, 1] = eps, -eps, -eps, eps
    sd["out_conv.weight"], sd["out_conv.bias"] = w, torch.zeros(channels)
    return sd


class DnCNN:
    """``channels`` (= in_channels = out_channels): 3 for colour images, 1 for grayscale ones.  The weights are packed for that
    channel count, and the samplers take images of that many channels only."""

    is_residual = True  # D(x) = x + R(x): the samplers add gain * R to their base

    def __init__(self, in_channels=3, out_channels=3, depth=20, bias=True, nf=64, pretrained=None, device=None):
        torch_ = _lib.require_cuda()
        if in_channels != out_channels or in_channels not in (1, 3) or nf != 64:
            raise ValueError("the sm_100a conv path is built for DnCNN with in = out = 3 (colour) or 1 (grayscale) channels, "
                             "nf = 64")
        if depth < 2:
            raise ValueError("depth must be >= 2")
        self.channels = int(in_channels)
        self.depth = int(depth)
        self.device = torch_.device("cuda", torch_.cuda.current_device()) if device is None else torch_.device(device)
        if pretrained is None:
            sd = random_dncnn_state_dict(0, depth, nf, channels=self.channels)
        elif isinstance(pretrained, str):
            sd = torch_.load(pretrained, map_location="cpu")
        else:
            sd = pretrained
        names = ["in_conv"] + ["conv_list.%d" % i for i in range(depth - 2)] + ["out_conv"]
        missing = [n for n in names if n + ".weight" not in sd]
        if missing:
            raise KeyError("state dict lacks %s" % missing[:3])
        self.state_dict_fp32 = {k: v.detach().to("cpu", torch_.float32).contiguous() for k, v in sd.items()}
        ws = [self.state_dict_fp32[n + ".weight"] for n in names]
        expect = [(nf, self.channels, 3, 3)] + [(nf, nf, 3, 3)] * (depth - 2) + [(self.channels, nf, 3, 3)]
        for w, e, n in zip(ws, expect, names):
            if tuple(w.shape) != e:
                raise ValueError("%s.weight has shape %s, expected %s" % (n, tuple(w.shape), e))
        bs = [self.state_dict_fp32.get(n + ".bias") if bias else None for n in names]
        lib = _lib.lib()
        self.packed = torch_.empty(lib.psgla_dncnn_packed_bytes(self.depth), dtype=torch_.uint8, device=self.device)
        FP = C.POINTER(C.c_float)
        warr = (FP * depth)(*[C.cast(w.data_ptr(), FP) for w in ws])
        barr = (FP * depth)(*[C.cast(b.data_ptr(), FP) if b is not None else FP() for b in bs])
        with torch_.cuda.device(self.device):
            _lib.check(lib.psgla_dncnn_pack_weights_ch(self.depth, self.channels, warr, barr, _lib.ptr(self.packed),
                                                       _lib.stream_ptr(self.device)), "psgla_dncnn_pack_weights_ch")
        self._ws = None
        self._den_in = None

    # workspace shared by every call with the same shape
    def buffers(self, shape: "_lib.ImgShape"):
        need = _lib.lib().psgla_dncnn_workspace_bytes(shape)
        if self._ws is None or self._ws.numel() < need:
            self._ws = torch.empty(need, dtype=torch.uint8, device=self.device)
        n_in = shape.B * shape.H * shape.W * 16
        if self._den_in is None or self._den_in.numel() < n_in:
            self._den_in = torch.empty(n_in, dtype=torch.bfloat16, device=self.device)
        return self._ws, self._den_in

    def residual_post(self, shape, den_in, base, post, x_out, sample=None, mean=None, mean2=None, next_pre=None):
        """``next_pre``: a ``_lib.NextPre`` -- the next iteration's inpainting "pre" fused into the last layer's epilogue."""
        ws, _ = self.buffers(shape)
        with torch.cuda.device(self.device):
            rc = _lib.lib().psgla_dncnn_residual_post_next(self.depth, _lib.ptr(self.packed), shape, _lib.ptr(den_in),
                                                           _lib.ptr(ws), ws.numel(), _lib.ptr(base), C.byref(post),
                                                           _lib.ptr(x_out), _lib.ptr(sample), _lib.ptr(mean), _lib.ptr(mean2),
                                                           C.byref(next_pre) if next_pre is not None else None,
                                                           _lib.stream_ptr(self.device))
        _lib.check(rc, "psgla_dncnn_residual_post_next")

    def forward(self, x, sigma=None):
        """D(x) = x + R(x), fp32 [B,C,H,W] in and out, C = ``channels`` (``sigma`` ignored, as in deepinv's DnCNN)."""
        if not x.is_cuda:
            raise RuntimeError("DnCNN.forward needs a CUDA tensor: there is no CPU path")
        _check_channels(x, self.channels, "DnCNN")
        x = x.to(torch.float32).contiguous()
        shape = _lib.ImgShape(int(x.shape[0]), self.channels, int(x.shape[2]), int(x.shape[3]))
        _, den_in = self.buffers(shape)
        out = torch.empty_like(x)
        with torch.cuda.device(self.device):
            _lib.check(_lib.lib().psgla_img_to_nhwc16(shape, _lib.ptr(x), 0.0, _lib.ptr(den_in), _lib.stream_ptr(self.device)),
                       "psgla_img_to_nhwc16")
        self.residual_post(shape, den_in, x, _lib.PostParams(1.0, 1.0, 0.0, 1.0), out)
        return out

    __call__ = forward
    apply_post = residual_post  # common name used by the samplers for both denoiser families


def _check_channels(x, channels, name):
    if x.dim() != 4 or x.shape[1] != channels:
        raise ValueError("%s was built for %d-channel images: expected a [B,%d,H,W] batch, got %s" %
                         (name, channels, channels, tuple(x.shape)))


# ----------------------------------------------------------------------------------------------------- DRUNet
def _drunet_keys(nb=4):
    keys = ["m_head.weight"]
    for s in (1, 2, 3):
        keys += ["m_down%d.%d.res.%d.weight" % (s, i, j) for i in range(nb) for j in (0, 2)] + ["m_down%d.%d.weight" % (s, nb)]
    keys += ["m_body.%d.res.%d.weight" % (i, j) for i in range(nb) for j in (0, 2)]
    for s in (3, 2, 1):
        keys += ["m_up%d.0.weight" % s] + ["m_up%d.%d.res.%d.weight" % (s, i, j) for i in range(1, nb + 1) for j in (0, 2)]
    return keys + ["m_tail.weight"]


DRUNET_KEYS = _drunet_keys()  # the 64 weight tensors of drunet_color.pth in state-dict order
GSDRUNET_KEYS = _drunet_keys(2)  # the 36 of the gradient-step DRUNet's network (nb = 2)


def _drunet_shape(key, nc=(64, 128, 256, 512), channels=3):
    if key == "m_head.weight":
        return (nc[0], channels + 1, 3, 3)  # the image channels, then the noise-level map
    if key == "m_tail.weight":
        return (channels, nc[0], 3, 3)
    if key.startswith("m_body"):
        return (nc[3], nc[3], 3, 3)
    s = int(key[len("m_down")]) if key.startswith("m_down") else int(key[len("m_up")])
    if ".res." in key:
        return (nc[s - 1], nc[s - 1], 3, 3)
    if key.startswith("m_down"):
        return (nc[s], nc[s - 1], 2, 2)  # strided conv, OIHW
    return (nc[s], nc[s - 1], 2, 2)      # transposed conv: [Cin][Cout][2][2]


def random_drunet_state_dict(seed=0, gain=0.5, nb=4, channels=3):
    """Seeded random-init DRUNet state dict on the CPU (checkpoints are unreachable offline): uniform
    +-gain*sqrt(3/fan_in), second conv of every residual block halved, tail quartered, so activations stay O(1).
    ``nb``: residual blocks per stage (2: the gradient-step DRUNet's network).  ``channels``: image channels, 3 or 1."""
    g = torch.Generator().manual_seed(seed)
    sd = {}
    for k in _drunet_keys(nb):
        shp = _drunet_shape(k, channels=channels)
        is_up = k.startswith("m_up") and ".res." not in k
        fan_in = shp[0] * 4 if is_up else shp[1] * shp[2] * shp[3]
        bound = gain * math.sqrt(3.0 / fan_in)
        if ".res.2." in k:
            bound *= 0.5
        if k == "m_tail.weight":
            bound *= 0.25
        sd[k] = (torch.rand(shp, generator=g) * 2 - 1) * bound
    return sd


class DRUNet:
    """``deepinv.models.DRUNet(in_channels=3, out_channels=3, pretrained=..., device=...)`` (sampling_images.py:136) on
    tcgen05 convolutions: the DPIR U-Net (KAIR UNetRes, nc = 64/128/256/512, 4 residual blocks per stage, no biases).
    ``forward(x, sigma)`` appends the constant noise-level channel and returns the denoised image.  ``pretrained``: a
    ``drunet_color.pth``-style state dict / path, or None for seeded random init.  H, W multiples of 8.
    ``channels`` (= in_channels = out_channels): 3 for colour images, 1 for grayscale ones (``drunet_gray.pth``-style: m_head
    takes the image and the noise-level map, m_tail gives one channel); the samplers take images of that many channels only."""

    is_residual = False  # the network outputs D(x) itself

    def __init__(self, in_channels=3, out_channels=3, pretrained=None, device=None):
        torch_ = _lib.require_cuda()
        if in_channels != out_channels or in_channels not in (1, 3):
            raise ValueError("the sm_100a DRUNet path is built for in = out = 3 (colour) or 1 (grayscale) channels")
        self.channels = int(in_channels)
        self.device = torch_.device("cuda", torch_.cuda.current_device()) if device is None else torch_.device(device)
        if pretrained is None:
            sd = random_drunet_state_dict(0, channels=self.channels)
        elif isinstance(pretrained, str):
            sd = torch_.load(pretrained, map_location="cpu")
        else:
            sd = pretrained
        missing = [k for k in DRUNET_KEYS if k not in sd]
        if missing:
            raise KeyError("state dict lacks %s" % missing[:3])
        ws = []
        for k in DRUNET_KEYS:
            w = sd[k].detach().to("cpu", torch_.float32).contiguous()
            want = _drunet_shape(k, channels=self.channels)
            if tuple(w.shape) != want:
                raise ValueError("%s has shape %s, expected %s" % (k, tuple(w.shape), want))
            ws.append(w)
        self.state_dict_fp32 = dict(zip(DRUNET_KEYS, ws))
        lib = _lib.lib()
        assert lib.psgla_drunet_num_weights() == len(ws)
        self.packed = torch_.empty(lib.psgla_drunet_packed_bytes(), dtype=torch_.uint8, device=self.device)
        FP = C.POINTER(C.c_float)
        warr = (FP * len(ws))(*[C.cast(w.data_ptr(), FP) for w in ws])
        with torch_.cuda.device(self.device):
            _lib.check(lib.psgla_drunet_pack_weights_ch(self.channels, warr, _lib.ptr(self.packed), _lib.stream_ptr(self.device)),
                       "psgla_drunet_pack_weights_ch")
        self._ws = None
        self._den_in = None

    def buffers(self, shape: "_lib.ImgShape"):
        need = _lib.lib().psgla_drunet_workspace_bytes(shape)
        if self._ws is None or self._ws.numel() < need:
            self._ws = torch.empty(need, dtype=torch.uint8, device=self.device)
        n_in = shape.B * shape.H * shape.W * 16
        if self._den_in is None or self._den_in.numel() < n_in:
            self._den_in = torch.empty(n_in, dtype=torch.bfloat16, device=self.device)
        return self._ws, self._den_in

    def apply_post(self, shape, den_in, base, post, x_out, sample=None, mean=None, mean2=None, next_pre=None):
        ws, _ = self.buffers(shape)
        with torch.cuda.device(self.device):
            rc = _lib.lib().psgla_drunet_denoise_post_next(_lib.ptr(self.packed), shape, _lib.ptr(den_in), _lib.ptr(ws),
                                                           ws.numel(), _lib.ptr(base), C.byref(post), _lib.ptr(x_out),
                                                           _lib.ptr(sample), _lib.ptr(mean), _lib.ptr(mean2),
                                                           C.byref(next_pre) if next_pre is not None else None,
                                                           _lib.stream_ptr(self.device))
        _lib.check(rc, "psgla_drunet_denoise_post_next")

    def forward(self, x, sigma):
        """D(x; sigma), fp32 [B,C,H,W] in and out, C = ``channels``.  The U-Net halves the resolution three times, so H and W must be multiples
        of 8; other sizes (CBSD68's 481 x 321) are replication-padded at the bottom / right to the next multiple, denoised and
        cropped -- KAIR's ``test_pad`` rule, which is what deepinv applies to small inputs (its rule for large ones, a 4-way
        overlapping split, cannot be verified offline: a documented deviation).  The samplers apply the same per-call padding to
        inpainting problems (restoration_algorithms._Run); deblurring problems must be cropped to multiples of 8."""
        if not x.is_cuda:
            raise RuntimeError("DRUNet.forward needs a CUDA tensor: there is no CPU path")
        _check_channels(x, self.channels, "DRUNet")
        sigma = float(sigma.reshape(-1)[0]) if isinstance(sigma, torch.Tensor) else float(sigma)
        x = x.to(torch.float32).contiguous()
        H0, W0 = int(x.shape[2]), int(x.shape[3])
        ph, pw = (-H0) % 8, (-W0) % 8
        if ph or pw:
            x = torch.nn.functional.pad(x, (0, pw, 0, ph), mode="replicate").contiguous()
        shape = _lib.ImgShape(int(x.shape[0]), self.channels, int(x.shape[2]), int(x.shape[3]))
        _, den_in = self.buffers(shape)
        out = torch.empty_like(x)
        with torch.cuda.device(self.device):
            _lib.check(_lib.lib().psgla_img_to_nhwc16(shape, _lib.ptr(x), sigma, _lib.ptr(den_in), _lib.stream_ptr(self.device)),
                       "psgla_img_to_nhwc16")
        self.apply_post(shape, den_in, x, _lib.PostParams(1.0, 0.0, 0.0, 1.0), out)  # out = 0 * x + 1 * D(x)
        return out[:, :, :H0, :W0].contiguous() if (ph or pw) else out

    __call__ = forward


# ----------------------------------------------------------------------------------------------------- GSDRUNet
def random_gsdrunet_state_dict(seed=0, gain=0.5):
    """Seeded random-init state dict of the gradient-step DRUNet's network (``random_drunet_state_dict`` with nb = 2)."""
    return random_drunet_state_dict(seed, gain, nb=2)


_GS_PREFIX = "student_grad.model."


def gsdrunet_weights(sd):
    """The 36 fp32 CPU tensors of GSDRUNET_KEYS from a state dict with KAIR keys.  A ``{"state_dict": ...}`` wrapper and
    the ``student_grad.model.`` prefix of deepinv's GSDRUNet module are stripped (both forms recalled, not verified against a
    deepinv checkpoint)."""
    if "state_dict" in sd and isinstance(sd["state_dict"], dict):
        sd = sd["state_dict"]
    sd = {(k[len(_GS_PREFIX):] if k.startswith(_GS_PREFIX) else k): v for k, v in sd.items()}
    missing = [k for k in GSDRUNET_KEYS if k not in sd]
    if missing:
        raise KeyError("state dict lacks %s" % missing[:3])
    ws = []
    for k in GSDRUNET_KEYS:
        w = sd[k].detach().to("cpu", torch.float32).contiguous()
        if tuple(w.shape) != _drunet_shape(k):
            raise ValueError("%s has shape %s, expected %s" % (k, tuple(w.shape), _drunet_shape(k)))
        ws.append(w)
    return ws


class GSDRUNet:
    """``deepinv.models.GSDRUNet(alpha=1.0, in_channels=3, out_channels=3, nb=2, nc=[64,128,256,512], act_mode="E",
    pretrained=..., device=...)``, the gradient-step denoiser (Prox-DRUNet is the same class from another checkpoint):
    ``D(x; sigma) = x - alpha grad g(x)`` with ``g(x) = 1/2 ||x - N(x)||^2`` and N the KAIR U-Net with 2 residual blocks per
    stage, ELU inside the blocks and no biases.  Each call runs N and its vector-Jacobian product on tcgen05 convolutions
    (csrc/gsdrunet.cu).  ``pretrained``: None (seeded random init), a checkpoint path or a state dict.  H, W multiples of 8."""

    is_residual = False  # D(x) itself
    channels = 3  # colour-only

    def __init__(self, alpha=1.0, in_channels=3, out_channels=3, nb=2, nc=(64, 128, 256, 512), act_mode="E", pretrained=None,
                 device=None):
        if in_channels != 3 or out_channels != 3 or nb != 2 or list(nc) != [64, 128, 256, 512] or act_mode != "E":
            raise ValueError("the sm_100a GSDRUNet path is built for in = out = 3 channels, nb = 2, nc = [64, 128, 256, 512], "
                             "act_mode = 'E'")
        self.alpha = float(alpha)
        if not math.isfinite(self.alpha):
            raise ValueError("alpha must be finite")
        torch_ = _lib.require_cuda()
        self.device = torch_.device("cuda", torch_.cuda.current_device()) if device is None else torch_.device(device)
        if pretrained is None:
            sd = random_gsdrunet_state_dict(0)
        elif isinstance(pretrained, str):
            sd = torch_.load(pretrained, map_location="cpu")
        else:
            sd = pretrained
        ws = gsdrunet_weights(sd)
        self.state_dict_fp32 = dict(zip(GSDRUNET_KEYS, ws))
        lib = _lib.lib()
        assert lib.psgla_gsdrunet_num_weights() == len(ws)
        self.packed = torch_.empty(lib.psgla_gsdrunet_packed_bytes(), dtype=torch_.uint8, device=self.device)
        FP = C.POINTER(C.c_float)
        warr = (FP * len(ws))(*[C.cast(w.data_ptr(), FP) for w in ws])
        with torch_.cuda.device(self.device):
            _lib.check(lib.psgla_gsdrunet_pack_weights(warr, _lib.ptr(self.packed), _lib.stream_ptr(self.device)),
                       "psgla_gsdrunet_pack_weights")
        self._ws = None
        self._den_in = None

    @staticmethod
    def check_size(H, W):
        if H % 8 or W % 8:
            raise ValueError("GSDRUNet needs H and W to be multiples of 8 (got %d x %d): crop the image; the gradient through "
                             "a padded input is not implemented" % (H, W))

    def buffers(self, shape: "_lib.ImgShape"):
        need = _lib.lib().psgla_gsdrunet_workspace_bytes(shape)
        if need == 0:
            raise ValueError("bad image shape for GSDRUNet")
        if self._ws is None or self._ws.numel() < need:
            self._ws = torch.empty(need, dtype=torch.uint8, device=self.device)
        n_in = shape.B * shape.H * shape.W * 16
        if self._den_in is None or self._den_in.numel() < n_in:
            self._den_in = torch.empty(n_in, dtype=torch.bfloat16, device=self.device)
        return self._ws, self._den_in

    def apply_post(self, shape, den_in, base, post, x_out, sample=None, mean=None, mean2=None, next_pre=None, x=None):
        """x_out = post.base_scale * base + post.gain * D(x), thinning, moments, optional fused next pre.  ``den_in``: bf16
        NHWC16 of x with the sigma map in channel 3; ``x``: x in fp32, None when it is ``base`` (PSGLA)."""
        ws, _ = self.buffers(shape)
        with torch.cuda.device(self.device):
            rc = _lib.lib().psgla_gsdrunet_denoise_post_next(_lib.ptr(self.packed), shape, _lib.ptr(den_in), _lib.ptr(x),
                                                             _lib.ptr(ws), ws.numel(), _lib.ptr(base), self.alpha, C.byref(post),
                                                             _lib.ptr(x_out), _lib.ptr(sample), _lib.ptr(mean), _lib.ptr(mean2),
                                                             C.byref(next_pre) if next_pre is not None else None,
                                                             _lib.stream_ptr(self.device))
        _lib.check(rc, "psgla_gsdrunet_denoise_post_next")

    def forward(self, x, sigma):
        """D(x; sigma), fp32 [B,3,H,W] in and out, H and W multiples of 8."""
        if not x.is_cuda:
            raise RuntimeError("GSDRUNet.forward needs a CUDA tensor: there is no CPU path")
        if x.dim() != 4 or x.shape[1] != 3:
            raise ValueError("expected a [B,3,H,W] colour batch, got %s" % (tuple(x.shape),))
        self.check_size(int(x.shape[2]), int(x.shape[3]))
        sigma = float(sigma.reshape(-1)[0]) if isinstance(sigma, torch.Tensor) else float(sigma)
        x = x.to(self.device, torch.float32).contiguous()
        shape = _lib.ImgShape(int(x.shape[0]), 3, int(x.shape[2]), int(x.shape[3]))
        _, den_in = self.buffers(shape)
        out = torch.empty_like(x)
        with torch.cuda.device(self.device):
            _lib.check(_lib.lib().psgla_img_to_nhwc16(shape, _lib.ptr(x), sigma, _lib.ptr(den_in), _lib.stream_ptr(self.device)),
                       "psgla_img_to_nhwc16")
        self.apply_post(shape, den_in, x, _lib.PostParams(1.0, 0.0, 0.0, 1.0), out)  # out = 0 * x + 1 * D(x)
        return out

    __call__ = forward


# ----------------------------------------------------------------------------------------------------- TV
class TVDenoiser:
    """``deepinv.models.TVDenoiser(verbose=False, tau=0.01, rho=1.99, n_it_max=1000, crit=1e-5)`` (sampling_images.py:139-140)
    on one cooperative CUDA launch per call (csrc/tv_prox.cu): the prox of ths * isotropic total variation (per channel and
    pixel) by over-relaxed Chambolle-Pock, fp32.  ``forward(y, ths)`` warm-starts from the previous call's primal / dual state
    like deepinv's: it restarts (x2 = y, u2 = 0) on the first call, after ``reset()`` or ``restart = True``, and when y's shape
    changes.  One difference: the stopping test ||x_prev - x2|| / ||x2|| < crit is evaluated per chain (per batch entry) and
    each chain stops on its own, so a chain's result does not depend on the chains next to it; for a single chain -- every
    run the reference makes -- this is deepinv's rule.  Any image size.

    ``x2`` / ``u2``: views of the state ([B,3,H,W] and [B,3,H,W,2]); ``last_iterations``: device int32 [B], the CP iteration
    count of each chain in the last call (no host synchronisation)."""

    is_residual = False  # D(y) itself: the samplers form (1 - alpha) Y + alpha D(Y)
    channels = 3  # colour-only

    def __init__(self, verbose=False, tau=0.01, rho=1.99, n_it_max=1000, crit=1e-5, device=None):
        torch_ = _lib.require_cuda()
        self.device = torch_.device("cuda", torch_.cuda.current_device()) if device is None else torch_.device(device)
        self.verbose = bool(verbose)
        self.tau, self.rho, self.n_it_max, self.crit = float(tau), float(rho), int(n_it_max), float(crit)
        self.restart = True
        self._shape = None
        self._state = None
        self._ws = None
        self._den_in = None
        self.last_iterations = None

    def reset(self):
        """The next call starts from x2 = y, u2 = 0."""
        self.restart = True

    @property
    def x2(self):
        if self._shape is None:
            return None
        B, _, H, W = self._shape
        return self._state[:B * 3 * H * W].view(B, 3, H, W)

    @property
    def u2(self):
        if self._shape is None:
            return None
        B, _, H, W = self._shape
        return self._state[B * 3 * H * W:].view(B, 3, H, W, 2)

    def buffers(self, shape: "_lib.ImgShape"):
        """(workspace, denoiser input): the samplers' "pre" writes the bf16 input every denoiser takes; the prox reads the
        fp32 base instead, so the second buffer is only written."""
        lib = _lib.lib()
        need = lib.psgla_tv_workspace_bytes(shape)
        if need == 0:
            raise ValueError("bad image shape for the TV prox")
        if self._ws is None or self._ws.numel() < need:
            self._ws = torch.empty(need, dtype=torch.uint8, device=self.device)
        n_in = shape.B * shape.H * shape.W * 16
        if self._den_in is None or self._den_in.numel() < n_in:
            self._den_in = torch.empty(n_in, dtype=torch.bfloat16, device=self.device)
        return self._ws, self._den_in

    def apply_post(self, shape, den_in, base, post, x_out, sample=None, mean=None, mean2=None, next_pre=None, ths=None):
        """x_out = post.base_scale * base + post.gain * TV_prox(base; ths), thinning and moments (the samplers' post).
        ``den_in`` is not read; the fused next-iteration pre is a conv-epilogue feature and is not offered."""
        if next_pre is not None:
            raise ValueError("the TV prox does not fuse the next iteration's pre")
        if ths is None:
            raise ValueError("the TV prox needs ths")
        ws, _ = self.buffers(shape)
        key = (shape.B, 3, shape.H, shape.W)
        restart = self.restart or self._shape != key
        if restart and self._shape != key:
            self._state = torch.empty(_lib.lib().psgla_tv_state_bytes(shape) // 4, dtype=torch.float32, device=self.device)
            self._shape = key
        if self.last_iterations is None or self.last_iterations.numel() != shape.B:
            self.last_iterations = torch.empty(shape.B, dtype=torch.int32, device=self.device)
        prm = _lib.TVParams(float(ths), self.tau, self.rho, self.crit, self.n_it_max, int(restart))
        with torch.cuda.device(self.device):
            rc = _lib.lib().psgla_tv_prox_post(C.byref(prm), shape, _lib.ptr(base), _lib.ptr(self._state), self._state.numel() * 4,
                                               _lib.ptr(ws), ws.numel(), C.byref(post), _lib.ptr(x_out), _lib.ptr(sample),
                                               _lib.ptr(mean), _lib.ptr(mean2), _lib.ptr(self.last_iterations),
                                               _lib.stream_ptr(self.device))
        _lib.check(rc, "psgla_tv_prox_post")
        self.restart = False
        if self.verbose:
            print("TV prox: %s Chambolle-Pock iterations" % self.last_iterations.tolist())

    def forward(self, y, ths):
        """TV_prox(y; ths), fp32 [B,3,H,W] in and out (``ths``: a number or a one-element tensor)."""
        if not y.is_cuda:
            raise RuntimeError("TVDenoiser.forward needs a CUDA tensor: there is no CPU path")
        if y.dim() != 4 or y.shape[1] != 3:
            raise ValueError("expected a [B,3,H,W] colour batch, got %s" % (tuple(y.shape),))
        ths = float(ths.reshape(-1)[0]) if isinstance(ths, torch.Tensor) else float(ths)
        y = y.to(self.device, torch.float32).contiguous()
        shape = _lib.ImgShape(int(y.shape[0]), 3, int(y.shape[2]), int(y.shape[3]))
        out = torch.empty_like(y)
        self.apply_post(shape, None, y, _lib.PostParams(1.0, 0.0, 0.0, 1.0), out, ths=ths)  # out = 0 * y + 1 * D(y)
        return out

    __call__ = forward
