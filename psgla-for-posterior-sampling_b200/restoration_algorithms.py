"""Drop-in for the Langevin samplers of the reference's ``restoration_algorithms.py``: ``psgla`` (:163-285) and
``pnpula`` (:38-160; ``pnp_ula`` is the script's ``--alg`` spelling, exported as an alias).

Same positional / keyword arguments and the same return triple ``(Xlist, Xlist_mmse, Xlist_mmse2)`` of device
tensors.  Per iteration the host issues two C-ABI calls: the fused Langevin "pre" kernel and the DnCNN layer chain
whose last layer's epilogue applies the denoiser term, thins samples and updates the running moments.
Extra keyword-only arguments:
  noise          tensor (n_iter, *init.shape) of N(0,1) draws to replay (e.g. the reference's torch.randn stream)
  rng            default: "torch_cuda" for a single chain (so that ``seed=k`` alone reproduces the reference's CUDA run), "philox"
                 when ``n_chains`` is given.  "philox": in-kernel Philox4x32-10, keyed by seed / chain id / iteration; "torch"
                 (draw ``torch.randn(im_shape, generator=Generator(device).manual_seed(seed))`` per iteration exactly
                 like the reference and replay it) or "torch_cuda" (the same stream as "torch" on a CUDA device, generated
                 bit for bit inside the fused kernel from the seed alone: no randn launch, no noise tensor)
  n_chains       run that many independent chains of the same problem (init broadcast); outputs gain a leading
                 chain axis
  chain_id0      global id of the first chain (Philox subsequence) when chains are sharded over GPUs
  store          "all" (default, the reference's behaviour: every thinned sample and every window mean is kept, N=10^4 /
                 n_inter=10 is 1 000 samples + 909 x 2 window moments per chain) or "stats" (statistics-only: no sample is
                 stored -- ``Xlist`` comes back empty -- and the window means are folded into their running average on the
                 device, so ``Xlist_mmse`` / ``Xlist_mmse2`` hold ONE tensor each: the mean over windows the reference's
                 post-processing forms anyway, sampling_images.py:427,436).  What batched runs (64 chains per image) need:
                 memory independent of n_iter.
The data term must be an ``InpaintingDataGrad`` / ``DeblurDataGrad`` and the denoiser a ``psgla_b200.DnCNN`` / ``DRUNet`` /
``GSDRUNet`` (``prior_grad`` a ``PriorGrad`` wrapping one); opaque callables raise ``TypeError`` -- there is no eager fallback.
``GSDRUNet`` needs image sides that are multiples of 8.
Images have the denoiser's channel count: 3 (colour), or 1 (grayscale, the reference's ``--grayscale`` runs) with a
``DnCNN`` / ``DRUNet`` built with ``in_channels = out_channels = 1``.  ``TVDenoiser`` and ``GSDRUNet`` are colour-only.
``psgla`` / ``psgla_run`` / ``pnp`` also take a ``psgla_b200.TVDenoiser`` (PSGLA-TV): each iteration is then the "pre" launch and
one cooperative launch of the TV prox with the post fused (csrc/tv_prox.cu), at any image size.  ``pnpula`` and ``red`` feed
the denoiser X instead of the fp32 base and reject it.
"""
from __future__ import annotations

import ctypes as C
import math

import numpy as np
import torch

from . import _lib
from .denoisers import DRUNet, DnCNN, GSDRUNet, TVDenoiser
from .operators import DeblurDataGrad, InpaintingDataGrad, PriorGrad

__all__ = ["psgla", "pnpula", "pnp_ula", "psgla_run", "pnpula_run", "pnp", "red"]


def _f(v):
    return float(v.item()) if isinstance(v, torch.Tensor) else float(v)


class _Run:
    """State shared by both samplers: buffers, thinning, running moments (restoration_algorithms.py:118-144)."""

    def __init__(self, init, data_grad, denoiser, n_iter, n_inter, n_inter_mmse, seed, noise, rng, n_chains, chain_id0,
                 store="all"):
        _lib.require_cuda()
        if store not in ("all", "stats"):
            raise ValueError("store must be 'all' or 'stats'")
        self.store = store
        if not isinstance(data_grad, (InpaintingDataGrad, DeblurDataGrad)):
            raise TypeError("data_grad must be an InpaintingDataGrad or DeblurDataGrad (structured callable); an opaque "
                            "callable cannot be fused into the CUDA kernels and there is no eager fallback")
        if not isinstance(denoiser, (DnCNN, DRUNet, GSDRUNet, TVDenoiser)):
            raise TypeError("denoiser must be a psgla_b200.DnCNN, DRUNet, GSDRUNet or (psgla / pnp only) TVDenoiser")
        if seed is None and noise is None:
            raise ValueError("seed=None: the reference fails with UnboundLocalError here "
                             "(restoration_algorithms.py:211-213,232); pass a seed or a noise tensor")
        if not init.is_cuda:
            raise RuntimeError("init must be a CUDA tensor: there is no CPU path")
        self.dg, self.den = data_grad, denoiser
        self.device = init.device
        x = init.detach().to(torch.float32)
        if x.dim() == 3:
            x = x[None]
        Cn = int(denoiser.channels)  # 3, or 1 for a grayscale DnCNN / DRUNet
        if x.dim() != 4 or x.shape[1] != Cn:
            raise ValueError("init must be a [B,%d,H,W] (or [%d,H,W]) %s image batch to match the %d-channel %s%s, got %s" %
                             (Cn, Cn, "colour" if Cn == 3 else "grayscale", Cn, type(denoiser).__name__,
                              " (colour-only)" if isinstance(denoiser, (TVDenoiser, GSDRUNet)) else "", tuple(init.shape)))
        self.squeeze = n_chains is None and x.shape[0] == 1
        B = int(n_chains) if n_chains is not None else int(x.shape[0])
        # DRUNet halves the resolution three times.  Sides that are not multiples of 8 (CBSD68: 481 x 321) are handled like KAIR's
        # test_pad, which deepinv's DRUNet applies per call: the network sees the image replication-padded at the bottom / right
        # and its output is cropped.  Here the whole problem is carried at the padded size -- the pad region is unobserved
        # (mask 0), its state never feeds back because the denoiser input's pad pixels are re-filled from the edge before every
        # network application (psgla_img_pad_replicate_nhwc16) -- and every returned tensor is cropped.  Inpainting only: the
        # circular blur of the deblurring problem is defined on the true image size.
        self.crop = None
        if isinstance(denoiser, GSDRUNet):
            denoiser.check_size(int(x.shape[2]), int(x.shape[3]))
        if isinstance(denoiser, DRUNet) and (x.shape[2] % 8 or x.shape[3] % 8):
            if not isinstance(data_grad, InpaintingDataGrad):
                raise RuntimeError("DRUNet needs H and W to be multiples of 8 for deblurring problems (crop the image, e.g. "
                                   "481 x 321 -> 480 x 320); inpainting problems are padded internally")
            self.crop = (int(x.shape[2]), int(x.shape[3]))
            ph, pw = (-x.shape[2]) % 8, (-x.shape[3]) % 8
            x = torch.nn.functional.pad(x, (0, pw, 0, ph), mode="replicate")
            if noise is not None:
                noise = torch.nn.functional.pad(noise.reshape((noise.shape[0], -1, Cn) + self.crop).to(self.device, torch.float32),
                                                (0, pw, 0, ph))
        self.X = x.expand(B, -1, -1, -1).contiguous().clone() if x.shape[0] != B else x.contiguous().clone()
        self.shape = _lib.ImgShape(B, Cn, int(x.shape[2]), int(x.shape[3]))
        self.base = torch.empty_like(self.X)
        _, self.den_in = denoiser.buffers(self.shape)
        self.n_iter, self.n_inter = int(n_iter), int(n_inter)
        self.n_inter_mmse = int(n_inter if n_inter_mmse is None else n_inter_mmse)
        if self.n_inter < 1:
            raise ZeroDivisionError("integer modulo by zero (n_inter must be >= 1, as in the reference)")
        n_samples = (self.n_iter + self.n_inter - 1) // self.n_inter
        self.samples = None
        if store == "all":
            self.samples = torch.empty((max(n_samples, 1),) + tuple(self.X.shape), dtype=torch.float32, device=self.device)
        self.n_windows, self.win_sum, self.win_sum2 = 0, None, None  # statistics-only: running sums of the window means
        self.mean = torch.zeros_like(self.X)
        self.mean2 = torch.zeros_like(self.X)
        # closed windows are copied into storage reserved in chunks, so that no allocator call (a device-wide
        # synchronisation when it reaches cudaMalloc) lands inside the iteration loop
        self._win_left = self.n_iter // (self.n_inter_mmse + 1)
        self._win_chunk, self._win_used = None, 0
        self.Xlist, self.Xlist_mmse, self.Xlist_mmse2 = [], [], []
        self.iter_mmse = 0
        self.seed = 0 if seed is None else int(seed)
        self.chain_id0 = int(chain_id0)
        self.noise = noise
        self.gen = None
        self.torch_threads = self.torch_step = 0
        if rng is None:
            rng = "torch_cuda" if n_chains is None else "philox"
        if noise is None and rng == "torch":
            self.gen = torch.Generator(device=self.device)
            self.gen.manual_seed(self.seed)
        elif noise is None and rng == "torch_cuda":
            # torch's launch policy for a randn of X.numel() floats on this device (restoration_algorithms.py:104,232 draw
            # one such tensor per iteration from a private generator, so iteration i starts at offset i * step)
            props = torch.cuda.get_device_properties(self.device)
            threads, step = C.c_uint32(), C.c_uint64()
            _lib.check(_lib.lib().psgla_torch_cuda_randn_policy(self.X.numel(), props.multi_processor_count,
                                                                props.max_threads_per_multi_processor,
                                                                C.byref(threads), C.byref(step)),
                       "psgla_torch_cuda_randn_policy")
            self.torch_threads, self.torch_step = threads.value, step.value
        elif noise is None and rng != "philox":
            raise ValueError("rng must be 'philox', 'torch' or 'torch_cuda'")
        if noise is not None and tuple(noise.shape[1:]) != tuple(self.X.shape) and not (
                self.X.shape[0] == 1 and tuple(noise.shape[1:]) == tuple(self.X.shape[1:])):
            raise ValueError("noise must have shape (n_iter, *init.shape)")
        if noise is not None and noise.shape[0] < self.n_iter:
            raise ValueError("noise holds %d draws but n_iter = %d" % (noise.shape[0], self.n_iter))
        H, W = int(self.X.shape[2]), int(self.X.shape[3])

        def operand(t, what, channels):
            t = t.to(self.device)
            if t.dim() == 3:
                t = t[None]
            want = self.crop if self.crop is not None else (H, W)
            if t.dim() != 4 or t.shape[0] not in (1, B) or t.shape[1] not in channels or tuple(t.shape[2:]) != want:
                raise ValueError("%s has shape %s; expected [1 or %d, %s, %d, %d] to match init" %
                                 (what, tuple(t.shape), B, "/".join(str(c) for c in channels), want[0], want[1]))
            if self.crop is not None:  # zero pad: the pad region is unobserved
                t = torch.nn.functional.pad(t, (0, W - want[1], 0, H - want[0]))
            return t.expand(-1, Cn, -1, -1).contiguous()

        if isinstance(data_grad, DeblurDataGrad):
            self.y = operand(data_grad.y, "the blurred observation y", (Cn,))
            self.mask = None
            # A^T(A x - y) = (A^T A) x - A^T y: A^T y is blurred once here, the iterations run the two-pass A^T A kernel
            # (half-widths above 4 take the four-pass kernel: aty = None)
            self.aty = data_grad.AT(self.y) if 1 <= data_grad.l <= 4 else None
        else:
            self.y = operand(data_grad.y, "the observation y", (1, Cn))
            self.mask = operand(data_grad.mask, "the mask", (1, Cn))

    def configure(self, pre, gain, base_scale=1.0):
        self.pre_params, self.gain, self.base_scale = pre, float(gain), float(base_scale)
        # the fused next-iteration pre is a conv-epilogue feature: the TV prox runs one pre launch per iteration
        self.fuse_next_pre = not isinstance(self.den, TVDenoiser)
        self._pre_done_for = None
        self._next_params = _lib.PreParams()

    def step(self, i):
        """Iteration i of the sampler.  Inpainting (``fuse_next_pre``): the conv launches alone -- the last layer's epilogue
        applies the denoiser term, thins, updates the moments AND evaluates iteration i + 1's Langevin "pre" on the fresh
        iterate; only the first iteration of a run of consecutive steps launches the stand-alone "pre" kernel.  Deblurring
        (a stencil: neighbours needed): "pre" kernel, then the conv launches."""
        fuse = self.fuse_next_pre and self.mask is not None and self.noise is None and self.gen is None
        if not fuse or self._pre_done_for != i:
            self.pre(i, self.pre_params)
        nxt = i + 1 if (fuse and i + 1 < self.n_iter) else None
        self.post(i, self.gain, next_iteration=nxt)
        self._pre_done_for = nxt

    def _out(self, t):
        if self.crop is not None:
            t = t[..., :self.crop[0], :self.crop[1]]
        if not self.squeeze:
            return t
        # the reference appends torch.squeeze(X): [3, H, W] for colour, [H, W] for a grayscale chain
        return t[0, 0] if self.shape.C == 1 else t[0]

    def z_for(self, i):
        if self.noise is not None:
            return self.noise[i].to(self.device, torch.float32).reshape(self.X.shape).contiguous()
        if self.gen is not None:
            return torch.randn(self.X.shape, generator=self.gen, dtype=torch.float32, device=self.device)
        return None

    def _stamp(self, pre, i):
        pre.seed, pre.chain_id0, pre.iteration = self.seed, self.chain_id0, i
        if self.torch_threads:
            pre.noise_mode, pre.torch_threads, pre.torch_offset = _lib.NOISE_TORCH_CUDA, self.torch_threads, i * self.torch_step
        else:
            pre.noise_mode = _lib.NOISE_PHILOX

    def pre(self, i, pre: "_lib.PreParams"):
        z = self.z_for(i)
        self._stamp(pre, i)
        lib = _lib.lib()
        with torch.cuda.device(self.device):
            st = _lib.stream_ptr(self.device)
            if self.mask is not None:
                rc = lib.psgla_img_pre_inpaint(C.byref(pre), self.shape, _lib.ptr(self.X), _lib.ptr(self.mask),
                                               int(self.mask.shape[0]), _lib.ptr(self.y), int(self.y.shape[0]),
                                               _lib.ptr(z), _lib.ptr(self.base), _lib.ptr(self.den_in), st)
                _lib.check(rc, "psgla_img_pre_inpaint")
            elif self.aty is not None:
                rc = lib.psgla_img_pre_deblur_ata(C.byref(pre), self.shape, _lib.ptr(self.X), self.dg._taps_c, self.dg.l,
                                                  _lib.ptr(self.aty), int(self.aty.shape[0]), _lib.ptr(z), _lib.ptr(self.base),
                                                  _lib.ptr(self.den_in), st)
                _lib.check(rc, "psgla_img_pre_deblur_ata")
            else:
                rc = lib.psgla_img_pre_deblur(C.byref(pre), self.shape, _lib.ptr(self.X), self.dg._taps_c, self.dg.l,
                                              _lib.ptr(self.y), int(self.y.shape[0]), _lib.ptr(z), _lib.ptr(self.base),
                                              _lib.ptr(self.den_in), st)
                _lib.check(rc, "psgla_img_pre_deblur")

    def post(self, i, gain, next_iteration=None):
        k = self.iter_mmse
        post = _lib.PostParams(float(gain), self.base_scale, float(np.float32(k / (k + 1))), float(np.float32(1 / (k + 1))))
        sample = self.samples[i // self.n_inter] if (self.samples is not None and i % self.n_inter == 0) else None
        nxt = None
        if next_iteration is not None:
            if self.noise is not None or self.gen is not None:
                raise RuntimeError("the fused next-iteration pre generates its noise in the kernel (rng 'philox' / 'torch_cuda')")
            C.memmove(C.byref(self._next_params), C.byref(self.pre_params), C.sizeof(_lib.PreParams))
            self._stamp(self._next_params, next_iteration)
            nxt = _lib.NextPre(C.pointer(self._next_params), _lib.ptr(self.mask), _lib.ptr(self.y), int(self.mask.shape[0]),
                               int(self.y.shape[0]), _lib.ptr(self.base), _lib.ptr(self.den_in))
        if self.crop is not None:  # re-fill the pad pixels of the network input from the image edge (KAIR test_pad)
            with torch.cuda.device(self.device):
                _lib.check(_lib.lib().psgla_img_pad_replicate_nhwc16(self.shape, self.crop[0], self.crop[1], _lib.ptr(self.den_in),
                                                                     _lib.stream_ptr(self.device)), "psgla_img_pad_replicate_nhwc16")
        if isinstance(self.den, TVDenoiser):  # ths = the level the pre carries for non-residual denoisers (pnp anneals it)
            self.den.apply_post(self.shape, self.den_in, self.base, post, self.X, sample, self.mean, self.mean2,
                                ths=self.pre_params.den_in_c3)
        elif isinstance(self.den, GSDRUNet):  # D is evaluated where the pre left the denoiser input: base (PSGLA) or X
            x = self.X if self.pre_params.alg == _lib.ALG_PNPULA else None
            self.den.apply_post(self.shape, self.den_in, self.base, post, self.X, sample, self.mean, self.mean2, next_pre=nxt, x=x)
        else:
            self.den.apply_post(self.shape, self.den_in, self.base, post, self.X, sample, self.mean, self.mean2, next_pre=nxt)
        if sample is not None:
            self.Xlist.append(self._out(sample))
        # window bookkeeping exactly as restoration_algorithms.py:128-144 / :255-271
        if self.iter_mmse <= self.n_inter_mmse - 1:
            self.iter_mmse += 1
        elif self.store == "stats":
            # statistics-only: fold the closed window into the running sums instead of keeping it (the reference's tail
            # averages the window means anyway, sampling_images.py:427,436); Xlist_mmse / Xlist_mmse2 come from finish()
            if self.win_sum is None:
                self.win_sum, self.win_sum2 = self.mean.clone(), self.mean2.clone()
            else:
                self.win_sum.add_(self.mean)
                self.win_sum2.add_(self.mean2)
            self.n_windows += 1
            self.iter_mmse = 0
        else:
            if self._win_chunk is None or self._win_used == self._win_chunk.shape[0]:
                per_window = 2 * self.mean.numel() * 4
                n = max(1, min(max(self._win_left, 1), (1 << 31) // per_window))
                self._win_chunk = torch.empty((n, 2) + tuple(self.mean.shape), dtype=torch.float32, device=self.device)
                self._win_used = 0
            slot = self._win_chunk[self._win_used]
            self._win_used += 1
            self._win_left -= 1
            slot[0].copy_(self.mean)
            slot[1].copy_(self.mean2)
            self.Xlist_mmse.append(self._out(slot[0]))
            self.Xlist_mmse2.append(self._out(slot[1]))
            self.iter_mmse = 0  # the next update has w_old = 0, which restarts the window without a memset


    def finish(self):
        """The reference's return triple.  Statistics-only runs return ([], [mean of the window means], [mean of the window
        second moments]) -- one tensor each, empty lists when no window closed."""
        if self.store == "stats" and self.n_windows:
            self.Xlist_mmse = [self._out(self.win_sum / self.n_windows)]
            self.Xlist_mmse2 = [self._out(self.win_sum2 / self.n_windows)]
        return self.Xlist, self.Xlist_mmse, self.Xlist_mmse2


def _save_online(path, name, i, run, extra):
    # restoration_algorithms.py:146-158 / :273-283 (the PNG previews need matplotlib and are not reproduced)
    d = {"Samples": run.Xlist, "Mmse": run.Xlist_mmse, "Mmse2": run.Xlist_mmse2, "n_iter": run.n_iter}
    d.update(extra)
    torch.save(d, (path or "") + "/" + (name or "") + "_sampling.pth")


def psgla_run(init, data_grad, denoiser, alpha, lambd, sig_float=0.0055, delta=4e-5, n_iter=5000, n_inter=1000,
              n_inter_mmse=1000, seed=None, *, noise=None, rng=None, n_chains=None, chain_id0=0, store="all"):
    """The stepping object behind ``psgla``: ``run.step(i)`` issues iteration i (one "pre" launch + the DnCNN layer
    chain); ``run.Xlist`` / ``run.Xlist_mmse`` / ``run.Xlist_mmse2`` are the reference's three lists."""
    run = _Run(init, data_grad, denoiser, n_iter, n_inter, n_inter_mmse, seed, noise, rng, n_chains, chain_id0, store)
    delta32 = float(np.float32(delta))
    sig32 = float(np.float32(sig_float))
    pre = _lib.PreParams()
    pre.alg = _lib.ALG_PSGLA
    pre.gain_data = (delta32 / _f(lambd)) / run.dg.sigma2
    pre.noise_scale = float(np.float32(np.float32(np.sqrt(2)) * np.float32(sig32)))
    pre.proj_gain, pre.c_min, pre.c_max, pre.x_gain = 0.0, 0.0, 0.0, 0.0
    if denoiser.is_residual:  # DnCNN: (1-alpha) Y + alpha (Y + R(Y)) = Y + alpha R(Y)
        pre.den_in_c3 = 0.0
        run.configure(pre, _f(alpha))
    else:  # DRUNet / TV: (1-alpha) Y + alpha D(Y; sig), sig = the noise-level map in channel 3 resp. ths (restoration_algorithms.py:238)
        pre.den_in_c3 = sig32
        run.configure(pre, _f(alpha), 1.0 - _f(alpha))
    return run


def psgla(init, data_grad, denoiser, alpha, lambd, sig_float=0.0055, delta=4e-5, n_iter=5000, n_inter=1000,
          n_inter_mmse=1000, seed=None, device=None, path=None, save_images_online=False, name=None, *, noise=None,
          rng=None, n_chains=None, chain_id0=0, store="all"):
    """PSGLA (restoration_algorithms.py:163-285):  Y = X + (delta/lambd) data_grad(X) + sqrt(2) sig Z;
    X = (1 - alpha) Y + alpha D(Y).  Returns (Xlist, Xlist_mmse, Xlist_mmse2)."""
    run = psgla_run(init, data_grad, denoiser, alpha, lambd, sig_float, delta, n_iter, n_inter, n_inter_mmse, seed,
                    noise=noise, rng=rng, n_chains=n_chains, chain_id0=chain_id0, store=store)
    print("delta = {}, sigma = {}".format(delta, sig_float))
    K = int(run.n_iter / 10)
    for i in range(run.n_iter):
        run.step(i)
        if save_images_online and i % K == 0:  # ZeroDivisionError for n_iter < 10 with the flag, as in the reference (:246)
            _save_online(path, name, i, run, {"lambda": lambd, "delta": delta})
    return run.finish()


def pnpula_run(init, data_grad, prior_grad, delta, lambd, n_iter=5000, n_inter=1000, n_inter_mmse=1000, seed=None,
               c_min=-1, c_max=2, *, noise=None, rng=None, n_chains=None, chain_id0=0, store="all"):
    """The stepping object behind ``pnpula`` (see ``psgla_run``)."""
    if not isinstance(prior_grad, PriorGrad):
        raise TypeError("prior_grad must be a PriorGrad(denoiser, alpha, s1, s2) structured callable")
    if isinstance(prior_grad.denoiser, TVDenoiser):
        raise TypeError("pnpula supports a psgla_b200.DnCNN or psgla_b200.DRUNet prior, not the TV prox")
    run = _Run(init, data_grad, prior_grad.denoiser, n_iter, n_inter, n_inter_mmse, seed, noise, rng, n_chains, chain_id0,
               store)
    delta_f, lambd_f = _f(delta), _f(lambd)
    pre = _lib.PreParams()
    pre.alg = _lib.ALG_PNPULA
    pre.gain_data = delta_f / run.dg.sigma2
    pre.noise_scale = float(np.float32(math.sqrt(2 * delta_f)))
    pre.proj_gain = delta_f / lambd_f
    pre.c_min, pre.c_max = float(c_min), float(c_max)
    g = delta_f * prior_grad.alpha / prior_grad.s2  # delta * prior_grad = g (D(X; s1) - X)   (sampling_images.py:156-157)
    if prior_grad.denoiser.is_residual:
        pre.x_gain, pre.den_in_c3 = 0.0, 0.0  # D(X) - X is the network output itself
    else:
        pre.x_gain, pre.den_in_c3 = -g, prior_grad.s1
    run.configure(pre, g)
    return run


def pnpula(init, data_grad, prior_grad, delta, lambd, n_iter=5000, n_inter=1000, n_inter_mmse=1000, seed=None,
           device=None, c_min=-1, c_max=2, path=None, save_images_online=False, name=None, *, noise=None, rng=None,
           n_chains=None, chain_id0=0, store="all"):
    """PnP-ULA (restoration_algorithms.py:38-160):
    X+ = X + delta (prior_grad(X) - (X - proj_[c_min,c_max] X)/lambd + data_grad(X)) + sqrt(2 delta) Z."""
    run = pnpula_run(init, data_grad, prior_grad, delta, lambd, n_iter, n_inter, n_inter_mmse, seed, c_min, c_max,
                     noise=noise, rng=rng, n_chains=n_chains, chain_id0=chain_id0, store=store)
    print("delta = {}".format(delta.float() if isinstance(delta, torch.Tensor) else delta))
    K = int(run.n_iter / 10)
    for i in range(run.n_iter):
        run.step(i)
        if save_images_online and i % K == 0:
            _save_online(path, name, i, run, {"c_min": c_min, "c_max": c_max, "lambda": lambd, "delta": delta})
    return run.finish()


pnp_ula = pnpula


def pnp(init, data_grad, Pb, denoiser, alpha, lambd, sig_float=0.0055, delta=1e-5, n_iter=500, device=None, path=None,
        save_images_online=False, name=None, *, n_chains=None):
    """PnP forward-backward (restoration_algorithms.py:386-463): PSGLA without the noise.  Y = X + (delta/lambd)
    data_grad(X); X = (1 - alpha) Y + alpha D(Y; sig_den), sig_den = 40/255 for the first n_iter // 10 iterations of an
    inpainting problem, else sig_float (only DRUNet reads it).  Returns (all iterates, [last iterate], [])."""
    run = psgla_run(init, data_grad, denoiser, alpha, lambd, sig_float, delta, n_iter, 1, max(int(n_iter), 1), seed=0,
                    rng="philox", n_chains=n_chains)
    run.pre_params.noise_scale = 0.0
    run.fuse_next_pre = False  # the noise-level map of iteration i + 1 is only known at iteration i + 1 (annealing schedule)
    print("delta = {}, sigma = {}".format(delta, sig_float))
    sig32 = float(np.float32(sig_float))
    for i in range(run.n_iter):
        if not denoiser.is_residual:
            run.pre_params.den_in_c3 = 40.0 / 255.0 if (Pb == "inpainting" and i < run.n_iter // 10) else sig32
        run.step(i)
    return run.Xlist, [run._out(run.X.clone())], []


def red(init, data_grad, Pb, denoiser, lambd, sig_float=0.0055, delta=1e-5, n_iter=500, device=None, path=None,
        save_images_online=False, name=None, *, n_chains=None):
    """RED (restoration_algorithms.py:465-529): X+ = X + delta data_grad(X) - delta lambd (X - D(X; sig_den)), sig_den =
    50/255 for the first 10 iterations of an inpainting problem.  Returns (all iterates, [last iterate], [])."""
    if not isinstance(denoiser, (DnCNN, DRUNet, GSDRUNet)):
        raise TypeError("denoiser must be a psgla_b200.DnCNN, DRUNet or GSDRUNet")
    run = _Run(init, data_grad, denoiser, n_iter, 1, max(int(n_iter), 1), 0, None, "philox", n_chains, 0)
    delta32 = float(np.float32(delta))
    g = delta32 * _f(lambd)
    pre = _lib.PreParams()
    pre.alg = _lib.ALG_PNPULA  # the denoiser sees X; the projection term is switched off
    pre.gain_data = delta32 / run.dg.sigma2
    pre.noise_scale, pre.proj_gain, pre.c_min, pre.c_max = 0.0, 0.0, 0.0, 0.0
    pre.x_gain = 0.0 if denoiser.is_residual else -g
    run.configure(pre, g)
    run.fuse_next_pre = False
    print("delta = {}, sigma = {}".format(delta, sig_float))
    sig32 = float(np.float32(sig_float))
    for i in range(run.n_iter):
        pre.den_in_c3 = 0.0 if denoiser.is_residual else (50.0 / 255.0 if (i < 10 and Pb == "inpainting") else sig32)
        run.step(i)
    return run.Xlist, [run._out(run.X.clone())], []
