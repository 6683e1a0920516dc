"""Image sets sharded over GPUs: the outer loop of the reference's driver script (sampling_images.py:265-277 iterates over
the dataset, :351/:358 runs one sampler per image, :371-442 reduces it to PSNR / SSIM / MMSE / std) for BATCHES of
independent chains per image -- BASELINE.json configs[4]: "64 chains per image, images sharded across 8 x B200".

``run_image_set`` deals the images round-robin over the ranks of the default ``torch.distributed`` group (image i belongs
to rank i % world_size; SURVEY.md section 8e), runs ``n_chains`` chains of every local image in statistics-only mode
(``store="stats"``: memory independent of the iteration count), reduces each image to the reference's summary numbers on the
device, and gathers the rows on rank 0.  The Philox subsequence of chain c of image i is ``i * n_chains + c`` whatever the
world size, so the gathered results do not depend on how many GPUs ran them.  No communication inside the sampling loop.
"""
from __future__ import annotations

import torch

from . import dist as _dist
from . import metrics as _metrics
from .denoisers import DnCNN, GSDRUNet, TVDenoiser
from .operators import PriorGrad, make_deblurring, make_inpainting
from .params import as_pnpula_kwargs, as_psgla_kwargs, sampler_params
from .restoration_algorithms import pnpula, psgla

__all__ = ["run_image_set", "load_image", "deal_round_robin", "ROW_FIELDS"]

# one gathered row per image
ROW_FIELDS = ("index", "psnr_mmse", "ssim_mmse", "psnr_chain_mean", "psnr_chain_min", "psnr_chain_max", "ssim_chain_mean",
              "psnr_observation", "std_mean", "std_max", "n_chains", "n_windows", "H", "W")


def load_image(path, device=None, n_channels=3):
    """An image file as the reference reads it (sampling_images.py:268-276: ``imread_uint`` -> uint8 -> float32 / 255 ->
    [1, n_channels, H, W]).  ``n_channels=3``: RGB.  ``n_channels=1`` (the reference's ``--grayscale`` runs): the file is read
    as ``cv2.imread(path, 0)``, which is KAIR's ``imread_uint(path, n_channels=1)`` as recalled -- that rule cannot be checked
    against KAIR here, so a colour file's conversion to gray may differ from the reference's."""
    import cv2
    import numpy as np
    if n_channels not in (1, 3):
        raise ValueError("n_channels must be 1 or 3")
    if n_channels == 1:
        gray = cv2.imread(path, 0)
        if gray is None:
            raise FileNotFoundError(path)
        t = torch.from_numpy(np.ascontiguousarray(np.float32(gray / 255.0))).float()[None, None]
        return t if device is None else t.to(device)
    bgr = cv2.imread(path, cv2.IMREAD_COLOR)
    if bgr is None:
        raise FileNotFoundError(path)
    rgb = cv2.cvtColor(bgr, cv2.COLOR_BGR2RGB)
    t = torch.from_numpy(np.ascontiguousarray(np.transpose(np.float32(rgb / 255.0), (2, 0, 1)))).float()[None]
    return t if device is None else t.to(device)


def deal_round_robin(n_items: int, rank: int, world_size: int):
    """Indices of the items rank ``rank`` owns: i with i % world_size == rank (SURVEY.md section 8e)."""
    if world_size < 1 or not (0 <= rank < world_size) or n_items < 0:
        raise ValueError("bad deal request")
    return list(range(rank, n_items, world_size))


def _sample_image(index, im, denoiser, problem, alg, n_chains, prm, seed, seed_ip, prop, sigma, l, blur_type, si, keep_maps):
    """All chains of ONE image on this rank's GPU -> (row tensor [len(ROW_FIELDS)] float64, maps or None)."""
    dev = denoiser.device
    im = im.to(dev, torch.float32)
    if im.dim() == 3:
        im = im[None]
    if problem == "inpainting":
        dg, init, y, _ = make_inpainting(im, prop=prop, sigma=sigma, seed_ip=seed_ip)
    elif problem == "deblurring":
        dg, init, y = make_deblurring(im, l=l, blur_type=blur_type, si=si, sigma=sigma, seed_ip=seed_ip)
    else:
        raise ValueError("problem must be 'inpainting' or 'deblurring'")
    kw = dict(n_chains=n_chains, chain_id0=index * n_chains, store="stats", rng="philox")
    if isinstance(denoiser, TVDenoiser):
        # every image starts the prox from x2 = y, u2 = 0, so a row does not depend on which images this rank ran before
        # it (the reference warm-starts across the images of its loop)
        denoiser.reset()
    if alg == "psgla":
        _, M, M2 = psgla(init, dg, denoiser, **as_psgla_kwargs(prm, seed=seed), **kw)
    elif alg in ("pnp_ula", "pnpula"):
        pg = PriorGrad(denoiser, prm["alpha"], prm["s1"], prm["s2"])
        k = as_pnpula_kwargs(prm, seed=seed)
        delta, lambd = k.pop("delta"), k.pop("lambd")
        _, M, M2 = pnpula(init, dg, pg, torch.tensor(delta, device=dev), torch.tensor(lambd, device=dev), **k, **kw)
    else:
        raise ValueError("alg must be 'psgla' or 'pnp_ula'")
    if not M:
        raise ValueError("no statistics window closed: n_iter = %d must exceed n_inter_mmse = %d" % (prm["N"], prm["n_inter_mmse"]))
    M, M2 = M[0], M2[0]  # [n_chains, C, H, W]: per-chain mean of the window means / second moments
    xmmse = M.mean(0)    # chains are exchangeable: the pooled posterior mean (sampling_images.py:427 over chains as well)
    var = M2.mean(0) - xmmse ** 2
    std = torch.sqrt(torch.clamp(var, min=0.0))  # :436-439
    p_pool, s_pool = _metrics.psnr_ssim(xmmse, im[0])
    p_chain, s_chain = _metrics.psnr_ssim(M, im[0])
    p_obs, _ = _metrics.psnr_ssim(y[0], im[0])
    n_windows = prm["N"] // (prm["n_inter_mmse"] + 1)
    row = torch.stack([torch.tensor(float(index), device=dev, dtype=torch.float64), p_pool[0].double(), s_pool[0].double(),
                       p_chain.double().mean(), p_chain.double().min(), p_chain.double().max(), s_chain.double().mean(),
                       p_obs[0].double(), std.double().mean(), std.double().max(),
                       torch.tensor(float(n_chains), device=dev, dtype=torch.float64),
                       torch.tensor(float(n_windows), device=dev, dtype=torch.float64),
                       torch.tensor(float(im.shape[2]), device=dev, dtype=torch.float64),
                       torch.tensor(float(im.shape[3]), device=dev, dtype=torch.float64)])
    return row, ((xmmse, std) if keep_maps else None)


def run_image_set(images, denoiser=None, problem="inpainting", alg="psgla", n_chains=64, n_iter=None, params=None, seed=0,
                  seed_ip=0, prop=0.5, sigma=1.0, l=4, blur_type="uniform", si=1.0, keep_maps=False, _sample=None):
    """Posterior sampling of a SET of images, ``n_chains`` independent chains each, sharded over the process group.

    images     list of [C, H, W] / [1, C, H, W] float tensors in [0, 1] (sizes may differ), the same list on every rank; C = the
               denoiser's channel count (1: grayscale images with a one-channel DnCNN / DRUNet)
    denoiser   this rank's ``psgla_b200.DnCNN`` / ``DRUNet`` / ``GSDRUNet`` / ``TVDenoiser`` (default: a DnCNN with the library's seeded
               weights; TV: psgla only, table row ``den="TV"``, the prox state is reset before each image)
    params     the dict of ``psgla_b200.sampler_params`` (default: the script's table for ``alg`` / the denoiser family, with
               ``N = n_iter`` when given)
    Returns, on rank 0, a list of dicts (one per image, in input order) with the keys of ``ROW_FIELDS`` (+ ``xmmse`` / ``std``
    maps of the images this rank ran when ``keep_maps``); ``None`` on the other ranks."""
    rank, ws = _dist.world()
    if _sample is None:
        if denoiser is None:
            denoiser = DnCNN()
        den_name = ("DnCNN" if isinstance(denoiser, DnCNN) else "TV" if isinstance(denoiser, TVDenoiser)
                    else "GSDRUNet" if isinstance(denoiser, GSDRUNet) else "DRUNet")
        prm = dict(params) if params is not None else sampler_params("pnp_ula" if alg in ("pnp_ula", "pnpula") else alg, den=den_name,
                                                                     sigma=sigma, N=n_iter)
        if n_iter is not None:
            prm["N"] = int(n_iter)

        def _sample(index, im):  # noqa: E306
            return _sample_image(index, im, denoiser, problem, alg, int(n_chains), prm, seed, seed_ip, prop, sigma, l, blur_type,
                                 si, keep_maps)
    mine = deal_round_robin(len(images), rank, ws)
    rows, maps = [], {}
    for i in mine:
        row, mp = _sample(i, images[i])
        rows.append(row.reshape(1, -1))
        if mp is not None:
            maps[i] = mp
    width = len(ROW_FIELDS)
    if rows:
        local = torch.cat(rows, 0)
    else:  # more ranks than images: an empty block of the right width and device
        ref_dev = denoiser.device if denoiser is not None else "cpu"
        local = torch.zeros((0, width), dtype=torch.float64, device=ref_dev)
    table = _dist.gather_to_rank0(local, n_total=len(images) if ws > 1 else None)
    if rank != 0:
        return None
    table = table[torch.argsort(table[:, 0])].cpu()
    out = []
    for r in table:
        d = {k: (int(v) if k in ("index", "n_chains", "n_windows", "H", "W") else float(v)) for k, v in zip(ROW_FIELDS, r.tolist())}
        if d["index"] in maps:
            d["xmmse"], d["std"] = maps[d["index"]]
        out.append(d)
    return out
