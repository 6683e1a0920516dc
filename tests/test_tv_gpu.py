"""-m gpu: the TV prox (csrc/tv_prox.cu, ``psgla_b200.TVDenoiser``) against the restated deepinv algorithm (tests/tv_reference.py,
PARITY UNPINNED against deepinv itself), and PSGLA-TV through the samplers.

Stated tolerances (observed values are printed by ``observed``; bounds are about 4x the values measured on a B200)
  * the prox with crit = 0 against the fp64 restatement: fp32 state and arithmetic, so the error grows with the iteration
    count; bounds on max |x2 - ref| and max |u2 - ref| / ths per (shape, n_it_max);
  * sampler iterates under replayed noise against the fp32 restatement: the prox stops at crit = 1e-5, and a stopping test on
    the other side of the threshold moves the result by about crit times the step; bound per iterate.
Bit-exact where the arithmetic is the same: a chain alone vs in a batch, a repeated call, the post against torch ops."""
import os

import numpy as np
import pytest
import torch

import psgla_b200 as P
from oracle import image_oracle as io_
from conftest import GOLDEN, observed
import tv_reference as TV

pytestmark = pytest.mark.gpu

S_TV = 10.0 / 255.0             # the table's TV row (sampling_images.py:181-184)
LAMBD_GAIN1 = S_TV ** 2 / (1.0 / 255.0) ** 2  # lambda = 100: data-step gain (delta / lambda) / sigma^2 = 1 at sigma = 1/255
TOL_SAMPLER = 2e-4


def _image(name, H=None, W=None):
    im = P.load_image(os.path.join(GOLDEN, name), device="cuda")
    return im if H is None else im[..., :H, :W].contiguous()


def _noisy(shape, seed, scale=S_TV):
    g = torch.Generator(device="cuda").manual_seed(seed)
    base = torch.rand(shape[:2] + (1, 1), generator=g, device="cuda")
    # a piecewise-smooth field plus noise: a prox that is neither the identity nor a constant
    H, W = shape[2], shape[3]
    yy = torch.linspace(0, 1, H, device="cuda")[:, None]
    xx = torch.linspace(0, 1, W, device="cuda")[None, :]
    field = base * (yy > 0.4) + (1 - base) * torch.sin(6 * xx) * 0.5
    return (field + scale * torch.randn(shape, generator=g, device="cuda")).contiguous()


def _prox(den, y, ths):
    """One psgla_tv_prox_post call through the Python object; returns (x_out, x2, u2, iterations)."""
    out = den.forward(y, ths)
    torch.cuda.synchronize()
    return out, den.x2.clone(), den.u2.clone(), den.last_iterations.cpu().tolist()


# bounds per CP iteration count, fp32 kernel vs fp64 restatement, at ths = 0.1: max |x2 - ref| and max |u2 - ref| / ths.  Largest
# values measured over the shapes below on a B200 (1000 W): x2 2.4e-7 / 4.6e-7 / 6.5e-7 / 2.0e-6 / 4.5e-6, u2 / ths 5.9e-5 / 8.3e-5
# / 1.3e-4 / 4.7e-4 / 5.4e-4 after 1 / 2 / 3 / 50 / 300 iterations.  The dual step multiplies x's rounding by sigma = 12.5.
X2_BOUND = {1: 1e-6, 2: 2e-6, 3: 3e-6, 50: 8e-6, 300: 2e-5}
U2_BOUND = {1: 2.5e-4, 2: 3.5e-4, 3: 5e-4, 50: 2e-3, 300: 2.5e-3}


@pytest.mark.parametrize("n_it", [1, 2, 3, 50, 300])
@pytest.mark.parametrize("B,H,W", [(1, 1, 1), (1, 1, 37), (1, 41, 1), (2, 33, 47), (1, 256, 256), (1, 321, 481), (1, 481, 321)])
def test_prox_against_fp64_oracle(B, H, W, n_it):
    y = _noisy((B, 3, H, W), seed=H * 1000 + W)
    ths = 0.1
    den = P.TVDenoiser(n_it_max=n_it, crit=0.0)
    out, x2, u2, iters = _prox(den, y, ths)
    ref = TV.TVDenoiser(n_it_max=n_it, crit=0.0)
    want = ref.forward(y.double(), ths)
    assert iters == [n_it] * B
    assert torch.equal(out, x2)
    observed("prox |x2 - fp64| n=%d %dx%dx%d" % (n_it, B, H, W), (x2.double() - want).abs().max().item(), X2_BOUND[n_it])
    observed("prox |u2 - fp64|/ths n=%d %dx%dx%d" % (n_it, B, H, W), (u2.double() - ref.u2).abs().max().item() / ths,
             U2_BOUND[n_it])


def test_iteration_count_at_default_crit():
    """crit = 1e-5 on a noisy 256^2 photograph at ths = s = 10/255: the count is within 1 of the restatement's in fp64 and fp32."""
    im = _image("set3c/butterfly.png")
    y = (im + S_TV * torch.randn(im.shape, generator=torch.Generator(device="cuda").manual_seed(0), device="cuda")).contiguous()
    den = P.TVDenoiser()
    _, x2, _, iters = _prox(den, y, S_TV)
    r64, r32 = TV.TVDenoiser(), TV.TVDenoiser()
    w64 = r64.forward(y.double(), S_TV)
    r32.forward(y, S_TV)
    print("CP iterations: kernel %d, fp64 %d, fp32 %d" % (iters[0], r64.calls[0][0], r32.calls[0][0]))
    assert abs(iters[0] - r64.calls[0][0]) <= 1 and abs(iters[0] - r32.calls[0][0]) <= 1
    assert 3 < iters[0] < 1000
    observed("prox |x2 - fp64| at crit 1e-5", (x2.double() - w64).abs().max().item(), 2e-4)


def test_warm_start_three_calls():
    """Three chained calls (the state carries over, y changes) against three chained calls of the restatement."""
    den = P.TVDenoiser(n_it_max=60, crit=0.0)
    ref = TV.TVDenoiser(n_it_max=60, crit=0.0)
    ex = eu = 0.0
    for call in range(3):
        y = _noisy((2, 3, 40, 56), seed=call)
        out, x2, u2, _ = _prox(den, y, 0.05)
        want = ref.forward(y.double(), 0.05)
        ex = max(ex, (out.double() - want).abs().max().item())
        eu = max(eu, (u2.double() - ref.u2).abs().max().item() / 0.05)
    observed("warm-started prox x2 vs fp64, 3 calls", ex, 2e-5)
    observed("warm-started prox u2 / ths vs fp64, 3 calls", eu, 5e-3)
    # a restart forgets the state: equal to a fresh object's first call
    den.reset()
    y = _noisy((2, 3, 40, 56), seed=9)
    assert torch.equal(den.forward(y, 0.05), P.TVDenoiser(n_it_max=60, crit=0.0).forward(y, 0.05))


def test_batch_independence_freezing_and_determinism():
    """Each chain of a B = 5 batch equals that chain run alone bit for bit (output, state, count); a constant chain stops at 3
    while the others go on; a repeated call is bit-identical."""
    y = torch.cat([_noisy((1, 3, 70, 90), seed=s, scale=0.05 * (s + 1)) for s in range(5)]).contiguous()
    y[2] = 0.3
    den = P.TVDenoiser()
    out, x2, u2, iters = _prox(den, y, S_TV)
    print("CP iterations per chain:", iters)
    assert iters[2] == 3 and all(n > 3 for i, n in enumerate(iters) if i != 2)
    for b in range(5):
        a = P.TVDenoiser()
        ob, xb, ub, nb = _prox(a, y[b:b + 1].contiguous(), S_TV)
        assert nb == [iters[b]], b
        assert torch.equal(ob[0], out[b]) and torch.equal(xb[0], x2[b]) and torch.equal(ub[0], u2[b]), b
    den.reset()
    out2, x22, u22, iters2 = _prox(den, y, S_TV)
    assert iters2 == iters and torch.equal(out2, out) and torch.equal(x22, x2) and torch.equal(u22, u2)


def test_post_bit_exact():
    """x_out = fma(gain, D, fl(base_scale * y)), sample = x_out, mean / mean2 = three rounded fp32 operations, with D the returned
    state x2; x_out aliasing y."""
    B, H, W = 3, 37, 53
    y = _noisy((B, 3, H, W), seed=5)
    y0 = y.clone()
    g = torch.Generator(device="cuda").manual_seed(6)
    mean0, mean20 = torch.rand(y.shape, generator=g, device="cuda"), torch.rand(y.shape, generator=g, device="cuda")
    mean, mean2, sample = mean0.clone(), mean20.clone(), torch.empty_like(y)
    den = P.TVDenoiser()
    shape = P._lib.ImgShape(B, 3, H, W)
    den.buffers(shape)
    w_old, w_new = float(np.float32(3 / 4)), float(np.float32(1 / 4))
    post = P._lib.PostParams(0.7, 0.3, w_old, w_new)
    den.apply_post(shape, None, y, post, y, sample, mean, mean2, ths=S_TV)  # x_out = y, in place
    torch.cuda.synchronize()
    D = den.x2.double()
    bs_y = (torch.tensor(0.3, dtype=torch.float32) * y0).double()
    want = (np.float32(0.7) * D + bs_y).float()  # the product is exact in fp64: only the final rounding remains
    assert torch.equal(y, want)
    assert torch.equal(sample, y)
    assert torch.equal(mean, w_old * mean0 + w_new * y)
    assert torch.equal(mean2, w_old * mean20 + w_new * (y * y))
    assert den.last_iterations.dtype == torch.int32 and den.last_iterations.is_cuda


def _replay_noise(shape, n_iter, seed=0):
    g = torch.Generator(device="cuda").manual_seed(seed)
    return torch.stack([torch.randn(shape, generator=g, device="cuda") for _ in range(n_iter)])


def _psgla_kw(n_iter, n_inter=1, n_mm=4, alpha=1.0):
    return dict(alpha=torch.tensor(alpha, device="cuda"), lambd=torch.tensor(LAMBD_GAIN1, device="cuda"), sig_float=S_TV,
                delta=S_TV ** 2, n_iter=n_iter, n_inter=n_inter, n_inter_mmse=n_mm, seed=0)


@pytest.mark.parametrize("problem,H,W", [("inpainting", 64, 64), ("deblurring", 48, 40)])
def test_psgla_tv_replay_against_oracle(problem, H, W):
    im = _image("set3c/leaves.png", H, W)
    if problem == "inpainting":
        dg, init, y, _ = P.make_inpainting(im)
        ref_dg = dg
    else:
        dg, init, y = P.make_deblurring(im, l=2, blur_type="uniform")
        h = P.blur_taps(2, "uniform")
        ref_dg = lambda x: io_.deblur_data_grad(x, h, 2, y, dg.sigma2)  # noqa: E731
    n_iter = 20
    noise = _replay_noise(im.shape, n_iter)
    kw = _psgla_kw(n_iter, alpha=0.9)
    ref = TV.TVDenoiser()
    Xr, Mr, M2r = io_.psgla(init, ref_dg, ref, device="cuda", noise=noise, **kw)
    den = P.TVDenoiser()
    Xg, Mg, M2g = P.psgla(init, dg, den, noise=noise, **kw)
    assert len(Xg) == len(Xr) == n_iter and len(Mg) == len(Mr) and len(M2g) == len(M2r)
    assert Xg[0].shape == (3, H, W)
    print("oracle CP iterations per PSGLA iteration:", [c[0] for c in ref.calls])
    observed("PSGLA-TV %s iterate vs oracle" % problem, max((a - b).abs().max().item() for a, b in zip(Xr + Mr + M2r, Xg + Mg + M2g)),
             TOL_SAMPLER)


def test_pnp_tv_annealed_threshold_against_oracle():
    """pnp anneals the denoiser level (40/255 for the first n_iter // 10 iterations of inpainting); the TV prox reads it as ths."""
    im = _image("set3c/starfish.png", 64, 64)
    dg, init, y, _ = P.make_inpainting(im)
    n_iter = 30
    kw = dict(alpha=0.9, lambd=LAMBD_GAIN1, sig_float=S_TV, delta=S_TV ** 2, n_iter=n_iter)
    ref = TV.TVDenoiser()
    Xr, Lr, _ = io_.pnp(init, dg, "inpainting", ref, device="cuda", **kw)
    Xg, Lg, _ = P.pnp(init, dg, "inpainting", P.TVDenoiser(), **kw)
    assert len(Xg) == len(Xr) == n_iter
    observed("pnp-TV iterate vs oracle", max((a - b).abs().max().item() for a, b in zip(Xr + Lr, Xg + Lg)), TOL_SAMPLER)
    # the annealed level matters: a run at a constant level differs
    Xc, _, _ = P.pnp(init, dg, "deblurring-like", P.TVDenoiser(), **kw)
    assert (Xc[0] - Xg[0]).abs().max().item() > 1e-3


def test_long_chain_castle_against_oracle():
    """One 481 x 321 chain (CBSD68's size, no padding), 50 PSGLA-TV inpainting iterations under replayed noise."""
    im = _image("set1c/castle.png")
    assert tuple(im.shape[2:]) == (481, 321)
    dg, init, y, _ = P.make_inpainting(im)
    n_iter = 50
    noise = _replay_noise(im.shape, n_iter, seed=1)
    kw = _psgla_kw(n_iter, n_inter=5, n_mm=9)
    Xr, Mr, M2r = io_.psgla(init, dg, TV.TVDenoiser(), device="cuda", noise=noise, **kw)
    Xg, Mg, M2g = P.psgla(init, dg, P.TVDenoiser(), noise=noise, **kw)
    assert len(Xg) == len(Xr) == 10 and len(Mg) == len(Mr) == 5
    observed("PSGLA-TV castle 50 it vs oracle", max((a - b).abs().max().item() for a, b in zip(Xr + Mr + M2r, Xg + Mg + M2g)),
             TOL_SAMPLER)


def test_batched_chains_stats_and_rng_modes():
    """n_chains, store="stats" and every rng mode run; chain c of a batched philox run equals a one-chain run with chain_id0 = c."""
    im = _image("set3c/butterfly.png", 48, 64)
    dg, init, y, _ = P.make_inpainting(im)
    kw = _psgla_kw(12, n_inter=3, n_mm=3)
    _, M, M2 = P.psgla(init, dg, P.TVDenoiser(), n_chains=3, rng="philox", store="stats", **kw)
    assert len(M) == 1 and M[0].shape == (3, 3, 48, 64)
    _, M1, _ = P.psgla(init, dg, P.TVDenoiser(), n_chains=1, chain_id0=1, rng="philox", store="stats", **kw)
    assert torch.equal(M1[0][0], M[0][1])
    for rng in ("torch", "torch_cuda"):
        X, _, _ = P.psgla(init, dg, P.TVDenoiser(), rng=rng, **kw)
        assert len(X) == 4 and torch.isfinite(X[-1]).all()
    Xa, _, _ = P.psgla(init, dg, P.TVDenoiser(), rng="torch", **kw)
    Xb, _, _ = P.psgla(init, dg, P.TVDenoiser(), rng="torch_cuda", **kw)
    assert all(torch.equal(a, b) for a, b in zip(Xa, Xb))


def test_run_image_set_rows_do_not_depend_on_earlier_images():
    """run_image_set resets the prox state before each image, so every row equals that image's row computed by a fresh
    denoiser (the reference warm-starts across images; here a row must not depend on which images a rank ran before it)."""
    ims = [_image("set3c/leaves.png", 40, 48)[0].cpu(), _image("set3c/starfish.png", 40, 48)[0].cpu()]
    prm = dict(P.sampler_params("psgla", den="TV", N=1000), N=12, n_inter=2, n_inter_mmse=2, lambd=LAMBD_GAIN1)
    res = P.run_image_set(ims, P.TVDenoiser(), problem="inpainting", alg="psgla", n_chains=2, params=prm, seed=3)
    from psgla_b200 import image_set
    for i, im in enumerate(ims):
        row, _ = image_set._sample_image(i, im, P.TVDenoiser(), "inpainting", "psgla", 2, prm, 3, 0, 0.5, 1.0, 4, "uniform", 1.0,
                                         False)
        got = [res[i][k] for k in P.image_set.ROW_FIELDS]
        assert got == [int(v) if k in ("index", "n_chains", "n_windows", "H", "W") else float(v)
                       for k, v in zip(P.image_set.ROW_FIELDS, row.tolist())], i
    assert P.sampler_params("psgla", den="TV")["lambd"] == 10.0  # the table itself is unchanged


def test_samplers_that_feed_x_reject_tv():
    tv = P.TVDenoiser()
    im = torch.rand(1, 3, 16, 16, device="cuda")
    dg, init, y, _ = P.make_inpainting(im)
    with pytest.raises(TypeError, match="DnCNN"):
        P.PriorGrad(tv, 1.0, 0.01, 1e-4)
    pg = object.__new__(P.PriorGrad)
    pg.denoiser, pg.alpha, pg.s1, pg.s2 = tv, 1.0, 0.01, 1e-4
    with pytest.raises(TypeError, match="DnCNN"):
        P.pnpula(init, dg, pg, 1e-5, 1e-4, n_iter=2, seed=0)
    with pytest.raises(TypeError, match="DnCNN"):
        P.red(init, dg, "inpainting", tv, 1.0, n_iter=2)
