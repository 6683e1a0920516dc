"""-m gpu: image path through the C ABI against the plain-PyTorch fp32 oracle (oracle/image_oracle.py).

Stated tolerances
  * elementwise / stencil kernels (fp32): 1e-5 relative to the tensor's scale (they fold constants, e.g. one multiply by
    (delta/lambd)/sigma^2 instead of the reference's divide-then-multiply);
  * one conv layer, bf16 operands with fp32 accumulation, against the fp64 sum of the same bf16 operands, element by element
    (tests/conv_reference.py): |got - ref| <= 2^-8 |ref| + tau S for bf16 outputs (2^-23 |ref| for the fp32 last layer), S =
    sum |w| |x| + |bias|, tau calibrated and at most 2^-10; and fewer than MISMATCH_MAX of the bf16 outputs differ from the
    correctly rounded reference;
  * DnCNN residual (20 layers, bf16 activations): <= 1e-2 relative L2 error of the residual;
  * sampler iterates under replayed noise, bf16 denoiser vs fp32 oracle: <= 1e-3 abs per iterate (images live in [0,1];
    observed 1e-4 .. 4e-4 over 50 .. 300 iterations with the Lipschitz-0.9 denoiser) and, where the denoiser term dominates
    (large-gain weights), <= 2 % of the denoiser term itself; thinning / window bookkeeping must match exactly."""
import os

import numpy as np
import pytest
import torch
import torch.nn.functional as F

import psgla_b200 as P
from oracle import image_oracle as io_
from conftest import observed
import conv_reference as CR

pytestmark = pytest.mark.gpu
G = np.load(os.path.join(os.path.dirname(__file__), "golden", "image_golden.npz"))
G20 = np.load(os.path.join(os.path.dirname(__file__), "golden", "image_golden_d20.npz"))
TOL_ITERATE = 1e-3  # abs, per iterate, bf16 tcgen05 denoiser vs the fp32 reference / oracle under the same noise, <= 25 iterations


def tol_iterate(n_iter):
    """The per-iterate bound over a horizon of n_iter iterations.  On unobserved pixels the PSGLA map X -> X + R(X + noise) is
    not contractive, so the bf16-vs-fp32 denoiser difference (~3e-5 per iteration) accumulates along the chain: observed
    1.1e-4 after 4 iterations, 2.7e-4 after 12, 1.7e-3 after 50, 6.8e-3 after 300 (gpurun_out r2f).  Bound: 4e-5 per iteration."""
    return max(TOL_ITERATE, 4e-5 * n_iter)


@pytest.fixture(scope="module")
def weights():
    return io_.make_dncnn_weights(seed=0, n_power_iter=10, spatial=16)


@pytest.fixture(scope="module")
def nets(weights):
    den = P.DnCNN(pretrained=weights)
    net = io_.DnCNN().cuda()
    net.load_state_dict(weights)
    return den, net.eval()


def test_umma_descriptor_selftest():
    lib = P._lib.lib()
    torch.manual_seed(0)
    a = torch.randn(136, 64, device="cuda").to(torch.bfloat16).contiguous()
    b = torch.randn(64, 64, device="cuda").to(torch.bfloat16).contiguous()
    for mode in (0, 2):  # A operand from shared memory (descriptor shift) / from tensor memory (copied by tcgen05.st)
        for shift in (0, 1, 2, 5, 8):
            d = torch.zeros(128, 64, device="cuda")
            P._lib.check(lib.psgla_selftest_umma(a.data_ptr(), b.data_ptr(), d.data_ptr(), shift, mode, None), "selftest")
            torch.cuda.synchronize()
            ref = a[shift:shift + 128].float() @ b.float().t()
            assert (d - ref).abs().max().item() < 1e-4, (mode, shift)


@pytest.mark.parametrize("B,H,W,layer", [(1, 8, 128, 1), (2, 40, 256, 5), (1, 33, 200, 3), (3, 5, 17, 2), (1, 1, 1, 4),
                                         (1, 8, 128, 0), (2, 37, 150, 0), (1, 8, 128, 19), (2, 37, 150, 19), (1, 321, 481, 7)])
def test_conv_layer_against_torch(B, H, W, layer):
    depth = 20
    lib = P._lib.lib()
    sd = P.random_dncnn_state_dict(3, depth, scale=3.0)
    den = P.DnCNN(depth=depth, pretrained=sd)
    names = ["in_conv"] + ["conv_list.%d" % i for i in range(depth - 2)] + ["out_conv"]
    w, bias = sd[names[layer] + ".weight"], sd[names[layer] + ".bias"]
    cin = w.shape[1]
    x = torch.randn(B, cin, H, W, device="cuda", generator=torch.Generator(device="cuda").manual_seed(1)).to(torch.bfloat16)
    cpad = 16 if layer == 0 else 64
    xin = torch.zeros(B, H, W, cpad, device="cuda", dtype=torch.bfloat16)
    xin[..., :cin] = x.permute(0, 2, 3, 1)
    last = layer == depth - 1
    ref, S = CR.reference("conv3", x, w, bias, relu=not last)
    shape = P._lib.ImgShape(B, 3, H, W)
    out = CR.Guarded((B, 3, H, W) if last else (B, H, W, 64), torch.float32 if last else torch.bfloat16)
    P._lib.check(lib.psgla_conv3x3_layer(den.packed.data_ptr(), depth, layer, shape, xin.data_ptr(), out.ptr(), int(not last), None), "conv")
    torch.cuda.synchronize()
    assert out.intact()
    CR.check("dncnn layer %d at %s" % (layer, (B, H, W)), out.tensor if last else out.tensor.permute(0, 3, 1, 2), ref, S)


def test_dncnn_forward_against_fp32_oracle(nets):
    den, net = nets
    for shape in ((2, 3, 64, 96), (1, 3, 130, 70)):
        x = torch.rand(*shape, device="cuda")
        with torch.no_grad():
            ref = net(x)
        got = den.forward(x, 2 / 255)
        r_ref, r_got = ref - x, got - x
        assert ((r_got - r_ref).norm() / r_ref.norm()).item() < 1e-2
        assert (got - ref).abs().max().item() < 1e-3


@pytest.mark.parametrize("shape", [(1, 3, 256, 256), (1, 3, 64, 64), (2, 3, 100, 200), (1, 3, 37, 150), (1, 3, 5, 17), (1, 3, 1, 1),
                                   (3, 3, 70, 256), (1, 3, 3, 130), (1, 3, 64, 300), (4, 3, 256, 256)])
@pytest.mark.parametrize("depth", [20, 5])
def test_fused_layer_pairs_equal_single_layers(shape, depth, monkeypatch):
    """Few chains: two hidden layers per launch (conv_fused2.cu, the intermediate rows stay in shared memory, the strips' edge pixels
    cross the CTA pair by st.async) must equal the per-layer launches BIT FOR BIT -- the intermediate is rounded to bf16 either
    way.  Shapes: R = 4 / 2 / 1 row blocks, ragged strips, images smaller than a tile, an odd number of hidden layers
    (depth 5: one pair + a single layer), and two shapes the fused path does not take (W > 256, more than one wave)."""
    sd = P.random_dncnn_state_dict(7, depth, scale=2.0)
    den = P.DnCNN(depth=depth, pretrained=sd)
    x = torch.rand(*shape, device="cuda", generator=torch.Generator(device="cuda").manual_seed(3))
    monkeypatch.setenv("PSGLA_CONV_FUSE2", "0")
    ref = den.forward(x, 2 / 255).clone()
    monkeypatch.setenv("PSGLA_CONV_FUSE2", "1")
    for _ in range(3):  # repeated: the launches overlap their predecessors' tails (PDL), a race would not repeat bit for bit
        got = den.forward(x, 2 / 255)
        torch.cuda.synchronize()
        assert torch.equal(got, ref), (got - ref).abs().max().item()
    assert torch.isfinite(ref).all() and (ref - x).abs().max().item() > 1e-3


def test_blur_against_reference_formulation():
    torch.manual_seed(0)
    im = torch.rand(2, 3, 45, 70, device="cuda")
    for l, bt in ((4, "uniform"), (2, "gaussian"), (7, "gaussian"), (0, "uniform")):
        h = P.blur_taps(l, bt, 1.3).reshape(-1)
        op = P.DeblurDataGrad(h, l, torch.zeros_like(im), 1.0)
        got = op.A(im)
        want = io_.blur_operators(h, l, 3, "cuda")[0](im)  # the reference's pad-circular + depthwise conv2d (sampling_images.py:329)
        assert (got - want).abs().max().item() < 1e-5


def _pre_inputs(B, H, W, seed=0):
    g = torch.Generator(device="cuda").manual_seed(seed)
    x = torch.rand(B, 3, H, W, device="cuda", generator=g) * 1.6 - 0.3
    z = torch.randn(B, 3, H, W, device="cuda", generator=g)
    im = torch.rand(1, 3, H, W, device="cuda", generator=g)
    return x, z, im


@pytest.mark.parametrize("H,W", [(16, 16), (33, 47), (64, 128)])
@pytest.mark.parametrize("alg", ["psgla", "pnp_ula"])
def test_pre_inpaint_against_oracle(H, W, alg):
    lib = P._lib.lib()
    B = 3
    x, z, im = _pre_inputs(B, H, W)
    dg, init, y, mask = P.make_inpainting(im)
    pre = P._lib.PreParams()
    if alg == "psgla":
        prm = io_.resolve_params("psgla")
        pre.alg, pre.gain_data, pre.noise_scale = 0, (prm["delta"] / prm["lambd"]) / dg.sigma2, float(np.sqrt(2) * prm["s"])
        want = x + (prm["delta"] / prm["lambd"]) * dg(x) + float(np.sqrt(2) * prm["s"]) * z
        den_want = want
    else:
        prm = io_.resolve_params("pnp_ula", s=5.0)
        pre.alg, pre.gain_data, pre.noise_scale = 1, prm["delta"] / dg.sigma2, float(np.sqrt(2 * prm["delta"]))
        pre.proj_gain, pre.c_min, pre.c_max = prm["delta"] / prm["lambd"], 0.1, 0.9
        proj = x.clamp(0.1, 0.9)
        want = x + prm["delta"] * (-(x - proj) / prm["lambd"] + dg(x)) + float(np.sqrt(2 * prm["delta"])) * z
        den_want = x
    base = torch.empty_like(x)
    den_in = torch.full((B, H, W, 16), 7.0, device="cuda", dtype=torch.bfloat16)
    m3, y3 = mask.expand(-1, 3, -1, -1).contiguous(), y.contiguous()
    P._lib.check(lib.psgla_img_pre_inpaint(pre, P._lib.ImgShape(B, 3, H, W), x.data_ptr(), m3.data_ptr(), 1, y3.data_ptr(), 1,
                                           z.data_ptr(), base.data_ptr(), den_in.data_ptr(), None), "pre")
    torch.cuda.synchronize()
    assert (base - want).abs().max().item() <= 1e-5 * max(1.0, want.abs().max().item())
    assert torch.equal(den_in[..., :3].float(), den_want.permute(0, 2, 3, 1).to(torch.bfloat16).float()) or \
        (den_in[..., :3].float() - den_want.permute(0, 2, 3, 1)).abs().max().item() < 2 ** -7
    assert torch.count_nonzero(den_in[..., 3:]).item() == 0


@pytest.mark.parametrize("form", ["four_pass", "ata"])
@pytest.mark.parametrize("H,W,l,bt", [(32, 32, 4, "uniform"), (45, 70, 2, "gaussian"), (64, 96, 4, "gaussian"), (256, 256, 4, "uniform"),
                                      (37, 300, 3, "gaussian"), (5, 7, 4, "uniform"), (130, 514, 1, "uniform")])
@pytest.mark.parametrize("alg", ["psgla", "pnp_ula"])
def test_pre_deblur_against_oracle(H, W, l, bt, form, alg):
    """Both deblurring "pre" kernels -- the four-pass A, A^T stencil and the row-streaming two-pass A^T A form with A^T y
    precomputed -- against the reference's pad-circular + conv2d formulation (sampling_images.py:329-338); sizes cover strips
    wider than 256 columns, widths not a multiple of 4, images smaller than the halo (multiple wrap-arounds)."""
    lib = P._lib.lib()
    B = 2
    x, z, im = _pre_inputs(B, H, W, seed=2)
    dd, init, y = P.make_deblurring(im, l=l, blur_type=bt, si=1.0)
    pre = P._lib.PreParams()
    if alg == "psgla":
        prm = io_.resolve_params("psgla")
        pre.alg, pre.gain_data, pre.noise_scale = 0, (prm["delta"] / prm["lambd"]) / dd.sigma2, float(np.sqrt(2) * prm["s"])
        grad = io_.deblur_data_grad(x.cpu(), dd.h1d, l, y.cpu(), dd.sigma2)  # the reference's conv2d formulation, on the host
        want = (x.cpu() + (prm["delta"] / prm["lambd"]) * grad + float(np.sqrt(2) * prm["s"]) * z.cpu()).cuda()
        den_want = want
    else:
        prm = io_.resolve_params("pnp_ula", s=5.0)
        pre.alg, pre.gain_data, pre.noise_scale = 1, prm["delta"] / dd.sigma2, float(np.sqrt(2 * prm["delta"]))
        pre.proj_gain, pre.c_min, pre.c_max = prm["delta"] / prm["lambd"], 0.1, 0.9
        grad = io_.deblur_data_grad(x.cpu(), dd.h1d, l, y.cpu(), dd.sigma2)
        xc = x.cpu()
        want = (xc + prm["delta"] * (-(xc - xc.clamp(0.1, 0.9)) / prm["lambd"] + grad) + float(np.sqrt(2 * prm["delta"])) * z.cpu()).cuda()
        den_want = x
    base = torch.full_like(x, float("nan"))
    den_in = torch.full((B, H, W, 16), 7.0, device="cuda", dtype=torch.bfloat16)
    shape = P._lib.ImgShape(B, 3, H, W)
    if form == "four_pass":
        P._lib.check(lib.psgla_img_pre_deblur(pre, shape, x.data_ptr(), dd._taps_c, l, y.data_ptr(), 1, z.data_ptr(), base.data_ptr(),
                                              den_in.data_ptr(), None), "pre_deblur")
    else:
        aty = dd.AT(y)
        P._lib.check(lib.psgla_img_pre_deblur_ata(pre, shape, x.data_ptr(), dd._taps_c, l, aty.data_ptr(), 1, z.data_ptr(),
                                                  base.data_ptr(), den_in.data_ptr(), None), "pre_deblur_ata")
    torch.cuda.synchronize()
    scale = max(1.0, want.abs().max().item())
    assert (base - want).abs().max().item() <= 2e-5 * scale
    assert (den_in[..., :3].float() - den_want.permute(0, 2, 3, 1)).abs().max().item() < 2 ** -7 * max(1.0, den_want.abs().max().item())
    assert torch.count_nonzero(den_in[..., 3:]).item() == 0


def test_pre_deblur_ata_philox_and_batched_observation():
    """In-kernel noise of the A^T A kernel == the library's dumped Philox stream; a per-chain A^T y (aty_B = B) is honoured."""
    lib = P._lib.lib()
    B, H, W, l = 3, 40, 64, 4
    x, _, im = _pre_inputs(B, H, W, seed=5)
    dd, _, y = P.make_deblurring(im, l=l, blur_type="uniform")
    yB = y.expand(B, -1, -1, -1).contiguous() * torch.tensor([1.0, 0.5, 2.0], device="cuda")[:, None, None, None]
    aty = dd.AT(yB)
    pre = P._lib.PreParams()
    pre.alg, pre.gain_data, pre.noise_scale, pre.seed, pre.chain_id0, pre.iteration = 0, 0.3, 0.7, 9, 4, 6
    shape = P._lib.ImgShape(B, 3, H, W)
    z = torch.empty(B, 3, H, W, device="cuda")
    P._lib.check(lib.psgla_img_noise(shape, 9, 4, 6, z.data_ptr(), None), "noise")
    outs = []
    for noise in (None, z):
        base = torch.empty_like(x)
        den_in = torch.empty((B, H, W, 16), device="cuda", dtype=torch.bfloat16)
        P._lib.check(lib.psgla_img_pre_deblur_ata(pre, shape, x.data_ptr(), dd._taps_c, l, aty.data_ptr(), B,
                                                  None if noise is None else noise.data_ptr(), base.data_ptr(), den_in.data_ptr(), None), "ata")
        outs.append(base)
    assert torch.equal(outs[0], outs[1])
    # canaries: outputs carved out of larger sentinel-filled buffers (odd sizes, width not a multiple of 4, strips > 256 columns)
    for Hc, Wc in ((19, 37), (9, 530)):
        xc, zc, imc = _pre_inputs(2, Hc, Wc, seed=8)
        ddc, _, yc = P.make_deblurring(imc, l=3, blur_type="gaussian", si=1.2)
        atyc = ddc.AT(yc)
        n = 2 * 3 * Hc * Wc
        big = torch.full((n + 2048,), 1234.5, device="cuda")
        bigd = torch.full((2 * Hc * Wc * 16 + 4096,), 7.0, device="cuda", dtype=torch.bfloat16)
        base_c, den_c = big[1024:1024 + n], bigd[2048:2048 + 2 * Hc * Wc * 16]
        P._lib.check(lib.psgla_img_pre_deblur_ata(pre, P._lib.ImgShape(2, 3, Hc, Wc), xc.data_ptr(), ddc._taps_c, 3, atyc.data_ptr(), 1,
                                                  zc.data_ptr(), base_c.data_ptr(), den_c.data_ptr(), None), "ata canary")
        torch.cuda.synchronize()
        assert torch.all(big[:1024] == 1234.5) and torch.all(big[1024 + n:] == 1234.5)
        assert torch.all(bigd[:2048] == 7.0) and torch.all(bigd[2048 + 2 * Hc * Wc * 16:] == 7.0)
        assert torch.isfinite(base_c).all() and not torch.any(base_c == 1234.5)
    want = x - 0.3 * (dd.A(dd.A(x)) - aty) + 0.7 * z
    assert (outs[0] - want).abs().max().item() < 2e-5 * max(1.0, want.abs().max().item())


def test_image_philox_noise_matches_pre_kernel():
    lib = P._lib.lib()
    for H, W in ((32, 64), (33, 47)):
        B = 2
        shape = P._lib.ImgShape(B, 3, H, W)
        z = torch.empty(B, 3, H, W, device="cuda")
        P._lib.check(lib.psgla_img_noise(shape, 42, 5, 11, z.data_ptr(), None), "noise")
        x = torch.zeros(B, 3, H, W, device="cuda")
        m = torch.zeros(1, 3, H, W, device="cuda")
        pre = P._lib.PreParams()
        pre.alg, pre.gain_data, pre.noise_scale, pre.seed, pre.chain_id0, pre.iteration = 0, 0.0, 1.0, 42, 5, 11
        base = torch.empty_like(x)
        den_in = torch.empty((B, H, W, 16), device="cuda", dtype=torch.bfloat16)
        P._lib.check(lib.psgla_img_pre_inpaint(pre, shape, x.data_ptr(), m.data_ptr(), 1, m.data_ptr(), 1, None, base.data_ptr(),
                                               den_in.data_ptr(), None), "pre")
        torch.cuda.synchronize()
        assert torch.equal(base, z)
        zz = z.double().cpu().numpy().reshape(-1)
        assert abs(zz.mean()) < 0.03 and abs(zz.var() - 1) < 0.05
    # chains are independent streams
    assert abs(np.corrcoef(z[0].cpu().numpy().reshape(-1), z[1].cpu().numpy().reshape(-1))[0, 1]) < 0.05


def _psgla_kw(prm, n_iter, n_inter, n_mm, alpha=1.0):
    return dict(alpha=torch.tensor(alpha, device="cuda"), lambd=torch.tensor(prm["lambd"], device="cuda"), sig_float=prm["s"],
                delta=prm["delta"], n_iter=n_iter, n_inter=n_inter, n_inter_mmse=n_mm, seed=0)


@pytest.mark.parametrize("problem", ["inpainting", "deblurring"])
def test_psgla_replay_against_oracle(nets, problem):
    den, net = nets
    torch.manual_seed(0)
    im = torch.rand(1, 3, 64, 64, device="cuda")
    if problem == "inpainting":
        dg, init, y, mask = P.make_inpainting(im)
    else:
        dg, init, y = P.make_deblurring(im, l=4, blur_type="uniform")
    prm = io_.resolve_params("psgla")
    n_iter, n_inter, n_mm = 50, 5, 4
    g = torch.Generator(device="cuda").manual_seed(0)
    noise = torch.stack([torch.randn(im.shape, generator=g, device="cuda") for _ in range(n_iter)])
    kw = _psgla_kw(prm, n_iter, n_inter, n_mm, alpha=0.8)
    Xr, Mr, M2r = io_.psgla(init, dg, net, device="cuda", noise=noise, **kw)
    Xg, Mg, M2g = P.psgla(init, dg, den, noise=noise, **kw)
    assert len(Xg) == len(Xr) == 10 and len(Mg) == len(Mr) == n_iter // (n_mm + 1) and len(M2g) == len(M2r)
    assert Xg[0].shape == Xr[0].shape == (3, 64, 64)
    observed("max |iterate - oracle|", max((a - b).abs().max().item() for a, b in zip(Xr + Mr + M2r, Xg + Mg + M2g)), tol_iterate(n_iter))
    # rng="torch" reproduces the reference's own generator stream on this device
    Xt, _, _ = P.psgla(init, dg, den, rng="torch", **kw)
    assert all(torch.equal(a, b) for a, b in zip(Xt, Xg))


def test_pnpula_replay_against_oracle(nets):
    den, net = nets
    torch.manual_seed(1)
    im = torch.rand(1, 3, 48, 80, device="cuda")
    dg, init, y = P.make_deblurring(im, l=4, blur_type="uniform")
    prm = io_.resolve_params("pnp_ula", s=5.0)
    n_iter, n_inter, n_mm = 30, 4, 5
    g = torch.Generator(device="cuda").manual_seed(2)
    noise = torch.stack([torch.randn(im.shape, generator=g, device="cuda") for _ in range(n_iter)])
    delta = torch.tensor(prm["delta"], dtype=torch.float32, device="cuda")
    lambd = torch.tensor(prm["lambd"], dtype=torch.float32, device="cuda")
    pg_ref = io_.make_prior_grad(net, 1.0, prm["s1"], prm["s2"], device="cuda")
    Xr, Mr, M2r = io_.pnpula(init, dg, pg_ref, delta, lambd, n_iter=n_iter, n_inter=n_inter, n_inter_mmse=n_mm, device="cuda", noise=noise)
    Xg, Mg, M2g = P.pnp_ula(init, dg, P.PriorGrad(den, 1.0, prm["s1"], prm["s2"]), delta, lambd, n_iter=n_iter, n_inter=n_inter,
                            n_inter_mmse=n_mm, seed=2, noise=noise)
    assert len(Xg) == len(Xr) and len(Mg) == len(Mr)
    observed("max |iterate - oracle|", max((a - b).abs().max().item() for a, b in zip(Xr + Mr + M2r, Xg + Mg + M2g)), tol_iterate(n_iter))


def test_golden_fixture_sampler_bookkeeping(nets):
    """The committed reference run (tests/golden, 16x16): same thinning / window counts and the same observation."""
    den, _ = nets
    im = torch.from_numpy(G["im"]).cuda()
    dg, init, y, mask = P.make_inpainting(im)  # CUDA generator stream differs from the CPU fixture: compare structure only
    alpha, lambd, s, delta, n_iter, n_inter, n_mm = G["psgla.params"]
    Xg, Mg, M2g = P.psgla(init, dg, den, float(alpha), float(lambd), float(s), float(delta), n_iter=int(n_iter), n_inter=int(n_inter),
                          n_inter_mmse=int(n_mm), seed=0)
    assert len(Xg) == G["psgla.X"].shape[0] and len(Mg) == G["psgla.M"].shape[0] and len(M2g) == G["psgla.M2"].shape[0]
    assert tuple(Xg[0].shape) == G["psgla.X"].shape[1:]
    # with the fixture's own mask / observation / noise the data term is the reference's: check the first pre step
    dgf = P.InpaintingDataGrad(torch.from_numpy(G["inp.mask"]).cuda(), torch.from_numpy(G["inp.y"]).cuda(), (1 / 255) ** 2)
    x0 = torch.from_numpy(G["inp.init"]).cuda()
    z0 = torch.from_numpy(G["psgla.noise"][0]).cuda()
    want = x0 + (float(delta) / float(lambd)) * dgf(x0) + float(np.sqrt(2) * s) * z0
    run = P.restoration_algorithms._Run(x0, dgf, den, 1, 1, 1, 0, torch.from_numpy(G["psgla.noise"][:1]).cuda(), "philox", None, 0)
    pre = P._lib.PreParams()
    pre.alg, pre.gain_data, pre.noise_scale = 0, (float(delta) / float(lambd)) / dgf.sigma2, float(np.sqrt(2) * s)
    run.pre(0, pre)
    assert (run.base - want).abs().max().item() < 1e-5


def test_batched_chains_and_philox_mode(nets):
    den, net = nets
    torch.manual_seed(0)
    im = torch.rand(1, 3, 32, 64, device="cuda")
    dg, init, y, mask = P.make_inpainting(im)
    prm = io_.resolve_params("psgla")
    kw = _psgla_kw(prm, 12, 3, 3)
    Xb, Mb, _ = P.psgla(init, dg, den, n_chains=4, **kw)
    assert Xb[0].shape == (4, 3, 32, 64) and len(Xb) == 4 and len(Mb) == 3
    assert not torch.equal(Xb[-1][0], Xb[-1][1])  # independent noise per chain
    # chain c of a batch == a single-chain run with chain_id0 = c (sharding invariance)
    X1, _, _ = P.psgla(init, dg, den, n_chains=1, chain_id0=2, **kw)
    assert (X1[-1][0] - Xb[-1][2]).abs().max().item() < 1e-6
    # replay of the library's own Philox stream through the fp32 oracle
    lib = P._lib.lib()
    zs = []
    for i in range(12):
        z = torch.empty(1, 3, 32, 64, device="cuda")
        P._lib.check(lib.psgla_img_noise(P._lib.ImgShape(1, 3, 32, 64), 0, 2, i, z.data_ptr(), None), "noise")
        zs.append(z)
    Xr, _, _ = io_.psgla(init, dg, net, device="cuda", noise=torch.stack(zs), **kw)
    observed("philox replay through the oracle", (Xr[-1] - X1[-1][0]).abs().max().item(), TOL_ITERATE)


def test_argument_errors(nets):
    den, _ = nets
    im = torch.rand(1, 3, 16, 16, device="cuda")
    dg, init, y, mask = P.make_inpainting(im)
    with pytest.raises(ValueError, match="seed=None"):
        P.psgla(init, dg, den, 1.0, 5.0, n_iter=10)
    with pytest.raises(TypeError):
        P.psgla(init, lambda x: x, den, 1.0, 5.0, n_iter=10, seed=0)
    with pytest.raises(ZeroDivisionError):
        P.psgla(init, dg, den, 1.0, 5.0, n_iter=5, n_inter=1, seed=0, save_images_online=True)


@pytest.mark.parametrize("n,H,W", [(1, 7, 7), (5, 37, 50), (3, 256, 256)])
def test_psnr_ssim_against_oracle(n, H, W):
    """Device PSNR / SSIM (sampling_images.py:373-384) against the oracle's NumPy restatement of skimage's definitions."""
    g = torch.Generator(device="cuda").manual_seed(n)
    ref = torch.rand(3, H, W, device="cuda", generator=g)
    imgs = (ref[None] + 0.1 * torch.randn(n, 3, H, W, device="cuda", generator=g)).clamp(0, 1)
    p, s = P.psnr_ssim(imgs, ref)
    torch.cuda.synchronize()
    for i in range(n):
        a, b = ref.permute(1, 2, 0).cpu().numpy(), imgs[i].permute(1, 2, 0).cpu().numpy()
        assert abs(p[i].item() - io_.psnr(a, b)) < 1e-3
        assert abs(s[i].item() - io_.ssim(a, b)) < 2e-4
    with pytest.raises(RuntimeError, match="7 x 7"):
        P.psnr_ssim(torch.rand(1, 3, 6, 20, device="cuda"), torch.rand(3, 6, 20, device="cuda"))


def test_posterior_summary_matches_reference_formulas(nets):
    den, net = nets
    torch.manual_seed(4)
    im = torch.rand(1, 3, 40, 48, device="cuda")
    dg, init, y, mask = P.make_inpainting(im, prop=0.5, sigma=1.0, seed_ip=0)
    s = 2 / 255
    X, M, M2 = P.psgla(init, dg, den, alpha=1.0, lambd=5.0, sig_float=s, delta=s * s, n_iter=44, n_inter=4, n_inter_mmse=3, seed=1)
    out = P.posterior_summary(im[0], X, M, M2)
    imn = im[0].permute(1, 2, 0).cpu().numpy()
    Mn = np.stack([m.permute(1, 2, 0).cpu().numpy() for m in M])
    mean_list = np.cumsum(Mn, axis=0) / np.arange(1, len(Mn) + 1)[:, None, None, None]  # sampling_images.py:414
    want = [io_.psnr(imn, mean_list[i]) for i in range(1, len(Mn))]
    assert np.allclose(out["psnr_running"].cpu().numpy(), want, atol=1e-3)
    xm = Mn.mean(0)
    assert abs(out["psnr_mmse"].item() - io_.psnr(imn, xm)) < 1e-3 and abs(out["ssim_mmse"].item() - io_.ssim(imn, xm)) < 2e-4
    var = np.stack([m.permute(1, 2, 0).cpu().numpy() for m in M2]).mean(0) - xm ** 2
    assert np.allclose(out["std"].permute(1, 2, 0).cpu().numpy(), np.sqrt(var * (var >= 0)), atol=1e-4)
    assert out["psnr_samples"].shape == (len(X),)


def test_final_psnr_ssim_parity_long_replay(nets):
    """North-star parity on the *result*: 300 PSGLA iterations with the reference's own torch.randn stream (rng="torch"),
    PSNR / SSIM of the MMSE estimate and the per-pixel std map against the fp32 oracle run on the same stream."""
    den, net = nets
    torch.manual_seed(8)
    low = torch.rand(1, 3, 8, 8, device="cuda")
    im = F.interpolate(low, size=(64, 64), mode="bicubic", align_corners=False).clamp(0, 1)
    dg, init, y, mask = P.make_inpainting(im, prop=0.5, sigma=1.0, seed_ip=0)
    prm = io_.resolve_params("psgla")
    kw = dict(alpha=torch.tensor(1.0, device="cuda"), lambd=torch.tensor(prm["lambd"], device="cuda"), sig_float=prm["s"],
              delta=prm["delta"], n_iter=300, n_inter=10, n_inter_mmse=10, seed=21)
    Xr, Mr, M2r = io_.psgla(init, dg, net, device="cuda", **kw)            # draws torch.randn(generator(seed)) per iteration
    Xg, Mg, M2g = P.psgla(init, dg, den, rng="torch", **kw)               # same generator, replayed into the kernels
    a, b = P.posterior_summary(im[0], Xr, Mr, M2r), P.posterior_summary(im[0], Xg, Mg, M2g)
    assert abs(a["psnr_mmse"].item() - b["psnr_mmse"].item()) < 0.05       # dB
    assert abs(a["ssim_mmse"].item() - b["ssim_mmse"].item()) < 1e-3
    assert (a["std"] - b["std"]).abs().max().item() < 5e-3
    assert (a["psnr_samples"] - b["psnr_samples"]).abs().max().item() < 0.1
    observed("300-iteration per-iterate error", max((u - v).abs().max().item() for u, v in zip(Xr, Xg)), tol_iterate(300))


def test_reference_edge_behaviours(nets, tmp_path):
    """Quirks of the reference's samplers that a drop-in must keep (restoration_algorithms.py:123,146-158,211-213,217-218,246)."""
    den, net = nets
    torch.manual_seed(0)
    im = torch.rand(1, 3, 16, 24, device="cuda")
    dg, init, y, mask = P.make_inpainting(im, prop=0.5, sigma=1.0, seed_ip=0)
    s = 2 / 255
    kw = dict(alpha=1.0, lambd=5.0, sig_float=s, delta=s * s)
    # fewer than 10 iterations run fine without the online-save flag ...
    X, M, M2 = P.psgla(init, dg, den, n_iter=5, n_inter=2, n_inter_mmse=1, seed=0, **kw)
    assert len(X) == 3 and len(M) == len(M2) == 2
    # ... and divide by zero with it (K = int(n_iter / 10) = 0), as in the reference
    with pytest.raises(ZeroDivisionError):
        P.psgla(init, dg, den, n_iter=5, n_inter=2, n_inter_mmse=1, seed=0, save_images_online=True, path=str(tmp_path), name="t", **kw)
    # the online dump: a dict with the reference's keys every n_iter / 10 iterations
    P.psgla(init, dg, den, n_iter=20, n_inter=5, n_inter_mmse=4, seed=0, save_images_online=True, path=str(tmp_path), name="run", **kw)
    d = torch.load(str(tmp_path / "run_sampling.pth"))
    assert set(d) >= {"Samples", "Mmse", "Mmse2", "n_iter", "lambda", "delta"} and d["n_iter"] == 20
    # n_inter_mmse=None falls back to n_inter (:217-218)
    Xa, Ma, _ = P.psgla(init, dg, den, n_iter=12, n_inter=3, n_inter_mmse=None, seed=4, **kw)
    Xb, Mb, _ = P.psgla(init, dg, den, n_iter=12, n_inter=3, n_inter_mmse=3, seed=4, **kw)
    assert len(Ma) == len(Mb) == 3 and all(torch.equal(a, b) for a, b in zip(Ma, Mb))
    # a 3-D init is accepted like the reference's squeeze conventions; results are squeezed [3, H, W] tensors
    Xc, _, _ = P.psgla(init[0], dg, den, n_iter=12, n_inter=3, n_inter_mmse=3, seed=4, **kw)
    assert Xc[0].shape == (3, 16, 24) and all(torch.equal(a, b) for a, b in zip(Xa, Xc))
    # no seed: the reference dies with UnboundLocalError at the first randn; here a ValueError up front
    with pytest.raises(ValueError, match="seed"):
        P.psgla(init, dg, den, n_iter=12, n_inter=3, **kw)
    # PnP-ULA keeps the function's own projection box [-1, 2] unless told otherwise (:38; sampling_images.py:358)
    prm = io_.resolve_params("pnp_ula", s=5.0)
    pg = P.PriorGrad(den, 1.0, prm["s1"], prm["s2"])
    big = init + 5.0  # far outside [-1, 2]: the projection term must pull it back
    Xu, _, _ = P.pnpula(big, dg, pg, torch.tensor(prm["delta"]), torch.tensor(prm["lambd"]), n_iter=12, n_inter=11, seed=0)
    Xw, _, _ = P.pnpula(big, dg, pg, torch.tensor(prm["delta"]), torch.tensor(prm["lambd"]), n_iter=12, n_inter=11, seed=0,
                        c_min=-100, c_max=100)
    assert (Xu[-1] - big[0]).abs().max() > (Xw[-1] - big[0]).abs().max()


@pytest.mark.parametrize("family", ["dncnn", "drunet"])
@pytest.mark.parametrize("alg,rng,B,H,W", [("psgla", "philox", 3, 40, 56), ("psgla", "torch_cuda", None, 33, 31),
                                           ("pnpula", "philox", 2, 24, 40), ("pnpula", "torch_cuda", None, 64, 64)])
def test_fused_next_pre_equals_separate_pre_kernel(weights, family, alg, rng, B, H, W):
    """Inpainting: the last layer's epilogue evaluates the next iteration's Langevin "pre" on the iterate it has just produced
    (psgla_*_post_next).  Same arithmetic, same noise element: samples and moments must equal, BIT FOR BIT, the run that
    launches the stand-alone pre kernel every iteration (run.fuse_next_pre = False)."""
    if family == "drunet":
        if H % 8 or W % 8:
            H, W = (H + 7) // 8 * 8, (W + 7) // 8 * 8
        den = P.DRUNet(pretrained=io_.make_drunet_weights(seed=0))
    else:
        den = P.DnCNN(pretrained=weights)
    torch.manual_seed(4)
    im = torch.rand(1, 3, H, W, device="cuda")
    dg, init, _, _ = P.make_inpainting(im, prop=0.5, sigma=1.0, seed_ip=0)

    def run(fuse):
        if alg == "psgla":
            r = P.psgla_run(init, dg, den, alpha=0.8, lambd=5.0, sig_float=2 / 255, delta=(2 / 255) ** 2, n_iter=7, n_inter=2,
                            n_inter_mmse=2, seed=3, rng=rng, n_chains=B)
        else:
            pg = P.PriorGrad(den, 1.0, 5 / 255, (5 / 255) ** 2)
            r = P.pnpula_run(init, dg, pg, delta=torch.tensor(1e-5, device="cuda"), lambd=torch.tensor(2e-5, device="cuda"),
                             n_iter=7, n_inter=2, n_inter_mmse=2, seed=3, rng=rng, n_chains=B)
        assert r.fuse_next_pre
        r.fuse_next_pre = fuse
        for i in range(r.n_iter):
            r.step(i)
        return r.finish()

    a = run(True)
    b = run(False)
    torch.cuda.synchronize()
    for la, lb in zip(a, b):
        assert len(la) == len(lb) and len(la) > 0
        for ta, tb in zip(la, lb):
            assert torch.equal(ta, tb)


def _d20_denoiser():
    seed, n_pi, spatial = (int(v) for v in G20["weights"])
    return io_.make_dncnn_weights(seed=seed, n_power_iter=n_pi, spatial=spatial)


def test_reference_fixture_replayed_through_cuda():
    """The UNMODIFIED reference's own outputs (tests/golden/image_golden_d20.npz: psgla on inpainting and pnpula with the
    script's default table on deblurring, full DnCNN depth 20 / 64 features, CPU fp32) against the CUDA path fed the same mask /
    observation / noise / weights: samples, window means and second moments within 1e-3, directly -- no oracle in between."""
    den = P.DnCNN(pretrained=_d20_denoiser())
    cu = lambda k: torch.from_numpy(G20[k]).cuda()  # noqa: E731
    alpha, lambd, s, delta, n_iter, n_inter, n_mm = G20["psgla.params"]
    dg = P.InpaintingDataGrad(cu("inp.mask"), cu("inp.y"), (1 / 255) ** 2)
    X, M, M2 = P.psgla(cu("inp.init"), dg, den, float(alpha), float(lambd), float(s), float(delta), n_iter=int(n_iter),
                       n_inter=int(n_inter), n_inter_mmse=int(n_mm), seed=7, noise=cu("psgla.noise"))
    for got, key in ((X, "psgla.X"), (M, "psgla.M"), (M2, "psgla.M2")):
        assert len(got) == G20[key].shape[0]
        observed("reference fixture " + key, (torch.stack(got) - cu(key)).abs().max().item(), TOL_ITERATE)
    # ... and rng="torch" on the CPU-seeded stream is NOT expected to match (CUDA generator), but the replay above is the
    # reference's stream.  PnP-ULA, default parameters: delta ~ 1e-10, so delta * data_grad ~ 1e-6 and the noise step
    # sqrt(2 delta) ~ 1.4e-5 sit a few fp32 ulps above X ~ 0.5 (6e-8); the prior term delta alpha / s2 = 0.11 carries the update.
    delta, lambd, alpha, s1, s2, n_iter, n_inter, n_mm, l = G20["ula.params"]
    dd = P.DeblurDataGrad(G20["deb.h"].reshape(-1), int(l), cu("deb.y"), (1 / 255) ** 2)
    pg = P.PriorGrad(den, float(alpha), float(s1), float(s2))
    X, M, M2 = P.pnpula(cu("deb.y"), dd, pg, torch.tensor(float(delta)), torch.tensor(float(lambd)), n_iter=int(n_iter),
                        n_inter=int(n_inter), n_inter_mmse=int(n_mm), seed=11, noise=cu("ula.noise"))
    for got, key in ((X, "ula.X"), (M, "ula.M"), (M2, "ula.M2")):
        assert len(got) == G20[key].shape[0]
        observed("reference fixture " + key, (torch.stack(got) - cu(key)).abs().max().item(), TOL_ITERATE)
    assert (torch.stack(X)[-1] - cu("deb.y")[0]).abs().max().item() > 1e-2  # the chain has moved (300 x the error): not a vacuous match


def test_pnpula_default_parameters_against_oracle(nets):
    """The parameters the bench times (sampling_images.py:147-168 defaults: s1 = 2/255/255, lambd = 4.7e-10, delta = 1.05e-10) on
    a 64 x 64 deblurring problem, 40 iterations, replayed noise, against the fp32 oracle."""
    den, net = nets
    torch.manual_seed(3)
    im = torch.rand(1, 3, 64, 64, device="cuda")
    dg, init, y = P.make_deblurring(im, l=4, blur_type="uniform")
    prm = P.sampler_params("pnp_ula", den="DnCNN")
    assert prm["delta"] < 1.1e-10 and prm["N"] == 100000 and prm["n_inter"] == 10
    n_iter = 40
    g = torch.Generator(device="cuda").manual_seed(5)
    noise = torch.stack([torch.randn(im.shape, generator=g, device="cuda") for _ in range(n_iter)])
    delta = torch.tensor(prm["delta"], dtype=torch.float32, device="cuda")
    lambd = torch.tensor(prm["lambd"], dtype=torch.float32, device="cuda")
    ref_dg = lambda x: io_.deblur_data_grad(x, dg.h1d, 4, y, dg.sigma2)  # noqa: E731  the reference's conv2d formulation
    pg_ref = io_.make_prior_grad(net, prm["alpha"], prm["s1"], prm["s2"], device="cuda")
    Xr, Mr, M2r = io_.pnpula(init, ref_dg, pg_ref, delta, lambd, n_iter=n_iter, n_inter=4, n_inter_mmse=5, device="cuda", noise=noise)
    Xg, Mg, M2g = P.pnp_ula(init, dg, P.PriorGrad(den, prm["alpha"], prm["s1"], prm["s2"]), delta, lambd, n_iter=n_iter, n_inter=4,
                            n_inter_mmse=5, seed=5, noise=noise)
    assert len(Xg) == len(Xr) == 10 and len(Mg) == len(Mr)
    observed("max |iterate - oracle|", max((a - b).abs().max().item() for a, b in zip(Xr + Mr + M2r, Xg + Mg + M2g)), tol_iterate(n_iter))
    assert (Xr[-1] - init[0]).abs().max().item() > 1e-3


def test_large_gain_denoiser_term_dominates():
    """Weights with per-layer gain ~0.93 (uniform +-2.3/sqrt(fan_in): the residual is ~25 % of the input instead of the 1e-3
    of the Lipschitz-0.9 stand-in), so that the denoiser term carries the iterate: one PSGLA iteration from the same state must
    reproduce the fp32 oracle's denoiser term X+ - Y to 2 % (bf16 activations through 20 layers), and 6 iterations stay within
    2 % of the accumulated term."""
    sd = P.random_dncnn_state_dict(11, 20, scale=2.3)
    den = P.DnCNN(pretrained=sd)
    net = io_.DnCNN().cuda()
    net.load_state_dict(sd)
    net.eval()
    torch.manual_seed(6)
    im = torch.rand(1, 3, 48, 64, device="cuda")
    dg, init, y, mask = P.make_inpainting(im)
    prm = io_.resolve_params("psgla")
    for n_iter in (1, 6):
        g = torch.Generator(device="cuda").manual_seed(1)
        noise = torch.stack([torch.randn(im.shape, generator=g, device="cuda") for _ in range(n_iter)])
        kw = _psgla_kw(prm, n_iter, 1, 1, alpha=1.0)
        Xr, _, _ = io_.psgla(init, dg, net, device="cuda", noise=noise, **kw)
        Xg, _, _ = P.psgla(init, dg, den, noise=noise, **kw)
        # the denoiser's share of the total displacement: the run with the denoiser switched off (alpha = 0) is Y alone
        kw0 = _psgla_kw(prm, n_iter, 1, 1, alpha=0.0)
        Y0, _, _ = io_.psgla(init, dg, net, device="cuda", noise=noise, **kw0)
        term = (Xr[-1] - Y0[-1])
        assert term.abs().mean().item() > 0.02  # it does dominate: the noise step is 0.011, the data step ~1e-3
        observed("large-gain relative error of the denoiser term, %d it" % n_iter, ((Xg[-1] - Xr[-1]).norm() / term.norm()).item(), 2e-2)


def test_dncnn_sampler_256_50_iterations_against_oracle(nets):
    """BASELINE size: a 256 x 256 PSGLA run (DnCNN, inpainting, the script's parameters), 50 iterations under replayed noise,
    every stored sample / window mean against the fp32 oracle on the same device."""
    den, net = nets
    torch.manual_seed(12)
    low = torch.rand(1, 3, 20, 20, device="cuda")
    im = F.interpolate(low, size=(256, 256), mode="bicubic", align_corners=False).clamp(0, 1)
    dg, init, y, mask = P.make_inpainting(im, prop=0.5, sigma=1.0, seed_ip=0)
    prm = io_.resolve_params("psgla")
    n_iter = 50
    g = torch.Generator(device="cuda").manual_seed(9)
    noise = torch.stack([torch.randn(im.shape, generator=g, device="cuda") for _ in range(n_iter)])
    kw = _psgla_kw(prm, n_iter, 10, 10, alpha=1.0)
    Xr, Mr, M2r = io_.psgla(init, dg, net, device="cuda", noise=noise, **kw)
    Xg, Mg, M2g = P.psgla(init, dg, den, noise=noise, **kw)
    assert len(Xg) == len(Xr) == 5 and len(Mg) == len(Mr) == 4
    observed("max |iterate - oracle| at 256 x 256", max((a - b).abs().max().item() for a, b in zip(Xr + Mr + M2r, Xg + Mg + M2g)), tol_iterate(n_iter))


def test_statistics_only_mode_equals_the_stored_run(nets):
    """store="stats" (no sample kept, window means folded on the device): Xlist is empty and the single returned mean / second
    moment equal the average of the window means of the storing run; also: shape validation rejects what the kernels cannot index."""
    den, _ = nets
    torch.manual_seed(2)
    im = torch.rand(1, 3, 32, 40, device="cuda")
    dg, init, y, mask = P.make_inpainting(im)
    kw = dict(alpha=1.0, lambd=5.0, sig_float=2 / 255, delta=(2 / 255) ** 2, n_iter=23, n_inter=2, n_inter_mmse=3, seed=4, n_chains=3)
    X, M, M2 = P.psgla(init, dg, den, **kw)
    Xs, Ms, M2s = P.psgla(init, dg, den, store="stats", **kw)
    assert Xs == [] and len(Ms) == len(M2s) == 1 and len(M) == 23 // 4
    assert (Ms[0] - torch.stack(M).mean(0)).abs().max().item() < 1e-6
    assert (M2s[0] - torch.stack(M2).mean(0)).abs().max().item() < 1e-6
    with pytest.raises(ValueError, match="colour image"):
        P.psgla(torch.rand(1, 1, 32, 40, device="cuda"), dg, den, 1.0, 5.0, n_iter=10, seed=0)
    with pytest.raises(ValueError, match="to match init"):
        P.psgla(torch.rand(1, 3, 32, 48, device="cuda"), dg, den, 1.0, 5.0, n_iter=10, seed=0)
    with pytest.raises(ValueError, match="n_iter"):
        P.psgla(init, dg, den, 1.0, 5.0, n_iter=10, seed=0, noise=torch.zeros(4, 1, 3, 32, 40, device="cuda"))
    with pytest.raises(ValueError, match="store"):
        P.psgla(init, dg, den, 1.0, 5.0, n_iter=10, seed=0, store="none")


def test_second_device_after_first():
    """Per-device caches (function attributes, SM counts): the library used on cuda:0 and then on cuda:1 in one process."""
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    sd = _d20_denoiser()
    outs = []
    for d in (0, 1):
        dev = torch.device("cuda", d)
        den = P.DnCNN(pretrained=sd, device=dev)
        x = torch.rand(1, 3, 40, 72, generator=torch.Generator().manual_seed(0)).to(dev)
        outs.append(den.forward(x, 0.01).cpu())
        D = P.Theorical_MMSE(*P.gaussian_mixt_example("cross"))
        fin, _ = P.run_chains("psgla", 50, np.zeros(2), 0.3, np.eye(2), 1, D, 2 / 3, n_chains=4096, seed=0, device=dev)
        outs.append(fin.cpu())
    assert torch.equal(outs[0], outs[2]) and torch.equal(outs[1], outs[3])


def test_run_image_set_equals_per_image_runs(nets):
    """psgla_b200.run_image_set (one process = world size 1 here; the dealing / gathering logic at world sizes 2 and 3 is
    tests/test_dist_gloo.py): three images of different sizes, 2 chains each, statistics-only mode.  Every row must equal what a
    direct psgla() call on that image with chain_id0 = index * n_chains gives -- the invariant that makes the result independent
    of how many GPUs share the set."""
    den, _ = nets
    g = torch.Generator().manual_seed(3)
    images = [torch.rand(3, 32, 40, generator=g), torch.rand(3, 24, 24, generator=g), torch.rand(1, 3, 40, 32, generator=g)]
    prm = dict(P.sampler_params("psgla", den="DnCNN", N=1000), N=14, n_inter=2, n_inter_mmse=2)
    res = P.run_image_set(images, den, problem="inpainting", alg="psgla", n_chains=2, params=prm, seed=5, keep_maps=True)
    assert [d["index"] for d in res] == [0, 1, 2] and all(d["n_chains"] == 2 and d["n_windows"] == 14 // 3 for d in res)
    for i, im in enumerate(images):
        imc = im.reshape(1, 3, im.shape[-2], im.shape[-1]).cuda()
        dg, init, y, _ = P.make_inpainting(imc, prop=0.5, sigma=1.0, seed_ip=0)
        X, M, M2 = P.psgla(init, dg, den, **P.as_psgla_kwargs(prm, seed=5), n_chains=2, chain_id0=2 * i, rng="philox")
        xmmse = torch.stack(M).mean(0).mean(0)  # mean over windows, then over the two chains
        assert (res[i]["xmmse"] - xmmse).abs().max().item() < 1e-6
        p, s = P.psnr_ssim(xmmse, imc[0])
        assert abs(res[i]["psnr_mmse"] - p.item()) < 1e-3 and abs(res[i]["ssim_mmse"] - s.item()) < 1e-4
        assert (res[i]["H"], res[i]["W"]) == (im.shape[-2], im.shape[-1])
    # deblurring + PnP-ULA through the same entry
    prm_u = dict(P.sampler_params("pnp_ula", den="DnCNN", N=1000), N=9, n_inter=2, n_inter_mmse=2)
    res_u = P.run_image_set(images[:1], den, problem="deblurring", alg="pnp_ula", n_chains=3, params=prm_u, seed=1)
    assert len(res_u) == 1 and res_u[0]["n_chains"] == 3 and np.isfinite(res_u[0]["psnr_mmse"])
