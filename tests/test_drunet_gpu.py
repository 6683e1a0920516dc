"""GPU parity tests of the DRUNet path: the general tcgen05 conv layers element by element against the fp64 sum of the same
bf16 operands (tests/conv_reference.py), then the whole denoiser and the samplers against the fp32 oracle."""
import numpy as np
import pytest
import torch
import torch.nn.functional as F

import conv_reference as CR
import psgla_b200 as P

pytestmark = pytest.mark.gpu
# abs, per iterate: the non-residual U-Net feeds its whole output (|D| ~ 0.5, ~70 bf16 layers) into the iterate, unlike DnCNN's
# small residual; set from the observed figures (pytest -s prints them)
TOL_DRUNET = 2e-3


def _bf(x):
    return x.to(torch.bfloat16)


def _nhwc(x):
    return x.permute(0, 2, 3, 1).contiguous()


def _run_layer(mode, x, w_taps, res1=None, res2=None, relu=False):
    """x: bf16 NCHW; w_taps: bf16 [taps][Cout][Cin]; returns the bf16 output as NCHW."""
    lib = P._lib.lib()
    B, Cin, H, W = x.shape
    Cout = w_taps.shape[1]
    Ho, Wo = {0: (H, W), 1: (H // 2, W // 2), 2: (2 * H, 2 * W)}[mode]
    xin = _nhwc(x)
    out = CR.Guarded((B, Ho, Wo, Cout), torch.bfloat16)
    r1 = _nhwc(res1) if res1 is not None else None
    r2 = _nhwc(res2) if res2 is not None else None
    P._lib.check(lib.psgla_convg_layer(mode, B, H, W, Cin, Cout, w_taps.data_ptr(), xin.data_ptr(),
                                       r1.data_ptr() if r1 is not None else None, r2.data_ptr() if r2 is not None else None,
                                       out.ptr(), int(relu), None), "psgla_convg_layer")
    torch.cuda.synchronize()
    assert out.intact()
    return out.tensor.permute(0, 3, 1, 2)


@pytest.mark.parametrize("B,H,W,Cin,Cout,res,relu", [
    (2, 20, 24, 128, 128, 0, True),    # PX = 24, 5 rows per tile (120 of 128 tile pixels used)
    (1, 9, 240, 128, 128, 1, False),   # two 128-pixel strips, ragged second strip
    (1, 64, 64, 256, 256, 2, False),   # N tile 256, two residual inputs
    (2, 8, 8, 512, 512, 1, True),      # deepest scale, 8 k-blocks
    (1, 7, 130, 64, 192, 0, False),    # N tile 64 x 3, odd extents
    (1, 1, 1, 128, 128, 0, False),
    (1, 5, 128, 128, 128, 1, True),    # CTA-pair kernel, one 130-pixel row box for the three horizontal taps; odd M-tile count
    (3, 3, 300, 128, 128, 2, True),    # same with three strips per row (ragged last strip), 27 M tiles
    (1, 4, 256, 256, 256, 0, False),   # row-box form at N tile 256
    (4, 80, 256, 128, 128, 1, True),   # resident-weights form: 320 tile pairs, several per CTA pair (activation ring wraps)
])
def test_conv3x3_general(B, H, W, Cin, Cout, res, relu):
    g = torch.Generator(device="cuda").manual_seed(0)
    x = _bf(torch.randn(B, Cin, H, W, device="cuda", generator=g))
    w = _bf(torch.randn(Cout, Cin, 3, 3, device="cuda", generator=g) / np.sqrt(9 * Cin))
    rs = [_bf(torch.randn(B, Cout, H, W, device="cuda", generator=g)) for _ in range(res)]
    ref, S = CR.reference("conv3", x, w, None, rs, relu)
    w_taps = w.permute(2, 3, 0, 1).reshape(9, Cout, Cin).contiguous()
    got = _run_layer(0, x, w_taps, *(rs + [None, None])[:2], relu=relu)
    CR.check("convg conv3x3 %s" % ((B, H, W, Cin, Cout, res, relu),), got, ref, S)


@pytest.mark.parametrize("B,H,W,Cin,Cout", [(2, 16, 40, 64, 128), (1, 8, 8, 256, 512), (1, 2, 260, 128, 256)])
def test_strided_down_conv(B, H, W, Cin, Cout):
    g = torch.Generator(device="cuda").manual_seed(1)
    x = _bf(torch.randn(B, Cin, H, W, device="cuda", generator=g))
    w = _bf(torch.randn(Cout, Cin, 2, 2, device="cuda", generator=g) / np.sqrt(4 * Cin))
    ref, S = CR.reference("down", x, w)
    got = _run_layer(1, x, w.permute(2, 3, 0, 1).reshape(4, Cout, Cin).contiguous())
    CR.check("convg down %s" % ((B, H, W, Cin, Cout),), got, ref, S)


@pytest.mark.parametrize("B,H,W,Cin,Cout,res", [(2, 8, 20, 128, 64, 0), (1, 4, 4, 512, 256, 0), (1, 3, 130, 256, 128, 0),
                                                 (3, 40, 136, 128, 64, 0)])  # 240 ragged tile pairs, quadrants merged into N
def test_transposed_up_conv(B, H, W, Cin, Cout, res):
    g = torch.Generator(device="cuda").manual_seed(2)
    x = _bf(torch.randn(B, Cin, H, W, device="cuda", generator=g))
    w = _bf(torch.randn(Cin, Cout, 2, 2, device="cuda", generator=g) / np.sqrt(Cin))  # ConvTranspose2d layout
    ref, S = CR.reference("up", x, w)
    got = _run_layer(2, x, w.permute(2, 3, 1, 0).reshape(4, Cout, Cin).contiguous())
    CR.check("convg up %s" % ((B, H, W, Cin, Cout),), got, ref, S)


def test_convg_argument_errors():
    lib = P._lib.lib()
    t = torch.zeros(16, device="cuda", dtype=torch.bfloat16)
    assert lib.psgla_convg_layer(0, 1, 4, 4, 48, 64, t.data_ptr(), t.data_ptr(), None, None, t.data_ptr(), 0, None) == -1
    assert lib.psgla_convg_layer(1, 1, 5, 4, 64, 128, t.data_ptr(), t.data_ptr(), None, None, t.data_ptr(), 0, None) == -1
    assert lib.psgla_convg_layer(7, 1, 4, 4, 64, 64, t.data_ptr(), t.data_ptr(), None, None, t.data_ptr(), 0, None) == -1


# ----------------------------------------------------------------------------------------------------- whole network
from oracle import image_oracle as io_  # noqa: E402
from conftest import observed  # noqa: E402


@pytest.fixture(scope="module")
def drunets():
    sd = io_.make_drunet_weights(seed=0)
    den = P.DRUNet(pretrained=sd)
    net = io_.DRUNet().cuda()
    net.load_state_dict(sd)
    net.eval()
    return den, net


def test_product_and_oracle_random_init_agree():
    """The product's own seeded random init is the oracle's (same generator stream, same scaling)."""
    a, b = P.random_drunet_state_dict(3), io_.make_drunet_weights(seed=3)
    assert list(a) == list(b) == P.DRUNET_KEYS
    for k in a:
        assert torch.equal(a[k], b[k]), k


@pytest.mark.parametrize("B,H,W", [(1, 64, 64), (2, 40, 72), (1, 256, 256)])
def test_drunet_forward_against_fp32_oracle(drunets, B, H, W):
    den, net = drunets
    x = torch.rand(B, 3, H, W, device="cuda", generator=torch.Generator(device="cuda").manual_seed(5))
    sigma = 5.0 / 255.0
    with torch.no_grad():
        ref = net(x, sigma)
    got = den.forward(x, sigma)
    torch.cuda.synchronize()
    assert torch.isfinite(got).all()
    # ~70 bf16 layers against fp32: relative error of the output stays at the percent level
    rel = ((got - ref).norm() / ref.norm()).item()
    assert rel < 3e-2, rel
    assert (got - ref).abs().max().item() < 5e-2 * max(1.0, ref.abs().max().item())


def test_drunet_sizes_not_multiple_of_8(drunets):
    """forward() pads by replication to the next multiple of 8 and crops (KAIR test_pad); the fused sampler path refuses."""
    den, net = drunets
    x = torch.rand(1, 3, 36, 61, device="cuda")
    got = den.forward(x, 0.02)
    xp = F.pad(x, (0, 3, 0, 4), mode="replicate")
    with torch.no_grad():
        want = net(xp, 0.02)[:, :, :36, :61]
    assert got.shape == x.shape
    assert ((got - want).norm() / want.norm()).item() < 3e-2
    dd, initd, _ = P.make_deblurring(x, l=2, blur_type="gaussian")
    with pytest.raises(RuntimeError, match="multiples of 8"):
        P.psgla(initd, dd, den, 1.0, 25.0, 5 / 255, (5 / 255) ** 2, n_iter=2, n_inter=1, n_inter_mmse=1, seed=0)


@pytest.mark.parametrize("alg", ["psgla", "pnpula"])
def test_drunet_samplers_on_sizes_not_multiple_of_8(drunets, alg):
    """CBSD68 is 481 x 321: inpainting samplers with DRUNet carry the problem at the padded size (pad region unobserved, the
    network input's pad pixels re-filled from the edge before every application = the per-call replication padding of the
    oracle's DRUNet) and return cropped tensors.  Replayed noise, against the fp32 oracle at the true size; philox / fused path too."""
    den, net = drunets
    torch.manual_seed(5)
    im = torch.rand(1, 3, 37, 50, device="cuda")
    dg, init, y, mask = P.make_inpainting(im, prop=0.5, sigma=1.0, seed_ip=0)
    n_iter = 5
    g = torch.Generator(device="cuda").manual_seed(0)
    noise = torch.stack([torch.randn(im.shape, generator=g, device="cuda") for _ in range(n_iter)])
    if alg == "psgla":
        prm = io_.resolve_params("psgla", den="DRUNet", lambd=25.0)
        kw = dict(alpha=torch.tensor(0.8, device="cuda"), lambd=torch.tensor(prm["lambd"], device="cuda"), sig_float=prm["s"],
                  delta=prm["delta"], n_iter=n_iter, n_inter=2, n_inter_mmse=2, seed=0)
        Xr, Mr, M2r = io_.psgla(init, dg, net, device="cuda", noise=noise, **kw)
        Xg, Mg, M2g = P.psgla(init, dg, den, noise=noise, **kw)
        Xp, Mp, _ = P.psgla(init, dg, den, n_chains=2, rng="philox", **kw)  # the fused next-pre path on a padded problem
    else:
        prm = io_.resolve_params("pnp_ula", den="DRUNet", s=5.0)
        delta = torch.tensor(prm["delta"], device="cuda", dtype=torch.float32)
        lambd = torch.tensor(prm["lambd"], device="cuda", dtype=torch.float32)
        Xr, Mr, M2r = io_.pnpula(init, dg, io_.make_prior_grad(net, 1.0, prm["s1"], prm["s2"], device="cuda"), delta, lambd,
                                 n_iter=n_iter, n_inter=2, n_inter_mmse=2, seed=0, device="cuda", noise=noise)
        Xg, Mg, M2g = P.pnpula(init, dg, P.PriorGrad(den, 1.0, prm["s1"], prm["s2"]), delta, lambd, n_iter=n_iter, n_inter=2,
                               n_inter_mmse=2, seed=0, noise=noise)
        Xp, Mp, _ = P.pnpula(init, dg, P.PriorGrad(den, 1.0, prm["s1"], prm["s2"]), delta, lambd, n_iter=n_iter, n_inter=2,
                             n_inter_mmse=2, seed=0, n_chains=2, rng="philox")
    torch.cuda.synchronize()
    assert len(Xr) == len(Xg) and len(Mr) == len(Mg) and Xg[0].shape == (3, 37, 50) and Mg[0].shape == (3, 37, 50)
    observed("DRUNet %s iterate on a padded 37 x 50 problem" % alg,
             max((a - b).abs().max().item() for a, b in zip(Xr + Mr + M2r, Xg + Mg + M2g)), TOL_DRUNET)
    assert Xp[0].shape == (2, 3, 37, 50) and all(torch.isfinite(t).all() for t in Xp + Mp)


def test_psgla_drunet_replay_against_oracle(drunets):
    """PSGLA with the non-residual denoiser: X+ = (1 - alpha) Y + alpha D(Y; s) (restoration_algorithms.py:238)."""
    den, net = drunets
    torch.manual_seed(0)
    im = torch.rand(1, 3, 32, 48, device="cuda")
    dg, init, y, mask = P.make_inpainting(im, prop=0.5, sigma=1.0, seed_ip=0)
    prm = io_.resolve_params("psgla", den="DRUNet", lambd=25.0)
    n_iter = 6
    g = torch.Generator(device="cuda").manual_seed(0)
    noise = torch.stack([torch.randn(im.shape, generator=g, device="cuda") for _ in range(n_iter)])
    for alpha in (1.0, 0.7):
        kw = dict(alpha=torch.tensor(alpha, device="cuda"), lambd=torch.tensor(prm["lambd"], device="cuda"),
                  sig_float=prm["s"], delta=prm["delta"], n_iter=n_iter, n_inter=2, n_inter_mmse=2, seed=0)
        Xr, Mr, M2r = io_.psgla(init, dg, net, device="cuda", noise=noise, **kw)
        Xg, Mg, M2g = P.psgla(init, dg, den, noise=noise, **kw)
        torch.cuda.synchronize()
        assert len(Xr) == len(Xg) and len(Mr) == len(Mg) == len(M2g)
        observed("DRUNet psgla iterate", max((a - b).abs().max().item() for a, b in zip(Xr + Mr, Xg + Mg)), TOL_DRUNET)


def test_pnpula_drunet_replay_against_oracle(drunets):
    """PnP-ULA with prior_grad = alpha (D(X; s1) - X) / s2 (sampling_images.py:156-157) and a non-residual denoiser."""
    den, net = drunets
    torch.manual_seed(1)
    im = torch.rand(1, 3, 32, 32, device="cuda")
    dg, init, y = P.make_deblurring(im, l=2, blur_type="gaussian", si=1.0, sigma=1.0, seed_ip=0)
    prm = io_.resolve_params("pnp_ula", den="DRUNet", s=5.0)
    n_iter = 5
    g = torch.Generator(device="cuda").manual_seed(0)
    noise = torch.stack([torch.randn(im.shape, generator=g, device="cuda") for _ in range(n_iter)])
    delta = torch.tensor(prm["delta"], device="cuda", dtype=torch.float32)
    lambd = torch.tensor(prm["lambd"], device="cuda", dtype=torch.float32)
    pg_ref = io_.make_prior_grad(net, 1.0, prm["s1"], prm["s2"], device="cuda")
    pg = P.PriorGrad(den, 1.0, prm["s1"], prm["s2"])
    Xr, Mr, _ = io_.pnpula(init, dg, pg_ref, delta, lambd, n_iter=n_iter, n_inter=1, n_inter_mmse=1, seed=0, device="cuda", noise=noise)
    Xg, Mg, _ = P.pnpula(init, dg, pg, delta, lambd, n_iter=n_iter, n_inter=1, n_inter_mmse=1, seed=0, noise=noise)
    torch.cuda.synchronize()
    assert len(Xr) == len(Xg) and len(Mr) == len(Mg)
    observed("DRUNet pnpula iterate", max((a - b).abs().max().item() for a, b in zip(Xr + Mr, Xg + Mg)), TOL_DRUNET)


@pytest.mark.parametrize("family", ["dncnn", "drunet"])
def test_pnp_and_red_against_oracle(drunets, family):
    """The deterministic siblings (restoration_algorithms.py:386-529) reuse the Langevin kernels with the noise switched
    off; DRUNet makes the sigma-annealing schedules (40/255 for n_iter // 10 iterations, 50/255 for 10) observable."""
    if family == "drunet":
        den, net = drunets
    else:
        sd = io_.make_dncnn_weights(seed=0, n_power_iter=5, spatial=16)
        den = P.DnCNN(pretrained=sd)
        net = io_.DnCNN().cuda()
        net.load_state_dict(sd)
    torch.manual_seed(2)
    im = torch.rand(1, 3, 32, 40, device="cuda")
    dg, init, y, mask = P.make_inpainting(im, prop=0.5, sigma=1.0, seed_ip=0)
    s = 5 / 255
    kw = dict(alpha=torch.tensor(0.8, device="cuda"), lambd=torch.tensor(25.0, device="cuda"), sig_float=s, delta=s * s, n_iter=22)
    Xr, Fr, _ = io_.pnp(init, dg, "inpainting", net, device="cuda", **kw)
    Xg, Fg, Eg = P.pnp(init, dg, "inpainting", den, **kw)
    assert Eg == [] and len(Fg) == 1 and len(Xg) == len(Xr) == 22
    observed(family + " pnp iterate", max((a - b).abs().max().item() for a, b in zip(Xr + Fr, Xg + Fg)), TOL_DRUNET)
    kw = dict(lambd=torch.tensor(3000.0, device="cuda"), sig_float=s, delta=1e-5, n_iter=14)
    Xr, Fr, _ = io_.red(init, dg, "inpainting", net, device="cuda", **kw)
    Xg, Fg, Eg = P.red(init, dg, "inpainting", den, **kw)
    assert Eg == [] and len(Xg) == 14
    observed(family + " red iterate", max((a - b).abs().max().item() for a, b in zip(Xr + Fr, Xg + Fg)), TOL_DRUNET)
