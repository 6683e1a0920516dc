"""GPU tests of grayscale (one-channel) images with one-channel DnCNN / DRUNet networks.

The main check embeds a grayscale network in a colour one (input channel 0 -- and DRUNet's noise-level channel 3 -- of the head,
output channel 0 of the tail, zeros elsewhere) and runs the colour path on an image whose channel 0 is the grayscale image:
every grayscale iterate, sample and window moment must equal channel 0 of the colour run bit for bit.  That rests on zero
weights adding exactly zero to the accumulator (checked on the first and last layers alone first), on the padded K / N columns
being independent, and on channel 0's element index and Philox counter not depending on the channel count.  Then the samplers
against the oracle restatement with one-channel networks under replayed noise, the one-channel layers against fp64, the
torch_cuda noise stream, batch independence, run_image_set and the rejections."""
import pytest
import torch

import conv_reference as CR
import psgla_b200 as P
from conftest import observed
from oracle import image_oracle as io_

pytestmark = pytest.mark.gpu
L = P._lib
BF = torch.bfloat16
SIG = 5 / 255


def tol_iterate(n_iter):
    return max(1e-3, 4e-5 * n_iter)  # test_image_gpu.py's bound for the samplers against the oracle


def embed_dncnn(sd1):
    """The colour DnCNN state dict that computes the grayscale network on channel 0 and zero on channels 1, 2."""
    sd3 = {k: v.clone() for k, v in sd1.items()}
    w = torch.zeros(sd1["in_conv.weight"].shape[0], 3, 3, 3)
    w[:, 0] = sd1["in_conv.weight"][:, 0]
    sd3["in_conv.weight"] = w
    w = torch.zeros(3, sd1["out_conv.weight"].shape[1], 3, 3)
    w[0] = sd1["out_conv.weight"][0]
    sd3["out_conv.weight"] = w
    b = torch.zeros(3)
    b[0] = sd1["out_conv.bias"][0]
    sd3["out_conv.bias"] = b
    return sd3


def embed_drunet(sd1):
    sd3 = {k: v.clone() for k, v in sd1.items()}
    w = torch.zeros(64, 4, 3, 3)
    w[:, 0], w[:, 3] = sd1["m_head.weight"][:, 0], sd1["m_head.weight"][:, 1]
    sd3["m_head.weight"] = w
    w = torch.zeros(3, 64, 3, 3)
    w[0] = sd1["m_tail.weight"][0]
    sd3["m_tail.weight"] = w
    return sd3


@pytest.fixture(scope="module")
def dncnn_pair():
    sd1 = P.lipschitz_dncnn_state_dict(3, channels=1)
    return P.DnCNN(1, 1, pretrained=sd1), P.DnCNN(pretrained=embed_dncnn(sd1)), sd1


@pytest.fixture(scope="module")
def drunet_pair():
    sd1 = P.random_drunet_state_dict(4, channels=1)
    return P.DRUNet(1, 1, pretrained=sd1), P.DRUNet(pretrained=embed_drunet(sd1)), sd1


def _colour(t1, seed):
    """[1,1,H,W] -> [1,3,H,W] with t1 in channel 0 and unrelated values in channels 1, 2."""
    g = torch.Generator(device=t1.device).manual_seed(seed)
    return torch.cat([t1, torch.rand((1, 2) + tuple(t1.shape[2:]), generator=g, device=t1.device)], 1).contiguous()


def _problems(problem, H, W, seed=0):
    """(grayscale data_grad, init, colour data_grad, init) with the grayscale problem in channel 0 of the colour one."""
    torch.manual_seed(seed)
    im1 = torch.rand(1, 1, H, W, device="cuda")
    if problem == "inpainting":
        dg1, init1, y1, mask1 = P.make_inpainting(im1, prop=0.5, sigma=1.0, seed_ip=seed)
        dg3 = P.InpaintingDataGrad(_colour(mask1, 1).round(), _colour(y1, 2), dg1.sigma2)
        return dg1, init1, dg3, _colour(init1, 3)
    dg1, init1, y1 = P.make_deblurring(im1, l=4, sigma=1.0, seed_ip=seed)
    dg3 = P.DeblurDataGrad(dg1.h1d, dg1.l, _colour(y1, 2), dg1.sigma2)
    return dg1, init1, dg3, _colour(init1, 3)


def _assert_channel0(gray, colour, squeeze):
    for lg, lc in zip(gray, colour):
        assert len(lg) == len(lc)
        for a, b in zip(lg, lc):
            want = b[0] if squeeze else b[:, 0:1]  # a single grayscale chain comes back as [H, W], like torch.squeeze
            assert a.shape == want.shape and torch.equal(a, want)


def _run(alg, den, dg, init, store, form=None, **kw):
    """form "unfused": the stand-alone pre kernel every iteration; "4pass": the four-pass deblurring pre."""
    prm = io_.resolve_params("psgla" if alg == "psgla" else "pnp_ula", s=5.0)
    common = dict(n_iter=9, n_inter=2, n_inter_mmse=2, store=store, **kw)
    if alg == "psgla":
        run = P.psgla_run(init, dg, den, alpha=torch.tensor(0.9, device="cuda"), lambd=torch.tensor(prm["lambd"], device="cuda"),
                          sig_float=prm["s"], delta=prm["delta"], **common)
    else:
        pg = P.PriorGrad(den, 1.0, SIG, SIG ** 2)
        run = P.pnpula_run(init, dg, pg, torch.tensor(1e-5, device="cuda"), torch.tensor(2e-5, device="cuda"), **common)
    if form == "unfused":
        run.fuse_next_pre = False
    elif form == "4pass":
        run.aty = None
    for i in range(run.n_iter):
        run.step(i)
    return run.finish()


# ---------------------------------------------------------------------------------------------- the zero-weight fact
def test_zero_weights_add_exactly_zero_on_first_and_last_layer(dncnn_pair):
    """First layer: the grayscale input (v, 0, 0, 0) under the grayscale packing == the colour input (v, a, b, 0) under the
    embedded colour packing, bit for bit.  Last layer: the raw grayscale conv == channel 0 of the embedded colour conv."""
    g1, g3, _ = dncnn_pair
    B, H, W = 2, 40, 136
    torch.manual_seed(0)
    x1 = torch.rand(B, 1, H, W, device="cuda")
    x3 = torch.cat([x1, torch.randn(B, 2, H, W, device="cuda")], 1).contiguous()
    lib = L.lib()
    ins, outs = [], []
    for den, x, C in ((g1, x1, 1), (g3, x3, 3)):
        sh = L.ImgShape(B, C, H, W)
        xin = torch.empty(B, H, W, 16, dtype=BF, device="cuda")
        L.check(lib.psgla_img_to_nhwc16(sh, x.data_ptr(), 0.0, xin.data_ptr(), None), "to_nhwc16")
        out = torch.empty(B, H, W, 64, dtype=BF, device="cuda")
        L.check(lib.psgla_conv3x3_layer(den.packed.data_ptr(), den.depth, 0, sh, xin.data_ptr(), out.data_ptr(), 1, None), "first")
        ins.append(xin)
        outs.append(out)
    assert torch.equal(ins[0][..., 1:3], torch.zeros_like(ins[0][..., 1:3])) and not torch.equal(ins[0], ins[1])
    assert torch.equal(outs[0], outs[1])
    hidden = (torch.randn(B, H, W, 64, device="cuda") * 0.5).relu().to(BF)
    raws = []
    for den, C in ((g1, 1), (g3, 3)):
        r = torch.empty(B, C, H, W, device="cuda")
        L.check(lib.psgla_conv3x3_layer(den.packed.data_ptr(), den.depth, den.depth - 1, L.ImgShape(B, C, H, W), hidden.data_ptr(),
                                        r.data_ptr(), 0, None), "last")
        raws.append(r)
    torch.cuda.synchronize()
    assert torch.equal(raws[0], raws[1][:, 0:1])


# ---------------------------------------------------------------------------------------------- bit-identity with colour
@pytest.mark.parametrize("family", ["dncnn", "drunet"])
@pytest.mark.parametrize("alg", ["psgla", "pnpula"])
@pytest.mark.parametrize("problem,form", [("inpainting", "fused"), ("inpainting", "unfused"), ("deblurring", "ata"),
                                          ("deblurring", "4pass")])
@pytest.mark.parametrize("store", ["all", "stats"])
def test_gray_equals_channel0_of_embedded_colour_run(family, alg, problem, form, store, dncnn_pair, drunet_pair):
    g1, g3, _ = dncnn_pair if family == "dncnn" else drunet_pair
    H, W = (40, 48) if family == "drunet" else (36, 52)
    dg1, init1, dg3, init3 = _problems(problem, H, W, seed=1)
    kw = dict(seed=7, n_chains=2, chain_id0=3, rng="philox", form=form)
    gray = _run(alg, g1, dg1, init1, store, **kw)
    colour = _run(alg, g3, dg3, init3, store, **kw)
    torch.cuda.synchronize()
    _assert_channel0(gray, colour, squeeze=False)
    assert gray[0 if store == "all" else 1][0].shape[1] == 1


@pytest.mark.parametrize("family", ["dncnn", "drunet"])
def test_gray_equals_channel0_under_replayed_noise(family, dncnn_pair, drunet_pair):
    """One chain with a replayed noise tensor (the colour run gets the grayscale draws in channel 0)."""
    g1, g3, _ = dncnn_pair if family == "dncnn" else drunet_pair
    dg1, init1, dg3, init3 = _problems("inpainting", 37, 50, seed=2)
    g = torch.Generator(device="cuda").manual_seed(5)
    z1 = torch.randn((9, 1, 1, 37, 50), generator=g, device="cuda")
    z3 = torch.cat([z1, torch.randn((9, 1, 2, 37, 50), generator=g, device="cuda")], 2)
    gray = _run("psgla", g1, dg1, init1, "all", seed=0, noise=z1)
    colour = _run("psgla", g3, dg3, init3, "all", seed=0, noise=z3)
    torch.cuda.synchronize()
    _assert_channel0(gray, colour, squeeze=True)


def test_pnp_red_gray_equal_channel0(drunet_pair):
    g1, g3, _ = drunet_pair
    dg1, init1, dg3, init3 = _problems("inpainting", 37, 50, seed=3)
    a = P.pnp(init1, dg1, "inpainting", g1, 0.5, 1.0, sig_float=SIG, delta=1e-5, n_iter=8)
    b = P.pnp(init3, dg3, "inpainting", g3, 0.5, 1.0, sig_float=SIG, delta=1e-5, n_iter=8)
    _assert_channel0(a, b, squeeze=True)
    a = P.red(init1, dg1, "inpainting", g1, 0.5, sig_float=SIG, delta=1e-5, n_iter=12)
    b = P.red(init3, dg3, "inpainting", g3, 0.5, sig_float=SIG, delta=1e-5, n_iter=12)
    _assert_channel0(a, b, squeeze=True)


# ---------------------------------------------------------------------------------------------- against the oracle
@pytest.fixture(scope="module")
def oracle_nets(dncnn_pair, drunet_pair):
    d = io_.DnCNN(in_channels=1, out_channels=1).cuda()
    d.load_state_dict(dncnn_pair[2])
    u = io_.DRUNet(in_channels=1, out_channels=1).cuda()
    u.load_state_dict(drunet_pair[2])
    return d.eval(), u.eval()


@pytest.mark.parametrize("family,problem,H,W", [("dncnn", "inpainting", 48, 64), ("dncnn", "deblurring", 48, 64),
                                                ("drunet", "inpainting", 37, 50), ("drunet", "deblurring", 40, 48)])
@pytest.mark.parametrize("alg", ["psgla", "pnpula"])
def test_samplers_against_oracle(family, problem, H, W, alg, dncnn_pair, drunet_pair, oracle_nets):
    den = (dncnn_pair if family == "dncnn" else drunet_pair)[0]
    net = oracle_nets[0 if family == "dncnn" else 1]
    dg, init, _, _ = _problems(problem, H, W, seed=4)
    n_iter = 12
    g = torch.Generator(device="cuda").manual_seed(6)
    noise = torch.randn((n_iter, 1, 1, H, W), generator=g, device="cuda")
    kw = dict(n_iter=n_iter, n_inter=3, n_inter_mmse=3)
    if alg == "psgla":
        prm = io_.resolve_params("psgla")
        a = dict(alpha=torch.tensor(0.9, device="cuda"), lambd=torch.tensor(prm["lambd"], device="cuda"), sig_float=prm["s"],
                 delta=prm["delta"])
        ref = io_.psgla(init, dg, net, device="cuda", noise=noise, **a, **kw)
        got = P.psgla(init, dg, den, noise=noise, seed=0, **a, **kw)
    else:
        delta, lambd = torch.tensor(1e-5, device="cuda"), torch.tensor(2e-5, device="cuda")
        ref = io_.pnpula(init, dg, io_.make_prior_grad(net, 1.0, SIG, SIG ** 2, device="cuda"), delta, lambd, device="cuda",
                         noise=noise, **kw)
        got = P.pnpula(init, dg, P.PriorGrad(den, 1.0, SIG, SIG ** 2), delta, lambd, noise=noise, seed=0, **kw)
    torch.cuda.synchronize()
    for lr, lg in zip(ref, got):
        assert len(lr) == len(lg)
    assert got[0][0].shape == (H, W)
    err = max((a - b).abs().max().item() for lr, lg in zip(ref, got) for a, b in zip(lr, lg))
    observed("gray %s %s %s: max |iterate - oracle|" % (family, alg, problem), err, tol_iterate(n_iter))


@pytest.mark.parametrize("family", ["dncnn", "drunet"])
def test_pnp_red_against_oracle(family, dncnn_pair, drunet_pair, oracle_nets):
    den = (dncnn_pair if family == "dncnn" else drunet_pair)[0]
    net = oracle_nets[0 if family == "dncnn" else 1]
    dg, init, _, _ = _problems("inpainting", 37, 50, seed=5)
    got = P.pnp(init, dg, "inpainting", den, 0.5, 1.0, sig_float=SIG, delta=1e-5, n_iter=10)
    ref = io_.pnp(init, dg, "inpainting", net, 0.5, 1.0, sig_float=SIG, delta=1e-5, n_iter=10, device="cuda")
    err = max((a - b).abs().max().item() for a, b in zip(ref[0], got[0]))
    observed("gray pnp %s: max |iterate - oracle|" % family, err, tol_iterate(10))
    got = P.red(init, dg, "inpainting", den, 0.5, sig_float=SIG, delta=1e-5, n_iter=12)
    ref = io_.red(init, dg, "inpainting", net, 0.5, sig_float=SIG, delta=1e-5, n_iter=12, device="cuda")
    err = max((a - b).abs().max().item() for a, b in zip(ref[0], got[0]))
    observed("gray red %s: max |iterate - oracle|" % family, err, tol_iterate(12))


# ---------------------------------------------------------------------------------------------- layers against fp64
def test_one_channel_dncnn_first_and_last_layer_against_fp64(dncnn_pair):
    den, _, sd1 = dncnn_pair
    lib = L.lib()
    B, H, W = 2, 33, 140
    torch.manual_seed(1)
    x = torch.rand(B, 1, H, W, device="cuda")
    sh = L.ImgShape(B, 1, H, W)
    xin = torch.empty(B, H, W, 16, dtype=BF, device="cuda")
    L.check(lib.psgla_img_to_nhwc16(sh, x.data_ptr(), 0.0, xin.data_ptr(), None), "to_nhwc16")
    out = CR.Guarded((B, H, W, 64), BF)
    L.check(lib.psgla_conv3x3_layer(den.packed.data_ptr(), den.depth, 0, sh, xin.data_ptr(), out.ptr(), 1, None), "first")
    ref, S = CR.reference("conv3", xin[..., :1].permute(0, 3, 1, 2), sd1["in_conv.weight"], sd1["in_conv.bias"], relu=True)
    torch.cuda.synchronize()
    assert out.intact()
    CR.check("gray dncnn first layer", out.tensor.permute(0, 3, 1, 2), ref, S)
    hidden = (torch.randn(B, H, W, 64, device="cuda") * 0.5).relu().to(BF)
    r = CR.Guarded((B, 1, H, W), torch.float32)
    L.check(lib.psgla_conv3x3_layer(den.packed.data_ptr(), den.depth, den.depth - 1, sh, hidden.data_ptr(), r.ptr(), 0, None),
            "last")
    ref, S = CR.reference("conv3", hidden.permute(0, 3, 1, 2), sd1["out_conv.weight"], sd1["out_conv.bias"])
    torch.cuda.synchronize()
    assert r.intact()
    CR.check("gray dncnn last layer", r.tensor, ref, S)


def test_one_channel_drunet_head_and_tail_against_fp64(drunet_pair):
    den, _, sd1 = drunet_pair
    lib = L.lib()
    B, H, W = 2, 40, 136
    torch.manual_seed(2)
    x = torch.rand(B, 1, H, W, device="cuda")
    sh = L.ImgShape(B, 1, H, W)
    xin = torch.empty(B, H, W, 16, dtype=BF, device="cuda")
    L.check(lib.psgla_img_to_nhwc16(sh, x.data_ptr(), SIG, xin.data_ptr(), None), "to_nhwc16")
    out = CR.Guarded((B, H, W, 64), BF)
    L.check(lib.psgla_drunet_layer(den.packed.data_ptr(), sh, 0, xin.data_ptr(), None, None, out.ptr(), None), "head")
    x2 = torch.stack([xin[..., 0], xin[..., 3]], 1)  # the image and the noise-level map, as the head sees them
    ref, S = CR.reference("conv3", x2, sd1["m_head.weight"])
    torch.cuda.synchronize()
    assert out.intact()
    CR.check("gray drunet head", out.tensor.permute(0, 3, 1, 2), ref, S)
    hidden = (torch.randn(B, H, W, 64, device="cuda") * 0.5).to(BF)
    r = CR.Guarded((B, 1, H, W), torch.float32)
    last = len(P.DRUNET_KEYS) - 1
    L.check(lib.psgla_drunet_layer(den.packed.data_ptr(), sh, last, hidden.data_ptr(), None, None, r.ptr(), None), "tail")
    ref, S = CR.reference("conv3", hidden.permute(0, 3, 1, 2), sd1["m_tail.weight"])
    torch.cuda.synchronize()
    assert r.intact()
    CR.check("gray drunet tail", r.tensor, ref, S)


# ---------------------------------------------------------------------------------------------- noise, batches, image sets
@pytest.mark.parametrize("problem,H,W", [("inpainting", 40, 52), ("inpainting", 33, 31), ("deblurring", 48, 36)])
def test_torch_cuda_stream_equals_torch_randn(problem, H, W, dncnn_pair):
    den = dncnn_pair[0]
    dg, init, _, _ = _problems(problem, H, W, seed=6)
    kw = dict(seed=3)
    for alg in ("psgla", "pnpula"):
        a = _run(alg, den, dg, init, "all", rng="torch", **kw)
        b = _run(alg, den, dg, init, "all", rng="torch_cuda", **kw)
        torch.cuda.synchronize()
        for la, lb in zip(a, b):
            assert len(la) == len(lb) and all(torch.equal(ta, tb) for ta, tb in zip(la, lb))


@pytest.mark.parametrize("family,problem", [("dncnn", "inpainting"), ("dncnn", "deblurring"), ("drunet", "inpainting")])
def test_batch_independence(family, problem, dncnn_pair, drunet_pair):
    den = (dncnn_pair if family == "dncnn" else drunet_pair)[0]
    dg, init, _, _ = _problems(problem, 40, 48, seed=7)
    B = 3
    full = _run("psgla", den, dg, init, "all", seed=2, n_chains=B, rng="philox")
    for b in range(B):
        one = _run("psgla", den, dg, init, "all", seed=2, n_chains=1, chain_id0=b, rng="philox")
        for lf, lo in zip(full, one):
            assert all(torch.equal(tf[b:b + 1], to) for tf, to in zip(lf, lo))


def test_run_image_set_gray_rows_equal_per_image_runs(dncnn_pair):
    den = dncnn_pair[0]
    g = torch.Generator().manual_seed(3)
    images = [torch.rand(1, 32, 40, generator=g), torch.rand(1, 1, 24, 28, generator=g)]
    prm = dict(P.sampler_params("psgla", den="DnCNN", N=1000), N=11, n_inter=2, n_inter_mmse=2)
    res = P.run_image_set(images, den, problem="inpainting", alg="psgla", n_chains=2, params=prm, seed=5, keep_maps=True)
    assert [d["index"] for d in res] == [0, 1]
    for i, im in enumerate(images):
        imc = im.reshape(1, 1, im.shape[-2], im.shape[-1]).cuda()
        dg, init, _, _ = P.make_inpainting(imc, prop=0.5, sigma=1.0, seed_ip=0)
        _, M, _ = P.psgla(init, dg, den, **P.as_psgla_kwargs(prm, seed=5), n_chains=2, chain_id0=2 * i, rng="philox")
        xmmse = torch.stack(M).mean(0).mean(0)
        assert res[i]["xmmse"].shape == (1, im.shape[-2], im.shape[-1])
        assert (res[i]["xmmse"] - xmmse).abs().max().item() < 1e-6
        p, s = P.psnr_ssim(xmmse, imc[0])
        assert abs(res[i]["psnr_mmse"] - p.item()) < 1e-3 and abs(res[i]["ssim_mmse"] - s.item()) < 1e-4


# ---------------------------------------------------------------------------------------------- rejections
def test_python_rejections(dncnn_pair, drunet_pair):
    g1, g3, sd1 = dncnn_pair
    dg1, init1, dg3, init3 = _problems("inpainting", 32, 40)
    kw = dict(alpha=1.0, lambd=5.0, n_iter=3, seed=0)
    with pytest.raises(ValueError, match="grayscale image"):
        P.psgla(init3, dg3, g1, **kw)
    with pytest.raises(ValueError, match="colour image"):
        P.psgla(init1, dg1, g3, **kw)
    with pytest.raises(ValueError, match="colour image"):
        P.psgla(init1, dg1, drunet_pair[1], **kw)
    with pytest.raises(ValueError, match="TVDenoiser \\(colour-only\\)"):
        P.psgla(init1, dg1, P.TVDenoiser(), **kw)
    with pytest.raises(ValueError, match="GSDRUNet \\(colour-only\\)"):
        P.psgla(init1, dg1, P.GSDRUNet(), **kw)
    with pytest.raises(ValueError, match="to match init"):  # a colour mask with a grayscale init
        P.psgla(init1, P.InpaintingDataGrad(dg3.mask, dg1.y, dg1.sigma2), g1, **kw)
    with pytest.raises(ValueError, match="in_conv.weight has shape"):
        P.DnCNN(1, 1, pretrained=P.random_dncnn_state_dict(0))
    with pytest.raises(ValueError, match="m_head.weight has shape"):
        P.DRUNet(1, 1, pretrained=P.random_drunet_state_dict(0))
    with pytest.raises(ValueError, match="in_conv.weight has shape"):
        P.DnCNN(pretrained=sd1)
    for bad in ((1, 3), (2, 2), (4, 4)):
        with pytest.raises(ValueError):
            P.DnCNN(*bad)
        with pytest.raises(ValueError):
            P.DRUNet(*bad)
    with pytest.raises(ValueError, match="1-channel"):
        g1.forward(torch.rand(1, 3, 16, 16, device="cuda"))
