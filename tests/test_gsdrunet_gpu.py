"""GPU tests of the gradient-step DRUNet (csrc/gsdrunet.cu): every forward and backward layer element by element against the
fp64 sum of the same bf16 operands (tests/conv_reference.py's criterion), the adjoint identity of every backward layer, the
whole denoiser against the fp64 restatement (tests/gs_reference.py), and the samplers against the oracle under replayed noise."""
import math

import pytest
import torch
import torch.nn.functional as F

import conv_reference as CR
import gs_reference as GS
import psgla_b200 as P
from conftest import observed
from oracle import image_oracle as io_

pytestmark = pytest.mark.gpu
KEYS = P.GSDRUNET_KEYS
SIGMA = 5 / 255
TOL_SAMPLER = 2e-3  # test_drunet_gpu.py's bound for the samplers with a non-residual U-Net denoiser


def _fwd_info(l):
    """(kind, input scale, output scale, act, n residual inputs) of forward layer l, from its state-dict key."""
    k = KEYS[l]
    if k == "m_head.weight":
        return "head", 0, 0, None, 0
    if k == "m_tail.weight":
        return "tail", 0, 0, None, 0
    stage = 3 if k.startswith("m_body") else int(k[len("m_down")] if k.startswith("m_down") else k[len("m_up")])
    if ".res." in k:
        s = 3 if k.startswith("m_body") else stage - 1
        if ".res.0." in k:
            return "conv3", s, s, "elu", 0
        last = k.startswith("m_body.1.") or (k.startswith("m_up") and ".2.res." in k)
        return "conv3", s, s, None, 2 if last else 1
    if k.startswith("m_down"):
        return "down", stage - 1, stage, None, 0
    return "up", stage, stage - 1, None, 0


def _bwd_nres(l):
    """Residual inputs of the adjoint of forward layer l (a first conv of a block: res1, + res2 for the first block of the body
    and of each encoder stage)."""
    k = KEYS[l]
    if ".res.0." not in k:
        return 0
    return 2 if (k.startswith("m_down") or k.startswith("m_body")) and ".0.res." in k else 1


@pytest.fixture(scope="module")
def gs():
    sd = P.random_gsdrunet_state_dict(0)
    return P.GSDRUNet(pretrained=sd), sd


def _bf(x):
    return x.to(torch.bfloat16)


def _nhwc(x):
    return x.permute(0, 2, 3, 1).contiguous()


def _nhwc16(x):
    out = torch.zeros(x.shape[0], x.shape[2], x.shape[3], 16, dtype=torch.bfloat16, device=x.device)
    out[..., :3] = _nhwc(x[:, :3]).to(torch.bfloat16)
    if x.shape[1] > 3:
        out[..., 3] = x[:, 3].to(torch.bfloat16)
    return out


def _lin(kind, x, w, adjoint):
    """The linear map of a layer (fp64 torch) or its adjoint."""
    if kind in ("head", "tail", "conv3"):
        return F.conv_transpose2d(x, w, padding=1) if adjoint else F.conv2d(x, w, padding=1)
    if kind == "down":
        return F.conv_transpose2d(x, w, stride=2) if adjoint else F.conv2d(x, w, stride=2)
    return F.conv2d(x, w, stride=2) if adjoint else F.conv_transpose2d(x, w, stride=2)


def _layer(den, shape, backward, idx, xin, out_shape, res1=None, res2=None, gate=None, fp32=False):
    lib = P._lib.lib()
    out = CR.Guarded(out_shape, torch.float32 if fp32 else torch.bfloat16)
    ptr = lambda t: t.data_ptr() if t is not None else None  # noqa: E731
    P._lib.check(lib.psgla_gsdrunet_layer(den.packed.data_ptr(), P._lib.ImgShape(*shape), backward, idx, xin.data_ptr(),
                                          ptr(res1), ptr(res2), ptr(gate), out.ptr(), None), "psgla_gsdrunet_layer")
    torch.cuda.synchronize()
    assert out.intact()
    return out.tensor


def _layer_case(den, sd, shape, backward, idx, g, unit_gate=False, zero_res=False):
    """Runs one layer on random operands; returns (got NCHW, ref fp64, S, the input NCHW, the linear operator's weight)."""
    B, _, H, W = shape
    fl = 35 - idx if backward else idx
    kind, s_in, s_out, act, nres = _fwd_info(fl)
    w = sd[KEYS[fl]].cuda()
    wb = CR.bf16_weights(w).double()
    if backward:
        s_in, s_out = s_out, s_in
        nres = _bwd_nres(fl)
    cin, cout = (wb.shape[1], wb.shape[0]) if kind != "up" else (wb.shape[0], wb.shape[1])
    if backward:
        cin, cout = cout, cin
    if kind == "head" and not backward:
        cin = 4
    if kind == "head" and backward:
        cout = 3
    hi, wi, ho, wo = H >> s_in, W >> s_in, H >> s_out, W >> s_out
    x = _bf(torch.randn(B, cin, hi, wi, device="cuda", generator=g))
    if (kind == "head" and not backward) or (kind == "tail" and backward):
        xin = _nhwc16(x.float())
    else:
        xin = _nhwc(x)
    gate = None
    is_gate = backward and kind == "conv3" and act is None  # the adjoint of a block's second conv
    rs = [_bf(torch.zeros(B, cout, ho, wo, device="cuda") if zero_res else torch.randn(B, cout, ho, wo, device="cuda", generator=g))
          for _ in range(nres)]
    if is_gate:
        t = torch.ones(B, cout, ho, wo, device="cuda") if unit_gate else torch.randn(B, cout, ho, wo, device="cuda", generator=g)
        gate = _bf(t.clamp_min(-1.0))  # an ELU output is > -1
    raw = (kind == "tail" and not backward) or (kind == "head" and backward)
    got = _layer(den, shape, backward, idx, xin, (B, 3, H, W) if raw else (B, ho, wo, cout),
                 res1=_nhwc(rs[0]) if nres >= 1 else None, res2=_nhwc(rs[1]) if nres >= 2 else None,
                 gate=_nhwc(gate) if gate is not None else None, fp32=raw)
    if not raw:
        got = got.permute(0, 3, 1, 2)
    x64 = x.double()
    ref = _lin(kind, x64, wb, backward)
    S = _lin(kind, x64.abs(), wb.abs(), backward)
    if kind == "head" and backward:
        ref, S = ref[:, :3], S[:, :3]
    for r in rs:
        ref, S = ref + r.double(), S + r.double().abs()
    if gate is not None:
        t64 = gate.double()
        d = torch.where(t64 > 0, torch.ones_like(t64), t64 + 1)
        ref, S = ref * d, S * d.abs()
    if act == "elu" and not backward:
        ref = F.elu(ref)  # the bound holds for the pre-activation and ELU is 1-Lipschitz
    return got, ref, S, x, wb, kind


ALL = [(b, i) for b in (0, 1) for i in range(36)]
SHAPES = [(1, 3, 64, 96), (1, 3, 16, 512)]  # scale 1 reaches the row-box / resident-weight 128-channel forms at W >= 256


@pytest.mark.parametrize("shape", SHAPES)
@pytest.mark.parametrize("backward,idx", ALL)
def test_gs_layer_against_fp64(gs, shape, backward, idx):
    den, sd = gs
    g = torch.Generator(device="cuda").manual_seed(100 * backward + idx)
    got, ref, S, *_ = _layer_case(den, sd, shape, backward, idx, g)
    CR.check("gs %s %d %s" % ("bwd" if backward else "fwd", idx, shape), got, ref, S)


SCALE0 = [(b, i) for b, i in ALL if (KEYS[35 - i if b else i].startswith(("m_head", "m_tail", "m_down1.0", "m_down1.1",
                                                                              "m_up1.1", "m_up1.2")))]


@pytest.mark.parametrize("backward,idx", SCALE0)
def test_gs_full_resolution_layers_2x320x480(gs, backward, idx):
    den, sd = gs
    g = torch.Generator(device="cuda").manual_seed(7 + 100 * backward + idx)
    got, ref, S, *_ = _layer_case(den, sd, (2, 3, 320, 480), backward, idx, g)
    CR.check("gs %s %d 2x320x480" % ("bwd" if backward else "fwd", idx), got, ref, S)


@pytest.mark.parametrize("idx", range(36))
def test_gs_backward_layer_is_the_adjoint(gs, idx):
    """<L^T g, h> = <g, L h> for backward layer idx with its gates at 1 and residual inputs at 0, L the library's own forward
    layer with zero residual inputs (for the ELU layers, whose forward is not linear, the fp64 conv of the bf16 weights)."""
    den, sd = gs
    shape = (1, 3, 32, 48)
    g = torch.Generator(device="cuda").manual_seed(300 + idx)
    lt_g, _, _, gin, wb, kind = _layer_case(den, sd, shape, 1, idx, g, unit_gate=True, zero_res=True)
    fl = 35 - idx
    kind_f, s_in, s_out, act, nres = _fwd_info(fl)
    B, _, H, W = shape
    cin = 4 if kind_f == "head" else (wb.shape[1] if kind_f != "up" else wb.shape[0])
    h = _bf(torch.randn(B, cin, H >> s_in, W >> s_in, device="cuda", generator=g))
    if kind_f == "head":
        h[:, 3] = 0  # the sigma channel's gradient is dropped
    if act == "elu":
        lh = _lin(kind_f, h.double(), wb, False)
    else:
        cout = gin.shape[1]
        zeros = [_nhwc(_bf(torch.zeros(B, cout, H >> s_out, W >> s_out, device="cuda"))) for _ in range(nres)]
        xin = _nhwc16(h.float()) if kind_f == "head" else _nhwc(h)
        raw = kind_f == "tail"
        out = _layer(den, shape, 0, fl, xin, (B, 3, H, W) if raw else (B, H >> s_out, W >> s_out, cout),
                     res1=zeros[0] if nres >= 1 else None, res2=zeros[1] if nres >= 2 else None, fp32=raw)
        lh = (out if raw else out.permute(0, 3, 1, 2)).double()
    lhs_t = lt_g.double() * h.double()[:, :lt_g.shape[1]]
    rhs_t = gin.double() * lh
    lhs, rhs = lhs_t.sum().item(), rhs_t.sum().item()
    scale = max(lhs_t.abs().sum().item(), rhs_t.abs().sum().item())
    observed("adjoint identity backward %d (relative to sum |terms|)" % idx, abs(lhs - rhs) / scale, 4e-3)


def _lib_network(den, x, sigma):
    """N(x) through the library's forward layers (the tensors psgla_gsdrunet_denoise_post_next computes internally)."""
    B, _, H, W = x.shape
    shape = (B, 3, H, W)
    xs4 = torch.cat((x, torch.full_like(x[:, :1], sigma)), 1)
    cur = _nhwc16(xs4)
    skips, li = [], 0

    def run(inp, r1=None, r2=None):
        nonlocal li
        kind, s_in, s_out, act, nres = _fwd_info(li)
        raw = kind == "tail"
        co = 3 if raw else (P.denoisers._drunet_shape(KEYS[li])[1 if kind == "up" else 0])
        out = _layer(den, shape, 0, li, inp, (B, 3, H, W) if raw else (B, H >> s_out, W >> s_out, co), res1=r1, res2=r2,
                     fp32=raw).clone()
        li += 1
        return out

    def blocks(h, skip):
        for blk in range(2):
            t = run(h)
            h = run(t, h, skip if blk == 1 else None)
        return h

    cur = run(cur)
    for s in range(3):
        skips.append(cur)
        cur = run(blocks(cur, None))
    skips.append(cur)
    cur = blocks(cur, cur)
    for s in (2, 1, 0):
        cur = blocks(run(cur), skips[s])
    return run(cur)


@pytest.mark.parametrize("shape", [(1, 64, 64), (2, 40, 72), (1, 256, 256)])
def test_gs_denoiser_against_fp64(gs, shape):
    den, sd = gs
    B, H, W = shape
    x = torch.rand(B, 3, H, W, device="cuda", generator=torch.Generator(device="cuda").manual_seed(1))
    got = den.forward(x, SIGMA)
    n_lib = _lib_network(den, x, SIGMA)
    torch.cuda.synchronize()
    sd64 = {k: v.double() for k, v in sd.items()}
    grad, n_ref, jtv_ref = GS.grad_g(sd64, x.double(), SIGMA)
    want = x.double() - den.alpha * grad
    rel = lambda a, b: ((a.double() - b).norm() / b.norm()).item()  # noqa: E731
    v_lib = x.double() - n_lib.double()
    jtv_lib = (got.double() - x.double()) / den.alpha + v_lib
    print("GSDRUNet %s: rel L2 error of N %.3g, of J^T v %.3g" % (shape, rel(n_lib, n_ref), rel(jtv_lib, jtv_ref)))
    observed("GSDRUNet x - D(x) rel L2 %s" % (shape,), rel(x.double() - got.double(), x.double() - want), 3e-2)


def test_gs_batch_position_invariance(gs):
    den, _ = gs
    g = torch.Generator(device="cuda").manual_seed(2)
    x = torch.rand(3, 3, 48, 64, device="cuda", generator=g)
    d3 = den.forward(x, SIGMA)
    for b in range(3):
        assert torch.equal(den.forward(x[b:b + 1].contiguous(), SIGMA)[0], d3[b]), b


def _inpaint(seed, H=32, W=48):
    torch.manual_seed(seed)
    im = torch.rand(1, 3, H, W, device="cuda")
    return P.make_inpainting(im, prop=0.5, sigma=1.0, seed_ip=0)


def _noise(n_iter, shape):
    g = torch.Generator(device="cuda").manual_seed(0)
    return torch.stack([torch.randn(shape, generator=g, device="cuda") for _ in range(n_iter)])


def test_psgla_gs_replay_against_oracle(gs):
    den, sd = gs
    ref = GS.GSDRUNet(sd)
    dg, init, y, mask = _inpaint(0)
    prm = io_.resolve_params("psgla", den="DRUNet", lambd=25.0)
    n_iter = 6
    noise = _noise(n_iter, init.shape)
    for alpha in (1.0, 0.7):
        kw = dict(alpha=torch.tensor(alpha, device="cuda"), lambd=torch.tensor(prm["lambd"], device="cuda"),
                  sig_float=prm["s"], delta=prm["delta"], n_iter=n_iter, n_inter=2, n_inter_mmse=2, seed=0)
        Xr, Mr, M2r = io_.psgla(init, dg, ref, device="cuda", noise=noise, **kw)
        Xg, Mg, M2g = P.psgla(init, dg, den, noise=noise, **kw)
        torch.cuda.synchronize()
        assert len(Xr) == len(Xg) and len(Mr) == len(Mg) == len(M2g)
        observed("GSDRUNet psgla iterate", max((a - b).abs().max().item() for a, b in zip(Xr + Mr, Xg + Mg)), TOL_SAMPLER)


def test_pnpula_gs_replay_against_oracle(gs):
    """PnP-ULA evaluates D at the chain state X, not at the sampler's base."""
    den, sd = gs
    ref = GS.GSDRUNet(sd)
    torch.manual_seed(1)
    im = torch.rand(1, 3, 32, 32, device="cuda")
    dg, init, y = P.make_deblurring(im, l=2, blur_type="gaussian", si=1.0, sigma=1.0, seed_ip=0)
    prm = io_.resolve_params("pnp_ula", den="DRUNet", s=5.0)
    n_iter = 5
    noise = _noise(n_iter, im.shape)
    delta = torch.tensor(prm["delta"], device="cuda", dtype=torch.float32)
    lambd = torch.tensor(prm["lambd"], device="cuda", dtype=torch.float32)
    Xr, Mr, _ = io_.pnpula(init, dg, io_.make_prior_grad(ref, 1.0, prm["s1"], prm["s2"], device="cuda"), delta, lambd,
                           n_iter=n_iter, n_inter=1, n_inter_mmse=1, seed=0, device="cuda", noise=noise)
    Xg, Mg, _ = P.pnpula(init, dg, P.PriorGrad(den, 1.0, prm["s1"], prm["s2"]), delta, lambd, n_iter=n_iter, n_inter=1,
                         n_inter_mmse=1, seed=0, noise=noise)
    torch.cuda.synchronize()
    assert len(Xr) == len(Xg) and len(Mr) == len(Mg)
    observed("GSDRUNet pnpula iterate", max((a - b).abs().max().item() for a, b in zip(Xr + Mr, Xg + Mg)), TOL_SAMPLER)


def test_pnp_and_red_gs_against_oracle(gs):
    den, sd = gs
    ref = GS.GSDRUNet(sd)
    dg, init, y, mask = _inpaint(2, 32, 40)
    s = 5 / 255
    kw = dict(alpha=torch.tensor(0.8, device="cuda"), lambd=torch.tensor(25.0, device="cuda"), sig_float=s, delta=s * s, n_iter=22)
    Xr, Fr, _ = io_.pnp(init, dg, "inpainting", ref, device="cuda", **kw)
    Xg, Fg, _ = P.pnp(init, dg, "inpainting", den, **kw)
    assert len(Xg) == len(Xr) == 22
    observed("GSDRUNet pnp iterate", max((a - b).abs().max().item() for a, b in zip(Xr + Fr, Xg + Fg)), TOL_SAMPLER)
    kw = dict(lambd=torch.tensor(3000.0, device="cuda"), sig_float=s, delta=1e-5, n_iter=14)
    Xr, Fr, _ = io_.red(init, dg, "inpainting", ref, device="cuda", **kw)
    Xg, Fg, _ = P.red(init, dg, "inpainting", den, **kw)
    assert len(Xg) == 14
    observed("GSDRUNet red iterate", max((a - b).abs().max().item() for a, b in zip(Xr + Fr, Xg + Fg)), TOL_SAMPLER)


@pytest.mark.parametrize("alg", ["psgla", "pnpula"])
def test_fused_next_pre_is_bit_identical(gs, alg):
    den, _ = gs
    dg, init, y, mask = _inpaint(3)
    outs = []
    for fuse in (True, False):
        if alg == "psgla":
            prm = io_.resolve_params("psgla", den="DRUNet", lambd=25.0)
            run = P.psgla_run(init, dg, den, alpha=0.9, lambd=prm["lambd"], sig_float=prm["s"], delta=prm["delta"], n_iter=5,
                              n_inter=1, n_inter_mmse=2, seed=4, n_chains=2, rng="philox")
        else:
            prm = io_.resolve_params("pnp_ula", den="DRUNet", s=5.0)
            run = P.pnpula_run(init, dg, P.PriorGrad(den, 1.0, prm["s1"], prm["s2"]), prm["delta"], prm["lambd"], n_iter=5,
                               n_inter=1, n_inter_mmse=2, seed=4, n_chains=2, rng="philox")
        assert run.fuse_next_pre
        run.fuse_next_pre = fuse
        for i in range(run.n_iter):
            run.step(i)
        outs.append(run.finish())
    for a, b in zip(outs[0], outs[1]):
        assert len(a) == len(b) and all(torch.equal(u, v) for u, v in zip(a, b))


def test_run_image_set_gs_row_equals_a_per_image_run(gs):
    den, _ = gs
    torch.manual_seed(6)
    ims = [torch.rand(3, 32, 40), torch.rand(3, 32, 40)]
    prm = dict(P.sampler_params("psgla", den="GSDRUNet", N=1000), N=6, n_inter=2, n_inter_mmse=2, lambd=25.0)
    gs_prm, dru_prm = P.sampler_params("psgla", den="GSDRUNet"), P.sampler_params("psgla", den="DRUNet")
    assert gs_prm.pop("den") == "GSDRUNet" and dru_prm.pop("den") == "DRUNet" and gs_prm == dru_prm
    res = P.run_image_set(ims, den, problem="inpainting", alg="psgla", n_chains=2, params=prm, seed=3)
    from psgla_b200 import image_set
    for i, im in enumerate(ims):
        row, _ = image_set._sample_image(i, im, den, "inpainting", "psgla", 2, prm, 3, 0, 0.5, 1.0, 4, "uniform", 1.0, False)
        got = [res[i][k] for k in P.image_set.ROW_FIELDS]
        assert got == [int(v) if k in ("index", "n_chains", "n_windows", "H", "W") else float(v)
                       for k, v in zip(P.image_set.ROW_FIELDS, row.tolist())], i


def test_gs_rejections_on_gpu(gs):
    den, _ = gs
    with pytest.raises(ValueError, match="multiples of 8"):
        den.forward(torch.rand(1, 3, 20, 24, device="cuda"), SIGMA)
    dg, init, y, mask = P.make_inpainting(torch.rand(1, 3, 37, 50, device="cuda"))
    with pytest.raises(ValueError, match="multiples of 8"):
        P.psgla(init, dg, den, alpha=1.0, lambd=1.0, n_iter=2, seed=0)
    with pytest.raises(ValueError, match="multiples of 8"):
        P.pnpula(init, dg, P.PriorGrad(den, 1.0, 0.01, 1e-4), 1e-5, 1.0, n_iter=2, seed=0)
    with pytest.raises(RuntimeError, match="CUDA"):
        den.forward(torch.rand(1, 3, 16, 16), SIGMA)
    lib = P._lib.lib()
    shape = P._lib.ImgShape(1, 3, 16, 16)
    x = torch.rand(1, 3, 16, 16, device="cuda")
    ws = torch.empty(lib.psgla_gsdrunet_workspace_bytes(shape), dtype=torch.uint8, device="cuda")
    den_in = torch.zeros(16 * 16 * 16, dtype=torch.bfloat16, device="cuda")
    post = P._lib.PostParams(1.0, 0.0, 0.0, 1.0)
    import ctypes
    for alpha, wsb, want in ((float("nan"), ws.numel(), -1), (1.0, ws.numel() - 1, -4), (1.0, ws.numel(), 0)):
        rc = lib.psgla_gsdrunet_denoise_post_next(den.packed.data_ptr(), shape, den_in.data_ptr(), None, ws.data_ptr(), wsb,
                                                  x.data_ptr(), alpha, ctypes.byref(post), x.data_ptr(), None, None, None,
                                                  None, None)
        assert rc == want, (alpha, wsb, rc)
    torch.cuda.synchronize()
    assert math.isfinite(float(x.sum()))
