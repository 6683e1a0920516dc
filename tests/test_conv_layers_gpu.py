"""-m gpu: every production conv layer element by element against an fp64 reference (tests/conv_reference.py), and the
per-layer entry points composed back into the production networks bit for bit.

DRUNet layers run through psgla_drunet_layer, i.e. exactly the kernel, ReLU and residual inputs the network uses for that
plan layer.  Inputs and residuals are independent random bf16 N(0, 1) tensors (never the input itself as the residual, so
that a misrouted or shifted residual shows), every output is NaN-poisoned before the call and sits between sentinel guards
that must come back bit-unchanged, and every case runs twice in a row: the layers that alternate their traversal direction
(conv64_hidden, the CTA-pair conv_gemm_layer kernels) walk their items once forward and once backward, and the two outputs
must be bit-identical.

Image shapes (B, H, W) of the DRUNet cases; scale s runs at (H >> s) x (W >> s), and the instantiations each reaches follow the
dispatch rules of conv_gemm_layer (PX = min(W_s, 128), ROWS = min(128 / PX, H_s)) and plan_items_pair:
  (2, 64, 64)    every plan layer.  Head: conv3x3_kernel<16, 64>; scale 0: conv3x3_ts2_kernel<64, 0 / 1 / 2> (one strip, padded
                 to two); scales 1-3: conv_gemm2_kernel<128 / 256, false> (PX 32 / 16 / 8); tail: conv3x3_ts_kernel<16, POST>.
  (1, 8, 8)      scale 3 is 1 x 1: PX = ROWS = 1, the one M tile paired with an empty padding tile (conv_gemm2_kernel<256, false>).
  (1, 40, 264)   scale 0: three 128-pixel strips, the last one 8 pixels wide, padded to four.  Scale 1 (20 x 132): PX = 128, ROWS = 1,
                 the row-box REUSE kernel with resident weights, conv_gemm2_kernel<128, true, *, true>, and a 4-pixel ragged tile.
                 Scale 2 (10 x 66): PX = 66, conv_gemm2_kernel<256, false>.  Scale 3 (5 x 33): PX = 33, ROWS = 3, the last tile
                 ragged in rows.
  (1, 16, 1024)  REUSE at N tile 256: scale 2 (256 channels, conv_gemm2_kernel<256, true>) and scale 3 (512 channels); scale 1
                 REUSE with resident weights over four tiles per row.
  (2, 320, 480)  the 64-channel residual layers (conv3x3_ts2_kernel<64, 1 / 2>) at the production image size.
"""
import math
import time

import pytest
import torch

import conv_reference as CR
import psgla_b200 as P

pytestmark = pytest.mark.gpu
L = P._lib
BF = torch.bfloat16


@pytest.fixture(scope="module", autouse=True)
def wall_time():
    t0 = time.perf_counter()
    yield
    print("\nOBSERVED tests/test_conv_layers_gpu.py wall time = %.1f s" % (time.perf_counter() - t0))


def _rand_bf16(g, *shape):
    return torch.randn(*shape, device="cuda", generator=g).to(BF)


def _nhwc(x):
    return x.permute(0, 2, 3, 1).contiguous()


def _bits(t):
    return t.view(torch.int16 if t.element_size() == 2 else torch.int32)


# ------------------------------------------------------------------------------------------------------------ DRUNet
@pytest.fixture(scope="module")
def drunet():
    sd = P.random_drunet_state_dict(11)
    return sd, P.DRUNet(pretrained=sd)


def drunet_spec(sd, l):
    """Layer l of the 64-entry plan, read off its state-dict key (independently of the library's own plan)."""
    key = P.DRUNET_KEYS[l]
    w = sd[key]
    spec = dict(key=key, w=w, relu=False, nres=0, head=key == "m_head.weight", tail=key == "m_tail.weight")
    if spec["head"] or spec["tail"]:
        spec.update(kind="conv3", cin=w.shape[1], cout=w.shape[0], scale=0)
    elif ".res." in key:
        second = ".res.2." in key
        last = key.startswith("m_body.3.") or (key.startswith("m_up") and ".4.res." in key)  # + the U-Net skip
        spec.update(kind="conv3", cin=w.shape[1], cout=w.shape[0], relu=not second, nres=(2 if last else 1) if second else 0)
    elif key.startswith("m_down"):
        spec.update(kind="down", cin=w.shape[1], cout=w.shape[0])
    else:
        spec.update(kind="up", cin=w.shape[0], cout=w.shape[1])  # ConvTranspose2d weight [Cin][Cout][2][2]
    if "scale" not in spec:
        spec["scale"] = int(math.log2(spec["cin"] // 64))
    return spec


def run_drunet_layer(den, shape, l, x, r1, r2, out_ptr):
    B, H, W = shape
    rc = L.lib().psgla_drunet_layer(den.packed.data_ptr(), L.ImgShape(B, 3, H, W), l, x.data_ptr(),
                                    None if r1 is None else r1.data_ptr(), None if r2 is None else r2.data_ptr(), out_ptr, None)
    L.check(rc, "psgla_drunet_layer(%d)" % l)


def drunet_layer_case(sd, den, shape, l, seed=0):
    """Runs plan layer l twice on random operands and checks it against the fp64 reference; returns the output."""
    sp = drunet_spec(sd, l)
    B, H, W = shape
    h, w = H >> sp["scale"], W >> sp["scale"]
    ho, wo = {"conv3": (h, w), "down": (h // 2, w // 2), "up": (2 * h, 2 * w)}[sp["kind"]]
    g = torch.Generator(device="cuda").manual_seed(1000 * l + seed)
    if sp["head"]:  # bf16 NHWC16: channels 0-2 the image, 3 the noise level, 4-15 zero
        x = torch.zeros(B, 16, h, w, device="cuda", dtype=BF)
        x[:, :4] = _rand_bf16(g, B, 4, h, w)
        x_ref = x[:, :4]
    else:
        x = x_ref = _rand_bf16(g, B, sp["cin"], h, w)
    res = [_rand_bf16(g, B, sp["cout"], ho, wo) for _ in range(sp["nres"])]
    ref, S = CR.reference(sp["kind"], x_ref, sp["w"], None, res, sp["relu"])
    out = CR.Guarded((B, 3, H, W) if sp["tail"] else (B, ho, wo, sp["cout"]), torch.float32 if sp["tail"] else BF)
    xn = _nhwc(x)
    rn = [_nhwc(r) for r in res] + [None, None]
    outs = []
    for _ in range(2):  # the second call walks the items in the other direction
        out.poison()
        run_drunet_layer(den, shape, l, xn, rn[0], rn[1], out.ptr())
        torch.cuda.synchronize()
        assert out.intact(), "layer %d wrote outside its output tensor" % l
        outs.append(out.tensor.clone())
    assert torch.equal(_bits(outs[0]), _bits(outs[1])), "layer %d: the two traversal directions disagree" % l
    got = outs[0] if sp["tail"] else outs[0].permute(0, 3, 1, 2)
    CR.check("drunet layer %d (%s) at %s" % (l, sp["key"], shape), got, ref, S)
    return outs[0]


@pytest.mark.parametrize("l", range(64))
def test_drunet_every_layer(drunet, l):
    """Every plan layer at (2, 64, 64): each tensor's packing and each kernel path the network takes."""
    drunet_layer_case(*drunet, (2, 64, 64), l)


@pytest.mark.parametrize("l", range(64))
@pytest.mark.parametrize("shape", [(1, 8, 8), (1, 40, 264), (1, 16, 1024)])
def test_drunet_layers_at_edge_shapes(drunet, shape, l):
    drunet_layer_case(*drunet, shape, l)


@pytest.mark.parametrize("l", [1, 2, 61, 62])
def test_drunet_residual_layers_production_size(drunet, l):
    """The 64-channel residual block convs (no residual / block input / block input + U-Net skip) at 2 x 320 x 480."""
    drunet_layer_case(*drunet, (2, 320, 480), l)


def test_drunet_layer_chain_equals_network(drunet):
    """The 64 layers chained through psgla_drunet_layer with KAIR's routing (residual blocks x + conv(relu(conv(x))), skips
    x4 / x3 / x2 / x1 added by the last conv of the body and of each decoder stage) == psgla_drunet_denoise_post with gain 1,
    base_scale 0 and a zero base, bit for bit: the per-layer tests cover what the network runs."""
    sd, den = drunet
    lib = L.lib()
    for shape in ((2, 64, 64), (1, 40, 264)):
        B, H, W = shape
        sh = L.ImgShape(B, 3, H, W)
        img = torch.rand(B, 3, H, W, device="cuda", generator=torch.Generator(device="cuda").manual_seed(4))
        den_in = torch.empty(B, H, W, 16, device="cuda", dtype=BF)
        L.check(lib.psgla_img_to_nhwc16(sh, img.data_ptr(), 5 / 255, den_in.data_ptr(), None), "to_nhwc16")

        def layer(l, x, r1=None, r2=None):
            sp = drunet_spec(sd, l)
            if sp["tail"]:
                out = torch.empty(B, 3, H, W, device="cuda")
            else:
                h, w = H >> sp["scale"], W >> sp["scale"]
                f = {"conv3": 1, "down": 0.5, "up": 2}[sp["kind"]]
                out = torch.empty(B, int(h * f), int(w * f), sp["cout"], device="cuda", dtype=BF)
            run_drunet_layer(den, shape, l, x, r1, r2, out.data_ptr())
            return out

        def blocks(l, cur, skip):
            for blk in range(4):
                t = layer(l, cur)
                cur = layer(l + 1, t, cur, skip if blk == 3 else None)
                l += 2
            return cur, l

        cur, l, skips = layer(0, den_in), 1, []
        for _ in range(3):  # encoder: x1, x2, x3 kept for the decoder
            skips.append(cur)
            cur, l = blocks(l, cur, None)
            cur, l = layer(l, cur), l + 1
        cur, l = blocks(l, cur, cur)  # body + x4
        for s in (2, 1, 0):
            cur, l = layer(l, cur), l + 1
            cur, l = blocks(l, cur, skips[s])
        assert l == 63
        chained = layer(63, cur)
        ws = torch.empty(lib.psgla_drunet_workspace_bytes(sh), dtype=torch.uint8, device="cuda")
        net = torch.full((B, 3, H, W), float("nan"), device="cuda")
        base = torch.zeros(B, 3, H, W, device="cuda")
        post = L.PostParams(1.0, 0.0, 0.0, 1.0)
        L.check(lib.psgla_drunet_denoise_post(den.packed.data_ptr(), sh, den_in.data_ptr(), ws.data_ptr(), ws.numel(), base.data_ptr(),
                                              post, net.data_ptr(), None, None, None, None), "denoise_post")
        torch.cuda.synchronize()
        assert torch.isfinite(chained).all() and chained.abs().max().item() > 1e-2
        assert torch.equal(chained, net), (shape, (chained - net).abs().max().item())


# ------------------------------------------------------------------------------------------------------------ DnCNN
def dncnn(depth, seed=3, scale=3.0):
    sd = P.random_dncnn_state_dict(seed, depth, scale=scale)
    return sd, P.DnCNN(depth=depth, pretrained=sd)


def dncnn_hidden_case(sd, den, shape, layer=1, seed=0):
    B, H, W = shape
    name = "conv_list.%d" % (layer - 1)
    w, bias = sd[name + ".weight"], sd[name + ".bias"]
    g = torch.Generator(device="cuda").manual_seed(seed)
    x = _rand_bf16(g, B, 64, H, W)
    ref, S = CR.reference("conv3", x, w, bias, relu=True)
    out = CR.Guarded((B, H, W, 64), BF)
    xn = _nhwc(x)
    outs = []
    for _ in range(2):
        out.poison()
        L.check(L.lib().psgla_conv3x3_layer(den.packed.data_ptr(), den.depth, layer, L.ImgShape(B, 3, H, W), xn.data_ptr(), out.ptr(),
                                            1, None), "conv3x3_layer")
        torch.cuda.synchronize()
        assert out.intact()
        outs.append(out.tensor.clone())
    assert torch.equal(_bits(outs[0]), _bits(outs[1]))
    CR.check("dncnn layer %d at %s" % (layer, shape), outs[0].permute(0, 3, 1, 2), ref, S)


@pytest.mark.parametrize("rows", [None, 1, 2, 4, 8, 16, 32])
def test_forced_item_plans(drunet, rows, monkeypatch):
    """PSGLA_CONV_ROWS (read per call) forces the pair kernel's R: block heights that do not divide the rows (40 and 45 rows),
    and at R = 1 on 64 x 64 images B = 1, 2, 3 chains give 64, 128 and 192 item pairs, i.e. fewer than the co-resident CTA
    pairs, between that count and its double, and more (PSGLA_VERBOSE=1 prints the count: 74 pairs on a 148-SM B200)."""
    if rows is None:
        monkeypatch.delenv("PSGLA_CONV_ROWS", raising=False)
    else:
        monkeypatch.setenv("PSGLA_CONV_ROWS", str(rows))
    sd_d, den_d = dncnn(20)
    drunet_layer_case(*drunet, (1, 40, 136), 2, seed=rows or 0)  # 64-channel residual layer (block input added)
    dncnn_hidden_case(sd_d, den_d, (1, 45, 136), seed=rows or 0)  # DnCNN hidden layer
    if rows == 1:
        for B in (1, 2, 3):
            drunet_layer_case(*drunet, (B, 64, 64), 62, seed=B)
            dncnn_hidden_case(sd_d, den_d, (B, 64, 64), seed=B)


@pytest.mark.parametrize("fuse2", ["0", "1"])
@pytest.mark.parametrize("shape", [(1, 96, 200), (6, 64, 64)])
@pytest.mark.parametrize("depth", [20, 5])
def test_dncnn_layer_chain_equals_network(depth, shape, fuse2, monkeypatch):
    """Layers 0 .. depth-1 through psgla_conv3x3_layer == psgla_dncnn_residual_post with gain 1 and a zero base, bit for bit --
    with the production buffer routing, the odd layers walking their items backwards and (PSGLA_CONV_FUSE2=1, few chains)
    hidden layers fused in pairs.  (1, 96, 200) takes the fused pairs, (6, 64, 64) has too many row blocks for one wave."""
    monkeypatch.setenv("PSGLA_CONV_FUSE2", fuse2)
    sd, den = dncnn(depth, seed=5, scale=2.0)
    lib = L.lib()
    B, H, W = shape
    sh = L.ImgShape(B, 3, H, W)
    img = torch.rand(B, 3, H, W, device="cuda", generator=torch.Generator(device="cuda").manual_seed(6))
    den_in = torch.empty(B, H, W, 16, device="cuda", dtype=BF)
    L.check(lib.psgla_img_to_nhwc16(sh, img.data_ptr(), 0.0, den_in.data_ptr(), None), "to_nhwc16")
    cur = den_in
    for layer in range(depth - 1):
        out = torch.empty(B, H, W, 64, device="cuda", dtype=BF)
        L.check(lib.psgla_conv3x3_layer(den.packed.data_ptr(), depth, layer, sh, cur.data_ptr(), out.data_ptr(), 1, None), "layer")
        cur = out
    chained = torch.empty(B, 3, H, W, device="cuda")
    L.check(lib.psgla_conv3x3_layer(den.packed.data_ptr(), depth, depth - 1, sh, cur.data_ptr(), chained.data_ptr(), 0, None), "last")
    ws = torch.empty(lib.psgla_dncnn_workspace_bytes(sh), dtype=torch.uint8, device="cuda")
    net = torch.full((B, 3, H, W), float("nan"), device="cuda")
    base = torch.zeros(B, 3, H, W, device="cuda")
    L.check(lib.psgla_dncnn_residual_post(depth, den.packed.data_ptr(), sh, den_in.data_ptr(), ws.data_ptr(), ws.numel(), base.data_ptr(),
                                          L.PostParams(1.0, 1.0, 0.0, 1.0), net.data_ptr(), None, None, None, None), "residual_post")
    torch.cuda.synchronize()
    assert torch.isfinite(chained).all() and chained.abs().max().item() > 1e-3
    assert torch.equal(chained, net), (chained - net).abs().max().item()


# ------------------------------------------------------------------------------------------------------------ post epilogue
def _check_post(name, r, base_term, gain, w_old, w_new, x_out, sample, m_in, m2_in, m_out, m2_out):
    """x_out within 1 fp32 ulp of fma(gain, r, base_term) (float64 has the product exactly; only the final rounding can differ
    from the kernel's single one), sample == x_out, and the moments bit-equal to the eager fp32 ops."""
    e = (torch.tensor(gain, dtype=torch.float32).double() * r.double() + base_term.double()).float()
    lo = torch.nextafter(e, torch.full_like(e, -float("inf")))
    hi = torch.nextafter(e, torch.full_like(e, float("inf")))
    assert bool(((x_out >= lo) & (x_out <= hi)).all()), "%s: x_out off fma(gain, r, base) by %.3g" % (
        name, (x_out - e).abs().max().item())
    assert torch.equal(_bits(sample), _bits(x_out)), name
    wo, wn = torch.tensor(w_old, dtype=torch.float32, device="cuda"), torch.tensor(w_new, dtype=torch.float32, device="cuda")
    assert torch.equal(_bits(m_out), _bits(wo * m_in + wn * x_out)), "%s: mean" % name
    assert torch.equal(_bits(m2_out), _bits(wo * m2_in + wn * (x_out * x_out))), "%s: mean2" % name


def _post_buffers(g, B, H, W):
    bufs = [CR.Guarded((B, 3, H, W), torch.float32) for _ in range(4)]  # x_out, sample, mean, mean2
    m_in = torch.rand(B, 3, H, W, device="cuda", generator=g)
    m2_in = torch.rand(B, 3, H, W, device="cuda", generator=g)
    bufs[2].tensor.copy_(m_in)
    bufs[3].tensor.copy_(m2_in)
    return bufs, m_in, m2_in


@pytest.mark.parametrize("shape", [(1, 256, 256), (3, 37, 150), (2, 1, 1)])
@pytest.mark.parametrize("depth", [20, 5])
def test_dncnn_post_epilogue_exact(depth, shape):
    """psgla_dncnn_last_layer_post_next (depth 20: the last layer walks its items backwards, depth 5: forwards) against the raw
    last-layer conv r of the same input: X+ = fma(gain, r, base), sample = X+, mean / mean2 = three rounded fp32 operations."""
    sd, den = dncnn(depth, seed=9, scale=2.0)
    lib = L.lib()
    B, H, W = shape
    sh = L.ImgShape(B, 3, H, W)
    g = torch.Generator(device="cuda").manual_seed(depth)
    hidden = _nhwc(_rand_bf16(g, B, 64, H, W).relu())
    r = CR.Guarded((B, 3, H, W), torch.float32)
    L.check(lib.psgla_conv3x3_layer(den.packed.data_ptr(), depth, depth - 1, sh, hidden.data_ptr(), r.ptr(), 0, None), "raw last layer")
    base = torch.randn(B, 3, H, W, device="cuda", generator=g)
    bufs, m_in, m2_in = _post_buffers(g, B, H, W)
    post = L.PostParams(0.8, 1.0, 0.75, 0.25)
    L.check(lib.psgla_dncnn_last_layer_post_next(depth, den.packed.data_ptr(), sh, hidden.data_ptr(), base.data_ptr(), post,
                                                 *[b.ptr() for b in bufs], None, None), "last_layer_post")
    torch.cuda.synchronize()
    assert r.intact() and all(b.intact() for b in bufs)
    _check_post("dncnn depth %d %s" % (depth, shape), r.tensor, base, 0.8, 0.75, 0.25, *[b.tensor for b in bufs[:2]], m_in, m2_in,
                bufs[2].tensor, bufs[3].tensor)


@pytest.mark.parametrize("shape", [(2, 64, 64), (3, 40, 136)])
def test_drunet_post_epilogue_exact(drunet, shape):
    """The DRUNet tail's post with (gain, base_scale) = (0.8, 0.2): X+ = fma(gain, r, fl(base_scale * base)), where r is the
    network output of the same input (gain 1, base_scale 0)."""
    _, den = drunet
    lib = L.lib()
    B, H, W = shape
    sh = L.ImgShape(B, 3, H, W)
    g = torch.Generator(device="cuda").manual_seed(B)
    img = torch.rand(B, 3, H, W, device="cuda", generator=g)
    den_in = torch.empty(B, H, W, 16, device="cuda", dtype=BF)
    L.check(lib.psgla_img_to_nhwc16(sh, img.data_ptr(), 0.02, den_in.data_ptr(), None), "to_nhwc16")
    ws = torch.empty(lib.psgla_drunet_workspace_bytes(sh), dtype=torch.uint8, device="cuda")
    r = CR.Guarded((B, 3, H, W), torch.float32)
    zero = torch.zeros(B, 3, H, W, device="cuda")
    L.check(lib.psgla_drunet_denoise_post(den.packed.data_ptr(), sh, den_in.data_ptr(), ws.data_ptr(), ws.numel(), zero.data_ptr(),
                                          L.PostParams(1.0, 0.0, 0.0, 1.0), r.ptr(), None, None, None, None), "raw")
    base = torch.randn(B, 3, H, W, device="cuda", generator=g)
    bufs, m_in, m2_in = _post_buffers(g, B, H, W)
    L.check(lib.psgla_drunet_denoise_post(den.packed.data_ptr(), sh, den_in.data_ptr(), ws.data_ptr(), ws.numel(), base.data_ptr(),
                                          L.PostParams(0.8, 0.2, 0.75, 0.25), *[b.ptr() for b in bufs], None), "post")
    torch.cuda.synchronize()
    assert r.intact() and all(b.intact() for b in bufs)
    base_term = torch.tensor(0.2, dtype=torch.float32, device="cuda") * base
    _check_post("drunet %s" % (shape,), r.tensor, base_term, 0.8, 0.75, 0.25, *[b.tensor for b in bufs[:2]], m_in, m2_in,
                bufs[2].tensor, bufs[3].tensor)


# ------------------------------------------------------------------------------------------------------------ layout helpers
@pytest.mark.parametrize("shape", [(2, 37, 50), (1, 1, 1), (3, 8, 130)])
def test_img_to_nhwc16_exact(shape):
    B, H, W = shape
    x = torch.randn(B, 3, H, W, device="cuda", generator=torch.Generator(device="cuda").manual_seed(H)) * 3
    c3 = 0.0173
    out = CR.Guarded((B, H, W, 16), BF)
    L.check(L.lib().psgla_img_to_nhwc16(L.ImgShape(B, 3, H, W), x.data_ptr(), c3, out.ptr(), None), "to_nhwc16")
    torch.cuda.synchronize()
    want = torch.zeros(B, H, W, 16, device="cuda", dtype=BF)
    want[..., :3] = x.permute(0, 2, 3, 1).to(BF)
    want[..., 3] = torch.tensor(c3, dtype=torch.float32).to(BF).item()
    assert out.intact()
    assert torch.equal(_bits(out.tensor), _bits(want))


@pytest.mark.parametrize("padded,H,W", [((2, 40, 56), 37, 50), ((1, 8, 8), 1, 1), ((3, 16, 136), 16, 130), ((1, 24, 8), 21, 8)])
def test_img_pad_replicate_exact(padded, H, W):
    """In-place replication padding of an NHWC16 batch (sizes that are not multiples of 8) == F.pad(mode="replicate")."""
    B, Hp, Wp = padded
    img = CR.Guarded((B, Hp, Wp, 16), BF)  # pad region NaN
    valid = _rand_bf16(torch.Generator(device="cuda").manual_seed(W), B, H, W, 16)
    img.tensor[:, :H, :W] = valid
    L.check(L.lib().psgla_img_pad_replicate_nhwc16(L.ImgShape(B, 3, Hp, Wp), H, W, img.ptr(), None), "pad_replicate")
    torch.cuda.synchronize()
    want = torch.nn.functional.pad(valid.permute(0, 3, 1, 2).float(), (0, Wp - W, 0, Hp - H), mode="replicate")
    assert img.intact()
    assert torch.equal(_bits(img.tensor), _bits(want.to(BF).permute(0, 2, 3, 1).contiguous()))
