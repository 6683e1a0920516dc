"""not-gpu: the gradient-step DRUNet restatement (tests/gs_reference.py) is the tested DRUNet architecture with ELU and two
blocks per stage, its gradient is the gradient of g, checkpoints load, and the C ABI and the Python class reject bad arguments
before any CUDA call."""
import ctypes

import pytest
import torch
import torch.nn.functional as F

import gs_reference as GS
from oracle import image_oracle as io_


@pytest.fixture(scope="module")
def built():
    import __graft_entry__ as g
    g.build()
    import psgla_b200
    return psgla_b200


def _small_sd(seed=0):
    from psgla_b200.denoisers import random_gsdrunet_state_dict
    return {k: v.double() for k, v in random_gsdrunet_state_dict(seed).items()}


def test_restatement_is_the_drunet_architecture(built):
    """With ReLU and nb = 4 the restatement is oracle.image_oracle.DRUNet bit for bit in fp64."""
    sd = io_.make_drunet_weights(seed=0)
    net = io_.DRUNet().double()
    net.load_state_dict({k: v.double() for k, v in sd.items()})
    x = torch.rand(2, 3, 16, 24, dtype=torch.float64, generator=torch.Generator().manual_seed(1))
    with torch.no_grad():
        want = net(x, 0.05)
    got = GS.network({k: v.double() for k, v in sd.items()}, x, 0.05, nb=4, act=F.relu)
    assert torch.equal(got, want)
    assert set(sd) == set(built.denoisers._drunet_keys(4))


def test_grad_g_is_the_gradient_of_g():
    sd = _small_sd()
    x = torch.rand(1, 3, 8, 8, dtype=torch.float64, generator=torch.Generator().manual_seed(2), requires_grad=True)

    def g_of(z):
        return 0.5 * ((z - GS.network(sd, z, 0.1)) ** 2).sum()

    g_auto = torch.autograd.grad(g_of(x), x)[0]
    assert torch.allclose(GS.grad_g(sd, x, 0.1)[0], g_auto, rtol=1e-12, atol=1e-14)  # v - J^T v
    assert torch.autograd.gradcheck(g_of, (x,), eps=1e-6, atol=1e-6)  # autograd's gradient against finite differences


def test_state_dict_loading(built):
    from psgla_b200.denoisers import GSDRUNET_KEYS, gsdrunet_weights, random_gsdrunet_state_dict
    sd = random_gsdrunet_state_dict(3)
    assert list(sd) == GSDRUNET_KEYS and len(GSDRUNET_KEYS) == 36
    ws = gsdrunet_weights(sd)
    wrapped = {"state_dict": {"student_grad.model." + k: v for k, v in sd.items()}}
    for a, b in zip(ws, gsdrunet_weights(wrapped)):
        assert torch.equal(a, b)
    with pytest.raises(KeyError):
        gsdrunet_weights({k: v for k, v in sd.items() if k != "m_tail.weight"})
    bad = dict(sd)
    bad["m_body.0.res.0.weight"] = torch.zeros(512, 512, 2, 2)
    with pytest.raises(ValueError):
        gsdrunet_weights(bad)


@pytest.mark.parametrize("kw", [dict(nb=4), dict(nc=[32, 64, 128, 256]), dict(act_mode="R"), dict(in_channels=1),
                                dict(out_channels=1), dict(alpha=float("nan")), dict(alpha=float("inf"))])
def test_gsdrunet_constructor_rejects(built, kw):
    with pytest.raises(ValueError):
        built.GSDRUNet(**kw)


def test_gsdrunet_abi_sizes(built):
    L = built._lib
    lib = L.lib()
    assert lib.psgla_gsdrunet_num_weights() == 36
    assert lib.psgla_gsdrunet_packed_bytes() > 2 * lib.psgla_drunet_packed_bytes() // 2
    s = L.ImgShape(2, 3, 64, 32)
    px = 2 * 64 * 32
    assert 1800 * px < lib.psgla_gsdrunet_workspace_bytes(s) < 2200 * px
    for bad in (L.ImgShape(0, 3, 8, 8), L.ImgShape(1, 3, 0, 8), L.ImgShape(1, 3, 8, -8)):
        assert lib.psgla_gsdrunet_workspace_bytes(bad) == 0


def test_gsdrunet_argument_errors_without_gpu(built):
    """psgla_gsdrunet_denoise_post_next / _layer / _pack_weights reject each bad argument on the host before any CUDA call (the
    fake pointers are never dereferenced)."""
    L = built._lib
    lib = L.lib()
    fake = 0x1000
    shape = L.ImgShape(1, 3, 16, 16)
    ws = lib.psgla_gsdrunet_workspace_bytes(shape)
    post = L.PostParams(1.0, 0.0, 0.0, 1.0)

    def call(shape=shape, packed=fake, den=fake, x=None, ws_ptr=fake, ws=ws, base=fake, alpha=1.0, post=post, out=fake,
             mean=None, mean2=None, nxt=None):
        return lib.psgla_gsdrunet_denoise_post_next(packed, shape, den, x, ws_ptr, ws, base, alpha,
                                                    ctypes.byref(post) if post is not None else None, out, None, mean, mean2,
                                                    nxt, None)

    for kw in (dict(packed=None), dict(den=None), dict(ws_ptr=None), dict(base=None), dict(post=None), dict(out=None),
               dict(mean=fake), dict(mean2=fake)):
        assert call(**kw) == -1, kw
    for a in (float("nan"), float("inf"), -float("inf")):
        assert call(alpha=a) == -1 and b"alpha" in lib.psgla_last_error()
    for bad in (L.ImgShape(0, 3, 16, 16), L.ImgShape(1, 1, 16, 16), L.ImgShape(1, 3, 0, 16), L.ImgShape(1, 3, 16, -8)):
        assert call(shape=bad) == -1 and b"shape" in lib.psgla_last_error()
    for bad in (L.ImgShape(1, 3, 12, 16), L.ImgShape(1, 3, 16, 20), L.ImgShape(1, 3, 481, 320)):
        assert call(shape=bad) == -1 and b"multiples of 8" in lib.psgla_last_error()
    assert call(ws=ws - 1) == -4 and b"workspace" in lib.psgla_last_error()
    nxt = L.NextPre(None, fake, fake, 1, 1, fake, fake)
    assert call(nxt=ctypes.byref(nxt)) == -1

    def layer(backward=0, idx=1, packed=fake, shape=shape, inp=fake, r1=None, r2=None, gate=None, out=fake):
        return lib.psgla_gsdrunet_layer(packed, shape, backward, idx, inp, r1, r2, gate, out, None)

    for kw in (dict(backward=2), dict(backward=-1), dict(idx=-1), dict(idx=36), dict(packed=None), dict(inp=None),
               dict(out=None), dict(shape=L.ImgShape(1, 3, 12, 16))):
        assert layer(**kw) == -1, kw
    # forward 1: first conv of a block (ELU, no inputs); forward 2: second conv (res1); forward 19: last body conv (res1 + res2)
    assert layer(idx=1, r1=fake) == -1 and layer(idx=1, gate=fake) == -1
    assert layer(idx=2) == -1 and layer(idx=2, r1=fake, r2=fake) == -1
    assert layer(idx=19, r1=fake) == -1
    # backward 1: adjoint of forward 34 (a second conv: gate only); backward 2: adjoint of 33 (a first conv: res1)
    assert layer(backward=1, idx=1) == -1 and layer(backward=1, idx=1, gate=fake, r1=fake) == -1
    assert layer(backward=1, idx=2) == -1 and layer(backward=1, idx=2, r1=fake, gate=fake) == -1
    # backward 34: adjoint of forward 1, the first conv of encoder 0: res1 and the held skip gradient
    assert layer(backward=1, idx=34, r1=fake) == -1
    assert lib.psgla_gsdrunet_pack_weights(None, fake, None) == -1
    arr = (ctypes.POINTER(ctypes.c_float) * 36)()
    assert lib.psgla_gsdrunet_pack_weights(arr, fake, None) == -1 and b"null" in lib.psgla_last_error()
