"""not-gpu: grayscale (one-channel) support on the host -- the seeded state dicts' channel keyword, the C ABI accepting C = 1 and
rejecting other channel counts before any CUDA call, and the colour-only entries (TV prox, gradient-step DRUNet) staying so."""
import ctypes

import pytest
import torch


@pytest.fixture(scope="module")
def built():
    import __graft_entry__ as g
    g.build()
    import psgla_b200
    return psgla_b200


def test_seeded_state_dicts_take_a_channel_count(built):
    D = built.denoisers
    for fn in (D.random_dncnn_state_dict, D.smoothing_dncnn_state_dict):
        c3, c1, dflt = fn(channels=3), fn(channels=1), fn()
        assert all(torch.equal(dflt[k], c3[k]) for k in dflt) and set(dflt) == set(c3) == set(c1)
        assert tuple(c1["in_conv.weight"].shape) == (64, 1, 3, 3) and tuple(c1["out_conv.weight"].shape) == (1, 64, 3, 3)
        assert tuple(c1["out_conv.bias"].shape) == (1,)
    c1 = D.lipschitz_dncnn_state_dict(0, depth=4, channels=1)
    assert tuple(c1["in_conv.weight"].shape) == (64, 1, 3, 3)
    d3, d1 = D.random_drunet_state_dict(0), D.random_drunet_state_dict(0, channels=1)
    assert all(torch.equal(d3[k], D.random_drunet_state_dict(0, channels=3)[k]) for k in d3)
    assert tuple(d1["m_head.weight"].shape) == (64, 2, 3, 3) and tuple(d1["m_tail.weight"].shape) == (1, 64, 3, 3)
    assert all(tuple(d1[k].shape) == tuple(d3[k].shape) for k in d3 if k not in ("m_head.weight", "m_tail.weight"))
    # the grayscale smoothing network carries the one channel on features 0, 3, 6, 9
    s1 = D.smoothing_dncnn_state_dict(channels=1)
    assert s1["in_conv.weight"][[0, 3, 6, 9], 0, 1, 1].tolist() == [1.0, -1.0, 1.0, -1.0]


def test_abi_channel_counts(built):
    """C = 2 and C = 4 are rejected by every image entry that takes C = 1, and packer channel counts other than 1 and 3 are
    rejected; C = 1 passes the shape checks (each call below then stops at a null pointer, still before any CUDA call); the TV
    prox and the gradient-step DRUNet reject C = 1."""
    L = built._lib
    lib = L.lib()
    fake = 0x1000  # never dereferenced
    pre = L.PreParams()
    post = L.PostParams(1.0, 1.0, 0.0, 1.0)
    taps = (ctypes.c_float * 9)(*([1 / 9] * 9))
    FP = ctypes.POINTER(ctypes.c_float)

    def calls(s, null=False):
        p = None if null else fake
        return {
            "pre_inpaint": lambda: lib.psgla_img_pre_inpaint(ctypes.byref(pre), s, p, fake, 1, fake, 1, None, fake, fake, None),
            "pre_deblur": lambda: lib.psgla_img_pre_deblur(ctypes.byref(pre), s, p, taps, 4, fake, 1, None, fake, fake, None),
            "pre_deblur_ata": lambda: lib.psgla_img_pre_deblur_ata(ctypes.byref(pre), s, p, taps, 4, fake, 1, None, fake, fake, None),
            "blur": lambda: lib.psgla_img_blur(s, p, taps, 4, fake, None),
            "noise": lambda: lib.psgla_img_noise(s, 0, 0, -1, fake, None),  # iteration -1: rejected after the shape check
            "to_nhwc16": lambda: lib.psgla_img_to_nhwc16(s, p, 0.0, fake, None),
            "conv3x3_layer": lambda: lib.psgla_conv3x3_layer(fake, 20, 0 if not null else -1, s, fake, fake, 1, None),
            "dncnn": lambda: lib.psgla_dncnn_residual_post_next(20, fake, s, p, fake, 1 << 40, fake, ctypes.byref(post), fake,
                                                                None, None, None, None, None),
            "drunet": lambda: lib.psgla_drunet_denoise_post_next(fake, s, p, fake, 1 << 40, fake, ctypes.byref(post), fake, None,
                                                                 None, None, None, None),
            "drunet_layer": lambda: lib.psgla_drunet_layer(fake, s, 0, p, None, None, fake, None),
        }

    for C in (2, 4, 0):
        for name, f in calls(L.ImgShape(1, C, 16, 16)).items():
            assert f() == -1, name
            assert b"[C = 1 or 3]" in lib.psgla_last_error(), (name, lib.psgla_last_error())
    for name, f in calls(L.ImgShape(1, 1, 16, 16), null=True).items():
        assert f() == -1, name
        assert b"C = 1 or 3" not in lib.psgla_last_error(), (name, lib.psgla_last_error())
    assert lib.psgla_tv_state_bytes(L.ImgShape(1, 1, 16, 16)) == 0 and lib.psgla_tv_workspace_bytes(L.ImgShape(1, 1, 16, 16)) == 0
    assert lib.psgla_gsdrunet_denoise_post_next(fake, L.ImgShape(1, 1, 16, 16), fake, None, fake, 1 << 40, fake, 1.0,
                                                ctypes.byref(post), fake, None, None, None, None, None) == -1
    assert b"[B>0][3][H>0][W>0]" in lib.psgla_last_error()
    ws = (FP * 64)(*([ctypes.cast(fake, FP)] * 64))
    for ch in (0, 2, 4, -1):
        assert lib.psgla_dncnn_pack_weights_ch(20, ch, ws, None, fake, None) == -1
        assert b"channels must be 3 or 1" in lib.psgla_last_error()
        assert lib.psgla_drunet_pack_weights_ch(ch, ws, fake, None) == -1
        assert b"channels must be 3 or 1" in lib.psgla_last_error()
    assert lib.psgla_dncnn_packed_bytes(20) > 0


def test_shape_helper_and_load_image(built, tmp_path):
    from psgla_b200 import operators
    s = operators._shape_of(torch.zeros(2, 1, 5, 7))
    assert (s.B, s.C, s.H, s.W) == (2, 1, 5, 7)
    for bad in ((2, 2, 5, 7), (2, 4, 5, 7), (1, 5, 7)):
        with pytest.raises(ValueError):
            operators._shape_of(torch.zeros(*bad))
    cv2 = pytest.importorskip("cv2")
    import numpy as np
    img = (np.arange(6 * 10 * 3).reshape(6, 10, 3) % 251).astype(np.uint8)
    path = str(tmp_path / "im.png")
    cv2.imwrite(path, img)
    g = built.load_image(path, n_channels=1)
    assert g.shape == (1, 1, 6, 10) and g.dtype == torch.float32
    assert torch.equal(g[0, 0], torch.from_numpy(np.float32(cv2.imread(path, 0) / 255.0)))
    assert built.load_image(path).shape == (1, 3, 6, 10)
    with pytest.raises(ValueError):
        built.load_image(path, n_channels=2)
