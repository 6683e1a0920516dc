"""ctypes binding of libpsgla_b200.so (the C ABI declared in include/psgla_b200.h).

There is deliberately no fallback: if the shared library is missing or a call fails, a
``RuntimeError`` is raised -- the product never computes on the CPU.
"""
from __future__ import annotations

import ctypes as C
import os
import threading

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libpsgla_b200.so")

GMM_MAX_COMPONENTS = 16
ALG_PSGLA, ALG_PNPULA = 0, 1
NOISE_PHILOX, NOISE_TORCH_CUDA = 0, 1


class GmmProblem(C.Structure):
    """psgla_gmm2d_problem"""
    _fields_ = [
        ("alg", C.c_int32), ("n_components", C.c_int32),
        ("delta", C.c_double), ("alpha", C.c_double), ("epsilon", C.c_double), ("sigma", C.c_double),
        ("A", C.c_double * 4), ("y", C.c_double * 2),
        ("mu", (C.c_double * 2) * GMM_MAX_COMPONENTS),
        ("Sigma", (C.c_double * 4) * GMM_MAX_COMPONENTS),
        ("pi", C.c_double * GMM_MAX_COMPONENTS),
    ]


class ImgShape(C.Structure):
    """psgla_img_shape"""
    _fields_ = [("B", C.c_int32), ("C", C.c_int32), ("H", C.c_int32), ("W", C.c_int32)]


class PreParams(C.Structure):
    """psgla_pre_params"""
    _fields_ = [("alg", C.c_int32), ("gain_data", C.c_float), ("noise_scale", C.c_float), ("proj_gain", C.c_float),
                ("c_min", C.c_float), ("c_max", C.c_float), ("x_gain", C.c_float), ("den_in_c3", C.c_float),
                ("seed", C.c_uint64), ("chain_id0", C.c_int64),
                ("iteration", C.c_int64), ("noise_mode", C.c_int32), ("torch_threads", C.c_uint32),
                ("torch_offset", C.c_uint64)]


class PostParams(C.Structure):
    """psgla_post_params"""
    _fields_ = [("gain", C.c_float), ("base_scale", C.c_float), ("w_old", C.c_float), ("w_new", C.c_float)]


class NextPre(C.Structure):
    """psgla_next_pre"""
    _fields_ = [("pre", C.POINTER(PreParams)), ("mask_dev", C.c_void_p), ("y_dev", C.c_void_p), ("mask_B", C.c_int32),
                ("y_B", C.c_int32), ("base_dev", C.c_void_p), ("den_in_dev", C.c_void_p)]


class TVParams(C.Structure):
    """psgla_tv_params"""
    _fields_ = [("ths", C.c_float), ("tau", C.c_float), ("rho", C.c_float), ("crit", C.c_float), ("n_it_max", C.c_int32),
                ("restart", C.c_int32)]


_vp, _i64, _u64, _int, _sz = C.c_void_p, C.c_int64, C.c_uint64, C.c_int, C.c_size_t

# name -> (restype, argtypes); every symbol include/psgla_b200.h declares
SIGNATURES = {
    "psgla_last_error": (C.c_char_p, []),
    "psgla_abi_version": (_int, []),
    "psgla_device_arch": (_int, []),
    "psgla_struct_size": (_int, [_int]),
    "psgla_philox4x32_10": (None, [C.POINTER(C.c_uint32), C.POINTER(C.c_uint32), C.POINTER(C.c_uint32)]),
    "psgla_gmm2d_run": (_int, [C.POINTER(GmmProblem), _int, _vp, _i64, _i64, _i64, _i64, _u64, _vp, _vp, _i64, _vp]),
    "psgla_gmm2d_last_launches": (_int, []),
    "psgla_gmm2d_denoise": (_int, [C.POINTER(GmmProblem), C.c_double, _int, _vp, _vp, _i64, _vp]),
    "psgla_gmm2d_noise": (_int, [_vp, _i64, _i64, _i64, _i64, _u64, _vp]),
    "psgla_gmm2d_sw2_workspace_bytes": (_sz, [_i64, _int]),
    "psgla_gmm2d_sorted_projections": (_int, [_vp, _int, _i64, C.POINTER(C.c_float), _int, _vp, _vp, _sz, _vp]),
    "psgla_gmm2d_sliced_w2": (_int, [_vp, _int, _i64, C.POINTER(C.c_float), _int, _vp, _vp, _sz, _vp, _vp]),
    "psgla_img_pre_inpaint": (_int, [C.POINTER(PreParams), ImgShape, _vp, _vp, _int, _vp, _int, _vp, _vp, _vp, _vp]),
    "psgla_img_pre_deblur": (_int, [C.POINTER(PreParams), ImgShape, _vp, C.POINTER(C.c_float), _int, _vp, _int, _vp,
                                    _vp, _vp, _vp]),
    "psgla_img_pre_deblur_ata": (_int, [C.POINTER(PreParams), ImgShape, _vp, C.POINTER(C.c_float), _int, _vp, _int, _vp,
                                        _vp, _vp, _vp]),
    "psgla_img_blur": (_int, [ImgShape, _vp, C.POINTER(C.c_float), _int, _vp, _vp]),
    "psgla_img_noise": (_int, [ImgShape, _u64, _i64, _i64, _vp, _vp]),
    "psgla_torch_cuda_randn_policy": (_int, [_i64, _int, _int, C.POINTER(C.c_uint32), C.POINTER(C.c_uint64)]),
    "psgla_img_noise_torch_cuda": (_int, [_i64, _u64, _u64, C.c_uint32, _vp, _vp]),
    "psgla_dncnn_packed_bytes": (_sz, [_int]),
    "psgla_dncnn_pack_weights": (_int, [_int, C.POINTER(C.POINTER(C.c_float)), C.POINTER(C.POINTER(C.c_float)), _vp, _vp]),
    "psgla_dncnn_pack_weights_ch": (_int, [_int, _int, C.POINTER(C.POINTER(C.c_float)), C.POINTER(C.POINTER(C.c_float)), _vp,
                                           _vp]),
    "psgla_dncnn_workspace_bytes": (_sz, [ImgShape]),
    "psgla_dncnn_residual_post": (_int, [_int, _vp, ImgShape, _vp, _vp, _sz, _vp, C.POINTER(PostParams), _vp, _vp, _vp,
                                         _vp, _vp]),
    "psgla_dncnn_residual_post_next": (_int, [_int, _vp, ImgShape, _vp, _vp, _sz, _vp, C.POINTER(PostParams), _vp, _vp, _vp,
                                              _vp, C.POINTER(NextPre), _vp]),
    "psgla_dncnn_last_layer_post_next": (_int, [_int, _vp, ImgShape, _vp, _vp, C.POINTER(PostParams), _vp, _vp, _vp, _vp,
                                                C.POINTER(NextPre), _vp]),
    "psgla_conv3x3_layer": (_int, [_vp, _int, _int, ImgShape, _vp, _vp, _int, _vp]),
    "psgla_img_pad_replicate_nhwc16": (_int, [ImgShape, _int, _int, _vp, _vp]),
    "psgla_img_to_nhwc16": (_int, [ImgShape, _vp, C.c_float, _vp, _vp]),
    "psgla_img_metrics_workspace_bytes": (_sz, [_int]),
    "psgla_img_psnr_ssim": (_int, [ImgShape, _vp, _vp, C.c_float, _vp, _sz, _vp, _vp, _vp]),
    "psgla_drunet_num_weights": (_int, []),
    "psgla_drunet_packed_bytes": (_sz, []),
    "psgla_drunet_pack_weights": (_int, [C.POINTER(C.POINTER(C.c_float)), _vp, _vp]),
    "psgla_drunet_pack_weights_ch": (_int, [_int, C.POINTER(C.POINTER(C.c_float)), _vp, _vp]),
    "psgla_drunet_workspace_bytes": (_sz, [ImgShape]),
    "psgla_drunet_denoise_post": (_int, [_vp, ImgShape, _vp, _vp, _sz, _vp, C.POINTER(PostParams), _vp, _vp, _vp, _vp, _vp]),
    "psgla_drunet_denoise_post_next": (_int, [_vp, ImgShape, _vp, _vp, _sz, _vp, C.POINTER(PostParams), _vp, _vp, _vp, _vp,
                                              C.POINTER(NextPre), _vp]),
    "psgla_drunet_layer": (_int, [_vp, ImgShape, _int, _vp, _vp, _vp, _vp, _vp]),
    "psgla_gsdrunet_num_weights": (_int, []),
    "psgla_gsdrunet_packed_bytes": (_sz, []),
    "psgla_gsdrunet_pack_weights": (_int, [C.POINTER(C.POINTER(C.c_float)), _vp, _vp]),
    "psgla_gsdrunet_workspace_bytes": (_sz, [ImgShape]),
    "psgla_gsdrunet_denoise_post_next": (_int, [_vp, ImgShape, _vp, _vp, _vp, _sz, _vp, C.c_float, C.POINTER(PostParams), _vp,
                                                _vp, _vp, _vp, C.POINTER(NextPre), _vp]),
    "psgla_gsdrunet_layer": (_int, [_vp, ImgShape, _int, _int, _vp, _vp, _vp, _vp, _vp, _vp]),
    "psgla_tv_state_bytes": (_sz, [ImgShape]),
    "psgla_tv_workspace_bytes": (_sz, [ImgShape]),
    "psgla_tv_prox_post": (_int, [C.POINTER(TVParams), ImgShape, _vp, _vp, _sz, _vp, _sz, C.POINTER(PostParams), _vp, _vp, _vp,
                                  _vp, _vp, _vp]),
    "psgla_mcmc_diag_workspace_bytes": (_sz, [_i64, _i64]),
    "psgla_mcmc_diag": (_int, [_vp, _i64, _i64, _i64, _vp, _sz, _vp, _vp, _vp, _vp]),
    "psgla_mcmc_diag_large_workspace_bytes": (_sz, [_i64, _i64, _i64]),
    "psgla_mcmc_diag_large": (_int, [_vp, _i64, _i64, _i64, _vp, _sz, _vp, _vp, _vp, _vp]),
    "psgla_mcmc_summary_workspace_bytes": (_sz, [_i64, _i64, _i64, _int]),
    "psgla_mcmc_summary": (_int, [_vp, _i64, _i64, _i64, C.POINTER(C.c_double), _int, C.c_double, _vp, _sz, _vp, _vp, _vp,
                                  _vp, _vp, _vp, _vp, _vp, _vp, _vp]),
    "psgla_selftest_umma": (_int, [_vp, _vp, _vp, _int, _int, _vp]),
    "psgla_selftest_umma2": (_int, [_vp, _vp, _vp, _int, _vp]),
    "psgla_convg_layer": (_int, [_int, _int, _int, _int, _int, _int, _vp, _vp, _vp, _vp, _vp, _int, _vp]),
    "psgla_selftest_mma_rate": (_int, [_int, _int, _int, _int, _vp, _vp]),
    "psgla_selftest_mma_rate2": (_int, [_int, _int, _int, _int, _vp, _vp]),
    "psgla_selftest_fp32_rate": (_int, [_int, _int, _int, _vp, C.POINTER(C.c_double), _vp]),
    "psgla_selftest_pipe_rate": (_int, [_int, _int, _int, _vp, C.POINTER(C.c_double), _vp]),
}

_lock = threading.Lock()
_lib = None


def lib() -> C.CDLL:
    """The loaded library; raises (never falls back) when it is absent."""
    global _lib
    if _lib is None:
        with _lock:
            if _lib is None:
                if not os.path.exists(LIB_PATH):
                    raise RuntimeError(
                        "libpsgla_b200.so is not built (%s). Run `python -c 'import __graft_entry__ as g; g.build()'` "
                        "or `python psgla-for-posterior-sampling_b200/build.py`. There is no CPU fallback." % LIB_PATH)
                handle = C.CDLL(LIB_PATH)
                for name, (res, args) in SIGNATURES.items():
                    fn = getattr(handle, name)  # AttributeError if the header and the library disagree
                    fn.restype = res
                    fn.argtypes = args
                for which, struct in enumerate((GmmProblem, ImgShape, PreParams, PostParams, NextPre, TVParams)):
                    if handle.psgla_struct_size(which) != C.sizeof(struct):
                        raise RuntimeError("ctypes layout of %s (%d bytes) disagrees with libpsgla_b200.so (%d bytes): "
                                           "rebuild the library" % (struct.__name__, C.sizeof(struct), handle.psgla_struct_size(which)))
                _lib = handle
    return _lib


def check(code: int, what: str) -> None:
    if code != 0:
        msg = lib().psgla_last_error()
        raise RuntimeError("%s failed with code %d: %s" % (what, code, msg.decode() if msg else "?"))


def require_cuda():
    import torch
    if not torch.cuda.is_available():
        raise RuntimeError("psgla_b200 needs a CUDA device (sm_100a); there is no CPU fallback")
    return torch


def stream_ptr(device=None) -> int:
    import torch
    return torch.cuda.current_stream(device).cuda_stream


def ptr(t) -> int:
    """Device pointer of a contiguous CUDA tensor (or None)."""
    if t is None:
        return None
    if not t.is_cuda or not t.is_contiguous():
        raise ValueError("expected a contiguous CUDA tensor")
    return t.data_ptr()
