"""not-gpu: the C-ABI library builds, loads, and exports exactly the symbols include/psgla_b200.h declares."""
import ctypes
import os
import re

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def built():
    import __graft_entry__ as g
    g.build()
    import psgla_b200
    return psgla_b200


def _header_functions():
    src = open(os.path.join(ROOT, "include", "psgla_b200.h")).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    return sorted(set(re.findall(r"\b(psgla_[a-z0-9_]+)\s*\(", src)))


def test_header_and_binding_agree(built):
    fns = _header_functions()
    assert len(fns) >= 17
    assert sorted(built._lib.SIGNATURES) == fns


def test_library_exports_every_symbol(built):
    handle = ctypes.CDLL(built._lib.LIB_PATH)
    for fn in _header_functions():
        assert hasattr(handle, fn), fn
    assert handle.psgla_abi_version() == 5


def test_struct_sizes_match_header(built):
    L = built._lib
    assert ctypes.sizeof(L.GmmProblem) == 8 + 4 * 8 + 4 * 8 + 2 * 8 + 16 * (2 + 4 + 1) * 8
    assert ctypes.sizeof(L.ImgShape) == 16
    assert ctypes.sizeof(L.PreParams) == 72
    assert ctypes.sizeof(L.PostParams) == 16
    assert ctypes.sizeof(L.NextPre) == 48
    for which, struct in enumerate((L.GmmProblem, L.ImgShape, L.PreParams, L.PostParams, L.NextPre)):  # as compiled into the .so
        assert L.lib().psgla_struct_size(which) == ctypes.sizeof(struct)


def test_argument_errors_without_gpu(built):
    lib = built._lib.lib()
    # null problem pointer: rejected on the host before any CUDA call
    rc = lib.psgla_gmm2d_run(None, 0, None, 1, 0, 1, 0, 0, None, None, 1, None)
    assert rc == -1 and b"null" in lib.psgla_last_error()
    assert lib.psgla_dncnn_packed_bytes(20) == 1024 * (19 + 18 * 73 + 19)
    assert lib.psgla_dncnn_packed_bytes(1) == 0


def test_no_cpu_fallback(built):
    import numpy as np
    import torch
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    D = built.Theorical_MMSE(*built.gaussian_mixt_example("cross"))
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        built.SnoPnP_ULA(10, np.zeros(2), np.zeros(2), 0.3, np.eye(2), 1, D, 2 / 3)
    with pytest.raises(TypeError, match="structured callable"):
        built.SnoPnP_ULA(10, np.zeros(2), np.zeros(2), 0.3, np.eye(2), 1, lambda x, e: x, 2 / 3)
    with pytest.raises(RuntimeError):
        built.DnCNN()


def test_product_does_not_import_oracle():
    pkg = os.path.join(ROOT, "psgla-for-posterior-sampling_b200")
    for f in os.listdir(pkg):
        if f.endswith(".py"):
            src = open(os.path.join(pkg, f)).read()
            assert "oracle" not in src.replace("# oracle", ""), f


def test_environment_selects_no_kernel_but_the_documented_switches():
    """The problem alone selects each kernel: the library reads PSGLA_CONV_FUSE2 (per-layer launches, which the bench times
    beside the fused pairs), PSGLA_CONV_ROWS (a test hook) and PSGLA_VERBOSE (diagnostics), and the package reads none."""
    names = set()
    csrc = os.path.join(ROOT, "psgla-for-posterior-sampling_b200", "csrc")
    for f in os.listdir(csrc):
        names.update(re.findall(r'getenv\(\s*"(PSGLA_\w*)"', open(os.path.join(csrc, f)).read()))
    pkg = os.path.join(ROOT, "psgla-for-posterior-sampling_b200")
    for f in os.listdir(pkg):
        if f.endswith(".py"):
            names.update(re.findall(r'os\.(?:environ\b[^"\'\n]*|getenv\(\s*)["\'](PSGLA_\w*)["\']', open(os.path.join(pkg, f)).read()))
    assert names == {"PSGLA_CONV_FUSE2", "PSGLA_CONV_ROWS", "PSGLA_VERBOSE"}


def test_philox_known_answers(built):
    """Random123's kat_vectors for philox4x32-10: the RNG the kernels inline is the published Philox."""
    import ctypes as C
    lib = built._lib.lib()
    kat = [
        ((0, 0, 0, 0), (0, 0), (0x6627e8d5, 0xe169c58d, 0xbc57ac4c, 0x9b00dbd8)),
        ((0xffffffff,) * 4, (0xffffffff, 0xffffffff), (0x408f276d, 0x41c83b0e, 0xa20bc7c6, 0x6d5451fd)),
        ((0x243f6a88, 0x85a308d3, 0x13198a2e, 0x03707344), (0xa4093822, 0x299f31d0), (0xd16cfe09, 0x94fdcceb, 0x5001e420, 0x24126ea1)),
    ]
    for ctr, key, want in kat:
        out = (C.c_uint32 * 4)()
        lib.psgla_philox4x32_10((C.c_uint32 * 4)(*ctr), (C.c_uint32 * 2)(*key), out)
        assert tuple(out) == want


def test_next_pre_argument_errors_without_gpu(built):
    """psgla_*_post_next validates the fused next-iteration pre descriptor on the host, before any CUDA call."""
    L = built._lib
    lib = L.lib()
    shape = L.ImgShape(1, 3, 8, 8)
    post = L.PostParams(1.0, 1.0, 0.0, 1.0)
    pre = L.PreParams()
    pre.alg = 7  # not a PSGLA_ALG_* value
    fake = 0x1000  # never dereferenced: the descriptor is rejected first
    bad_alg = L.NextPre(ctypes.pointer(pre), fake, fake, 1, 1, fake, fake)
    rc = lib.psgla_dncnn_residual_post_next(20, fake, shape, fake, fake, 1 << 30, fake, ctypes.byref(post), fake, None, None, None,
                                            ctypes.byref(bad_alg), None)
    assert rc == -1 and b"alg=7" in lib.psgla_last_error()
    pre.alg = 0
    null_mask = L.NextPre(ctypes.pointer(pre), None, fake, 1, 1, fake, fake)
    rc = lib.psgla_drunet_denoise_post_next(fake, shape, fake, fake, 1 << 30, fake, ctypes.byref(post), fake, None, None, None,
                                            ctypes.byref(null_mask), None)
    assert rc == -1 and b"psgla_next_pre" in lib.psgla_last_error()
    bad_b = L.NextPre(ctypes.pointer(pre), fake, fake, 2, 1, fake, fake)  # mask_B must be 1 or B
    rc = lib.psgla_dncnn_residual_post_next(20, fake, shape, fake, fake, 1 << 30, fake, ctypes.byref(post), fake, None, None, None,
                                            ctypes.byref(bad_b), None)
    assert rc == -1 and b"mask_B" in lib.psgla_last_error()


def test_drunet_layer_argument_errors_without_gpu(built):
    """psgla_drunet_layer rejects, on the host before any CUDA call, a layer index out of range, null pointers, a shape the network
    rejects, and every residual pattern the network would not pass for that layer: res1 (the block input) exactly on the second
    conv of each residual block, res2 (the U-Net skip) exactly on the last such conv of the body and of each decoder stage."""
    L = built._lib
    lib = L.lib()
    shape = L.ImgShape(1, 3, 16, 16)
    fake = 0x1000  # never dereferenced: every call below is rejected first
    for layer in (-1, 64, 1 << 20):
        assert lib.psgla_drunet_layer(fake, shape, layer, fake, None, None, fake, None) == -1
        assert b"layer" in lib.psgla_last_error()
    assert lib.psgla_drunet_layer(None, shape, 0, fake, None, None, fake, None) == -1 and b"null" in lib.psgla_last_error()
    assert lib.psgla_drunet_layer(fake, shape, 0, fake, None, None, None, None) == -1 and b"null" in lib.psgla_last_error()
    for bad in (L.ImgShape(1, 3, 12, 16), L.ImgShape(1, 3, 16, 20), L.ImgShape(0, 3, 16, 16), L.ImgShape(1, 4, 16, 16)):
        assert lib.psgla_drunet_layer(fake, bad, 1, fake, None, None, fake, None) == -1
    keys = built.DRUNET_KEYS
    assert len(keys) == lib.psgla_drunet_num_weights() == 64
    n_roles = {0: 0, 1: 0, 2: 0}
    for layer, key in enumerate(keys):
        want = 0
        if ".res.2." in key:
            want = 2 if key.startswith("m_body.3.") or (key.startswith("m_up") and ".4.res." in key) else 1
        n_roles[want] += 1
        for r1, r2 in ((None, None), (fake, None), (fake, fake), (None, fake)):
            if (r1 is not None) + (r2 is not None) == want and (r2 is None or r1 is not None):
                continue  # what the network passes: not called here (it would launch)
            assert lib.psgla_drunet_layer(fake, shape, layer, fake, r1, r2, fake, None) == -1, (layer, key, r1, r2)
            assert b"residual" in lib.psgla_last_error(), key
    assert n_roles == {0: 64 - 28, 1: 24, 2: 4}


def _sass(obj):
    import shutil
    import subprocess
    cuobjdump = shutil.which("cuobjdump") or "/usr/local/cuda/bin/cuobjdump"
    if not os.path.exists(cuobjdump):
        pytest.skip("cuobjdump not available")
    return subprocess.run([cuobjdump, "-sass", obj], capture_output=True, text=True, check=True).stdout


def test_sass_is_blackwell_native(built):
    """What the build produced, read back from the objects (no GPU needed): the conv kernels issue tcgen05 MMAs (UTCHMMA, the
    CTA-pair ones .2CTA), move tiles by TMA (UTMALDG / UTMASTG) and read accumulators from tensor memory (LDTM); nothing falls
    back to the legacy warp-level mma.sync (HMMA); and the weight-resident conv kernels read their bias vector with shared-space
    loads -- as generic LD.E loads behind every chunk's staging store they cost the hidden layers 13 % (DESIGN.md section 4)."""
    build_dir = os.path.join(os.path.dirname(built._lib.LIB_PATH), "build")
    conv_tc = _sass(os.path.join(build_dir, "conv_tc.o"))
    conv_gemm = _sass(os.path.join(build_dir, "conv_gemm.o"))
    fused2 = _sass(os.path.join(build_dir, "conv_fused2.o"))
    for name, text in (("conv_tc", conv_tc), ("conv_gemm", conv_gemm), ("conv_fused2", fused2)):
        assert text.count("UTCHMMA") > 0, name
        assert text.count("UTCHMMA.2CTA") > 0, name
        assert text.count("UTMALDG") > 0, name
        assert text.count("LDTM") > 0, name
        assert len(re.findall(r"\bHMMA\b", text)) == 0, name
    assert conv_tc.count("UTMASTG") > 0 and conv_tc.count("STTM") > 0
    # per kernel of conv_tc.o: generic 128-bit loads (the old bias path) only where a residual / bias pointer may be global
    for fn, body in re.findall(r"Function : (\S+)\n(.*?)(?=\n\s*Function : |\Z)", conv_tc, flags=re.S):
        if "conv3x3_ts2_kernelILi64ELi0E" in fn or "conv3x3_ts2_kernelILi64ELi1E" in fn:
            assert body.count("LD.E.128") == 0, fn
    gmm = _sass(os.path.join(build_dir, "gmm2d.o"))
    assert gmm.count("FFMA2") > 0 and gmm.count("MUFU") > 0
