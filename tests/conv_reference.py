"""fp64 reference of one convolution layer and the element-wise acceptance criterion of the conv-layer tests.

The reference takes exactly the operands the kernel sees: the bf16 input / residual tensors themselves and the weights
rounded fp32 -> bf16 to nearest-even as the packers round them.  It sums in float64, so its own error (~1e-16 relative) is
negligible, and it also returns S = sum |w| |x| + |bias| + sum |res|, the scale of the fp32 accumulation error.

Criterion, per element:
  bf16 output  |got - ref| <= 2^-8 |ref| + TAU * S    (one bf16 rounding of the output + fp32 accumulation)
  fp32 output  |got - ref| <= 2^-23 |ref| + TAU * S
and for bf16 outputs the fraction of elements with got != bf16_rn(ref) stays below MISMATCH_MAX (a wrong rounding mode or a
systematic bias moves half of them).  A bound on max |got - ref| relative to max |ref| cannot see a dropped bias of 1e-2 next
to outputs of 10; this one can, because it is tight where the outputs are small.

TAU is 4 x the largest value measured over the 307 cases of tests/test_conv_layers_gpu.py, test_drunet_gpu.py and
test_image_gpu.py (2.9e-7, a 512-channel 3 x 3 layer; on one B200 at its 1000 W power limit), and it must stay at most
2^-10 = 2 K 2^-24 for the largest K here (9 x 512 = 4 608 terms), a bound that even a truncating fp32 accumulation meets.
MISMATCH_MAX is 4 x the largest measured mismatch fraction (1.2e-3, a 256-channel layer; same device).  check() prints each
case's figures (pytest -s).
"""
import torch
import torch.nn.functional as F

from conftest import observed

BF16_U = 2.0 ** -8
FP32_U = 2.0 ** -23
TAU_MAX = 2.0 ** -10
TAU = 1.2e-6
MISMATCH_MAX = 5e-3
assert TAU <= TAU_MAX

GUARD_BYTES = 1024
SENTINEL = 0xA5


def bf16_weights(w):
    """fp32 -> bf16, round to nearest even (what psgla_dncnn_pack_weights / psgla_drunet_pack_weights store)."""
    return w.float().to(torch.bfloat16)


def reference(kind, x, w, bias=None, res=(), relu=False):
    """kind: "conv3" (3x3, zero pad 1), "down" (2x2 stride 2) or "up" (2x2 stride-2 transposed, w in ConvTranspose2d layout).
    x, res: bf16 NCHW on the device; w: fp32 or bf16 (rounded here as the packers round it); bias: fp32 or None.
    Returns (ref, S) in float64 NCHW."""
    x64 = x.double()
    w64 = bf16_weights(w).to(x.device).double()
    b64 = None if bias is None else bias.to(x.device).double()
    if kind == "conv3":
        op = lambda a, k, b: F.conv2d(a, k, b, padding=1)  # noqa: E731
    elif kind == "down":
        op = lambda a, k, b: F.conv2d(a, k, b, stride=2)  # noqa: E731
    elif kind == "up":
        op = lambda a, k, b: F.conv_transpose2d(a, k, b, stride=2)  # noqa: E731
    else:
        raise ValueError(kind)
    ref = op(x64, w64, b64)
    S = op(x64.abs(), w64.abs(), None if b64 is None else b64.abs())
    for r in res:
        ref = ref + r.double()
        S = S + r.double().abs()
    if relu:
        ref = ref.relu()
    return ref, S


def tau_of(got, ref, S, rel):
    """Smallest tau with |got - ref| <= rel |ref| + tau S everywhere (inf where S = 0 and got != ref)."""
    excess = ((got.double() - ref).abs() - rel * ref.abs()).clamp_min(0)
    t = torch.where(S > 0, excess / S.clamp_min(1e-300), torch.where(excess > 0, float("inf"), 0.0))
    return t.max().item()


def check(name, got, ref, S):
    """got: the kernel's output as NCHW, bf16 or fp32.  Asserts the criterion above; returns (tau, mismatch fraction)."""
    assert got.shape == ref.shape, (got.shape, ref.shape)
    assert torch.isfinite(got).all(), "%s: non-finite output" % name
    if got.dtype == torch.bfloat16:
        tau = tau_of(got, ref, S, BF16_U)
        want = ref.float().to(torch.bfloat16)  # fp64 -> fp32 -> bf16: double rounding only at exact fp32 ties
        mism = (got.view(torch.int16) != want.view(torch.int16)).double().mean().item()
        observed("tau %s" % name, tau, TAU * (1 + 1e-9))
        observed("bf16 mismatch %s" % name, mism, MISMATCH_MAX)
        return tau, mism
    assert got.dtype == torch.float32
    tau = tau_of(got, ref, S, FP32_U)
    observed("tau %s" % name, tau, TAU * (1 + 1e-9))
    return tau, 0.0


class Guarded:
    """An output tensor inside a larger allocation: GUARD_BYTES of sentinel bytes on either side, the tensor itself starting
    on a 1 KB boundary and filled with NaN before every call.  intact() says whether the guards are bit-unchanged."""

    def __init__(self, shape, dtype, device="cuda"):
        self.shape, self.dtype = tuple(shape), dtype
        n = 1
        for s in shape:
            n *= s
        self.nbytes = n * torch.empty(0, dtype=dtype).element_size()
        self.raw = torch.empty(3 * GUARD_BYTES + self.nbytes, dtype=torch.uint8, device=device)
        self.off = 2 * GUARD_BYTES - self.raw.data_ptr() % GUARD_BYTES  # front guard of 1..2 KB, tensor 1 KB aligned
        self.end = self.off + self.nbytes
        self.tensor = self.raw[self.off:self.end].view(dtype).view(self.shape)
        self.poison()

    def poison(self):
        self.raw.fill_(SENTINEL)
        self.tensor.fill_(float("nan"))
        return self.tensor

    def intact(self):
        return bool((self.raw[:self.off] == SENTINEL).all().item() and (self.raw[self.end:] == SENTINEL).all().item())

    def ptr(self):
        return self.tensor.data_ptr()
