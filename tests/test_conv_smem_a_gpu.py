"""3x3 convolutions over pre-split inputs (the shared-memory A kernel of fod_conv2d_nhwc) against the same layer fed fp32.

A pre-split input holds, per pixel and 16 channels, [16 x fp16 hi | 16 x fp16 lo] of x * 2^e with 2^e the scale the
kernel derives from x_amax.  Those are exactly the halves the kernel forms itself from fp32 x, and the MMAs run in the
same order, so the outputs must be bit-identical: torch.equal, no tolerance."""
import pytest
import torch

from faster_orefsdet_b200 import ops
from tests.util import amax_per_image, presplit

pytestmark = pytest.mark.gpu
DEV = "cuda"
MAGS = [1e-3, 30.0, 0.7]   # per-image magnitudes: every image gets its own scale


def _layer(n, h, w, cin, cout, seed):
    g = torch.Generator().manual_seed(seed)
    x = torch.randn(n, cin, h, w, generator=g)
    x *= torch.tensor(MAGS[:n]).view(n, 1, 1, 1)
    wt = torch.randn(cout, cin, 3, 3, generator=g) / (9 * cin) ** 0.5
    b = torch.randn(cout, generator=g) * 0.1
    x = x.to(DEV).contiguous(memory_format=torch.channels_last)
    return x, ops.conv2d_pack(wt.to(DEV)), b.to(DEV)


def _in_wide_buffer(x, lead, trail):
    """x as a channel slice of a wider NHWC buffer whose other channels hold NaN"""
    n, c, h, w = x.shape
    buf = torch.full((n, h, w, lead + c + trail), float("nan"), device=x.device)
    buf[..., lead:lead + c] = x.permute(0, 2, 3, 1)
    return buf.permute(0, 3, 1, 2)[:, lead:lead + c]


@pytest.mark.parametrize("n,h,w,cin,cout", [
    (2, 20, 20, 64, 64),     # stem_2 (partial tiles)
    (3, 37, 53, 64, 64),     # OSA2 64 -> 64, neither side a tile multiple
    (2, 37, 53, 128, 64),    # OSA2 128 -> 64
    (3, 80, 80, 112, 80),    # OSA3 112 -> 80: the last chunk half outside Cin; 75 tile pairs leave a last-wave tail
    (2, 20, 24, 80, 80),     # OSA3 80 -> 80 (27 chunks in parts of 14)
    (2, 20, 20, 256, 96),    # OSA4 256 -> 96
    (3, 8, 16, 96, 96),      # OSA4 96 -> 96, one tile per image: an odd tile count
    (2, 20, 20, 64, 32),     # a single 32-column slab: epilogue warps without columns
    (2, 20, 20, 384, 112),   # OSA5 384 -> 112 does not fit the shared-memory A stages: the tensor-memory path
])
def test_presplit_3x3_is_bit_identical_to_fp32_input(n, h, w, cin, cout):
    x, pk, b = _layer(n, h, w, cin, cout, 1000 + cin + cout)
    amax = amax_per_image(x)
    ya_ref, ya = ops.new_amax(DEV, n), ops.new_amax(DEV, n)
    ref = ops.conv2d_nhwc(x, pk, b, cout, 3, True, x_amax=amax, y_amax=ya_ref)
    xp = _in_wide_buffer(presplit(x, amax), 16, 48)
    y = ops.conv2d_nhwc(xp, pk, b, cout, 3, True, x_amax=amax, y_amax=ya, x_presplit=True)
    assert torch.equal(y, ref)
    assert torch.equal(ya, ya_ref)
    assert torch.isfinite(y).all()


def test_presplit_3x3_split_output_is_bit_identical():
    n, h, w, cin, cout = 3, 37, 53, 64, 64
    x, pk, b = _layer(n, h, w, cin, cout, 7)
    amax = amax_per_image(x)
    outs = []
    for xin, pre in ((x, False), (presplit(x, amax), True)):
        y = torch.empty((n, h, w, cout), device=DEV).permute(0, 3, 1, 2)
        yb, ya = torch.empty((n,), device=DEV), ops.new_amax(DEV, n)
        ops.conv2d_nhwc_split(xin, pk, b, cout, 3, y, amax, y_amax=ya, x_presplit=pre, y_bound=yb, y_l1=2.5, y_beta=0.1)
        outs.append((y.contiguous().view(torch.int32), yb, ya))
    for a, r in zip(outs[1], outs[0]):
        assert torch.equal(a, r)


@pytest.mark.parametrize("n,h,w,cout", [(2, 37, 53, 128), (3, 40, 40, 128), (2, 20, 20, 256)])
def test_presplit_stride2_is_bit_identical_to_fp32_input(n, h, w, cout):
    """stem_3: stride 2 over an input pre-split at a single bound"""
    cin = 64
    x, pk, b = _layer(n, h, w, cin, cout, 300 + h + cout)
    amax = amax_per_image(x)
    ho, wo = (h - 1) // 2 + 1, (w - 1) // 2 + 1
    outs = []
    for xin, pre in ((x, -1), (_in_wide_buffer(presplit(x, amax), 32, 16), 0)):
        y = torch.empty((n, ho, wo, cout), device=DEV).permute(0, 3, 1, 2)
        ya = ops.new_amax(DEV, n)
        ops.conv2d_nhwc_split(xin, pk, b, cout, 3, y, amax, y_amax=ya, x_presplit_from=pre,
                              slice_ch=[0] if pre == 0 else None, stride=2)
        outs.append((y, ya))
    assert torch.equal(outs[1][0], outs[0][0])
    assert torch.equal(outs[1][1], outs[0][1])
