"""Shared helpers for the tests: golden fixtures, synthetic weights, comparisons."""
import os

import numpy as np
import torch

from faster_orefsdet_b200 import ops, synth

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def golden(name):
    return np.load(os.path.join(GOLDEN, name + ".npz"))


def head_param_shapes():
    shapes = {}
    with open(os.path.join(GOLDEN, "head_param_shapes.txt")) as f:
        for line in f:
            parts = line.split()
            shapes[parts[0]] = tuple(int(x) for x in parts[1:])
    return shapes


def head_state_dict():
    """The synthetic head weights the golden vectors were produced with."""
    return synth.state_dict(head_param_shapes())


def t(x):
    return torch.from_numpy(np.ascontiguousarray(x))


def assert_close(a, b, rtol=1e-4, atol=1e-5, what=""):
    a = a.detach().cpu().double() if torch.is_tensor(a) else torch.as_tensor(a).double()
    b = b.detach().cpu().double() if torch.is_tensor(b) else torch.as_tensor(b).double()
    assert a.shape == b.shape, f"{what}: shape {tuple(a.shape)} vs {tuple(b.shape)}"
    if a.numel() == 0:
        return
    err = (a - b).abs()
    tol = atol + rtol * b.abs()
    bad = err > tol
    assert not bad.any(), (f"{what}: {int(bad.sum())}/{a.numel()} elements off; max abs err "
                           f"{float(err.max()):.3e}, max rel {float((err / (b.abs() + 1e-12)).max()):.3e}")


def amax_per_image(x):
    """max |x| of every image of an fp32 [N,C,H,W] map, as the [1, N] per-image bound layout of ops.conv2d_nhwc"""
    return ops.absmax(x.contiguous(memory_format=torch.channels_last), per_image=True).reshape(1, -1)


def presplit(x, amax):
    """fp32 NHWC view [N,C,H,W] -> the split operand format at the scale of amax ([1, N]), as an fp32 NHWC view."""
    n, c, h, w = x.shape
    _, ex = torch.frexp(amax.reshape(-1))                                  # amax = m * 2^ex, m in [0.5, 1)
    scale = ((141 - ex.to(torch.int32)) << 23).view(torch.float32)      # 2^(14 - ex): max|x| * 2^e in [2^13, 2^14)
    xs = x.permute(0, 2, 3, 1) * scale.view(n, 1, 1, 1)
    hi = xs.half()
    lo = (xs - hi.float()).half()
    packed = torch.cat([hi.reshape(n, h, w, c // 16, 16), lo.reshape(n, h, w, c // 16, 16)], dim=-1)
    return packed.contiguous().view(torch.float32).reshape(n, h, w, c).permute(0, 3, 1, 2)
