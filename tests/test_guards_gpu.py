"""Memory-safety checks of every C-ABI kernel without compute-sanitizer (it is closed on this GPU pool, see
profiles/r2_sanitizer.md): every device buffer the operator wrappers allocate is placed between two guard bands of a
known byte pattern, and what `torch.empty` would leave uninitialised is pre-filled with a pattern.

  * out-of-bounds WRITES of a kernel show up as a damaged guard band (memcheck's job);
  * READS of memory the kernel was never given valid data for (rows beyond a count, padding of a tile) show up as
    outputs that change with the fill pattern - each case runs once with 0xA5 bytes and once with 0xFF bytes (NaN as
    fp32, -1 as integers) and the valid parts of the results must be bit-identical (initcheck's job);
  * races between the warp roles of the tensor-core kernels would show up as run-to-run differences: each case is also
    repeated and compared bit for bit (a weak stand-in for racecheck; the hand-off protocols themselves are exercised at
    many shapes by the parity tests).
"""
import math

import pytest
import torch

from faster_orefsdet_b200 import fold, ops, synth
from tests.util import head_state_dict

pytestmark = pytest.mark.gpu
DEV = "cuda"
GUARD = 4096          # elements on each side (a multiple of 16 bytes for every dtype)


class GuardedTorch:
    """Stand-in for the ``torch`` module inside faster_orefsdet_b200.ops: empty / zeros allocate between guard bands."""

    def __init__(self, fill_byte):
        self.fill_byte = fill_byte
        self.allocs = []

    def __getattr__(self, name):
        return getattr(torch, name)

    def _alloc(self, shape, dtype, device, zero, pin_memory=False):
        if isinstance(shape, int):
            shape = (shape,)
        if device is None or torch.device(device).type != "cuda" or pin_memory:
            return (torch.zeros if zero else torch.empty)(shape, dtype=dtype, device=device, pin_memory=pin_memory)
        n = int(math.prod(shape))
        buf = torch.empty(n + 2 * GUARD, dtype=dtype, device=device)
        buf.view(torch.uint8).fill_(0x5C)
        mid = buf[GUARD:GUARD + n]
        if zero:
            mid.zero_()
        else:
            mid.view(torch.uint8).fill_(self.fill_byte)
        self.allocs.append((buf, n))
        return mid.view(shape)

    def empty(self, *shape, dtype=None, device=None, pin_memory=False):
        shape = shape[0] if len(shape) == 1 and not isinstance(shape[0], int) else shape
        return self._alloc(tuple(shape), dtype or torch.float32, device, False, pin_memory)

    def zeros(self, *shape, dtype=None, device=None, pin_memory=False):
        shape = shape[0] if len(shape) == 1 and not isinstance(shape[0], int) else shape
        return self._alloc(tuple(shape), dtype or torch.float32, device, True, pin_memory)

    def check(self):
        torch.cuda.synchronize()
        for buf, n in self.allocs:
            b = buf.view(torch.uint8)
            es = buf.element_size()
            assert bool((b[:GUARD * es] == 0x5C).all()), "guard band BEFORE a buffer was overwritten"
            assert bool((b[(GUARD + n) * es:] == 0x5C).all()), "guard band AFTER a buffer was overwritten"


def run_guarded(monkeypatch, fn, valid):
    """fn() -> outputs; valid(outputs) -> list of tensors that must not depend on uninitialised memory."""
    results = []
    for fill in (0xA5, 0xFF, 0xA5):
        g = GuardedTorch(fill)
        monkeypatch.setattr(ops, "torch", g)
        out = fn()
        g.check()
        results.append([t.contiguous().reshape(-1).clone() for t in valid(out)])
        monkeypatch.undo()
    for other in results[1:]:
        for a, b in zip(results[0], other):
            assert a.shape == b.shape and torch.equal(a.view(torch.uint8), b.view(torch.uint8)), "result depends on uninitialised memory or differs between runs"


def _boxes(n, seed, lo=20.0, hi=300.0, wmin=8.0, wmax=90.0):
    ctr = synth.tensor((n, 2), seed, lo, hi)
    wh = synth.tensor((n, 2), seed + 1, wmin, wmax)
    return torch.cat((ctr - wh / 2, ctr + wh / 2), 1)


def test_decode_and_nms_stay_inside_their_buffers(monkeypatch):
    sizes, strides, P = [(40, 48), (20, 24), (10, 12)], (8, 16, 32), 3
    hm = [synth.tensor((P, 1, h, w), 21 + l, -9.0, 3.0).to(DEV) for l, (h, w) in enumerate(sizes)]
    reg = [synth.tensor((P, 4, h, w), 31 + l, 0.0, 9.0).to(DEV) for l, (h, w) in enumerate(sizes)]
    status = torch.zeros(1, dtype=torch.int32, device=DEV)

    def fn():
        boxes, scores, loc, lc, cc = ops.decode_topk(hm, reg, strides, 1e-5, 1000, status)
        keep, pb, ps, pc = ops.nms_proposals(boxes, scores, cc, 0.6, 256, 320, status)
        return boxes, scores, loc, lc, cc, keep, pb, ps, pc

    def valid(o):
        boxes, scores, loc, lc, cc, keep, pb, ps, pc = o
        out = [lc, cc, pc]
        for p in range(P):
            n, m = int(cc[p]), int(pc[p])
            out += [boxes[p, :n], scores[p, :n], loc[p, :n], keep[p, :m], pb[p, :m], ps[p, :m]]
        return out

    run_guarded(monkeypatch, fn, valid)
    assert int(status.item()) == 0


@pytest.mark.parametrize("n", [1, 65, 700, 5000])
def test_batched_nms_stays_inside_its_buffers(monkeypatch, n):
    boxes, scores = _boxes(n, 11 + n).to(DEV), synth.tensor((n,), 13 + n, 0.0, 1.0).to(DEV)
    idxs = (synth.tensor((n,), 14, 0.0, 1.0) * 3).long().to(DEV)
    run_guarded(monkeypatch, lambda: ops.batched_nms(boxes, scores, idxs, 0.6), lambda k: [k])


def test_roi_relation_final_stay_inside_their_buffers(monkeypatch):
    sd = head_state_dict()
    feats = synth.features(2, 128, 160, 33)
    fl = [feats[k].to(DEV).contiguous(memory_format=torch.channels_last) for k in ("p3", "p4", "p5")]
    C, cap = 2, 130                                    # two units per problem, the second one ragged
    P = 2 * C
    bx = _boxes(P * cap, 90, 10.0, 120.0, 4.0, 200.0).reshape(P, cap, 4).to(DEV)
    counts = torch.tensor([130, 3, 0, 129], dtype=torch.int32, device=DEV)
    sup = synth.tensor((C, 128, 8, 8), 73, -1.0, 1.0)
    w_fold, w_out, b_out = fold.fold_relation_weights(sd)
    bias = fold.fold_class_bias(sd, sup).to(DEV)
    w_fold, w_out, b_out = ops.relation_pack(w_fold.to(DEV)), w_out.to(DEV), b_out.to(DEV)
    xa = torch.cat([ops.absmax(f) for f in fl])
    hw = torch.tensor([[128, 160]] * 2, dtype=torch.int32, device=DEV)
    status = torch.zeros(1, dtype=torch.int32, device=DEV)

    def fn():
        dense = ops.roi_align(fl, (8, 16, 32), bx, counts, C, 8)
        small = ops.roi_align(fl, (8, 16, 32), bx, counts, C, 4)
        tiled = ops.roi_align(fl, (8, 16, 32), bx, counts, C, 8, tiled=True)
        db, ds, lg, dl = ops.relation_head(tiled, w_fold, bias, w_out, b_out, bx, counts, C, (10.0, 10.0, 5.0, 5.0),
                                           want_raw=True, x_amax=xa)
        fin = ops.final_detect(db, ds, counts, C, 0.0, 0.9, 100, hw, None, status)
        return dense, small, tiled, db, ds, lg, dl, fin

    def valid(o):
        dense, small, tiled, db, ds, lg, dl, (ob, os_, ocls, orow, oc) = o
        out = [oc]
        back = ops.untile_pooled(tiled, cap)
        for p in range(P):
            n = int(counts[p])
            out += [dense[p, :n], small[p, :n], back[p, :n], db[p, :n], ds[p, :n], lg[p, :n], dl[p, :n]]
        for b in range(2):
            m = int(oc[b])
            out += [ob[b, :m], os_[b, :m], ocls[b, :m], orow[b, :m]]
        return out

    run_guarded(monkeypatch, fn, valid)
    assert int(status.item()) == 0


def test_roi_align_14_wide_stays_inside_its_buffers(monkeypatch):
    """Resolution 14 over 1024-channel stride-16 maps (the ROI pooling of the FsodRCNN path), ragged counts, boxes of
    every kind including sampling grids beyond the tap tables."""
    from tests.test_ops_gpu import roi14_case
    f, bx, counts = roi14_case(1024, 13, 17, 2, 950)
    fd, bd, cd = f.to(DEV), bx.to(DEV), counts.to(DEV)

    def valid(pooled):
        return [pooled[p, :int(counts[p])] for p in range(bx.shape[0])]

    run_guarded(monkeypatch, lambda: ops.roi_align([fd], [16], bd, cd, 2, 14), valid)


@pytest.mark.parametrize("sizes,B,C",[(((25, 42), (13, 21), (7, 11)), 2, 3), (((8, 16),), 1, 1), (((1, 1), (5, 3)), 1, 7)])
def test_correlate_levels_stays_inside_its_buffers(monkeypatch, sizes, B, C):
    sd = head_state_dict()
    qs = [synth.tensor((B, 128, h, w), 150 + h + 3 * i, -1.5, 1.5).to(DEV) for i, (h, w) in enumerate(sizes)]
    taps = [ops.support_taps(synth.tensor((C, 128, 5, 6), 160 + i, -0.6, 0.8).to(DEV)).cpu() for i in range(len(sizes))]
    w3, b3 = sd["conv3.weight"].to(DEV), sd["conv3.bias"].to(DEV)
    run_guarded(monkeypatch, lambda: ops.correlate_levels(qs, taps, w3, b3, want_amax=True),
                lambda o: list(o[0]) + list(o[1]))


@pytest.mark.parametrize("shape", [(2, 64, 19, 23, 64, 3, 1), (1, 128, 9, 40, 8, 3, 1), (3, 32, 17, 18, 96, 1, 1), (2, 64, 21, 22, 128, 3, 2)])
def test_conv_and_group_norm_stay_inside_their_buffers(monkeypatch, shape):
    n, cin, h, w, cout, k, stride = shape
    x = synth.tensor((n, cin, h, w), 700 + cin, -2.0, 2.0).to(DEV).contiguous(memory_format=torch.channels_last)
    wt = synth.tensor((cout, cin, k, k), 701 + cout, -0.2, 0.2).to(DEV)
    bias = synth.tensor((cout,), 702, -0.1, 0.1).to(DEV)
    gamma, beta = synth.tensor((cout,), 703, 0.8, 1.2).to(DEV), synth.tensor((cout,), 704, -0.1, 0.1).to(DEV)

    def fn():
        pk = ops.conv2d_pack(wt)
        am = ops.new_amax(DEV)
        y = ops.conv2d_nhwc(x, pk, bias, cout, k, relu=True, stride=stride, y_amax=am)
        out = [y, am]
        if cout % 32 == 0:
            out.append(ops.group_norm_nhwc(y, 32 if cout % 128 == 0 else 8, gamma, beta, 1e-5, relu=True))
        return out

    run_guarded(monkeypatch, fn, lambda o: o)


@pytest.mark.parametrize("hw", [(37, 51), (320, 416)])
def test_stem_kernels_stay_inside_their_buffers(monkeypatch, hw):
    """stem_1 from uint8 images, FMA and tensor-core kernel: odd sizes (the last tile row / column is clipped by the TMA
    store) and more tiles than SMs; the two runs of each pattern double as a run-to-run check of the tensor-core hand-offs."""
    h, w_ = hw
    n = 3
    x = synth.tensor((n, 3, h, w_), 810, 0.0, 255.99).to(torch.uint8).to(DEV)
    mean, std = [103.53, 116.28, 123.675], [1.0, 1.0, 1.0]
    w = synth.tensor((64, 3, 3, 3), 811, -0.3, 0.3).to(DEV)
    b = synth.tensor((64,), 812, -1.0, 1.0).to(DEV)
    w32 = torch.cat((w.permute(0, 2, 3, 1).reshape(64, 27), torch.zeros(64, 5, device=DEV)), 1).reshape(64, 32, 1, 1).contiguous()

    def fn():
        pk = ops.conv2d_pack(w32)
        a1, a2 = ops.new_amax(DEV, n), ops.new_amax(DEV, n)
        return [ops.stem1_u8_tc(x, mean, std, pk, b, y_amax=a1), a1, ops.stem1_u8(x, mean, std, w, b, y_amax=a2), a2]

    run_guarded(monkeypatch, fn, lambda o: o)
