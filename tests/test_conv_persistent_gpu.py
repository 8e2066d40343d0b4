"""The persistent tensor-core convolution (fod_conv2d_nhwc) against float64 where every CTA pair works through several
work units.

The kernels run min(pair_units, SMs / 2) CTA pairs; pair k takes the pair-units k, k + pairs, k + 2 pairs, ..., one
pair-unit being (two adjacent tiles of 8 x 16 output pixels, one group of <= 128 output channels).  From one unit to the
next a pair changes image (operand scale, per-image bounds, a_gate / a_shift rows), tile (TMA origins, residual row,
colsum index, store), channel group (bias, weight rows), and every ring (input, weights, shared-memory A, accumulator)
starts where the previous unit left it.  Every case restates the launch arithmetic (``schedule``) and asserts the regime
it exists for, so a change of tile size or SM count fails here instead of quietly testing something else.

The images of a batch are scaled more than 10^6 apart (MAGS): a scale, bound or row taken from another unit's image
then overflows fp16 or drops the lo half and the per-image check fails by orders of magnitude."""
import math
from typing import NamedTuple, Optional

import pytest
import torch
import torch.nn.functional as F

from faster_orefsdet_b200 import ops
from tests.util import amax_per_image, presplit

gpu = pytest.mark.gpu
DEV = "cuda"
TILE_H, TILE_W, PART_CHUNKS, CHUNK = 8, 16, 16, 32       # conv_tc.cu: kTileH, kTileW, kPartChunks, kChunk
RING_STAGES = {"input": 3, "tmem_b": 6, "smem_a": 2, "acc": 2}
MAGS = (2e3, 3e-4, 5e2, 1e-4, 1e3, 2e-4)   # per-image magnitudes: neighbours differ by >= 1.6e6 either way
BAR = 2e-5                                  # of each image's own output maximum (test_conv_gpu.py measures ~5e-7)


# ------------------------------------------------------------------------------------------------------------ schedule
class Schedule(NamedTuple):
    tiles_per_img: int
    tiles: int
    n_group: int
    n_groups: int
    pair_units: int
    pairs: int
    min_units: int        # units of the pairs outside the last wave, and of those in it
    max_units: int
    last_wave: int        # pair-units in the last wave (pairs that run max_units)
    odd_tiles: bool       # the second CTA of the last pair recomputes the last tile and stores nothing
    chunks: int           # 32-channel chunks x taps of one unit
    parts: int            # partial sums of one unit
    chunks_per_part: int
    smem_b_stages: Optional[int]   # B ring depth of the shared-memory A pipeline (None: the layer cannot take it)
    steps: dict           # ring -> uses per unit: a ring's stage at the start of a unit moves iff steps % depth != 0

    @property
    def group_changes(self):
        """the channel group of a pair's units changes from one unit to the next (bias, weight rows)"""
        return self.pairs % self.n_groups != 0

    def shifts(self, ring):
        stages = self.smem_b_stages if ring == "smem_b" else RING_STAGES[ring]
        return self.steps[ring] % stages != 0


def schedule(n, h, w, cin, cout, k, stride=1, sms=None):
    """conv2d_nhwc_impl's launch arithmetic for an [n, cin, h, w] input"""
    if sms is None:
        sms = torch.cuda.get_device_properties(0).multi_processor_count
    pad = k // 2
    ho, wo = (h + 2 * pad - k) // stride + 1, (w + 2 * pad - k) // stride + 1
    tiles_per_img = math.ceil(wo / TILE_W) * math.ceil(ho / TILE_H)
    tiles = n * tiles_per_img
    n_group = min((cout + 15) // 16 * 16, 128)
    n_groups = math.ceil(cout / n_group)
    pair_units = math.ceil(tiles / 2) * n_groups
    pairs = min(pair_units, sms // 2)
    cin_chunks = math.ceil(cin / CHUNK)
    chunks = k * k * cin_chunks
    parts = math.ceil(chunks / PART_CHUNKS)
    cpp = math.ceil(chunks / parts)
    parts = math.ceil(chunks / cpp)
    max_units = math.ceil(pair_units / pairs)
    # smem_a_layout: 6 B stages up to n_group 64, 3 at 80 / 96, 2 at n_group 128 with stride 2; 3x3 layers only
    smem_b = None
    if k == 3:
        smem_b = 6 if n_group <= 64 else 3 if n_group <= 96 else 2 if stride == 2 else None
    steps = {"input": cin_chunks * (k * k if stride == 2 else 1),   # stride 2: one input stage per tap
             "tmem_b": chunks,
             "smem_a": cin_chunks * (3 if stride == 2 else 1),      # stride 2: one A stage per tap row
             "smem_b": 3 * cin_chunks,                               # one weight stage per tap row
             "acc": parts}
    return Schedule(tiles_per_img, tiles, n_group, n_groups, pair_units, pairs, pair_units // pairs, max_units,
                    pair_units - (max_units - 1) * pairs, tiles % 2 == 1, chunks, parts, cpp, smem_b, steps)


def _assert_regime(s, what, shifting=(), **want):
    """every pair runs at least two units, and the schedule has the properties the case exists for"""
    assert s.min_units >= 2, f"{what}: a pair runs {s.min_units} unit(s) ({s})"
    for key, v in want.items():
        assert getattr(s, key) == v, f"{what}: {key} = {getattr(s, key)}, the case exists for {v} ({s})"
    for ring in shifting:
        assert s.shifts(ring), f"{what}: the {ring} ring starts every unit at the same stage ({s})"


def test_schedule_restates_the_launch_arithmetic():
    """The helper itself, on shapes whose schedule is known (148 SMs)"""
    s = schedule(3, 80, 80, 112, 80, 3, sms=148)          # 150 tiles: one pair of 74 gets a second unit
    assert (s.tiles, s.pair_units, s.pairs, s.min_units, s.max_units, s.last_wave) == (150, 75, 74, 1, 2, 1)
    assert (s.n_group, s.chunks, s.parts, s.chunks_per_part, s.smem_b_stages) == (80, 36, 3, 12, 3)
    s = schedule(1, 10, 10, 384, 112, 3, sms=148)         # 108 chunks in 7 parts of <= 16
    assert (s.tiles, s.pairs, s.chunks, s.parts, s.chunks_per_part, s.smem_b_stages) == (2, 1, 108, 7, 16, None)
    s = schedule(1, 10, 12, 720, 512, 1, sms=148)         # four groups, 23 chunks in 2 parts
    assert (s.n_group, s.n_groups, s.pair_units, s.chunks, s.parts, s.chunks_per_part) == (128, 4, 4, 23, 2, 12)
    s = schedule(201, 14, 14, 256, 512, 3, 2, sms=148)    # ROI rows: one tile per image
    assert (s.tiles_per_img, s.odd_tiles, s.pair_units, s.min_units, s.max_units, s.last_wave) == (1, True, 404, 5, 6, 34)
    assert s.group_changes and s.steps["input"] == 72 and not s.shifts("input")
    assert schedule(2, 40, 40, 64, 128, 3, 2, sms=148).smem_b_stages == 2
    assert schedule(2, 40, 40, 64, 48, 3, sms=148).shifts("smem_b") is False


# ------------------------------------------------------------------------------------------------ inputs and reference
def _gen(seed):
    return torch.Generator(device=DEV).manual_seed(seed)


def _mags(n, mags=MAGS):
    return torch.tensor([mags[i % len(mags)] for i in range(n)], device=DEV).view(n, 1, 1, 1)


def _input(n, c, h, w, seed, mags=MAGS):
    x = torch.randn(n, c, h, w, generator=_gen(seed), device=DEV) * _mags(n, mags)
    return x.contiguous(memory_format=torch.channels_last)


def _weights(cout, cin, k, seed):
    """weights of unit gain, and a bias that differs per channel (bias[c] = (c / 64 - 1) * 1e-4): a bias kept from
    another channel group shows in the small images"""
    wt = torch.randn(cout, cin, k, k, generator=_gen(seed), device=DEV) / (k * k * cin) ** 0.5
    b = (torch.arange(cout, device=DEV, dtype=torch.float32) / 64.0 - 1.0) * 1e-4
    return wt, b


def _ref(x, wt, b=None, stride=1, relu=False, residual=None, up2=False):
    """float64 convolution (+ residual, nearest-2x upsampled if up2) (+ ReLU) on x's device; ATen's im2col + DGEMM"""
    with torch.backends.cudnn.flags(enabled=False):
        y = F.conv2d(x.double().contiguous(), wt.double(), None if b is None else b.double(), stride=stride,
                     padding=wt.shape[-1] // 2)
    if residual is not None:
        r = residual.double()
        if up2:
            r = r.repeat_interleave(2, 2).repeat_interleave(2, 3)[:, :, :y.shape[2], :y.shape[3]]
        y = y + r
    return y.relu() if relu else y


def _check(y, ref, what, bar=BAR):
    """per image: max |y - ref| <= bar * max |ref| of that image; returns the worst ratio"""
    n = y.shape[0]
    err = (y.double() - ref).abs().reshape(n, -1).amax(1)
    scale = ref.abs().reshape(n, -1).amax(1)
    rel = err / scale.clamp_min(1e-300)
    i = int(torch.nan_to_num(rel, nan=math.inf).argmax())
    worst = float(rel[i])
    assert worst <= bar, (f"{what}: image {i} of {n}: max abs err {float(err[i]):.3e} vs its output scale "
                          f"{float(scale[i]):.3e} ({worst:.2e} > {bar:.0e})")
    print(f"{what}: {worst:.2e} of {bar:.0e}")
    return worst


def _check_y_amax(y, ya, what):
    """the per-image y_amax is a maximum of the very fp32 values stored: exactly y[i].abs().amax()"""
    want = y.abs().amax((1, 2, 3))
    bad = (ya != want).nonzero().flatten().tolist()
    assert not bad, f"{what}: y_amax of images {bad[:8]}: {ya[bad[:8]].tolist()} vs {want[bad[:8]].tolist()}"


def _nhwc_out(n, c, h, w):
    return torch.empty((n, h, w, c), device=DEV).permute(0, 3, 1, 2)


@gpu
def test_float64_reference_on_the_device_matches_the_cpu():
    x = _input(2, 48, 13, 21, 1)
    wt, b = _weights(40, 48, 3, 2)
    r = torch.randn(2, 40, 7, 11, generator=_gen(3), device=DEV)
    for stride, res, up2 in ((1, None, False), (2, None, False), (1, r, True)):
        dev = _ref(x, wt, b, stride, True, res, up2)
        with torch.no_grad():
            cpu = F.conv2d(x.cpu().double(), wt.cpu().double(), b.cpu().double(), stride=stride, padding=1)
            if res is not None:
                cpu = cpu + F.interpolate(res.cpu().double(), scale_factor=2.0, mode="nearest")[:, :, :13, :21]
        assert torch.allclose(dev.cpu(), cpu.relu(), rtol=1e-12, atol=1e-12 * float(cpu.abs().max()))


# ------------------------------------------------------------------------------------------------------- the case table
# id, (n, h, w, cin, cout, k, stride), relu, both pipelines, regime, rings whose stage at the start of a unit must move
CASES = [
    # stem_2: 3-4 units per pair, 2 parts; Cin = 64 moves only the input ring (2 chunks over 3 stages)
    ("a", (3, 128, 160, 64, 64, 3, 1), True, True, dict(min_units=3, max_units=4, parts=2, smem_b_stages=6), ("input",)),
    # 3 chunks: 27 chunks over 6 B stages, 3 A stages over 2 (the A parity flips), 9 tap rows over 6 B stages
    ("b", (4, 96, 112, 96, 64, 3, 1), False, True, dict(min_units=2, max_units=3, parts=2, smem_b_stages=6),
     ("tmem_b", "smem_a", "smem_b")),
    # n_group 80 (3 B stages; 3 x Cin-chunks tap rows can never move a 3-deep ring); Cin 112: the last chunk is half
    # outside Cin; 3 parts move the accumulator ring; odd tile count: rank 1 recomputes the last tile after earlier units
    ("c", (3, 120, 136, 112, 80, 3, 1), True, True,
     dict(min_units=2, max_units=3, n_group=80, parts=3, odd_tiles=True, smem_b_stages=3), ("input", "acc")),
    # n_group 96; 72 chunks in 5 parts of 15 move the accumulator ring, 8 chunks the input ring
    ("d96", (3, 120, 136, 256, 96, 3, 1), False, True, dict(min_units=2, n_group=96, parts=5, smem_b_stages=3),
     ("input", "acc")),
    # 27 chunks in parts of 14: the first part ends inside a tap row of the shared-memory pipeline
    ("d80", (3, 120, 136, 80, 80, 3, 1), True, True, dict(min_units=2, n_group=80, chunks=27, chunks_per_part=14),
     ("tmem_b", "smem_a")),
    # the shared-memory pipeline at the n_group the model does not use; 16 / 32 columns: the second epilogue phase is idle
    ("e32", (3, 128, 160, 32, 32, 3, 1), False, True, dict(min_units=3, n_group=32, parts=1, smem_b_stages=6),
     ("input", "tmem_b", "smem_a", "smem_b", "acc")),
    ("e48", (3, 128, 160, 64, 48, 3, 1), True, True, dict(min_units=3, n_group=48, smem_b_stages=6), ("input",)),
    ("e16", (3, 128, 160, 64, 16, 3, 1), False, True, dict(min_units=3, n_group=16, smem_b_stages=6), ("input",)),
    # stride 2, n_group 128: 2 B stages; 96 -> 128 puts 9 tap rows per unit on them (and on the 2 A stages)
    ("f64", (3, 200, 232, 64, 128, 3, 2), True, True, dict(min_units=2, n_group=128, smem_b_stages=2), ()),
    ("f96", (3, 200, 232, 96, 128, 3, 2), True, True, dict(min_units=2, n_group=128, smem_b_stages=2),
     ("tmem_b", "smem_a", "smem_b")),
    # 384 -> 112: 108 chunks in 7 parts of <= 16, N = 112 (tensor memory only)
    ("g", (2, 128, 160, 384, 112, 3, 1), False, False, dict(min_units=2, n_group=112, parts=7, chunks_per_part=16), ("acc",)),
    # several channel groups, the last one partial (144 = 128 + 16; 74 pairs keep their group) ...
    ("h144", (2, 128, 160, 128, 144, 3, 1), True, False, dict(min_units=4, n_groups=2), ("input", "acc")),
    # ... and three groups, which a pair's units cycle through (bias and weight rows change every unit)
    ("h272", (2, 128, 160, 544, 272, 1, 1), False, False, dict(min_units=6, n_groups=3, group_changes=True),
     ("input", "tmem_b")),
    # one chunk per unit; one part per unit (the accumulator stage alternates every unit)
    ("i48", (2, 128, 160, 32, 48, 1, 1), False, False, dict(min_units=2, chunks=1, parts=1), ("input", "tmem_b", "acc")),
    ("i256", (2, 128, 160, 352, 256, 1, 1), True, False, dict(min_units=4, chunks=11, parts=1), ("input", "tmem_b", "acc")),
    # FsodRCNN ROI rows (res5 / conv_1): one tile per image, so the two CTAs of a pair hold different images; 201 bounds
    ("j512", (201, 14, 14, 256, 512, 3, 2), True, False,
     dict(tiles_per_img=1, min_units=5, max_units=6, odd_tiles=True, group_changes=True), ("acc",)),
    ("j256", (201, 7, 7, 256, 256, 3, 1), False, False, dict(tiles_per_img=1, min_units=2, max_units=3, odd_tiles=True),
     ("input", "acc")),
]


@gpu
@pytest.mark.parametrize("name,shape,relu,both,regime,shifting", CASES, ids=[c[0] for c in CASES])
def test_persistent_conv_matches_float64(name, shape, relu, both, regime, shifting):
    n, h, w, cin, cout, k, stride = shape
    _assert_regime(schedule(*shape), name, shifting, **regime)
    seed = 17 * cin + cout + k + stride
    x = _input(n, cin, h, w, seed)
    wt, b = _weights(cout, cin, k, seed + 1)
    pk = ops.conv2d_pack(wt)
    amax = amax_per_image(x)
    ya = ops.new_amax(DEV, n)
    y = ops.conv2d_nhwc(x, pk, b, cout, k, relu, stride=stride, x_amax=amax, y_amax=ya)
    _check(y, _ref(x, wt, b, stride, relu), name)
    _check_y_amax(y, ya, name)
    if both:   # the same input pre-split: the shared-memory A pipeline runs the same MMAs in the same order
        xp = presplit(x, amax)
        ya2 = ops.new_amax(DEV, n)
        if stride == 1:
            y2 = ops.conv2d_nhwc(xp, pk, b, cout, 3, relu, x_amax=amax, y_amax=ya2, x_presplit=True)
        else:   # stride 2 reads a pre-split input as a single slice through the split entry point (always ReLU)
            y2 = ops.conv2d_nhwc_split(xp, pk, b, cout, 3, _nhwc_out(n, cout, *y.shape[2:]), amax, y_amax=ya2,
                                       x_presplit_from=0, slice_ch=[0], stride=2)
        assert torch.equal(y2, y), f"{name}: the pre-split input gives other bits"
        assert torch.equal(ya2, ya)
    for i in (1, n - 1):   # alone, image i sits at another unit index on another pair
        yi = ops.conv2d_nhwc(x[i:i + 1], pk, b, cout, k, relu, stride=stride, x_amax=amax[:, i:i + 1].contiguous())
        assert torch.equal(yi[0], y[i]), f"{name}: image {i} alone differs from its slice of the batch"


@gpu
def test_batch_wide_y_amax_is_the_maximum_over_the_batch():
    n, h, w, cin, cout = 2, 128, 160, 352, 256
    _assert_regime(schedule(n, h, w, cin, cout, 1), "batch-wide y_amax")
    x = _input(n, cin, h, w, 5)
    wt, b = _weights(cout, cin, 1, 6)
    ya = ops.new_amax(DEV, 1)
    y = ops.conv2d_nhwc(x, ops.conv2d_pack(wt), b, cout, 1, x_amax=amax_per_image(x), y_amax=ya)
    assert torch.equal(ya, y.abs().amax().reshape(1))


# --------------------------------------------------------------------------------- epilogue extras and their consumers
def _tile_sums(y):
    """float64 per-tile channel sums of [N,C,Ho,Wo], as the colsum layout [N, tiles, C]: sum, sum of squares, sum of |y|"""
    n, c, ho, wo = y.shape
    ty, tx = math.ceil(ho / TILE_H), math.ceil(wo / TILE_W)
    p = torch.zeros((n, c, ty * TILE_H, tx * TILE_W), dtype=torch.float64, device=y.device)
    p[:, :, :ho, :wo] = y
    p = p.reshape(n, c, ty, TILE_H, tx, TILE_W).permute(0, 2, 4, 1, 3, 5).reshape(n, ty * tx, c, TILE_H * TILE_W)
    return p.sum(-1), (p * p).sum(-1), p.abs().sum(-1)


@gpu
@pytest.mark.parametrize("path", ["tmem", "smem"])
def test_colsum_colsumsq_are_the_tile_sums_of_the_output(path):
    """Per-tile channel sums against float64 sums of the kernel's own output; buffers preset with NaN, with guards on
    both sides: every tile's entry is written, nothing outside [N, tiles, C] is (not by the recomputed odd last tile)"""
    n, h, w = 3, 120, 136
    cin, cout, k = (544, 272, 1) if path == "tmem" else (112, 80, 3)
    s = schedule(n, h, w, cin, cout, k)
    _assert_regime(s, f"colsum {path}", odd_tiles=True, **(dict(group_changes=True) if path == "tmem" else dict(smem_b_stages=3)))
    x = _input(n, cin, h, w, 31 + k)
    wt, b = _weights(cout, cin, k, 32 + k)
    amax = amax_per_image(x)
    total, guard = n * s.tiles_per_img * cout, 2 * cout
    bufs = [torch.full((total + 2 * guard,), float("nan"), device=DEV) for _ in range(2)]
    cs, cq = (bb[guard:guard + total].view(n, s.tiles_per_img, cout) for bb in bufs)
    xin = x if path == "tmem" else presplit(x, amax)
    y = ops.conv2d_nhwc(xin, ops.conv2d_pack(wt), b, cout, k, True, x_amax=amax, colsum=cs, colsumsq=cq,
                        x_presplit=path == "smem")
    _check(y, _ref(x, wt, b, 1, True), f"colsum {path}: output")
    for bb in bufs:
        assert bool(bb[:guard].isnan().all()) and bool(bb[guard + total:].isnan().all()), "written outside [N, tiles, C]"
    s1, s2, sa = _tile_sums(y)
    for got, want, mag, what in ((cs, s1, sa, "colsum"), (cq, s2, s2, "colsumsq")):
        assert bool(torch.isfinite(got).all()), f"{what}: {int((~torch.isfinite(got)).sum())} entries not written"
        err = (got.double() - want).abs() - 1e-5 * mag
        assert float(err.max()) <= 0, f"{what} ({path}): {int((err > 0).sum())} entries off, first at {(err > 0).nonzero()[0].tolist()}"


@gpu
def test_conv_groupnorm_relu_conv_in_the_persistent_regime():
    """CenterNetHead tower: 3x3 128 -> 128 with colsum / colsumsq -> group_norm_affine with one bound per map -> 1x1
    48-column consumer applying act(x * scale + shift) to its operand; against float64 GroupNorm"""
    n, h, w, c = 2, 128, 160, 128
    _assert_regime(schedule(n, h, w, c, c, 3), "tower", parts=3)
    _assert_regime(schedule(n, h, w, c, 48, 1), "consumer", n_group=48)
    x = _input(n, c, h, w, 41)
    w1, b1 = _weights(c, c, 3, 42)
    gamma = 0.5 + torch.rand(c, generator=_gen(43), device=DEV)
    beta = torch.rand(c, generator=_gen(44), device=DEV) - 0.5
    w2, b2 = _weights(48, c, 1, 45)
    t_ref = _ref(x, w1, b1)
    g_ref = F.group_norm(t_ref, 32, gamma.double(), beta.double(), 1e-5).relu()
    y_ref = _ref(g_ref, w2, b2)
    tiles = ops.conv2d_tiles_per_image(h, w)
    cs, cq = torch.zeros((n, tiles, c), device=DEV), torch.zeros((n, tiles, c), device=DEV)
    a_t = ops.new_amax(DEV, n)
    t = ops.conv2d_nhwc(x, ops.conv2d_pack(w1), b1, c, 3, x_amax=amax_per_image(x), y_amax=a_t, colsum=cs, colsumsq=cq)
    _check(t, t_ref, "tower conv")
    scale, shift, a_g = ops.group_norm_affine(cs, cq, h * w, 32, gamma, beta, 1e-5, x_amax=a_t)
    assert a_g.shape == (n,) and bool((a_g.double() >= g_ref.amax((1, 2, 3)) * (1 - 1e-5)).all())
    y = ops.conv2d_nhwc(t, ops.conv2d_pack(w2), b2, 48, 1, x_amax=a_g.view(1, n), a_gate=scale, a_shift=shift, a_relu=True)
    _check(y, y_ref, "GroupNorm + ReLU consumer")


@gpu
@pytest.mark.parametrize("c", [112, 256, 384, 512])
def test_ese_gate_from_colsum_and_its_gated_consumer(c):
    """OSA concat 1x1 with colsum -> ese_gate at the backbone's widths (partial blocks of 32 outputs, 160 tiles per
    image) -> the next layer with the gate on its operand (a_gate needs Cin % 32 == 0: not 112, which the model gates
    outside the kernel).  Magnitudes 3 and 3e-6: the first image's gate does not saturate."""
    n, h, w, cin = 2, 128, 160, 256
    mags = (3.0, 3e-6)
    _assert_regime(schedule(n, h, w, cin, c, 1), f"eSE {c}")
    x = _input(n, cin, h, w, 50 + c, mags)
    wt, b = _weights(c, cin, 1, 51 + c)
    fw = torch.randn(c, c, 1, 1, generator=_gen(52 + c), device=DEV) * (3.0 / c ** 0.5)
    fb = torch.randn(c, generator=_gen(53 + c), device=DEV) * 0.5
    y_ref = _ref(x, wt, b, relu=True)
    g_ref = F.relu6(F.conv2d(y_ref.mean((2, 3), keepdim=True), fw.double(), fb.double()) + 3.0) / 6.0
    colsum = torch.full((n, ops.conv2d_tiles_per_image(h, w), c), float("nan"), device=DEV)
    ya = ops.new_amax(DEV, n)
    y = ops.conv2d_nhwc(x, ops.conv2d_pack(wt), b, c, 1, True, x_amax=amax_per_image(x), y_amax=ya, colsum=colsum)
    _check(y, y_ref, f"eSE {c}: concat 1x1")
    gate = ops.ese_gate(colsum, h * w, fw, fb)
    err = float((gate.double() - g_ref.view(n, c)).abs().max())
    print(f"eSE {c}: gate {err:.2e} of 1e-5")
    assert err <= 1e-5, f"eSE {c}: gate off by {err:.3e}"
    if c % 32 == 0:
        w2, b2 = _weights(64, c, 1, 54 + c)
        _assert_regime(schedule(n, h, w, c, 64, 1), f"eSE {c} consumer")
        out = ops.conv2d_nhwc(y, ops.conv2d_pack(w2), b2, 64, 1, x_amax=ya.view(1, n), a_gate=gate)
        _check(out, _ref(y_ref * g_ref, w2, b2), f"eSE {c}: gated consumer")


@gpu
def test_split_handoff_at_several_units_per_pair():
    """conv2d_nhwc_split writing the consumer's operand format: the stored bytes are presplit(fp32 output of the same
    layer, published bound), and the pre-split consumer (shared-memory A pipeline) matches float64 of both layers"""
    n, h, w, c1, c2 = 3, 128, 160, 64, 80
    _assert_regime(schedule(n, h, w, c1, c1, 3), "producer")
    _assert_regime(schedule(n, h, w, c1, c2, 3), "consumer", smem_b_stages=3)
    x = _input(n, c1, h, w, 61)
    w1, b1 = _weights(c1, c1, 3, 62)
    w2, b2 = _weights(c2, c1, 3, 63)
    pk1 = ops.conv2d_pack(w1)
    amax = amax_per_image(x)
    l1 = float(w1.double().abs().sum((1, 2, 3)).max()) * 1.001
    beta = float(b1.abs().max()) * 1.001
    ys, yb, ya = _nhwc_out(n, c1, h, w), torch.empty((n,), device=DEV), ops.new_amax(DEV, n)
    ops.conv2d_nhwc_split(x, pk1, b1, c1, 3, ys, amax, y_amax=ya, y_bound=yb, y_l1=l1, y_beta=beta)
    yf = ops.conv2d_nhwc(x, pk1, b1, c1, 3, True, x_amax=amax)
    r1 = _ref(x, w1, b1, relu=True)
    assert bool((yb >= yf.amax((1, 2, 3))).all()), "a published bound below its image's maximum"
    _check_y_amax(yf, ya, "split producer")
    want = presplit(yf, yb.view(1, n)).permute(0, 2, 3, 1).contiguous().view(torch.int32)
    got = ys.permute(0, 2, 3, 1).contiguous().view(torch.int32)
    bad = (got != want).nonzero()
    assert bad.numel() == 0, f"{bad.shape[0]} stored words differ from the split of the fp32 output, first at {bad[0].tolist()}"
    y2 = ops.conv2d_nhwc(ys, ops.conv2d_pack(w2), b2, c2, 3, True, x_amax=yb.view(1, n), x_presplit=True)
    _check(y2, _ref(r1, w2, b2, relu=True), "pre-split consumer of a split hand-off")


@gpu
def test_concat_1x1_over_mixed_slices_with_per_image_bounds():
    """1x1 over a concat buffer: an fp32 slice and three slices stored pre-split, each at its own per-image bound
    (x_presplit_from / slice_ch), two channel groups, 4-5 units per pair"""
    n, h, w, c0, sc, cout = 2, 128, 160, 128, 80, 256
    cin = c0 + 3 * sc
    _assert_regime(schedule(n, h, w, cin, cout, 1), "concat 1x1", n_groups=2)
    starts = [0, c0, c0 + sc, c0 + 2 * sc]
    xs = [_input(n, c0 if k == 0 else sc, h, w, 70 + k) * f for k, f in enumerate((1.0, 0.3, 3.0, 0.7))]
    buf = torch.empty((n, h, w, cin), device=DEV).permute(0, 3, 1, 2)
    amax = torch.zeros((4, n), device=DEV)
    for k, xk in enumerate(xs):
        amax[k] = amax_per_image(xk).view(-1)
        end = starts[k] + xk.shape[1]
        buf[:, starts[k]:end] = xk if k == 0 else presplit(xk, amax[k:k + 1])
    wt, b = _weights(cout, cin, 1, 75)
    y = ops.conv2d_nhwc_split(buf, ops.conv2d_pack(wt), b, cout, 1, _nhwc_out(n, cout, h, w), amax, x_presplit_from=c0,
                              slice_ch=starts)
    _check(y, _ref(torch.cat(xs, 1), wt, b, relu=True), "concat 1x1 over mixed slices")


@gpu
@pytest.mark.parametrize("up2", [False, True])
def test_residual_in_the_epilogue_at_several_units_per_pair(up2):
    """FPN lateral: 1x1 + (nearest 2x upsampled) coarser map in the epilogue; odd output size under upsampling"""
    n, h, w, cin, cout = 2, 127, 159, 96, 256
    _assert_regime(schedule(n, h, w, cin, cout, 1), "residual", n_groups=2)
    x = _input(n, cin, h, w, 81)
    wt, b = _weights(cout, cin, 1, 82)
    rs = ((h + 1) // 2, (w + 1) // 2) if up2 else (h, w)
    r = _input(n, cout, *rs, 83)
    ya = ops.new_amax(DEV, n)
    y = ops.conv2d_nhwc(x, ops.conv2d_pack(wt), b, cout, 1, x_amax=amax_per_image(x), y_amax=ya, residual=r,
                        residual_upsample2=up2)
    _check(y, _ref(x, wt, b, residual=r, up2=up2), f"residual{' + up2' if up2 else ''}")
    _check_y_amax(y, ya, "residual")


# --------------------------------------------------------------------------------------------------- fod_absmax_rows
@gpu
@pytest.mark.parametrize("rows,length", [(1, 3), (1, 4099), (1, 1_000_003), (3, 113_676), (201, 12_544), (3_200, 1_000)])
def test_absmax_rows_is_exact(rows, length):
    """The per-row bound the split format's scale comes from: a value below the true maximum overflows fp16.  The
    maximum sits in the first element, the last, the middle, or (one row of n % 4 != 0) the tail block 0 reads; all-zero
    rows report 0"""
    x = torch.randn(rows, length, generator=_gen(rows + length), device=DEV)
    r = torch.arange(rows, device=DEV)
    where = torch.tensor([0, length - 1, length // 2 + 1], device=DEV)
    for rot in range(3):      # row i has its maximum (of either sign) at where[(i + rot) % 3]
        xt = x.clone()
        xt[r, where[(r + rot) % 3]] = (9.0 + r) * (1.0 - 2.0 * (r % 2))
        if rows > 1:
            xt[1] = 0.0
        got, want = ops.absmax(xt, per_image=True), xt.abs().amax(1)
        assert torch.equal(got, want), f"rows {(got != want).nonzero().flatten()[:8].tolist()} differ (rotation {rot})"
    assert torch.equal(ops.absmax(torch.zeros(rows, length, device=DEV), per_image=True), torch.zeros(rows, device=DEV))
