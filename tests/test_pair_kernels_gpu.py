"""The CTA-pair tensor-core kernels in the modes the model runs them in: the relation head with per-image operand
bounds, and the correlation reporting the bound of every map it writes."""
import pytest
import torch

from faster_orefsdet_b200 import fold, ops, synth
from oracle import head_oracle as O
from tests.util import assert_close, head_state_dict

pytestmark = pytest.mark.gpu
DEV = "cuda"
CFG = O.HeadConfig()


def test_relation_head_per_image_bounds():
    """x_amax [k, B] (roi_heads.detect_raw): the rows of image b are scaled by column b alone.  Three images whose pooled
    magnitudes lie two orders of magnitude apart, ragged counts (full, empty, one row, across a unit boundary), two
    classes: every image against float64, and each image's rows bit-identical to a call that holds that image alone."""
    sd = head_state_dict()
    B, C, cap = 3, 2, 200
    P = B * C
    mags = torch.tensor([1.0, 1e-2, 1e-4]).repeat_interleave(C)
    counts = torch.tensor([200, 1, 0, 129, 128, 57], dtype=torch.int32)
    pooled = synth.tensor((P, cap, 64, 128), 81, -1.0, 1.5) * mags.view(P, 1, 1, 1)
    ctr = synth.tensor((P * cap, 2), 82, 30.0, 280.0)
    wh = synth.tensor((P * cap, 2), 83, 8.0, 150.0)
    bx = torch.cat((ctr - wh / 2, ctr + wh / 2), 1).reshape(P, cap, 4)
    sup = synth.tensor((C, 128, 8, 8), 84, -1.0, 1.0)
    amax = pooled.reshape(B, -1).abs().amax(1)
    x_amax = torch.stack((0.5 * amax, amax))          # [k = 2, B]: the larger row bounds each image
    w_fold, w_out, b_out = fold.fold_relation_weights(sd)
    packed = ops.relation_pack(w_fold.to(DEV))
    bias, w_out, b_out = fold.fold_class_bias(sd, sup).to(DEV), w_out.to(DEV), b_out.to(DEV)

    def run(problems, bounds):
        return ops.relation_head(pooled[problems].to(DEV), packed, bias, w_out, b_out, bx[problems].to(DEV),
                                 counts[problems].to(DEV), C, CFG.bbox_reg_weights, want_raw=True,
                                 x_amax=bounds.contiguous().to(DEV))

    db, ds, logits, deltas = run(slice(None), x_amax)
    torch.cuda.synchronize()
    sd64 = {k: v.double() for k, v in sd.items()}
    for p in range(P):
        n = int(counts[p])
        if n < cap:
            assert float(ds[p, n:].abs().max()) == 0.0
        if n == 0:
            continue
        x = pooled[p, :n].reshape(n, 8, 8, 128).permute(0, 3, 1, 2).double()
        ref_logits, ref_deltas = O.relation_head(x, sup[p % C:p % C + 1].double(), sd64)
        assert_close(logits[p, :n], ref_logits, what=f"logits p{p}")
        assert_close(deltas[p, :n], ref_deltas, atol=2e-5, what=f"deltas p{p}")
        sc, bb = O.score_and_decode(ref_logits, ref_deltas, bx[p, :n].double(), CFG)
        assert_close(ds[p, :n], sc, what=f"scores p{p}")
        assert_close(db[p, :n], bb, atol=2e-3, what=f"boxes p{p}")
    for b in range(B):
        mine = slice(b * C, (b + 1) * C)
        alone = run(mine, x_amax[:, b:b + 1])
        for name, got, want in zip(("boxes", "scores", "logits", "deltas"), (db, ds, logits, deltas), alone):
            assert torch.equal(got[mine], want), f"image {b}: {name} depend on the batch mates"


def test_correlate_levels_amax_is_the_max_of_each_map():
    """want_amax: per level and problem, the returned bound equals attn[l][p].amax() bit for bit.  The levels are not
    multiples of the 8 x 16 tile, and the weights put every padding pixel of a tile above every pixel of the map
    (q > 0, so s > 0, against W3 <= 0 and b3 = 10: a map stays below 10, a pixel with no input in reach is 10), so a
    bound that counted padding pixels would be 10."""
    sizes, B, C = ((13, 21), (7, 11), (4, 5)), 2, 3
    qs = [synth.tensor((B, 128, h, w), 450 + 3 * i, 0.5, 1.5).to(DEV) for i, (h, w) in enumerate(sizes)]
    taps = [ops.support_taps(synth.tensor((C, 128, 3, 4), 460 + i, -0.6, 0.8).to(DEV)).cpu() for i in range(len(sizes))]
    w3 = -synth.tensor((128, 256), 470, 0.0, 0.02)
    b3 = torch.full((128,), 10.0)
    attn, amax = ops.correlate_levels(qs, taps, w3.to(DEV), b3.to(DEV), want_amax=True)
    torch.cuda.synchronize()
    for l, (h, w) in enumerate(sizes):
        assert attn[l].shape == (B * C, 128, h, w) and amax[l].shape == (B * C,)
        want = attn[l].amax(dim=(1, 2, 3))
        assert float(want.max()) < 10.0 and float(want.min()) > 0.0
        assert torch.equal(amax[l], want), f"level {l}: {amax[l].tolist()} vs {want.tolist()}"
