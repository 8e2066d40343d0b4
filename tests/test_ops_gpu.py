"""GPU parity: every C-ABI kernel against the CPU oracle on the same seeded inputs.
Index outputs bit-exact, floating point within 1e-4 relative (north_star)."""
import numpy as np
import pytest
import torch

from faster_orefsdet_b200 import fold, ops, synth
from oracle import head_oracle as O
from tests.util import assert_close, golden, head_state_dict, t

pytestmark = pytest.mark.gpu
DEV = "cuda"
CFG = O.HeadConfig()


def _boxes(n, seed, lo=20.0, hi=300.0, wmin=8.0, wmax=90.0):
    ctr = synth.tensor((n, 2), seed, lo, hi)
    wh = synth.tensor((n, 2), seed + 1, wmin, wmax)
    return torch.cat((ctr - wh / 2, ctr + wh / 2), 1)


# ----------------------------------------------------------------------------------------- NMS
@pytest.mark.parametrize("n", [0, 1, 63, 64, 65, 700, 3000, 8192])
def test_batched_nms_single_class_bit_exact(n):
    boxes = _boxes(n, 11 + n)
    scores = torch.round(synth.tensor((n,), 13 + n, 0.0, 1.0) * 256) / 256     # ties
    for thr in (0.6, 0.9):
        ref = O.batched_nms_coordinate_trick(boxes, scores, torch.zeros(n, dtype=torch.long), thr)
        got = ops.batched_nms(boxes.to(DEV), scores.to(DEV), None, thr)
        assert np.array_equal(got.cpu().numpy(), ref.numpy())


def test_batched_nms_golden_reference_vectors():
    g = golden("ops")
    n = 700
    boxes = _boxes(n, 11)
    scores = torch.round(synth.tensor((n,), 13, 0.0, 1.0) * 64) / 64
    boxes[100:140] = boxes[60:100]
    idxs = (synth.tensor((n,), 14, 0.0, 1.0) * 3).long()
    for thr in (0.6, 0.9):
        k1 = ops.batched_nms(boxes.to(DEV), scores.to(DEV), None, thr)
        k3 = ops.batched_nms(boxes.to(DEV), scores.to(DEV), idxs.to(DEV), thr)
        assert np.array_equal(k1.cpu().numpy(), g[f"nms1_keep_{thr}"])
        assert np.array_equal(k3.cpu().numpy(), g[f"nms3_keep_{thr}"])
    eb = torch.tensor([[0, 0, 10, 10], [0, 0, 10, 6], [0, 0, 5, 9], [0, 0, 9, 10.0]])
    es = torch.tensor([0.9, 0.8, 0.7, 0.6])
    for thr in (0.6, 0.9, 0.45):
        k = ops.batched_nms(eb.to(DEV), es.to(DEV), None, thr)
        assert np.array_equal(k.cpu().numpy(), g[f"nms_edge_keep_{thr}"])


def test_batched_nms_all_equal_scores_and_identical_boxes():
    n = 500
    boxes = _boxes(n, 77)
    boxes[250:] = boxes[:250]
    scores = torch.full((n,), 0.5)
    ref = O.batched_nms_coordinate_trick(boxes, scores, torch.zeros(n, dtype=torch.long), 0.6)
    got = ops.batched_nms(boxes.to(DEV), scores.to(DEV), None, 0.6)
    assert np.array_equal(got.cpu().numpy(), ref.numpy())


@pytest.mark.parametrize("max_cluster", [1, 2, 4])
def test_nms_every_cluster_size(max_cluster, monkeypatch):
    """One, two and four CTAs per problem run the same sweep on differently split data (own suppression words, exchanged
    chunk pairs, shared survivor / alive-list array): each must reproduce the oracle on a full sweep without early stop
    (3000 candidates, almost nothing suppressed at first) and on the duplicated-box list."""
    monkeypatch.setenv("FOD_NMS_MAX_CLUSTER", str(max_cluster))
    n = 500
    boxes = _boxes(n, 77)
    boxes[250:] = boxes[:250]
    scores = torch.full((n,), 0.5)
    ref = O.batched_nms_coordinate_trick(boxes, scores, torch.zeros(n, dtype=torch.long), 0.6)
    got = ops.batched_nms(boxes.to(DEV), scores.to(DEV), None, 0.6)
    assert np.array_equal(got.cpu().numpy(), ref.numpy())
    cap = 3000
    pb = _boxes(cap, 300, 30.0, 600.0, 20.0, 60.0).unsqueeze(0)
    ps = synth.tensor((cap,), 301, 0.01, 1.0).unsqueeze(0)
    status = ops.new_status(DEV)
    keep, ob, os_, oc = ops.nms_proposals(pb.to(DEV), ps.to(DEV), torch.tensor([cap], dtype=torch.int32, device=DEV), 0.6, -1, cap,
                                          status)
    ops.check_status(status)
    ref = O.proposal_nms_topk(pb[0], ps[0], O.HeadConfig(post_nms_topk=10 ** 9))
    m = int(oc[0])
    assert m == ref.numel() and np.array_equal(keep[0, :m].cpu().numpy(), ref.numpy())


@pytest.mark.parametrize("post_topk,ties", [(256, False), (256, True), (2000, False), (-1, False)])
def test_nms_proposals_bit_exact(post_topk, ties):
    P, cap = 5, 3000
    counts = [3000, 2400, 0, 1, 777]
    boxes = torch.zeros((P, cap, 4))
    scores = torch.zeros((P, cap))
    for p in range(P):
        n = counts[p]
        boxes[p, :n] = _boxes(n, 100 + p, 30.0, 600.0, 60.0, 180.0)
        s = synth.tensor((n,), 200 + p, 0.01, 1.0)
        scores[p, :n] = torch.round(s * 50) / 50 if ties else s
    cfg = O.HeadConfig(post_nms_topk=post_topk if post_topk > 0 else 10 ** 9)
    roi_cap = 3000
    status = ops.new_status(DEV)
    keep, ob, os_, oc = ops.nms_proposals(boxes.to(DEV), scores.to(DEV), torch.tensor(counts, dtype=torch.int32, device=DEV),
                                          0.6, post_topk, roi_cap, status)
    ops.check_status(status)
    for p in range(P):
        n = counts[p]
        ref = O.proposal_nms_topk(boxes[p, :n], scores[p, :n], cfg)
        m = int(oc[p])
        assert m == ref.numel(), (p, m, ref.numel())
        assert np.array_equal(keep[p, :m].cpu().numpy(), ref.numpy())
        assert np.array_equal(ob[p, :m].cpu().numpy(), boxes[p, :n][ref].numpy())
        assert np.array_equal(os_[p, :m].cpu().numpy(), scores[p, :n][ref].numpy())


def test_nms_proposals_overflow_flag():
    P, cap = 1, 512
    boxes = _boxes(cap, 5, 30.0, 3000.0, 5.0, 10.0).unsqueeze(0)       # nothing overlaps
    scores = torch.full((1, cap), 0.5)                                  # everything ties
    status = ops.new_status(DEV)
    _, _, _, oc = ops.nms_proposals(boxes.to(DEV), scores.to(DEV), None, 0.6, 256, 300, status)
    assert int(status.item()) & 2
    assert int(oc[0]) == 300


# ----------------------------------------------------------------------------------------- decode
def _decode_case(sizes, strides, P, seed, ties):
    hm, reg = [], []
    for l, (h, w) in enumerate(sizes):
        x = synth.tensor((P, 1, h, w), seed + l, -9.0, 3.0)
        if ties:
            x = torch.round(x * 8) / 8
        x[:, :, :1] = -20.0
        hm.append(x)
        reg.append(synth.tensor((P, 4, h, w), seed + 10 + l, 0.0, 9.0))
    return hm, reg


@pytest.mark.parametrize("ties", [False, True])
@pytest.mark.parametrize("channels_last", [False, True])
def test_decode_topk_bit_exact_on_probabilities(ties, channels_last):
    sizes, strides, P = [(40, 48), (20, 24), (10, 12)], (8, 16, 32), 3
    hm, reg = _decode_case(sizes, strides, P, 21, ties)
    prob = [h.sigmoid() for h in hm]                       # identical scores on both sides
    status = ops.new_status(DEV)
    regd = [r.to(DEV) for r in reg]
    if channels_last:
        regd = [r.contiguous(memory_format=torch.channels_last) for r in regd]
    boxes, scores, loc, lc, cc = ops.decode_topk([x.to(DEV) for x in prob], regd, strides, CFG.inference_th, 1000,
                                                 status, hm_is_logit=False)
    ops.check_status(status)
    for p in range(P):
        off = 0
        for l in range(3):
            ref_loc, ref_boxes, ref_scores = _oracle_decode_prob(prob[l][p, 0], reg[l][p], strides[l])
            n = ref_loc.numel()
            assert int(lc[p, l]) == n
            assert np.array_equal(loc[p, off:off + n].cpu().numpy(), ref_loc.numpy())
            assert np.array_equal(boxes[p, off:off + n].cpu().numpy(), ref_boxes.numpy())
            # torch's CPU sqrt goes through MKL VML on large tensors and is not correctly rounded
            # (about 0.6 % of elements are 1 ulp off); numpy's is, like CUDA's sqrt.rn.
            exact = np.sqrt(prob[l][p, 0].reshape(-1).numpy()[ref_loc.numpy()])
            assert np.array_equal(scores[p, off:off + n].cpu().numpy(), exact)
            assert_close(scores[p, off:off + n].cpu(), ref_scores, rtol=2e-7, atol=0, what="scores vs oracle")
            off += n
        assert int(cc[p]) == off


def _oracle_decode_prob(prob, reg, stride):
    return O.decode_level(prob, reg, stride, CFG, is_logit=False)


def test_decode_topk_from_logits_matches_oracle_set():
    sizes, strides, P = [(80, 80), (40, 40), (20, 20)], (8, 16, 32), 2
    hm, reg = _decode_case(sizes, strides, P, 31, False)
    status = ops.new_status(DEV)
    boxes, scores, loc, lc, cc = ops.decode_topk([x.to(DEV) for x in hm], [r.to(DEV) for r in reg], strides,
                                                 CFG.inference_th, 1000, status)
    ops.check_status(status)
    for p in range(P):
        off = 0
        for l in range(3):
            ref_loc, ref_boxes, ref_scores = O.decode_level(hm[l][p, 0], reg[l][p], strides[l], CFG)
            n = int(lc[p, l])
            assert n == ref_loc.numel()
            got = set(loc[p, off:off + n].cpu().tolist())
            want = set(ref_loc.tolist())
            # GPU expf vs CPU exp differ in the last ulp: allow a handful of swaps right at the k-th value
            assert len(got ^ want) <= 4, len(got ^ want)
            common = sorted(got & want)
            gi = {v: i for i, v in enumerate(loc[p, off:off + n].cpu().tolist())}
            ri = {v: i for i, v in enumerate(ref_loc.tolist())}
            gsel = torch.tensor([gi[v] for v in common])
            rsel = torch.tensor([ri[v] for v in common])
            assert_close(scores[p, off:off + n].cpu()[gsel], ref_scores[rsel], what="scores")
            assert_close(boxes[p, off:off + n].cpu()[gsel], ref_boxes[rsel], atol=1e-3, what="boxes")
            off += n


def test_decode_topk_taps_equals_conv_then_decode():
    """The 3x3 output convolutions folded into the decode (nine shifted sums of per-tap products from one 1x1 contraction)
    against F.conv2d + decode_level of the oracle: same candidate set, boxes and scores."""
    sd = head_state_dict()
    P = 3
    wh, bh = sd["proposal_generator.centernet_head.agn_hm.weight"], sd["proposal_generator.centernet_head.agn_hm.bias"]
    wr, br = sd["proposal_generator.centernet_head.bbox_pred.weight"], sd["proposal_generator.centernet_head.bbox_pred.bias"]
    w9 = torch.cat((wh.permute(0, 2, 3, 1).reshape(9, 128), torch.zeros((3, 128)),   # row tap | 12 + tap*4 + j
                    wr.permute(2, 3, 0, 1).reshape(36, 128)), 0).reshape(48, 128, 1, 1).contiguous()
    pk = ops.conv2d_pack(w9.to(DEV))
    sizes, strides, scales = [(40, 48), (20, 24), (7, 9)], (8, 16, 32), (1.0, 0.9, 1.1)
    taps, ts = [], []
    for l, (h, w) in enumerate(sizes):
        t_ = synth.tensor((P, 128, h, w), 400 + l, 0.0, 1.2)            # tower output (post ReLU)
        ts.append(t_)
        taps.append(ops.conv2d_nhwc(t_.to(DEV).contiguous(memory_format=torch.channels_last), pk, None, 48, 1))
    status = ops.new_status(DEV)
    bias5 = torch.cat((bh, br)).tolist()
    boxes, scores, loc, lc, cc = ops.decode_topk_taps(taps, bias5, strides, CFG.inference_th, 1000, status, reg_scale=scales)
    ops.check_status(status)
    for p in range(P):
        off = 0
        for l in range(3):
            hm = torch.nn.functional.conv2d(ts[l][p:p + 1], wh, bh, padding=1)[0, 0]
            reg = torch.relu(torch.nn.functional.conv2d(ts[l][p:p + 1], wr, br, padding=1)[0] * scales[l])
            ref_loc, ref_boxes, ref_scores = O.decode_level(hm, reg, strides[l], CFG)
            n = int(lc[p, l])
            got, want = set(loc[p, off:off + n].cpu().tolist()), set(ref_loc.tolist())
            assert abs(n - ref_loc.numel()) <= 2 and len(got ^ want) <= 4        # summation order at the k-th value
            gi = {v: i for i, v in enumerate(loc[p, off:off + n].cpu().tolist())}
            ri = {v: i for i, v in enumerate(ref_loc.tolist())}
            common = sorted(got & want)
            gsel, rsel = torch.tensor([gi[v] for v in common]), torch.tensor([ri[v] for v in common])
            assert_close(scores[p, off:off + n].cpu()[gsel], ref_scores[rsel], what="scores")
            assert_close(boxes[p, off:off + n].cpu()[gsel], ref_boxes[rsel], atol=2e-3, what="boxes")
            off += n
        assert int(cc[p]) == off


# ----------------------------------------------------------------------------------------- correlation
def test_support_taps_match_oracle():
    for size in (32, 16, 8, 7, 5):
        proto = synth.tensor((3, 128, size, size + 1), 40 + size, -1.0, 1.0)
        taps = ops.support_taps(proto.to(DEV)).cpu()
        for c in range(3):
            k11, k13, k31 = O.support_taps(proto[c:c + 1])
            assert_close(taps[c, 0], k11, what="k11")
            assert_close(taps[c, 1:4], k13.t(), what="k13")
            assert_close(taps[c, 4:7], k31.t(), what="k31")


@pytest.mark.parametrize("hw", [(80, 80), (20, 20), (25, 42), (7, 9), (1, 1)])
def test_correlate_matches_oracle(hw):
    sd = head_state_dict()
    B, C = 2, 3
    H, W = hw
    q = synth.tensor((B, 128, H, W), 50 + H, -1.5, 1.5)
    proto = synth.tensor((C, 128, 8, 8), 60, -0.6, 0.8)
    taps = ops.support_taps(proto.to(DEV))
    attn = ops.correlate(q.to(DEV), taps, sd["conv3.weight"].to(DEV), sd["conv3.bias"].to(DEV)).cpu()
    assert attn.shape == (B * C, 128, H, W)
    for b in range(B):
        for c in range(C):
            k11, k13, k31 = O.support_taps(proto[c:c + 1])
            ref = O.correlate_level(q[b:b + 1], k11, k13, k31, sd["conv3.weight"], sd["conv3.bias"])
            assert_close(attn[b * C + c], ref[0], what=f"attn b{b} c{c}")


@pytest.mark.parametrize("sizes,B,C", [(((80, 80), (40, 40), (20, 20)), 2, 1), (((25, 42), (13, 21), (7, 11)), 3, 2),
                                       (((8, 16),), 1, 1), (((1, 1), (5, 3)), 1, 3), (((100, 168), (50, 84), (25, 42)), 1, 2)])
def test_correlate_levels_tensor_core_matches_oracle(sizes, B, C):
    """One persistent tcgen05 launch over all levels (3xTF32) against the fp32 CPU oracle."""
    sd = head_state_dict()
    qs = [synth.tensor((B, 128, h, w), 150 + h + 3 * i, -1.5, 1.5) for i, (h, w) in enumerate(sizes)]
    protos = [synth.tensor((C, 128, 8 // (i + 1) + 1, 8 // (i + 1) + 2), 160 + i, -0.6, 0.8) for i in range(len(sizes))]
    taps = [ops.support_taps(p.to(DEV)) for p in protos]
    outs = ops.correlate_levels([q.to(DEV) for q in qs], taps, sd["conv3.weight"].to(DEV), sd["conv3.bias"].to(DEV))
    torch.cuda.synchronize()
    for l, (q, proto) in enumerate(zip(qs, protos)):
        got = outs[l].cpu()
        assert got.shape == (B * C, 128) + tuple(sizes[l])
        for b in range(B):
            for c in range(C):
                k11, k13, k31 = O.support_taps(proto[c:c + 1])
                ref = O.correlate_level(q[b:b + 1], k11, k13, k31, sd["conv3.weight"], sd["conv3.bias"])
                assert_close(got[b * C + c], ref[0], what=f"attn level{l} b{b} c{c}")


@pytest.mark.parametrize("C", [7, 10])
def test_correlate_levels_many_classes_matches_oracle(C):
    """BASELINE.json configs[2] is 10-way: the taps ride in the launch parameters six sets at a time, so C > 2 takes
    several launches with class_begin > 0 (three levels) - every (image, class) map against the oracle."""
    sd = head_state_dict()
    sizes, B = ((20, 24), (10, 12), (5, 6)), 2
    qs = [synth.tensor((B, 128, h, w), 350 + h + 3 * i, -1.5, 1.5) for i, (h, w) in enumerate(sizes)]
    protos = [synth.tensor((C, 128, 8 // (i + 1) + 1, 8 // (i + 1) + 2), 360 + i, -0.6, 0.8) for i in range(len(sizes))]
    taps = [ops.support_taps(p.to(DEV)).cpu() for p in protos]
    outs = ops.correlate_levels([q.to(DEV) for q in qs], taps, sd["conv3.weight"].to(DEV), sd["conv3.bias"].to(DEV))
    torch.cuda.synchronize()
    for l, (q, proto) in enumerate(zip(qs, protos)):
        got = outs[l].cpu()
        assert got.shape == (B * C, 128) + tuple(sizes[l])
        for b in range(B):
            for c in range(C):
                k11, k13, k31 = O.support_taps(proto[c:c + 1])
                ref = O.correlate_level(q[b:b + 1], k11, k13, k31, sd["conv3.weight"], sd["conv3.bias"])
                assert_close(got[b * C + c], ref[0], what=f"attn level{l} b{b} c{c}")
    # a single level takes six classes per launch: same maps
    one = ops.correlate_levels([qs[0].to(DEV)], taps[:1], sd["conv3.weight"].to(DEV), sd["conv3.bias"].to(DEV))[0]
    assert torch.equal(one, outs[0])


def test_correlate_levels_is_reentrant_across_streams():
    """Two episodes correlated concurrently on two streams must not see each other's taps (the taps are launch
    parameters, not a device symbol)."""
    sd = head_state_dict()
    w3, b3 = sd["conv3.weight"].to(DEV), sd["conv3.bias"].to(DEV)
    B, C = 8, 2
    qs = [synth.tensor((B, 128, 80, 80), 370, -1.5, 1.5).to(DEV), synth.tensor((B, 128, 40, 40), 371, -1.5, 1.5).to(DEV)]
    tap_sets = []
    for e in range(2):
        protos = [synth.tensor((C, 128, 9, 10), 380 + 10 * e + i, -0.6, 0.8) for i in range(2)]
        tap_sets.append([ops.support_taps(p.to(DEV)).cpu() for p in protos])
    ref = [[t.clone() for t in ops.correlate_levels(qs, tp, w3, b3)] for tp in tap_sets]
    torch.cuda.synchronize()
    streams = [torch.cuda.Stream(), torch.cuda.Stream()]
    for rnd in range(4):
        got = [None, None]
        for e in range(2):
            with torch.cuda.stream(streams[e]):
                got[e] = ops.correlate_levels(qs, tap_sets[e], w3, b3)
        torch.cuda.synchronize()
        for e in range(2):
            for a, b in zip(got[e], ref[e]):
                assert torch.equal(a, b), (rnd, e)


def test_correlate_golden_reference_maps():
    g = golden("full_small")
    sd = head_state_dict()
    protos = synth.prototypes(list(g["class_ids"]), int(g["shots"]), int(g["proto_seed"]))
    h, w = g["sizes"][0]
    feats = synth.features(1, int(h), int(w), int(g["feat_seed"]))
    for l, name in enumerate(("p3", "p4", "p5")):
        taps = ops.support_taps(protos[name][1].to(DEV))
        attn = ops.correlate(feats[name].to(DEV), taps, sd["conv3.weight"].to(DEV), sd["conv3.bias"].to(DEV))
        assert_close(attn[0].cpu(), t(g[f"img0_attn{l}"]), what=f"attn{l} vs reference")


# ----------------------------------------------------------------------------------------- ROI head
def test_roi_align_matches_reference_and_oracle():
    g = golden("ops")
    feats = synth.features(2, 256, 320, 31)
    fl = [feats["p3"], feats["p4"], feats["p5"]]
    bx = t(g["pool_boxes"])                                  # [2, 96, 4]
    want_lv = O.assign_levels(bx.reshape(-1, 4)).reshape(2, -1)
    for res in (8, 4):
        pooled, lv = ops.roi_align([f.to(DEV) for f in fl], (8, 16, 32), bx.to(DEV), None, 1, res, want_levels=True)
        assert np.array_equal(lv.cpu().numpy(), want_lv.numpy())
        got = pooled.cpu().reshape(2 * 96, res, res, 128).permute(0, 3, 1, 2)
        assert_close(got[:, ::8], t(golden("roi_pool")[f"pool_out{res}"]), what=f"roi_align{res} vs reference")
        assert_close(got, O.roi_pool(fl, [bx[0], bx[1]], res), what=f"roi_align{res} vs oracle")


def test_roi_align_respects_counts_and_classes():
    feats = synth.features(2, 128, 160, 33)
    fl = [feats["p3"], feats["p4"], feats["p5"]]
    C, cap = 2, 16
    bx = _boxes(2 * C * cap, 90, 10.0, 120.0, 4.0, 200.0).reshape(2 * C, cap, 4)
    counts = torch.tensor([16, 3, 0, 9], dtype=torch.int32)
    pooled = ops.roi_align([f.to(DEV) for f in fl], (8, 16, 32), bx.to(DEV), counts.to(DEV), C, 8).cpu()
    for p in range(2 * C):
        n = int(counts[p])
        img = p // C
        ref = O.roi_pool([f[img:img + 1] for f in fl], [bx[p, :n]], 8) if n else torch.zeros((0, 128, 8, 8))
        got = pooled[p, :n].reshape(n, 8, 8, 128).permute(0, 3, 1, 2)
        assert_close(got, ref, what=f"problem {p}")
    # the tiled operand layout of the relation head holds the same rows
    tiled = ops.roi_align([f.to(DEV) for f in fl], (8, 16, 32), bx.to(DEV), counts.to(DEV), C, 8, tiled=True)
    back = ops.untile_pooled(tiled, cap).cpu()
    for p in range(2 * C):
        n = int(counts[p])
        assert torch.equal(back[p, :n], pooled[p, :n])


def _roi_stress_boxes(n, seed, height, width):
    """Boxes of every kind the pooling has a separate path for: ordinary proposals, slivers and elongated boxes (bins
    longer than the tile halo: taps read from the map), boxes larger than their level expects (sampling grid beyond the
    tap tables: per-ROI list kernel), boxes partly / entirely outside the image, zero-area and inverted boxes."""
    base = _boxes(n, seed, 0.0, float(max(height, width)), 6.0, 260.0)
    kind = (synth.tensor((n,), seed + 7, 0.0, 1.0) * 10).floor()
    ctr = (base[:, :2] + base[:, 2:]) / 2
    wh = base[:, 2:] - base[:, :2]
    wh = torch.where((kind == 1)[:, None], wh * torch.tensor([6.0, 0.15]), wh)       # long and flat
    wh = torch.where((kind == 2)[:, None], wh * torch.tensor([0.1, 5.0]), wh)        # tall and thin
    wh = torch.where((kind == 3)[:, None], wh * 8.0, wh)                             # far beyond the image
    wh = torch.where((kind == 4)[:, None], wh * 0.0, wh)                             # zero area
    wh = torch.where((kind == 5)[:, None], wh * torch.tensor([-1.0, 1.0]), wh)       # inverted in x
    ctr = torch.where((kind == 6)[:, None], ctr - float(max(height, width)), ctr)    # left of / above the image
    ctr = torch.where((kind == 7)[:, None], ctr + float(max(height, width)), ctr)    # right of / below the image
    return torch.cat((ctr - wh / 2, ctr + wh / 2), 1)


@pytest.mark.parametrize("height,width,C", [(256, 320, 1), (200, 312, 3), (640, 640, 2)])
def test_roi_align_tile_stationary_is_bit_identical_to_per_roi(height, width, C):
    """The tile-stationary kernel (fod_roi_align, resolution 8) against the one-CTA-per-ROI kernel on the same inputs:
    every valid row bit-identical, rows beyond the count untouched, both output layouts; and against the oracle."""
    B, cap = 3, 300                                          # 300 > 256: two scan passes per problem
    feats = synth.features(B, height, width, 71 + C)
    fl = [feats["p3"], feats["p4"], feats["p5"]]
    bx = _roi_stress_boxes(B * C * cap, 300 + C, height, width).reshape(B * C, cap, 4)
    counts = torch.tensor([cap, 257, 0, 1, 256, 129, 40, cap, 7][:B * C], dtype=torch.int32)
    fd = [f.to(DEV) for f in fl]
    for tiled in (False, True):
        shape = (B * C, 3, 256, 128, 32) if tiled else (B * C, cap, 64, 128)
        out_t = torch.full(shape, -7.0, device=DEV)
        out_r = torch.full(shape, -7.0, device=DEV)
        _, lv_t = ops.roi_align(fd, (8, 16, 32), bx.to(DEV), counts.to(DEV), C, 8, out=out_t, tiled=tiled, want_levels=True)
        _, lv_r = ops.roi_align(fd, (8, 16, 32), bx.to(DEV), counts.to(DEV), C, 8, out=out_r, tiled=tiled, want_levels=True,
                                per_roi=True)
        assert torch.equal(lv_t, lv_r)
        assert torch.equal(out_t, out_r), f"tiled={tiled}: {(out_t != out_r).sum().item()} elements differ"
        if not tiled:
            got = out_t.cpu()
            for p in range(B * C):
                n = int(counts[p])
                assert torch.all(got[p, n:] == -7.0)
                if n and p % 2 == 0:
                    ok = (bx[p, :n, 2] > bx[p, :n, 0]) & (bx[p, :n, 3] > bx[p, :n, 1])     # the oracle's level rule needs a positive area
                    ref = O.roi_pool([f[p // C:p // C + 1] for f in fl], [bx[p, :n][ok]], 8)
                    assert_close(got[p, :n].reshape(n, 8, 8, 128).permute(0, 3, 1, 2)[ok], ref, what=f"problem {p} vs oracle")


def test_roi_align_tile_stationary_resumes_after_a_full_task_list():
    """300 small boxes crowded into one corner: every ROI's eight bin rows start inside the same 8 x 8-pixel tile, more
    tasks than one pass of the tile-stationary kernel holds (it stops at the first ROI that does not fit and resumes)."""
    feats = synth.features(2, 256, 320, 77)
    fl = [feats["p3"], feats["p4"], feats["p5"]]
    bx = _boxes(2 * 300, 91, 12.0, 44.0, 6.0, 30.0).reshape(2, 300, 4)
    counts = torch.tensor([300, 290], dtype=torch.int32, device=DEV)
    fd = [f.to(DEV) for f in fl]
    out_t = ops.roi_align(fd, (8, 16, 32), bx.to(DEV), counts, 1, 8)
    out_r = ops.roi_align(fd, (8, 16, 32), bx.to(DEV), counts, 1, 8, per_roi=True)
    for p, n in enumerate((300, 290)):
        assert torch.equal(out_t[p, :n], out_r[p, :n])
    ref = O.roi_pool([f[:1] for f in fl], [bx[0]], 8)
    assert_close(out_t[0].cpu().reshape(300, 8, 8, 128).permute(0, 3, 1, 2), ref, what="crowded boxes vs oracle")


def test_relation_head_matches_reference_and_oracle():
    g = golden("ops")
    sd = head_state_dict()
    feats = synth.features(2, 256, 320, 31)
    fl = [feats["p3"], feats["p4"], feats["p5"]]
    bx = t(g["pool_boxes"])
    sup = synth.tensor((5, 128, 8, 8), 41, -1.0, 1.0)
    w_fold, w_out, b_out = fold.fold_relation_weights(sd)
    bias = fold.fold_class_bias(sd, sup.mean(0, True))
    pooled = ops.roi_align([f.to(DEV) for f in fl], (8, 16, 32), bx.to(DEV), None, 1, 8)
    counts = torch.tensor([96, 70], dtype=torch.int32, device=DEV)
    db, ds, logits, deltas = ops.relation_head(pooled, w_fold.to(DEV), bias.to(DEV), w_out.to(DEV), b_out.to(DEV),
                                               bx.to(DEV), counts, 1, CFG.bbox_reg_weights, want_raw=True)
    ref_logits, ref_deltas = t(g["rel_logits"]).reshape(2, 96, 2), t(g["rel_deltas"]).reshape(2, 96, 4)
    for p, n in enumerate((96, 70)):
        assert_close(logits[p, :n].cpu(), ref_logits[p, :n], what="logits vs reference")
        assert_close(deltas[p, :n].cpu(), ref_deltas[p, :n], what="deltas vs reference")
        sc, bb = O.score_and_decode(ref_logits[p, :n], ref_deltas[p, :n], bx[p, :n], CFG)
        assert_close(ds[p, :n].cpu(), sc, what="scores")
        assert_close(db[p, :n].cpu(), bb, atol=2e-3, what="boxes")
        assert float(ds[p, n:].abs().max()) == 0.0 if n < 96 else True


def test_relation_head_tensor_core_multi_class_ragged_counts():
    """tcgen05 fp16-split contraction: several classes, roi_cap not a multiple of 128, empty / 1-row / full problems."""
    sd = head_state_dict()
    B, C, cap = 3, 2, 320
    P = B * C
    counts = torch.tensor([320, 0, 1, 129, 256, 37], dtype=torch.int32)
    pooled = synth.tensor((P, cap, 64, 128), 71, -1.0, 1.5)
    bx = _boxes(P * cap, 72, 30.0, 280.0, 8.0, 150.0).reshape(P, cap, 4)
    sup = synth.tensor((C, 128, 8, 8), 73, -1.0, 1.0)
    w_fold, w_out, b_out = fold.fold_relation_weights(sd)
    bias = fold.fold_class_bias(sd, sup)
    db, ds, logits, deltas = ops.relation_head(pooled.to(DEV), ops.relation_pack(w_fold.to(DEV)), bias.to(DEV), w_out.to(DEV),
                                               b_out.to(DEV), bx.to(DEV), counts.to(DEV), C, CFG.bbox_reg_weights,
                                               want_raw=True)
    torch.cuda.synchronize()
    for p in range(P):
        n = int(counts[p])
        if n == 0:
            continue
        x = pooled[p, :n].reshape(n, 8, 8, 128).permute(0, 3, 1, 2).contiguous()
        ref_logits, ref_deltas = O.relation_head(x, sup[p % C:p % C + 1], sd)
        assert_close(logits[p, :n].cpu(), ref_logits, what=f"logits p{p}")
        assert_close(deltas[p, :n].cpu(), ref_deltas, atol=2e-5, what=f"deltas p{p}")
        sc, bb = O.score_and_decode(ref_logits, ref_deltas, bx[p, :n], CFG)
        assert_close(ds[p, :n].cpu(), sc, what=f"scores p{p}")
        assert_close(db[p, :n].cpu(), bb, atol=2e-3, what=f"boxes p{p}")
        if n < cap:
            assert float(ds[p, n:].abs().max()) == 0.0


def test_relation_head_ten_classes_per_class_bias():
    """C = 10 (BASELINE.json configs[2]): every problem must pick its own class's folded bias."""
    sd = head_state_dict()
    B, C, cap = 2, 10, 130
    P = B * C
    counts = torch.tensor([(37 * p + 5) % (cap + 1) for p in range(P)], dtype=torch.int32)
    pooled = synth.tensor((P, cap, 64, 128), 171, -1.0, 1.5)
    bx = _boxes(P * cap, 172, 30.0, 280.0, 8.0, 150.0).reshape(P, cap, 4)
    sup = synth.tensor((C, 128, 8, 8), 173, -1.0, 1.0)
    w_fold, w_out, b_out = fold.fold_relation_weights(sd)
    bias = fold.fold_class_bias(sd, sup)
    db, ds, logits, deltas = ops.relation_head(pooled.to(DEV), ops.relation_pack(w_fold.to(DEV)), bias.to(DEV), w_out.to(DEV),
                                               b_out.to(DEV), bx.to(DEV), counts.to(DEV), C, CFG.bbox_reg_weights,
                                               want_raw=True)
    torch.cuda.synchronize()
    for p in range(P):
        n = int(counts[p])
        if n == 0:
            continue
        x = pooled[p, :n].reshape(n, 8, 8, 128).permute(0, 3, 1, 2).contiguous()
        ref_logits, ref_deltas = O.relation_head(x, sup[p % C:p % C + 1], sd)
        assert_close(logits[p, :n].cpu(), ref_logits, what=f"logits p{p}")
        assert_close(deltas[p, :n].cpu(), ref_deltas, atol=2e-5, what=f"deltas p{p}")
        sc, bb = O.score_and_decode(ref_logits, ref_deltas, bx[p, :n], CFG)
        assert_close(ds[p, :n].cpu(), sc, what=f"scores p{p}")
        assert_close(db[p, :n].cpu(), bb, atol=2e-3, what=f"boxes p{p}")


# ----------------------------------------------------------------------------------------- final detect
@pytest.mark.parametrize("C,cap", [(1, 64), (3, 64), (10, 320)])
def test_final_detect_bit_exact(C, cap):
    B = 3
    P = B * C
    boxes = _boxes(P * cap, 300, 10.0, 300.0, 10.0, 120.0).reshape(P, cap, 4)      # some stick out of the image
    scores = synth.tensor((P, cap), 301, 0.0, 1.0)
    scores = torch.round(scores * 40) / 40
    boxes[0, 3, 1] = float("nan")
    boxes[0, 4, 2] = float("inf")
    scores[1 % P, 5] = float("inf")
    counts = torch.tensor([(cap - 7 * p) % (cap + 1) for p in range(P)], dtype=torch.int32)
    if C == 10:
        counts[::3] = cap      # 10-way: full problems too (up to 3 200 rows per image enter the class-wise NMS)
    image_hw = torch.tensor([[256, 320]] * B, dtype=torch.int32)
    out_hw = torch.tensor([[256, 320], [300, 500], [128, 160]], dtype=torch.int32)
    for sthr, nthr, topk in ((0.0, 0.9, 100), (0.3, 0.5, 10)):
        cfg = O.HeadConfig(score_thresh_test=sthr, nms_thresh_test=nthr, detections_per_image=topk)
        status = ops.new_status(DEV)
        ob, os_, ocls, orow, oc = ops.final_detect(boxes.to(DEV), scores.to(DEV), counts.to(DEV), C, sthr, nthr, topk,
                                                   image_hw.to(DEV), out_hw.to(DEV), status)
        ops.check_status(status)
        for b in range(B):
            rb, rs, rc = [], [], []
            for c in range(C):
                n = int(counts[b * C + c])
                rb.append(boxes[b * C + c, :n])
                rs.append(scores[b * C + c, :n])
                rc.append(torch.full((n,), c, dtype=torch.long))
            fb, fs, fc, _ = O.final_detect(torch.cat(rb), torch.cat(rs), torch.cat(rc), (256, 320), cfg)
            pb, ps, pc = O.postprocess(fb, fs, fc, (256, 320), int(out_hw[b, 0]), int(out_hw[b, 1]))
            m = int(oc[b])
            assert m == pb.shape[0], (b, m, pb.shape[0])
            assert np.array_equal(ob[b, :m].cpu().numpy(), pb.numpy())
            assert np.array_equal(os_[b, :m].cpu().numpy(), ps.numpy())
            assert np.array_equal(ocls[b, :m].cpu().numpy(), pc.numpy())


def test_final_detect_golden_reference():
    g = golden("ops")
    pb, pr = t(g["frcnn_in_boxes"]), t(g["frcnn_in_probs"])
    n = pb.shape[0]
    hw = torch.tensor([[256, 320]], dtype=torch.int32, device=DEV)
    for tag, sthr, nthr, topk in (("frcnn", 0.0, 0.9, 100), ("frcnn2", 0.3, 0.5, 10)):
        status = ops.new_status(DEV)
        ob, os_, ocls, orow, oc = ops.final_detect(pb.reshape(1, n, 4).to(DEV), pr[:, 0].reshape(1, n).to(DEV), None,
                                                   1, sthr, nthr, topk, hw, None, status)
        m = int(oc[0])
        assert np.array_equal(ob[0, :m].cpu().numpy(), g[f"{tag}_boxes"])
        assert np.array_equal(os_[0, :m].cpu().numpy(), g[f"{tag}_scores"])
