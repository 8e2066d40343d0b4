"""Serving throughput of FsodRCNN: the plain ``model(batch)`` loop against the submit-ahead loop
(``q = model.submit(batch k+1); model(p_k)``), alternating in one process, plus the host time of one ``submit`` and the
device RPN proposal selection (``ops.rpn_proposals``) against the eager ``FsodRPN.predict_proposals`` on the same inputs.

Workload of bench.py::fsodrcnn_record: Base-FSOD-C4.yaml, 2-way episode, batch 16 x 640 x 640, synthetic weights.  Both
loops read the same pinned host images, so every host-to-device copy and the device-to-host copy of the detections are
inside the timed region.  Prints one JSON object (and writes it to --out), with the card's name, power limit and
maximum SM clock read by nvidia-smi in the same run.

    python tools/bench_fsodrcnn_serving.py --steps 20 --rounds 3 --out results.json
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import torch  # noqa: E402

from faster_orefsdet_b200 import ops, synth  # noqa: E402


def build_model(dev):
    from faster_orefsdet_b200.compat import META_ARCH_REGISTRY
    from faster_orefsdet_b200.config import get_cfg
    import faster_orefsdet_b200.modeling  # noqa: F401
    cfg = get_cfg()
    cfg.merge_from_file(os.path.join(ROOT, "configs/fsod/Base-FSOD-C4.yaml"))
    cfg.merge_from_list(["MODEL.DEVICE", str(dev)])
    m = META_ARCH_REGISTRY.get("FsodRCNN")(cfg).to(dev).eval()
    m.load_state_dict(synth.state_dict({k: tuple(v.shape) for k, v in m.state_dict().items()}))
    sup = {"res4_avg": {}, "res5_avg": {}}
    for j, c in enumerate((3, 9)):               # the episode of bench.py::fsodrcnn_record
        sup["res4_avg"][c] = synth.tensor((1, 1024, 14, 14), 341 + 2 * j, 0.0, 1.2)
        sup["res5_avg"][c] = synth.tensor((1, 2048, 7, 7), 342 + 2 * j, 0.0, 1.0)
    m.set_prototypes(sup)
    return m


def gpu_info():
    try:
        return subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv"],
                              capture_output=True, text=True, timeout=60).stdout.strip()
    except (OSError, subprocess.SubprocessError) as e:
        return f"nvidia-smi failed: {e}"


def plain_loop(m, batches, steps):
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for k in range(steps):
        out = m(batches[k % len(batches)])
    torch.cuda.synchronize()
    return (time.perf_counter() - t0) * 1e3 / steps, out


def submit_loop(m, batches, steps):
    """steps batches, batch k+1 submitted before batch k is collected; returns (ms per batch, ms of host time per
    submit call, last result)."""
    torch.cuda.synchronize()
    sub = []
    t0 = time.perf_counter()
    s0 = time.perf_counter()
    p = m.submit(batches[0])
    sub.append(time.perf_counter() - s0)
    for k in range(1, steps):
        s0 = time.perf_counter()
        q = m.submit(batches[k % len(batches)])
        sub.append(time.perf_counter() - s0)
        m(p)
        p = q
    out = m(p)
    torch.cuda.synchronize()
    return (time.perf_counter() - t0) * 1e3 / steps, statistics.median(sub) * 1e3, out


def rpn_times(m, batch, iters):
    """CUDA-event time per call of the eager selection and of ops.rpn_proposals, one class, on the RPN head output of
    one batch (the same inputs for both)."""
    rpn = m.proposal_generator
    with torch.no_grad():
        images = m.preprocess_image(batch)
        res4, gates, bounds = m._rpn_gates(m.backbone(images.tensor))
        logits, deltas = rpn.rpn_head([res4], [gates[0]], [bounds[0]])
        anchors = rpn.anchor_generator([res4])
        A = logits[0].shape[1]
        lg = [logits[0].permute(0, 2, 3, 1).flatten(1)]
        dl = [deltas[0].reshape(deltas[0].shape[0], -1, 4, deltas[0].shape[-2], deltas[0].shape[-1]).permute(0, 3, 4, 1, 2).flatten(1, -2)]
        hw = torch.tensor(images.image_sizes, dtype=torch.int32, device=res4.device)

        def eager():
            return rpn.predict_proposals(anchors, lg, dl, images.image_sizes)

        def device():
            return ops.rpn_proposals(logits, deltas, anchors, hw, rpn.pre_nms_topk, rpn.box_weights, rpn.min_box_size,
                                     rpn.nms_thresh, rpn.post_nms_topk)

        res = {}
        for name, fn in (("eager_predict_proposals", eager), ("rpn_proposals", device)):
            for _ in range(3):
                fn()
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(iters):
                r = fn()
            e1.record()
            torch.cuda.synchronize()
            res[name] = e0.elapsed_time(e1) / iters
            if name == "eager_predict_proposals":
                ref = r
            else:
                ob, ol, oc = r
                res["outputs_equal"] = all(int(oc[i]) == len(p) and torch.equal(ob[i, :len(p)], p.proposal_boxes.tensor)
                                           and torch.equal(ol[i, :len(p)], p.objectness_logits) for i, p in enumerate(ref))
    res["problems"], res["anchors_per_problem"] = int(res4.shape[0]), int(res4.shape[2] * res4.shape[3] * A)
    return res


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--steps", type=int, default=20, help="batches per timed loop")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--rounds", type=int, default=3, help="alternations of the two loops")
    ap.add_argument("--batch", type=int, default=16)
    ap.add_argument("--size", type=int, default=640)
    ap.add_argument("--rpn-iters", type=int, default=20)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("bench_fsodrcnn_serving: needs a CUDA device")
    dev = torch.device("cuda", 0)
    info = gpu_info()
    m = build_model(dev)
    batches = [[{"image": synth.ore_image(args.size, args.size, 7000 + 17 * k + i).pin_memory()} for i in range(args.batch)]
               for k in range(2)]
    with torch.no_grad():
        for _ in range(args.warmup):
            plain_loop(m, batches, 2)
            submit_loop(m, batches, 2)
        plain, piped, sub = [], [], []
        for _ in range(args.rounds):
            ms, out_plain = plain_loop(m, batches, args.steps)
            plain.append(ms)
            ms, sub_ms, out_piped = submit_loop(m, batches, args.steps)
            piped.append(ms)
            sub.append(sub_ms)
        rpn = rpn_times(m, batches[0], args.rpn_iters)
    same = all(torch.equal(a["instances"].pred_boxes.tensor, b["instances"].pred_boxes.tensor)
               and torch.equal(a["instances"].scores, b["instances"].scores) for a, b in zip(out_plain, out_piped))
    pm, qm = statistics.median(plain), statistics.median(piped)
    res = {"workload": f"FsodRCNN R50-C4 (Base-FSOD-C4.yaml), 2-way, batch {args.batch} x {args.size}x{args.size}, "
                       f"pinned host images, {args.steps} batches per loop, {args.rounds} alternating rounds",
           "gpu": info,
           "plain_ms_per_batch": pm, "plain_images_per_s": args.batch / (pm * 1e-3), "plain_ms_rounds": plain,
           "submit_ahead_ms_per_batch": qm, "submit_ahead_images_per_s": args.batch / (qm * 1e-3), "submit_ahead_ms_rounds": piped,
           "submit_host_ms": statistics.median(sub),
           "last_batch_results_equal": same,
           "rpn_selection_ms_per_class": rpn}
    line = json.dumps(res)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
