#!/usr/bin/env python
"""Benchmark of the B200 detection head (BASELINE.json metric: query images/sec, VoVNet FSOD, 640x640).

    python bench.py --gpus N --steps K --warmup W          # this repo's CUDA path
    python bench.py --impl reference [...]                 # the reference's CPU path (oracle port) on host cores
    python bench.py [...] --dump-outputs DIR               # + the detections of the last timed step as DIR/<name>.npy

One step = one pass of the whole detector (backbone + support-guided head) over one batch of
synthetic 640x640 ore-shaped query images, 1-way 25-shot, random-init (synthetic) weights.
Prints ONE JSON line (rank 0).  See DESIGN.md "Measurement" for every field.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import torch  # noqa: E402

from faster_orefsdet_b200 import synth  # noqa: E402

def _ncu_traffic():
    """DRAM bytes per launch (dram__bytes_read.sum + dram__bytes_write.sum) of the kernels, from the committed summary
    of the `ncu --set full` captures (profiles/traffic.json, written by tools/ncu_summary.py next to the capture it
    came from): {"kernels": {name: bytes}, "conv_layers": {"H,W,Cin,Cout,k,s": bytes}, "batch": 64, "source": ...}."""
    p = os.path.join(ROOT, "profiles", "traffic.json")
    if not os.path.exists(p):
        return {"kernels": {}, "conv_layers": {}, "batch": None, "source": None}
    with open(p) as f:
        return json.load(f)


HEAD_KERNELS = ("correlate_levels", "decode_topk", "nms_proposals", "roi_align", "relation_head", "roi_relation_head",
                "final_detect")
METRIC = "query_images_per_sec"
UNIT = "images/s"
IMG = 640
SHOTS = 25
BATCH = 64            # BASELINE.json configs[1]
M_PIXELS = 8400       # p3+p4+p5 pixels at 640x640


def _peaks():
    """(HBM GB/s, dense bf16 TFLOP/s sustained, source).  The sustained tensor figure is the one for a kernel timed
    inside a long step (B200_PROFILING.md)."""
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            d = json.load(f)
        return float(d["hbm_gbs"]), float(d.get("bf16_tflops_sustained", d.get("bf16_tflops", 1410.0))), "measured (MEASURED_PEAKS.json)"
    return 6650.0, 1410.0, "fallback (B200_PROFILING.md)"


def _cfg(device):
    from faster_orefsdet_b200.config import get_cfg
    cfg = get_cfg()
    cfg.merge_from_file(os.path.join(ROOT, "configs/fsod/finetune_vovnet.yaml"))
    cfg.merge_from_list(["MODEL.DEVICE", device, "INPUT.FS.SUPPORT_SHOT", SHOTS])
    return cfg


def _workload(batch):
    """The workload both arms are measured on (BASELINE.json configs[1])."""
    return (f"finetune_vovnet.yaml 1-way {SHOTS}-shot inference, batch {batch} synthetic 640x640 ore queries per GPU "
            f"(BASELINE.json configs[1])")


def _images(batch, seed0, n_distinct=8):
    base = [synth.ore_image(IMG, IMG, seed0 + i) for i in range(n_distinct)]
    out = []
    for i in range(batch):           # distinct content per slot: roll a base image
        out.append(torch.roll(base[i % n_distinct], shifts=(7 * (i // n_distinct), 13 * (i // n_distinct)), dims=(1, 2)))
    return out


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled while the timed region runs."""

    def __init__(self, index):
        self.index, self.proc, self.lines = index, None, []

    def start(self):
        q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
             "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
             "clocks_event_reasons.sw_power_cap")
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader,nounits", "-lms", "100",
                                          "-i", str(self.index)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except OSError:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        sm, mx, reasons = [], [], set()
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 8:
                continue
            try:
                sm.append(float(f[0]))
                mx.append(float(f[1]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[4:8]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


# ------------------------------------------------------------------------------------------ CPU arm
def cpu_reference_rate(n_images, warmup, threads):
    """The reference's CPU path restated (oracle/ head + the same VoVNet/FPN module on CPU), batch-1
    loop like the reference (fewx/data/build.py:195, fsod_cen.py:438).  Returns images/s."""
    from faster_orefsdet_b200.modeling import META_ARCH_REGISTRY
    from oracle import head_oracle as O
    torch.set_num_threads(threads)
    cfg = _cfg("cuda")
    # the detector is only constructed (on the host) for its backbone module and parameter shapes;
    # its CUDA head is never called here
    det = META_ARCH_REGISTRY.get(cfg.MODEL.META_ARCHITECTURE)(cfg).eval()
    sd = synth.state_dict({k: tuple(v.shape) for k, v in det.state_dict().items()})
    det.load_state_dict(sd)
    backbone = det.backbone
    protos = synth.prototypes([1], SHOTS, 7)
    ocfg = O.HeadConfig()
    mean = torch.tensor(cfg.MODEL.PIXEL_MEAN).view(3, 1, 1)
    imgs = _images(n_images + warmup, 1000)
    t0 = None
    with torch.no_grad():
        for i, im in enumerate(imgs):
            if i == warmup:
                t0 = time.perf_counter()
            feats = backbone(((im.float() - mean) / 1.0).unsqueeze(0))
            O.detect_image(feats, protos, sd, (IMG, IMG), ocfg)
    dt = time.perf_counter() - t0
    return n_images / dt, dt


def run_reference_arm(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    threads = len(os.sched_getaffinity(0))
    per_step = 16                                 # bounded sample: images per step (~1 s of host work per step)
    rate, dt = cpu_reference_rate(per_step * args.steps, min(args.warmup, 2), threads)
    line = {
        "impl": "reference", "metric": METRIC, "value": rate, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": dt / args.steps * 1e3, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": _workload(BATCH), "batch_per_gpu": BATCH, "ways": 1, "shots": SHOTS,
                   "execution": "reference CPU path (MODEL.DEVICE=cpu semantics): batch-1 loop on the host cores, oracle head + "
                                "PyTorch-CPU VoVNet/FPN",
                   "sample": f"{per_step} images of the workload per step"},
        "cpu_baseline": {"value": rate, "unit": UNIT, "cores": threads, "kind": "port",
                         "sample": f"{per_step * args.steps} images 640x640, batch-1 loop, oracle head + PyTorch-CPU VoVNet/FPN"},
        "e2e": {"value": rate, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line))


# ------------------------------------------------------------------------------------------ GPU arm
class KernelTimer:
    """CUDA-event timing of every C-ABI launch on torch's current stream."""

    def __init__(self):
        self.records = {}
        self.launches = 0
        self.enabled = False

    # kernels of this library per C-ABI call (memsets are not counted)
    kernels_per_call = {"group_norm_nhwc": 2, "roi_align": 3, "decode_topk_taps": 2}   # statistics + apply; tap tables + tile pooling + per-ROI list; keys + select

    def wrap(self, ops_mod, names):
        for n in names:
            fn = getattr(ops_mod, n)

            def timed(*a, __fn=fn, __n=n, **k):
                if not self.enabled:
                    return __fn(*a, **k)
                s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                # keep the GPU busy (~0.2 ms spin) while the host enqueues this call's launches, so that the two events
                # bracket kernel time and not the host's launch latency (this pass is eager; the timed region is a graph)
                torch.cuda._sleep(400_000)
                s.record()
                r = __fn(*a, **k)
                e.record()
                tag = None
                if __n in ("conv2d_nhwc", "conv2d_nhwc_split"):      # (N, H, W, Cin, Cout, ksize, stride) of this layer
                    x = a[0]
                    tag = (x.shape[0], x.shape[2], x.shape[3], x.shape[1], int(a[3]), int(a[4]), int(k.get("stride", 1)))
                self.records.setdefault({"decode_topk_taps": "decode_topk", "conv2d_nhwc_split": "conv2d_nhwc"}.get(__n, __n), []).append((s, e, tag))
                self.launches += self.kernels_per_call.get(__n, 1)
                return r
            setattr(ops_mod, n, timed)

    def summary(self):
        return {n: (sum(s.elapsed_time(e) for s, e, _ in ev), len(ev)) for n, ev in self.records.items()}

    def conv_layers(self):
        """per layer shape: [total ms, launches, flops per launch] (2*N*Ho*Wo*Cin*Cout*k*k, fp32 convolution flops)"""
        out = {}
        for s, e, tag in self.records.get("conv2d_nhwc", []):
            n, h, w, cin, cout, ks, st = tag
            ho, wo = (h - 1) // st + 1, (w - 1) // st + 1
            ent = out.setdefault(tag, [0.0, 0, 2.0 * n * ho * wo * cin * cout * ks * ks])
            ent[0] += s.elapsed_time(e)
            ent[1] += 1
        return out


def fsodrcnn_record(dev, steps):
    """SURVEY 8f#3, the R50-C4 FsodRCNN path (Base-FSOD-C4.yaml: attention RPN, 1000 -> 100 proposals, relation head):
    model(batched_inputs) on 16 synthetic 640x640 images already on the device, 2-way episode, timed with CUDA events
    after three warm-up calls; parity of this path is pinned by tests/test_fsodrcnn_gpu.py."""
    from faster_orefsdet_b200.compat import META_ARCH_REGISTRY
    from faster_orefsdet_b200.config import get_cfg
    import faster_orefsdet_b200.modeling  # noqa: F401
    cfg = get_cfg()
    cfg.merge_from_file(os.path.join(ROOT, "configs/fsod/Base-FSOD-C4.yaml"))
    cfg.merge_from_list(["MODEL.DEVICE", str(dev)])
    m = META_ARCH_REGISTRY.get("FsodRCNN")(cfg).to(dev).eval()      # (detectron2's build_model does the .to())
    m.load_state_dict(synth.state_dict({k: tuple(v.shape) for k, v in m.state_dict().items()}))
    sup = {"res4_avg": {}, "res5_avg": {}}
    for j, c in enumerate((3, 9)):
        sup["res4_avg"][c] = synth.tensor((1, 1024, 14, 14), 341 + 2 * j, 0.0, 1.2)
        sup["res5_avg"][c] = synth.tensor((1, 2048, 7, 7), 342 + 2 * j, 0.0, 1.0)
    m.set_prototypes(sup)
    nb = 16
    batches = [[{"image": synth.ore_image(IMG, IMG, 7000 + 17 * k + i).to(dev)} for i in range(nb)] for k in range(2)]
    with torch.no_grad():
        for k in range(3):
            out = m(batches[k % 2])
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for k in range(steps):
            out = m(batches[k % 2])
        e1.record()
        torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / steps
    return {"workload": f"FsodRCNN R50-C4 (Base-FSOD-C4.yaml), 2-way episode, batch {nb} x {IMG}x{IMG}, through model(batched_inputs)",
            "ms_per_step": ms, "images_per_s": nb / (ms * 1e-3), "steps": steps,
            "detections": int(sum(len(o["instances"]) for o in out))}


DUMP_LIMIT_BYTES = 64 << 20


def dump_outputs(out_dir, arrays):
    """Writes each host tensor as out_dir/<name>.npy, float32 kept and integers widened to float64 (exact), so that two
    builds can be compared output for output on the same seeded inputs."""
    import numpy as np
    arrays = {n: v.numpy() if v.dtype == torch.float32 else v.numpy().astype(np.float64) for n, v in arrays.items()}
    total = sum(a.nbytes for a in arrays.values())
    if total > DUMP_LIMIT_BYTES:
        raise SystemExit(f"--dump-outputs: {total} bytes of detections exceed {DUMP_LIMIT_BYTES}; use a smaller --batch")
    os.makedirs(out_dir, exist_ok=True)
    for n, a in arrays.items():
        np.save(os.path.join(out_dir, n + ".npy"), a)


def run_gpu_arm(args):
    import torch.distributed as dist
    from faster_orefsdet_b200 import ops
    from faster_orefsdet_b200.modeling import build_model

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    B = args.batch
    model = build_model(_cfg(f"cuda:{local}")).eval()
    shapes = {k: tuple(v.shape) for k, v in model.state_dict().items()}
    model.load_state_dict(synth.state_dict(shapes))

    # prototypes: rank 0 owns the episode, one NCCL broadcast hands it to the other ranks
    bcast_ms = 0.0
    if rank == 0:
        model.set_prototypes(synth.prototypes([1], SHOTS, 7))
    if world > 1:
        torch.cuda.synchronize()
        dist.barrier()
        t0 = time.perf_counter()
        model.sync_prototypes(0)
        torch.cuda.synchronize()
        bcast_ms = (time.perf_counter() - t0) * 1e3

    # inputs: NSETS distinct batches so consecutive steps never re-read the same bytes from L2
    NSETS = 4
    host_sets = [[im.pin_memory() for im in _images(B, 1000 + 100 * s + 17 * rank)] for s in range(NSETS)]
    dev_sets = [torch.stack(hs).to(dev) for hs in host_sets]
    sizes = [(IMG, IMG)] * B
    timer = KernelTimer()
    timer.wrap(ops, ["correlate_levels", "decode_topk", "decode_topk_taps", "group_norm_affine", "nms_proposals", "roi_align", "relation_head", "final_detect",
                     "conv2d_nhwc", "conv2d_nhwc_split", "group_norm_nhwc", "stem_patches", "stem_patches_u8", "stem1_u8", "stem1_u8_tc", "maxpool3x3s2_nhwc", "ese_gate"])

    def step_resident(i):      # raw uint8 images resident in HBM -> padded detections on the device
        return model.detect_from_uint8(dev_sets[i % NSETS], sizes, sizes)

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize()

    with torch.no_grad():
        for i in range(args.warmup):
            out = step_resident(i)
        if world > 1:     # the job's final gather once untimed as well: NCCL sets its channels up lazily on the first call
            packed = torch.cat((out[0], out[1].unsqueeze(-1), out[2].unsqueeze(-1).float()), -1)
            dist.all_gather([torch.empty_like(packed) for _ in range(world)], packed)
        barrier()
        clocks = ClockSampler(local)
        if rank == 0:
            clocks.start()
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        ev0.record()
        for i in range(args.steps):
            out = step_resident(args.warmup + i)
        if world > 1:     # detections are gathered once at the end (fixed-size padded block per image)
            packed = torch.cat((out[0], out[1].unsqueeze(-1), out[2].unsqueeze(-1).float()), -1)
            gathered = [torch.empty_like(packed) for _ in range(world)]
            dist.all_gather(gathered, packed)
        ev1.record()
        barrier()
        clk = clocks.stop() if rank == 0 else None
        ms = ev0.elapsed_time(ev1)
        # what the caller of the timed path received from its last step, copied out before a later replay can reuse
        # the graph's output buffers
        last = dict(zip(("boxes", "scores", "classes", "counts"), (v.cpu() for v in out))) \
            if args.dump_outputs and rank == 0 else None
        # Per-kernel durations: the timed region replays one CUDA graph per step, inside which events cannot be read,
        # so the same K steps are re-run eagerly right here (same inputs, same kernels, same launch parameters) with
        # CUDA events around every C-ABI call on torch's current stream.
        graph_mode = model.USE_CUDA_GRAPH
        model.USE_CUDA_GRAPH = False
        step_resident(0)
        timer.enabled = True
        for i in range(args.steps):
            step_resident(args.warmup + i)
        torch.cuda.synchronize()
        timer.enabled = False
        model.USE_CUDA_GRAPH = graph_mode
        ksum = timer.summary()
        launches = timer.launches
        layers = timer.conv_layers()

        # ---- end-to-end through the public API: host images in, host detections out.  Every step copies its 64 pinned
        # host images to the device and reads its detections back, all inside the timed region.  `pipelined`: the serving
        # loop of INTEGRATION.md - model.submit(batch k+1) starts the next batch's copies before model(staged k) runs, so
        # the PCIe transfer rides under the current batch's kernels; `serial`: model(batched_inputs) alone, each call
        # waits for its own copies first.
        from faster_orefsdet_b200.modeling import roi_heads as _rh
        inputs = [[{"image": im} for im in hs] for hs in host_sets]

        def consume(res):
            n_det = 0
            for r in res:
                inst = r["instances"].to("cpu")          # host views of the one padded transfer the detector made
                n_det += len(inst.scores)
            return _rh.LAST_D2H_BYTES + 4                # + the head's status word

        def run_e2e(n_steps, first, pipelined):
            d2h = 0
            if not pipelined:
                for i in range(n_steps):
                    d2h = consume(model(inputs[(first + i) % NSETS]))
                return d2h
            nxt = model.submit(inputs[first % NSETS])
            for i in range(n_steps):
                cur = nxt
                if i + 1 < n_steps:
                    nxt = model.submit(inputs[(first + i + 1) % NSETS])
                d2h = consume(model(cur))
            return d2h

        e2e = {}
        for mode in ("serial", "pipelined"):
            run_e2e(max(args.warmup, 3), 0, mode == "pipelined")
            barrier()
            t0 = time.perf_counter()
            d2h_bytes = run_e2e(args.steps, args.warmup, mode == "pipelined")
            barrier()
            e2e[mode] = time.perf_counter() - t0
        e2e_s = e2e["pipelined"]

        # ---- the other BASELINE.json configurations as sub-records (N = 1 only; outside the headline region; parity for
        # the same shapes is pinned by tests/test_model_gpu.py::test_config3_* / test_config4_*)
        cfg_records = {}
        if world == 1 and not args.no_configs:
            pg = model.proposal_generator
            keep = (pg.pre_nms_topk_test, pg.post_nms_topk_test)
            for name, (cb, ch, cw, ways, shots, pre, post) in (
                    ("C3", (32, IMG, IMG, 10, 10, keep[0], keep[1])),      # 10 ways x 10 shots, batch 32, 640x640
                    ("C4", (16, 800, 1344, 1, SHOTS, 2000, 2000))):        # 1333x800 (padded 800x1344), top-k 2000, batch 16
                pg.pre_nms_topk_test, pg.post_nms_topk_test = pre, post
                model.set_prototypes(synth.prototypes(list(range(1, ways + 1)), shots, 7))
                xs = [torch.stack([synth.ore_image(ch, cw, 5000 + 31 * k + i) for i in range(4)]).repeat(cb // 4, 1, 1, 1).to(dev)
                      for k in range(2)]
                for k in range(2):          # distinct content per slot
                    for i in range(cb):
                        xs[k][i] = torch.roll(xs[k][i], shifts=(5 * (i // 4), 11 * (i // 4)), dims=(1, 2))
                szs = [(ch, cw)] * cb
                for k in range(3):
                    model.detect_from_uint8(xs[k % 2], szs, szs)
                torch.cuda.synchronize()
                c0, c1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                n_cfg = max(args.steps // 2, 3)
                c0.record()
                for k in range(n_cfg):
                    res = model.detect_from_uint8(xs[k % 2], szs, szs)
                c1.record()
                torch.cuda.synchronize()
                cms = c0.elapsed_time(c1) / n_cfg
                # head kernels of this configuration, eagerly with events (same method as the headline's per-kernel table)
                model.USE_CUDA_GRAPH = False
                model.detect_from_uint8(xs[0], szs, szs)
                timer.records, timer.enabled = {}, True
                for k in range(3):
                    model.detect_from_uint8(xs[k % 2], szs, szs)
                torch.cuda.synchronize()
                timer.enabled = False
                model.USE_CUDA_GRAPH = graph_mode
                hk = {n: tot / 3 for n, (tot, cnt) in timer.summary().items() if n in HEAD_KERNELS}
                cfg_records[name] = {"workload": f"{ways}-way {shots}-shot, batch {cb} x {ch}x{cw}, PRE/POST_NMS_TOPK {pre}/{post}",
                                     "ms_per_step": cms, "images_per_s": cb / (cms * 1e-3), "steps": n_cfg,
                                     "detections": int(res[3].sum()), "head_ms_per_step": sum(hk.values()), "head_kernels_ms": hk}
                del xs
            pg.pre_nms_topk_test, pg.post_nms_topk_test = keep
            model.set_prototypes(synth.prototypes([1], SHOTS, 7))
            cfg_records["FsodRCNN"] = fsodrcnn_record(dev, max(args.steps // 2, 3))

        # ---- BASELINE.json configs[4] as written (strong scaling): ONE global batch of 256 queries sharded 256 / G with the
        # InferenceSampler formula (d2!/data/samplers/distributed_sampler.py:191-194), prototypes broadcast by rank 0 and the
        # padded detections of all ranks gathered (fewx/evaluation/coco_evaluation.py:131-137) INSIDE the timed region
        strong = None
        if not args.no_strong:
            from faster_orefsdet_b200 import dist_utils
            G = 256
            lo, hi = dist_utils.shard_range(G, rank, world)
            nb = hi - lo
            shard_sets = [torch.stack(_images(G, 7000 + 100 * k)[lo:hi]).to(dev) for k in range(2)]
            ssz = [(IMG, IMG)] * nb

            def strong_steps(n_steps):
                tot = None
                for k in range(n_steps):
                    ob, os_, ocls, oc = model.detect_from_uint8(shard_sets[k % 2], ssz, ssz)
                    if world > 1:
                        ob, os_, ocls, oc = dist_utils.gather_detections(ob, os_, ocls, oc, G)
                    tot = oc
                return tot

            strong_steps(3)
            barrier()
            # the episode: rank 0 broadcasts the prototypes (NCCL); a new bank means new device buffers and new tap values
            # baked into launch parameters, so the first step after it re-captures the CUDA graph - timed as `setup`
            s0, s1, s2 = (torch.cuda.Event(enable_timing=True) for _ in range(3))
            n_strong = max(args.steps, 4) // 2 * 2          # even: the last step always runs input set 1
            s0.record()
            if world > 1:
                model.sync_prototypes(0)
            strong_steps(1)
            s1.record()
            tot = strong_steps(n_strong)
            s2.record()
            barrier()
            strong = {"n_det": int(tot.sum()), "n_img": int(tot.numel()), "batch_per_gpu": nb, "steps": n_strong,
                      "ms": s1.elapsed_time(s2), "setup_ms": s0.elapsed_time(s1)}
            del shard_sets

    vals = [ms, e2e_s * 1e3, e2e["serial"] * 1e3, strong["ms"] if strong else 0.0, strong["setup_ms"] if strong else 0.0]
    t = torch.tensor(vals, dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms, e2e_ms, e2e_serial_ms = float(t[0]), float(t[1]), float(t[2])
    if strong:
        strong["ms"], strong["setup_ms"] = float(t[3]), float(t[4])
    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    peak, tensor_peak, peak_src = _peaks()
    traffic = _ncu_traffic()
    # algorithmic bytes per launch (DESIGN.md "Measurement"; SURVEY section 8d), 1-way, B images of 640x640
    lvl_px = [6400, 1600, 400]
    alg = {
        "correlate_levels": 1024.0 * M_PIXELS * B,          # one persistent launch over the three levels
        "decode_topk": (20.0 * M_PIXELS + 28.0 * 2400) * B,
        "nms_proposals": (20.0 * 2400 + 8.0 * 256) * B,
        "roi_align": (512.0 * M_PIXELS + 16.0 * 256 + 256 * 32768.0) * B,   # + pooled rows, materialised while R1/R2 are two kernels
        "relation_head": (256 * 32768.0 + 40.0 * 256) * B + 2 * 4.19e6,    # pooled rows + tf32 hi/lo weight planes
        "final_detect": 20.0 * 256 * B,
    }
    kernels, extractor = {}, {}
    for n, (tot_ms, cnt) in ksum.items():
        per_launch_ms = tot_ms / max(cnt, 1)
        if n not in alg:      # feature-extractor kernels (convolutions on the tensor cores and their memory-bound glue)
            extractor[n] = {"ms_per_step": tot_ms / args.steps, "launches_per_step": cnt / args.steps}
            continue
        gbs = alg[n] / (per_launch_ms * 1e-3) / 1e9
        kernels[n] = {"ms_per_step": tot_ms / args.steps, "launches_per_step": cnt / args.steps,
                      "achieved_gbs": gbs, "frac": gbs / peak}
    # the convolution kernel: per layer shape, and the launch with the largest share of the step
    conv_ms = sum(v[0] for v in layers.values()) / args.steps
    conv_flops = sum(v[2] * v[1] for v in layers.values()) / args.steps
    top = max(layers, key=lambda t: layers[t][0]) if layers else None
    conv_roof = None
    if top is not None:
        t_ms, cnt, fl = layers[top]
        ach = fl / (t_ms / cnt * 1e-3) / 1e12
        # fp32-accurate arithmetic on the tensor cores = 3 fp16 MMAs per product (hi.hi + lo.hi + hi.lo), fp16 runs at the
        # bf16 rate: the ceiling of this arithmetic is peak / 3
        conv_roof = {"bound": "tensor", "kernel": "conv_tc_kernel (fod_conv2d_nhwc)",
                     "launch": "N%d %dx%d %d->%d k%d s%d" % top, "achieved": ach, "peak": tensor_peak, "unit": "TFLOP/s",
                     "frac": ach / tensor_peak,
                     "traffic": traffic["conv_layers"].get(",".join(str(v) for v in top[1:])) if B == traffic["batch"] else None,
                     "algorithmic_flops": fl, "issued_f16_tflops": 3 * ach, "frac_of_split_ceiling": ach / (tensor_peak / 3),
                     "all_layers": {"ms_per_step": conv_ms, "launches_per_step": sum(v[1] for v in layers.values()) / args.steps,
                                    "achieved": conv_flops / (conv_ms * 1e-3) / 1e12, "frac": conv_flops / (conv_ms * 1e-3) / 1e12 / tensor_peak},
                     "peak_source": peak_src + ", dense bf16 sustained"}
        extractor["conv2d_nhwc"]["fp32_tflops"] = conv_flops / (conv_ms * 1e-3) / 1e12
        # the layers by their share of the step (shape, launches per step, ms per step, fp32-equivalent TFLOP/s)
        extractor["conv2d_nhwc"]["layers"] = [
            {"shape": "N%d %dx%d %d->%d k%d s%d" % tag, "launches": v[1] / args.steps, "ms_per_step": v[0] / args.steps,
             "tflops": v[2] / (v[0] / v[1] * 1e-3) / 1e12}
            for tag, v in sorted(layers.items(), key=lambda kv: -kv[1][0])]
    # DRAM traffic per launch of the same kernels from the committed `ncu --set full` captures
    # (dram__bytes_read.sum + dram__bytes_write.sum, batch 64, 1-way; profiles/r1_ncu_v2_summary.md)
    ncu_traffic = traffic["kernels"] if B == traffic["batch"] else {}
    dom = max(kernels, key=lambda n: kernels[n]["ms_per_step"])
    head_ms = sum(k["ms_per_step"] for k in kernels.values())
    head_alg_bytes = 13.2e6 * B
    cpu_threads = len(os.sched_getaffinity(0))
    cpu_rate, cpu_dt = (None, None)
    if world == 1 and not args.no_cpu_baseline:
        cpu_rate, cpu_dt = cpu_reference_rate(args.cpu_images, 2, cpu_threads)
    total_images = B * world * args.steps
    line = {
        "metric": METRIC, "value": total_images / (ms * 1e-3), "unit": UNIT, "n_gpus": world, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": _workload(B), "batch_per_gpu": B, "ways": 1, "shots": SHOTS,
                   "implementation": "VoVNet-19-slim-eSE+FPN + CenterNetHead convolutions on tcgen05 (fp16-split operands, 3 MMAs "
                                     "per product = fp32 accuracy) + CUDA head",
                   "l2": f"inputs rotate over {NSETS} distinct batches ({NSETS * B * 3 * IMG * IMG / 1e6:.0f} MB) and the "
                         f"backbone activations (> 1 GB per step) exceed the 126 MB L2",
                   "execution": ("stem eager, everything behind it one CUDA-graph replay per step" if graph_mode else "eager") +
                                "; per-kernel durations from an eager re-run of the same steps inside this process",
                   "parallelism": f"query batch sharded, {world} rank(s); prototypes broadcast once "
                                  f"({bcast_ms:.2f} ms, outside the timed region), detections all-gathered once at the end"},
        "e2e": {"value": total_images / (e2e_ms * 1e-3), "unit": UNIT, "h2d_bytes_per_step": B * 3 * IMG * IMG,
                "d2h_bytes_per_step": d2h_bytes,
                "api": "staged = model.submit(next batched_inputs) [async H2D of the next batch from pinned host uint8 images]; "
                       "model(staged) -> Instances.to('cpu'); every step's H2D and D2H lie inside the timed region",
                "serial": {"value": total_images / (e2e_serial_ms * 1e-3), "unit": UNIT,
                           "api": "model(batched_inputs) alone: copies, kernels, transfer and Instances of one batch in series"}},
        "gpu_launches": launches,
        # The path north_star names is the HEAD: `roofline` is its dominant kernel (largest share of the head's time)
        # against the HBM roof; the step-dominant kernel overall is the feature extractor's tensor-core convolution
        # (an "(f)" row of SURVEY section 8), reported under `step_dominant` against the tensor roof.
        "roofline": {"bound": "hbm", "kernel": dom, "achieved": kernels[dom]["achieved_gbs"], "peak": peak, "unit": "GB/s",
                     "frac": kernels[dom]["frac"], "traffic": ncu_traffic.get(dom), "algorithmic_bytes": alg[dom],
                     "ms_per_launch": kernels[dom]["ms_per_step"] / max(kernels[dom]["launches_per_step"], 1),
                     "scope": "dominant kernel of the support-guided head (the hot path)", "peak_source": peak_src,
                     "traffic_source": traffic.get("source")},
        "step_dominant": conv_roof,
        "head": {"ms_per_step": head_ms, "images_per_s": B / (head_ms * 1e-3),
                 "achieved_gbs": head_alg_bytes / (head_ms * 1e-3) / 1e9, "frac": head_alg_bytes / (head_ms * 1e-3) / 1e9 / peak,
                 "share_of_step": head_ms / (ms / args.steps), "kernels": kernels,
                 "dominant_hbm_kernel": {"kernel": dom, "achieved": kernels[dom]["achieved_gbs"], "peak": peak, "unit": "GB/s",
                                         "frac": kernels[dom]["frac"], "traffic": ncu_traffic.get(dom),
                                         "algorithmic_bytes": alg[dom]}},
        "feature_extractor": extractor,
        "clocks": clk,
    }
    if cfg_records:
        line["configs"] = cfg_records
    if strong:
        sm = strong["ms"] / strong["steps"]
        line["strong"] = {"workload": "BASELINE.json configs[4]: one global batch of 256 synthetic 640x640 queries sharded 256/G "
                                      "(InferenceSampler formula); every step all-gathers the padded detections of all ranks; "
                                      "episode_setup_ms = NCCL prototype broadcast + the first step behind it (which "
                                      "re-captures the CUDA graph for the new bank), once per episode",
                          "global_batch": 256, "batch_per_gpu": strong["batch_per_gpu"], "steps": strong["steps"],
                          "ms_per_step": sm, "images_per_s": 256 / (sm * 1e-3), "scaling": "strong",
                          "episode_setup_ms": strong["setup_ms"],
                          "images_per_s_incl_setup": 256 * strong["steps"] / ((strong["ms"] + strong["setup_ms"]) * 1e-3),
                          "images_gathered": strong["n_img"], "detections": strong["n_det"]}
    if cpu_rate is not None:
        line["cpu_baseline"] = {"value": cpu_rate, "unit": UNIT, "cores": cpu_threads, "kind": "port",
                                "sample": f"{args.cpu_images} images 640x640 after 2 warm-up, batch-1 loop, oracle head + "
                                          f"PyTorch-CPU VoVNet/FPN, {cpu_dt:.1f} s"}
    if last is not None:
        dump_outputs(args.dump_outputs, last)
    print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--batch", type=int, default=BATCH)
    ap.add_argument("--cpu-images", type=int, default=200)      # ~12 s of host work on 16 cores
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-configs", action="store_true", help="skip the C3 / C4 sub-records")
    ap.add_argument("--no-strong", action="store_true", help="skip the strong-scaling (global batch 256) sub-record")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the padded detections of the last timed step (rank 0) as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.impl == "reference":
        run_reference_arm(args)
    else:
        run_gpu_arm(args)


if __name__ == "__main__":
    main()
