#!/usr/bin/env python
"""Images/s of the batched test-time path (fused.InferHotPath, SURVEY 3.2): RPN proposals at the test configuration
(1000 / 1000 / 1000) -> per stage FPN RoIAlign of the 1000 boxes per image -> arg-max refine between stages ->
detections (softmax, per-class decode, class-offset NMS, top 100) with packed records.

  python scripts/bench_infer.py --gpus 1 --stages 1 3 --steps 50 --warmup 5
  python scripts/bench_infer.py --gpus 2 ...           # re-launches itself under torch.distributed.run

Workload: config-2 geometry (batch 8 per GPU, 800x1333 padded to 800x1344, fp32 NHWC 256-channel FPN maps, RPN maps
as bench.py draws them).  The RCNN heads' convolutions / FCs stay out of the timed region: each stage's head returns
fixed synthetic outputs drawn with the config-1 recipe (logits N(0, 2.5) with +2 on the background, deltas N(0, 0.5)).
The feature maps (731 MB per step) exceed the 126 MB L2, so no flush is needed between steps.

Reported per stage count: the CUDA-graph step time (median of per-step CUDA events), images/s, kernel launches per step
(an eager step under torch.profiler), the phase split from an event-bracketed eager step (proposals, RoIAlign per
stage, refine, detect) with the device kernel times of the detect phase, candidate and detection counts per image,
RoIAlign bytes against a measured HBM rate, and the reference's own per-image call sequence on the drop-in functions
(rpn_predict_single_image -> BasicRoIExtractor -> refine_bboxes_single_image -> predict_bboxes_single_image) on the
same inputs.  With --gpus N the records are all-gathered (dist.gather_detections) inside the timed loop.  One JSON line.
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

B = 8
NC = 21
ROI_BYTES = 256 * 7 * 7 * 4                       # one RoI's fp32 output: 50 176 B
HBM_GBS = 6544.0                                  # B200 HBM copy rate measured by torch copy_ of 1 Gi bf16 (BASELINE.md)
RPN_TEST = dict(pre_nms=1000, post_nms=1000, max_num=1000, nms_iou=0.7, min_bbox_size=0)
RCNN_TEST = dict(min_score=0.05, nms_iou=0.5, max_per_img=100, nms_type="official")
STDS = ((0.1, 0.1, 0.2, 0.2), (0.05, 0.05, 0.1, 0.1), (0.033, 0.033, 0.067, 0.067))


def gpu_info(index):
    q = "name,power.limit,clocks.max.sm"
    try:
        out = subprocess.run(["nvidia-smi", "-i", str(index), "--query-gpu=" + q, "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=20).stdout.strip()
        name, power, clk = [v.strip() for v in out.split(",")]
        return dict(name=name, power_limit=power, sm_max_clock=clk)
    except Exception as e:                                              # report, do not guess
        return dict(error="nvidia-smi query failed: %s" % e)


def head_outputs(torch, dev, P, stages, seed):
    rng = np.random.default_rng(seed)
    outs = []
    for _ in range(stages):
        cls = rng.normal(0, 2.5, (B * P, NC)).astype(np.float32)
        cls[:, 0] += 2.0
        reg = rng.normal(0, 0.5, (B * P, 4 * NC)).astype(np.float32)
        outs.append((torch.from_numpy(cls).to(dev), torch.from_numpy(reg).to(dev)))
    return outs


def run_stages(S, args, torch, dev, rank, world, w, cls, reg, feats, img_hw):
    from b200det import dist as bdist, fused
    hp = fused.InferHotPath(B, w["grids"], dev, feat_channels=256, num_classes=NC, num_stages=S, rpn_test=RPN_TEST,
                            rcnn_test=RCNN_TEST, stage_stds=STDS)
    P, M = hp.P, hp.M
    fixed = head_outputs(torch, dev, P, S, seed=2019 + 31 + rank)
    heads = [(lambda x, t=t: t) for t in fixed]
    rec = torch.zeros((B, M, 6), dtype=torch.float32, device=dev)
    step = lambda: hp.step(cls, reg, feats, img_hw, heads, records=rec)
    for _ in range(max(args.warmup, 2)):
        out = step()
    hp.check()
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(graph, stream=side):
            out = step()
    torch.cuda.current_stream().wait_stream(side)
    for _ in range(3):
        graph.replay()
    torch.cuda.synchronize()

    def one():
        graph.replay()
        if world > 1:
            bdist.gather_detections(rec, hp.det_count)

    def barrier():
        if world > 1:
            torch.distributed.barrier()
        torch.cuda.synchronize()

    # ---- step time: per-step CUDA events around graph replays (+ the all-gather when N > 1)
    barrier()
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
    for a, b in ev:
        a.record()
        one()
        b.record()
    barrier()
    per = np.array([a.elapsed_time(b) for a, b in ev])
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    e0.record()
    for _ in range(args.steps):
        one()
    e1.record()
    barrier()
    back_to_back = e0.elapsed_time(e1) / args.steps
    hp.check()
    ms = float(np.median(per))

    # ---- phase split: event-bracketed eager steps (launch gaps included)
    names, split = None, []
    for _ in range(10):
        marks = []
        start = torch.cuda.Event(enable_timing=True)
        start.record()

        def mark(name):
            e = torch.cuda.Event(enable_timing=True)
            e.record()
            marks.append((name, e))
        hp.step(cls, reg, feats, img_hw, heads, records=rec, mark=mark)
        torch.cuda.synchronize()
        names = [n for n, _ in marks]
        prev, row = start, []
        for _, e in marks:
            row.append(prev.elapsed_time(e))
            prev = e
        split.append(row)
    split = np.median(np.array(split), 0)
    phases = {n: float(v) for n, v in zip(names, split) if not n.startswith("head")}     # heads: fixed tensors, ~0
    eager_ms = float(split.sum())

    # ---- launches and device kernel times of one eager step (a profiled run of its own)
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        hp.step(cls, reg, feats, img_hw, heads, records=rec)
        torch.cuda.synchronize()
    kernels, launches = {}, 0
    for e in prof.events():
        if e.device_type != torch.autograd.DeviceType.CUDA:
            continue
        launches += 1
        k = e.name if len(e.name) < 80 else e.name[:77] + "..."
        kernels[k] = kernels.get(k, 0.0) + e.device_time_total           # us
    kernels = dict(sorted(kernels.items(), key=lambda kv: -kv[1]))

    # ---- sizes: proposals, candidates (foreground softmax >= min_score, rows < count), detections
    count = hp.proposals.count.cpu().numpy()
    c_last = fixed[-1][0].view(B, P, NC)
    sm = torch.softmax(c_last, -1)[..., 1:] >= float(np.float32(RCNN_TEST["min_score"]))
    cand = [int(sm[b, :int(count[b])].sum()) for b in range(B)]
    dets = hp.det_count.cpu().numpy()
    rois = int(count.sum())
    roi_bytes = rois * ROI_BYTES
    ra_ms = [phases["roi_align%d" % s] for s in range(S)]

    # ---- the reference's own call sequence on the drop-in functions, eager, image by image
    ref = None
    if not args.no_reference and rank == 0:
        ref = reference_arm(S, torch, dev, w, cls, reg, feats, fixed, P, hp, args)
    return {
        "stages": S, "ms_per_step": ms, "ms_per_step_back_to_back": back_to_back, "value": B * world / (ms / 1e3),
        "unit": "images/s", "per_gpu": B / (ms / 1e3), "steps": args.steps, "step_ms_p10_p90": [float(np.percentile(per, 10)),
                                                                                                 float(np.percentile(per, 90))],
        "launches_per_step": launches, "launches_note": "kernels + memsets of one eager step (torch.profiler)", "eager_ms": eager_ms, "phases_ms": phases,
        "detect_frac_of_graph_step": phases["detect"] / ms, "detect_kernels_us": {k: v for k, v in kernels.items()
                                                                                 if "rcnn" in k or "k_nms" in k},
        "kernels_us": kernels,
        "counts": {"proposals_mean": float(count.mean()), "candidates_mean": float(np.mean(cand)), "candidates_max": int(max(cand)),
                   "detections_mean": float(dets.mean()), "detections_max": int(dets.max())},
        "roi_align": {"bytes_per_roi": ROI_BYTES, "rois_per_stage": rois, "out_bytes_per_stage": roi_bytes,
                      "ms_per_stage": ra_ms, "out_gbs": [roi_bytes / (t / 1e3) / 1e9 for t in ra_ms], "hbm_gbs": HBM_GBS,
                      "out_frac_of_hbm": [roi_bytes / (t / 1e3) / 1e9 / HBM_GBS for t in ra_ms],
                      "note": "output bytes only (feature reads come on top); eager phase times"},
        "reference": ref,
    }


def reference_arm(S, torch, dev, w, cls, reg, feats, fixed, P, hp, args):
    import types
    from b200det import anchor, heads, region
    strides = list(w["strides"])
    creators = [anchor.AnchorCreator(base=s, scales=[8], aspect_ratios=[0.5, 1.0, 2.0]) for s in strides]
    for c in creators:
        c.to(dev)
    rpn = types.SimpleNamespace(anchor_strides=strides, anchor_scales=[8], anchor_ratios=[0.5, 1.0, 2.0], target_means=[0.0] * 4,
                                target_stds=[1.0] * 4, use_sigmoid=True, cls_channels=1, anchor_creators=creators)
    bbox_heads = [types.SimpleNamespace(use_sigmoid=False, reg_class_agnostic=False, num_classes=NC, target_means=[0.0] * 4,
                                        target_stds=list(STDS[s])) for s in range(S)]
    extractor = region.BasicRoIExtractor([dict(type="RoIAlign", spatial_scale=1.0 / st, sampling_ratio=2) for st in strides[:4]],
                                         output_size=(7, 7))
    meta = dict(img_shape=tuple(w["img_shape"]) + (3,), pad_shape=tuple(w["pad_shape"]) + (3,), scale_factor=1.0)

    def one_batch():
        res = []
        anchors = [ac(s, g) for ac, s, g in zip(creators, strides, w["grids"])]
        for b in range(B):
            props, _, _ = heads.rpn_predict_single_image(rpn, [c[b] for c in cls], [r[b] for r in reg], anchors, meta, RPN_TEST)
            for s in range(S):
                k = int(props.shape[1])
                extractor.forward_single_image([f[b] for f in feats], props)
                co, ro = fixed[s][0][b * P:b * P + k], fixed[s][1][b * P:b * P + k]
                if s + 1 < S:
                    props = heads.refine_bboxes_single_image(bbox_heads[s], props, co.argmax(1), ro, None, meta)
                else:
                    res.append(heads.predict_bboxes_single_image(bbox_heads[s], props, co, ro, meta["img_shape"], RCNN_TEST))
        torch.cuda.synchronize()
        return res

    one_batch()
    ts = []
    for _ in range(args.ref_reps):
        t0 = time.perf_counter()
        res = one_batch()
        ts.append(time.perf_counter() - t0)
    ms = 1e3 * float(np.median(ts))
    # same inputs, same results: per image the detection count, labels and scores of the batched path
    same = True
    for b, (bx, sc, lb) in enumerate(res):
        k = int(hp.det_count[b])
        same &= k == int(sc.numel()) and torch.equal(lb, hp.det_label[b, :k]) and \
            bool(torch.allclose(sc, hp.det_score[b, :k], rtol=1e-5, atol=1e-7))
    return {"ms_per_batch": ms, "value": B / (ms / 1e3), "unit": "images/s", "reps": args.ref_reps,
            "detections_equal_batched_path": bool(same),
            "what": "eager, image by image: heads.rpn_predict_single_image -> region.BasicRoIExtractor.forward_single_image -> "
                    "(heads.refine_bboxes_single_image with cls_out.argmax(1)) -> heads.predict_bboxes_single_image; host clock "
                    "around a synchronised batch"}


def main(args):
    import torch
    import torch.distributed as dist

    import b200det
    from b200det import _C, workload
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench_infer.py needs a CUDA device: the path has no CPU fallback")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    sys.stdout.flush()
    real_stdout = os.dup(1)
    os.dup2(2, 1)                                                      # NCCL banners go to stderr; fd 1 keeps the JSON line
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    _C.lib()
    w = workload.config2(B=B, K=1, seed=workload.SEED + rank)
    T = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(dev)
    cls, reg = [T(c) for c in w["cls"]], [T(r) for r in w["reg"]]
    feats = [T(f).contiguous(memory_format=torch.channels_last) for f in w["feats"]]
    del w["feats"]
    img_hw = torch.tensor([[float(w["img_shape"][0]), float(w["img_shape"][1])]] * B, device=dev)
    runs = [run_stages(S, args, torch, dev, rank, world, w, cls, reg, feats, img_hw) for S in args.stages]
    if rank == 0:
        sys.stdout.flush()
        os.dup2(real_stdout, 1)
        print(json.dumps({
            "metric": "images/s of the test-time path (proposals -> RoIAlign -> refine -> detections), R50-FPN 800x1333",
            "gpu": gpu_info(local), "n_gpus": world, "images_per_gpu": B, "scaling": "weak", "dtype": "f32", "data": "synthetic",
            "warmup": max(args.warmup, 2), "cuda_graph": True,
            "allgather": None if world == 1 else {"in_timed_loop": True, "what": "dist.gather_detections of the [8, 100, 6] "
                                                  "records + counts after every replay"},
            "workload": "batch 8/GPU, 800x1333 (pad 800x1344), 256-channel fp32 NHWC FPN maps, RPN test 1000/1000/1000 @ 0.7, "
                        "RCNN test min_score 0.05, NMS 0.5, 100 per image, 21 classes, fixed synthetic head outputs (config-1 recipe)",
            "runs": runs}), flush=True)
        os.dup2(2, 1)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--stages", type=int, nargs="+", default=[1, 3], choices=[1, 2, 3])
    ap.add_argument("--steps", type=int, default=50, help="timed graph replays (the median of their per-step times is reported)")
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--ref-reps", type=int, default=5, help="timed batches of the reference call sequence")
    ap.add_argument("--no-reference", action="store_true")
    a = ap.parse_args()
    if a.steps < 20:
        ap.error("--steps must be at least 20 (the step time is a median)")
    if a.gpus > 1 and "WORLD_SIZE" not in os.environ:
        cmd = [sys.executable, "-m", "torch.distributed.run", "--standalone", "--nproc_per_node", str(a.gpus)] + sys.argv
        sys.exit(subprocess.call(cmd))
    main(a)
