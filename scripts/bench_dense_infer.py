#!/usr/bin/env python
"""Images/s of the batched one-stage test path (fused.DenseInferHotPath): head maps -> packed detections for RetinaNet
(BASELINE config 4) and FCOS / ATSS (config 5), both in one command.

  python scripts/bench_dense_infer.py --gpus 1 --steps 50 --warmup 5
  python scripts/bench_dense_infer.py --gpus 2 ...     # re-launches itself under torch.distributed.run

Workloads (batch 8 per GPU, 800x1333 padded to 800x1344, strides 8..128):
  retina  201 600 anchors (9 per cell), 20 classes, sigmoid, strict NMS, pre_nms 1000, min_score 0.05, NMS 0.5, top 100;
  fcos    22 400 points, 20 classes, centerness, strict NMS, pre_nms 1000, min_score 0.05, NMS 0.6, top 100.
Inputs are seeded synthetic head maps (not tuned to the result): class logits = -4.6 (the focal-loss prior bias,
p = 0.01) + N(0, 0.8) noise, plus per image 20 objects (sizes 32..400 px, random classes) that add a Gaussian bump of
height 7 to their class on every level, radius about the object size over the stride; RetinaNet deltas N(0, 0.2); FCOS
ltrb = |N(0.1, 0.05)| (x 300 px), centerness logits N(-1, 1) + the same bumps.  Candidates and detections per image are
reported, because the NMS cost follows them.

Reported per head (one JSON line per head): the CUDA-graph step time (median of per-step CUDA events; L2 flushed before
every step by a 256 MB memset outside the events, and also without the flush), images/s, kernel launches per step (an
eager step under torch.profiler), the phase split of an event-bracketed eager step (selection, candidates, NMS, gather;
FCOS also decode), the eager arms on the same inputs (the per-image drop-in image by image, and for RetinaNet
batched.anchor_head_predict_fast), and the GPU name and power limit read in the same run.  With --gpus N the records are
all-gathered (dist.gather_detections) inside the timed loop.
"""
import argparse
import json
import os
import subprocess
import sys
import time
import types

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

B = 8
C = 20
STRIDES = (8, 16, 32, 64, 128)
GRIDS = [(100, 168), (50, 84), (25, 42), (13, 21), (7, 11)]
IMG = (800.0, 1333.0)
SCALES = [4 * 2 ** (i / 3) for i in range(3)]
RATIOS = [0.5, 1.0, 2.0]
RETINA_CFG = dict(pre_nms=1000, min_bbox_size=0, min_score=0.05, nms_iou=0.5, max_per_img=100, nms_type="strict")
FCOS_CFG = dict(pre_nms=1000, min_bbox_size=0, min_score=0.05, nms_iou=0.6, max_per_img=100, nms_type="strict")
FLUSH_BYTES = 256 << 20


def gpu_info(index):
    q = "name,power.limit,clocks.max.sm"
    try:
        out = subprocess.run(["nvidia-smi", "-i", str(index), "--query-gpu=" + q, "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=20).stdout.strip()
        name, power, clk = [v.strip() for v in out.split(",")]
        return dict(name=name, power_limit=power, sm_max_clock=clk)
    except Exception as e:                                              # report, do not guess
        return dict(error="nvidia-smi query failed: %s" % e)


def synth_logits(rng, per_cell, objects):
    """[B, per_cell * C, H, W] per level: prior bias + noise + one Gaussian bump per object on its class channel(s)."""
    out = []
    for s, (H, W) in zip(STRIDES, GRIDS):
        x = (-4.6 + 0.8 * rng.standard_normal((B, per_cell, C, H, W))).astype(np.float32)
        yy, xx = np.mgrid[0:H, 0:W].astype(np.float32)
        for b, objs in enumerate(objects):
            for (cx, cy, size, c) in objs:
                r = max(size / s / 2.0, 0.5)
                bump = 7.0 * np.exp(-(((xx + 0.5) * s - cx) ** 2 + ((yy + 0.5) * s - cy) ** 2) / (2 * (r * s) ** 2))
                x[b, :, c] += bump.astype(np.float32)
        out.append(x.reshape(B, per_cell * C, H, W))
    return out


def make_inputs(rng):
    objects = [[(rng.uniform(0, IMG[1]), rng.uniform(0, IMG[0]), rng.uniform(32, 400), int(rng.integers(C)))
                for _ in range(20)] for _ in range(B)]
    ret_cls = synth_logits(rng, 9, objects)
    ret_reg = [(0.2 * rng.standard_normal((B, 36, H, W))).astype(np.float32) for H, W in GRIDS]
    fc_cls = synth_logits(rng, 1, objects)
    fc_reg = [np.abs(0.1 + 0.05 * rng.standard_normal((B, 4, H, W))).astype(np.float32) for H, W in GRIDS]
    fc_ctr = [(-1.0 + rng.standard_normal((B, 1, H, W))).astype(np.float32) for H, W in GRIDS]
    return dict(retina=(ret_cls, ret_reg, None), fcos=(fc_cls, fc_reg, fc_ctr))


def run_head(head, args, torch, dev, rank, world, maps):
    from b200det import dist as bdist, fused
    cls, reg, ctr = maps
    cfg = RETINA_CFG if head == "retina" else FCOS_CFG
    hp = fused.DenseInferHotPath(B, GRIDS, dev, head=head, num_classes=C + 1, test_cfg=cfg, strides=STRIDES,
                                 anchor_scales=SCALES, anchor_ratios=RATIOS, use_centerness=True)
    img_hw = torch.tensor([list(IMG)] * B, device=dev)
    rec = torch.zeros((B, hp.M, 6), dtype=torch.float32, device=dev)
    step = lambda: hp.step(cls, reg, img_hw, ctr_outs=ctr, records=rec)
    for _ in range(max(args.warmup, 2)):
        step()
    hp.check()
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(graph, stream=side):
            step()
    torch.cuda.current_stream().wait_stream(side)
    for _ in range(3):
        graph.replay()
    torch.cuda.synchronize()
    flush = torch.empty(FLUSH_BYTES, dtype=torch.uint8, device=dev)

    def one():
        graph.replay()
        if world > 1:
            bdist.gather_detections(rec, hp.det_count)

    def barrier():
        if world > 1:
            torch.distributed.barrier()
        torch.cuda.synchronize()

    def timed(do_flush):
        barrier()
        ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
        for a, b in ev:
            if do_flush:
                flush.zero_()
            a.record()
            one()
            b.record()
        barrier()
        return np.array([a.elapsed_time(b) for a, b in ev])

    per = timed(True)
    per_warm = timed(False)
    hp.check()
    ms = float(np.median(per))

    # ---- phase split: event-bracketed eager steps; the detection call records two events inside itself
    split, names = [], None
    dev_ev = [torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)]
    for e in dev_ev:
        e.record()
    torch.cuda.synchronize()
    for _ in range(10):
        flush.zero_()
        marks = []
        start = torch.cuda.Event(enable_timing=True)
        start.record()

        def mark(name):
            e = torch.cuda.Event(enable_timing=True)
            e.record()
            marks.append((name, e))
        hp.step(cls, reg, img_hw, ctr_outs=ctr, records=rec, mark=mark, detect_events=dev_ev)
        torch.cuda.synchronize()
        pts = [(n, e) for n, e in marks if n != "detect"] + [("candidates", dev_ev[0]), ("nms", dev_ev[1]),
                                                              ("gather", marks[-1][1])]
        names = [n for n, _ in pts]
        prev, row = start, []
        for _, e in pts:
            row.append(prev.elapsed_time(e))
            prev = e
        split.append(row)
    split = np.median(np.array(split), 0)
    phases = {n: float(v) for n, v in zip(names, split)}

    # ---- launches and device kernel times of one eager step (a profiled run of its own)
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        step()
        torch.cuda.synchronize()
    kernels, launches = {}, 0
    for e in prof.events():
        if e.device_type != torch.autograd.DeviceType.CUDA:
            continue
        launches += 1
        k = e.name if len(e.name) < 80 else e.name[:77] + "..."
        kernels[k] = kernels.get(k, 0.0) + e.device_time_total           # us
    kernels = dict(sorted(kernels.items(), key=lambda kv: -kv[1]))

    # ---- sizes: selected rows, NMS candidates (the detect call's own test, recomputed here), detections
    sel = hp.step(cls, reg, img_hw, ctr_outs=ctr, records=rec)
    torch.cuda.synchronize()
    rows = sel["sel_count"].cpu().numpy()
    cand = candidates(torch, hp, head, cls, sel, cfg)
    dets = hp.det_count.cpu().numpy()

    arms = None
    if not args.no_reference and rank == 0:
        arms = eager_arms(head, torch, dev, hp, cls, reg, ctr, cfg, args)
    return {
        "head": head, "ms_per_step": ms, "value": B * world / (ms / 1e3), "unit": "images/s", "per_gpu": B / (ms / 1e3),
        "steps": args.steps, "step_ms_p10_p90": [float(np.percentile(per, 10)), float(np.percentile(per, 90))],
        "l2": "flushed (256 MB memset outside the events) before every timed step",
        "ms_per_step_l2_not_flushed": float(np.median(per_warm)),
        "launches_per_step": launches, "launches_note": "kernels + memsets + memcpys of one eager step (torch.profiler)",
        "phases_ms": phases, "phases_note": "eager step, L2 flushed, launch gaps included; candidates = count + write + offset "
                                            "boxes, nms = b2d_nms, gather = records",
        "kernels_us": kernels,
        "counts": {"rows_mean": float(rows.mean()), "candidates_mean": float(np.mean(cand)), "candidates_max": int(max(cand)),
                   "detections_mean": float(dets.mean()), "detections_max": int(dets.max())},
        "eager_arms": arms,
    }


def candidates(torch, hp, head, cls, sel, cfg):
    """(row, class) pairs passing the strict test of the detect call, per image (host-side recount for the report)."""
    thr = float(np.float32(cfg["min_score"]))
    out = []
    for b in range(B):
        n = int(sel["sel_count"][b])
        rows = sel["sel_rows"][b, :n].long()
        if head == "retina":
            flat = torch.cat([c[b].reshape(C, -1) for c in cls], dim=1)
            s = flat.index_select(1, rows).sigmoid()
        else:
            s = hp.score[b].index_select(1, rows)
        out.append(int((s.max(0).values >= thr).sum()))
    return out


def eager_arms(head, torch, dev, hp, cls, reg, ctr, cfg, args):
    from b200det import anchor, batched, heads
    meta = dict(img_shape=(int(IMG[0]), int(IMG[1]), 3), pad_shape=(800, 1344, 3), scale_factor=1.0)
    if head == "retina":
        creators = [anchor.AnchorCreator(base=s, scales=SCALES, aspect_ratios=RATIOS) for s in STRIDES]
        me = types.SimpleNamespace(anchor_strides=list(STRIDES), anchor_scales=SCALES, anchor_ratios=RATIOS,
                                   target_means=[0.0] * 4, target_stds=[1.0] * 4, use_sigmoid=True, cls_channels=C,
                                   num_classes=C + 1, anchor_creators=creators)
        anchors = [torch.empty((4, 9) + g, device=dev) for g in GRIDS]
        per_image = lambda: [heads.anchor_head_predict_single_image(me, [c[b] for c in cls], [r[b] for r in reg], anchors,
                                                                    meta, cfg) for b in range(B)]
        fast = lambda: list(zip(*batched.anchor_head_predict_fast(me, cls, reg, [meta] * B, cfg)))
        arms = [("per_image", per_image, "heads.anchor_head_predict_single_image, image by image"),
                ("anchor_head_predict_fast", fast, "batched.anchor_head_predict_fast (batched selection, one "
                                                    "utils.multiclass_nms per image)")]
    else:
        per_image = lambda: [heads.fcos_predict_single_image([c[b] for c in cls], [r[b] for r in reg], [c[b] for c in ctr],
                                                             list(STRIDES), meta, cfg, 0.0, 300.0, True) for b in range(B)]
        arms = [("per_image", per_image, "heads.fcos_predict_single_image, image by image")]
    res = {}
    for name, fn, what in arms:
        fn()
        torch.cuda.synchronize()
        ts = []
        for _ in range(args.ref_reps):
            t0 = time.perf_counter()
            out = fn()
            torch.cuda.synchronize()
            ts.append(time.perf_counter() - t0)
        ms = 1e3 * float(np.median(ts))
        same = True
        for b, (bx, sc, lb) in enumerate(out):
            k = int(hp.det_count[b])
            same &= k == int(sc.numel()) and torch.equal(lb, hp.det_label[b, :k]) and \
                bool(torch.allclose(sc, hp.det_score[b, :k], rtol=1e-5, atol=1e-7)) and \
                bool(torch.allclose(bx, hp.det_box[b, :, :k], rtol=1e-5, atol=1e-3))
        res[name] = {"ms_per_batch": ms, "value": B / (ms / 1e3), "unit": "images/s", "reps": args.ref_reps,
                     "detections_equal_graph_path": bool(same), "what": what + "; host clock around a synchronised batch"}
    return res


def main(args):
    import torch
    import torch.distributed as dist

    import b200det  # noqa: F401
    from b200det import _C
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench_dense_infer.py needs a CUDA device: the path has no CPU fallback")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    sys.stdout.flush()
    real_stdout = os.dup(1)
    os.dup2(2, 1)                                                      # NCCL banners go to stderr; fd 1 keeps the JSON lines
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    _C.lib()
    rng = np.random.default_rng(2019 + 7 * rank)
    host = make_inputs(rng)
    T = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(dev)
    gpu = gpu_info(local)
    lines = []
    for head in args.heads:
        cls, reg, ctr = host[head]
        maps = ([T(c) for c in cls], [T(r) for r in reg], [T(c) for c in ctr] if ctr is not None else None)
        run = run_head(head, args, torch, dev, rank, world, maps)
        lines.append(dict({
            "metric": "images/s of the one-stage test path (head maps -> packed detections), %s" %
                      ("RetinaNet config 4" if head == "retina" else "FCOS/ATSS config 5"),
            "gpu": gpu, "n_gpus": world, "images_per_gpu": B, "scaling": "weak", "dtype": "f32", "data": "synthetic",
            "warmup": max(args.warmup, 2), "cuda_graph": True,
            "allgather": None if world == 1 else {"in_timed_loop": True, "what": "dist.gather_detections of the [8, 100, 6] "
                                                  "records + counts after every replay"},
            "workload": ("batch 8/GPU, 800x1333 (pad 800x1344), 201600 anchors, 20 classes, sigmoid, strict, pre_nms 1000, "
                         "min_score 0.05, NMS 0.5, top 100" if head == "retina" else
                         "batch 8/GPU, 800x1333 (pad 800x1344), 22400 points, 20 classes, centerness, strict, pre_nms 1000, "
                         "min_score 0.05, NMS 0.6, top 100"),
            "input_bytes_per_step": int(sum(t.numel() * 4 for t in maps[0]) + sum(t.numel() * 4 for t in maps[1]) +
                                        (sum(t.numel() * 4 for t in maps[2]) if maps[2] is not None else 0))}, **run))
        del maps
        torch.cuda.empty_cache()
    if rank == 0:
        sys.stdout.flush()
        os.dup2(real_stdout, 1)
        for ln in lines:
            print(json.dumps(ln), flush=True)
        if args.out:
            with open(args.out, "w") as f:
                for ln in lines:
                    f.write(json.dumps(ln) + "\n")
        os.dup2(2, 1)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--heads", nargs="+", default=["retina", "fcos"], choices=["retina", "fcos"])
    ap.add_argument("--steps", type=int, default=50, help="timed graph replays (the median of their per-step times is reported)")
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--ref-reps", type=int, default=5, help="timed batches of each eager arm")
    ap.add_argument("--no-reference", action="store_true")
    ap.add_argument("--out", default=None, help="also write the JSON lines to this file")
    a = ap.parse_args()
    if a.steps < 20:
        ap.error("--steps must be at least 20 (the step time is a median)")
    if a.gpus > 1 and "WORLD_SIZE" not in os.environ:
        cmd = [sys.executable, "-m", "torch.distributed.run", "--standalone", "--nproc_per_node", str(a.gpus)] + sys.argv
        sys.exit(subprocess.call(cmd))
    main(a)
