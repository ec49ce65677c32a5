#!/usr/bin/env python
"""Detection past 16384 candidates per image: the cost of max_candidates on the batched test paths.

  python scripts/bench_detect_candidates.py --steps 30 --warmup 3

One GPU, batch 8, 800x1333 images padded to 800x1344.  Workloads (seeded synthetic head outputs):
  infer_0.05 / infer_0.001   fused.InferHotPath, faster_rcnn at 81 classes (config 2 geometry, 1000 proposals), official
                             NMS 0.5, top 100; the RCNN head is replaced by fixed logits N(0, 2) with +3 on the
                             background and deltas N(0, 0.2);
  retina_0.05 / retina_0.01  fused.DenseInferHotPath, RetinaNet at config 4 (strides 8..128, 9 anchors, 80 classes,
                             sigmoid), official NMS 0.5, pre_nms 1000, top 100; logits -4.6 + N(0, 0.8) plus 20 objects
                             per image as Gaussian bumps of height 7 on their class.
Per workload and cap (the default 16384 where it does not overflow, and the exact bound) it reports the CUDA-graph
step time and the detect phase of event-bracketed eager steps (medians), the candidates per image (mean and max, from
the same scores the kernels test), how many images needed the continuation and the rounds they took, and the time of
the continuation kernel (torch.profiler) -- its idle cost when no image continues.  The last entries time adversarial
image sets of 2^20 candidates per image, 16 500 near-duplicates on top: behind them 1024-candidate groups of
near-duplicates, one survivor per round, at max_per_img 100 (99 rounds) and 16 384 (one round per group, about 1 000),
and boxes that overlap nothing at max_per_img 16 384 (16 rounds, each filtering the rest against 1024 kept boxes).
A round takes a block of at most 1024 candidates and keeps at least one, so an image takes at most
min(max_per_img - kept in round 0, ceil((candidates - 16384) / 1024)) rounds.
Prints one JSON line.
"""
import argparse
import ctypes
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

B = 8
IMG = (800.0, 1333.0)
RET_STRIDES = (8, 16, 32, 64, 128)
RET_GRIDS = [(100, 168), (50, 84), (25, 42), (13, 21), (7, 11)]
RET_SCALES = [4 * 2 ** (i / 3) for i in range(3)]


def gpu_info():
    try:
        out = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=20).stdout.strip()
        name, power, clk = [v.strip() for v in out.split(",")]
        return dict(name=name, power_limit=power, sm_max_clock=clk)
    except Exception as e:
        return dict(error="nvidia-smi query failed: %s" % e)


def kernel_us(torch, fn, names, reps=5):
    """Mean device time per call of the kernels whose name contains one of `names` (torch.profiler, its own run)."""
    from torch.profiler import ProfilerActivity, profile
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(reps):
            fn()
        torch.cuda.synchronize()
    tot = {n: 0.0 for n in names}
    for e in prof.events():
        if e.device_type.name == "CUDA":
            for n in names:
                if n in e.name:
                    tot[n] += e.device_time
    return {n: round(v / reps, 2) for n, v in tot.items()}


def time_path(torch, hp, step, mark_before, steps, warmup):
    """(graph step ms, eager detect-phase ms): medians over `steps`."""
    for _ in range(max(warmup, 2)):
        step(None)
    torch.cuda.synchronize()
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g, stream=side):
            step(None)
    torch.cuda.current_stream().wait_stream(side)
    g.replay()
    torch.cuda.synchronize()
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
    for a, b in ev:
        a.record()
        g.replay()
        b.record()
    torch.cuda.synchronize()
    step_ms = float(np.median([a.elapsed_time(b) for a, b in ev]))
    det = []
    for _ in range(steps):
        evs = {}

        def mark(name):
            e = torch.cuda.Event(enable_timing=True)
            e.record()
            evs[name] = e
        step(mark)
        torch.cuda.synchronize()
        det.append(evs[mark_before].elapsed_time(evs["detect"]))
    return step_ms, float(np.median(det))


def rounds_of(torch, _C, hp):
    if hp.cap <= 16384:
        return None
    r = torch.zeros(B, dtype=torch.int32, device=hp.det_ws.device)
    _C.call("b2d_detect_continuation_rounds", _C.ptr(r), _C.ptr(hp.det_ws), hp.cap, B, _C.stream())
    torch.cuda.synchronize()
    return r.cpu().tolist()


def stats(cands):
    return dict(mean=round(float(np.mean(cands)), 1), max=int(np.max(cands)))


def bench_infer(torch, dev, args, min_score):
    from b200det import _C, fused, workload
    NC, C = 81, 16
    w = workload.config2(B=B, K=1, seed=2019, channels=C, img_shape=(800, 1333), pad_shape=(800, 1344))
    T = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(dev)
    cls, reg = [T(c) for c in w["cls"]], [T(r) for r in w["reg"]]
    feats = [T(f).contiguous(memory_format=torch.channels_last) for f in w["feats"]]
    img_hw = torch.tensor([list(IMG)] * B, device=dev)
    rcnn = dict(min_score=min_score, nms_iou=0.5, max_per_img=100, nms_type="official")
    res = []
    for full in (False, True):
        hp = fused.InferHotPath(B, w["grids"], dev, feat_channels=C, num_classes=NC, rcnn_test=rcnn,
                                max_candidates=(1 << 20) if full else 16384)
        P = hp.P
        g = torch.Generator(device=dev).manual_seed(5)
        logits = torch.randn((B * P, NC), device=dev, generator=g) * 2.0
        logits[:, 0] += 3.0
        deltas = torch.randn((B * P, 4 * NC), device=dev, generator=g) * 0.2
        heads = [lambda x: (logits, deltas)]
        step = lambda mark: hp.step(cls, reg, feats, img_hw, heads, mark=mark)
        out = step(None)
        torch.cuda.synchronize()
        n = out["stages"][0]["count"].cpu().numpy()
        sm = torch.softmax(logits, 1)[:, 1:] >= np.float32(min_score)
        cands = [int(sm[b * P:b * P + n[b]].sum()) for b in range(B)]
        if not full and max(cands) > 16384:
            res.append(dict(cap=hp.cap, overflow=True, candidates=stats(cands)))
            continue
        step_ms, det_ms = time_path(torch, hp, step, "head0", args.steps, args.warmup)
        hp.check()
        r = rounds_of(torch, _C, hp)
        k = kernel_us(torch, lambda: step(None), ["k_det_continue", "k_nms_scan", "k_select", "k_hist", "k_compact"])
        res.append(dict(cap=hp.cap, step_ms=round(step_ms, 4), detect_ms=round(det_ms, 4), candidates=stats(cands),
                        continued_images=None if r is None else int(sum(v > 0 for v in r)), rounds=r, kernels_us=k))
    return res


def retina_logits(torch, dev, g, C):
    out = []
    objs = [[(float(torch.rand(1, generator=g, device=dev)) * IMG[1], float(torch.rand(1, generator=g, device=dev)) * IMG[0],
              32 + 368 * float(torch.rand(1, generator=g, device=dev)), int(torch.randint(C, (1,), generator=g, device=dev)))
             for _ in range(20)] for _ in range(B)]
    for s, (H, W) in zip(RET_STRIDES, RET_GRIDS):
        x = -4.6 + 0.8 * torch.randn((B, 9, C, H, W), device=dev, generator=g)
        yy, xx = torch.meshgrid(torch.arange(H, device=dev, dtype=torch.float32),
                                torch.arange(W, device=dev, dtype=torch.float32), indexing="ij")
        for b in range(B):
            for (cx, cy, size, c) in objs[b]:
                r = max(size / s / 2.0, 0.5)
                x[b, :, c] += 7.0 * torch.exp(-(((xx + 0.5) * s - cx) ** 2 + ((yy + 0.5) * s - cy) ** 2) / (2 * (r * s) ** 2))
        out.append(x.reshape(B, 9 * C, H, W).contiguous())
    return out


def bench_retina(torch, dev, args, min_score):
    from b200det import _C, fused
    C = 80
    g = torch.Generator(device=dev).manual_seed(4)
    cls = retina_logits(torch, dev, g, C)
    reg = [(0.2 * torch.randn((B, 36, H, W), device=dev, generator=g)).contiguous() for H, W in RET_GRIDS]
    img_hw = torch.tensor([list(IMG)] * B, device=dev)
    cfg = dict(pre_nms=1000, min_bbox_size=0, min_score=min_score, nms_iou=0.5, max_per_img=100, nms_type="official")
    res = []
    for full in (False, True):
        hp = fused.DenseInferHotPath(B, RET_GRIDS, dev, head="retina", num_classes=C + 1, test_cfg=cfg, strides=RET_STRIDES,
                                     anchor_scales=RET_SCALES, max_candidates=(1 << 20) if full else 16384)
        step = lambda mark: hp.step(cls, reg, img_hw, mark=mark)
        out = step(None)
        torch.cuda.synchronize()
        cands = []
        for b in range(B):
            n = int(out["sel_count"][b])
            rows = out["sel_rows"][b, :n].long()
            x = torch.cat([c[b].reshape(C, -1) for c in cls], 1)[:, rows]
            cands.append(int((torch.sigmoid(x) >= np.float32(min_score)).sum()))
        if not full and max(cands) > 16384:
            res.append(dict(cap=hp.cap, overflow=True, candidates=stats(cands)))
            continue
        step_ms, det_ms = time_path(torch, hp, step, "selection", args.steps, args.warmup)
        hp.check()
        r = rounds_of(torch, _C, hp)
        k = kernel_us(torch, lambda: step(None), ["k_det_continue", "k_nms_scan", "k_select", "k_hist", "k_compact"])
        res.append(dict(cap=hp.cap, step_ms=round(step_ms, 4), detect_ms=round(det_ms, 4), candidates=stats(cands),
                        continued_images=None if r is None else int(sum(v > 0 for v in r)), rounds=r, kernels_us=k))
    return res


def bench_adversarial(torch, dev, args, M, distinct):
    """b2d_dense_detect on B images of 2^20 candidates (one channel, given scores, linearly decreasing): 16 500
    near-duplicates on top (round 0 keeps one), then either groups of 1024 near-duplicates (one survivor per block, so
    min(M - 1, groups) rounds) or boxes that overlap nothing (every block kept: ceil((M - 1) / 1024) rounds, each
    filtering the remaining list against 1024 kept boxes)."""
    from b200det import _C
    top, gsz = 16500, 1024
    cap = n = 1 << 20
    i = torch.arange(n, device=dev)
    jit = torch.randint(0, 2, (4, n), generator=torch.Generator(device=dev).manual_seed(1), device=dev).float()
    if distinct:
        k = torch.clamp(i - top + 1, min=0)                          # 0: the top duplicates
        gx, gy, side = (k % 1024) * 20.0, (k // 1024) * 20.0, 10.0
        jit = jit * (k == 0)[None].float()
    else:
        g = torch.clamp((i - top) // gsz, min=-1)                    # -1: the top duplicates
        gx, gy, side = (g + 1) % 1000 * 100.0, (g + 1) // 1000 * 100.0, 60.0
    box = torch.stack([gx + jit[0], gy + jit[1], gx + side + jit[2], gy + side + jit[3]])
    boxes = box[None].expand(B, 4, n).contiguous()
    score = torch.full((B, 2, n), -1.0, device=dev)
    score[:, 0] = torch.linspace(0.99, 0.01, n, device=dev)
    rows = torch.arange(n, dtype=torch.int32, device=dev)[None].expand(B, n).contiguous()
    counts = torch.full((B,), n, dtype=torch.int32, device=dev)
    lv = _C.DenseLevels()
    lv.num_levels = 1
    lv.offset[0], lv.img_stride[0], lv.class_stride[0], lv.base[0] = 0, 2 * n, n, score.data_ptr()
    ws = torch.empty(_C.lib().b2d_rcnn_detect_workspace_bytes(cap, B), dtype=torch.uint8, device=dev)
    ob, osc = torch.zeros((B, 4, M), device=dev), torch.zeros((B, M), device=dev)
    ol, oc = torch.zeros((B, M), dtype=torch.int64, device=dev), torch.zeros(B, dtype=torch.int32, device=dev)
    ovf = torch.zeros(1, dtype=torch.int32, device=dev)

    def call():
        _C.call("b2d_dense_detect", _C.ptr(ob), _C.ptr(osc), _C.ptr(ol), _C.ptr(oc), _C.ptr(boxes), n, _C.ptr(counts),
                _C.ptr(rows), ctypes.byref(lv), 2, 0, None, 0, (_C.c_ull * 2)(3, 0), 0.0, 0, 0.5, M, 0, cap, B, _C.ptr(ovf),
                _C.ptr(ws), ws.numel(), None, _C.stream())
    call()
    torch.cuda.synchronize()
    reps = 5 if M <= 100 else 2
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(reps)]
    for a, b in ev:
        a.record()
        call()
        b.record()
    torch.cuda.synchronize()
    r = torch.zeros(B, dtype=torch.int32, device=dev)
    _C.call("b2d_detect_continuation_rounds", _C.ptr(r), _C.ptr(ws), cap, B, _C.stream())
    torch.cuda.synchronize()
    k = kernel_us(torch, call, ["k_det_continue", "k_nms_scan", "k_select", "k_hist", "k_compact"], reps=1)
    return dict(candidates_per_image=n, max_per_img=M, boxes="distinct" if distinct else "groups of 1024 duplicates",
                detected=oc.cpu().tolist(), rounds=r.cpu().tolist(),
                call_ms=round(float(np.median([a.elapsed_time(b) for a, b in ev])), 3), kernels_us=k)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=30)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--only", default="")
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        sys.exit("bench_detect_candidates: needs a CUDA device")
    import b200det                                                     # noqa: F401 (builds / loads the library)
    dev = torch.device("cuda:0")
    res = dict(bench="detect_candidates", batch=B, gpu=gpu_info())
    todo = args.only.split(",") if args.only else ["infer", "retina", "adversarial"]
    if "infer" in todo:
        for ms in (0.05, 0.001):
            res["infer_%g" % ms] = bench_infer(torch, dev, args, ms)
    if "retina" in todo:
        for ms in (0.05, 0.01):
            res["retina_%g" % ms] = bench_retina(torch, dev, args, ms)
    if "adversarial" in todo:
        res["adversarial"] = bench_adversarial(torch, dev, args, 100, False)
        res["adversarial_max_rounds"] = bench_adversarial(torch, dev, args, 16384, False)
        res["adversarial_distinct"] = bench_adversarial(torch, dev, args, 16384, True)
    print(json.dumps(res))


if __name__ == "__main__":
    main()
