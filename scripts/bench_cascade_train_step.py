"""Benchmark of the batched cascade training step, forward + backward: BASELINE config 3 (cascade_rcnn_r50_fpn, batch 8,
800x1333, workload.config2 inputs, fp32 channels_last 256-channel FPN maps, 21 classes, 3 stages) through
fused.CascadeTrainHotPath.step + backward, each form captured as one CUDA graph.  The stage heads return fixed seeded
outputs (the recipe of scripts/bench_infer.py), so head layers are not timed.  Also reports, eager with CUDA events on
the same step's samples, the one RoIAlign backward over all three stages (b2d_roi_align_bwd_multi) against what a user
would otherwise run: three b2d_roi_align_bwd_batched calls and two additions of the gradient pyramids.  Prints one JSON
line (and writes it to --out if given)."""
import argparse
import ctypes
import json
import os
import subprocess
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

NC = 21


def card():
    """Name and power limit of the GPU the numbers were taken on (read-only nvidia-smi query)."""
    try:
        out = subprocess.run(["nvidia-smi", "-i", str(torch.cuda.current_device()), "--query-gpu=name,power.limit",
                              "--format=csv,noheader"], capture_output=True, text=True, timeout=10).stdout.strip()
        name, limit = [v.strip() for v in out.split(",")[:2]]
        return name, limit
    except Exception:
        return torch.cuda.get_device_name(), None


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--out", help="also write the JSON line to this file")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_cascade_train_step.py needs a CUDA device: the path has no CPU fallback")
    from b200det import _C, fused, workload

    dev = torch.device("cuda:0")
    B, K, C, S = 8, 8, 256, 3
    w = workload.config2(B=B, K=K, channels=C)
    T = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(dev)
    cls, reg = [T(c) for c in w["cls"]], [T(r) for r in w["reg"]]
    feats = [T(f).contiguous(memory_format=torch.channels_last) for f in w["feats"]]
    gt, gl = T(w["gt"]), T(w["gt_label"])
    gcount = torch.full((B,), K, dtype=torch.int32, device=dev)
    img_hw = torch.tensor([[float(w["img_shape"][0]), float(w["img_shape"][1])]] * B, device=dev)
    cp = fused.CascadeTrainHotPath(B, w["grids"], dev, gt_ld=K, feat_channels=C, num_classes=NC, num_stages=S, layout=1)
    m = cp.m
    rng = np.random.default_rng(2019 + 31)
    fixed = []
    for _ in range(S):
        c = rng.normal(0, 2.5, (B * m, NC)).astype(np.float32)
        c[:, 0] += 2.0
        fixed.append((T(c), T(rng.normal(0, 0.5, (B * m, 4 * NC)).astype(np.float32))))
    heads = [(lambda x, o=o: o) for o in fixed]
    gen = torch.Generator(device=dev).manual_seed(2019)
    g_cls = torch.randn(cp.tar_cls.shape, device=dev, generator=gen)
    g_reg = torch.randn(cp.tar_reg.shape, device=dev, generator=gen)
    g_roi = [torch.randn(ra.out.shape, device=dev, generator=gen) for ra in cp.roi_align]

    step = lambda: cp.step(cls, reg, feats, gt, gcount, gl, img_hw, heads)
    bwd = lambda: cp.backward(g_cls, g_reg, g_roi)
    for _ in range(max(args.warmup, 2)):
        step()
        bwd()
    torch.cuda.synchronize()

    def capture(fn):
        side = torch.cuda.Stream()
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side):
            g = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g, stream=side):
                fn()
        torch.cuda.current_stream().wait_stream(side)
        for _ in range(3):
            g.replay()
        torch.cuda.synchronize()
        return g

    g_fwd = capture(step)
    g_step = capture(lambda: (step(), bwd()))

    def timed(fn, n):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize()
        a.record()
        for _ in range(n):
            fn()
        b.record()
        torch.cuda.synchronize()
        return a.elapsed_time(b) / n

    fwd_ms, step_ms = timed(g_fwd.replay, args.steps), timed(g_step.replay, args.steps)
    fwd_ms2, step_ms2 = timed(g_fwd.replay, args.steps), timed(g_step.replay, args.steps)     # alternated: spread

    # the RoIAlign backward alone, on the last replay's samples: one call over the three stages against three batched
    # calls into three pyramids plus two pyramid additions (eager, events around back-to-back calls)
    st = cp._bwd_buffers()
    cfg = cp.roi_align[0].cfg
    lds = (_C.c_ll * S)(*([m] * S))
    gouts = (_C.c_void_p * S)(*[g.data_ptr() for g in g_roi])
    rois = (_C.c_void_p * S)(*[t.tar_box.data_ptr() for t in cp.targets])
    counts = (_C.c_void_p * S)(*[t.n_chosen.data_ptr() for t in cp.targets])
    multi = lambda: _C.call("b2d_roi_align_bwd_multi", fused._ptrs(st["dfeat"]), S, gouts, rois, lds, counts, B,
                            ctypes.byref(cfg), _C.ptr(st["ws"]), st["ws"].numel(), _C.stream())
    nb = _C.lib().b2d_roi_align_bwd_batched_workspace_bytes(m, B, ctypes.byref(cfg))
    ws1 = torch.empty(nb, dtype=torch.uint8, device=dev)
    pyr = [[torch.empty_like(d) for d in st["dfeat"]] for _ in range(S)]

    def separate():
        for s in range(S):
            t = cp.targets[s]
            _C.call("b2d_roi_align_bwd_batched", fused._ptrs(pyr[s]), _C.ptr(g_roi[s]), _C.ptr(t.tar_box), m,
                    _C.ptr(t.n_chosen), B, ctypes.byref(cfg), _C.ptr(ws1), ws1.numel(), _C.stream())
        for s in range(1, S):
            for a, b in zip(pyr[0], pyr[s]):
                a.add_(b)

    multi(); separate()
    torch.cuda.synchronize()
    # the two differ by summation order only; relative to |sum| + 1e-6 the difference is largest where the stages' terms
    # nearly cancel (the element-wise tolerance is tested in tests/test_gpu_cascade_train.py)
    max_rel = max(float(((a - b).abs() / (b.abs() + 1e-6)).max()) for a, b in zip(st["dfeat"], pyr[0]))
    multi_ms, sep_ms = timed(multi, args.steps), timed(separate, args.steps)
    multi_ms2, sep_ms2 = timed(multi, args.steps), timed(separate, args.steps)
    pyr_bytes = sum(d.numel() * 4 for d in st["dfeat"])

    name, limit = card()
    step_best = min(step_ms, step_ms2)
    res = {
        "metric": "images/sec of the batched cascade train step forward + backward, R50-FPN 800x1333, 3 stages (config 3)",
        "value": B / (step_best * 1e-3), "unit": "images/s", "batch": B, "stages": S, "classes": NC, "channels": C,
        "fwd_graph_ms": min(fwd_ms, fwd_ms2), "fwd_bwd_graph_ms": step_best,
        "fwd_images_per_s": B / (min(fwd_ms, fwd_ms2) * 1e-3),
        "backward_in_step_ms": step_best - min(fwd_ms, fwd_ms2),
        "runs_ms": {"fwd": [fwd_ms, fwd_ms2], "fwd_bwd": [step_ms, step_ms2]},
        "roi_align_bwd_ms": {"multi_one_call": [multi_ms, multi_ms2], "three_batched_plus_two_additions": [sep_ms, sep_ms2],
                             "max_rel_diff": max_rel,
                             "note": "eager, CUDA events around %d back-to-back calls of each, alternated, on the last "
                                     "step's samples" % args.steps},
        "rois_per_stage": [int(t.n_chosen.sum()) for t in cp.targets],
        "multi_workspace_bytes": int(st["ws"].numel()), "batched_workspace_bytes": int(nb),
        "gradient_pyramid_bytes": pyr_bytes,
        "gpu": name, "power_limit": limit,
        "l2": "inputs per step and gradient maps (%d MB) exceed the 126 MB L2; no flush between replays" % (pyr_bytes >> 20),
        "steps": args.steps, "warmup": max(args.warmup, 2),
    }
    line = json.dumps(res)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
