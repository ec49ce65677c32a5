"""Benchmark of the batched training step, forward + backward: BASELINE config 2 (faster_rcnn_r50_fpn, batch 8, 800x1333,
workload.config2 inputs, fp32 channels_last FPN maps) through fused.TrainHotPath.step + TrainHotPath.backward, both as
one CUDA graph, with seeded upstream gradients of the step's three differentiable outputs (rpn_tar_cls, rpn_tar_reg,
roi_feats).  Reports the forward graph step, the forward + backward graph step, the two backward kernels alone (CUDA
events, eager: b2d_scatter_head_grads and b2d_roi_align_bwd_batched), images/s, and the eager alternative of a
reference user: refpath.BatchedCallSequence forward plus torch autograd of the same linear functional of its outputs.
Prints one JSON line (and writes it to --out if given)."""
import argparse
import ctypes
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


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
    ap.add_argument("--eager-steps", type=int, default=10)
    ap.add_argument("--out", help="also write the JSON line to this file")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_train_step.py needs a CUDA device: the path has no CPU fallback")
    from b200det import _C, fused, refpath, workload

    dev = torch.device("cuda:0")
    B, K, C = 8, 8, 256
    w = workload.config2(B=B, K=K, channels=C)
    T = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(dev)
    cls, reg = [T(c) for c in w["cls"]], [T(r) for r in w["reg"]]
    feats = [T(f).contiguous(memory_format=torch.channels_last) for f in w["feats"]]
    gt, gl = T(w["gt"]), T(w["gt_label"])
    gcount = torch.full((B,), K, dtype=torch.int32, device=dev)
    img_hw = torch.tensor([[float(w["img_shape"][0]), float(w["img_shape"][1])]] * B, device=dev)
    hp = fused.TrainHotPath(B, w["grids"], dev, gt_ld=K, feat_channels=C, layout=1, overlap=True)
    gen = torch.Generator(device=dev).manual_seed(2019)
    g_cls = torch.randn(hp.tar_cls.shape, device=dev, generator=gen)
    g_reg = torch.randn(hp.tar_reg.shape, device=dev, generator=gen)
    g_feat = torch.randn(hp.roi_align.out.shape, device=dev, generator=gen)

    step = lambda: hp.step(cls, reg, feats, gt, gcount, gl, img_hw)
    bwd = lambda: hp.backward(g_cls, g_reg, g_feat)
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

    # the two backward kernels alone, on the last replay's samples (eager, events around each call)
    st = hp._bwd_buffers()
    rt, bt = hp.rpn_targets, hp.roi_targets
    scatter = lambda: _C.call("b2d_scatter_head_grads", fused._ptrs(st["dcls"]), fused._ptrs(st["dreg"]), _C.ptr(g_cls),
                              _C.ptr(g_reg), ctypes.byref(hp.pyr.c), 1, _C.ptr(rt.chosen), _C.ptr(rt.n_chosen), rt.max_num,
                              B, _C.stream())
    k6 = lambda: _C.call("b2d_roi_align_bwd_batched", fused._ptrs(st["dfeat"]), _C.ptr(g_feat), _C.ptr(bt.tar_box),
                         hp.roi_align.ld, _C.ptr(bt.n_chosen), B, ctypes.byref(hp.roi_align.cfg), _C.ptr(st["ws"]),
                         st["ws"].numel(), _C.stream())
    scatter(); k6()
    scatter_ms, k6_ms = timed(scatter, args.steps), timed(k6, args.steps)
    head_bytes = sum(t.numel() * 4 for t in st["dcls"] + st["dreg"])

    # eager alternative: the reference call sequence on the drop-in, autograd of the same linear functional
    seq = refpath.BatchedCallSequence(w["strides"], dev)
    metas = [dict(img_shape=(w["img_shape"][0], w["img_shape"][1], 3), pad_shape=(w["pad_shape"][0], w["pad_shape"][1], 3),
                  scale_factor=1.0) for _ in range(B)]
    gtl, gll = [gt[i] for i in range(B)], [gl[i] for i in range(B)]
    ld = hp.roi_align.ld
    wc, wr = g_cls.reshape(1, -1), g_reg.permute(1, 0, 2).reshape(4, -1)

    def eager_step():
        lc = [c.detach().requires_grad_(True) for c in cls]
        lr = [r.detach().requires_grad_(True) for r in reg]
        lf = [f.detach().requires_grad_(True) for f in feats]
        out = seq.step(lc, lr, lf, gtl, gll, metas)
        tc, tr = out["rpn_targets"][0], out["rpn_targets"][1]
        loss = (tc * wc[:, :tc.shape[1]]).sum() + (tr * wr[:, :tr.shape[1]]).sum()
        for b, o in enumerate(out["roi_feats"]):
            loss = loss + (o * g_feat[b * ld:b * ld + o.shape[0]]).sum()
        loss.backward()

    eager_step(); eager_step()
    torch.cuda.synchronize()
    ts = []
    for _ in range(args.eager_steps):
        t0 = time.perf_counter()
        eager_step()
        torch.cuda.synchronize()
        ts.append(time.perf_counter() - t0)
    eager_ms = float(np.median(ts)) * 1e3

    name, limit = card()
    step_best = min(step_ms, step_ms2)
    res = {
        "metric": "images/sec of the batched train step forward + backward, R50-FPN 800x1333 (config 2)",
        "value": B / (step_best * 1e-3), "unit": "images/s", "batch": B,
        "fwd_graph_ms": min(fwd_ms, fwd_ms2), "fwd_bwd_graph_ms": step_best,
        "backward_in_step_ms": step_best - min(fwd_ms, fwd_ms2),
        "runs_ms": {"fwd": [fwd_ms, fwd_ms2], "fwd_bwd": [step_ms, step_ms2]},
        "kernels_ms": {"scatter_head_grads": scatter_ms, "roi_align_bwd_batched": k6_ms,
                       "note": "eager, CUDA events around %d back-to-back calls of each, on the last step's samples" % args.steps},
        "scatter_store_bytes": head_bytes, "scatter_store_gbs": head_bytes / (scatter_ms * 1e-3) / 1e9,
        "rois": int(bt.n_chosen.sum()), "channels": C,
        "eager_reference": {"ms_per_step": eager_ms, "value": B / (eager_ms * 1e-3), "unit": "images/s",
                            "note": "refpath.BatchedCallSequence forward + torch autograd backward of the same linear "
                                    "functional, channels_last features, median host wall clock incl. synchronisation"},
        "gpu": name, "power_limit": limit,
        "l2": "inputs per step (755 MB) and gradient maps (774 MB) exceed the 126 MB L2; no flush between replays",
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
