"""Dev micro-benchmarks of single stages on the config-2 workload (not the judged bench)."""
import os, sys, time
import numpy as np
import torch
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import b200det
from b200det import _C, fused, workload

def timeit(fn, n=20, warm=3):
    for _ in range(warm): fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(n): fn()
    e1.record(); torch.cuda.synchronize()
    return e0.elapsed_time(e1) / n * 1e3   # us

def main():
    dev = torch.device("cuda:0")
    B, K = 8, 8
    w = workload.config2(B=B, K=K)
    T = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(dev)
    cls, reg = [T(c) for c in w["cls"]], [T(r) for r in w["reg"]]
    feats = [T(f).contiguous(memory_format=torch.channels_last) for f in w["feats"]]
    gt, gl = T(w["gt"]), T(w["gt_label"])
    gcount = torch.full((B,), K, dtype=torch.int32, device=dev)
    img_hw = torch.tensor([[800.0, 1333.0]] * B, device=dev)
    hp = fused.TrainHotPath(B, w["grids"], dev, gt_ld=K, feat_channels=256, layout=1)
    out = hp.step(cls, reg, feats, gt, gcount, gl, img_hw)
    torch.cuda.synchronize()
    bt = out["rcnn"]
    which = sys.argv[1:] or ["stages"]
    if "roil2" in which:
        # same RoIs, but every image reads the features of image 0 -> after warm-up all taps are L2 hits
        import ctypes
        m = int(bt.n_chosen[0])
        rois1 = bt.tar_box[0, :, :m].contiguous()
        rois = rois1.repeat(1, 8).contiguous()
        R = rois.shape[1]
        outb = torch.empty((R, 256, 7, 7), device=dev)
        cfg = hp.roi_align.cfg
        fn = lambda: _C.call("b2d_roi_align_fwd", _C.ptr(outb), fused._ptrs(feats), _C.ptr(rois), R, None, None, R,
                             ctypes.byref(cfg), _C.stream())
        print("L2-resident roi_align: %.1f us for %d rois" % (timeit(fn), R))
    if "stages" in which:
        print("proposals %.1f us" % timeit(lambda: hp.proposals(cls, reg, img_hw)))
        print("rpn_targets %.1f us" % timeit(lambda: hp.rpn_targets(gt, gcount, None, img_hw=img_hw)))
        print("roi_targets %.1f us" % timeit(lambda: hp.roi_targets(gt, gcount, gl, boxes=out["props"], box_count=out["prop_count"])))
        print("roi_align %.1f us" % timeit(lambda: hp.roi_align(feats, bt.tar_box, bt.n_chosen)))
        print("step %.1f us" % timeit(lambda: hp.step(cls, reg, feats, gt, gcount, gl, img_hw)))

def graph_bench(groups, overlap):
    dev = torch.device("cuda:0")
    B, K = 8, 8
    w = workload.config2(B=B, K=K)
    T = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(dev)
    cls, reg = [T(c) for c in w["cls"]], [T(r) for r in w["reg"]]
    feats = [T(f).contiguous(memory_format=torch.channels_last) for f in w["feats"]]
    gt, gl = T(w["gt"]), T(w["gt_label"])
    gcount = torch.full((B,), K, dtype=torch.int32, device=dev)
    img_hw = torch.tensor([[800.0, 1333.0]] * B, device=dev)
    hp = fused.TrainHotPath(B, w["grids"], dev, gt_ld=K, feat_channels=256, layout=1, groups=groups, overlap=overlap)
    step = lambda: hp.step(cls, reg, feats, gt, gcount, gl, img_hw)
    for _ in range(3): step()
    torch.cuda.synchronize()
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        step()
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g, stream=side):
            step()
    torch.cuda.current_stream().wait_stream(side)
    us = timeit(g.replay, n=30, warm=5)
    print("graph groups=%d overlap=%s: %.1f us/step -> %.0f img/s" % (groups, overlap, us, 8e6 / us))


if __name__ == "__main__":
    if sys.argv[1:2] == ["graph"]:
        for gr, ov in [(1, False), (1, True), (2, True), (4, True), (8, True)]:
            graph_bench(gr, ov)
        sys.exit(0)
    main()
