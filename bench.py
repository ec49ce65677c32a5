#!/usr/bin/env python
"""bench.py -- images/sec of RPN proposal + target assignment + RoIAlign, R50-FPN at
800x1333 (BASELINE.json metric, config faster_rcnn_r50_fpn, train path).

  python bench.py --gpus N --steps K --warmup W              # B200 kernels
  python bench.py --impl reference --gpus N --steps K ...    # CPU reference arm (oracle port)

One step = one pass of the hot path over a batch of 8 images per GPU (weak scaling):
proposals (K3+K4) -> RPN anchor targets (K2, sampler, K8, head gather) -> RoI targets
(K2 + GT prepend, sampler, K8) -> FPN RoIAlign of the 512 sampled RoIs/image (K5).
Inputs are synthetic (SURVEY 8(d)), 755 MB per step and GPU, i.e. larger than the
126 MB L2, so no explicit flush is needed between iterations.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

IMGS_PER_GPU = 8
K_GT = 8
METRIC = "images/sec of RPN proposal+assign+RoIAlign, R50-FPN 800x1333"
WORKLOAD = "faster_rcnn_r50_fpn train path: batch 8/GPU at 800x1333 (pad 800x1344), 268569 anchors x 8 GT, " \
           "2000 proposals/img, 256 RPN + 512 RCNN samples, RoIAlign 7x7x256 on 512 RoIs/img"


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return float(d["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


def ncu_traffic(stage):
    """dram__bytes_read.sum + dram__bytes_write.sum per launch of the stage's dominant kernel, from the
    committed ncu --set full capture (profiles/traffic.json, written by scripts/profile_summary.py)."""
    p = os.path.join(ROOT, "profiles", "traffic.json")
    if not os.path.exists(p):
        return None
    return json.load(open(p)).get(stage)


class ClockSampler(threading.Thread):
    """SM clock and throttle reasons DURING the timed region (B200_PROFILING.md).  NVML through pynvml (sub-millisecond
    per query, so that even a 6 ms timed region is sampled); `nvidia-smi` as a fallback."""

    _BITS = {"hw_slowdown": 0x8, "hw_thermal_slowdown": 0x40, "sw_thermal_slowdown": 0x20, "sw_power_cap": 0x4}

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.rows, self.stop_flag = index, [], False          # rows: (t, sm_mhz, sm_max_mhz, [reasons])
        self.spin = False                                                   # True while a timed region runs: no sleep between queries
        self.window = None
        self.nvml = None
        try:
            import pynvml
            pynvml.nvmlInit()
            vis = os.environ.get("CUDA_VISIBLE_DEVICES")
            phys = int(vis.split(",")[index]) if vis and all(v.strip().isdigit() for v in vis.split(",")) else index
            self.handle = pynvml.nvmlDeviceGetHandleByIndex(phys)
            self.max_mhz = float(pynvml.nvmlDeviceGetMaxClockInfo(self.handle, pynvml.NVML_CLOCK_SM))
            self.nvml = pynvml
        except Exception:
            self.nvml = None
        self.q = "clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
                 "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def run(self):
        while not self.stop_flag:
            try:
                if self.nvml is not None:
                    n = self.nvml
                    mhz = float(n.nvmlDeviceGetClockInfo(self.handle, n.NVML_CLOCK_SM))
                    mask = int(n.nvmlDeviceGetCurrentClocksEventReasons(self.handle))
                    self.rows.append((time.perf_counter(), mhz, self.max_mhz, [k for k, b in self._BITS.items() if mask & b]))
                    if not self.spin:
                        time.sleep(0.0005)
                    continue
                out = subprocess.run(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.q,
                                      "--format=csv,noheader,nounits"], capture_output=True, text=True, timeout=5).stdout
                c = [v.strip() for v in out.strip().split(",")]
                if len(c) >= 6 and c[0].replace(".", "").isdigit():
                    names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
                    self.rows.append((time.perf_counter(), float(c[0]), float(c[1]),
                                      [k for k, v in zip(names, c[2:6]) if v.lower().startswith("active")]))
            except Exception:
                pass
            time.sleep(0.05)

    def summary(self):
        rows = self.rows
        inside = [r for r in rows if self.window and self.window[0] <= r[0] <= self.window[1]]
        lw = getattr(self, "load_window", None)
        loaded = [r for r in rows if lw and lw[0] <= r[0] <= lw[1]]      # timed region + the untimed continuation of the same load
        use = inside or loaded
        if not use and self.window and rows:             # fall back to the samples closest to the region
            mid = 0.5 * (self.window[0] + self.window[1])
            use = sorted(rows, key=lambda r: abs(r[0] - mid))[:8]
        if not use:
            use = rows
        sm = [r[1] for r in use]
        mx = [r[2] for r in use]
        reasons = sorted({k for r in use for k in r[3]})
        return dict(sm_mhz=float(np.median(sm)) if sm else None, sm_max_mhz=max(mx) if mx else None, reasons=reasons,
                    samples=len(sm), samples_in_timed_region=len(inside), samples_under_load=len(loaded),
                    mean_sample_interval_ms=(1e3 * (rows[-1][0] - rows[0][0]) / max(len(rows) - 1, 1)) if len(rows) > 1 else None,
                    source="nvml" if self.nvml is not None else "nvidia-smi")


def touched_cell_bytes(rois_b4n, counts, grids, strides, C, finest=56.0):
    """Bytes of distinct feature cells the bilinear taps of these RoIs touch (per-image union),
    the input term of the RoIAlign algorithmic traffic (SURVEY 8(d)), fp32."""
    total = 0
    for b in range(rois_b4n.shape[0]):
        r = rois_b4n[b][:, :counts[b]].astype(np.float32)
        s = np.sqrt((r[2] - r[0] + 1) * (r[3] - r[1] + 1))
        lv = np.clip(np.floor(np.log2(s / finest + 1e-6)), 0, 3).astype(int)
        for l in range(4):
            H, W = grids[l]
            m = np.zeros((H, W), bool)
            rr = r[:, lv == l] / strides[l]
            if rr.shape[1] == 0:
                continue
            x0, y0 = rr[0], rr[1]
            rw, rh = np.maximum(rr[2] - x0, 1), np.maximum(rr[3] - y0, 1)
            k = (np.arange(14) + 0.5) / 14.0
            xs = np.clip(x0[:, None] + rw[:, None] * k[None], 0, W - 1)     # [n,14]
            ys = np.clip(y0[:, None] + rh[:, None] * k[None], 0, H - 1)
            xl, yl = np.floor(xs).astype(int), np.floor(ys).astype(int)
            xh, yh = np.minimum(xl + 1, W - 1), np.minimum(yl + 1, H - 1)
            for yy in (yl, yh):
                for xx in (xl, xh):
                    m[yy[:, :, None], xx[:, None, :]] = True
            total += int(m.sum()) * C * 4
    return total


DUMP_FEAT_ROWS = 512


def dump_outputs(path, out):
    """Write what one TrainHotPath.step returned to `path`/<name>.npy as float32 (the integer outputs are counts, labels
    and indices, all exact in float32), so that two builds can be compared output for output.  Entries past an image's
    count are zeroed: a caller never reads them and they may hold what an earlier step left.  roi_feats (205 MB at
    batch 8) is stored as a fixed, seeded sample of DUMP_FEAT_ROWS rows (25.7 MB), their indices in roi_feats_rows."""
    import torch

    rpn, rcnn = out["rpn"], out["rcnn"]
    pc, rn, bn = (t.cpu().numpy() for t in (out["prop_count"], rpn.n_chosen, rcnn.n_chosen))

    def upto(t, n):
        a = t.cpu().numpy()
        keep = np.arange(a.shape[-1])[None, :] < n[:, None]                     # [B, last axis]
        return np.where(keep.reshape((a.shape[0],) + (1,) * (a.ndim - 2) + (a.shape[-1],)), a, 0)

    arrays = {"props": upto(out["props"], pc), "scores": upto(out["scores"], pc), "prop_count": pc,
              "rpn_count": rn, "rpn_label": upto(rpn.tar_label, rn), "rpn_param": upto(rpn.tar_param, rn),
              "rpn_tar_cls": upto(out["rpn_tar_cls"], rn), "rpn_tar_reg": upto(out["rpn_tar_reg"], rn),
              "roi_count": bn, "roi_box": upto(rcnn.tar_box, bn), "roi_label": upto(rcnn.tar_label, bn),
              "roi_param": upto(rcnn.tar_param, bn)}
    feats = out["roi_feats"]
    ld = feats.shape[0] // len(bn)
    rows = np.sort(np.random.default_rng(0).choice(feats.shape[0], min(DUMP_FEAT_ROWS, feats.shape[0]), replace=False))
    sample = feats.index_select(0, torch.from_numpy(rows).to(feats.device)).cpu().numpy()
    sample[rows % ld >= bn[rows // ld]] = 0
    arrays["roi_feats"], arrays["roi_feats_rows"] = sample, rows
    os.makedirs(path, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(path, name + ".npy"), np.ascontiguousarray(a, dtype=np.float32))


def workload_config(world):
    """`config` of the JSON line: the workload only (identical for both arms; what the B200 arm does with it is `run_config`)."""
    return {"workload": WORKLOAD, "global_batch": IMGS_PER_GPU * world, "parallelism": "per-image partition, dp%d" % world,
            "l2": "inputs per step (755 MB/GPU) exceed the 126 MB L2; no flush needed"}


# --------------------------------------------------------------------------- reference arm
def run_reference(args):
    """The reference's CPU implementation of the path, timed on the host cores: the oracle
    port (the Python reference itself does not travel to the GPU box)."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    import oracle
    from oracle import pipeline as opipe
    from b200det import workload  # host-side input generator only
    oracle.set_num_threads(os.cpu_count())
    cores = oracle.num_threads()
    # one step = one GPU's batch (8 images) run image by image, as the reference's per-image loops do; with more than ~25
    # steps requested the sample shrinks to 2 images per step so that the run stays within a few minutes
    imgs = IMGS_PER_GPU if (args.steps + max(args.warmup, 1)) <= 25 else 2
    w = workload.config2(B=imgs, K=K_GT)
    path = opipe.ImagePath(w["grids"], w["strides"], w["img_shape"])
    per_img = [([c[b] for c in w["cls"]], [r[b] for r in w["reg"]], [f[b] for f in w["feats"]], w["gt"][b], w["gt_label"][b])
               for b in range(imgs)]
    for _ in range(max(args.warmup, 1)):
        for a in per_img:
            path.run(*a)
    t0 = time.perf_counter()
    for i in range(args.steps):
        for a in per_img:
            path.run(*a, seed=i)
    dt = time.perf_counter() - t0
    val = imgs * args.steps / dt
    sample = "%d images per step (one GPU's batch of the workload), %d steps; C port of the reference path with OpenMP" % (imgs, args.steps)
    print(json.dumps({
        "impl": "reference", "metric": METRIC, "value": val, "unit": "images/s", "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": 1e3 * dt / args.steps, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic", "config": workload_config(max(int(args.gpus), 1)),
        "cpu_baseline": {"value": val, "unit": "images/s", "cores": cores, "kind": "port", "sample": sample},
        "e2e": {"value": val, "unit": "images/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0}))


def bind_to_gpu_numa_node(index):
    """Pin this process (and with it the first-touch placement of its pinned host buffers) to the CPUs local to GPU
    `index`: at N = 8 the eight H2D streams otherwise cross the socket interconnect.  Best effort, silent on failure."""
    try:
        import pynvml
        pynvml.nvmlInit()
        vis = os.environ.get("CUDA_VISIBLE_DEVICES")
        phys = int(vis.split(",")[index]) if vis and all(v.strip().isdigit() for v in vis.split(",")) else index
        h = pynvml.nvmlDeviceGetHandleByIndex(phys)
        words = (os.cpu_count() + 63) // 64
        mask = pynvml.nvmlDeviceGetCpuAffinity(h, words)
        cpus = {64 * i + b for i, wd in enumerate(mask) for b in range(64) if (int(wd) >> b) & 1}
        cpus &= set(os.sched_getaffinity(0))
        if cpus:
            os.sched_setaffinity(0, cpus)
            return len(cpus)
    except Exception:
        pass
    return 0


# --------------------------------------------------------------------------- B200 arm
def run_b200(args):
    import torch
    import torch.distributed as dist

    import b200det
    from b200det import _C, fused, workload

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the B200 path has no CPU fallback")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    numa_cpus = bind_to_gpu_numa_node(local) if world > 1 else 0
    # NCCL prints its version banner on stdout (NCCL_DEBUG=VERSION/WARN): keep fd 1 for the one JSON line
    sys.stdout.flush()
    real_stdout = os.dup(1)
    os.dup2(2, 1)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    _C.lib()
    B = IMGS_PER_GPU
    w = workload.config2(B=B, K=K_GT, seed=workload.SEED + rank)
    grids, strides = w["grids"], w["strides"]
    host = lambda a: torch.from_numpy(np.ascontiguousarray(a)).pin_memory()
    h_cls, h_reg, h_feat = [host(c) for c in w["cls"]], [host(r) for r in w["reg"]], [host(f) for f in w["feats"]]
    h_gt, h_gl = host(w["gt"]), host(w["gt_label"])
    cls, reg = [t.to(dev) for t in h_cls], [t.to(dev) for t in h_reg]
    feats_nchw = [t.to(dev) for t in h_feat]
    feats = [f.contiguous(memory_format=torch.channels_last) for f in feats_nchw]     # B200-native layout (NHWC)
    gt, gl = h_gt.to(dev), h_gl.to(dev)
    gcount = torch.full((B,), K_GT, dtype=torch.int32, device=dev)
    img_hw = torch.tensor([[float(w["img_shape"][0]), float(w["img_shape"][1])]] * B, device=dev)
    hp = fused.TrainHotPath(B, grids, dev, gt_ld=K_GT, feat_channels=256, layout=1, overlap=True, groups=args.groups)

    def step():
        return hp.step(cls, reg, feats, gt, gcount, gl, img_hw)

    # warm-up (also sets the kernel attributes before graph capture)
    for _ in range(max(args.warmup, 3)):
        out = step()
    torch.cuda.synchronize()
    graph = None
    if not args.no_graph:
        side = torch.cuda.Stream()
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side):
            step()
            graph = torch.cuda.CUDAGraph()
            with torch.cuda.graph(graph, stream=side):
                out = step()
        torch.cuda.current_stream().wait_stream(side)
        for _ in range(3):
            graph.replay()
        torch.cuda.synchronize()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    sampler = ClockSampler(local)
    sampler.start()

    def timed(fn, n):
        """n calls of fn bracketed by barrier + synchronize on both sides, timed with CUDA events on the launching stream."""
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        barrier()
        a.record()
        for _ in range(n):
            fn()
        b.record()
        barrier()
        return a.elapsed_time(b)

    # ---- the all-gather of SURVEY 8(e) inside the timed loop (N > 1): the merge kernel itself writes the rank's proposals
    # as packed [B, P, 5] records (no packing kernel); two graphs alternate between two record buffers, and after every
    # replay the records are all-gathered over NCCL on a side stream while the next replay already runs
    if world > 1:
        P = hp.proposals.P
        rec = [torch.zeros((B, P, 5), dtype=torch.float32, device=dev) for _ in range(2)]
        gout = [torch.empty((world * B, P, 5), dtype=torch.float32, device=dev) for _ in range(2)]
        s_comm = torch.cuda.Stream()
        ev_done = [torch.cuda.Event() for _ in range(2)]
        state = {"it": 0}
        graphs = []
        for k in range(2):
            fn = (lambda k=k: hp.step(cls, reg, feats, gt, gcount, gl, img_hw, records=rec[k]))
            fn()
            torch.cuda.synchronize()
            if args.no_graph:
                graphs.append(fn)
                continue
            side = torch.cuda.Stream()
            side.wait_stream(torch.cuda.current_stream())
            with torch.cuda.stream(side):
                g2 = torch.cuda.CUDAGraph()
                with torch.cuda.graph(g2, stream=side):
                    fn()
            torch.cuda.current_stream().wait_stream(side)
            graphs.append(g2.replay)

        def run_step():
            k = state["it"] & 1
            state["it"] += 1
            cur = torch.cuda.current_stream()
            cur.wait_event(ev_done[k])                                  # the gather that last read rec[k]
            graphs[k]()
            s_comm.wait_stream(cur)
            with torch.cuda.stream(s_comm):
                dist.all_gather_into_tensor(gout[k], rec[k])
                ev_done[k].record(s_comm)

        for _ in range(4):
            run_step()
        torch.cuda.current_stream().wait_stream(s_comm)
        torch.cuda.synchronize()
    else:
        def run_step():
            graph.replay() if graph is not None else step()

    def run_all():
        run_step()

    # wake the clock sampler BEFORE the region and wait until it is spinning: on boxes with a coarse timer its 0.5 ms idle
    # sleep lasts longer than the whole timed region (seen: 0 samples inside although a query takes 3 us)
    sampler.spin = True
    n_rows, t_wake = len(sampler.rows), time.perf_counter()
    while len(sampler.rows) < n_rows + 3 and time.perf_counter() - t_wake < 0.5:
        time.sleep(0.001)
    barrier()
    t_host0 = time.perf_counter()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(args.steps):
        run_all()
    if world > 1:
        torch.cuda.current_stream().wait_stream(s_comm)                 # the last gather ends inside the timed region
    e1.record()
    barrier()
    sampler.window = (t_host0, time.perf_counter())
    ms = e0.elapsed_time(e1)
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, out)                            # out: the buffers every step writes
    # The timed region is a few milliseconds; where an NVML query takes longer than that (box-dependent) no sample can
    # fall inside it.  The identical load is therefore kept up, UNTIMED, for ~240 more steps while the sampler keeps
    # spinning; those samples are reported separately (clocks.samples_under_load) and only used when the region has none.
    for _ in range(max(1, 240 // max(args.steps, 1))):   # a FIXED count (every rank issues the same collectives): ~240 more steps
        for _ in range(args.steps):
            run_all()
        torch.cuda.synchronize()
    if world > 1:
        torch.cuda.current_stream().wait_stream(s_comm)
    barrier()
    sampler.spin = False
    sampler.load_window = (t_host0, time.perf_counter())
    # ---- the same step fed with the reference layout: fp32 NCHW features -> b2d_nchw_to_nhwc (4 launches) -> step
    nhwc_buf = [torch.empty_like(f, memory_format=torch.channels_last) for f in feats_nchw]

    def step_nchw():
        for f, o in zip(feats_nchw, nhwc_buf):
            _C.call("b2d_nchw_to_nhwc", _C.ptr(o), _C.ptr(f), f.shape[0], f.shape[1], f.shape[2], f.shape[3], _C.stream())
        return hp.step(cls, reg, nhwc_buf, gt, gcount, gl, img_hw)

    step_nchw()
    torch.cuda.synchronize()
    graph_nchw = None
    if not args.no_graph:
        side = torch.cuda.Stream()
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side):
            step_nchw()
            graph_nchw = torch.cuda.CUDAGraph()
            with torch.cuda.graph(graph_nchw, stream=side):
                step_nchw()
        torch.cuda.current_stream().wait_stream(side)
        graph_nchw.replay()
    nchw_ms = timed((lambda: graph_nchw.replay()) if graph_nchw is not None else step_nchw, args.steps) / args.steps
    # ---- strong scaling (N > 1): the global batch of BASELINE config 2 (8 images) split per image over the ranks
    strong_ms = None
    if world > 1 and B % world == 0:
        Bs = B // world
        hps = fused.TrainHotPath(Bs, grids, dev, gt_ld=K_GT, feat_channels=256, layout=1, overlap=True)
        sl = slice(0, Bs)
        args_s = ([t[sl] for t in cls], [t[sl] for t in reg], [f[sl] for f in feats], gt[sl], gcount[sl], gl[sl], img_hw[sl])
        for _ in range(3):
            hps.step(*args_s)
        torch.cuda.synchronize()
        side = torch.cuda.Stream()
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side):
            hps.step(*args_s)
            gs = torch.cuda.CUDAGraph()
            with torch.cuda.graph(gs, stream=side):
                hps.step(*args_s)
        torch.cuda.current_stream().wait_stream(side)
        gs.replay()
        strong_ms = timed(lambda: gs.replay(), args.steps) / args.steps
    # ---- two batches in flight (VERDICT r1 item 4): a second, independent TrainHotPath instance (own workspaces, outputs and
    # sampler counter) and graph; the two graphs are replayed alternately on two streams, so step i+1's latency-bound
    # proposal chain runs beside step i's RoIAlign.  Reported next to `value`, which stays one batch in flight (what a
    # training step can do).
    inflight = None
    if rank == 0 and world == 1 and graph is not None:
        hp2 = fused.TrainHotPath(B, grids, dev, gt_ld=K_GT, feat_channels=256, layout=1, overlap=True, groups=args.groups, seed=7)
        for _ in range(3):
            hp2.step(cls, reg, feats, gt, gcount, gl, img_hw)
        torch.cuda.synchronize()
        s2 = torch.cuda.Stream()
        s2.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(s2):
            hp2.step(cls, reg, feats, gt, gcount, gl, img_hw)
            graph2 = torch.cuda.CUDAGraph()
            with torch.cuda.graph(graph2, stream=s2):
                hp2.step(cls, reg, feats, gt, gcount, gl, img_hw)
        torch.cuda.current_stream().wait_stream(s2)
        s1 = torch.cuda.Stream()
        pair = ((s1, graph), (s2, graph2))

        def two_in_flight(n):
            cur = torch.cuda.current_stream()
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            torch.cuda.synchronize()
            a.record(cur)
            for st, _ in pair:
                st.wait_event(a)
            for i in range(n):
                st, g = pair[i & 1]
                with torch.cuda.stream(st):
                    g.replay()
            for st, _ in pair:
                cur.wait_stream(st)
            b.record(cur)
            torch.cuda.synchronize()
            return a.elapsed_time(b)

        two_in_flight(4)
        ms2 = two_in_flight(args.steps) / args.steps
        inflight = {"batches_in_flight": 2, "ms_per_step": ms2, "value": B / (ms2 / 1e3), "unit": "images/s",
                    "note": "two independent step graphs replayed alternately on two streams (total time / steps)"}
        del hp2, graph2
    # ---- what a reference user gets after install(): the reference's own per-image call sequence
    # (lib/detectors/cascade_rcnn.py:106-131) on the drop-in's reference-signature functions, eager, fp32 NCHW features
    # as the reference FPN emits them, and channels_last features (install(channels_last=True))
    dropin = None
    if rank == 0 and not args.no_dropin:
        from b200det import refpath
        seq = refpath.TrainCallSequence(strides, dev)
        metas = [dict(img_shape=(w["img_shape"][0], w["img_shape"][1], 3), pad_shape=(w["pad_shape"][0], w["pad_shape"][1], 3),
                      scale_factor=1.0) for _ in range(B)]
        gtl, gll = [gt[i] for i in range(B)], [gl[i] for i in range(B)]
        dropin = {}

        def host_median(fn, n_it):
            """median host wall time of one call, device work included (a scheduling hiccup of the host does not
            triple a 1 ms measurement, as it does with a mean over 20 calls)"""
            ts = []
            for _ in range(n_it):
                t0 = time.perf_counter()
                fn()
                torch.cuda.synchronize()
                ts.append(time.perf_counter() - t0)
            return float(np.median(ts))

        for name, ff in (("nchw", feats_nchw), ("channels_last", feats)):
            fn = lambda: seq.step(cls, reg, ff, gtl, gll, metas)
            fn(); fn()
            torch.cuda.synchronize()
            dt = host_median(fn, 5)
            dropin[name] = {"value": B / dt, "unit": "images/s", "ms_per_step": dt * 1e3}
        # the same sequence with the three per-image loops rebound at the METHOD level (batched.py; what install() binds
        # onto RPNHead.predict_bboxes_from_output / AnchorHead.loss / BBoxHead.bbox_targets): one batched pass per loop
        seqb = refpath.BatchedCallSequence(strides, dev)
        for name, ff in (("batched_nchw", feats_nchw), ("batched_channels_last", feats)):
            fn = lambda: seqb.step(cls, reg, ff, gtl, gll, metas)
            fn(); fn()
            torch.cuda.synchronize()
            dt = host_median(fn, 20)
            dropin[name] = {"value": B / dt, "unit": "images/s", "ms_per_step": dt * 1e3}
        dropin["note"] = "reference call sequence (AnchorHead.loss targets / predict_bboxes_from_output / bbox_targets / " \
                         "BasicRoIExtractor) on the drop-in, eager, median host wall clock per call incl. its syncs; nchw / channels_last: " \
                         "the reference's per-image Python loops on the rebound functions; batched_*: the loops themselves " \
                         "rebound (one batched pass + one sync each), as install() does"
    # ---- per-stage device times (eager, CUDA events on the launching stream)
    stages = ["proposals", "rpn_targets", "roi_targets", "roi_align"]
    evs = [[torch.cuda.Event(enable_timing=True) for _ in range(5)] for _ in range(args.steps)]
    for it in range(args.steps):
        ev = evs[it]
        ev[0].record()
        props, scores, count = hp.proposals(cls, reg, img_hw)
        ev[1].record()
        rt = hp.rpn_targets(gt, gcount, None, img_hw=img_hw)
        _C.call("b2d_gather_head_outputs", _C.ptr(hp.tar_cls), _C.ptr(hp.tar_reg), fused._ptrs(cls), fused._ptrs(reg),
                __import__("ctypes").byref(hp.pyr.c), 1, _C.ptr(rt.chosen), _C.ptr(rt.n_chosen), rt.max_num, B, _C.stream())
        ev[2].record()
        bt = hp.roi_targets(gt, gcount, gl, boxes=props, box_count=count)
        ev[3].record()
        hp.roi_align(feats, bt.tar_box, bt.n_chosen)
        ev[4].record()
    torch.cuda.synchronize()
    stage_ms = {s: float(np.mean([evs[it][i].elapsed_time(evs[it][i + 1]) for it in range(args.steps)]))
                for i, s in enumerate(stages)}
    # ---- the same RoIAlign on bf16 NHWC features (north_star: "NHWC bf16/fp32 features"; reported separately: it halves
    # the input bytes but cannot meet the 1e-5 parity bar against the fp32 reference)
    bf16_ms = None
    if rank == 0:
        feats16 = [f.to(torch.bfloat16).contiguous(memory_format=torch.channels_last) for f in feats[:4]]
        ra16 = fused.BatchedRoIAlign(B, hp.roi_align.ld, [(256, g[0], g[1]) for g in grids[:4]], list(strides[:4]), dev, layout=2)
        bt16 = out["rcnn"]
        for _ in range(3):
            ra16(feats16, bt16.tar_box, bt16.n_chosen)
        g0, g1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        g0.record()
        for _ in range(args.steps):
            ra16(feats16, bt16.tar_box, bt16.n_chosen)
        g1.record()
        torch.cuda.synchronize()
        bf16_ms = g0.elapsed_time(g1) / args.steps
        del feats16, ra16
    # ---- SURVEY 8(d)(ii): the same RoIAlign on ALL 2000 proposals per image ("stress": 16 000 RoIs, 803 MB of output)
    k2000_ms = None
    if rank == 0:
        ra2k = fused.BatchedRoIAlign(B, hp.proposals.P, [(256, g[0], g[1]) for g in grids[:4]], list(strides[:4]), dev, layout=1)
        for _ in range(2):
            ra2k(feats, hp.proposals.props, hp.proposals.count)
        g0, g1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        g0.record()
        for _ in range(5):
            ra2k(feats, hp.proposals.props, hp.proposals.count)
        g1.record()
        torch.cuda.synchronize()
        k2000_ms = g0.elapsed_time(g1) / 5
        del ra2k
    # ---- end-to-end through the public API with HOST buffers (fp32 NCHW, the reference layout):
    # TrainHotPath.step_from_host = pinned host inputs -> H2D -> NCHW->NHWC -> hot path -> D2H of the results
    def e2e_step():
        return hp.step_from_host(h_cls, h_reg, h_feat, h_gt, h_gl, gcount, img_hw)

    for _ in range(3):
        h_out = e2e_step()
    torch.cuda.synchronize()
    h2d = sum(t.numel() * t.element_size() for t in h_cls + h_reg + h_feat + [h_gt, h_gl])
    d2h = sum(t.numel() * t.element_size() for t in h_out.values())
    n_e2e = max(3, min(args.steps, 10))
    barrier()
    f0, f1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    f0.record()
    for _ in range(n_e2e):
        e2e_step()
    f1.record()
    barrier()
    e2e_ms = f0.elapsed_time(f1) / n_e2e
    # ---- the same call with the host feature maps in channels_last memory format (what install(channels_last=True) makes
    # the FPN emit): step_from_host then fetches only the cells under the sampled RoIs' taps from the pinned host maps
    # (csrc/roi_fetch.cu) instead of copying the pyramid.  Bytes moved are counted on the device (cells x C x 4).
    h_feat_cl = [fused.pinned_channels_last(t) for t in h_feat]
    hp_s = hp if hp.groups == 1 else fused.TrainHotPath(B, grids, dev, gt_ld=K_GT, feat_channels=256, layout=1, overlap=True)

    def e2e_sparse_step():
        return hp_s.step_from_host(h_cls, h_reg, h_feat_cl, h_gt, h_gl, gcount, img_hw)

    for _ in range(3):
        e2e_sparse_step()
    torch.cuda.synchronize()
    cells0 = int(hp_s.roi_align.cells_moved[0])
    barrier()
    f0.record()
    for _ in range(n_e2e):
        e2e_sparse_step()
    f1.record()
    barrier()
    e2e_sparse_ms = f0.elapsed_time(f1) / n_e2e
    cells_step = (int(hp_s.roi_align.cells_moved[0]) - cells0) / n_e2e
    h2d_sparse = sum(t.numel() * t.element_size() for t in h_cls + [h_gt, h_gl]) + int(cells_step * 256 * 4)
    # the same with two host batches in flight: two TrainHotPath instances on two streams, called alternately, so that the
    # objectness copy + chains of one batch run under the other's cell fetch (the PCIe link stays busy); secondary number
    e2e_if2_ms = None
    if rank == 0 and world == 1:
        pair = [(hp_s, torch.cuda.Stream(device=dev)),
                (fused.TrainHotPath(B, grids, dev, gt_ld=K_GT, feat_channels=256, layout=1, overlap=True, seed=7), torch.cuda.Stream(device=dev))]
        cur0 = torch.cuda.current_stream()

        def two_host_batches(n):
            for _, st_ in pair:
                st_.wait_stream(cur0)
            for i in range(n):
                hp_i, st_ = pair[i % 2]
                with torch.cuda.stream(st_):
                    hp_i.step_from_host(h_cls, h_reg, h_feat_cl, h_gt, h_gl, gcount, img_hw)
            for _, st_ in pair:
                cur0.wait_stream(st_)

        two_host_batches(4)
        torch.cuda.synchronize()
        n2 = 2 * max(2, n_e2e // 2)
        f0.record()
        two_host_batches(n2)
        f1.record()
        torch.cuda.synchronize()
        e2e_if2_ms = f0.elapsed_time(f1) / n2
        del pair
    if getattr(hp_s, "last_reg_zero_copy", False):
        # regression deltas are read at the selected anchors only, from the mapped host maps: 4 values per anchor of the
        # per-level top-k and per RPN sample, counted as the 32-byte sectors such reads move over PCIe
        h2d_sparse += B * (sum(min(2000, n) for n in hp_s.pyr.level_sizes) + 256) * 4 * 32
    else:
        h2d_sparse += sum(t.numel() * t.element_size() for t in h_reg)
    # the same with the RoI features (the input of the next stage, 205 MB) read back to the host as well
    e2e_feats_ms = None
    if rank == 0:
        hp2 = fused.TrainHotPath(B, grids, dev, gt_ld=K_GT, feat_channels=256, layout=1, overlap=True)
        fn = lambda: hp2.step_from_host(h_cls, h_reg, h_feat_cl, h_gt, h_gl, gcount, img_hw, with_roi_feats=True)
        for _ in range(2):
            fn()
        torch.cuda.synchronize()
        f0.record()
        for _ in range(3):
            fn()
        f1.record()
        torch.cuda.synchronize()
        e2e_feats_ms = f0.elapsed_time(f1) / 3
        del hp2
    sampler.stop_flag = True
    sampler.join(timeout=2)
    # ---- reduce over ranks (max time)
    t = torch.tensor([ms, e2e_ms, nchw_ms, strong_ms or 0.0, e2e_sparse_ms], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms, e2e_ms, nchw_ms, strong_ms = float(t[0]), float(t[1]), float(t[2]), (float(t[3]) if strong_ms is not None else None)
    e2e_sparse_ms = float(t[4])
    total_imgs = B * world
    value = total_imgs * args.steps / (ms / 1e3)
    e2e_val = total_imgs / (e2e_ms / 1e3)
    e2e_sparse_val = total_imgs / (e2e_sparse_ms / 1e3)

    if rank == 0:
        peak, peak_src = peaks()
        bt = out["rcnn"]
        counts = bt.n_chosen.cpu().numpy()
        rois = bt.tar_box.cpu().numpy()
        C = 256
        in_bytes = touched_cell_bytes(rois, counts, grids[:4], strides[:4], C)
        out_bytes = int(counts.sum()) * C * 49 * 4
        roi_bytes = in_bytes + out_bytes + int(counts.sum()) * 16
        # dominant KERNEL of the step: the RoIAlign stage is one launch (k_roi_align_*), 2x the next largest
        # kernel (k_nms_mask_sym); the other stages are chains of several smaller kernels (see stage_ms).
        dom = "roi_align"
        # per-step algorithmic bytes of every stage (SURVEY 8(d)), batch of 8
        n_anchor = hp.pyr.total
        stage_bytes = {
            "proposals": B * (n_anchor * 4 + (4 * 2000 + 819) * 16 + 2000 * 20),
            "rpn_targets": B * (n_anchor * 12 + 256 * 36),
            "roi_targets": B * (2008 * 12 + 2000 * 16 + 512 * 44),
            "roi_align": roi_bytes,
        }
        ach = stage_bytes[dom] / (stage_ms[dom] / 1e3) / 1e9
        path_bytes = sum(stage_bytes.values())
        roofline = {"bound": "hbm", "kernel": {"roi_align": "k_roi_align_win<float>", "proposals": "k_rpn_front + k_rpn_back (K3+K4)",
                                               "rpn_targets": "k_assign_colmax/label (K2)", "roi_targets": "k_assign (K2)"}[dom],
                    "achieved": ach, "peak": peak, "unit": "GB/s", "frac": ach / peak, "traffic": ncu_traffic(dom),
                    "peak_source": peak_src, "algorithmic_bytes_per_launch": stage_bytes[dom],
                    "stage_ms": stage_ms, "stage_algorithmic_bytes": stage_bytes,
                    "stage_ms_note": "eager per-stage CUDA-event times (launch gaps included); the step time above is the "
                                     "CUDA-graph replay",
                    "path_frac": (path_bytes / ((ms / args.steps) / 1e3) / 1e9) / peak,
                    "roi_align_all_2000_proposals": None if k2000_ms is None else {
                        "ms": k2000_ms, "rois": int(hp.proposals.count.sum()), "out_bytes": int(hp.proposals.count.sum()) * C * 49 * 4,
                        "note": "SURVEY 8(d)(ii) stress: every proposal, not the 512 sampled; eager, CUDA events"},
                    "roi_align_bf16_features": None if bf16_ms is None else {
                        "ms": bf16_ms, "algorithmic_bytes": in_bytes // 2 + out_bytes + int(counts.sum()) * 16,
                        "achieved": (in_bytes // 2 + out_bytes + int(counts.sum()) * 16) / (bf16_ms / 1e3) / 1e9,
                        "frac": (in_bytes // 2 + out_bytes + int(counts.sum()) * 16) / (bf16_ms / 1e3) / 1e9 / peak,
                        "note": "same kernel, bf16 NHWC inputs, fp32 accumulation and output; not the parity path"}}
        cpu = None
        if world == 1 and not args.no_cpu:
            import oracle
            from oracle import pipeline as opipe
            oracle.set_num_threads(os.cpu_count())
            path = opipe.ImagePath(grids, strides, w["img_shape"])
            a = ([c[0] for c in w["cls"]], [r[0] for r in w["reg"]], [f[0] for f in w["feats"]], w["gt"][0], w["gt_label"][0])
            path.run(*a)
            t0, n = time.perf_counter(), 0
            while n < 3 or (time.perf_counter() - t0 < 10 and n < 40):
                path.run(*a, seed=n)
                n += 1
            dt = time.perf_counter() - t0
            cpu = {"value": n / dt, "unit": "images/s", "cores": oracle.num_threads(), "kind": "port",
                   "sample": "image 0 of the batch, %d repetitions (%.1f s); C port of the reference path, OpenMP" % (n, dt)}
        sys.stdout.flush()
        os.dup2(real_stdout, 1)
        print(json.dumps({
            "metric": METRIC, "value": value, "unit": "images/s", "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3),
            "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
            "data": "synthetic", "config": workload_config(world),
            "run_config": {"features": "fp32 NHWC (channels_last) resident in HBM", "cuda_graph": graph is not None,
                           "image_groups": hp.groups, "host_cpus_bound_to_gpu_numa_node": numa_cpus},
            "e2e": {"value": e2e_sparse_val, "unit": "images/s", "h2d_bytes_per_step": h2d_sparse, "d2h_bytes_per_step": d2h,
                    "ms_per_step": e2e_sparse_ms,
                    "layout": "TrainHotPath.step_from_host on pinned host buffers, feature maps fp32 channels_last (NHWC strides; what "
                              "install(channels_last=True) makes the reference FPN emit): GT + head maps H2D (copy stream) -> hot path; the "
                              "feature cells under the sampled RoIs' bilinear taps (%.3f of the pyramid, counted on the device) are fetched "
                              "from the mapped host maps by b2d_fetch_marked_cells, the rest never crosses PCIe -> RoIAlign -> D2H of "
                              "proposals / targets.  Results bit-identical to e2e_nchw (tests)." % (
                                  cells_step / float(B * sum(g[0] * g[1] for g in grids[:4])))},
            "e2e_in_flight_2": None if e2e_if2_ms is None else {
                "value": B / (e2e_if2_ms / 1e3), "unit": "images/s", "ms_per_step": e2e_if2_ms, "batches_in_flight": 2,
                "note": "two TrainHotPath instances on two streams, step_from_host called alternately (total time / steps)"},
            "e2e_nchw": {"value": e2e_val, "unit": "images/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                         "ms_per_step": e2e_ms, "layout": "the same call with pinned host fp32 NCHW feature maps (the reference FPN's default "
                                                          "layout): H2D of the whole pyramid (copy stream) -> NCHW->NHWC -> hot path -> D2H; "
                                                          "the PCIe link is the bound (h2d bytes / ms)"},
            "value_nchw": {"value": total_imgs / (nchw_ms / 1e3), "unit": "images/s", "ms_per_step": nchw_ms,
                           "note": "the same step fed with fp32 NCHW features (the reference FPN's layout): + 4 x b2d_nchw_to_nhwc; "
                                   "install(channels_last=True) makes the FPN emit NHWC and removes them"},
            "dropin": dropin,
            "in_flight_2": inflight,
            "strong": None if strong_ms is None else {"global_batch": B, "images_per_gpu": B // world, "ms_per_step": strong_ms,
                                                      "value": B / (strong_ms / 1e3), "unit": "images/s",
                                                      "note": "BASELINE config 2: batch 8 split per image over the ranks"},
            "allgather": None if world == 1 else {"in_timed_loop": True, "bytes_per_rank_and_step": B * hp.proposals.P * 20,
                                                  "what": "proposals [B, 2000, 5] fp32 per rank, written as packed records by the merge kernel; NCCL "
                                                          "all_gather on a side stream after every step, next to the following step (two alternating graphs)"},
            "e2e_with_roi_feats": None if e2e_feats_ms is None else {
                "value": B / (e2e_feats_ms / 1e3), "unit": "images/s (this rank)", "ms_per_step": e2e_feats_ms,
                "d2h_bytes_per_step": d2h + B * 512 * 256 * 49 * 4},
            "gpu_launches": (hp.launches + (1 if world > 1 else 0)) * args.steps, "roofline": roofline, "cpu_baseline": cpu,
            "clocks": sampler.summary()}),
            flush=True)
        os.dup2(2, 1)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--groups", type=int, default=int(os.environ.get("B2D_GROUPS", "1")),
                    help="image groups with staggered stream priorities inside one step (fused.TrainHotPath)")
    ap.add_argument("--no-graph", action="store_true")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-dropin", action="store_true", help="skip the reference-call-sequence measurement")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the outputs of the last timed step (rank 0) to DIR/<name>.npy, float32")
    a = ap.parse_args()
    if a.impl == "reference":
        run_reference(a)
    else:
        run_b200(a)
