"""Batched (all images, all levels, one launch per stage) form of the hot path --
SURVEY 8(f) rank 1: what RPNHead.predict_bboxes_from_output, AnchorHead.loss's target
part, BBoxHead.bbox_targets and BasicRoIExtractor.forward compute per image in Python
loops (lib/heads/anchor_head.py:152-199,268-289; lib/heads/rpn_head.py:68-120;
lib/heads/bbox_head.py:47-52; lib/region.py:301-306) runs here as ~20 kernel launches
per batch with no host synchronisation, no allocation and no [N,K] temporaries, so a
whole step can be captured in a CUDA graph.

Every stage is also reachable through the reference-signature functions in
anchor.py / bbox.py / region.py / utils.py; this module only batches them.
"""
import ctypes
import os

import numpy as np
import torch

from . import _C


def _ptrs(tensors):
    arr = (_C.c_void_p * _C.MAX_LEVELS)()
    for i, t in enumerate(tensors):
        arr[i] = t.data_ptr()
    return arr


def pinned_channels_last(t):
    """Pinned host copy of a [B,C,H,W] tensor in channels_last memory format (NHWC strides): the host-side layout
    TrainHotPath.step_from_host fetches sparsely."""
    B, C, H, W = t.shape
    h = torch.empty((B, H, W, C), dtype=t.dtype, pin_memory=True).permute(0, 3, 1, 2)
    h.copy_(t)
    return h


def _batch_view(obj, b0, b1, rows_per_image=None):
    """Shallow copy of a batched stage object restricted to images [b0, b1): every tensor
    attribute is re-sliced along dim 0 (views, no copies), so a sub-batch can run on its own
    stream while the full-batch object keeps owning the memory."""
    import copy
    v = copy.copy(obj)
    rows_per_image = rows_per_image or {}
    for k, t in list(vars(obj).items()):
        if isinstance(t, torch.Tensor) and t.dim() >= 1 and k not in ("ws", "step_cell"):
            r = rows_per_image.get(k, 1)
            v.__dict__[k] = t[b0 * r:b1 * r]
    v.B, v.b0 = b1 - b0, getattr(obj, "b0", 0) + b0
    return v


class AnchorPyramid(object):
    """Closed-form anchors of an anchor head (lib/heads/anchor_head.py:33-36): per level
    stride == base size, shared scales/ratios; nothing is materialised."""

    def __init__(self, strides, grids, scales=(8,), ratios=(0.5, 1.0, 2.0), center_lt=False):
        self.strides, self.grids = list(strides), [tuple(int(v) for v in g) for g in grids]
        levels = []
        for s, g in zip(self.strides, self.grids):
            ws = [np.float32(s * sc * np.sqrt(ar)) for sc in scales for ar in ratios]   # lib/anchor.py:92-99
            hs = [np.float32(s * sc / np.sqrt(ar)) for sc in scales for ar in ratios]
            levels.append(dict(stride=s, H=g[0], W=g[1], ws=ws, hs=hs, center_lt=center_lt))
        self.num_anchors = len(scales) * len(ratios)
        self.c = _C.make_pyramid(levels)
        self.total = int(self.c.total)
        self.level_sizes = [self.num_anchors * g[0] * g[1] for g in self.grids]


class RpnProposals(object):
    """K3 + K4 over a batch: (cls_outs, reg_outs) -> props [B,4,P], scores [B,P], count [B]."""

    def __init__(self, pyramid, B, cfg, means, stds, device, score_mode=0, cls_channels=1, do_nms=True,
                 scale_factor=1.0):
        self.pyr, self.B = pyramid, B
        get = (lambda k, d=0: cfg.get(k, d)) if hasattr(cfg, "get") else (lambda k, d=0: getattr(cfg, k, d))
        c = _C.RpnCfg()
        c.pre_nms, c.post_nms, c.max_num = int(get("pre_nms")), int(get("post_nms")), int(get("max_num"))
        c.score_mode, c.num_cls_channels, c.do_nms = int(score_mode), int(cls_channels), int(bool(do_nms))
        c.nms_thr_f = _C.floor_f32(float(get("nms_iou", 0.7)))
        c.min_size = float(np.float32(scale_factor * get("min_bbox_size", 0)))
        for i in range(4):
            c.means[i], c.stds[i] = float(means[i]), float(stds[i])
        self.cfg = c
        nbytes = _C.lib().b2d_rpn_proposals_workspace_bytes(ctypes.byref(self.pyr.c), B, ctypes.byref(c))
        if nbytes == 0:
            raise _C.B200DetError("rpn_proposals: unsupported configuration (a level needs a pre-NMS top-k <= 16384)")
        self.ws = torch.empty(nbytes, dtype=torch.uint8, device=device)
        post = [(c.post_nms if 0 < c.post_nms < k else k) for k in
                [(c.pre_nms if 0 < c.pre_nms < n else n) for n in pyramid.level_sizes]]
        self.P = c.max_num if c.max_num > 0 else sum(post)
        self.props = torch.zeros((B, 4, self.P), dtype=torch.float32, device=device)
        self.scores = torch.zeros((B, self.P), dtype=torch.float32, device=device)
        self.count = torch.zeros(B, dtype=torch.int32, device=device)
        self.prov = torch.zeros((B, self.P), dtype=torch.int32, device=device)
        self.launches = 0                       # kernels + memset nodes per call: reported by the library after the first call

    def slice(self, b0, b1):
        v = _batch_view(self, b0, b1)
        nbytes = _C.lib().b2d_rpn_proposals_workspace_bytes(ctypes.byref(self.pyr.c), v.B, ctypes.byref(self.cfg))
        v.ws = torch.empty(nbytes, dtype=torch.uint8, device=self.ws.device)
        return v

    def __call__(self, cls_outs, reg_outs, img_hw, records=None, targets=None, after_select=None):
        """records: optional fp32 [B, P, 5] tensor that receives (x1, y1, x2, y2, score) rows (zero past count): the
        packed detection record of SURVEY 8(e), written by the merge itself so that an all-gather can start right
        after the step without a packing kernel.
        targets: optional (BatchedTargets in its fused form, gt, gt_count, gt_label): bbox_target on the proposals in the
        same library call (b2d_rpn_proposals_targets; the tail of the proposal kernel when that runs as clusters)."""
        self.cfg.records = records.data_ptr() if records is not None else None
        self.cfg.event_after_select = after_select.cuda_event if after_select is not None else None
        if targets is not None:
            bt, gt, gt_count, gt_label = targets
            ta = bt.target_args(gt, gt_count, gt_label)
            _C.call("b2d_rpn_proposals_targets", _C.ptr(self.props), _C.ptr(self.scores), _C.ptr(self.count), _C.ptr(self.prov),
                    _ptrs(cls_outs), _ptrs(reg_outs), ctypes.byref(self.pyr.c), _C.ptr(img_hw), self.B,
                    ctypes.byref(self.cfg), _C.ptr(self.ws), self.ws.numel(), ctypes.byref(ta), _C.stream())
            self.launches = int(_C.lib().b2d_last_launch_count())
            return self.props, self.scores, self.count
        _C.call("b2d_rpn_proposals", _C.ptr(self.props), _C.ptr(self.scores), _C.ptr(self.count), _C.ptr(self.prov),
                _ptrs(cls_outs), _ptrs(reg_outs), ctypes.byref(self.pyr.c), _C.ptr(img_hw), self.B,
                ctypes.byref(self.cfg), _C.ptr(self.ws), self.ws.numel(), _C.stream())
        self.launches = int(_C.lib().b2d_last_launch_count())
        return self.props, self.scores, self.count


class BatchedTargets(object):
    """K2 + sampler + K8 over a batch, for anchors (pyramid mode) or proposals (+ GT prepend)."""

    def __init__(self, B, n_boxes, gt_ld, assigner, sampler, means, stds, device, pyramid=None, border=0.0,
                 prepend_gt=False, seed=0):
        self.B, self.N, self.gt_ld, self.pyr = B, int(n_boxes), int(gt_ld), pyramid
        self.pos_iou, self.neg_iou, self.min_pos = (np.float32(assigner[k]) for k in ("pos_iou", "neg_iou", "min_pos_iou"))
        self.max_num, self.pos_num = int(sampler["max_num"]), int(sampler["pos_num"])
        self.border, self.prepend, self.seed = float(border), int(bool(prepend_gt)), int(seed)
        self.out_ld = self.N + (self.gt_ld if prepend_gt else 0)
        i32, f32, i64 = torch.int32, torch.float32, torch.int64
        self.labels = torch.empty((B, self.out_ld), dtype=i64, device=device)
        self.iou = torch.empty((B, self.out_ld), dtype=f32, device=device)
        self.census = torch.zeros((B, 4), dtype=i32, device=device)
        self.pos_list = torch.empty((B, self.out_ld), dtype=i32, device=device)
        self.colmax = torch.empty((B, self.gt_ld), dtype=i32, device=device)
        self.chosen = torch.empty((B, self.max_num), dtype=i32, device=device)
        self.n_chosen = torch.zeros(B, dtype=i32, device=device)
        self.tar_box = torch.zeros((B, 4, self.max_num), dtype=f32, device=device)
        self.tar_gt = torch.zeros((B, 4, self.max_num), dtype=f32, device=device)
        self.tar_param = torch.zeros((B, 4, self.max_num), dtype=f32, device=device)
        self.tar_label = torch.zeros((B, self.max_num), dtype=i64, device=device)
        self.tar_is_gt = torch.zeros((B, self.max_num), dtype=i64, device=device)
        self.means, self.stds = _C.host_f4(means, [0, 0, 0, 0]), _C.host_f4(stds, [1, 1, 1, 1])
        # per-step counter of the device sampler, in DEVICE memory: a CUDA-graph replay re-reads it, a by-value
        # seed would be frozen by the capture (every replay would keep the same positives / negative walk)
        self.step_cell = torch.zeros(1, dtype=torch.int64, device=device)
        self.auto_bump = True                   # False: the owner (TrainHotPath) advances a shared cell once per step
        self.b0 = 0
        small = pyramid is None and self.N <= 4096 and self.gt_ld <= 512
        # bbox_target in one launch (b2d_roi_targets_fused) when the problem fits one CTA per image
        self.fused = small and self.max_num <= 1024
        # kernels: roi_targets_small | assign_small | (colmax_rect, label_rows) | (fill, colmax, label); then sample, encode
        self.launches = 1 if self.fused else (3 if small else (4 if pyramid is not None else 5))      # (+1: counter, if auto_bump)

    def reset_step(self):
        """Restart the device sampler's step counter (tests: the same random stream again)."""
        self.step_cell.zero_()

    def target_args(self, gt, gt_count, gt_label):
        """The arguments of b2d_roi_targets_fused as the struct b2d_rpn_proposals_targets takes (fused form only)."""
        assert self.fused
        a = _C.RoiTargetArgs()
        dp = lambda t: t.data_ptr() if t is not None else None
        a.labels, a.max_iou, a.out_ld = dp(self.labels), dp(self.iou), self.out_ld
        a.gt, a.gt_ld, a.gt_count, a.gt_label = dp(gt), self.gt_ld, dp(gt_count), dp(gt_label)
        a.pos_iou, a.neg_iou, a.min_pos_iou = float(self.pos_iou), float(self.neg_iou), float(self.min_pos)
        a.prepend_gt, a.census, a.pos_list, a.pos_cap = self.prepend, dp(self.census), dp(self.pos_list), self.out_ld
        a.chosen, a.n_chosen, a.max_num, a.pos_num = dp(self.chosen), dp(self.n_chosen), self.max_num, self.pos_num
        a.seed = (self.seed * 1000003 + 0x632BE59BD9B4E019 * self.b0) & 0xFFFFFFFFFFFFFFFF
        a.seed_step = dp(self.step_cell)
        a.tar_box, a.tar_gt, a.tar_param = dp(self.tar_box), dp(self.tar_gt), dp(self.tar_param)
        a.tar_label, a.tar_is_gt = dp(self.tar_label), dp(self.tar_is_gt)
        for i in range(4):
            a.means[i], a.stds[i] = self.means[i], self.stds[i]
        return a

    def slice(self, b0, b1):
        return _batch_view(self, b0, b1)

    def __call__(self, gt, gt_count, gt_label=None, boxes=None, box_count=None, img_hw=None, tail_stream=None):
        """tail_stream: optional stream for the sampler + encode kernels (they start when the assignment is done)."""
        pyr = ctypes.byref(self.pyr.c) if boxes is None else None
        box_ld = boxes.shape[-1] if boxes is not None else 0
        if self.auto_bump:
            _C.call("b2d_counter_add", _C.ptr(self.step_cell), 1, _C.stream())
        base_seed = (self.seed * 1000003 + 0x632BE59BD9B4E019 * self.b0) & 0xFFFFFFFFFFFFFFFF
        if self.fused and boxes is not None:
            _C.call("b2d_roi_targets_fused", _C.ptr(self.labels), _C.ptr(self.iou), self.out_ld, _C.ptr(boxes), box_ld,
                    _C.ptr(box_count), self.N, _C.ptr(gt), self.gt_ld, _C.ptr(gt_count), _C.ptr(gt_label), self.B,
                    float(self.pos_iou), float(self.neg_iou), float(self.min_pos), self.prepend, _C.ptr(self.census),
                    _C.ptr(self.pos_list), self.out_ld, _C.ptr(self.chosen), _C.ptr(self.n_chosen), self.max_num,
                    self.pos_num, base_seed, _C.ptr(self.step_cell),
                    _C.ptr(self.tar_box), _C.ptr(self.tar_gt), _C.ptr(self.tar_param), _C.ptr(self.tar_label),
                    _C.ptr(self.tar_is_gt), self.means, self.stds, _C.stream())
            return self
        _C.call("b2d_assign_max_iou", _C.ptr(self.labels), _C.ptr(self.iou), self.out_ld, _C.ptr(boxes), box_ld,
                _C.ptr(box_count), self.N, pyr, _C.ptr(img_hw), self.border, _C.ptr(gt), self.gt_ld, _C.ptr(gt_count),
                self.B, float(self.pos_iou), float(self.neg_iou), float(self.min_pos), self.prepend,
                _C.ptr(self.census), _C.ptr(self.pos_list), self.out_ld, _C.ptr(self.colmax), self.colmax.numel() * 4,
                _C.stream())
        cnt, cnt_add = (box_count, gt_count) if (self.prepend and box_count is not None) else \
            ((None, gt_count) if self.prepend else (box_count, None))
        n = self.N if cnt is None else 0
        if tail_stream is not None:
            tail_stream.wait_stream(torch.cuda.current_stream())
            with torch.cuda.stream(tail_stream):
                self._sample_encode(cnt, cnt_add, n, base_seed, boxes, box_ld, pyr, gt, gt_count, gt_label)
            return self
        self._sample_encode(cnt, cnt_add, n, base_seed, boxes, box_ld, pyr, gt, gt_count, gt_label)
        return self

    def _sample_encode(self, cnt, cnt_add, n, base_seed, boxes, box_ld, pyr, gt, gt_count, gt_label):
        _C.call("b2d_sample_labels", _C.ptr(self.chosen), _C.ptr(self.n_chosen), _C.ptr(self.labels), self.out_ld,
                _C.ptr(cnt), _C.ptr(cnt_add), n, _C.ptr(self.census), _C.ptr(self.pos_list), self.out_ld, self.B,
                self.max_num, self.pos_num, base_seed, _C.ptr(self.step_cell), _C.stream())
        _C.call("b2d_encode_targets", _C.ptr(self.tar_box), _C.ptr(self.tar_gt), _C.ptr(self.tar_param),
                _C.ptr(self.tar_label), _C.ptr(self.tar_is_gt), _C.ptr(self.chosen), _C.ptr(self.n_chosen),
                self.max_num, _C.ptr(self.labels), self.out_ld, _C.ptr(boxes), box_ld, pyr, _C.ptr(gt), self.gt_ld,
                _C.ptr(gt_count), _C.ptr(gt_label), self.prepend, self.means, self.stds, self.B, _C.stream())
        return self


class BatchedRoIAlign(object):
    """K5 over a batch: rois [B,4,ld] + counts -> [B*ld, C, PH, PW] (image-major rows)."""

    def __init__(self, B, ld, feat_shapes, strides, device, out_size=(7, 7), sampling_ratio=2, finest_scale=56,
                 layout=1):
        cfg = _C.RoiCfg()
        cfg.num_levels, cfg.C = len(strides), int(feat_shapes[0][0])
        cfg.PH, cfg.PW, cfg.sampling_ratio, cfg.aligned = int(out_size[0]), int(out_size[1]), int(sampling_ratio), 0
        cfg.layout, cfg.finest_scale = int(layout), float(finest_scale)
        for l, (s, shp) in enumerate(zip(strides, feat_shapes)):
            cfg.H[l], cfg.W[l], cfg.spatial_scale[l] = int(shp[1]), int(shp[2]), 1.0 / float(s)
        self.cfg, self.B, self.ld = cfg, B, ld
        self.out = torch.zeros((B * ld, cfg.C, cfg.PH, cfg.PW), dtype=torch.float32, device=device)
        self.launches = 1

    def slice(self, b0, b1):
        return _batch_view(self, b0, b1, rows_per_image={"out": self.ld})

    def __call__(self, feats, rois, counts):
        _C.call("b2d_roi_align_fwd_batched", _C.ptr(self.out), _ptrs(feats), _C.ptr(rois), self.ld, _C.ptr(counts),
                self.B, ctypes.byref(self.cfg), _C.stream())
        return self.out

    def fetch_touched(self, dev_feats, host_feats, rois, counts):
        """Bring the cells these RoIs read -- and only those -- from channels-last PINNED HOST feature maps into the
        device maps (b2d_roi_mark_cells + b2d_fetch_marked_cells, csrc/roi_fetch.cu): 59 % of the pyramid at config 2.
        Returns the device counter of cells moved so far (cumulative)."""
        if not hasattr(self, "_bitmap"):
            n = _C.lib().b2d_roi_cell_bitmap_bytes(self.B, ctypes.byref(self.cfg))
            self._bitmap = torch.zeros(n, dtype=torch.uint8, device=self.out.device)
            self.cells_moved = torch.zeros(1, dtype=torch.int64, device=self.out.device)
        for d, h in zip(dev_feats, host_feats):
            if not (h.is_pinned() and d.is_cuda and d.shape == h.shape and d.dtype == h.dtype and d.stride() == h.stride()
                    and h.is_contiguous(memory_format=torch.channels_last)):
                raise _C.B200DetError("fetch_touched: host maps must be pinned channels_last tensors matching the device maps")
        _C.call("b2d_roi_mark_cells", _C.ptr(self._bitmap), _C.ptr(rois), self.ld, _C.ptr(counts), self.B,
                ctypes.byref(self.cfg), _C.stream())
        _C.call("b2d_fetch_marked_cells", _ptrs(dev_feats), _ptrs(host_feats), _C.ptr(self._bitmap), self.B,
                ctypes.byref(self.cfg), _C.ptr(self.cells_moved), _C.stream())
        return self.cells_moved


class TrainHotPath(object):
    """faster_rcnn_r50_fpn train path (BASELINE config 2): RPN proposals (K3+K4), RPN
    anchor targets (K2, sampler, K8, head-output gather), RoI targets on the proposals
    (K2 + GT prepend, sampler, K8) and FPN RoIAlign of the sampled RoIs (K5).
    Mirrors CascadeRCNN.forward_train lines 106-131 (lib/detectors/cascade_rcnn.py)
    minus convolutions and losses."""

    def __init__(self, B, grids, device, strides=(4, 8, 16, 32, 64), gt_ld=64, feat_channels=256,
                 rpn_proposal=None, rpn_assigner=None, rpn_sampler=None, rcnn_assigner=None, rcnn_sampler=None,
                 rpn_stds=(1.0, 1.0, 1.0, 1.0), rcnn_stds=(0.1, 0.1, 0.2, 0.2), allowed_border=0, layout=1, seed=0,
                 groups=1, overlap=False, order=None):
        z4 = (0.0, 0.0, 0.0, 0.0)
        self.order = order or os.environ.get("B2D_STEP_ORDER", "rpn_first")
        self.ev_select = torch.cuda.Event()
        self.ev_select.record()                              # (creates the CUDA event behind the handle)
        self.fuse_targets = os.environ.get("B2D_FUSE_TARGETS", "0") != "0"      # bbox_target as the tail of the proposal kernel (measured r2: 258.8 vs 251.2 us separate -> off)
        rpn_proposal = rpn_proposal or dict(pre_nms=2000, post_nms=2000, max_num=2000, nms_iou=0.7, min_bbox_size=0)
        rpn_assigner = rpn_assigner or dict(pos_iou=0.7, neg_iou=0.3, min_pos_iou=0.3)
        rpn_sampler = rpn_sampler or dict(max_num=256, pos_num=128)
        rcnn_assigner = rcnn_assigner or dict(pos_iou=0.5, neg_iou=0.5, min_pos_iou=0.5)
        rcnn_sampler = rcnn_sampler or dict(max_num=512, pos_num=128)
        self.B, self.device = B, device
        self.pyr = AnchorPyramid(strides, grids)
        self.proposals = RpnProposals(self.pyr, B, rpn_proposal, z4, rpn_stds, device)
        self.rpn_targets = BatchedTargets(B, self.pyr.total, gt_ld, rpn_assigner, rpn_sampler, z4, rpn_stds, device,
                                          pyramid=self.pyr, border=allowed_border, seed=seed)
        self.roi_targets = BatchedTargets(B, self.proposals.P, gt_ld, rcnn_assigner, rcnn_sampler, z4, rcnn_stds,
                                          device, prepend_gt=True, seed=seed + 1)
        # one device-side step counter for both samplers (graph-replay safe): starts at 1 and is advanced once per step
        # AFTER both samplers have read it, on a side stream next to RoIAlign (off the critical path)
        self.step_cell = torch.ones(1, dtype=torch.int64, device=device)
        self.s_bump = torch.cuda.Stream(device=device)
        for t in (self.rpn_targets, self.roi_targets):
            t.step_cell, t.auto_bump = self.step_cell, False
        roi_strides = list(strides[:4])
        shapes = [(feat_channels, g[0], g[1]) for g in grids[:4]]
        self.roi_align = BatchedRoIAlign(B, rcnn_sampler["max_num"], shapes, roi_strides, device, layout=layout)
        m = rpn_sampler["max_num"]
        self.tar_cls = torch.zeros((B, 1, m), dtype=torch.float32, device=device)
        self.tar_reg = torch.zeros((B, 4, m), dtype=torch.float32, device=device)
        # Stream plan.  The proposal chain (top-k -> NMS scan -> merge) is a sequence of small,
        # latency-bound grids, the RPN-target and RoIAlign kernels are throughput-bound, and the
        # images are independent, so the batch is cut into `groups` sub-batches whose chains
        # (proposals -> RoI targets -> RoIAlign) run on their own streams next to the RPN-target
        # chain: latency-bound kernels of one group fill the SMs the others leave idle.  Under
        # CUDA-graph capture the fork/join below becomes parallel graph branches.
        groups = max(1, min(int(groups), B))
        while B % groups:
            groups -= 1
        self.groups = groups
        self.subs = []
        if groups > 1 or overlap:
            per = B // groups
            for g in range(groups):
                b0, b1 = g * per, (g + 1) * per
                self.subs.append((b0, b1, self.proposals.slice(b0, b1) if groups > 1 else self.proposals,
                                  self.roi_targets.slice(b0, b1) if groups > 1 else self.roi_targets,
                                  self.roi_align.slice(b0, b1) if groups > 1 else self.roi_align,
                                  # Priorities stagger the groups: group 0's chain wins every SM slot it asks for, so it
                                  # reaches its RoIAlign (HBM-bound) while the later groups are still in their NMS masks
                                  # (ALU-bound) -- the two overlap instead of running back to back.  RoIAlign streams
                                  # rank below every chain, the RPN-target chain (off the critical path) lowest.
                                  torch.cuda.Stream(device=device, priority=-4 + min(g, 2)),       # proposal / target chain
                                  torch.cuda.Stream(device=device, priority=-2 + min(g, 1))))      # RoIAlign (throughput)
            # RPN-target chain: its two ALU-bound kernels (colmax 17 us + label rows 35 us at config 2) should run
            # while the proposal chains sit in hist / compact / select (latency-bound, ~50 us, SMs idle): lowest
            # priority (the small critical kernels always get their SM slots) but enqueued first, see step()
            self.s_rpn = torch.cuda.Stream(device=device, priority=int(os.environ.get("B2D_RPN_PRIO", "0")))
            # optional: the sampler / encode / gather tail of the RPN-target chain on its own stream ABOVE RoIAlign in
            # priority (B2D_RPN_TAIL_PRIO, e.g. -5), with slim sampler CTAs (B2D_SAMPLE_THREADS=128) that fit the hole a
            # retiring RoIAlign CTA leaves -- so that the tail is not starved when RoIAlign starts before K2 has finished
            tp = os.environ.get("B2D_RPN_TAIL_PRIO", "")
            self.s_tail = torch.cuda.Stream(device=device, priority=int(tp)) if tp else None
        self.launches = 0

    def reset_step(self):
        """Restart the samplers' step counter (tests: the same random stream again)."""
        self.step_cell.fill_(1)

    def _rpn_target_chain(self, cls_outs, reg_outs, gt, gt_count, img_hw):
        tail = getattr(self, "s_tail", None)
        rt = self.rpn_targets(gt, gt_count, None, img_hw=img_hw, tail_stream=tail)
        cur = torch.cuda.current_stream()
        with torch.cuda.stream(tail if tail is not None else cur):
            _C.call("b2d_gather_head_outputs", _C.ptr(self.tar_cls), _C.ptr(self.tar_reg), _ptrs(cls_outs), _ptrs(reg_outs),
                    ctypes.byref(self.pyr.c), 1, _C.ptr(rt.chosen), _C.ptr(rt.n_chosen), rt.max_num, self.B, _C.stream())
        if tail is not None:
            cur.wait_stream(tail)                        # the chain's stream ends where its tail ends (joins below see both)
        return rt

    def step(self, cls_outs, reg_outs, feats, gt, gt_count, gt_label, img_hw, feats_ready=None, records=None,
             before_roi_align=None):
        """One pass of the hot path over the batch (device-resident inputs).  `feats_ready`: optional
        CUDA event after which `feats` may be read (lets the proposal / target chains start while
        the feature maps are still arriving, see step_from_host).  `before_roi_align(rois, counts)`: optional
        callable run on RoIAlign's stream once the sampled RoIs exist (step_from_host: fetch of the touched cells)."""
        if not self.subs:
            if feats_ready is not None:
                torch.cuda.current_stream().wait_event(feats_ready)
            ride = self.roi_targets.fused and self.fuse_targets
            props, scores, count = self.proposals(cls_outs, reg_outs, img_hw, records=records,
                                                  targets=(self.roi_targets, gt, gt_count, gt_label) if ride else None)
            rt = self._rpn_target_chain(cls_outs, reg_outs, gt, gt_count, img_hw)
            bt = self.roi_targets if ride else self.roi_targets(gt, gt_count, gt_label, boxes=props, box_count=count)
            _C.call("b2d_counter_add", _C.ptr(self.step_cell), 1, _C.stream())      # both samplers have read it
            if before_roi_align is not None:
                before_roi_align(bt.tar_box, bt.n_chosen)
            self.roi_align(feats, bt.tar_box, bt.n_chosen)
        else:
            cur = torch.cuda.current_stream()
            # Graph nodes launch in creation order.  order "rpn_first" (default): the RPN-target kernels (ALU-bound,
            # thousands of CTAs) are enqueued before the proposal stage; "chain_first": the proposal stage's cluster
            # kernels (1024-thread CTAs that need whole SMs) first.  Measured at config 2 (r2l): 257 vs 275 us per step --
            # enqueued second, the RPN-target grid only gets the SMs the clusters leave and spills into RoIAlign.
            rpn_first = self.order == "rpn_first"
            self.s_rpn.wait_stream(cur)
            if rpn_first:
                with torch.cuda.stream(self.s_rpn):
                    rt = self._rpn_target_chain(cls_outs, reg_outs, gt, gt_count, img_hw)
            for gi, (b0, b1, prop, tgt, ra, st, st_lo) in enumerate(self.subs):
                st.wait_stream(cur)
                ride = tgt.fused and self.fuse_targets
                ev = self.ev_select if (gi == 0 and self.order == "rpn_after_select") else None
                with torch.cuda.stream(st):
                    p, _, c = prop([t[b0:b1] for t in cls_outs], [t[b0:b1] for t in reg_outs], img_hw[b0:b1],
                                   records=records[b0:b1] if records is not None else None,
                                   targets=(tgt, gt[b0:b1], gt_count[b0:b1], gt_label[b0:b1]) if ride else None,
                                   after_select=ev)
                if gi == 0 and not rpn_first:
                    if self.order == "rpn_late":         # behind the proposal stage: next to RoI targets + RoIAlign
                        self.s_rpn.wait_stream(st)
                    if ev is not None:                   # behind the selection kernel, beside NMS / merge / RoI targets
                        self.s_rpn.wait_event(ev)
                    with torch.cuda.stream(self.s_rpn):
                        rt = self._rpn_target_chain(cls_outs, reg_outs, gt, gt_count, img_hw)
                with torch.cuda.stream(st):
                    t2 = tgt if ride else tgt(gt[b0:b1], gt_count[b0:b1], gt_label[b0:b1], boxes=p, box_count=c)
                st_lo.wait_stream(st)
                if feats_ready is not None:
                    st_lo.wait_event(feats_ready)
                with torch.cuda.stream(st_lo):
                    if before_roi_align is not None:
                        if self.groups != 1:
                            raise _C.B200DetError("before_roi_align needs groups == 1")
                        before_roi_align(t2.tar_box, t2.n_chosen)
                    ra([f[b0:b1] for f in feats], t2.tar_box, t2.n_chosen)
            # the step counter moves on once every sampler of the step has read it: side stream, next to RoIAlign
            for sub in self.subs:
                self.s_bump.wait_stream(sub[-2])
            self.s_bump.wait_stream(self.s_rpn)
            with torch.cuda.stream(self.s_bump):
                _C.call("b2d_counter_add", _C.ptr(self.step_cell), 1, _C.stream())
            for sub in self.subs:
                cur.wait_stream(sub[-1])
            cur.wait_stream(self.s_rpn)
            cur.wait_stream(self.s_bump)
        self.launches = (sum(sub[2].launches for sub in self.subs) if self.groups > 1 else self.proposals.launches) + \
            ((0 if (self.roi_targets.fused and self.fuse_targets) else self.roi_targets.launches) + 1) * self.groups + \
            self.rpn_targets.launches + 1 + 1
        return dict(props=self.proposals.props, scores=self.proposals.scores, prop_count=self.proposals.count,
                    rpn=self.rpn_targets, rpn_tar_cls=self.tar_cls, rpn_tar_reg=self.tar_reg, rcnn=self.roi_targets,
                    roi_feats=self.roi_align.out)

    # ------------------------------------------------------------------ host-buffer entry
    def step_from_host(self, h_cls, h_reg, h_feats, h_gt, h_gt_label, gt_count, img_hw, h_out=None,
                       with_roi_feats=False, sparse=None):
        """End-to-end form of step(): inputs are pinned HOST tensors in the reference's layout
        (head maps [B,A*C,H,W] / [B,4A,H,W], FPN features fp32 NCHW [B,C,H,W], GT [B,4,K] and
        labels [B,K]); results land in pinned host tensors (`h_out`, allocated on first use).
        The H2D copies run on a copy stream in the order GT, head maps, features (largest level
        first); the proposal and target chains start as soon as the head maps have landed, each
        feature level is transposed to NHWC (b2d_nchw_to_nhwc) while the next one is still in
        flight, and only RoIAlign waits for the features.  gt_count / img_hw are device tensors.
        The RoI features (the input of the next GPU stage, 205 MB at config 2) stay on the device
        unless with_roi_feats is set; a one-element probe of them is always read back.

        `sparse` (default: chosen by the layout of h_feats): when the host feature maps are channels_last
        ([B,C,H,W] tensors with NHWC strides, what `install(channels_last=True)` makes the FPN emit) they are not
        copied at all -- once the sampled RoIs exist, the cells under their bilinear taps are fetched straight from
        the pinned host maps by the SMs (BatchedRoIAlign.fetch_touched) and RoIAlign reads those.  Same results,
        ~0.6 of the bytes over PCIe at config 2.  NCHW host maps take the full copy + transposition."""
        dev, B = self.device, self.B
        cl = all(t.dim() == 4 and t.is_contiguous(memory_format=torch.channels_last) and not t.is_contiguous()
                 for t in h_feats)
        if sparse is None:
            sparse = cl and all(t.is_pinned() for t in h_feats)
        if sparse:
            return self._step_from_host_sparse(h_cls, h_reg, h_feats, h_gt, h_gt_label, gt_count, img_hw, h_out,
                                               with_roi_feats)
        if not hasattr(self, "_stage"):
            st = dict(cls=[torch.empty(t.shape, dtype=t.dtype, device=dev) for t in h_cls],
                      reg=[torch.empty(t.shape, dtype=t.dtype, device=dev) for t in h_reg],
                      feat=[torch.empty(t.shape, dtype=t.dtype, device=dev) for t in h_feats],
                      nhwc=[torch.empty(t.shape, dtype=t.dtype, device=dev).contiguous(memory_format=torch.channels_last)
                            for t in h_feats],
                      gt=torch.empty(h_gt.shape, dtype=h_gt.dtype, device=dev),
                      gl=torch.empty(h_gt_label.shape, dtype=h_gt_label.dtype, device=dev),
                      s_copy=torch.cuda.Stream(device=dev), s_xpose=torch.cuda.Stream(device=dev, priority=0),
                      ev_heads=torch.cuda.Event(), ev_feat=[torch.cuda.Event() for _ in h_feats],
                      ev_ready=torch.cuda.Event())
            self._stage = st
        st = self._stage
        if h_out is None:
            h_out = self._host_results(with_roi_feats)
        cur = torch.cuda.current_stream()
        sc, sx = st["s_copy"], st["s_xpose"]
        sc.wait_stream(cur)
        sx.wait_stream(cur)
        with torch.cuda.stream(sc):
            st["gt"].copy_(h_gt, non_blocking=True)
            st["gl"].copy_(h_gt_label, non_blocking=True)
            for d, h in zip(st["cls"] + st["reg"], list(h_cls) + list(h_reg)):
                d.copy_(h, non_blocking=True)
            st["ev_heads"].record(sc)
            for l in sorted(range(len(h_feats)), key=lambda i: -h_feats[i].numel()):
                st["feat"][l].copy_(h_feats[l], non_blocking=True)
                st["ev_feat"][l].record(sc)
        with torch.cuda.stream(sx):
            for l in sorted(range(len(h_feats)), key=lambda i: -h_feats[i].numel()):
                sx.wait_event(st["ev_feat"][l])
                f = st["feat"][l]
                _C.call("b2d_nchw_to_nhwc", _C.ptr(st["nhwc"][l]), _C.ptr(f), f.shape[0], f.shape[1], f.shape[2],
                        f.shape[3], _C.stream())
            st["ev_ready"].record(sx)
        cur.wait_event(st["ev_heads"])
        out = self.step(st["cls"], st["reg"], st["nhwc"], st["gt"], gt_count, st["gl"], img_hw, feats_ready=st["ev_ready"])
        return self._read_back(out, h_out)

    def _host_results(self, with_roi_feats):
        if not hasattr(self, "_h_out"):
            pin = lambda t: torch.empty(t.shape, dtype=t.dtype).pin_memory()
            rt, bt = self.rpn_targets, self.roi_targets
            self._h_out = dict(props=pin(self.proposals.props), scores=pin(self.proposals.scores),
                               prop_count=pin(self.proposals.count), rpn_label=pin(rt.tar_label),
                               rpn_param=pin(rt.tar_param), rpn_tar_cls=pin(self.tar_cls), rpn_tar_reg=pin(self.tar_reg),
                               roi_label=pin(bt.tar_label), roi_param=pin(bt.tar_param), roi_count=pin(bt.n_chosen),
                               roi_probe=torch.empty(1).pin_memory())
        if with_roi_feats and "roi_feats" not in self._h_out:
            self._h_out["roi_feats"] = torch.empty(self.roi_align.out.shape, dtype=self.roi_align.out.dtype).pin_memory()
        return self._h_out

    @staticmethod
    def _read_back(out, h_out):
        pairs = [("props", out["props"]), ("scores", out["scores"]), ("prop_count", out["prop_count"]),
                 ("rpn_label", out["rpn"].tar_label), ("rpn_param", out["rpn"].tar_param),
                 ("rpn_tar_cls", out["rpn_tar_cls"]), ("rpn_tar_reg", out["rpn_tar_reg"]),
                 ("roi_label", out["rcnn"].tar_label), ("roi_param", out["rcnn"].tar_param),
                 ("roi_count", out["rcnn"].n_chosen), ("roi_feats", out["roi_feats"]),
                 ("roi_probe", out["roi_feats"][0, 0, 0, :1])]
        for k, t in pairs:
            if k in h_out:
                h_out[k].copy_(t, non_blocking=True)
        return h_out

    def _step_from_host_sparse(self, h_cls, h_reg, h_feats, h_gt, h_gt_label, gt_count, img_hw, h_out, with_roi_feats):
        """step_from_host for channels_last pinned host feature maps: GT + objectness maps by H2D copy (8.6 MB at
        config 2), proposal / target chains, then only the cells the sampled RoIs touch are fetched from the host maps.
        The regression maps (34 MB) are not copied either when they are pinned: the kernels read them only at the
        selected anchors (k_rpn_front's decode of the per-level top-k, b2d_gather_head_outputs at the 256 samples) and
        take those 4-byte values straight from the mapped host maps (`self.reg_zero_copy`, default on)."""
        dev = self.device
        if self.groups != 1:
            raise _C.B200DetError("step_from_host(sparse): image groups are not supported")
        if not hasattr(self, "_stage_sparse"):
            self._stage_sparse = dict(
                cls=[torch.empty(t.shape, dtype=t.dtype, device=dev) for t in h_cls],
                reg=None,
                # zero-filled once: cells no RoI has touched yet are never read, but stay finite for debuggers
                nhwc=[torch.zeros(t.shape, dtype=t.dtype, device=dev).contiguous(memory_format=torch.channels_last)
                      for t in h_feats],
                gt=torch.empty(h_gt.shape, dtype=h_gt.dtype, device=dev),
                gl=torch.empty(h_gt_label.shape, dtype=h_gt_label.dtype, device=dev),
                s_copy=torch.cuda.Stream(device=dev), ev_heads=torch.cuda.Event())
        st = self._stage_sparse
        if h_out is None:
            h_out = self._host_results(with_roi_feats)
        cur = torch.cuda.current_stream()
        sc = st["s_copy"]
        sc.wait_stream(cur)
        zc_reg = getattr(self, "reg_zero_copy", True) and all(t.is_pinned() and t.is_contiguous() for t in h_reg)
        if not zc_reg and st["reg"] is None:
            st["reg"] = [torch.empty(t.shape, dtype=t.dtype, device=dev) for t in h_reg]
        with torch.cuda.stream(sc):
            st["gt"].copy_(h_gt, non_blocking=True)
            st["gl"].copy_(h_gt_label, non_blocking=True)
            for d, h in zip(st["cls"] + ([] if zc_reg else st["reg"]), list(h_cls) + ([] if zc_reg else list(h_reg))):
                d.copy_(h, non_blocking=True)
            st["ev_heads"].record(sc)
        cur.wait_event(st["ev_heads"])
        fetch = lambda rois, counts: self.roi_align.fetch_touched(st["nhwc"], h_feats, rois, counts)
        out = self.step(st["cls"], list(h_reg) if zc_reg else st["reg"], st["nhwc"], st["gt"], gt_count, st["gl"], img_hw,
                        before_roi_align=fetch)
        self.last_reg_zero_copy = zc_reg
        return self._read_back(out, h_out)


class CascadeHotPath(object):
    """The stage loop of CascadeRCNN.forward_train (lib/detectors/cascade_rcnn.py:119-153; BASELINE config 3) minus
    the head convolutions and losses, batched: per stage bbox_target on the current boxes (b2d_roi_targets_fused,
    thresholds .5/.6/.7) -> FPN RoIAlign of the sampled RoIs (K5) -> [RCNN head: the caller's reg_out] ->
    BBoxHead.refine_bboxes (b2d_refine_bboxes, stage stds, GT columns dropped) -> next stage's boxes; and the RoIAlign
    backward of every stage (K6).  Allocation- and sync-free after construction (CUDA-graph capturable)."""

    def __init__(self, B, n_props, grids, device, strides=(4, 8, 16, 32), gt_ld=64, feat_channels=256,
                 thresholds=(0.5, 0.6, 0.7),
                 stage_stds=((0.1, 0.1, 0.2, 0.2), (0.05, 0.05, 0.1, 0.1), (0.033, 0.033, 0.067, 0.067)),
                 sampler=None, num_classes=21, layout=1, seed=0):
        sampler = sampler or dict(max_num=512, pos_num=128)
        z4 = (0.0, 0.0, 0.0, 0.0)
        self.B, self.m, self.C = B, int(sampler["max_num"]), int(num_classes)
        shapes = [(feat_channels, g[0], g[1]) for g in grids[:len(strides)]]
        self.stages = []
        n = int(n_props)
        for s, (thr, sd) in enumerate(zip(thresholds, stage_stds)):
            tg = BatchedTargets(B, n, gt_ld, dict(pos_iou=thr, neg_iou=thr, min_pos_iou=thr), sampler, z4, sd, device,
                                prepend_gt=True, seed=seed + s)
            ra = BatchedRoIAlign(B, self.m, shapes, list(strides), device, layout=layout)
            refined = torch.zeros((B, 4, self.m), dtype=torch.float32, device=device)
            rcount = torch.zeros(B, dtype=torch.int32, device=device)
            self.stages.append((tg, ra, refined, rcount, _C.host_f4(sd, [1, 1, 1, 1])))
            n = self.m
        self.step_cell = torch.zeros(1, dtype=torch.int64, device=device)        # one step counter for all stages
        for st in self.stages:
            st[0].step_cell, st[0].auto_bump = self.step_cell, False
        self.roi_img = torch.arange(B, dtype=torch.int32, device=device).repeat_interleave(self.m).contiguous()
        self.rois_flat = [torch.zeros((4, B * self.m), dtype=torch.float32, device=device) for _ in self.stages]
        mf = torch.channels_last if layout != 0 else torch.contiguous_format
        self.grads = [[torch.zeros((B,) + shp, dtype=torch.float32, device=device).contiguous(memory_format=mf) for shp in shapes]
                      for _ in self.stages]
        self.bwd_cfg = self.stages[0][1].cfg
        nb = _C.lib().b2d_roi_align_bwd_workspace_bytes(B * self.m, B, ctypes.byref(self.bwd_cfg))
        self.bwd_ws = torch.empty(nb, dtype=torch.uint8, device=device)
        self.zero4 = _C.host_f4(z4, [0, 0, 0, 0])
        self.launches = len(self.stages) * (1 + 1 + 1) + 1

    def step(self, props, prop_count, feats, gt, gt_count, gt_label, img_hw, reg_outs):
        """props [B,4,n_props] + prop_count; reg_outs[s]: the stage head's regression output [B, max_num, 4*num_classes]
        (rows in the order of the stage's sampled RoIs).  Returns the per-stage (targets, roi features, refined boxes,
        counts)."""
        outs = []
        boxes, count = props, prop_count
        _C.call("b2d_counter_add", _C.ptr(self.step_cell), 1, _C.stream())
        for s, (tg, ra, refined, rcount, stds) in enumerate(self.stages):
            bt = tg(gt, gt_count, gt_label, boxes=boxes, box_count=count)
            ra(feats, bt.tar_box, bt.n_chosen)
            _C.call("b2d_refine_bboxes", _C.ptr(refined), _C.ptr(rcount), _C.ptr(bt.tar_box), self.m, _C.ptr(bt.n_chosen),
                    self.m, _C.ptr(bt.tar_label), _C.ptr(reg_outs[s]), self.C, _C.ptr(bt.tar_is_gt), self.zero4, stds, 1,
                    _C.ptr(img_hw), self.B, _C.stream())
            outs.append((bt, ra.out, refined, rcount))
            boxes, count = refined, rcount
        return outs

    def backward(self, grad_feats):
        """grad_feats[s] [B*max_num, C, 7, 7] (zero rows for unused slots) -> per-stage feature gradients (K6);
        the caller (autograd in the reference) adds the stages."""
        for s, (tg, ra, _, _, _) in enumerate(self.stages):
            self.rois_flat[s].copy_(tg.tar_box.permute(1, 0, 2).reshape(4, -1))
            arr = (_C.c_void_p * _C.MAX_LEVELS)()
            for i, g in enumerate(self.grads[s]):
                arr[i] = g.data_ptr()
            _C.call("b2d_roi_align_bwd", arr, _C.ptr(grad_feats[s]), _C.ptr(self.rois_flat[s]), self.B * self.m,
                    _C.ptr(self.roi_img), None, self.B * self.m, self.B, ctypes.byref(self.bwd_cfg), _C.ptr(self.bwd_ws),
                    self.bwd_ws.numel(), _C.stream())
        return self.grads


class InferHotPath(object):
    """CascadeRCNN.forward_test (SURVEY 3.2, lib/detectors/cascade_rcnn.py:157-200) minus the backbone, neck and head
    layers, batched: RPN proposals at the test configuration (K3 + K4) -> per stage FPN RoIAlign of the current boxes (K5)
    -> [the caller's stage head] -> between stages BBoxHead.refine_bboxes with the arg-max labels
    (b2d_refine_bboxes_argmax) -> after the last stage BBoxHead.predict_bboxes_single_image on that stage's input boxes
    (b2d_rcnn_detect: softmax, per-class decode + clamp, class-offset NMS, top max_per_img).  num_stages = 1 is
    faster_rcnn_r50_fpn, 3 the cascade.  Everything is allocated here; step() reads nothing back to the host, so a step
    (head modules included) can be captured in one CUDA graph after a first eager call."""

    def __init__(self, B, grids, device, strides=(4, 8, 16, 32, 64), feat_channels=256, num_classes=21, num_stages=1,
                 rpn_test=None, rcnn_test=None,
                 stage_stds=((0.1, 0.1, 0.2, 0.2), (0.05, 0.05, 0.1, 0.1), (0.033, 0.033, 0.067, 0.067)),
                 reg_class_agnostic=False, layout=1):
        rpn_test = rpn_test or dict(pre_nms=1000, post_nms=1000, max_num=1000, nms_iou=0.7, min_bbox_size=0)
        rcnn_test = rcnn_test or dict(min_score=0.05, nms_iou=0.5, max_per_img=100, nms_type='official')
        if not 1 <= num_stages <= len(stage_stds):
            raise ValueError("num_stages must be in 1..%d (one stds tuple per stage)" % len(stage_stds))
        if not 2 <= int(num_classes) <= 128:
            # b2d_rcnn_detect holds a row's classes in one warp; without this check the first step would only fail at
            # the detection call, after the proposals, RoIAlign and the caller's head (or in the middle of a graph capture)
            raise _C.B200DetError("InferHotPath: 2..128 classes (background included) supported, got %d" % int(num_classes))
        z4 = (0.0, 0.0, 0.0, 0.0)
        self.B, self.device, self.S = B, device, int(num_stages)
        self.NC, self.reg_c = int(num_classes), 1 if reg_class_agnostic else int(num_classes)
        self.pyr = AnchorPyramid(strides, grids)
        self.proposals = RpnProposals(self.pyr, B, rpn_test, z4, (1.0, 1.0, 1.0, 1.0), device)
        self.P = P = self.proposals.P
        shapes = [(feat_channels, g[0], g[1]) for g in grids[:4]]
        self.roi_align = [BatchedRoIAlign(B, P, shapes, list(strides[:4]), device, layout=layout) for _ in range(self.S)]
        self.stds = [_C.host_f4(sd, [1, 1, 1, 1]) for sd in stage_stds[:self.S]]
        self.zero4 = _C.host_f4(z4, [0, 0, 0, 0])
        self.boxes = [torch.zeros((B, 4, P), dtype=torch.float32, device=device) for _ in range(self.S - 1)]
        self.counts = [torch.zeros(B, dtype=torch.int32, device=device) for _ in range(self.S - 1)]
        get = (lambda k, d=None: rcnn_test.get(k, d)) if hasattr(rcnn_test, "get") else (lambda k, d=None: getattr(rcnn_test, k, d))
        mode = get('nms_type', 'official')
        self.min_score, self.nms_thr = float(np.float32(get('min_score'))), _C.floor_f32(float(get('nms_iou')))
        self.strict = int(mode == 'strict')
        self.cap = max(1, min(16384, P * ((self.NC - 1) if not self.strict else 1)))
        mpi = get('max_per_img')
        self.M = M = max(1, min(int(mpi) if mpi is not None else self.cap, self.cap))
        self.det_box = torch.zeros((B, 4, M), dtype=torch.float32, device=device)
        self.det_score = torch.zeros((B, M), dtype=torch.float32, device=device)
        self.det_label = torch.zeros((B, M), dtype=torch.int64, device=device)
        self.det_count = torch.zeros(B, dtype=torch.int32, device=device)
        self.overflow = torch.zeros(1, dtype=torch.int32, device=device)
        self.det_ws = torch.empty(_C.lib().b2d_rcnn_detect_workspace_bytes(self.cap, B), dtype=torch.uint8, device=device)

    def step(self, cls_outs, reg_outs, feats, img_hw, heads, records=None, mark=None):
        """cls_outs / reg_outs: the RPN head maps per level ([B,A,H,W], [B,4A,H,W]); feats: the first four FPN maps
        (channels_last for layout 1); img_hw fp32 [B,2]; heads[s](roi_feats [B*P,C,7,7]) -> (cls_out [B*P, num_classes]
        logits, reg_out [B*P, 4*num_classes] or [B*P, 4]); records: optional fp32 [B, max_per_img, 6] that receives the
        packed detections of dist.pack_detections (the payload of dist.gather_detections); mark(name): optional
        callable run after each phase (e.g. to record a CUDA event).  Returns the detections (boxes [B,4,M], scores
        [B,M], labels int64 [B,M], count int32 [B]) and per stage the input boxes, counts and RoI features."""
        if records is not None and (tuple(records.shape) != (self.B, self.M, 6) or records.dtype != torch.float32
                                    or not records.is_contiguous()):
            raise _C.B200DetError("InferHotPath.step: records must be contiguous fp32 [%d, %d, 6]" % (self.B, self.M))
        props, _, count = self.proposals(cls_outs, reg_outs, img_hw)
        if mark is not None:
            mark("proposals")
        boxes, stages = props, []
        for s in range(self.S):
            roi_feats = self.roi_align[s](feats, boxes, count)
            if mark is not None:
                mark("roi_align%d" % s)
            cls_out, reg_out = heads[s](roi_feats)
            cls_out, reg_out = _C.f32c(cls_out), _C.f32c(reg_out)
            if tuple(cls_out.shape) != (self.B * self.P, self.NC) or tuple(reg_out.shape) != (self.B * self.P, 4 * self.reg_c):
                raise _C.B200DetError("InferHotPath.step: stage %d head returned %s / %s, expected [%d, %d] / [%d, %d]"
                                      % (s, tuple(cls_out.shape), tuple(reg_out.shape), self.B * self.P, self.NC,
                                         self.B * self.P, 4 * self.reg_c))
            if mark is not None:
                mark("head%d" % s)
            stages.append(dict(boxes=boxes, count=count, roi_feats=roi_feats, cls_out=cls_out, reg_out=reg_out))
            if s + 1 < self.S:
                _C.call("b2d_refine_bboxes_argmax", _C.ptr(self.boxes[s]), _C.ptr(self.counts[s]), _C.ptr(boxes), self.P,
                        _C.ptr(count), self.P, _C.ptr(cls_out), self.NC, _C.ptr(reg_out), self.reg_c, self.zero4,
                        self.stds[s], _C.ptr(img_hw), self.B, _C.stream())
                boxes, count = self.boxes[s], self.counts[s]
                if mark is not None:
                    mark("refine%d" % s)
        last = stages[-1]
        args = [_C.ptr(self.det_box), _C.ptr(self.det_score), _C.ptr(self.det_label), _C.ptr(self.det_count)]
        if records is not None:
            args.append(_C.ptr(records))
        args += [_C.ptr(boxes), self.P, _C.ptr(count), self.P, _C.ptr(last["cls_out"]), _C.ptr(last["reg_out"]), self.NC,
                 self.reg_c, self.zero4, self.stds[-1], _C.ptr(img_hw), self.min_score, self.nms_thr, self.M, self.strict,
                 self.cap, self.B, _C.ptr(self.overflow), _C.ptr(self.det_ws), self.det_ws.numel(), _C.stream()]
        _C.call("b2d_rcnn_detect_records" if records is not None else "b2d_rcnn_detect", *args)
        if mark is not None:
            mark("detect")
        return dict(boxes=self.det_box, scores=self.det_score, labels=self.det_label, count=self.det_count,
                    records=records, stages=stages)

    def check(self):
        """Synchronise and raise if the last step had an image with more than 16384 (box, class) candidates (its
        candidates past the cap were dropped in enumeration order)."""
        torch.cuda.synchronize(self.device)
        if int(self.overflow[0]):
            raise _C.B200DetError("rcnn_detect: more than 16384 (box, class) candidates; raise min_score")


class DenseInferHotPath(object):
    """The test path of the one-stage detectors after the head convolutions, batched: RetinaNet
    (AnchorHead.predict_single_image, lib/heads/anchor_head.py:207-258; BASELINE config 4) and FCOS / ATSS
    (FCOSHead.predict_single_image, lib/heads/fcos_head.py:570-631; config 5).
      head='retina': per-level top pre_nms on the best class score, decode, clamp, size filter (RpnProposals with
                     score_mode 2 / 3 and do_nms off) -> b2d_dense_detect on the logit maps read in place;
      head='fcos':   b2d_fcos_decode -> b2d_dense_select (per-level filter + top pre_nms) -> b2d_dense_detect on the
                     sigmoid scores with the centerness as score factor.
    b2d_dense_detect is utils.multiclass_nms for all images at once: candidate test, ordered compaction, class-offset NMS,
    the first max_per_img survivors, and optionally the packed records of dist.pack_detections.
    num_classes counts the background as the reference heads do: a sigmoid head (RetinaNet with use_sigmoid, FCOS) has
    num_classes - 1 class channels and 1-based labels, a softmax head num_classes channels with channel 0 the background.
    Everything is allocated here; step() reads nothing back to the host, so a step can be captured in one CUDA graph after
    a first eager call.  More than 16384 (box, class) candidates in an image set a device flag that check() raises."""

    def __init__(self, B, grids, device, head="retina", num_classes=21, test_cfg=None, strides=(8, 16, 32, 64, 128),
                 use_sigmoid=True, anchor_scales=tuple(4 * 2 ** (i / 3) for i in range(3)), anchor_ratios=(0.5, 1.0, 2.0),
                 center_lt=False, target_means=(0.0, 0.0, 0.0, 0.0), target_stds=(1.0, 1.0, 1.0, 1.0), reg_mean=0.0,
                 reg_std=300.0, use_centerness=True, scale_factor=1.0):
        if head not in ("retina", "fcos"):
            raise _C.B200DetError("DenseInferHotPath: head must be 'retina' or 'fcos', got %r" % (head,))
        test_cfg = test_cfg or dict(pre_nms=1000, min_bbox_size=0, min_score=0.05, nms_iou=0.5, max_per_img=100,
                                    nms_type="strict")
        get = (lambda k, d=None: test_cfg.get(k, d)) if hasattr(test_cfg, "get") else (lambda k, d=None: getattr(test_cfg, k, d))
        mode = get("nms_type", "official")
        if mode not in ("official", "strict"):
            raise _C.B200DetError("DenseInferHotPath: nms_type must be 'official' or 'strict'")
        self.B, self.device, self.head = int(B), device, head
        self.grids = [tuple(int(v) for v in g) for g in grids]
        self.L = len(self.grids)
        sigmoid = head == "fcos" or bool(use_sigmoid)
        self.C = C = int(num_classes) - 1 if sigmoid else int(num_classes)
        if not 1 <= C <= 128:
            raise _C.B200DetError("DenseInferHotPath: 1..128 class channels supported, got %d" % C)
        self.pre = int(get("pre_nms", 0) or 0)
        min_bbox = float(get("min_bbox_size", 0) or 0)
        self.min_score = float(np.float32(get("min_score", -1)))
        self.nms_thr = _C.floor_f32(float(get("nms_iou")))
        self.strict = int(mode == "strict")
        chans = list(range(0, C)) if sigmoid else list(range(1, C))
        mask = [0, 0]
        for c in chans:
            mask[c >> 6] |= 1 << (c & 63)
        self.chan = (_C.c_ull * 2)(*mask)
        self.label_add = 1 if sigmoid else 0
        self.lv = _C.DenseLevels()
        if head == "retina":
            self.transform = 1 if sigmoid else 2
            self.pyr = AnchorPyramid(strides, self.grids, tuple(anchor_scales), tuple(anchor_ratios), center_lt)
            self.A = self.pyr.num_anchors
            sel_cfg = dict(pre_nms=self.pre, post_nms=0, max_num=0, nms_iou=0.5, min_bbox_size=min_bbox)
            self.select = RpnProposals(self.pyr, B, sel_cfg, target_means, target_stds, device,
                                       score_mode=2 if sigmoid else 3, cls_channels=C, do_nms=False, scale_factor=scale_factor)
            self.P = self.select.P
            self.lv.num_levels = self.L
            for l, n in enumerate(self.pyr.level_sizes):              # cls_l.view(B, C, -1): [B][C][A*H*W]
                self.lv.offset[l], self.lv.img_stride[l], self.lv.class_stride[l] = int(self.pyr.c.lv[l].offset), C * n, n
        else:
            from . import heads
            self.transform, self.centerness = 0, bool(use_centerness)
            self.pyr_c = heads._point_pyramid(self.grids, strides, 8)
            self.total = T = int(self.pyr_c.total)
            sizes = [h * w for h, w in self.grids]
            self.sizes = (_C.c_int * _C.MAX_LEVELS)(*sizes)
            self.P = sum(min(self.pre, n) if self.pre > 0 else n for n in sizes)
            self.reg_mean, self.reg_std = float(reg_mean), float(reg_std)
            self.min_size = float(np.float32(scale_factor * min_bbox))
            self.boxes = torch.zeros((B, 4, T), dtype=torch.float32, device=device)
            self.key = torch.zeros((B, T), dtype=torch.float32, device=device)
            self.score = torch.zeros((B, C, T), dtype=torch.float32, device=device)
            self.ctrs = torch.zeros((B, T), dtype=torch.float32, device=device) if self.centerness else None
            self.sel_idx = torch.zeros((B, self.P), dtype=torch.int32, device=device)
            self.sel_count = torch.zeros(B, dtype=torch.int32, device=device)
            self.sel_boxes = torch.zeros((B, 4, self.P), dtype=torch.float32, device=device)
            nb = _C.lib().b2d_dense_select_workspace_bytes(self.sizes, self.L, B, self.pre)
            if nb == 0:
                raise _C.B200DetError("DenseInferHotPath: unsupported selection (1..8 levels, a level top-k <= 16384)")
            self.sel_ws = torch.empty(nb, dtype=torch.uint8, device=device)
            self.lv.num_levels = 1                                    # score [B][C][total] as one level
            self.lv.offset[0], self.lv.img_stride[0], self.lv.class_stride[0] = 0, C * T, T
            self.lv.base[0] = self.score.data_ptr()
        self.cap = max(1, min(16384, self.P * (len(chans) if not self.strict else 1)))
        mpi = get("max_per_img")
        self.M = M = max(1, min(int(mpi) if mpi is not None else self.cap, self.cap))
        self.det_box = torch.zeros((B, 4, M), dtype=torch.float32, device=device)
        self.det_score = torch.zeros((B, M), dtype=torch.float32, device=device)
        self.det_label = torch.zeros((B, M), dtype=torch.int64, device=device)
        self.det_count = torch.zeros(B, dtype=torch.int32, device=device)
        self.overflow = torch.zeros(1, dtype=torch.int32, device=device)
        self.det_ws = torch.empty(_C.lib().b2d_rcnn_detect_workspace_bytes(self.cap, B), dtype=torch.uint8, device=device)

    def _check_maps(self, what, maps, per_cell):
        if maps is None or len(maps) != self.L:
            raise _C.B200DetError("DenseInferHotPath.step: %s needs %d levels" % (what, self.L))
        for (h, w), t in zip(self.grids, maps):
            if (tuple(t.shape) != (self.B, per_cell, h, w) or t.dtype != torch.float32 or not t.is_contiguous()
                    or not t.is_cuda):
                raise _C.B200DetError("DenseInferHotPath.step: %s level of shape %s (%s), expected contiguous fp32 CUDA "
                                      "[%d, %d, %d, %d]" % (what, tuple(t.shape), t.dtype, self.B, per_cell, h, w))

    def step(self, cls_outs, reg_outs, img_hw, ctr_outs=None, records=None, mark=None, detect_events=None):
        """cls_outs / reg_outs (/ ctr_outs for FCOS with centerness): the head maps per level, contiguous fp32 --
        RetinaNet [B, A*C, H, W] / [B, 4A, H, W], FCOS [B, C, H, W] / [B, 4, H, W] / [B, 1, H, W]; img_hw fp32 [B, 2];
        records: optional fp32 [B, max_per_img, 6] that receives the packed detections of dist.pack_detections;
        mark(name): optional callable run after each phase; detect_events: optional two torch.cuda.Event (already
        recorded once) that the detection call records after its candidate stage and after its NMS.  Returns the
        detections (boxes [B,4,M], scores [B,M], labels int64 [B,M], count int32 [B]) and the selected rows."""
        B = self.B
        if tuple(img_hw.shape) != (B, 2) or img_hw.dtype != torch.float32 or not img_hw.is_contiguous():
            raise _C.B200DetError("DenseInferHotPath.step: img_hw must be contiguous fp32 [%d, 2]" % B)
        if records is not None and (tuple(records.shape) != (B, self.M, 6) or records.dtype != torch.float32
                                    or not records.is_contiguous()):
            raise _C.B200DetError("DenseInferHotPath.step: records must be contiguous fp32 [%d, %d, 6]" % (B, self.M))
        if self.head == "retina":
            self._check_maps("cls_outs", cls_outs, self.A * self.C)
            self._check_maps("reg_outs", reg_outs, 4 * self.A)
            boxes, count, rows = self.select(cls_outs, reg_outs, img_hw)[0], self.select.count, self.select.prov
            for l, t in enumerate(cls_outs):
                self.lv.base[l] = t.data_ptr()
            factor = None
            if mark is not None:
                mark("selection")
        else:
            self._check_maps("cls_outs", cls_outs, self.C)
            self._check_maps("reg_outs", reg_outs, 4)
            if self.centerness:
                self._check_maps("ctr_outs", ctr_outs, 1)
            _C.call("b2d_fcos_decode", _C.ptr(self.boxes), _C.ptr(self.key), _C.ptr(self.score), _C.ptr(self.ctrs),
                    _ptrs(cls_outs), _ptrs(reg_outs), _ptrs(ctr_outs) if self.centerness else None, ctypes.byref(self.pyr_c),
                    self.C, self.reg_mean, self.reg_std, self.min_size, _C.ptr(img_hw), B, _C.stream())
            if mark is not None:
                mark("decode")
            _C.call("b2d_dense_select", _C.ptr(self.sel_idx), _C.ptr(self.sel_count), _C.ptr(self.sel_boxes), _C.ptr(self.key),
                    _C.ptr(self.boxes), self.sizes, self.L, B, self.pre, _C.ptr(self.sel_ws), self.sel_ws.numel(), _C.stream())
            boxes, count, rows, factor = self.sel_boxes, self.sel_count, self.sel_idx, self.ctrs
            if mark is not None:
                mark("selection")
        ev = None
        if detect_events is not None:
            ev = (_C.c_void_p * 2)(*[e.cuda_event for e in detect_events])
        args = [_C.ptr(self.det_box), _C.ptr(self.det_score), _C.ptr(self.det_label), _C.ptr(self.det_count)]
        if records is not None:
            args.append(_C.ptr(records))
        args += [_C.ptr(boxes), self.P, _C.ptr(count), _C.ptr(rows), ctypes.byref(self.lv), self.C, self.transform,
                 _C.ptr(factor), self.total if factor is not None else 0, self.chan, self.min_score, self.label_add,
                 self.nms_thr, self.M, self.strict, self.cap, B, _C.ptr(self.overflow), _C.ptr(self.det_ws),
                 self.det_ws.numel(), ev, _C.stream()]
        _C.call("b2d_dense_detect_records" if records is not None else "b2d_dense_detect", *args)
        if mark is not None:
            mark("detect")
        return dict(boxes=self.det_box, scores=self.det_score, labels=self.det_label, count=self.det_count,
                    records=records, sel_boxes=boxes, sel_count=count, sel_rows=rows)

    def check(self):
        """Synchronise and raise if the last step had an image with more than 16384 (box, class) candidates (its
        candidates past the cap were dropped in enumeration order)."""
        torch.cuda.synchronize(self.device)
        if int(self.overflow[0]):
            raise _C.B200DetError("dense_detect: more than 16384 (box, class) candidates in an image; raise min_score")
