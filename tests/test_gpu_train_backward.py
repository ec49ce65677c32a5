"""Backward of the batched train step (fused.TrainHotPath.backward, fused.TrainStepFn): the head-map gradients of the RPN
target gather (b2d_scatter_head_grads) against torch autograd of the reference's index, the FPN feature gradients of the
sampled RoIs (b2d_roi_align_bwd_batched, K6) against the oracle, the unbatched K6 entry and region.roi_align_levels, and
the step + backward as one CUDA graph and as an autograd node.  GPU only."""
import ctypes

import numpy as np
import pytest
import torch

import oracle

pytestmark = pytest.mark.gpu

if torch.cuda.is_available():
    from b200det import _C, fused, region as bregion, workload
    DEV = torch.device("cuda:0")

SCALES = [1 / 4, 1 / 8, 1 / 16, 1 / 32]


def T(a):
    return torch.from_numpy(np.ascontiguousarray(a)).to(DEV)


def N(t):
    return t.detach().cpu().numpy()


def same_bits(a, b):
    return a.shape == b.shape and torch.equal(a.contiguous().view(torch.int32), b.contiguous().view(torch.int32))


def config2_path(B, C, layout=1, overlap=False, groups=1, seed=0, K=8):
    w = workload.config2(B=B, K=K, channels=C)
    hp = fused.TrainHotPath(B, w["grids"], DEV, gt_ld=K, feat_channels=C, layout=layout, overlap=overlap, groups=groups,
                            seed=seed)
    mf = torch.channels_last if layout == 1 else torch.contiguous_format
    inputs = dict(cls=[T(c) for c in w["cls"]], reg=[T(r) for r in w["reg"]],
                  feats=[T(f).contiguous(memory_format=mf) for f in w["feats"]],
                  gt=T(w["gt"]), gt_count=torch.full((B,), K, dtype=torch.int32, device=DEV), gt_label=T(w["gt_label"]),
                  img_hw=torch.tensor([[800.0, 1333.0]] * B, device=DEV))
    return hp, inputs, w


def small_path(layout=1, C=128):
    """A 96 x 128 pyramid whose images hold fewer labelled anchors than the RPN sampler asks for, and fewer proposals
    + GT than the RoI sampler asks for: n_chosen < max_num on both sides, unequal between the images."""
    B, K = 2, 3
    strides = (4, 8, 16, 32, 64)
    grids = workload.fpn_grids((96, 128), strides)
    rng = np.random.default_rng(41)
    hp = fused.TrainHotPath(B, grids, DEV, strides=strides, gt_ld=K, feat_channels=C, layout=layout, seed=5,
                            rpn_proposal=dict(pre_nms=150, post_nms=150, max_num=150, nms_iou=0.7, min_bbox_size=0),
                            rpn_sampler=dict(max_num=2048, pos_num=1024), rcnn_sampler=dict(max_num=512, pos_num=128))
    gt = np.zeros((B, 4, K), np.float32)
    gl = np.zeros((B, K), np.int64)
    for b in range(B):
        gt[b], gl[b] = workload.synth_gt(rng, K, 96 - 32 * b, 128)
    mf = torch.channels_last if layout == 1 else torch.contiguous_format
    inputs = dict(cls=[T(rng.standard_normal((B, 3) + g, dtype=np.float32)) for g in grids],
                  reg=[T(0.5 * rng.standard_normal((B, 12) + g, dtype=np.float32)) for g in grids],
                  feats=[T(rng.standard_normal((B, C) + g, dtype=np.float32)).contiguous(memory_format=mf) for g in grids[:4]],
                  gt=T(gt), gt_count=torch.full((B,), K, dtype=torch.int32, device=DEV), gt_label=T(gl),
                  img_hw=torch.tensor([[96.0, 128.0], [64.0, 128.0]], device=DEV))
    return hp, inputs, grids


def run_step(hp, x):
    return hp.step(x["cls"], x["reg"], x["feats"], x["gt"], x["gt_count"], x["gt_label"], x["img_hw"])


def upstream(hp, seed, poison=True):
    """Seeded upstream gradients of the step's three differentiable outputs; entries past the counts are NaN."""
    g = torch.Generator(device=DEV).manual_seed(seed)
    g_cls = torch.randn(hp.tar_cls.shape, device=DEV, generator=g)
    g_reg = torch.randn(hp.tar_reg.shape, device=DEV, generator=g)
    g_feat = torch.randn(hp.roi_align.out.shape, device=DEV, generator=g)
    if poison:
        poison_past_counts(hp, g_cls, g_reg, g_feat)
    return g_cls, g_reg, g_feat


def poison_past_counts(hp, g_cls, g_reg, g_feat):
    m, ld = hp.tar_cls.shape[2], hp.roi_align.ld
    n_rpn, n_roi = N(hp.rpn_targets.n_chosen), N(hp.roi_targets.n_chosen)
    for b in range(hp.B):
        g_cls[b, :, n_rpn[b]:m] = float("nan")
        g_reg[b, :, n_rpn[b]:m] = float("nan")
        g_feat[b * ld + n_roi[b]:(b + 1) * ld] = float("nan")


def head_grads_reference(cls_maps, reg_maps, chosen, n_chosen, g_cls, g_reg, C=1):
    """torch autograd of the reference's gather (lib/anchor.py:49-56 on the views of refpath.rpn_targets_single_image)."""
    cl = [c.detach().clone().requires_grad_(True) for c in cls_maps]
    rl = [r.detach().clone().requires_grad_(True) for r in reg_maps]
    loss = 0
    for b in range(cl[0].shape[0]):
        n = int(n_chosen[b])
        idx = chosen[b, :n].long()
        cls_out = torch.cat([x[b].view(C, -1) for x in cl], dim=1)
        reg_out = torch.cat([x[b].view(4, -1) for x in rl], dim=1)
        loss = loss + (cls_out[:, idx] * g_cls[b, :, :n]).sum() + (reg_out[:, idx] * g_reg[b, :, :n]).sum()
    loss.backward()
    return [x.grad for x in cl], [x.grad for x in rl]


def compacted(hp):
    bt = hp.roi_targets
    n = N(bt.n_chosen)
    rois = torch.cat([bt.tar_box[b, :, :n[b]] for b in range(hp.B)], 1).contiguous()
    img = torch.cat([torch.full((int(n[b]),), b, dtype=torch.int32, device=DEV) for b in range(hp.B)])
    rows = torch.cat([torch.arange(b * hp.roi_align.ld, b * hp.roi_align.ld + int(n[b]), device=DEV) for b in range(hp.B)])
    return rois, img, rows


def feat_grads_reference(hp, feats, g_feat):
    """region.roi_align_levels(...).backward on the compacted RoI list (the unbatched K6 entry)."""
    rois, img, rows = compacted(hp)
    fs = [f.detach().clone().requires_grad_(True) for f in feats]
    bregion.roi_align_levels(fs, rois, img, SCALES).backward(g_feat[rows])
    return [f.grad for f in fs]


# ------------------------------------------------------------------ head-map gradients (b2d_scatter_head_grads)
@pytest.mark.parametrize("case", ["config2", "small"])
def test_head_map_gradients_equal_autograd_of_the_gather(case):
    hp, x, _ = config2_path(2, 16) if case == "config2" else small_path(C=16)
    out = run_step(hp, x)
    rt = out["rpn"]
    n = N(rt.n_chosen)
    if case == "small":
        assert (n < rt.max_num).all() and n[0] != n[1], n
    g_cls, g_reg, g_feat = upstream(hp, 1)
    dcls, dreg, _ = hp.backward(g_cls, g_reg, g_feat)
    ref_cls, ref_reg = head_grads_reference(x["cls"], x["reg"], rt.chosen, n, g_cls, g_reg)
    for a, b in zip(dcls + dreg, ref_cls + ref_reg):
        assert same_bits(a, b)
    # the forward gathered the values at the anchors the backward scatters to
    for b in range(hp.B):
        k = int(n[b])
        flat = torch.cat([c[b].reshape(-1) for c in x["cls"]])
        torch.testing.assert_close(out["rpn_tar_cls"][b, 0, :k], flat[rt.chosen[b, :k].long()], rtol=0, atol=0)


def test_scatter_head_grads_two_class_channels_direct():
    """b2d_scatter_head_grads with cls_channels = 2 (a softmax RPN), ragged sample lists incl. an empty and a full one,
    NaN past the counts: bit-identical to autograd of the gather, and the adjoint of b2d_gather_head_outputs."""
    B, C, m = 4, 2, 300
    pyr = fused.AnchorPyramid((4, 8, 16, 32, 64), workload.fpn_grids((100, 150)))
    A, total = pyr.num_anchors, pyr.total
    rng = np.random.default_rng(9)
    counts = np.array([m, 0, 57, 211], np.int32)
    chosen = np.full((B, m), -1, np.int32)
    for b in range(B):
        chosen[b, :counts[b]] = np.sort(rng.choice(total, counts[b], replace=False))
    chosen[2, counts[2]:] = rng.integers(0, total, m - counts[2])          # stale rows: never read
    cls = [T(rng.standard_normal((B, A * C) + g, dtype=np.float32)) for g in pyr.grids]
    reg = [T(rng.standard_normal((B, 4 * A) + g, dtype=np.float32)) for g in pyr.grids]
    g_cls = torch.randn((B, C, m), device=DEV)
    g_reg = torch.randn((B, 4, m), device=DEV)
    for b in range(B):
        g_cls[b, :, counts[b]:] = float("nan")
        g_reg[b, :, counts[b]:] = float("nan")
    dcls = [torch.full_like(c, float("nan")) for c in cls]
    dreg = [torch.full_like(r, float("nan")) for r in reg]
    ch, nc = T(chosen), T(counts)
    _C.call("b2d_scatter_head_grads", fused._ptrs(dcls), fused._ptrs(dreg), _C.ptr(g_cls), _C.ptr(g_reg),
            ctypes.byref(pyr.c), C, _C.ptr(ch), _C.ptr(nc), m, B, _C.stream())
    ref_cls, ref_reg = head_grads_reference(cls, reg, ch, counts, g_cls, g_reg, C=C)
    for a, b in zip(dcls + dreg, ref_cls + ref_reg):
        assert same_bits(a, b)
    # adjoint: <gather(x), g> == <x, scatter(g)> on the live entries
    tc, tr = torch.zeros((B, C, m), device=DEV), torch.zeros((B, 4, m), device=DEV)
    _C.call("b2d_gather_head_outputs", _C.ptr(tc), _C.ptr(tr), fused._ptrs(cls), fused._ptrs(reg), ctypes.byref(pyr.c), C,
            _C.ptr(ch), _C.ptr(nc), m, B, _C.stream())
    lhs = sum(float((tc[b, :, :counts[b]].double() * g_cls[b, :, :counts[b]].double()).sum() +
                    (tr[b, :, :counts[b]].double() * g_reg[b, :, :counts[b]].double()).sum()) for b in range(B))
    rhs = sum(float((a.double() * g.double()).sum()) for a, g in zip(cls + reg, dcls + dreg))
    assert abs(lhs - rhs) <= 1e-9 * max(1.0, abs(lhs))


# ------------------------------------------------------------------ feature gradients (b2d_roi_align_bwd_batched)
def test_feature_gradients_vs_oracle_config2_geometry():
    B, C = 2, 128
    hp, x, w = config2_path(B, C)
    run_step(hp, x)
    g_cls, g_reg, g_feat = upstream(hp, 2)
    _, _, dfeat = hp.backward(g_cls, g_reg, g_feat)
    bt, ld = hp.roi_targets, hp.roi_align.ld
    for b in range(B):
        n = int(bt.n_chosen[b])
        rois = N(bt.tar_box[b, :, :n])
        go = N(g_feat[b * ld:b * ld + n])
        lv = oracle.level_map(rois)
        for l, s in enumerate((4, 8, 16, 32)):
            m = lv == l
            ref = oracle.roi_align_bwd(go[m], (C,) + tuple(w["grids"][l]), np.ascontiguousarray(rois[:, m]), 1.0 / s)
            np.testing.assert_allclose(N(dfeat[l][b]), ref, rtol=1e-5, atol=5e-6)


def test_feature_gradients_full_size_bit_identical_to_unbatched():
    B, C = 2, 256
    hp, x, _ = config2_path(B, C)
    run_step(hp, x)
    g_cls, g_reg, g_feat = upstream(hp, 3)
    _, _, dfeat = hp.backward(g_cls, g_reg, g_feat)
    for a, b in zip(dfeat, feat_grads_reference(hp, x["feats"], g_feat)):
        assert same_bits(a, b)


@pytest.mark.parametrize("layout", [1, 0])
def test_rows_past_the_counts_change_nothing(layout):
    hp, x, _ = small_path(layout=layout)
    run_step(hp, x)
    n = N(hp.roi_targets.n_chosen)
    assert (n < hp.roi_align.ld).all(), n
    clean = upstream(hp, 4, poison=False)
    got = [[t.clone() for t in ts] for ts in hp.backward(*clean)]
    poisoned = [t.clone() for t in clean]
    poison_past_counts(hp, *poisoned)
    again = hp.backward(*poisoned)
    for ga, gb in zip(got, again):
        for a, b in zip(ga, gb):
            assert same_bits(a, b)
    assert not any(torch.isnan(t).any() for ts in again for t in ts)
    if layout == 1:
        assert all(t.is_contiguous(memory_format=torch.channels_last) for t in again[2])
    else:
        assert all(t.is_contiguous() for t in again[2])
    # layout 1 runs the same K6 form as the unbatched entry (bit-identical); NCHW gradients take the generic
    # torchvision-ordered kernel, the reference path transposes to NHWC first (rounding only)
    for a, b in zip(again[2], feat_grads_reference(hp, x["feats"], clean[2])):
        if layout == 1:
            assert same_bits(a, b)
        else:
            torch.testing.assert_close(a, b, rtol=1e-5, atol=5e-6)


def _ragged_case(rng, B, ld, counts, grids, C, layout):
    Wimg, Himg = 4.0 * grids[0][1], 4.0 * grids[0][0]
    rois = np.full((B, 4, ld), np.nan, np.float32)                     # stale slots: NaN boxes, never read
    for b in range(B):
        k = counts[b]
        w = np.exp(rng.uniform(np.log(2.0), np.log(0.9 * Wimg), k)); h = np.exp(rng.uniform(np.log(2.0), np.log(0.9 * Himg), k))
        cx, cy = rng.uniform(-10, Wimg + 10, k), rng.uniform(-10, Himg + 10, k)
        rois[b, :, :k] = np.stack([cx - w / 2, cy - h / 2, cx + w / 2, cy + h / 2])
    cfg = _C.RoiCfg()
    cfg.num_levels, cfg.C, cfg.PH, cfg.PW, cfg.sampling_ratio, cfg.aligned = len(grids), C, 7, 7, 2, 0
    cfg.layout, cfg.finest_scale = layout, 56.0
    for l, g in enumerate(grids):
        cfg.H[l], cfg.W[l], cfg.spatial_scale[l] = g[0], g[1], 1.0 / (4 * 2 ** l)
    go = rng.standard_normal((B * ld, C, 7, 7)).astype(np.float32)
    for b in range(B):
        go[b * ld + counts[b]:(b + 1) * ld] = np.nan
    return T(rois), cfg, T(go)


def _k6_pair(rois, counts, go, cfg, B, ld, grids, C):
    mf = torch.channels_last if cfg.layout == 1 else torch.contiguous_format
    mk = lambda: [torch.full((B, C) + tuple(g), float("nan"), device=DEV).contiguous(memory_format=mf) for g in grids]
    gb, gu = mk(), mk()
    ws = torch.empty(_C.lib().b2d_roi_align_bwd_batched_workspace_bytes(ld, B, ctypes.byref(cfg)), dtype=torch.uint8, device=DEV)
    _C.call("b2d_roi_align_bwd_batched", fused._ptrs(gb), _C.ptr(go), _C.ptr(rois), ld, _C.ptr(T(counts)), B,
            ctypes.byref(cfg), _C.ptr(ws), ws.numel(), _C.stream())
    flat = torch.cat([rois[b, :, :counts[b]] for b in range(B)], 1).contiguous()
    img = torch.cat([torch.full((int(counts[b]),), b, dtype=torch.int32, device=DEV) for b in range(B)])
    rows = torch.cat([torch.arange(b * ld, b * ld + int(counts[b]), device=DEV) for b in range(B)])
    gout = go[rows].contiguous()
    R = flat.shape[1]
    ws2 = torch.empty(_C.lib().b2d_roi_align_bwd_workspace_bytes(R, B, ctypes.byref(cfg)), dtype=torch.uint8, device=DEV)
    _C.call("b2d_roi_align_bwd", fused._ptrs(gu), _C.ptr(gout), _C.ptr(flat), R, _C.ptr(img), None, R, B, ctypes.byref(cfg),
            _C.ptr(ws2), ws2.numel(), _C.stream())
    return gb, gu


@pytest.mark.parametrize("layout", [1, 0])
@pytest.mark.parametrize("form", ["2", "1", "0"])
def test_batched_k6_equals_unbatched_on_the_compacted_list(form, layout, setknob):
    """b2d_roi_align_bwd_batched against b2d_roi_align_bwd on the compacted list under every B2D_ROI_BWD_TILE form:
    ragged counts incl. an empty image, NaN boxes and gradient rows in the unused slots."""
    setknob(B2D_ROI_BWD_TILE=form)
    rng = np.random.default_rng(17)
    B, ld, C = 4, 96, 128
    grids = [(48, 80), (24, 40), (12, 20), (6, 10)]
    counts = np.array([37, 0, 96, 11], np.int32)
    rois, cfg, go = _ragged_case(rng, B, ld, counts, grids, C, layout)
    gb, gu = _k6_pair(rois, counts, go, cfg, B, ld, grids, C)
    for a, b in zip(gb, gu):
        assert same_bits(a, b)
        assert not torch.isnan(a).any()


def test_batched_k6_takes_the_patch_fallback_of_the_compacted_list(setknob):
    """The patch form's scratch budget follows the RoIs present, not the slots: three ~7 600-cell patches in 2 x 64 slots
    overflow the budget of 3 RoIs (16 K cells) but not that of 128 slots, and the batched call must fall back to the tile
    kernel exactly as the compacted call does (bit-identical to it)."""
    setknob(B2D_ROI_BWD_TILE=2)
    B, ld, C = 2, 64, 128
    grids = [(80, 100)]
    counts = np.array([3, 0], np.int32)
    rois = np.full((B, 4, ld), np.nan, np.float32)
    rois[0, :, :3] = np.array([[0, 0, 388, 312], [0, 0, 390, 310], [4, 2, 392, 316]], np.float32).T
    cfg = _C.RoiCfg()
    cfg.num_levels, cfg.C, cfg.PH, cfg.PW, cfg.sampling_ratio, cfg.aligned, cfg.layout, cfg.finest_scale = 1, C, 7, 7, 2, 0, 1, 56.0
    cfg.H[0], cfg.W[0], cfg.spatial_scale[0] = 80, 100, 0.25
    go = np.random.default_rng(3).standard_normal((B * ld, C, 7, 7)).astype(np.float32)
    gb, gu = _k6_pair(T(rois), counts, T(go), cfg, B, ld, grids, C)
    assert same_bits(gb[0], gu[0])
    setknob(B2D_ROI_BWD_TILE=1)
    _, gt_ = _k6_pair(T(rois), counts, T(go), cfg, B, ld, grids, C)
    assert same_bits(gu[0], gt_[0]), "the compacted call itself takes the tile fallback here"


# ------------------------------------------------------------------ graph capture and autograd
def test_step_and_backward_in_one_cuda_graph():
    B, C = 4, 128
    hp, x, _ = config2_path(B, C, overlap=True, groups=2, seed=3)
    run_step(hp, x)
    g_cls, g_reg, g_feat = upstream(hp, 5, poison=False)
    hp.backward(g_cls, g_reg, g_feat)                                   # first call: buffers
    torch.cuda.synchronize()
    hp.reset_step()
    out = run_step(hp, x)
    eager = [t.clone() for ts in hp.backward(g_cls, g_reg, g_feat) for t in ts]
    eager_chosen = (out["rpn"].chosen.clone(), out["rcnn"].tar_box.clone(), out["roi_feats"].clone())
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(graph, stream=side):
            run_step(hp, x)
            grads = hp.backward(g_cls, g_reg, g_feat)
    torch.cuda.current_stream().wait_stream(side)
    hp.reset_step()
    graph.replay()
    torch.cuda.synchronize()
    flat = [t for ts in grads for t in ts]
    assert all(same_bits(a, b) for a, b in zip(flat, eager))
    assert same_bits(hp.rpn_targets.chosen, eager_chosen[0]) and same_bits(hp.roi_targets.tar_box, eager_chosen[1])
    assert same_bits(hp.roi_align.out, eager_chosen[2])
    graph.replay()
    torch.cuda.synchronize()
    rt = hp.rpn_targets
    assert not torch.equal(rt.chosen, eager_chosen[0]), "a replay draws fresh samples"
    ref_cls, ref_reg = head_grads_reference(x["cls"], x["reg"], rt.chosen, N(rt.n_chosen), g_cls, g_reg)
    for a, b in zip(list(grads[0]) + list(grads[1]), ref_cls + ref_reg):
        assert same_bits(a, b)
    for a, b in zip(grads[2], feat_grads_reference(hp, x["feats"], g_feat)):
        assert same_bits(a, b)


@pytest.mark.parametrize("overlap", [False, True])
def test_autograd_entry_matches_explicit_backward(overlap):
    B, C = 2, 128
    hp, x, _ = config2_path(B, C, overlap=overlap)
    cls = [c.clone().requires_grad_(True) for c in x["cls"]]
    reg = [r.clone().requires_grad_(True) for r in x["reg"]]
    feats = [f.clone().requires_grad_(l != 3) for l, f in enumerate(x["feats"])]
    out = hp.step_autograd(cls, reg, feats, x["gt"], x["gt_count"], x["gt_label"], x["img_hw"])
    g_cls, g_reg, g_feat = upstream(hp, 6, poison=False)
    loss = (out["rpn_tar_cls"] * g_cls).sum() + (out["rpn_tar_reg"] * g_reg).sum() + (out["roi_feats"] * g_feat).sum()
    loss.backward()
    dcls, dreg, dfeat = hp.backward(g_cls, g_reg, g_feat)
    for leaf, g in zip(cls + reg + feats[:3], list(dcls) + list(dreg) + list(dfeat[:3])):
        assert same_bits(leaf.grad, g)
    assert feats[3].grad is None


def test_backward_refuses_bf16_features():
    hp, x, _ = small_path(layout=2, C=128)
    g = (torch.zeros(hp.tar_cls.shape, device=DEV), torch.zeros(hp.tar_reg.shape, device=DEV),
         torch.zeros(hp.roi_align.out.shape, device=DEV))
    with pytest.raises(_C.B200DetError, match="bf16"):
        hp.backward(*g)
    assert not hasattr(hp, "_bwd")
