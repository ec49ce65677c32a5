"""The cascade training step (fused.CascadeTrainHotPath): RoIAlign backward over several RoI sets in one call
(b2d_roi_align_bwd_multi) against the unbatched K6 entry, the batched one and the oracle; the forward against TrainHotPath
(stage 0) and the oracle (later stages); the backward, graph capture and the autograd entry.  GPU only."""
import ctypes

import numpy as np
import pytest
import torch

import oracle

pytestmark = pytest.mark.gpu

if torch.cuda.is_available():
    from b200det import _C, fused, workload
    DEV = torch.device("cuda:0")

THRESHOLDS = (0.5, 0.6, 0.7)
STDS = ((0.1, 0.1, 0.2, 0.2), (0.05, 0.05, 0.1, 0.1), (0.033, 0.033, 0.067, 0.067))


def T(a):
    return torch.from_numpy(np.ascontiguousarray(a)).to(DEV)


def N(t):
    return t.detach().cpu().numpy()


def same_bits(a, b):
    return a.shape == b.shape and torch.equal(a.contiguous().view(torch.int32), b.contiguous().view(torch.int32))


# ------------------------------------------------------------------ b2d_roi_align_bwd_multi
def roi_cfg(grids, C, layout):
    cfg = _C.RoiCfg()
    cfg.num_levels, cfg.C, cfg.PH, cfg.PW, cfg.sampling_ratio, cfg.aligned = len(grids), C, 7, 7, 2, 0
    cfg.layout, cfg.finest_scale = layout, 56.0
    for l, g in enumerate(grids):
        cfg.H[l], cfg.W[l], cfg.spatial_scale[l] = g[0], g[1], 1.0 / (4 * 2 ** l)
    return cfg


def ragged_set(rng, B, ld, counts, grids, C):
    """One RoI set: rois [B,4,ld] and grad_out [B*ld,C,7,7], NaN in every slot at or past counts[b] (never read)."""
    Wimg, Himg = 4.0 * grids[0][1], 4.0 * grids[0][0]
    rois = np.full((B, 4, ld), np.nan, np.float32)
    for b in range(B):
        k = counts[b]
        w = np.exp(rng.uniform(np.log(2.0), np.log(0.9 * Wimg), k)); h = np.exp(rng.uniform(np.log(2.0), np.log(0.9 * Himg), k))
        cx, cy = rng.uniform(-10, Wimg + 10, k), rng.uniform(-10, Himg + 10, k)
        rois[b, :, :k] = np.stack([cx - w / 2, cy - h / 2, cx + w / 2, cy + h / 2])
    go = rng.standard_normal((B * ld, C, 7, 7)).astype(np.float32)
    for b in range(B):
        go[b * ld + counts[b]:(b + 1) * ld] = np.nan
    return T(rois), T(np.asarray(counts, np.int32)), T(go)


def grad_maps(B, C, grids, layout):
    mf = torch.channels_last if layout == 1 else torch.contiguous_format
    return [torch.full((B, C) + tuple(g), float("nan"), device=DEV).contiguous(memory_format=mf) for g in grids]


def k6_multi(sets, cfg, B, grids, C):
    """sets: [(rois [B,4,ld], counts [B], grad_out [B*ld,...])] -> summed gradient maps (b2d_roi_align_bwd_multi)."""
    S = len(sets)
    lds = (_C.c_ll * S)(*[r.shape[2] for r, _, _ in sets])
    ws = torch.empty(_C.lib().b2d_roi_align_bwd_multi_workspace_bytes(S, lds, B, ctypes.byref(cfg)), dtype=torch.uint8,
                     device=DEV)
    out = grad_maps(B, C, grids, cfg.layout)
    _C.call("b2d_roi_align_bwd_multi", fused._ptrs(out), S, (_C.c_void_p * S)(*[g.data_ptr() for _, _, g in sets]),
            (_C.c_void_p * S)(*[r.data_ptr() for r, _, _ in sets]), lds,
            (_C.c_void_p * S)(*[c.data_ptr() for _, c, _ in sets]), B, ctypes.byref(cfg), _C.ptr(ws), ws.numel(), _C.stream())
    return out


def k6_batched(rois, counts, go, cfg, B, grids, C):
    ld = rois.shape[2]
    ws = torch.empty(_C.lib().b2d_roi_align_bwd_batched_workspace_bytes(ld, B, ctypes.byref(cfg)), dtype=torch.uint8, device=DEV)
    out = grad_maps(B, C, grids, cfg.layout)
    _C.call("b2d_roi_align_bwd_batched", fused._ptrs(out), _C.ptr(go), _C.ptr(rois), ld, _C.ptr(counts), B, ctypes.byref(cfg),
            _C.ptr(ws), ws.numel(), _C.stream())
    return out


def k6_compacted(sets, cfg, B, grids, C):
    """b2d_roi_align_bwd on the compacted RoI lists of the sets, concatenated set-major."""
    flat, img, rows = [], [], []
    for rois, counts, go in sets:
        ld, n = rois.shape[2], N(counts)
        for b in range(B):
            flat.append(rois[b, :, :n[b]])
            img.append(torch.full((int(n[b]),), b, dtype=torch.int32, device=DEV))
            rows.append(go[b * ld:b * ld + int(n[b])])
    flat, img, gout = torch.cat(flat, 1).contiguous(), torch.cat(img), torch.cat(rows).contiguous()
    R = flat.shape[1]
    ws = torch.empty(_C.lib().b2d_roi_align_bwd_workspace_bytes(R, B, ctypes.byref(cfg)), dtype=torch.uint8, device=DEV)
    out = grad_maps(B, C, grids, cfg.layout)
    _C.call("b2d_roi_align_bwd", fused._ptrs(out), _C.ptr(gout), _C.ptr(flat), R, _C.ptr(img), None, R, B, ctypes.byref(cfg),
            _C.ptr(ws), ws.numel(), _C.stream())
    return out


GRIDS = [(48, 80), (24, 40), (12, 20), (6, 10)]


def three_sets(rng, B, C):
    """S = 3 with different ld: an image without RoIs in the first set, the whole second set empty, ragged counts."""
    return [ragged_set(rng, B, 96, [37, 0, 96, 11], GRIDS, C),
            ragged_set(rng, B, 40, [0, 0, 0, 0], GRIDS, C),
            ragged_set(rng, B, 64, [64, 5, 0, 30], GRIDS, C)]


@pytest.mark.parametrize("layout", [1, 0])
@pytest.mark.parametrize("form", ["2", "1", "0"])
def test_multi_k6_equals_unbatched_on_the_set_major_concatenation(form, layout, setknob):
    setknob(B2D_ROI_BWD_TILE=form)
    B, C = 4, 128
    sets = three_sets(np.random.default_rng(23), B, C)
    cfg = roi_cfg(GRIDS, C, layout)
    got, want = k6_multi(sets, cfg, B, GRIDS, C), k6_compacted(sets, cfg, B, GRIDS, C)
    for a, b in zip(got, want):
        assert same_bits(a, b)
        assert not torch.isnan(a).any()


def test_multi_k6_takes_the_patch_fallback_of_the_compacted_list(setknob):
    """Three overlapping ~7 600-cell patches, two in one set and one in another, overflow the scratch budget of 3 RoIs
    (16 K cells) but not that of the 160 slots: the call must fall back to the tile kernel as the compacted call does."""
    setknob(B2D_ROI_BWD_TILE=2)
    B, C = 2, 128
    grids = [(80, 100)]
    boxes = np.array([[0, 0, 388, 312], [0, 0, 390, 310], [4, 2, 392, 316]], np.float32).T
    rng = np.random.default_rng(3)
    sets = []
    for ld, cols in ((64, [0, 1]), (96, [2])):
        rois = np.full((B, 4, ld), np.nan, np.float32)
        rois[0, :, :len(cols)] = boxes[:, cols]
        counts = [len(cols), 0]
        go = rng.standard_normal((B * ld, C, 7, 7)).astype(np.float32)
        sets.append((T(rois), T(np.asarray(counts, np.int32)), T(go)))
    cfg = roi_cfg(grids, C, 1)
    got, want = k6_multi(sets, cfg, B, grids, C), k6_compacted(sets, cfg, B, grids, C)
    assert same_bits(got[0], want[0])
    setknob(B2D_ROI_BWD_TILE=1)
    tile = k6_compacted(sets, cfg, B, grids, C)
    assert same_bits(want[0], tile[0]), "the compacted call itself takes the tile fallback here"


def test_multi_k6_is_the_sum_of_the_sets():
    B, C = 4, 128
    sets = three_sets(np.random.default_rng(29), B, C)
    cfg = roi_cfg(GRIDS, C, 1)
    got = k6_multi(sets, cfg, B, GRIDS, C)
    parts = [k6_batched(r, c, g, cfg, B, GRIDS, C) for r, c, g in sets]
    for l in range(len(GRIDS)):
        torch.testing.assert_close(got[l], sum(p[l] for p in parts), rtol=1e-5, atol=5e-6)


def test_multi_k6_one_image_vs_oracle():
    B, C = 1, 64
    rng = np.random.default_rng(31)
    sets = [ragged_set(rng, B, 50, [50], GRIDS, C), ragged_set(rng, B, 30, [17], GRIDS, C),
            ragged_set(rng, B, 20, [20], GRIDS, C)]
    got = k6_multi(sets, roi_cfg(GRIDS, C, 1), B, GRIDS, C)
    want = [np.zeros((C,) + g, np.float32) for g in GRIDS]
    for rois, counts, go in sets:
        k = int(counts[0])
        r, g = N(rois[0, :, :k]), N(go[:k])
        lv = oracle.level_map(r)
        for l, g_ in enumerate(GRIDS):
            m = lv == l
            want[l] += oracle.roi_align_bwd(g[m], (C,) + g_, np.ascontiguousarray(r[:, m]), 1.0 / (4 * 2 ** l))
    for l in range(len(GRIDS)):
        np.testing.assert_allclose(N(got[l][0]), want[l], rtol=1e-5, atol=5e-6)


@pytest.mark.parametrize("layout", [1, 0])
def test_multi_k6_one_set_is_the_batched_entry(layout):
    B, C = 4, 128
    rois, counts, go = ragged_set(np.random.default_rng(37), B, 96, [37, 0, 96, 11], GRIDS, C)
    cfg = roi_cfg(GRIDS, C, layout)
    one = k6_multi([(rois, counts, go)], cfg, B, GRIDS, C)
    again = k6_multi([(rois, counts, go)], cfg, B, GRIDS, C)
    ref = k6_batched(rois, counts, go, cfg, B, GRIDS, C)
    for a, b, c in zip(one, again, ref):
        assert same_bits(a, c) and same_bits(a, b)


def test_multi_k6_refuses_bad_arguments():
    B, C = 2, 128
    cfg = roi_cfg(GRIDS, C, 1)
    rois, counts, go = ragged_set(np.random.default_rng(1), B, 8, [3, 2], GRIDS, C)
    out = grad_maps(B, C, GRIDS, 1)
    ok = _C.lib().b2d_roi_align_bwd_multi_workspace_bytes(1, (_C.c_ll * 1)(8), B, ctypes.byref(cfg))
    ws = torch.empty(ok, dtype=torch.uint8, device=DEV)

    def call(S, ld=8, nbytes=ok, null=False):
        n = max(S, 1)
        p = lambda t: (_C.c_void_p * n)(*([None if null else t.data_ptr()] * n))
        _C.call("b2d_roi_align_bwd_multi", fused._ptrs(out), S, p(go), p(rois), (_C.c_ll * n)(*([ld] * n)), p(counts), B,
                ctypes.byref(cfg), _C.ptr(ws), nbytes, _C.stream())

    call(1)
    for kw in (dict(S=0), dict(S=5), dict(S=1, ld=0), dict(S=1, nbytes=ok - 1), dict(S=1, null=True)):
        with pytest.raises(_C.B200DetError):
            call(**kw)


# ------------------------------------------------------------------ CascadeTrainHotPath
B3, K3, C3, NC = 2, 8, 64, 21


def config3_inputs(B=B3, C=C3, K=K3):
    w = workload.config2(B=B, K=K, channels=C)
    x = dict(cls=[T(c) for c in w["cls"]], reg=[T(r) for r in w["reg"]],
             feats=[T(f).contiguous(memory_format=torch.channels_last) for f in w["feats"]],
             gt=T(w["gt"]), gt_count=torch.full((B,), K, dtype=torch.int32, device=DEV), gt_label=T(w["gt_label"]),
             img_hw=torch.tensor([[800.0, 1333.0]] * B, device=DEV))
    return w, x


def fixed_heads(B, m, reg_c, seed=2019):
    """Seeded head outputs (the recipe of scripts/bench_infer.py): the heads' layers are not part of the path."""
    rng = np.random.default_rng(seed)
    outs = []
    for _ in range(3):
        cls = rng.normal(0, 2.5, (B * m, NC)).astype(np.float32)
        cls[:, 0] += 2.0
        reg = rng.normal(0, 0.5, (B * m, 4 * reg_c)).astype(np.float32)
        outs.append((T(cls), T(reg)))
    return [(lambda f, o=o: o) for o in outs], outs


def cascade_path(w, seed=3, agnostic=False, **kw):
    return fused.CascadeTrainHotPath(B3, w["grids"], DEV, gt_ld=K3, feat_channels=C3, num_classes=NC,
                                     reg_class_agnostic=agnostic, seed=seed, **kw)


def run(cp, x, heads):
    return cp.step(x["cls"], x["reg"], x["feats"], x["gt"], x["gt_count"], x["gt_label"], x["img_hw"], heads)


@pytest.mark.parametrize("agnostic", [False, True])
def test_cascade_step_stage0_is_train_hot_path_and_later_stages_match_the_oracle(agnostic):
    from oracle import sampler_spec
    w, x = config3_inputs()
    seed = 3
    cp = cascade_path(w, seed=seed, agnostic=agnostic)
    reg_c = 1 if agnostic else NC
    heads, outs = fixed_heads(B3, cp.m, reg_c)
    out = run(cp, x, heads)
    hp = fused.TrainHotPath(B3, w["grids"], DEV, gt_ld=K3, feat_channels=C3, seed=seed)
    ref = hp.step(x["cls"], x["reg"], x["feats"], x["gt"], x["gt_count"], x["gt_label"], x["img_hw"])
    torch.cuda.synchronize()
    # ---- stage 0 and the RPN side: TrainHotPath at the same seed
    for k in ("props", "scores", "prop_count", "rpn_tar_cls", "rpn_tar_reg", "roi_feats"):
        assert same_bits(out[k], ref[k]), k
    for a, b in ((out["rpn"], ref["rpn"]), (out["rcnn"], ref["rcnn"])):
        assert torch.equal(a.n_chosen, b.n_chosen)
        for b_ in range(B3):
            n = int(a.n_chosen[b_])
            assert torch.equal(a.chosen[b_, :n], b.chosen[b_, :n])
            for f in ("tar_box", "tar_gt", "tar_param"):
                assert same_bits(getattr(a, f)[b_, :, :n], getattr(b, f)[b_, :, :n]), f
            assert torch.equal(a.tar_label[b_, :n], b.tar_label[b_, :n])
    # ---- stages 1 and 2 against the oracle, on the boxes the previous stage refined
    gt, gl = N(x["gt"]), N(x["gt_label"])
    feats_np = w["feats"]
    m = cp.m
    for s in range(1, 3):
        prev, st = out["stages"][s - 1], out["stages"][s]
        pb = prev["targets"]
        bt = st["targets"]
        for b in range(B3):
            # refine of the previous stage: its sampled boxes decoded with its reg_out at the sampled labels, GT dropped
            k0 = int(pb.n_chosen[b])
            want0 = N(pb.chosen[b, :k0])
            tb0 = N(pb.tar_box[b, :, :k0])
            lab = N(pb.tar_label[b, :k0])
            reg_np = N(outs[s - 1][1])[b * m:b * m + k0].reshape(k0, 4, reg_c)
            reg = reg_np[np.arange(k0), :, 0 if agnostic else lab].T
            keep = N(pb.tar_is_gt[b, :k0]) == 0
            dec = oracle.param2bbox(np.ascontiguousarray(tb0[:, keep]), np.ascontiguousarray(reg[:, keep]), [0.0] * 4,
                                    list(STDS[s - 1]), (800, 1333))
            kr = int(prev["count"][b])
            assert kr == int(keep.sum()) and want0.shape[0] == k0
            np.testing.assert_allclose(N(prev["boxes"][b, :, :kr]), dec, rtol=1e-5, atol=1e-5)
            cur = np.ascontiguousarray(N(prev["boxes"][b, :, :kr]))
            # this stage's targets and RoI features
            olab, _ = oracle.assign_max_iou(cur, gt[b], THRESHOLDS[s], THRESHOLDS[s], THRESHOLDS[s])
            full = np.concatenate([np.arange(1, K3 + 1), olab]).astype(np.int64)
            assert np.array_equal(N(bt.labels[b, :full.shape[0]]), full), (s, b)
            want = sampler_spec.sample(full, m, 128, ((seed + 1 + s) * 1000003 + 1) & 0xFFFFFFFFFFFFFFFF, image_index=b)
            k = int(bt.n_chosen[b])
            assert np.array_equal(N(bt.chosen[b, :k]), want), (s, b)
            tb = np.concatenate([gt[b], cur], 1)[:, want]
            np.testing.assert_array_equal(N(bt.tar_box[b, :, :k]), tb)
            tg = gt[b][:, np.maximum(full[want] - 1, 0)]
            np.testing.assert_allclose(N(bt.tar_param[b, :, :k]), oracle.bbox2param(tb, tg, [0.0] * 4, list(STDS[s])),
                                       rtol=1e-5, atol=1e-5)
            rf = oracle.roi_extract([f[b] for f in feats_np], tb)
            assert np.array_equal(N(st["roi_feats"][b * m:b * m + k]).view(np.uint32), rf.view(np.uint32)), (s, b)
    assert out["stages"][2]["boxes"] is None


def head_grads_reference(cls_maps, reg_maps, chosen, n_chosen, g_cls, g_reg):
    """torch autograd of the reference's gather (lib/anchor.py:49-56)."""
    cl = [c.detach().clone().requires_grad_(True) for c in cls_maps]
    rl = [r.detach().clone().requires_grad_(True) for r in reg_maps]
    loss = 0
    for b in range(cl[0].shape[0]):
        n = int(n_chosen[b])
        idx = chosen[b, :n].long()
        cls_out = torch.cat([x[b].view(1, -1) for x in cl], dim=1)
        reg_out = torch.cat([x[b].view(4, -1) for x in rl], dim=1)
        loss = loss + (cls_out[:, idx] * g_cls[b, :, :n]).sum() + (reg_out[:, idx] * g_reg[b, :, :n]).sum()
    loss.backward()
    return [x.grad for x in cl], [x.grad for x in rl]


def upstream(cp, seed, poison=True):
    g = torch.Generator(device=DEV).manual_seed(seed)
    g_cls = torch.randn(cp.tar_cls.shape, device=DEV, generator=g)
    g_reg = torch.randn(cp.tar_reg.shape, device=DEV, generator=g)
    g_roi = [torch.randn(ra.out.shape, device=DEV, generator=g) for ra in cp.roi_align]
    if poison:
        n_rpn = N(cp.rpn_targets.n_chosen)
        for b in range(cp.B):
            g_cls[b, :, n_rpn[b]:] = float("nan")
            g_reg[b, :, n_rpn[b]:] = float("nan")
            for t, g_ in zip(cp.targets, g_roi):
                g_[b * cp.m + int(t.n_chosen[b]):(b + 1) * cp.m] = float("nan")
    return g_cls, g_reg, g_roi


def feat_grads_reference(cp, g_roi):
    """b2d_roi_align_bwd on the concatenated stage RoIs (set-major, stages whose gradient is None left out)."""
    cfg = cp.roi_align[0].cfg
    grids = [(cfg.H[l], cfg.W[l]) for l in range(cfg.num_levels)]
    sets = [(t.tar_box, t.n_chosen, g) for t, g in zip(cp.targets, g_roi) if g is not None]
    return k6_compacted(sets, cfg, cp.B, grids, cfg.C)


def test_cascade_backward_vs_references():
    w, x = config3_inputs()
    cp = cascade_path(w)
    heads, _ = fixed_heads(B3, cp.m, NC)
    out = run(cp, x, heads)
    g_cls, g_reg, g_roi = upstream(cp, 11)
    dcls, dreg, dfeat = cp.backward(g_cls, g_reg, g_roi)
    rt = out["rpn"]
    ref_cls, ref_reg = head_grads_reference(x["cls"], x["reg"], rt.chosen, N(rt.n_chosen), g_cls, g_reg)
    for a, b in zip(list(dcls) + list(dreg), ref_cls + ref_reg):
        assert same_bits(a, b)
    for a, b in zip(dfeat, feat_grads_reference(cp, g_roi)):
        assert same_bits(a, b)
        assert a.is_contiguous(memory_format=torch.channels_last) and not torch.isnan(a).any()
    # a stage left out; then no stage at all (zero feature gradient)
    part = [g_roi[0], None, g_roi[2]]
    for a, b in zip(cp.backward(g_cls, g_reg, part)[2], feat_grads_reference(cp, part)):
        assert same_bits(a, b)
    assert all(not t.any() for t in cp.backward(g_cls, g_reg, [None] * 3)[2])


def test_cascade_step_and_backward_in_one_cuda_graph():
    w, x = config3_inputs()
    cp = cascade_path(w, seed=5)
    heads, _ = fixed_heads(B3, cp.m, NC)
    run(cp, x, heads)
    g_cls, g_reg, g_roi = upstream(cp, 12, poison=False)
    cp.backward(g_cls, g_reg, g_roi)                                    # first call: buffers
    torch.cuda.synchronize()
    cp.reset_step()
    out = run(cp, x, heads)
    eager = [t.clone() for ts in cp.backward(g_cls, g_reg, g_roi) for t in ts]
    # later stages can take every candidate (the same index list each step): their samples are compared by box
    samples = lambda: [cp.rpn_targets.chosen.clone()] + [t.tar_box.clone() for t in cp.targets]
    eager_samples = samples()
    eager_feats = [st["roi_feats"].clone() for st in out["stages"]]
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(graph, stream=side):
            gout = run(cp, x, heads)
            grads = cp.backward(g_cls, g_reg, g_roi)
    torch.cuda.current_stream().wait_stream(side)
    cp.reset_step()
    graph.replay()
    torch.cuda.synchronize()
    assert all(same_bits(a, b) for a, b in zip([t for ts in grads for t in ts], eager))
    assert all(torch.equal(a, b) for a, b in zip(samples(), eager_samples))
    assert all(same_bits(st["roi_feats"], f) for st, f in zip(gout["stages"], eager_feats))
    graph.replay()
    torch.cuda.synchronize()
    for a, b in zip(samples(), eager_samples):
        assert not torch.equal(a, b), "a replay draws fresh samples in the RPN and in every stage"
    for a, b in zip(grads[2], feat_grads_reference(cp, g_roi)):
        assert same_bits(a, b)


class StageHead(torch.nn.Module):
    def __init__(self, C, reg_c, seed):
        super().__init__()
        torch.manual_seed(seed)
        self.cls = torch.nn.Linear(C * 49, NC).to(DEV)
        self.reg = torch.nn.Linear(C * 49, 4 * reg_c).to(DEV)

    def forward(self, x):
        f = x.flatten(1)
        return self.cls(f), self.reg(f)


def autograd_case(stages_in_loss=(0, 1, 2)):
    w, x = config3_inputs()
    cp = cascade_path(w, seed=7)
    heads = [StageHead(C3, NC, 100 + s) for s in range(3)]
    cls = [c.clone().requires_grad_(True) for c in x["cls"]]
    reg = [r.clone().requires_grad_(True) for r in x["reg"]]
    feats = [f.clone().requires_grad_(True) for f in x["feats"]]
    out = cp.step_autograd(cls, reg, feats, x["gt"], x["gt_count"], x["gt_label"], x["img_hw"], heads)
    seen = [None] * 3
    for s, st in enumerate(out["stages"]):
        st["roi_feats"].register_hook(lambda g, s=s: seen.__setitem__(s, g.clone()))
    gen = torch.Generator(device=DEV).manual_seed(13)
    g_cls = torch.randn(cp.tar_cls.shape, device=DEV, generator=gen)
    g_reg = torch.randn(cp.tar_reg.shape, device=DEV, generator=gen)
    loss = (out["rpn_tar_cls"] * g_cls).sum() + (out["rpn_tar_reg"] * g_reg).sum()
    for s in stages_in_loss:
        st = out["stages"][s]
        loss = loss + st["cls_out"].square().mean() + (st["reg_out"] * 0.5).sum()
    return cp, heads, out, (cls, reg, feats), seen, (g_cls, g_reg), loss


@pytest.mark.parametrize("stages_in_loss", [(0, 1, 2), (0, 2)])
def test_cascade_autograd_matches_explicit_backward(stages_in_loss, monkeypatch):
    cp, heads, out, (cls, reg, feats), seen, (g_cls, g_reg), loss = autograd_case(stages_in_loss)
    calls = []
    real = _C.call
    monkeypatch.setattr(_C, "call", lambda name, *a: (calls.append(name), real(name, *a))[1])
    loss.backward()
    monkeypatch.undo()
    assert calls.count("b2d_roi_align_bwd_multi") == 1 and "b2d_roi_align_bwd_batched" not in calls, calls
    leaf = [t.grad.clone() for t in cls + reg + feats]
    for s in range(3):
        assert (seen[s] is None) == (s not in stages_in_loss)
    dcls, dreg, dfeat = cp.backward(g_cls, g_reg, seen)
    for a, b in zip(leaf, list(dcls) + list(dreg) + list(dfeat)):
        assert same_bits(a, b)
    # head parameters: autograd of the same loss terms on the stage features alone
    for s in range(3):
        h = heads[s]
        if s not in stages_in_loss:
            assert h.cls.weight.grad is None
            continue
        co, ro = h(out["stages"][s]["roi_feats"].detach())
        want = torch.autograd.grad(co.square().mean() + (ro * 0.5).sum(), list(h.parameters()))
        for p, g in zip(h.parameters(), want):
            assert same_bits(p.grad, g)


def test_cascade_autograd_backward_after_a_later_step_raises():
    cp, heads, out, (cls, reg, feats), _, _, loss = autograd_case()
    x = config3_inputs()[1]
    cp.step_autograd(cls, reg, feats, x["gt"], x["gt_count"], x["gt_label"], x["img_hw"], heads)
    with pytest.raises(_C.B200DetError, match="another step"):
        loss.backward()


def test_cascade_wrong_head_shape_raises_before_refine(monkeypatch):
    w, x = config3_inputs()
    cp = cascade_path(w)
    heads, outs = fixed_heads(B3, cp.m, NC)
    heads[0] = lambda f: (outs[0][0], outs[0][1][:, :4])
    calls = []
    real = _C.call
    monkeypatch.setattr(_C, "call", lambda name, *a: (calls.append(name), real(name, *a))[1])
    with pytest.raises(_C.B200DetError, match="stage 0 head"):
        run(cp, x, heads)
    assert "b2d_refine_bboxes" not in calls


def test_cascade_constructor_refusals():
    w = workload.config2(B=1, K=2, channels=128, with_feats=False)
    for kw in (dict(layout=2), dict(num_stages=0), dict(num_stages=4), dict(num_stages=3, thresholds=(0.5, 0.6)),
               dict(num_stages=2, stage_stds=((0.1, 0.1, 0.2, 0.2),))):
        with pytest.raises(_C.B200DetError):
            fused.CascadeTrainHotPath(1, w["grids"], DEV, gt_ld=2, feat_channels=128, **kw)
