"""GPU parity of the batched one-stage test path (fused.DenseInferHotPath): RetinaNet (BASELINE config 4) and FCOS /
ATSS (config 5) head maps -> packed detections.  B = 1 against the reference's golden outputs; ragged batches image by
image against the per-image drop-ins (heads.anchor_head_predict_single_image / heads.fcos_predict_single_image); records,
CUDA-graph replay, no host synchronisation, empty images and the candidate overflow flag."""
import json
import os
import sys
import types

import numpy as np
import pytest
import torch

from conftest import load_golden

pytestmark = pytest.mark.gpu

if torch.cuda.is_available():
    import b200det
    from b200det import _C, fused, heads as bheads
    DEV = torch.device("cuda:0")

FCOS_STRIDES = [8, 16, 32, 64, 128]
FCOS_CFGS = [dict(pre_nms=1000, min_bbox_size=0, min_score=0.05, nms_iou=0.6, nms_type="strict", max_per_img=100),
             dict(pre_nms=50, min_bbox_size=40, min_score=0.3, nms_iou=0.5, nms_type="official", max_per_img=60)]


def T(a):
    return torch.from_numpy(np.ascontiguousarray(a)).to(DEV)


def N(t):
    return t.detach().cpu().numpy()


def _gin():
    sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden"))
    import inputs as gin
    return gin


def _assert_dets(out, b, box, score, label, records=None):
    k = int(out["count"][b])
    assert k == int(score.shape[0]), (b, k, tuple(score.shape))
    assert np.array_equal(N(out["labels"][b, :k]), N(label) if torch.is_tensor(label) else label)
    np.testing.assert_allclose(N(out["scores"][b, :k]), N(score) if torch.is_tensor(score) else score, rtol=1e-5, atol=1e-7)
    np.testing.assert_allclose(N(out["boxes"][b, :, :k]), N(box) if torch.is_tensor(box) else box, rtol=1e-5, atol=1e-3)
    if records is not None:
        r = N(records[b])
        assert np.array_equal(r[:k, :4], N(out["boxes"][b, :, :k]).T)
        assert np.array_equal(r[:k, 4], N(out["scores"][b, :k]))
        assert np.array_equal(r[:k, 5], N(out["labels"][b, :k]).astype(np.float32))
        assert (r[k:] == 0).all()
    return k


# ------------------------------------------------------------------ 1. RetinaNet vs the reference
@pytest.mark.parametrize("i", [0, 1])
def test_retinanet_b1_vs_reference(i):
    """config-4 sizes (201 600 anchors x 20 classes): heads2 ret_* (strict at pre 1000; official with min_bbox_size 24)."""
    gin = _gin()
    g = load_golden("heads2")
    cls, reg = gin.retina_inputs(20)
    cfg = json.loads(str(g["ret_cfgs"][i]))
    hp = fused.DenseInferHotPath(1, gin.RETINA_GRIDS, DEV, head="retina", num_classes=21, test_cfg=cfg,
                                 strides=gin.RETINA_STRIDES, anchor_scales=gin.RETINA_SCALES)
    rec = torch.full((1, hp.M, 6), -7.0, device=DEV)
    out = hp.step([T(x)[None] for x in cls], [T(x)[None] for x in reg], torch.tensor([[800.0, 1333.0]], device=DEV),
                  records=rec)
    hp.check()
    assert _assert_dets(out, 0, g["ret_bbox%d" % i], g["ret_score%d" % i], g["ret_label%d" % i], rec) > 0


def test_retinanet_softmax_head_b1_vs_reference():
    g = load_golden("heads2")
    cfg = json.loads(str(g["sm_cfg"]))
    grids = [(20, 28), (10, 14), (5, 7)]
    hp = fused.DenseInferHotPath(1, grids, DEV, head="retina", num_classes=5, test_cfg=cfg, strides=(8, 16, 32),
                                 use_sigmoid=False, anchor_scales=(8,))
    out = hp.step([T(g["sm_cls%d" % k])[None] for k in range(3)], [T(g["sm_reg%d" % k])[None] for k in range(3)],
                  torch.tensor([[160.0, 213.0]], device=DEV))
    hp.check()
    assert _assert_dets(out, 0, g["sm_bbox"], g["sm_score"], g["sm_label"]) > 0


# ------------------------------------------------------------------ 2. FCOS vs the reference
@pytest.mark.parametrize("i", [0, 1])
def test_fcos_b1_vs_reference(i):
    g = load_golden("heads")
    cls = [T(g["fc_cls%d" % l])[None] for l in range(5)]
    reg = [T(g["fc_reg%d" % l])[None] for l in range(5)]
    ctr = [T(g["fc_ctr%d" % l])[None] for l in range(5)]
    grids = [tuple(c.shape[-2:]) for c in cls]
    img = tuple(int(v) for v in g["fc_img"])
    hp = fused.DenseInferHotPath(1, grids, DEV, head="fcos", num_classes=int(cls[0].shape[1]) + 1, test_cfg=FCOS_CFGS[i],
                                 strides=FCOS_STRIDES, reg_mean=0.0, reg_std=300.0, use_centerness=True)
    out = hp.step(cls, reg, torch.tensor([[float(img[0]), float(img[1])]], device=DEV), ctr_outs=ctr)
    hp.check()
    assert _assert_dets(out, 0, g["fc_bbox%d" % i], g["fc_score%d" % i], g["fc_label%d" % i]) > 0


# ------------------------------------------------------------------ 3. + 4. ragged batches vs the per-image drop-ins
RET_GRIDS, RET_STRIDES = [(40, 52), (20, 26), (10, 13)], [8, 16, 32]
RET_SCALES = [4 * 2 ** (i / 3) for i in range(3)]
IMGS = [(300.0, 400.0), (277.0, 389.0), (318.0, 350.0)]


def _retina_case(use_sigmoid, seed, B=3):
    rng = np.random.default_rng(seed)
    C = 6 if use_sigmoid else 7
    cls = [rng.standard_normal((B, 9 * C) + g).astype(np.float32) * 2.0 - 1.0 for g in RET_GRIDS]
    if B > 2 and use_sigmoid:
        # image 2, level 0: many tied logits.  (Not for softmax: there equal sets of logits in a different channel order
        # give scores that differ in the last bit with the summation order, which the reference does not fix.)
        cls[0][2] = np.round(cls[0][2] * 2.0) / 2.0
    reg = [(0.3 * rng.standard_normal((B, 36) + g)).astype(np.float32) for g in RET_GRIDS]
    head = types.SimpleNamespace(anchor_strides=RET_STRIDES, anchor_scales=RET_SCALES, anchor_ratios=[0.5, 1.0, 2.0],
                                 target_means=[0.0] * 4, target_stds=[1.0] * 4, use_sigmoid=use_sigmoid, cls_channels=C,
                                 num_classes=C + 1 if use_sigmoid else C, anchor_creators=None)
    return [T(c) for c in cls], [T(r) for r in reg], head


@pytest.mark.parametrize("use_sigmoid", [True, False])
@pytest.mark.parametrize("mode", ["official", "strict"])
def test_retinanet_ragged_batch_equals_per_image(use_sigmoid, mode):
    cls, reg, head = _retina_case(use_sigmoid, 11)
    B = 3
    cfg = dict(pre_nms=300, min_bbox_size=0, min_score=0.3, nms_iou=0.5, max_per_img=100, nms_type=mode)
    hp = fused.DenseInferHotPath(B, RET_GRIDS, DEV, head="retina", num_classes=head.num_classes, test_cfg=cfg,
                                 strides=RET_STRIDES, use_sigmoid=use_sigmoid, anchor_scales=RET_SCALES)
    rec = torch.full((B, hp.M, 6), -7.0, device=DEV)
    out = hp.step(cls, reg, torch.tensor(IMGS, device=DEV), records=rec)
    hp.check()
    anchors = [torch.empty((4, 9) + g, device=DEV) for g in RET_GRIDS]
    for b in range(B):
        meta = dict(img_shape=(int(IMGS[b][0]), int(IMGS[b][1]), 3), scale_factor=1.0)
        bx, sc, lb = bheads.anchor_head_predict_single_image(head, [c[b] for c in cls], [r[b] for r in reg], anchors, meta, cfg)
        assert _assert_dets(out, b, bx, sc, lb, rec) > 3, b


FC_GRIDS = [(40, 52), (20, 26), (10, 13), (5, 7), (3, 4)]


def _fcos_case(seed, B=3, C=5):
    rng = np.random.default_rng(seed)
    cls = [(rng.standard_normal((B, C) + g) * 2.0 - 2.0).astype(np.float32) for g in FC_GRIDS]
    reg = [np.abs(0.05 + 0.05 * rng.standard_normal((B, 4) + g)).astype(np.float32) for g in FC_GRIDS]
    ctr = [rng.standard_normal((B, 1) + g).astype(np.float32) for g in FC_GRIDS]
    # image 1, level 1 (520 points, pre_nms 300): all but 100 boxes below min_bbox_size -> the ascending-index branch
    small = np.full((4,) + FC_GRIDS[1], 0.003, np.float32)
    small.reshape(4, -1)[:, rng.choice(520, 100, replace=False)] = 0.05
    if B > 2:
        reg[1][1] = small
        cls[0][2] = np.round(cls[0][2] * 2.0) / 2.0                  # image 2, level 0: tied keys
        ctr[0][2] = 0.5
    return [T(c) for c in cls], [T(r) for r in reg], [T(c) for c in ctr]


@pytest.mark.parametrize("centerness", [True, False])
@pytest.mark.parametrize("mode", ["official", "strict"])
def test_fcos_ragged_batch_equals_per_image(centerness, mode):
    cls, reg, ctr = _fcos_case(5)
    B, C = 3, int(cls[0].shape[1])
    cfg = dict(pre_nms=300, min_bbox_size=8, min_score=0.2, nms_iou=0.5, max_per_img=80, nms_type=mode)
    hp = fused.DenseInferHotPath(B, FC_GRIDS, DEV, head="fcos", num_classes=C + 1, test_cfg=cfg, strides=FCOS_STRIDES,
                                 reg_mean=0.0, reg_std=300.0, use_centerness=centerness)
    rec = torch.full((B, hp.M, 6), -7.0, device=DEV)
    out = hp.step(cls, reg, torch.tensor(IMGS, device=DEV), ctr_outs=ctr if centerness else None, records=rec)
    hp.check()
    # the ascending-index branch was taken: image 1 keeps fewer than pre_nms points of level 1
    key1 = N(hp.key[1, 2080:2600])
    assert 0 < (key1 > -np.inf).sum() < 300
    for b in range(B):
        meta = dict(img_shape=(int(IMGS[b][0]), int(IMGS[b][1]), 3), scale_factor=1.0)
        bx, sc, lb = bheads.fcos_predict_single_image([c[b] for c in cls], [r[b] for r in reg], [c[b] for c in ctr],
                                                      FCOS_STRIDES, meta, cfg, 0.0, 300.0, use_centerness=centerness)
        assert _assert_dets(out, b, bx, sc, lb, rec) > 3, b


# ------------------------------------------------------------------ 5. graph replay and no host synchronisation
def _graph_vs_eager(hp, step):
    out = step()                                                    # first eager call (module load, kernel attributes)
    torch.cuda.synchronize()
    torch.cuda.set_sync_debug_mode("error")
    try:
        out = step()
    finally:
        torch.cuda.set_sync_debug_mode(0)
    hp.check()
    eager = {k: out[k].clone() for k in ("boxes", "scores", "labels", "count", "records")}
    for k in eager:
        out[k].zero_()
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(graph, stream=side):
            step()
    torch.cuda.current_stream().wait_stream(side)
    for k in eager:
        out[k].zero_()
    graph.replay()
    graph.replay()
    torch.cuda.synchronize()
    for k, v in eager.items():
        assert torch.equal(out[k], v), k
    assert int(eager["count"].sum()) > 0


def test_graph_replay_equals_eager_and_step_never_syncs_retina():
    cls, reg, head = _retina_case(True, 3)
    cfg = dict(pre_nms=300, min_bbox_size=0, min_score=0.3, nms_iou=0.5, max_per_img=100, nms_type="official")
    hp = fused.DenseInferHotPath(3, RET_GRIDS, DEV, head="retina", num_classes=7, test_cfg=cfg, strides=RET_STRIDES,
                                 anchor_scales=RET_SCALES)
    rec = torch.zeros((3, hp.M, 6), device=DEV)
    hw = torch.tensor(IMGS, device=DEV)
    _graph_vs_eager(hp, lambda: hp.step(cls, reg, hw, records=rec))


def test_graph_replay_equals_eager_and_step_never_syncs_fcos():
    cls, reg, ctr = _fcos_case(8)
    cfg = dict(pre_nms=300, min_bbox_size=8, min_score=0.2, nms_iou=0.5, max_per_img=80, nms_type="strict")
    hp = fused.DenseInferHotPath(3, FC_GRIDS, DEV, head="fcos", num_classes=6, test_cfg=cfg, strides=FCOS_STRIDES)
    rec = torch.zeros((3, hp.M, 6), device=DEV)
    hw = torch.tensor(IMGS, device=DEV)
    _graph_vs_eager(hp, lambda: hp.step(cls, reg, hw, ctr_outs=ctr, records=rec))


# ------------------------------------------------------------------ 6. edge cases
def test_image_without_candidates_gives_count_zero_and_zero_records():
    cls, reg, head = _retina_case(True, 4, B=2)
    with torch.no_grad():
        for c in cls:
            c[1].fill_(-20.0)                                        # sigmoid ~ 2e-9 < min_score
    cfg = dict(pre_nms=300, min_bbox_size=0, min_score=0.05, nms_iou=0.5, max_per_img=100, nms_type="official")
    hp = fused.DenseInferHotPath(2, RET_GRIDS, DEV, head="retina", num_classes=7, test_cfg=cfg, strides=RET_STRIDES,
                                 anchor_scales=RET_SCALES)
    rec = torch.full((2, hp.M, 6), -7.0, device=DEV)
    out = hp.step(cls, reg, torch.tensor(IMGS[:2], device=DEV), records=rec)
    hp.check()
    assert int(out["count"][0]) > 0 and int(out["count"][1]) == 0
    assert (N(rec[1]) == 0).all() and (N(out["labels"][1]) == 0).all() and (N(out["scores"][1]) == 0).all()


def test_more_than_16384_candidates_sets_the_flag_and_check_raises():
    rng = np.random.default_rng(9)
    C = 20
    cls = [T(rng.standard_normal((1, 9 * C) + g).astype(np.float32)) for g in RET_GRIDS]
    reg = [T((0.3 * rng.standard_normal((1, 36) + g)).astype(np.float32)) for g in RET_GRIDS]
    cfg = dict(pre_nms=1000, min_bbox_size=0, min_score=0.01, nms_iou=0.5, max_per_img=100, nms_type="official")
    hp = fused.DenseInferHotPath(1, RET_GRIDS, DEV, head="retina", num_classes=C + 1, test_cfg=cfg, strides=RET_STRIDES,
                                 anchor_scales=RET_SCALES)
    assert hp.cap == 16384 and hp.P * C > 16384
    hp.step(cls, reg, torch.tensor([IMGS[0]], device=DEV))
    with pytest.raises(_C.B200DetError, match="16384"):
        hp.check()


def test_unsupported_configurations_raise_before_any_kernel():
    cfg = dict(pre_nms=100, min_bbox_size=0, min_score=0.05, nms_iou=0.5, max_per_img=100, nms_type="official")
    with pytest.raises(_C.B200DetError, match="class channels"):
        fused.DenseInferHotPath(1, RET_GRIDS, DEV, head="retina", num_classes=130, test_cfg=cfg, strides=RET_STRIDES)
    big = dict(cfg, pre_nms=17000)
    with pytest.raises(_C.B200DetError, match="16384"):
        fused.DenseInferHotPath(1, [(150, 150)], DEV, head="fcos", num_classes=3, test_cfg=big, strides=[8])
    hp = fused.DenseInferHotPath(1, FC_GRIDS, DEV, head="fcos", num_classes=6, test_cfg=cfg, strides=FCOS_STRIDES)
    cls, reg, ctr = _fcos_case(1, B=1)
    hw = torch.tensor([IMGS[0]], device=DEV)
    with pytest.raises(_C.B200DetError, match="cls_outs"):
        hp.step(cls[:4], reg, hw, ctr_outs=ctr)
    with pytest.raises(_C.B200DetError, match="ctr_outs"):
        hp.step(cls, reg, hw)
    with pytest.raises(_C.B200DetError, match="records"):
        hp.step(cls, reg, hw, ctr_outs=ctr, records=torch.zeros((1, hp.M, 5), device=DEV))
