"""The class-dependent detection kernels at COCO width (80 / 81 classes) and at the 128-class limit.

The candidate kernels hold a row's classes four per lane (class c = 32 r + lane, r = 0..3) and the NMS channels in a
two-word bitmap.  At 20 / 21 classes the lane groups r = 2, 3, the second bitmap word, cross-group arg-max ties and the
class-minor candidate order across groups never run; these tests run them against plain references kept in this file:
numpy in float64 wherever a score is computed, and the C oracle (oracle.topk_desc, param2bbox, batched_nms,
anchor_head_loss) where it defines the semantics.

An fp32 kernel and a float64 reference must never disagree about a decision only through rounding, so the references
assert a margin at every decision point (score against min_score, IoU against the NMS threshold, the k-th against the
(k+1)-th key of a top-k, near-equal scores whose order matters).  Exact ties are built only from equal logits, for
which both sides compute bit-equal scores; logits are drawn on a 1/8 grid for that reason."""
import numpy as np
import pytest
import torch

import oracle

pytestmark = [pytest.mark.gpu, pytest.mark.skipif(not torch.cuda.is_available(), reason="needs a CUDA device")]

if torch.cuda.is_available():
    import b200det
    from b200det import _C, fused, heads as bheads, utils as butils, workload
    DEV = torch.device("cuda:0")

EPS_SCORE = 1e-6          # relative: two float64 scores closer than this could order either way in fp32
EPS_IOU = 2e-4            # absolute, boxes decoded on both sides: a one-ulp difference moves an offset box (label x max
                          # coordinate) by < 1e-4 IoU at these sizes
EPS_IOU_SAME = 1e-6       # the same fp32 boxes on both sides: only the IoU arithmetic rounds


def T(a):
    return torch.from_numpy(np.ascontiguousarray(a)).to(DEV)


def N(t):
    return t.detach().cpu().numpy()


def _q(x):
    """Logits on a 1/8 grid: equal values give bit-equal scores on both sides, distinct ones are far apart."""
    return (np.round(np.asarray(x) * 8.0) / 8.0).astype(np.float32)


def _sigmoid64(x):
    return 1.0 / (1.0 + np.exp(-np.asarray(x, np.float64)))


def _softmax64(x, axis):
    x = np.asarray(x, np.float64)
    e = np.exp(x - x.max(axis, keepdims=True))
    return e / e.sum(axis, keepdims=True)


# ------------------------------------------------------------------ margins
def _margin(v, thr, eps, what):
    v = np.asarray(v, np.float64).reshape(-1)
    bad = np.abs(v - thr) <= eps * max(1.0, abs(thr))
    assert not bad.any(), "%s: %d value(s) within %g of the threshold %r; change the seed" % (what, int(bad.sum()), eps, thr)


def _order_margin(s, what, eps=EPS_SCORE):
    """s: float64 keys in their decided (descending) order: adjacent distinct keys must be clearly apart."""
    s = np.asarray(s, np.float64)
    if s.size < 2:
        return
    d = np.abs(s[:-1] - s[1:])
    bad = (d > 0) & (d <= eps * np.maximum(np.abs(s[:-1]), np.abs(s[1:])))
    assert not bad.any(), "%s: %d near-tied adjacent key(s); change the seed" % (what, int(bad.sum()))


def _topk_margin(key64, k, what):
    """Top-k on float64 keys: the kept ones and the first left out must be strictly ordered or exactly tied."""
    key64 = np.asarray(key64, np.float64)
    srt = np.sort(key64[np.isfinite(key64)])[::-1]
    _order_margin(srt[:k + 1], what)


def _iou_one(a, b):
    """IoU of box a [4] with boxes b [m, 4] as torchvision computes it (no +1), in float64."""
    w = np.maximum(0.0, np.minimum(a[2], b[:, 2]) - np.maximum(a[0], b[:, 0]))
    h = np.maximum(0.0, np.minimum(a[3], b[:, 3]) - np.maximum(a[1], b[:, 1]))
    inter = w * h
    with np.errstate(invalid="ignore", divide="ignore"):
        return inter / ((a[2] - a[0]) * (a[3] - a[1]) + (b[:, 2] - b[:, 0]) * (b[:, 3] - b[:, 1]) - inter)


def _nms_margins(cb, s64, lab, keep, thr, max_num, eps_iou, eps_score):
    """Class-offset NMS replayed per class in float64 on the offset boxes both sides compute: every IoU that a kept box
    tests against a live candidate is clear of the threshold, a live candidate it suppresses is not near-tied with it in
    score, and the first max_num + 1 survivors are strictly ordered or exactly tied."""
    if len(s64) == 0:
        return
    mx = np.float32(cb.max())
    off = (lab.astype(np.float32) * mx).astype(np.float32)
    nb = (cb + off[:, None]).astype(np.float32).astype(np.float64)
    s32 = s64.astype(np.float32)
    for c in np.unique(lab):
        idx = np.nonzero(lab == c)[0]
        order = idx[np.lexsort((idx, -s32[idx]))]                     # score descending, ties by candidate index
        b, s = nb[order], s64[order]
        alive = np.ones(order.size, bool)
        for p in range(order.size):
            if not alive[p]:
                continue
            rest = np.nonzero(alive[p + 1:])[0] + p + 1
            if rest.size == 0:
                break
            iou = _iou_one(b[p], b[rest])
            near = np.abs(iou - thr) <= eps_iou
            assert not near.any(), "class %d: IoU within %g of %g; change the seed" % (c, eps_iou, thr)
            ds = np.abs(s[rest] - s[p])
            tied = (iou > thr) & (ds > 0) & (ds <= eps_score * s[p])
            assert not tied.any(), "class %d: a suppression between near-tied scores; change the seed" % c
            alive[rest[iou > thr]] = False
    _order_margin(s64[keep[:max_num + 1]], "survivor order", eps_score)


def _ref_detect(boxes, prob, chans, min_score, mode, nms_iou, max_num, factor=None, label_add=0, eps_iou=EPS_IOU,
                eps_score=EPS_SCORE):
    """utils.multiclass_nms (lib/utils.py:224-269) on float64 raw scores.  boxes fp32 [n, 4] or [n, 4, C]; prob float64
    [n, C]; factor float64 [n] or None.  Candidates in row-major, class-minor order; 'official' tests every NMS channel
    against min_score, 'strict' takes the first maximum over all channels.  -> (boxes [k, 4], float64 scores [k],
    labels [k], (rows, channels) of the candidates).  eps_iou / eps_score: the NMS margins (exact fp32 inputs and
    products, as in utils.multiclass_nms, need eps_score 0: both sides compare the same fp32 values)."""
    n, C = prob.shape
    cm = np.zeros(C, bool)
    cm[[int(c) for c in chans if 0 <= int(c) < C]] = True
    ms = float(np.float32(min_score))
    if mode == "official":
        _margin(prob[:, cm], ms, EPS_SCORE, "score vs min_score")
        ii, cc = np.nonzero((prob >= ms) & cm[None, :])
    else:
        cc_all = np.argmax(prob, 1)
        best = prob[np.arange(n), cc_all]
        if C > 1:
            second = np.where(np.arange(C)[None, :] == cc_all[:, None], -np.inf, prob).max(1)
            gap = best - second
            bad = (gap > 0) & (gap <= EPS_SCORE * best)
            assert not bad.any(), "strict: %d row(s) with a near-tied maximum; change the seed" % int(bad.sum())
        _margin(best[cm[cc_all]], ms, EPS_SCORE, "best score vs min_score")
        ii = np.nonzero(cm[cc_all] & (best >= ms))[0]
        cc = cc_all[ii]
    s64 = prob[ii, cc] * (np.asarray(factor, np.float64)[ii] if factor is not None else 1.0)
    cb = (boxes[ii] if boxes.ndim == 2 else boxes[ii, :, cc]).astype(np.float32)
    if ii.size == 0:
        return np.zeros((0, 4), np.float32), np.zeros(0), np.zeros(0, np.int64), (ii, cc)
    keep = oracle.batched_nms(np.ascontiguousarray(cb), s64.astype(np.float32), cc.astype(np.int64), nms_iou)
    _nms_margins(cb, s64, cc, keep, nms_iou, max_num, eps_iou, eps_score)
    keep = keep[:max_num]
    return cb[keep], s64[keep], cc[keep].astype(np.int64) + label_add, (ii, cc)


def _assert_dets(out, b, box, score, label, records=None):
    """Packed detections of image b against the reference: count and labels exact, scores rtol 1e-5, boxes atol 1e-3."""
    k = int(out["count"][b])
    assert k == score.shape[0], (b, k, score.shape)
    assert np.array_equal(N(out["labels"][b, :k]), label), b
    np.testing.assert_allclose(N(out["scores"][b, :k]), score, rtol=1e-5)
    np.testing.assert_allclose(N(out["boxes"][b, :, :k]), box.T, rtol=0, atol=1e-3)
    if records is not None:
        r = N(records[b])
        assert np.array_equal(r[:k, :4], N(out["boxes"][b, :, :k]).T)
        assert np.array_equal(r[:k, 4], N(out["scores"][b, :k]))
        assert np.array_equal(r[:k, 5], N(out["labels"][b, :k]).astype(np.float32))
        assert (r[k:] == 0).all()
    return k


def _tie_classes(c0, C):
    return [c0 + 32 * g for g in range(4) if c0 + 32 * g < C]


# ------------------------------------------------------------------ 1. utils.multiclass_nms
def _chan_sets(C):
    return {"fg": list(range(1, C)), "all": list(range(0, C)), "pair": [63, 64], "high": list(range(64, C)),
            "sparse": list(range(1, C, 6))}                              # odd classes 1, 7, ..., in both bitmap words


def _mc_case(C, n, per_class, use_factor, seed):
    rng = np.random.default_rng(seed)
    cx, cy = rng.uniform(0, 300, n), rng.uniform(0, 250, n)
    w, h = rng.uniform(8, 100, n), rng.uniform(8, 100, n)
    base = np.stack([cx - w / 2, cy - h / 2, cx + w / 2, cy + h / 2], 1).astype(np.float32)
    bbox = (base[:, :, None] + rng.normal(0, 3, (n, 4, C))).astype(np.float32) if per_class else base
    logit = _q(rng.normal(-4, 1.5, (n, C)))
    ties = rng.choice(n, 24, replace=False)
    for t, r in enumerate(ties):                 # row maximum tied across classes c0, c0 + 32, c0 + 64, c0 + 96
        logit[r, _tie_classes((7 * t) % 32, C)] = 3.0 + t / 8.0
    score = _sigmoid64(logit).astype(np.float32)
    fac = _sigmoid64(_q(rng.normal(0, 1, n) / 2)).astype(np.float32) if use_factor else None
    return bbox, score, fac, ties


MC_RUNS = [("official", 1500, True, False), ("official", 200, False, True), ("strict", 1500, True, False),
           ("strict", 200, False, True), ("strict", 17000, True, True)]


@pytest.mark.parametrize("chans", ["fg", "all", "pair", "high", "sparse"])
@pytest.mark.parametrize("C", [64, 65, 81, 128])
@pytest.mark.parametrize("mode,n,use_factor,per_class", MC_RUNS)
def test_multiclass_nms_wide_vs_reference(C, chans, mode, n, use_factor, per_class):
    """b2d_multiclass_nms, and b2d_multiclass_candidates + NMS when n x |channels| > 16384, at 64..128 classes, with
    NMS-channel sets in either bitmap word, official and strict, with and without score factor, shared and per-class
    boxes; rows whose maximum is tied across the four lane groups."""
    chan = _chan_sets(C)[chans]
    bbox, score, fac, ties = _mc_case(C, n, per_class, use_factor, seed=1000 * C + n)
    thr, ms, mn = 0.6, 0.2, 100
    kb, ks, kl = butils.multiclass_nms(T(bbox.reshape(n, -1)), T(score), chan, thr, ms, mn,
                                       T(fac) if use_factor else None, mode=mode)
    rb, rs, rl, _ = _ref_detect(bbox, score.astype(np.float64), chan, ms, mode, thr, mn,
                                fac.astype(np.float64) if use_factor else None, eps_iou=EPS_IOU_SAME, eps_score=0.0)
    assert np.array_equal(N(kl), rl)
    np.testing.assert_allclose(N(ks), rs, rtol=1e-5)
    np.testing.assert_allclose(N(kb), rb, rtol=0, atol=1e-3)
    # the tied rows, named explicitly: strict keeps the first tied class; official keeps equal scores in class order
    got_s, got_l = N(ks), N(kl)
    cm = set(c for c in chan if c < C)
    seen = 0
    for t, r in enumerate(ties):
        cls = _tie_classes((7 * t) % 32, C)
        v = np.float32(score[r, cls[0]] * (fac[r] if use_factor else np.float32(1)))
        at = np.nonzero(got_s == v)[0]
        if mode == "strict":
            assert set(got_l[at].tolist()) <= ({cls[0]} if cls[0] in cm else set()), (r, cls, got_l[at])
        else:
            assert np.all(np.diff(got_l[at]) > 0), (r, cls, got_l[at])
            assert set(got_l[at].tolist()) <= set(cls) & cm
        seen += at.size
    if mode == "official" and chans in ("fg", "all"):
        assert seen >= 24


def test_multiclass_nms_rejects_129_classes():
    bbox = T(np.tile(np.array([[0, 0, 10, 10]], np.float32), (5, 1)))
    with pytest.raises(AssertionError):
        butils.multiclass_nms(bbox, torch.full((5, 129), 0.5, device=DEV), range(129), 0.5, 0.1, 10)
    kb, ks, kl = butils.multiclass_nms(bbox, torch.full((5, 128), 0.5, device=DEV), range(128), 0.5, 0.1, 10)
    assert kl.tolist() == list(range(10))                               # one box, 128 tied classes: class order


# ------------------------------------------------------------------ 2. DenseInferHotPath at width
IMGS = [(300.0, 400.0), (277.0, 389.0), (318.0, 350.0)]
RET_GRIDS, RET_STRIDES = [(40, 52), (20, 26), (10, 13)], [8, 16, 32]
RET_SCALES = [4 * 2 ** (i / 3) for i in range(3)]
FC_GRIDS, FC_STRIDES = [(40, 52), (20, 26), (10, 13), (5, 7), (3, 4)], [8, 16, 32, 64, 128]


def _select_retina(cls, reg, anchors, img, pre, min_size, sigmoid):
    """AnchorHead.predict_single_image's per-level selection for one image: key = best class logit (sigmoid) or
    max over c >= 1 of the float64 softmax, top pre (ties to the lowest index), decode + clamp, min-size filter.
    cls[l] [A*C, H, W], reg[l] [4A, H, W], anchors[l] fp32 [4, A*H*W] -> flat rows, boxes fp32 [k, 4]."""
    rows, boxes, off = [], [], 0
    for c_l, r_l, a_l in zip(cls, reg, anchors):
        n = a_l.shape[1]
        x = c_l.reshape(-1, n)
        if sigmoid:
            key = x.max(0)                                       # fp32 values: no rounding
        else:
            key = _softmax64(x, 0)[1:].max(0)
        k = min(pre, n) if pre > 0 else n
        _topk_margin(key, k, "level key")
        idx = oracle.topk_desc(key.astype(np.float32), k) if k < n else np.arange(n)
        d = np.ascontiguousarray(r_l.reshape(4, -1)[:, idx])
        bx = oracle.param2bbox(np.ascontiguousarray(a_l[:, idx]), d, img_size=img)
        if min_size > 0:
            w, h = (bx[2] - bx[0]) + np.float32(1), (bx[3] - bx[1]) + np.float32(1)
            _margin(np.concatenate([w, h]), min_size, 1e-5, "box size vs min_bbox_size")
            ok = (w >= np.float32(min_size)) & (h >= np.float32(min_size))
            idx, bx = idx[ok], bx[:, ok]
        rows.append(idx + off)
        boxes.append(bx.T)
        off += n
    return np.concatenate(rows), np.concatenate(boxes).astype(np.float32)


def _retina_detect_reference(cls, rows, boxes, cfg, C, sigmoid):
    """multiclass_nms of the selected rows: boxes are the selection's (the GPU's, once they matched the reference's,
    so that the NMS margins need only cover the IoU arithmetic)."""
    x = np.concatenate([c.reshape(C, -1) for c in cls], 1)[:, rows].T.astype(np.float64)      # [k, C]
    prob = _sigmoid64(x) if sigmoid else _softmax64(x, 1)
    chans = range(0, C) if sigmoid else range(1, C)
    return _ref_detect(boxes, prob, chans, cfg["min_score"], cfg["nms_type"], cfg["nms_iou"], cfg["max_per_img"],
                       label_add=1 if sigmoid else 0, eps_iou=EPS_IOU_SAME)


def _retina_inputs(C, seed, B, grids, mean, bg=0.0):
    rng = np.random.default_rng(seed)
    cls = []
    for g in grids:
        x = rng.normal(mean, 1.5, (B, C, 9) + g)
        x[:, 0] += bg
        cls.append(_q(x).reshape(B, 9 * C, *g))                  # channel c * A + a: class-major, as view(C, -1) reads it
    reg = [(0.3 * rng.standard_normal((B, 36) + g)).astype(np.float32) for g in grids]
    return cls, reg


def _run_retina(C_ch, sigmoid, cfg, seed, grids=RET_GRIDS, strides=RET_STRIDES, imgs=IMGS, mean=-6.0, bg=0.0,
                min_dets=20):
    B = len(imgs)
    cls, reg = _retina_inputs(C_ch, seed, B, grids, mean, bg)
    anchors = [oracle.anchor_grid(s, g, scales=RET_SCALES).reshape(4, -1) for s, g in zip(strides, grids)]
    sels = [_select_retina([c[b] for c in cls], [r[b] for r in reg], anchors, (int(imgs[b][0]), int(imgs[b][1])),
                           cfg["pre_nms"], cfg.get("min_bbox_size", 0), sigmoid) for b in range(B)]
    hp = fused.DenseInferHotPath(B, grids, DEV, head="retina", num_classes=C_ch + 1 if sigmoid else C_ch, test_cfg=cfg,
                                 strides=strides, use_sigmoid=sigmoid, anchor_scales=RET_SCALES)
    rec = torch.full((B, hp.M, 6), -7.0, device=DEV)
    out = hp.step([T(c) for c in cls], [T(r) for r in reg], torch.tensor(imgs, device=DEV), records=rec)
    hp.check()
    for b, (rows, boxes) in enumerate(sels):
        n = int(out["sel_count"][b])
        assert n == rows.size, (b, n, rows.size)
        assert np.array_equal(N(out["sel_rows"][b, :n]), rows), b
        got = N(out["sel_boxes"][b, :, :n]).T.copy()
        np.testing.assert_allclose(got, boxes, rtol=0, atol=1e-3)
        db, ds, dl, _ = _retina_detect_reference([c[b] for c in cls], rows, got, cfg, C_ch, sigmoid)
        assert _assert_dets(out, b, db, ds, dl, rec) >= min_dets, b


RET_CFG = dict(pre_nms=300, min_bbox_size=0, min_score=0.05, nms_iou=0.5, max_per_img=100)


@pytest.mark.parametrize("mode", ["official", "strict"])
@pytest.mark.parametrize("C_ch", [80, 128, 79])
def test_dense_retinanet_sigmoid_wide_vs_reference(C_ch, mode):
    """RetinaNet sigmoid heads with 80 and 128 class channels (score mode 2 through k_class_max), and 79 channels,
    whose channel loop leaves a tail of two (classes 77, 78) after the four-wide steps from class 1."""
    _run_retina(C_ch, True, dict(RET_CFG, nms_type=mode), seed={80: 2, 128: 128, 79: 8}[C_ch])


@pytest.mark.parametrize("mode", ["official", "strict"])
def test_dense_retinanet_softmax_81_vs_reference(mode):
    """Softmax anchor head with 81 channels: the selection key is max over c >= 1 of the softmax (score mode 3,
    load_logit), the detection scores the softmax over all 81."""
    cfg = dict(pre_nms=100, min_bbox_size=12, min_score=0.05, nms_iou=0.5, max_per_img=100, nms_type=mode)
    _run_retina(81, False, cfg, seed=81, mean=0.0, bg=1.0, min_dets=10)


def test_dense_retinanet_config4_80_classes():
    """DESIGN's config 4: 800x1333 image on the 800x1344 pyramid, strides 8..128, 9 anchors x 80 classes, B = 2."""
    strides = [8, 16, 32, 64, 128]
    grids = [(-(-800 // s), -(-1344 // s)) for s in strides]
    for mode in ("official", "strict"):
        cfg = dict(pre_nms=1000, min_bbox_size=0, min_score=0.05, nms_iou=0.5, max_per_img=100, nms_type=mode)
        _run_retina(80, True, cfg, seed=4, grids=grids, strides=strides, imgs=[(800.0, 1333.0)] * 2)


def _fcos_inputs(C, seed, B):
    rng = np.random.default_rng(seed)
    cls = [_q(rng.normal(-6, 1.5, (B, C) + g)) for g in FC_GRIDS]
    reg = [np.abs(0.05 + 0.05 * rng.standard_normal((B, 4) + g)).astype(np.float32) for g in FC_GRIDS]
    ctr = [rng.choice(np.array([-1.0, 0.0, 0.5, 2.0], np.float32), (B, 1) + g) for g in FC_GRIDS]
    return cls, reg, ctr


def _fcos_select(cls, reg, ctr, img, cfg, C):
    """FCOSHead.predict_single_image's selection for one image: ltrb decode + clamp (fp32, the reference's order),
    strict min-size test, key max_c sigmoid(cls) [* sigmoid(ctr)] in float64, per level the top pre_nms valid points
    (ties to the lowest index) or all valid points in index order -> flat rows, boxes fp32 [k, 4]."""
    f32 = np.float32
    std, mean, min_size = f32(300.0), f32(0.0), f32(cfg.get("min_bbox_size", 0))
    my, mx = f32(img[0]) - f32(1), f32(img[1]) - f32(1)
    rows, boxes, off = [], [], 0
    for (H, W), s, c_l, r_l, t_l in zip(FC_GRIDS, FC_STRIDES, cls, reg, ctr):
        s = f32(s)
        px = np.tile(np.arange(W, dtype=f32) * s + s / f32(2.0), H)
        py = np.repeat(np.arange(H, dtype=f32) * s + s / f32(2.0), W)
        l_, t_, r_, b_ = [(r_l[k].reshape(-1) * std + mean).astype(f32) for k in range(4)]
        x1, y1 = np.minimum(np.maximum(px - l_, f32(0)), mx), np.minimum(np.maximum(py - t_, f32(0)), my)
        x2, y2 = np.minimum(np.maximum(r_ + px, f32(0)), mx), np.minimum(np.maximum(b_ + py, f32(0)), my)
        w, h = (x2 - x1) + f32(1), (y2 - y1) + f32(1)
        if min_size > 0:
            _margin(np.concatenate([w, h]), float(min_size), 1e-5, "box size vs min_bbox_size")
        ok = (w > min_size) & (h > min_size)
        key = _sigmoid64(c_l.reshape(C, -1).max(0))
        if t_l is not None:
            key = key * _sigmoid64(t_l.reshape(-1))
        key = np.where(ok, key, -np.inf)
        valid = np.nonzero(ok)[0]
        pre = cfg["pre_nms"]
        if 0 < pre < valid.size:
            _topk_margin(key, pre, "level key")
            idx = oracle.topk_desc(key.astype(np.float32), pre)
        else:
            idx = valid
        rows.append(idx + off)
        boxes.append(np.stack([x1, y1, x2, y2], 1)[idx])
        off += H * W
    return np.concatenate(rows), np.concatenate(boxes).astype(np.float32)


def _fcos_detect_reference(cls, ctr, rows, boxes, cfg, C):
    """multiclass_nms over all C channels of the selected points, the centerness as score factor."""
    x = np.concatenate([c.reshape(C, -1) for c in cls], 1)[:, rows].T
    fac = _sigmoid64(np.concatenate([t.reshape(-1) for t in ctr])[rows]) if ctr[0] is not None else None
    return _ref_detect(boxes, _sigmoid64(x), range(C), cfg["min_score"], cfg["nms_type"], cfg["nms_iou"],
                       cfg["max_per_img"], factor=fac, label_add=1, eps_iou=EPS_IOU_SAME)


@pytest.mark.parametrize("centerness", [True, False])
@pytest.mark.parametrize("mode", ["official", "strict"])
def test_dense_fcos_80_classes_vs_reference(centerness, mode):
    C, B = 80, 3
    cls, reg, ctr = _fcos_inputs(C, 80 + 2 * centerness, B)
    cfg = dict(pre_nms=300, min_bbox_size=8, min_score=0.05, nms_iou=0.5, max_per_img=80, nms_type=mode)
    ctr_b = [[c[b] for c in ctr] if centerness else [None] * 5 for b in range(B)]
    sels = [_fcos_select([c[b] for c in cls], [r[b] for r in reg], ctr_b[b], IMGS[b], cfg, C) for b in range(B)]
    hp = fused.DenseInferHotPath(B, FC_GRIDS, DEV, head="fcos", num_classes=C + 1, test_cfg=cfg, strides=FC_STRIDES,
                                 reg_mean=0.0, reg_std=300.0, use_centerness=centerness)
    rec = torch.full((B, hp.M, 6), -7.0, device=DEV)
    out = hp.step([T(c) for c in cls], [T(r) for r in reg], torch.tensor(IMGS, device=DEV),
                  ctr_outs=[T(c) for c in ctr] if centerness else None, records=rec)
    hp.check()
    for b, (rows, boxes) in enumerate(sels):
        n = int(out["sel_count"][b])
        assert n == rows.size, (b, n, rows.size)
        assert np.array_equal(N(out["sel_rows"][b, :n]), rows), b
        got = N(out["sel_boxes"][b, :, :n]).T.copy()
        np.testing.assert_allclose(got, boxes, rtol=0, atol=1e-3)
        db, ds, dl, _ = _fcos_detect_reference([c[b] for c in cls], ctr_b[b], rows, got, cfg, C)
        assert _assert_dets(out, b, db, ds, dl, rec) >= 20, b


def test_dense_class_limit():
    cfg = dict(pre_nms=100, min_bbox_size=0, min_score=0.05, nms_iou=0.5, max_per_img=100, nms_type="official")
    with pytest.raises(_C.B200DetError, match="128 class channels"):
        fused.DenseInferHotPath(1, RET_GRIDS, DEV, head="retina", num_classes=130, test_cfg=cfg, strides=RET_STRIDES)
    hp = fused.DenseInferHotPath(1, RET_GRIDS, DEV, head="retina", num_classes=129, test_cfg=cfg, strides=RET_STRIDES)
    assert hp.C == 128


# ------------------------------------------------------------------ 3. RCNN test path
STDS = ((0.1, 0.1, 0.2, 0.2), (0.05, 0.05, 0.1, 0.1), (0.033, 0.033, 0.067, 0.067))
IMG = (800, 1333)


class Head(torch.nn.Module):
    """Deterministic stand-in for a stage's RCNN head: 7x7 mean-pool, then seeded fc layers written as products and sums
    (no cuBLAS algorithm choice)."""

    def __init__(self, C, NC, reg_c, seed, scale=6.0):
        super().__init__()
        g = torch.Generator().manual_seed(seed)
        self.wc = (torch.randn((NC, C), generator=g) * scale).to(DEV)
        self.wr = (torch.randn((4 * reg_c, C), generator=g) * 0.5).to(DEV)
        self.bias = torch.zeros(NC, device=DEV)
        self.bias[0] = 1.0

    def forward(self, x):
        p = x.mean((2, 3))
        return (p[:, None, :] * self.wc[None]).sum(-1) + self.bias, (p[:, None, :] * self.wr[None]).sum(-1)


def _rcnn_reference(boxes, cls_out, reg_out, stds, img, cfg):
    """BBoxHead.predict_bboxes_single_image: float64 softmax, per-class param2bbox + clamp, multiclass_nms over 1..C-1."""
    n, C = cls_out.shape
    reg_c = reg_out.shape[1] // 4
    param = np.ascontiguousarray(reg_out.T).reshape(4, reg_c, n)
    per = np.stack([oracle.param2bbox(np.ascontiguousarray(boxes), np.ascontiguousarray(param[:, c]), [0.0] * 4, list(stds),
                                      img) for c in range(reg_c)], 2)                      # [4, n, reg_c]
    bx = per.transpose(1, 0, 2)
    bx = np.repeat(bx, C, 2) if reg_c == 1 else bx
    return _ref_detect(bx, _softmax64(cls_out, 1), range(1, C), cfg["min_score"], cfg.get("nms_type", "official"),
                       cfg["nms_iou"], cfg["max_per_img"])


def _refine_reference(boxes, cls_out, reg_out, stds, img):
    n = boxes.shape[1]
    label = np.argmax(cls_out, 1)
    reg_c = reg_out.shape[1] // 4
    d = reg_out.reshape(n, 4, reg_c)[np.arange(n), :, label if reg_c > 1 else 0].T
    return oracle.param2bbox(np.ascontiguousarray(boxes), np.ascontiguousarray(d), [0.0] * 4, list(stds), img)


@pytest.mark.parametrize("stages,agnostic", [(1, False), (3, False), (3, True)])
def test_infer_hot_path_81_classes_vs_reference(stages, agnostic):
    """faster_rcnn (1 stage) and the cascade (3 stages, arg-max refine over 81 logits), per-class and class-agnostic
    regression, B = 2 at config-2 geometry; each stage checked from the GPU's own stage inputs."""
    B, C, NC = 2, 16, 81
    w = workload.config2(B=B, K=1, seed=17 + stages, channels=C, img_shape=IMG, pad_shape=(800, 1344))
    feats = [T(f).contiguous(memory_format=torch.channels_last) for f in w["feats"]]
    img_hw = torch.tensor([[float(IMG[0]), float(IMG[1])]] * B, device=DEV)
    rcnn = dict(min_score=0.05, nms_iou=0.5, max_per_img=100, nms_type="official")
    hp = fused.InferHotPath(B, w["grids"], DEV, feat_channels=C, num_classes=NC, num_stages=stages,
                            reg_class_agnostic=agnostic, rcnn_test=rcnn)
    heads = [Head(C, NC, 1 if agnostic else NC, seed=30 + s) for s in range(stages)]
    rec = torch.full((B, hp.M, 6), -7.0, device=DEV)
    out = hp.step([T(c) for c in w["cls"]], [T(r) for r in w["reg"]], feats, img_hw, heads, records=rec)
    hp.check()
    P = hp.P
    for s in range(stages - 1):
        cur, nxt = out["stages"][s], out["stages"][s + 1]
        for b in range(B):
            n = int(cur["count"][b])
            assert int(nxt["count"][b]) == n
            ref = _refine_reference(N(cur["boxes"][b, :, :n]), N(cur["cls_out"][b * P:b * P + n]),
                                    N(cur["reg_out"][b * P:b * P + n]), STDS[s], IMG)
            np.testing.assert_allclose(N(nxt["boxes"][b, :, :n]), ref, rtol=1e-5, atol=1e-3)
    last, total = out["stages"][-1], 0
    for b in range(B):
        n = int(last["count"][b])
        db, ds, dl, _ = _rcnn_reference(N(last["boxes"][b, :, :n]), N(last["cls_out"][b * P:b * P + n]),
                                        N(last["reg_out"][b * P:b * P + n]), STDS[stages - 1], IMG, rcnn)
        total += _assert_dets(out, b, db, ds, dl, rec)
    assert total > 20


def test_infer_hot_path_class_limit():
    w = workload.config2(B=1, K=1, channels=8, img_shape=(160, 213), pad_shape=(160, 224))
    with pytest.raises(_C.B200DetError, match="128 classes"):
        fused.InferHotPath(1, w["grids"], DEV, feat_channels=8, num_classes=129)
    hp = fused.InferHotPath(1, w["grids"], DEV, feat_channels=8, num_classes=128)
    assert hp.NC == 128


def _rcnn_detect_case(B, n, C, seed):
    rng = np.random.default_rng(seed)
    cx, cy = rng.uniform(0, 560, (B, n)), rng.uniform(0, 380, (B, n))
    w, h = rng.uniform(16, 120, (B, n)), rng.uniform(16, 120, (B, n))
    props = np.stack([cx - w / 2, cy - h / 2, cx + w / 2, cy + h / 2], 1).astype(np.float32)        # [B, 4, n]
    logit = _q(rng.normal(0, 1, (B, n, C)))
    ties = []
    for b in range(B):
        for t, r in enumerate(rng.choice(n, 32, replace=False)):
            c0 = t                                               # lanes 0..31: every lane position of the first group
            logit[b, r, _tie_classes(c0, C)] = 4.0 + (t % 8) / 8.0
            ties.append((b, r, c0))
    reg = (0.3 * rng.standard_normal((B, n, 4 * C))).astype(np.float32)
    return props, logit, reg, ties


@pytest.mark.parametrize("mode", ["strict", "official"])
def test_rcnn_detect_128_classes_cross_group_ties(mode):
    """b2d_rcnn_detect at C = 128: rows whose maximum is tied at classes c, c+32, c+64, c+96 (c = 0 included: the
    background wins strict mode there).  Strict keeps the first tied class; official keeps the tied classes of a row in
    ascending class order."""
    B, n, C = 2, 300, 128
    props, logit, reg, ties = _rcnn_detect_case(B, n, C, seed=128)
    img = (400, 600)
    cfg = dict(min_score=0.05, nms_iou=0.5, max_per_img=100, nms_type=mode)
    stds = STDS[0]
    b_, s_, l_, cnt, ovf = bheads.rcnn_detect(T(props), T(logit), T(reg), img, [0.0] * 4, list(stds), **cfg)
    torch.cuda.synchronize()
    assert int(ovf[0]) == 0
    out = dict(boxes=b_, scores=s_, labels=l_, count=cnt)
    for b in range(B):
        db, ds, dl, (ii, cc) = _rcnn_reference(props[b], logit[b], reg[b], stds, img, cfg)
        _assert_dets(out, b, db, ds, dl)
        tied = [(r, c0) for (bb, r, c0) in ties if bb == b]
        for r, c0 in tied:
            got = cc[ii == r]
            if mode == "strict":
                assert got.tolist() == ([] if c0 == 0 else [c0]), (r, c0, got)
            else:
                grp = [c for c in _tie_classes(c0, C) if c >= 1]
                assert set(grp) <= set(got.tolist()), (r, c0, got)
        assert int(cnt[b]) >= 20


def test_refine_argmax_128_logits_takes_the_first_maximum():
    """b2d_refine_bboxes_argmax over 128 logits: maxima tied at 0/32/64/96 and at 5/69 give the first index, as
    torch.argmax; random rows give np.argmax."""
    B, ld, NC = 2, 64, 128
    rng = np.random.default_rng(5)
    cls = _q(rng.normal(0, 1, (B, ld, NC)))
    crafted = [([0, 32, 64, 96], 0), ([5, 69], 5), ([31, 63, 95, 127], 31), ([64, 96], 64), ([100, 127], 100),
               ([1, 33, 65, 97], 1)]
    for k, (idx, first) in enumerate(crafted):
        cls[:, k, idx] = 5.0
    counts = np.array([ld, 50], np.int32)
    cls[1, 50:] = np.nan                                         # past the count: never read
    props = np.tile(np.array([[10.0], [20.0], [110.0], [220.0]], np.float32), (B, 1, ld))
    reg = np.zeros((B, ld, 4, NC), np.float32)
    reg[:, :, 0, :] = 0.05 * np.arange(NC, dtype=np.float32)    # dx grows with the class: the refined x1 names the label
    reg = reg.reshape(B, ld, 4 * NC)
    out = torch.full((B, 4, ld), -7.0, device=DEV)
    cnt = torch.full((B,), -1, dtype=torch.int32, device=DEV)
    img_hw = torch.tensor([[400.0, 600.0]] * B, device=DEV)
    stds = _C.host_f4(STDS[0], [1, 1, 1, 1])
    d_props, d_counts, d_cls, d_reg = T(props), T(counts), T(cls), T(reg)
    _C.call("b2d_refine_bboxes_argmax", _C.ptr(out), _C.ptr(cnt), _C.ptr(d_props), ld, _C.ptr(d_counts), ld, _C.ptr(d_cls), NC,
            _C.ptr(d_reg), NC, _C.host_f4(None, [0, 0, 0, 0]), stds, _C.ptr(img_hw), B, _C.stream())
    torch.cuda.synchronize()
    assert np.array_equal(N(cnt), counts)
    for b in range(B):
        n = int(counts[b])
        lab = np.argmax(cls[b, :n], 1)
        assert lab[:len(crafted)].tolist() == [first for _, first in crafted]
        ref = _refine_reference(props[b, :, :n], cls[b, :n], reg[b, :n], STDS[0], (400, 600))
        np.testing.assert_allclose(N(out[b, :, :n]), ref, rtol=1e-5, atol=1e-3)
        assert (N(out[b, :, n:]) == -7.0).all()


# ------------------------------------------------------------------ 4. losses at width
def test_anchor_head_loss_80_classes_vs_oracle():
    """Focal + smooth-L1 sums and both gradients at 80 classes (RetinaNet on COCO), on a 400x672 pyramid."""
    rng = np.random.default_rng(80)
    strides = [8, 16, 32, 64, 128]
    grids = [(-(-400 // s), -(-672 // s)) for s in strides]
    scales = [4.0, 4.0 * 2 ** (1 / 3), 4.0 * 2 ** (2 / 3)]
    pyr = fused.AnchorPyramid(strides, grids, scales=scales)
    B, K, C, A = 2, 10, 80, 9
    gt = np.zeros((B, 4, K), np.float32)
    for b in range(B):
        x1 = rng.uniform(0, 500, K); y1 = rng.uniform(0, 300, K)
        gt[b] = np.stack([x1, y1, np.minimum(x1 + rng.uniform(20, 250, K), 671), np.minimum(y1 + rng.uniform(20, 160, K), 399)])
    gl = rng.integers(1, C + 1, (B, K)).astype(np.int64)
    gl[0, :4] = [64, 65, 80, 33]                                 # labels in the upper lane groups
    cls_np = [rng.normal(-2, 1.5, (B, A * C) + g).astype(np.float32) for g in grids]
    reg_np = [rng.normal(0, 0.4, (B, A * 4) + g).astype(np.float32) for g in grids]
    anc = np.concatenate([oracle.anchor_grid(s, gr, scales=scales).reshape(4, -1) for s, gr in zip(strides, grids)], 1)
    labs = np.stack([oracle.assign_max_iou(anc, gt[b], 0.5, 0.4, 0.0)[0] for b in range(B)])
    cls = [T(c).requires_grad_(True) for c in cls_np]
    reg = [T(r).requires_grad_(True) for r in reg_np]
    closs, rloss = bheads.anchor_head_calc_loss(cls, reg, T(labs), pyr, T(gt), T(gl), beta=1.0 / 9.0)
    (closs + rloss).backward()
    f = s1 = 0.0
    npos, dcs, drs = 0, [], []
    for b in range(B):
        fb, sb, nb, dc, dr = oracle.anchor_head_loss([c[b] for c in cls_np], [r[b] for r in reg_np], labs[b], anc, gt[b], gl[b])
        f += fb; s1 += sb; npos += nb; dcs.append(dc); drs.append(dr)
    assert npos > 50
    np.testing.assert_allclose(float(closs.detach()), f / npos, rtol=1e-5)
    np.testing.assert_allclose(float(rloss.detach()), s1 / npos, rtol=1e-5)
    for l in range(5):
        np.testing.assert_allclose(N(cls[l].grad), np.stack([dcs[b][l] for b in range(B)]) / npos, rtol=1e-4, atol=1e-7)
        np.testing.assert_allclose(N(reg[l].grad), np.stack([drs[b][l] for b in range(B)]) / npos, rtol=1e-4, atol=1e-7)


@pytest.mark.parametrize("use_sigmoid,C", [(False, 81), (True, 80), (False, 128), (True, 128)])
@pytest.mark.parametrize("layout", ["rows", "transposed"])
def test_sampled_cross_entropy_wide_vs_float64(use_sigmoid, C, layout):
    """sampled_cross_entropy at 80..128 classes against float64 torch on the CPU, forward and gradient."""
    import torch.nn.functional as F
    rng = np.random.default_rng(C + use_sigmoid)
    n = 777
    x = rng.normal(0, 2, (n, C)).astype(np.float32)
    lab = rng.integers(0, C + 1 if use_sigmoid else C, n).astype(np.int64)
    lab[:8] = np.minimum([C - 1, 63, 64, 65, 96, 127, 0, C], C if use_sigmoid else C - 1)     # both lane-group edges
    base = T(x) if layout == "rows" else T(np.ascontiguousarray(x.T))
    base.requires_grad_(True)
    pred = base if layout == "rows" else base.t()
    loss = bheads.sampled_cross_entropy(pred, T(lab), use_sigmoid, 0.5)
    loss.backward()
    ref_in = torch.from_numpy(x.astype(np.float64)).requires_grad_(True)
    tl = torch.from_numpy(lab)
    if use_sigmoid:
        ref = F.binary_cross_entropy_with_logits(ref_in, F.one_hot(tl, C + 1)[:, 1:].double(), reduction="none").sum() * 0.5
    else:
        ref = F.cross_entropy(ref_in, tl, reduction="none").sum() * 0.5
    ref.backward()
    np.testing.assert_allclose(float(loss), float(ref), rtol=1e-5)
    got = N(base.grad) if layout == "rows" else N(base.grad).T
    np.testing.assert_allclose(got, ref_in.grad.numpy(), rtol=1e-4, atol=1e-6)
