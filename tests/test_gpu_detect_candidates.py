"""Detection past 16384 candidates per image: b2d_rcnn_detect / b2d_dense_detect with cap > 16384 and the
max_candidates option of fused.InferHotPath / DenseInferHotPath.

With cap > 16384 the NMS runs on the 16384 best candidates of every image (round 0) and, for an image that keeps fewer
than max_per_img there, continues greedily over the rest in blocks (the continuation).  The result must be that of one
greedy NMS over every candidate.

The references here compare exactly, not within margins: scores are values both sides compute bit-equal (given fp32
values, 0.5 = sigmoid(0), 0 = sigmoid(-200), 1/k from k tied maxima of a softmax) and boxes are decoded with zero
size deltas and 1/8-grid centre deltas on integer proposals, so every IoU decision is taken on identical fp32 boxes.
The reference NMS runs oracle.nms per class on the class-offset boxes of lib/utils.py:211-221 (offsets keep the
classes apart, so this is batched_nms) and merges the survivors by score, then candidate index."""
import ctypes

import numpy as np
import pytest
import torch

import oracle

pytestmark = [pytest.mark.gpu, pytest.mark.skipif(not torch.cuda.is_available(), reason="needs a CUDA device")]

if torch.cuda.is_available():
    import b200det
    from b200det import _C, fused, workload
    DEV = torch.device("cuda:0")

BIG = 1 << 17                      # a cap above 16384 for the library-level calls
THR = 0.5


def T(a):
    return torch.from_numpy(np.ascontiguousarray(a)).to(DEV)


def N(t):
    return t.detach().cpu().numpy()


# ------------------------------------------------------------------ references
def _batched_ref(cb, cs, cc, M, thr=THR):
    """batched_nms (class-offset boxes, fp32) -> the first M kept candidate indices, score order, ties by index."""
    if cs.size == 0:
        return np.zeros(0, np.int64)
    cb = np.ascontiguousarray(cb, np.float32)
    mx = np.float32(cb.max())
    off = (cc.astype(np.int64).astype(np.float32) * mx).astype(np.float32)
    nb = (cb + off[:, None]).astype(np.float32)
    keep = []
    for c in np.unique(cc):
        idx = np.nonzero(cc == c)[0]
        keep.append(idx[oracle.nms(np.ascontiguousarray(nb[idx]), np.ascontiguousarray(cs[idx]), thr)])
    keep = np.concatenate(keep)
    keep = keep[np.lexsort((keep, -cs[keep].astype(np.float64)))]
    return keep[:M]


def _dense_ref(boxes_4n, score_cn, n, min_score, M, strict=False, factor=None):
    """utils.multiclass_nms on given fp32 scores [C][n] and boxes [4][n], every channel an NMS channel."""
    s = score_cn[:, :n].T                                                   # [n, C]
    if strict:
        cc = s.argmax(1)
        ii = np.nonzero(s[np.arange(n), cc] >= np.float32(min_score))[0]
        cc = cc[ii]
    else:
        ii, cc = np.nonzero(s >= np.float32(min_score))
    cs = s[ii, cc].astype(np.float32)
    if factor is not None:
        cs = (cs * factor[ii]).astype(np.float32)
    cb = boxes_4n[:, ii].T
    k = _batched_ref(cb, cs, cc, M)
    return cb[k], cs[k], cc[k], ii.size


def _assert_same(out, b, box, score, label):
    k = int(out["count"][b])
    assert k == score.shape[0], (b, k, score.shape[0])
    assert np.array_equal(N(out["labels"][b, :k]), label), b
    np.testing.assert_allclose(N(out["scores"][b, :k]), score, rtol=1e-5, atol=0)
    np.testing.assert_allclose(N(out["boxes"][b, :, :k]), box.T, rtol=0, atol=1e-5)
    return k


# ------------------------------------------------------------------ library calls
def _outs(B, M):
    return dict(boxes=torch.zeros((B, 4, M), device=DEV), scores=torch.zeros((B, M), device=DEV),
                labels=torch.zeros((B, M), dtype=torch.int64, device=DEV), count=torch.zeros(B, dtype=torch.int32, device=DEV),
                records=torch.full((B, M, 6), -7.0, device=DEV), overflow=torch.full((1,), 5, dtype=torch.int32, device=DEV))


def _rounds(ws, cap, B):
    r = torch.full((B,), -1, dtype=torch.int32, device=DEV)
    _C.call("b2d_detect_continuation_rounds", _C.ptr(r), _C.ptr(ws), cap, B, _C.stream())
    return N(r)


def dense_detect(boxes, score, counts, min_score, M, cap, strict=False, factor=None, transform=0):
    """b2d_dense_detect_records on one level: boxes fp32 [B][4][ld], class values [B][C][ld] (rows = 0..count-1)."""
    B, C, ld = score.shape
    bx, sc, cnt = T(boxes), T(score), T(np.asarray(counts, np.int32))
    rows = T(np.tile(np.arange(ld, dtype=np.int32), (B, 1)))
    fac = T(factor) if factor is not None else None
    lv = _C.DenseLevels()
    lv.num_levels = 1
    lv.offset[0], lv.img_stride[0], lv.class_stride[0], lv.base[0] = 0, C * ld, ld, sc.data_ptr()
    mask = [0, 0]
    for c in range(C):
        mask[c >> 6] |= 1 << (c & 63)
    ws = torch.empty(_C.lib().b2d_rcnn_detect_workspace_bytes(cap, B), dtype=torch.uint8, device=DEV)
    o = _outs(B, M)
    _C.call("b2d_dense_detect_records", _C.ptr(o["boxes"]), _C.ptr(o["scores"]), _C.ptr(o["labels"]), _C.ptr(o["count"]),
            _C.ptr(o["records"]), _C.ptr(bx), ld, _C.ptr(cnt), _C.ptr(rows), ctypes.byref(lv), C, transform, _C.ptr(fac),
            ld if fac is not None else 0, (_C.c_ull * 2)(*mask), float(np.float32(min_score)), 0, _C.floor_f32(THR), M,
            int(strict), cap, B, _C.ptr(o["overflow"]), _C.ptr(ws), ws.numel(), None, _C.stream())
    torch.cuda.synchronize()
    o["rounds"] = _rounds(ws, cap, B) if cap > 16384 else None
    return o


def rcnn_detect(props, logits, reg, img, min_score, M, cap, strict=False, stds=(1.0, 1.0, 1.0, 1.0)):
    """b2d_rcnn_detect_records: props [B][4][n], logits [B][n][C], reg [B][n][4 * reg_c]."""
    B, n, C = logits.shape
    reg_c = reg.shape[2] // 4
    ws = torch.empty(_C.lib().b2d_rcnn_detect_workspace_bytes(cap, B), dtype=torch.uint8, device=DEV)
    o = _outs(B, M)
    img_hw = T(np.array([img] * B, np.float32))
    pr, lg, rg = T(props), T(logits), T(reg)                     # held until the call has run
    _C.call("b2d_rcnn_detect_records", _C.ptr(o["boxes"]), _C.ptr(o["scores"]), _C.ptr(o["labels"]), _C.ptr(o["count"]),
            _C.ptr(o["records"]), _C.ptr(pr), n, None, n, _C.ptr(lg), _C.ptr(rg), C, reg_c,
            _C.host_f4(None, [0, 0, 0, 0]), _C.host_f4(stds, [1, 1, 1, 1]), _C.ptr(img_hw), float(np.float32(min_score)),
            _C.floor_f32(THR), M, int(strict), cap, B, _C.ptr(o["overflow"]), _C.ptr(ws), ws.numel(), _C.stream())
    torch.cuda.synchronize()
    return o


def _bitwise(a, b):
    for k in ("boxes", "scores", "labels", "count", "records", "overflow"):
        assert torch.equal(a[k], b[k]), k


# ------------------------------------------------------------------ 1. same result where both caps apply
def _random_dense(B, C, ld, seed):
    rng = np.random.default_rng(seed)
    cx, cy = rng.uniform(0, 600, (B, ld)), rng.uniform(0, 400, (B, ld))
    w, h = rng.uniform(8, 90, (B, ld)), rng.uniform(8, 90, (B, ld))
    boxes = np.stack([cx - w / 2, cy - h / 2, cx + w / 2, cy + h / 2], 1).astype(np.float32)
    score = rng.uniform(0, 1, (B, C, ld)).astype(np.float32) ** 3
    return boxes, score


@pytest.mark.parametrize("strict", [False, True])
@pytest.mark.parametrize("use_factor", [False, True])
def test_dense_big_cap_matches_default_cap(strict, use_factor):
    B, C, ld = 3, 80, 3000
    boxes, score = _random_dense(B, C, ld, seed=11 + strict + 2 * use_factor)
    counts = [3000, 1700, 0]
    fac = np.random.default_rng(4).uniform(0.2, 1, (B, ld)).astype(np.float32) if use_factor else None
    ms = 0.9 if not strict else 0.05                            # official: ~3.5 % of 240 000 values, under 16384 per image
    a = dense_detect(boxes, score, counts, ms, 100, 16384, strict, fac)
    b = dense_detect(boxes, score, counts, ms, 100, BIG, strict, fac)
    assert int(a["overflow"][0]) == 0 and int(a["count"].sum()) > 100
    _bitwise(a, b)
    assert (b["rounds"] == 0).all()


@pytest.mark.parametrize("strict", [False, True])
@pytest.mark.parametrize("agnostic", [False, True])
def test_rcnn_big_cap_matches_default_cap(strict, agnostic):
    B, n, C = 2, 1000, 81
    rng = np.random.default_rng(21 + strict + 2 * agnostic)
    props = _int_props(rng, B, n)
    logits = rng.normal(0, 2.5, (B, n, C)).astype(np.float32)
    logits[:, :, 0] += 2.0
    reg = (0.3 * rng.standard_normal((B, n, 4 * (1 if agnostic else C)))).astype(np.float32)
    stds = (0.1, 0.1, 0.2, 0.2)
    a = rcnn_detect(props, logits, reg, (800, 1333), 0.05, 100, 16384, strict, stds)
    b = rcnn_detect(props, logits, reg, (800, 1333), 0.05, 100, 30000, strict, stds)
    assert int(a["overflow"][0]) == 0 and int(a["count"].sum()) > 100
    _bitwise(a, b)


# ------------------------------------------------------------------ 2. beyond the old cap
def _int_props(rng, B, n, W=1300, H=790):
    x1, y1 = rng.integers(0, W - 200, (B, n)), rng.integers(0, H - 200, (B, n))
    w, h = rng.integers(8, 200, (B, n)), rng.integers(8, 200, (B, n))
    return np.stack([x1, y1, x1 + w, y1 + h], 1).astype(np.float32)


def _rcnn_exact_case(B, n, C, reg_c, seed):
    """Softmax scores 1/k: every row has k tied maxima (logit 0) among the classes, the rest at -200 (exp underflows to 0
    on both sides).  Size deltas 0 and centre deltas on a 1/8 grid with stds 1: decoded boxes are exact."""
    rng = np.random.default_rng(seed)
    props = _int_props(rng, B, n)
    logits = np.full((B, n, C), -200.0, np.float32)
    for b in range(B):
        k = rng.integers(1, C + 1, n)
        for i in range(n):
            logits[b, i, rng.choice(C, k[i], replace=False)] = 0.0
    reg = np.zeros((B, n, 4 * reg_c), np.float32)
    reg[:, :, :2 * reg_c] = np.round(rng.normal(0, 0.1, (B, n, 2 * reg_c)) * 8) / 8
    return props, logits, reg


def _rcnn_ref(props, logits, reg, img, min_score, M):
    """oracle.rcnn_detect's candidate stage (the C param2bbox + clamp) with the per-class reference NMS."""
    n, C = logits.shape
    e = np.exp(logits - logits.max(1, keepdims=True), dtype=np.float32)
    score = (e / e.sum(1, keepdims=True, dtype=np.float32)).astype(np.float32)
    reg_c = reg.shape[1] // 4
    param = np.ascontiguousarray(reg.T).reshape(4, reg_c, n)
    boxes = np.stack([oracle.param2bbox(props, np.ascontiguousarray(param[:, c, :]), img_size=img) for c in range(reg_c)], 1)
    chosen = score >= np.float32(min_score)
    chosen[:, 0] = False
    ii, cc = np.nonzero(chosen)
    cb = boxes[:, cc if reg_c > 1 else np.zeros_like(cc), ii].T.astype(np.float32)
    cs = score[ii, cc]
    k = _batched_ref(cb, cs, cc, M)
    return cb[k], cs[k], cc[k], ii.size


@pytest.mark.parametrize("min_score", [0.0, 0.001, 0.01])
@pytest.mark.parametrize("agnostic", [False, True])
def test_rcnn_81_classes_beyond_16384_vs_reference(min_score, agnostic):
    B, n, C = 2, 600, 81
    props, logits, reg = _rcnn_exact_case(B, n, C, 1 if agnostic else C, seed=int(1000 * min_score) + agnostic)
    img = (790, 1310)
    out = rcnn_detect(props, logits, reg, img, min_score, 100, BIG)
    assert int(out["overflow"][0]) == 0
    for b in range(B):
        db, ds, dl, ncand = _rcnn_ref(props[b], logits[b], reg[b], img, min_score, 100)
        assert 20000 <= ncand <= 100000, ncand
        assert _assert_same(out, b, db, ds, dl) == 100


@pytest.mark.parametrize("min_score", [0.0, 0.001, 0.01])
@pytest.mark.parametrize("strict", [False, True])
def test_dense_80_classes_beyond_16384_vs_reference(min_score, strict):
    """RetinaNet-like rows: 80 sigmoid channels of logits 0 or -200 (scores exactly 0.5 and 0), and FCOS-like rows: given
    scores with a centerness factor.  20 000 - 100 000 candidates per image."""
    B, C = 2, 80
    rng = np.random.default_rng(7 + strict)
    ld = 1200 if not strict else 30000
    boxes = _int_props(rng, B, ld).astype(np.float32)
    logit = np.where(rng.uniform(0, 1, (B, C, ld)) < 0.25, 0.0, -200.0).astype(np.float32)
    counts = [ld, ld - 100]
    out = dense_detect(boxes, logit, counts, min_score, 100, BIG, strict, transform=1)
    assert int(out["overflow"][0]) == 0
    for b in range(B):
        sc = np.where(logit[b] == 0, np.float32(0.5), np.float32(0.0)).astype(np.float32)
        db, ds, dl, ncand = _dense_ref(boxes[b], sc, counts[b], min_score, 100, strict)
        assert 20000 <= ncand <= 100000, ncand
        _assert_same(out, b, db, ds, dl)
    # given scores (transform 0) with a score factor, FCOS style
    score = (np.round(rng.uniform(0, 1, (B, C, 1200)) ** 2 * 64) / 64).astype(np.float32)
    fac = (np.round(rng.uniform(0.25, 1, (B, 1200)) * 16) / 16).astype(np.float32)
    bx = _int_props(rng, B, 1200)
    out = dense_detect(bx, score, [1200, 1100], min_score, 100, BIG, strict, fac)
    for b, n in enumerate([1200, 1100]):
        db, ds, dl, ncand = _dense_ref(bx[b], score[b], n, min_score, 100, strict, fac[b])
        _assert_same(out, b, db, ds, dl)


# ------------------------------------------------------------------ 3. continuation rounds
def _dups(rng, n, x, y, s=60):
    """n near-duplicates of the box (x, y, x + s, y + s): jitter of at most 1 pixel, IoU > 0.9 with each other."""
    j = rng.integers(0, 2, (4, n))
    return np.stack([x + j[0], y + j[1], x + s + j[2], y + s + j[3]]).astype(np.float32)


def _spread(rng, n, x0=2000, y0=0):
    """n boxes on a grid, none overlapping another."""
    i = np.arange(n)
    x, y = x0 + (i % 200) * 20, y0 + (i // 200) * 20
    return np.stack([x, y, x + 10, y + 10]).astype(np.float32)


def _case(parts, C=2):
    """parts: (boxes [4][m], score, class) in rank order -> boxes [4][n], scores [C][n] (other channels -1)."""
    boxes = np.concatenate([p[0] for p in parts], 1)
    n = boxes.shape[1]
    score = np.full((C, n), -1.0, np.float32)
    o = 0
    for bx, s, c in parts:
        m = bx.shape[1]
        score[c, o:o + m] = s
        o += m
    return boxes, score


def _run_case(images, M, C=2, min_score=0.0):
    ld = max(b.shape[1] for b, _ in images)
    B = len(images)
    boxes = np.zeros((B, 4, ld), np.float32)
    score = np.full((B, C, ld), -1.0, np.float32)
    for b, (bx, sc) in enumerate(images):
        boxes[b, :, :bx.shape[1]] = bx
        score[b, :, :bx.shape[1]] = sc
    counts = [bx.shape[1] for bx, _ in images]
    out = dense_detect(boxes, score, counts, min_score, M, BIG)
    assert int(out["overflow"][0]) == 0
    for b in range(B):
        db, ds, dl, _ = _dense_ref(boxes[b], score[b], counts[b], min_score, M)
        _assert_same(out, b, db, ds, dl)
    return out


def _decreasing(m, hi, lo):
    return np.linspace(hi, lo, m, dtype=np.float32)


def test_continuation_one_round():
    """16 900 near-duplicates on top (one survivor in round 0), 3000 separate boxes behind them."""
    rng = np.random.default_rng(1)
    bx, sc = _case([(_dups(rng, 16900, 100, 100), _decreasing(16900, 0.99, 0.6), 0),
                    (_spread(rng, 3000), _decreasing(3000, 0.5, 0.1), 1)])
    out = _run_case([(bx, sc)], 100)
    assert int(out["count"][0]) == 100 and out["rounds"][0] == 1


def test_continuation_many_rounds():
    """Groups of 700 near-duplicates, each group a block and a half: one or two survivors per round."""
    rng = np.random.default_rng(2)
    parts = [(_dups(rng, 16500, 100, 100), _decreasing(16500, 0.99, 0.9), 0)]
    for g in range(12):
        parts.append((_dups(rng, 700, 300 + 100 * g, 300), _decreasing(700, 0.8 - 0.05 * g, 0.78 - 0.05 * g), g % 2))
    bx, sc = _case(parts)
    out = _run_case([(bx, sc)], 8)
    assert int(out["count"][0]) == 8 and out["rounds"][0] >= 3


def test_continuation_max_per_img_at_block_boundary():
    """The first continuation block is 1023 duplicates of one box and one separate box: max_per_img = 3 is reached on the
    block's last candidate; the candidates behind it stay out."""
    rng = np.random.default_rng(3)
    bx, sc = _case([(_dups(rng, 16400, 100, 100), _decreasing(16400, 0.99, 0.9), 0),
                    (_dups(rng, 1023, 400, 400), _decreasing(1023, 0.8, 0.7), 0),
                    (_spread(rng, 1), np.float32([0.65]), 1),
                    (_spread(rng, 500, 6000), _decreasing(500, 0.6, 0.1), 1)])
    out = _run_case([(bx, sc)], 3)
    assert int(out["count"][0]) == 3 and out["rounds"][0] == 1


def test_continuation_equal_scores_across_the_boundary():
    """Every candidate at score 0.5: round 0 takes the 16384 lowest indices (duplicates of one box), the continuation
    the separate boxes behind them in index order."""
    rng = np.random.default_rng(4)
    n_dup = 16384 + 300
    bx = np.concatenate([_dups(rng, n_dup, 100, 100), _spread(rng, 2000)], 1)
    sc = np.full((2, bx.shape[1]), -1.0, np.float32)
    sc[0] = 0.5
    out = _run_case([(bx, sc)], 100)
    assert int(out["count"][0]) == 100 and out["rounds"][0] == 1
    assert int(N(out["boxes"][0, 0, 0])) in (100, 101)


def test_continuation_mixed_batch():
    """One image within 16384 candidates, one in continuation, one without candidates."""
    rng = np.random.default_rng(5)
    small = _case([(_spread(rng, 5000), _decreasing(5000, 0.9, 0.1), 1)])
    cont = _case([(_dups(rng, 17000, 100, 100), _decreasing(17000, 0.99, 0.6), 0),
                  (_spread(rng, 800), _decreasing(800, 0.5, 0.1), 1)])
    empty = (np.zeros((4, 10), np.float32), np.full((2, 10), -1.0, np.float32))
    out = _run_case([small, cont, empty], 100)
    assert list(N(out["count"])) == [100, 100, 0]
    assert list(out["rounds"]) == [0, 1, 0]
    assert (N(out["records"][2]) == 0).all()


def test_continuation_with_more_than_a_block_kept_in_round_0():
    """max_per_img = 2000: round 0 keeps 1501 boxes (1500 separate ones and one of the near-duplicates behind them),
    more than one 1024-box chunk, so the first filter of the continuation runs two passes; 1000 separate boxes with
    lower scores then fill the detections up to 2000."""
    rng = np.random.default_rng(6)
    bx, sc = _case([(_spread(rng, 1500), _decreasing(1500, 0.99, 0.9), 1),
                    (_dups(rng, 16000, 100, 100), _decreasing(16000, 0.89, 0.6), 0),
                    (_spread(rng, 1000, 6000), _decreasing(1000, 0.5, 0.1), 0)])
    out = _run_case([(bx, sc)], 2000)
    assert int(out["count"][0]) == 2000 and out["rounds"][0] == 1


# ------------------------------------------------------------------ 4. the hot paths
IMG = (800, 1333)


def _infer_inputs(B, C, seed=2019):
    w = workload.config2(B=B, K=1, seed=seed, channels=C, img_shape=IMG, pad_shape=(800, 1344))
    cls, reg = [T(c) for c in w["cls"]], [T(r) for r in w["reg"]]
    feats = [T(f).contiguous(memory_format=torch.channels_last) for f in w["feats"]]
    img_hw = torch.tensor([[float(IMG[0]), float(IMG[1])]] * B, device=DEV)
    return w, cls, reg, feats, img_hw


@pytest.mark.parametrize("stages", [1, 3])
def test_infer_hot_path_full_cap_is_exact(stages):
    """Uniform logits at 81 classes, min_score 0.01: every foreground class of every proposal is a candidate (P * 80 per
    image, far past 16384).  With max_candidates = P * 80 nothing overflows and the detections are those of the
    reference on the last stage's boxes; with the default the flag is set and check() raises."""
    B, C, NC = 2, 8, 81
    w, cls, reg, feats, img_hw = _infer_inputs(B, C)
    rcnn = dict(min_score=0.01, nms_iou=THR, max_per_img=100, nms_type="official")
    probe = fused.InferHotPath(B, w["grids"], DEV, feat_channels=C, num_classes=NC, num_stages=stages, rcnn_test=rcnn)
    P = probe.P
    hp = fused.InferHotPath(B, w["grids"], DEV, feat_channels=C, num_classes=NC, num_stages=stages, rcnn_test=rcnn,
                            max_candidates=P * (NC - 1))
    assert hp.cap == P * (NC - 1) and probe.cap == 16384
    flat = (torch.zeros((B * P, NC), device=DEV), torch.zeros((B * P, 4 * NC), device=DEV))
    heads = [lambda x: flat] * stages
    rec = torch.full((B, hp.M, 6), -7.0, device=DEV)
    out = hp.step(cls, reg, feats, img_hw, heads, records=rec)
    hp.check()
    last = out["stages"][-1]
    for b in range(B):
        n = int(last["count"][b])
        assert n * (NC - 1) > 16384
        props = N(last["boxes"][b, :, :n])
        db, ds, dl, ncand = _rcnn_ref(props, np.zeros((n, NC), np.float32), np.zeros((n, 4 * NC), np.float32), IMG, 0.01, 100)
        assert ncand == n * (NC - 1)
        assert _assert_same(out, b, db, ds, dl) == 100
        r = N(rec[b])
        assert np.array_equal(r[:, 4], N(out["scores"][b])) and np.array_equal(r[:, 5], N(out["labels"][b]).astype(np.float32))
    probe.step(cls, reg, feats, img_hw, heads)
    with pytest.raises(_C.B200DetError, match="more than 16384"):
        probe.check()
    small = fused.InferHotPath(B, w["grids"], DEV, feat_channels=C, num_classes=NC, num_stages=stages, rcnn_test=rcnn,
                               max_candidates=20000)
    small.step(cls, reg, feats, img_hw, heads)
    with pytest.raises(_C.B200DetError, match="more than 20000"):
        small.check()


def test_infer_hot_path_full_cap_graph_replay():
    """A captured step with cap = P * 80 replays bitwise equal to an eager step."""
    B, C, NC = 2, 8, 81
    w, cls, reg, feats, img_hw = _infer_inputs(B, C, seed=7)
    rcnn = dict(min_score=0.001, nms_iou=THR, max_per_img=100, nms_type="official")
    hp = fused.InferHotPath(B, w["grids"], DEV, feat_channels=C, num_classes=NC, rcnn_test=rcnn, max_candidates=1 << 20)
    P = hp.P
    assert hp.cap == P * (NC - 1)
    g_ = torch.Generator(device=DEV).manual_seed(3)
    logits = torch.randn((B * P, NC), device=DEV, generator=g_) * 0.5
    deltas = torch.randn((B * P, 4 * NC), device=DEV, generator=g_) * 0.2
    heads = [lambda x: (logits, deltas)]
    rec = torch.zeros((B, hp.M, 6), device=DEV)
    hp.step(cls, reg, feats, img_hw, heads, records=rec)
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        gout = hp.step(cls, reg, feats, img_hw, heads, records=rec)
    for t in (gout["boxes"], gout["scores"], rec):
        t.zero_()
    g.replay()
    torch.cuda.synchronize()
    got = [t.clone() for t in (gout["boxes"], gout["scores"], gout["labels"], gout["count"], rec)]
    hp.check()
    eout = hp.step(cls, reg, feats, img_hw, heads, records=rec)
    torch.cuda.synchronize()
    for a, e in zip(got, (eout["boxes"], eout["scores"], eout["labels"], eout["count"], rec)):
        assert torch.equal(a, e)
    assert int(got[3].min()) == 100


RET_GRIDS, RET_STRIDES = [(40, 52), (20, 26), (10, 13)], [8, 16, 32]
RET_SCALES = [4 * 2 ** (i / 3) for i in range(3)]


def test_dense_hot_path_full_cap_is_exact():
    """RetinaNet, 80 classes, min_score 0.01, logits 0 or -200 (scores 0.5 / 0): about a third of P * 80 candidates per
    image.  The default cap overflows; max_candidates = P * 80 gives the reference's detections."""
    rng = np.random.default_rng(9)
    C, B = 80, 2
    cls = [T(np.where(rng.uniform(0, 1, (B, 9 * C) + g) < 0.3, 0.0, -200.0).astype(np.float32)) for g in RET_GRIDS]
    reg = [T((0.3 * rng.standard_normal((B, 36) + g)).astype(np.float32)) for g in RET_GRIDS]
    img_hw = torch.tensor([[300.0, 400.0]] * B, device=DEV)
    cfg = dict(pre_nms=1000, min_bbox_size=0, min_score=0.01, nms_iou=THR, max_per_img=100, nms_type="official")
    kw = dict(head="retina", num_classes=C + 1, test_cfg=cfg, strides=RET_STRIDES, anchor_scales=RET_SCALES)
    dflt = fused.DenseInferHotPath(B, RET_GRIDS, DEV, **kw)
    hp = fused.DenseInferHotPath(B, RET_GRIDS, DEV, max_candidates=dflt.P * C, **kw)
    assert dflt.cap == 16384 and hp.cap == dflt.P * C
    dflt.step(cls, reg, img_hw)
    with pytest.raises(_C.B200DetError, match="more than 16384"):
        dflt.check()
    out = hp.step(cls, reg, img_hw)
    hp.check()
    for b in range(B):
        n = int(out["sel_count"][b])
        rows = N(out["sel_rows"][b, :n])
        x = np.concatenate([N(c[b]).reshape(C, -1) for c in cls], 1)[:, rows]       # [C][n] logits of the rows
        sc = np.where(x == 0, np.float32(0.5), np.float32(0.0)).astype(np.float32)
        db, ds, dl, ncand = _dense_ref(N(out["sel_boxes"][b, :, :n]), sc, n, 0.01, 100)
        assert ncand > 16384
        _assert_same(out, b, db, ds, dl + 1)


def test_infer_overflow_case_is_exact_with_max_candidates():
    """The overflow case of test_gpu_infer (seed-5 inputs, 21 classes, uniform logits, min_score 0.01: 20 candidates
    per proposal, more than 16384 per image): the default overflows; max_candidates = P * 20 gives the reference's
    detections.  The case's random deltas are replaced by zeros: decoded boxes are then exact on both sides, so every
    NMS decision can be compared exactly (the overflow comes from the logits alone)."""
    B, C, NC = 2, 8, 21
    w, cls, reg, feats, img_hw = _infer_inputs(B, C, seed=5)
    rcnn = dict(min_score=0.01, nms_iou=THR, max_per_img=100, nms_type="official")
    dflt = fused.InferHotPath(B, w["grids"], DEV, feat_channels=C, num_classes=NC, rcnn_test=rcnn)
    P = dflt.P
    deltas = np.zeros((B * P, 4 * NC), np.float32)
    flat = (torch.zeros((B * P, NC), device=DEV), T(deltas))
    dflt.step(cls, reg, feats, img_hw, [lambda x: flat])
    with pytest.raises(_C.B200DetError, match="more than 16384"):
        dflt.check()
    hp = fused.InferHotPath(B, w["grids"], DEV, feat_channels=C, num_classes=NC, rcnn_test=rcnn, max_candidates=P * (NC - 1))
    out = hp.step(cls, reg, feats, img_hw, [lambda x: flat])
    hp.check()
    st = out["stages"][-1]
    stds = (0.1, 0.1, 0.2, 0.2)
    for b in range(B):
        n = int(st["count"][b])
        assert n * (NC - 1) > 16384
        props = N(st["boxes"][b, :, :n])
        d = deltas[b * P:b * P + n]
        param = np.ascontiguousarray(d.T).reshape(4, NC, n)
        boxes = np.stack([oracle.param2bbox(props, np.ascontiguousarray(param[:, c, :]), [0.0] * 4, list(stds), IMG)
                          for c in range(NC)], 1)                  # [4, NC, n]
        ii, cc = np.nonzero(np.ones((n, NC), bool)[:, 1:])
        cc = cc + 1
        cb = boxes[:, cc, ii].T.astype(np.float32)
        cs = np.full(ii.size, np.float32(1.0) / np.float32(NC), np.float32)
        k = _batched_ref(cb, cs, cc, 100)
        kk = int(out["count"][b])
        assert kk == 100
        assert np.array_equal(N(out["labels"][b, :kk]), cc[k])
        np.testing.assert_allclose(N(out["scores"][b, :kk]), cs[k], rtol=1e-6)
        np.testing.assert_allclose(N(out["boxes"][b, :, :kk]), cb[k].T, rtol=0, atol=1e-5)


def test_dense_overflow_case_is_exact_with_max_candidates():
    """The overflow case of test_gpu_dense_infer (RetinaNet, 20 classes, min_score 0.01): the default overflows;
    max_candidates = P * 20 gives the reference's detections.  The reference scores are sigmoid(x) = 1 / (1 + exp(-x))
    evaluated by torch on the device, the kernels' own formula, so the candidate test and the order are exact."""
    rng = np.random.default_rng(9)
    C = 20
    cls = [T(rng.standard_normal((1, 9 * C) + g).astype(np.float32)) for g in RET_GRIDS]
    reg = [T((0.3 * rng.standard_normal((1, 36) + g)).astype(np.float32)) for g in RET_GRIDS]
    cfg = dict(pre_nms=1000, min_bbox_size=0, min_score=0.01, nms_iou=0.5, max_per_img=100, nms_type="official")
    kw = dict(head="retina", num_classes=C + 1, test_cfg=cfg, strides=RET_STRIDES, anchor_scales=RET_SCALES)
    img = torch.tensor([[300.0, 400.0]], device=DEV)
    dflt = fused.DenseInferHotPath(1, RET_GRIDS, DEV, **kw)
    dflt.step(cls, reg, img)
    with pytest.raises(_C.B200DetError, match="16384"):
        dflt.check()
    hp = fused.DenseInferHotPath(1, RET_GRIDS, DEV, max_candidates=dflt.P * C, **kw)
    assert hp.cap == dflt.P * C
    out = hp.step(cls, reg, img)
    hp.check()
    n = int(out["sel_count"][0])
    rows = out["sel_rows"][0, :n].long()
    x = torch.cat([c[0].reshape(C, -1) for c in cls], 1)[:, rows]
    sc = N(1.0 / (1.0 + torch.exp(-x)))
    db, ds, dl, ncand = _dense_ref(N(out["sel_boxes"][0, :, :n]), sc, n, 0.01, 100)
    assert ncand > 16384
    assert _assert_same(out, 0, db, ds, dl + 1) == 100


@pytest.mark.parametrize("bad", [0, -1, (1 << 20) + 1, 1.5, True, "all"])
def test_bad_max_candidates_rejected(bad):
    w = workload.config2(B=1, K=1, channels=8, img_shape=(160, 213), pad_shape=(160, 224))
    with pytest.raises(_C.B200DetError, match="max_candidates"):
        fused.InferHotPath(1, w["grids"], DEV, feat_channels=8, num_classes=81, max_candidates=bad)
    with pytest.raises(_C.B200DetError, match="max_candidates"):
        fused.DenseInferHotPath(1, RET_GRIDS, DEV, head="retina", num_classes=81, strides=RET_STRIDES, max_candidates=bad)


def test_library_rejects_caps_past_the_maximum():
    assert _C.lib().b2d_rcnn_detect_workspace_bytes(_C.DET_MAX_CAP + 1, 1) == 0
    boxes = np.zeros((1, 4, 4), np.float32)
    score = np.full((1, 2, 4), 0.5, np.float32)
    with pytest.raises(_C.B200DetError):
        dense_detect(boxes, score, [4], 0.0, 4, _C.DET_MAX_CAP + 1)
    with pytest.raises(_C.B200DetError, match="max_per_img"):
        dense_detect(boxes, score, [4], 0.0, 16385, BIG)
