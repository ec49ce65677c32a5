"""GPU parity of the batched test-time path (fused.InferHotPath, SURVEY 3.2): RPN proposals at the test configuration
-> per stage RoIAlign -> the stage head -> arg-max refine between stages -> detections with packed records after the
last stage.  Every stage is compared with the CPU oracle starting from the GPU's own stage inputs, so last-bit
differences of one stage do not cascade into the next."""
import numpy as np
import pytest
import torch

import oracle

pytestmark = pytest.mark.gpu

if torch.cuda.is_available():
    import b200det
    from b200det import _C, fused, workload
    DEV = torch.device("cuda:0")

STDS = ((0.1, 0.1, 0.2, 0.2), (0.05, 0.05, 0.1, 0.1), (0.033, 0.033, 0.067, 0.067))
RPN_TEST = dict(pre_nms=1000, post_nms=1000, max_num=1000, nms_iou=0.7, min_bbox_size=0)
RCNN_TEST = dict(min_score=0.05, nms_iou=0.5, max_per_img=100, nms_type="official")
IMG = (800, 1333)


def T(a):
    return torch.from_numpy(np.ascontiguousarray(a)).to(DEV)


def N(t):
    return t.detach().cpu().numpy()


class InferPath(object):
    """CPU oracle of SURVEY 3.2 for ONE image, composed only of existing oracle functions (rpn_proposals, roi_extract,
    param2bbox, rcnn_detect).  Each stage method takes its inputs -- boxes and the head's outputs -- as arrays, so a
    test can feed it the GPU's stage inputs."""

    def __init__(self, grids, strides, img_shape, num_stages=1, rpn_test=RPN_TEST, rcnn_test=RCNN_TEST, stage_stds=STDS):
        self.anchors = [oracle.anchor_grid(s, g, scales=[8]).reshape(4, -1) for s, g in zip(strides, grids)]
        self.offs = np.cumsum([0] + [a.shape[1] for a in self.anchors])
        self.img, self.strides = tuple(img_shape[:2]), tuple(strides)
        self.rpn_test, self.rcnn_test, self.stds = rpn_test, rcnn_test, stage_stds[:num_stages]

    def proposals(self, cls, reg):
        """cls[l] [A,H,W], reg[l] [4A,H,W] -> boxes [4,k], scores [k], provenance (anchor index in the pyramid) [k]."""
        b, s, lv, ix = oracle.rpn_proposals([c.reshape(-1) for c in cls], [r.reshape(4, -1) for r in reg], self.anchors,
                                            self.rpn_test, [0, 0, 0, 0], [1, 1, 1, 1], self.img)
        return b, s, self.offs[lv] + ix

    def roi_feats(self, feats, boxes):
        return oracle.roi_extract(feats, np.ascontiguousarray(boxes), strides=self.strides[:4])

    def refine(self, s, boxes, cls_out, reg_out):
        """BBoxHead.refine_bboxes with the test-time labels argmax(cls_out) (lib/detectors/cascade_rcnn.py:186-190)."""
        n = boxes.shape[1]
        label = np.argmax(cls_out, 1)
        reg_c = reg_out.shape[1] // 4
        d = reg_out.reshape(n, 4, reg_c)[np.arange(n), :, label if reg_c > 1 else 0].T
        return oracle.param2bbox(np.ascontiguousarray(boxes), np.ascontiguousarray(d), [0.0] * 4, list(self.stds[s]), self.img)

    def detect(self, boxes, cls_out, reg_out):
        c = self.rcnn_test
        return oracle.rcnn_detect(np.ascontiguousarray(boxes), cls_out, reg_out, self.img, [0.0] * 4, list(self.stds[-1]),
                                  c["min_score"], c["nms_iou"], c["max_per_img"], c["nms_type"])


class Head(torch.nn.Module):
    """Deterministic stand-in for a stage's RCNN head: 7x7 mean-pool, then seeded fc layers written as products and sums
    (no cuBLAS algorithm choice: eager and graph-captured calls compute the same bits)."""

    def __init__(self, C, NC, reg_c, seed, scale=6.0):
        super().__init__()
        g = torch.Generator().manual_seed(seed)
        self.wc = (torch.randn((NC, C), generator=g) * scale).to(DEV)
        self.wr = (torch.randn((4 * reg_c, C), generator=g) * 0.5).to(DEV)
        self.bias = torch.zeros(NC, device=DEV)
        self.bias[0] = 1.0                                                   # background a little ahead, as trained heads are

    def forward(self, x):
        p = x.mean((2, 3))
        return (p[:, None, :] * self.wc[None]).sum(-1) + self.bias, (p[:, None, :] * self.wr[None]).sum(-1)


def _inputs(B, channels, seed=2019, pad=(800, 1344)):
    w = workload.config2(B=B, K=1, seed=seed, channels=channels, img_shape=IMG, pad_shape=pad)
    cls, reg = [T(c) for c in w["cls"]], [T(r) for r in w["reg"]]
    feats = [T(f).contiguous(memory_format=torch.channels_last) for f in w["feats"]]
    img_hw = torch.tensor([[float(IMG[0]), float(IMG[1])]] * B, device=DEV)
    return w, cls, reg, feats, img_hw


def _check_detections(op, hp, out, b, n, records=None):
    st = out["stages"][-1]
    P = hp.P
    kb, ks, kl = op.detect(N(st["boxes"][b, :, :n]), N(st["cls_out"][b * P:b * P + n]), N(st["reg_out"][b * P:b * P + n]))
    k = int(out["count"][b])
    assert k == ks.shape[0], (b, k, ks.shape)
    assert np.array_equal(N(out["labels"][b, :k]), kl)
    np.testing.assert_allclose(N(out["scores"][b, :k]), ks, rtol=1e-5, atol=1e-7)
    np.testing.assert_allclose(N(out["boxes"][b, :, :k]), kb, rtol=1e-5, atol=1e-3)
    if records is not None:
        r = N(records[b])
        assert np.array_equal(r[:k, :4], N(out["boxes"][b, :, :k]).T)
        assert np.array_equal(r[:k, 4], N(out["scores"][b, :k]))
        assert np.array_equal(r[:k, 5], N(out["labels"][b, :k]).astype(np.float32))
        assert (r[k:] == 0).all()
    return k


def test_one_stage_config2_vs_oracle():
    """faster_rcnn_r50_fpn test path at config-2 geometry (800x1344 pyramid, 1000 proposals), B = 2, 64 channels."""
    B, C, NC = 2, 64, 21
    w, cls, reg, feats, img_hw = _inputs(B, C)
    hp = fused.InferHotPath(B, w["grids"], DEV, feat_channels=C, num_classes=NC)
    head = Head(C, NC, NC, seed=1)
    rec = torch.full((B, hp.M, 6), -7.0, device=DEV)
    out = hp.step(cls, reg, feats, img_hw, [head], records=rec)
    hp.check()
    op = InferPath(w["grids"], w["strides"], IMG)
    st = out["stages"][0]
    total = 0
    for b in range(B):
        ob, osc, oprov = op.proposals([c[b] for c in w["cls"]], [r[b] for r in w["reg"]])
        n = int(st["count"][b])
        assert n == ob.shape[1], (b, n, ob.shape)
        assert np.array_equal(N(hp.proposals.prov[b, :n]), oprov)
        np.testing.assert_allclose(N(st["boxes"][b, :, :n]), ob, rtol=1e-5, atol=1e-3)
        np.testing.assert_allclose(N(hp.proposals.scores[b, :n]), osc, rtol=1e-5, atol=1e-7)
        ref = op.roi_feats([f[b] for f in w["feats"]], N(st["boxes"][b, :, :n]))
        got = N(st["roi_feats"][b * hp.P:b * hp.P + n])
        assert np.array_equal(got.view(np.uint32), ref.view(np.uint32)), b
        total += _check_detections(op, hp, out, b, n, rec)
    assert total > 0                                            # the head's logits put some classes above 0.05


@pytest.mark.parametrize("agnostic", [False, True])
def test_three_stages_argmax_refine_vs_oracle(agnostic):
    """Cascade test path: per stage the refined boxes equal param2bbox with np.argmax labels of the same logits, the
    stage's stds and the clamp (per-class deltas differ per class, so a wrong label moves the box), nothing is dropped,
    and the last stage's detections match the oracle."""
    B, C, NC = 2, 16, 21
    w, cls, reg, feats, img_hw = _inputs(B, C, seed=7)
    hp = fused.InferHotPath(B, w["grids"], DEV, feat_channels=C, num_classes=NC, num_stages=3, reg_class_agnostic=agnostic)
    heads = [Head(C, NC, 1 if agnostic else NC, seed=10 + s) for s in range(3)]
    out = hp.step(cls, reg, feats, img_hw, heads)
    hp.check()
    op = InferPath(w["grids"], w["strides"], IMG, num_stages=3)
    P = hp.P
    for s in range(2):
        cur, nxt = out["stages"][s], out["stages"][s + 1]
        for b in range(B):
            n = int(cur["count"][b])
            assert int(nxt["count"][b]) == n
            ref = op.refine(s, N(cur["boxes"][b, :, :n]), N(cur["cls_out"][b * P:b * P + n]), N(cur["reg_out"][b * P:b * P + n]))
            np.testing.assert_allclose(N(nxt["boxes"][b, :, :n]), ref, rtol=1e-5, atol=1e-3)
            if s == 0:
                assert np.array_equal(N(nxt["roi_feats"][b * P:b * P + n]).view(np.uint32),
                                      op.roi_feats([f[b] for f in w["feats"]], N(nxt["boxes"][b, :, :n])).view(np.uint32))
    for b in range(B):
        _check_detections(op, hp, out, b, int(out["stages"][-1]["count"][b]))


def test_argmax_ties_take_the_first_index():
    """b2d_refine_bboxes_argmax on crafted logits: equal maxima resolve to the lowest class index (torch.argmax), the
    background wins a tie with a foreground class; rows past the count are neither read (NaN logits there) nor written."""
    B, ld, NC = 2, 8, 5
    rows = np.array([[0, 0, 0, 0, 0],                  # all equal -> 0 (background)
                     [3, 1, 3, 3, 2],                  # background tied with foreground -> 0
                     [1, 4, 2, 4, 4],                  # foreground ties -> 1
                     [-1, -2, -3, -4, 5],              # last class
                     [2, 2, 7, 7, -7],                 # -> 2
                     [-5, -5, -5, -5, -5],
                     [0, 1, 0, 1, 0],
                     [9, 9, 9, 9, 9.5]], np.float32)
    cls = np.stack([rows, rows[::-1]]).copy()
    counts = np.array([ld, 5], np.int32)
    cls[1, 5:] = np.nan
    props = np.tile(np.array([[10.0], [20.0], [110.0], [220.0]], np.float32), (B, 1, ld))
    # per-class deltas dx = 0.1 * class: the refined x1 identifies the label
    reg = np.zeros((B, ld, 4, NC), np.float32)
    reg[:, :, 0, :] = 0.1 * np.arange(NC, dtype=np.float32)
    reg = reg.reshape(B, ld, 4 * NC)
    out = torch.full((B, 4, ld), -7.0, device=DEV)
    cnt = torch.full((B,), -1, dtype=torch.int32, device=DEV)
    img_hw = torch.tensor([[400.0, 600.0]] * B, device=DEV)
    stds = _C.host_f4(STDS[0], [1, 1, 1, 1])
    d_props, d_counts, d_cls, d_reg = T(props), T(counts), T(cls), T(reg)          # locals: they must outlive the launch
    _C.call("b2d_refine_bboxes_argmax", _C.ptr(out), _C.ptr(cnt), _C.ptr(d_props), ld, _C.ptr(d_counts), ld, _C.ptr(d_cls), NC,
            _C.ptr(d_reg), NC, _C.host_f4(None, [0, 0, 0, 0]), stds, _C.ptr(img_hw), B, _C.stream())
    torch.cuda.synchronize()
    assert np.array_equal(N(cnt), counts)
    for b in range(B):
        n = int(counts[b])
        lab = np.argmax(cls[b, :n], 1)
        assert lab.tolist() == ([0, 0, 1, 4, 2, 0, 1, 4] if b == 0 else [4, 1, 0, 2, 4])
        d = reg[b, :n].reshape(n, 4, NC)[np.arange(n), :, lab].T
        ref = oracle.param2bbox(np.ascontiguousarray(props[b, :, :n]), np.ascontiguousarray(d), [0.0] * 4, list(STDS[0]), (400, 600))
        np.testing.assert_allclose(N(out[b, :, :n]), ref, rtol=1e-5, atol=1e-3)
        assert (N(out[b, :, n:]) == -7.0).all()


def test_cuda_graph_replay_equals_eager_step():
    """One captured step (heads included), new inputs copied into the same buffers, replay: bitwise what an eager step
    computes on those inputs."""
    B, C, NC = 2, 16, 21
    w, cls, reg, feats, img_hw = _inputs(B, C, seed=3)
    w2 = _inputs(B, C, seed=4)
    hp = fused.InferHotPath(B, w["grids"], DEV, feat_channels=C, num_classes=NC, num_stages=3)
    heads = [Head(C, NC, NC, seed=20 + s) for s in range(3)]
    rec = torch.zeros((B, hp.M, 6), device=DEV)
    hp.step(cls, reg, feats, img_hw, heads, records=rec)           # first call outside the capture
    torch.cuda.synchronize()
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g, stream=side):
            gout = hp.step(cls, reg, feats, img_hw, heads, records=rec)
    torch.cuda.current_stream().wait_stream(side)
    for dst, src in zip(cls + reg + feats, w2[1] + w2[2] + w2[3]):
        dst.copy_(src)
    g.replay()
    torch.cuda.synchronize()
    pick = lambda o: [o["boxes"], o["scores"], o["labels"], o["count"], rec] + \
        [t for st in o["stages"] for t in (st["boxes"], st["count"], st["roi_feats"], st["cls_out"])]
    got = [t.clone() for t in pick(gout)]
    assert int(got[3].sum()) > 0
    eout = hp.step(cls, reg, feats, img_hw, heads, records=rec)
    torch.cuda.synchronize()
    for a, e in zip(got, pick(eout)):
        assert torch.equal(a, e)


def test_empty_image_and_candidate_overflow():
    """An image whose foreground scores all stay below min_score gets count 0 and all-zero records; head outputs with
    more than 16384 candidates in an image set the device flag without raising inside step(), check() then raises."""
    B, C, NC = 2, 8, 21
    w, cls, reg, feats, img_hw = _inputs(B, C, seed=5)
    hp = fused.InferHotPath(B, w["grids"], DEV, feat_channels=C, num_classes=NC)
    P = hp.P
    rng = np.random.default_rng(9)
    logits = rng.normal(0, 2.5, (B * P, NC)).astype(np.float32)
    logits[:P, 0] += 40.0                                          # image 0: background everywhere
    deltas = rng.normal(0, 0.5, (B * P, 4 * NC)).astype(np.float32)
    fixed = (T(logits), T(deltas))
    rec = torch.full((B, hp.M, 6), -7.0, device=DEV)
    out = hp.step(cls, reg, feats, img_hw, [lambda x: fixed], records=rec)
    hp.check()
    assert int(out["count"][0]) == 0 and (N(rec[0]) == 0).all()
    op = InferPath(w["grids"], w["strides"], IMG)
    assert _check_detections(op, hp, out, 1, int(out["stages"][0]["count"][1]), rec) > 0
    # uniform logits: every foreground class scores 1/21 >= 0.01, i.e. 20 candidates per proposal
    hp2 = fused.InferHotPath(B, w["grids"], DEV, feat_channels=C, num_classes=NC,
                             rcnn_test=dict(min_score=0.01, nms_iou=0.5, max_per_img=100, nms_type="official"))
    flat = (torch.zeros((B * P, NC), device=DEV), fixed[1])
    out2 = hp2.step(cls, reg, feats, img_hw, [lambda x: flat])
    torch.cuda.synchronize()
    assert int(out2["stages"][0]["count"].max()) * (NC - 1) > 16384
    with pytest.raises(_C.B200DetError, match="more than 16384"):
        hp2.check()


_NCCL_WORKER = r'''
import os, sys, numpy as np, torch, torch.distributed as dist
sys.path.insert(0, %(root)r)
import b200det
from b200det import dist as bdist, fused, workload
rank, world = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"])
torch.cuda.set_device(rank)
dev = torch.device("cuda", rank)
dist.init_process_group("nccl", rank=rank, world_size=world, device_id=dev)
B, C, NC = 2, 8, 21
w = workload.config2(B=B, K=1, seed=100 + rank, channels=C)
T = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(dev)
feats = [T(f).contiguous(memory_format=torch.channels_last) for f in w["feats"]]
img_hw = torch.tensor([[800.0, 1333.0]] * B, device=dev)
hp = fused.InferHotPath(B, w["grids"], dev, feat_channels=C, num_classes=NC)
rng = np.random.default_rng(rank)
fixed = (T(rng.normal(0, 2.5, (B * hp.P, NC)).astype(np.float32)), T(rng.normal(0, 0.5, (B * hp.P, 4 * NC)).astype(np.float32)))
rec = torch.zeros((B, hp.M, 6), device=dev)
out = hp.step([T(c) for c in w["cls"]], [T(r) for r in w["reg"]], feats, img_hw, [lambda x: fixed], records=rec)
hp.check()
allrec, allcnt = bdist.gather_detections(rec, out["count"])
assert allrec.shape == (world * B, hp.M, 6), allrec.shape
for g in range(world * B):
    r, slot = g %% world, g // world
    if r == rank:
        assert torch.equal(allrec[g], rec[slot]) and int(allcnt[g]) == int(out["count"][slot])
        assert int(allcnt[g]) > 0
dist.barrier(); dist.destroy_process_group()
print("rank", rank, "ok")
'''


def test_nccl_world2_gather_inference_records(tmp_path):
    """The records InferHotPath writes are the payload of dist.gather_detections over NCCL (two ranks, two GPUs).
    Skipped on a 1-GPU box."""
    import os, subprocess, sys
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    script = tmp_path / "w.py"
    script.write_text(_NCCL_WORKER % dict(root=root))
    procs = []
    for r in range(2):
        env = dict(os.environ, RANK=str(r), WORLD_SIZE="2", MASTER_ADDR="127.0.0.1", MASTER_PORT="29591")
        procs.append(subprocess.Popen([sys.executable, str(script)], env=env, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True))
    outs = [p.communicate(timeout=300)[0] for p in procs]
    assert all(p.returncode == 0 for p in procs), "\n".join(outs)
