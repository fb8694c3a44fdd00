"""ClipSimilarity.predict_many_iou / FusionEngine.predict_many_iou / dc_predict_many_iou: every grounding query of a
batch scored against its ground truth in one call. Query q's (inter, union) must equal what binary_iou_counts counts on
predict_many's prediction row and the isin mask of the query's ids, and metrics.grounding_scores of them must be
trainMetricPC's result."""
import ctypes

import numpy as np
import pytest
import torch

from dropclip_b200 import _lib
from dropclip_b200.engine import FusionEngine, gt_csr
from dropclip_b200.metrics import binary_iou_counts, grounding_scores, trainMetricPC
from dropclip_b200.similarity import ClipSimilarity
from tests.test_predict_many import BATCHES, VARIANTS, _batch, _cs, _split


# ---------------------------------------------------------------------------------------------- host (CPU)
def test_gt_csr_keeps_query_order_and_sorts_and_dedupes_each_list():
    off, ids = gt_csr([[[3, 1, 3], []], [(np.int64(7), -2)], [iter([5])]], [2, 1, 1], torch.int64)
    assert off.dtype == np.int32 and ids.dtype == np.int64
    assert off.tolist() == [0, 2, 2, 4, 5]
    assert ids.tolist() == [1, 3, -2, 7, 5]
    off, ids = gt_csr([], [], torch.int32)
    assert off.tolist() == [0] and ids.size == 0


def test_gt_csr_rejects_ids_outside_the_label_dtype_and_miscounted_lists():
    assert gt_csr([[[-2 ** 31, 2 ** 31 - 1]]], [1], torch.int32)[1].tolist() == [-2 ** 31, 2 ** 31 - 1]
    for bad in (2 ** 31, -2 ** 31 - 1):
        with pytest.raises(ValueError):
            gt_csr([[[1, bad]]], [1], torch.int32)
    assert gt_csr([[[2 ** 31, -2 ** 63]]], [1], torch.int64)[1].tolist() == [-2 ** 63, 2 ** 31]
    with pytest.raises(ValueError):
        gt_csr([[[2 ** 63]]], [1], torch.int64)
    with pytest.raises(ValueError):  # scene 0 has two queries
        gt_csr([[[1]]], [2], torch.int64)
    with pytest.raises(ValueError):  # one list per scene
        gt_csr([[[1]], [[2]]], [1], torch.int64)
    with pytest.raises(TypeError):  # ids are integers
        gt_csr([[[1.5]]], [1], torch.int64)


def test_engine_predict_many_iou_host_checks():
    """FusionEngine.predict_many_iou checks every index, count, mode, label and id rule before anything reaches the
    device (the engine here has no library: any device work would raise AttributeError)."""
    eng = object.__new__(FusionEngine)
    x, t = torch.zeros(6, 64), torch.zeros(5, 64)
    lab = torch.zeros(6, dtype=torch.int32)
    P = _lib.DC_GROUND_PAIRED
    pos, negs, ids = [[0], [0]], [[[1]], [[1]]], [[[1]], [[2]]]
    args = (P, 0.1, True, 0.7)
    with pytest.raises(IndexError):  # scene 1's positive column outside its 2 prompts
        FusionEngine.predict_many_iou(eng, x, [4, 2], t, [3, 2], [[0], [2]], negs, lab, ids, *args)
    with pytest.raises(ValueError):  # paired needs a negative for every query
        FusionEngine.predict_many_iou(eng, x, [4, 2], t, [3, 2], [[0, 1], [0]], [[[1], []], [[1]]], lab,
                                      [[[1], [2]], [[2]]], *args)
    with pytest.raises(ValueError):  # point counts do not sum to the rows
        FusionEngine.predict_many_iou(eng, x, [4, 3], t, [3, 2], pos, negs, lab, ids, *args)
    with pytest.raises(ValueError):  # labels of another dtype
        FusionEngine.predict_many_iou(eng, x, [4, 2], t, [3, 2], pos, negs, lab.float(), ids, *args)
    with pytest.raises(ValueError):
        FusionEngine.predict_many_iou(eng, x, [4, 2], t, [3, 2], pos, negs, lab.to(torch.uint8), ids, *args)
    with pytest.raises(ValueError):  # one label per feature row
        FusionEngine.predict_many_iou(eng, x, [4, 2], t, [3, 2], pos, negs, lab[:5], ids, *args)
    with pytest.raises(ValueError):  # an id outside int32
        FusionEngine.predict_many_iou(eng, x, [4, 2], t, [3, 2], pos, negs, lab, [[[1]], [[2 ** 31]]], *args)
    with pytest.raises(ValueError):  # one id list per query
        FusionEngine.predict_many_iou(eng, x, [4, 2], t, [3, 2], pos, negs, lab, [[[1]], []], *args)
    with pytest.raises(AttributeError):  # every check passed: the next step is the library
        FusionEngine.predict_many_iou(eng, x, [4, 2], t, [3, 2], pos, negs, lab.long(), [[[1]], [[2 ** 31]]], *args)


def test_clip_predict_many_iou_checks_before_the_device():
    cs = object.__new__(ClipSimilarity)
    cs.method, cs.threshold, cs.norm_vis_feat = "paired", 0.7, True
    with pytest.raises(RuntimeError):  # CPU features: no CPU fallback
        cs.predict_many_iou(torch.zeros(4, 64), [4], torch.zeros(4, dtype=torch.int64), [{"a": [1]}])


def test_grounding_scores_against_the_reference_metric():
    """grounding_scores of the per-instance counts equals oracle.metrics_ref.train_metric_pc (utils/misc.py:21-50) on
    the same masks: Pr@k exactly, mIoU up to the order of the fp32 sum."""
    from oracle import metrics_ref
    rng = np.random.default_rng(4)
    preds, gts = [], []
    for n in [0, 1, 50, 1000, 3000, 7, 200, 200]:
        preds.append(torch.from_numpy(rng.random(n) < rng.random()).float())
        gts.append(torch.from_numpy(rng.random(n) < rng.random()))
    preds.append(gts[-1].float())  # IoU 1
    gts.append(gts[-1].clone())
    inter = torch.tensor([int((p.bool() & g).sum()) for p, g in zip(preds, gts)])
    union = torch.tensor([int((p.bool() | g).sum()) for p, g in zip(preds, gts)])
    for pr_ious in ([0.25, 0.5, 0.75], [0.0, 0.9]):
        miou, prs = grounding_scores(inter, union, pr_ious)
        want_miou, want_prs = metrics_ref.train_metric_pc([p.clone() for p in preds], gts, pr_ious=pr_ious)
        assert abs(float(miou) - float(want_miou)) <= 1e-5 * abs(float(want_miou))
        assert [float(p) for p in prs] == [float(p) for p in want_prs]
    assert grounding_scores(torch.zeros(0, dtype=torch.int64), torch.zeros(0, dtype=torch.int64)) == trainMetricPC([], [])


# ---------------------------------------------------------------------------------------------- GPU
def _ground_truth(counts, queries, label_dtype, seed):
    """Labels in [-3, 8) (negative ones included) and, per query, 0, 1 or 3 ids, with repeats and with ids no point
    carries (8, and the largest id of the label dtype)."""
    rng = np.random.default_rng(seed)
    labels = torch.from_numpy(rng.integers(-3, 8, size=sum(counts))).to(label_dtype).cuda()
    absent = torch.iinfo(label_dtype).max
    patterns = [lambda i: [], lambda i: [i % 11 - 3], lambda i: [5, -2, 1], lambda i: [4, 4, -3, 4],
                lambda i: [absent, 2, 8], lambda i: [8]]
    obj = [{t: patterns[(s + i) % len(patterns)](i) for i, t in enumerate(qs)} for s, qs in enumerate(queries)]
    return labels, obj


def _expected(res, labels, counts, obj):
    """binary_iou_counts over predict_many's prediction rows and the isin masks of the query ids."""
    preds, gts = [], []
    for (pred, _), lab, o in zip(res, _split(labels, counts), obj):
        for row, ids in zip(pred, o.values()):
            preds.append(row)
            gts.append(torch.isin(lab, torch.tensor(sorted(set(ids)), dtype=lab.dtype, device=lab.device)))
    if not preds:
        return torch.zeros(0, dtype=torch.int64), torch.zeros(0, dtype=torch.int64)
    if sum(p.numel() for p in preds) == 0:
        return torch.zeros(len(preds), dtype=torch.int64), torch.zeros(len(preds), dtype=torch.int64)
    inter, union = binary_iou_counts(preds, gts, 0.35, in_place=False)
    return inter.cpu(), union.cpu()


def _check_counts(cs, feat, counts, labels, obj, method, qneg, thr=0.7):
    queries = [list(o) for o in obj]
    res = cs.predict_many(feat.clone(), counts, queries, qneg=qneg, method=method, threshold=thr)
    x = feat.clone()
    inter, union = cs.predict_many_iou(x, counts, labels, obj, qneg=qneg, method=method, threshold=thr)
    n_q = sum(len(q) for q in queries)
    assert inter.shape == union.shape == (n_q,) and inter.dtype == union.dtype == torch.int64 and inter.is_cuda
    want_i, want_u = _expected(res, labels, counts, obj)
    assert torch.equal(inter.cpu(), want_i), f"{method} {qneg}: intersections differ"
    assert torch.equal(union.cpu(), want_u), f"{method} {qneg}: unions differ"
    assert bool((inter <= union).all())


@pytest.mark.gpu
@pytest.mark.parametrize("batch", list(BATCHES))
@pytest.mark.parametrize("dname,dim,lname", [("f16", 768, "i64"), ("f32", 768, "i32"), ("f16", 512, "i32"),
                                             ("f32", 512, "i64")])
def test_predict_many_iou_counts_equal_binary_iou_counts(batch, dname, dim, lname):
    dtype = torch.float32 if dname == "f32" else torch.float16
    label_dtype = torch.int32 if lname == "i32" else torch.int64
    cs = _cs(dim, dtype)
    shapes = BATCHES[batch]
    feat, counts, queries = _batch(cs, shapes, dim, dtype, seed=len(shapes) + dim)
    labels, obj = _ground_truth(counts, queries, label_dtype, seed=dim)
    one_point = any(n == 1 and q for n, q in shapes)
    for method, qneg in VARIANTS:
        if method == "argmax" and qneg is not None and one_point:
            x = feat.clone()
            with pytest.raises(IndexError):
                cs.predict_many_iou(x, counts, labels, obj, qneg=qneg, method=method)
            assert torch.equal(x, feat)  # raised before any scene was normalised
            keep = [s for s, (n, q) in enumerate(shapes) if not (n == 1 and q)]
            rows, labs = _split(feat, counts), _split(labels, counts)
            _check_counts(cs, torch.cat([rows[s] for s in keep]).contiguous(), [counts[s] for s in keep],
                          torch.cat([labs[s] for s in keep]), [obj[s] for s in keep], method, qneg)
        else:
            _check_counts(cs, feat, counts, labels, obj, method, qneg)


@pytest.mark.gpu
@pytest.mark.parametrize("dname", ["f32", "f16"])
@pytest.mark.parametrize("norm", [True, False])
def test_predict_many_iou_normalises_in_place_like_predict_many(dname, norm):
    dtype = torch.float32 if dname == "f32" else torch.float16
    cs = _cs(768, dtype, norm_vis_feat=norm)
    feat, counts, queries = _batch(cs, [(1000, 5), (300, 0), (2000, 3)], 768, dtype, seed=9)
    labels, obj = _ground_truth(counts, queries, torch.int64, seed=1)
    x1, x2 = feat.clone(), feat.clone()
    cs.predict_many(x1, counts, queries)
    cs.predict_many_iou(x2, counts, labels, obj)
    assert torch.equal(x1, x2)
    assert torch.equal(_split(x2, counts)[1], _split(feat, counts)[1])  # no queries: untouched


@pytest.mark.gpu
@pytest.mark.parametrize("negatives_mode", ["scene", "generic"])
def test_validation_loop_through_predict_many_iou(negatives_mode):
    """validate_grounding's loop (tools/validate_upper_bound.py:200-221) over a batch of 4 scenes: trainMetricPC over
    predict_many's rows and the per-query ground-truth masks against grounding_scores(*predict_many_iou(...))."""
    cs = _cs(768, torch.float16, method="paired", threshold=0.7)
    rng = np.random.default_rng(5)
    outputs, labels, scene_queries = [], [], []
    for s, n in enumerate([4000, 2500, 3000, 1000]):
        obj_queries = {f"scene {s} object {i}": [i + 1] for i in range(3 + s)}
        obj_queries[f"scene {s} pair"] = [1, 2]
        emb = cs.model.encode_text(cs._tok(list(obj_queries))).float().cpu()
        label = torch.from_numpy(rng.integers(0, 3 + s + 1, size=n))
        out = torch.zeros((n, 768))
        for i in range(3 + s):
            out[label == i + 1] = emb[i]
        out += 0.03 * torch.from_numpy(rng.standard_normal((n, 768)).astype(np.float32))
        outputs.append(out)
        labels.append(label.cuda())
        scene_queries.append(obj_queries)
    qneg = "scene" if negatives_mode == "scene" else []
    batch = torch.cat(outputs).cuda().half()
    counts = [o.shape[0] for o in outputs]
    res = cs.predict_many(batch.clone(), counts, [list(q) for q in scene_queries], qneg)
    pred_list, gt_list = [], []
    for (pred, _), label_d, obj_queries in zip(res, labels, scene_queries):
        for row, obj_ids in zip(pred, obj_queries.values()):
            gt = torch.zeros_like(label_d)
            for obj in obj_ids:
                gt[label_d == obj] = True
            pred_list.append(row)
            gt_list.append(gt)
    iou, prs = trainMetricPC(pred_list, gt_list, pr_ious=[0.25, 0.5, 0.75], sigmoid=False)
    iou2, prs2 = grounding_scores(*cs.predict_many_iou(batch.clone(), counts, torch.cat(labels), scene_queries, qneg))
    assert float(iou) > 0.5
    assert iou2.dtype == iou.dtype and torch.equal(iou2.cpu(), iou.cpu())  # bit for bit
    assert [p.item() for p in prs2] == [p.item() for p in prs]


def _lib_call(x, labels, gt_off, gt_ids, inter, union):
    """dc_predict_many_iou on one scene of 64 points, two queries (paired, one negative each)."""
    lib = _lib.load()
    text = torch.nn.functional.normalize(torch.randn(2, x.shape[1]), dim=-1).half().cuda()
    c = lambda a: a.ctypes.data_as(ctypes.c_void_p)  # noqa: E731
    point_off, prompt_off, query_off = np.array([0, 64]), np.array([0, 2], np.int32), np.array([0, 2], np.int32)
    pos, neg_off, neg_cols = np.array([0, 1], np.int32), np.array([0, 1, 2], np.int32), np.array([1, 0], np.int32)
    ws_bytes = lib.dc_predict_many_iou_workspace(1, c(point_off), c(prompt_off), c(query_off), 2, int(gt_ids.size),
                                                 x.shape[1], _lib.DC_F16, _lib.DC_F16)
    ws = torch.empty(ws_bytes, dtype=torch.uint8, device="cuda")
    _lib.check(lib.dc_predict_many_iou(
        _lib.ptr(x), _lib.DC_F16, _lib.ptr(text), _lib.DC_F16, x.shape[1], 1, c(point_off), c(prompt_off), c(query_off),
        c(pos), c(neg_off), c(neg_cols), _lib.ptr(labels), _lib.torch_dtype_code(labels.dtype), c(gt_off),
        c(gt_ids) if gt_ids.size else None, _lib.DC_GROUND_PAIRED, 0.1, 1, 0.7, _lib.ptr(inter), _lib.ptr(union),
        _lib.ptr(ws), ws_bytes, _lib.current_stream()))


@pytest.mark.gpu
def test_predict_many_iou_errors_before_any_row_changes():
    cs = _cs(768, torch.float16)
    feat, counts, queries = _batch(cs, [(500, 4), (1, 3), (200, 2)], 768, torch.float16, seed=21)
    labels, obj = _ground_truth(counts, queries, torch.int32, seed=2)

    def raises(exc, rows, *args, match=None, **kw):
        x = rows.clone()
        with pytest.raises(exc, match=match):
            cs.predict_many_iou(x, *args, **kw)
        assert torch.equal(x, rows)

    raises(IndexError, feat, counts, labels, obj, method="argmax")  # a one-point scene with queries
    raises(ValueError, feat, counts, labels.float(), obj)
    raises(ValueError, feat, counts, labels[:-1], obj)
    raises(RuntimeError, feat, counts, labels.cpu(), obj)
    raises(ValueError, feat, [500, 1, 199], labels, obj)
    bad = [dict(o) for o in obj]
    bad[2][queries[2][0]] = [2 ** 31]  # outside int32
    raises(ValueError, feat, counts, labels, bad)
    assert cs.predict_many_iou(feat.clone(), counts, labels.long(), bad) is not None  # fine for int64 labels
    raises(RuntimeError, feat[:500], [500], labels[:500], [{f"q{i}": [1] for i in range(1537)}], qneg=None,
           match="0..1536 prompts")
    x = feat.clone()
    assert cs.predict_many_iou(x, counts, labels, obj, method="other") is None
    assert torch.equal(x, feat)
    with pytest.raises(RuntimeError):
        cs.predict_many_iou(feat.cpu(), counts, labels, obj)
    # the library's own checks of the host tables: ids not ascending, gt_off decreasing
    x = feat[:64].clone()
    lab = labels[:64].contiguous()
    inter = torch.full((2,), -7, dtype=torch.int64, device="cuda")
    union = inter.clone()
    with pytest.raises(_lib.DropClipError, match="strictly ascending"):
        _lib_call(x, lab, np.array([0, 2, 3], np.int32), np.array([3, 3, 1]), inter, union)
    with pytest.raises(_lib.DropClipError, match="must not decrease"):
        _lib_call(x, lab, np.array([0, 2, 1], np.int32), np.array([1, 3]), inter, union)
    assert torch.equal(x, feat[:64]) and (inter == -7).all() and (union == -7).all()
    _lib_call(x, lab, np.array([0, 2, 3], np.int32), np.array([1, 3, 2]), inter, union)
    assert (inter >= 0).all() and (union >= inter).all()


@pytest.mark.gpu
def test_predict_many_iou_edge_cases():
    cs = _cs(768, torch.float16)
    feat, counts, queries = _batch(cs, [(500, 4), (0, 3), (200, 0)], 768, torch.float16, seed=22)
    labels, obj = _ground_truth(counts, queries, torch.int64, seed=3)
    # S = 0, and no queries at all
    i, u = cs.predict_many_iou(feat[:0].clone(), [], labels[:0], [])
    assert i.shape == u.shape == (0,)
    i, u = cs.predict_many_iou(feat[:200].clone(), [200], labels[:200], [{}])
    assert i.shape == u.shape == (0,)
    # every scene empty: 0 / 0 for each query
    i, u = cs.predict_many_iou(feat[:0].clone(), [0, 0], labels[:0], [{"a": [1], "b": [2, 3]}, {}])
    assert i.tolist() == [0, 0] and u.tolist() == [0, 0]
    # the empty scene's queries report 0 / 0 among the others
    i, u = cs.predict_many_iou(feat.clone(), counts, labels, obj)
    assert i.shape == (7,) and i[4:].tolist() == [0, 0, 0] and u[4:].tolist() == [0, 0, 0]
    _check_counts(cs, feat, counts, labels, obj, "paired", "scene")


@pytest.mark.gpu
def test_predict_many_iou_on_a_side_stream():
    """Issued on a non-default stream behind a long kernel: the call returns while the stream is still busy (no host
    synchronisation inside it) and gives the default stream's counts."""
    eng = FusionEngine("cuda")
    g = torch.Generator().manual_seed(2)
    counts, p_counts = [3000, 129, 10_000], [5, 21, 3]
    feats = torch.randn((sum(counts), 768), generator=g).half().cuda()
    text = torch.randn((sum(p_counts), 768), generator=g)
    text = (text / text.norm(dim=-1, keepdim=True)).half().cuda()
    labels = torch.randint(0, 6, (sum(counts),), generator=g).cuda()
    pos = [[0, 1, 2], list(range(21)), [2]]
    negs = [[[3, 4]] * 3, [[j for j in range(21) if j != i] for i in range(21)], [[0, 1]]]
    gt = [[[0], [1, 2], []], [[i % 6] for i in range(21)], [[5, 4, 3]]]
    args = (pos, negs, labels, gt, _lib.DC_GROUND_PAIRED, 0.1, True, 0.7)
    want = eng.predict_many_iou(feats.clone(), counts, text, p_counts, *args)
    torch.cuda.synchronize()
    side = torch.cuda.Stream()
    x = feats.clone()
    torch.cuda.synchronize()
    with torch.cuda.stream(side):
        torch.cuda._sleep(200_000_000)  # ~0.1 s of spinning ahead of the call
        got = eng.predict_many_iou(x, counts, text, p_counts, *args)
        busy = not side.query()
    side.synchronize()
    assert busy, "predict_many_iou waited for the stream"
    assert torch.equal(want[0], got[0]) and torch.equal(want[1], got[1])
    assert int(want[1].sum()) > 0
