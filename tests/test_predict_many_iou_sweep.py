"""ClipSimilarity.predict_many_iou_sweep / FusionEngine.predict_many_iou_sweep / dc_predict_many_iou_sweep: the grounding
counts of a batch at many thresholds in one call. Row t must equal, bit for bit, what predict_many_iou returns at
thresholds[t] on a fresh copy of the features."""
import ctypes

import numpy as np
import pytest
import torch

from dropclip_b200 import _lib
from dropclip_b200.engine import SWEEP_MAX_THRESHOLDS, FusionEngine, threshold_table
from dropclip_b200.metrics import grounding_scores
from dropclip_b200.similarity import ClipSimilarity
from tests.test_predict_many import BATCHES, VARIANTS, _batch, _cs, _split
from tests.test_predict_many_iou import _expected, _ground_truth

INF, NAN = float("inf"), float("nan")
# unsorted, with duplicates, falsy entries (the default threshold), +-inf, NaN and 1.0
THRESHOLDS = [0.7, 0.3, 0.7, 0.0, INF, 0.95, -INF, NAN, 1.0, 0.3, 0.05, None, 0.5000001]


# ---------------------------------------------------------------------------------------------- host (CPU)
def test_threshold_table_keeps_the_callers_order_and_rounds_to_fp32():
    t = threshold_table([0.7, 0.1, 0.7, INF, -INF, NAN, 1e39, 3, np.float32(0.2)])
    assert t.dtype == np.float32 and t.flags.c_contiguous
    want = [ctypes.c_float(x).value for x in (0.7, 0.1, 0.7, INF, -INF)]  # the scalar calls' rounding
    assert t[:5].tolist() == want
    assert np.isnan(t[5]) and t[6] == np.inf and t[7] == 3.0 and t[8] == np.float32(0.2)
    assert threshold_table(iter([0.25])).tolist() == [0.25]
    assert threshold_table(np.array([0.5, 0.25])).tolist() == [0.5, 0.25]
    # no default: 0 stays 0; with one, a falsy entry is `threshold or default`, as the scalar call reads it
    assert threshold_table([0, 0.0, 0.5]).tolist() == [0.0, 0.0, 0.5]
    got = threshold_table([0, 0.0, None, 0.5, NAN, -0.0], default=0.7)
    assert got[:4].tolist() == [np.float32(0.7)] * 3 + [0.5] and np.isnan(got[4]) and got[5] == np.float32(0.7)


def test_threshold_table_limits():
    with pytest.raises(ValueError):
        threshold_table([])
    with pytest.raises(ValueError):
        threshold_table([0.5] * (SWEEP_MAX_THRESHOLDS + 1))
    assert threshold_table([0.5] * SWEEP_MAX_THRESHOLDS).size == SWEEP_MAX_THRESHOLDS == 1024
    with pytest.raises(TypeError):  # None is only a default where ClipSimilarity supplies one
        threshold_table([None])


def _levels(thresholds):
    """dc_sweep_levels (pure host code): (levels, rank)."""
    lib = _lib.load()
    thr = np.asarray(thresholds, dtype=np.float32)
    levels, rank, n = np.empty(thr.size, np.float32), np.empty(thr.size, np.int32), ctypes.c_int(-1)
    _lib.check(lib.dc_sweep_levels(thr.ctypes.data_as(ctypes.c_void_p), thr.size, levels.ctypes.data_as(ctypes.c_void_p),
                                   rank.ctypes.data_as(ctypes.c_void_p), ctypes.byref(n)))
    return levels[:n.value], rank


def test_sweep_levels_sort_dedupe_and_rank_in_the_callers_order():
    thr = [0.7, 0.3, 0.7, INF, -INF, NAN, 1.0, 0.3, -0.0, 0.0]
    levels, rank = _levels(thr)
    assert levels.tolist()[:2] == [-INF, 0.0] and levels.tolist()[2:] == [np.float32(0.3), np.float32(0.7), 1.0, INF]
    assert rank.tolist() == [3, 2, 3, 5, 0, 5, 4, 2, 1, 1]  # NaN shares +inf's level, -0 shares +0's
    # every entry: x > thresholds[t] exactly when x exceeds levels[rank[t]], for x on and around each level
    xs = np.concatenate([levels, np.nextafter(levels, np.float32(np.inf)), np.nextafter(levels, np.float32(-np.inf)),
                         np.float32([NAN])])
    for t, v in enumerate(np.float32(thr)):
        assert np.array_equal(xs > v, xs > levels[rank[t]])
    rng = np.random.default_rng(0)
    thr = np.round(rng.random(1024), 2).astype(np.float32)  # about 100 distinct values
    levels, rank = _levels(thr)
    assert np.array_equal(levels, np.unique(thr)) and np.array_equal(levels[rank], thr)
    levels, rank = _levels([0.5])
    assert levels.tolist() == [0.5] and rank.tolist() == [0]


def test_library_rejects_threshold_counts_before_any_device_work():
    lib = _lib.load()
    one = np.float32([0.5] * 1025)
    p = one.ctypes.data_as(ctypes.c_void_p)
    n = ctypes.c_int()
    for count in (0, 1025):
        with pytest.raises(_lib.DropClipError, match="1..1024 thresholds"):
            _lib.check(lib.dc_sweep_levels(p, count, p, p, ctypes.byref(n)))
        with pytest.raises(_lib.DropClipError, match="1..1024 thresholds"):  # checked before anything else is read
            _lib.check(lib.dc_predict_many_iou_sweep(None, 0, None, 0, 64, 1, None, None, None, None, None, None, None, 0,
                                                     None, None, 1, 0.1, 1, p, count, None, None, None, 0, None))
        assert lib.dc_predict_many_iou_sweep_workspace(0, None, None, None, 0, 0, count, 64, 0, 0) == 0
    with pytest.raises(_lib.DropClipError, match="null pointer"):
        _lib.check(lib.dc_predict_many_iou_sweep(None, 0, None, 0, 64, 1, None, None, None, None, None, None, None, 0,
                                                 None, None, 1, 0.1, 1, None, 3, None, None, None, 0, None))


def test_engine_predict_many_iou_sweep_host_checks():
    """FusionEngine.predict_many_iou_sweep checks the thresholds and every rule of predict_many_iou before anything
    reaches the device (the engine here has no library: any device work would raise AttributeError)."""
    eng = object.__new__(FusionEngine)
    x, t = torch.zeros(6, 64), torch.zeros(5, 64)
    lab = torch.zeros(6, dtype=torch.int32)
    P = _lib.DC_GROUND_PAIRED
    pos, negs, ids = [[0], [0]], [[[1]], [[1]]], [[[1]], [[2]]]
    sweep = FusionEngine.predict_many_iou_sweep
    for thr in ([], [0.5] * 1025):
        with pytest.raises(ValueError):
            sweep(eng, x, [4, 2], t, [3, 2], pos, negs, lab, ids, P, 0.1, True, thr)
    args = (P, 0.1, True, [0.5, 0.2])
    with pytest.raises(IndexError):  # scene 1's positive column outside its 2 prompts
        sweep(eng, x, [4, 2], t, [3, 2], [[0], [2]], negs, lab, ids, *args)
    with pytest.raises(ValueError):  # point counts do not sum to the rows
        sweep(eng, x, [4, 3], t, [3, 2], pos, negs, lab, ids, *args)
    with pytest.raises(ValueError):  # labels of another dtype
        sweep(eng, x, [4, 2], t, [3, 2], pos, negs, lab.float(), ids, *args)
    with pytest.raises(ValueError):  # an id outside int32
        sweep(eng, x, [4, 2], t, [3, 2], pos, negs, lab, [[[1]], [[2 ** 31]]], *args)
    with pytest.raises(AttributeError):  # every check passed: the next step is the library
        sweep(eng, x, [4, 2], t, [3, 2], pos, negs, lab, ids, P, 0.1, True, [0.5] * 1024)


def test_clip_predict_many_iou_sweep_checks_before_the_device():
    cs = object.__new__(ClipSimilarity)
    cs.method, cs.threshold, cs.norm_vis_feat = "paired", 0.7, True
    x, lab = torch.zeros(4, 64), torch.zeros(4, dtype=torch.int64)
    for thr in ([], [0.5] * 1025):
        with pytest.raises(ValueError):
            cs.predict_many_iou_sweep(x, [4], lab, [{"a": [1]}], thr)
    with pytest.raises(RuntimeError):  # CPU features: no CPU fallback
        cs.predict_many_iou_sweep(x, [4], lab, [{"a": [1]}], [0.5])


# ---------------------------------------------------------------------------------------------- GPU
def _loop(cs, feat, counts, labels, obj, thresholds, **kw):
    """One predict_many_iou per threshold, each on a fresh copy of the features: (inter, union) (T, sum Q) on the host."""
    rows = [cs.predict_many_iou(feat.clone(), counts, labels, obj, threshold=t, **kw) for t in thresholds]
    return torch.stack([r[0] for r in rows]).cpu(), torch.stack([r[1] for r in rows]).cpu()


def _check_sweep(cs, feat, counts, labels, obj, thresholds, **kw):
    x = feat.clone()
    inter, union = cs.predict_many_iou_sweep(x, counts, labels, obj, thresholds, **kw)
    n_q = sum(len(o) for o in obj)
    assert inter.shape == union.shape == (len(thresholds), n_q)
    assert inter.dtype == union.dtype == torch.int64 and inter.is_cuda and union.is_cuda
    want_i, want_u = _loop(cs, feat, counts, labels, obj, thresholds, **kw)
    assert torch.equal(inter.cpu(), want_i), f"{kw}: intersections differ"
    assert torch.equal(union.cpu(), want_u), f"{kw}: unions differ"
    return inter.cpu(), union.cpu()


@pytest.mark.gpu
@pytest.mark.parametrize("batch", list(BATCHES))
@pytest.mark.parametrize("dname,dim,lname", [("f16", 768, "i64"), ("f32", 768, "i32"), ("f16", 512, "i32"),
                                             ("f32", 512, "i64")])
def test_sweep_rows_equal_predict_many_iou(batch, dname, dim, lname):
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
                cs.predict_many_iou_sweep(x, counts, labels, obj, THRESHOLDS, qneg=qneg, method=method)
            assert torch.equal(x, feat)  # raised before any scene was normalised
            keep = [s for s, (n, q) in enumerate(shapes) if not (n == 1 and q)]
            rows, labs = _split(feat, counts), _split(labels, counts)
            args = (torch.cat([rows[s] for s in keep]).contiguous(), [counts[s] for s in keep],
                    torch.cat([labs[s] for s in keep]), [obj[s] for s in keep])
        else:
            args = (feat, counts, labels, obj)
        inter, union = _check_sweep(cs, *args, THRESHOLDS, qneg=qneg, method=method)
        if method == "argmax" and qneg is not None:  # the prediction does not depend on the threshold
            assert (inter == inter[0]).all() and (union == union[0]).all()


@pytest.mark.gpu
@pytest.mark.parametrize("n_thr", [1, 2, 101, 1024])
def test_sweep_threshold_counts(n_thr):
    cs = _cs(768, torch.float16)
    feat, counts, queries = _batch(cs, [(3000, 5), (129, 3), (0, 2), (700, 1)], 768, torch.float16, seed=n_thr)
    labels, obj = _ground_truth(counts, queries, torch.int64, seed=n_thr)
    rng = np.random.default_rng(n_thr)
    thr = np.round(rng.random(n_thr), 3).tolist()  # duplicates from T = 101 on
    thr[:min(n_thr, 4)] = [0.7, NAN, -INF, 0.0][:n_thr] if n_thr > 1 else [0.35]
    _check_sweep(cs, feat, counts, labels, obj, thr)


@pytest.mark.gpu
@pytest.mark.parametrize("dname", ["f16", "f32"])
def test_sweep_at_the_normalised_scores_themselves(dname):
    """Thresholds equal to normalised scores predict_many returns, so x > thr is decided at equality for some points."""
    dtype = torch.float32 if dname == "f32" else torch.float16
    cs = _cs(512, dtype)
    feat, counts, queries = _batch(cs, [(2000, 4), (500, 2)], 512, dtype, seed=13)
    labels, obj = _ground_truth(counts, queries, torch.int32, seed=13)
    res = cs.predict_many(feat.clone(), counts, queries)
    sims = torch.cat([s.reshape(-1) for _, s in res]).cpu().numpy()
    picked = np.random.default_rng(1).choice(sims, 40, replace=False).tolist() + [float(sims.max()), float(sims.min())]
    picked = [t for t in picked if t != 0.0]  # 0.0 would mean the default threshold
    inter, union = _check_sweep(cs, feat, counts, labels, obj, picked)
    assert int(union.sum()) > 0 and int(inter.sum()) > 0


@pytest.mark.gpu
def test_sweep_where_max_equals_min():
    """A scene whose rows are all equal: every score of its queries is the same, so min-max takes the x / max branch
    (x = 1); thresholds just below, at and above 1."""
    cs = _cs(768, torch.float16)
    feat, counts, queries = _batch(cs, [(300, 3), (1000, 2)], 768, torch.float16, seed=17)
    feat[:300] = feat[0]
    labels, obj = _ground_truth(counts, queries, torch.int64, seed=17)
    below = float(np.nextafter(np.float32(1), np.float32(0)))
    inter, union = _check_sweep(cs, feat, counts, labels, obj, [below, 1.0, 1.5, 0.5, -INF])
    # below 1 and -inf predict all 300 points of scene 0 (union 300), 1.0 and 1.5 none (inter 0)
    assert union[0, :3].tolist() == union[4, :3].tolist() == [300] * 3
    assert inter[1, :3].tolist() == inter[2, :3].tolist() == [0] * 3


@pytest.mark.gpu
@pytest.mark.parametrize("dname", ["f32", "f16"])
@pytest.mark.parametrize("norm", [True, False])
def test_sweep_normalises_in_place_like_one_predict_many_iou(dname, norm):
    dtype = torch.float32 if dname == "f32" else torch.float16
    cs = _cs(768, dtype, norm_vis_feat=norm)
    feat, counts, queries = _batch(cs, [(1000, 5), (300, 0), (2000, 3)], 768, dtype, seed=9)
    labels, obj = _ground_truth(counts, queries, torch.int64, seed=1)
    x1, x2 = feat.clone(), feat.clone()
    cs.predict_many_iou(x1, counts, labels, obj)
    cs.predict_many_iou_sweep(x2, counts, labels, obj, THRESHOLDS)
    assert torch.equal(x1, x2)
    assert torch.equal(_split(x2, counts)[1], _split(feat, counts)[1])  # no queries: untouched


@pytest.mark.gpu
def test_grounding_scores_per_row_equal_the_loop():
    cs = _cs(768, torch.float16, method="paired", threshold=0.7)
    feat, counts, queries = _batch(cs, [(4000, 6), (2500, 4), (3000, 5)], 768, torch.float16, seed=5)
    labels, obj = _ground_truth(counts, queries, torch.int64, seed=5)
    thresholds = [0.05 * i for i in range(1, 20)]
    inter, union = cs.predict_many_iou_sweep(feat.clone(), counts, labels, obj, thresholds)
    for t, thr in enumerate(thresholds):
        miou, prs = grounding_scores(*cs.predict_many_iou(feat.clone(), counts, labels, obj, threshold=thr))
        miou_t, prs_t = grounding_scores(inter[t], union[t])
        assert torch.equal(miou_t.cpu(), miou.cpu())
        assert [p.item() for p in prs_t] == [p.item() for p in prs]
    # and the single call agrees with binary_iou_counts over predict_many's rows
    res = cs.predict_many(feat.clone(), counts, queries, threshold=0.7)
    want_i, want_u = _expected(res, labels, counts, obj)
    t = thresholds.index(0.05 * 14)  # fp32(0.7000000000000001) == fp32(0.7)
    assert torch.equal(inter[t].cpu(), want_i) and torch.equal(union[t].cpu(), want_u)


@pytest.mark.gpu
def test_sweep_errors_before_any_row_changes():
    cs = _cs(768, torch.float16)
    feat, counts, queries = _batch(cs, [(500, 4), (1, 3), (200, 2)], 768, torch.float16, seed=21)
    labels, obj = _ground_truth(counts, queries, torch.int32, seed=2)

    def raises(exc, rows, *args, match=None, **kw):
        x = rows.clone()
        with pytest.raises(exc, match=match):
            cs.predict_many_iou_sweep(x, *args, **kw)
        assert torch.equal(x, rows)

    raises(ValueError, feat, counts, labels, obj, [])
    raises(ValueError, feat, counts, labels, obj, [0.5] * 1025)
    raises(IndexError, feat, counts, labels, obj, [0.5], method="argmax")  # a one-point scene with queries
    raises(ValueError, feat, counts, labels.float(), obj, [0.5])
    raises(ValueError, feat, counts, labels[:-1], obj, [0.5])
    raises(RuntimeError, feat, counts, labels.cpu(), obj, [0.5])
    raises(ValueError, feat, [500, 1, 199], labels, obj, [0.5])
    raises(RuntimeError, feat[:500], [500], labels[:500], [{f"q{i}": [1] for i in range(1537)}], [0.5], qneg=None,
           match="0..1536 prompts")
    x = feat.clone()
    assert cs.predict_many_iou_sweep(x, counts, labels, obj, [0.5], method="other") is None
    assert torch.equal(x, feat)


@pytest.mark.gpu
def test_sweep_edge_cases_and_workspace():
    cs = _cs(768, torch.float16)
    feat, counts, queries = _batch(cs, [(500, 4), (0, 3), (200, 0)], 768, torch.float16, seed=22)
    labels, obj = _ground_truth(counts, queries, torch.int64, seed=3)
    # S = 0, and no queries at all
    i, u = cs.predict_many_iou_sweep(feat[:0].clone(), [], labels[:0], [], [0.5, 0.2])
    assert i.shape == u.shape == (2, 0)
    i, u = cs.predict_many_iou_sweep(feat[:200].clone(), [200], labels[:200], [{}], [0.5])
    assert i.shape == u.shape == (1, 0)
    # every scene empty: 0 / 0 for each query and threshold
    i, u = cs.predict_many_iou_sweep(feat[:0].clone(), [0, 0], labels[:0], [{"a": [1], "b": [2, 3]}, {}], [0.5, NAN, 0.1])
    assert i.shape == (3, 2) and not i.any() and not u.any()
    # the empty scene's queries report 0 / 0 among the others
    i, u = _check_sweep(cs, feat, counts, labels, obj, THRESHOLDS)
    assert not i[:, 4:].any() and not u[:, 4:].any()
    # the workspace: dc_predict_many_iou's, plus 8 (T + 1) bytes of histograms per query and the two tables
    lib = _lib.load()
    c = lambda a: a.ctypes.data_as(ctypes.c_void_p)  # noqa: E731
    point_off, prompt_off, query_off = np.array([0, 500, 500, 700]), np.array([0, 4, 7, 7], np.int32), np.array(
        [0, 4, 7, 7], np.int32)
    tables = (3, c(point_off), c(prompt_off), c(query_off), 21, 9)
    base = lib.dc_predict_many_iou_workspace(*tables, 768, _lib.DC_F16, _lib.DC_F16)
    for n_thr in (1, 13, 1024):
        extra = lib.dc_predict_many_iou_sweep_workspace(*tables, n_thr, 768, _lib.DC_F16, _lib.DC_F16) - base
        hist = -(-8 * (n_thr + 1) * 7 // 256) * 256
        assert hist <= extra <= hist + -(-(8 * n_thr + 16) // 256) * 256


@pytest.mark.gpu
def test_sweep_on_a_side_stream():
    """Issued on a non-default stream behind a long kernel: the call returns while the stream is still busy (no host
    synchronisation inside it) and gives the default stream's counts, which equal the single calls'."""
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
    args = (pos, negs, labels, gt, _lib.DC_GROUND_PAIRED, 0.1, True)
    thr = [0.7, 0.2, 0.9, 0.2]
    want = eng.predict_many_iou_sweep(feats.clone(), counts, text, p_counts, *args, thr)
    for t, th in enumerate(thr):
        single = eng.predict_many_iou(feats.clone(), counts, text, p_counts, *args, th)
        assert torch.equal(want[0][t], single[0]) and torch.equal(want[1][t], single[1])
    torch.cuda.synchronize()
    side = torch.cuda.Stream()
    x = feats.clone()
    torch.cuda.synchronize()
    with torch.cuda.stream(side):
        torch.cuda._sleep(200_000_000)  # ~0.1 s of spinning ahead of the call
        got = eng.predict_many_iou_sweep(x, counts, text, p_counts, *args, thr)
        busy = not side.query()
    side.synchronize()
    assert busy, "predict_many_iou_sweep waited for the stream"
    assert torch.equal(want[0], got[0]) and torch.equal(want[1], got[1])
    assert int(want[1].sum()) > 0
