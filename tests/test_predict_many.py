"""ClipSimilarity.predict_many / FusionEngine.predict_many / dc_predict_many: every text query of a batch of scenes
grounded in one call. Scene s's result must equal what predict_queries returns for that scene alone."""
import numpy as np
import pytest
import torch

from dropclip_b200.similarity import ClipSimilarity, batch_query_columns, query_columns

GENERIC = ClipSimilarity.NEGATIVE_PROMPT_GENERIC
VARIANTS = [("paired", "scene"), ("paired", []), ("argmax", "scene"), ("argmax", []), ("paired", None)]


# ---------------------------------------------------------------------------------------------- prompt tables (CPU)
def test_batch_query_columns_dedupes_globally_and_keeps_scene_local_columns():
    scenes = [["a", "b"], [], ["b", "c", "b"], ["d"]]
    texts, gather, counts, pos, negs = batch_query_columns(scenes, "scene", GENERIC)
    assert texts == ["a", "b", "c", "d"] + GENERIC  # every distinct text once, in order of appearance
    assert counts == [2, 0, 2, 5]
    off = np.concatenate([[0], np.cumsum(counts)])
    for s, queries in enumerate(scenes):
        t_s, p_s, n_s = query_columns(queries, "scene", GENERIC)
        assert [texts[gather[j]] for j in range(off[s], off[s + 1])] == t_s  # the scene's own table
        assert pos[s] == p_s and negs[s] == n_s  # columns local to the scene's table
    assert pos[2] == [0, 1, 0] and negs[2] == [[1], [0, 0], [1]]
    assert pos[3] == [0] and negs[3] == [[1, 2, 3, 4]]  # generic negatives when the scene has no other text


def test_batch_query_columns_shared_list_and_none():
    texts, gather, counts, pos, negs = batch_query_columns([["a"], ["b", "x"]], ["x", "y"], GENERIC)
    assert texts == ["a", "x", "y", "b"] and counts == [3, 3]
    assert [texts[g] for g in gather] == ["a", "x", "y", "b", "x", "y"]
    assert pos == [[0], [0, 1]] and negs == [[[1, 2]], [[1, 2], [1, 2]]]
    texts, gather, counts, pos, negs = batch_query_columns([["a", "a"], []], None, GENERIC)
    assert texts == ["a"] and gather == [0] and counts == [1, 0] and pos == [[0, 0], []] and negs == [None, None]
    assert batch_query_columns([], "scene", GENERIC) == ([], [], [], [], [])


def test_engine_predict_many_host_checks():
    """FusionEngine.predict_many checks every index, count and mode rule before anything reaches the device."""
    from dropclip_b200 import _lib
    from dropclip_b200.engine import FusionEngine
    eng = object.__new__(FusionEngine)  # no engine, no GPU needed here
    x, t = torch.zeros(6, 64), torch.zeros(5, 64)
    P = _lib.DC_GROUND_PAIRED
    args = (0.1, True, 0.7)
    with pytest.raises(IndexError):  # scene 1's positive column outside its 2 prompts
        FusionEngine.predict_many(eng, x, [4, 2], t, [3, 2], [[0], [2]], [[[1]], [[0]]], P, *args)
    with pytest.raises(IndexError):  # scene 0's negative column outside its 3 prompts
        FusionEngine.predict_many(eng, x, [4, 2], t, [3, 2], [[0], [0]], [[[3]], [[1]]], P, *args)
    with pytest.raises(ValueError):  # paired needs a negative for every query
        FusionEngine.predict_many(eng, x, [4, 2], t, [3, 2], [[0, 1], [0]], [[[1], []], [[1]]], P, *args)
    with pytest.raises(ValueError):  # raw takes none
        FusionEngine.predict_many(eng, x, [4, 2], t, [3, 2], [[0], [0]], [[[1]], [[1]]], _lib.DC_GROUND_RAW, *args)
    with pytest.raises(ValueError):  # point counts do not sum to the rows
        FusionEngine.predict_many(eng, x, [4, 3], t, [3, 2], [[0], [0]], [[[1]], [[1]]], P, *args)
    with pytest.raises(ValueError):  # prompt counts do not sum to the prompt rows
        FusionEngine.predict_many(eng, x, [4, 2], t, [3, 3], [[0], [0]], [[[1]], [[1]]], P, *args)
    with pytest.raises(ValueError):  # one list per scene
        FusionEngine.predict_many(eng, x, [4, 2], t, [3, 2], [[0]], [[[1]]], P, *args)


def test_clip_predict_many_checks_before_the_device():
    cs = object.__new__(ClipSimilarity)
    cs.method, cs.threshold, cs.norm_vis_feat = "paired", 0.7, True
    with pytest.raises(RuntimeError):  # CPU features: no CPU fallback
        cs.predict_many(torch.zeros(4, 64), [4], [["a"]])


# ---------------------------------------------------------------------------------------------- GPU
class ExactNormTower:
    """encode_text = a fixed row per text; every row has 256 entries of +-1/16 and zeros elsewhere, so its norm is
    exactly 1 in any summation order. torch's row-norm reduction order depends on how many rows a tensor has, so the
    batch's one prompt table and a scene's own table would otherwise differ in the last bits; with these rows both
    calls see the same embeddings, the condition under which predict_many equals predict_queries."""

    def __init__(self, dim, dtype, vocab=4096, seed=17):
        rng = np.random.default_rng(seed)
        table = np.zeros((vocab, dim), dtype=np.float32)
        for r in range(vocab):
            table[r, rng.choice(dim, 256, replace=False)] = rng.choice([-1.0, 1.0], 256) / 16
        self.table = torch.from_numpy(table).to(dtype).cuda()
        self.ids = {}

    def tokenize(self, texts):
        texts = [texts] if isinstance(texts, str) else texts
        return torch.tensor([self.ids.setdefault(t, len(self.ids)) for t in texts], dtype=torch.long)

    def encode_text(self, tok):
        return self.table[tok.cuda()].clone()

    def eval(self):
        return self

    def to(self, *_):
        return self


def _cs(dim, dtype, **kw):
    tower = ExactNormTower(dim, dtype)
    return ClipSimilarity(model=tower, tokenize=tower.tokenize, device="cuda", **kw)


def _batch(cs, shapes, dim, dtype, seed):
    """Scenes (N_s, Q_s): rows near the scene's query embeddings plus noise, concatenated in scene order."""
    g = torch.Generator().manual_seed(seed)
    feats, queries = [], []
    for s, (n, q) in enumerate(shapes):
        qs = [f"scene {seed} {s} object {i}" for i in range(q)]
        f = 0.05 * torch.randn((n, dim), generator=g)
        if q and n:
            emb = cs.model.encode_text(cs._tok(qs)).float().cpu()
            owner = torch.randint(0, q + 1, (n,), generator=g)
            near = owner < q
            f[near] += 0.6 * emb[owner[near]]
        feats.append(f)
        queries.append(qs)
    return torch.cat(feats).to(dtype).cuda().contiguous(), [n for n, _ in shapes], queries


def _split(x, counts):
    return list(torch.split(x, counts))


BATCHES = {
    "s1": [(3000, 21)],
    "s3": [(127, 1), (0, 21), (129, 300)],  # 300 scene-negative prompts: two column blocks, ld widened for the batch
    "s16": [(128, 21), (129, 1), (0, 0), (3000, 21), (1, 21), (127, 21), (200_000, 21), (3000, 0),
            (128, 1), (129, 21), (0, 1), (3000, 21), (127, 1), (1, 1), (500, 40), (128, 21)],
}
WORST = {}


def _compare(cs, feat, counts, queries, method, qneg, thr=0.7):
    x = feat.clone()
    res = cs.predict_many(x, counts, queries, qneg=qneg, method=method, threshold=thr)
    assert len(res) == len(counts)
    worst = 0.0
    for s, (rows, n, qs) in enumerate(zip(_split(feat, counts), counts, queries)):
        xs = rows.clone()
        want = cs.predict_queries(xs, qs, qneg=qneg, method=method, threshold=thr)
        pred, sims = res[s]
        wp, ws = want
        assert sims.shape == ws.shape == (len(qs), n) and pred.shape == wp.shape
        assert sims.dtype == torch.float32 and pred.dtype == torch.bool
        assert torch.equal(_split(x, counts)[s], xs), f"scene {s}: rows normalised differently"
        if sims.numel():
            worst = max(worst, (sims - ws).abs().max().item())
            if method == "argmax" and qneg is not None:
                assert torch.equal(pred, wp), f"scene {s}"
            else:
                sure = (ws - thr).abs() > 1e-5
                assert torch.equal(pred[sure], wp[sure]), f"scene {s}"
    assert worst <= 1e-6, worst
    return worst


@pytest.mark.gpu
@pytest.mark.parametrize("batch", list(BATCHES))
@pytest.mark.parametrize("dname,dim", [("f16", 768), ("f32", 768), ("f16", 512), ("f32", 512)])
def test_predict_many_vs_predict_queries_per_scene(batch, dname, dim):
    dtype = torch.float32 if dname == "f32" else torch.float16
    cs = _cs(dim, dtype)
    shapes = BATCHES[batch]
    feat, counts, queries = _batch(cs, shapes, dim, dtype, seed=len(shapes) + dim)
    one_point = any(n == 1 and q for n, q in shapes)
    for method, qneg in VARIANTS:
        if method == "argmax" and qneg is not None and one_point:
            x = feat.clone()
            with pytest.raises(IndexError):
                cs.predict_many(x, counts, queries, qneg=qneg, method=method)
            assert torch.equal(x, feat)  # raised before any scene was normalised
            keep = [s for s, (n, q) in enumerate(shapes) if not (n == 1 and q)]
            rows = _split(feat, counts)
            sub = torch.cat([rows[s] for s in keep]).contiguous()
            w = _compare(cs, sub, [counts[s] for s in keep], [queries[s] for s in keep], method, qneg)
        else:
            w = _compare(cs, feat, counts, queries, method, qneg)
        WORST[(batch, dname, dim, method, str(qneg))] = w
    print(f"\n{batch} {dname} {dim}: largest score difference against predict_queries "
          f"{max(v for k, v in WORST.items() if k[:3] == (batch, dname, dim)):.3e}")


@pytest.mark.gpu
@pytest.mark.parametrize("dname", ["f32", "f16"])
def test_engine_predict_many_bit_equal_to_predict_queries(dname):
    """The embedding-level form on the same prompt rows: bit-equal scores and predictions, every mode."""
    from dropclip_b200 import _lib
    from dropclip_b200.engine import FusionEngine
    dtype = torch.float32 if dname == "f32" else torch.float16
    eng = FusionEngine("cuda")
    g = torch.Generator().manual_seed(8)
    counts, p_counts = [700, 0, 129, 5000], [6, 3, 280, 1]
    feats = torch.randn((sum(counts), 768), generator=g).to(dtype).cuda()
    text = torch.randn((sum(p_counts), 768), generator=g)
    text = (text / text.norm(dim=-1, keepdim=True)).to(dtype).cuda()
    pos = [[0, 2, 5], [1], list(range(0, 280, 7)), [0, 0]]
    negs = [[[1, 2], [0], [1, 3, 4, 1]], [[0, 2]], [[j for j in range(280) if j != p] for p in range(0, 280, 7)], [[0], [0]]]
    for mode in (_lib.DC_GROUND_PAIRED, _lib.DC_GROUND_ARGMAX, _lib.DC_GROUND_RAW):
        nl = None if mode == _lib.DC_GROUND_RAW else negs
        x = feats.clone()
        res = eng.predict_many(x, counts, text, p_counts, pos, nl, mode, 0.1, True, 0.6)
        rows, trows = _split(feats, counts), _split(text, p_counts)
        for s in range(len(counts)):
            xs = rows[s].clone()
            ws, wp = eng.predict_queries(xs, trows[s], pos[s], None if nl is None else nl[s], mode, 0.1, True, 0.6)
            score, pred = res[s]
            # bit patterns: scene 3's argmax query has its positive as its only negative, so both give 0 / 0 = NaN
            assert torch.equal(score.view(torch.int32), ws.view(torch.int32)) and torch.equal(pred, wp), f"mode {mode} scene {s}"
            assert torch.equal(_split(x, counts)[s], xs)


@pytest.mark.gpu
@pytest.mark.parametrize("dname", ["f32", "f16"])
@pytest.mark.parametrize("norm", [True, False])
def test_predict_many_normalises_in_place_like_predict_queries(dname, norm):
    dtype = torch.float32 if dname == "f32" else torch.float16
    cs = _cs(768, dtype, norm_vis_feat=norm)
    feat, counts, queries = _batch(cs, [(1000, 5), (300, 0), (2000, 3)], 768, dtype, seed=9)
    x1 = feat.clone()
    cs.predict_many(x1, counts, queries)
    x2 = [r.clone() for r in _split(feat, counts)]
    for xs, qs in zip(x2, queries):
        cs.predict_queries(xs, qs)
    assert torch.equal(x1, torch.cat(x2))
    assert torch.equal(_split(x1, counts)[1], _split(feat, counts)[1])  # no queries: untouched, as predict_queries
    if norm:
        assert not torch.equal(x1, feat)


@pytest.mark.gpu
@pytest.mark.parametrize("dname", ["f32", "f16"])
def test_predict_many_edge_cases(dname):
    dtype = torch.float32 if dname == "f32" else torch.float16
    cs = _cs(768, dtype)
    feat, counts, queries = _batch(cs, [(500, 4), (1, 3), (200, 2)], 768, dtype, seed=21)
    # S = 0
    assert cs.predict_many(feat[:0].clone(), [], []) == []
    # every scene empty: (Q_s, 0) and (0, N_s) shapes
    res = cs.predict_many(feat[:0].clone(), [0, 0], [["a", "b"], []])
    assert [tuple(p.shape) for p, _ in res] == [(2, 0), (0, 0)] and all(p.dtype == torch.bool for p, _ in res)
    res = cs.predict_many(feat[:3].clone(), [3], [[]])
    assert res[0][0].shape == (0, 3) and res[0][1].shape == (0, 3)
    # argmax with a one-point scene that has queries: IndexError, features bit-unchanged
    x = feat.clone()
    with pytest.raises(IndexError):
        cs.predict_many(x, counts, queries, method="argmax")
    assert torch.equal(x, feat)
    # ... but a one-point scene without queries is fine
    res = cs.predict_many(feat[:501].clone(), [500, 1], [queries[0], []], method="argmax")
    assert res[1][0].shape == (0, 1)
    # unknown method: None per scene, features untouched
    x = feat.clone()
    assert cs.predict_many(x, counts, queries, method="other") == [None] * 3
    assert torch.equal(x, feat)
    # CPU and non-contiguous features: RuntimeError; counts that do not sum to the rows: ValueError
    with pytest.raises(RuntimeError):
        cs.predict_many(feat.cpu(), counts, queries)
    with pytest.raises(RuntimeError):
        cs.predict_many(feat[:, :128].repeat(1, 2).t(), [256], [["a"]])
    x = feat.clone()
    with pytest.raises(ValueError):
        cs.predict_many(x, [500, 1, 199], queries)
    assert torch.equal(x, feat)
    # more than 1536 prompts in one scene: the library's error
    many = [f"q{i}" for i in range(1537)]
    with pytest.raises(RuntimeError, match="0..1536 prompts"):
        cs.predict_many(feat[:500].clone(), [500], [many], qneg=None)


@pytest.mark.gpu
@pytest.mark.parametrize("dname", ["f32", "f16"])
def test_predict_many_vs_cpu_oracle(dname):
    from oracle import similarity_ref
    dtype = torch.float32 if dname == "f32" else torch.float16
    cs = _cs(768, dtype)
    feat, counts, queries = _batch(cs, [(700, 5), (0, 2), (1500, 21), (129, 1)], 768, dtype, seed=3)
    tol = dict(rtol=1e-3, atol=1e-5) if dname == "f32" else dict(rtol=0, atol=6e-3)
    for method, qneg in VARIANTS:
        res = cs.predict_many(feat.clone(), counts, queries, qneg=qneg, method=method, threshold=0.7)
        for s, (rows, qs) in enumerate(zip(_split(feat, counts), queries)):
            if not rows.shape[0]:
                continue
            for q, t in enumerate(qs):
                negs = None if qneg is None else ([x for x in qs if x != t] if qneg == "scene" else qneg) or GENERIC
                qp = cs.model.encode_text(cs._tok([t])).cpu()
                qn = None if negs is None else cs.model.encode_text(cs._tok(negs)).cpu()
                vis = rows.cpu().clone() if dname == "f32" else rows.cpu().float()
                _, ws = similarity_ref.predict_from_embeds(vis, qp.float(), None if qn is None else qn.float(),
                                                           method=method, threshold=0.7)
                np.testing.assert_allclose(res[s][1][q].cpu().numpy(), ws.numpy().reshape(-1), **tol,
                                           err_msg=f"{method} {qneg} scene {s} query {q}")


@pytest.mark.gpu
@pytest.mark.parametrize("negatives_mode", ["scene", "generic"])
def test_validation_loop_through_predict_many(negatives_mode):
    """validate_grounding's loop (tools/validate_upper_bound.py:200-220) over a batch of 4 scenes: the per-scene,
    per-query predict loop feeding trainMetricPC against one predict_many per batch."""
    from dropclip_b200.metrics import trainMetricPC
    cs = _cs(768, torch.float16, method="paired", threshold=0.7)
    rng = np.random.default_rng(5)
    outputs, labels, scene_queries = [], [], []
    for s, n in enumerate([4000, 2500, 3000, 1000]):
        obj_queries = {f"scene {s} object {i}": [i + 1] for i in range(3 + s)}
        emb = cs.model.encode_text(cs._tok(list(obj_queries))).float().cpu()
        label = torch.from_numpy(rng.integers(0, len(obj_queries) + 1, size=n))
        out = torch.zeros((n, 768))
        for i in range(len(obj_queries)):
            out[label == i + 1] = emb[i]
        out += 0.03 * torch.from_numpy(rng.standard_normal((n, 768)).astype(np.float32))
        outputs.append(out)
        labels.append(label.cuda())
        scene_queries.append(obj_queries)
    pred_list, gt_list = [], []
    for out, label_d, obj_queries in zip(outputs, labels, scene_queries):
        output_d = out.cuda()
        for text_query, obj_ids in obj_queries.items():
            negatives = [] if negatives_mode == "generic" else [x for x in obj_queries if x != text_query]
            pred, _ = cs.predict(output_d.half(), text_query, negatives)
            gt = torch.zeros_like(label_d)
            for obj in obj_ids:
                gt[label_d == obj] = True
            pred_list.append(pred)
            gt_list.append(gt)
    iou, prs = trainMetricPC(pred_list, gt_list, pr_ious=[0.25, 0.5, 0.75], sigmoid=False)
    batch = torch.cat(outputs).cuda().half()
    res = cs.predict_many(batch, [o.shape[0] for o in outputs], [list(q) for q in scene_queries],
                          "scene" if negatives_mode == "scene" else [])
    pred_list2 = [row for pred, _ in res for row in pred]
    iou2, prs2 = trainMetricPC(pred_list2, gt_list, pr_ious=[0.25, 0.5, 0.75], sigmoid=False)
    assert abs(float(iou) - float(iou2)) < 1e-3 and float(iou) > 0.5
    assert [float(p) for p in prs] == [float(p) for p in prs2]


@pytest.mark.gpu
def test_predict_many_on_a_side_stream():
    """Issued on a non-default stream behind a long kernel: the call returns while the stream is still busy (no host
    synchronisation inside it) and gives the default stream's results."""
    from dropclip_b200 import _lib
    from dropclip_b200.engine import FusionEngine
    eng = FusionEngine("cuda")
    g = torch.Generator().manual_seed(2)
    counts, p_counts = [3000, 129, 10_000], [5, 21, 3]
    feats = torch.randn((sum(counts), 768), generator=g).half().cuda()
    text = torch.randn((sum(p_counts), 768), generator=g)
    text = (text / text.norm(dim=-1, keepdim=True)).half().cuda()
    pos = [[0, 1, 2], list(range(21)), [2]]
    negs = [[[3, 4]] * 3, [[j for j in range(21) if j != i] for i in range(21)], [[0, 1]]]
    want = eng.predict_many(feats.clone(), counts, text, p_counts, pos, negs, _lib.DC_GROUND_PAIRED, 0.1, True, 0.7)
    torch.cuda.synchronize()
    side = torch.cuda.Stream()
    x = feats.clone()
    torch.cuda.synchronize()
    with torch.cuda.stream(side):
        torch.cuda._sleep(200_000_000)  # ~0.1 s of spinning ahead of the call
        got = eng.predict_many(x, counts, text, p_counts, pos, negs, _lib.DC_GROUND_PAIRED, 0.1, True, 0.7)
        busy = not side.query()
    side.synchronize()
    assert busy, "predict_many waited for the stream"
    for (ws, wp), (gs, gp) in zip(want, got):
        assert torch.equal(ws, gs) and torch.equal(wp, gp)
