"""ClipSimilarity.predict_queries / FusionEngine.predict_queries / dc_predict_queries: every text query of a scene
grounded from one similarity GEMM. Row q must equal what ClipSimilarity.predict returns for query q alone."""
import numpy as np
import pytest
import torch

from dropclip_b200.similarity import ClipSimilarity, query_columns

GENERIC = ClipSimilarity.NEGATIVE_PROMPT_GENERIC


# ---------------------------------------------------------------------------------------------- column table (CPU)
def test_query_columns_dedupes_texts_in_order_of_appearance():
    texts, pos, negs = query_columns(["a", "b", "a", "c"], None, GENERIC)
    assert texts == ["a", "b", "c"] and pos == [0, 1, 0, 2] and negs is None


def test_query_columns_scene_negatives_are_the_other_query_texts():
    queries = ["a", "b", "a", "c"]
    texts, pos, negs = query_columns(queries, "scene", GENERIC)
    assert texts == ["a", "b", "c"] and pos == [0, 1, 0, 2]
    for q, t in enumerate(queries):
        assert [texts[j] for j in negs[q]] == [x for x in queries if x != t]  # repeats kept, as the reference encodes them
    assert negs == [[1, 2], [0, 0, 2], [1, 2], [0, 1, 0]]


def test_query_columns_shared_list_and_generic():
    texts, pos, negs = query_columns(["a", "b"], ["x", "a", "y"], GENERIC)
    assert texts == ["a", "b", "x", "y"] and pos == [0, 1] and negs == [[2, 0, 3], [2, 0, 3]]
    texts, pos, negs = query_columns(["a", "b"], [], GENERIC)
    assert texts == ["a", "b"] + GENERIC and negs == [[2, 3, 4, 5]] * 2


def test_query_columns_scene_without_other_texts_falls_back_to_generic():
    for queries in (["a"], ["a", "a"]):
        texts, pos, negs = query_columns(queries, "scene", GENERIC)
        assert texts == ["a"] + GENERIC and pos == [0] * len(queries) and negs == [[1, 2, 3, 4]] * len(queries)


def test_query_columns_rejects_other_qneg():
    with pytest.raises(AssertionError):
        query_columns(["a"], "all", GENERIC)
    with pytest.raises(AssertionError):
        query_columns(["a"], ("b",), GENERIC)


def test_engine_query_csr_and_index_range_checks():
    from dropclip_b200.engine import FusionEngine, query_csr
    pos, off, cols = query_csr([0, 2], [[1, 2], [0]], 3)
    assert pos.dtype == off.dtype == cols.dtype == np.int32
    assert pos.tolist() == [0, 2] and off.tolist() == [0, 2, 3] and cols.tolist() == [1, 2, 0]
    pos, off, cols = query_csr([1], None, 2)
    assert off.tolist() == [0, 0] and cols.size == 0
    for p, n in (([3], [[0]]), ([-1], [[0]]), ([0], [[3]]), ([0], [[-1]])):
        with pytest.raises(IndexError):
            query_csr(p, n, 3)
    with pytest.raises(ValueError):
        query_csr([0, 1], [[2]], 3)
    # FusionEngine.predict_queries checks before anything reaches the device (no engine, no GPU needed here)
    from dropclip_b200 import _lib
    eng = object.__new__(FusionEngine)
    x, t = torch.zeros(4, 64), torch.zeros(3, 64)
    with pytest.raises(IndexError):
        FusionEngine.predict_queries(eng, x, t, [3], [[0]], _lib.DC_GROUND_PAIRED, 0.1, True, 0.7)
    with pytest.raises(IndexError):
        FusionEngine.predict_queries(eng, x, t, [0], [[1, 7]], _lib.DC_GROUND_PAIRED, 0.1, True, 0.7)
    with pytest.raises(ValueError):
        FusionEngine.predict_queries(eng, x, t, [0, 1], [[1], []], _lib.DC_GROUND_PAIRED, 0.1, True, 0.7)
    with pytest.raises(ValueError):
        FusionEngine.predict_queries(eng, x, t, [0], [[1]], _lib.DC_GROUND_RAW, 0.1, True, 0.7)


# ---------------------------------------------------------------------------------------------- GPU
def _cs(dim, dtype, **kw):
    from tests.test_gpu_parity import make_cs
    return make_cs(dim, dtype, **kw)


def _flat(t):
    return t.reshape(-1).cpu().numpy()


@pytest.mark.gpu
@pytest.mark.parametrize("case", [("g0", 11, 3000, 768, 4), ("g1", 12, 2000, 512, 31), ("g2", 13, 1, 768, 4)])
@pytest.mark.parametrize("dname", ["f32", "f16"])
def test_predict_queries_vs_reference_golden(case, dname):
    """test_grounding_vs_reference_golden's cases, bars and pred bands through predict_queries with one query."""
    from tests import golden_io as gio
    from tests.test_oracle_golden import ground_inputs
    name, seed, n, dim, nneg = case
    dtype = torch.float32 if dname == "f32" else torch.float16
    g = gio.load("ground.npz")
    feat, emb, prompts, _ = ground_inputs(name, seed, n, dim, nneg, dtype)
    cs = _cs(dim, dtype)
    tol = dict(rtol=1e-3, atol=1e-5) if dname == "f32" else dict(rtol=0, atol=6e-3)
    for method in ("paired", "argmax"):
        x = feat.clone().cuda()
        if n == 1 and method == "argmax":
            with pytest.raises(IndexError):
                cs.predict_queries(x, [prompts[0]], qneg=prompts[1:], method=method)
            continue
        pred, sims = cs.predict_queries(x, [prompts[0]], qneg=prompts[1:], method=method, threshold=0.7)
        assert sims.shape == (1, n) and pred.shape == (1, n)
        assert sims.dtype == torch.float32 and pred.dtype == torch.bool
        want = g[f"{name}_{dname}_{method}_sims"]
        np.testing.assert_allclose(_flat(sims[0]), want, **tol)
        gold_pred = gio.unpack(g[f"{name}_{dname}_{method}_pred"], n).astype(bool)
        if method == "paired":
            sure = np.abs(want - 0.7) > (1e-3 if dname == "f32" else 2e-2)
            assert np.array_equal(_flat(pred[0])[sure], gold_pred[sure])
        elif dname == "f32":
            assert (_flat(pred[0]) != gold_pred).mean() < 2e-3
        if name == "g0" and method == "paired":
            np.testing.assert_allclose(x[:8].float().cpu().numpy(), g[f"{name}_{dname}_normed_head"],
                                       rtol=1e-6 if dname == "f32" else 1e-3)
    x = feat.clone().cuda()
    pred, sims = cs.predict_queries(x, [prompts[0]], qneg=None, threshold=0.7)
    np.testing.assert_allclose(_flat(sims[0]), g[f"{name}_{dname}_noneg_sims"], **tol)
    x = feat.clone().cuda()
    pred, sims = cs.predict_queries(x, [prompts[0]], qneg=[], method="paired")
    np.testing.assert_allclose(_flat(sims[0]), g[f"{name}_{dname}_generic_sims"], **tol)


def _scene(q, n, dim, dtype, seed):
    """n points of which a share lies near each of q query embeddings (fake text tower), plus noise."""
    from oracle import ref_shim
    rng = np.random.default_rng(seed)
    queries = [f"object {seed} {i}" for i in range(q)]
    emb = ref_shim.FakeTextTower(dim, dtype).encode_text(ref_shim.fake_tokenize(queries)).float()
    emb /= emb.norm(dim=-1, keepdim=True)
    owner = torch.from_numpy(rng.integers(0, q + 1, size=n))
    feat = 0.05 * torch.from_numpy(rng.standard_normal((n, dim)).astype(np.float32))
    near = owner < q
    feat[near] += 0.6 * emb[owner[near]]
    return feat.to(dtype), queries


def _negatives(queries, q, qneg):
    if qneg == "scene":
        return [x for x in queries if x != queries[q]]
    return qneg


VARIANTS = [("paired", "scene"), ("paired", []), ("argmax", "scene"), ("argmax", []), ("paired", None)]


def _check_rows_vs_predict(cs, feat, queries, method, qneg, thr=0.7):
    """Every row of predict_queries against predict on a clone; returns the normalised features."""
    x = feat.clone().cuda()
    pred, sims = cs.predict_queries(x, queries, qneg=qneg, method=method, threshold=thr)
    n = feat.shape[0]
    assert sims.shape == (len(queries), n) and pred.shape == (len(queries), n)
    assert sims.dtype == torch.float32 and pred.dtype == torch.bool
    text = None
    for q, t in enumerate(queries):
        xq = feat.clone().cuda()
        negs = _negatives(queries, q, qneg)
        wp, ws = cs.predict(xq, t, negs, method=method, threshold=thr)
        np.testing.assert_allclose(_flat(sims[q]), _flat(ws), rtol=0, atol=1e-5, err_msg=f"query {q}")
        got_p, want_p = _flat(pred[q]), _flat(wp)
        if method == "argmax" and negs is not None:
            # decided by S_pos >= max S_neg: compare wherever the margin exceeds 1e-6
            texts = [t] + (negs if negs else list(cs.NEGATIVE_PROMPT_GENERIC))
            emb = cs.model.encode_text(cs._tok(texts)).float()
            emb /= emb.norm(dim=-1, keepdim=True)
            s = xq.float() @ emb.T
            margin = (s[:, 0] - s[:, 1:].max(1).values).abs().cpu().numpy()
            sure = margin > 1e-6
        else:
            sure = np.abs(_flat(ws) - thr) > 1e-4
        assert np.array_equal(got_p[sure], want_p[sure]), f"query {q}"
    return x


@pytest.mark.gpu
@pytest.mark.parametrize("q", [2, 21, 300])
@pytest.mark.parametrize("dname,dim", [("f16", 768), ("f32", 768), ("f16", 512), ("f32", 512)])
def test_predict_queries_vs_per_query_predict(q, dname, dim):
    """Q = 300 crosses the GEMM's 256-column blocks (scene negatives: 300 distinct prompts)."""
    dtype = torch.float32 if dname == "f32" else torch.float16
    n = 3000 if q < 300 else 1200
    feat, queries = _scene(q, n, dim, dtype, seed=q + dim)
    cs = _cs(dim, dtype)
    for method, qneg in VARIANTS:
        _check_rows_vs_predict(cs, feat, queries, method, qneg)


@pytest.mark.gpu
@pytest.mark.parametrize("dname", ["f32", "f16"])
def test_predict_queries_vs_cpu_oracle(dname):
    from oracle import ref_shim, similarity_ref
    dtype = torch.float32 if dname == "f32" else torch.float16
    dim, n = 768, 2000
    feat, queries = _scene(21, n, dim, dtype, seed=3)
    cs = _cs(dim, dtype)
    tower = ref_shim.FakeTextTower(dim, dtype)
    tol = dict(rtol=1e-3, atol=1e-5) if dname == "f32" else dict(rtol=0, atol=6e-3)
    for method, qneg in VARIANTS:
        pred, sims = cs.predict_queries(feat.clone().cuda(), queries, qneg=qneg, method=method, threshold=0.7)
        for q, t in enumerate(queries):
            negs = _negatives(queries, q, qneg)
            qp = tower.encode_text(ref_shim.fake_tokenize(t))
            qn = None if negs is None else tower.encode_text(ref_shim.fake_tokenize(negs if negs else GENERIC))
            vis = feat.clone() if dname == "f32" else feat.float()  # fp16 replay in fp32, as the install test does
            wp, ws = similarity_ref.predict_from_embeds(vis, qp.float(), None if qn is None else qn.float(),
                                                        method=method, threshold=0.7)
            np.testing.assert_allclose(_flat(sims[q]), ws.numpy().reshape(-1), **tol, err_msg=f"{method} {qneg} query {q}")


@pytest.mark.gpu
@pytest.mark.parametrize("dname", ["f32", "f16"])
@pytest.mark.parametrize("norm", [True, False])
def test_predict_queries_normalises_in_place_once(dname, norm):
    dtype = torch.float32 if dname == "f32" else torch.float16
    feat, queries = _scene(5, 1000, 768, dtype, seed=9)
    cs = _cs(768, dtype, norm_vis_feat=norm)
    x1, x2 = feat.clone().cuda(), feat.clone().cuda()
    cs.predict_queries(x1, queries)
    cs.predict(x2, queries[0], queries[1:])
    assert torch.equal(x1, x2)
    if norm:
        assert not torch.equal(x1.cpu(), feat)


@pytest.mark.gpu
@pytest.mark.parametrize("dname", ["f32", "f16"])
def test_predict_queries_edge_cases(dname):
    dtype = torch.float32 if dname == "f32" else torch.float16
    feat, queries = _scene(4, 500, 768, dtype, seed=21)
    cs = _cs(768, dtype)
    # one point: (Q, 1) rows equal predict's 0-d results; argmax raises IndexError like predict
    for qneg in ("scene", [], None):
        pred, sims = cs.predict_queries(feat[:1].clone().cuda(), queries, qneg=qneg)
        assert sims.shape == (4, 1) and pred.shape == (4, 1)
        for q in range(4):
            wp, ws = cs.predict(feat[:1].clone().cuda(), queries[q], _negatives(queries, q, qneg))
            assert abs(sims[q, 0].item() - ws.item()) <= 1e-5 and pred[q, 0].item() == wp.item()
    with pytest.raises(IndexError):
        cs.predict_queries(feat[:1].clone().cuda(), queries, method="argmax")
    # no points
    for method in ("paired", "argmax"):
        pred, sims = cs.predict_queries(feat[:0].clone().cuda(), queries, method=method)
        assert sims.shape == (4, 0) and pred.shape == (4, 0) and pred.dtype == torch.bool
    # constant features: max == min, the v / max branch
    const = feat[:1].repeat(300, 1).contiguous()
    for method, qneg in VARIANTS:
        _check_rows_vs_predict(cs, const, queries, method, qneg)
    # a single query (scene: generic negatives) and repeated query texts
    for method, qneg in VARIANTS:
        _check_rows_vs_predict(cs, feat, queries[:1], method, qneg)
        _check_rows_vs_predict(cs, feat, [queries[0], queries[1], queries[0], queries[0]], method, qneg)
        _check_rows_vs_predict(cs, feat, [queries[2]] * 3, method, qneg)
    # a method predict does not know: None, like predict; features untouched
    x = feat.clone().cuda()
    assert cs.predict_queries(x, queries, method="other") is None
    assert torch.equal(x.cpu(), feat)
    # CPU and non-contiguous features: RuntimeError (no CPU fallback)
    with pytest.raises(RuntimeError):
        cs.predict_queries(feat.clone(), queries)
    with pytest.raises(RuntimeError):
        cs.predict_queries(feat.clone().cuda().t(), queries)


@pytest.mark.gpu
@pytest.mark.parametrize("negatives_mode", ["scene", "generic"])
def test_validation_loop_through_predict_queries(negatives_mode):
    """The loop body of validate_grounding (tools/validate_upper_bound.py:200-220) per query, against one
    predict_queries call per scene feeding trainMetricPC: same IoU and Pr@k."""
    from dropclip_b200.metrics import trainMetricPC
    from oracle import ref_shim
    tower = ref_shim.FakeTextTower(768, torch.float16)
    cs = _cs(768, torch.float16, method="paired", threshold=0.7)
    rng = np.random.default_rng(5)
    obj_queries = {f"a photo of object {i}": [i + 1] for i in range(6)}
    emb = tower.encode_text(ref_shim.fake_tokenize(list(obj_queries))).float()
    emb /= emb.norm(dim=-1, keepdim=True)
    n = 4000
    label = torch.from_numpy(rng.integers(0, 7, size=n))
    output = torch.zeros((n, 768))
    for i in range(6):
        output[label == i + 1] = emb[i]
    output += 0.03 * torch.from_numpy(rng.standard_normal((n, 768)).astype(np.float32))
    output_d, label_d = output.cuda(), label.cuda()
    pred_list, sims_list, gt_list = [], [], []
    for text_query, obj_ids in obj_queries.items():
        negatives = [] if negatives_mode == "generic" else [x for x in list(obj_queries.keys()) if x != text_query]
        pred, sims_norm = cs.predict(output_d.half(), text_query, negatives)
        gt = torch.zeros_like(label_d, device=label_d.device)
        for obj in obj_ids:
            gt[label_d == obj] = True
        pred_list.append(pred)
        sims_list.append(sims_norm)
        gt_list.append(gt)
    iou, prs = trainMetricPC(pred_list, gt_list, pr_ious=[0.25, 0.5, 0.75], sigmoid=False)
    # the same loop as one call per scene
    pred, sims = cs.predict_queries(output_d.half(), list(obj_queries), "scene" if negatives_mode == "scene" else [])
    for q in range(len(obj_queries)):
        np.testing.assert_allclose(_flat(sims[q]), _flat(sims_list[q]), rtol=0, atol=1e-5)
        sure = np.abs(_flat(sims_list[q]) - 0.7) > 1e-4
        assert np.array_equal(_flat(pred[q])[sure], _flat(pred_list[q])[sure])
    iou2, prs2 = trainMetricPC(list(pred), gt_list, pr_ious=[0.25, 0.5, 0.75], sigmoid=False)
    assert abs(float(iou) - float(iou2)) < 1e-3 and float(iou) > 0.5
    assert [float(p) for p in prs] == [float(p) for p in prs2]


@pytest.mark.gpu
def test_engine_predict_queries_with_ablation_tables():
    """benchmarks/ablation.py's grounding tables: positives = the objects present in the scene, negatives = every other
    object except the table (object 0). Each row equals FusionEngine.predict for that object."""
    from dropclip_b200 import _lib
    from dropclip_b200.engine import FusionEngine
    eng = FusionEngine("cuda")
    n_objects, n, dim = 12, 5000, 768
    g = torch.Generator().manual_seed(4)
    q = torch.randn((n_objects, dim), generator=g)
    q /= q.norm(dim=-1, keepdim=True)
    labels = torch.randint(0, n_objects - 2, (n,), generator=g)  # the last two objects are absent
    feats = (q[labels] + 0.1 * torch.randn((n, dim), generator=g)).half().cuda()
    qd = q.cuda()
    present = [int(k) for k in torch.unique(labels).tolist() if k > 0]
    negs = [[j for j in range(1, n_objects) if j != k] for k in present]
    for mode in (_lib.DC_GROUND_PAIRED, _lib.DC_GROUND_ARGMAX):
        score, pred = eng.predict_queries(feats.clone(), qd, present, negs, mode, 0.1, True, 0.6)
        assert score.shape == (len(present), n) and pred.shape == (len(present), n) and pred.dtype == torch.uint8
        for i, k in enumerate(present):
            text = torch.cat([qd[k:k + 1], qd[negs[i]]])
            ws, wp = eng.predict(feats.clone(), text, mode, 0.1, True, 0.6)
            np.testing.assert_allclose(score[i].cpu().numpy(), ws.cpu().numpy(), rtol=0, atol=1e-5)
            if mode == _lib.DC_GROUND_PAIRED:
                sure = (ws - 0.6).abs().cpu().numpy() > 1e-4
            else:
                xn = feats.clone()
                xn = (xn.float() / xn.float().norm(dim=-1, keepdim=True)).half().float()
                s = xn @ text.T
                sure = (s[:, 0] - s[:, 1:].max(1).values).abs().cpu().numpy() > 1e-6
            assert np.array_equal(pred[i].cpu().numpy()[sure], wp.cpu().numpy()[sure])
