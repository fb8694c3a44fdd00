"""Drop-in for the reference's `models/similarity.py` (class ClipSimilarity).

Same constructor, class constants, method names, argument defaults and quirks (q15-q20): `x or
self.x` defaulting, in-place normalisation of `vis_feats`, `.squeeze()`-shaped results. The text
tower stays whatever CLIP model the caller loads (out of scope, SURVEY.md §2 #8); everything after
`encode_text` - the point x prompt GEMM, paired softmax, min-max, threshold - runs in libdropclip's
tcgen05 kernel with a fused epilogue, so the (N x P) similarity matrix is never written unless
`compute_similarity` is asked for it.

Reference lines mirrored: models/similarity.py:1-101.
"""
from __future__ import annotations

import torch

from . import _lib
from .engine import FusionEngine, threshold_table

DEVICE = torch.device("cuda")  # the reference's expression always evaluates to 'cuda' (quirk q20)


def query_columns(queries, qneg, generic):
    """The prompt table of ClipSimilarity.predict_queries: (texts, pos, neg_lists). `texts` holds every distinct text
    once (queries first, in order of appearance); query q's positive prompt is texts[pos[q]] and its negatives are
    texts[j] for j in neg_lists[q], in the order predict(vis_feats, queries[q], qneg_q) would encode them:
      qneg == "scene": qneg_q = [x for x in queries if x != queries[q]] (the reference's evaluation loops), `generic`
                       when that is empty;
      qneg a list:     the same negatives for every query, `generic` for [];
      qneg None:       no negatives, neg_lists is None."""
    texts, col = [], {}

    def column(t):
        if t not in col:
            col[t] = len(texts)
            texts.append(t)
        return col[t]

    pos = [column(t) for t in queries]
    if qneg is None:
        return texts, pos, None
    if isinstance(qneg, str) and qneg == "scene":
        per_query = [[x for x in queries if x != t] or list(generic) for t in queries]
    else:
        assert isinstance(qneg, list), "qneg argument should be list or None"
        shared = list(qneg) if len(qneg) else list(generic)
        per_query = [shared] * len(queries)
    return texts, pos, [[column(x) for x in negs] for negs in per_query]


def batch_query_columns(scene_queries, qneg, generic):
    """The prompt tables of ClipSimilarity.predict_many: (texts, gather, prompt_counts, pos, neg_lists). Scene s gets
    the table query_columns(scene_queries[s], qneg, generic) = (texts_s, pos[s], neg_lists[s]), with pos[s] and
    neg_lists[s] local to it; `texts` holds every distinct text of the batch once, in order of appearance, and the
    scene tables one after the other are texts[gather[j]] (scene s: prompt_counts[s] = len(texts_s) entries). So one
    encode_text of `texts` and one index_select with `gather` give every scene its prompt rows."""
    texts, col = [], {}
    gather, prompt_counts, pos, neg_lists = [], [], [], []
    for queries in scene_queries:
        texts_s, pos_s, negs_s = query_columns(list(queries), qneg, generic)
        for t in texts_s:
            if t not in col:
                col[t] = len(texts)
                texts.append(t)
        gather += [col[t] for t in texts_s]
        prompt_counts.append(len(texts_s))
        pos.append(pos_s)
        neg_lists.append(negs_s)
    return texts, gather, prompt_counts, pos, neg_lists



def _load_clip(model_name, device):
    """The reference imports its vendored CLIP (`models.features.clip`); use it when importable."""
    try:
        from models.features.clip import clip  # the reference tree on sys.path
    except Exception as exc:  # pragma: no cover - depends on the caller's environment
        raise ImportError(
            "ClipSimilarity needs the CLIP text tower of the host application "
            "(`models.features.clip`); pass `model=` / `tokenize=` to use another encoder") from exc
    model, _ = clip.load(model_name, device=device)
    return model, clip.tokenize


class ClipSimilarity(object):

    NEGATIVE_PROMPT_GENERIC = ["object", "thing", "texture", "stuff"]
    SOFTMAX_TEMP = 0.1

    def __init__(self, model_name="ViT-L/14@336px", method="paired", threshold=0.7, norm_vis_feat=True, device=DEVICE,
                 model=None, tokenize=None):
        self.device = device
        self.threshold = threshold
        self.method = method
        self.norm_vis_feat = norm_vis_feat
        if model is None:
            model, tokenize = _load_clip(model_name, device)
            print(f"Loaded CLIP model {model_name}")
        self.model = model.eval().to(device)
        self.tokenize = tokenize
        self._engine = None

    # ------------------------------------------------------------------ helpers
    def _eng(self) -> FusionEngine:
        if getattr(self, "_engine", None) is None:
            self._engine = FusionEngine(self.device)
        return self._engine

    def _tok(self, text):
        tok = getattr(self, "tokenize", None)
        if tok is None:
            from models.features.clip import clip
            tok = clip.tokenize
        return tok(text)

    def _encode(self, qpos, qneg):
        """models/similarity.py:33-45: tokenise, encode, L2-normalise (tiny P x C tensors)."""
        qp = self.model.encode_text(self._tok(qpos).to(self.device))
        qp /= qp.norm(dim=-1, keepdim=True)
        if qneg is None:
            return qp, None
        assert isinstance(qneg, list), "qneg argument should be list or None"
        if not len(qneg):
            qneg = self.NEGATIVE_PROMPT_GENERIC
        qn = self.model.encode_text(self._tok(qneg).to(self.device))
        qn /= qn.norm(dim=-1, keepdim=True)
        return qp, qn

    def _check_feats(self, x):
        if not (isinstance(x, torch.Tensor) and x.is_cuda):
            raise RuntimeError("dropclip_b200 grounding needs CUDA feature tensors; there is no CPU fallback")
        if x.dtype not in (torch.float16, torch.float32) or x.dim() != 2 or not x.is_contiguous():
            raise RuntimeError("vis_feats must be a contiguous (N, C) fp16 or fp32 tensor")

    # ------------------------------------------------------------------ a15
    @torch.no_grad()
    def compute_similarity(self, vis_feat_norm, qpos, qneg=None, softmax_temp=None, method="paired"):
        softmax_temp = softmax_temp or self.SOFTMAX_TEMP
        self._check_feats(vis_feat_norm)
        qp, qn = self._encode(qpos, qneg)
        eng = self._eng()
        text = qp if qn is None else torch.cat([qp, qn], dim=0)
        text = text.to(vis_feat_norm.device)
        if qn is not None and method == "paired":
            out, _, _ = eng.ground(vis_feat_norm, text, _lib.DC_GROUND_PAIRED, softmax_temp, normalize=False)
            return out.view(-1, 1).to(vis_feat_norm.dtype)
        if qn is not None and method != "argmax":
            return None  # the reference falls off the end of the if/elif chain
        out, _, _ = eng.ground(vis_feat_norm, text, _lib.DC_GROUND_RAW, softmax_temp, normalize=False)
        return out.to(vis_feat_norm.dtype)

    # ------------------------------------------------------------------ a16
    @torch.no_grad()
    def predict(self, vis_feats, qpos, qneg=None, norm_vis_feat=None, method=None, threshold=None):
        method = method or self.method
        threshold = threshold or self.threshold
        norm_vis_feat = norm_vis_feat or self.norm_vis_feat
        self._check_feats(vis_feats)
        qp, qn = self._encode(qpos, qneg)
        eng = self._eng()
        text = (qp if qn is None else torch.cat([qp, qn], dim=0)).to(vis_feats.device)
        n = vis_feats.shape[0]
        if qneg is None or (qneg is not None and method == "paired"):
            mode = _lib.DC_GROUND_RAW if qn is None else _lib.DC_GROUND_PAIRED
            sims, pred = eng.predict(vis_feats, text, mode, self.SOFTMAX_TEMP, bool(norm_vis_feat), threshold)
            pred = pred.view(torch.bool)
            if n == 1:  # .squeeze() in the reference makes these 0-d (quirk q18)
                pred, sims = pred.reshape(()), sims.reshape(())
            return pred, sims
        elif qneg is not None and method == "argmax":
            if n == 1:
                raise IndexError("too many indices for tensor of dimension 1")  # reference behaviour (q18)
            out, pred = eng.predict(vis_feats, text, _lib.DC_GROUND_ARGMAX, self.SOFTMAX_TEMP, bool(norm_vis_feat), threshold)
            return pred.view(torch.bool), out

    @torch.no_grad()
    def predict_queries(self, vis_feats, queries, qneg="scene", norm_vis_feat=None, method=None, threshold=None):
        """`predict` for every text query of a scene in one library call. Returns (pred (Qq,N) bool, sims (Qq,N) fp32):
        row q is predict(vis_feats.clone(), queries[q], qneg_q, norm_vis_feat, method, threshold) flattened to (N,), with
        qneg_q = every other query text for qneg == "scene" (the reference's evaluation loops, tools/validate_upper_bound.py
        :200-218; the generic negatives when there is none), the same list for every query when qneg is a list, no
        negatives for None. Every distinct text is encoded once, the features are normalised in place once and
        multiplied with the prompt rows once. None where predict returns None."""
        method = method or self.method
        threshold = threshold or self.threshold
        norm_vis_feat = norm_vis_feat or self.norm_vis_feat
        self._check_feats(vis_feats)
        queries = list(queries)
        texts, pos, negs = query_columns(queries, qneg, self.NEGATIVE_PROMPT_GENERIC)
        if negs is None:
            mode = _lib.DC_GROUND_RAW
        elif method == "paired":
            mode = _lib.DC_GROUND_PAIRED
        elif method == "argmax":
            mode = _lib.DC_GROUND_ARGMAX
        else:
            return None  # predict falls off the end of its if/elif chain
        n = vis_feats.shape[0]
        if mode == _lib.DC_GROUND_ARGMAX and n == 1 and queries:
            raise IndexError("too many indices for tensor of dimension 1")  # predict's behaviour (q18)
        if not queries:
            return (torch.empty((0, n), dtype=torch.bool, device=vis_feats.device),
                    torch.empty((0, n), dtype=torch.float32, device=vis_feats.device))
        text = self.model.encode_text(self._tok(texts).to(self.device))
        text /= text.norm(dim=-1, keepdim=True)
        score, pred = self._eng().predict_queries(vis_feats, text.to(vis_feats.device), pos, negs, mode, self.SOFTMAX_TEMP,
                                                  bool(norm_vis_feat), threshold)
        return pred.view(torch.bool), score

    @torch.no_grad()
    def predict_many(self, vis_feats, counts, queries, qneg="scene", norm_vis_feat=None, method=None, threshold=None):
        """`predict_queries` for every scene of a batch in one library call. vis_feats (sum N, C) holds the scenes' rows
        in scene order (a collated sparse batch), counts[s] = N_s, queries[s] the query texts of scene s; qneg applies to
        every scene as in predict_queries. Returns one entry per scene: what predict_queries(rows of scene s,
        queries[s], qneg, norm_vis_feat, method, threshold) returns, a (pred (Q_s, N_s) bool, sims (Q_s, N_s) fp32) pair
        (views into one score and one pred buffer) or None for a method predict does not know.
        Every distinct text of the batch is encoded in one encode_text call. The rows of the scenes with queries are
        normalised in place once (a scene without queries is left as it is, as predict_queries leaves it).
        Unlike a loop of predict_queries, which would have normalised the scenes before the failing one, every error
        is raised before any row changes: IndexError when method == "argmax" and a scene with queries has one point,
        RuntimeError for CPU or non-contiguous features, ValueError when counts do not sum to the rows."""
        method = method or self.method
        threshold = threshold or self.threshold
        norm_vis_feat = norm_vis_feat or self.norm_vis_feat
        batch = self._batch_prompts(vis_feats, counts, queries, qneg, method)
        if batch is None:
            return [None] * len(counts)  # predict falls off the end of its if/elif chain
        counts, mode, text, prompt_counts, pos, negs = batch
        res = self._eng().predict_many(vis_feats, counts, text, prompt_counts, pos, negs, mode, self.SOFTMAX_TEMP,
                                       bool(norm_vis_feat), threshold)
        return [(pred.view(torch.bool), score) for score, pred in res]

    @torch.no_grad()
    def predict_many_iou(self, vis_feats, counts, labels, obj_queries, qneg="scene", norm_vis_feat=None, method=None,
                         threshold=None):
        """predict_many scored against the point labels in one library call, for the grounding evaluation loops
        (engine/distil.py:436-493, tools/validate_upper_bound.py:200-221): returns (inter, union), int64 CUDA tensors of
        shape (sum Q,). obj_queries[s] maps each text query of scene s to its object ids (the reference's mapping);
        the queries of a scene are its keys in order, scene after scene. For query q with ids `ids` of scene s,
        inter = |pred & gt| and union = |pred | gt|, where pred is the row predict_many(vis_feats, counts, [list(o) for o in
        obj_queries], qneg, ...) returns for the query and gt = isin(labels of scene s, ids): what trainMetricPC counts
        for that query, at any of its thresholds in (0, 1] without sigmoid. metrics.grounding_scores(inter, union) then
        gives trainMetricPC's mIoU and Pr@k. Neither the scores nor the predictions are returned.
        labels (sum N,) int32 / int64 CUDA tensor in feature-row order. Defaults, the in-place normalisation and the
        errors follow predict_many, and every error is raised before any row changes; ValueError also for labels of
        another dtype or count, and for an id outside the labels' dtype. None for a method predict does not know."""
        return self._many_iou("predict_many_iou", vis_feats, counts, labels, obj_queries, qneg, norm_vis_feat, method,
                              threshold or self.threshold)

    @torch.no_grad()
    def predict_many_iou_sweep(self, vis_feats, counts, labels, obj_queries, thresholds, qneg="scene", norm_vis_feat=None,
                               method=None):
        """predict_many_iou at many thresholds in one library call, to choose the threshold on a validation set or to
        report mIoU / Pr@k against it: returns (inter, union), int64 CUDA tensors of shape (T, sum Q). Row t equals
        predict_many_iou(vis_feats.clone(), counts, labels, obj_queries, qneg, norm_vis_feat, method,
        threshold=thresholds[t]) on the rows as passed, and metrics.grounding_scores(inter[t], union[t]) gives that
        call's mIoU and Pr@k. Everything before the threshold comparison (normalisation, GEMM, scoring, min-max) runs
        once. thresholds: 1..1024 numbers in the caller's order, duplicates allowed; a falsy entry (0, 0.0, None) means
        self.threshold, as for the single call, and each entry is rounded to fp32 as the single call rounds it. A NaN or
        +inf entry predicts no point (inter 0, union |gt|); -inf every point whose score is not NaN. With method
        "argmax" every row is the same. Defaults, the in-place normalisation (done once), empty scenes and the errors
        follow predict_many_iou; ValueError also for no thresholds or more than 1024, raised before any row changes."""
        return self._many_iou("predict_many_iou_sweep", vis_feats, counts, labels, obj_queries, qneg, norm_vis_feat,
                              method, threshold_table(thresholds, self.threshold))

    def _many_iou(self, fn, vis_feats, counts, labels, obj_queries, qneg, norm_vis_feat, method, threshold):
        """FusionEngine.predict_many_iou / predict_many_iou_sweep (`fn`) at `threshold` (one or a table) from the
        reference's text -> ids mappings; None for a method predict does not know."""
        method = method or self.method
        norm_vis_feat = norm_vis_feat or self.norm_vis_feat
        obj_queries = [dict(o) for o in obj_queries]
        batch = self._batch_prompts(vis_feats, counts, [list(o) for o in obj_queries], qneg, method)
        if batch is None:
            return None  # predict falls off the end of its if/elif chain
        counts, mode, text, prompt_counts, pos, negs = batch
        gt_ids = [[list(ids) for ids in o.values()] for o in obj_queries]
        return getattr(self._eng(), fn)(vis_feats, counts, text, prompt_counts, pos, negs, labels, gt_ids, mode,
                                        self.SOFTMAX_TEMP, bool(norm_vis_feat), threshold)

    def _batch_prompts(self, vis_feats, counts, queries, qneg, method):
        """The checks and the prompt tables of predict_many: (counts, mode, text, prompt_counts, pos, negs), or None for a
        method predict does not know. Every distinct text of the batch is encoded in one encode_text call."""
        self._check_feats(vis_feats)
        counts = [int(c) for c in counts]
        scene_queries = [list(q) for q in queries]
        if len(scene_queries) != len(counts):
            raise ValueError(f"{len(counts)} point counts but {len(scene_queries)} query lists")
        if any(c < 0 for c in counts) or sum(counts) != vis_feats.shape[0]:
            raise ValueError(f"point counts {counts} do not sum to the {vis_feats.shape[0]} feature rows")
        texts, gather, prompt_counts, pos, negs = batch_query_columns(scene_queries, qneg, self.NEGATIVE_PROMPT_GENERIC)
        if qneg is None:
            mode = _lib.DC_GROUND_RAW
        elif method == "paired":
            mode = _lib.DC_GROUND_PAIRED
        elif method == "argmax":
            mode = _lib.DC_GROUND_ARGMAX
        else:
            return None
        if mode == _lib.DC_GROUND_ARGMAX and any(n == 1 and q for n, q in zip(counts, scene_queries)):
            raise IndexError("too many indices for tensor of dimension 1")  # predict's behaviour (q18)
        if texts:
            emb = self.model.encode_text(self._tok(texts).to(self.device))
            emb /= emb.norm(dim=-1, keepdim=True)
            text = emb.index_select(0, torch.tensor(gather, dtype=torch.long, device=emb.device)).to(vis_feats.device)
        else:
            text = vis_feats.new_empty((0, vis_feats.shape[1]))
        return counts, mode, text, prompt_counts, pos, None if qneg is None else negs


# ---------------------------------------------------------------------- a18
@torch.no_grad()
def class_similarity(vis_feat: torch.Tensor, txt_feat: torch.Tensor, return_sims: bool = True, engine: FusionEngine = None):
    """`_get_similarity` + the arg max that follows it in the reference's evaluation loops
    (engine/distil.py:244-246,289-290, tools/validate_upper_bound.py:59-61,101-102):

        txt_feat /= txt_feat.norm(dim=-1, keepdim=True)       # IN PLACE on the class table the caller passes
        sims = vis_feat @ txt_feat.T                          # (M, K) fp32, vis_feat is NOT normalised
        pred = torch.max(sims, 1)[1]                          # (M,) int64

    One tcgen05 GEMM whose epilogue keeps each row's arg max, so the (M, K) matrix is written only when
    `return_sims` (the reference feeds it to the cross-entropy criterion, engine/distil.py:302).
    Returns (sims | None, pred)."""
    if not (isinstance(vis_feat, torch.Tensor) and vis_feat.is_cuda and isinstance(txt_feat, torch.Tensor) and txt_feat.is_cuda):
        raise RuntimeError("dropclip_b200 grounding needs CUDA tensors; there is no CPU fallback")
    if vis_feat.dim() != 2 or txt_feat.dim() != 2 or vis_feat.shape[1] != txt_feat.shape[1]:
        raise RuntimeError(f"mat1 and mat2 shapes cannot be multiplied ({tuple(vis_feat.shape)} and {tuple(txt_feat.T.shape)})")
    txt_feat /= txt_feat.norm(dim=-1, keepdim=True)  # K x C, tiny; in place like the reference
    eng = engine or FusionEngine(vis_feat.device)
    x = vis_feat if vis_feat.dtype in (torch.float16, torch.float32) else vis_feat.float()
    x = x.contiguous()
    if x.shape[0] == 0:
        return (torch.empty((0, txt_feat.shape[0]), dtype=torch.float32, device=x.device) if return_sims else None,
                torch.empty(0, dtype=torch.int64, device=x.device))
    sims, pred, _ = eng.ground(x, txt_feat, _lib.DC_GROUND_CLASS, 0.1, normalize=False, want_matrix=return_sims)
    if sims is not None and vis_feat.dtype != torch.float32 and vis_feat.dtype == txt_feat.dtype:
        sims = sims.to(vis_feat.dtype)
    return sims, pred


def _get_similarity(vis_feat, txt_feat):
    """Name and signature of the closure in engine/distil.py:244-246 / tools/validate_upper_bound.py:59-61."""
    return class_similarity(vis_feat, txt_feat, return_sims=True)[0]
