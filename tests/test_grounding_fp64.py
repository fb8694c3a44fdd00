"""The grounding kernels against an fp64 evaluation of the formulas in include/dropclip.h.

The reference below is plain torch float64 (on the GPU for speed) and never calls libdropclip:
  - feature rows as the library multiplies them: fp16 rows normalised with the correctly rounded fp16 norm and the
    fp16-rounded quotient (the library's promise), fp32 rows normalised in fp64; prompt rows exactly as received;
  - S = Y . T^T, then per query RAW v = S[pos]; PAIRED v = 1 / (m + sum_j exp((S[j] - S[pos]) / T)), NaN -> 0;
    ARGMAX v = S[pos] - mean(S[neg]), pred = S[pos] >= max(S[neg]); CLASS the first index of the row maximum;
  - the per-query min-max (v - min) / (max - min), or v / max when the extrema coincide (ARGMAX: the raw extrema).

Every comparison is against a bound derived below (s_bound, score64, minmax64), not a measured tolerance, and discrete
outputs are compared only where the fp64 margin exceeds the bound. The largest error and the largest error / bound of
each group are printed (pytest -s)."""
import math
import zlib

import numpy as np
import pytest
import torch

from dropclip_b200 import _lib
from dropclip_b200.similarity import ClipSimilarity, batch_query_columns, query_columns

RAW, PAIRED, ARGMAX, CLASS = _lib.DC_GROUND_RAW, _lib.DC_GROUND_PAIRED, _lib.DC_GROUND_ARGMAX, _lib.DC_GROUND_CLASS
PAIRS = [("f16", "f16"), ("f16", "f32"), ("f32", "f16"), ("f32", "f32")]  # (features, prompts)
DT = {"f16": torch.float16, "f32": torch.float32}
U24, U23, U22 = 2.0 ** -24, 2.0 ** -23, 2.0 ** -22
WORST = {}  # group -> [largest error, largest error / bound, values compared, values inside the bound's margin]


# ---------------------------------------------------------------------------------------------------- reference
def fp16_unit_rows(x):
    """fp16 rows divided by their correctly rounded fp16 norm, the fp32 quotient rounded to fp16 (the library's
    normalisation of fp16 features). torch's d.half() rounds through fp32, so the nearest of three neighbours is
    picked in fp64."""
    d = x.double().pow(2).sum(-1, keepdim=True).sqrt()
    h0 = d.float().half()
    bits = h0.view(torch.int16)
    cands = torch.stack([h0, (bits + 1).view(torch.float16), (bits - 1).clamp_min(0).view(torch.float16)], 0)
    pick = (cands.double() - d).abs().nan_to_num(nan=float("inf")).argmin(0, keepdim=True)
    nrm = torch.where(torch.isfinite(h0) & (h0 > 0), cands.gather(0, pick)[0], h0)
    return (x.float() / nrm.float()).half()


def rows64(x, normalize):
    """The feature rows the library multiplies, in fp64."""
    if not normalize:
        return x.double()
    if x.dtype == torch.float16:
        return fp16_unit_rows(x).double()
    x = x.double()
    return x / x.norm(dim=-1, keepdim=True)


def s_bound(y, t, x32, t32, norm32):
    """Bound of |S_kernel - Y.T^T| per entry. A = sum_k |y_k t_k| (<= 1 for unit rows).
    - An fp32 operand v enters as hi + lo (hi = fp16(v), lo = fp16(v - hi)): |v - hi - lo| <= 2^-22 |v| + 2^-25 (lo is
      an fp16 subnormal below 2^-14, spacing 2^-24): 2^-22 A + 2^-25 |other row|_1. With both operands split, lo.lo and
      the cross terms are left out: 2^-21 A.
    - fp32 features normalised by the library: the fp32 norm and quotient, 2^-23 A.
    - Products of fp16 values are exact in fp32. Each MMA instruction adds 16 of them to the fp32 accumulator and
      rounds (or truncates) once, by at most 2^-23 of the running sum, itself at most 1.01 A; n_terms * dim / 16
      instructions. (About 2e-6 for unit rows of width 768 if these errors cancelled like random signs; this bound does
      not assume that.)"""
    a = y.abs() @ t.abs().T
    n_terms = 1 + int(x32) + int(t32)
    e = (n_terms * y.shape[1] // 16) * U23 * 1.01 * a
    if x32:
        e += U22 * a + 2.0 ** -25 * t.abs().sum(1)[None, :]
    if t32:
        e += U22 * a + 2.0 ** -25 * y.abs().sum(1)[:, None]
    if x32 and t32:
        e += 2 * U22 * a
    if norm32:
        e += U23 * a
    return e


def score64(S, eS, pos, negs, mode, temp):
    """fp64 scores of one query and their bounds given |dS| <= eS: (v, ev, pred, sure_pred, raw_differ).
    PAIRED: every exponent moves by at most (eS_j + eS_pos) / T, plus the rounding of its fp32 argument (scale and
    bias rounded, 2^-22 (|S_j| + |S_pos|) / T) and ex2.approx (2^-21), so |dv| <= v (e^d - 1); the fp32 sums of m
    terms and the reciprocal add (m + 4) 2^-23 v; an fp32 sum that overflows gives v = 0 where fp64 keeps < 4e-38.
    ARGMAX: eS_pos + max eS_neg, plus the fp32 mean of m values, (m + 2) 2^-24 (mean |S_neg| + |v|)."""
    sp, ep = S[:, pos], eS[:, pos]
    raw_differ = None
    if mode == RAW:
        return sp, ep, None, None, raw_differ
    sn, en = S[:, negs], eS[:, negs]
    m = len(negs)
    if mode == PAIRED:
        t32 = float(np.float32(temp))
        v = torch.nan_to_num(1.0 / (m + torch.exp((sn - sp[:, None]) / t32).sum(1)), nan=0.0)
        d = ((en + ep[:, None]) / t32 + U22 * (sn.abs() + sp.abs()[:, None]) / t32).max(1).values + 2.0 ** -21
        return v, v * (torch.expm1(d) + (m + 4) * U23) + 4e-38, None, None, raw_differ
    v = sp - sn.mean(1)
    ev = ep + en.max(1).values + (m + 2) * U24 * (sn.abs().mean(1) + v.abs())
    nmax = sn.max(1).values
    sure = (sp - nmax).abs() > ep + en.max(1).values
    raw = torch.cat([sp[:, None], sn], 1)
    return v, ev, sp >= nmax, sure, bool(raw.max() != raw.min())


def minmax64(v, ev, mode, raw_differ):
    """The library's per-query min-max of v and its bound: with R = max - min > 4 E (E = max ev), the extrema move by
    at most E, so |d out| <= (ev + E (1 + 2 |out|)) / (R - 2 E), plus three fp32 roundings. Extrema that coincide (one
    point) give v / max or, for ARGMAX with distinct raw extrema, 0 / 0 in both. None: R is inside the noise."""
    mn, mx = v.min(), v.max()
    r = mx - mn
    differ = raw_differ if mode == ARGMAX else bool(mx != mn)
    out = (v - mn) / r if differ else v / mx
    e = ev.max()
    if r == 0 and (differ or mx.abs() > e):
        return out, torch.full_like(v, 4 * U24)
    if r <= 4 * e:  # also v / max with max in the noise (a paired score whose fp32 sum overflows)
        return None, None
    return out, (ev + e * (1 + 2 * out.abs())) / (r - 2 * e) + 4 * U24


def close(group, got, want, bound, what=""):
    got, want = got.double().reshape(want.shape), want
    nan = torch.isnan(want)
    assert torch.equal(torch.isnan(got), nan), f"{group} {what}: NaN where the reference has none (or the reverse)"
    err = (got - want).abs().masked_fill(nan, 0.0)
    ratio = (err / bound.expand_as(err)).masked_fill(nan, 0.0)
    w = WORST.setdefault(group, [0.0, 0.0, 0, 0])
    w[0], w[1], w[2] = max(w[0], err.max().item() if err.numel() else 0.0), max(w[1], ratio.max().item() if err.numel() else 0.0), w[2] + err.numel()
    if err.numel():
        k = int(ratio.argmax())
        assert ratio.max().item() <= 1.0, (f"{group} {what}: error {err.reshape(-1)[k].item():.3e} at {k} is "
                                           f"{ratio.max().item():.2f} x the bound {bound.expand_as(err).reshape(-1)[k].item():.3e}")


def same_where(group, got, want, sure, what=""):
    got = got.reshape(want.shape)
    w = WORST.setdefault(group, [0.0, 0.0, 0, 0])
    w[2], w[3] = w[2] + want.numel(), w[3] + int(sure.sum())
    bad = (got.bool() != want.bool()) & sure
    assert not bool(bad.any()), f"{group} {what}: {int(bad.sum())} decisions differ outside the bound's margin"


def report(title):
    print(f"\n{title}: largest error, largest error / bound, values, margins decided")
    for g, (e, r, n, s) in sorted(WORST.items()):
        print(f"  {g:<34} {e:.3e} {r:6.3f} {n:>10} {s:>10}")


def check_query(group, out, pred, v, ev, mode, raw_differ, pred_ref, sure_pred, thr, what):
    """A query's min-max normalised scores and predictions (dc_predict, dc_predict_queries, dc_predict_many)."""
    want, tol = minmax64(v, ev, mode, raw_differ)
    if want is None:
        WORST.setdefault(group + " (range in noise)", [0.0, 0.0, 0, 0])[2] += 1
        return
    close(group, out, want, tol, what)
    if mode == ARGMAX:
        same_where(group + " pred", pred, pred_ref, sure_pred, what)
    else:
        same_where(group + " pred", pred, want > thr, (want - thr).abs() > tol, what)


# ---------------------------------------------------------------------------------------------------- inputs
def prompt_rows(p, dim, dtype, gen):
    t = torch.randn((p, dim), generator=gen, device="cuda")
    return (t / t.norm(dim=-1, keepdim=True)).to(dtype)


def feature_rows(n, dim, dtype, t, gen, strong=None):
    """Noise rows pulled toward a random prompt row each (scores spread over the whole range); `strong` rows pulled
    hard toward one prompt row."""
    x = torch.randn((n, dim), generator=gen, device="cuda")
    if t.shape[0] and n:
        owner = torch.randint(0, t.shape[0], (n,), generator=gen, device="cuda")
        x += torch.rand((n, 1), generator=gen, device="cuda") * 1.5 * math.sqrt(dim) * t.float()[owner]
        if strong is not None:
            x[: max(1, n // 6)] += 4.0 * math.sqrt(dim) * t.float()[strong]
    return x.to(dtype).contiguous()


def gen(*key):
    return torch.Generator(device="cuda").manual_seed(zlib.crc32(repr(key).encode()))


def engine():
    from dropclip_b200.engine import FusionEngine
    return FusionEngine("cuda")


def sims64(x0, t, normalize):
    y = rows64(x0, normalize)
    tt = t.double()
    return y @ tt.T, s_bound(y, tt, x0.dtype == torch.float32, t.dtype == torch.float32,
                             normalize and x0.dtype == torch.float32)


# ---------------------------------------------------------------------------------------------------- CPU
def test_reference_matches_the_cpu_oracle():
    """The fp64 reference (fp32 path: rows normalised in fp64) equals oracle/similarity_ref evaluated on fp64 inputs."""
    from oracle import similarity_ref
    g = torch.Generator().manual_seed(5)
    for n, p, dim in ((1, 2, 64), (7, 5, 64), (300, 33, 128)):
        x = torch.randn((n, dim), generator=g, dtype=torch.float64)
        emb = torch.randn((p, dim), generator=g, dtype=torch.float64)
        t = emb / emb.norm(dim=-1, keepdim=True)
        S = rows64(x, True) @ t.T
        eS = torch.zeros_like(S)
        for temp in (1e-3, 0.1, 10.0):
            v = score64(S, eS, 0, list(range(1, p)), PAIRED, float(np.float32(temp)))[0]
            torch.testing.assert_close(v, similarity_ref.paired_softmax(S, float(np.float32(temp)))[:, 0], rtol=1e-10, atol=1e-300)
        if n < 2:
            continue
        for method, mode, qn in (("paired", PAIRED, emb[1:]), ("argmax", ARGMAX, emb[1:]), ("paired", RAW, None)):
            want_pred, want = similarity_ref.predict_from_embeds(x.clone(), emb[:1].clone(), qn, method=method, threshold=0.7)
            Sq = S if qn is not None else S[:, :1]
            v, ev, pred, sure, raw_differ = score64(Sq, torch.zeros_like(Sq), 0, list(range(1, Sq.shape[1])), mode,
                                                    similarity_ref.SOFTMAX_TEMP)
            out, _ = minmax64(v, ev, mode, raw_differ)
            torch.testing.assert_close(out, want.double(), rtol=0, atol=2.0 ** -24)  # the oracle returns fp32
            assert torch.equal(pred if mode == ARGMAX else out > 0.7, want_pred)
        sims, idx = similarity_ref.class_similarity(x, emb.clone())
        torch.testing.assert_close(sims, rows64(x, False) @ t.T, rtol=1e-12, atol=1e-12)
        assert torch.equal(idx, torch.topk(sims, 1, dim=1).indices[:, 0])


def test_bounds_catch_a_doubled_product():
    """The S bound is far below the error of counting hi.t twice (fp32 features, fp16 prompts)."""
    g = torch.Generator().manual_seed(1)
    x = torch.randn((200, 768), generator=g)
    t = torch.randn((20, 768), generator=g)
    t = (t / t.norm(dim=-1, keepdim=True)).half()
    y = rows64(x, True)
    S = y @ t.double().T
    e = s_bound(y, t.double(), True, False, True)
    assert e.max().item() < 2e-5
    hi = y.float().half().double()
    assert ((2 * hi @ t.double().T + (y - hi) @ t.double().T - S).abs() > e).float().mean().item() > 0.99


# ---------------------------------------------------------------------------------------------------- GPU: dtype pairs
class Tower:
    """encode_text: a fixed random row per text in the prompt dtype, on the GPU (a CLIP model on CUDA returns fp16
    embeddings whatever the dtype of the point features)."""

    def __init__(self, dim, dtype, seed=3):
        g = torch.Generator().manual_seed(seed)
        self.table = torch.randn((4096, dim), generator=g).to(dtype).cuda()
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


def encoded(cs, texts):
    """The prompt rows ClipSimilarity hands the library for `texts` (encode_text, then the in-place row norm)."""
    e = cs.model.encode_text(cs._tok(texts).to(cs.device))
    e /= e.norm(dim=-1, keepdim=True)
    return e


@pytest.mark.gpu
@pytest.mark.parametrize("dim", [512, 768, 1024])
@pytest.mark.parametrize("fd,td", PAIRS)
def test_dtype_pairs(fd, td, dim):
    """Every public grounding call at every (features, prompts) dtype pair. fp32 features with fp16 prompts is what a
    CLIP model on CUDA (fp16) and a 3D network (fp32) give together."""
    fdt, tdt = DT[fd], DT[td]
    tower = Tower(dim, tdt)
    cs = ClipSimilarity(model=tower, tokenize=tower.tokenize, device="cuda", method="paired", threshold=0.7)
    g = gen("pairs", fd, td, dim)
    queries = [f"object {i}" for i in range(6)]
    qneg = ["wall", "floor", "chair", "table", "lamp"]
    n = 3000
    x0 = feature_rows(n, dim, fdt, encoded(cs, queries + qneg).float(), g)
    tag = f"{fd}x{td}"
    thr = 0.7

    # compute_similarity: RAW matrix and the paired score, not min-max normalised, cast to the feature dtype
    xn = x0.clone()
    xn /= xn.norm(dim=-1, keepdim=True)
    # compute_similarity returns the feature dtype: rounding the kernel's value (within e of s) to fp16 adds
    # 2^-11 (|s| + e), 2^-25 below 2^-14
    r16 = (lambda s, e: e + 2.0 ** -11 * (s.abs() + e) + 2.0 ** -25) if fdt == torch.float16 else (lambda s, e: e)
    qp, qn = cs._encode(queries[0], qneg)
    S, eS = sims64(xn, torch.cat([qp, qn]), False)
    raw = cs.compute_similarity(xn.clone(), queries[0], qneg, method="argmax")
    close(f"compute_similarity RAW {tag}", raw, S, r16(S, eS))
    raw1 = cs.compute_similarity(xn.clone(), queries[0])
    close(f"compute_similarity RAW {tag}", raw1, S[:, :1], r16(S[:, :1], eS[:, :1]))
    v, ev, *_ = score64(S, eS, 0, list(range(1, S.shape[1])), PAIRED, cs.SOFTMAX_TEMP)
    got = cs.compute_similarity(xn.clone(), queries[0], qneg, method="paired")
    close(f"compute_similarity PAIRED {tag}", got, v, r16(v, ev))

    # predict: RAW, PAIRED, ARGMAX (features normalised in place by the library)
    for method, negs, mode in (("paired", None, RAW), ("paired", qneg, PAIRED), ("argmax", qneg, ARGMAX)):
        qp, qn = cs._encode(queries[1], negs)
        S, eS = sims64(x0, qp if qn is None else torch.cat([qp, qn]), True)
        v, ev, pref, sure, rd = score64(S, eS, 0, list(range(1, S.shape[1])), mode, cs.SOFTMAX_TEMP)
        pred, out = cs.predict(x0.clone(), queries[1], negs, method=method, threshold=thr)
        check_query(f"predict {tag}", out, pred, v, ev, mode, rd, pref, sure, thr, method)

    # predict_queries and predict_many: every query of the scene, scene negatives and none
    texts, pos, negl = query_columns(queries, "scene", cs.NEGATIVE_PROMPT_GENERIC)
    S, eS = sims64(x0, encoded(cs, texts), True)
    for method, mode in (("paired", PAIRED), ("argmax", ARGMAX)):
        pred, out = cs.predict_queries(x0.clone(), queries, "scene", method=method, threshold=thr)
        for q in range(len(queries)):
            v, ev, pref, sure, rd = score64(S, eS, pos[q], negl[q], mode, cs.SOFTMAX_TEMP)
            check_query(f"predict_queries {tag}", out[q], pred[q], v, ev, mode, rd, pref, sure, thr, f"{method} q{q}")
    pred, out = cs.predict_queries(x0.clone(), queries, None, threshold=thr)
    for q in range(len(queries)):
        v, ev, *_ = score64(S, eS, pos[q], None, RAW, cs.SOFTMAX_TEMP)
        check_query(f"predict_queries {tag}", out[q], pred[q], v, ev, RAW, None, None, None, thr, f"raw q{q}")

    counts = [1000, 0, 2000]
    scene_q = [queries[:3], ["x"], queries[2:]]
    texts, gather, pcounts, pos, negl = batch_query_columns(scene_q, "scene", cs.NEGATIVE_PROMPT_GENERIC)
    emb = encoded(cs, texts).index_select(0, torch.tensor(gather, device="cuda"))
    res = cs.predict_many(x0.clone(), counts, scene_q, "scene", method="paired", threshold=thr)
    r0 = p0 = 0
    for s, (ns, ps) in enumerate(zip(counts, pcounts)):
        if ns:
            S, eS = sims64(x0[r0:r0 + ns], emb[p0:p0 + ps], True)
            for q in range(len(scene_q[s])):
                v, ev, pref, sure, rd = score64(S, eS, pos[s][q], negl[s][q], PAIRED, cs.SOFTMAX_TEMP)
                check_query(f"predict_many {tag}", res[s][1][q], res[s][0][q], v, ev, PAIRED, rd, pref, sure, thr,
                            f"scene {s} q{q}")
        r0, p0 = r0 + ns, p0 + ps

    # class_similarity: un-normalised features against the class table it normalises in place
    table = tower.table[:40].clone()
    sims, idx = cs_class(x0, table)
    S, eS = sims64(x0, table, False)
    close(f"class_similarity {tag}", sims, S, r16(S, eS) if tdt == torch.float16 else eS)  # fp16 x fp16: fp16 sims
    check_argmax(f"class_similarity {tag}", idx, S, eS)
    report(f"dtype pair {tag}, dim {dim}")


def cs_class(x, table):
    from dropclip_b200.similarity import class_similarity
    sims, idx = class_similarity(x.clone(), table)  # `table` now holds the normalised rows the library used
    return sims.float(), idx


def check_argmax(group, idx, S, eS):
    """First index of the row maximum, where the fp64 gap to the runner-up exceeds both entries' bounds."""
    top = torch.topk(S, min(2, S.shape[1]), dim=1)
    want = top.indices[:, 0]
    if S.shape[1] == 1:
        sure = torch.ones_like(want, dtype=torch.bool)
    else:
        sure = (top.values[:, 0] - top.values[:, 1]) > 2 * eS.max(1).values
    w = WORST.setdefault(group + " argmax", [0.0, 0.0, 0, 0])
    w[2], w[3] = w[2] + want.numel(), w[3] + int(sure.sum())
    assert torch.equal(idx[sure], want[sure]), f"{group}: {int((idx[sure] != want[sure]).sum())} arg max indices differ"


# ---------------------------------------------------------------------------------------------------- GPU: dc_ground
GROUND_P = [2, 33, 255, 256, 257, 300, 511, 512, 513, 1000]


@pytest.mark.gpu
@pytest.mark.parametrize("fd,td", PAIRS)
@pytest.mark.parametrize("p", GROUND_P)
def test_ground_prompt_blocks(p, fd, td):
    """dc_ground's epilogue (no min-max) for every width of the last 256-column block and the carry rows between
    blocks: PAIRED at three temperatures, ARGMAX, CLASS and the RAW matrix. A strong negative sits in the last block."""
    dim = (512, 768, 1024)[GROUND_P.index(p) % 3]
    fdt, tdt = DT[fd], DT[td]
    g = gen("ground", p, fd, td)
    t = prompt_rows(p, dim, tdt, g)
    x0 = feature_rows(3000, dim, fdt, t, g, strong=max(1, p - 3))
    eng = engine()
    tag = f"{fd}x{td}"
    S, eS = sims64(x0, t, True)
    negs = list(range(1, p))
    for temp in (1e-3, 0.1, 10.0):
        out, _, _ = eng.ground(x0.clone(), t, PAIRED, temp, normalize=True)
        v, ev, *_ = score64(S, eS, 0, negs, PAIRED, temp)
        close(f"ground PAIRED T={temp:g} {tag}", out, v, ev, f"P={p}")
    out, pred, _ = eng.ground(x0.clone(), t, ARGMAX, 0.1, normalize=True)
    v, ev, pref, sure, _ = score64(S, eS, 0, negs, ARGMAX, 0.1)
    close(f"ground ARGMAX {tag}", out, v, ev, f"P={p}")
    same_where(f"ground ARGMAX {tag} pred", pred, pref, sure, f"P={p}")
    out, _, _ = eng.ground(x0.clone(), t, RAW, 0.1, normalize=True)
    close(f"ground RAW {tag}", out, S, eS, f"P={p}")
    S, eS = sims64(x0, t, False)
    sims, idx, _ = eng.ground(x0.clone(), t, CLASS, 0.1, normalize=False)
    close(f"ground CLASS {tag}", sims, S, eS, f"P={p}")
    check_argmax(f"ground CLASS {tag}", idx, S, eS)
    _, idx2, _ = eng.ground(x0.clone(), t, CLASS, 0.1, normalize=False, want_matrix=False)
    assert torch.equal(idx2, idx)
    report(f"dc_ground P={p} dim={dim} {tag}")


# ---------------------------------------------------------------------------------------------------- GPU: query_scores_kernel
TILE_P = [47, 48, 95, 96, 191, 192, 383, 384, 1535, 1536]
TILE_N = [1, 31, 32, 33, 255, 256, 257, 20_000]


def check_queries(group, score, pred, S, eS, pos, negl, mode, temp, thr, what=""):
    for q in range(len(pos)):
        v, ev, pref, sure, rd = score64(S, eS, pos[q], None if negl is None else negl[q], mode, temp)
        check_query(group, score[q], pred[q], v, ev, mode, rd, pref, sure, thr, f"{what} q{q}")


@pytest.mark.gpu
@pytest.mark.parametrize("p", TILE_P)
def test_query_scores_row_tiles(p):
    """dc_predict_queries at each tile_rows boundary of the scoring pass (256 -> 128 -> 64 -> 32 staged rows, then
    past 48 KB of shared memory up to the 1536-prompt limit), odd and even P (S stored by scalars or float4), and
    N around the 32-row warps and 256-thread blocks. Three queries share a negative list of P - 3 prompts."""
    k = TILE_P.index(p)
    dim = (512, 768, 1024)[k % 3]
    fd, td = PAIRS[k % 4]
    g = gen("tiles", p)
    t = prompt_rows(p, dim, DT[td], g)
    eng = engine()
    pos = [0, 1, 2]
    shared = list(range(3, p))
    group = f"predict_queries {fd}x{td}"
    for n in TILE_N:
        x0 = feature_rows(n, dim, DT[fd], t, g, strong=p - 1)
        S, eS = sims64(x0, t, True)
        for mode, temp in ((RAW, 0.1), (ARGMAX, 0.1), (PAIRED, 1e-3), (PAIRED, 0.1), (PAIRED, 10.0)):
            negl = None if mode == RAW else [shared] * 3
            score, pred = eng.predict_queries(x0.clone(), t, pos, negl, mode, temp, True, 0.5)
            check_queries(f"{group} mode {mode} T={temp:g}", score, pred, S, eS, pos, negl, mode, temp, 0.5, f"P={p} N={n}")
    report(f"query_scores_kernel P={p} dim={dim} {fd}x{td}")


@pytest.mark.gpu
@pytest.mark.parametrize("fd,td", PAIRS)
def test_query_scores_scene_negatives_385(fd, td):
    """385 queries, each with the other 384 as negatives: more than 48 KB of staged rows through scene negatives."""
    p, dim = 385, 768
    g = gen("scene385", fd, td)
    t = prompt_rows(p, dim, DT[td], g)
    x0 = feature_rows(1500, dim, DT[fd], t, g)
    S, eS = sims64(x0, t, True)
    eng = engine()
    pos = list(range(p))
    negl = [[j for j in range(p) if j != q] for q in range(p)]
    for mode in (PAIRED, ARGMAX):
        score, pred = eng.predict_queries(x0.clone(), t, pos, negl, mode, 0.1, True, 0.7)
        check_queries(f"predict_queries 385 scene {fd}x{td} mode {mode}", score, pred, S, eS, pos, negl, mode, 0.1, 0.7)
    report(f"385 scene negatives {fd}x{td}")


# ---------------------------------------------------------------------------------------------------- GPU: dc_predict_many
def check_many(group, res, x0, t, counts, pcounts, pos, negl, mode, temp, thr):
    r0 = p0 = 0
    for s, (ns, ps) in enumerate(zip(counts, pcounts)):
        score, pred = res[s]
        assert score.shape == (len(pos[s]), ns)
        if ns and pos[s]:
            S, eS = sims64(x0[r0:r0 + ns], t[p0:p0 + ps], True)
            check_queries(group, score, pred, S, eS, pos[s], None if negl is None else negl[s], mode, temp, thr,
                          f"scene {s}")
        r0, p0 = r0 + ns, p0 + ps


@pytest.mark.gpu
@pytest.mark.parametrize("fd,td", PAIRS)
@pytest.mark.parametrize("pw", [1533, 1534, 1535, 1536])
def test_predict_many_ragged(pw, fd, td):
    """The widest scene pads S's row stride by 3, 2, 1, 0 columns; beside it scenes of 2 prompts, a scene without
    points, one with a single point and one without queries (its rows must stay untouched). Every block is checked
    against fp64 on its own."""
    dim = (512, 768, 1024, 768)[pw - 1533]
    g = gen("many", pw, fd, td)
    counts = [500, 3000, 0, 1, 700, 129]
    pcounts = [2, pw, 2, 2, 3, 2]
    t = torch.cat([prompt_rows(c, dim, DT[td], g) for c in pcounts])
    x0 = feature_rows(sum(counts), dim, DT[fd], t[:8], g)
    pos = [[0, 1], [0, 1, 2], [0, 1], [0, 1], [], [1, 0]]
    negl = [[[1], [0]], [list(range(3, pw))] * 3, [[1], [0]], [[1], [0]], [], [[0], [1]]]
    eng = engine()
    for mode, temp in ((RAW, 0.1), (PAIRED, 0.1), (ARGMAX, 0.1), (PAIRED, 1e-3)):
        x = x0.clone()
        res = eng.predict_many(x, counts, t, pcounts, pos, None if mode == RAW else negl, mode, temp, True, 0.6)
        r4 = sum(counts[:4])
        assert torch.equal(x[r4:r4 + counts[4]], x0[r4:r4 + counts[4]]), "a scene without queries was changed"
        check_many(f"predict_many {fd}x{td} mode {mode} T={temp:g}", res, x0, t, counts, pcounts, pos,
                   None if mode == RAW else negl, mode, temp, 0.6)
    report(f"predict_many widest P={pw} {fd}x{td}")


# ---------------------------------------------------------------------------------------------------- GPU: widths
@pytest.mark.gpu
@pytest.mark.parametrize("fd,td", PAIRS)
@pytest.mark.parametrize("dim", [64, 2048])
def test_widths_64_and_2048(dim, fd, td):
    """One K block (fewer than the operand ring's stages) and the longest K loop of the ABI's common widths."""
    g = gen("width", dim, fd, td)
    t = prompt_rows(300, dim, DT[td], g)
    x0 = feature_rows(1000, dim, DT[fd], t, g, strong=297)
    eng = engine()
    tag = f"{fd}x{td} dim {dim}"
    S, eS = sims64(x0, t, True)
    out, _, _ = eng.ground(x0.clone(), t, PAIRED, 0.1, normalize=True)
    v, ev, *_ = score64(S, eS, 0, list(range(1, 300)), PAIRED, 0.1)
    close(f"ground PAIRED {tag}", out, v, ev)
    out, pred, _ = eng.ground(x0.clone(), t, ARGMAX, 0.1, normalize=True)
    v, ev, pref, sure, _ = score64(S, eS, 0, list(range(1, 300)), ARGMAX, 0.1)
    close(f"ground ARGMAX {tag}", out, v, ev)
    same_where(f"ground ARGMAX {tag} pred", pred, pref, sure)
    Sc, eSc = sims64(x0, t, False)
    sims, idx, _ = eng.ground(x0.clone(), t, CLASS, 0.1, normalize=False)
    close(f"ground CLASS {tag}", sims, Sc, eSc)
    check_argmax(f"ground CLASS {tag}", idx, Sc, eSc)
    pos, negl = [0, 5, 9], [list(range(10, 300))] * 3
    for mode in (PAIRED, ARGMAX):
        score, pred = eng.predict_queries(x0.clone(), t, pos, negl, mode, 0.1, True, 0.7)
        check_queries(f"predict_queries {tag}", score, pred, S, eS, pos, negl, mode, 0.1, 0.7)
        counts, pcounts = [129, 871], [5, 295]
        tb = torch.cat([t[:5], t[5:]])
        res = eng.predict_many(x0.clone(), counts, tb, pcounts, [[0, 1, 2, 3, 4], [0, 7]],
                               [[[j for j in range(5) if j != q] for q in range(5)], [list(range(8, 295))] * 2],
                               mode, 0.1, True, 0.7)
        check_many(f"predict_many {tag}", res, x0, tb, counts, pcounts, [[0, 1, 2, 3, 4], [0, 7]],
                   [[[j for j in range(5) if j != q] for q in range(5)], [list(range(8, 295))] * 2], mode, 0.1, 0.7)
    report(f"widths {tag}")


# ---------------------------------------------------------------------------------------------------- GPU: limits
@pytest.mark.gpu
@pytest.mark.parametrize("fd", ["f16", "f32"])
def test_limits_raise_before_any_row_changes(fd):
    """1537 prompts in a scene and 65536 queries in all are refused before the features are normalised."""
    g = gen("limits", fd)
    dim = 512
    t = prompt_rows(1537, dim, torch.float32, g)
    x0 = feature_rows(300, dim, DT[fd], t[:4], g)
    eng = engine()
    for call in (
            lambda x: eng.predict_queries(x, t, [0], [list(range(1, 1537))], PAIRED, 0.1, True, 0.7),
            lambda x: eng.predict_queries(x, t[:4], [0] * 65536, None, RAW, 0.1, True, 0.7),
            lambda x: eng.predict_many(x, [100, 200], t, [1537, 0], [[0], []], [[list(range(1, 1537))], []], PAIRED,
                                       0.1, True, 0.7),
            lambda x: eng.predict_many(x, [100, 200], t[:4], [2, 2], [[0] * 32768, [1] * 32768], None, RAW, 0.1, True,
                                       0.7)):
        x = x0.clone()
        with pytest.raises(RuntimeError):
            call(x)
        torch.cuda.synchronize()
        assert torch.equal(x, x0)
    # the limits themselves are accepted
    x = x0.clone()
    score, _ = eng.predict_queries(x, t[:1536], [0], [list(range(1, 1536))], PAIRED, 0.1, True, 0.7)
    assert score.shape == (1, 300) and not torch.equal(x, x0)
    score, _ = eng.predict_queries(x0[:2].clone(), t[:4], [0] * 65535, None, RAW, 0.1, True, 0.7)
    assert score.shape == (65535, 2)
