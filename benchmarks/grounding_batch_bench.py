"""Grounding every text query of a batch of scenes: a loop of `ClipSimilarity.predict_queries` over the scenes (what
the reference's evaluation loops become per scene, engine/distil.py:436-458, tools/validate_upper_bound.py:200-218)
against one `ClipSimilarity.predict_many` call.

Four batches, fp16 features, C = 768, scene negatives:
  (a) val16:   16 scenes x 10 k points x 21 queries (the validation shape: per-scene launches and host work dominate)
  (b) val64:   64 x 10 k x 21
  (c) ragged8: 8 scenes, N in [1 k, 100 k], Q in [1, 40] (seeded)
  (d) big4:    4 x 200 k x 21, 256 MB of L2-overwriting writes before every pass
The two paths alternate within one run, each pass timed by a host clock around work that ends in a device synchronise,
after two warm-up rounds; the median and the spread of --runs passes are reported. The text tower is a table lookup
(grounding_queries_bench.TableTower), so the timings cover everything after a real tower's encode_text.
Outputs are compared in the same run: every scene's predict_many result against predict_queries on a clone of its
rows; the largest score difference is reported, and predictions must be equal wherever the score is further than 1e-5
from the threshold. Prints one JSON line."""
import argparse
import json
import os
import statistics
import sys
import time

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(HERE))
sys.path.insert(0, HERE)
import numpy as np  # noqa: E402
import torch  # noqa: E402

from dropclip_b200.similarity import ClipSimilarity  # noqa: E402
from grounding_queries_bench import TableTower, gpu_info  # noqa: E402

THR = 0.7


def make_batch(shapes, dim, tower, seed):
    g = torch.Generator(device="cuda").manual_seed(seed)
    feats, queries = [], []
    for s, (n, q) in enumerate(shapes):
        qs = [f"scene {s} object {i}" for i in range(q)]
        emb = tower.encode_text(tower.tokenize(qs)).float()
        emb /= emb.norm(dim=-1, keepdim=True)
        owner = torch.randint(0, q + 1, (n,), generator=g, device="cuda")
        f = 0.05 * torch.randn((n, dim), generator=g, device="cuda")
        near = owner < q
        f[near] += 0.6 * emb[owner[near]]
        feats.append(f.half())
        queries.append(qs)
    return torch.cat(feats).contiguous(), [n for n, _ in shapes], queries


def loop(cs, x, counts, queries):
    return [cs.predict_queries(xs, qs) for xs, qs in zip(torch.split(x, counts), queries)]


def check(cs, feat, counts, queries):
    """predict_many against predict_queries per scene on clones; returns the largest score difference."""
    res = cs.predict_many(feat.clone(), counts, queries)
    worst = 0.0
    for (pred, sims), xs, qs in zip(res, torch.split(feat, counts), queries):
        wp, ws = cs.predict_queries(xs.clone(), qs)
        worst = max(worst, (sims - ws).abs().max().item())
        sure = (ws - THR).abs() > 1e-5
        if not torch.equal(pred[sure], wp[sure]):
            raise AssertionError("predictions differ away from the threshold")
    return worst


def bench_batch(name, shapes, runs, flush_l2, dim=768):
    tower = TableTower(dim)
    cs = ClipSimilarity(model=tower, tokenize=tower.tokenize, device="cuda", method="paired", threshold=THR)
    feat, counts, queries = make_batch(shapes, dim, tower, seed=len(shapes))
    max_diff = check(cs, feat, counts, queries)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda") if flush_l2 else None
    paths = {"predict_queries_loop": lambda x: loop(cs, x, counts, queries),
             "predict_many": lambda x: cs.predict_many(x, counts, queries)}
    times = {k: [] for k in paths}
    for it in range(runs + 2):  # two warm-up rounds
        for k, fn in paths.items():
            x = feat.clone()
            if flush is not None:
                flush.zero_()  # 256 MB > the 126 MB L2: S and the features come from HBM
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            fn(x)
            torch.cuda.synchronize()
            if it >= 2:
                times[k].append((time.perf_counter() - t0) * 1e3)
    med = {k: statistics.median(v) for k, v in times.items()}
    return {"batch": name, "scenes": len(shapes), "n_points": counts, "n_queries": [len(q) for q in queries], "dim": dim,
            "dtype": "fp16", "negatives": "scene",
            "l2": "256 MB overwritten before every pass" if flush_l2 else "not flushed", "runs": runs,
            "predict_queries_loop_ms": round(med["predict_queries_loop"], 3), "predict_many_ms": round(med["predict_many"], 3),
            "speedup": round(med["predict_queries_loop"] / med["predict_many"], 2),
            "predict_queries_loop_ms_range": [round(min(times["predict_queries_loop"]), 3), round(max(times["predict_queries_loop"]), 3)],
            "predict_many_ms_range": [round(min(times["predict_many"]), 3), round(max(times["predict_many"]), 3)],
            "max_score_diff": max_diff}


def main():
    ap = argparse.ArgumentParser(description=__doc__.splitlines()[0])
    ap.add_argument("--runs", type=int, default=9, help="timed passes per path and batch (median reported, >= 7)")
    ap.add_argument("--batches", default="val16,val64,ragged8,big4")
    args = ap.parse_args()
    if args.runs < 7:
        ap.error("--runs must be at least 7")
    if not torch.cuda.is_available():
        raise SystemExit("grounding_batch_bench.py needs a CUDA device")
    rng = np.random.default_rng(8)
    ragged = list(zip(rng.integers(1_000, 100_001, 8).tolist(), rng.integers(1, 41, 8).tolist()))
    batches = {"val16": ([(10_000, 21)] * 16, False), "val64": ([(10_000, 21)] * 64, False),
               "ragged8": (ragged, False), "big4": ([(200_000, 21)] * 4, True)}
    res = {"bench": "grounding_batch", **gpu_info(), "batches": []}
    for b in args.batches.split(","):
        shapes, flush = batches[b]
        res["batches"].append(bench_batch(b, shapes, args.runs, flush))
    print(json.dumps(res))


if __name__ == "__main__":
    main()
