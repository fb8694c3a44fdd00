"""Grounding every text query of a scene: the per-query `ClipSimilarity.predict` loop of the reference's evaluation
scripts (tools/validate_upper_bound.py:200-218, scene negatives) against one `ClipSimilarity.predict_queries` call.

Three shapes, fp16 features, C = 768:
  (a) eval:    N = 10 k,  Q = 21  (the evaluation size: launches and host work dominate)
  (b) q21:     N = 200 k, Q = 21  (throughput; 256 MB of L2-overwriting writes before every pass)
  (c) q256:    N = 200 k, Q = 256 (as (b); 256 distinct prompts fill the GEMM's widest tile)
The two paths alternate within one run, each pass timed by a host clock around work that ends in a device synchronise,
after warm-up; the median of --runs passes is reported. The text tower is a table lookup defined here (one fixed
random embedding per text), so the timings cover everything after a real tower's encode_text.
Outputs are compared in the same run: per-query predict on a clone of the features against predict_queries, scores
within 1e-5, predictions equal wherever the score is further than 1e-4 from the threshold.
Prints one JSON line."""
import argparse
import json
import os
import statistics
import subprocess
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np  # noqa: E402
import torch  # noqa: E402

from dropclip_b200.similarity import ClipSimilarity  # noqa: E402

THR = 0.7


class TableTower:
    """encode_text(tokens) = a fixed random fp16 row per token; tokenize assigns each new text the next row."""

    def __init__(self, dim, vocab=4096, seed=7):
        g = torch.Generator().manual_seed(seed)
        self.table = torch.randn((vocab, dim), generator=g).half().cuda()
        self.ids = {}

    def tokenize(self, texts):
        texts = [texts] if isinstance(texts, str) else texts
        return torch.tensor([self.ids.setdefault(t, len(self.ids)) for t in texts], dtype=torch.long)

    def encode_text(self, tok):
        return self.table[tok.to(self.table.device)]

    def eval(self):
        return self

    def to(self, *_):
        return self


def gpu_info():
    info = {"gpu": torch.cuda.get_device_name(0)}
    try:
        r = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30)
        power, clock = r.stdout.strip().splitlines()[0].split(",")
        info["power_limit"] = power.strip()
        info["max_sm_clock"] = clock.strip()
    except Exception as exc:  # pragma: no cover - depends on the machine
        info["power_limit"] = f"unknown ({exc!r})"
    return info


def make_scene(n, q, dim, tower, seed):
    queries = [f"object {i}" for i in range(q)]
    emb = tower.encode_text(tower.tokenize(queries)).float()
    emb /= emb.norm(dim=-1, keepdim=True)
    g = torch.Generator(device="cuda").manual_seed(seed)
    owner = torch.randint(0, q + 1, (n,), generator=g, device="cuda")
    feat = 0.05 * torch.randn((n, dim), generator=g, device="cuda")
    near = owner < q
    feat[near] += 0.6 * emb[owner[near]]
    return feat.half(), queries


def loop(cs, x, queries):
    """The reference's loop body: predict(output.half(), query, the scene's other queries) per query. `output.half()`
    of fp16 features is the tensor itself, so every call normalises the same rows in place again."""
    out = []
    for t in queries:
        out.append(cs.predict(x, t, [y for y in queries if y != t]))
    return out


def check(cs, feat, queries):
    """Per-query predict on a clone of the features against predict_queries; returns the largest score difference."""
    pred, sims = cs.predict_queries(feat.clone(), queries)
    worst = 0.0
    for q, t in enumerate(queries):
        wp, ws = cs.predict(feat.clone(), t, [y for y in queries if y != t])
        worst = max(worst, (sims[q] - ws).abs().max().item())
        sure = (ws - THR).abs() > 1e-4
        if not torch.equal(pred[q][sure], wp[sure]):
            raise AssertionError(f"query {q}: predictions differ away from the threshold")
    if worst > 1e-5:
        raise AssertionError(f"scores differ by {worst:.3e} > 1e-5")
    return worst


def bench_shape(name, n, q, runs, flush_l2, dim=768):
    tower = TableTower(dim)
    cs = ClipSimilarity(model=tower, tokenize=tower.tokenize, device="cuda", method="paired", threshold=THR)
    feat, queries = make_scene(n, q, dim, tower, seed=n + q)
    max_diff = check(cs, feat, queries)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda") if flush_l2 else None
    paths = {"per_query_loop": lambda x: loop(cs, x, queries), "predict_queries": lambda x: cs.predict_queries(x, queries)}
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
    return {"shape": name, "n_points": n, "n_queries": q, "dim": dim, "dtype": "fp16", "negatives": "scene",
            "l2": "256 MB overwritten before every pass" if flush_l2 else "not flushed",
            "runs": runs, "per_query_loop_ms": round(med["per_query_loop"], 3), "predict_queries_ms": round(med["predict_queries"], 3),
            "speedup": round(med["per_query_loop"] / med["predict_queries"], 2),
            "per_query_loop_ms_all": [round(v, 3) for v in times["per_query_loop"]],
            "predict_queries_ms_all": [round(v, 3) for v in times["predict_queries"]],
            "outputs_agree": True, "max_score_diff": max_diff}


def main():
    ap = argparse.ArgumentParser(description=__doc__.splitlines()[0])
    ap.add_argument("--runs", type=int, default=7, help="timed passes per path and shape (median reported, >= 5)")
    ap.add_argument("--shapes", default="eval,q21,q256")
    args = ap.parse_args()
    if args.runs < 5:
        ap.error("--runs must be at least 5")
    if not torch.cuda.is_available():
        raise SystemExit("grounding_queries_bench.py needs a CUDA device")
    shapes = {"eval": (10_000, 21, False), "q21": (200_000, 21, True), "q256": (200_000, 256, True)}
    res = {"bench": "grounding_queries", **gpu_info(), "shapes": []}
    for s in args.shapes.split(","):
        n, q, flush = shapes[s]
        res["shapes"].append(bench_shape(s, n, q, args.runs, flush))
    print(json.dumps(res))


if __name__ == "__main__":
    main()
