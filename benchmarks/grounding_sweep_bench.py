"""The grounding evaluation of a batch of scenes at T thresholds (choosing `sim_norm_thresh` on a validation set, or
reporting mIoU / Pr@k against it): T `ClipSimilarity.predict_many_iou` calls, each on a fresh clone of the features
(`predict` normalises them in place, quirk q15), against one `ClipSimilarity.predict_many_iou_sweep` on one clone.
T in {1, 11, 101}; the four batches and the batch builder of grounding_eval_bench.py (fp16 features, C = 768, scene
negatives, paired method, int64 labels):
  (a) val16:   16 scenes x 10 k points x 21 queries
  (b) val64:   64 x 10 k x 21 (1344 queries)
  (c) ragged8: 8 scenes, N in [1 k, 100 k], Q in [1, 40] (seeded)
  (d) big4:    4 x 200 k x 21, 256 MB of L2-overwriting writes before every pass
Also timed in the same run, with the clone outside the timed region as the other grounding benchmarks time them:
one `predict_many` and one `predict_many_iou` (to compare with their recorded ranges), and the sweep at T = 1 (its
difference to `predict_many_iou` is the cost of the histogram pass over the counting pass).
Every path alternates with the others within one run, each pass timed by a host clock around work that ends in a device
synchronise, after two warm-up rounds; the median and the range of --runs passes are reported. Before timing, the sweep
must give the loop's (inter, union) for every threshold and query. Prints one JSON line with the GPU's name and power
limit."""
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
from grounding_eval_bench import THR, make_batch  # noqa: E402
from grounding_queries_bench import TableTower, gpu_info  # noqa: E402

SWEEPS = {1: [THR], 11: [0.05 + 0.09 * i for i in range(11)], 101: [0.01 * i for i in range(1, 102)]}


def loop(cs, feat, counts, labels, obj, thresholds):
    rows = [cs.predict_many_iou(feat.clone(), counts, labels, obj, threshold=t) for t in thresholds]
    return torch.stack([r[0] for r in rows]), torch.stack([r[1] for r in rows])


def sweep(cs, feat, counts, labels, obj, thresholds):
    return cs.predict_many_iou_sweep(feat.clone(), counts, labels, obj, thresholds)


def bench_batch(name, shapes, runs, flush_l2, dim=768):
    tower = TableTower(dim)
    cs = ClipSimilarity(model=tower, tokenize=tower.tokenize, device="cuda", method="paired", threshold=THR)
    feat, counts, labels, obj = make_batch(shapes, dim, tower, seed=len(shapes))
    queries = [list(o) for o in obj]
    for t, thr in SWEEPS.items():
        want, got = loop(cs, feat, counts, labels, obj, thr), sweep(cs, feat, counts, labels, obj, thr)
        if not (torch.equal(want[0], got[0]) and torch.equal(want[1], got[1])):
            raise AssertionError(f"{name}, T = {t}: the sweep's counts differ from the loop's")
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda") if flush_l2 else None
    # (clone inside the timed region, path)
    paths = {"predict_many": (False, lambda x: cs.predict_many(x, counts, queries)),
             "predict_many_iou": (False, lambda x: cs.predict_many_iou(x, counts, labels, obj)),
             "sweep_T1_clone_outside": (False, lambda x: cs.predict_many_iou_sweep(x, counts, labels, obj, [THR]))}
    for t, thr in SWEEPS.items():
        paths[f"loop_T{t}"] = (True, lambda x, thr=thr: loop(cs, feat, counts, labels, obj, thr))
        paths[f"sweep_T{t}"] = (True, lambda x, thr=thr: sweep(cs, feat, counts, labels, obj, thr))
    times = {k: [] for k in paths}
    for it in range(runs + 2):  # two warm-up rounds
        for k, (clone_inside, fn) in paths.items():
            x = None if clone_inside else feat.clone()
            if flush is not None:
                flush.zero_()  # 256 MB > the 126 MB L2: S and the features come from HBM
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            fn(x)
            torch.cuda.synchronize()
            if it >= 2:
                times[k].append((time.perf_counter() - t0) * 1e3)
    ms = {k: {"median": round(statistics.median(v), 3), "range": [round(min(v), 3), round(max(v), 3)]}
          for k, v in times.items()}
    speedup = {f"T{t}": round(ms[f"loop_T{t}"]["median"] / ms[f"sweep_T{t}"]["median"], 2) for t in SWEEPS}
    return {"batch": name, "scenes": len(shapes), "n_points": counts, "n_queries": [len(o) for o in obj], "dim": dim,
            "dtype": "fp16", "labels": "int64", "negatives": "scene",
            "l2": "256 MB overwritten before every pass" if flush_l2 else "not flushed", "runs": runs,
            "thresholds": {f"T{t}": [min(v), max(v)] for t, v in SWEEPS.items()}, "ms": ms, "loop_over_sweep": speedup}


def main():
    ap = argparse.ArgumentParser(description=__doc__.splitlines()[0])
    ap.add_argument("--runs", type=int, default=9, help="timed passes per path and batch (median reported, >= 7)")
    ap.add_argument("--batches", default="val16,val64,ragged8,big4")
    args = ap.parse_args()
    if args.runs < 7:
        ap.error("--runs must be at least 7")
    if not torch.cuda.is_available():
        raise SystemExit("grounding_sweep_bench.py needs a CUDA device")
    rng = np.random.default_rng(8)
    ragged = list(zip(rng.integers(1_000, 100_001, 8).tolist(), rng.integers(1, 41, 8).tolist()))
    batches = {"val16": ([(10_000, 21)] * 16, False), "val64": ([(10_000, 21)] * 64, False),
               "ragged8": (ragged, False), "big4": ([(200_000, 21)] * 4, True)}
    res = {"bench": "grounding_sweep", **gpu_info(), "batches": []}
    for b in args.batches.split(","):
        shapes, flush = batches[b]
        res["batches"].append(bench_batch(b, shapes, args.runs, flush))
    print(json.dumps(res))


if __name__ == "__main__":
    main()
