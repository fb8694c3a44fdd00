"""The grounding evaluation of a batch of scenes, from the point features to mIoU and Pr@k: the loop INTEGRATION.md §4
shows (one `ClipSimilarity.predict_many`, then per query a ground-truth mask built from the point labels and
`trainMetricPC` over the lists, engine/distil.py:436-493, tools/validate_upper_bound.py:200-221) against one
`ClipSimilarity.predict_many_iou` followed by `metrics.grounding_scores`.

The four batches of grounding_batch_bench.py, fp16 features, C = 768, scene negatives, paired method:
  (a) val16:   16 scenes x 10 k points x 21 queries
  (b) val64:   64 x 10 k x 21 (1344 queries)
  (c) ragged8: 8 scenes, N in [1 k, 100 k], Q in [1, 40] (seeded)
  (d) big4:    4 x 200 k x 21, 256 MB of L2-overwriting writes before every pass
Point labels are int64 object ids (0: background; the points near query i's embedding carry id i + 1), and query i
has one to three ids (i + 1, then i + 2 and i + 3 for every second and third query).
The two paths alternate within one run, each pass timed by a host clock around work that ends in a device synchronise,
after two warm-up rounds; the median and the range of --runs passes are reported. The text tower is a table lookup
(grounding_queries_bench.TableTower), so the timings cover everything after a real tower's encode_text.
In the same run the two paths must give equal (inter, union) counts for every query, a bit-equal mIoU and equal Pr@k.
Prints one JSON line with the GPU's name and power limit."""
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

from dropclip_b200.metrics import binary_iou_counts, grounding_scores, trainMetricPC  # noqa: E402
from dropclip_b200.similarity import ClipSimilarity  # noqa: E402
from grounding_queries_bench import TableTower, gpu_info  # noqa: E402

THR = 0.7
PR_IOUS = [0.25, 0.5, 0.75]


def make_batch(shapes, dim, tower, seed):
    g = torch.Generator(device="cuda").manual_seed(seed)
    feats, labels, obj = [], [], []
    for s, (n, q) in enumerate(shapes):
        qs = [f"scene {s} object {i}" for i in range(q)]
        emb = tower.encode_text(tower.tokenize(qs)).float()
        emb /= emb.norm(dim=-1, keepdim=True)
        owner = torch.randint(0, q + 1, (n,), generator=g, device="cuda")
        f = 0.05 * torch.randn((n, dim), generator=g, device="cuda")
        near = owner < q
        f[near] += 0.6 * emb[owner[near]]
        feats.append(f.half())
        labels.append(torch.where(near, owner + 1, 0))
        obj.append({t: [i + 1 + k for k in range(1 + i % 3)] for i, t in enumerate(qs)})
    return torch.cat(feats).contiguous(), [n for n, _ in shapes], torch.cat(labels), obj


def loop_path(cs, x, counts, labels, obj):
    """INTEGRATION.md §4: predict_many, a ground-truth mask per query, trainMetricPC over the lists."""
    res = cs.predict_many(x, counts, [list(o) for o in obj])
    pred_list, gt_list = [], []
    for (preds, _), label_d, obj_queries in zip(res, torch.split(labels, counts), obj):
        for pred, obj_ids in zip(preds, obj_queries.values()):
            gt = torch.zeros_like(label_d)
            for ob in obj_ids:
                gt[label_d == ob] = True
            pred_list.append(pred)
            gt_list.append(gt)
    return trainMetricPC(pred_list, gt_list, pr_ious=PR_IOUS, sigmoid=False), pred_list, gt_list


def fused_path(cs, x, counts, labels, obj):
    counts_iou = cs.predict_many_iou(x, counts, labels, obj)
    return grounding_scores(*counts_iou, pr_ious=PR_IOUS), counts_iou


def check(cs, feat, counts, labels, obj):
    """Equal counts per query, bit-equal mIoU and equal Pr@k; returns the metrics."""
    (miou, prs), pred_list, gt_list = loop_path(cs, feat.clone(), counts, labels, obj)
    (miou2, prs2), (inter2, union2) = fused_path(cs, feat.clone(), counts, labels, obj)
    inter, union = binary_iou_counts(pred_list, gt_list, 0.35, in_place=False)
    if not (torch.equal(inter, inter2) and torch.equal(union, union2)):
        raise AssertionError("per-query counts differ")
    if not (torch.equal(miou, miou2) and [p.item() for p in prs] == [p.item() for p in prs2]):
        raise AssertionError(f"metrics differ: {miou.item()} {[p.item() for p in prs]} / {miou2.item()} "
                             f"{[p.item() for p in prs2]}")
    return {"miou": round(miou.item(), 4), "pr": [round(p.item(), 4) for p in prs]}


def bench_batch(name, shapes, runs, flush_l2, dim=768):
    tower = TableTower(dim)
    cs = ClipSimilarity(model=tower, tokenize=tower.tokenize, device="cuda", method="paired", threshold=THR)
    feat, counts, labels, obj = make_batch(shapes, dim, tower, seed=len(shapes))
    metrics = check(cs, feat, counts, labels, obj)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda") if flush_l2 else None
    paths = {"loop": lambda x: loop_path(cs, x, counts, labels, obj), "fused": lambda x: fused_path(cs, x, counts, labels, obj)}
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
    return {"batch": name, "scenes": len(shapes), "n_points": counts, "n_queries": [len(o) for o in obj], "dim": dim,
            "dtype": "fp16", "labels": "int64", "negatives": "scene",
            "l2": "256 MB overwritten before every pass" if flush_l2 else "not flushed", "runs": runs,
            "loop_ms": round(med["loop"], 3), "predict_many_iou_ms": round(med["fused"], 3),
            "speedup": round(med["loop"] / med["fused"], 2),
            "loop_ms_range": [round(min(times["loop"]), 3), round(max(times["loop"]), 3)],
            "predict_many_iou_ms_range": [round(min(times["fused"]), 3), round(max(times["fused"]), 3)], **metrics}


def main():
    ap = argparse.ArgumentParser(description=__doc__.splitlines()[0])
    ap.add_argument("--runs", type=int, default=9, help="timed passes per path and batch (median reported, >= 7)")
    ap.add_argument("--batches", default="val16,val64,ragged8,big4")
    args = ap.parse_args()
    if args.runs < 7:
        ap.error("--runs must be at least 7")
    if not torch.cuda.is_available():
        raise SystemExit("grounding_eval_bench.py needs a CUDA device")
    rng = np.random.default_rng(8)
    ragged = list(zip(rng.integers(1_000, 100_001, 8).tolist(), rng.integers(1, 41, 8).tolist()))
    batches = {"val16": ([(10_000, 21)] * 16, False), "val64": ([(10_000, 21)] * 64, False),
               "ragged8": (ragged, False), "big4": ([(200_000, 21)] * 4, True)}
    res = {"bench": "grounding_eval", **gpu_info(), "batches": []}
    for b in args.batches.split(","):
        shapes, flush = batches[b]
        res["batches"].append(bench_batch(b, shapes, args.runs, flush))
    print(json.dumps(res))


if __name__ == "__main__":
    main()
