"""Pixel-level fusion (use_obj_prior=0) over a stream of scenes: a loop of `MultiviewFeatureFusion.fuse` against one
`MultiviewFeatureFusion.fuse_many` over the same scenes, i.e. the pixel arm of the reference's ablation driver
(scripts/run_eval.py:205-220) before and after.

Two sizes, N = 100 k points, 480 x 640, C = 768 fp32 patch maps of 24 x 32, sim kernel max, norm_feat:
  (a) v8:  16 scenes x 8 views
  (b) v73:  8 scenes x 73 views (MV-TOD)
The scenes are built by `scenes.make_scene(..., pixel_features=True, feature_dtype=torch.float32)` and handed over as
host numpy arrays and CPU tensors, as run_eval.py hands them. The two paths alternate within one run; each pass over
all scenes is timed by a host clock around work that ends in a device synchronise, after one warm-up round, and the
median and range of --runs passes are reported as scenes/s. Host -> device bytes per scene are computed from the
shapes (the int64 instance maps travel as one byte per pixel); the pinned host -> device copy rate measured in the same
run is their bound. Before any number is printed every output of the stream is compared with `fuse` on the same
scene: visibility and returned rows exactly; features and similarity weights bit for bit is not promised on the
tcgen05 path (its atomics add in no fixed order), so their largest difference is reported and must stay within 1e-5.
Prints one JSON line."""
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

from dropclip_b200.feature_fusion import MultiviewFeatureFusion  # noqa: E402
from dropclip_b200.scenes import MVTOD_INTRINSIC, make_scene  # noqa: E402
from grounding_queries_bench import gpu_info  # noqa: E402


def scene_args(seed, n_views, n_points):
    sc = make_scene(seed, n_views=n_views, n_points=n_points, pixel_features=True, feature_dtype=torch.float32, device="cuda")
    return (sc.points, sc.colors, sc.labels, sc.depths, sc.seg_masks, sc.camera_poses, sc.mv_features, sc.query_embeddings)


def h2d_bytes(a):
    points, colors, labels, depths, segs, poses, feats, query = a
    n = (points.nbytes + colors.nbytes + labels.nbytes + sum(d.nbytes for d in depths) + sum(s.size for s in segs)
         + sum(f.numel() * 4 for f in feats) + query.numel() * 4)
    return n + len(poses) * 16 * 8 + 9 * 8  # inverse poses and intrinsics in fp64 (offset tables not counted)


def pinned_h2d_gbps(nbytes=256 << 20, reps=9):
    src = torch.empty(nbytes, dtype=torch.uint8, pin_memory=True)
    dst = torch.empty(nbytes, dtype=torch.uint8, device="cuda")
    rates = []
    for i in range(reps + 1):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        dst.copy_(src, non_blocking=True)
        b.record()
        b.synchronize()
        if i:
            rates.append(nbytes / (a.elapsed_time(b) * 1e-3) / 1e9)
    return statistics.median(rates)


def compare(M, scenes):
    """Every fuse_many output against fuse; returns (largest feature difference, largest weight difference, bitwise)."""
    worst_f = worst_w = 0.0
    bitwise = True
    for a, ((f2, v2, w2), rows2) in zip(scenes, M.fuse_many(scenes, device="cuda")):
        (f1, v1, w1), rows1 = M.fuse(*a, device="cuda")
        if not torch.equal(v1, v2) or not all(x.dtype == y.dtype and np.array_equal(x, y) for x, y in zip(rows1, rows2)):
            raise AssertionError("visibility or returned rows differ between fuse and fuse_many")
        for x, y, name in ((f1, f2, "f"), (w1, w2, "w")):
            if not torch.equal(x.isnan(), y.isnan()):
                raise AssertionError("NaN rows differ between fuse and fuse_many")
            bitwise &= torch.equal(x.view(torch.int32), y.view(torch.int32))
            diff = (x - y)[~x.isnan()].abs()
            d = float(diff.max()) if diff.numel() else 0.0
            if name == "f":
                worst_f = max(worst_f, d)
            else:
                worst_w = max(worst_w, d)
    if max(worst_f, worst_w) > 1e-5:
        raise AssertionError(f"fuse_many differs from fuse by {max(worst_f, worst_w):.3e}")
    return worst_f, worst_w, bitwise


def bench_size(name, n_scenes, n_views, n_points, runs):
    M = MultiviewFeatureFusion(MVTOD_INTRINSIC, use_visibility=1, use_similarity=1, use_sim_kernel="max", use_obj_prior=0,
                               norm_feat=True, device="cuda")
    scenes = [scene_args(1234 + i, n_views, n_points) for i in range(n_scenes)]
    torch.cuda.synchronize()
    worst_f, worst_w, bitwise = compare(M, scenes)

    def loop():
        return [M.fuse(*a, device="cuda") for a in scenes]

    def many():
        return list(M.fuse_many(scenes, device="cuda"))

    times = {"fuse_loop": [], "fuse_many": []}
    for it in range(runs + 1):  # one warm-up round
        for k, fn in (("fuse_loop", loop), ("fuse_many", many)):
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            out = fn()
            torch.cuda.synchronize()
            dt = time.perf_counter() - t0
            del out
            if it:
                times[k].append(n_scenes / dt)
    per_scene = statistics.median(h2d_bytes(a) for a in scenes)
    res = {"size": name, "scenes": n_scenes, "views": n_views, "points": n_points, "image": [480, 640], "dim": 768,
           "patch": [24, 32], "runs": runs, "h2d_mb_per_scene": round(per_scene / 1e6, 1),
           "max_feature_diff": worst_f, "max_weight_diff": worst_w, "bitwise_equal": bitwise}
    for k, v in times.items():
        res[f"{k}_scenes_per_s"] = round(statistics.median(v), 2)
        res[f"{k}_scenes_per_s_range"] = [round(min(v), 2), round(max(v), 2)]
    res["speedup"] = round(res["fuse_many_scenes_per_s"] / res["fuse_loop_scenes_per_s"], 3)
    return res


def main():
    ap = argparse.ArgumentParser(description=__doc__.splitlines()[0])
    ap.add_argument("--runs", type=int, default=7, help="timed passes per path and size (median reported, >= 5)")
    ap.add_argument("--sizes", default="v8,v73")
    args = ap.parse_args()
    if args.runs < 5:
        ap.error("--runs must be at least 5")
    if not torch.cuda.is_available():
        raise SystemExit("pixel_stream_bench.py needs a CUDA device")
    sizes = {"v8": (16, 8, 100_000), "v73": (8, 73, 100_000)}
    res = {"bench": "pixel_stream", **gpu_info(), "pinned_h2d_gb_per_s": None, "sizes": []}
    res["pinned_h2d_gb_per_s"] = round(pinned_h2d_gbps(), 1)
    for s in args.sizes.split(","):
        r = bench_size(s, *sizes[s], args.runs)
        r["h2d_bound_scenes_per_s"] = round(res["pinned_h2d_gb_per_s"] * 1e9 / (r["h2d_mb_per_scene"] * 1e6), 1)
        res["sizes"].append(r)
    print(json.dumps(res))


if __name__ == "__main__":
    main()
