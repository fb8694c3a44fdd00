"""aggregate_views_many against the per-view loop it replaces (the previous aggregate_views_blender_new, copied below),
at 480x640 with 21 objects per view and voxel sizes {None, 0.02, 0.04, 0.06, 0.08}.

The two arms alternate within each pass; every timed output of the batched call is checked bit-equal with the loop's.
The split of one batched call (host instance-map build, H2D, kernels, D2H) comes from a separate profiled pass.
Prints one JSON line per case with the card name and power limit read in the same run.

    python benchmarks/aggregate_bench.py [--passes 7] [--loop-passes-large 3]
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import time

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

from dropclip_b200 import _lib  # noqa: E402
from dropclip_b200._lib import check, current_stream, ptr  # noqa: E402
from dropclip_b200.geometry import aggregate_views_many, binary_masks_to_seg, voxel_down_trace  # noqa: E402

SIZES = [None, 0.02, 0.04, 0.06, 0.08]
INTR = {"fx": 600.0, "fy": 600.0, "cx": 319.5, "cy": 239.5, "height": 480, "width": 640}


def per_view_loop(scene, camera_intrinsic, depth_trunc=25.0, voxel_size=None):
    """The previous aggregate_views_blender_new: one view at a time (host instance map, pageable copies, gathers)."""
    dev = torch.device("cuda")
    from dropclip_b200.projections import backproject
    col_to_ins = scene["col_to_ins"]
    all_p, all_c, all_l = [], [], []
    for _, stuff in scene["views"].items():
        rgb = stuff["rgb"]
        depth = np.ascontiguousarray(stuff["depth"], dtype=np.float32)
        _, binary_masks, colors = zip(*stuff["annos"])
        seg = binary_masks_to_seg(np.stack(binary_masks), np.asarray([col_to_ins[x] for x in colors]))
        d = torch.from_numpy(depth).to(dev)
        valid_m = (d < float(depth_trunc)).reshape(-1)
        d0 = torch.where(d >= float(depth_trunc), torch.zeros_like(d), d)
        keep = (d0 > 0).reshape(-1)
        pts = backproject(d0, camera_intrinsic, o3d_rounding=True)[0].reshape(-1, 3)[keep]
        pts = (pts * torch.tensor([1.0, -1.0, -1.0], dtype=torch.float64, device=dev)).contiguous()
        world = np.ascontiguousarray(np.asarray(stuff["camera"]["world_matrix"]), dtype=np.float64).reshape(16)
        out = torch.empty_like(pts)
        check(_lib.load().dc_transform_points(ptr(pts), pts.shape[0], world.ctypes.data_as(_lib.c_void_p), ptr(out),
                                              current_stream()))
        all_p.append(out)
        all_c.append(torch.from_numpy(np.ascontiguousarray(rgb)).to(dev).reshape(-1, rgb.shape[-1])[keep].to(torch.float64))
        all_l.append(torch.from_numpy(np.ascontiguousarray(seg)).to(dev).reshape(-1)[valid_m].to(torch.int64))
    pts, cols, labs = torch.cat(all_p), torch.cat(all_c), torch.cat(all_l)
    if voxel_size is None:
        return pts.cpu().numpy(), cols.cpu().numpy() / 255.0, labs.cpu().numpy()
    cols = torch.from_numpy(cols.cpu().numpy() / 255.0).to(dev)
    p, c, l, _ = voxel_down_trace(pts, cols, labs, voxel_size)
    return p.cpu().numpy(), c.cpu().numpy(), l.cpu().numpy()


def make_scene(seed, n_views, h=480, w=640, n_obj=21):
    """Blocky instance maps (objects are 40x40-pixel cells), smooth depth 0.5-3 m, camera on a circle."""
    rng = np.random.default_rng(seed)
    col_to_ins = {(i, 0, 7): i for i in range(n_obj)}
    views = {}
    yy, xx = np.mgrid[0:h, 0:w]
    for v in range(n_views):
        cells = rng.integers(0, n_obj, size=(h // 40 + 1, w // 40 + 1))
        seg = cells[yy // 40, xx // 40]
        annos = [(f"o{i}", seg == i, (i, 0, 7)) for i in range(n_obj) if (seg == i).any()]
        depth = (1.5 + 0.8 * np.sin(xx / 97.0 + v) * np.cos(yy / 61.0) + rng.normal(0, 0.01, (h, w))).astype(np.float32)
        a = 2 * np.pi * v / n_views
        pose = np.eye(4)
        pose[:3, :3] = [[np.cos(a), 0, np.sin(a)], [0, 1, 0], [-np.sin(a), 0, np.cos(a)]]
        pose[:3, 3] = (2 * np.sin(a), 0.3, 2 * np.cos(a))
        views[v] = {"rgb": rng.integers(0, 256, size=(h, w, 3), dtype=np.uint8), "depth": depth, "annos": annos,
                    "camera": {"world_matrix": pose}}
    return {"col_to_ins": col_to_ins, "views": views}


def timed(fn):
    torch.cuda.synchronize()
    t = time.perf_counter()
    r = fn()
    torch.cuda.synchronize()
    return r, (time.perf_counter() - t) * 1e3


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 else "unknown"


def split(scenes):
    """One profiled batched call: host time outside device work, and device time per activity kind."""
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CPU, ProfilerActivity.CUDA]) as prof:
        _, total = timed(lambda: aggregate_views_many(scenes, INTR, 25.0, SIZES))
    kinds = {"h2d_ms": 0.0, "d2h_ms": 0.0, "kernels_ms": 0.0}
    for e in prof.events():
        dt = getattr(e, "device_time", None) or getattr(e, "cuda_time", 0.0)
        if e.device_type != torch.autograd.DeviceType.CUDA or not dt:
            continue
        name = e.name.lower()
        if "htod" in name or "host to device" in name:
            kinds["h2d_ms"] += dt / 1e3
        elif "dtoh" in name or "device to host" in name:
            kinds["d2h_ms"] += dt / 1e3
        elif "memcpy" not in name and "memset" not in name:
            kinds["kernels_ms"] += dt / 1e3
    kinds["profiled_call_ms"] = total
    return kinds


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--passes", type=int, default=7)
    ap.add_argument("--loop-passes-large", type=int, default=3, help="loop passes for the 8-scene case (about 1 min each)")
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    gpu = card()
    rows = []
    for n_views, n_scenes in ((8, 1), (73, 1), (73, 8)):
        scenes = [make_scene(100 * n_views + s, n_views) for s in range(n_scenes)]
        aggregate_views_many(scenes, INTR, 25.0, SIZES)  # warm-up: module load, pinned pools
        per_view_loop(scenes[0], INTR, 25.0, SIZES[1])
        t_many, t_loop = [], []
        loop_passes = args.passes if n_scenes == 1 else min(args.passes, args.loop_passes_large)
        torch.cuda.reset_peak_memory_stats()
        for p in range(args.passes):
            out, t = timed(lambda: aggregate_views_many(scenes, INTR, 25.0, SIZES))
            t_many.append(t)
            if p < loop_passes:
                ref, t = timed(lambda: [[per_view_loop(sc, INTR, 25.0, vs) for vs in SIZES] for sc in scenes])
                t_loop.append(t)
                for s in range(n_scenes):
                    for k in range(len(SIZES)):
                        assert all(np.array_equal(a, b) and a.dtype == b.dtype for a, b in zip(out[s][k], ref[s][k])), \
                            f"batched result differs: scene {s}, size {SIZES[k]}"
        peak = torch.cuda.max_memory_allocated() / 2**30
        row = {"case": f"V={n_views}, {n_scenes} scene(s), 480x640, 21 objects, sizes {SIZES}", "gpu": gpu,
               "many_ms": {"median": statistics.median(t_many), "min": min(t_many), "max": max(t_many), "passes": len(t_many)},
               "loop_ms": {"median": statistics.median(t_loop), "min": min(t_loop), "max": max(t_loop), "passes": len(t_loop)},
               "bit_equal": True, "peak_device_GiB": round(peak, 2),
               "points_per_scene": int(out[0][0][0].shape[0]),
               "voxels_per_scene": [int(out[0][k][0].shape[0]) for k in range(1, len(SIZES))],
               "split_one_call": split(scenes)}
        print(json.dumps(row), flush=True)
        rows.append(row)
        del scenes, out, ref
    if args.out:
        os.makedirs(os.path.dirname(args.out) or ".", exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(rows, f, indent=1)


if __name__ == "__main__":
    main()
