#!/usr/bin/env python
"""Benchmark of the hot path: object-level multi-view fusion with semantic view selection
(BASELINE.json configs[1]): per GPU a batch of 64 synthetic MV-TOD-shaped scenes, V=73 views of
480x640, N=100k points, Q=21 objects, C=768, production flags of tools/preprocess_data.py:177-185.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]

One "step" = one pass of the hot path over one batch. `value` = scenes/s with inputs resident in
HBM; `e2e` = the same metric through the reference-shaped call MultiviewFeatureFusion.fuse() with
host numpy inputs (pinned staging + H2D + D2H inside the timed region). `--impl reference` times
the CPU restatement of the reference's own torch/numpy path (oracle/fusion_ref.py; the reference is
pure Python and is not part of this repository) on the host cores.

`--dump-outputs DIR` writes what the last timed step computed (rank 0) as DIR/<name>.npy, float32 or
float64, under 64 MB in all; see dump_outputs(). The inputs are generated from fixed seeds, so two
builds run with the same arguments can be compared output for output.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time
import zlib

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402
import torch  # noqa: E402

WORKLOAD = "mvtod_object_fusion_sim_max_batch64_V73_N100k_Q21_C768"


def positive_int(s):
    v = int(s)
    if v < 1:
        raise argparse.ArgumentTypeError("must be >= 1")
    return v


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=positive_int, default=10,
                    help="timed steps of the headline, one-stream, full-output, uint8-map and e2e loops")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--scenes", type=int, default=64, help="scenes per GPU per step")
    ap.add_argument("--unique", type=int, default=64, help="distinct generated scenes per GPU (replicated to --scenes if fewer)")
    ap.add_argument("--job-scenes", type=int, default=-1, help="distinct scenes of the configs[2] job (-1: 1000 at N>1, 256 at N=1; 0: skip)")
    ap.add_argument("--views", type=int, default=73)
    ap.add_argument("--points", type=int, default=100_000)
    ap.add_argument("--objects", type=int, default=21)
    ap.add_argument("--e2e-scenes", type=int, default=4, help="scenes per e2e step through the host API")
    ap.add_argument("--e2e-batch", type=int, default=4, help="scenes per launch sequence of the e2e pipeline")
    ap.add_argument("--e2e-slots", type=int, default=12, help="pinned scene slots (= distinct scenes) of the e2e pipeline")
    ap.add_argument("--e2e-pipeline-scenes", type=int, default=480, help="scenes timed through the e2e pipeline per GPU")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-extras", action="store_true", help="skip the supplementary configs 4/5 (pixel-level fusion, grounding)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the outputs of the last timed step as DIR/<name>.npy (rank 0)")
    return ap.parse_args()


# ---------------------------------------------------------------------------------------------- clocks
class ClockSampler:
    """SM clock and throttle reasons sampled in-process through NVML while the step loop runs.
    (An external `nvidia-smi -lms 20` poller was measured to slow the kernels by ~1.6x; NVML calls
    from a Python thread every 10 ms do not.)"""

    def __init__(self, gpu_index: int):
        self.gpu = gpu_index
        self.sm, self.reasons = [], set()
        self.max_mhz = None
        self._stop = threading.Event()
        self._thread = None

    def _run(self):
        try:
            import pynvml as nv
            nv.nvmlInit()
            visible = os.environ.get("CUDA_VISIBLE_DEVICES")
            idx = int(visible.split(",")[self.gpu]) if visible and visible.split(",")[self.gpu].isdigit() else self.gpu
            h = nv.nvmlDeviceGetHandleByIndex(idx)
            self.max_mhz = float(nv.nvmlDeviceGetMaxClockInfo(h, nv.NVML_CLOCK_SM))
            names = {"hw_slowdown": nv.nvmlClocksThrottleReasonHwSlowdown,
                     "hw_thermal_slowdown": nv.nvmlClocksThrottleReasonHwThermalSlowdown,
                     "sw_thermal_slowdown": nv.nvmlClocksThrottleReasonSwThermalSlowdown,
                     "sw_power_cap": nv.nvmlClocksThrottleReasonSwPowerCap}
            while not self._stop.is_set():
                self.sm.append(float(nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM)))
                bits = nv.nvmlDeviceGetCurrentClocksThrottleReasons(h)
                for k, m in names.items():
                    if bits & m:
                        self.reasons.add(k)
                self._stop.wait(0.01)
        except Exception as exc:  # pragma: no cover - NVML missing
            self.error = repr(exc)

    def start(self):
        self._thread = threading.Thread(target=self._run, daemon=True)
        self._thread.start()

    def stop(self):
        self._stop.set()
        if self._thread is not None:
            self._thread.join(2.0)
        if not self.sm:
            return {"sm_mhz": None, "sm_max_mhz": self.max_mhz, "reasons": [], "samples": 0,
                    "note": getattr(self, "error", "no samples")}
        busy = sorted(self.sm)[len(self.sm) // 2:]
        return {"sm_mhz": float(np.median(busy)), "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons),
                "samples": len(self.sm)}


# ---------------------------------------------------------------------------------------------- reference arm / CPU baseline
def cpu_scene(args, seed=1234):
    from dropclip_b200.scenes import make_scene
    dev = "cuda" if torch.cuda.is_available() else "cpu"
    sc = make_scene(seed, n_views=args.views, n_points=args.points, n_objects=args.objects, device=dev)
    return sc


def cpu_model() -> str:
    try:
        for line in open("/proc/cpuinfo"):
            if line.startswith("model name"):
                return line.split(":", 1)[1].strip()
    except OSError:
        pass
    return "unknown"


def host_cores() -> int:
    try:
        return len(os.sched_getaffinity(0))
    except (AttributeError, OSError):
        return os.cpu_count() or 1


class cpu_threads:
    """Pins every thread pool the reference's CPU path touches, whatever the launcher put in the environment
    (torchrun exports OMP_NUM_THREADS=1; a bare `python` leaves the BLAS pools at one thread per core):
    numpy's BLAS (the 4x4 . 4xN np.dot per view, utils/transforms.py:56) and OpenMP pools through threadpoolctl,
    torch's intra-op pool through torch.set_num_threads."""

    def __init__(self, blas: int, torch_threads: int):
        self.blas, self.torch_threads = blas, torch_threads

    def __enter__(self):
        from threadpoolctl import threadpool_limits
        self._prev = torch.get_num_threads()
        torch.set_num_threads(self.torch_threads)
        self._lim = [threadpool_limits(limits=self.blas, user_api="blas"),
                     threadpool_limits(limits=max(self.blas, self.torch_threads), user_api="openmp")]
        return self

    def __exit__(self, *exc):
        for lim in self._lim:
            lim.restore_original_limits()
        torch.set_num_threads(self._prev)
        return False


def cpu_modes():
    """Thread configurations of the CPU arm. The reference's per-view np.dot is a 4x4 . 4xN product: a BLAS pool of one
    thread per core spends its time spinning at barriers on it (measured 13x slower than one BLAS thread on a 16-core
    box), so "the reference on all cores" is not one number. Every mode is timed and the FASTEST is reported."""
    n = host_cores()
    return {"blas%d_torch%d" % (n, n): (n, n), "blas1_torch%d" % n: (1, n), "blas1_torch1": (1, 1)}


def one_cpu_scene(sc):
    from oracle import fusion_ref
    K = fusion_ref.intrinsic_matrix(sc.intrinsic)
    H, W = sc.intrinsic["height"], sc.intrinsic["width"]
    t0 = time.perf_counter()
    fusion_ref.fuse_object_level(sc.points, sc.colors, sc.labels, sc.depths, sc.seg_masks, sc.camera_poses,
                                 sc.mv_features, sc.query_embeddings, K, H, W, use_visibility=False,
                                 use_similarity=True, sim_method="max", return_obj=True, device="cpu")
    return time.perf_counter() - t0


def pick_cpu_mode(sc, repeats=2):
    """Seconds per scene of every thread mode (one warm-up, then the best of `repeats`); returns (best name, table)."""
    table = {}
    for name, (blas, tt) in cpu_modes().items():
        with cpu_threads(blas, tt):
            one_cpu_scene(sc)  # warm-up: page faults, pool start-up
            table[name] = min(one_cpu_scene(sc) for _ in range(repeats))
    best = min(table, key=table.get)
    return best, table


def workload_config(args, world):
    """The `config` object of both arms (the driver compares them key by key)."""
    return {"workload": WORKLOAD, "scenes_per_gpu": args.scenes, "unique_scenes_per_gpu": args.unique,
            "views": args.views, "points": args.points, "objects": args.objects, "feat_dim": 768,
            "image": "480x640", "seg_dtype": "int64", "mask_dtype": "uint8", "feature_dtype": "fp16",
            "flags": "use_obj_prior=1,use_similarity=1,use_visibility=0,sim_kernel=max,return_obj=True",
            "parallelism": "scene-parallel x%d, no data-path collective; one all_gather of the fused features per run" % world}


def run_reference(args):
    """The reference's own CPU path (oracle/fusion_ref.py, the pinned restatement of utils/feature_fusion.py:272-343 -
    the reference is pure Python and is not part of this repository) on rank 0's host cores: one scene of the
    workload per step, in the fastest of the thread modes of cpu_modes()."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    sc = cpu_scene(args)
    best, table = pick_cpu_mode(sc)
    blas, tt = cpu_modes()[best]
    with cpu_threads(blas, tt):
        for _ in range(args.warmup):
            one_cpu_scene(sc)
        t0 = time.perf_counter()
        for _ in range(args.steps):
            one_cpu_scene(sc)
        dt = time.perf_counter() - t0
    val = args.steps / dt
    world = int(os.environ.get("WORLD_SIZE", "1"))
    line = {
        "impl": "reference", "metric": "fused_scenes_per_sec", "value": val, "unit": "scenes/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * dt / args.steps, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f64+f32", "data": "synthetic",
        "points_per_sec": val * args.points,
        "config": workload_config(args, world),
        "cpu_baseline": {"value": val, "unit": "scenes/s", "cores": max(blas, tt), "kind": "port",
                         "threads": {"blas": blas, "torch": tt}, "mode": best, "host_cores": host_cores(),
                         "cpu_model": cpu_model(),
                         "modes_scenes_per_s": {k: 1.0 / v for k, v in table.items()},
                         "sample": "1 scene of the workload per step (V=%d, N=%d), oracle/fusion_ref.fuse_object_level, "
                                   "fastest of the thread modes listed" % (args.views, args.points)},
        "e2e": {"value": val, "unit": "scenes/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line))


# ---------------------------------------------------------------------------------------------- our arm
def algorithmic_bytes(b, mask_elem=1):
    """SURVEY.md §8(d) per-scene figures x the scenes of one launch (DESIGN.md §5)."""
    HW = b.height * b.width
    seg_elem = b.segs.element_size()
    vis = sum(24 * n + v * n * (4 + mask_elem) for n, v in zip(b.n_points, b.n_views))
    seg = sum(v * HW * seg_elem for v in b.n_views)
    fe = b.feats.element_size()
    dim = int(b.feats.shape[1])
    wmean = b.total_rows * dim * fe + sum(q * v * 4 + q * dim * 4 for q, v in zip(b.n_queries, b.n_views))
    score_flops = 2 * b.total_rows * dim * max(b.n_queries)
    return {"project_visibility": vis, "seg_histogram": seg, "segmented_wmean": wmean, "view_score_flops": score_flops}


def _fit(name, a, cap, dtype=np.float32):
    """`a` (a CUDA tensor) as a host array of `dtype`: in full if it has at most `cap` elements, otherwise flattened and
    sampled at sorted indices drawn from a generator seeded by the name and the size (the same for equal sizes)."""
    flat = a.reshape(-1)
    if flat.numel() > cap:
        seed = (zlib.crc32(name.encode()), flat.numel())
        idx = np.unique(np.random.default_rng(seed).integers(0, flat.numel(), size=cap))
        a = flat[torch.from_numpy(idx).to(flat.device)]
    return a.cpu().numpy().astype(dtype)


def dump_outputs(out_dir, b, res, comp):
    """The results of one step as a caller of the device-resident path receives them: fused object features (sum Q, C),
    view weights (wobj layout), per-view status flags, the keep flag of every point, kept points per scene, and the
    compacted (V, N') uint8 visibility masks as per-(scene, view) visible counts plus a seeded sample of their elements.
    Counts and status flags are written as float64 (exact for any count). Each array is capped (_fit) so that all of them
    stay under 64 MB whatever the batch size.
    An object seen in no view has an all-NaN feature row, as in the reference; it is written as `object_seen` = 0 and a
    row of zeros. Any other non-finite value is written as it is and reported on stderr."""
    fused = res["fused"]
    unseen = torch.isnan(fused).all(1)
    fused = fused.masked_fill(unseen[:, None], 0.0)
    _, kept_off, _, out_off, cmask, _ = comp
    kept = kept_off.cpu().numpy()
    out = out_off.cpu().numpy()
    cmask = cmask[:int(out[-1])]
    counts = [cmask[int(out[s]):int(out[s + 1])].view(v, int(kept[s + 1] - kept[s])).sum(1, dtype=torch.int64)
              for s, v in enumerate(b.n_views)]
    arrays = {
        "fused_features": _fit("fused_features", fused, 1 << 21),
        "object_seen": _fit("object_seen", ~unseen, 1 << 17),
        "view_weights": _fit("view_weights", res["weight_obj"], 1 << 20),
        "view_status": _fit("view_status", res["view_status"][:b.total_views], 1 << 17, np.float64),
        "any_visible": _fit("any_visible", res["any_visible"], 1 << 23),
        "kept_points_per_scene": np.diff(kept).astype(np.float64),
        "visible_points_per_view": _fit("visible_points_per_view", torch.cat(counts), 1 << 17, np.float64),
        "visibility_mask_sample": _fit("visibility_mask_sample", cmask, 1 << 21),
    }
    total = sum(a.nbytes for a in arrays.values())
    assert total <= 64_000_000, total
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)
    bad = {name: int((~np.isfinite(a)).sum()) for name, a in arrays.items() if not np.isfinite(a).all()}
    if bad:
        sys.stderr.write("bench.py: non-finite values in the dumped outputs (count per array): %s\n" % bad)


def run_ours(args):
    import torch.distributed as dist
    from dropclip_b200.engine import FusionEngine, batch_from_device
    from dropclip_b200.feature_fusion import MultiviewFeatureFusion
    from dropclip_b200.scenes import make_scene

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)

    eng = FusionEngine(dev)
    # ---- synthetic batch, generated on the device; scene ids are sharded rank::world (weak scaling)
    uniq = []
    for i in range(args.unique):
        sid = 1234 + rank * args.scenes + i
        uniq.append(make_scene(sid, n_views=args.views, n_points=args.points, n_objects=args.objects, device=str(dev),
                               as_torch=True))
    scenes = [uniq[i % args.unique] for i in range(args.scenes)]
    batch = batch_from_device(scenes, dev, seg_dtype=torch.int64)  # torch.cat copies: every scene has its own memory
    torch.cuda.synchronize()

    def step(b=None):
        b = batch if b is None else b
        # the object branch (instance histograms -> scores -> weighted mean) runs on the engine's side stream beside the
        # visibility branch; it is joined after the compaction below has been enqueued on this stream
        res = eng.fuse_object_level(b, 0.05, False, True, "max", torch.uint8, join=False)
        # device-resident consumer: sizes and block layout of the compacted masks stay on the GPU (no host sync)
        comp = eng.compact_visibility(b, res["any_visible"], res["records"], res["rank"], torch.uint8, host_sizes=False)
        res["join"]()
        return res, comp

    gathered = torch.empty((world,) + (batch.total_queries, 768), dtype=torch.float32, device=dev) if world > 1 else None

    def gather_once(res):
        # SURVEY 8(e): the per-scene object features of all ranks are gathered ONCE per run/eval (NCCL over NVLink),
        # not per step; it sits inside the timed region, after the last step
        if world > 1:
            dist.all_gather_into_tensor(gathered, res["fused"])

    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()  # samples every 10 ms through warm-up and the timed region (same load)
    # Results stay referenced across steps exactly like in the timed loop below: the host runs ahead of the GPU
    # (the step has no sync), so two generations of outputs are alive at a time and the caching allocator must
    # own both before timing starts (a cudaMalloc of the 467 MB mask inside the timed region costs 20-150 ms).
    res = comp = None
    for _ in range(args.warmup):
        res, comp = step()
    gather_once(res)
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    eng.launches = 0
    eng.profile = {}
    torch.cuda.synchronize()
    start, end = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    start.record()
    for _ in range(args.steps):
        res, comp = step()
    gather_once(res)
    end.record()
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    clocks = sampler.stop() if rank == 0 else None
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, batch, res, comp)
    ms = torch.tensor([start.elapsed_time(end)], device=dev)
    if world > 1:
        dist.all_reduce(ms, op=dist.ReduceOp.MAX)
    ms_total = float(ms.item())
    launches = eng.launches
    prof = eng.profile_ms()
    eng.profile = None
    ms_step = ms_total / args.steps
    scenes_per_s = world * args.scenes / (ms_step * 1e-3)
    points_per_s = scenes_per_s * args.points

    # ---- roofline of the dominant kernel (live CUDA-event durations from the timed region)
    alg = algorithmic_bytes(batch)
    resident_gb = batch.h2d_bytes() / 1e9  # inputs of the timed step (before the uint8 variant below replaces the maps)
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    hbm_peak = float(peaks.get("hbm_gbs", 6650.0))
    peak_src = "measured" if "hbm_gbs" in peaks else "fallback"
    kernels = {}
    for name in ("project_visibility", "seg_histogram", "segmented_wmean"):
        if name in prof and prof[name] > 0:
            gbs = alg[name] / (prof[name] * 1e-3) / 1e9
            kernels[name] = {"ms": prof[name], "alg_bytes": alg[name], "gbs": gbs, "frac": gbs / hbm_peak}
    if "view_score" in prof:
        kernels["view_score"] = {"ms": prof["view_score"], "flops": alg["view_score_flops"],
                                 "tflops": alg["view_score_flops"] / (prof["view_score"] * 1e-3) / 1e12}
    # the HBM-dominant kernel: the one with the most algorithmic bytes (81 % of the step's). In the two-stream step its
    # live duration is measured while the issue-bound visibility filter shares the SMs and the bus with it.
    top = max(("project_visibility", "seg_histogram"), key=lambda k: kernels.get(k, {}).get("alg_bytes", 0.0))
    traffic, traffic_src = None, None
    try:  # DRAM bytes per launch of the same kernel at this workload, from the committed ncu --set full capture
        tj = json.load(open(os.path.join(ROOT, "profiles", "r02_traffic.json" if eng.overlap else "r01_traffic.json")))
        if args.scenes == 64 and args.views == 73 and args.points == 100000 and top in tj:
            traffic, traffic_src = tj[top]["bytes_per_launch"], tj[top]["source"]
    except Exception:
        pass
    try:  # what ncu says limits the projection/visibility kernel (it is issue-bound, not HBM-bound; DESIGN.md section 6)
        if "project_visibility" in kernels and "limiter" in tj.get("project_visibility", {}):
            kernels["project_visibility"]["limiter"] = tj["project_visibility"]["limiter"]
            kernels["project_visibility"]["dram_traffic"] = tj["project_visibility"]["bytes_per_launch"]
    except Exception:
        pass
    roofline = {"bound": "hbm", "kernel": top, "achieved": kernels[top]["gbs"], "peak": hbm_peak, "unit": "GB/s",
                "frac": kernels[top]["frac"], "traffic": traffic, "traffic_source": traffic_src, "peak_source": peak_src,
                "share_of_step": kernels[top]["ms"] / ms_step, "kernels": kernels}
    step_alg = sum(alg[k] for k in ("project_visibility", "seg_histogram", "segmented_wmean", "unpack_compact") if k in alg)
    roofline["whole_step"] = {"alg_bytes": step_alg, "gbs": step_alg / (ms_step * 1e-3) / 1e9,
                              "frac": step_alg / (ms_step * 1e-3) / 1e9 / hbm_peak}
    if eng.overlap:
        # the same kernels with the two branches on ONE stream (each kernel alone on the GPU): the figure to hold against
        # the ncu captures, which serialise kernels
        try:
            eng.overlap = False
            keep_a = None
            for _ in range(3):
                keep_a = step()
            torch.cuda.synchronize()
            eng.profile = {}
            a0, a1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a0.record()
            for _ in range(args.steps):
                keep_a = step()
            a1.record()
            torch.cuda.synchronize()
            pa = eng.profile_ms()
            roofline["one_stream"] = {
                "ms_per_step": a0.elapsed_time(a1) / args.steps,
                "kernels": {k: {"ms": pa[k], "gbs": alg[k] / (pa[k] * 1e-3) / 1e9, "frac": alg[k] / (pa[k] * 1e-3) / 1e9 / hbm_peak}
                            for k in ("project_visibility", "seg_histogram") if k in pa and pa[k] > 0}}
            del keep_a
        finally:
            eng.profile = None
            eng.overlap = True
        roofline["concurrency"] = ("object branch (instance histograms: HBM-bound bulk-copy ring kernel, one CTA per SM) on a second "
                                   "stream beside the point branch (visibility filter: issue-bound, two CTAs per SM); kernel "
                                   "durations above are live, i.e. measured while the two share the SMs and the bus")
    if roofline["frac"] > 1.0:
        roofline["note"] = ("the measured peak is a COPY bandwidth (reads and writes share the bus); this kernel only reads, "
                            "and a read-only stream sustains more than the copy figure (HBM3e nominal ~7.7 TB/s)")

    # ---- the API's full output, resident: int64 masks (the reference's dtype, utils/feature_fusion.py:86) and the
    # compacted points / labels rows (:277-281) written by the step as well (headline: uint8 masks, no row outputs)
    full = None
    try:
        def full_step():
            r = eng.fuse_object_level(batch, 0.05, False, True, "max", torch.uint8, join=False)
            c = eng.compact_visibility(batch, r["any_visible"], r["records"], r["rank"], torch.int64,
                                       extra_rows=(batch.points, batch.labels), host_sizes=False)
            r["join"]()
            return r, c
        keep_f = None
        for _ in range(max(3, args.warmup)):
            keep_f = full_step()
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        f0, f1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        f0.record()
        for _ in range(args.steps):
            keep_f = full_step()
        f1.record()
        torch.cuda.synchronize()
        ms_f = torch.tensor([f0.elapsed_time(f1)], device=dev)
        if world > 1:
            dist.all_reduce(ms_f, op=dist.ReduceOp.MAX)
        ms_full = float(ms_f.item()) / args.steps
        full = {"mask_dtype": "int64", "row_outputs": "points f64 (N',3), labels i64 (N',)", "ms_per_step": ms_full,
                "value": world * args.scenes / (ms_full * 1e-3), "unit": "scenes/s",
                "extra_write_bytes": int(batch.off_host["mask"][-1]) * 7 + batch.total_points * 32}
        del keep_f
        torch.cuda.empty_cache()
    except Exception as exc:  # never let the supplementary measurement break the contract line
        full = {"error": repr(exc)}

    # ---- the same step with the instance maps resident as uint8: this is what the library's own staging
    # (SceneBatch.from_host -> dc_host_gather_narrow_i64_u8) leaves in HBM for the reference's int64 maps; the
    # headline `value` above keeps them int64, the dtype the reference hands over
    alt = None
    try:
        del res, comp
        batch.segs = batch.segs.to(torch.uint8)
        torch.cuda.empty_cache()
        res = comp = None
        for _ in range(max(3, args.warmup)):
            res, comp = step()
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        a0, a1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a0.record()
        for _ in range(args.steps):
            res, comp = step()
        a1.record()
        torch.cuda.synchronize()
        ms_alt = torch.tensor([a0.elapsed_time(a1)], device=dev)
        if world > 1:
            dist.all_reduce(ms_alt, op=dist.ReduceOp.MAX)
        ms_alt_step = float(ms_alt.item()) / args.steps
        alt = {"seg_dtype": "uint8", "ms_per_step": ms_alt_step, "value": world * args.scenes / (ms_alt_step * 1e-3),
               "unit": "scenes/s", "note": "instance maps narrowed at staging time (1 byte per pixel in HBM)"}
        del res, comp
    except Exception as exc:  # never let the supplementary measurement break the contract line
        alt = {"error": repr(exc)}

    # ---- BASELINE configs[2]: a job of DISTINCT scenes (no replay) sharded rank::world, fused batch by batch; each batch is
    # generated on the device right before its (timed) pass, so the job needs the memory of one batch only
    job = None
    try:
        job_total = args.job_scenes if args.job_scenes >= 0 else (1000 if world > 1 else 256)
        if job_total > 0:
            mine = list(range(rank, job_total, world))
            # allocator warm-up (not a replay of job scenes): one untimed pass over the resident batch so that both stream
            # pools own their blocks again after the empty_cache() above; otherwise the first job pass pays 4 cudaMallocs
            # (22-25 ms, benchmarks/job_probe.py) inside its timed region
            warm = step()
            torch.cuda.synchronize()
            del warm
            job_ms, done, pass_ms, host_ms = 0.0, 0, [], []
            t_gen = time.perf_counter()
            for b0 in range(0, len(mine), args.scenes):
                ids = mine[b0:b0 + args.scenes]
                scs = [make_scene(100_000 + sid, n_views=args.views, n_points=args.points, n_objects=args.objects,
                                  device=str(dev), as_torch=True) for sid in ids]
                jb = batch_from_device(scs, dev, seg_dtype=torch.int64)
                del scs
                torch.cuda.synchronize()
                j0, j1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                j0.record()
                h0 = time.perf_counter()
                jr = step(jb)
                host_ms.append(round((time.perf_counter() - h0) * 1e3, 3))
                j1.record()
                torch.cuda.synchronize()
                job_ms += j0.elapsed_time(j1)
                pass_ms.append(round(j0.elapsed_time(j1), 3))
                done += len(ids)
                del jb, jr
            wall = time.perf_counter() - t_gen
            if world > 1:  # per-rank evidence on stderr (the JSON line carries rank 0's passes)
                sys.stderr.write("[rank %d] job pass ms %s host enqueue ms %s\n" % (rank, pass_ms, host_ms))
            t = torch.tensor([job_ms, float(done)], device=dev, dtype=torch.float64)
            tmax = t[:1].clone()
            if world > 1:
                dist.all_reduce(tmax, op=dist.ReduceOp.MAX)
                dist.all_reduce(t, op=dist.ReduceOp.SUM)
            job = {"workload": "configs[2]: %d distinct scenes (seeds 100000+i, no replay), sharded rank::world over %d GPU(s), "
                               "batches of %d scenes per launch sequence" % (job_total, world, args.scenes),
                   "scenes": int(t[1].item()), "gpu_ms_max_over_ranks": float(tmax.item()),
                   "value": float(t[1].item()) / (float(tmax.item()) * 1e-3), "unit": "scenes/s",
                   "wall_s_incl_generation": wall, "pass_ms_rank0": pass_ms, "host_enqueue_ms_rank0": host_ms,
                   "note": "device time of the fusion passes (inputs of a batch resident when its pass starts), max over ranks"}
            torch.cuda.empty_cache()
    except Exception as exc:  # never let the supplementary measurement break the contract line
        job = {"error": repr(exc)}

    # ---- end to end through the reference-shaped host API
    e2e = None
    if not args.no_e2e:
        host = [make_scene(1234 + rank * args.scenes + i, n_views=args.views, n_points=args.points, n_objects=args.objects,
                           device=str(dev)) for i in range(args.e2e_scenes)]
        M = MultiviewFeatureFusion(host[0].intrinsic, use_visibility=0, use_similarity=1, use_sim_kernel="max",
                                   use_obj_prior=1, norm_feat=False, device=dev)

        def e2e_step():
            outs = []
            for s in host:
                (f, w, vis), (p, c, l) = M.fuse(s.points, s.colors, s.labels, s.depths, s.seg_masks, s.camera_poses,
                                                s.mv_features, s.query_embeddings, return_obj=True, device=dev)
                outs.append((f.cpu(), w.cpu(), vis))  # device->host read of the step's results
            return outs

        outs = None
        for _ in range(max(3, args.warmup)):
            outs = e2e_step()  # results stay referenced across steps, exactly like in the timed loop (pinned-buffer reuse)
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        n_e2e = args.steps
        up0 = M._staging.bytes_uploaded
        t0 = time.perf_counter()
        for _ in range(n_e2e):
            outs = e2e_step()
        torch.cuda.synchronize()
        dt = torch.tensor([time.perf_counter() - t0], device=dev)
        if world > 1:
            dist.all_reduce(dt, op=dist.ReduceOp.MAX)
        h2d = (M._staging.bytes_uploaded - up0) // n_e2e  # bytes that crossed PCIe (instance maps travel as uint8)
        host_in = sum(sum(d.nbytes for d in s.depths) + sum(m.nbytes for m in s.seg_masks) + s.points.nbytes + s.labels.nbytes
                      + s.colors.nbytes + sum(f.numel() * f.element_size() for f in s.mv_features)
                      + s.query_embeddings.numel() * 4 + len(s.depths) * 64 for s in host)
        d2h = sum(f.numel() * 4 + w.numel() * 4 + vis.numel() * 8 + vis.shape[1] * (24 + 24 + 8) for f, w, vis in outs) \
            + sum(s.points.shape[0] * 8 for s in host)
        # same scenes through the overlapped scene loop (staging of scene i+1 under the fusion of scene i)
        def many_step():
            return [(f.cpu(), w.cpu(), vis) for (f, w, vis), _ in M.fuse_many(
                [(s.points, s.colors, s.labels, s.depths, s.seg_masks, s.camera_poses, s.mv_features, s.query_embeddings)
                 for s in host], return_obj=True, device=dev)]
        for _ in range(4):
            outs_many = many_step()
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        t1 = time.perf_counter()
        for _ in range(n_e2e):
            t_dbg = time.perf_counter()
            outs_many = many_step()
            if os.environ.get("DC_BENCH_DEBUG"):
                print("many_step ms", (time.perf_counter() - t_dbg) * 1e3, file=sys.stderr)
        torch.cuda.synchronize()
        dt_many = torch.tensor([time.perf_counter() - t1], device=dev)
        if world > 1:
            dist.all_reduce(dt_many, op=dist.ReduceOp.MAX)
        fuse_many_rate = world * args.e2e_scenes * n_e2e / float(dt_many.item())
        ref_shaped = {"value": world * args.e2e_scenes * n_e2e / float(dt.item()), "unit": "scenes/s",
                      "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": int(d2h), "host_input_bytes_per_step": int(host_in),
                      "scenes_per_step": args.e2e_scenes, "steps": n_e2e,
                      "api": "MultiviewFeatureFusion.fuse(pageable host numpy inputs, return_obj=True), one call per scene "
                             "like tools/preprocess_data.py:268", "fuse_many_scenes_per_s": fuse_many_rate}
        M = None
        torch.cuda.empty_cache()
        e2e = e2e_pipeline(args, dev, host, world, dist if world > 1 else None)
        e2e["reference_shaped_fuse"] = ref_shaped

        del host

    # ---- BASELINE configs 4 and 5 (supplementary; rank 0, N=1)
    extras = None
    if rank == 0 and world == 1 and not args.no_extras:
        try:
            extras = other_configs(dev, eng)
        except Exception as exc:  # never let a supplementary measurement break the contract line
            extras = {"error": repr(exc)}

    # ---- CPU baseline (rank 0, N=1): one scene of the workload through the oracle port
    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        sc = cpu_scene(args)
        best, table = pick_cpu_mode(sc, repeats=3)
        blas, tt = cpu_modes()[best]
        cpu = {"value": 1.0 / table[best], "unit": "scenes/s", "cores": max(blas, tt), "kind": "port",
               "threads": {"blas": blas, "torch": tt}, "mode": best, "host_cores": host_cores(), "cpu_model": cpu_model(),
               "modes_scenes_per_s": {k: 1.0 / v for k, v in table.items()},
               "sample": "1 scene of the workload (V=%d, N=%d) through oracle/fusion_ref.fuse_object_level, fastest of the "
                         "thread modes listed (best of 3 after 1 warm-up each), %.2f s/scene" % (args.views, args.points, table[best])}

    if rank == 0:
        line = {
            "metric": "fused_scenes_per_sec", "value": scenes_per_s, "unit": "scenes/s", "n_gpus": world,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_step, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f64+f32(f16 tensor operands)", "data": "synthetic",
            "points_per_sec": points_per_s, "point_views_per_sec": points_per_s * args.views,
            "config": dict(workload_config(args, world), l2="inputs per step (%.1f GB) exceed the 126 MB L2; no explicit flush" % resident_gb),
            "roofline": roofline, "cpu_baseline": cpu, "e2e": e2e, "gpu_launches": launches, "clocks": clocks,
            "resident_uint8_instance_maps": alt, "resident_full_output": full, "distinct_scene_job": job,
            "other_configs": extras,
        }
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


def e2e_pipeline(args, dev, host, world, dist):
    """End to end through FusionPipeline (the throughput form of the scene loop, tools/preprocess_data.py:188-297):
    every scene's inputs start in pinned HOST memory (library-owned PinnedSceneSlot, what a loader fills), and per scene
    the timed region holds its H2D copies, the batched launch sequences and the D2H read of every result
    (object features, weights, compacted uint8 visibility mask, keep flags) into host memory."""
    import threading
    from dropclip_b200.pipeline import FusionPipeline
    from dropclip_b200.scenes import make_scene
    rank = int(os.environ.get("RANK", "0"))
    n_slots, B = args.e2e_slots, args.e2e_batch
    cores = None
    if world > 1 and not os.environ.get("DC_BENCH_NO_PIN"):
        # every rank keeps its pipeline threads (and the pinned slots it allocates from here on) on its own slice of the host
        # cores - the cores NVML reports as local to its GPU when the box exposes that (shard.pin_rank_cores)
        from dropclip_b200 import shard
        local = int(os.environ.get("LOCAL_RANK", "0"))
        cores = shard.pin_rank_cores(local, int(os.environ.get("LOCAL_WORLD_SIZE", world)), local)
    pipe = FusionPipeline(host[0].intrinsic, device=dev, batch_scenes=B, n_slots=n_slots, max_views=args.views,
                          max_points=max(s.points.shape[0] for s in host), max_queries=args.objects)
    slots, fill_s, fill_bytes = [], 0.0, 0
    for i in range(n_slots):
        sc = host[i] if i < len(host) else make_scene(1234 + rank * args.scenes + i, n_views=args.views, n_points=args.points,
                                                      n_objects=args.objects, device=str(dev))
        sl = pipe.acquire()
        t0 = time.perf_counter()
        sl.fill(sc.points, sc.colors, sc.labels, sc.depths, sc.seg_masks, sc.camera_poses, sc.mv_features, sc.query_embeddings)
        fill_s += time.perf_counter() - t0
        fill_bytes += sum(d.nbytes for d in sc.depths) + sum(m.nbytes for m in sc.seg_masks) + sc.points.nbytes
        slots.append(sl)
    for sl in slots:
        pipe.release(sl)
    # the bound: this box's pinned host->device rate, one plain copy stream, measured here
    probe = torch.empty_like(slots[0].t_depths, device=dev)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for _ in range(8):
        probe.copy_(slots[0].t_depths, non_blocking=True)
    torch.cuda.synchronize()
    pcie_h2d = 8 * probe.numel() * 4 / (time.perf_counter() - t0) / 1e9
    hprobe = torch.empty(probe.shape, dtype=probe.dtype, pin_memory=True)
    t0 = time.perf_counter()
    for _ in range(4):
        hprobe.copy_(probe, non_blocking=True)
    torch.cuda.synchronize()
    pcie_d2h = 4 * probe.numel() * 4 / (time.perf_counter() - t0) / 1e9
    # the same copy with ALL ranks of the box copying at once: the host's memory system feeds every GPU's DMA engine, so
    # this, not the solo rate, bounds a rank's H2D rate at N > 1
    pcie_h2d_all = pcie_h2d
    if dist is not None:
        dist.barrier()
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        for _ in range(8):
            probe.copy_(slots[0].t_depths, non_blocking=True)
        torch.cuda.synchronize()
        mine = torch.tensor([8 * probe.numel() * 4 / (time.perf_counter() - t0) / 1e9], device=dev)
        dist.all_reduce(mine, op=dist.ReduceOp.MIN)
        pcie_h2d_all = float(mine.item())
        dist.barrier()
    del probe, hprobe
    done = [0]
    res_bytes = [0]

    def consume():
        for r in pipe.results():
            if r.error is not None:
                raise r.error
            res_bytes[0] += r.mv_feats_obj.nbytes + r.weight_obj.nbytes + r.visibility_mask.nbytes + r.keep.nbytes
            done[0] += 1

    th = threading.Thread(target=consume, daemon=True)
    th.start()

    def run(n):
        n0 = done[0]
        for i in range(n):
            pipe.submit(pipe.acquire(), tag=i)
        t_wait = time.perf_counter()
        while done[0] < n0 + n:
            time.sleep(0.0002)
            if pipe._error is not None or time.perf_counter() - t_wait > 120:
                raise RuntimeError(f"pipeline stopped: {pipe._error!r}")

    run(3 * n_slots)  # warm-up: allocator pools, arenas, host threads
    torch.cuda.synchronize()
    if dist is not None:
        dist.barrier()
    n_scenes = args.e2e_pipeline_scenes
    h0, d0, l0 = pipe.h2d_bytes, pipe.d2h_bytes, pipe.launches
    t0 = time.perf_counter()
    run(n_scenes)
    torch.cuda.synchronize()
    dt = torch.tensor([time.perf_counter() - t0], device=dev)
    if dist is not None:
        dist.all_reduce(dt, op=dist.ReduceOp.MAX)
    dt = float(dt.item())
    h2d, d2h, launches = pipe.h2d_bytes - h0, pipe.d2h_bytes - d0, pipe.launches - l0
    pipe.finish()
    th.join(10)
    pipe.close()
    rate = world * n_scenes / dt
    return {"value": rate, "unit": "scenes/s", "scenes_per_step": B, "scenes_timed_per_gpu": n_scenes,
            "h2d_bytes_per_step": int(h2d // n_scenes * B), "d2h_bytes_per_step": int(d2h // n_scenes * B),
            "h2d_gbs_per_gpu": h2d / dt / 1e9, "d2h_gbs_per_gpu": d2h / dt / 1e9,
            "bound": {"kind": "pcie_h2d", "pinned_h2d_gbs": pcie_h2d, "pinned_d2h_gbs": pcie_d2h,
                      "pinned_h2d_gbs_all_ranks_at_once": pcie_h2d_all,
                      "frac_of_bound": (h2d / dt / 1e9) / pcie_h2d_all, "frac_of_solo_rate": (h2d / dt / 1e9) / pcie_h2d,
                      "host_cores_per_rank": len(cores) if cores else host_cores(),
                      "note": "plain pinned->device copies of one slot's depth block on this box, measured in this run: alone, "
                              "and with every rank copying at the same time (slowest rank; the bound at N > 1)"},
            "host_fill": {"gbs": fill_bytes / fill_s / 1e9, "ms_per_scene": 1e3 * fill_s / n_slots,
                          "note": "PinnedSceneSlot.fill() from the reference's pageable numpy containers (int64 maps narrowed "
                                  "to uint8 on the way), outside the timed region: a loader writes the slot once"},
            "gpu_launches": launches, "distinct_scenes_per_gpu": n_slots,
            "api": "FusionPipeline.submit(PinnedSceneSlot): inputs in library-owned pinned host memory; per scene H2D copies + "
                   "batched launch sequences + D2H of (Q,C) features, (Q,V) weights, compacted (V,N') uint8 mask, keep flags"}


def other_configs(dev, eng):
    """BASELINE.json configs 4 and 5 on one GPU, as supplementary numbers next to the headline (CUDA events, median of 5
    after 3 warm-ups): pixel-level fusion of one scene (use_obj_prior=0, V=8, sim kernel max, norm_feat) and 3D grounding
    of 200 k points x 256 prompts (fp16, paired softmax, in-place normalisation + GEMM + min-max threshold)."""
    from dropclip_b200.engine import batch_from_device
    from dropclip_b200.scenes import make_scene
    out = {}

    def median_ms(fn, reps=5, warm=3):
        ts = []
        for it in range(warm + reps):
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            fn()
            b.record()
            torch.cuda.synchronize()
            if it >= warm:
                ts.append(a.elapsed_time(b))
        return sorted(ts)[len(ts) // 2]

    sc = make_scene(1234, n_views=8, n_points=100_000, n_objects=21, device=str(dev), as_torch=True, pixel_features=True,
                    feature_dtype=torch.float32)
    patches = torch.stack(sc["mv_features"]).contiguous()
    sc_obj = dict(sc)
    sc_obj["mv_features"] = [torch.zeros((1, 768), device=dev, dtype=torch.float16) for _ in range(8)]
    b = batch_from_device([sc_obj], dev)
    b.feats = patches
    mask, _, _ = eng.visibility(b, 0.05, torch.uint8)
    ms = median_ms(lambda: eng.pixel_fuse(b, mask, "max", True, normalize=True))
    pairs = int(mask.sum().item())
    out["pixel_level_fusion"] = {"workload": "configs[3]: 1 scene, V=8, N=100k, C=768, Q=21, 24x32 patch maps, sim max, norm_feat",
                                 "ms_per_scene": ms, "visible_point_views": pairs,
                                 "tap_tflops": 2.0 * 16 * 768 * pairs / (ms * 1e-3) / 1e12,
                                 "kernel": "dc_pixel_fuse_mma (tcgen05: pairs sorted by bicubic footprint, 128-pair tiles)"}
    del b, mask, patches, sc, sc_obj
    try:  # the same at the full view set
        sc = make_scene(1234, n_views=73, n_points=100_000, n_objects=21, device=str(dev), as_torch=True, pixel_features=True,
                        feature_dtype=torch.float32)
        patches = torch.stack(sc["mv_features"]).contiguous()
        sc_obj = dict(sc)
        sc_obj["mv_features"] = [torch.zeros((1, 768), device=dev, dtype=torch.float16) for _ in range(73)]
        b = batch_from_device([sc_obj], dev)
        b.feats = patches
        mask, _, _ = eng.visibility(b, 0.05, torch.uint8)
        ms73 = median_ms(lambda: eng.pixel_fuse(b, mask, "max", True, normalize=True))
        pairs73 = int(mask.sum().item())
        out["pixel_level_fusion_V73"] = {"workload": "1 scene, V=73, N=100k, C=768, Q=21, sim max, norm_feat", "ms_per_scene": ms73,
                                         "visible_point_views": pairs73, "tap_tflops": 2.0 * 16 * 768 * pairs73 / (ms73 * 1e-3) / 1e12}
        del b, mask, patches, sc, sc_obj
    except Exception as exc:
        out["pixel_level_fusion_V73"] = {"error": repr(exc)}
    torch.cuda.empty_cache()

    from dropclip_b200 import _lib as lib_mod
    n, p, c = 200_000, 256, 768
    g = torch.Generator(device=dev).manual_seed(0)
    x0 = torch.randn((n, c), generator=g, device=dev).half()
    t = torch.randn((p, c), generator=g, device=dev)
    t = (t / t.norm(dim=-1, keepdim=True)).half()
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    ts = []
    for it in range(8):
        x = x0.clone()
        flush.zero_()  # 256 MB > L2: the features come from HBM
        a, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        vals, pred = eng.predict(x, t, lib_mod.DC_GROUND_PAIRED, 0.1, True, 0.7)
        e.record()
        torch.cuda.synchronize()
        if it >= 3:
            ts.append(a.elapsed_time(e))
    ms = sorted(ts)[len(ts) // 2]
    out["grounding"] = {"workload": "configs[4]: 200k points x 256 prompts x 768, fp16, paired softmax, predict() = dc_predict "
                                    "(in-place normalisation + tcgen05 GEMM with fused epilogue + min-max threshold)",
                        "ms": ms, "points_per_s": n / (ms * 1e-3), "useful_tflops": 2.0 * n * p * c / (ms * 1e-3) / 1e12,
                        "gemm_kernel_ncu": {"us": 70.8, "tensor_pipe_active_pct": 65.6, "dram_read_mb": 307.8,
                                            "source": "profiles/r02_ncu_ground_final_raw.csv (ncu --set full, cold cache)"}}
    del x0, x, t, flush
    torch.cuda.empty_cache()
    try:
        sys.path.insert(0, os.path.join(ROOT, "benchmarks"))
        import ablation
        out["voxel_size_ablation"] = ablation.run(dev)
    except Exception as exc:
        out["voxel_size_ablation"] = {"error": repr(exc)}
    return out


def main():
    args = parse()
    if args.impl == "reference":
        if args.dump_outputs:
            raise SystemExit("--dump-outputs writes the outputs of --impl ours")
        run_reference(args)
    else:
        if not torch.cuda.is_available():
            raise SystemExit("bench.py needs a CUDA device; there is no CPU fallback (use --impl reference for the CPU arm)")
        run_ours(args)


if __name__ == "__main__":
    main()
