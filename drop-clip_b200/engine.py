"""Scene-batched device engine under the reference-shaped classes.

A `SceneBatch` holds a ragged batch of scenes in HBM in the layout the C ABI takes
(concatenated arrays + int64 prefix offsets, DESIGN.md §3); `FusionEngine` strings the CUDA
kernels together on the current stream. The reference processes one scene per call and one
view per Python iteration (utils/feature_fusion.py:88,303); one scene is only ~10^2 MB of
traffic, so batching scenes is what lets the kernels run at HBM speed instead of launch speed.
torch is used for allocation, streams and copies only.
"""
from __future__ import annotations

from dataclasses import dataclass, field
from typing import Dict, List, Optional, Sequence

import ctypes
import os

import numpy as np
import torch

from . import _lib
from ._lib import check, current_stream, ptr

_TORCH_TO_NP = {torch.float32: np.dtype(np.float32), torch.float64: np.dtype(np.float64), torch.int64: np.dtype(np.int64),
                torch.int32: np.dtype(np.int32), torch.uint8: np.dtype(np.uint8), torch.float16: np.dtype(np.float16)}
SIM_KERNELS = {None: _lib.DC_SIM_NONE, "max": _lib.DC_SIM_MAX, "mean": _lib.DC_SIM_MEAN}
MIN_BINS = 256  # instance ids are stored as uint8 labels downstream (tools/preprocess_data.py:294); more bins when Q > 256
MAX_BINS = MIN_BINS  # kept for callers that size count tables for the common case


def hist_bins(max_queries: int) -> int:
    """Bins of the per-view instance histogram: every id the reference can index (ids < Q, quirk q7) needs one."""
    return max(MIN_BINS, (int(max_queries) + 31) // 32 * 32)


def _prefix(counts: Sequence[int]) -> np.ndarray:
    out = np.zeros(len(counts) + 1, dtype=np.int64)
    np.cumsum(np.asarray(counts, dtype=np.int64), out=out[1:])
    return out


def _labels_as_int64(labels) -> np.ndarray:
    """Point labels as int64 object ids for the scatter kernel. The reference compares `label == obj`
    (utils/feature_fusion.py:133) in the caller's dtype, so a non-integral or non-finite float label matches no
    object: it becomes -1 (a zero row) instead of being truncated onto a neighbouring id."""
    arr = np.asarray(labels).reshape(-1)
    if arr.dtype == np.int64:
        return arr
    if arr.dtype.kind == "f":
        with np.errstate(invalid="ignore"):
            ok = np.isfinite(arr) & (arr == np.floor(arr)) & (np.abs(arr) < 2.0 ** 62)
        return np.where(ok, arr, -1).astype(np.int64)
    if arr.dtype.kind == "b":
        return arr.astype(np.int64)
    if arr.dtype.kind == "u" and arr.dtype.itemsize == 8:
        return np.where(arr < np.uint64(2 ** 63), arr, np.uint64(0)).astype(np.int64) - (arr >= np.uint64(2 ** 63))
    return arr.astype(np.int64)


def query_csr(pos, neg_lists, n_prompts: int):
    """Host column table of FusionEngine.predict_queries: (pos int32 [Q], neg_off int32 [Q+1], neg_cols int32) from
    query q's positive row pos[q] and negative rows neg_lists[q] (neg_lists None: no query has negatives). Every index
    must lie in [0, n_prompts): IndexError otherwise, before anything reaches the device."""
    pos_a = np.asarray(list(pos), dtype=np.int64).reshape(-1)
    q = pos_a.size
    if neg_lists is None:
        neg_lists = [()] * q
    neg_lists = [np.asarray(list(x), dtype=np.int64).reshape(-1) for x in neg_lists]
    if len(neg_lists) != q:
        raise ValueError(f"{q} positive columns but {len(neg_lists)} negative lists")
    cols = np.concatenate(neg_lists) if q else np.zeros(0, dtype=np.int64)
    for what, a in (("positive", pos_a), ("negative", cols)):
        bad = (a < 0) | (a >= n_prompts)
        if bad.any():
            raise IndexError(f"{what} prompt index {int(a[bad][0])} outside [0, {n_prompts})")
    off = _prefix([x.size for x in neg_lists])
    if off[-1] >= 2 ** 31:
        raise ValueError("too many negative columns for one call")
    return pos_a.astype(np.int32), off.astype(np.int32), cols.astype(np.int32)


def intrinsic_matrix(intr: Dict[str, float]) -> np.ndarray:
    """utils/feature_fusion.py:35-40, always promoted to fp64 (K @ fp64 points is fp64 anyway)."""
    return np.asarray([[intr["fx"], 0, intr["cx"]], [0, intr["fy"], intr["cy"]], [0, 0, 1]], dtype=np.float64)


@dataclass
class SceneBatch:
    """Ragged scene batch resident on one GPU."""

    device: torch.device
    height: int
    width: int
    n_scenes: int
    # host-side extents
    n_points: List[int]
    n_views: List[int]
    n_queries: List[int]
    feat_rows: List[int]  # per view (stacked over scenes)
    # device arrays
    points: torch.Tensor  # (sum N, 3) f64
    depths: torch.Tensor  # (TV, H, W) f32
    inv_poses: torch.Tensor  # (TV, 16) f64 (inverted in the pose dtype on the host, then widened: exact)
    intrinsics: torch.Tensor  # (S, 9) f64
    segs: Optional[torch.Tensor] = None  # (TV, H, W) u8 / i32 / i64
    labels: Optional[torch.Tensor] = None  # (sum N,) i64
    feats: Optional[torch.Tensor] = None  # (TR, C) f16 / f32  or (TV, ph, pw, C) f32 for the pixel path
    queries: Optional[torch.Tensor] = None  # (sum Q, C) f32
    # offsets (device int64) + host mirrors
    off: Dict[str, torch.Tensor] = field(default_factory=dict)
    off_host: Dict[str, np.ndarray] = field(default_factory=dict)

    @property
    def total_points(self) -> int:
        return int(self.off_host["point"][-1])

    @property
    def total_views(self) -> int:
        return int(self.off_host["view"][-1])

    @property
    def total_queries(self) -> int:
        return int(self.off_host["query"][-1])

    @property
    def total_rows(self) -> int:
        return int(self.off_host["feat"][-1])

    def h2d_bytes(self) -> int:
        n = 0
        for t in (self.points, self.depths, self.inv_poses, self.intrinsics, self.segs, self.labels, self.feats,
                  self.queries):
            if t is not None:
                n += t.numel() * t.element_size()
        for t in self.off.values():
            n += t.numel() * t.element_size()
        return n

    @staticmethod
    def offsets_for(n_points, n_views, n_queries, feat_rows):
        host = {
            "point": _prefix(n_points),
            "view": _prefix(n_views),
            "query": _prefix(n_queries),
            "mask": _prefix([v * n for v, n in zip(n_views, n_points)]),
            "wobj": _prefix([q * v for q, v in zip(n_queries, n_views)]),
            "feat": _prefix(feat_rows),
        }
        host["view_scene"] = np.repeat(np.arange(len(n_views), dtype=np.int32), np.asarray(n_views, dtype=np.int64))
        return host

    @classmethod
    def from_host(cls, scenes: Sequence, device="cuda", pixel_features: bool = False,
                  inv_poses: Optional[Sequence] = None, staging: Optional["PinnedStaging"] = None,
                  narrow_segs: bool = True) -> "SceneBatch":
        """Uploads scenes given in the reference's own containers (numpy arrays and lists, torch
        feature tensors). `scenes[i]` needs attributes/keys points, depths, camera_poses, intrinsic
        and optionally labels, seg_masks, mv_features, query_embeddings.

        The camera->world poses are inverted here with np.linalg.inv in their own dtype, exactly
        like utils/transforms.py:54 does on the host (a 4x4 per view), and stored as fp64 on the device:
        widening an fp32 inverse is what np.dot does with it (exact), and fp64 poses stay fp64."""
        dev = torch.device(device)
        get = (lambda s, k: s.get(k)) if isinstance(scenes[0], dict) else (lambda s, k: getattr(s, k, None))
        intr0 = get(scenes[0], "intrinsic")
        H, W = int(intr0["height"]), int(intr0["width"])
        n_points = [int(np.asarray(get(s, "points")).shape[0]) for s in scenes]
        n_views = [len(get(s, "depths")) for s in scenes]
        has_q = get(scenes[0], "query_embeddings") is not None
        has_f = get(scenes[0], "mv_features") is not None
        n_queries = [int(get(s, "query_embeddings").shape[0]) if has_q else 0 for s in scenes]
        feat_rows: List[int] = []
        if has_f and not pixel_features:
            for s in scenes:
                feat_rows += [int(f.shape[0]) for f in get(s, "mv_features")]
        else:
            feat_rows = [0] * sum(n_views)
        host = cls.offsets_for(n_points, n_views, n_queries, feat_rows)
        if staging is not None:
            staging.begin()
        up = staging.upload if staging is not None else (lambda a: torch.as_tensor(a).to(dev, non_blocking=False))

        pts_l = [np.ascontiguousarray(get(s, "points"), dtype=np.float64).reshape(-1, 3) for s in scenes]
        pts = pts_l[0] if len(pts_l) == 1 else np.concatenate(pts_l)  # one scene: no extra 2.4 MB host copy
        dlist = [d for s in scenes for d in get(s, "depths")]
        if staging is not None and dlist:
            depths_dev = staging.upload_list(dlist, torch.float32, (H, W))
        else:
            depths = np.stack([np.asarray(d, dtype=np.float32) for d in dlist]) if dlist else np.zeros((0, H, W), np.float32)
            depths_dev = None
        if inv_poses is None:
            poses = [np.asarray(p) for s in scenes for p in get(s, "camera_poses")]
            if poses and all(p.shape == (4, 4) and p.dtype == poses[0].dtype for p in poses):
                # one stacked call: the same LAPACK routine per matrix, bit-identical to per-view np.linalg.inv, 5x less overhead
                inv = list(np.linalg.inv(np.stack(poses)))
            else:
                inv = [np.linalg.inv(p) for p in poses]
        else:
            inv = [np.asarray(p) for ps in inv_poses for p in ps]
        # np.dot(inv_pose, fp64 points) promotes an fp32 inverse to fp64 (exact); an fp64 pose stays fp64 end to end
        inv = np.stack([np.asarray(m, dtype=np.float64) for m in inv]).reshape(-1, 16) if inv else np.zeros((0, 16), np.float64)
        K = np.stack([intrinsic_matrix(get(s, "intrinsic")).reshape(9) for s in scenes])
        b = cls(device=dev, height=H, width=W, n_scenes=len(scenes), n_points=n_points, n_views=n_views,
                n_queries=n_queries, feat_rows=feat_rows, points=up(pts),
                depths=depths_dev if depths_dev is not None else up(depths), inv_poses=up(inv), intrinsics=up(K))
        if get(scenes[0], "seg_masks") is not None:
            segs = [np.asarray(m) for s in scenes for m in get(s, "seg_masks")]
            if segs:
                dt = segs[0].dtype
                if dt not in (np.uint8, np.int32, np.int64):
                    dt = np.int64
                if staging is not None:
                    tdt = {np.dtype(np.uint8): torch.uint8, np.dtype(np.int32): torch.int32,
                           np.dtype(np.int64): torch.int64}[np.dtype(dt)]
                    narrowed = False
                    if narrow_segs and tdt == torch.int64 and all(
                            isinstance(m, np.ndarray) and m.dtype == np.int64 and m.flags.c_contiguous for m in segs):
                        # instance ids fit a byte in every valid input (ids index the Q <= 256 query rows, quirk
                        # q7): ship 1 byte per pixel instead of 8; fall back to int64 if some id does not fit
                        b.segs, narrowed = staging.upload_list(segs, tdt, (H, W), narrow_to_u8=True)
                    if not narrowed:
                        b.segs = staging.upload_list(segs, tdt, (H, W))
                else:
                    b.segs = up(np.stack([m.astype(dt, copy=False) for m in segs]))
        if get(scenes[0], "labels") is not None:
            lab_l = [_labels_as_int64(get(s, "labels")) for s in scenes]
            b.labels = up(lab_l[0] if len(lab_l) == 1 else np.concatenate(lab_l))
        if has_f:
            fl = [f for s in scenes for f in get(s, "mv_features")]
            host_np = lambda f, dt: (not f.is_cuda) and f.dtype == dt and f.is_contiguous()
            if pixel_features:
                if staging is not None and fl and all(host_np(f, torch.float32) and f.shape == fl[0].shape for f in fl):
                    # equally shaped patch maps: the multi-threaded gather into pinned memory (no pageable H2D copies)
                    b.feats = staging.upload_list([f.numpy() for f in fl], torch.float32, tuple(fl[0].shape))
                else:
                    b.feats = torch.stack([f.to(dev, torch.float32) for f in fl]).contiguous()
            else:
                dt = torch.float16 if fl[0].dtype == torch.float16 else torch.float32
                if fl and fl[0].is_cuda:
                    b.feats = torch.cat([f.to(dt) for f in fl]).to(dev).contiguous()
                elif fl and all(host_np(f, dt) for f in fl):
                    b.feats = up(np.concatenate([f.numpy() for f in fl]))  # numpy: no OpenMP region (see upload())
                elif fl:
                    b.feats = up(torch.cat([f.to(dt) for f in fl]))
        if has_q:
            ql = [get(s, "query_embeddings").to(torch.float32) for s in scenes]
            b.queries = torch.cat(ql).to(dev).contiguous() if ql[0].is_cuda else up(torch.cat(ql))
        b.off_host = host
        if staging is not None:
            keys = list(host)
            b.off = dict(zip(keys, staging.upload_packed([host[k] for k in keys])))  # one copy for the seven offset arrays
            staging.end()
        else:
            b.off = {k: up(v) for k, v in host.items()}
        return b


def batch_from_device(scenes: Sequence[dict], device="cuda", seg_dtype=torch.int64) -> SceneBatch:
    """Builds a SceneBatch from scenes that already live on the GPU (`scenes.make_scene(...,
    as_torch=True)`): used by the benchmark so that synthetic data never crosses PCIe. The
    inverse poses are still taken on the host with np.linalg.inv (4x4 per view), as in
    utils/transforms.py:54."""
    dev = torch.device(device)
    intr0 = scenes[0]["intrinsic"]
    H, W = int(intr0["height"]), int(intr0["width"])
    n_points = [int(s["points"].shape[0]) for s in scenes]
    n_views = [int(s["depths"].shape[0]) for s in scenes]
    n_queries = [int(s["query_embeddings"].shape[0]) for s in scenes]
    feat_rows = [int(f.shape[0]) for s in scenes for f in s["mv_features"]]
    host = SceneBatch.offsets_for(n_points, n_views, n_queries, feat_rows)
    inv = np.stack([np.linalg.inv(p) for s in scenes for p in s["camera_poses"].cpu().numpy()]).astype(np.float64)
    K = np.stack([intrinsic_matrix(s["intrinsic"]).reshape(9) for s in scenes])
    fdt = scenes[0]["mv_features"][0].dtype
    b = SceneBatch(
        device=dev, height=H, width=W, n_scenes=len(scenes), n_points=n_points, n_views=n_views, n_queries=n_queries,
        feat_rows=feat_rows,
        points=torch.cat([s["points"] for s in scenes]).to(dev, torch.float64).contiguous(),
        depths=torch.cat([s["depths"] for s in scenes]).to(dev, torch.float32).contiguous(),
        inv_poses=torch.from_numpy(inv.reshape(-1, 16)).to(dev), intrinsics=torch.from_numpy(K).to(dev),
        segs=torch.cat([s["seg_masks"].to(seg_dtype) for s in scenes]).to(dev).contiguous(),
        labels=torch.cat([s["labels"] for s in scenes]).to(dev, torch.int64).contiguous(),
        feats=torch.cat([f.to(fdt) for s in scenes for f in s["mv_features"]]).to(dev).contiguous(),
        queries=torch.cat([s["query_embeddings"] for s in scenes]).to(dev, torch.float32).contiguous())
    b.off_host = host
    b.off = {k: torch.from_numpy(v).to(dev) for k, v in host.items()}
    return b


class PinnedStaging:
    """Reusable pinned host buffers so that host->device copies of numpy inputs run at PCIe speed
    and asynchronously on the current stream. Slots are handed out in call order between
    begin() and end(); begin() waits until the copies of the previous round have drained before
    the buffers are overwritten."""

    def __init__(self, device="cuda"):
        self.device = torch.device(device)
        self._bufs: List[torch.Tensor] = []
        self._slot = 0
        self._event: Optional[torch.cuda.Event] = None
        self.bytes_uploaded = 0

    def begin(self):
        if self._event is not None:
            self._event.synchronize()
        self._slot = 0

    def end(self):
        self._event = torch.cuda.Event()
        self._event.record()

    def _pinned(self, numel: int, dtype: torch.dtype) -> torch.Tensor:
        if self._slot == len(self._bufs):
            self._bufs.append(torch.empty(max(numel, 1), dtype=dtype, pin_memory=True))
        buf = self._bufs[self._slot]
        if buf.dtype != dtype or buf.numel() < numel:
            buf = torch.empty(max(numel, 1), dtype=dtype, pin_memory=True)
            self._bufs[self._slot] = buf
        self._slot += 1
        return buf

    @staticmethod
    def _host_threads() -> int:
        """Threads for the host staging helpers: the cores this process may use, shared between the ranks of
        the node when launched under torchrun (LOCAL_WORLD_SIZE), at most 16 (more does not add bandwidth)."""
        try:
            cores = len(os.sched_getaffinity(0))
        except (AttributeError, OSError):
            cores = os.cpu_count() or 1
        ranks = max(1, int(os.environ.get("LOCAL_WORLD_SIZE", "1") or 1))
        return max(1, min(16, cores // ranks))

    def upload_list(self, arrays, dtype: torch.dtype, item_shape, group_bytes: int = 32 << 20,
                    narrow_to_u8: bool = False):
        """Stacks a list of equally-shaped host arrays straight into one pinned buffer and uploads it
        group by group, so the H2D copy of group g overlaps the host copy of group g+1. Contiguous
        numpy arrays of the right dtype go through libdropclip's multi-threaded gather-copy (one call
        per group); anything else through per-item tensor copies.

        With `narrow_to_u8` (int64 instance maps) the values are narrowed to uint8 while being
        staged; returns (tensor, ok) where ok is False if some value does not fit [0, 255] - the
        caller then uploads the int64 maps as they are."""
        n = len(arrays)
        numel = int(np.prod(item_shape)) if len(item_shape) else 1
        out_dtype = torch.uint8 if narrow_to_u8 else dtype
        buf = self._pinned(n * numel, out_dtype)
        view = buf[: n * numel].view((n,) + tuple(item_shape))
        out = torch.empty((n,) + tuple(item_shape), dtype=out_dtype, device=self.device)
        np_dtype = _TORCH_TO_NP[dtype]
        fast = all(isinstance(a, np.ndarray) and a.dtype == np_dtype and a.flags.c_contiguous and a.size == numel
                   for a in arrays)
        if narrow_to_u8 and not (fast and dtype == torch.int64):
            raise ValueError("narrow_to_u8 needs contiguous int64 numpy arrays")
        item_bytes = numel * buf.element_size()
        per_group = max(1, group_bytes // max(1, item_bytes if not narrow_to_u8 else numel * 8))
        lib, threads, ok = _lib.load(), self._host_threads(), True
        for g0 in range(0, n, per_group):
            g1 = min(n, g0 + per_group)
            if fast:
                srcs = (ctypes.c_void_p * (g1 - g0))(*[a.ctypes.data for a in arrays[g0:g1]])
                dst = ctypes.c_void_p(view[g0].data_ptr())
                if narrow_to_u8:
                    bad = ctypes.c_int(0)
                    check(lib.dc_host_gather_narrow_i64_u8(srcs, g1 - g0, numel, dst, threads, ctypes.byref(bad)))
                    if bad.value:
                        ok = False
                        break
                else:
                    check(lib.dc_host_gather_copy(srcs, g1 - g0, item_bytes, dst, threads))
            else:
                for i in range(g0, g1):
                    a = arrays[i]
                    t = a if isinstance(a, torch.Tensor) else torch.from_numpy(np.asarray(a))
                    view[i].copy_(t.reshape(item_shape))  # converts dtype if needed
            out[g0:g1].copy_(view[g0:g1], non_blocking=True)
        self.bytes_uploaded += n * item_bytes
        return (out, ok) if narrow_to_u8 else out

    def download(self, t: torch.Tensor) -> torch.Tensor:
        """Async device->host copy into a reusable pinned buffer; valid until the next download()."""
        n = t.numel()
        buf = getattr(self, "_down", None)
        if buf is None or buf.dtype != t.dtype or buf.numel() < n:
            buf = torch.empty(max(n, 1), dtype=t.dtype, pin_memory=True)
            self._down = buf
        view = buf[:n].view(t.shape)
        view.copy_(t, non_blocking=True)
        return view

    def upload_packed(self, arrays: Sequence[np.ndarray]) -> List[torch.Tensor]:
        """Several small host arrays in ONE pinned buffer and ONE H2D copy; returns device views (16-byte aligned)
        with the arrays' dtypes and shapes. Each separate small upload costs ~60 us of host time."""
        arrays = [np.ascontiguousarray(a) for a in arrays]
        offs, total = [], 0
        for a in arrays:
            offs.append(total)
            total += (a.nbytes + 15) // 16 * 16
        buf = self._pinned(max(total, 16), torch.uint8)
        host = buf[:max(total, 16)].numpy()
        for a, o in zip(arrays, offs):
            host[o:o + a.nbytes] = a.reshape(-1).view(np.uint8)
        dev = buf[:max(total, 16)].to(self.device, non_blocking=True)
        self.bytes_uploaded += total
        out = []
        for a, o in zip(arrays, offs):
            tdt = {v: k for k, v in _TORCH_TO_NP.items()}[a.dtype]
            out.append(dev[o:o + a.nbytes].view(tdt).view(a.shape) if a.nbytes else torch.empty(a.shape, dtype=tdt, device=self.device))
        return out

    def upload(self, arr) -> torch.Tensor:
        t = arr if isinstance(arr, torch.Tensor) else torch.from_numpy(np.ascontiguousarray(arr))
        t = t.contiguous()
        if self._slot == len(self._bufs):
            self._bufs.append(torch.empty(max(t.numel(), 1), dtype=t.dtype, pin_memory=True))
        buf = self._bufs[self._slot]
        if buf.dtype != t.dtype or buf.numel() < t.numel():
            buf = torch.empty(max(t.numel(), 1), dtype=t.dtype, pin_memory=True)
            self._bufs[self._slot] = buf
        self._slot += 1
        view = buf[:t.numel()].view(t.shape)
        # A torch CPU copy_ of more than 32 k elements opens an OpenMP parallel region, and libgomp's workers then
        # SPIN for a few milliseconds on every core - exactly the cores the staging helpers of the next upload_list
        # need (measured: the helper calls of one scene took 7.9 ms behind such a copy, 3.3 ms without). A plain
        # single-threaded memcpy through numpy is as fast for these few MB and leaves the cores alone.
        nbytes = t.numel() * t.element_size()
        if not t.is_cuda and nbytes >= (1 << 20):
            # a few MB (points, colours, labels, object features): the staging pool copies them in 256 KB slices
            srcs = (ctypes.c_void_p * 1)(t.data_ptr())
            check(_lib.load().dc_host_gather_copy(srcs, 1, nbytes, ctypes.c_void_p(view.data_ptr()), self._host_threads()))
        elif t.dtype in _TORCH_TO_NP and not t.is_cuda:
            np.copyto(view.numpy(), t.detach().numpy())
        else:
            view.copy_(t)
        self.bytes_uploaded += t.numel() * t.element_size()
        return view.to(self.device, non_blocking=True)


class _Tick:
    """Records a (start, end) CUDA event pair for one launch group when the engine's profile is enabled.
    (A module-level class: building a class object per call leaves cyclic garbage behind, and the collector's
    pauses showed up as multi-millisecond gaps between launches.)"""
    __slots__ = ("eng", "name", "a", "b")

    def __init__(self, eng, name):
        self.eng, self.name = eng, name

    def __enter__(self):
        if self.eng.profile is not None:
            self.a = torch.cuda.Event(enable_timing=True)
            self.b = torch.cuda.Event(enable_timing=True)
            self.a.record()
        return self

    def __exit__(self, *exc):
        if self.eng.profile is not None:
            self.b.record()
            self.eng.profile.setdefault(self.name, []).append((self.a, self.b))
        return False


def _no_join():
    return None


class FusionEngine:
    """Launch sequences over a SceneBatch. Every method only enqueues work on the current stream."""

    def __init__(self, device="cuda"):
        self.lib = _lib.load()
        if not torch.cuda.is_available():
            raise RuntimeError("dropclip_b200 needs a CUDA device (sm_100a); there is no CPU path")
        self.device = torch.device(device)
        self.launches = 0  # kernels launched by this engine (bench.py's gpu_launches)
        # object-level similarity weights below this are re-evaluated in fp64 (dc_view_weights); inf = every row
        self.refine_below = 0.02
        self.profile: Optional[Dict[str, list]] = None  # name -> [(start_event, end_event)] when enabled
        # object branch and visibility branch of fuse_object_level on two streams (DC_OVERLAP=0: one stream)
        self._side: Dict[Optional[int], "torch.cuda.Stream"] = {}
        self._events: Dict[Optional[int], tuple] = {}
        self._out_stream: Optional["torch.cuda.Stream"] = None
        self.overlap = os.environ.get("DC_OVERLAP", "1") != "0"

    @property
    def overlap(self) -> bool:
        return self._overlap

    @overlap.setter
    def overlap(self, on: bool):
        # the library shapes the two kernels that share the SMs accordingly (include/dropclip.h: dc_set_stream_overlap)
        self._overlap = bool(on)
        self.lib.dc_set_stream_overlap(int(self._overlap))

    def _alloc_out(self, shape, dtype, device) -> torch.Tensor:
        """Result tensors of the object branch. While that branch is being enqueued on the side stream
        (fuse_object_level) they still come from the CALLER's stream pool: they outlive the join, so the caller's
        allocator may recycle them in its own stream order with no cross-stream bookkeeping (record_stream would park
        every freed block behind an event, the pools would grow while the host runs ahead, and the resulting
        cudaMallocs inside the step loop contend between the ranks of a node: 2.78 -> 3.4-3.8 ms per step at N=2).
        Branch-local scratch stays in the side stream's pool."""
        if self._out_stream is None:
            return torch.empty(shape, dtype=dtype, device=device)
        with torch.cuda.stream(self._out_stream):
            return torch.empty(shape, dtype=dtype, device=device)

    def _tick(self, name: str):
        """Context manager recording CUDA events around a launch group on the current stream."""
        return _Tick(self, name)

    def profile_ms(self) -> Dict[str, float]:
        """Mean duration per recorded launch group (call after a synchronize)."""
        return {k: sum(a.elapsed_time(b) for a, b in v) / len(v) for k, v in (self.profile or {}).items()}

    # ------------------------------------------------------------------ (1)+(2)
    def visibility(self, b: SceneBatch, threshold: float = 0.05, mask_dtype=torch.uint8, point_object: bool = False):
        """Returns (mask [flat, mask layout], any_visible [sum N] u8, point_object | None)."""
        total_mask = int(b.off_host["mask"][-1])
        mask = torch.empty(total_mask, dtype=mask_dtype, device=b.device)
        any_vis = torch.empty(b.total_points, dtype=torch.uint8, device=b.device)
        pobj = torch.empty(total_mask, dtype=torch.int32, device=b.device) if point_object else None
        segs = b.segs if point_object else None
        with self._tick("project_visibility"):
            check(self.lib.dc_project_visibility(
                ptr(b.points), ptr(b.off["point"]), ptr(b.off["view"]), ptr(b.depths), ptr(b.inv_poses), ptr(b.intrinsics),
                ptr(b.off["mask"]), b.n_scenes, max(b.n_points, default=0), max(b.n_views, default=0), b.height, b.width,
                float(threshold), ptr(mask), mask.element_size(), ptr(any_vis), ptr(segs),
                _lib.torch_dtype_code(segs.dtype) if segs is not None else _lib.DC_I64, ptr(pobj), current_stream()))
        self.launches += 1
        return mask, any_vis, pobj

    def visibility_sorted(self, b: SceneBatch, threshold: float = 0.05):
        """Sorted-gather variant: returns (records [words, sum N] u32, rank [sum N] i64, any_visible)."""
        n = b.total_points
        words = (max(b.n_views, default=0) + 31) // 32
        records = torch.empty((max(words, 1), max(n, 1)), dtype=torch.int32, device=b.device)
        rank = torch.empty(max(n, 1), dtype=torch.int64, device=b.device)
        any_vis = torch.empty(max(n, 1), dtype=torch.uint8, device=b.device)
        ws_bytes = self.lib.dc_visibility_sorted_workspace(n, b.n_scenes, max(b.n_views, default=0))
        ws = torch.empty(ws_bytes, dtype=torch.uint8, device=b.device)
        with self._tick("project_visibility"):
            check(self.lib.dc_project_visibility_sorted(
                ptr(b.points), ptr(b.off["point"]), ptr(b.off["view"]), ptr(b.depths), ptr(b.inv_poses), ptr(b.intrinsics),
                b.n_scenes, n, max(b.n_points, default=0), max(b.n_views, default=0), b.height, b.width, float(threshold),
                ptr(records), ptr(rank), ptr(any_vis), ptr(ws), ws_bytes, current_stream()))
        self.launches += 7 + self.lib.dc_visibility_sorted_groups(b.n_scenes, max(b.n_points, default=0), max(b.n_views, default=0))
        return records, rank, any_vis[:n]

    def unpack_visibility(self, b: SceneBatch, records, rank, mask_dtype=torch.uint8):
        mask = torch.empty(int(b.off_host["mask"][-1]), dtype=mask_dtype, device=b.device)
        check(self.lib.dc_unpack_visibility(ptr(records), ptr(rank), ptr(b.off["point"]), ptr(b.off["view"]), ptr(b.off["mask"]),
                                            b.n_scenes, b.total_points, max(b.n_points, default=0), ptr(mask),
                                            mask.element_size(), current_stream()))
        self.launches += 1
        return mask

    def compact_visibility(self, b: SceneBatch, any_vis, records, rank, out_dtype=torch.uint8,
                           extra_rows: Sequence[torch.Tensor] = (), host_sizes: bool = True, wide_unpack: bool = True):
        """Drops never-visible points and expands the bit records straight into the compacted masks.
        Returns (new_index, kept_off, kept_host, out_off_host, compacted mask, compacted rows).

        With `host_sizes=False` nothing is read back: the outputs are allocated at their upper bound (the
        uncompacted sizes), the block layout stays on the device (kept_off, and out_off returned in place of
        out_off_host) and kept_host is None - the form a device-resident consumer uses (bench.py's step)."""
        n = b.total_points
        new_index = torch.empty(max(n, 1), dtype=torch.int64, device=b.device)
        kept_off = torch.empty(b.n_scenes + 1, dtype=torch.int64, device=b.device)
        ws_bytes = self.lib.dc_compact_workspace(n)
        ws = torch.empty(ws_bytes, dtype=torch.uint8, device=b.device)
        check(self.lib.dc_compact_scan(ptr(any_vis), n, ptr(b.off["point"]), b.n_scenes, ptr(new_index), ptr(kept_off),
                                       ptr(ws), ws_bytes, current_stream()))
        self.launches += 4
        if host_sizes:
            kept_host = kept_off.cpu().numpy()
            out_off_host = _prefix([v * k for v, k in zip(b.n_views, np.diff(kept_host))])
            out_off = torch.from_numpy(out_off_host).to(b.device)
            mask_elems, n_kept = int(out_off_host[-1]), int(kept_host[-1])
        else:
            kept_host, out_off_host = None, None
            out_off = torch.empty(b.n_scenes + 1, dtype=torch.int64, device=b.device)
            check(self.lib.dc_compact_mask_offsets(ptr(kept_off), ptr(b.off["view"]), b.n_scenes, ptr(out_off), current_stream()))
            self.launches += 1
            mask_elems, n_kept = int(b.off_host["mask"][-1]), n
        cmask_buf = torch.empty(max(mask_elems, 1), dtype=out_dtype, device=b.device)  # empty tensors have a null data_ptr
        cmask = cmask_buf[:mask_elems]
        uws_bytes = self.lib.dc_unpack_compact_workspace(n, cmask.element_size()) if wide_unpack else 0
        uws = torch.empty(uws_bytes, dtype=torch.uint8, device=b.device) if uws_bytes else None
        with self._tick("unpack_compact"):
            check(self.lib.dc_unpack_visibility_compact(ptr(records), ptr(rank), ptr(b.off["point"]), ptr(b.off["view"]),
                                                        ptr(any_vis), ptr(new_index), ptr(kept_off), ptr(out_off), b.n_scenes, n,
                                                        max(b.n_points, default=0), ptr(cmask_buf), cmask.element_size(),
                                                        ptr(uws), uws_bytes, current_stream()))
        self.launches += 2 if uws_bytes else 1
        rows_out = []
        for t in extra_rows:
            t2 = t.reshape(n, -1)
            o_buf = torch.empty((max(n_kept, 1), t2.shape[1]), dtype=t.dtype, device=b.device)
            check(self.lib.dc_compact_rows(ptr(t2), t2.shape[1] * t2.element_size(), ptr(any_vis), ptr(new_index), n,
                                           ptr(o_buf), current_stream()))
            self.launches += 1
            rows_out.append(o_buf[:n_kept])
        return new_index, kept_off, kept_host, (out_off_host if host_sizes else out_off), cmask, rows_out

    def seg_tables(self, b: SceneBatch):
        """Instance histograms and the feature-row <-> object binding of every view."""
        tv = b.total_views
        nbins = hist_bins(max(b.n_queries, default=0))
        counts = self._alloc_out((tv, nbins), torch.int32, b.device)
        outside = self._alloc_out((max(tv, 1), 4), torch.int64, b.device)
        with self._tick("seg_histogram"):
            check(self.lib.dc_seg_histogram(ptr(b.segs), _lib.torch_dtype_code(b.segs.dtype), tv, b.height * b.width,
                                            nbins, ptr(counts), ptr(outside), current_stream()))
        row_object = self._alloc_out(max(b.total_rows, 1), torch.int32, b.device)
        total_wobj = int(b.off_host["wobj"][-1])
        object_row = self._alloc_out(max(total_wobj, 1), torch.int32, b.device)
        status = self._alloc_out(max(tv, 1), torch.int32, b.device)
        check(self.lib.dc_view_table(ptr(counts), ptr(outside), ptr(b.off["feat"]), ptr(b.off["view_scene"]),
                                     ptr(b.off["view"]), ptr(b.off["query"]), ptr(b.off["wobj"]), tv, b.total_rows,
                                     total_wobj, nbins, ptr(row_object), ptr(object_row), ptr(status),
                                     current_stream()))
        self.launches += 2
        return counts, outside, row_object, object_row, status

    # ------------------------------------------------------------------ (3)+(4)
    def view_scores(self, b: SceneBatch):
        """Cosine scores of every feature row against its scene's queries (utils/feature_fusion.py:106-124): returns
        (sims [rows, ld] f32, ld, workspace holding the normalised fp16 planes). Independent of the instance tables, so
        the two-stream step runs it ahead of the histogram pass."""
        dim = int(b.feats.shape[1])
        max_q = max(b.n_queries)
        ld = self.lib.dc_view_score_ld(max_q)
        sims = torch.empty((max(b.total_rows, 1), ld), dtype=torch.float32, device=b.device)
        fdt = _lib.torch_dtype_code(b.feats.dtype)
        ws_bytes = self.lib.dc_view_score_workspace(b.total_rows, b.total_queries, dim, fdt)
        ws = torch.empty(ws_bytes + 1024, dtype=torch.uint8, device=b.device)
        shift = (-ws.data_ptr()) % 1024
        ws = ws[shift:shift + ws_bytes]
        with self._tick("view_score"):
            check(self.lib.dc_view_score(ptr(b.feats), fdt, b.total_rows, dim, ptr(b.off["feat"]), ptr(b.off["view"]),
                                         ptr(b.queries), ptr(b.off["query"]), b.total_queries, b.n_scenes, max_q,
                                         ptr(sims), ld, ptr(ws), ws_bytes, current_stream()))
        self.launches += 4
        return sims, ld, ws

    def object_features(self, b: SceneBatch, tables, use_visibility: bool, use_similarity: bool, sim_kernel, scores=None):
        """Returns (fused [sum Q, C] f32, weight_obj [wobj layout] f32). `scores`: result of view_scores(b) if the caller
        has already enqueued it."""
        counts, _, row_object, object_row, _ = tables
        dim = int(b.feats.shape[1])
        max_q = max(b.n_queries)
        total_wobj = int(b.off_host["wobj"][-1])
        weight = self._alloc_out(max(total_wobj, 1), torch.float32, b.device)
        weight.zero_()  # on the branch's own stream
        sims, ld = None, 0
        kern = SIM_KERNELS[sim_kernel] if use_similarity else _lib.DC_SIM_NONE
        if use_similarity:
            sims, ld, ws = scores if scores is not None else self.view_scores(b)
        view_mm = torch.empty(self.lib.dc_view_weights_scratch(b.total_views, b.total_rows) // 4 + 1, dtype=torch.int32,
                              device=b.device) if use_similarity else None
        check(self.lib.dc_view_weights(ptr(sims), ld, ptr(b.off["feat"]), ptr(b.off["view_scene"]), ptr(b.off["view"]),
                                       ptr(b.off["query"]), ptr(b.off["wobj"]), ptr(row_object), ptr(counts), int(counts.shape[1]),
                                       b.total_views, kern, int(bool(use_visibility)), ptr(weight),
                                       ptr(b.feats) if use_similarity else None, _lib.torch_dtype_code(b.feats.dtype), dim,
                                       ptr(b.queries) if use_similarity else None, b.total_rows, ptr(view_mm),
                                       ptr(ws) if (use_similarity and b.feats.dtype == torch.float16) else None,
                                       float(self.refine_below), current_stream()))
        fused = self._alloc_out((b.total_queries, dim), torch.float32, b.device)
        with self._tick("segmented_wmean"):
            check(self.lib.dc_segmented_wmean(ptr(b.feats), _lib.torch_dtype_code(b.feats.dtype), dim, ptr(object_row),
                                              ptr(weight), ptr(b.off["view"]), ptr(b.off["query"]), ptr(b.off["wobj"]),
                                              b.n_scenes, max_q, ptr(fused), current_stream()))
        self.launches += 4 if use_similarity else 2  # weights (+ memset node, + refinement), weighted mean
        return fused, weight

    def compact_rows(self, t: torch.Tensor, any_vis, new_index, n_kept: int) -> torch.Tensor:
        """out[new_index[j]] = t[j] for the kept points; rows of any byte width."""
        n = int(any_vis.shape[0])
        t2 = t.reshape(n, -1)
        o_buf = torch.empty((max(n_kept, 1), t2.shape[1]), dtype=t.dtype, device=t.device)
        check(self.lib.dc_compact_rows(ptr(t2), t2.shape[1] * t2.element_size(), ptr(any_vis), ptr(new_index), n, ptr(o_buf),
                                       current_stream()))
        self.launches += 1
        return o_buf[:n_kept]

    def scatter_to_points(self, b: SceneBatch, fused, labels, point_off, n_scenes, max_points, skip_first=True):
        if labels.dtype != torch.int64 or not labels.is_contiguous():
            raise TypeError(f"scatter_to_points: labels must be a contiguous int64 tensor (got {labels.dtype}); the kernel reads 8 bytes per point")
        if fused.dtype != torch.float32:
            raise TypeError("scatter_to_points: fused features must be fp32")
        dim = int(fused.shape[1])
        n_rows = int(labels.shape[0])
        out = torch.empty((max(n_rows, 1), dim), dtype=torch.float32, device=fused.device)
        if n_rows > 0:
            check(self.lib.dc_scatter_to_points(ptr(fused), ptr(b.off["query"]), ptr(labels), ptr(point_off), n_scenes,
                                                max_points, dim, int(skip_first), ptr(out), current_stream()))
            self.launches += 1
        return out[:n_rows]

    # ------------------------------------------------------------------ compaction
    def compact(self, b: SceneBatch, any_vis, mask, extra_rows: Sequence[torch.Tensor] = (), out_dtype=None):
        """Drops never-visible points. Returns (new_index, kept_off (device), kept_off (host), mask offsets
        (host), compacted mask, compacted rows). `out_dtype=torch.int64` widens a uint8 mask while
        compacting (the reference's visibility mask is int64)."""
        n = b.total_points
        new_index = torch.empty(max(n, 1), dtype=torch.int64, device=b.device)
        kept_off = torch.empty(b.n_scenes + 1, dtype=torch.int64, device=b.device)
        ws_bytes = self.lib.dc_compact_workspace(n)
        ws = torch.empty(ws_bytes, dtype=torch.uint8, device=b.device)
        check(self.lib.dc_compact_scan(ptr(any_vis), n, ptr(b.off["point"]), b.n_scenes, ptr(new_index), ptr(kept_off),
                                       ptr(ws), ws_bytes, current_stream()))
        self.launches += 4
        kept_host = kept_off.cpu().numpy()  # sizes of the outputs: one small D2H, like the reference's .cpu() at :278
        n_kept = np.diff(kept_host)
        out_off_host = _prefix([v * k for v, k in zip(b.n_views, n_kept)])
        out_off = torch.from_numpy(out_off_host).to(b.device)
        widen = out_dtype is not None and out_dtype != mask.dtype
        if widen and not (mask.dtype == torch.uint8 and out_dtype == torch.int64):
            raise ValueError("compact: only uint8 -> int64 widening is supported")
        n_mask = int(out_off_host[-1])
        cmask_buf = torch.empty(max(n_mask, 1), dtype=out_dtype if widen else mask.dtype, device=b.device)
        check(self.lib.dc_compact_mask(ptr(mask), 18 if widen else mask.element_size(), ptr(b.off["mask"]), ptr(b.off["point"]),
                                       ptr(b.off["view"]), ptr(any_vis), ptr(new_index), ptr(kept_off), ptr(out_off),
                                       b.n_scenes, max(b.n_points, default=0), max(b.n_views, default=0), ptr(cmask_buf),
                                       current_stream()))
        self.launches += 1
        cmask = cmask_buf[:n_mask]
        rows_out = []
        for t in extra_rows:
            t2 = t.reshape(n, -1)
            o_buf = torch.empty((max(int(kept_host[-1]), 1), t2.shape[1]), dtype=t.dtype, device=b.device)
            check(self.lib.dc_compact_rows(ptr(t2), t2.shape[1] * t2.element_size(), ptr(any_vis), ptr(new_index), n,
                                           ptr(o_buf), current_stream()))
            self.launches += 1
            rows_out.append(o_buf[:int(kept_host[-1])])
        return new_index, kept_off, kept_host, out_off_host, cmask, rows_out

    # ------------------------------------------------------------------ whole object-level pass
    def fuse_object_level(self, b: SceneBatch, threshold=0.05, use_visibility=False, use_similarity=True,
                          sim_kernel="max", mask_dtype=torch.uint8, sorted_gather: bool = True, join: bool = True):
        """Device-resident hot path of fuse_obj_prior (utils/feature_fusion.py:272-335) for a batch:
        visibility -> instance tables -> view scores -> weights -> segmented weighted mean.
        With `sorted_gather` the visibility result is returned as bit records (+ rank) to be expanded
        by compact_visibility / unpack_visibility; otherwise as the full (V,N) mask blocks.
        `join=False`: the object branch is still running on the side stream when this returns; the caller enqueues its
        own consumers of the visibility result first and then calls out["join"]() before touching fused / weight_obj."""
        out = {}
        if not (self.overlap and sorted_gather):
            if sorted_gather:
                out["records"], out["rank"], out["any_visible"] = self.visibility_sorted(b, threshold)
            else:
                out["mask"], out["any_visible"], _ = self.visibility(b, threshold, mask_dtype)
            tables = self.seg_tables(b)
            fused, weight = self.object_features(b, tables, use_visibility, use_similarity, sim_kernel)
            out.update({"fused": fused, "weight_obj": weight, "view_status": tables[4], "join": _no_join})
            return out
        # Two branches that share no data until the caller combines them: instance tables -> scores -> weighted mean
        # (HBM-bound: the int64 maps) on the side stream, point visibility (issue-bound) on the current stream. The
        # histogram kernel is shaped to sit beside the filter's CTAs on every SM (csrc/seg_table.cu), so the two
        # overlap instead of alternating. Branch-local scratch comes from the side stream's allocator pool; everything
        # handed back is allocated from the caller's pool (_alloc_out).
        main = torch.cuda.current_stream(b.device)
        side = self._side_stream(b.device)
        fork_evt, join_evt = self._events[torch.device(b.device).index]  # reused every call (no event churn on the host)
        fork_evt.record(main)
        side.wait_event(fork_evt)
        self._out_stream = main
        try:
            with torch.cuda.stream(side):
                # scores first: they do not need the tables, and the point branch starts with its latency-bound sort passes
                scores = self.view_scores(b) if use_similarity else None
                tables = self.seg_tables(b)
                fused, weight = self.object_features(b, tables, use_visibility, use_similarity, sim_kernel, scores)
                del scores
        finally:
            self._out_stream = None
        join_evt.record(side)
        out["records"], out["rank"], out["any_visible"] = self.visibility_sorted(b, threshold)

        def join_now():
            main.wait_event(join_evt)

        # the tables stay referenced by the result until the caller drops it (after the join): their blocks belong to the
        # caller's stream pool and must not be recycled while the side stream may still read them
        out.update({"fused": fused, "weight_obj": weight, "view_status": tables[4], "tables": tables, "join": join_now})
        if join:
            join_now()
            out["join"] = _no_join
        return out

    def _side_stream(self, device):
        key = torch.device(device).index
        if key not in self._side:
            # high priority: the object branch ends in a chain of small kernels that should not queue behind filter CTAs
            self._side[key] = torch.cuda.Stream(device=device, priority=-1)
            self._events[key] = (torch.cuda.Event(), torch.cuda.Event())
        return self._side[key]

    # ------------------------------------------------------------------ pixel-level path
    def pixel_fuse(self, b: SceneBatch, mask_u8, sim_kernel, norm_feat: bool, spatial_order: bool = True, normalize: bool = False):
        """aggregate_features (utils/feature_fusion.py:138-250): returns (sum_features [sum N, C] f32,
        similarity weights [mask layout] f32 | None). `b.feats` is the (TV, ph, pw, C) patch stack.
        `normalize`: return the final features of fuse_points (:266-268) instead of the sums (fused division)."""
        tv, ph, pw, dim = b.feats.shape
        kern = SIM_KERNELS[sim_kernel]
        # the tensor-core path keeps 84 bytes of sort / operand records per (point, view) of the mask: batches beyond
        # ~40 M mask elements (several full-size scenes at once) take the SIMT kernel instead of a multi-GB workspace
        use_mma = (dim in (512, 768, 1024) and b.total_points > 0 and os.environ.get("DC_PIXEL_PATH", "mma") != "simt"
                   and b.feats.dtype == torch.float32 and int(b.off_host["mask"][-1]) <= 40_000_000)
        if use_mma:
            return self._pixel_fuse_mma(b, mask_u8, kern, norm_feat, normalize)
        sums = torch.empty((b.total_points, dim), dtype=torch.float32, device=b.device)
        weight = torch.empty(int(b.off_host["mask"][-1]), dtype=torch.float32, device=b.device) \
            if kern != _lib.DC_SIM_NONE else None
        segs = b.segs if kern != _lib.DC_SIM_NONE else None
        perm = self.spatial_sort(b)[0] if spatial_order and b.total_points > 0 else None
        max_q = max(b.n_queries, default=0) if kern != _lib.DC_SIM_NONE else 0
        ws_bytes = self.lib.dc_pixel_fuse_workspace(int(tv), int(ph), int(pw), max_q) if kern != _lib.DC_SIM_NONE else 0
        ws = torch.empty(max(ws_bytes, 1), dtype=torch.uint8, device=b.device)
        check(self.lib.dc_pixel_fuse(
            ptr(b.points), ptr(b.off["point"]), ptr(b.off["view"]), ptr(b.inv_poses), ptr(b.intrinsics), ptr(b.off["mask"]),
            ptr(mask_u8), ptr(segs), _lib.torch_dtype_code(segs.dtype) if segs is not None else _lib.DC_I64,
            ptr(b.feats), int(ph), int(pw), int(dim), ptr(b.queries) if kern else None,
            ptr(b.off["query"]) if kern else None, kern, int(bool(norm_feat)), b.n_scenes, max(b.n_points, default=0),
            max(b.n_views, default=0), b.height, b.width, ptr(perm), ptr(sums), ptr(weight), int(bool(normalize)), int(tv), max_q, ptr(ws), ws_bytes,
            current_stream()))
        self.launches += 3 if kern != _lib.DC_SIM_NONE else 1
        return sums, weight

    def _pixel_fuse_mma(self, b: SceneBatch, mask_u8, kern: int, norm_feat: bool, normalize: bool):
        """The tcgen05 form of pixel_fuse (dc_pixel_fuse_mma): pairs sorted by bicubic footprint, 128-pair MMA tiles."""
        tv, ph, pw, dim = b.feats.shape
        mask_elems = int(b.off_host["mask"][-1])
        sums = torch.empty((b.total_points, dim), dtype=torch.float32, device=b.device)
        has_sim = kern != _lib.DC_SIM_NONE
        weight = torch.empty(max(mask_elems, 1), dtype=torch.float32, device=b.device)[:mask_elems] if has_sim else None
        max_q = max(b.n_queries, default=0) if has_sim else 0
        ws_bytes = self.lib.dc_pixel_fuse_mma_workspace(int(tv), mask_elems, int(ph), int(pw), int(dim), max_q)
        ws = torch.empty(ws_bytes + 256, dtype=torch.uint8, device=b.device)
        shift = (-ws.data_ptr()) % 256
        segs = b.segs if has_sim else None
        # Morton rank of the points: pairs are grouped by spatial region so that the rows being accumulated stay in L2
        rank = self.spatial_sort(b)[1] if b.total_points * dim * 4 > (48 << 20) else None
        check(self.lib.dc_pixel_fuse_mma(
            ptr(b.points), ptr(b.off["point"]), ptr(b.off["view"]), ptr(b.inv_poses), ptr(b.intrinsics), ptr(b.off["mask"]),
            ptr(mask_u8), ptr(segs), _lib.torch_dtype_code(segs.dtype) if segs is not None else _lib.DC_I64, ptr(b.feats),
            int(ph), int(pw), int(dim), ptr(b.queries) if has_sim else None, ptr(b.off["query"]) if has_sim else None, kern,
            int(bool(norm_feat)), b.n_scenes, max(b.n_points, default=0), max(b.n_views, default=0), b.height, b.width,
            ptr(rank), ptr(sums), ptr(weight), int(bool(normalize)), int(tv), b.total_points, mask_elems, max_q,
            ctypes.c_void_p(ws.data_ptr() + shift), ws_bytes, current_stream()))
        self.launches += 12 + int(has_sim) + int(bool(norm_feat)) + int(bool(normalize))
        return sums, weight

    def spatial_sort(self, b: SceneBatch):
        """(perm, rank): counting sort of every scene's points by Morton cell (order inside a cell is arbitrary)."""
        n = b.total_points
        perm = torch.empty(max(n, 1), dtype=torch.int64, device=b.device)
        rank = torch.empty(max(n, 1), dtype=torch.int64, device=b.device)
        ws_bytes = self.lib.dc_spatial_sort_workspace(b.n_scenes)
        ws = torch.empty(ws_bytes, dtype=torch.uint8, device=b.device)
        check(self.lib.dc_spatial_sort(ptr(b.points), ptr(b.off["point"]), b.n_scenes, n, max(b.n_points, default=0), ptr(perm),
                                       ptr(rank), ptr(ws), ws_bytes, current_stream()))
        self.launches += 5
        return perm, rank

    def pixel_normalize(self, b: SceneBatch, sums, mask_u8, weight):
        check(self.lib.dc_pixel_normalize(ptr(sums), ptr(b.off["point"]), ptr(b.off["view"]), ptr(b.off["mask"]),
                                          ptr(mask_u8), ptr(weight), b.n_scenes, max(b.n_points, default=0),
                                          int(sums.shape[1]), current_stream()))
        self.launches += 1
        return sums

    # ------------------------------------------------------------------ (6) grounding
    def ground(self, feats: torch.Tensor, text: torch.Tensor, mode: int, softmax_temp: float = 0.1,
               normalize: bool = True, want_matrix: bool = True):
        """feats (N,C) fp16/fp32 CUDA tensor (normalised IN PLACE when `normalize`), text (P,C) already
        normalised prompt embeddings (any P: the kernel walks the prompt axis in blocks of 256), prompt 0 positive.
        Returns (out, pred|None, minmax[4]); DC_GROUND_CLASS: out = (N,P) raw similarities (None unless
        `want_matrix`) and pred = (N,) int64 index of each row's maximum."""
        n, dim = feats.shape
        p = int(text.shape[0])
        dev = feats.device
        is_f32 = feats.dtype == torch.float32
        code = _lib.torch_dtype_code(feats.dtype)
        if is_f32:
            planes = torch.empty((2, max(n, 1), dim), dtype=torch.float16, device=dev)
            x_hi, x_lo = planes[0], planes[1]
            check(self.lib.dc_row_normalize(ptr(feats), code, n, dim, int(normalize), ptr(x_hi), ptr(x_lo), current_stream()))
        else:
            x_hi, x_lo = feats, None  # fp16 rows are normalised in place by dc_ground (a separate pass before the GEMM)
        t32 = text.to(torch.float32).contiguous()
        tplanes = torch.empty((2, p, dim), dtype=torch.float16, device=dev)
        t_lo = tplanes[1] if text.dtype == torch.float32 else None
        check(self.lib.dc_row_normalize(ptr(t32), _lib.DC_F32, p, dim, 0, ptr(tplanes[0]), ptr(tplanes[1]), current_stream()))
        minmax = torch.empty(4, dtype=torch.float32, device=dev)
        check(self.lib.dc_ground_init_minmax(ptr(minmax), current_stream()))
        pred = argmax_idx = None
        if mode in (_lib.DC_GROUND_RAW, _lib.DC_GROUND_CLASS):
            out = torch.empty((n, p), dtype=torch.float32, device=dev) if (want_matrix or mode == _lib.DC_GROUND_RAW) else None
            ld = p
            if mode == _lib.DC_GROUND_CLASS:
                argmax_idx = torch.empty(n, dtype=torch.int64, device=dev)
        else:
            out = torch.empty(n, dtype=torch.float32, device=dev)
            ld = 1
            if mode == _lib.DC_GROUND_ARGMAX:
                pred = torch.empty(n, dtype=torch.uint8, device=dev)
        ws_bytes = self.lib.dc_ground_workspace(n, p, mode)
        ws = torch.empty(ws_bytes, dtype=torch.uint8, device=dev) if ws_bytes else None
        check(self.lib.dc_ground(ptr(x_hi), ptr(x_lo), n, ptr(tplanes[0]), ptr(t_lo), p, dim, mode, float(softmax_temp),
                                 int(bool(normalize) and not is_f32), ptr(out), ld, ptr(pred), ptr(argmax_idx), ptr(minmax),
                                 ptr(ws), ws_bytes, current_stream()))
        self.launches += 3 + (p + 255) // 256
        return out, (argmax_idx if mode == _lib.DC_GROUND_CLASS else pred), minmax

    def predict(self, feats: torch.Tensor, text: torch.Tensor, mode: int, softmax_temp: float, normalize: bool, threshold: float):
        """ClipSimilarity.predict after the text tower (models/similarity.py:77-101) in one library call and two
        allocations: returns (score (N,) fp32 min-max normalised, pred (N,) uint8). `feats` is normalised in place."""
        n, dim = feats.shape
        p = int(text.shape[0])
        dev = feats.device
        text = text.contiguous()
        if text.dtype not in (torch.float16, torch.float32):
            text = text.float()
        fcode, tcode = _lib.torch_dtype_code(feats.dtype), _lib.torch_dtype_code(text.dtype)
        ws_bytes = self.lib.dc_predict_workspace(n, p, dim, fcode, tcode, mode)
        res = torch.empty(max(n, 1) * 5 + 256, dtype=torch.uint8, device=dev)  # score fp32 + pred u8 in one allocation
        ws = torch.empty(ws_bytes + 256, dtype=torch.uint8, device=dev)
        shift = (-ws.data_ptr()) % 256
        out = res[:4 * n].view(torch.float32)
        pred = res[4 * max(n, 1):4 * max(n, 1) + n]
        check(self.lib.dc_predict(ptr(feats), fcode, n, ptr(text), tcode, p, dim, mode, float(softmax_temp), int(bool(normalize)),
                                  float(threshold), ctypes.c_void_p(res.data_ptr()), ctypes.c_void_p(res.data_ptr() + 4 * max(n, 1)),
                                  None, ctypes.c_void_p(ws.data_ptr() + shift), ws_bytes, current_stream()))
        self.launches += 3 + int(tcode == _lib.DC_F32) + int(fcode == _lib.DC_F32 or bool(normalize)) + (p + 255) // 256 - 1
        return out, pred

    def predict_queries(self, feats: torch.Tensor, text: torch.Tensor, pos, neg_lists, mode: int, softmax_temp: float,
                        normalize: bool, threshold: float):
        """`predict` for Qq queries over one prompt table in one library call: the (N, P) similarity matrix is computed
        once and every query is scored from its own columns. text (P,C) already normalised rows; pos[q] is query q's
        positive row, neg_lists[q] its negative rows (None: no negatives, RAW). Row q of the result equals
        predict(feats, text[[pos[q]] + neg_lists[q]], ...). Returns (score (Qq,N) fp32, pred (Qq,N) uint8)."""
        n_prompts = int(text.shape[0])
        pos_a, off, cols = query_csr(pos, neg_lists, n_prompts)
        if (mode == _lib.DC_GROUND_RAW) != (cols.size == 0) or (mode != _lib.DC_GROUND_RAW and (np.diff(off) == 0).any()):
            raise ValueError("raw mode takes no negatives; paired and argmax need negatives for every query")
        n, dim = feats.shape
        q = int(pos_a.size)
        dev = feats.device
        if q == 0:
            return torch.empty((0, n), dtype=torch.float32, device=dev), torch.empty((0, n), dtype=torch.uint8, device=dev)
        text = text.contiguous()
        if text.dtype not in (torch.float16, torch.float32):
            text = text.float()
        fcode, tcode = _lib.torch_dtype_code(feats.dtype), _lib.torch_dtype_code(text.dtype)
        ws_bytes = self.lib.dc_predict_queries_workspace(n, n_prompts, q, int(cols.size), dim, fcode, tcode)
        res = torch.empty(max(q * n, 1) * 5 + 256, dtype=torch.uint8, device=dev)  # score fp32 + pred u8 in one allocation
        ws = torch.empty(ws_bytes + 256, dtype=torch.uint8, device=dev)
        shift = (-ws.data_ptr()) % 256
        score = res[:4 * q * n].view(torch.float32).view(q, n)
        pred = res[4 * max(q * n, 1):4 * max(q * n, 1) + q * n].view(q, n)
        c_i32 = lambda a: a.ctypes.data_as(ctypes.c_void_p)  # noqa: E731
        check(self.lib.dc_predict_queries(
            ptr(feats), fcode, n, ptr(text), tcode, n_prompts, dim, c_i32(pos_a), c_i32(off), c_i32(cols) if cols.size else None,
            q, mode, float(softmax_temp), int(bool(normalize)), float(threshold), ctypes.c_void_p(res.data_ptr()),
            ctypes.c_void_p(res.data_ptr() + 4 * max(q * n, 1)), ctypes.c_void_p(ws.data_ptr() + shift), ws_bytes,
            current_stream()))
        if n > 0:
            self.launches += 4 + int(tcode == _lib.DC_F32) + int(fcode == _lib.DC_F32 or bool(normalize)) + (n_prompts + 255) // 256 - 1
        else:
            self.launches += 1
        return score, pred

    def predict_many(self, feats: torch.Tensor, counts, text: torch.Tensor, prompt_counts, pos, neg_lists, mode: int,
                     softmax_temp: float, normalize: bool, threshold: float):
        """`predict_queries` for every scene of a batch in one library call. feats (sum N, C) holds the scenes' rows in
        scene order, counts[s] = N_s; text (sum P, C) the scenes' prompt blocks (already normalised rows),
        prompt_counts[s] = P_s; pos[s] / neg_lists[s] (None: no negatives, RAW) index scene s's prompt block as in
        predict_queries. Every index, count and mode rule is checked before anything reaches the device. Returns one
        (score (Q_s, N_s) fp32, pred (Q_s, N_s) uint8) pair per scene, views into one score and one pred buffer; each
        equals predict_queries(rows of scene s, text block of scene s, pos[s], neg_lists[s], ...)."""
        counts = [int(c) for c in counts]
        prompt_counts = [int(p) for p in prompt_counts]
        s_n = len(counts)
        if len(prompt_counts) != s_n or len(pos) != s_n or (neg_lists is not None and len(neg_lists) != s_n):
            raise ValueError(f"{s_n} scenes but {len(prompt_counts)} prompt counts, {len(pos)} positive lists"
                             + ("" if neg_lists is None else f", {len(neg_lists)} negative lists"))
        if any(c < 0 for c in counts) or sum(counts) != feats.shape[0]:
            raise ValueError(f"point counts {counts} do not sum to the {feats.shape[0]} feature rows")
        if any(p < 0 for p in prompt_counts) or sum(prompt_counts) != text.shape[0]:
            raise ValueError(f"prompt counts {prompt_counts} do not sum to the {text.shape[0]} prompt rows")
        tables = [query_csr(pos[s], None if neg_lists is None else neg_lists[s], prompt_counts[s]) for s in range(s_n)]
        for _, off, cols in tables:
            raw = mode == _lib.DC_GROUND_RAW
            if off.size > 1 and (raw != (cols.size == 0) or (not raw and (np.diff(off) == 0).any())):
                raise ValueError("raw mode takes no negatives; paired and argmax need negatives for every query")
        q_counts = [int(t[0].size) for t in tables]
        dev = feats.device
        cells = [q * n for q, n in zip(q_counts, counts)]
        res = torch.empty(max(sum(cells), 1) * 5 + 256, dtype=torch.uint8, device=dev)  # score fp32 + pred u8 in one allocation
        pred_base = 4 * max(sum(cells), 1)
        out, at = [], 0
        for q, n, c in zip(q_counts, counts, cells):
            out.append((res[4 * at:4 * (at + c)].view(torch.float32).view(q, n), res[pred_base + at:pred_base + at + c].view(q, n)))
            at += c
        if s_n == 0 or sum(q_counts) == 0:
            return out
        n_total, dim = feats.shape
        text = text.contiguous()
        if text.dtype not in (torch.float16, torch.float32):
            text = text.float()
        point_off = _prefix(counts).astype(np.int64)
        prompt_off = _prefix(prompt_counts).astype(np.int32)
        query_off = _prefix(q_counts).astype(np.int32)
        pos_a = np.concatenate([t[0] for t in tables]).astype(np.int32)
        cols = np.concatenate([t[2] for t in tables]).astype(np.int32)
        off = _prefix([int(t[1][-1]) for t in tables])
        neg_off = np.concatenate([[0]] + [t[1][1:] + off[s] for s, t in enumerate(tables)]).astype(np.int32)
        fcode, tcode = _lib.torch_dtype_code(feats.dtype), _lib.torch_dtype_code(text.dtype)
        c_p = lambda a: a.ctypes.data_as(ctypes.c_void_p)  # noqa: E731
        ws_bytes = self.lib.dc_predict_many_workspace(s_n, c_p(point_off), c_p(prompt_off), c_p(query_off), int(cols.size),
                                                      dim, fcode, tcode)
        ws = torch.empty(ws_bytes + 256, dtype=torch.uint8, device=dev)
        shift = (-ws.data_ptr()) % 256
        check(self.lib.dc_predict_many(
            ptr(feats) if n_total else None, fcode, ptr(text) if text.shape[0] else None, tcode, dim, s_n, c_p(point_off),
            c_p(prompt_off), c_p(query_off), c_p(pos_a), c_p(neg_off), c_p(cols) if cols.size else None, mode,
            float(softmax_temp), int(bool(normalize)), float(threshold), ctypes.c_void_p(res.data_ptr()),
            ctypes.c_void_p(res.data_ptr() + pred_base), ctypes.c_void_p(ws.data_ptr() + shift), ws_bytes, current_stream()))
        return out

    def minmax_threshold(self, values, minmax, use_raw: bool, threshold: float, want_pred: bool):
        pred = torch.empty(values.numel(), dtype=torch.uint8, device=values.device) if want_pred else None
        check(self.lib.dc_minmax_threshold(ptr(values), values.numel(), ptr(minmax), int(use_raw), float(threshold),
                                           int(want_pred), ptr(pred), current_stream()))
        self.launches += 1
        return pred

    # ------------------------------------------------------------------ (5) voxelisation
    def voxelize(self, xyz: torch.Tensor, sample_off: torch.Tensor, voxel_size: float, labels=None, ignore_label=-100):
        """Batch sparse_quantize. xyz (sum N,3) fp32, sample_off (B+1) int64 device.
        Returns dict(coords, unique_map, inverse_map, voxel_labels, voxel_off) in the C-ABI layout."""
        total = int(xyz.shape[0])
        nb = int(sample_off.numel()) - 1
        dev = xyz.device
        coords = torch.empty((max(total, 1), 3), dtype=torch.int32, device=dev)
        umap = torch.empty(max(total, 1), dtype=torch.int64, device=dev)
        imap = torch.empty(max(total, 1), dtype=torch.int64, device=dev)
        vlab = torch.empty(max(total, 1), dtype=torch.int32, device=dev) if labels is not None else None
        voff = torch.empty(nb + 1, dtype=torch.int64, device=dev)
        ws_bytes = self.lib.dc_voxelize_workspace(total)
        ws = torch.empty(ws_bytes, dtype=torch.uint8, device=dev)
        check(self.lib.dc_voxelize(ptr(xyz), ptr(sample_off), nb, total, float(voxel_size), ptr(labels), int(ignore_label),
                                   ptr(coords), ptr(umap), ptr(imap), ptr(vlab), ptr(voff), ptr(ws), ws_bytes,
                                   current_stream()))
        self.launches += 10
        return {"coords": coords, "unique_map": umap, "inverse_map": imap, "voxel_labels": vlab, "voxel_off": voff}

    def voxel_gather(self, rows: torch.Tensor, sample_off, vox, n_voxels_total: int):
        rows = rows.contiguous()
        width = int(rows.shape[1])
        out = torch.empty((n_voxels_total, width), dtype=rows.dtype, device=rows.device)
        check(self.lib.dc_voxel_gather(ptr(rows), width * rows.element_size(), ptr(sample_off), ptr(vox["voxel_off"]),
                                       ptr(vox["unique_map"]), int(sample_off.numel()) - 1, int(rows.shape[0]), ptr(out),
                                       current_stream()))
        self.launches += 1
        return out
