"""Drop-in for the reference's `utils/feature_fusion.py` (class MultiviewFeatureFusion).

Same constructor arguments, method names, positional order, return containers, dtypes and
devices as the reference (SURVEY.md §8a rows a1-a9, quirks q1-q14); the arithmetic runs in
libdropclip's CUDA kernels through `engine.FusionEngine`. There is no CPU path: a non-CUDA
`device` raises.

Reference lines mirrored: utils/feature_fusion.py:15-350.
"""
from __future__ import annotations

from typing import Dict, Optional, Tuple

import numpy as np
import torch

from . import _lib
from .engine import FusionEngine, PinnedStaging, SceneBatch

__all__ = ["MultiviewFeatureFusion"]


def _require_cuda(device) -> torch.device:
    dev = torch.device(device)
    if dev.type != "cuda":
        raise RuntimeError(f"dropclip_b200 runs on CUDA devices only (got device={device!r}); there is no CPU fallback")
    return dev


class MultiviewFeatureFusion:
    def __init__(
        self,
        camera_intrinsic: Dict[str, float],
        visibility_threshold: float = 0.05,
        image_size: Tuple[float] = (480, 640),
        patch_size: int = 14,
        feature_size: int = 768,
        use_visibility: bool = True,
        use_similarity: bool = True,
        use_sim_kernel: Optional[str] = None,
        use_obj_prior: bool = True,
        norm_feat: bool = True,
        device="cuda",
    ):
        self.visibility_threshold = visibility_threshold
        self.height, self.width = image_size
        self.feature_size = feature_size
        self.patch_size = patch_size
        self.camera_intrinsic = camera_intrinsic
        self.K = np.asarray([
            [camera_intrinsic["fx"], 0, camera_intrinsic["cx"]],
            [0, camera_intrinsic["fy"], camera_intrinsic["cy"]],
            [0, 0, 1],
        ])
        self.device = device
        self.use_obj_prior = use_obj_prior
        self.norm_feat = norm_feat
        self.use_visibility = use_visibility
        self.use_similarity = use_similarity
        if self.use_similarity:
            assert use_sim_kernel is not None, "Remember to set similarity kernel for `use_similarity=True`"
            self.sim_method = use_sim_kernel
        self._engine: Optional[FusionEngine] = None
        self._staging: Optional[PinnedStaging] = None

    # ------------------------------------------------------------------ helpers
    def _eng(self, device) -> FusionEngine:
        dev = _require_cuda(device)
        if self._engine is None or self._engine.device != dev:
            self._engine = FusionEngine(dev)
            self._staging = PinnedStaging(dev)
        return self._engine

    def _sim_kernel(self):
        if not self.use_similarity:
            return None
        if self.sim_method not in ("max", "mean"):
            raise ValueError("Please set method in [mean, max]")
        return self.sim_method

    def _scene(self, points, depths, camera_poses, labels=None, seg_masks=None, mv_features=None, query=None):
        intr = dict(self.camera_intrinsic)
        intr["height"], intr["width"] = int(self.height), int(self.width)
        return {"points": points, "depths": depths, "camera_poses": camera_poses, "labels": labels,
                "seg_masks": seg_masks, "mv_features": mv_features, "query_embeddings": query, "intrinsic": intr}

    def calculate_sim(self, pos, neg, eps=1e-6):
        """utils/feature_fusion.py:65-73 (tiny tensor expression kept for API parity; the fused
        paths evaluate the same formula inside the CUDA epilogues)."""
        if self.sim_method == "max":
            return torch.clip(pos - torch.max(neg, dim=-1)[0], eps).squeeze().float()
        elif self.sim_method == "mean":
            return torch.clip(pos - neg.mean(-1), eps).squeeze().float()
        else:
            raise ValueError("Please set method in [mean, max]")

    @staticmethod
    def _cvt_o3d_coords(pts):
        pts[:, 1] = -pts[:, 1]
        pts[:, 2] = -pts[:, 2]
        return pts

    # ------------------------------------------------------------------ a3
    def get_visibility_mask(self, points, depths, camera_poses, device=None):
        """(V,N) int64 tensor on the CPU, like the reference (quirk q5)."""
        device = device or self.device
        eng = self._eng(device)
        if len(depths) == 0 or points.shape[0] == 0:
            return torch.zeros((len(depths), points.shape[0]), dtype=int)
        b = SceneBatch.from_host([self._scene(points, depths, camera_poses)], eng.device, staging=self._staging)
        records, rank, _ = eng.visibility_sorted(b, self.visibility_threshold)
        mask = eng.unpack_visibility(b, records, rank, torch.int64)
        staged = self._staging.download(mask.view(len(depths), points.shape[0]))
        torch.cuda.current_stream().synchronize()
        return staged.clone()

    # ------------------------------------------------------------------ a6
    @staticmethod
    def reconstruct_per_obj_feat(pc, label, feat, obj_ids):
        """out[label == obj_ids[i]] = feat[i] for i >= 1, zeros elsewhere; CPU fp32 (N,C).
        Runs the scatter kernel when a GPU is present (the reference does this on the CPU)."""
        with torch.no_grad():
            n = pc.shape[0]
            ids = list(obj_ids)
            if ids != list(range(len(ids))):
                # arbitrary id lists: remap labels to row indices first
                lut = {o: i for i, o in enumerate(ids)}
                label = np.asarray([lut.get(int(x), -1) for x in np.asarray(label).reshape(-1)], dtype=np.int64)
            eng = FusionEngine("cuda")
            dev = eng.device
            fused = feat.to(dev, torch.float32).contiguous()
            labels = torch.from_numpy(np.asarray(label).astype(np.int64).reshape(-1)).to(dev)
            q_off = torch.tensor([0, fused.shape[0]], dtype=torch.int64, device=dev)
            p_off = torch.tensor([0, n], dtype=torch.int64, device=dev)
            out = torch.empty((n, fused.shape[1]), dtype=torch.float32, device=dev)
            _lib.check(eng.lib.dc_scatter_to_points(_lib.ptr(fused), _lib.ptr(q_off), _lib.ptr(labels), _lib.ptr(p_off), 1, n,
                                                   int(fused.shape[1]), 1, _lib.ptr(out), _lib.current_stream()))
            return out.cpu()

    # ------------------------------------------------------------------ a7 / a8 (pixel level)
    @torch.no_grad()
    def aggregate_features(self, points, depths, seg_masks, camera_poses, mv_features, query_embeddings=None, device=None):
        device = device or self.device
        eng = self._eng(device)
        if self.use_similarity:
            assert query_embeddings is not None, "Must provide query embeddings for using similarity."
        b = self._pixel_batch(eng, self._staging, points, depths, seg_masks, camera_poses, mv_features, query_embeddings)
        mask, _, _ = eng.visibility(b, self.visibility_threshold, torch.uint8)
        sums, weight = eng.pixel_fuse(b, mask, self._sim_kernel(), self.norm_feat)
        n_views, n_pts = len(depths), points.shape[0]
        vis = mask.view(n_views, n_pts).to(torch.int64)
        simw = weight.view(n_views, n_pts) if self.use_similarity else None
        return sums, vis, simw

    def _pixel_batch(self, eng, staging, points, depths, seg_masks, camera_poses, mv_features, query_embeddings):
        """Host -> device upload of one scene with its patch maps (pinned staging, async H2D on the current stream).
        The reference normalises its own upsampled copy of the maps under norm_feat, so nothing is written back."""
        segs = [s.cpu().numpy() if isinstance(s, torch.Tensor) else s for s in seg_masks]
        feats = [f.float() for f in mv_features]
        assert feats[0].shape[-1] == self.feature_size
        q = query_embeddings if self.use_similarity else None
        return SceneBatch.from_host([self._scene(points, depths, camera_poses, None, segs, feats, q)], eng.device,
                                    pixel_features=True, staging=staging)

    def _stage_pix(self, eng, staging, points, colors, labels, depths, seg_masks, camera_poses, mv_features, query_embeddings):
        """Staging half of fuse_points: the scene and the rows it hands back, uploaded on the current stream."""
        b = self._pixel_batch(eng, staging, points, depths, seg_masks, camera_poses, mv_features, query_embeddings)
        self._stage_rows(b, staging, points, colors, labels)
        return b

    def _finish_pix(self, eng, b, points, colors, labels):
        """Finishing half of fuse_points on the current stream. Every compaction is enqueued at its upper bound (all
        points kept) and laid out from the kept count on the device, so the one host wait, for that count, also covers
        the read-back of the returned rows."""
        n_views = b.total_views
        kern = self._sim_kernel()
        host_rows = {"points": points, "colors": colors, "labels": labels}
        if b.total_points == 0:  # an empty cloud: the projection and fusion launches need at least one point
            feats = torch.empty((0, int(b.feats.shape[-1])), dtype=torch.float32, device=b.device)
            vis = torch.empty((n_views, 0), dtype=torch.int64, device=b.device)
            simw = torch.empty((n_views, 0), dtype=torch.float32, device=b.device) if kern is not None else None
            keep = np.zeros(0, dtype=bool)
            return (feats, vis, simw), tuple(arr[keep] for arr in host_rows.values())
        mask, any_vis, _ = eng.visibility(b, self.visibility_threshold, torch.uint8)
        # the division by sum_v visibility / sum_v similarity (:266-268) is fused into the fusion kernel
        sums, weight = eng.pixel_fuse(b, mask, kern, self.norm_feat, normalize=True)
        masks = [(mask, torch.int64)] + ([(weight.view(torch.int32), None)] if weight is not None else [])
        dev_rows = b.row_sources
        names = list(dev_rows)
        kept_off, masks_out, rows_out = eng.compact_unsized(b, any_vis, masks, [sums] + [dev_rows[k] for k in names])
        kept_host = self._pinned_like(kept_off)
        kept_host.copy_(kept_off, non_blocking=True)
        outs = {}
        for k, t in zip(names, rows_out[1:]):
            outs[k] = self._pinned_like(t)
            outs[k].copy_(t, non_blocking=True)
        keep_host = None
        if len(names) < 3:  # some array could not travel as raw rows: filter it on the host like the reference
            keep_host = self._pinned_like(any_vis)
            keep_host.copy_(any_vis, non_blocking=True)
        torch.cuda.current_stream().synchronize()
        n_kept = int(kept_host[-1])
        vis = masks_out[0][: n_views * n_kept].view(n_views, n_kept)
        simw = masks_out[1][: n_views * n_kept].view(torch.float32).view(n_views, n_kept) if weight is not None else None
        final = []
        for name, arr in host_rows.items():
            if name in outs:
                final.append(outs[name].numpy()[:n_kept].view(arr.dtype).reshape((n_kept,) + tuple(np.shape(arr)[1:])))
            else:
                final.append(arr[keep_host.numpy().astype(bool)])
        return (rows_out[0][:n_kept], vis, simw), tuple(final)

    def fuse_points(self, points, colors, labels, depths, seg_masks, camera_poses, mv_features, query_embeddings, device=None):
        device = device or self.device
        eng = self._eng(device)
        b = self._stage_pix(eng, self._staging, points, colors, labels, depths, seg_masks, camera_poses, mv_features,
                            query_embeddings)
        return self._finish_pix(eng, b, points, colors, labels)

    # ------------------------------------------------------------------ a4 (object level)
    def _stage_obj(self, eng, staging, points, labels, depths, seg_masks, camera_poses, mv_features, query_embeddings,
                   colors=None):
        """Host -> device upload of one scene (pinned staging, chunked async H2D on the current stream)."""
        feats = list(mv_features)
        for f in feats:
            if f.shape[-1] != 768:  # quirk q11: the object path is hard-wired to 768 channels
                raise RuntimeError(f"The expanded size of the tensor (768) must match the existing size ({f.shape[-1]})")
        segs = [s.cpu().numpy() if isinstance(s, torch.Tensor) else s for s in seg_masks]
        b = SceneBatch.from_host([self._scene(points, depths, camera_poses, labels, segs, feats, query_embeddings)],
                                 eng.device, staging=staging)
        self._stage_rows(b, staging, points, colors, labels)
        return b

    @staticmethod
    def _stage_rows(b, staging, points, colors, labels):
        """Rows that are only filtered and handed back (points[keep], colors[keep], labels[keep]) travel as raw bytes, so
        that the filtering can run on the device: b.row_sources maps each array that can to its (N, row) device tensor."""
        n_pts = b.total_points
        b.row_sources = {}
        for name, arr in (("points", points), ("colors", colors), ("labels", labels)):
            if name == "points" and isinstance(arr, np.ndarray) and arr.dtype == np.float64:
                b.row_sources[name] = b.points
            elif name == "labels" and b.labels is not None and isinstance(arr, np.ndarray) and arr.dtype == np.int64:
                b.row_sources[name] = b.labels.view(-1, 1)
            elif isinstance(arr, np.ndarray) and arr.ndim >= 1 and arr.shape[0] == n_pts and n_pts > 0 and \
                    arr.dtype.kind in "fiub" and arr.size > 0:
                # any fixed-width dtype travels as raw bytes (uint8 colours, int32 / uint8 labels, fp16 points ...)
                b.row_sources[name] = staging.upload(np.ascontiguousarray(arr).reshape(n_pts, -1).view(np.uint8))
        staging.end()

    @staticmethod
    def _pinned_like(t: torch.Tensor) -> torch.Tensor:
        """Fresh pinned host tensor (torch's caching host allocator recycles the blocks once the caller
        drops the result), so results are handed out without a second host copy."""
        return torch.empty(t.shape, dtype=t.dtype, pin_memory=True)

    def _finish_obj(self, eng, staging, b, points, colors, labels, depths, mv_features, query_embeddings, return_obj):
        n_views = len(mv_features)
        n_objects = query_embeddings.shape[0]
        res = eng.fuse_object_level(b, self.visibility_threshold, self.use_visibility, self.use_similarity,
                                    self._sim_kernel(), torch.uint8)
        status_host = self._pinned_like(res["view_status"][:n_views])
        status_host.copy_(res["view_status"][:n_views], non_blocking=True)  # read after the sync inside compact_visibility
        # The rows returned next to the features (points[keep], colors[keep], labels[keep]) are compacted on
        # the device as raw bytes and read back, instead of a host-side boolean take (3-4 ms per scene).
        host_rows = {"points": points, "colors": colors, "labels": labels}
        dev_rows = getattr(b, "row_sources", {})
        names = list(dev_rows)
        new_index, kept_off, kept_host, out_off_host, cmask, rows_out = eng.compact_visibility(
            b, res["any_visible"], res["records"], res["rank"], torch.int64, [dev_rows[k] for k in names])
        n_kept = int(kept_host[-1])
        status = status_host.numpy()
        if (status & 1).any():
            v = int(np.flatnonzero(status & 1)[0])
            raise IndexError(f"index out of bounds: view {v} contains an instance id outside [0, {n_objects})")
        if (status & 2).any():
            v = int(np.flatnonzero(status & 2)[0])
            rows = mv_features[v].shape[0]
            raise IndexError(f"index {rows} is out of bounds for dimension 0 with size {rows}")
        # int64 mask widened on the device (58 MB at V=73, N=100k: ~1 ms over PCIe instead of a ~4 ms
        # uint8 -> int64 conversion on the host), straight into the pinned tensor that is returned
        visibility_mask = self._pinned_like(cmask.view(len(depths), n_kept))
        visibility_mask.copy_(cmask.view(len(depths), n_kept), non_blocking=True)
        outs = {}
        for k, t in zip(names, rows_out):
            h = self._pinned_like(t)
            h.copy_(t, non_blocking=True)
            outs[k] = h
        keep = None
        if len(names) < 3:  # some array could not travel as raw rows: filter it on the host like the reference
            keep = np.flatnonzero(res["any_visible"].cpu().numpy())
        weight_obj = res["weight_obj"][: n_objects * n_views].view(n_objects, n_views)
        mv_feats_obj = res["fused"]
        if not return_obj:
            k_off = torch.tensor([0, n_kept], dtype=torch.int64, device=eng.device)
            # the scatter kernel reads int64 ids: compact the batch's own int64 copy of the labels, never the caller's
            # raw rows (int32 / uint8 / float labels are returned in their dtype but must not be reinterpreted)
            if "labels" in names and dev_rows["labels"].dtype == torch.int64:
                lab_dev = rows_out[names.index("labels")].reshape(-1)
            else:
                lab_dev = eng.compact_rows(b.labels, res["any_visible"], new_index, n_kept).reshape(-1)
            mv_feats = eng.scatter_to_points(b, mv_feats_obj, lab_dev, k_off, 1, n_kept, skip_first=True).cpu()
        else:
            mv_feats = mv_feats_obj
        torch.cuda.current_stream().synchronize()
        final = []
        for name, arr in host_rows.items():
            if name in outs:
                final.append(outs[name].numpy().view(arr.dtype).reshape((n_kept,) + tuple(np.shape(arr)[1:])))
            else:
                final.append(arr.take(keep, axis=0) if isinstance(arr, np.ndarray) else np.asarray(arr)[keep])
        return (mv_feats, weight_obj, visibility_mask), tuple(final)

    @torch.no_grad()
    def fuse_obj_prior(self, points, colors, labels, depths, seg_masks, camera_poses, mv_features, query_embeddings,
                       return_obj=False, device=None):
        # like the reference, the visibility stage runs on self.device, the rest on `device` (q5)
        device = device or self.device
        eng = self._eng(device)
        b = self._stage_obj(eng, self._staging, points, labels, depths, seg_masks, camera_poses, mv_features, query_embeddings,
                            colors)
        return self._finish_obj(eng, self._staging, b, points, colors, labels, depths, mv_features, query_embeddings,
                                return_obj)

    @torch.no_grad()
    def fuse_many(self, scenes, return_obj=True, device=None):
        """Throughput form of `fuse`: `scenes` is an iterable of argument tuples (points, colors, labels, depths,
        seg_masks, camera_poses, mv_features, query_embeddings); yields exactly what `fuse(*args, device=device)`
        returns, in order. The host->device staging of scene i+1 runs on a side stream in a helper thread while scene i
        is fused and read back, so the loop runs at the speed of the slower of the two (PCIe/host-copy bound at MV-TOD
        sizes). Both levels are covered. At object level `return_obj` is passed to each `fuse`; at pixel level
        (use_obj_prior=0) it has no meaning, as `fuse_points` has no such argument, and is ignored. A scene that fails
        raises when the loop reaches it, after every earlier scene was yielded, with the exception `fuse` raises for it.
        This is what the reference's scene loops (tools/preprocess_data.py:188-297, scripts/run_eval.py:205-220) become."""
        from concurrent.futures import ThreadPoolExecutor
        device = device or self.device
        eng = self._eng(device)
        dev = eng.device
        if getattr(self, "_many_stagings", None) is None or self._many_stagings[0].device != dev:
            self._many_stagings = [PinnedStaging(dev), PinnedStaging(dev)]  # pinned buffers are expensive: keep them
        stagings = self._many_stagings
        dev_index = dev.index if dev.index is not None else torch.cuda.current_device()
        # one persistent side stream: the caching allocator keeps a pool per stream, so a fresh stream per call would
        # cudaMalloc every staging buffer again (measured: +6 device allocations and ~150 ms per call)
        if getattr(self, "_many_stream", None) is None or self._many_stream.device != torch.device("cuda", dev_index):
            self._many_stream = torch.cuda.Stream(device=dev)
        side = self._many_stream

        def stage(k, args, ready):
            torch.cuda.set_device(dev_index)
            points, colors, labels, depths, seg_masks, camera_poses, mv_features, query = args
            with torch.cuda.stream(side):
                side.wait_event(ready)  # device inputs the caller produced before handing the scene over
                if self.use_obj_prior:
                    b = self._stage_obj(eng, stagings[k % 2], points, labels, depths, seg_masks, camera_poses, mv_features,
                                        query, colors)
                else:
                    b = self._stage_pix(eng, stagings[k % 2], points, colors, labels, depths, seg_masks, camera_poses,
                                        mv_features, query)
                ev = torch.cuda.Event()
                ev.record(side)
            return b, ev

        def submit(k, args):
            ready = torch.cuda.Event()
            ready.record()
            return pool.submit(stage, k, args, ready)

        it = iter(scenes)
        with ThreadPoolExecutor(max_workers=1) as pool:
            k = 0
            try:
                cur_args = next(it)
            except StopIteration:
                return
            fut = submit(k, cur_args)
            while True:
                b, ev = fut.result()
                try:
                    nxt_args = next(it)
                    fut = submit(k + 1, nxt_args)
                except StopIteration:
                    nxt_args, fut = None, None
                torch.cuda.current_stream().wait_event(ev)
                points, colors, labels, depths, seg_masks, camera_poses, mv_features, query = cur_args
                if self.use_obj_prior:
                    yield self._finish_obj(eng, stagings[k % 2], b, points, colors, labels, depths, mv_features, query,
                                           return_obj)
                else:
                    yield self._finish_pix(eng, b, points, colors, labels)
                if fut is None:
                    return
                cur_args, k = nxt_args, k + 1

    @torch.no_grad()
    def fuse(self, *args, **kwargs):
        if self.use_obj_prior:
            return self.fuse_obj_prior(*args, **kwargs)
        else:
            return self.fuse_points(*args, **kwargs)
