"""GPU versions of the Open3D / SciPy glue the fusion path leans on (`utils/geometry.py`).

The reference delegates these to un-vendored native libraries (open3d 0.15.2, scipy cKDTree), so
parity is anchored on their published semantics and checked against numpy/scipy restatements
(tests/test_gpu_parity.py) - "parity unpinned" for the Open3D ones (DESIGN.md §2).

Reference lines: pc_voxel_down utils/geometry.py:350-352, find_closest_indices :390-401,
rgbd_to_pointcloud_o3d :21-36 (and utils/projections.py:41-56), remove_table_mask :294-300.
"""
from __future__ import annotations

from dataclasses import dataclass

import numpy as np
import torch

from . import _lib
from ._lib import check, current_stream, ptr


def _dev():
    if not torch.cuda.is_available():
        raise RuntimeError("dropclip_b200 needs a CUDA device (sm_100a); there is no CPU path")
    return torch.device("cuda")


def _f64(x) -> torch.Tensor:
    t = x if isinstance(x, torch.Tensor) else torch.from_numpy(np.ascontiguousarray(x, dtype=np.float64))
    return t.to(_dev(), torch.float64).reshape(-1, 3).contiguous()


def _workspace(n: int, size_fn: str = "dc_sort_workspace") -> torch.Tensor:
    return torch.empty(getattr(_lib.load(), size_fn)(int(n)), dtype=torch.uint8, device=_dev())


def voxel_down(points, voxel_size: float, return_first_index: bool = False):
    """Open3D `voxel_down_sample`: one output point per occupied voxel = mean of its points.
    Returns a CUDA fp64 tensor (M,3) (voxels ordered by voxel index)."""
    lib = _lib.load()
    pts = _f64(points)
    n = pts.shape[0]
    out = torch.empty((max(n, 1), 3), dtype=torch.float64, device=pts.device)
    first = torch.empty(max(n, 1), dtype=torch.int64, device=pts.device)
    cnt = torch.zeros(1, dtype=torch.int64, device=pts.device)
    ws = _workspace(n)
    check(lib.dc_voxel_down_mean(ptr(pts), n, float(voxel_size), ptr(out), ptr(first), ptr(cnt), ptr(ws), ws.numel(),
                                 current_stream()))
    m = int(cnt.item())
    return (out[:m], first[:m]) if return_first_index else out[:m]


def voxel_down_trace(points, colors, labels, voxel_size: float):
    """Open3D `voxel_down_sample_and_trace` followed by the label majority vote of
    aggregate_views_blender_new (utils/geometry.py:186-201), on the device: returns CUDA tensors
    (points (M,3) f64, colors (M,3) f64, labels (M,) i64, counts (M,) i64), voxels ordered by voxel index."""
    lib = _lib.load()
    pts = _f64(points)
    n = pts.shape[0]
    dev = pts.device
    cols = _f64(colors) if colors is not None else None
    labs = None
    if labels is not None:
        labs = (labels if isinstance(labels, torch.Tensor) else torch.from_numpy(np.ascontiguousarray(labels))).to(dev, torch.int64)
        labs = labs.reshape(-1).contiguous()
    out_p = torch.empty((max(n, 1), 3), dtype=torch.float64, device=dev)
    out_c = torch.empty((max(n, 1), 3), dtype=torch.float64, device=dev) if cols is not None else None
    out_l = torch.empty(max(n, 1), dtype=torch.int64, device=dev) if labs is not None else None
    counts = torch.empty(max(n, 1), dtype=torch.int64, device=dev)
    m_dev = torch.zeros(1, dtype=torch.int64, device=dev)
    ws = _workspace(n, "dc_voxel_down_trace_workspace")
    check(lib.dc_voxel_down_trace(ptr(pts), ptr(cols), ptr(labs), n, float(voxel_size), ptr(out_p), ptr(out_c), ptr(out_l),
                                  None, ptr(counts), ptr(m_dev), ptr(ws), ws.numel(), current_stream()))
    m = int(m_dev.item())
    return out_p[:m], (out_c[:m] if out_c is not None else None), (out_l[:m] if out_l is not None else None), counts[:m]


def binary_masks_to_seg(masks, obj_ids=None):
    """utils/image.py:11-15 (host numpy; defines the instance-map dtype the hot path receives)."""
    if obj_ids is None:
        obj_ids = np.arange(masks.shape[0], dtype=np.uint8)
    return np.max(masks * obj_ids[:, None, None], axis=0)


def aggregate_views_blender_new(scene, camera_intrinsic, depth_trunc=25.0, voxel_size=None):
    """utils/geometry.py:120-204: back-project every view's valid pixels (depth < depth_trunc), flip to the
    Blender camera convention, move to the world frame, concatenate, and - with `voxel_size` - voxel-grid
    down-sample with mean position / colour and majority-vote instance label. Same arguments and return
    triple (numpy points, colors, labels) as the reference; all arithmetic on the device. Voxels come out
    ordered by voxel index (Open3D's order is its hash map's iteration order)."""
    return aggregate_views_many([scene], camera_intrinsic, depth_trunc, [voxel_size])[0][0]


_MASK_DTYPES = (np.dtype(np.bool_), np.dtype(np.uint8))
_MAX_SORT_ELEMS = 1 << 31


class _View:
    """One view's host inputs, checked and laid out for the staging calls."""

    def __init__(self, view, col_to_ins):
        self.depth = np.ascontiguousarray(view["depth"], dtype=np.float32)
        if self.depth.ndim != 2:
            raise ValueError(f"aggregate_views_many: a depth map must be 2-D, got shape {self.depth.shape}")
        self.h, self.w = self.depth.shape
        n = self.h * self.w
        _, masks, colors = zip(*view["annos"])  # a view without annotations raises ValueError here, as in the reference
        ids = np.asarray([col_to_ins[x] for x in colors])
        rgb = np.asarray(view["rgb"])
        if rgb.ndim < 1 or rgb.shape[-1] != 3 or rgb.size != 3 * n:
            raise ValueError(f"aggregate_views_many: rgb of shape {rgb.shape} does not hold 3 channels per depth pixel")
        self.rgb = np.ascontiguousarray(rgb) if rgb.dtype == np.uint8 else rgb.astype(np.float64)  # exact widening
        world = np.ascontiguousarray(np.asarray(view["camera"]["world_matrix"]), dtype=np.float64).reshape(16)
        self.world = world
        arrs = [m if isinstance(m, np.ndarray) else np.asarray(m) for m in masks]
        shape = arrs[0].shape
        if ids.dtype == np.int64 and len(shape) == 2 and arrs[0].size == n and \
                all(a.dtype in _MASK_DTYPES and a.shape == shape for a in arrs):
            self.masks, self.ids, self.seg = [np.ascontiguousarray(a) for a in arrs], ids, None
        else:  # any other mask / id type: numpy builds the map, exactly as the reference does
            seg = binary_masks_to_seg(np.stack(masks), ids)
            if seg.size != n:
                raise IndexError(f"aggregate_views_many: instance map of shape {seg.shape} does not match the depth map "
                                 f"{self.depth.shape}")
            self.masks, self.ids = None, None
            self.seg = torch.from_numpy(np.ascontiguousarray(seg)).reshape(-1).to(torch.int64).numpy()


def _pointers(arrays):
    return (_lib.c_void_p * max(len(arrays), 1))(*[a.ctypes.data for a in arrays])


def _stage_segs(views, pix_off, n_pix, threads):
    """Instance maps of every view in one pinned buffer: uint8 when every value fits, int64 otherwise."""
    lib = _lib.load()
    fast = [i for i, v in enumerate(views) if v.masks is not None]
    slow = [i for i, v in enumerate(views) if v.masks is None]
    masks = [m for i in fast for m in views[i].masks]
    ids = np.concatenate([views[i].ids for i in fast]) if fast else np.zeros(1, dtype=np.int64)
    mask_off = np.zeros(len(fast) + 1, dtype=np.int64)
    mask_off[1:] = np.cumsum([len(views[i].masks) for i in fast])
    pixels = np.asarray([views[i].h * views[i].w for i in fast] or [0], dtype=np.int64)
    offs = np.asarray([pix_off[i] for i in fast] or [0], dtype=np.int64)
    ptrs = _pointers(masks)
    narrow = all(v.seg.size == 0 or (v.seg.min() >= 0 and v.seg.max() <= 255) for v in (views[i] for i in slow))
    for dtype, code in ((torch.uint8, _lib.DC_U8), (torch.int64, _lib.DC_I64)):
        if dtype == torch.uint8 and not narrow:
            continue
        buf = torch.empty(max(n_pix, 1), dtype=dtype, pin_memory=True)
        bad = _lib.c_int(0)
        check(lib.dc_host_masks_to_seg(ptrs, ids.ctypes.data, mask_off.ctypes.data, len(fast), pixels.ctypes.data,
                                       offs.ctypes.data, code, _lib.c_void_p(buf.data_ptr()), threads, _lib.ctypes.byref(bad)))
        if bad.value:
            continue
        host = buf.numpy()
        for i in slow:
            host[pix_off[i]:pix_off[i + 1]] = views[i].seg
        return buf, code
    raise AssertionError("unreachable: int64 maps always fit")


def _stage_rows(arrays, item_elems, dtype, n_total, threads):
    """Concatenates same-dtype host arrays into one pinned buffer (runs of equal sizes per staging call)."""
    lib = _lib.load()
    buf = torch.empty(max(n_total, 1), dtype=dtype, pin_memory=True)
    esize = buf.element_size()
    pos, i = 0, 0
    while i < len(arrays):
        j = i
        while j < len(arrays) and item_elems[j] == item_elems[i]:
            j += 1
        if item_elems[i]:
            check(lib.dc_host_gather_copy(_pointers(arrays[i:j]), j - i, item_elems[i] * esize,
                                          _lib.c_void_p(buf.data_ptr() + pos * esize), threads))
        pos += (j - i) * item_elems[i]
        i = j
    return buf


def aggregate_views_many(scenes, camera_intrinsic, depth_trunc=25.0, voxel_sizes=(None,)):
    """`aggregate_views_blender_new` for a batch of scenes at every voxel size of a sweep in one call.

    `scenes` holds scene dicts in the reference layout (views[v] = {rgb, depth, annos=[(_, mask, colour)],
    camera: {world_matrix}}, plus col_to_ins) that share `camera_intrinsic`; `voxel_sizes` holds T entries, each a
    float or None (no down-sampling), duplicates allowed. Returns out[s][t] = (points, colors, labels) numpy arrays,
    bit-equal to aggregate_views_blender_new(scenes[s], camera_intrinsic, depth_trunc, voxel_sizes[t]).

    The instance maps are built on the host (bool / uint8 masks in one threaded pass, other types by numpy) and
    shipped as uint8 when every value fits; compaction, back-projection and one segmented voxel-down-trace over
    all (scene, distinct voxel size) pairs run on the device. The host waits for the result sizes, then for the
    read-back into pinned memory. Every error is raised before any device work; the sort indexes points with
    int32, so pixels x distinct voxel sizes must stay below 2^31 (ValueError otherwise)."""
    from .engine import PinnedStaging
    lib = _lib.load()
    scenes = list(scenes)
    if not scenes:
        return []
    sizes = list(voxel_sizes)
    size_index, distinct = [], []
    for v in sizes:
        if v is None:
            size_index.append(None)
            continue
        f = float(v)
        if not f > 0.0:  # 0, negative, NaN: the library's argument error, as the single-scene call raised it
            raise _lib.DropClipError(-1, f"aggregate_views_many: voxel_size must be positive, got {v!r}")
        if f not in distinct:
            distinct.append(f)
        size_index.append(distinct.index(f))
    trunc32 = _lib.c_float(float(depth_trunc))  # the reference compares fp32 depths with the fp32 image of the scalar
    if distinct and trunc32.value != trunc32.value:
        raise ValueError("aggregate_views_many: depth_trunc is NaN, so no pixel is labelled and the label vote has no input")
    views, scene_view_off = [], [0]
    for sc in scenes:
        vs = sc["views"]
        if len(vs) == 0:
            raise ValueError("aggregate_views_many: a scene has no views")
        views.extend(_View(stuff, sc["col_to_ins"]) for _, stuff in vs.items())
        scene_view_off.append(len(views))
    pix = [v.h * v.w for v in views]
    pix_off = np.zeros(len(views) + 1, dtype=np.int64)
    pix_off[1:] = np.cumsum(pix)
    n_pix = int(pix_off[-1])
    if n_pix >= _MAX_SORT_ELEMS or n_pix * len(distinct) >= _MAX_SORT_ELEMS:
        raise ValueError(f"aggregate_views_many: {n_pix} pixels x {len(distinct)} distinct voxel sizes reach 2^31; "
                         "split the batch")
    if len(scenes) > 65535:
        raise ValueError("aggregate_views_many: at most 65535 scenes per call")

    threads = PinnedStaging._host_threads()
    S, V, U = len(scenes), len(views), len(distinct)
    seg_buf, seg_code = _stage_segs(views, pix_off, n_pix, threads)
    depth_buf = _stage_rows([v.depth for v in views], pix, torch.float32, n_pix, threads)
    rgb_u8 = all(v.rgb.dtype == np.uint8 for v in views)
    rgbs = [v.rgb if rgb_u8 else v.rgb.astype(np.float64, copy=False) for v in views]
    rgb_buf = _stage_rows(rgbs, [3 * p for p in pix], torch.uint8 if rgb_u8 else torch.float64, 3 * n_pix, threads)
    hw = np.asarray([[v.h, v.w] for v in views], dtype=np.int32).reshape(-1)
    poses = np.concatenate([v.world for v in views])
    k4 = np.asarray([camera_intrinsic["fx"], camera_intrinsic["fy"], camera_intrinsic["cx"], camera_intrinsic["cy"]],
                    dtype=np.float64)
    svo = np.asarray(scene_view_off, dtype=np.int32)
    vsz = np.asarray(distinct or [0.0], dtype=np.float64)

    dev = _dev()
    d_depth = depth_buf.to(dev, non_blocking=True)
    d_seg = seg_buf.to(dev, non_blocking=True)
    d_rgb = rgb_buf.to(dev, non_blocking=True)
    rows = max(n_pix, 1)
    pts = torch.empty((rows, 3), dtype=torch.float64, device=dev)
    cols = torch.empty((rows, 3), dtype=torch.float64, device=dev)
    labs = torch.empty(rows, dtype=torch.int64, device=dev)
    offs = torch.empty(2 * (S + 1) + U * S + 1, dtype=torch.int64, device=dev)  # point_off, label_off, vox_off
    vrows = max(U * n_pix, 1)
    v_pts = torch.empty((vrows, 3), dtype=torch.float64, device=dev) if U else None
    v_cols = torch.empty((vrows, 3), dtype=torch.float64, device=dev) if U else None
    v_labs = torch.empty(vrows, dtype=torch.int64, device=dev) if U else None
    ws = torch.empty(lib.dc_aggregate_views_workspace(S, V, n_pix, U), dtype=torch.uint8, device=dev)
    cp = _lib.c_void_p
    check(lib.dc_aggregate_views(ptr(d_depth), ptr(d_seg), seg_code, ptr(d_rgb), _lib.DC_U8 if rgb_u8 else _lib.DC_F64,
                                 cp(pix_off.ctypes.data), cp(hw.ctypes.data), cp(svo.ctypes.data), cp(poses.ctypes.data),
                                 cp(k4.ctypes.data), trunc32, cp(vsz.ctypes.data), S, V, U, ptr(pts), ptr(cols), ptr(labs),
                                 cp(offs.data_ptr()), cp(offs.data_ptr() + 8 * (S + 1)), ptr(v_pts), ptr(v_cols), ptr(v_labs),
                                 cp(offs.data_ptr() + 16 * (S + 1)), ptr(ws), ws.numel(), current_stream()))
    h_offs = torch.empty(offs.shape, dtype=torch.int64, pin_memory=True)
    h_offs.copy_(offs, non_blocking=True)
    torch.cuda.current_stream().synchronize()  # the sizes of every result
    o = h_offs.numpy()
    pt_off, lab_off, vox_off = o[:S + 1], o[S + 1:2 * (S + 1)], o[2 * (S + 1):]

    def back(t, n):
        h = torch.empty((n,) + tuple(t.shape[1:]), dtype=t.dtype, pin_memory=True)
        if n:
            h.copy_(t[:n], non_blocking=True)
        return h

    h_pts, h_cols, h_labs = back(pts, int(pt_off[S])), back(cols, int(pt_off[S])), back(labs, int(lab_off[S]))
    m = int(vox_off[U * S]) if U else 0
    h_vp, h_vc, h_vl = (back(v_pts, m), back(v_cols, m), back(v_labs, m)) if U else (None, None, None)
    torch.cuda.current_stream().synchronize()  # the read-back
    out = []
    for s in range(S):
        handed, res = set(), []
        for u in size_index:
            if u is None:
                a, b, la, lb = pt_off[s], pt_off[s + 1], lab_off[s], lab_off[s + 1]
                r = (h_pts.numpy()[a:b], h_cols.numpy()[a:b], h_labs.numpy()[la:lb])
            else:
                a, b = vox_off[u * S + s], vox_off[u * S + s + 1]
                r = (h_vp.numpy()[a:b], h_vc.numpy()[a:b], h_vl.numpy()[a:b])
            if u in handed:  # a repeated size gets arrays of its own
                r = tuple(x.copy() for x in r)
            handed.add(u)
            res.append(r)
        out.append(res)
    return out


def pc_voxel_down(pc, voxel_size=0.0075):
    return voxel_down(pc, voxel_size).cpu().numpy()


def nearest_index(query, ref, return_dist2: bool = False):
    lib = _lib.load()
    q, r = _f64(query), _f64(ref)
    out = torch.empty(q.shape[0], dtype=torch.int64, device=q.device)
    d2 = torch.empty(q.shape[0], dtype=torch.float64, device=q.device) if return_dist2 else None
    check(lib.dc_nearest_index(ptr(q), q.shape[0], ptr(r), r.shape[0], ptr(out), ptr(d2), current_stream()))
    return (out, d2) if return_dist2 else out


def find_closest_indices(full_pc, filtered_pc, eps=None):
    """For each point of `filtered_pc` the index of its nearest neighbour in `full_pc`."""
    if eps is None:
        return nearest_index(filtered_pc, full_pc).cpu().numpy()
    idx, d2 = nearest_index(filtered_pc, full_pc, True)
    idx, dist = idx.cpu().numpy(), np.sqrt(d2.cpu().numpy())
    return idx[np.argwhere(dist <= eps)]


@dataclass
class PointCloud:
    """Stand-in for the open3d.geometry.PointCloud the reference returns (points / colors arrays)."""
    points: np.ndarray
    colors: np.ndarray


def rgbd_to_pointcloud_o3d(rgb, depth, camera_intrinsics, depth_scale=1.0, depth_trunc=25.0):
    """Open3D create_from_rgbd_image semantics: pixels with 0 < depth/scale < trunc, row-major,
    x = (u - cx) * z / fx, y = (v - cy) * z / fy, colours / 255."""
    dev = _dev()
    d = torch.as_tensor(np.ascontiguousarray(depth, dtype=np.float32)).to(dev) / float(depth_scale)
    d = torch.where(d >= float(depth_trunc), torch.zeros_like(d), d)
    keep = (d > 0).reshape(-1)
    from .projections import backproject
    pts = backproject(d, camera_intrinsics, o3d_rounding=True)[0].reshape(-1, 3)[keep]
    col = torch.as_tensor(np.ascontiguousarray(rgb)).to(dev).reshape(-1, rgb.shape[-1])[keep]
    # true division on the host: torch's CUDA div-by-scalar multiplies by the reciprocal (1 ulp off)
    return PointCloud(points=pts.cpu().numpy(), colors=col.cpu().numpy().astype(np.float64) / 255.0)


def remove_table_mask(points, colors, labels):
    keep = labels > 0
    return points[keep], colors[keep], labels[keep]
