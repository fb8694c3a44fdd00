"""Drop-in for the metric reductions of `utils/misc.py` that follow the grounding kernel
(SURVEY.md §8f-2): `trainMetricPC` (utils/misc.py:21-50) and `intersectionAndUnionGPU`
(utils/misc.py:186-199, duplicate at :449-462).

Same signatures, return containers and in-place side effects as the reference; the counting runs in
libdropclip (`csrc/metrics.cu`) for all instances of a call in one launch, the handful of floating
point operations that follow are written like the reference. CUDA tensors only - there is no CPU path.
"""
from __future__ import annotations

from typing import List, Sequence

import torch

from . import _lib
from ._lib import check, current_stream, ptr

__all__ = ["trainMetricPC", "intersectionAndUnionGPU", "binary_iou_counts", "grounding_scores"]


def _require_cuda(t: torch.Tensor, what: str):
    if not t.is_cuda:
        raise RuntimeError(f"dropclip_b200.metrics.{what} needs CUDA tensors; there is no CPU fallback")


def binary_iou_counts(preds: Sequence[torch.Tensor], gts: Sequence[torch.Tensor], threshold: float, sigmoid: bool = False,
                      in_place: bool = True):
    """(inter, union) int64 tensors of shape (len(preds),): per-instance |pred & gt| and |pred | gt| after the
    reference's thresholding. With `in_place` and no sigmoid the callers' prediction tensors are binarised
    like `pred[pred < thr] = 0; pred[pred >= thr] = 1` does in the reference (utils/misc.py:36-37)."""
    lib = _lib.load()
    n = len(preds)
    dev = preds[0].device
    flat_p = [p.squeeze() if p.dim() else p for p in preds]
    sizes = [int(p.numel()) for p in flat_p]
    for p, g in zip(flat_p, gts):
        _require_cuda(p, "trainMetricPC")
        if g.numel() != p.numel():
            raise RuntimeError(f"The size of tensor a ({p.numel()}) must match the size of tensor b ({g.numel()})")
    pred = torch.cat([p.reshape(-1).to(torch.float32) for p in flat_p]) if n else torch.empty(0, device=dev)
    gt_dtype = gts[0].dtype
    if gt_dtype == torch.bool:
        gt = torch.cat([g.reshape(-1).view(torch.uint8) for g in gts])
    elif gt_dtype in (torch.uint8, torch.int32, torch.int64, torch.float32):
        gt = torch.cat([g.reshape(-1) for g in gts])
    else:
        gt = torch.cat([(g.reshape(-1) != 0).view(torch.uint8) for g in gts])
    off = torch.zeros(n + 1, dtype=torch.int64)
    off[1:] = torch.cumsum(torch.tensor(sizes, dtype=torch.int64), 0)
    off_dev = off.to(dev)
    inter = torch.empty(n, dtype=torch.int64, device=dev)
    union = torch.empty(n, dtype=torch.int64, device=dev)
    write_back = bool(in_place and not sigmoid)
    check(lib.dc_binary_iou_counts(ptr(pred), ptr(gt), _lib.torch_dtype_code(gt.dtype), ptr(off_dev), n, max(sizes, default=0),
                                   float(threshold), int(bool(sigmoid)), int(write_back), ptr(inter), ptr(union),
                                   current_stream()))
    if write_back:  # the reference binarises the tensors it was handed (squeeze() returns a view)
        o = off.tolist()
        for i, p in enumerate(preds):
            p.copy_(pred[o[i]:o[i + 1]].view(p.shape).to(p.dtype))
    return inter, union


@torch.no_grad()
def trainMetricPC(output, target, threshold=0.35, pr_ious=[0.25, 0.5, 0.75], sigmoid=False):
    assert len(output) == len(target)
    if len(output) == 0:
        return grounding_scores((), (), pr_ious)
    return grounding_scores(*binary_iou_counts(list(output), list(target), threshold, sigmoid), pr_ious)


@torch.no_grad()
def grounding_scores(inter, union, pr_ious=[0.25, 0.5, 0.75]):
    """trainMetricPC's mIoU and Pr@k (percent) from per-instance |pred & gt| and |pred | gt| counts, e.g. the
    (inter, union) of binary_iou_counts or of ClipSimilarity.predict_many_iou."""
    count = 1e-6 + len(inter)
    if len(inter) == 0:  # the reference's accumulators stay python floats
        return 100. * (0.0 / (count + 1e-6)), [100. * (0.0 / count) for _ in pr_ious]
    iou = inter / (union + 1e-6)  # int64 / fp32 -> fp32, as in the reference
    mean_iou = iou.sum()          # (the reference adds the instances one by one in fp32)
    mean_prec: List[torch.Tensor] = [(iou > pr_iou).float().sum() for pr_iou in pr_ious]
    mean_iou = mean_iou / (count + 1e-6)
    mean_prec = [prec / count for prec in mean_prec]
    return 100. * mean_iou, [100. * x for x in mean_prec]


def intersectionAndUnionGPU(output, target, K, ignore_index=255):
    # 'K' classes, output and target sizes are N or N * L or N * H * W, each value in range 0 to K - 1.
    assert (output.dim() in [1, 2, 3, 4])
    assert output.shape == target.shape
    _require_cuda(output, "intersectionAndUnionGPU")
    output = output.view(-1)  # raises for non-contiguous inputs exactly like the reference
    target = target.view(-1)
    lib = _lib.load()
    if output.dtype not in (torch.uint8, torch.int32, torch.int64) or target.dtype != output.dtype:
        # other dtypes: do the reference's in-place masking here, count on an int64 image
        output[target == ignore_index] = ignore_index
        out_k, tgt_k = output.to(torch.int64), target.to(torch.int64)
    else:
        out_k, tgt_k = output, target
    dev = output.device
    res = torch.empty((3, K), dtype=torch.float32, device=dev)
    ws_bytes = lib.dc_class_iou_workspace(int(K))
    ws = torch.empty(ws_bytes, dtype=torch.uint8, device=dev)
    check(lib.dc_class_iou_hist(ptr(out_k), ptr(tgt_k), _lib.torch_dtype_code(out_k.dtype), out_k.numel(), int(K),
                                int(ignore_index), ptr(res[0]), ptr(res[1]), ptr(res[2]), ptr(ws), ws_bytes,
                                current_stream()))
    return res[0], res[1], res[2]
