"""Headline step on one stream (register-staged instance-histogram kernel) and on two streams (bulk-copy ring kernel
beside the visibility filter), alternated. Checks first that both histogram kernels return identical tables.

    python benchmarks/overlap_probe.py [scenes] [unique]
"""
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch

from dropclip_b200.engine import FusionEngine, batch_from_device
from dropclip_b200.scenes import make_scene

n_scenes = int(sys.argv[1]) if len(sys.argv) > 1 else 64
n_unique = int(sys.argv[2]) if len(sys.argv) > 2 else 16
dev = torch.device("cuda", 0)
eng = FusionEngine(dev)
uniq = [make_scene(1234 + i, n_views=73, n_points=100_000, n_objects=21, device="cuda:0", as_torch=True) for i in range(n_unique)]
batch = batch_from_device([uniq[i % n_unique] for i in range(n_scenes)], dev, seg_dtype=torch.int64)
torch.cuda.synchronize()

eng.overlap = False
ref = [t.clone() for t in eng.seg_tables(batch)]
eng.overlap = True
got = eng.seg_tables(batch)
torch.cuda.synchronize()
for name, a, b in zip(("counts", "outside", "row_object", "object_row", "status"), ref, got):
    assert torch.equal(a, b), f"ring histogram differs from the register-staged kernel: {name}"
print("ring == register-staged tables: ok")


def step():
    res = eng.fuse_object_level(batch, 0.05, False, True, "max", torch.uint8, join=False)
    comp = eng.compact_visibility(batch, res["any_visible"], res["records"], res["rank"], torch.uint8, host_sizes=False)
    res["join"]()
    return res, comp


base = None
for overlap in (False, True, False, True):
    eng.overlap = overlap
    keep = None
    for _ in range(3):
        keep = step()
    torch.cuda.synchronize()
    eng.profile = {}
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    import time
    h0 = time.perf_counter()
    for _ in range(10):
        keep = step()
    host_ms = (time.perf_counter() - h0) * 100
    b.record()
    torch.cuda.synchronize()
    prof = eng.profile_ms()
    eng.profile = None
    res, comp = keep
    sig = (res["fused"].double().nan_to_num().sum().item(), res["weight_obj"].double().sum().item(), comp[4].sum().item())
    if base is None:
        base = sig
    assert sig == base, (sig, base)
    print(f"overlap={overlap}: {a.elapsed_time(b) / 10:.3f} ms/step (host enqueue {host_ms:.2f} ms/step)  "
          + "  ".join(f"{k}={v:.3f}" for k, v in prof.items()), flush=True)
