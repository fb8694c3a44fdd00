"""Instance-histogram pass alone on the headline batch (int64 maps): the register-staged kernel the library takes in
one-stream mode against the bulk-copy ring kernel it takes in two-stream mode. Both must return identical tables."""
import os, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
from dropclip_b200.engine import FusionEngine, batch_from_device
from dropclip_b200.scenes import make_scene
dev = torch.device("cuda", 0)
eng = FusionEngine(dev)
uniq = [make_scene(1234 + i, n_views=73, n_points=1000, n_objects=21, device="cuda:0", as_torch=True) for i in range(16)]
batch = batch_from_device([uniq[i % 16] for i in range(64)], dev, seg_dtype=torch.int64)
gb = batch.segs.numel() * 8 / 1e9
tables = {}
for overlap, name in ((False, "register-staged"), (True, "ring")):
    eng.overlap = overlap
    for _ in range(3): got = eng.seg_tables(batch)
    torch.cuda.synchronize()
    tables[name] = [t.clone() for t in got]
    eng.profile = {}
    for _ in range(10): eng.seg_tables(batch)
    torch.cuda.synchronize()
    ms = eng.profile_ms()["seg_histogram"]
    eng.profile = None
    print(f"{name} (overlap={overlap}): {ms:.3f} ms  {gb / ms:.2f} TB/s", flush=True)
for field, a, b in zip(("counts", "outside", "row_object", "object_row", "status"), tables["register-staged"], tables["ring"]):
    assert torch.equal(a, b), f"ring histogram differs from the register-staged kernel: {field}"
print("tables equal: ok")
