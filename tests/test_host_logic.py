"""CPU-only tests: the C-ABI library loads and exports every declared symbol, host-side layout
logic, install aliasing, and the N>1 sharding/gather path on gloo with world_size 2."""
import os
import re
import subprocess
import sys
import time

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def header_symbols():
    text = open(os.path.join(ROOT, "include", "dropclip.h")).read()
    return sorted(set(re.findall(r"^DC_API\s+[\w\s\*]+?\b(dc_\w+)\s*\(", text, flags=re.M)))


def test_library_builds_loads_and_exports_every_declared_symbol():
    from dropclip_b200 import _lib, build
    lib_path = build.build()
    out = subprocess.run(["nm", "-D", "--defined-only", lib_path], capture_output=True, text=True, check=True).stdout
    exported = sorted(set(re.findall(r"\sT\s+(dc_\w+)", out)))
    declared = header_symbols()
    assert len(declared) >= 28
    assert exported == declared, (set(declared) ^ set(exported))
    assert sorted(_lib.SIGNATURES) == declared
    lib = _lib.load()
    assert lib.dc_abi_version() == 2
    assert lib.dc_last_error() is not None
    # pure host queries only: no compute call without a GPU
    assert lib.dc_view_score_ld(21) == 32 and lib.dc_view_score_ld(200) == 256
    assert lib.dc_compact_workspace(100000) > 0 and lib.dc_voxelize_workspace(10000) > 0


def test_library_targets_sm100a_with_tensor_core_and_tma_instructions():
    from dropclip_b200 import build
    sass = subprocess.run(["cuobjdump", "-sass", build.build()], capture_output=True, text=True, check=True).stdout
    assert "sm_100a" in sass
    for mnemonic in ("UTCHMMA", "UTMALDG", "LDTM"):
        assert mnemonic in sass, mnemonic
    # the instance-histogram ring kernel of the two-stream step streams its input with 1-D bulk copies onto mbarriers
    ring = sass[sass.index("seg_histogram_ring_kernel"):]
    ring = ring[:ring.index("Function :", 10)] if "Function :" in ring[10:] else ring
    assert "UBLKCP.S.G" in ring and "SYNCS.ARRIVE.TRANS64" in ring and "SYNCS.PHASECHK.TRANS64.TRYWAIT" in ring


_NO_GPU_SCRIPT = r"""
import sys
sys.path.insert(0, {root!r})
import numpy as np, pytest, torch
assert not torch.cuda.is_available()
from dropclip_b200.engine import FusionEngine
from dropclip_b200.feature_fusion import MultiviewFeatureFusion
with pytest.raises(RuntimeError):
    FusionEngine("cuda")
M = MultiviewFeatureFusion({{"fx": 1.0, "fy": 1.0, "cx": 0.0, "cy": 0.0}}, use_similarity=False, device="cpu")
with pytest.raises(RuntimeError):
    M.get_visibility_mask(np.zeros((3, 3)), [np.zeros((480, 640), np.float32)], [np.eye(4, dtype=np.float32)])
"""


def test_no_cpu_fallback_without_gpu():
    """Runs in a child process with every CUDA device hidden, so that it checks the same on a machine that has a GPU."""
    r = subprocess.run([sys.executable, "-c", _NO_GPU_SCRIPT.format(root=ROOT)], env=dict(os.environ, CUDA_VISIBLE_DEVICES=""),
                       capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stdout + r.stderr


def test_product_package_never_imports_the_oracle():
    pkg = os.path.join(ROOT, "drop-clip_b200")
    for fn in os.listdir(pkg):
        if fn.endswith(".py"):
            src = open(os.path.join(pkg, fn)).read()
            assert not re.search(r"^\s*(from|import)\s+oracle\b", src, flags=re.M), fn


def test_environment_reaches_only_the_known_switches():
    """Launch sequences and results follow from the arguments: the library's only environment read is the DC_SEG_MODE
    test seam, and the package reads DC_OVERLAP (INTEGRATION.md) and DC_PIXEL_PATH (the pixel path's A/B seam)."""
    csrc = os.path.join(ROOT, "drop-clip_b200", "csrc")
    reads = []
    for fn in sorted(os.listdir(csrc)):
        if ".cu" in fn:
            reads += re.findall(r"\bgetenv\s*\(\s*([^)]*)\)", open(os.path.join(csrc, fn)).read())
    assert reads == ['"DC_SEG_MODE"'], reads
    pkg = os.path.join(ROOT, "drop-clip_b200")
    names = set()
    for fn in os.listdir(pkg):
        if fn.endswith(".py"):
            src = open(os.path.join(pkg, fn)).read()
            names |= set(re.findall(r"\b(?:os\.environ(?:\.get)?\s*[\[(]|os\.getenv\s*\()\s*[\"'](\w+)[\"']", src))
    assert {n for n in names if n.startswith("DC_")} == {"DC_OVERLAP", "DC_PIXEL_PATH"}, names


def test_batch_offsets_layout():
    from dropclip_b200.engine import SceneBatch
    off = SceneBatch.offsets_for([5, 0, 7], [2, 3, 1], [4, 4, 2], [3, 3, 1, 1, 1, 2])
    assert off["point"].tolist() == [0, 5, 5, 12]
    assert off["view"].tolist() == [0, 2, 5, 6]
    assert off["mask"].tolist() == [0, 10, 10, 17]
    assert off["wobj"].tolist() == [0, 8, 20, 22]
    assert off["feat"].tolist() == [0, 3, 6, 7, 8, 9, 11]
    assert off["view_scene"].tolist() == [0, 0, 1, 1, 1, 2]


def test_install_aliases_reference_module_names():
    from dropclip_b200 import install
    saved = {k: sys.modules.get(k) for k in install.ALIASES}
    try:
        install.install(voxelizer=True)
        import importlib
        ff = importlib.import_module("utils.feature_fusion")
        ms = importlib.import_module("models.similarity")
        pj = importlib.import_module("utils.projections")
        assert ff.MultiviewFeatureFusion.__module__ == "dropclip_b200.feature_fusion"
        assert ms.ClipSimilarity.NEGATIVE_PROMPT_GENERIC == ["object", "thing", "texture", "stuff"]
        assert ms.ClipSimilarity.SOFTMAX_TEMP == 0.1
        assert hasattr(pj, "depth_to_pointcloud") and hasattr(pj, "pool_multiview_features")
        import MinkowskiEngine as ME
        assert callable(ME.utils.sparse_quantize) and callable(ME.utils.sparse_collate)
    finally:
        for k, v in saved.items():
            if v is None:
                sys.modules.pop(k, None)
            else:
                sys.modules[k] = v
        sys.modules.pop("MinkowskiEngine", None)
        sys.modules.pop("MinkowskiEngine.utils", None)


def test_reference_signatures_are_mirrored():
    import inspect
    from dropclip_b200.feature_fusion import MultiviewFeatureFusion as M
    from dropclip_b200.similarity import ClipSimilarity as C
    sig = inspect.signature(M.__init__)
    assert list(sig.parameters)[1:] == ["camera_intrinsic", "visibility_threshold", "image_size", "patch_size",
                                        "feature_size", "use_visibility", "use_similarity", "use_sim_kernel",
                                        "use_obj_prior", "norm_feat", "device"]
    assert sig.parameters["visibility_threshold"].default == 0.05 and sig.parameters["image_size"].default == (480, 640)
    assert list(inspect.signature(M.fuse_obj_prior).parameters)[1:] == [
        "points", "colors", "labels", "depths", "seg_masks", "camera_poses", "mv_features", "query_embeddings",
        "return_obj", "device"]
    assert list(inspect.signature(M.fuse_points).parameters)[1:] == [
        "points", "colors", "labels", "depths", "seg_masks", "camera_poses", "mv_features", "query_embeddings", "device"]
    assert list(inspect.signature(C.predict).parameters)[1:] == ["vis_feats", "qpos", "qneg", "norm_vis_feat", "method",
                                                                 "threshold"]
    assert list(inspect.signature(C.compute_similarity).parameters)[1:] == ["vis_feat_norm", "qpos", "qneg",
                                                                            "softmax_temp", "method"]


def test_shard_tables():
    from dropclip_b200 import shard
    assert shard.strided_shard(10, 1, 4) == [1, 5, 9]
    # tools/preprocess_data.py:711-716: chunk = ceil((110 - 100) / 3) = 4, inclusive ranges that share their boundary id
    assert shard.reference_chunks(100, 110, 3) == [(100, 104), (104, 108), (108, 110)]
    parts = [shard.contiguous_shard(100, 110, r, 3) for r in range(3)]
    assert sum(parts, []) == list(range(100, 111)) and [len(p) for p in parts] == [5, 4, 2]
    for r, (lo, hi) in enumerate(shard.reference_chunks(100, 110, 3)):  # each rank stays inside the reference's range
        assert set(parts[r]) <= set(range(lo, hi + 1))
    bal = shard.balanced_shard([9, 1, 1, 1, 8, 2, 2, 2], 2)
    assert sorted(sum(bal, [])) == list(range(8))
    loads = [sum([9, 1, 1, 1, 8, 2, 2, 2][i] for i in b) for b in bal]
    assert abs(loads[0] - loads[1]) <= 1


def test_scene_writer_restart_semantics(tmp_path):
    from dropclip_b200 import shard
    per_obj = np.random.default_rng(0).standard_normal((4, 8)).astype(np.float32)
    per_obj[0] = np.nan
    q = np.ones((4, 8), np.float32)
    p = shard.write_scene(str(tmp_path), 12, per_obj, q, np.zeros((5, 3)), np.zeros((5, 3)), np.arange(5), np.ones((2, 5)))
    z = shard.read_scene(p)
    assert np.array_equal(z["multiview/per_obj"][0], q[0]) and np.array_equal(z["multiview/per_obj"][1:], per_obj[1:])
    assert z["pointcloud/label"].dtype == np.uint8 and z["pointcloud/vis_mask"].dtype == np.float32
    assert z["multiview/obj_ids"].dtype == np.uint8 and z["pointcloud/xyz"].dtype == np.float32
    assert shard.pending_scenes(str(tmp_path), [11, 12, 13]) == [11, 13]
    # a file the REFERENCE wrote (tools/preprocess_data.py:191 names it {id}.h5py) is honoured by the restart check
    open(str(tmp_path / "000013.h5py"), "wb").close()
    assert shard.pending_scenes(str(tmp_path), [11, 12, 13]) == [11]


def _gloo_worker(rank, world, port, q):
    import torch.distributed as dist
    from dropclip_b200 import shard
    dist.init_process_group("gloo", init_method=f"tcp://127.0.0.1:{port}", rank=rank, world_size=world)
    try:
        n_scenes = 7
        mine = shard.strided_shard(n_scenes, rank, world)
        feats = [torch.full((3 + (i % 3), 16), float(i)) for i in mine]  # ragged Q per scene
        allf = shard.gather_object_features(mine, feats, q_max=5)
        assert sorted(allf) == list(range(n_scenes))
        for i, f in allf.items():
            assert f.shape == (3 + (i % 3), 16) and bool((f == float(i)).all())
        m = shard.reduce_metric_sums(torch.tensor([float(rank + 1), 2.0]))
        assert torch.allclose(m, torch.tensor([(1 + 2) / 2.0, 2.0]))
        assert shard.max_over_ranks(float(rank)) == float(world - 1)
        q.put((rank, "ok"))
    finally:
        dist.destroy_process_group()


def test_scene_parallel_gather_and_reduce_on_gloo_world2():
    import torch.multiprocessing as mp
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = 29500 + os.getpid() % 2000
    procs = [ctx.Process(target=_gloo_worker, args=(r, 2, port, q)) for r in range(2)]
    for p in procs:
        p.start()
    for p in procs:
        p.join(120)
        assert p.exitcode == 0
    assert sorted(q.get(timeout=5)[0] for _ in range(2)) == [0, 1]


def test_host_staging_helpers_copy_and_narrow():
    """dc_host_gather_copy / dc_host_gather_narrow_i64_u8 are pure host code: exercised without a GPU."""
    import ctypes
    import numpy as np
    from dropclip_b200 import _lib
    lib = _lib.load()
    rng = np.random.default_rng(3)
    for n_items, shape, threads in ((1, (7,), 1), (5, (33, 17), 4), (9, (480, 640), 16)):
        numel = int(np.prod(shape))
        arrs = [rng.random(shape, dtype=np.float32) for _ in range(n_items)]
        dst = np.empty((n_items,) + shape, dtype=np.float32)
        srcs = (ctypes.c_void_p * n_items)(*[a.ctypes.data for a in arrs])
        _lib.check(lib.dc_host_gather_copy(srcs, n_items, numel * 4, ctypes.c_void_p(dst.ctypes.data), threads))
        assert np.array_equal(dst, np.stack(arrs))
        segs = [rng.integers(0, 256, size=shape, dtype=np.int64) for _ in range(n_items)]
        out = np.empty((n_items,) + shape, dtype=np.uint8)
        bad = ctypes.c_int(7)
        srcs = (ctypes.c_void_p * n_items)(*[a.ctypes.data for a in segs])
        _lib.check(lib.dc_host_gather_narrow_i64_u8(srcs, n_items, numel, ctypes.c_void_p(out.ctypes.data), threads,
                                                    ctypes.byref(bad)))
        assert bad.value == 0 and np.array_equal(out, np.stack(segs).astype(np.uint8))
        for weird in (256, -1, 2 ** 40, -2 ** 62):
            segs[-1].reshape(-1)[numel // 2] = weird
            _lib.check(lib.dc_host_gather_narrow_i64_u8(srcs, n_items, numel, ctypes.c_void_p(out.ctypes.data), threads,
                                                        ctypes.byref(bad)))
            assert bad.value == 1
    assert lib.dc_host_gather_copy(None, 1, 4, None, 1) != 0  # null pointers are rejected, not dereferenced


@pytest.mark.parametrize("name", ["r01_bench_final.json", "r02_bench_final.json", "r02_bench_one_stream.json", "r02_bench_n2.json",
                                  "r02_bench_n4.json"])
def test_committed_bench_line_has_the_contract_keys(name):
    """profiles/rNN_bench_*.json are lines printed by bench.py on B200s; their shape is the driver's contract."""
    import json
    path = os.path.join(ROOT, "profiles", name)
    d = json.loads(open(path).read())
    if d["n_gpus"] > 1:
        d.setdefault("cpu_baseline", None)
        assert d["cpu_baseline"] is None  # rank 0 at N = 1 only
        d["cpu_baseline"] = {"value": 0, "unit": "", "cores": 0, "kind": "port", "sample": ""}
    if name.startswith("r02"):
        assert d["e2e"]["bound"]["kind"] == "pcie_h2d" and 0 < d["e2e"]["bound"]["frac_of_bound"] <= 1.05
        assert d["distinct_scene_job"]["scenes"] in (256, 1000) and d["resident_full_output"]["mask_dtype"] == "int64"
    for k in ("metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling", "vs_baseline",
              "dtype", "data", "config", "roofline", "cpu_baseline", "e2e", "gpu_launches", "clocks"):
        assert k in d, k
    assert d["metric"] == "fused_scenes_per_sec" and d["unit"] == "scenes/s" and d["scaling"] == "weak" and d["vs_baseline"] is None
    assert "workload" in d["config"] and "model" not in d["config"]
    r = d["roofline"]
    assert r["bound"] in ("hbm", "tensor") and abs(r["frac"] - r["achieved"] / r["peak"]) < 1e-9 and r["traffic"]
    assert {"value", "unit", "cores", "kind", "sample"} <= set(d["cpu_baseline"]) and d["cpu_baseline"]["kind"] in ("port", "reference")
    assert {"value", "unit", "h2d_bytes_per_step", "d2h_bytes_per_step"} <= set(d["e2e"]) and d["e2e"]["h2d_bytes_per_step"] > 0
    assert d["gpu_launches"] > 0 and {"sm_mhz", "sm_max_mhz", "reasons"} <= set(d["clocks"])
    if "one_stream" in r:  # two-stream step: the dominant kernel's live window lies inside the step, the step's bytes below the peak
        assert r["kernel"] == "seg_histogram" and r["kernels"]["seg_histogram"]["ms"] < d["ms_per_step"]
        assert 0 < r["whole_step"]["frac"] < 1 and r["one_stream"]["ms_per_step"] > d["ms_per_step"]


def test_host_staging_pool_survives_fork():
    """The staging helpers keep a persistent worker pool; a forked child (multiprocessing 'fork') has none of the
    parent's threads and must rebuild it instead of waiting for workers that do not exist."""
    import ctypes
    import numpy as np
    from dropclip_b200 import _lib
    lib = _lib.load()
    arrs = [np.full(5000, i, dtype=np.float32) for i in range(40)]
    srcs = (ctypes.c_void_p * 40)(*[a.ctypes.data for a in arrs])
    dst = np.empty((40, 5000), dtype=np.float32)
    assert lib.dc_host_gather_copy(srcs, 40, 20000, ctypes.c_void_p(dst.ctypes.data), 8) == 0
    pid = os.fork()
    if pid == 0:
        ok = 1
        try:
            out = np.empty((40, 5000), dtype=np.float32)
            rc = lib.dc_host_gather_copy(srcs, 40, 20000, ctypes.c_void_p(out.ctypes.data), 8)
            ok = 0 if (rc == 0 and np.array_equal(out, np.stack(arrs))) else 2
        finally:
            os._exit(ok)
    deadline = time.time() + 30
    while time.time() < deadline:
        done, status = os.waitpid(pid, os.WNOHANG)
        if done:
            assert os.WIFEXITED(status) and os.WEXITSTATUS(status) == 0
            break
        time.sleep(0.05)
    else:
        os.kill(pid, 9)
        raise AssertionError("forked child hung in the staging helper")
    assert np.array_equal(dst, np.stack(arrs))
