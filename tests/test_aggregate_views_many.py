"""geometry.aggregate_views_many: the host instance-map builder, the argument checks, and (GPU) every batched result
against the restatement in oracle/projections_ref.py and against single-scene calls."""
import ctypes

import numpy as np
import pytest
import torch

from oracle import projections_ref as pr


def _lib():
    from dropclip_b200 import _lib
    return _lib


def _masks_to_seg(views, out_dtype):
    """dc_host_masks_to_seg over a list of (masks, ids) views; returns (maps, out_of_range)."""
    L = _lib()
    lib = L.load()
    flat = [np.ascontiguousarray(m) for ms, _ in views for m in ms]
    ids = np.concatenate([np.asarray(i, dtype=np.int64) for _, i in views])
    mask_off = np.cumsum([0] + [len(ms) for ms, _ in views]).astype(np.int64)
    pixels = np.asarray([ms[0].size for ms, _ in views], dtype=np.int64)
    pix_off = np.cumsum([0] + list(pixels)).astype(np.int64)
    dst = np.zeros(max(int(pix_off[-1]), 1), dtype=np.uint8 if out_dtype == L.DC_U8 else np.int64)
    ptrs = (ctypes.c_void_p * len(flat))(*[m.ctypes.data for m in flat])
    bad = ctypes.c_int(0)
    L.check(lib.dc_host_masks_to_seg(ptrs, ids.ctypes.data, mask_off.ctypes.data, len(views), pixels.ctypes.data,
                                     pix_off.ctypes.data, out_dtype, dst.ctypes.data, 4, ctypes.byref(bad)))
    return [dst[pix_off[v]:pix_off[v + 1]] for v in range(len(views))], bad.value


@pytest.mark.parametrize("dtype", [np.bool_, np.uint8])
def test_host_masks_to_seg_vs_numpy(dtype):
    L = _lib()
    rng = np.random.default_rng(0)
    cases = []
    for k, (h, w) in zip((21, 1, 5, 3), ((48, 64), (7, 9), (33, 50), (10, 10))):
        ms = [(rng.random((h, w)) < 0.3).astype(dtype) for _ in range(k)]  # overlapping masks
        if dtype == np.uint8:
            ms[0][0, :5] = (0, 2, 17, 255, 1)  # non-binary uint8 values multiply like numpy
        cases.append((ms, rng.integers(0, 12, size=k)))
    full = [np.ones((6, 8), dtype=dtype) for _ in range(3)]  # full coverage: max(ids), no 0
    cases.append((full, np.asarray([-4, -2, -9])))
    got, bad = _masks_to_seg(cases, L.DC_I64)
    assert bad == 0
    for (ms, ids), g in zip(cases, got):
        want = pr.binary_masks_to_seg_ref(np.stack(ms), np.asarray(ids, dtype=np.int64))
        assert want.dtype == np.int64 and np.array_equal(g, want.reshape(-1))
    assert np.array_equal(got[-1], np.full(48, -2))
    # narrow output: fits only without the negative ids (and, for uint8 masks, without the 255 * id products)
    for case in cases[:-1]:
        want = pr.binary_masks_to_seg_ref(np.stack(case[0]), np.asarray(case[1], dtype=np.int64)).reshape(-1)
        small, bad = _masks_to_seg([case], L.DC_U8)
        assert bad == int(want.max() > 255)
        if not bad:
            assert np.array_equal(small[0], want)
    assert _masks_to_seg(cases[-1:], L.DC_U8)[1] == 1
    big = [(cases[1][0], np.asarray([300]))]  # ids > 255
    assert _masks_to_seg(big, L.DC_U8)[1] == 1
    g, bad = _masks_to_seg(big, L.DC_I64)
    assert bad == 0 and np.array_equal(g[0], pr.binary_masks_to_seg_ref(np.stack(big[0][0]), big[0][1]).reshape(-1))


def test_host_masks_to_seg_rejects_view_without_masks():
    L = _lib()
    lib = L.load()
    z = np.zeros(2, dtype=np.int64)
    dst = np.zeros(4, dtype=np.uint8)
    bad = ctypes.c_int(0)
    rc = lib.dc_host_masks_to_seg((ctypes.c_void_p * 1)(), z.ctypes.data, z.ctypes.data, 1, np.asarray([4]).ctypes.data,
                                  z.ctypes.data, L.DC_U8, dst.ctypes.data, 1, ctypes.byref(bad))
    assert rc == -1


def _scene(seed, n_views=3, h=30, w=40, n_obj=5, id_base=0, rgb_float=False, f32_pose=False, uint8_masks=False):
    rng = np.random.default_rng(seed)
    ids = list(range(id_base, id_base + n_obj))
    col_to_ins = {(i % 256, i // 256, 7): i for i in ids}
    views = {}
    for v in range(n_views):
        seg = rng.integers(0, n_obj, size=(h, w))
        annos = [(f"o{i}", (seg == k).astype(np.uint8 if uint8_masks else bool), (i % 256, i // 256, 7))
                 for k, i in enumerate(ids) if (seg == k).any()]
        depth = rng.uniform(0.5, 3.0, size=(h, w)).astype(np.float32)
        a = np.deg2rad(rng.uniform(0, 360))
        pose = np.eye(4)
        pose[:3, :3] = [[np.cos(a), -np.sin(a), 0], [np.sin(a), np.cos(a), 0], [0, 0, 1]]
        pose[:3, 3] = rng.uniform(-1, 1, 3)
        rgb = rng.integers(0, 256, size=(h, w, 3), dtype=np.uint8)
        views[v] = {"rgb": rgb.astype(np.float32) if rgb_float else rgb, "depth": depth, "annos": annos,
                    "camera": {"world_matrix": pose.astype(np.float32) if f32_pose else pose}}
    return {"col_to_ins": col_to_ins, "views": views}


INTR = {"fx": 35.0, "fy": 36.5, "cx": 19.5, "cy": 14.25, "height": 30, "width": 40}


def test_argument_checks_before_device_work(monkeypatch):
    from dropclip_b200 import geometry as geo
    L = _lib()
    called = []
    monkeypatch.setattr(geo, "_dev", lambda: called.append(1))
    sc = _scene(1)
    for bad in (0.0, -0.1, float("nan")):
        with pytest.raises(L.DropClipError):
            geo.aggregate_views_many([sc], INTR, 25.0, [None, bad])
    empty = _scene(2)
    empty["views"][1]["annos"] = []
    with pytest.raises(ValueError):
        geo.aggregate_views_many([sc, empty], INTR, 25.0, [None])
    with pytest.raises(ValueError):
        geo.aggregate_views_many([sc], INTR, float("nan"), [0.1])
    rgba = _scene(3)
    rgba["views"][0]["rgb"] = np.zeros((30, 40, 4), dtype=np.uint8)
    with pytest.raises(ValueError):
        geo.aggregate_views_many([rgba], INTR, 25.0, [None])
    # 2^31 sort elements: a zero-stride depth map of 2^29 pixels at 4 distinct sizes (no memory behind it)
    huge = _scene(4, n_views=1)
    v0 = huge["views"][0]
    v0["depth"] = np.broadcast_to(np.float32(1), (1 << 14, 1 << 15))
    v0["rgb"] = np.broadcast_to(np.uint8(0), (1 << 14, 1 << 15, 3))
    v0["annos"] = [("o", np.broadcast_to(True, (1 << 14, 1 << 15)), (0, 0, 7))]
    huge["col_to_ins"] = {(0, 0, 7): 0}
    with pytest.raises(ValueError, match="2\\^31"):
        geo.aggregate_views_many([huge], INTR, 25.0, [0.1, 0.2, 0.3, 0.4])
    assert not called


# ---------------------------------------------------------------------------------------------- GPU
@pytest.fixture(autouse=True)
def _release_cached_memory():
    """The full-size case caches several GB in torch's allocator; hand it back so that later tests in the session
    do not pay for freeing it (a cudaFree synchronises the device) inside their own calls."""
    yield
    if torch.cuda.is_available():
        torch.cuda.synchronize()
        torch.cuda.empty_cache()


def _check_vs_ref(scene, got, trunc, vs):
    wp, wc, wl = pr.aggregate_views_ref(scene, INTR, trunc, vs)
    p, c, l = got
    assert p.shape == wp.shape and c.shape == wc.shape and l.shape == wl.shape
    assert np.array_equal(l, wl)
    if vs is None:
        assert np.array_equal(c, wc) and np.allclose(p, wp, rtol=0, atol=1e-12)
    else:
        assert np.allclose(p, wp, rtol=0, atol=1e-11) and np.allclose(c, wc, rtol=0, atol=1e-12)


def _same(a, b):
    return all(x.dtype == y.dtype and x.shape == y.shape and np.array_equal(x, y, equal_nan=True) for x, y in zip(a, b))


@pytest.mark.gpu
@pytest.mark.parametrize("n_scenes,sizes", [(1, [None]), (1, [0.2]), (3, [None, 0.2, 0.2, 1.0]),
                                            (8, [0.5, None, 0.1, None, 0.5])])
def test_many_vs_reference_and_single_calls(n_scenes, sizes):
    from dropclip_b200 import geometry as geo
    scenes = [_scene(10 + s, n_views=1 + (s * 5) % 7) for s in range(n_scenes)]  # ragged view counts
    out = geo.aggregate_views_many(scenes, INTR, 25.0, sizes)
    assert len(out) == n_scenes and all(len(r) == len(sizes) for r in out)
    for s, sc in enumerate(scenes):
        for t, vs in enumerate(sizes):
            _check_vs_ref(sc, out[s][t], 25.0, vs)
            assert _same(out[s][t], geo.aggregate_views_blender_new(sc, INTR, 25.0, vs))
    if sizes.count(0.5) == 2:  # duplicates are equal but do not share memory
        a, b = out[0][0], out[0][4]
        assert _same(a, b) and not np.shares_memory(a[0], b[0])


@pytest.mark.gpu
def test_depth_quirks():
    from dropclip_b200 import geometry as geo
    sc = _scene(30, n_views=4)
    d = sc["views"][0]["depth"]
    d[0, :6] = (0.0, -1.0, np.nan, 25.0, 30.0, np.inf)  # 0 / negative labelled but not kept; NaN, >= trunc neither
    d[5, 5] = -0.0
    sc["views"][1]["depth"][:] = 0.0                     # a view with no kept pixel (all labelled)
    sc["views"][2]["depth"][:] = np.nan                  # a view with no valid pixel
    nothing = _scene(31, n_views=2)
    for v in nothing["views"].values():
        v["depth"][:] = 40.0                             # a scene with no kept pixel
    sizes = [None, 0.3, 0.05]
    out = geo.aggregate_views_many([sc, nothing], INTR, 25.0, sizes)
    for t, vs in enumerate(sizes):
        _check_vs_ref(sc, out[0][t], 25.0, vs)
        # no point: the restatement cannot take a min bound; the single-scene call returns empty arrays
        assert _same(out[1][t], geo.aggregate_views_blender_new(nothing, INTR, 25.0, vs))
    _check_vs_ref(nothing, out[1][0], 25.0, None)
    assert out[0][0][2].shape[0] > out[0][0][0].shape[0]  # labels outnumber points
    assert all(x.shape[0] == 0 for x in out[1][1])
    # trunc is compared in fp32, like the reference's fp32 depth against a Python float
    t = float(np.float32(1.3)) + 1e-9
    sc2 = _scene(32, n_views=2)
    sc2["views"][0]["depth"][:3, :3] = np.float32(1.3)
    r = geo.aggregate_views_many([sc2], INTR, t, [None, 0.2])[0]
    _check_vs_ref(sc2, r[0], t, None)
    _check_vs_ref(sc2, r[1], t, 0.2)


@pytest.mark.gpu
def test_variants_labels_poses_rgb():
    from dropclip_b200 import geometry as geo
    scenes = [_scene(40, rgb_float=True), _scene(41, f32_pose=True, id_base=300), _scene(42, uint8_masks=True),
              _scene(43, n_obj=40, n_views=2)]  # > 32 labels in a coarse voxel: the quadratic vote
    # full coverage: a pixel under every mask of its view takes max(ids) without the 0
    v = scenes[0]["views"][0]
    v["annos"] = v["annos"] + [("all", np.ones((30, 40), dtype=bool), (4, 0, 7))]
    # a mask type outside bool / uint8 goes through numpy
    v = scenes[2]["views"][1]
    v["annos"] = [(n, m.astype(np.int32), c) for n, m, c in v["annos"]]
    sizes = [None, 5.0, 0.1]
    out = geo.aggregate_views_many(scenes, INTR, 25.0, sizes)
    for s, sc in enumerate(scenes):
        for t, vs in enumerate(sizes):
            _check_vs_ref(sc, out[s][t], 25.0, vs)
            assert _same(out[s][t], geo.aggregate_views_blender_new(sc, INTR, 25.0, vs))
    assert out[1][0][2].max() >= 300
    assert len(np.unique(out[3][0][2])) > 32 and out[3][1][0].shape[0] <= 8


@pytest.mark.gpu
def test_full_size_scene():
    """480x640 at 73 views (22.4 M pixels), 21 objects."""
    from dropclip_b200 import geometry as geo
    sc = _scene(50, n_views=73, h=480, w=640, n_obj=21)
    intr = {"fx": 600.0, "fy": 600.0, "cx": 319.5, "cy": 239.5}
    sizes = [None, 0.02, 0.08]
    out = geo.aggregate_views_many([sc], intr, 25.0, sizes)[0]
    p, c, l = out[0]
    assert p.shape == (73 * 480 * 640, 3) and l.shape == (73 * 480 * 640,)
    wp, wc, wl = pr.aggregate_views_ref(sc, intr, 25.0, None)
    assert wp.shape == p.shape and np.allclose(p, wp, rtol=0, atol=1e-12) and np.array_equal(l, wl) and np.array_equal(c, wc)
    for t, vs in enumerate(sizes[1:], 1):
        got = out[t]
        assert got[0].shape[0] < p.shape[0] and _same(got, geo.aggregate_views_many([sc], intr, 25.0, [vs])[0][0])
        assert set(np.unique(got[2])) <= set(np.unique(l))
