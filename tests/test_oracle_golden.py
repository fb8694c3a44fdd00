"""Pins the oracle: every restatement under oracle/ must reproduce the vectors that the
unmodified reference produced (tests/make_golden.py), and - when /root/reference is present -
the reference itself on fresh inputs."""
import numpy as np
import pytest
import torch

from oracle import c_oracle, fusion_ref, projections_ref, ref_shim, similarity_ref
from tests import golden_io as gio

FUSE = ["fuse_s0.npz", "fuse_s1.npz", "fuse_s2.npz"]
FLAGS = {"sim_max": (0, 1, "max"), "sim_mean": (0, 1, "mean"), "vis": (1, 0, None), "none": (0, 0, None),
         "both": (1, 1, "max")}


@pytest.mark.parametrize("name", FUSE)
def test_numpy_visibility_matches_reference(name):
    z = gio.load(name)
    sc = gio.scene_of(z)
    K = fusion_ref.intrinsic_matrix(sc.intrinsic)
    H, W = sc.intrinsic["height"], sc.intrinsic["width"]
    got = fusion_ref.visibility_mask(sc.points, sc.depths, sc.camera_poses, K, H, W).numpy()
    assert np.array_equal(got, gio.unpack(z["vis"], sc.n_points))


@pytest.mark.parametrize("name", FUSE)
def test_c_visibility_matches_reference_bit_exact(name):
    z = gio.load(name)
    sc = gio.scene_of(z)
    K = fusion_ref.intrinsic_matrix(sc.intrinsic)
    got = c_oracle.visibility_mask(sc.points, sc.depths, None, K, inv_poses=sc.inv_poses)
    assert np.array_equal(got, gio.unpack(z["vis"], sc.n_points))
    adv = z["adv_points"]
    got = c_oracle.visibility_mask(adv, sc.depths, None, K, inv_poses=sc.inv_poses)
    assert np.array_equal(got, gio.unpack(z["adv_vis"], adv.shape[0]))


def test_c_projection_is_the_dgemm_fma_chain():
    """np.dot / @ on this numpy are k-ascending FMA chains; the C oracle must agree on every
    pixel coordinate and depth, not only on the final mask."""
    z = gio.load("fuse_s1.npz")
    sc = gio.scene_of(z)
    K = fusion_ref.intrinsic_matrix(sc.intrinsic)
    for v in range(sc.n_views):
        pix, zd = fusion_ref.project_to_pixels(sc.points, sc.camera_poses[v], K)
        _, cpix, czd = c_oracle.visibility_view(sc.points, sc.depths[v], np.linalg.inv(sc.camera_poses[v]), K,
                                                want_pixels=True)
        assert np.array_equal(pix, cpix)
        assert np.array_equal(zd.view(np.int64), czd.view(np.int64))


@pytest.mark.parametrize("name", FUSE)
@pytest.mark.parametrize("tag", list(FLAGS))
def test_object_level_fusion_matches_reference(name, tag):
    z = gio.load(name)
    sc = gio.scene_of(z)
    uv, us, kern = FLAGS[tag]
    K = fusion_ref.intrinsic_matrix(sc.intrinsic)
    H, W = sc.intrinsic["height"], sc.intrinsic["width"]
    (feat, w, vis), (p, c, l) = fusion_ref.fuse_object_level(
        sc.points, sc.colors, sc.labels, sc.depths, sc.seg_masks, sc.camera_poses, sc.mv_features,
        sc.query_embeddings, K, H, W, use_visibility=uv, use_similarity=us, sim_method=kern, return_obj=True)
    np.testing.assert_allclose(w.numpy(), z[f"obj_{tag}_weight"], rtol=1e-6, atol=0)
    np.testing.assert_allclose(feat.numpy(), z[f"obj_{tag}_feat"], rtol=1e-5, atol=1e-7, equal_nan=True)
    if tag == "sim_max":
        assert np.array_equal(p, z["kept_points"])
        assert np.array_equal(l, z["kept_labels"].astype(np.int64))
        assert np.array_equal(vis.numpy(), gio.unpack(z["kept_vis"], p.shape[0]))


@pytest.mark.parametrize("name", ["pixel_p0.npz", "pixel_p1.npz"])
def test_pixel_level_fusion_matches_reference(name):
    z = gio.load(name)
    sc = gio.scene_of(z, pixel=True)
    K = fusion_ref.intrinsic_matrix(sc.intrinsic)
    H, W = sc.intrinsic["height"], sc.intrinsic["width"]
    segs = [torch.from_numpy(s) for s in sc.seg_masks]
    for tag, (us, kern, nf) in {"sim_max_norm": (1, "max", True), "sim_mean_raw": (1, "mean", False),
                                "vis_norm": (0, None, True)}.items():
        feats = [f.clone() for f in sc.mv_features]
        (feat, vis, simw), (p, _, _) = fusion_ref.fuse_pixel_level(
            sc.points, sc.colors, sc.labels, sc.depths, segs, sc.camera_poses, feats, sc.query_embeddings, K, H, W,
            use_similarity=us, sim_method=kern, norm_feat=nf, feature_size=feats[0].shape[-1])
        assert p.shape[0] == int(z[f"pix_{tag}_npts"][0])
        assert np.array_equal(vis.numpy(), gio.unpack(z[f"pix_{tag}_vis"], p.shape[0]))
        np.testing.assert_allclose(feat.numpy(), z[f"pix_{tag}_feat"], rtol=1e-5, atol=1e-6, equal_nan=True)
        if simw is not None:
            np.testing.assert_allclose(simw.numpy(), z[f"pix_{tag}_simw"], rtol=1e-6, atol=1e-8)


def ground_inputs(name, seed, n, dim, nneg, dtype):
    rng = np.random.default_rng(seed)
    base = rng.standard_normal((n, dim)).astype(np.float32)
    prompts = [f"prompt {seed} {i}" for i in range(1 + nneg)]
    tower = ref_shim.FakeTextTower(dim, dtype)
    emb = tower.encode_text(ref_shim.fake_tokenize(prompts))
    pos = emb[0].float()
    feat = torch.from_numpy(base) * 0.05
    feat[: max(1, n // 3)] += pos / pos.norm() * 0.6
    return feat.to(dtype), emb, prompts, tower


GROUND = [("g0", 11, 3000, 768, 4), ("g1", 12, 2000, 512, 31), ("g2", 13, 1, 768, 4)]


def close(a, b, dname):
    """fp32 GEMM results move by an ulp with the BLAS thread count; fp16 ones by an fp16 ulp."""
    tol = dict(rtol=2e-5, atol=2e-6) if dname == "f32" else dict(rtol=0, atol=4e-3)
    np.testing.assert_allclose(np.atleast_1d(a), np.atleast_1d(b), **tol)


def same_pred(pred, sims, gold_pred, thr, dname):
    margin = 1e-4 if dname == "f32" else 1e-2
    sure = np.abs(np.atleast_1d(sims) - thr) > margin
    assert np.array_equal(np.atleast_1d(pred)[sure], gold_pred[sure])


@pytest.mark.parametrize("case", GROUND)
@pytest.mark.parametrize("dname", ["f32", "f16"])
def test_grounding_matches_reference(case, dname):
    name, seed, n, dim, nneg = case
    dtype = torch.float32 if dname == "f32" else torch.float16
    g = gio.load("ground.npz")
    feat, emb, prompts, tower = ground_inputs(name, seed, n, dim, nneg, dtype)
    for method in ("paired", "argmax"):
        if n == 1 and method == "argmax":
            with pytest.raises(IndexError):
                similarity_ref.predict_from_embeds(feat.clone(), emb[:1], emb[1:], method=method)
            continue
        pred, sims = similarity_ref.predict_from_embeds(feat.clone(), emb[:1], emb[1:], method=method)
        close(sims.numpy(), g[f"{name}_{dname}_{method}_sims"], dname)
        if method == "paired":
            same_pred(pred.numpy(), sims.numpy(), gio.unpack(g[f"{name}_{dname}_{method}_pred"], n).astype(bool), 0.7, dname)
    pred, sims = similarity_ref.predict_from_embeds(feat.clone(), emb[:1], None)
    close(sims.numpy(), g[f"{name}_{dname}_noneg_sims"], dname)
    generic = tower.encode_text(ref_shim.fake_tokenize(["object", "thing", "texture", "stuff"]))
    pred, sims = similarity_ref.predict_from_embeds(feat.clone(), emb[:1], generic, method="paired")
    close(sims.numpy(), g[f"{name}_{dname}_generic_sims"], dname)


def test_paired_closed_form_equals_softmax():
    # seeded (numpy stream: stable across machines); exp() of the two forms rounds differently, a few fp32 ulps apart
    raw = torch.from_numpy(np.random.default_rng(20260118).standard_normal((1000, 9)).astype(np.float32)) * 0.3
    a = similarity_ref.paired_softmax(raw)
    b = similarity_ref.paired_closed_form(raw)
    np.testing.assert_allclose(a.numpy(), b.numpy(), rtol=5e-6)


def test_c_transform_is_np_dot():
    """oracle_transform (visibility_ref.c) == np.dot(M, [p;1])[:3] on this host, for fp64 and promoted fp32 matrices, and ==
    the golden output of the unmodified transform_pointcloud_to_world_frame."""
    z = gio.load("proj.npz")
    np.testing.assert_array_equal(c_oracle.transform(z["regrad"], z["pose"]), z["world"])
    np.testing.assert_array_equal(c_oracle.transform(z["world"], np.linalg.inv(z["pose"])), z["cam"])
    rng = np.random.default_rng(0)
    pts = rng.uniform(-9, 9, size=(513, 3))
    M = rng.standard_normal((4, 4))
    for mat in (M, M.astype(np.float32)):
        want = np.dot(mat, np.vstack([pts.T, np.ones((1, pts.shape[0]))]))[:3, :].T
        np.testing.assert_array_equal(c_oracle.transform(pts, mat), want)


def test_projection_helpers_match_reference():
    z = gio.load("proj.npz")
    intr = gio.intr_of(z)
    np.testing.assert_array_equal(projections_ref.back_project(z["depth"], intr), z["backproj"])
    np.testing.assert_array_equal(projections_ref.pixels_of(z["regrad"], intr), z["pixels"])
    np.testing.assert_array_equal(projections_ref.to_world(z["regrad"], z["pose"]), z["world"])
    u, f = projections_ref.unique_max_pool(z["pool_in_pts"], z["pool_in_feat"])
    np.testing.assert_array_equal(u, z["pool_pts"])
    np.testing.assert_array_equal(f, z["pool_feat"])
    pm = projections_ref.nearest_patch_map(torch.from_numpy(z["patch_in"]), (60, 80, 3)).numpy()
    np.testing.assert_array_equal(pm, z["patch_map"])


def test_sparse_quantize_restatement_properties():
    """ME is absent (parity unpinned): check the published contract as properties."""
    rng = np.random.default_rng(3)
    xyz = (rng.uniform(-3, 3, size=(5000, 3))).astype(np.float32)
    lab = rng.integers(0, 5, size=5000).astype(np.int32)
    feat = rng.standard_normal((5000, 7)).astype(np.float32)
    coords, f, vl, um, im = projections_ref.sparse_quantize_ref(xyz, feat, lab, ignore_label=0, quantization_size=0.25)
    q = c_oracle.quantize(xyz, 0.25)
    assert np.array_equal(q, np.floor(xyz / np.float32(0.25)).astype(np.int32))
    assert np.array_equal(coords[im], q)
    assert np.array_equal(q[um], coords)
    assert len({tuple(c) for c in coords}) == coords.shape[0] == len({tuple(c) for c in q})
    assert np.all(np.diff(um) > 0)  # first-occurrence order
    assert np.array_equal(f, feat[um])
    for j in rng.integers(0, coords.shape[0], size=200):
        labs = np.unique(lab[im == j])
        assert vl[j] == (labs[0] if labs.size == 1 else 0)


def test_restatement_against_reference_golden():
    """The live comparison below against the reference's stored values (tests/golden/live_restatement.npz): masks and
    kept points bit for bit; features and weights to the fp32 GEMM's thread-count ulps, as in the other golden tests."""
    from tests.make_golden_live import SCENE, restatement_scene, scene_digest
    z = gio.load("live_restatement.npz")
    sc = restatement_scene()
    assert scene_digest(sc) == str(z["inputs_sha"]), "small_scene() no longer generates the stored inputs"
    H, W = SCENE["height"], SCENE["width"]
    K = fusion_ref.intrinsic_matrix(sc.intrinsic)
    (of, ow, ov), (op, _, _) = fusion_ref.fuse_object_level(
        sc.points, sc.colors, sc.labels, sc.depths, sc.seg_masks, sc.camera_poses, sc.mv_features,
        sc.query_embeddings, K, H, W, return_obj=True)
    assert op.shape[0] == int(z["n_kept"][0]) and np.array_equal(op, z["points"])
    assert np.array_equal(ov.numpy(), gio.unpack(z["vis"], op.shape[0]))
    np.testing.assert_allclose(ow.numpy(), z["weight"], rtol=1e-6, atol=0)
    np.testing.assert_allclose(of.numpy(), z["feat"], rtol=1e-5, atol=1e-7, equal_nan=True)
    cm = c_oracle.visibility_mask(sc.points, sc.depths, sc.camera_poses, K)
    assert np.array_equal(cm, gio.unpack(z["vis_full"], sc.n_points))


def test_c_visibility_with_fp64_poses_against_reference_golden():
    """The C oracle on fp64 poses and on their fp32 roundings against the reference's masks for the same inputs
    (tests/golden/live_fp64_poses.npz), bit for bit."""
    from tests.make_golden_live import fp64_pose_digest
    z = gio.load("live_fp64_poses.npz")
    sc, poses64, pts = gio.fp64_pose_case()
    assert fp64_pose_digest(sc, poses64, pts) == str(z["inputs_sha"]), "fp64_pose_case() no longer generates the stored inputs"
    poses32 = [p.astype(np.float32) for p in poses64]
    K = fusion_ref.intrinsic_matrix(sc.intrinsic)
    ref64, ref32 = gio.unpack(z["vis64"], pts.shape[0]), gio.unpack(z["vis32"], pts.shape[0])
    assert np.array_equal(c_oracle.visibility_mask(pts, sc.depths, poses64, K), ref64)
    assert np.array_equal(c_oracle.visibility_mask(pts, sc.depths, poses32, K), ref32)
    assert (ref64 != ref32).sum() > 100, "the case must distinguish fp64 poses from their fp32 roundings"


@pytest.mark.needs_reference
def test_restatement_against_live_reference():
    from dropclip_b200.scenes import small_scene
    ff, _, _, _ = ref_shim.load()
    sc = small_scene(777, n_views=3, n_points=1200, n_objects=5, height=96, width=128)
    H, W = 96, 128
    M = ff.MultiviewFeatureFusion(sc.intrinsic, image_size=(H, W), use_visibility=0, use_similarity=1,
                                  use_sim_kernel="max", use_obj_prior=1, norm_feat=False, device="cpu")
    (rf, rw, rv), (rp, _, _) = M.fuse(sc.points, sc.colors, sc.labels, sc.depths, sc.seg_masks, sc.camera_poses,
                                      sc.mv_features, sc.query_embeddings, return_obj=True, device="cpu")
    K = fusion_ref.intrinsic_matrix(sc.intrinsic)
    (of, ow, ov), (op, _, _) = fusion_ref.fuse_object_level(
        sc.points, sc.colors, sc.labels, sc.depths, sc.seg_masks, sc.camera_poses, sc.mv_features,
        sc.query_embeddings, K, H, W, return_obj=True)
    assert torch.equal(rv, ov) and np.array_equal(rp, op)
    assert torch.equal(rw, ow)
    np.testing.assert_array_equal(rf.numpy(), of.numpy())
    cm = c_oracle.visibility_mask(sc.points, sc.depths, sc.camera_poses, K)
    full = M.get_visibility_mask(sc.points, sc.depths, sc.camera_poses).numpy()
    assert np.array_equal(cm, full)


@pytest.mark.needs_reference
def test_c_visibility_with_fp64_poses_against_live_reference():
    """utils/transforms.py:54-58 inverts and multiplies in the pose's dtype: the C oracle fed the fp64 inverse must
    reproduce the unmodified reference on fp64 poses (and differ from the run on their fp32 roundings)."""
    ff, _, _, _ = ref_shim.load()
    sc, poses64, pts = gio.fp64_pose_case()
    poses32 = [p.astype(np.float32) for p in poses64]
    M = ff.MultiviewFeatureFusion(sc.intrinsic, image_size=(120, 160), use_similarity=False, device="cpu")
    K = fusion_ref.intrinsic_matrix(sc.intrinsic)
    ref64 = M.get_visibility_mask(pts, sc.depths, poses64).numpy()
    ref32 = M.get_visibility_mask(pts, sc.depths, poses32).numpy()
    assert np.array_equal(c_oracle.visibility_mask(pts, sc.depths, poses64, K), ref64)
    assert np.array_equal(c_oracle.visibility_mask(pts, sc.depths, poses32, K), ref32)
    assert (ref64 != ref32).sum() > 100, "the case must distinguish fp64 poses from their fp32 roundings"
