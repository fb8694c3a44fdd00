"""Boundary evidence (SURVEY 8b): (i) every mirrored callable has the signature of the LIVE reference object
(`inspect.signature`, build container only); (ii) a reference caller - the grounding loop of
tools/validate_upper_bound.py:164-221 / engine/distil.py:430-460 - runs against the module names the reference
imports (`models.similarity`, `utils.misc`) after `dropclip_b200.install.install()`; (iii) the project_2d_features_to_3d
branches (center_crop / subsample_step / transform_coords, utils/projections.py:118-145) against outputs of the
unmodified reference; (iv) sparse_collate (data/dataset_blender.py:450-461)."""
import inspect
import json
import os
import sys
import types

import numpy as np
import pytest
import torch

from tests import golden_io as gio


def _params(fn):
    return [(n, p.default, p.kind) for n, p in inspect.signature(fn).parameters.items()]


def test_signatures_equal_the_reference_golden():
    """The live comparison below against the reference's signatures stored in tests/golden/reference_signatures.json
    (tests/make_golden_live.py): every mirrored callable, static or not, defaults included."""
    from tests.make_golden_live import our_modules, signatures
    want = json.load(open(os.path.join(gio.GOLDEN, "reference_signatures.json")))
    got = json.loads(json.dumps(signatures(*our_modules(), ours=True)))  # tuples -> lists, as stored
    assert sorted(got) == sorted(want)
    for key in want:
        assert got[key] == want[key], key
    import dropclip_b200.similarity as oms
    assert str(inspect.signature(oms.ClipSimilarity.__init__).parameters["device"].default) == "cuda"


@pytest.mark.needs_reference
def test_signatures_equal_the_live_reference():
    from oracle import ref_shim
    ff, pj, ms, tf = ref_shim.load()
    import utils.misc as misc
    import dropclip_b200.feature_fusion as off
    import dropclip_b200.metrics as om
    import dropclip_b200.projections as opj
    import dropclip_b200.similarity as oms
    import dropclip_b200.transforms as otf
    R, O = ff.MultiviewFeatureFusion, off.MultiviewFeatureFusion
    for name in ("__init__", "calculate_sim", "_cvt_o3d_coords", "get_visibility_mask", "reconstruct_per_obj_feat",
                 "aggregate_features", "fuse_points", "fuse_obj_prior", "fuse"):
        assert _params(getattr(O, name)) == _params(getattr(R, name)), name
        assert isinstance(inspect.getattr_static(O, name), type(inspect.getattr_static(R, name))), name  # staticmethod or not
    for name in ("depth_to_pointcloud", "pointcloud_to_pixel", "_cvt_regrad_coord", "_cvt_blender_coord", "apply_pca",
                 "project_2d_features_to_3d", "rgbd_to_pointcloud_o3d", "pool_multiview_features", "fuse_multiview_features",
                 "fuse_multiview_features_obj_prior"):
        got, want = _params(getattr(opj, name)), _params(getattr(pj, name))
        if name == "project_2d_features_to_3d":  # the default is the module's own function object
            got = [(n, getattr(d, "__name__", d), k) for n, d, k in got]
            want = [(n, getattr(d, "__name__", d), k) for n, d, k in want]
        assert got == want, name
    for name in ("transform_pointcloud_to_world_frame", "transform_pointcloud_to_camera_frame", "reconstruct_feature_map"):
        assert _params(getattr(otf, name)) == _params(getattr(tf, name)), name
    assert _params(otf.CoordTransform2d.__init__) == _params(tf.CoordTransform2d.__init__)
    RC, OC = ms.ClipSimilarity, oms.ClipSimilarity
    for name in ("compute_similarity", "predict"):
        assert _params(getattr(OC, name)) == _params(getattr(RC, name)), name
    ours, ref = _params(OC.__init__), _params(RC.__init__)
    assert [(n, k) for n, _, k in ours[:len(ref)]] == [(n, k) for n, _, k in ref]  # extra trailing keywords only (model=, tokenize=)
    assert [d for _, d, _ in ours[1:5]] == [d for _, d, _ in ref[1:5]]             # model_name, method, threshold, norm_vis_feat
    assert str(ours[5][1]) == "cuda" and all(d is None for _, d, _ in ours[len(ref):])
    assert (OC.NEGATIVE_PROMPT_GENERIC, OC.SOFTMAX_TEMP) == (RC.NEGATIVE_PROMPT_GENERIC, RC.SOFTMAX_TEMP)
    for name in ("trainMetricPC", "intersectionAndUnionGPU"):
        assert _params(getattr(om, name)) == _params(getattr(misc, name)), name


def test_sparse_collate_prepends_the_batch_index():
    """ME.utils.sparse_collate as data/dataset_blender.py:450-461 calls it: (sum M, 1 + 3) int32 coordinates with the
    sample index in column 0, features and labels concatenated in sample order."""
    from dropclip_b200.voxelize import sparse_collate
    rng = np.random.default_rng(3)
    coords = [torch.from_numpy(rng.integers(-50, 50, size=(m, 3)).astype(np.int32)) for m in (5, 0, 7)]
    feats = [torch.from_numpy(rng.standard_normal((c.shape[0], 6)).astype(np.float32)) for c in coords]
    labels = [torch.from_numpy(rng.integers(0, 9, size=c.shape[0]).astype(np.int32)) for c in coords]
    bc, bf, bl = sparse_collate(coords, feats, labels, dtype=torch.int32)
    assert bc.dtype == torch.int32 and bc.shape == (12, 4) and bf.shape == (12, 6) and bl.shape == (12,)
    assert bc[:, 0].tolist() == [0] * 5 + [2] * 7
    assert torch.equal(bc[:5, 1:], coords[0]) and torch.equal(bc[5:, 1:], coords[2])
    assert torch.equal(bf, torch.cat(feats)) and torch.equal(bl, torch.cat(labels))
    bc2, bf2 = sparse_collate([c.numpy() for c in coords], [f.numpy() for f in feats])
    assert torch.equal(bc2, bc) and torch.equal(bf2, bf)


@pytest.mark.gpu
def test_project_2d_features_to_3d_branches_vs_reference_golden():
    from dropclip_b200 import projections as opj
    from tests.make_golden_proj_branches import CASES, INTR, case_inputs
    g = gio.load("proj_branches.npz")
    cvt = {"regrad": opj._cvt_regrad_coord, "blender": opj._cvt_blender_coord, None: None}
    for name in CASES:
        depth, feats, ext, kw = case_inputs(name)
        kw["transform_coords"] = cvt[kw["transform_coords"]]
        if kw.get("transform_to_world"):
            kw["camera_extrinsics"] = ext
        pc, f = opj.project_2d_features_to_3d(depth.copy(), feats.copy(), INTR, **kw)
        want_pc, want_f = g[name + "_pc"], g[name + "_feat"]
        assert pc.shape == want_pc.shape and pc.dtype == want_pc.dtype, (name, pc.shape, pc.dtype, want_pc.shape, want_pc.dtype)
        assert np.array_equal(pc, want_pc), name                       # fp64 arithmetic in the reference's order: bit-exact
        assert f.shape == want_f.shape and np.array_equal(np.asarray(f), want_f), name


class _Args:
    sim_method, sim_norm_thresh, sim_negatives = "paired", 0.7, "scene"


@pytest.mark.gpu
@pytest.mark.parametrize("negatives_mode", ["scene", "generic"])
def test_validate_grounding_loop_runs_through_install(negatives_mode):
    """The body of validate_grounding (tools/validate_upper_bound.py:175-221): construct ClipSimilarity the way the
    reference does (positional defaults -> it loads `models.features.clip`), call predict(output.half(), query,
    negatives) per text query, score with trainMetricPC - all through the reference's module names after install()."""
    from dropclip_b200 import install
    from oracle import metrics_ref, ref_shim, similarity_ref
    saved = {k: sys.modules.get(k) for k in ("models", "models.features", "models.features.clip", "models.similarity",
                                             "utils", "utils.feature_fusion", "utils.projections")}
    tower = ref_shim.FakeTextTower(768, torch.float16)

    class _Model:
        def encode_text(self, tok):
            return tower.encode_text(tok).cuda()

        def eval(self):
            return self

        def to(self, *_):
            return self

    clip_mod = types.ModuleType("models.features.clip.clip")
    clip_mod.load = lambda name, device=None, jit=False: (_Model(), None)
    clip_mod.tokenize = ref_shim.fake_tokenize
    pkg = types.ModuleType("models.features.clip")
    pkg.clip = clip_mod
    try:
        for name in ("models", "models.features"):
            sys.modules[name] = types.ModuleType(name)
        sys.modules["models.features.clip"] = pkg
        sys.modules["models.features.clip.clip"] = clip_mod
        install.install()
        from models.similarity import ClipSimilarity  # the reference's import line (tools/validate_upper_bound.py:25)
        from dropclip_b200.metrics import trainMetricPC
        args = _Args()
        args.sim_negatives = negatives_mode
        CLIP = ClipSimilarity(device='cuda', method=args.sim_method, threshold=args.sim_norm_thresh)  # :175-176
        rng = np.random.default_rng(5)
        obj_queries = {f"a photo of object {i}": [i + 1] for i in range(6)}
        emb = tower.encode_text(ref_shim.fake_tokenize(list(obj_queries))).float()
        emb /= emb.norm(dim=-1, keepdim=True)
        n = 4000
        label = torch.from_numpy(rng.integers(0, 7, size=n))
        output = torch.zeros((n, 768))
        for i in range(6):
            output[label == i + 1] = emb[i]
        output += 0.03 * torch.from_numpy(rng.standard_normal((n, 768)).astype(np.float32))
        output_d, label_d = output.cuda(), label.cuda()
        pred_list, gt_list, want_pred, want_gt = [], [], [], []
        for text_query, obj_ids in obj_queries.items():                       # :200-218
            if args.sim_negatives == "generic":
                negatives = []
            elif args.sim_negatives == "scene":
                negatives = [x for x in list(obj_queries.keys()) if x != text_query]
            pred, sims_norm = CLIP.predict(output_d.half(), text_query, negatives)
            gt = torch.zeros_like(label_d, device=label_d.device)
            for obj in obj_ids:
                gt[label_d == obj] = True
            pred_list.append(pred)
            gt_list.append(gt)
            # the oracle on the CPU, same call shape (fp16 features, fp16 prompt rows from the tower)
            qp = tower.encode_text(ref_shim.fake_tokenize(text_query))
            qn = tower.encode_text(ref_shim.fake_tokenize(negatives if negatives else CLIP.NEGATIVE_PROMPT_GENERIC))
            wp, ws = similarity_ref.predict_from_embeds(output.half().float(), qp.float(), qn.float(), method="paired", threshold=0.7)
            np.testing.assert_allclose(sims_norm.cpu().numpy(), ws.numpy(), rtol=0, atol=6e-3)
            want_pred.append(wp)
            want_gt.append(gt.cpu())
        iou, (pr25, pr50, pr75) = trainMetricPC(pred_list, gt_list, pr_ious=[0.25, 0.5, 0.75], sigmoid=False)  # :220
        w_iou, (w25, w50, w75) = metrics_ref.train_metric_pc(want_pred, want_gt, pr_ious=[0.25, 0.5, 0.75], sigmoid=False)
        assert abs(float(iou) - float(w_iou)) < 2e-2 and float(iou) > 0.5
        assert (float(pr25), float(pr50)) == (float(w25), float(w50))
    finally:
        install.uninstall()
        for k, v in saved.items():
            if v is None:
                sys.modules.pop(k, None)
            else:
                sys.modules[k] = v
        sys.modules.pop("models.features.clip.clip", None)
