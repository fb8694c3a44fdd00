"""`MultiviewFeatureFusion.fuse_many` at pixel level (use_obj_prior=0) against a loop of `fuse()` on the same arguments.

Every yielded element is compared with what `fuse()` returns: the visibility and the filtered rows exactly, the features
and similarity weights bit for bit (as int32 views, so that NaN rows compare equal) wherever the kernel sums in a fixed
order - the SIMT kernels (other widths, DC_PIXEL_PATH=simt). The tcgen05 path adds each pair's row to its point with
global float atomics and sums the norms and denominators the same way (csrc/pixel_fuse.cu), so two `fuse()` calls on the
same scene may already differ there by fp32 reordering; those two outputs are held to a reordering bound instead."""
import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

H, W = 96, 128
U = 2.0 ** -24  # fp32 unit roundoff


def _mvff(dim, us, kern, uv, nf):
    from dropclip_b200.feature_fusion import MultiviewFeatureFusion
    from dropclip_b200.scenes import scaled_intrinsic
    return MultiviewFeatureFusion(scaled_intrinsic(H, W), image_size=(H, W), feature_size=dim, use_visibility=uv,
                                  use_similarity=us, use_sim_kernel=kern, use_obj_prior=0, norm_feat=nf, device="cuda")


def _args(sc):
    return (sc.points, sc.colors, sc.labels, sc.depths, sc.seg_masks, sc.camera_poses, sc.mv_features, sc.query_embeddings)


def _scene(seed, v, n, dim, n_objects=6):
    from dropclip_b200.scenes import small_scene
    return small_scene(seed, n_views=v, n_points=n, n_objects=n_objects, height=H, width=W, feat_dim=dim,
                       feature_dtype=torch.float32, pixel_features=True, patch_hw=(6, 8))


def _sequence(dim):
    """Scenes of 1, 3 and 8 views, an empty cloud, a cloud no view sees, and every input container the drop-in takes."""
    a = _args(_scene(11, 3, 1500, dim))
    b = list(_args(_scene(12, 8, 2200, dim)))
    b[1] = (b[1] * 255).astype(np.uint8)  # uint8 colours
    b[2] = b[2].astype(np.int32)
    b[6] = [f.cuda() for f in b[6]]  # patch maps already on the device
    c = list(_args(_scene(13, 1, 900, dim)))
    c[2] = c[2].astype(np.uint8)
    c[4] = [s.astype(np.uint8) for s in c[4]]
    empty = list(_args(_scene(14, 3, 700, dim)))
    empty[0], empty[1], empty[2] = empty[0][:0], empty[1][:0], empty[2][:0]
    far = list(_args(_scene(15, 3, 800, dim)))
    far[0] = far[0] + 1000.0  # every point projects off-image or fails the depth test
    d = list(_args(_scene(16, 3, 1200, dim)))
    d[4] = [s.copy() for s in d[4]]
    d[4][1][:4, :4] = 300  # an id above 255: the maps travel as int64 (and the id binds no query)
    e = list(_args(_scene(17, 8, 1600, dim)))
    e[4] = [s.astype(np.int32) for s in e[4]]
    return [a, tuple(b), tuple(c), tuple(empty), tuple(far), tuple(d), tuple(e)]


def _reorder_bound(args, n_views, nf):
    """|got - want| allowed between two tcgen05 runs: fp32 sums of at most V terms in another order, each term at most the
    largest interpolated value (bicubic overshoot < 2x the largest tap) times its share of the weights, twice (the
    denominator is such a sum too), with the norms under norm_feat summed in another order as well."""
    m = 1.0 if nf else 2.0 * max(float(f.abs().max()) for f in args[6])
    return 16.0 * max(n_views, 1) * U * m


def _same(got, want, args, exact, nf):
    (f1, v1, w1), (p1, c1, l1) = want
    (f2, v2, w2), (p2, c2, l2) = got
    assert f2.is_cuda and v2.is_cuda and f2.dtype == f1.dtype == torch.float32 and tuple(f2.shape) == tuple(f1.shape)
    assert v2.dtype == torch.int64 and torch.equal(v1, v2)
    assert (w1 is None) == (w2 is None)
    if w1 is not None:
        assert w2.is_cuda and w2.dtype == torch.float32 and tuple(w2.shape) == tuple(w1.shape)
    for a, b, src in ((p1, p2, args[0]), (c1, c2, args[1]), (l1, l2, args[2])):
        assert type(a) is type(b) and a.dtype == b.dtype == src.dtype and a.shape == b.shape and np.array_equal(a, b)
    pairs = [(f1, f2, _reorder_bound(args, v1.shape[0], nf))] + ([(w1, w2, 16.0 * U)] if w1 is not None else [])
    for a, b, bound in pairs:
        if exact:
            assert torch.equal(a.view(torch.int32), b.view(torch.int32))
        else:
            assert torch.equal(a.isnan(), b.isnan())
            d = (a - b)[~a.isnan()].abs()
            assert d.numel() == 0 or float(d.max()) <= bound


FLAGS = [(1, "max", 1, True), (1, "mean", 0, False), (0, None, 1, True), (0, None, 0, False)]
PATHS = [(768, "mma"), (768, "simt"), (64, "mma")]  # tcgen05 / SIMT tile kernel / generic kernel (width 64)


@pytest.mark.parametrize("dim,path", PATHS)
@pytest.mark.parametrize("us,kern,uv,nf", FLAGS)
def test_fuse_many_equals_a_loop_of_fuse(dim, path, us, kern, uv, nf, monkeypatch):
    monkeypatch.setenv("DC_PIXEL_PATH", path)
    exact = path == "simt" or dim not in (512, 768, 1024)
    seq = _sequence(dim)
    M = _mvff(dim, us, kern, uv, nf)
    want = [M.fuse(*a, device="cuda") for a in seq]
    got = list(M.fuse_many(seq, return_obj=False, device="cuda"))
    assert len(got) == len(want) == len(seq)
    for a, g, w in zip(seq, got, want):
        _same(g, w, a, exact, nf)
    # the empty cloud and the cloud no view sees
    for i in (3, 4):
        (f, v, s), (p, c, l) = got[i]
        assert tuple(f.shape) == (0, dim) and tuple(v.shape) == (len(seq[i][3]), 0) and p.shape == (0, 3) and l.shape == (0,)
        assert (s is None) == (not us)


def test_fuse_many_on_a_generator_consumes_one_scene_ahead():
    seq = _sequence(768)[:3]
    M = _mvff(768, 1, "max", 1, True)
    want = [M.fuse(*a, device="cuda") for a in seq]
    handed = []

    def lazily():
        for i, a in enumerate(seq):
            handed.append(i)
            yield a

    out = M.fuse_many(lazily(), device="cuda")
    for i, (a, w) in enumerate(zip(seq, want)):
        g = next(out)
        assert handed == list(range(min(i + 2, len(seq))))  # scene i + 1 is staged while scene i is finished
        _same(g, w, a, False, True)
    with pytest.raises(StopIteration):
        next(out)


@pytest.mark.parametrize("where", ["staging", "finishing"])
def test_a_failing_scene_raises_after_the_earlier_scenes_were_yielded(where):
    seq = _sequence(768)[:3]
    bad = list(seq[1])
    if where == "staging":
        bad[6] = [f[..., :64].contiguous() for f in bad[6]]  # wrong channel count: the upload's check fails
    else:
        bad[1] = bad[1][:5]  # colours that do not match the cloud: the host filter fails
    seq = [seq[0], tuple(bad), seq[2]]
    M = _mvff(768, 1, "max", 1, True)
    with pytest.raises(Exception) as single:
        M.fuse(*seq[1], device="cuda")
    first = M.fuse(*seq[0], device="cuda")
    out = M.fuse_many(seq, device="cuda")
    _same(next(out), first, seq[0], False, True)
    with pytest.raises(type(single.value)):
        next(out)


def test_empty_iterable_and_the_side_stream_is_kept_between_calls():
    M = _mvff(768, 1, "max", 1, True)
    assert list(M.fuse_many([], device="cuda")) == []
    seq = _sequence(768)[:2]
    list(M.fuse_many(seq, device="cuda"))
    stream, stagings = M._many_stream, M._many_stagings
    again = list(M.fuse_many(seq, device="cuda"))
    assert M._many_stream is stream and M._many_stagings is stagings and len(again) == 2
