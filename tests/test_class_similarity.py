"""a18: `_get_similarity` + arg max of the reference's evaluation loops (engine/distil.py:244-246,289-290,
tools/validate_upper_bound.py:59-61,101-102) against outputs of the unmodified reference closure
(tests/golden/class_sim.npz, generator tests/make_golden_class_sim.py), and the prompt axis beyond one 256-column
GEMM block (models/similarity.py:47-61 has no prompt limit)."""
import numpy as np
import pytest
import torch

from tests import golden_io as gio
from tests.make_golden_class_sim import CASES, class_inputs


def _rows(m):
    return slice(None, None, max(1, m // 512))


@pytest.mark.parametrize("case", CASES)
def test_oracle_class_similarity_vs_reference_golden(case):
    from oracle import similarity_ref
    name, seed, m, k, c = case
    g = gio.load("class_sim.npz")
    x, table = class_inputs(seed, m, k, c)
    sims, pred = similarity_ref.class_similarity(x, table)
    np.testing.assert_allclose(sims[_rows(m)].numpy(), g[f"{name}_sims_rows"], rtol=1e-5, atol=1e-5)
    sure = g[f"{name}_margin"] > 1e-4
    assert np.array_equal(pred.numpy()[sure], g[f"{name}_pred"].astype(np.int64)[sure])
    np.testing.assert_allclose(table.numpy(), g[f"{name}_table_after"], rtol=1e-6)


@pytest.mark.gpu
@pytest.mark.parametrize("case", CASES)
def test_class_similarity_vs_reference_golden(case):
    from dropclip_b200.similarity import _get_similarity, class_similarity
    name, seed, m, k, c = case
    g = gio.load("class_sim.npz")
    x, table = class_inputs(seed, m, k, c)
    xd, td = x.cuda(), table.cuda()
    sims, pred = class_similarity(xd, td)
    assert sims.shape == (m, k) and sims.dtype == torch.float32 and pred.shape == (m,) and pred.dtype == torch.int64
    want = g[f"{name}_sims_rows"]
    got = sims[_rows(m)].cpu().numpy()
    assert np.abs(got - want).max() <= 1e-3 * np.abs(want).max(), np.abs(got - want).max()
    np.testing.assert_allclose(got, want, rtol=1e-3, atol=2e-5)
    sure = g[f"{name}_margin"] > 1e-4  # rows whose two best classes are closer than fp32 summation noise may flip
    assert sure.mean() > 0.99
    assert np.array_equal(pred.cpu().numpy()[sure], g[f"{name}_pred"].astype(np.int64)[sure])
    # arg max of OUR matrix is exactly what the epilogue kept (first index on ties)
    assert torch.equal(pred, torch.max(sims, 1)[1])
    np.testing.assert_allclose(td.cpu().numpy(), g[f"{name}_table_after"], rtol=2e-6)  # class table normalised in place
    # without the matrix: same arg max, nothing of size M x K written
    none, pred2 = class_similarity(xd, table.cuda(), return_sims=False)
    assert none is None and torch.equal(pred2, pred)
    assert torch.equal(_get_similarity(xd, table.cuda()), sims)


@pytest.mark.gpu
def test_class_similarity_empty_and_fp16_and_errors():
    from dropclip_b200.similarity import class_similarity
    t = torch.randn((44, 768), device="cuda")
    s, p = class_similarity(torch.empty((0, 768), device="cuda"), t.clone())
    assert s.shape == (0, 44) and p.shape == (0,) and p.dtype == torch.int64
    x = torch.randn((300, 768), device="cuda").half()
    s, p = class_similarity(x, t.clone().half())
    ref = x.float() @ (t / t.norm(dim=-1, keepdim=True)).half().float().T
    assert s.dtype == torch.float16 and (s.float() - ref).abs().max().item() < 3e-2
    with pytest.raises(RuntimeError):
        class_similarity(torch.randn((4, 512), device="cuda"), t)
    with pytest.raises(RuntimeError):
        class_similarity(torch.randn((4, 768)), t)


@pytest.mark.gpu
@pytest.mark.parametrize("n_prompts", [257, 1000])
def test_more_than_256_prompts(n_prompts):
    """use_kernel_neg == 'all' concatenates the whole class table (tools/preprocess_data.py:253-257); the reference has
    no prompt limit. The 256-column GEMM blocks combine their partial sums / maxima / arg max through the carry rows."""
    from oracle import ref_shim, similarity_ref
    from tests.test_gpu_parity import make_cs
    dim, n = 768, 3000
    rng = np.random.default_rng(31)
    prompts = [f"class {i}" for i in range(n_prompts)]
    tower = ref_shim.FakeTextTower(dim, torch.float32)
    emb = tower.encode_text(ref_shim.fake_tokenize(prompts))
    x = torch.from_numpy(rng.standard_normal((n, dim)).astype(np.float32))
    x[: n // 3] += 4.0 * emb[0] / emb[0].norm()
    x[n // 3: n // 2] += 4.0 * emb[n_prompts - 3] / emb[n_prompts - 3].norm()  # a strong negative in the LAST block
    cs = make_cs(dim, torch.float32)
    for method in ("paired", "argmax"):
        want_pred, want = similarity_ref.predict_from_embeds(x.clone(), emb[:1].clone(), emb[1:].clone(), method=method)
        xd = x.clone().cuda()
        pred, sims = cs.predict(xd, prompts[0], qneg=prompts[1:], method=method, threshold=0.7)
        np.testing.assert_allclose(sims.cpu().numpy(), want.numpy(), rtol=1e-3, atol=1e-5)
        if method == "paired":
            sure = (want - 0.7).abs() > 1e-3
            assert torch.equal(pred.cpu()[sure], want_pred[sure])
        else:
            assert (pred.cpu() != want_pred).float().mean().item() < 2e-3
    xn = x.clone().cuda()
    xn /= xn.norm(dim=-1, keepdim=True)
    raw = cs.compute_similarity(xn, prompts[0], prompts[1:], method="argmax")
    t = torch.cat([emb[:1], emb[1:]]).clone()
    t /= t.norm(dim=-1, keepdim=True)
    ref = xn.cpu() @ t.T
    assert raw.shape == (n, n_prompts) and (raw.cpu() - ref).abs().max().item() < 2e-5
    from dropclip_b200.similarity import class_similarity
    sims, idx = class_similarity(x.clone().cuda(), emb.clone().cuda())
    assert torch.equal(idx, torch.max(sims, 1)[1])
    rs = x @ t.T
    top2 = torch.topk(rs, 2, dim=1).values
    sure = (top2[:, 0] - top2[:, 1]) > 1e-4
    assert torch.equal(idx.cpu()[sure], rs.argmax(1)[sure])


@pytest.mark.gpu
@pytest.mark.parametrize("dim", [512, 768, 1024])
def test_ground_normalises_fp16_rows_in_place(dim):
    """predict() normalises fp16 features in place (models/similarity.py:77) in a pass before the GEMM, which walks the
    tiles last to first: every mode must leave the same normalised rows, torch's own fp16 result to an ulp, for full
    tiles, ragged tails and row counts below one tile."""
    from dropclip_b200 import _lib
    from dropclip_b200.engine import FusionEngine
    eng = FusionEngine("cuda")
    g = torch.Generator(device="cuda").manual_seed(dim)
    for n, p in ((1, 5), (31, 40), (127, 5), (128, 256), (129, 33), (1000, 256), (70_001, 200)):
        x0 = (torch.randn((n, dim), generator=g, device="cuda") * 3).half()
        t = torch.randn((p, dim), generator=g, device="cuda")
        t = (t / t.norm(dim=-1, keepdim=True)).half()
        ref = x0.float()
        ref = (ref / ref.norm(dim=-1, keepdim=True).half().float()).half()
        rows = []
        for mode in (_lib.DC_GROUND_PAIRED, _lib.DC_GROUND_ARGMAX, _lib.DC_GROUND_RAW):
            x = x0.clone()
            eng.ground(x, t, mode, 0.1, normalize=True)
            torch.cuda.synchronize()
            assert (x.float() - ref.float()).abs().max().item() <= 2e-3, (n, p, mode)
            rows.append(x)
        assert all(torch.equal(r.view(torch.int16), rows[0].view(torch.int16)) for r in rows[1:]), (n, p)


@pytest.mark.gpu
def test_fp16_row_normalisation_is_the_correctly_rounded_one():
    """In-place normalisation of fp16 features (models/similarity.py:77: `x /= x.norm(dim=-1, keepdim=True)`): the kernel's
    fp32 fast path with its exactness test and fp64 fall-back must give, for EVERY row, the correctly rounded fp16 norm and
    the fp16-rounded IEEE quotient - checked against an fp64 evaluation in torch, including rows whose norm sits next to an
    fp16 rounding boundary, zero rows, tiny and huge rows."""
    from dropclip_b200 import _lib
    from dropclip_b200.engine import FusionEngine
    eng = FusionEngine("cuda")
    g = torch.Generator(device="cuda").manual_seed(77)
    n, c = 120_000, 768
    x = (torch.randn((n, c), generator=g, device="cuda") * torch.rand((n, 1), generator=g, device="cuda") * 4).half()
    x[5] = 0
    x[6] = 6e-8     # subnormal fp16 entries
    x[7] = 2000.0   # norm overflows fp16 -> inf -> rows of zeros, like torch
    # rows engineered onto a rounding boundary of the norm: one large entry, the rest zero => norm = |entry| exactly
    x[8] = 0
    x[8, 3] = 1.0009765625
    d = x.double().pow(2).sum(-1, keepdim=True).sqrt()                     # fp64 error << fp16 spacing
    # correctly rounded fp16 of d. (d.half() goes through fp32 in torch - a double rounding that lands on the wrong
    # neighbour for ~1 row in 10^4 -, so the nearest of the three candidate fp16 values is picked in fp64.)
    h0 = d.float().half()
    bits = h0.view(torch.int16)
    cands = torch.stack([h0, (bits + 1).view(torch.float16), (bits - 1).clamp_min(0).view(torch.float16)], 0)
    pick = (cands.double() - d).abs().nan_to_num(nan=float("inf")).argmin(0, keepdim=True)
    want_nrm = torch.where(torch.isfinite(h0) & (h0 > 0), cands.gather(0, pick)[0], h0)
    want = (x.float() / want_nrm.float()).half()                            # IEEE fp32 division, rounded to fp16
    y = x.clone()
    t = torch.randn((4, c), generator=g, device="cuda").half()
    eng.ground(y, t, _lib.DC_GROUND_RAW, 0.1, normalize=True)
    torch.cuda.synchronize()
    same = (y.view(torch.int16) == want.view(torch.int16)) | (torch.isnan(y) & torch.isnan(want))
    assert bool(same.all()), f"{int((~same).any(-1).sum())} rows differ"
