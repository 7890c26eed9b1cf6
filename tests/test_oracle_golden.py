"""CPU: the oracle against the golden fixtures produced by the REAL reference (oracle/make_golden.py)."""
import os
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "oracle"))
import stego_oracle as O  # noqa: E402

GOLD = os.path.join(ROOT, "tests", "golden")


def _load(name):
    return torch.load(os.path.join(GOLD, name))


def _kat_inputs():
    torch.manual_seed(1234)
    return (torch.randn(2, 384, 28, 28), torch.randn(2, 384, 28, 28), torch.randn(2, 70, 28, 28),
            torch.randn(2, 70, 28, 28))


def test_kat_c0_known_answers():
    """SURVEY.md §4.3 known-answer values."""
    g = _load("corr_kat_c0.pt")
    feats, feats_pos, code, code_pos = _kat_inputs()
    code.requires_grad_(True)
    code_pos.requires_grad_(True)
    cfg = O.LossCfg()
    torch.manual_seed(99)
    c1, c2, perms = O.draw_loss_randomness(2, cfg)
    assert torch.equal(c1, g["coords1"]) and torch.equal(c2, g["coords2"]) and torch.equal(torch.stack(perms), g["perms"])
    out = O.correlation_loss(feats, feats_pos, code, code_pos, c1, c2, perms, cfg)
    total = .67 * out[0] + .25 * out[2] + .63 * out[4].mean()
    total.backward()
    assert abs(out[0].item() - 0.0001824702339945361) < 2e-8
    assert abs(out[2].item() - 0.005728472955524921) < 2e-8
    assert abs(out[4].mean().item() - 0.022114580497145653) < 2e-8
    assert abs(total.item() - 0.015486558899283409) < 2e-8
    assert torch.allclose(torch.stack([out[1].mean(), out[3].mean(), out[5].mean()]), g["cd_means"], atol=1e-8)
    assert abs(code.grad.norm().item() - 0.000311240553855896) < 1e-9
    assert abs(code_pos.grad.norm().item() - 2.0298446543165483e-05) < 1e-10
    assert torch.allclose(code.grad.reshape(-1)[::97], g["code_grad_sub"], atol=1e-10)
    assert torch.allclose(code_pos.grad.reshape(-1)[::97], g["code_pos_grad_sub"], atol=1e-11)
    assert torch.allclose(out[1].reshape(-1)[::211], g["intra_cd_sub"], atol=1e-6)
    assert torch.allclose(out[4].reshape(-1)[::211], g["neg_loss_sub"], atol=1e-6)
    assert out[1].shape == (2, 11, 11, 11, 11) and out[4].shape == (10, 11, 11, 11, 11)


def test_small_case_full_gradients():
    g = _load("corr_small.pt")
    cfg = O.LossCfg()
    code, code_pos = g["code"].clone().requires_grad_(True), g["code_pos"].clone().requires_grad_(True)
    out = O.correlation_loss(g["feats"], g["feats_pos"], code, code_pos, g["coords1"], g["coords2"], list(g["perms"]), cfg)
    total = O.weighted_correspondence_loss(out, cfg)
    total.backward()
    assert abs(total.item() - g["total"].item()) < 1e-6 * abs(g["total"].item()) + 1e-8
    assert torch.allclose(code.grad, g["code_grad"], rtol=1e-4, atol=1e-9)
    assert torch.allclose(code_pos.grad, g["code_pos_grad"], rtol=1e-4, atol=1e-9)
    assert torch.allclose(out[3].reshape(-1)[::53], g["inter_cd_sub"], atol=1e-6)


def test_cluster_lookup_kat():
    g = _load("cluster_lookup_kat.pt")
    torch.manual_seed(7)
    _ = torch.randn(27, 70)  # ClusterLookup.__init__ draws the centroids first
    x = torch.randn(2, 70, 28, 28)
    loss, probs = O.cluster_lookup(x, g["clusters"], None)
    assert abs(loss.item() - (-0.23893260955810547)) < 1e-7
    assert int(probs.argmax(1).sum()) == 20458
    assert torch.equal(probs.argmax(1).to(torch.int16), g["argmax"])
    lp = O.cluster_lookup(x, g["clusters"], 2.0, log_probs=True)
    assert abs(lp.sum().item() - g["log_probs_sum"].item()) < 0.5  # sum of 42k terms of magnitude ~3.3
    assert torch.allclose(lp.reshape(-1)[::101], g["log_probs_sub"], atol=1e-5)


def test_vit_tokens_golden():
    g = _load("vit_small8_32px.pt")
    sd = O.perturb_vit_state(O.vit_random_state("vit_small", 8, seed=3))
    torch.manual_seed(11)
    img = torch.randn(2, 3, 32, 32)
    with torch.no_grad():
        tok = O.vit_forward(sd, img, "vit_small", 8)
    assert tok.shape == g["tokens"].shape == (2, 17, 384)
    assert torch.allclose(tok, g["tokens"], atol=2e-5)


def test_super_perm_golden():
    g = _load("super_perm.pt")
    for size, want in zip((1, 2, 5, 16, 32), g["draws"]):
        torch.manual_seed(1000 + size)
        got = torch.stack([O.super_perm_from_randperm(torch.randperm(size, dtype=torch.long)) for _ in range(3)])
        assert torch.equal(got, want)
    assert O.super_perm_from_randperm(torch.tensor([0])).tolist() == [0]


def test_sample_semantics_probe():
    """SURVEY.md §4.3: 3x4 ramp, corner coords -> [0, 8, 3, 11] (grid permutation, x->width, y->height)."""
    t = torch.arange(12.).reshape(1, 1, 3, 4)
    coords = torch.tensor([[[[-1., -1.], [1., -1.]], [[-1., 1.], [1., 1.]]]])
    assert O.bilinear_sample(t, coords).reshape(-1).tolist() == [0., 8., 3., 11.]


def test_clamp_gradient_is_inclusive():
    x = torch.tensor([0.0, -1e-6, 1e-6], requires_grad=True)
    x.clamp(0.0).sum().backward()
    assert x.grad.tolist() == [1.0, 0.0, 1.0]


def test_oracle_matches_real_reference():
    """Every check of oracle/check_against_reference.py, against the reference's outputs stored (sampled) by
    make_golden.py: the same max|diff| bound on the stored elements, shape and norm of the whole tensor."""
    import check_against_reference as C
    gold = _load("reference_checks.pt")
    got = C.oracle_outputs()
    bad = []
    for k, tol in C.TOL.items():
        g, w = got[k], gold[k]
        assert tuple(g.shape) == w["shape"], k
        if tol is None:
            ok = torch.equal(g.reshape(-1).to(w["val"].dtype), w["val"])
        else:
            flat = g.reshape(-1)
            sub = flat[w["idx"].long()] if "idx" in w else flat
            scale = tol * max(w["absmax"], 1.0)
            ok = ((sub - w["val"]).abs().max().item() <= scale and
                  abs(flat.double().norm().item() - w["norm"]) <= scale * flat.numel() ** 0.5)
        if not ok:
            bad.append(k)
    assert not bad, bad


def test_knn_oracle_against_brute_force():
    """oracle.knn_descriptors / knn_indices (restating src/precompute_knns.py:19, 83-92) against an independent
    argsort of the full similarity matrix; row i must list itself first (cosine similarity 1)."""
    g = torch.Generator().manual_seed(5)
    fmap = torch.randn(97, 64, 4, 4, generator=g)
    d = O.knn_descriptors(fmap)
    assert torch.allclose(d.norm(dim=1), torch.ones(97), atol=1e-6)
    assert torch.allclose(d, torch.nn.functional.normalize(fmap.mean([2, 3]), dim=1))
    idx, val = O.knn_indices(d, 10, n_batches=16)
    sims = d @ d.t()
    order = torch.argsort(sims, dim=1, descending=True, stable=True)[:, :10]
    assert (idx[:, 0] == torch.arange(97)).all()
    assert torch.equal(idx, order)
    assert torch.allclose(val, sims.gather(1, order))


def test_crf_oracle_lattice_and_mean_field_sanity():
    """oracle/crf_oracle.py (parity UNPINNED: pydensecrf is absent): the permutohedral filter tracks exact Gaussian filtering
    (correlation > 0.99 in 2-D, > 0.85 in 5-D: the lattice is an approximation by construction), symmetric normalisation
    makes K 1 ~ 1-homogeneous, and mean-field on uniform unaries stays uniform."""
    import numpy as np
    import crf_oracle as CO
    rng = np.random.default_rng(0)
    for d, n, lo in ((2, 500, 0.99), (5, 400, 0.85)):
        f = (rng.random((d, n)) * 6).astype(np.float32)
        x = rng.random((n, 3)).astype(np.float32)
        a = CO.Permutohedral(f).compute(x)
        b = CO.brute_force_filter(f, x)
        assert np.corrcoef(a.ravel(), b.ravel())[0, 1] > lo
    k = CO.DenseKernel(CO.gaussian_features(12, 16, 1.0))
    U = np.full((12 * 16, 4), -np.log(0.25), np.float32)
    Q = CO.mean_field(U, [k], [3.0], 5)
    assert np.abs(Q - 0.25).max() < 1e-5
    # reverse blur order is the transpose of the filter: <K x, y> == <x, K^T y>
    lat = CO.Permutohedral((rng.random((3, 200)) * 4).astype(np.float32))
    x, y = rng.random((200, 1)).astype(np.float32), rng.random((200, 1)).astype(np.float32)
    assert abs((lat.compute(x) * y).sum() - (x * lat.compute(y, reverse=True)).sum()) < 1e-2 * abs((lat.compute(x) * y).sum())


def test_contrastive_crf_loss_golden():
    """oracle.contrastive_crf_loss against the reference's ContrastiveCRFLoss (modules.py:437-469) run by make_golden.py."""
    g = _load("contrastive_crf_loss.pt")
    torch.manual_seed(51)
    gd = torch.rand(2, 3, 56, 56) * 4 - 2
    cl = torch.nn.functional.normalize(torch.randn(2, 70, 56, 56), dim=1).requires_grad_(True)
    torch.manual_seed(52)
    coords = torch.cat([torch.randint(0, 56, size=[1, 300]), torch.randint(0, 56, size=[1, 300])], 0)
    out = O.contrastive_crf_loss(gd, cl, coords, .5, .15, .05, 10.0, 3.0, 0.00)
    grad, = torch.autograd.grad(out.mean(), cl)
    assert torch.allclose(out.detach().reshape(-1)[::97], g["out_sub"], atol=1e-6)
    assert abs(out.detach().abs().sum().item() - g["out_abs_sum"].item()) < 1e-5 * g["out_abs_sum"].item()
    assert torch.allclose(grad.reshape(-1)[::53], g["grad_sub"], atol=1e-9, rtol=1e-5)


def test_crf_oracle_against_exact_dense_mean_field():
    """Independent check of the CRF restatement's conventions (sign of the Potts message, symmetric normalisation, kernel
    weights, softmax update) that does not go through the lattice: exact O(N^2) Gaussian kernels on a 16 x 20 frame, the
    same 10 mean-field iterations.  The lattice only approximates the filter, so the marginals agree to ~1e-2 and the labels
    on >= 95 % of the pixels — on a problem where the CRF changes most of the unary labels."""
    import numpy as np
    import crf_oracle as CO
    rng = np.random.default_rng(1)
    H, W, C = 16, 20, 4
    base = rng.integers(0, 255, (2, 2, 3))
    img = np.clip(np.kron(base, np.ones((H // 2, W // 2, 1))) + rng.normal(0, 2.0, (H, W, 3)), 0, 255).astype(np.uint8)
    probs = rng.dirichlet(np.ones(C) * 0.7, H * W).T.reshape(C, H, W).astype(np.float32)
    U = CO.unary_from_softmax(probs).T.copy()
    feats = [CO.gaussian_features(H, W, 1.0), CO.bilateral_features(img, 8.0, 6.0)]
    weights = [3.0, 4.0]
    Q_lat = CO.mean_field(U, [CO.DenseKernel(f) for f in feats], weights, 10)

    def exact(f):
        f = f.T.astype(np.float64)
        K = np.exp(-0.5 * ((f[:, None] - f[None]) ** 2).sum(-1))
        n = 1.0 / np.sqrt(K.sum(1) + 1e-20)
        return n[:, None] * K * n[None, :]
    Ks = [exact(f) for f in feats]
    Q = CO.exp_and_normalize(-U).astype(np.float64)
    for _ in range(10):
        t = -U.astype(np.float64)
        for K, w in zip(Ks, weights):
            t = t + w * (K @ Q)
        e = np.exp(t - t.max(1, keepdims=True))
        Q = e / e.sum(1, keepdims=True)
    assert (Q.argmax(1) != (-U).argmax(1)).mean() > 0.3          # the CRF does something here
    assert (Q.argmax(1) == Q_lat.argmax(1)).mean() >= 0.95
    assert np.abs(Q - Q_lat).mean() < 0.02
