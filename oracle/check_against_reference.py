"""Pin the oracle: compare oracle/stego_oracle.py function-by-function with the REAL reference code.
Run:  STEGO_REFERENCE_SRC=<reference checkout>/src python oracle/check_against_reference.py

Exit status 0 iff every check passes.  `reference_outputs` computes the reference's side of every check and
`oracle_outputs` the oracle's side on the same seeded inputs; oracle/make_golden.py stores sampled reference outputs in
tests/golden/reference_checks.pt, against which tests/test_oracle_golden.py repeats the same checks without the reference.
"""
from __future__ import annotations

import os
import sys
import types

import torch

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import stego_oracle as O  # noqa: E402

CCL_CASES = [(True, True, False), (False, True, False), (True, False, True)]  # (pointwise, zero_clamp, stabalize)
VIT_CASES = [("vit_small", 224), ("vit_small", 96), ("vit_base", 64)]
CCL_NAMES = ["intra", "intra_cd", "inter", "inter_cd", "neg", "neg_cd"]


def _ccl_tag(pointwise, zero_clamp, stab):
    return f"loss[pw={pointwise},zc={zero_clamp},st={stab}]"


# check name -> max|diff| tolerance relative to max(max|reference|, 1); None = bit-exact
TOL = {"norm": 1e-6, "tensor_correlation": 1e-5, "sample": 1e-5, "sample(corners)": 1e-6,
       **{f"super_perm(size={s})": None for s in (1, 2, 5, 32)},
       **{f"{_ccl_tag(*c)}.{n}": 2e-6 for c in CCL_CASES for n in CCL_NAMES},
       **{f"{_ccl_tag(*c)}.{n}": 1e-5 for c in CCL_CASES for n in ("dcode", "dcode_pos")},
       "ClusterLookup.clusters": None, "ClusterLookup.loss": 1e-6, "ClusterLookup.argmax": None,
       "ClusterLookup.log_probs(alpha=2)": 1e-5, "ClusterLookup.softmax(alpha=3)": 1e-6,
       **{f"ViT {a}/8 @{r} tokens": 2e-5 for a, r in VIT_CASES},
       "head code (dropout masks replayed)": 1e-5, "head returned feats": 1e-6,
       "ContrastiveCRFLoss": 1e-6, "ContrastiveCRFLoss d/dclusters": 1e-6}


def _cfg_ns(cfg: O.LossCfg):
    return types.SimpleNamespace(**cfg.__dict__)


def _basic_inputs():
    torch.manual_seed(0)
    t = torch.randn(3, 20, 9, 13)
    coords = torch.rand(3, 5, 7, 2) * 2.4 - 1.2  # includes out-of-range coords (border clamp)
    a, b = torch.randn(2, 16, 5, 5), torch.randn(2, 16, 4, 6)
    corner = torch.tensor([[[[-1., -1.], [1., -1.]], [[-1., 1.], [1., 1.]]]]).repeat(3, 1, 1, 1)
    return t, coords, a, b, corner


def _ccl_inputs():
    torch.manual_seed(7)
    B, E, D, h = 3, 48, 70, 14
    feats, feats_pos = torch.randn(B, E, h, h), torch.randn(B, E, h, h)
    code = torch.randn(B, D, h, h, requires_grad=True)
    code_pos = torch.randn(B, D, h, h, requires_grad=True)
    return feats, feats_pos, code, code_pos


def _head_inputs():
    """modules.py:109-116 with plain torch layers on the oracle's head state (the layer constructors draw from the
    global generator before the features are drawn)."""
    torch.manual_seed(5)
    E, D, B, h = 384, 70, 2, 6
    hp = O.head_random_state(E, D, seed=4)
    c1 = torch.nn.Sequential(torch.nn.Conv2d(E, D, (1, 1)))
    c2 = torch.nn.Sequential(torch.nn.Conv2d(E, E, (1, 1)), torch.nn.ReLU(), torch.nn.Conv2d(E, D, (1, 1)))
    c1.load_state_dict({k[len("cluster1."):]: v for k, v in hp.items() if k.startswith("cluster1.")})
    c2.load_state_dict({k[len("cluster2."):]: v for k, v in hp.items() if k.startswith("cluster2.")})
    f = torch.randn(B, E, h, h)
    return hp, c1, c2, f


def _crf_inputs():
    torch.manual_seed(31)
    gd = torch.rand(2, 3, 20, 24)
    cl_ = torch.nn.functional.normalize(torch.randn(2, 70, 20, 24), dim=1).requires_grad_(True)
    return gd, cl_


def reference_outputs(ref, vits) -> dict:
    """The reference's side of every check in TOL (ref, vits: the reference's modules / vision_transformer)."""
    out = {}
    t, coords, a, b, corner = _basic_inputs()
    out["norm"] = ref.norm(t)
    out["tensor_correlation"] = ref.tensor_correlation(a, b)
    out["sample"] = ref.sample(t, coords)
    out["sample(corners)"] = ref.sample(t, corner)
    for size in (1, 2, 5, 32):
        torch.manual_seed(123 + size)
        out[f"super_perm(size={size})"] = torch.stack([ref.super_perm(size, torch.device("cpu")) for _ in range(4)])
    for pointwise, zero_clamp, stab in CCL_CASES:
        cfg = O.LossCfg(pointwise=pointwise, zero_clamp=zero_clamp, stabalize=stab)
        feats, feats_pos, code, code_pos = _ccl_inputs()
        torch.manual_seed(99)
        want = ref.ContrastiveCorrelationLoss(_cfg_ns(cfg))(feats, feats_pos, None, None, code, code_pos)
        gw = torch.autograd.grad(O.weighted_correspondence_loss(want, cfg), [code, code_pos])
        tag = _ccl_tag(pointwise, zero_clamp, stab)
        for name, v in zip(CCL_NAMES, want):
            out[f"{tag}.{name}"] = v
        out[f"{tag}.dcode"], out[f"{tag}.dcode_pos"] = gw
    torch.manual_seed(7)
    cl = ref.ClusterLookup(70, 27)
    x = torch.randn(2, 70, 28, 28)
    wl_, wp_ = cl(x, None)
    out["ClusterLookup.clusters"] = cl.clusters
    out["ClusterLookup.loss"] = wl_
    out["ClusterLookup.argmax"] = wp_.argmax(1)
    out["ClusterLookup.log_probs(alpha=2)"] = cl(x, 2.0, log_probs=True)
    out["ClusterLookup.softmax(alpha=3)"] = cl(x, 3.0)[1]
    for arch, res in VIT_CASES:
        sd = O.perturb_vit_state(O.vit_random_state(arch, 8, seed=3))
        model = vits.__dict__[arch](patch_size=8, num_classes=0)
        model.load_state_dict(sd, strict=True)
        model.eval()
        torch.manual_seed(11)
        img = torch.randn(1, 3, res, res)
        with torch.no_grad():
            feat, _, _ = model.get_intermediate_feat(img, n=1)
        out[f"ViT {arch}/8 @{res} tokens"] = feat[0]
    _, c1, c2, f = _head_inputs()
    drop = torch.nn.Dropout2d(p=.1)
    torch.manual_seed(21)
    code = c1(drop(f))  # modules.py:109
    code = code + c2(drop(f))  # modules.py:111
    out["head code (dropout masks replayed)"] = code
    out["head returned feats"] = drop(f)  # modules.py:116
    # ContrastiveCRFLoss (modules.py:437-469), train_config.yml:131-137 parameters; coords replayed from the seed
    crf = ref.ContrastiveCRFLoss(200, .5, .15, .05, 10.0, 3.0, 0.00)
    gd, cl_ = _crf_inputs()
    torch.manual_seed(32)
    want = crf(gd, cl_)
    out["ContrastiveCRFLoss"] = want
    out["ContrastiveCRFLoss d/dclusters"], = torch.autograd.grad(want.mean(), cl_)
    return {k: v.detach() for k, v in out.items()}


def oracle_outputs() -> dict:
    """The oracle's side of every check in TOL, on the inputs `reference_outputs` uses."""
    out = {}
    t, coords, a, b, corner = _basic_inputs()
    out["norm"] = O.l2_normalize(t)
    out["tensor_correlation"] = O.correlation(a, b)
    out["sample"] = O.bilinear_sample(t, coords)
    out["sample(corners)"] = O.bilinear_sample(t, corner)
    for size in (1, 2, 5, 32):
        torch.manual_seed(123 + size)
        out[f"super_perm(size={size})"] = torch.stack(
            [O.super_perm_from_randperm(torch.randperm(size, dtype=torch.long)) for _ in range(4)])
    for pointwise, zero_clamp, stab in CCL_CASES:
        cfg = O.LossCfg(pointwise=pointwise, zero_clamp=zero_clamp, stabalize=stab)
        feats, feats_pos, code, code_pos = _ccl_inputs()
        torch.manual_seed(99)
        c1, c2, perms = O.draw_loss_randomness(feats.shape[0], cfg)
        got = O.correlation_loss(feats, feats_pos, code, code_pos, c1, c2, perms, cfg)
        gg = torch.autograd.grad(O.weighted_correspondence_loss(got, cfg), [code, code_pos])
        tag = _ccl_tag(pointwise, zero_clamp, stab)
        for name, v in zip(CCL_NAMES, got):
            out[f"{tag}.{name}"] = v
        out[f"{tag}.dcode"], out[f"{tag}.dcode_pos"] = gg
    torch.manual_seed(7)
    clusters = torch.randn(27, 70)  # ClusterLookup.__init__ (modules.py:122)
    x = torch.randn(2, 70, 28, 28)
    gl_, gp_ = O.cluster_lookup(x, clusters, None)
    out["ClusterLookup.clusters"] = clusters
    out["ClusterLookup.loss"] = gl_
    out["ClusterLookup.argmax"] = gp_.argmax(1)
    out["ClusterLookup.log_probs(alpha=2)"] = O.cluster_lookup(x, clusters, 2.0, log_probs=True)
    out["ClusterLookup.softmax(alpha=3)"] = O.cluster_lookup(x, clusters, 3.0)[1]
    for arch, res in VIT_CASES:
        sd = O.perturb_vit_state(O.vit_random_state(arch, 8, seed=3))
        torch.manual_seed(11)
        img = torch.randn(1, 3, res, res)
        with torch.no_grad():
            out[f"ViT {arch}/8 @{res} tokens"] = O.vit_forward(sd, img, arch, 8)
    hp, _, _, f = _head_inputs()
    torch.manual_seed(21)
    masks = [O.draw_dropout2d_mask(f.shape[0], f.shape[1]) for _ in range(3)]
    got_feat, got_code = O.head_forward(f, hp, masks)
    out["head code (dropout masks replayed)"] = got_code
    out["head returned feats"] = got_feat
    gd, cl_ = _crf_inputs()
    torch.manual_seed(32)
    coords = torch.cat([torch.randint(0, 20, size=[1, 200]), torch.randint(0, 24, size=[1, 200])], 0)
    got = O.contrastive_crf_loss(gd, cl_, coords, .5, .15, .05, 10.0, 3.0, 0.00)
    out["ContrastiveCRFLoss"] = got
    out["ContrastiveCRFLoss d/dclusters"], = torch.autograd.grad(got.mean(), cl_)
    return {k: v.detach() for k, v in out.items()}


def close(got, want, tol, what) -> bool:
    """max|got - want| <= tol * max(max|want|, 1), or bit-exact when tol is None."""
    if tol is None:
        ok = torch.equal(got, want)
        print(f"  {'ok ' if ok else 'BAD'} {what} (bit-exact)")
        return ok
    err = (got - want).abs().max().item()
    scale = want.abs().max().item() + 1e-30
    ok = err <= tol * max(scale, 1.0)
    print(f"  {'ok ' if ok else 'BAD'} {what}: max|diff|={err:.3e} (scale {scale:.3e})")
    return ok


def run_checks() -> bool:
    import reference_shim
    ref, vits = reference_shim.import_reference()
    torch.set_num_threads(max(1, os.cpu_count() or 1))
    want = reference_outputs(ref, vits)
    got = oracle_outputs()
    ok = all([close(got[k], want[k], tol, k) for k, tol in TOL.items()])
    print("ORACLE PINNED AGAINST REFERENCE" if ok else "ORACLE MISMATCH")
    return ok


if __name__ == "__main__":
    sys.exit(0 if run_checks() else 1)
