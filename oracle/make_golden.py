"""Generate tests/golden/*.pt from the REAL reference (its src directory named by $STEGO_REFERENCE_SRC).

    STEGO_REFERENCE_SRC=<reference checkout>/src python oracle/make_golden.py [--out DIR]
    STEGO_REFERENCE_SRC=<reference checkout>/src python oracle/make_golden.py --gpu [--out DIR]   (on a CUDA device)

The first form writes the CPU fixtures, the second reference_gpu.pt: the reference run in PyTorch eager (fp32) on the
GPU, whose random draws come from the CUDA generator and so cannot be made on the host.

The reference ships no tests or golden vectors (SURVEY.md §4.1), so these fixtures are outputs of the
reference's own code (imported through oracle/reference_shim.py) on seeded inputs.  Large inputs are NOT
stored: they are regenerated from the recorded seeds with the CPU generator (same torch build on the GPU
box), only outputs / sub-sampled outputs are stored, so the fixtures stay small.
"""
from __future__ import annotations

import argparse
import ast
import os
import sys
import tempfile
import textwrap
import types

import torch

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, HERE)
sys.path.insert(0, os.path.dirname(HERE))
import check_against_reference as C  # noqa: E402
import lightning_harness as H  # noqa: E402
import reference_shim  # noqa: E402
import stego_oracle as O  # noqa: E402

OUT = os.path.join(HERE, "..", "tests", "golden")


def sampled(t, k, seed=0):
    """`t` in full when it has at most k elements, else k elements at fixed random positions (`idx`); `absmax` and `norm`
    always describe the whole tensor."""
    t = t.detach()
    flat = t.reshape(-1)
    d = dict(shape=tuple(t.shape), absmax=flat.abs().max().double().item() if flat.is_floating_point() else None,
             norm=flat.double().norm().item() if flat.is_floating_point() else None)
    if flat.numel() <= k:
        d["val"] = flat.clone().cpu()
    else:
        idx = torch.randperm(flat.numel(), generator=torch.Generator().manual_seed(seed))[:k].sort().values.to(flat.device)
        d["idx"], d["val"] = idx.int().cpu(), flat[idx].clone().cpu()
    return d


def kat_inputs():
    """SURVEY.md §4.3 recipe (config c0 shapes)."""
    torch.manual_seed(1234)
    feats = torch.randn(2, 384, 28, 28)
    feats_pos = torch.randn(2, 384, 28, 28)
    code = torch.randn(2, 70, 28, 28)
    code_pos = torch.randn(2, 70, 28, 28)
    return feats, feats_pos, code, code_pos


def small_inputs():
    g = torch.Generator().manual_seed(4321)
    B, E, D, h = 3, 64, 70, 12
    basis_f, basis_c = torch.randn(8, E, generator=g), torch.randn(8, D, generator=g)
    z = torch.randn(B, 8, h, h, generator=g)
    zp = z + 0.3 * torch.randn(B, 8, h, h, generator=g)
    mk = lambda zz, bs, C: torch.einsum("bkhw,kc->bchw", zz, bs) + 0.1 * torch.randn(B, C, h, h, generator=g)
    return mk(z, basis_f, E), mk(zp, basis_f, E), mk(z, basis_c, D), mk(zp, basis_c, D)


def main(out_dir):
    ref, vits = reference_shim.import_reference()
    os.makedirs(out_dir, exist_ok=True)
    torch.set_num_threads(1)
    cfg = O.LossCfg()
    ns = types.SimpleNamespace(**cfg.__dict__)

    # ---- 1. KAT (§4.3): scalars, grad statistics, sub-sampled grads --------------------------------
    feats, feats_pos, code, code_pos = kat_inputs()
    code.requires_grad_(True)
    code_pos.requires_grad_(True)
    torch.manual_seed(99)
    o = ref.ContrastiveCorrelationLoss(ns)(feats, feats_pos, None, None, code, code_pos)
    loss = .67 * o[0] + .25 * o[2] + .63 * o[4].mean()
    loss.backward()
    torch.manual_seed(99)
    c1, c2, perms = O.draw_loss_randomness(2, cfg)
    torch.save(dict(
        recipe="manual_seed(1234); feats, feats_pos = randn(2,384,28,28) x2; code, code_pos = randn(2,70,28,28) x2; "
               "manual_seed(99); ContrastiveCorrelationLoss(shipped cfg)",
        pos_intra_loss=o[0].detach(), pos_inter_loss=o[2].detach(), neg_inter_loss_mean=o[4].mean().detach(),
        cd_means=torch.stack([o[1].mean(), o[3].mean(), o[5].mean()]).detach(), total=loss.detach(),
        code_grad_norm=code.grad.norm(), code_grad_sum=code.grad.sum(),
        code_pos_grad_norm=code_pos.grad.norm(), code_pos_grad_sum=code_pos.grad.sum(),
        code_grad_sub=code.grad.reshape(-1)[::97].clone(), code_pos_grad_sub=code_pos.grad.reshape(-1)[::97].clone(),
        intra_cd_sub=o[1].detach().reshape(-1)[::211].clone(), neg_loss_sub=o[4].detach().reshape(-1)[::211].clone(),
        coords1=c1, coords2=c2, perms=torch.stack(perms)), os.path.join(out_dir, "corr_kat_c0.pt"))

    # ---- 2. small correlated case with full inputs -------------------------------------------------
    f, fp, c, cp = small_inputs()
    c.requires_grad_(True)
    cp.requires_grad_(True)
    torch.manual_seed(5)
    o = ref.ContrastiveCorrelationLoss(ns)(f, fp, None, None, c, cp)
    loss = .67 * o[0] + .25 * o[2] + .63 * o[4].mean()
    loss.backward()
    torch.manual_seed(5)
    c1, c2, perms = O.draw_loss_randomness(3, cfg)
    torch.save(dict(feats=f, feats_pos=fp, code=c.detach(), code_pos=cp.detach(), coords1=c1, coords2=c2,
                    perms=torch.stack(perms), pos_intra_loss=o[0].detach(), pos_inter_loss=o[2].detach(),
                    neg_inter_loss_mean=o[4].mean().detach(), total=loss.detach(),
                    cd_means=torch.stack([o[1].mean(), o[3].mean(), o[5].mean()]).detach(),
                    inter_cd_sub=o[3].detach().reshape(-1)[::53].clone(), neg_loss_sub=o[4].detach().reshape(-1)[::53].clone(),
                    code_grad=c.grad.clone(), code_pos_grad=cp.grad.clone()), os.path.join(out_dir, "corr_small.pt"))

    # ---- 3. ClusterLookup KAT ----------------------------------------------------------------------
    torch.manual_seed(7)
    cl = ref.ClusterLookup(70, 27)
    x = torch.randn(2, 70, 28, 28)
    l, p = cl(x, None)
    lp = cl(x, 2.0, log_probs=True)
    torch.save(dict(recipe="manual_seed(7); ClusterLookup(70,27); x = randn(2,70,28,28)",
                    clusters=cl.clusters.detach().clone(), cluster_loss=l.detach(), argmax=p.argmax(1).to(torch.int16),
                    log_probs_sum=lp.sum().detach(), log_probs_sub=lp.detach().reshape(-1)[::101].clone()),
               os.path.join(out_dir, "cluster_lookup_kat.pt"))

    # ---- 4. ViT-S/8 tokens on a 32x32 image (pos-embed interpolation path) -------------------------
    sd = O.perturb_vit_state(O.vit_random_state("vit_small", 8, seed=3))
    model = vits.vit_small(patch_size=8, num_classes=0)
    model.load_state_dict(sd)
    model.eval()
    torch.manual_seed(11)
    img = torch.randn(2, 3, 32, 32)
    with torch.no_grad():
        feat, _, _ = model.get_intermediate_feat(img, n=1)
    torch.save(dict(recipe="sd = perturb_vit_state(vit_random_state('vit_small', 8, seed=3)); manual_seed(11); "
                           "img = randn(2,3,32,32); get_intermediate_feat(img)[0][0]",
                    tokens=feat[0].clone()), os.path.join(out_dir, "vit_small8_32px.pt"))

    # ---- 5. super_perm draws -----------------------------------------------------------------------
    rows = []
    for size in (1, 2, 5, 16, 32):
        torch.manual_seed(1000 + size)
        rows.append(torch.stack([ref.super_perm(size, torch.device("cpu")) for _ in range(3)]))
    torch.save(dict(recipe="for size in (1,2,5,16,32): manual_seed(1000+size); 3 x super_perm(size)",
                    draws=rows), os.path.join(out_dir, "super_perm.pt"))
    # ---- 6. ContrastiveCRFLoss (modules.py:437-469) at the training call's shapes (56 x 56, 70 channels), 300 samples
    torch.manual_seed(51)
    gd = torch.rand(2, 3, 56, 56) * 4 - 2
    cl = torch.nn.functional.normalize(torch.randn(2, 70, 56, 56), dim=1).requires_grad_(True)
    crf = ref.ContrastiveCRFLoss(300, .5, .15, .05, 10.0, 3.0, 0.00)
    torch.manual_seed(52)
    out = crf(gd, cl)
    g, = torch.autograd.grad(out.mean(), cl)
    torch.save(dict(recipe="manual_seed(51); guidance = rand(2,3,56,56)*4-2; clusters = normalize(randn(2,70,56,56), dim=1); "
                           "ContrastiveCRFLoss(300, .5, .15, .05, 10, 3, 0) under manual_seed(52) (coords = randint(56,[1,300]) x 2); "
                           "grad of out.mean()",
                    out_sub=out.detach().reshape(-1)[::97].clone(), out_mean=out.detach().mean(), out_abs_sum=out.detach().abs().sum(),
                    grad_sub=g.reshape(-1)[::53].clone(), grad_abs_sum=g.abs().sum()),
               os.path.join(out_dir, "contrastive_crf_loss.pt"))

    # ---- 7. every check of oracle/check_against_reference.py: the reference's side, sampled ---------------------------
    want = C.reference_outputs(ref, vits)
    torch.save({k: sampled(want[k].to(torch.int16) if k == "ClusterLookup.argmax" else want[k],
                                   1 << 30 if tol is None else 128) for k, tol in C.TOL.items()},
               os.path.join(out_dir, "reference_checks.pt"))

    # ---- 8. the reference's own LitUnsupervisedSegmenter.training_step (one step, CPU) --------------------------------
    B, res = 2, 64
    ts = H.load_reference_segmenter("reference")
    with tempfile.TemporaryDirectory() as td:
        ck = os.path.join(td, "dino.pth")
        H.write_random_dino_checkpoint(ck, "vit_small")
        from stego_b200.config import make_cfg
        torch.manual_seed(0)
        m = ts.LitUnsupervisedSegmenter(27, make_cfg(pretrained_weights=ck))
    H.load_trainable_state(m, H.trainable_state())
    m.train()
    batch = H.make_batch(B, res, "cpu")
    torch.manual_seed(777)
    loss = m.training_step(batch, 0).detach()
    params = dict(m.named_parameters())
    torch.save(dict(recipe="H.trainable_state() in the reference segmenter (random ViT checkpoint, seed 3); "
                           "H.make_batch(2, 64); manual_seed(777); training_step(batch, 0)",
                    loss=float(loss), logged={k: float(v) for k, v in m.logged.items()},
                    grad={k: sampled(params[k].grad, 512, i) for i, k in enumerate(H.trainable_state())},
                    param={k: sampled(params[k], 512, i) for i, k in enumerate(H.trainable_state())}),
               os.path.join(out_dir, "reference_training_step.pt"))

    # ---- 9. kNN: `get_feats` (src/precompute_knns.py:15-21) and the slab loop (:83-92), lifted as text and executed ---
    text = open(os.path.join(H.reference_src(), "precompute_knns.py")).read()
    tree = ast.parse(text)
    get_feats_src = next(ast.get_source_segment(text, n) for n in tree.body
                         if isinstance(n, ast.FunctionDef) and n.name == "get_feats")
    lines = text.splitlines()
    first = next(i for i, l in enumerate(lines) if "normed_feats = get_feats(par_model, loader)" in l)
    last = next(i for i, l in enumerate(lines) if "nearest_neighbors = torch.cat(all_nns, dim=0)" in l)
    loop_src = textwrap.dedent("\n".join(lines[first:last + 1]))
    feats_maps = knn_inputs()
    it = iter(feats_maps)
    env = dict(torch=torch, F=torch.nn.functional, tqdm=lambda x: x, n_batches=4)
    orig_cuda, orig_empty = torch.Tensor.cuda, torch.cuda.empty_cache
    torch.Tensor.cuda = lambda self, *a, **k: self  # get_feats moves the batch to the GPU; this runs on the host
    torch.cuda.empty_cache = lambda: None
    try:
        exec(get_feats_src, env)
        env["par_model"] = type("ParModel", (), {"forward": staticmethod(lambda img: next(it))})()
        env["loader"] = [dict(img=torch.zeros(8, 3, 4, 4)) for _ in feats_maps]
        exec(loop_src, env)
    finally:
        torch.Tensor.cuda, torch.cuda.empty_cache = orig_cuda, orig_empty
    torch.save(dict(recipe="knn_inputs(): 5 model outputs [8, 32, 5, 5]; n_batches = 4",
                    normed_feats=env["normed_feats"].clone(), nearest_neighbors=env["nearest_neighbors"].to(torch.int16)),
               os.path.join(out_dir, "reference_knn.pt"))
    for f_ in sorted(os.listdir(out_dir)):
        print(f_, os.path.getsize(os.path.join(out_dir, f_)))


def knn_inputs():
    g = torch.Generator().manual_seed(0)
    return [torch.randn(8, 32, 5, 5, generator=g) for _ in range(5)]  # "model outputs" of 5 loader batches: n = 40


def featurizer_inputs(dev):
    torch.manual_seed(6)
    return torch.randn(2, 3, 64, 96, device=dev)


def main_gpu(out_dir):
    """The reference on cuda:0 in PyTorch eager, fp32 (TF32 off)."""
    from stego_b200.config import make_cfg
    torch.backends.cuda.matmul.allow_tf32 = False
    torch.backends.cudnn.allow_tf32 = False
    torch.set_float32_matmul_precision("highest")
    dev = torch.device("cuda:0")
    ts = H.load_reference_segmenter("reference")
    out = {}
    with tempfile.TemporaryDirectory() as td:
        ck = os.path.join(td, "dino.pth")
        H.write_random_dino_checkpoint(ck, "vit_small")
        # DinoFeaturizer (src/modules.py:98-106): feat_type "KK" / "feat", and return_class_feat
        img = featurizer_inputs(dev)
        for feat_type in ("KK", "feat"):
            torch.manual_seed(0)
            ref = ts._modules.DinoFeaturizer(70, make_cfg(dino_feat_type=feat_type, pretrained_weights=ck)).to(dev).eval()
            H.load_trainable_state(ref, H.trainable_state(), prefix="net.")
            with torch.no_grad():
                rf, rc = ref(img)
                out[f"featurizer_{feat_type}"] = dict(feats=sampled(rf, 1024, 1), code=sampled(rc, 1024, 2))
                if feat_type == "feat":
                    out["featurizer_class_feat"] = sampled(ref(img, return_class_feat=True), 1024, 3)
        # two training steps of the reference's LitUnsupervisedSegmenter over its own modules.py
        B, res = 4, 64
        batch = H.make_batch(B, res, dev)
        torch.manual_seed(0)
        m = ts.LitUnsupervisedSegmenter(27, make_cfg(pretrained_weights=ck)).to(dev)
        H.load_trainable_state(m, H.trainable_state())
        m.train()
        torch.manual_seed(777)
        losses = []
        for s in range(2):
            losses.append(float(m.training_step(batch, s).detach()))
            m.global_step += 1
        params = dict(m.named_parameters())
        out["training_step"] = dict(
            recipe="H.trainable_state() in the reference segmenter (random ViT checkpoint, seed 3); H.make_batch(4, 64, "
                   "cuda); manual_seed(777); training_step x 2", losses=losses, logged={k: float(v) for k, v in m.logged.items()},
            grad={k: sampled(params[k].grad, 2048, i) for i, k in enumerate(H.trainable_state())})
    out["device"] = torch.cuda.get_device_name(dev)
    os.makedirs(out_dir, exist_ok=True)
    torch.save(out, os.path.join(out_dir, "reference_gpu.pt"))
    print("reference_gpu.pt", os.path.getsize(os.path.join(out_dir, "reference_gpu.pt")))


if __name__ == "__main__":
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=OUT)
    ap.add_argument("--gpu", action="store_true")
    a = ap.parse_args()
    main_gpu(a.out) if a.gpu else main(a.out)
