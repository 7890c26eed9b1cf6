"""CPU: pins the oracle's restatement of the training step (oracle/stego_oracle.py::training_losses, adam_step —
src/train_segmentation.py:112-245, 373-383) and of the kNN helpers against what the REFERENCE's own code computed on
the same seeded inputs: its LitUnsupervisedSegmenter.training_step executed unmodified through the stub-Lightning
harness (oracle/lightning_harness.py), and its precompute_knns.py statements, stored by oracle/make_golden.py under
tests/golden/."""
import os
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "oracle"))
GOLD = os.path.join(ROOT, "tests", "golden")


def _sub(t, s):
    """The elements of `t` that the stored sample `s` (make_golden.sampled) holds."""
    flat = t.reshape(-1)
    return flat[s["idx"].long()] if "idx" in s else flat


def test_oracle_training_step_matches_reference_training_step():
    import lightning_harness as H
    import stego_oracle as O
    gold = torch.load(os.path.join(GOLD, "reference_training_step.pt"))
    B, E = 2, 384
    sd = O.perturb_vit_state(O.vit_random_state("vit_small", 8, seed=3))  # the checkpoint the reference loaded
    p0 = H.trainable_state()
    batch = H.make_batch(B, 64, "cpu")
    # the draws the reference step made (Dropout2d x3 for net(img), x3 for net(img_pos), rand x2, randperm x5)
    torch.manual_seed(777)
    masks = [O.draw_dropout2d_mask(B, E) for _ in range(3)]
    masks_pos = [O.draw_dropout2d_mask(B, E) for _ in range(3)]
    c1, c2, perms = O.draw_loss_randomness(B, O.LossCfg())
    with torch.no_grad():
        f = O.vit_image_feat(sd, batch["img"], "vit_small", 8)
        fp = O.vit_image_feat(sd, batch["img_pos"], "vit_small", 8)
    hp = {k[len("net."):]: v.clone().requires_grad_(True) for k, v in p0.items() if k.startswith("net.")}
    probes = {k: v.clone().requires_grad_(True) for k, v in p0.items() if not k.startswith("net.")}
    out = O.training_losses(f, fp, hp, probes, batch["label"], masks, masks_pos, c1, c2, perms, O.LossCfg(), 27)
    out["total"].backward()
    assert abs(gold["loss"] - out["total"].item()) < 2e-6 * abs(out["total"].item())
    for k_log, k_or in [("loss/pos_intra", "pos_intra"), ("loss/pos_inter", "pos_inter"), ("loss/neg_inter", "neg_inter"),
                        ("loss/linear", "linear"), ("loss/cluster", "cluster"), ("cd/pos_intra", "cd_intra"),
                        ("cd/pos_inter", "cd_inter"), ("cd/neg_inter", "cd_neg")]:
        assert abs(gold["logged"][k_log] - out[k_or].item()) < 1e-5 * abs(out[k_or].item()) + 1e-7, k_log
    want_g = {("net." + k): v.grad for k, v in hp.items()}
    want_g.update({k: v.grad for k, v in probes.items()})
    for k in p0:
        gs, ps = gold["grad"][k], gold["param"][k]
        g, w = gs["val"], _sub(want_g[k], gs)
        assert (g - w).norm() <= 1e-4 * w.norm() + 1e-10, k
        assert abs(gs["norm"] - want_g[k].double().norm().item()) <= 1e-4 * want_g[k].norm().item() + 1e-10, k
        # the reference's torch.optim.Adam update vs the oracle's adam_step on the reference's gradient
        assert ("idx" in gs) == ("idx" in ps) and ("idx" not in gs or torch.equal(gs["idx"], ps["idx"]))
        p = _sub(p0[k], ps).clone()
        O.adam_step(p, g, torch.zeros_like(p), torch.zeros_like(p), 1, 5e-4 if k.startswith("net.") else 5e-3)
        assert (ps["val"] - p).abs().max().item() < 1e-7, k


def test_knn_oracle_matches_lifted_reference_lines():
    """The kNN restatement (oracle knn_descriptors / knn_indices) against the reference's own statements: `get_feats`
    (src/precompute_knns.py:15-21) and the slab loop (:83-92), lifted as TEXT from the reference file and executed by
    make_golden.py on the same 40 descriptors."""
    import make_golden
    import stego_oracle as O
    gold = torch.load(os.path.join(GOLD, "reference_knn.pt"))
    want_feats, want_nn = gold["normed_feats"], gold["nearest_neighbors"].long()
    desc = torch.cat([O.knn_descriptors(f) for f in make_golden.knn_inputs()], 0)
    assert torch.allclose(desc, want_feats, atol=1e-7)
    idx, _ = O.knn_indices(desc, k=30, n_batches=4)
    assert idx.shape == want_nn.shape == (40, 30)
    assert torch.equal(idx, want_nn)
