"""Parity of the path bench.py measures: `training_step` repeated on the same model — eager first step, CUDA-graph
capture on the second, graph replays afterwards, the parameter update overlapped on the side stream — against

  * the autograd-stitched path (cfg.fused_step=False) stepping a twin model with the same random draws, and
  * the oracle (oracle/stego_oracle.py) stepping its own copy of the trainable parameters with torch-Adam arithmetic,

after EVERY step: losses, all nine gradients, all nine parameters.  Batches alternate between two different inputs so
that a stale baked pointer, a missed memset or a value captured instead of re-read would show.

Then the same comparison at the BASELINE.json sizes (c1 ViT-S/8 224² B=32, c2 ViT-B/8 320² B=32, c3 ViT-B/8 448² B=16)
against the oracle run in fp32 ON THE GPU (TF32 off), twice: on the CUDA backbone's own features (isolates everything
after the backbone: asserted at the north-star 1e-3) and from the images through the oracle's fp32 ViT (image -> loss,
image -> gradient error, which includes the bf16-operand backbone error: reported and bounded).
"""
import pytest
import torch

from _parity_util import (NAMES, OracleStepper, feats_from_tokens, fp32_strict, grads_of, lr_of, make_batch, make_model,
                          oracle_vit_feats, params_of, peek_draws, record, rel)

pytestmark = pytest.mark.gpu


def _check_losses(model, loss, out, tol=1e-3):
    logged = {k: float(v) for k, v in model.logged.items()}
    elem_scale = 0.05  # typical |loss element|: the call means nearly cancel on random features
    assert abs(logged["loss/linear"] - out["linear"].item()) < 1e-4 * abs(out["linear"].item()) + 1e-6
    assert abs(logged["loss/cluster"] - out["cluster"].item()) < 2e-4 * abs(out["cluster"].item()) + 1e-6
    for k_log, k_or in [("loss/pos_intra", "pos_intra"), ("loss/pos_inter", "pos_inter"), ("loss/neg_inter", "neg_inter")]:
        assert abs(logged[k_log] - out[k_or].item()) < tol * abs(out[k_or].item()) + tol * elem_scale, (k_log, logged[k_log], out[k_or].item())
    assert abs(float(loss) - out["total"].item()) < tol * abs(out["total"].item())


@pytest.mark.parametrize("reset_at", [None, 2], ids=["plain", "reset_probe_steps=2"])
def test_multistep_graph_replay_vs_autograd_vs_oracle(cuda_dev, reset_at):
    """6 steps: eager, capture, 4 replays (reset_probe_steps fires inside the replayed regime)."""
    arch, res, B, nsteps = "vit_small", 64, 4, 6
    fused, _ = make_model(arch, cuda_dev, fused=True, reset_probe_steps=reset_at)
    twin, _ = make_model(arch, cuda_dev, fused=False, reset_probe_steps=reset_at)
    for k, v in params_of(fused).items():
        assert torch.equal(v, params_of(twin)[k])
    batches = [make_batch(B, res, cuda_dev, seed=1), make_batch(B, res, cuda_dev, seed=2)]
    orc = OracleStepper(params_of(fused), "cpu")
    h = res // 8
    torch.manual_seed(777)
    worst = dict(grad=0.0, param=0.0, twin_param=0.0)
    for s in range(nsteps):
        batch = batches[s % 2]
        draws = peek_draws(fused, B, cuda_dev)
        gpu_state, cpu_state = torch.cuda.get_rng_state(cuda_dev), torch.get_rng_state()
        p_before = params_of(fused)
        # the twin starts every step from the fused model's parameters and Adam moments: left on its own trajectory it
        # drifts from the fused one (Adam's update is sign-like for tiny gradients, and hidden activations at the ReLU /
        # clamp kinks land on either side), which after a few steps moves hidden-layer gradients by more than the bound
        with torch.no_grad():
            for buf in ("param", "exp_avg", "exp_avg_sq"):
                getattr(twin._flat, buf).copy_(getattr(fused._flat, buf))
        loss = fused.training_step(batch, s)
        g_f, p_f = grads_of(fused), params_of(fused)
        after_state = torch.cuda.get_rng_state(cuda_dev)
        # twin (autograd path): same generator states -> same draws, and it must leave the generators where the fused
        # path left them (RNG-stream parity with the reference's call order)
        torch.cuda.set_rng_state(gpu_state, cuda_dev)
        torch.set_rng_state(cpu_state)
        loss_t = twin.training_step(batch, s)
        g_t, p_t = grads_of(twin), params_of(twin)
        assert torch.equal(torch.cuda.get_rng_state(cuda_dev), after_state), f"step {s}: RNG consumption differs"
        assert fused._fused.step_idx == s + 1 and twin._fused is None
        if s >= 2:
            assert fused._fused.ws.graph is not None  # replay regime
        assert abs(float(loss) - float(loss_t)) < 2e-5 * abs(float(loss_t)), (s, float(loss), float(loss_t))
        for k in NAMES:
            # both paths run the same kernels; they differ in accumulation order (atomics) and both sit ~2e-4 from the
            # oracle on the hidden-layer weight gradient (bf16 dgrad operand), measured 3e-4 from each other
            worst["twin_grad"] = max(worst.get("twin_grad", 0.0), rel(g_f[k], g_t[k]))
            assert rel(g_f[k], g_t[k]) < 3e-3, (s, k, rel(g_f[k], g_t[k]))
            worst["twin_param"] = max(worst["twin_param"], rel(p_f[k], p_t[k]))
            assert rel(p_f[k], p_t[k]) < 2e-4, (s, k, rel(p_f[k], p_t[k]))
        # oracle on the same backbone features and the same draws
        with torch.no_grad():
            tok = fused.net.backbone_tokens(torch.cat([batch["img"], batch["img_pos"]], 0)).float().cpu()
        out = orc.losses(feats_from_tokens(tok, 2 * B, h, h), B, batch["label"].cpu(), draws)
        _check_losses(fused, loss, out)
        g_o = orc.grads()
        for k in NAMES:
            worst["grad"] = max(worst["grad"], rel(g_f[k], g_o[k]))
            assert rel(g_f[k], g_o[k]) < 1e-3, (s, k, rel(g_f[k], g_o[k]))
        # torch-Adam arithmetic (bias correction with the per-optimiser step count) on the gradients the kernels were
        # given: the update direction of Adam is sign-like for tiny gradients, so the oracle's own gradients (1e-3
        # away) cannot be used to check the update itself; this also keeps the oracle on the model's trajectory
        orc.adam(g_f)
        resetting = reset_at is not None and s == reset_at
        if resetting:
            for k in ("linear_probe.weight", "linear_probe.bias", "cluster_probe.clusters"):
                # the twin re-initialised with the same generator states: identical new values
                assert torch.equal(p_f[k], p_t[k]), k
                assert not torch.allclose(p_f[k], p_before[k]), k
                orc.adopt(k, p_f[k])
        for k in NAMES:
            # parameter DELTAS of this step (lr-sized)
            if resetting and not k.startswith("net."):
                continue
            d_f = p_f[k].cpu() - p_before[k].cpu()
            d_o = orc.p[k].detach() - p_before[k].cpu()
            worst["param"] = max(worst["param"], rel(d_f, d_o))
            assert rel(d_f, d_o) < 1e-4, (s, k, rel(d_f, d_o))
            assert rel(p_f[k], orc.p[k]) < 1e-5, (s, k)
    if reset_at is not None:
        assert fused.optimizers()[1].steps == nsteps - reset_at - 1 and fused.optimizers()[0].steps == nsteps
    record(f"multistep_{'reset' if reset_at is not None else 'plain'}", dict(steps=nsteps, worst=worst))


def test_flush_and_optimizer_state_dict(cuda_dev):
    """The overlapped update is visible after flush(); FusedAdam round-trips through torch.optim.Adam's layout."""
    model, _ = make_model("vit_small", cuda_dev, fused=True)
    batch = make_batch(2, 64, cuda_dev)
    p0 = params_of(model)
    for s in range(3):
        model.training_step(batch, s)
    sd = model.state_dict()  # flushes
    assert not torch.equal(sd["linear_probe.weight"], p0["linear_probe.weight"])
    opt = model.optimizers()[1]
    osd = opt.state_dict()
    ref = torch.optim.Adam(list(model.linear_probe.parameters()), lr=5e-3)
    ref.load_state_dict(osd)  # torch accepts the layout
    assert int(ref.state_dict()["state"][0]["step"]) == 3
    opt.reset_state()
    assert opt.steps == 0
    opt.load_state_dict(osd)
    assert opt.steps == 3 and rel(opt.state_dict()["state"][0]["exp_avg"], osd["state"][0]["exp_avg"]) == 0.0
    # set_to_none zero_grad must not break the raw-pointer step
    model.zero_grad(set_to_none=True)
    model.training_step(batch, 3)
    assert grads_of(model)["linear_probe.weight"].abs().sum() > 0


FULL = {"c1": ("vit_small", 224, 32), "c2": ("vit_base", 320, 32), "c3": ("vit_base", 448, 16)}


@pytest.mark.parametrize("cfg_name", ["c1", "c2", "c3"])
def test_fullsize_step_vs_gpu_fp32_oracle(cuda_dev, cfg_name):
    arch, res, B = FULL[cfg_name]
    fp32_strict()
    model, sd = make_model(arch, cuda_dev, fused=True)
    batches = [make_batch(B, res, cuda_dev, seed=1), make_batch(B, res, cuda_dev, seed=2)]
    orc = OracleStepper(params_of(model), "cuda")
    h = res // 8
    torch.manual_seed(777)
    nsteps = 3  # eager, capture, replay: the compared step is a graph replay
    for s in range(nsteps):
        batch = batches[s % 2]
        draws = peek_draws(model, B, cuda_dev)
        loss = model.training_step(batch, s)
        g = grads_of(model)
        if s < nsteps - 1:
            orc.adam(g)  # keep the oracle's parameters on the model's trajectory (exact: same gradients)
            for k in NAMES:
                assert rel(params_of(model)[k], orc.p[k]) < 1e-5
            continue
        imgs = torch.cat([batch["img"], batch["img_pos"]], 0)
        with torch.no_grad():
            tok = model.net.backbone_tokens(imgs).float()
        f_cuda = feats_from_tokens(tok, 2 * B, h, h)
        # (a) everything after the backbone, on identical features
        out = orc.losses(f_cuda, B, batch["label"], draws)
        _check_losses(model, loss, out)
        g_same = orc.grads()
        same = {k: rel(g[k], g_same[k]) for k in NAMES}
        for k in NAMES:
            assert same[k] < 1e-3, (k, same[k])
        # (b) image -> loss / gradient: the oracle's own fp32 ViT (GPU, TF32 off) instead of the CUDA backbone
        f_orc = oracle_vit_feats(sd, imgs, arch, "cuda", chunk=8 if res < 400 else 4)
        feat_err = rel(f_cuda, f_orc)
        assert feat_err < 1e-2, feat_err
        out_i = orc.losses(f_orc, B, batch["label"], draws, round_bf16=False)  # the all-fp32 reference step
        g_img = orc.grads()
        img = {k: rel(g[k], g_img[k]) for k in NAMES}
        loss_err = abs(float(loss) - out_i["total"].item()) / abs(out_i["total"].item())
        corr_err = abs(float(model.logged["loss/total"] - model.logged["loss/linear"] - model.logged["loss/cluster"])
                       - out_i["corr"].item()) / max(abs(out_i["corr"].item()), 1e-3)
        record(f"fullsize_{cfg_name}", dict(
            config=dict(arch=arch, res=res, batch=B, tokens=h * h + 1, compared_step=s, regime="cuda-graph replay"),
            oracle="oracle/stego_oracle.py on cuda, fp32, TF32 off",
            backbone_feature_rel_l2=feat_err, total_loss=float(loss), oracle_total_loss_from_images=out_i["total"].item(),
            image_to_loss_rel=loss_err, image_to_corr_loss_rel=corr_err,
            grad_rel_same_features=same, grad_rel_from_images=img))
        print(f"[{cfg_name}] backbone rel-L2 {feat_err:.2e}; image->loss {loss_err:.2e} (corr term {corr_err:.2e}); "
              f"grads same-features max {max(same.values()):.2e}, from images max {max(img.values()):.2e}")
        assert loss_err < 5e-3, loss_err
        for k in NAMES:
            assert img[k] < 0.2, (k, img[k])  # bf16-operand backbone vs fp32 backbone: reported above, bounded here
