#!/usr/bin/env python
"""bench.py — STEGO correspondence-distillation training step on B200 (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--config c1|c2|c3|c4] [--impl ours|reference|torch-eager]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 ... bench.py --gpus N ...

A "step" is one full training step of the hot path on one synthetic batch per GPU: 2x frozen DINO ViT
forward, seg head fwd/bwd, correspondence loss fwd/bwd (self + KNN + 5 random negatives), linear + cluster
probes fwd/bwd, one gradient all-reduce (N > 1), three fused Adam updates.  Nothing is skipped or cached.

One JSON line on rank 0:
  value      images/s, whole job, inputs already resident in HBM (device timed, CUDA events, max over ranks)
  e2e        same metric through the public API with pinned-host inputs copied H2D and the loss read back
             D2H inside the timed region, every step
  roofline   the dominant kernel of the step, timed live with CUDA events; achieved = algorithmic FLOPs/launch
             / measured duration; peak from MEASURED_PEAKS.json (burst figure: kernel timed alone)
  corr_roofline  the named correlation+loss kernel against BOTH the bf16 tensor peak and the HBM peak
  cpu_baseline   the oracle port (CPU restatement of the reference, oracle/stego_oracle.py) on the host cores,
                 bounded sample
  sustained      the same device-resident loop run for >= 5 s with its own clock record
`--impl reference` times the reference's CPU path alone (rank 0 only; the REAL reference classes from baseline/_ref
through oracle/lightning_harness.py when that copy is present — `cpu_baseline.kind` "reference" — else the oracle port)
and prints the same line shape.  `--impl torch-eager` runs the unmodified reference modules.py / vision_transformer.py /
training_step text in PyTorch eager ON THE GPU (fp32 defaults and bf16 autocast) plus the library kernels (cuBLAS
GEMMs, SDPA) at the step's shapes: the "reference PyTorch path on B200" comparator (SURVEY.md §2.2, BASELINE.md §5).
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

CONFIGS = {
    # BASELINE.json configs[1..3]; batch is PER GPU (reference DDP semantics: DataLoader batch_size per process)
    "c1": dict(model_type="vit_small", res=224, batch=32, desc="ViT-S/8 224x224 batch=32/GPU self+knn+5 random, bf16"),
    "c2": dict(model_type="vit_base", res=320, batch=32, desc="ViT-B/8 320x320 batch=32/GPU, bf16"),
    "c3": dict(model_type="vit_base", res=448, batch=16, desc="ViT-B/8 448x448 batch=16/GPU, bf16"),
    # BASELINE.json configs[4]: eval probes + dense CRF on 1024x2048 frames (code 128x256)
    "c4": dict(model_type=None, res=None, batch=4, desc="eval path: upsample + linear probe + ClusterLookup log-probs, "
                                                        "1024x2048 frames from a 70x128x256 code, fp32 (value / e2e: the fused "
                                                        "probe call; eval_pipeline: + flip-TTA, confusion counts, dense CRF)"),
}
N_CLASSES = 27


def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return dict(hbm=d["hbm_gbs"], tf_burst=d["bf16_tflops"], tf_sust=d.get("bf16_tflops_sustained", d["bf16_tflops"]),
                    source="measured (MEASURED_PEAKS.json)")
    return dict(hbm=6650.0, tf_burst=1590.0, tf_sust=1400.0, source="fallback (B200_PROFILING.md)")


# ----------------------------------------------------------------------------------------------------
# algorithmic work (BASELINE.md §4, SURVEY.md §8d)
# ----------------------------------------------------------------------------------------------------
def vit_dims(model_type, res):
    E, heads = (384, 6) if model_type == "vit_small" else (768, 12)
    hw = (res // 8) ** 2
    return E, heads, hw, hw + 1


def step_flops_per_image(model_type, res):
    E, heads, hw, N = vit_dims(model_type, res)
    gemm = 12 * (2 * N * E * 3 * E + 2 * N * E * E + 2 * 2 * N * E * 4 * E)
    attn = 12 * (2 * 2 * N * N * E)
    patch = 2 * hw * 192 * E
    vit = gemm + attn + patch
    D = 70
    head_fwd = 2 * hw * E * D * 2 + 2 * hw * E * E
    head_bwd = 2 * hw * E * D * 2 + 2 * hw * E * E * 2 + 2 * hw * D * E
    corr = 7 * 2 * 121 * 121 * E + 3 * 7 * 2 * 121 * 121 * D
    return 2 * vit + 2 * (head_fwd + head_bwd) + corr


# ----------------------------------------------------------------------------------------------------
# clocks sampling (B200_PROFILING.md recipe)
# ----------------------------------------------------------------------------------------------------
class ClockSampler:
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "100", "-i", str(self.index)], stdout=subprocess.PIPE, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if self.proc is None:
            return dict(sm_mhz=None, sm_max_mhz=None, reasons=["nvidia-smi unavailable"])
        time.sleep(0.15)
        self.proc.terminate()
        sm, mx, reasons = [], None, set()
        for r in self.rows:
            try:
                sm.append(float(r[1]))
                mx = float(r[2])
                for name, v in zip(["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"], r[4:8]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
            except Exception:
                pass
        sm.sort()
        return dict(sm_mhz=(sm[len(sm) // 2] if sm else None), sm_max_mhz=mx, reasons=sorted(reasons), samples=len(sm))


# ----------------------------------------------------------------------------------------------------
# CPU baseline: the oracle port of the reference step on the host cores (bounded sample)
# ----------------------------------------------------------------------------------------------------
def cpu_step_fn(model_type, res, batch):
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import stego_oracle as O
    E = 384 if model_type == "vit_small" else 768
    sd = O.vit_random_state(model_type, 8, seed=0)
    hp = {k: v.requires_grad_(True) for k, v in O.head_random_state(E, 70, seed=1).items()}
    g = torch.Generator().manual_seed(2)
    probes = {"linear_probe.weight": (torch.randn(N_CLASSES, 70, 1, 1, generator=g) * 0.1).requires_grad_(True),
              "linear_probe.bias": torch.zeros(N_CLASSES, requires_grad=True),
              "cluster_probe.clusters": torch.randn(N_CLASSES, 70, generator=g).requires_grad_(True)}
    params = list(hp.values()) + list(probes.values())
    lrs = [5e-4] * len(hp) + [5e-3] * len(probes)  # train_segmentation.py:379-381
    state = [(torch.zeros_like(p), torch.zeros_like(p)) for p in params]
    cfg = O.LossCfg()
    img = torch.randn(batch, 3, res, res, generator=g)
    img_pos = torch.randn(batch, 3, res, res, generator=g)
    label = torch.randint(-1, N_CLASSES, (batch, res, res), generator=g)
    it = [0]

    def step():
        it[0] += 1
        with torch.no_grad():
            f = O.vit_image_feat(sd, img, model_type, 8)
            fp = O.vit_image_feat(sd, img_pos, model_type, 8)
        masks = [O.draw_dropout2d_mask(batch, E) for _ in range(3)]
        masks_pos = [O.draw_dropout2d_mask(batch, E) for _ in range(3)]
        c1, c2, perms = O.draw_loss_randomness(batch, cfg)
        out = O.training_losses(f, fp, hp, probes, label, masks, masks_pos, c1, c2, perms, cfg, N_CLASSES)
        for p in params:
            p.grad = None
        out["total"].backward()
        with torch.no_grad():
            for p, (m, v), lr in zip(params, state, lrs):
                O.adam_step(p, p.grad, m, v, it[0], lr)
        return float(out["total"].detach())

    return step, torch.get_num_threads()


def time_cpu(model_type, res, batch, steps, warmup, budget_s=150.0):
    """Returns (images/s, s/step, threads, steps actually timed).  The thread count is the fastest of
    {all usable host threads, 32, 16, 8} on one probe step each (small torch CPU ops collapse when a 128-thread pool
    is oversubscribed, and the baseline should be the reference path at its best); the step count is capped so
    that the whole CPU leg stays within `budget_s` seconds."""
    step, _ = cpu_step_fn(model_type, res, batch)
    try:
        avail = len(os.sched_getaffinity(0))
    except Exception:
        avail = os.cpu_count() or 1
    cands = sorted({c for c in (avail, 32, 16, 8) if c <= avail}) or [avail]  # ascending: cheap probes first
    torch.set_num_threads(cands[0])
    step()  # warm-up (allocator, MKL init)
    best_t, best_c = None, cands[0]
    t_spent = 0.0
    for c in cands:
        if best_t is not None and t_spent > budget_s / 3:
            break
        torch.set_num_threads(c)
        t0 = time.perf_counter()
        step()
        dt = time.perf_counter() - t0
        t_spent += dt
        if best_t is None or dt < best_t:
            best_t, best_c = dt, c
        elif dt > 1.5 * best_t:
            break  # more threads are already making it slower (oversubscribed pool): do not probe the larger counts
    torch.set_num_threads(best_c)
    steps = max(1, min(steps, int(max(budget_s - t_spent, 1.0) / max(best_t, 1e-3))))
    t0 = time.perf_counter()
    for _ in range(steps):
        step()
    dt = (time.perf_counter() - t0) / steps
    return batch / dt, dt, best_c, steps


def reference_step_fn(model_type, res, batch, device, autocast=False):
    """One training step of the REAL reference (src/train_segmentation.py:112-245 over src/modules.py and
    src/dino/vision_transformer.py, all unmodified, from baseline/_ref) behind the stub-Lightning harness.  Returns
    step() or None when the reference copy is not present."""
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import lightning_harness as H
    if not H.available():
        return None
    import tempfile
    from stego_b200.config import make_cfg
    import contextlib
    ts = H.load_reference_segmenter("reference")
    with tempfile.TemporaryDirectory() as td, contextlib.redirect_stdout(sys.stderr):  # the reference prints to stdout;
        ck = os.path.join(td, "dino.pth")                                              # stdout carries ONE JSON line
        H.write_random_dino_checkpoint(ck, model_type, seed=0, perturb=False)
        cfg = make_cfg(model_type=model_type, res=res, batch_size=batch, pretrained_weights=ck)
        torch.manual_seed(0)
        m = ts.LitUnsupervisedSegmenter(N_CLASSES, cfg)
    m = m.to(device)
    m.train()
    b = H.make_batch(batch, res, device, seed=2)
    it = [0]

    def step():
        if autocast:
            with torch.autocast("cuda", dtype=torch.bfloat16):
                loss = m.training_step(b, it[0])
        else:
            loss = m.training_step(b, it[0])
        m.global_step += 1
        it[0] += 1
        return loss

    return step


def time_reference_cpu(model_type, res, batch, steps, warmup, budget_s=150.0):
    """The reference itself on the host cores (all threads torch picks; probed like time_cpu).  None if unavailable."""
    step = reference_step_fn(model_type, res, batch, "cpu")
    if step is None:
        return None
    try:
        avail = len(os.sched_getaffinity(0))
    except Exception:
        avail = os.cpu_count() or 1
    cands = sorted({c for c in (avail, 64, 32, 16) if c <= avail}) or [avail]
    torch.set_num_threads(cands[0])
    step()
    best_t, best_c, t_spent = None, cands[0], 0.0
    for c in cands:
        if best_t is not None and t_spent > budget_s / 3:
            break
        torch.set_num_threads(c)
        t0 = time.perf_counter()
        step()
        dt = time.perf_counter() - t0
        t_spent += dt
        if best_t is None or dt < best_t:
            best_t, best_c = dt, c
        elif dt > 1.5 * best_t:
            break
    torch.set_num_threads(best_c)
    for _ in range(max(0, min(warmup, 1))):
        step()
    steps = max(1, min(steps, int(max(budget_s - t_spent, 1.0) / max(best_t, 1e-3))))
    t0 = time.perf_counter()
    for _ in range(steps):
        step()
    dt = (time.perf_counter() - t0) / steps
    return batch / dt, dt, best_c, steps


def run_torch_eager(args, cfgd, workload):
    """The reference PyTorch path on the B200: unmodified reference modules in eager mode (what PyTorch 2.11 dispatches
    — cuBLAS / cuDNN / ATen), fp32 (PyTorch defaults: TF32 off for matmul) and under bf16 autocast, plus the library
    kernels at the step's GEMM / attention shapes.  One JSON line; `value` is the bf16-autocast images/s."""
    import torch.nn.functional as F
    model_type, res, B = cfgd["model_type"], cfgd["res"], cfgd["batch"]
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    out = {}
    for name, ac in (("fp32", False), ("bf16_autocast", True)):
        try:
            step = reference_step_fn(model_type, res, B, dev, autocast=ac)
            if step is None:
                print(json.dumps({"impl": "torch-eager", "unavailable": "baseline/_ref (reference copy) not present"}))
                return
            for _ in range(max(args.warmup, 3)):
                step()
            torch.cuda.synchronize()
            s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            s.record()
            for _ in range(args.steps):
                step()
            e.record()
            torch.cuda.synchronize()
            ms = s.elapsed_time(e) / args.steps
            out[name] = {"images_per_s": B / (ms / 1e3), "ms_per_step": ms}
        except torch.cuda.OutOfMemoryError as ex:
            out[name] = {"error": "out of memory: " + str(ex)[:120]}
        torch.cuda.empty_cache()
    # library kernels at this config's shapes (2B images through the ViT)
    E, heads, hw, N = vit_dims(model_type, res)
    M = 2 * B * N
    flush = torch.zeros(64 * 1024 * 1024, device=dev)
    lib = {}

    def mm(name, Nn, K):
        a = torch.randn(M, K, device=dev).bfloat16()
        w = (torch.randn(Nn, K, device=dev) * K ** -0.5).bfloat16()
        bias = torch.randn(Nn, device=dev).bfloat16()
        ms = time_kernel(lambda: F.linear(a, w, bias), flush=flush)
        lib[name] = {"ms": ms, "tflops": 2.0 * M * Nn * K / ms / 1e9}

    mm("cublas_qkv", 3 * E, E)
    mm("cublas_proj", E, E)
    mm("cublas_fc1", 4 * E, E)
    mm("cublas_fc2", E, 4 * E)
    q = torch.randn(2 * B, heads, N, 64, device=dev).bfloat16()
    k, v = torch.randn_like(q), torch.randn_like(q)
    ms = time_kernel(lambda: F.scaled_dot_product_attention(q, k, v), flush=flush)
    lib["sdpa_bf16"] = {"ms": ms, "tflops": 2.0 * 2 * 2 * B * N * N * E / ms / 1e9}
    xr = torch.randn(M, E, device=dev)
    ln = torch.nn.LayerNorm(E, eps=1e-6).to(dev)
    ms = time_kernel(lambda: ln(xr), flush=flush)
    lib["aten_layernorm_fp32"] = {"ms": ms}
    best = out.get("bf16_autocast", {}).get("images_per_s") or out.get("fp32", {}).get("images_per_s")
    print(json.dumps({
        "impl": "torch-eager", "metric": "train-step images/sec", "value": best, "unit": "images/s", "n_gpus": 1,
        "steps": args.steps, "warmup": max(args.warmup, 3), "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "bf16 autocast (value) / fp32", "data": "synthetic",
        "config": {"workload": workload, "global_batch": B, "parallelism": "dp1",
                   "what": "unmodified reference modules.py + dino/vision_transformer.py + training_step text "
                           "(baseline/_ref) in PyTorch eager on the B200"},
        "modes": out, "library_kernels": lib}))


# ----------------------------------------------------------------------------------------------------
# per-kernel timing (roofline)
# ----------------------------------------------------------------------------------------------------
def time_kernel(fn, iters=10, flush=None):
    """Average device time of fn() in ms: CUDA events on the launching (current) stream, L2 flushed between."""
    for _ in range(3):
        fn()
    torch.cuda.synchronize()
    tot = 0.0
    for _ in range(iters):
        if flush is not None:
            flush.add_(1.0)  # > L2 (126 MB) write: evicts the previous iteration's working set
        s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s.record()
        fn()
        e.record()
        e.synchronize()
        tot += s.elapsed_time(e)
    return tot / iters


def kernel_rooflines(cfgd, peaks, dev):
    """Time the step's main kernels in isolation at the bench shapes."""
    from stego_b200 import corr, ops
    from stego_b200.config import make_cfg
    model_type, res, Bq = cfgd["model_type"], cfgd["res"], cfgd["batch"]
    E, heads, hw, N = vit_dims(model_type, res)
    B2 = 2 * Bq  # img ++ img_pos share one ViT pass
    M = B2 * N
    flush = torch.zeros(64 * 1024 * 1024, device=dev)  # 256 MB
    g = torch.Generator(device=dev).manual_seed(0)
    rnd = lambda *s: torch.randn(*s, device=dev, generator=g)
    x_bf = rnd(M, E).bfloat16()
    out = {}

    def gemm_case(name, Nn, K, **kw):
        a = rnd(M, K).bfloat16()
        w = (rnd(Nn, K) * K ** -0.5).bfloat16()
        bias = rnd(Nn)
        o = torch.empty(M, Nn, device=dev, dtype=torch.float32 if kw.get("residual") else torch.bfloat16)
        res_ = o if kw.get("residual") else None
        act = kw.get("act", 0)
        ms = time_kernel(lambda: ops.gemm(a, w, o, M=M, N=Nn, K=K, bias=bias, act=act, residual=res_), flush=flush)
        fl = 2.0 * M * Nn * K
        by = M * K * 2 + Nn * K * 2 + M * Nn * (8 if res_ is not None else 2)
        out[name] = dict(ms=ms, tflops=fl / ms / 1e9, gbs=by / ms / 1e6, flops=fl, bytes=by, launches_per_step=12)

    gemm_case("gemm_qkv", 3 * E, E)
    gemm_case("gemm_proj", E, E, residual=True)
    gemm_case("gemm_fc1_gelu", 4 * E, E, act=1)
    gemm_case("gemm_fc2", E, 4 * E, residual=True)
    if os.environ.get("STEGO_BENCH_DIAG"):
        gemm_case("diag_fc1_noact", 4 * E, E)
        gemm_case("diag_proj_bf16out", E, E)
        gemm_case("diag_fc2_bf16out", E, 4 * E)
    qkv = rnd(M, 3 * E).bfloat16()
    ao = torch.empty(M, E, device=dev, dtype=torch.bfloat16)
    ms = time_kernel(lambda: ops.attention(qkv, ao, B2, N, E, heads), flush=flush)
    fl = 2.0 * 2 * B2 * N * N * E
    out["attention"] = dict(ms=ms, tflops=fl / ms / 1e9, gbs=(M * 4 * E * 2) / ms / 1e6, flops=fl, bytes=M * 4 * E * 2,
                            launches_per_step=12)
    # head-dim-64 attention needs one exponential per 256 tensor flops; MUFU.EX2 issues 16 / clk / SM, so the exponentials
    # alone cap the kernel at 4096 flop/clk/SM, half the nominal tensor rate (profiles/r2_attention_v3.md).  Tile-padded count: 128-row query
    # tiles x 64-key tiles, what the kernel actually evaluates.
    n_exp = float(B2 * heads) * (-(-N // 128) * 128) * (-(-N // 64) * 64)
    sm_count = torch.cuda.get_device_properties(dev).multi_processor_count
    out["attention"]["exp_per_launch"] = n_exp
    out["attention"]["exp_per_clk_per_sm_needed_at_peak"] = 16.0
    out["attention"]["exp_rate_gexp_s"] = n_exp / ms / 1e6
    out["attention"]["sm_count"] = sm_count
    xr = rnd(M, E)
    gam, bet = rnd(E), rnd(E)
    ms = time_kernel(lambda: ops.layernorm(xr, gam, bet, x_bf), flush=flush)
    out["layernorm"] = dict(ms=ms, gbs=(M * E * 6) / ms / 1e6, bytes=M * E * 6, launches_per_step=25)

    # correlation + loss (the BASELINE.json-named kernel): tiles -> fd/cd einsums -> loss partials
    cfg = make_cfg()
    spec = corr.LossSpec(cfg)
    h = res // 8
    feats = rnd(Bq, h, h, E).bfloat16().permute(0, 3, 1, 2)
    feats_pos = rnd(Bq, h, h, E).bfloat16().permute(0, 3, 1, 2)
    code = rnd(Bq, h, h, 72)[..., :70].permute(0, 3, 1, 2)
    code_pos = rnd(Bq, h, h, 72)[..., :70].permute(0, 3, 1, 2)
    c1, c2 = torch.rand(Bq, 11, 11, 2, device=dev) * 2 - 1, torch.rand(Bq, 11, 11, 2, device=dev) * 2 - 1
    perms = torch.stack([torch.randperm(Bq, device=dev) for _ in range(5)])
    ft = corr.build_tiles(feats, feats_pos, c1, c2, perms, spec, E)
    ct = corr.build_tiles(code, code_pos, c1, c2, perms, spec, corr.CODE_PAD)
    from stego_b200 import _lib
    partials = torch.empty(7, Bq, 8, device=dev)
    stats = torch.empty(7, 4, device=dev)
    soc, shf = corr._i32(spec.slot_of_call), corr._f32(spec.shifts)

    def corr_fwd():
        _lib.check(_lib.load().stego_corr_loss_fwd(_lib.ptr(ft), _lib.ptr(ct), Bq, 11, E, 70, 7, 7, soc, shf, 1, 1, 0,
                                                   _lib.ptr(partials), _lib.ptr(stats), 0, 0, 0, _lib.stream()), "corr_fwd")

    ms = time_kernel(corr_fwd, flush=flush)
    S = 121
    fl = Bq * (7 * 2 * S * S * E + 7 * 2 * S * S * 70)  # fd + cd forward einsums (algorithmic, SURVEY §8d)
    by = Bq * (2 * hw * E * 2 + 2 * hw * 70 * 2)         # feats, feats_pos, code, code_pos once (bf16 algorithmic)
    out["corr_loss_fwd"] = dict(ms=ms, tflops=fl / ms / 1e9, gbs=by / ms / 1e6, flops=fl, bytes=by, launches_per_step=1)
    ms = time_kernel(lambda: corr.build_tiles(feats, feats_pos, c1, c2, perms, spec, E), flush=flush)
    out["sample_norm_feats"] = dict(ms=ms, gbs=(Bq * 2 * hw * E * 2) / ms / 1e6, bytes=Bq * 2 * hw * E * 2,
                                    launches_per_step=1)
    return out


# ----------------------------------------------------------------------------------------------------
# dense correlation sweep (SURVEY.md §8d "dense stress variant", labelled NON-REFERENCE: the reference samples S = 121
# points per image; S = h w is its plotting script's use of the same einsum, src/plot_dino_correspondence.py:45,49)
# ----------------------------------------------------------------------------------------------------
def run_corr_sweep(args):
    """`tensor_correlation` (einsum nchw,ncij->nhwij) as one batched tcgen05 GEMM launch, S x S x E per image, for S from
    the reference's 121 sampled points up to the full feature map of c1 / c2 / c3.  TFLOP/s are ALGORITHMIC (2 S^2 E per
    image) against the measured bf16 peak; `split3` is the fp32-input path (bf16 hi/lo split: 3x the tensor work for
    ~2^-16 relative error), `bf16` the single pass on bf16 features (what the frozen backbone emits)."""
    from stego_b200 import ops
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    peaks = load_peaks()
    flush = torch.zeros(64 * 1024 * 1024, device=dev)
    rows = []
    for name, E, S, B in [("S=121 (reference: 11x11 samples), ViT-S", 384, 121, 32), ("S=121, ViT-B", 768, 121, 32),
                          ("S=400", 384, 400, 32), ("S=784 = 28x28 (c1 dense)", 384, 784, 32),
                          ("S=1600 = 40x40 (c2 dense)", 768, 1600, 32), ("S=3136 = 56x56 (c3 dense)", 768, 3136, 16)]:
        g = torch.Generator(device=dev).manual_seed(S)
        f = torch.nn.functional.normalize(torch.randn(B, S, E, device=dev, generator=g), dim=2)
        ld = (S + 3) // 4 * 4
        out = torch.empty(B, S, ld, device=dev)
        res = {}
        for mode in ("bf16", "split3"):
            if mode == "bf16":
                a = f.bfloat16().contiguous()
                b = a
            else:
                hi = f.bfloat16()
                lo = (f - hi.float()).bfloat16()
                a = torch.cat([hi, lo, hi], 2).contiguous()
                b = torch.cat([hi, hi, lo], 2).contiguous()
            ms = time_kernel(lambda: ops.gemm_batched(a, b, out[:, :, :S]), flush=flush)
            fl = 2.0 * B * S * S * E
            res[mode] = {"ms": ms, "algorithmic_tflops": fl / ms / 1e9, "frac_of_bf16_peak": fl / ms / 1e9 / peaks["tf_burst"],
                         "tensor_work_tflops": fl * (3 if mode == "split3" else 1) / ms / 1e9}
        want = torch.einsum("nsc,ntc->nst", f[:2].double(), f[:2].double())
        err = (out[:2, :, :S].double() - want).abs().max().item()
        rows.append({"case": name, "E": E, "S": S, "images": B, "max_abs_err_split3_vs_fp64": err, **res})
    print(json.dumps({"metric": "correlation-einsum TFLOP/s vs bf16 peak (dense sweep, NON-REFERENCE sizes beyond S=121)",
                      "peak_tflops": peaks["tf_burst"], "peak_source": peaks["source"] + ", burst", "rows": rows}))


# ----------------------------------------------------------------------------------------------------
# configs[4]: fused eval probes (HBM-bound; metric frames/s)
# ----------------------------------------------------------------------------------------------------
def run_c4(args, rank, world, local):
    import torch.nn.functional as F
    B, h, w, H, W, C, n = CONFIGS["c4"]["batch"], 128, 256, 1024, 2048, 70, N_CLASSES
    workload = f"c4: {CONFIGS['c4']['desc']}; synthetic N(0,1) code, random probes"
    g = torch.Generator().manual_seed(7)
    lin = torch.nn.Conv2d(C, n, (1, 1))
    clusters = torch.randn(n, C, generator=g)
    if args.impl == "reference":
        if rank != 0:
            return
        sys.path.insert(0, os.path.join(ROOT, "oracle"))
        import stego_oracle as O
        code = torch.randn(1, C, h, w, generator=g)

        def step():
            with torch.no_grad():
                up = F.interpolate(code, (H, W), mode="bilinear", align_corners=False)
                a = torch.log_softmax(F.conv2d(up, lin.weight, lin.bias), dim=1)
                b = O.cluster_lookup(up, clusters, 2.0, log_probs=True)
            return a, b

        step()
        nst = max(1, min(args.steps, 10))
        t0 = time.perf_counter()
        for _ in range(nst):
            step()
        dt = (time.perf_counter() - t0) / nst
        v = 1.0 / dt
        print(json.dumps({"impl": "reference", "metric": "eval-probe frames/sec", "value": v, "unit": "frames/s",
                          "n_gpus": args.gpus, "steps": nst, "warmup": 1, "ms_per_step": dt * 1e3, "higher_is_better": True,
                          "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
                          "config": {"workload": workload, "global_batch": 1, "parallelism": "cpu"},
                          "cpu_baseline": {"value": v, "unit": "frames/s", "cores": torch.get_num_threads(), "kind": "port",
                                           "sample": "1 frame per step: F.interpolate + conv1x1 + log_softmax + ClusterLookup "
                                                     "(eval_segmentation.py:128-131 op sequence) on the host"},
                          "e2e": {"value": v, "unit": "frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}))
        return
    import torch.distributed as dist
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    from stego_b200 import _lib
    from stego_b200.eval import fused_probe_log_probs
    from stego_b200.modules import ClusterLookup
    lin = lin.to(dev)
    clu = ClusterLookup(C, n).to(dev)
    with torch.no_grad():
        clu.clusters.copy_(clusters)
    host_code = torch.randn(B, h, w, C, generator=torch.Generator().manual_seed(100 + rank)).pin_memory()
    code = host_code.to(dev).permute(0, 3, 1, 2)
    host_arg = torch.empty(2, B, H, W, dtype=torch.uint8).pin_memory()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def run(nsteps, e2e):
        barrier()
        s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s.record()
        for _ in range(nsteps):
            if e2e:  # host code in, per-pixel class maps out (what the eval loop keeps after the CRF / argmax)
                c = host_code.to(dev, non_blocking=True).permute(0, 3, 1, 2)
                _, _, la, ca = fused_probe_log_probs(c, lin, clu, (H, W), 2.0, want_argmax=True)
                host_arg[0].copy_(la, non_blocking=True)
                host_arg[1].copy_(ca, non_blocking=True)
                torch.cuda.current_stream().synchronize()
            else:
                fused_probe_log_probs(code, lin, clu, (H, W), 2.0)
        e.record()
        barrier()
        ms = torch.tensor([s.elapsed_time(e)], device=dev)
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return ms.item()

    run(args.warmup, False)
    model.check_update_health()  # N > 1: every rank made every peer-memory rendezvous of the warm-up
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    l0 = _lib.launch_count()
    ms_dev = run(args.steps, False)
    launches = _lib.launch_count() - l0
    clocks = sampler.stop() if rank == 0 else None
    run(min(args.warmup, 3), True)
    ms_e2e = run(args.steps, True)

    # the whole eval inner loop of src/eval_segmentation.py:119-141 on the device, once per frame batch: flip-TTA average of
    # the two codes + upsample + both probes + confusion counts of the raw predictions (ONE fused call), then dense CRF on
    # the linear and on the cluster log-probabilities (run_crf=True: 2 CRFs per frame), argmax, UnsupervisedMetrics.update
    def eval_pipeline(nsteps):
        from stego_b200 import crf as gcrf
        from stego_b200.eval import UnsupervisedMetrics
        g2 = torch.Generator().manual_seed(200 + rank)
        img = torch.randn(B, 3, H, W, generator=g2).to(dev)
        code2 = torch.randn(B, h, w, C, generator=g2).to(dev).permute(0, 3, 1, 2)
        label = torch.randint(-1, n, (B, H, W), generator=g2).to(dev)
        lin_m = UnsupervisedMetrics("final/linear/", n, 0, False, device=dev)
        clu_m = UnsupervisedMetrics("final/cluster/", n, 0, True, device=dev)
        raw_lin = torch.zeros(n, n, dtype=torch.int64, device=dev)
        raw_clu = torch.zeros(n, n, dtype=torch.int64, device=dev)
        t_crf = 0.0
        barrier()
        s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s.record()
        for _ in range(nsteps):
            lp, cp = fused_probe_log_probs(code, lin, clu, (H, W), 2.0, code_flipped=code2, label=label,
                                           linear_confusion=raw_lin, cluster_confusion=raw_clu)
            c0, c1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            c0.record()
            lin_pred = gcrf.batched_crf(None, img, lp).argmax(1)
            clu_pred = gcrf.batched_crf(None, img, cp).argmax(1)
            c1.record()
            lin_m.update(lin_pred, label)
            clu_m.update(clu_pred, label)
            c1.synchronize()
            t_crf += c0.elapsed_time(c1)
        e.record()
        barrier()
        ms = s.elapsed_time(e)
        return ms, t_crf, clu_m.compute()

    pipe = None
    if rank == 0 and not args.no_kernel_rooflines:
        eval_pipeline(1)
        pms, pcrf, pmetrics = eval_pipeline(2)
        pipe = {"frames_per_s": 2 * B / (pms / 1e3), "ms_per_frame": pms / (2 * B), "crf_ms_per_frame_two_crfs": pcrf / (2 * B),
                "what": "flip-TTA + upsample + linear & cluster probes + confusion counts (one fused call), dense CRF on both "
                        "probes' log-probabilities (10 mean-field iterations each, permutohedral lattice), argmax, "
                        "UnsupervisedMetrics.update + Hungarian — synthetic noise frames: worst case for the bilateral lattice",
                "cluster_metrics_on_noise": pmetrics}
    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return
    peaks = load_peaks()
    frames = B * world * args.steps
    value = frames / (ms_dev / 1e3)
    by = B * (h * w * C * 4 + 2 * n * H * W * 4)  # algorithmic bytes per step and GPU: read code, write both maps
    gbs = by * args.steps / (ms_dev / 1e3) / 1e9
    line = {"metric": "eval-probe frames/sec", "value": value, "unit": "frames/s", "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms_dev / args.steps, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": workload, "global_batch": B * world, "parallelism": f"dp{world}",
                       "l2": "each step writes 1.8 GB of outputs (> 126 MB L2); no explicit flush"},
            "e2e": {"value": frames / (ms_e2e / 1e3), "unit": "frames/s", "h2d_bytes_per_step": B * h * w * C * 4,
                    "d2h_bytes_per_step": 2 * B * H * W, "ms_per_step": ms_e2e / args.steps},
            "gpu_launches": int(launches), "clocks": clocks,
            "roofline": {"kernel": "eval_probe_vec4_kernel (+ eval_prep_kernel, both inside the timed call)", "bound": "hbm", "achieved": gbs, "peak": peaks["hbm"], "unit": "GB/s",
                         "frac": gbs / peaks["hbm"], "traffic": None, "algorithmic_bytes_per_launch": by,
                         "peak_source": peaks["source"]},
            **({"eval_pipeline": pipe} if pipe else {})}
    if not args.no_cpu_baseline and world == 1:  # the CPU arm is reported at N = 1 only
        sys.path.insert(0, os.path.join(ROOT, "oracle"))
        import stego_oracle as O
        cc = torch.randn(1, C, h, w)
        lc = lin.cpu()
        t0 = time.perf_counter()
        with torch.no_grad():
            up = F.interpolate(cc, (H, W), mode="bilinear", align_corners=False)
            torch.log_softmax(F.conv2d(up, lc.weight, lc.bias), dim=1)
            O.cluster_lookup(up, clusters, 2.0, log_probs=True)
        dt = time.perf_counter() - t0
        line["cpu_baseline"] = {"value": 1.0 / dt, "unit": "frames/s", "cores": torch.get_num_threads(), "kind": "port",
                                "sample": "1 frame, reference op sequence (interpolate + conv1x1 + log_softmax + ClusterLookup)"}
    print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


# ----------------------------------------------------------------------------------------------------
def dump_outputs(out_dir, model, loss):
    """What the caller of training_step holds after the last timed step: the returned loss, the logged values and the
    trainable parameters with their gradients (fp32; < 8 MB for ViT-B), as <name>.npy with '/' in a name written '.'."""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    arrays = {"loss": loss, **{"logged." + k.replace("/", "."): v for k, v in model.logged.items()}}
    for n, p in model.named_parameters():
        if p.grad is not None:  # the parameters the step trains (the decoder has none without the rec term)
            arrays["param." + n], arrays["grad." + n] = p, p.grad
    for name, t in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), torch.as_tensor(t).detach().float().cpu().numpy())


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--config", default="c1", choices=sorted(CONFIGS))
    ap.add_argument("--exchange", default="p2p", choices=["p2p", "nccl"],
                    help="N > 1: fused peer-memory all-reduce + Adam (default) or NCCL all-reduce + Adam launches")
    ap.add_argument("--impl", default="ours", choices=["ours", "reference", "torch-eager"])
    ap.add_argument("--sustain-seconds", type=float, default=5.0, help="length of the extra sustained-clock run (0 = skip)")
    ap.add_argument("--batch", type=int, default=None, help="override the per-GPU batch")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-kernel-rooflines", action="store_true")
    ap.add_argument("--breakdown", action="store_true", help="also report per-phase device time of the step")
    ap.add_argument("--corr-sweep", action="store_true", help="dense tensor_correlation sweep (S = 121 ... h w) and exit")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last one computed (loss, logged values, the trainable "
                         "parameters and their gradients) as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be >= 1")
    if args.dump_outputs and (args.corr_sweep or args.config == "c4" or args.impl != "ours"):
        ap.error("--dump-outputs applies to the training step (--config c1|c2|c3, --impl ours)")
    cfgd = dict(CONFIGS[args.config])
    if args.batch:
        cfgd["batch"] = args.batch
    rank = int(os.environ.get("RANK", 0))
    world = int(os.environ.get("WORLD_SIZE", 1))
    local = int(os.environ.get("LOCAL_RANK", 0))
    if args.corr_sweep:
        return run_corr_sweep(args) if rank == 0 else None
    if args.config == "c4":
        return run_c4(args, rank, world, local)
    model_type, res, B = cfgd["model_type"], cfgd["res"], cfgd["batch"]
    workload = f"{args.config}: {cfgd['desc']}; synthetic N(0,1) images, random-init weights"

    if args.impl == "torch-eager":
        if rank != 0:
            return
        return run_torch_eager(args, cfgd, workload)

    if args.impl == "reference":
        # the reference's own CPU implementation of the path, rank 0 only, bounded sample per step: the REAL reference
        # (baseline/_ref through the stub-Lightning harness) when that copy travelled with the repo, else the oracle port
        if rank != 0:
            return
        os.environ["CUDA_VISIBLE_DEVICES"] = ""  # a CPU arm: the reference's unconditional .cuda() must not find a GPU
        sample_b = {"c1": 8, "c2": 2, "c3": 1}.get(args.config, 2)
        kind = "reference"
        r = time_reference_cpu(model_type, res, sample_b, max(1, args.steps), max(1, min(args.warmup, 2)))
        if r is None:
            kind, sample_b = "port", 2
            r = time_cpu(model_type, res, sample_b, max(1, args.steps), max(1, min(args.warmup, 2)))
        v, dt, cores, nst = r
        what = ("the reference's own LitUnsupervisedSegmenter.training_step (baseline/_ref, unmodified, stub Lightning base)"
                if kind == "reference" else "the oracle port")
        print(json.dumps({
            "impl": "reference", "metric": "train-step images/sec", "value": v, "unit": "images/s", "n_gpus": args.gpus,
            "steps": nst, "warmup": args.warmup, "ms_per_step": dt * 1e3, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": workload, "global_batch": sample_b, "parallelism": "cpu"},
            "cpu_baseline": {"value": v, "unit": "images/s", "cores": cores, "kind": kind,
                             "sample": f"batch {sample_b} per step of the {args.config} workload (full step: 2x ViT fwd, "
                                       f"head, loss, probes, backward, 3x Adam) with {what} on {cores} host threads"},
            "e2e": {"value": v, "unit": "images/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}))
        return

    import torch.distributed as dist
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        # the one collective is a <= 2.8 MB all-reduce that runs on a side stream UNDER the next step's frozen backbone:
        # two channels are plenty for it, and every SM NCCL does not occupy stays with the persistent GEMM / attention CTAs
        os.environ.setdefault("NCCL_MAX_NCHANNELS", "2")
        dist.init_process_group("nccl", device_id=dev)
    from stego_b200 import _lib
    from stego_b200.config import make_cfg
    from stego_b200.segmenter import LitUnsupervisedSegmenter
    cfg = make_cfg(model_type=model_type, res=res, batch_size=B, random_backbone_init=True, p2p_update=args.exchange == "p2p")
    torch.manual_seed(0)  # seed_everything(0) on every rank, like the reference (train_segmentation.py:403)
    model = LitUnsupervisedSegmenter(N_CLASSES, cfg).to(dev)
    model.train()
    model.configure_optimizers()
    gdata = torch.Generator().manual_seed(1000 + rank)  # data differs per rank
    host = dict(img=torch.randn(B, 3, res, res, generator=gdata).pin_memory(),
                img_pos=torch.randn(B, 3, res, res, generator=gdata).pin_memory(),
                label=torch.randint(-1, N_CLASSES, (B, res, res), generator=gdata).pin_memory())
    batch = {k: v.to(dev) for k, v in host.items()}
    # the same batch as the public API also accepts it: bf16 images (patchify rounds the fp32 image to bf16 — the GEMM
    # operand — anyway) and uint8 labels (classes 0..26, 255 = ignore instead of -1): 2.4x fewer bytes over PCIe.  The
    # images here are rounded to bf16 on the host, so this path gives the same loss as the fp32/int64 one would on
    # bf16-representable pixels.
    lab8 = host["label"].clone()
    lab8[lab8 < 0] = 255
    host_compact = dict(img=host["img"].bfloat16().pin_memory(), img_pos=host["img_pos"].bfloat16().pin_memory(),
                        label=lab8.to(torch.uint8).pin_memory())
    h2d_of = lambda hb: sum(v.numel() * v.element_size() for v in hb.values())
    h2d = h2d_of(host)
    loss_host = torch.zeros(1).pin_memory()
    loss_ring = [torch.zeros(1).pin_memory(), torch.zeros(1).pin_memory()]

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    copy_stream = torch.cuda.Stream(device=dev)

    def stage_batch(hb):
        """H2D copy of one step's inputs from pinned host memory on a side stream (overlaps the previous step)."""
        with torch.cuda.stream(copy_stream):
            b = {k: v.to(dev, non_blocking=True) for k, v in hb.items()}
            ev = torch.cuda.Event()
            ev.record(copy_stream)
        return b, ev

    host_ms = [0.0]
    last_loss = [None]

    def run(nsteps, e2e, hb=None):
        barrier()
        s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s.record()
        if e2e:
            hb = hb if hb is not None else host
            # every step: inputs come from pinned host memory (H2D inside the timed region, prefetched one step
            # ahead on a copy stream like a pin_memory DataLoader) and the step's loss is read back to the host
            # (D2H, one step delayed so the host never stalls the launch queue).
            pending = []
            nxt = stage_batch(hb)
            for i in range(nsteps):
                b, ev = nxt
                torch.cuda.current_stream().wait_event(ev)
                for t in b.values():
                    t.record_stream(torch.cuda.current_stream())
                if i + 1 < nsteps:
                    nxt = stage_batch(hb)
                loss = model.training_step(b, i)
                slot = loss_ring[i % 2]
                slot.copy_(loss.detach().reshape(1), non_blocking=True)
                done = torch.cuda.Event()
                done.record()
                pending.append((done, slot))
                if len(pending) > 1:
                    d0, s0 = pending.pop(0)
                    d0.synchronize()
                    loss_host.copy_(s0)  # the host really reads the value
            for d0, s0 in pending:
                d0.synchronize()
                loss_host.copy_(s0)
        else:
            t_host = time.perf_counter()
            for i in range(nsteps):
                last_loss[0] = model.training_step(batch, i)
            host_ms[0] = (time.perf_counter() - t_host) * 1e3 / max(nsteps, 1)  # CPU time to ENQUEUE one step
        model.flush()  # the last step's parameter update (side stream) belongs to the timed region too
        e.record()
        barrier()
        ms = torch.tensor([s.elapsed_time(e)], device=dev)
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return ms.item()

    run(args.warmup, False)
    model.check_update_health()  # N > 1: every rank made every peer-memory rendezvous of the warm-up
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    l0 = _lib.launch_count()
    ms_dev = run(args.steps, False)
    host_enqueue_ms = host_ms[0]
    launches = _lib.launch_count() - l0
    clocks = sampler.stop() if rank == 0 else None
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, model, last_loss[0])
    run(min(args.warmup, 3), True, host_compact)
    ms_e2e = run(args.steps, True, host_compact)
    run(min(args.warmup, 3), True, host)
    ms_e2e_full = run(args.steps, True, host)
    # sustained regime: the same device-resident loop for >= --sustain-seconds, with its own clock record (a 20-step
    # timed region is ~0.1 s of burst clocks)
    sustained = None
    if args.sustain_seconds > 0:
        n_sus = max(args.steps, int(args.sustain_seconds * 1e3 / (ms_dev / args.steps)) + 1)
        sampler2 = ClockSampler(local)
        if rank == 0:
            sampler2.start()
        ms_sus = run(n_sus, False)
        clocks2 = sampler2.stop() if rank == 0 else None
        sustained = {"steps": n_sus, "seconds": ms_sus / 1e3, "ms_per_step": ms_sus / n_sus,
                     "value": B * world * n_sus / (ms_sus / 1e3), "unit": "images/s", "clocks": clocks2}
    phases = None
    if args.breakdown:
        model.profile_marks = []
        run(args.steps, False)
        marks, model.profile_marks = model.profile_marks, None
        phases = {}
        for (n0, e0), (n1, e1) in zip(marks[:-1], marks[1:]):
            if n1 != "start":
                phases[n1] = phases.get(n1, 0.0) + e0.elapsed_time(e1) / args.steps
    loss_val = float(loss_host.item())

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    peaks = load_peaks()
    img_per_step = B * world
    value = img_per_step * args.steps / (ms_dev / 1e3)
    e2e_value = img_per_step * args.steps / (ms_e2e / 1e3)
    e2e_full_value = img_per_step * args.steps / (ms_e2e_full / 1e3)
    fl_img = step_flops_per_image(model_type, res)
    line = {
        "metric": "train-step images/sec", "value": value, "unit": "images/s", "n_gpus": world, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": ms_dev / args.steps, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
        "config": {"workload": workload, "global_batch": img_per_step, "per_gpu_batch": B, "res": res,
                   "parallelism": f"dp{world}",
                   "exchange": ("none (1 GPU)" if world == 1 else
                                "all-reduce fused into Adam over NVLink peer memory (csrc/p2p_update.cu), on the side stream under "
                                "the next step's backbone" if getattr(model, "_peer", None) is not None else
                                "NCCL all-reduce + 3 Adam launches on the side stream"),
                   "l2": "per-step working set (>5 GB of activations) exceeds the 126 MB L2; no explicit flush between steps"},
        "e2e": {"value": e2e_value, "unit": "images/s", "h2d_bytes_per_step": h2d_of(host_compact), "d2h_bytes_per_step": 4,
                "ms_per_step": ms_e2e / args.steps,
                "inputs": "LitUnsupervisedSegmenter.training_step with pinned-host bf16 images + uint8 labels (255 = "
                          "ignore) copied H2D every step, loss read back D2H every step"},
        "e2e_fp32_int64_inputs": {"value": e2e_full_value, "unit": "images/s", "h2d_bytes_per_step": h2d,
                                  "d2h_bytes_per_step": 4, "ms_per_step": ms_e2e_full / args.steps,
                                  "inputs": "the reference DataLoader's dtypes: fp32 images + int64 labels"},
        **({"sustained": sustained} if sustained else {}),
        "gpu_launches": int(launches), "host_enqueue_ms_per_step": round(host_enqueue_ms, 3), "clocks": clocks,
        "last_loss": loss_val,
        **({"phase_ms": {k: round(v, 4) for k, v in phases.items()}} if phases else {}),
        "step_tensor_roofline": {"flops_per_image": fl_img, "achieved_tflops": value / world * fl_img / 1e12,
                                 "peak_tflops_sustained": peaks["tf_sust"],
                                 "frac": value / world * fl_img / 1e12 / peaks["tf_sust"], "peak_source": peaks["source"]},
    }
    if not args.no_kernel_rooflines:
        ks = kernel_rooflines(cfgd, peaks, dev)
        step_ms = ms_dev / args.steps
        for k, v in ks.items():
            v["share_of_step"] = v["ms"] * v["launches_per_step"] / step_ms
        dom = max((k for k in ks if "tflops" in ks[k] and k != "corr_loss_fwd" and not k.startswith("diag_")),
                  key=lambda k: ks[k]["share_of_step"])
        d = ks[dom]
        traffic = None
        traffic_src = None
        tpath = os.path.join(ROOT, "profiles", "ncu_traffic_r2.json")
        if os.path.exists(tpath):
            # dram__bytes_read.sum + dram__bytes_write.sum per launch from the committed `ncu --set full` capture of
            # THIS build's kernels at these shapes (a profiler cannot run inside the timed region); see `traffic_source`
            tj = json.load(open(tpath))
            if tj.get("config") == args.config and not args.batch:
                traffic = tj["bytes_per_launch"].get(dom)
                traffic_src = tj.get("source")
        line["roofline"] = {"kernel": dom, "bound": "tensor", "achieved": d["tflops"], "peak": peaks["tf_burst"],
                            "unit": "TFLOP/s", "frac": d["tflops"] / peaks["tf_burst"], "traffic": traffic, "traffic_source": traffic_src,
                            "algorithmic_bytes_per_launch": d["bytes"],
                            "algorithmic_flops_per_launch": d["flops"], "ms_per_launch": d["ms"],
                            "share_of_step": d["share_of_step"], "peak_source": peaks["source"] + ", burst"}
        if dom == "attention" and (clocks or {}).get("sm_mhz") and "exp_per_launch" in d:
            # second ceiling of this kernel: the MUFU pipe (16 ex2 / clk / SM at the clock sampled during the run)
            mufu_peak = 16.0 * d["sm_count"] * clocks["sm_mhz"] * 1e6 / 1e9  # Gexp/s
            line["roofline"]["mufu"] = {"exp_per_launch": d["exp_per_launch"], "achieved_gexp_s": d["exp_rate_gexp_s"],
                                        "peak_gexp_s": mufu_peak, "frac": d["exp_rate_gexp_s"] / mufu_peak,
                                        "note": "head_dim 64: 256 tensor flop per exponential, so the MUFU pipe caps this kernel at "
                                                "4096 flop/clk/SM (1.19 PFLOP/s at 1965 MHz, half the nominal tensor rate); frac here = share of that second ceiling"}
        c = ks["corr_loss_fwd"]
        line["corr_roofline"] = {"kernel": "corr_loss_fwd (fd+cd einsums + loss reduction, 7 calls x B images)",
                                 "ms_per_launch": c["ms"], "achieved_tflops": c["tflops"],
                                 "frac_of_bf16_tensor_peak": c["tflops"] / peaks["tf_burst"],
                                 "achieved_gbs_algorithmic": c["gbs"], "frac_of_hbm_peak": c["gbs"] / peaks["hbm"],
                                 "bound": "hbm/latency (S=121: intensity << ridge, SURVEY.md §8d)"}
        line["kernels"] = {k: {kk: (round(vv, 4) if isinstance(vv, float) else vv) for kk, vv in v.items()
                               if kk in ("ms", "tflops", "gbs", "share_of_step")} for k, v in ks.items()}
    if not args.no_cpu_baseline and world == 1:  # the CPU arm is reported at N = 1 only
        # the reference's own training_step on the host cores when its copy travelled with the repo (baseline/_ref, made by
        # __graft_entry__.build()); the oracle port otherwise
        sample_b = {"c1": 4, "c2": 2, "c3": 1}.get(args.config, 2)
        try:
            r = time_reference_cpu(model_type, res, sample_b, 2, 0, budget_s=30.0)
        except Exception as ex:  # the baseline must never take the bench line down
            sys.stderr.write(f"cpu_baseline: reference step failed ({ex!r}); timing the oracle port instead\n")
            r = None
        if r is not None:
            v, dt, cores, nst = r
            line["cpu_baseline"] = {"value": v, "unit": "images/s", "cores": cores, "kind": "reference",
                                    "sample": f"{nst} steps of batch {sample_b} of the {args.config} workload: the reference's "
                                              f"LitUnsupervisedSegmenter.training_step (baseline/_ref, unmodified; Lightning / "
                                              f"Hydra stubbed) on {cores} host threads"}
        else:
            v, dt, cores, nst = time_cpu(model_type, res, 2, 3, 1, budget_s=30.0)
            line["cpu_baseline"] = {"value": v, "unit": "images/s", "cores": cores, "kind": "port",
                                    "sample": f"{nst} steps of batch 2 of the {args.config} workload with the oracle port "
                                              f"(full step incl. 2x ViT fwd) on {cores} host threads"}
    print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
