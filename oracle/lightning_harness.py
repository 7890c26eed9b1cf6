"""Run the REFERENCE's own `LitUnsupervisedSegmenter` (src/train_segmentation.py:53-383, text unmodified) without
Lightning / Hydra / torchmetrics / matplotlib installed.  TEST INFRASTRUCTURE ONLY.

What it is for
  * the drop-in check SURVEY.md §7.3(9) asks for: the reference `training_step` text executed over
    `stego_b200.modules` (`from modules import *` resolves to the B200 package) — `modules_impl="stego_b200"`;
  * the "reference PyTorch path" comparator: the same class over the reference's own `modules.py`
    (`modules_impl="reference"`) on the B200 (PyTorch eager, fp32 or bf16 autocast) and on the host CPU.

Nothing here is product code and nothing under stego_b200/ imports it.  The reference sources are never copied
into the repository: they are read at run time from the directory $STEGO_REFERENCE_SRC names (the reference's `src`)
or from a git-ignored `baseline/_ref/src`.  oracle/make_golden.py runs the reference through this harness and stores
what the tests compare against under tests/golden/.

The stubs replace exactly the third-party names `train_segmentation.py` imports (`:1-16`):
  utils.*            -> nn, F, torch, np, os, join, plt + no-op UnsupervisedMetrics / colormaps / resize / one_hot_feats
  data.*             -> random
  hydra / omegaconf  -> identity decorator / plain containers
  pytorch_lightning  -> LightningModule = nn.Module + optimizers() / manual_backward() / log() / global_step
  seaborn            -> empty module
"""
from __future__ import annotations

import importlib.util
import os
import random
import sys
import types
from typing import Optional

import numpy as np
import torch
import torch.nn as nn
import torch.nn.functional as F

_HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(_HERE)


def reference_src() -> Optional[str]:
    for c in [os.environ.get("STEGO_REFERENCE_SRC", ""), os.path.join(ROOT, "baseline", "_ref", "src")]:
        if c and os.path.isfile(os.path.join(c, "train_segmentation.py")):
            return c
    return None


def available() -> bool:
    return reference_src() is not None


# --------------------------------------------------------------------------------------------------
# stub modules
# --------------------------------------------------------------------------------------------------
class _NoMetrics:
    """utils.UnsupervisedMetrics (src/utils.py:203-274) is only constructed by the segmenter's __init__ on the
    training path; validation is out of scope here."""

    def __init__(self, *a, **k):
        pass

    def update(self, *a, **k):
        pass

    def compute(self):
        return {}

    def reset(self):
        pass


def _resize(classes, size):
    """src/utils.py:61-62."""
    return F.interpolate(classes, (size, size), mode="bilinear", align_corners=False)


def _one_hot_feats(labels, n_classes):
    """src/utils.py:65-66."""
    return F.one_hot(labels, n_classes).permute(0, 3, 1, 2).to(torch.float32)


def _stub_utils():
    m = types.ModuleType("utils")
    m.nn, m.F, m.torch, m.np, m.os, m.join = nn, F, torch, np, os, os.path.join
    m.plt = None
    m.UnsupervisedMetrics = _NoMetrics
    m.create_pascal_label_colormap = lambda: np.zeros((512, 3), dtype=np.uint8)
    m.create_cityscapes_colormap = lambda: np.zeros((512, 3), dtype=np.uint8)
    m.resize = _resize
    m.one_hot_feats = _one_hot_feats
    m.load_model = lambda *a, **k: (_ for _ in ()).throw(RuntimeError("load_model: not available in the harness"))
    m.prep_args = lambda: None
    m._stego_stub = True
    return m


class _LightningModule(nn.Module):
    """The slice of pl.LightningModule the reference's training path touches."""

    def __init__(self):
        super().__init__()
        self.global_step = 0
        self.logged = {}
        self._optimizers = None
        self.trainer = types.SimpleNamespace(optimizers=None, is_global_zero=True)
        self.logger = types.SimpleNamespace(experiment=types.SimpleNamespace(
            add_histogram=lambda *a, **k: None, close=lambda: None, _get_file_writer=lambda: None))

    def save_hyperparameters(self, *a, **k):
        pass

    def optimizers(self):
        if self._optimizers is None:
            self._optimizers = list(self.configure_optimizers())
            self.trainer.optimizers = self._optimizers
        return tuple(self.trainer.optimizers)

    def manual_backward(self, loss):
        loss.backward()

    def log(self, name, value, **_kw):
        self.logged[name] = value.detach() if torch.is_tensor(value) else value

    def log_dict(self, d, **_kw):
        for k, v in d.items():
            self.log(k, v)


def _stub_lightning():
    pl = types.ModuleType("pytorch_lightning")
    pl.LightningModule = _LightningModule
    pl.Trainer = object
    loggers = types.ModuleType("pytorch_lightning.loggers")
    loggers.TensorBoardLogger = object
    utilities = types.ModuleType("pytorch_lightning.utilities")
    seed = types.ModuleType("pytorch_lightning.utilities.seed")
    seed.seed_everything = lambda s: (random.seed(s), np.random.seed(s), torch.manual_seed(s))
    callbacks = types.ModuleType("pytorch_lightning.callbacks")
    callbacks.ModelCheckpoint = object
    pl.loggers, pl.utilities, pl.callbacks = loggers, utilities, callbacks
    utilities.seed = seed
    return {"pytorch_lightning": pl, "pytorch_lightning.loggers": loggers, "pytorch_lightning.utilities": utilities,
            "pytorch_lightning.utilities.seed": seed, "pytorch_lightning.callbacks": callbacks}


def _stub_misc():
    hydra = types.ModuleType("hydra")
    hydra.main = lambda *a, **k: (lambda fn: fn)
    omega = types.ModuleType("omegaconf")
    omega.DictConfig = dict
    omega.OmegaConf = types.SimpleNamespace(set_struct=lambda *a, **k: None, to_yaml=lambda c: str(c))
    data = types.ModuleType("data")
    data.random = random
    sns = types.ModuleType("seaborn")
    return {"hydra": hydra, "omegaconf": omega, "data": data, "seaborn": sns}


def _stego_modules_shim():
    """`modules` as the B200 package: what `from modules import *` sees when stego_b200 replaces src/modules.py."""
    if ROOT not in sys.path:
        sys.path.insert(0, ROOT)
    import stego_b200.modules as ours
    m = types.ModuleType("modules")
    for k in ours.__all__:
        setattr(m, k, getattr(ours, k))
    m.__all__ = list(ours.__all__)
    return m


_OWNED = ["utils", "data", "modules", "hydra", "omegaconf", "seaborn", "pytorch_lightning", "pytorch_lightning.loggers",
          "pytorch_lightning.utilities", "pytorch_lightning.utilities.seed", "pytorch_lightning.callbacks",
          "train_segmentation", "dino", "dino.vision_transformer", "dino.utils"]


def load_reference_segmenter(modules_impl: str = "reference"):
    """Import the reference's train_segmentation.py with the stubs in place and return its module object
    (`.LitUnsupervisedSegmenter` is the reference class, text unmodified).

    modules_impl = "reference": `modules` is the reference's own src/modules.py (PyTorch eager).
    modules_impl = "stego_b200": `modules` is stego_b200.modules (the drop-in under test).
    The module objects are private to this call (sys.modules is restored), so both flavours can coexist."""
    src = reference_src()
    if src is None:
        raise RuntimeError("reference sources not found: set STEGO_REFERENCE_SRC to the reference's src directory")
    saved = {k: sys.modules.get(k) for k in _OWNED}
    saved_path = list(sys.path)
    try:
        for k in _OWNED:
            sys.modules.pop(k, None)
        sys.modules["utils"] = _stub_utils()
        sys.modules.update(_stub_lightning())
        sys.modules.update(_stub_misc())
        sys.path.insert(0, src)
        if modules_impl == "reference":
            if not torch.cuda.is_available():
                # src/modules.py:32 calls .cuda() unconditionally; in a process without a GPU keep modules on the CPU
                nn.Module.cuda = lambda self, device=None: self
            spec = importlib.util.spec_from_file_location("modules", os.path.join(src, "modules.py"))
            mod = importlib.util.module_from_spec(spec)
            sys.modules["modules"] = mod
            spec.loader.exec_module(mod)
        elif modules_impl == "stego_b200":
            sys.modules["modules"] = _stego_modules_shim()
        else:
            raise ValueError(modules_impl)
        spec = importlib.util.spec_from_file_location("train_segmentation", os.path.join(src, "train_segmentation.py"))
        ts = importlib.util.module_from_spec(spec)
        sys.modules["train_segmentation"] = ts
        spec.loader.exec_module(ts)
        ts._modules = sys.modules["modules"]
        return ts
    finally:
        sys.path[:] = saved_path
        for k, v in saved.items():
            if v is None:
                sys.modules.pop(k, None)
            else:
                sys.modules[k] = v


def write_random_dino_checkpoint(path: str, arch: str, seed: int = 3, perturb: bool = True) -> dict:
    """A checkpoint file in the layout DinoFeaturizer loads (src/modules.py:46-58: torch.load(path)["teacher"]) holding
    the random ViT state the oracle tests use — avoids the weight download (no network)."""
    sys.path.insert(0, _HERE)
    import stego_oracle as O
    sd = O.vit_random_state(arch, 8, seed=seed)
    if perturb:
        sd = O.perturb_vit_state(sd)
    torch.save({"teacher": sd}, path)
    return sd


def trainable_state(n_feats: int = 384, dim: int = 70, n_classes: int = 27, seed: int = 4) -> dict:
    """Seeded values for the nine trainable parameters (named as in LitUnsupervisedSegmenter.named_parameters()), so that a
    stored reference run and a later run of this project start from the same state without storing it."""
    sys.path.insert(0, _HERE)
    import stego_oracle as O
    sd = {"net." + k: v for k, v in O.head_random_state(n_feats, dim, seed=seed).items()}
    g = torch.Generator().manual_seed(seed + 1)
    b = 1.0 / dim ** 0.5
    sd["linear_probe.weight"] = (torch.rand(n_classes, dim, 1, 1, generator=g) * 2 - 1) * b
    sd["linear_probe.bias"] = (torch.rand(n_classes, generator=g) * 2 - 1) * b
    sd["cluster_probe.clusters"] = torch.randn(n_classes, dim, generator=g)
    return sd


def load_trainable_state(model: nn.Module, sd: dict, prefix: str = "") -> None:
    """Copy `sd` (keys as trainable_state returns them, `prefix` stripped) into the model's parameters in place."""
    params = dict(model.named_parameters())
    with torch.no_grad():
        for k, v in sd.items():
            if k.startswith(prefix):
                params[k[len(prefix):]].copy_(v)


def make_batch(B: int, res: int, device, seed: int = 1, n_classes: int = 27) -> dict:
    """The dict `training_step` reads (src/train_segmentation.py:121-128): ind, img, img_aug, coord_aug, img_pos,
    label, label_pos (the aug / *_pos label entries are only touched when their loss weights are non-zero)."""
    g = torch.Generator().manual_seed(seed)
    img = torch.randn(B, 3, res, res, generator=g)
    img_pos = img + 0.3 * torch.randn(B, 3, res, res, generator=g)
    label = torch.randint(-1, n_classes, (B, res, res), generator=g)
    b = dict(ind=torch.arange(B), img=img, img_pos=img_pos, label=label, label_pos=label.clone(),
             img_aug=img[:, :, :8, :8].clone(), coord_aug=torch.zeros(B, 8, 8, 2))
    return {k: v.to(device) for k, v in b.items()}
