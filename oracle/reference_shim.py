"""Import the REAL reference (mhamilton723/STEGO): its `src` directory is named by $STEGO_REFERENCE_SRC.

TEST INFRASTRUCTURE ONLY: oracle/check_against_reference.py and oracle/make_golden.py use it; the tests read what
make_golden.py stored under tests/golden/ instead.
`src/modules.py:3` does `from utils import *`, and `src/utils.py` imports matplotlib / wget /
torch._six / torchmetrics which are not installed; modules.py only needs nn, F, torch, np, os, join
from it, so a stub `utils` module is pre-seeded (SURVEY.md §8c).  Nothing is copied from the reference.
"""
from __future__ import annotations

import os
import sys
import types

REFERENCE_SRC = os.environ.get("STEGO_REFERENCE_SRC", "")


def available() -> bool:
    return bool(REFERENCE_SRC) and os.path.isdir(REFERENCE_SRC)


def import_reference():
    """Returns (modules, vision_transformer) of the reference."""
    if not available():
        raise RuntimeError("reference sources not found: set STEGO_REFERENCE_SRC to the reference's src directory")
    if REFERENCE_SRC not in sys.path:
        sys.path.insert(0, REFERENCE_SRC)
    if "utils" not in sys.modules or not getattr(sys.modules["utils"], "_stego_stub", False):
        import numpy as np
        import torch
        import torch.nn as nn
        import torch.nn.functional as F
        stub = types.ModuleType("utils")
        stub.nn, stub.F, stub.torch, stub.np, stub.os, stub.join = nn, F, torch, np, os, os.path.join
        stub._stego_stub = True
        sys.modules["utils"] = stub
    import dino.vision_transformer as vits  # noqa: E402
    import modules  # noqa: E402
    return modules, vits
