"""TEST INFRASTRUCTURE ONLY — imports the UNMODIFIED reference from a checkout of andrewjong/SwapNet named by the
environment variable SWAPNET_REFERENCE, so that the golden vectors under tests/golden/ can be generated from it
(tests/tools/make_golden*.py).  Recipe: SURVEY.md App. C.
"""
from __future__ import annotations

import argparse
import os
import sys
import tempfile
import types

import torch

REF = os.path.abspath(os.environ["SWAPNET_REFERENCE"]) if os.environ.get("SWAPNET_REFERENCE") else None


def available() -> bool:
    return REF is not None and os.path.isdir(os.path.join(REF, "models"))


def _install_stubs() -> None:
    if "adabound" not in sys.modules:  # optimizers/__init__.py:4 imports it unconditionally
        m = types.ModuleType("adabound")

        class AdaBound(torch.optim.Adam):
            pass

        m.AdaBound = AdaBound
        sys.modules["adabound"] = m
    if "seaborn" not in sys.modules:  # util/draw_rois.py:4 (texture only)
        m = types.ModuleType("seaborn")
        m.color_palette = lambda name=None, n=12: [(0.5, 0.5, 0.5)] * (n or 12)
        sys.modules["seaborn"] = m


def import_reference():
    """Put the reference first on sys.path (its packages are called models/modules/...)."""
    assert available(), "set SWAPNET_REFERENCE to a checkout of the reference"
    _install_stubs()
    if REF not in sys.path:
        sys.path.insert(0, REF)
    for name in ("models", "modules", "optimizers", "options", "datasets", "util"):
        mod = sys.modules.get(name)
        if mod is not None and not getattr(mod, "__file__", "").startswith(REF):
            raise RuntimeError(f"a non-reference package '{name}' is already imported")
    import models  # noqa: F401
    import modules  # noqa: F401

    return sys.modules["models"], sys.modules["modules"]


def warp_opt(batch_size: int, **over) -> argparse.Namespace:
    d = dict(model="warp", gpu_id=None, is_train=True, checkpoints_dir=tempfile.mkdtemp(prefix="sn_ref_"),
             name="warp", no_confirm=True, body_representation="rgb", body_channels=12,
             cloth_representation="labels", cloth_channels=19, texture_channels=3, init_type="kaiming",
             init_gain=0.02, discriminator="basic", n_layers_D=3, norm="instance", gan_mode="vanilla",
             gan_label_mode="smooth", lambda_gan=1.0, lambda_discriminator=1.0, lambda_gp=10,
             optimizer_G="AdamW", optimizer_D="AdamW", lr=1e-4, d_lr=4e-4, weight_decay=0, d_weight_decay=0.01,
             b1=0.9, b2=0.999, warp_mode="gan", lambda_ce=100, continue_train=False, load_epoch="latest",
             verbose=False, batch_size=batch_size)
    d.update(over)
    return argparse.Namespace(**d)


def texture_opt(batch_size: int, size: int, **over) -> argparse.Namespace:
    o = warp_opt(batch_size, model="texture", name="texture", netG="swapnet", crop_size=size, load_size=size,
                 lambda_l1=10, lambda_content=0, lambda_style=0)
    for k, v in over.items():
        setattr(o, k, v)
    return o
