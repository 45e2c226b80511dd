"""Import the reference's own in-tree modules (authoring container only).

`/root/reference` does not exist on the GPU box; callers must check `available()` first.
Only the fairscale import (used for grad-checkpointing, clip_model.py:10) needs a shim
(SURVEY.md §8c).  Nothing here copies reference code: it imports it in place.
"""
from __future__ import annotations

import os
import sys
import types

REF_ROOT = "/root/reference"


def available() -> bool:
    return os.path.isdir(os.path.join(REF_ROOT, "starvector"))


def load():
    """Returns (VisionTransformer, LayerNorm, Adapter) classes of the reference."""
    if not available():
        raise RuntimeError("/root/reference is not mounted")
    for n in ("fairscale", "fairscale.nn", "fairscale.nn.checkpoint",
              "fairscale.nn.checkpoint.checkpoint_activations"):
        sys.modules.setdefault(n, types.ModuleType(n))
    sys.modules["fairscale.nn.checkpoint.checkpoint_activations"].checkpoint_wrapper = lambda m, **k: m
    if REF_ROOT not in sys.path:
        sys.path.insert(0, REF_ROOT)
    from starvector.model.image_encoder.clip_model import VisionTransformer, LayerNorm
    from starvector.model.adapters.adapter import Adapter
    return VisionTransformer, LayerNorm, Adapter


def load_validator_base():
    """The reference's starvector/validation/svg_validator_base.py, imported from its file with stand-ins for what it imports
    but the registry does not need (omegaconf, svgpathtools, the metrics package, cairosvg-backed data utils)."""
    import importlib.util

    if not available():
        raise RuntimeError("the reference checkout is not available")

    def stub(name, **attrs):
        m = types.ModuleType(name)
        m.__dict__.update(attrs)
        sys.modules[name] = m
        return m

    stub("omegaconf", OmegaConf=type("OmegaConf", (), {"save": staticmethod(lambda **k: None), "load": staticmethod(lambda p: {"metrics": {}})}))
    stub("svgpathtools", svgstr2paths=lambda s: None)
    for n in ("starvector", "starvector.validation", "starvector.metrics", "starvector.data"):
        stub(n).__path__ = []
    stub("starvector.metrics.metrics", SVGMetrics=lambda cfg: None)
    stub("starvector.data.util", rasterize_svg=lambda *a, **k: None, clean_svg=lambda s: s, use_placeholder=lambda: "<svg></svg>")
    path = os.path.join(REF_ROOT, "starvector", "validation", "svg_validator_base.py")
    spec = importlib.util.spec_from_file_location("starvector.validation.svg_validator_base", path)
    mod = importlib.util.module_from_spec(spec)
    sys.modules[spec.name] = mod
    spec.loader.exec_module(mod)
    return mod
