"""Record what the reference's own code returns where tests compare against it, so that those tests run without it.

Run from the repo root, with the reference checkout where `oracle/ref_shim.py` looks for it:
    python -m oracle.make_golden_reference

Writes
  * tests/golden/tiny_v1_reference_vision.pt: ``LayerNorm(VisionTransformer(img))`` and ``Adapter`` of that, both reference
    modules (clip_model.py, adapters/adapter.py) in bf16 on the tiny v1 weights of tests/golden/tiny_v1_{norm}.pt, for both
    adapter norms.  They are computed with oneDNN switched off: its AMX and AVX kernels round bf16 matmuls differently, so
    bits taken with it would only hold on hosts of one CPU family, while ATen's own kernels give the same bits on every
    AVX2 or AVX-512 host.
  * tests/golden/validator_registry.json: the interface of the reference's validator registry
    (validation/svg_validator_base.py) that starvector_b200/validator.py registers with: the module path, the abstract
    methods of ``SVGValidator`` and the attribute of a class that ``register_validator`` files it under.
"""
from __future__ import annotations

import json
import os
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

from oracle import ref_shim  # noqa: E402
from oracle.make_golden import GOLDEN_DIR, reference_vision  # noqa: E402
from starvector_b200.config import dims_tiny  # noqa: E402
from starvector_b200.weights import synthetic_images, synthetic_state_dict  # noqa: E402


def vision() -> None:
    torch.set_num_threads(1)
    out = {}
    with torch.backends.mkldnn.flags(enabled=False):
        for norm_id, norm in ((0, "layer_norm"), (1, "batch_norm")):
            d = dims_tiny(adapter_norm=norm_id)
            vit_out, adapter_out = reference_vision(d, synthetic_state_dict(d, seed=0, init="randomized"), synthetic_images(d, 2, seed=1), norm)
            out[norm] = {"vit_out": vit_out, "adapter_out": adapter_out}
    path = os.path.join(GOLDEN_DIR, "tiny_v1_reference_vision.pt")
    torch.save(out, path)
    print("wrote", path, os.path.getsize(path) // 1024, "KiB")


def validator_registry() -> None:
    mod = ref_shim.load_validator_base()
    probe = type("RegistryProbe", (mod.SVGValidator,), {"generate_svg": lambda self, batch: []})
    assert mod.register_validator(probe) is probe
    key = next(k for k, v in mod.validator_registry.items() if v is probe)
    out = {"module": mod.__name__, "abstract_methods": sorted(mod.SVGValidator.__abstractmethods__),
           "registry_key": next(a for a in ("__name__", "__qualname__", "__module__") if getattr(probe, a) == key)}
    path = os.path.join(GOLDEN_DIR, "validator_registry.json")
    with open(path, "w") as f:
        json.dump(out, f, indent=1)
        f.write("\n")
    print("wrote", path, out)


if __name__ == "__main__":
    vision()                      # before the validator's stand-in modules shadow the reference's `starvector` package
    validator_registry()
