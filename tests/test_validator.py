"""Validator backend (starvector_b200/validator.py): the reference's registry accepts it and `generate_svg` follows
starvector_hf_validator.py:77-88.  The model is a recording stand-in: no GPU is needed for the contract."""
import abc
import json
import os
import sys
import types

import pytest
import torch

from starvector_b200 import validator as V


class _FakeCore:
    def __init__(self):
        self.calls = []
        self.processor = object()
        self.svg_transformer = types.SimpleNamespace(tokenizer=lambda text, add_special_tokens=False: {"input_ids": [7, 8, 9]})

    def generate_im2svg(self, batch, **kw):
        self.calls.append((batch, kw))
        return ["<svg></svg>"] * batch["image"].shape[0]


class _FakeModel:
    def __init__(self):
        self.model = _FakeCore()
        self.device = torch.device("cpu")


def _load_reference_base(golden_dir):
    """A stand-in for the reference's svg_validator_base module, built from what oracle/make_golden_reference.py recorded of
    it (tests/golden/validator_registry.json): its import path, the abstract methods of `SVGValidator` and the class attribute
    `register_validator` files a class under."""
    with open(os.path.join(golden_dir, "validator_registry.json")) as f:
        spec = json.load(f)
    pkg, _, leaf = spec["module"].rpartition(".")
    saved = {k: sys.modules.get(k) for k in ("starvector", pkg, spec["module"])}
    for n in ("starvector", pkg):
        m = types.ModuleType(n)
        m.__path__ = []
        sys.modules[n] = m
    mod = types.ModuleType(spec["module"])
    mod.validator_registry = {}
    mod.SVGValidator = abc.ABCMeta("SVGValidator", (abc.ABC,), {n: abc.abstractmethod(lambda self, *a, **k: None)
                                                                for n in spec["abstract_methods"]})

    def register_validator(cls):
        mod.validator_registry[getattr(cls, spec["registry_key"])] = cls
        return cls

    mod.register_validator = register_validator
    sys.modules[spec["module"]] = mod
    setattr(sys.modules[pkg], leaf, mod)
    return mod, saved


def test_generate_svg_follows_the_hf_backend():
    class Base:
        task = "im2svg"

    cls = V.make_validator_class(Base)
    v = cls.__new__(cls)
    v.bind_model(_FakeModel())
    assert v.svg_end_token_id == 7 and v.processor is v.model.model.processor
    cfg = {"temperature": 0, "max_length": 300, "num_beams": 1, "top_p": 0.95}
    out = v.generate_svg({"image": torch.zeros(3, 3, 8, 8)}, cfg)
    assert out == ["<svg></svg>"] * 3
    batch, kw = v.model.model.calls[0]
    assert kw["temperature"] == 1.0 and kw["do_sample"] is False and kw["max_length"] == 300     # :78-80
    assert batch["image"].dtype == torch.bfloat16
    assert cfg["temperature"] == 0                                                              # the caller's config is not mutated
    v.task = "text2svg"
    with pytest.raises(NotImplementedError):
        v.generate_svg({"image": torch.zeros(1, 3, 8, 8)}, cfg)


def test_registers_with_the_reference_registry(golden_dir):
    mod, saved = _load_reference_base(golden_dir)
    try:
        cls = V.register()
        assert mod.validator_registry[V.ENGINE_NAME] is cls and issubclass(cls, mod.SVGValidator)
        assert cls.__abstractmethods__ == frozenset()                     # generate_svg, the only abstract method, is provided
        assert V.register() is cls                                        # idempotent
        # validate.py:8-12 resolves full class names through the same registry; the short name goes through the wrapper
        vm = types.ModuleType("validate")
        vm.get_validator = lambda name, config: mod.validator_registry.get(config.model.generation_engine)
        V.install_short_name(vm)
        cfg = types.SimpleNamespace(model=types.SimpleNamespace(generation_engine="b200"))
        assert vm.get_validator("b200", cfg) is cls and cfg.model.generation_engine == V.ENGINE_NAME
    finally:
        for k, v in saved.items():
            if v is None:
                sys.modules.pop(k, None)
            else:
                sys.modules[k] = v
