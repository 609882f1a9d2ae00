"""Import the reference's own ``python_coreml_stable_diffusion.unet`` UNMODIFIED.

TEST INFRASTRUCTURE ONLY (see ``oracle/__init__.py``).

The reference network definitions (``unet.py``, ``attention.py``, ``layer_norm.py``,
``controlnet.py``) need exactly two things that are not installed in this image:

* ``diffusers.ModelMixin`` / ``diffusers.configuration_utils.{ConfigMixin, register_to_config}``
  (reference ``unet.py:9-10``, ``controlnet.py:6-7``)
* ``coremltools.models.utils._macos_version`` (reference ``unet.py:26``)

Both are replaced by the minimal stand-ins below (SURVEY.md section 8c lists the exact
requirements).  No reference source is copied: the modules are imported from where they lie
(``$B200SD_REFERENCE`` or ``baseline/_ref``).  Only the golden-fixture generators under
``tests/golden/`` need the reference tree; the tests compare against the fixtures they wrote and
``oracle.restated``.
"""
from __future__ import annotations

import functools
import inspect
import os
import sys
import types

import torch.nn as nn

_REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
_CANDIDATES = [
    os.environ.get("B200SD_REFERENCE", ""),
    os.path.join(_REPO, "baseline", "_ref"),
]


def reference_root():
    for c in _CANDIDATES:
        if c and os.path.isfile(os.path.join(c, "python_coreml_stable_diffusion", "unet.py")):
            return c
    return None


def available() -> bool:
    return reference_root() is not None


class _Config(dict):
    """attr-dict: supports cfg.x, cfg.x = v, cfg.get('x')."""

    def __getattr__(self, k):
        try:
            return self[k]
        except KeyError as e:  # pragma: no cover
            raise AttributeError(k) from e

    def __setattr__(self, k, v):
        self[k] = v


def _register_to_config(init):
    sig = inspect.signature(init)

    @functools.wraps(init)
    def wrapper(self, *args, **kwargs):
        bound = sig.bind(self, *args, **kwargs)
        cfg = _Config()
        for name, p in sig.parameters.items():
            if name == "self" or p.kind is inspect.Parameter.VAR_KEYWORD:
                continue
            if p.default is not inspect.Parameter.empty:
                cfg[name] = p.default
        for name, v in bound.arguments.items():
            if name == "self":
                continue
            if sig.parameters[name].kind is inspect.Parameter.VAR_KEYWORD:
                cfg.update(v)
            else:
                cfg[name] = v
        # must be visible as soon as nn.Module.__init__ has run (unet.py:847 writes to it)
        object.__setattr__(self, "_b200sd_pending_config", cfg)
        init(self, *args, **kwargs)

    return wrapper


class _ModelMixin(nn.Module):
    def __init__(self, *a, **k):
        super().__init__()
        cfg = self.__dict__.pop("_b200sd_pending_config", None)
        object.__setattr__(self, "config", cfg if cfg is not None else _Config())


class _ConfigMixin:
    pass


def _install_shims():
    if "diffusers" not in sys.modules:
        d = types.ModuleType("diffusers")
        d.ModelMixin = _ModelMixin
        cu = types.ModuleType("diffusers.configuration_utils")
        cu.ConfigMixin = _ConfigMixin
        cu.register_to_config = _register_to_config
        d.configuration_utils = cu
        d.__b200sd_shim__ = True
        sys.modules["diffusers"] = d
        sys.modules["diffusers.configuration_utils"] = cu
    if "coremltools" not in sys.modules:
        c = types.ModuleType("coremltools")
        m = types.ModuleType("coremltools.models")
        u = types.ModuleType("coremltools.models.utils")
        u._macos_version = lambda: (99, 0)
        m.utils = u
        c.models = m
        c.__b200sd_shim__ = True
        sys.modules["coremltools"] = c
        sys.modules["coremltools.models"] = m
        sys.modules["coremltools.models.utils"] = u


@functools.lru_cache(maxsize=1)
def load():
    """Returns the reference modules (unet, attention, layer_norm, controlnet)."""
    root = reference_root()
    if root is None:
        raise FileNotFoundError("reference tree not found (set B200SD_REFERENCE)")
    _install_shims()
    if root not in sys.path:
        sys.path.insert(0, root)
    import importlib

    unet = importlib.import_module("python_coreml_stable_diffusion.unet")
    attention = importlib.import_module("python_coreml_stable_diffusion.attention")
    layer_norm = importlib.import_module("python_coreml_stable_diffusion.layer_norm")
    controlnet = importlib.import_module("python_coreml_stable_diffusion.controlnet")
    return types.SimpleNamespace(unet=unet, attention=attention, layer_norm=layer_norm,
                                 controlnet=controlnet, root=root)


def build_unet(cfg: dict, state_dict: dict | None = None, xl: bool = False, impl: str | None = None):
    """Instantiate the reference UNet (reference ``torch2coreml.py:915-918`` construction:
    ``unet_cls(**config).eval()`` + ``load_state_dict``) on CPU/fp32."""
    ref = load()
    if impl is not None:
        ref.unet.ATTENTION_IMPLEMENTATION_IN_EFFECT = ref.unet.AttentionImplementations[impl]
    cls = ref.unet.UNet2DConditionModelXL if xl else ref.unet.UNet2DConditionModel
    model = cls(**cfg).eval()
    if state_dict is not None:
        # load_state_dict pre-hooks mutate their input (unet.py:121-138): hand them a copy
        model.load_state_dict({k: v.clone().float() for k, v in state_dict.items()})
    return model


def set_attention_impl(impl: str):
    ref = load()
    ref.unet.ATTENTION_IMPLEMENTATION_IN_EFFECT = ref.unet.AttentionImplementations[impl]


def build_controlnet(cfg: dict, state_dict: dict | None = None):
    """Instantiate the reference ControlNetModel (controlnet.py:49-189) on CPU/fp32."""
    ref = load()
    model = ref.controlnet.ControlNetModel(**cfg).eval()
    if state_dict is not None:
        model.load_state_dict({k: v.clone().float() for k, v in state_dict.items()})
    return model
