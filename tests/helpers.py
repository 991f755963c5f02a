"""Shared test helpers: golden loading, seeded weights, error metrics. The oracle is imported ONLY by tests."""
import os
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, "oracle")):
    if p not in sys.path:
        sys.path.insert(0, p)

import sdb200  # noqa: E402,F401
from sdb200 import arch  # noqa: E402

GOLDEN = os.path.join(ROOT, "tests", "golden")
CFGS = {"unet": {"tiny": arch.TINY_UNET, "sdv1": arch.SD_V1_UNET},
        "vae": {"tiny": arch.TINY_VAE, "sdv1": arch.SD_V1_VAE},
        "clip": {"tiny": arch.TINY_CLIP, "sdv1": arch.SD_V1_CLIP},
        "safety": {"tiny": arch.TINY_SAFETY, "sdv1": arch.SD_V1_SAFETY}}
_SHAPES = {"unet": arch.unet_param_shapes, "vae": arch.vae_param_shapes, "clip": arch.clip_param_shapes,
           "safety": arch.safety_param_shapes}
_cache = {}
_DRAWS = {"randn": torch.randn, "rand": torch.rand}


def _redraw(o):
    if isinstance(o, dict):
        kind = set(o) - {"seed"}
        if "seed" in o and len(kind) == 1 and kind <= set(_DRAWS):
            kind = kind.pop()
            return _DRAWS[kind](o[kind], generator=torch.Generator().manual_seed(o["seed"]))
        return {k: _redraw(v) for k, v in o.items()}
    if isinstance(o, list):
        return [_redraw(v) for v in o]
    return o


def golden(name):
    """A fixture stores a seeded random input as the draw that made it, {"randn" or "rand": shape, "seed": s}
    (oracle/make_golden.py); it is drawn again here, bit for bit the tensor the reference was given."""
    return _redraw(torch.load(os.path.join(GOLDEN, name), weights_only=True))


def weights(kind, tag, seed):
    key = (kind, tag, seed)
    if key not in _cache:
        _cache[key] = arch.random_state_dict(_SHAPES[kind](CFGS[kind][tag]), seed)
    return _cache[key]


def rel_l2(a, b):
    a = a.detach().double().cpu().flatten()
    b = b.detach().double().cpu().flatten()
    return float((a - b).norm() / b.norm().clamp_min(1e-30))
