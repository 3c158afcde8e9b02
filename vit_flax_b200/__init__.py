"""vit_flax_b200 -- B200-native forward pass of conceptofmind/vit-flax's ``vit_flax/vit.py``.

Public surface = the reference's: ``ViT(...)``, ``.init(rngs, x)``, ``.apply(variables, x)``.
Importing this package does not need a GPU; computing anything does (no CPU fallback).
"""
from .params import count_params, flatten_params, init_params, perturb_params  # noqa: F401
from .checkpoint import load_params, save_params  # noqa: F401
from .optim import adamw  # noqa: F401
from .simple_vit import SimpleViT  # noqa: F401
from .train import Trainer  # noqa: F401
from .vit import ViT  # noqa: F401

__all__ = ["ViT", "SimpleViT", "init_params", "perturb_params", "flatten_params", "count_params", "load_params", "save_params",
           "adamw", "Trainer"]
