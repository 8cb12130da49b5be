"""Generative models (mentflow/generate)."""
from .base import GenerativeModel
from .build import build_flow, build_generator
from .nn import NNGenerator
from .nsf import NSFGenerator, conditioner_masks, layer_order

WrappedZukoFlow = NSFGenerator  # the reference's name for the object build_generator returns
