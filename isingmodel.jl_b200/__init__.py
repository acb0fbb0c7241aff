"""isingmodel.jl_b200 — B200 (sm_100a) implementation of the spin-update hot path of Wandao123/IsingModel.jl.

The compute lives in ``libising_b200.so`` (hand-written CUDA, C ABI in ``include/ising_b200.h``); this package
is the thin host side that mirrors the reference's module layout (src/IsingModel.jl:3-15):
``SpinSystems``, ``SingleSpinFlip``, ``MultiSpinFlip``, ``OnBipartiteGraph``, ``SamplingHelper``.
There is no CPU fallback: without the built library or without a CUDA device every call raises.
"""
from . import _lib  # noqa: F401
from . import SpinSystems, SingleSpinFlip, OnBipartiteGraph, MultiSpinFlip, SamplingHelper  # noqa: F401
from . import sharding, rowshard, tempering, cluster  # noqa: F401
from .cluster import SwendsenWang  # noqa: F401
from ._lib import IsbError, build, context  # noqa: F401

__all__ = ["SpinSystems", "SingleSpinFlip", "MultiSpinFlip", "OnBipartiteGraph", "SamplingHelper", "sharding", "rowshard", "tempering",
           "cluster", "SwendsenWang", "IsbError", "build", "context"]
