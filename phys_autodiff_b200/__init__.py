"""phys_autodiff_b200 -- B200-native (sm_100a) hot path of modular-ngp/phys-autodiff.

The product is the CUDA library ``libphysad_b200.so`` (C-ABI in include/physad_b200.h, sources in
csrc/).  This package is the thin Python host side used by the tests and bench.py: a ctypes
binding (``capi``) and a mirror of the reference's operator names (``ops``) that works on torch
CUDA tensors (device memory + streams only; no torch math on the library's path).  ``autograd.DeepMLP``
wraps a deep network as a ``torch.nn.Module``: the network, its Jacobian and the weight gradient run in
the library's kernels, and torch runs only the caller's loss on the outputs.

There is no CPU fallback: importing works anywhere (so the CPU test tier can check the exported
symbols), but every compute call needs the built library and a B200.
"""
from . import capi  # noqa: F401
from .capi import Grid, MLPConfig, PhysWeights, PhysadError, build_library, library_path  # noqa: F401

__all__ = ["capi", "ops", "autograd", "Grid", "MLPConfig", "PhysWeights", "PhysadError", "build_library", "library_path"]


def __getattr__(name):
    if name in ("ops", "autograd"):
        import importlib
        return importlib.import_module("." + name, __name__)
    raise AttributeError(name)
