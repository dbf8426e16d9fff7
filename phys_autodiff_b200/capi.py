"""ctypes binding of include/physad_b200.h -- one Python function per exported symbol."""
from __future__ import annotations

import ctypes as C
import os
import subprocess
from dataclasses import dataclass

_HERE = os.path.dirname(os.path.abspath(__file__))
_ROOT = os.path.dirname(_HERE)
_LIB = None

_F = C.POINTER(C.c_float)
_D = C.POINTER(C.c_double)


class PhysadError(RuntimeError):
    pass


class CGrid(C.Structure):
    _fields_ = [("nx", C.c_int), ("ny", C.c_int), ("nz", C.c_int), ("hx", C.c_float), ("hy", C.c_float),
                ("hz", C.c_float), ("dt", C.c_float), ("periodic", C.c_int)]


class CPhysWeights(C.Structure):
    _fields_ = [("w_sigma", C.c_float), ("w_u", C.c_float)]


class CMlpConfig(C.Structure):
    _fields_ = [("In", C.c_int), ("H", C.c_int), ("Out", C.c_int), ("norm", C.c_int)]


class CSlab(C.Structure):
    _fields_ = [("z_begin", C.c_int), ("z_end", C.c_int)]


@dataclass
class Grid:
    """phys::GridSpec (reference include/phys.h:8-13)."""
    nx: int
    ny: int
    nz: int
    hx: float = 1.0
    hy: float = 1.0
    hz: float = 1.0
    dt: float = 1.0
    periodic: bool = True

    @property
    def N(self) -> int:
        return self.nx * self.ny * self.nz

    def c(self) -> CGrid:
        return CGrid(self.nx, self.ny, self.nz, self.hx, self.hy, self.hz, self.dt, int(self.periodic))


@dataclass
class PhysWeights:
    """phys::PhysWeights (reference include/phys.h:15-18)."""
    w_sigma: float = 1.0
    w_u: float = 1.0

    def c(self) -> CPhysWeights:
        return CPhysWeights(self.w_sigma, self.w_u)


@dataclass
class MLPConfig:
    """phys::MLPDims + CoordNorm (reference include/mlp_grid.h:13-31)."""
    In: int = 4
    H: int = 64
    Out: int = 4
    minus_one_to_one: bool = True

    def c(self) -> CMlpConfig:
        return CMlpConfig(self.In, self.H, self.Out, int(self.minus_one_to_one))


# every symbol include/physad_b200.h declares (tests/test_boundary.py checks the two lists agree)
EXPORTS = [
    "physad_abi_version", "physad_last_error", "physad_error_string",
    "physad_ctx_create", "physad_ctx_destroy", "physad_ctx_sm_count", "physad_set_weights",
    "physad_mlp_forward_dev", "physad_mlp_forward_host", "physad_mlp_backward_dev", "physad_mlp_backward_host",
    "physad_mlp_grid_infer_dev", "physad_mlp_grid_infer_host",
    "physad_set_weights_deep", "physad_set_deep_mode", "physad_deep_tc_layer_bytes", "physad_deep_tc_pack_layer", "physad_mlp_grid_infer_deep_dev", "physad_mlp_generate_fields_deep_dev", "physad_deep_loss_host",
    "physad_mlp_generate_fields_dev", "physad_mlp_generate_fields_host",
    "physad_phys_residuals_dev", "physad_phys_residuals_host",
    "physad_phys_loss_dev", "physad_phys_loss_host", "physad_phys_loss_slab_dev",
    "physad_phys_backward_dev", "physad_phys_backward_host",
    "physad_phys_backward_from_fields_dev", "physad_phys_backward_from_fields_host",
    "physad_fused_loss_dev", "physad_fused_loss_host", "physad_fused_loss_slab_host", "physad_finalize_loss",
    "physad_set_exact_residuals", "physad_set_fused_variant", "physad_launch_count", "physad_mlp_random_init",
    "physad_fused_loss_grad_dev", "physad_fused_loss_grad_slab_dev", "physad_fused_loss_grad_host", "physad_plan_ranges", "physad_xchg_export", "physad_xchg_connect", "physad_xchg_disconnect", "physad_fused_loss_allreduce_dev",
    "physad_xchg_status", "physad_set_fused_trace", "physad_set_advection",
    "physad_mlp_generate_fields_lp_dev", "physad_phys_loss_lp_dev", "physad_tangent_loss_dev", "physad_tangent_loss_host",
    "physad_tangent_loss_grad_dev", "physad_tangent_loss_grad_host",
    "physad_deep_grad_len", "physad_deep_loss_grad_dev", "physad_deep_loss_grad_host",
    "physad_deep_tangent_loss_dev", "physad_deep_tangent_loss_grad_dev", "physad_deep_tangent_loss_grad_host",
    "physad_mlp_forward_deep_dev", "physad_mlp_forward_deep_host", "physad_deep_data_loss_grad_dev",
    "physad_deep_data_loss_grad_host", "physad_grid_input_scales", "physad_deep_tangent_points_loss_dev",
    "physad_deep_tangent_points_loss_grad_dev", "physad_deep_tangent_points_loss_grad_host",
    "physad_deep_pair_loss_grad_dev", "physad_deep_pair_loss_grad_host",
    "physad_mlp_jacobian_deep_dev", "physad_mlp_jacobian_deep_host", "physad_deep_deriv_loss_grad_dev",
    "physad_deep_deriv_loss_grad_host", "physad_mlp_vjp_deep_dev", "physad_mlp_vjp_deep_host",
    "physad_mlp_jacobian_vjp_deep_dev", "physad_mlp_jacobian_vjp_deep_host",
]


def library_path() -> str:
    # PHYSAD_LIB: tuning aid (A/B runs of experimental builds of the same sources on one box)
    return os.environ.get("PHYSAD_LIB") or os.path.join(_HERE, "libphysad_b200.so")


def build_library(verbose: bool = False) -> str:
    """Compile csrc/ for sm_100a into phys_autodiff_b200/libphysad_b200.so (in-tree)."""
    cmd = ["make", "-C", os.path.join(_HERE, "csrc"), "-j4"]
    r = subprocess.run(cmd, capture_output=not verbose, text=True)
    if r.returncode != 0:
        raise PhysadError("building libphysad_b200.so failed:\n" + (r.stdout or "") + (r.stderr or ""))
    return library_path()


def lib() -> C.CDLL:
    """Load the CUDA library; fail loudly when it is missing (there is no fallback path)."""
    global _LIB
    if _LIB is None:
        path = library_path()
        if not os.path.exists(path):
            raise PhysadError(f"{path} is missing: run `python -c 'import __graft_entry__ as g; g.build()'` "
                              "(nvcc, sm_100a). phys_autodiff_b200 has no CPU or PyTorch fallback.")
        _LIB = C.CDLL(path)
        _LIB.physad_last_error.restype = C.c_char_p
        _LIB.physad_error_string.restype = C.c_char_p
        _LIB.physad_launch_count.restype = C.c_uint64
        _LIB.physad_finalize_loss.restype = None
        _LIB.physad_deep_tc_layer_bytes.restype = C.c_size_t
        _LIB.physad_deep_grad_len.restype = C.c_size_t
    return _LIB


def check(rc: int, what: str = "") -> None:
    if rc != 0:
        L = lib()
        raise PhysadError(f"{what or 'physad call'} failed with status {rc} "
                          f"({L.physad_error_string(rc).decode()}): {L.physad_last_error().decode()}")


def ptr(x):
    """Raw address of a torch tensor / numpy array / int / None as c_void_p."""
    if x is None:
        return C.c_void_p(0)
    if isinstance(x, int):
        return C.c_void_p(x)
    if hasattr(x, "data_ptr"):
        return C.c_void_p(x.data_ptr())
    return C.c_void_p(x.ctypes.data)
