"""Host-side mirror of the reference's operator interface over the C-ABI.

Two layers, both thin:

* ``Context`` -- device-resident calls (torch CUDA tensors are used only as device buffers and for
  their stream; all arithmetic happens in libphysad_b200.so) plus the multi-GPU slab driver.
* module-level functions with the reference's names (``mlp_grid_infer_cuda``,
  ``mlp_generate_fields_cuda``, ``cuda_phys_residuals_fused`` ...) taking/returning host numpy
  arrays -- the host-pointer contract of the reference API (include/phys.h:66), so parity tests
  read like the reference's own tests.
"""
from __future__ import annotations

import ctypes as C
from typing import Optional, Sequence

import numpy as np

from . import capi
from .capi import Grid, MLPConfig, PhysWeights, CSlab, check, ptr


def slab_for_rank(nz: int, rank: int, world: int) -> tuple[int, int]:
    """Contiguous z-plane range of `rank` (z is the slowest index, so every output array of a rank
    is one contiguous block).  Remainder planes are spread over the first ranks."""
    return (rank * nz) // world, ((rank + 1) * nz) // world


def _f32(a) -> np.ndarray:
    return np.ascontiguousarray(a, dtype=np.float32)


class Context:
    """Owns a physad_ctx: resident weights, reduction scratch and staging buffers of one GPU."""

    def __init__(self, device: Optional[int] = None):
        self._lib = capi.lib()
        self._h = C.c_void_p()
        check(self._lib.physad_ctx_create(C.byref(self._h), C.c_int(-1 if device is None else device)), "ctx_create")
        self.cfg: Optional[MLPConfig] = None
        self.hidden_layers: Optional[int] = None   # L of the network set by set_weights_deep
        self._peers = None  # (rank, world) once connect_peers() has mapped the peers' exchange buffers

    def close(self):
        if self._h:
            self._lib.physad_ctx_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # -- bookkeeping -------------------------------------------------------------------------
    @property
    def sm_count(self) -> int:
        return int(self._lib.physad_ctx_sm_count(self._h))

    @property
    def launch_count(self) -> int:
        return int(self._lib.physad_launch_count(self._h))

    def set_exact_residuals(self, on: bool) -> bool:
        """False (default): residual arithmetic in fp32 with FMAs like the reference's own CUDA kernels;
        True: in double exactly as the CPU reference (bit-identical residuals, ~5 % slower)."""
        return bool(self._lib.physad_set_exact_residuals(self._h, C.c_int(int(on))))

    def set_advection(self, upwind: bool) -> bool:
        """Advection scheme of the stage-wise physics operators: False = central (the reference), True = first-order
        upwind (additive switch).  Returns the previous setting."""
        return bool(self._lib.physad_set_advection(self._h, C.c_int(int(upwind))))

    def set_fused_variant(self, v: int) -> int:
        return int(self._lib.physad_set_fused_variant(self._h, C.c_int(v)))

    def connect_peers(self, group=None) -> bool:
        """Map every rank's exchange buffer (CUDA IPC over NVLink) so the fused kernel can all-reduce its
        two sums itself.  torch.distributed is used only to all-gather the 64-byte handles.  Returns
        False (and leaves the NCCL path in place) for a single rank, or -- consistently on every rank --
        when any rank could not export or map a buffer (e.g. CUDA IPC not permitted in the container)."""
        import torch
        import torch.distributed as dist
        if not dist.is_initialized() or dist.get_world_size(group) == 1:
            return False
        world, rank = dist.get_world_size(group), dist.get_rank(group)
        buf = C.create_string_buffer(64)
        ok = self._lib.physad_xchg_export(self._h, buf) == 0
        handles = [None] * world
        dist.all_gather_object(handles, bytes(buf.raw) if ok else None, group=group)
        if ok and all(h is not None for h in handles):
            blob = C.create_string_buffer(b"".join(handles), 64 * world)
            ok = self._lib.physad_xchg_connect(self._h, C.c_int(rank), C.c_int(world), blob) == 0
        else:
            ok = False
        flag = torch.tensor([1 if ok else 0], device="cuda")
        dist.all_reduce(flag, op=dist.ReduceOp.MIN, group=group)   # also orders: nobody launches an exchange
        if not bool(flag.item()):                                  # before every rank has mapped every buffer
            self._lib.physad_xchg_disconnect(self._h)
            self._peers = None
            return False
        self._peers = (rank, world)
        return True

    def xchg_status(self) -> bool:
        """True if an in-kernel exchange since the last call gave up waiting for a peer (synchronises the device)."""
        v = C.c_int(0)
        check(self._lib.physad_xchg_status(self._h, C.byref(v)), "xchg_status")
        return bool(v.value)

    def set_fused_trace(self, buf=None) -> None:
        """Diagnostics: per-block timeline of the following fused launches into `buf` (a zeroed int64/uint64 CUDA tensor
        of blocks x 18 x 2 elements, see include/physad_b200.h); None switches it off."""
        if buf is None:
            check(self._lib.physad_set_fused_trace(self._h, None, C.c_int(0)), "set_fused_trace")
        else:
            check(self._lib.physad_set_fused_trace(self._h, ptr(buf), C.c_int(buf.numel() // 36)), "set_fused_trace")
        self._trace_keep = buf

    def disconnect_peers(self) -> None:
        self._lib.physad_xchg_disconnect(self._h)
        self._peers = None

    def set_weights(self, cfg: MLPConfig, W1, b1, W2, b2) -> None:
        W1, b1, W2, b2 = _f32(W1), _f32(b1), _f32(W2), _f32(b2)
        assert W1.size == cfg.H * cfg.In and b1.size == cfg.H and W2.size == cfg.Out * cfg.H and b2.size == cfg.Out
        c = cfg.c()
        check(self._lib.physad_set_weights(self._h, C.byref(c), ptr(W1), ptr(b1), ptr(W2), ptr(b2)), "set_weights")
        self.cfg = cfg
        self.hidden_layers = None   # a plain set_weights replaces any deep network

    # -- helpers -------------------------------------------------------------------------------
    @staticmethod
    def _stream():
        import torch
        return C.c_void_p(torch.cuda.current_stream().cuda_stream)

    @staticmethod
    def _slab(g: Grid, slab):
        z0, z1 = (0, g.nz) if slab is None else slab
        return CSlab(z0, z1), (z1 - z0) * g.ny * g.nx

    @staticmethod
    def _empty(n, dtype=None):
        import torch
        return torch.empty(n, dtype=dtype or torch.float32, device="cuda")

    # -- MLP -------------------------------------------------------------------------------------
    def mlp_forward(self, x):
        """y[B,Out] = MLP(x[B,In]) on device tensors (mlp_forward<ExecCuda>, include/mlp.h:5-6)."""
        B = x.shape[0]
        y = self._empty(B * self.cfg.Out)
        check(self._lib.physad_mlp_forward_dev(self._h, ptr(x), ptr(y), C.c_size_t(B), self._stream()), "mlp_forward")
        return y.view(B, self.cfg.Out)

    def mlp_grid_infer(self, g: Grid, t: float, slab=None):
        cs, n = self._slab(g, slab)
        out = self._empty(n * 4)
        cg = g.c()
        check(self._lib.physad_mlp_grid_infer_dev(self._h, C.byref(cg), C.byref(cs), C.c_float(t), ptr(out),
                                                  self._stream()), "mlp_grid_infer")
        return out.view(n, 4)

    def mlp_generate_fields(self, g: Grid, t: float, dt: float, slab=None):
        cs, n = self._slab(g, slab)
        s = [self._empty(n) for _ in range(3)]
        u = [self._empty(3 * n) for _ in range(3)]
        cg = g.c()
        check(self._lib.physad_mlp_generate_fields_dev(self._h, C.byref(cg), C.byref(cs), C.c_float(t), C.c_float(dt),
                                                       ptr(s[0]), ptr(s[1]), ptr(s[2]), ptr(u[0]), ptr(u[1]), ptr(u[2]),
                                                       self._stream()), "mlp_generate_fields")
        return s[0], s[1], s[2], u[0], u[1], u[2]

    # -- reduced-precision field I/O (additive) ---------------------------------------------------------
    @staticmethod
    def _lp(dtype):
        import torch
        return {"f16": (1, torch.float16), "bf16": (2, torch.bfloat16)}[dtype]

    def mlp_generate_fields_lp(self, g: Grid, t: float, dt: float, dtype: str = "bf16", slab=None):
        """The six fields as 16-bit device tensors (dtype 'f16' | 'bf16'): strict-fp32 MLP, rounded to nearest-even on the store."""
        code, td = self._lp(dtype)
        cs, n = self._slab(g, slab)
        s = [self._empty(n, td) for _ in range(3)]
        u = [self._empty(3 * n, td) for _ in range(3)]
        cg = g.c()
        check(self._lib.physad_mlp_generate_fields_lp_dev(self._h, C.byref(cg), C.byref(cs), C.c_float(t), C.c_float(dt), C.c_int(code),
                                                          ptr(s[0]), ptr(s[1]), ptr(s[2]), ptr(u[0]), ptr(u[1]), ptr(u[2]),
                                                          self._stream()), "mlp_generate_fields_lp")
        return s[0], s[1], s[2], u[0], u[1], u[2]

    def phys_loss_lp_acc(self, g: Grid, fields: Sequence, dtype: str = "bf16", want_residuals: bool = False):
        """Loss sums (and fp32 residuals) from 16-bit fields; arithmetic after the load is the fp32 path's."""
        import torch
        code, td = self._lp(dtype)
        assert all(f.dtype == td for f in fields)
        acc = self._empty(2, torch.float64)
        R = [self._empty(g.N) for _ in range(4)] if want_residuals else [None] * 4
        cg = g.c()
        check(self._lib.physad_phys_loss_lp_dev(self._h, C.byref(cg), C.c_int(code), *[ptr(f) for f in fields], ptr(acc),
                                                *[ptr(r) for r in R], self._stream()), "phys_loss_lp")
        return (acc, tuple(R)) if want_residuals else acc

    # -- deeper MLPs (additive, BASELINE config 5) -----------------------------------------------------
    def set_weights_deep(self, cfg: MLPConfig, hidden_layers: int, W1, b1, Wh, bh, W2, b2) -> None:
        """L = hidden_layers >= 1 hidden layers of width H; Wh: (L-1) x [H x H] row-major, bh: (L-1) x H."""
        W1, b1, W2, b2 = _f32(W1), _f32(b1), _f32(W2), _f32(b2)
        Wh = _f32(Wh if Wh is not None else np.zeros(0)); bh = _f32(bh if bh is not None else np.zeros(0))
        assert Wh.size == (hidden_layers - 1) * cfg.H * cfg.H and bh.size == (hidden_layers - 1) * cfg.H
        c = cfg.c()
        check(self._lib.physad_set_weights_deep(self._h, C.byref(c), C.c_int(hidden_layers), ptr(W1), ptr(b1),
                                                ptr(Wh) if Wh.size else None, ptr(bh) if bh.size else None, ptr(W2), ptr(b2)),
              "set_weights_deep")
        self.cfg = cfg
        self.hidden_layers = hidden_layers

    def deep_loss(self, g: Grid, pw: PhysWeights, t: float, dt: float):
        """(L_sigma, L_u) of the deep network set by set_weights_deep, in one call (fields stay in context scratch)."""
        ls, lu = C.c_float(), C.c_float()
        cg, cw = g.c(), pw.c()
        check(self._lib.physad_deep_loss_host(self._h, C.byref(cg), C.byref(cw), C.c_float(t), C.c_float(dt), C.byref(ls),
                                              C.byref(lu)), "deep_loss")
        return np.float32(ls.value), np.float32(lu.value)

    # -- closed loop of deeper networks (additive) -------------------------------------------------------------
    def deep_grad_len(self) -> int:
        """P(H, L) = 9H + 4 + (L-1)(H^2 + H): the gradient length of the network set by set_weights_deep."""
        return int(self._lib.physad_deep_grad_len(C.c_int(self.cfg.H), C.c_int(self.hidden_layers or 1)))

    def deep_loss_grad_acc(self, g: Grid, pw: PhysWeights, t: float, dt: float, slab=None, out=None):
        """Device form: a float64 device tensor [acc_sigma, acc_u, grad(P)] of the slab (None = whole grid) for the deep
        network; grad = dW1 | db1 | dWh | dbh | dW2 | db2, scaled by 2w/N of the whole grid, so the slabs' tensors add up."""
        import torch
        out = out if out is not None else self._empty(self.deep_grad_len() + 2, torch.float64)
        cs, _ = self._slab(g, slab)
        cg, cw = g.c(), pw.c()
        check(self._lib.physad_deep_loss_grad_dev(self._h, C.byref(cg), C.byref(cs), C.byref(cw), C.c_float(t), C.c_float(dt),
                                                  ptr(out), ptr(out[2:]), self._stream()), "deep_loss_grad")
        return out

    def deep_loss_grad(self, g: Grid, pw: PhysWeights, t: float, dt: float, group=None):
        """(L_sigma, L_u, grad float64 ndarray[P]) of the deep network.  With torch.distributed initialised each rank
        differentiates its z-slab (field planes two around it recomputed locally) and ONE all-reduce of P+2 doubles
        combines them."""
        import torch.distributed as dist
        world, rank = (dist.get_world_size(group), dist.get_rank(group)) if dist.is_initialized() else (1, 0)
        buf = self.deep_loss_grad_acc(g, pw, t, dt, slab_for_rank(g.nz, rank, world))
        if world > 1:
            dist.all_reduce(buf, op=dist.ReduceOp.SUM, group=group)
        h = buf.cpu().numpy()
        ls, lu = self.finalize(h[:2], pw, g.N)
        return ls, lu, h[2:].copy()

    def deep_loss_grad_host(self, g: Grid, pw: PhysWeights, t: float, dt: float):
        """Host-buffer form with the context's deep weights: (L_sigma, L_u, dW1, db1, dWh, dbh, dW2, db2), float32."""
        H, nl = self.cfg.H, (self.hidden_layers or 1) - 1
        d = [np.empty(n, np.float32) for n in (4 * H, H, nl * H * H, nl * H, 4 * H, 4)]
        ls, lu = C.c_float(), C.c_float()
        cg, cw = g.c(), pw.c()
        check(self._lib.physad_deep_loss_grad_host(self._h, C.byref(cg), C.byref(cw), C.c_float(t), C.c_float(dt), C.byref(ls),
                                                   C.byref(lu), *[ptr(x) if x.size else None for x in d]),
              "deep_loss_grad_host")
        return (np.float32(ls.value), np.float32(lu.value), *d)

    # -- analytic loss of deeper networks and its closed loop (additive) ---------------------------------------
    def deep_tangent_loss_acc(self, g: Grid, t: float, slab=None, acc=None, residuals=None):
        """Analytic (forward-mode) loss of the deep network set by set_weights_deep: the device sums
        {sum Rs^2, sum |Ru|^2} of the slab (None = whole grid); residuals: four slab-sized float32 device tensors or None."""
        import torch
        cs, _ = self._slab(g, slab)
        if acc is None:
            acc = self._empty(2, torch.float64)
        R = residuals if residuals is not None else [None] * 4
        cg = g.c()
        check(self._lib.physad_deep_tangent_loss_dev(self._h, C.byref(cg), C.byref(cs), C.c_float(t), ptr(acc),
                                                     *[ptr(r) for r in R], self._stream()), "deep_tangent_loss")
        return acc

    def deep_tangent_loss_grad_acc(self, g: Grid, pw: PhysWeights, t: float, slab=None, out=None):
        """Device form: a float64 device tensor [acc_sigma, acc_u, grad(P)] of the analytic loss of the deep network for
        the slab (None = whole grid); grad = dW1 | db1 | dWh | dbh | dW2 | db2, scaled by 2w/N of the whole grid, so the
        slabs' tensors add up."""
        import torch
        out = out if out is not None else self._empty(self.deep_grad_len() + 2, torch.float64)
        cs, _ = self._slab(g, slab)
        cg, cw = g.c(), pw.c()
        check(self._lib.physad_deep_tangent_loss_grad_dev(self._h, C.byref(cg), C.byref(cs), C.byref(cw), C.c_float(t),
                                                          ptr(out), ptr(out[2:]), self._stream()), "deep_tangent_loss_grad")
        return out

    def deep_tangent_loss_grad(self, g: Grid, pw: PhysWeights, t: float, group=None):
        """(L_sigma, L_u, grad float64 ndarray[P]) of the analytic loss of the deep network.  With torch.distributed
        initialised each rank differentiates its z-slab and ONE all-reduce of P+2 doubles combines them."""
        import torch.distributed as dist
        world, rank = (dist.get_world_size(group), dist.get_rank(group)) if dist.is_initialized() else (1, 0)
        buf = self.deep_tangent_loss_grad_acc(g, pw, t, slab_for_rank(g.nz, rank, world))
        if world > 1:
            dist.all_reduce(buf, op=dist.ReduceOp.SUM, group=group)
        h = buf.cpu().numpy()
        ls, lu = self.finalize(h[:2], pw, g.N)
        return ls, lu, h[2:].copy()

    def deep_tangent_loss_grad_host(self, g: Grid, pw: PhysWeights, t: float):
        """Host-buffer form with the context's deep weights: (L_sigma, L_u, dW1, db1, dWh, dbh, dW2, db2) of the analytic
        loss, float32."""
        H, nl = self.cfg.H, (self.hidden_layers or 1) - 1
        d = [np.empty(n, np.float32) for n in (4 * H, H, nl * H * H, nl * H, 4 * H, 4)]
        ls, lu = C.c_float(), C.c_float()
        cg, cw = g.c(), pw.c()
        check(self._lib.physad_deep_tangent_loss_grad_host(self._h, C.byref(cg), C.byref(cw), C.c_float(t), C.byref(ls),
                                                           C.byref(lu), *[ptr(x) if x.size else None for x in d]),
              "deep_tangent_loss_grad_host")
        return (np.float32(ls.value), np.float32(lu.value), *d)

    # -- deeper networks at arbitrary points: forward and data-fit loss (additive) -----------------------------------------
    def mlp_forward_deep(self, x):
        """y[B, 4] = MLP(x[B, 4]) of the network set by set_weights_deep, on device tensors.  x: float32 CUDA tensor of the
        network's inputs (x, y, z, t), already normalised like mlp_forward's; any B (strict fp32, bit-identical to
        mlp_grid_infer_deep at the grid's own coordinates)."""
        x = x.contiguous()
        B = x.numel() // 4
        y = self._empty(B * 4)
        check(self._lib.physad_mlp_forward_deep_dev(self._h, ptr(x), ptr(y), C.c_size_t(B), self._stream()), "mlp_forward_deep")
        return y.view(B, 4)

    def mlp_forward_deep_host(self, x) -> np.ndarray:
        """Host-array form of mlp_forward_deep: x [B, 4] (or flat) -> y float32 [B, 4]."""
        x = _f32(x)
        B = x.size // 4
        y = np.empty((B, 4), np.float32)
        check(self._lib.physad_mlp_forward_deep_host(self._h, ptr(x), ptr(y), C.c_size_t(B)), "mlp_forward_deep_host")
        return y

    @staticmethod
    def _lam(lam):
        """The C-ABI's lam: 4 host floats, or NULL (None) for 1/4 each."""
        if lam is None:
            return None
        lam = [float(v) for v in lam]
        assert len(lam) == 4
        return (C.c_float * 4)(*lam)

    def deep_data_loss_grad_acc(self, x, target, lam=None, n_norm=None, out=None):
        """Device form of the data-fit loss L_d = (1/n_norm) sum_i sum_o lam[o] (y_io - target_io)^2 of the deep network at
        the points x (float32 CUDA tensors x, target [B, 4]): a float64 device tensor [acc, grad(P)] with acc the
        un-normalised weighted sum and grad = dW1 | db1 | dWh | dbh | dW2 | db2 scaled by 2 lam[o] / n_norm, so the tensors
        of shards with the same n_norm add up and grad adds to the physics gradient.  lam None: 1/4 each (the mean squared
        error); n_norm None: B (1 for an empty shard)."""
        import torch
        x, target = x.contiguous(), target.contiguous()
        B = x.numel() // 4
        assert target.numel() == 4 * B
        out = out if out is not None else self._empty(self.deep_grad_len() + 1, torch.float64)
        n = max(B, 1) if n_norm is None else int(n_norm)
        check(self._lib.physad_deep_data_loss_grad_dev(self._h, ptr(x), ptr(target), C.c_size_t(B), self._lam(lam), C.c_size_t(n),
                                                       ptr(out), ptr(out[1:]), self._stream()), "deep_data_loss_grad")
        return out

    def deep_data_loss_grad(self, x, target, lam=None, n_global=None, group=None):
        """(L_d, grad float64 ndarray[P]) of the data-fit loss over the points of every rank.  With torch.distributed
        initialised each rank passes its own points; n_global (default: the sum of B over ranks, one all-reduce of one
        integer) normalises, and ONE all-reduce of P+1 doubles combines the ranks."""
        import torch
        import torch.distributed as dist
        world = dist.get_world_size(group) if dist.is_initialized() else 1
        B = x.numel() // 4
        if n_global is None:
            if world > 1:
                nb = torch.tensor([B], dtype=torch.int64, device=x.device)
                dist.all_reduce(nb, op=dist.ReduceOp.SUM, group=group)
                n_global = int(nb.item())
            else:
                n_global = B
        n_global = max(int(n_global), 1)
        buf = self.deep_data_loss_grad_acc(x, target, lam, n_global)
        if world > 1:
            dist.all_reduce(buf, op=dist.ReduceOp.SUM, group=group)
        h = buf.cpu().numpy()
        return float(h[0] / n_global), h[1:].copy()

    def deep_data_loss_grad_host(self, x, target, lam=None):
        """Host-array form with n_norm = B: (L_d, dW1, db1, dWh, dbh, dW2, db2), float32."""
        x, target = _f32(x), _f32(target)
        B = x.size // 4
        assert target.size == 4 * B
        H, nl = self.cfg.H, (self.hidden_layers or 1) - 1
        d = [np.empty(n, np.float32) for n in (4 * H, H, nl * H * H, nl * H, 4 * H, 4)]
        loss = C.c_float()
        check(self._lib.physad_deep_data_loss_grad_host(self._h, ptr(x), ptr(target), C.c_size_t(B), self._lam(lam), C.byref(loss),
                                                        *[ptr(a) if a.size else None for a in d]), "deep_data_loss_grad_host")
        return (np.float32(loss.value), *d)

    # -- analytic loss of deeper networks at arbitrary points (collocation points; additive) -------------------------------
    @staticmethod
    def _dcdx(dcdx):
        """The C-ABI's dcdx: 3 host floats, dc/dx of the three space inputs (grid_input_scales gives a grid's)."""
        d = [float(v) for v in dcdx]
        assert len(d) == 3
        return (C.c_float * 3)(*d)

    def deep_tangent_points_loss_acc(self, x, dcdx, acc=None, residuals=None):
        """Analytic loss of the deep network set by set_weights_deep at the points x (float32 CUDA tensor [B, 4] of network
        inputs (x, y, z, t), already normalised; the fourth is the grid calls' time input): the device sums
        {sum Rs^2, sum |Ru|^2} over the points; residuals: a float32 CUDA tensor [B, 4] (R_sigma, R_ux, R_uy, R_uz per
        point) or None."""
        import torch
        x = x.contiguous()
        B = x.numel() // 4
        acc = acc if acc is not None else self._empty(2, torch.float64)
        if residuals is not None:
            assert residuals.is_contiguous() and residuals.numel() == 4 * B
        check(self._lib.physad_deep_tangent_points_loss_dev(self._h, ptr(x), C.c_size_t(B), self._dcdx(dcdx), ptr(acc),
                                                            ptr(residuals), self._stream()), "deep_tangent_points_loss")
        return acc

    def deep_tangent_points_loss_grad_acc(self, x, dcdx, pw: PhysWeights, n_norm=None, out=None):
        """Device form: a float64 device tensor [acc_sigma, acc_u, grad(P)] of the analytic loss at the points x, with
        grad = dW1 | db1 | dWh | dbh | dW2 | db2 scaled by 2w/n_norm, so the tensors of shards with the same n_norm add up and
        grad adds to the data-fit and grid gradients.  n_norm None: B (1 for an empty shard)."""
        import torch
        x = x.contiguous()
        B = x.numel() // 4
        out = out if out is not None else self._empty(self.deep_grad_len() + 2, torch.float64)
        n = max(B, 1) if n_norm is None else int(n_norm)
        cw = pw.c()
        check(self._lib.physad_deep_tangent_points_loss_grad_dev(self._h, ptr(x), C.c_size_t(B), self._dcdx(dcdx), C.byref(cw),
                                                                 C.c_size_t(n), ptr(out), ptr(out[2:]), self._stream()),
              "deep_tangent_points_loss_grad")
        return out

    def deep_tangent_points_loss_grad(self, x, dcdx, pw: PhysWeights, n_global=None, group=None):
        """(L_sigma, L_u, grad float64 ndarray[P]) of the analytic loss over the points of every rank.  With
        torch.distributed initialised each rank passes its own points; n_global (default: the sum of B over ranks, one
        all-reduce of one integer) normalises, and ONE all-reduce of P+2 doubles combines the ranks."""
        import torch
        import torch.distributed as dist
        world = dist.get_world_size(group) if dist.is_initialized() else 1
        B = x.numel() // 4
        if n_global is None:
            if world > 1:
                nb = torch.tensor([B], dtype=torch.int64, device=x.device)
                dist.all_reduce(nb, op=dist.ReduceOp.SUM, group=group)
                n_global = int(nb.item())
            else:
                n_global = B
        n_global = max(int(n_global), 1)
        buf = self.deep_tangent_points_loss_grad_acc(x, dcdx, pw, n_global)
        if world > 1:
            dist.all_reduce(buf, op=dist.ReduceOp.SUM, group=group)
        h = buf.cpu().numpy()
        ls, lu = self.finalize(h[:2], pw, n_global)
        return ls, lu, h[2:].copy()

    def deep_tangent_points_loss_grad_host(self, x, dcdx, pw: PhysWeights):
        """Host-array form with n_norm = B: x [B, 4] (or flat) -> (L_sigma, L_u, dW1, db1, dWh, dbh, dW2, db2), float32."""
        x = _f32(x)
        B = x.size // 4
        H, nl = self.cfg.H, (self.hidden_layers or 1) - 1
        d = [np.empty(n, np.float32) for n in (4 * H, H, nl * H * H, nl * H, 4 * H, 4)]
        ls, lu = C.c_float(), C.c_float()
        cw = pw.c()
        check(self._lib.physad_deep_tangent_points_loss_grad_host(self._h, ptr(x), C.c_size_t(B), self._dcdx(dcdx), C.byref(cw),
                                                                  C.byref(ls), C.byref(lu), *[ptr(a) if a.size else None for a in d]),
              "deep_tangent_points_loss_grad_host")
        return (np.float32(ls.value), np.float32(lu.value), *d)

    def set_deep_mode(self, mode: int) -> None:
        """0: strict fp32 (bit-exact, default); 1: hidden layers on the tensor cores with three-term bf16 operands (~1e-6)."""
        check(self._lib.physad_set_deep_mode(self._h, C.c_int(mode)), "set_deep_mode")

    def mlp_grid_infer_deep(self, g: Grid, t: float, slab=None):
        cs, n = self._slab(g, slab)
        out = self._empty(n * 4)
        cg = g.c()
        check(self._lib.physad_mlp_grid_infer_deep_dev(self._h, C.byref(cg), C.byref(cs), C.c_float(t), ptr(out),
                                                       self._stream()), "mlp_grid_infer_deep")
        return out.view(n, 4)

    def mlp_generate_fields_deep(self, g: Grid, t: float, dt: float, slab=None):
        cs, n = self._slab(g, slab)
        s = [self._empty(n) for _ in range(3)]
        u = [self._empty(3 * n) for _ in range(3)]
        cg = g.c()
        check(self._lib.physad_mlp_generate_fields_deep_dev(self._h, C.byref(cg), C.byref(cs), C.c_float(t), C.c_float(dt),
                                                            ptr(s[0]), ptr(s[1]), ptr(s[2]), ptr(u[0]), ptr(u[1]), ptr(u[2]),
                                                            self._stream()), "mlp_generate_fields_deep")
        return s[0], s[1], s[2], u[0], u[1], u[2]

    # -- physics on supplied device fields -----------------------------------------------------------
    def phys_residuals(self, g: Grid, fields: Sequence):
        R = [self._empty(g.N) for _ in range(4)]
        cg = g.c()
        check(self._lib.physad_phys_residuals_dev(self._h, C.byref(cg), *[ptr(f) for f in fields], *[ptr(r) for r in R],
                                                  self._stream()), "phys_residuals")
        return tuple(R)

    def phys_loss_acc(self, g: Grid, fields: Sequence, want_residuals: bool = False):
        import torch
        acc = self._empty(2, torch.float64)
        R = [self._empty(g.N) for _ in range(4)] if want_residuals else [None] * 4
        cg = g.c()
        check(self._lib.physad_phys_loss_dev(self._h, C.byref(cg), *[ptr(f) for f in fields], ptr(acc),
                                             *[ptr(r) for r in R], self._stream()), "phys_loss")
        return (acc, tuple(R)) if want_residuals else acc

    def phys_loss(self, g: Grid, pw: PhysWeights, fields: Sequence, want_residuals: bool = False):
        out = self.phys_loss_acc(g, fields, want_residuals)
        acc = out[0] if want_residuals else out
        ls, lu = self.finalize(acc.cpu().numpy(), pw, g.N)
        return (ls, lu, out[1]) if want_residuals else (ls, lu)

    def phys_loss_slab_acc(self, g: Grid, slab, fields_local: Sequence, halo_lo, halo_hi, want_residuals: bool = False):
        """One rank's share of the loss on supplied fields: `fields_local` hold the slab's planes, `halo_lo/hi`
        ([4, ny, nx] float32 device tensors) the time-t planes below / above it.  Returns the device sums."""
        import torch
        cs, n = self._slab(g, slab)
        acc = self._empty(2, torch.float64)
        R = [self._empty(n) for _ in range(4)] if want_residuals else [None] * 4
        cg = g.c()
        check(self._lib.physad_phys_loss_slab_dev(self._h, C.byref(cg), C.byref(cs), *[ptr(f) for f in fields_local],
                                                  ptr(halo_lo), ptr(halo_hi), ptr(acc), *[ptr(r) for r in R],
                                                  self._stream()), "phys_loss_slab")
        return (acc, tuple(R)) if want_residuals else acc

    @staticmethod
    def halo_sources(g: Grid, slab):
        """Global plane indices (wrap/clamp applied) a slab needs below and above itself."""
        z0, z1 = slab
        if g.periodic:
            return (z0 - 1) % g.nz, z1 % g.nz
        return max(z0 - 1, 0), min(z1, g.nz - 1)

    def phys_loss_sharded(self, g: Grid, pw: PhysWeights, fields_local: Sequence, group=None, want_residuals: bool = False):
        """Multi-GPU loss on externally supplied, z-sharded fields: every rank holds its slab of the six fields;
        the two time-t boundary planes of every slab are all-gathered (2 x 4 x ny x nx floats per rank), each
        rank picks its two halo planes, runs the stencil + reduction on its slab, and one all-reduce of two
        doubles combines the sums."""
        import torch
        import torch.distributed as dist
        world, rank = (dist.get_world_size(group), dist.get_rank(group)) if dist.is_initialized() else (1, 0)
        slabs = [slab_for_rank(g.nz, r, world) for r in range(world)]
        z0, z1 = slabs[rank]
        pln = g.nx * g.ny
        s_0, u_0 = fields_local[1], fields_local[4]
        n = (z1 - z0) * pln

        def plane(zl):  # [4, pln]: sigma_t, ux_t, uy_t, uz_t of local plane zl
            return torch.stack([s_0[zl * pln:(zl + 1) * pln]] + [u_0[c * n + zl * pln: c * n + (zl + 1) * pln] for c in range(3)])
        mine = torch.stack([plane(0), plane(z1 - z0 - 1)]) if z1 > z0 else torch.zeros(2, 4, pln, device="cuda")
        if world > 1:
            gathered = [torch.empty_like(mine) for _ in range(world)]
            dist.all_gather(gathered, mine.contiguous(), group=group)
        else:
            gathered = [mine]
        lo_z, hi_z = self.halo_sources(g, (z0, z1))

        def fetch(zg):  # boundary plane zg is the first or the last plane of its owner's slab
            owner = next(r for r, (a, b) in enumerate(slabs) if a <= zg < b)
            a, b = slabs[owner]
            if zg == a:
                return gathered[owner][0]
            if zg == b - 1:
                return gathered[owner][1]
            raise capi.PhysadError("halo plane is not a slab boundary plane (slab thinner than the stencil?)")
        if z1 > z0:
            # planes inside my own slab (single rank, or clamp at the domain edge) come from my own arrays
            halo_lo = plane(lo_z - z0) if z0 <= lo_z < z1 else fetch(lo_z)
            halo_hi = plane(hi_z - z0) if z0 <= hi_z < z1 else fetch(hi_z)
            out = self.phys_loss_slab_acc(g, (z0, z1), fields_local, halo_lo.contiguous(), halo_hi.contiguous(), want_residuals)
        else:
            out = (torch.zeros(2, dtype=torch.float64, device="cuda"), tuple([self._empty(0)] * 4)) if want_residuals \
                else torch.zeros(2, dtype=torch.float64, device="cuda")
        acc = out[0] if want_residuals else out
        if world > 1:
            dist.all_reduce(acc, op=dist.ReduceOp.SUM, group=group)
        ls, lu = self.finalize(self._read_acc(acc), pw, g.N)
        return (ls, lu, out[1]) if want_residuals else (ls, lu)

    def phys_backward(self, g: Grid, pw: PhysWeights, R: Sequence):
        G = [self._empty(g.N) for _ in range(4)]
        cg, cw = g.c(), pw.c()
        check(self._lib.physad_phys_backward_dev(self._h, C.byref(cg), C.byref(cw), *[ptr(r) for r in R],
                                                 *[ptr(x) for x in G], self._stream()), "phys_backward")
        return tuple(G)

    def phys_backward_from_fields(self, g: Grid, pw: PhysWeights, fields: Sequence):
        G = [self._empty(g.N) for _ in range(4)]
        cg, cw = g.c(), pw.c()
        check(self._lib.physad_phys_backward_from_fields_dev(self._h, C.byref(cg), C.byref(cw), *[ptr(f) for f in fields],
                                                             *[ptr(x) for x in G], self._stream()),
              "phys_backward_from_fields")
        return tuple(G)

    # -- the metric path --------------------------------------------------------------------------------
    def fused_loss_acc(self, g: Grid, t: float, dt: float, slab=None, acc=None, residuals=None):
        """Enqueue the fused kernel for a slab; returns the device tensor {sum Rs^2, sum |Ru|^2}."""
        import torch
        cs, _ = self._slab(g, slab)
        if acc is None:
            acc = self._empty(2, torch.float64)
        R = residuals if residuals is not None else [None] * 4
        cg = g.c()
        check(self._lib.physad_fused_loss_dev(self._h, C.byref(cg), C.byref(cs), C.c_float(t), C.c_float(dt), ptr(acc),
                                              *[ptr(r) for r in R], self._stream()), "fused_loss")
        return acc

    def prepare_fused(self, g: Grid, t: float, dt: float, slab=None, acc=None, residuals=None, allreduce=False):
        """Pre-marshal one fused launch (ctypes structs, pointers) and return a zero-argument callable that
        enqueues it on the current stream: the per-step host cost matters once a slab takes ~0.2 ms.
        allreduce=True uses the in-kernel peer-memory all-reduce (needs connect_peers())."""
        import torch
        cs, _ = self._slab(g, slab)
        if acc is None:
            acc = self._empty(2, torch.float64)
        R = residuals if residuals is not None else [None] * 4
        cg = g.c()
        if allreduce and not self._peers:
            raise capi.PhysadError("prepare_fused(allreduce=True) needs connect_peers() first")
        fn, h = (self._lib.physad_fused_loss_allreduce_dev if allreduce else self._lib.physad_fused_loss_dev), self._h
        args = (C.byref(cg), C.byref(cs), C.c_float(t), C.c_float(dt), ptr(acc), *[ptr(r) for r in R])
        keep = (cg, cs, acc, R)

        def launch(_keep=keep):
            rc = fn(h, *args, C.c_void_p(torch.cuda.current_stream().cuda_stream))
            if rc:
                check(rc, "fused_loss")
            return acc
        return launch

    def _read_acc(self, acc):
        """16-byte device -> pinned host read of the two sums, then a stream sync."""
        import torch
        if getattr(self, "_pinned_acc", None) is None:
            self._pinned_acc = torch.empty(2, dtype=torch.float64).pin_memory()
        self._pinned_acc.copy_(acc, non_blocking=True)
        torch.cuda.current_stream().synchronize()
        return self._pinned_acc.numpy()

    def finalize(self, acc, pw: PhysWeights, n_global: int):
        a = (C.c_double * 2)(float(acc[0]), float(acc[1]))
        ls, lu = C.c_float(), C.c_float()
        cw = pw.c()
        self._lib.physad_finalize_loss(a, C.byref(cw), C.c_size_t(n_global), C.byref(ls), C.byref(lu))
        return np.float32(ls.value), np.float32(lu.value)

    def fused_loss(self, g: Grid, pw: PhysWeights, t: float, dt: float, group=None, want_residuals: bool = False):
        """Whole path.  With torch.distributed initialised, each rank evaluates its z-slab and one
        all-reduce (sum, 2 doubles) combines the partial sums (SURVEY.md section 8e); residuals, if
        requested, stay sharded."""
        import torch
        import torch.distributed as dist
        world, rank = (dist.get_world_size(group), dist.get_rank(group)) if dist.is_initialized() else (1, 0)
        slab = slab_for_rank(g.nz, rank, world)
        n = (slab[1] - slab[0]) * g.ny * g.nx
        R = [self._empty(n) for _ in range(4)] if want_residuals else None
        if world > 1 and self._peers == (rank, world):
            acc = self.prepare_fused(g, t, dt, slab=slab, residuals=R, allreduce=True)()   # exchange inside the kernel
        else:
            acc = self.fused_loss_acc(g, t, dt, slab=slab, residuals=R)
            if world > 1:
                dist.all_reduce(acc, op=dist.ReduceOp.SUM, group=group)
        ls, lu = self.finalize(self._read_acc(acc), pw, g.N)
        return (ls, lu, tuple(R)) if want_residuals else (ls, lu)

    # -- analytic (tangent) loss: additive, NOT the parity path ---------------------------------------------
    def tangent_loss_acc(self, g: Grid, t: float, slab=None, acc=None, residuals=None):
        """Forward-mode derivatives through the MLP instead of finite differences (include/physad_b200.h); returns the
        device sums {sum Rs^2, sum |Ru|^2} of the slab."""
        import torch
        cs, _ = self._slab(g, slab)
        if acc is None:
            acc = self._empty(2, torch.float64)
        R = residuals if residuals is not None else [None] * 4
        cg = g.c()
        check(self._lib.physad_tangent_loss_dev(self._h, C.byref(cg), C.byref(cs), C.c_float(t), ptr(acc),
                                                *[ptr(r) for r in R], self._stream()), "tangent_loss")
        return acc

    # -- closed loop of the analytic loss: its sums + gradient with respect to the MLP weights (additive) -----
    def tangent_loss_grad_acc(self, g: Grid, pw: PhysWeights, t: float, slab=None, out=None):
        """Device form: a float64 device tensor [acc_sigma, acc_u, grad(9H+4)] of the slab (None = whole grid); grad =
        dW1 | db1 | dW2 | db2, already scaled by 2w/N of the whole grid, so the slabs' tensors add up (all-reduce)."""
        import torch
        out = out if out is not None else self._empty(9 * self.cfg.H + 6, torch.float64)
        cs, _ = self._slab(g, slab)
        cg, cw = g.c(), pw.c()
        check(self._lib.physad_tangent_loss_grad_dev(self._h, C.byref(cg), C.byref(cs), C.byref(cw), C.c_float(t), ptr(out),
                                                     ptr(out[2:]), self._stream()), "tangent_loss_grad")
        return out

    def tangent_loss_grad(self, g: Grid, pw: PhysWeights, t: float, group=None):
        """(L_sigma, L_u, grad float64 ndarray[9H+4]) of the analytic loss for the weights set by set_weights().  With
        torch.distributed initialised each rank differentiates its z-slab and ONE all-reduce of 9H+6 doubles combines them."""
        import torch.distributed as dist
        world, rank = (dist.get_world_size(group), dist.get_rank(group)) if dist.is_initialized() else (1, 0)
        buf = self.tangent_loss_grad_acc(g, pw, t, slab_for_rank(g.nz, rank, world))
        if world > 1:
            dist.all_reduce(buf, op=dist.ReduceOp.SUM, group=group)
        h = buf.cpu().numpy()
        ls, lu = self.finalize(h[:2], pw, g.N)
        return ls, lu, h[2:].copy()

    def tangent_loss_grad_host(self, g: Grid, cfg: MLPConfig, W1, b1, W2, b2, pw: PhysWeights, t: float):
        """Host-buffer form: weights in, (L_sigma, L_u, dW1, db1, dW2, db2) of the analytic loss out (float32)."""
        W1, b1, W2, b2 = _f32(W1), _f32(b1), _f32(W2), _f32(b2)
        d = [np.empty(4 * cfg.H, np.float32), np.empty(cfg.H, np.float32), np.empty(4 * cfg.H, np.float32), np.empty(4, np.float32)]
        ls, lu = C.c_float(), C.c_float()
        cg, cc, cw = g.c(), cfg.c(), pw.c()
        check(self._lib.physad_tangent_loss_grad_host(self._h, C.byref(cg), C.byref(cc), ptr(W1), ptr(b1), ptr(W2), ptr(b2),
                                                      C.byref(cw), C.c_float(t), C.byref(ls), C.byref(lu),
                                                      *[ptr(x) for x in d]), "tangent_loss_grad_host")
        self.cfg = cfg
        return (np.float32(ls.value), np.float32(lu.value), *d)

    # -- closed loop: loss + gradient with respect to the MLP weights (additive) ----------------------------
    def fused_loss_grad_acc(self, g: Grid, pw: PhysWeights, t: float, dt: float, acc=None, grad=None):
        """Device form: returns (acc[2], grad[9H+4]) float64 device tensors; grad = dW1 | db1 | dW2 | db2."""
        import torch
        acc = acc if acc is not None else self._empty(2, torch.float64)
        grad = grad if grad is not None else self._empty(9 * self.cfg.H + 4, torch.float64)
        cg, cw = g.c(), pw.c()
        check(self._lib.physad_fused_loss_grad_dev(self._h, C.byref(cg), C.byref(cw), C.c_float(t), C.c_float(dt),
                                                   ptr(acc), ptr(grad), self._stream()), "fused_loss_grad")
        return acc, grad

    def fused_loss_grad_slab_acc(self, g: Grid, pw: PhysWeights, t: float, dt: float, slab, out=None):
        """One slab's SUMS: returns a float64 device tensor [acc_sigma, acc_u, grad(9H+4)] (all-reduce it over ranks)."""
        import torch
        out = out if out is not None else self._empty(9 * self.cfg.H + 6, torch.float64)
        cs, _ = self._slab(g, slab)
        cg, cw = g.c(), pw.c()
        check(self._lib.physad_fused_loss_grad_slab_dev(self._h, C.byref(cg), C.byref(cs), C.byref(cw), C.c_float(t),
                                                        C.c_float(dt), ptr(out), ptr(out[2:]), self._stream()),
              "fused_loss_grad_slab")
        return out

    def fused_loss_grad(self, g: Grid, pw: PhysWeights, t: float, dt: float, group=None):
        """(L_sigma, L_u, grad float64 ndarray[9H+4]) of the weights set by set_weights().  With torch.distributed
        initialised each rank differentiates its z-slab (fields two planes around it recomputed locally) and ONE
        all-reduce of 9H+6 doubles combines the sums."""
        import torch.distributed as dist
        world, rank = (dist.get_world_size(group), dist.get_rank(group)) if dist.is_initialized() else (1, 0)
        if world == 1:
            acc, grad = self.fused_loss_grad_acc(g, pw, t, dt)
            gh = grad.cpu().numpy()
            ls, lu = self.finalize(self._read_acc(acc), pw, g.N)
            return ls, lu, gh
        buf = self.fused_loss_grad_slab_acc(g, pw, t, dt, slab_for_rank(g.nz, rank, world))
        dist.all_reduce(buf, op=dist.ReduceOp.SUM, group=group)
        h = buf.cpu().numpy()
        ls, lu = self.finalize(h[:2], pw, g.N)
        return ls, lu, h[2:].copy()

    def fused_loss_grad_host(self, g: Grid, cfg: MLPConfig, W1, b1, W2, b2, pw: PhysWeights, t: float, dt: float):
        """Host-buffer form: weights in, (L_sigma, L_u, dW1, db1, dW2, db2) out (float32, the reference's layouts)."""
        W1, b1, W2, b2 = _f32(W1), _f32(b1), _f32(W2), _f32(b2)
        d = [np.empty(4 * cfg.H, np.float32), np.empty(cfg.H, np.float32), np.empty(4 * cfg.H, np.float32), np.empty(4, np.float32)]
        ls, lu = C.c_float(), C.c_float()
        cg, cc, cw = g.c(), cfg.c(), pw.c()
        check(self._lib.physad_fused_loss_grad_host(self._h, C.byref(cg), C.byref(cc), ptr(W1), ptr(b1), ptr(W2), ptr(b2),
                                                    C.byref(cw), C.c_float(t), C.c_float(dt), C.byref(ls), C.byref(lu),
                                                    *[ptr(x) for x in d]), "fused_loss_grad_host")
        self.cfg = cfg
        return (np.float32(ls.value), np.float32(lu.value), *d)

    # -- host-buffer forms (the reference's contract) -----------------------------------------------------
    def fused_loss_host(self, g: Grid, cfg: MLPConfig, W1, b1, W2, b2, pw: PhysWeights, t: float, dt: float,
                        want_residuals: bool = False):
        W1, b1, W2, b2 = _f32(W1), _f32(b1), _f32(W2), _f32(b2)
        R = [np.empty(g.N, np.float32) for _ in range(4)] if want_residuals else [None] * 4
        ls, lu = C.c_float(), C.c_float()
        cg, cc, cw = g.c(), cfg.c(), pw.c()
        check(self._lib.physad_fused_loss_host(self._h, C.byref(cg), C.byref(cc), ptr(W1), ptr(b1), ptr(W2), ptr(b2),
                                               C.byref(cw), C.c_float(t), C.c_float(dt), C.byref(ls), C.byref(lu),
                                               *[ptr(r) for r in R]), "fused_loss_host")
        self.cfg = cfg
        return (np.float32(ls.value), np.float32(lu.value)) + ((tuple(R),) if want_residuals else ())

    def prepare_step_host(self, g: Grid, cfg: MLPConfig, W1, b1, W2, b2, pw: PhysWeights, t: float, dt: float, slab=None):
        """One rank's whole step through the host-buffer C-ABI call (weights in, two losses out), pre-marshalled.
        With connect_peers() done the losses are global (in-kernel exchange); otherwise they are this slab's."""
        W1, b1, W2, b2 = _f32(W1), _f32(b1), _f32(W2), _f32(b2)
        cs, _ = self._slab(g, slab)
        cg, cc, cw = g.c(), cfg.c(), pw.c()
        ls, lu = C.c_float(), C.c_float()
        fn, h = self._lib.physad_fused_loss_slab_host, self._h
        args = (C.byref(cg), C.byref(cs), C.byref(cc), ptr(W1), ptr(b1), ptr(W2), ptr(b2), C.byref(cw), C.c_float(t),
                C.c_float(dt), C.c_int(1 if self._peers else 0), C.byref(ls), C.byref(lu))
        keep = (cg, cs, cc, cw, W1, b1, W2, b2)
        self.cfg = cfg

        def step(_keep=keep):
            rc = fn(h, *args)
            if rc:
                check(rc, "fused_loss_slab_host")
            return ls.value, lu.value
        return step

    def mlp_forward_host(self, x: np.ndarray) -> np.ndarray:
        x = _f32(x)
        B = x.size // self.cfg.In
        y = np.empty(B * self.cfg.Out, np.float32)
        check(self._lib.physad_mlp_forward_host(self._h, ptr(x), ptr(y), C.c_size_t(B)), "mlp_forward_host")
        return y

    def mlp_backward_host(self, x: np.ndarray, y_target: np.ndarray):
        """MSE weight gradients (dW1, db1, dW2, db2) -- mlp_backward<ExecCuda>, include/mlp.h:8-9."""
        x, y_target = _f32(x), _f32(y_target)
        c = self.cfg
        B = x.size // c.In
        dW1 = np.empty(c.H * c.In, np.float32); db1 = np.empty(c.H, np.float32)
        dW2 = np.empty(c.Out * c.H, np.float32); db2 = np.empty(c.Out, np.float32)
        check(self._lib.physad_mlp_backward_host(self._h, ptr(x), ptr(y_target), ptr(dW1), ptr(db1), ptr(dW2), ptr(db2),
                                                 C.c_size_t(B)), "mlp_backward_host")
        return dW1, db1, dW2, db2

    def mlp_grid_infer_host(self, g: Grid, t: float) -> np.ndarray:
        out = np.empty(g.N * 4, np.float32)
        cg = g.c()
        check(self._lib.physad_mlp_grid_infer_host(self._h, C.byref(cg), C.c_float(t), ptr(out)), "mlp_grid_infer_host")
        return out

    def mlp_generate_fields_host(self, g: Grid, t: float, dt: float):
        N = g.N
        s = [np.empty(N, np.float32) for _ in range(3)]
        u = [np.empty(3 * N, np.float32) for _ in range(3)]
        cg = g.c()
        check(self._lib.physad_mlp_generate_fields_host(self._h, C.byref(cg), C.c_float(t), C.c_float(dt), ptr(s[0]),
                                                        ptr(s[1]), ptr(s[2]), ptr(u[0]), ptr(u[1]), ptr(u[2])),
              "mlp_generate_fields_host")
        return s[0], s[1], s[2], u[0], u[1], u[2]

    def phys_residuals_host(self, g: Grid, fields, timed: bool = False):
        fields = [_f32(f) for f in fields]
        R = [np.empty(g.N, np.float32) for _ in range(4)]
        ms = C.c_float(-1.0)
        cg = g.c()
        check(self._lib.physad_phys_residuals_host(self._h, C.byref(cg), *[ptr(f) for f in fields], *[ptr(r) for r in R],
                                                   C.byref(ms) if timed else None), "phys_residuals_host")
        return (tuple(R), ms.value) if timed else tuple(R)

    def phys_loss_host(self, g: Grid, pw: PhysWeights, fields, want_residuals: bool = False):
        fields = [_f32(f) for f in fields]
        R = [np.empty(g.N, np.float32) for _ in range(4)] if want_residuals else [None] * 4
        ls, lu = C.c_float(), C.c_float()
        cg, cw = g.c(), pw.c()
        check(self._lib.physad_phys_loss_host(self._h, C.byref(cg), C.byref(cw), *[ptr(f) for f in fields], C.byref(ls),
                                              C.byref(lu), *[ptr(r) for r in R]), "phys_loss_host")
        return (np.float32(ls.value), np.float32(lu.value)) + ((tuple(R),) if want_residuals else ())

    def phys_backward_host(self, g: Grid, pw: PhysWeights, R):
        R = [_f32(r) for r in R]
        G = [np.empty(g.N, np.float32) for _ in range(4)]
        cg, cw = g.c(), pw.c()
        check(self._lib.physad_phys_backward_host(self._h, C.byref(cg), C.byref(cw), *[ptr(r) for r in R],
                                                  *[ptr(x) for x in G]), "phys_backward_host")
        return tuple(G)

    def phys_backward_from_fields_host(self, g: Grid, pw: PhysWeights, fields):
        fields = [_f32(f) for f in fields]
        G = [np.empty(g.N, np.float32) for _ in range(4)]
        cg, cw = g.c(), pw.c()
        check(self._lib.physad_phys_backward_from_fields_host(self._h, C.byref(cg), C.byref(cw), *[ptr(f) for f in fields],
                                                              *[ptr(x) for x in G]), "phys_backward_from_fields_host")
        return tuple(G)


def mlp_random_init(H: int, seed: int = 42, scale: float = 0.5, In: int = 4, Out: int = 4):
    """phys::mlp_random_init (reference include/mlp_grid.h:34): returns (W1, b1, W2, b2). Host only."""
    W1 = np.empty(H * In, np.float32); b1 = np.empty(H, np.float32)
    W2 = np.empty(Out * H, np.float32); b2 = np.empty(Out, np.float32)
    f = capi.lib().physad_mlp_random_init
    f.restype = None
    f(C.c_int(In), C.c_int(H), C.c_int(Out), C.c_uint(seed), C.c_float(scale), ptr(W1), ptr(b1), ptr(W2), ptr(b2))
    return W1, b1, W2, b2


def grid_input_scales(g: Grid, norm) -> np.ndarray:
    """dc/dx of the three space inputs (float32 [3]) exactly as the grid's analytic calls form them: the dcdx with which
    points of the grid's domain give the grid's physics.  norm: 1 / True = MinusOneToOne, 0 / False = ZeroToOne.
    Host-only, no GPU."""
    out = np.empty(3, np.float32)
    cg = g.c()
    check(capi.lib().physad_grid_input_scales(C.byref(cg), C.c_int(int(norm)), ptr(out)), "grid_input_scales")
    return out


# ---- reference-named host functions (one shared context, like the C++ layer) -----------------------
_CTX: Optional[Context] = None


def default_context() -> Context:
    global _CTX
    if _CTX is None:
        _CTX = Context()
    return _CTX


def mlp_infer_cuda(cfg: MLPConfig, w, coords: np.ndarray) -> np.ndarray:
    c = default_context()
    c.set_weights(cfg, *w)
    return c.mlp_forward_host(coords)


def mlp_grid_infer_cuda(g: Grid, cfg: MLPConfig, w, t: float) -> np.ndarray:
    c = default_context()
    c.set_weights(cfg, *w)
    return c.mlp_grid_infer_host(g, t)


def mlp_generate_fields_cuda(g: Grid, cfg: MLPConfig, w, t: float, dt: float):
    c = default_context()
    c.set_weights(cfg, *w)
    return c.mlp_generate_fields_host(g, t, dt)


def cuda_phys_residuals_fused(g: Grid, fields):
    return default_context().phys_residuals_host(g, fields)


cuda_phys_residuals_nonfused = cuda_phys_residuals_fused


def cuda_phys_residuals_fused_timed(g: Grid, fields):
    return default_context().phys_residuals_host(g, fields, timed=True)


def cuda_phys_loss_forward_fused(g: Grid, pw: PhysWeights, fields, want_residuals: bool = False):
    return default_context().phys_loss_host(g, pw, fields, want_residuals)


cuda_phys_loss_forward_nonfused = cuda_phys_loss_forward_fused


def cuda_phys_loss_backward_nonfused(g: Grid, pw: PhysWeights, R):
    return default_context().phys_backward_host(g, pw, R)


def cuda_phys_loss_backward_fused(g: Grid, pw: PhysWeights, fields):
    return default_context().phys_backward_from_fields_host(g, pw, fields)


def mlp_phys_loss_fused_cuda(g: Grid, cfg: MLPConfig, w, pw: PhysWeights, t: float, dt: float, want_residuals: bool = False):
    return default_context().fused_loss_host(g, cfg, *w, pw, t, dt, want_residuals)


def mlp_phys_loss_tangent_cuda(g: Grid, cfg: MLPConfig, w, pw: PhysWeights, t: float):
    """Analytic forward-mode physics loss (additive, NOT the parity path): (L_sigma, L_u) with derivatives propagated
    through the MLP instead of finite differences."""
    c = default_context()
    W1, b1, W2, b2 = (_f32(a) for a in w)
    ls, lu = C.c_float(), C.c_float()
    cg, cc, cw = g.c(), cfg.c(), pw.c()
    check(c._lib.physad_tangent_loss_host(c._h, C.byref(cg), C.byref(cc), ptr(W1), ptr(b1), ptr(W2), ptr(b2), C.byref(cw),
                                          C.c_float(t), C.byref(ls), C.byref(lu)), "tangent_loss_host")
    c.cfg = cfg
    return np.float32(ls.value), np.float32(lu.value)


def mlp_phys_loss_grad_cuda(g: Grid, cfg: MLPConfig, w, pw: PhysWeights, t: float, dt: float):
    """Closed loop (additive): losses and d(L_sigma + L_u)/d(W1, b1, W2, b2)."""
    return default_context().fused_loss_grad_host(g, cfg, *w, pw, t, dt)


def mlp_phys_loss_deep_grad_cuda(g: Grid, cfg: MLPConfig, L: int, w, pw: PhysWeights, t: float, dt: float):
    """Closed loop of a deep network (additive): w = (W1, b1, Wh, bh, W2, b2) ->
    (L_sigma, L_u, dW1, db1, dWh, dbh, dW2, db2)."""
    c = default_context()
    c.set_weights_deep(cfg, L, *w)
    return c.deep_loss_grad_host(g, pw, t, dt)


def mlp_phys_loss_tangent_grad_cuda(g: Grid, cfg: MLPConfig, w, pw: PhysWeights, t: float):
    """Closed loop of the analytic loss (additive): (L_sigma, L_u, dW1, db1, dW2, db2)."""
    return default_context().tangent_loss_grad_host(g, cfg, *w, pw, t)


def mlp_phys_loss_deep_tangent_grad_cuda(g: Grid, cfg: MLPConfig, L: int, w, pw: PhysWeights, t: float):
    """Closed loop of the analytic loss of a deep network (additive): w = (W1, b1, Wh, bh, W2, b2) ->
    (L_sigma, L_u, dW1, db1, dWh, dbh, dW2, db2)."""
    c = default_context()
    c.set_weights_deep(cfg, L, *w)
    return c.deep_tangent_loss_grad_host(g, pw, t)


def mlp_infer_deep_cuda(cfg: MLPConfig, L: int, w, coords: np.ndarray) -> np.ndarray:
    """A deep network at arbitrary points (additive): w = (W1, b1, Wh, bh, W2, b2), coords [N, 4] -> y float32 [N, 4]."""
    c = default_context()
    c.set_weights_deep(cfg, L, *w)
    return c.mlp_forward_deep_host(coords)


def mlp_data_loss_deep_grad_cuda(cfg: MLPConfig, L: int, w, x: np.ndarray, target: np.ndarray, lam=None):
    """Data-fit loss of a deep network and its gradient (additive): w = (W1, b1, Wh, bh, W2, b2) ->
    (L_d, dW1, db1, dWh, dbh, dW2, db2), L_d = mean over the points of sum_o lam[o] (y_o - target_o)^2 (lam None: 1/4 each)."""
    c = default_context()
    c.set_weights_deep(cfg, L, *w)
    return c.deep_data_loss_grad_host(x, target, lam)


def mlp_phys_loss_deep_tangent_points_grad_cuda(cfg: MLPConfig, L: int, w, x: np.ndarray, dcdx, pw: PhysWeights):
    """Analytic loss of a deep network at arbitrary points and its gradient (additive): w = (W1, b1, Wh, bh, W2, b2),
    x [B, 4] network inputs -> (L_sigma, L_u, dW1, db1, dWh, dbh, dW2, db2), the losses the mean over the points."""
    c = default_context()
    c.set_weights_deep(cfg, L, *w)
    return c.deep_tangent_points_loss_grad_host(x, dcdx, pw)
