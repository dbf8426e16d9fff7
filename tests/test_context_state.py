"""Context state: every entry point against the network the context holds, and every cache against a fresh context.

A context keeps more than its weights: which network it holds (one hidden layer, or L hidden layers from
physad_set_weights_deep), caches keyed on the geometry (coordinate tables, the fused plan), buffers that only grow, the
lazy device copy of the weights, the host-result sequence number of physad_fused_loss_slab_host, and the switches
(exact residuals, advection, deep mode).  The other GPU tests share one context and set weights right before each use,
so none of them sees a call made in a state left behind by another.  Here:

  A  every entry point x every weight state (none, one hidden layer, L = 1, L > 1, back to one layer, after a refused
     set_weights*): refused with the right status and nothing written, or equal to the CPU checker at the tolerance the
     other tests use for that call AND bitwise equal to the same call on a fresh context;
  B  one context walked through a scripted sequence of states; after every step a fixed set of probes is bitwise equal to
     a fresh context brought straight to that state (or refused the same way);
  C  physad_mlp_backward over its row limit: refused without leaking stream-ordered memory.
"""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

from helpers import max_rel_to_max
from oracle import Grid as OGrid
from test_deep_grad import DeepChecker, _deep_weights
from test_deep_tangent import TangentChecker
from test_tangent_grad import tangent_grad_ref

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
E_INVALID, E_UNSUPPORTED, E_NOWEIGHTS = -1, -2, -3
TOL_FIELD, TOL_LOSS, TOL_GRAD = 1e-5, 1e-4, 1e-4
T, DT = 0.25, 2e-3
WS, WU = 1.3, 0.7
MLP_ROWS = 300          # not a multiple of the 256-row blocks


# ---- fixtures and helpers ---------------------------------------------------------------------------------------------
def _cc(tmp_path_factory, name, src):
    out = str(tmp_path_factory.mktemp(name) / ("lib" + name + ".so"))
    subprocess.run([os.environ.get("CC", "gcc"), "-std=c11", "-O3", "-ffp-contract=off", "-fPIC", "-shared", "-o", out,
                    os.path.join(ROOT, "tests", src), "-lm"], check=True, capture_output=True)
    return out


@pytest.fixture(scope="module")
def deep_chk(tmp_path_factory):
    return DeepChecker(_cc(tmp_path_factory, "state_deepgrad", "deep_grad_checker.c"))


@pytest.fixture(scope="module")
def tan_chk(tmp_path_factory):
    return TangentChecker(_cc(tmp_path_factory, "state_deeptangent", "deep_tangent_checker.c"))


@pytest.fixture(scope="module")
def fresh():
    """Factory of new contexts, all closed at the end of the module."""
    import torch
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    from phys_autodiff_b200 import ops
    made = []

    def make():
        c = ops.Context()
        made.append(c)
        return c
    yield make
    for c in made:
        c.close()


def _same(a, b):
    """Bitwise equality of two lists of arrays (any dtype)."""
    return len(a) == len(b) and all(x.dtype == y.dtype and x.shape == y.shape and
                                    np.array_equal(x.view(np.uint8), y.view(np.uint8)) for x, y in zip(a, b))


class Result:
    def __init__(self, rc, msg, outs, untouched):
        self.rc, self.msg, self.outs, self.untouched = rc, msg, outs, untouched

    def __repr__(self):
        return f"Result(rc={self.rc}, msg={self.msg!r})"


class Call:
    """One C-ABI call with every output pre-filled with 0xFF bytes (a NaN in every float type), so a refused call can be
    checked to have written nothing."""

    def __init__(self, ctx):
        self.ctx, self.outs = ctx, []

    def dev(self, n, dtype=None):
        import torch
        t = torch.empty(n, dtype=dtype or torch.float32, device="cuda")
        t.view(torch.uint8).fill_(0xFF)
        self.outs.append(t)
        return t

    def host(self, n, dtype=np.float32):
        a = np.full(n * np.dtype(dtype).itemsize, 0xFF, np.uint8).view(dtype)
        self.outs.append(a)
        return a

    def run(self, name, *args):
        import torch
        torch.cuda.synchronize()
        return self.collect(getattr(self.ctx._lib, "physad_" + name)(self.ctx._h, *args))

    def collect(self, rc):
        import torch
        msg = self.ctx._lib.physad_last_error().decode() if rc else ""
        torch.cuda.synchronize()
        outs = []
        for o in self.outs:
            if not hasattr(o, "cpu"):
                outs.append(o.copy())
            elif o.element_size() == 2:
                outs.append(o.cpu().view(torch.int16).numpy())    # 16-bit floats: their bits
            else:
                outs.append(o.cpu().numpy())
        untouched = all((o.view(np.uint8) == 0xFF).all() for o in outs)
        return Result(rc, msg, outs, untouched)


class Case:
    """Grid, inputs and marshalled arguments shared by every probe of one (shape, H) case."""

    def __init__(self, shape, H, m1p1, periodic=True, h=(1.0, 1.0, 1.0)):
        import torch
        from phys_autodiff_b200 import Grid, PhysWeights
        self.shape, self.H, self.m1p1 = shape, H, m1p1
        self.og = OGrid(*shape, *h, 2e-3, periodic)
        self.g = Grid(*shape, *h, 2e-3, periodic)
        self.cg, self.cw = self.g.c(), PhysWeights(WS, WU).c()
        self.N = self.g.N
        rng = np.random.default_rng(H)
        self.x = rng.uniform(-1, 1, MLP_ROWS * 4).astype(np.float32)
        self.y = rng.uniform(-1, 1, MLP_ROWS * 4).astype(np.float32)
        self.xd, self.yd = torch.from_numpy(self.x).cuda(), torch.from_numpy(self.y).cuda()
        nz = shape[2]
        self.slab = (1, nz - 1) if nz > 2 else (0, nz)
        self.split = max(1, nz // 2)

    def cs(self, z0, z1):
        from phys_autodiff_b200.capi import CSlab
        s = CSlab(z0, z1)
        self._keep = getattr(self, "_keep", []) + [s]
        return C.byref(s)


def _p(x):
    from phys_autodiff_b200.capi import ptr
    return ptr(x)


def _stream():
    import torch
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


def _two(res_holder):
    """Addresses of the two float32 losses of a host form (one 2-element host output)."""
    return _p(res_holder), _p(res_holder.ctypes.data + 4)


# ---- the entry points -------------------------------------------------------------------------------------------------
# Each takes (context, Case) and returns a Result.  Host forms that can take new weights are called with cfg = NULL, so
# they run on whatever network the context holds.
def _mlp_forward_dev(ctx, k):
    c = Call(ctx)
    y = c.dev(MLP_ROWS * 4)
    return c.run("mlp_forward_dev", _p(k.xd), _p(y), C.c_size_t(MLP_ROWS), _stream())


def _mlp_forward_host(ctx, k):
    c = Call(ctx)
    y = c.host(MLP_ROWS * 4)
    return c.run("mlp_forward_host", _p(k.x), _p(y), C.c_size_t(MLP_ROWS))


def _mlp_backward_dev(ctx, k):
    c = Call(ctx)
    d = [c.dev(n) for n in (4 * k.H, k.H, 4 * k.H, 4)]
    return c.run("mlp_backward_dev", _p(k.xd), _p(k.yd), *[_p(a) for a in d], C.c_size_t(MLP_ROWS), _stream())


def _mlp_backward_host(ctx, k):
    c = Call(ctx)
    d = [c.host(n) for n in (4 * k.H, k.H, 4 * k.H, 4)]
    return c.run("mlp_backward_host", _p(k.x), _p(k.y), *[_p(a) for a in d], C.c_size_t(MLP_ROWS))


def _grid_infer_dev(ctx, k):
    c = Call(ctx)
    out = c.dev(4 * k.N)
    return c.run("mlp_grid_infer_dev", C.byref(k.cg), None, C.c_float(T), _p(out), _stream())


def _grid_infer_host(ctx, k):
    c = Call(ctx)
    out = c.host(4 * k.N)
    return c.run("mlp_grid_infer_host", C.byref(k.cg), C.c_float(T), _p(out))


def _fields_dev(ctx, k):
    c = Call(ctx)
    f = [c.dev(n * k.N) for n in (1, 1, 1, 3, 3, 3)]
    return c.run("mlp_generate_fields_dev", C.byref(k.cg), None, C.c_float(T), C.c_float(DT), *[_p(a) for a in f], _stream())


def _fields_host(ctx, k):
    c = Call(ctx)
    f = [c.host(n * k.N) for n in (1, 1, 1, 3, 3, 3)]
    return c.run("mlp_generate_fields_host", C.byref(k.cg), C.c_float(T), C.c_float(DT), *[_p(a) for a in f])


def _fields_lp_dev(ctx, k):
    import torch
    c = Call(ctx)
    f = [c.dev(n * k.N, torch.bfloat16) for n in (1, 1, 1, 3, 3, 3)]
    return c.run("mlp_generate_fields_lp_dev", C.byref(k.cg), None, C.c_float(T), C.c_float(DT), C.c_int(2),
                 *[_p(a) for a in f], _stream())


def _fused_loss_dev(ctx, k, name="fused_loss_dev"):
    import torch
    c = Call(ctx)
    acc = c.dev(2, torch.float64)
    R = [c.dev(k.N) for _ in range(4)]
    return c.run(name, C.byref(k.cg), None, C.c_float(T), C.c_float(DT), _p(acc), *[_p(r) for r in R], _stream())


def _fused_loss_allreduce_dev(ctx, k):
    return _fused_loss_dev(ctx, k, "fused_loss_allreduce_dev")


def _tangent_loss_dev(ctx, k, name="tangent_loss_dev"):
    import torch
    c = Call(ctx)
    acc = c.dev(2, torch.float64)
    R = [c.dev(k.N) for _ in range(4)]
    return c.run(name, C.byref(k.cg), None, C.c_float(T), _p(acc), *[_p(r) for r in R], _stream())


def _tangent_loss_grad_dev(ctx, k, name="tangent_loss_grad_dev", P=None):
    import torch
    c = Call(ctx)
    acc, grad = c.dev(2, torch.float64), c.dev(P or 9 * k.H + 4, torch.float64)
    return c.run(name, C.byref(k.cg), None, C.byref(k.cw), C.c_float(T), _p(acc), _p(grad), _stream())


def _fused_loss_grad_dev(ctx, k):
    import torch
    c = Call(ctx)
    acc, grad = c.dev(2, torch.float64), c.dev(9 * k.H + 4, torch.float64)
    return c.run("fused_loss_grad_dev", C.byref(k.cg), C.byref(k.cw), C.c_float(T), C.c_float(DT), _p(acc), _p(grad),
                 _stream())


def _slab_pair(ctx, k, name, P):
    """Two complementary slabs in one probe: outputs acc0, grad0, acc1, grad1."""
    import torch
    c = Call(ctx)
    bufs = [(c.dev(2, torch.float64), c.dev(P, torch.float64)) for _ in range(2)]
    rc = 0
    for (z0, z1), (acc, grad) in zip(((0, k.split), (k.split, k.shape[2])), bufs):
        rc = rc or getattr(ctx._lib, "physad_" + name)(ctx._h, C.byref(k.cg), k.cs(z0, z1), C.byref(k.cw), C.c_float(T),
                                                         C.c_float(DT), _p(acc), _p(grad), _stream())
    return c.collect(rc)


def _fused_loss_grad_slab_dev(ctx, k):
    return _slab_pair(ctx, k, "fused_loss_grad_slab_dev", 9 * k.H + 4)


NULL_W = (None, None, None, None, None)   # cfg, W1, b1, W2, b2


def _fused_loss_host(ctx, k):
    c = Call(ctx)
    l2 = c.host(2)
    R = [c.host(k.N) for _ in range(4)]
    return c.run("fused_loss_host", C.byref(k.cg), *NULL_W, C.byref(k.cw), C.c_float(T), C.c_float(DT), *_two(l2),
                 *[_p(r) for r in R])


def _fused_loss_slab_host(ctx, k, slab=None):
    c = Call(ctx)
    l2 = c.host(2)
    return c.run("fused_loss_slab_host", C.byref(k.cg), k.cs(*(slab or k.slab)), *NULL_W, C.byref(k.cw), C.c_float(T),
                 C.c_float(DT), C.c_int(0), *_two(l2))


def _tangent_loss_host(ctx, k):
    c = Call(ctx)
    l2 = c.host(2)
    return c.run("tangent_loss_host", C.byref(k.cg), *NULL_W, C.byref(k.cw), C.c_float(T), *_two(l2))


def _fused_loss_grad_host(ctx, k, name="fused_loss_grad_host", dt=True):
    c = Call(ctx)
    l2 = c.host(2)
    d = [c.host(n) for n in (4 * k.H, k.H, 4 * k.H, 4)]
    ts = (C.c_float(T), C.c_float(DT)) if dt else (C.c_float(T),)
    return c.run(name, C.byref(k.cg), *NULL_W, C.byref(k.cw), *ts, *_two(l2), *[_p(a) for a in d])


def _tangent_loss_grad_host(ctx, k):
    return _fused_loss_grad_host(ctx, k, "tangent_loss_grad_host", dt=False)


ONE_LAYER = {
    "mlp_forward_dev": _mlp_forward_dev, "mlp_forward_host": _mlp_forward_host,
    "mlp_backward_dev": _mlp_backward_dev, "mlp_backward_host": _mlp_backward_host,
    "mlp_grid_infer_dev": _grid_infer_dev, "mlp_grid_infer_host": _grid_infer_host,
    "mlp_generate_fields_dev": _fields_dev, "mlp_generate_fields_host": _fields_host,
    "mlp_generate_fields_lp_dev": _fields_lp_dev,
    "fused_loss_dev": _fused_loss_dev, "fused_loss_allreduce_dev": _fused_loss_allreduce_dev,
    "tangent_loss_dev": _tangent_loss_dev, "tangent_loss_grad_dev": _tangent_loss_grad_dev,
    "fused_loss_grad_dev": _fused_loss_grad_dev, "fused_loss_grad_slab_dev": _fused_loss_grad_slab_dev,
    "fused_loss_host": _fused_loss_host, "fused_loss_slab_host": _fused_loss_slab_host,
    "tangent_loss_host": _tangent_loss_host, "fused_loss_grad_host": _fused_loss_grad_host,
    "tangent_loss_grad_host": _tangent_loss_grad_host,
}


def _plen(H, L):
    return 9 * H + 4 + (L - 1) * (H * H + H)


def _deep_grid_infer(ctx, k):
    c = Call(ctx)
    out = c.dev(4 * k.N)
    return c.run("mlp_grid_infer_deep_dev", C.byref(k.cg), None, C.c_float(T), _p(out), _stream())


def _deep_fields(ctx, k):
    c = Call(ctx)
    f = [c.dev(n * k.N) for n in (1, 1, 1, 3, 3, 3)]
    return c.run("mlp_generate_fields_deep_dev", C.byref(k.cg), None, C.c_float(T), C.c_float(DT), *[_p(a) for a in f],
                 _stream())


def _deep_loss_host(ctx, k):
    c = Call(ctx)
    l2 = c.host(2)
    return c.run("deep_loss_host", C.byref(k.cg), C.byref(k.cw), C.c_float(T), C.c_float(DT), *_two(l2))


def _deep_loss_grad_dev(ctx, k):
    import torch
    c = Call(ctx)
    acc, grad = c.dev(2, torch.float64), c.dev(_plen(k.H, k.L), torch.float64)
    return c.run("deep_loss_grad_dev", C.byref(k.cg), None, C.byref(k.cw), C.c_float(T), C.c_float(DT), _p(acc), _p(grad),
                 _stream())


def _deep_loss_grad_slab_dev(ctx, k):
    return _slab_pair(ctx, k, "deep_loss_grad_dev", _plen(k.H, k.L))


def _deep_host_grad(ctx, k, name, dt):
    c = Call(ctx)
    l2 = c.host(2)
    H, nl = k.H, k.L - 1
    d = [c.host(n) for n in (4 * H, H, nl * H * H, nl * H, 4 * H, 4)]
    ts = (C.c_float(T), C.c_float(DT)) if dt else (C.c_float(T),)
    return c.run(name, C.byref(k.cg), C.byref(k.cw), *ts, *_two(l2), *[_p(a) if a.size else None for a in d])


def _deep_loss_grad_host(ctx, k):
    return _deep_host_grad(ctx, k, "deep_loss_grad_host", True)


def _deep_tangent_loss_dev(ctx, k):
    return _tangent_loss_dev(ctx, k, "deep_tangent_loss_dev")


def _deep_tangent_loss_grad_dev(ctx, k):
    return _tangent_loss_grad_dev(ctx, k, "deep_tangent_loss_grad_dev", _plen(k.H, k.L))


def _deep_tangent_loss_grad_host(ctx, k):
    return _deep_host_grad(ctx, k, "deep_tangent_loss_grad_host", False)


# deep entry point -> its one-hidden-layer twin (bit-identical at L = 1, as documented) or None
DEEP = {
    "mlp_grid_infer_deep_dev": (_deep_grid_infer, "mlp_grid_infer_dev"),
    "mlp_generate_fields_deep_dev": (_deep_fields, "mlp_generate_fields_dev"),
    "deep_loss_host": (_deep_loss_host, None),
    "deep_loss_grad_dev": (_deep_loss_grad_dev, "fused_loss_grad_dev"),
    "deep_loss_grad_dev[slabs]": (_deep_loss_grad_slab_dev, "fused_loss_grad_slab_dev"),
    "deep_loss_grad_host": (_deep_loss_grad_host, "fused_loss_grad_host"),
    "deep_tangent_loss_dev": (_deep_tangent_loss_dev, "tangent_loss_dev"),
    "deep_tangent_loss_grad_dev": (_deep_tangent_loss_grad_dev, "tangent_loss_grad_dev"),
    "deep_tangent_loss_grad_host": (_deep_tangent_loss_grad_host, "tangent_loss_grad_host"),
}


# ---- CPU checks of a call that worked ---------------------------------------------------------------------------------
def _fields_of(y, N):
    """Six field arrays of three AoS [N, 4] network outputs (t - dt, t, t + dt)."""
    y = [a.reshape(N, 4) for a in y]
    return [a[:, 0].copy() for a in y] + [np.concatenate([a[:, 1], a[:, 2], a[:, 3]]) for a in y]


def _slices():
    t = np.float32(T)
    return float(t - np.float32(DT)), float(t), float(t + np.float32(DT))


def _one_layer_check(name, r, k, w, port):
    """r: a Result of one-hidden-layer entry point `name` for the weights w = (W1, b1, W2, b2); asserts the checker's
    answer at the tolerance the other tests use for the same call."""
    import torch
    og, H, N, m1p1 = k.og, k.H, k.N, k.m1p1
    o = r.outs
    if name.startswith("mlp_forward"):
        assert _same([o[0]], [port.mlp_forward(k.x, *w, MLP_ROWS, 4, H, 4)])
    elif name.startswith("mlp_backward"):
        assert _same(o, list(port.mlp_backward(k.x, k.y, *w, MLP_ROWS, 4, H, 4)))
    elif name.startswith("mlp_grid_infer"):
        assert _same([o[0]], [port.mlp_grid_infer(og, w, T, m1p1)])
    elif name in ("mlp_generate_fields_dev", "mlp_generate_fields_host"):
        assert _same(o, list(port.generate_fields(og, w, T, DT, m1p1)))
    elif name == "mlp_generate_fields_lp_dev":
        want = [torch.from_numpy(f).to(torch.bfloat16).view(torch.int16).numpy() for f in port.generate_fields(og, w, T, DT, m1p1)]
        assert _same(o, want)
    elif name in ("fused_loss_dev", "fused_loss_host"):
        want = port.fused_loss(og, w, T, DT, WS, WU, m1p1, want_residuals=True)
        for a, b in zip(o[-4:], want["R"]):
            assert max_rel_to_max(a, b) <= TOL_FIELD
        if name == "fused_loss_dev":
            got = (o[0][0], o[0][1]), (want["acc_sigma"], want["acc_u"])
        else:
            got = (o[0][0], o[0][1]), (want["loss_sigma"], want["loss_u"])
        for a, b in zip(*got):
            assert abs(a - b) <= TOL_LOSS * abs(b) + 1e-30, (a, b)
    elif name == "fused_loss_slab_host":
        want = port.fused_loss(og, w, T, DT, WS, WU, m1p1, want_residuals=True)
        pl = og.nx * og.ny
        sl = slice(k.slab[0] * pl, k.slab[1] * pl)
        acc = [float(np.sum(want["R"][0][sl].astype(np.float64) ** 2)),
               float(sum(np.sum(want["R"][j][sl].astype(np.float64) ** 2) for j in (1, 2, 3)))]
        for a, b in zip(o[0], (WS * acc[0] / N, WU * acc[1] / N)):
            assert abs(a - b) <= TOL_LOSS * abs(b) + 1e-30, (a, b)
    elif name in ("tangent_loss_dev", "tangent_loss_host"):
        want = port.tangent_loss(og, w, T, m1p1, want_residuals=True)
        if name == "tangent_loss_dev":
            for a, b in zip(o[1:], want["R"]):
                assert max_rel_to_max(a, b) <= TOL_FIELD
            ref = (want["acc_sigma"], want["acc_u"])
            tol = 1e-6
        else:
            ref = (WS * want["acc_sigma"] / N, WU * want["acc_u"] / N)
            tol = 1e-5
        for a, b in zip(o[0], ref):
            assert abs(a - b) <= tol * abs(b) + 1e-30, (a, b)
    elif name.startswith("tangent_loss_grad"):
        want = tangent_grad_ref(og, np.concatenate([np.asarray(a, np.float64) for a in w]), H, T, WS, WU, m1p1)
        grad = o[1] if name.endswith("_dev") else np.concatenate(o[1:]).astype(np.float64)
        assert np.abs(grad - want["grad"]).max() <= TOL_GRAD * np.abs(want["grad"]).max()
        ref = (want["acc_sigma"], want["acc_u"]) if name.endswith("_dev") else (want["loss_sigma"], want["loss_u"])
        for a, b in zip(o[0], ref):
            assert abs(a - b) <= 1e-5 * abs(b) + 1e-30, (a, b)
    elif name.startswith("fused_loss_grad"):
        want = port.phys_loss_grad(og, w, T, DT, WS, WU, m1p1)
        if name == "fused_loss_grad_slab_dev":
            acc, grad = o[0] + o[2], o[1] + o[3]
        elif name == "fused_loss_grad_dev":
            acc, grad = o[0], o[1]
        else:
            acc, grad = None, np.concatenate(o[1:]).astype(np.float64)
        assert np.abs(grad - want["grad"]).max() <= TOL_GRAD * np.abs(want["grad"]).max()
        ls, lu = (WS * acc[0] / N, WU * acc[1] / N) if acc is not None else o[0]
        assert abs(ls - want["loss_sigma"]) <= TOL_LOSS * want["loss_sigma"]
        assert abs(lu - want["loss_u"]) <= TOL_LOSS * want["loss_u"]
    else:
        raise AssertionError(name)


def _deep_check(name, r, k, w, port, deep_chk, tan_chk):
    """The same for a deep entry point and deep weights w = (W1, b1, Wh, bh, W2, b2) of k.L hidden layers."""
    og, H, L, N, m1p1 = k.og, k.H, k.L, k.N, k.m1p1
    o = r.outs
    if name in ("mlp_grid_infer_deep_dev", "mlp_generate_fields_deep_dev", "deep_loss_host"):
        ys = [port.mlp_grid_infer_deep(og, H, L, *w, t, m1p1) for t in _slices()]
        if name == "mlp_grid_infer_deep_dev":
            assert _same([o[0]], [ys[1]])
        elif name == "mlp_generate_fields_deep_dev":
            assert _same(o, _fields_of(ys, N))
        else:
            want = port.phys_loss_forward(og, WS, WU, _fields_of(ys, N))
            for a, b in zip(o[0], want):
                assert abs(a - b) <= TOL_LOSS * abs(b) + 1e-30, (a, b)
    elif name.startswith("deep_loss_grad"):
        want = deep_chk.phys_loss_grad_deep(og, H, L, w, T, DT, WS, WU, m1p1)
        if name == "deep_loss_grad_dev[slabs]":
            acc, grad = o[0] + o[2], o[1] + o[3]
        elif name == "deep_loss_grad_dev":
            acc, grad = o[0], o[1]
        else:
            acc, grad = None, np.concatenate(o[1:]).astype(np.float64)
        assert np.abs(grad - want["grad"]).max() <= TOL_GRAD * np.abs(want["grad"]).max()
        ls, lu = (WS * acc[0] / N, WU * acc[1] / N) if acc is not None else o[0]
        assert abs(ls - want["loss_sigma"]) <= TOL_LOSS * want["loss_sigma"]
        assert abs(lu - want["loss_u"]) <= TOL_LOSS * want["loss_u"]
    elif name.startswith("deep_tangent"):
        theta = np.concatenate([np.asarray(a, np.float64).ravel() for a in w if a is not None])
        want = tan_chk.loss_grad(og, H, L, theta, T, WS, WU, m1p1)
        if name == "deep_tangent_loss_dev":
            rmax = max(np.abs(a).max() for a in want["R"])
            for a, b in zip(o[1:], want["R"]):
                assert np.abs(a - b).max() <= TOL_FIELD * rmax
        else:
            grad = o[1] if name.endswith("_dev") else np.concatenate(o[1:]).astype(np.float64)
            assert np.abs(grad - want["grad"]).max() <= TOL_GRAD * np.abs(want["grad"]).max()
        ref = (want["acc_sigma"], want["acc_u"]) if name.endswith("_dev") else (want["loss_sigma"], want["loss_u"])
        tol = 1e-6 if name.endswith("_dev") else 1e-5     # the host form's losses are rounded to float
        for a, b in zip(o[0], ref):
            assert abs(a - b) <= tol * abs(b) + 1e-30, (a, b)
    else:
        raise AssertionError(name)


# ---- part A: entry point x weight state --------------------------------------------------------------------------------
# (H, shape, ZeroToOne/MinusOneToOne, periodic); 48 is a padded width, which only the one-hidden-layer paths take
A_CASES = [(32, (33, 18, 7), True, True), (64, (20, 9, 4), False, False), (128, (33, 18, 7), False, True),
           (48, (20, 9, 4), True, True)]
DEEP_L = {32: 3, 64: 2, 128: 4}          # L > 1 per width
OTHER_H = {32: 64, 64: 128, 128: 32}     # the width set_weights switches back to


def _cfg(H, m1p1):
    from phys_autodiff_b200 import MLPConfig
    return MLPConfig(4, H, 4, m1p1)


def _case(H, shape, m1p1, per, L=1):
    k = Case(shape, H, m1p1, per)
    k.L = L
    return k


def _one_w(port, H, seed=777):
    return port.mlp_random_init(H, seed, 0.25)


_FRESH_ONE = {}


def _fresh_one(fresh, port, name, H, shape, m1p1, per, seed=777):
    """`name` on a new context given only set_weights(H): the reference row of every comparison (cached)."""
    key = (name, H, shape, m1p1, per, seed)
    if key not in _FRESH_ONE:
        c = fresh()
        c.set_weights(_cfg(H, m1p1), *_one_w(port, H, seed))
        r = ONE_LAYER[name](c, _case(H, shape, m1p1, per))
        assert r.rc == 0 or (name == "fused_loss_allreduce_dev" and r.rc == E_INVALID), (name, r)
        _FRESH_ONE[key] = r
        c.close()
    return _FRESH_ONE[key]


def _expect_works(name, r, ref):
    """A one-hidden-layer call that must run: bitwise the fresh context's result.  The in-kernel all-reduce has no peers
    on one process, so it must fail on that (and not on the network) instead."""
    if name == "fused_loss_allreduce_dev":
        assert r.rc == E_INVALID and "xchg_connect" in r.msg and r.untouched, r
        return
    assert r.rc == 0, (name, r)
    assert _same(r.outs, ref.outs), name


@pytest.mark.parametrize("name", list(ONE_LAYER) + list(DEEP))
def test_no_weights_is_refused(fresh, name):
    c = fresh()
    fn = ONE_LAYER[name] if name in ONE_LAYER else DEEP[name][0]
    k = _case(32, (20, 9, 4), True, True)
    r = fn(c, k)
    assert r.rc == E_NOWEIGHTS and r.untouched, r


@pytest.mark.parametrize("name", list(ONE_LAYER))
def test_one_hidden_layer_network(fresh, port, name):
    """set_weights(H): the call matches its checker and a second fresh context bit for bit."""
    for H, shape, m1p1, per in A_CASES:
        ref = _fresh_one(fresh, port, name, H, shape, m1p1, per)
        c = fresh()
        c.set_weights(_cfg(H, m1p1), *_one_w(port, H))
        r = ONE_LAYER[name](c, _case(H, shape, m1p1, per))
        _expect_works(name, r, ref)
        if name != "fused_loss_allreduce_dev":
            _one_layer_check(name, r, _case(H, shape, m1p1, per), _one_w(port, H), port)
        c.close()


@pytest.mark.parametrize("name", list(DEEP))
def test_deep_calls_refuse_a_one_hidden_layer_network(fresh, port, name):
    c = fresh()
    c.set_weights(_cfg(64, True), *_one_w(port, 64))
    r = DEEP[name][0](c, _case(64, (20, 9, 4), True, True))
    assert r.rc == E_NOWEIGHTS and r.untouched, r


@pytest.mark.parametrize("name", list(ONE_LAYER) + list(DEEP))
def test_deep_network_of_one_hidden_layer(fresh, port, name):
    """set_weights_deep(H, 1) is set_weights(H): every one-hidden-layer call bitwise as there, every deep call bitwise its
    one-hidden-layer twin (and its checker where it has no twin)."""
    for H, shape, m1p1, per in A_CASES[:3]:
        W1, b1, W2, b2 = _one_w(port, H)
        c = fresh()
        c.set_weights_deep(_cfg(H, m1p1), 1, W1, b1, None, None, W2, b2)
        k = _case(H, shape, m1p1, per, L=1)
        if name in ONE_LAYER:
            _expect_works(name, ONE_LAYER[name](c, k), _fresh_one(fresh, port, name, H, shape, m1p1, per))
        else:
            fn, twin = DEEP[name]
            r = fn(c, k)
            assert r.rc == 0, r
            if twin is None:
                _deep_check(name, r, k, (W1, b1, None, None, W2, b2), port, None, None)
            else:
                ref = _fresh_one(fresh, port, twin, H, shape, m1p1, per)
                assert _same([a for a in r.outs if a.size], ref.outs), name
        c.close()


@pytest.mark.parametrize("name", list(ONE_LAYER))
def test_one_hidden_layer_call_refuses_a_deeper_network(fresh, port, name):
    """set_weights_deep(H, L > 1): the call would otherwise evaluate 4 -> H -> 4 built from the first and last layers."""
    for H, shape, m1p1, per in A_CASES[:3]:
        L = DEEP_L[H]
        c = fresh()
        c.set_weights_deep(_cfg(H, m1p1), L, *_deep_weights(H, L, 777, 0.25, port))
        r = ONE_LAYER[name](c, _case(H, shape, m1p1, per, L))
        assert r.rc == E_UNSUPPORTED and "one-hidden-layer" in r.msg, (H, L, r)
        assert r.untouched, (H, L, "a refused call wrote its outputs")
        c.close()


@pytest.mark.parametrize("name", list(DEEP))
def test_deep_call_on_a_deeper_network(fresh, port, deep_chk, tan_chk, name):
    """set_weights_deep(H, L > 1): every deep call matches its checker and a fresh context bit for bit."""
    for H, shape, m1p1, per in A_CASES[:3]:
        L = DEEP_L[H]
        w = _deep_weights(H, L, 777, 0.25, port)
        rs = []
        for _ in range(2):
            c = fresh()
            c.set_weights_deep(_cfg(H, m1p1), L, *w)
            rs.append(DEEP[name][0](c, _case(H, shape, m1p1, per, L)))
            c.close()
        assert rs[0].rc == 0 and rs[1].rc == 0, rs
        assert _same(rs[0].outs, rs[1].outs), name
        _deep_check(name, rs[0], _case(H, shape, m1p1, per, L), w, port, deep_chk, tan_chk)


@pytest.mark.parametrize("name", list(ONE_LAYER) + list(DEEP))
def test_set_weights_after_a_deeper_network(fresh, port, name):
    """set_weights_deep(H, L > 1) then set_weights(H'): the context is a fresh one given only set_weights(H')."""
    for H, shape, m1p1, per in A_CASES[:3]:
        L, H2 = DEEP_L[H], OTHER_H[H]
        c = fresh()
        c.set_weights_deep(_cfg(H, m1p1), L, *_deep_weights(H, L, 777, 0.25, port))
        k = _case(H, shape, m1p1, per, L)
        pre = (ONE_LAYER[name] if name in ONE_LAYER else DEEP[name][0])(c, k)   # leaves its caches behind
        c.set_weights(_cfg(H2, m1p1), *_one_w(port, H2, 5))
        assert c.hidden_layers is None
        k2 = _case(H2, shape, m1p1, per)
        if name in ONE_LAYER:
            assert pre.rc == E_UNSUPPORTED
            _expect_works(name, ONE_LAYER[name](c, k2), _fresh_one(fresh, port, name, H2, shape, m1p1, per, 5))
        else:
            assert pre.rc == 0
            r = DEEP[name][0](c, k2)
            assert r.rc == E_NOWEIGHTS and r.untouched, r
        c.close()


def _all_probes(c, k):
    out = {n: fn(c, k) for n, fn in ONE_LAYER.items()}
    out.update({n: fn(c, k) for n, (fn, _) in DEEP.items()})
    return out


@pytest.mark.parametrize("H", [32, 64, 128])
def test_refused_set_weights_keep_the_network(fresh, port, H):
    """A refused set_weights_deep (H = 48, L = 17, null Wh) or set_weights (norm = 2) changes nothing: every entry point
    gives, bit for bit, what it gave before (refusals included), and Context mirrors the C state."""
    from phys_autodiff_b200 import MLPConfig, PhysadError
    from phys_autodiff_b200.capi import CMlpConfig
    _, shape, m1p1, per = next(a for a in A_CASES if a[0] == H)
    L = DEEP_L[H]
    c = fresh()
    w = _deep_weights(H, L, 777, 0.25, port)
    c.set_weights_deep(_cfg(H, m1p1), L, *w)
    k = _case(H, shape, m1p1, per, L)
    before = _all_probes(c, k)
    assert all(before[n].rc == E_UNSUPPORTED for n in ONE_LAYER) and all(before[n].rc == 0 for n in DEEP)
    W1, b1, W2, b2 = _one_w(port, 48)
    bad = CMlpConfig(4, 48, 4, 1)
    rc = c._lib.physad_set_weights_deep(c._h, C.byref(bad), C.c_int(17), _p(W1), _p(b1), None, None, _p(W2), _p(b2))
    assert rc != 0
    with pytest.raises(PhysadError):
        c.set_weights_deep(MLPConfig(4, 48, 4, True), 17, W1, b1, np.zeros(16 * 48 * 48, np.float32),
                           np.zeros(16 * 48, np.float32), W2, b2)
    assert c.hidden_layers == L and c.cfg == _cfg(H, m1p1)
    with pytest.raises(PhysadError, match="norm"):
        c.set_weights(MLPConfig(4, H, 4, 2), *_one_w(port, H, 9))
    assert c.hidden_layers == L and c.cfg == _cfg(H, m1p1)
    after = _all_probes(c, k)
    for n in before:
        assert before[n].rc == after[n].rc and _same(before[n].outs, after[n].outs), n


# ---- part B: one context through a sequence of states, against fresh contexts ------------------------------------------
class State:
    def __init__(self, grid, m1p1=True, net=None, mode=0, exact=0, adv=0):
        self.grid, self.m1p1, self.net, self.mode, self.exact, self.adv = grid, m1p1, net, mode, exact, adv

    def but(self, **kw):
        s = State(self.grid, self.m1p1, self.net, self.mode, self.exact, self.adv)
        for a, v in kw.items():
            setattr(s, a, v)
        return s

    @property
    def H(self):
        return self.net[1] if self.net else 32

    @property
    def L(self):
        return self.net[2] if self.net and self.net[0] == "deep" else 1


def _weights(port, net):
    if net[0] == "one":
        return _one_w(port, net[1], net[2])
    return _deep_weights(net[1], net[2], net[3], 0.25, port)


def _apply(c, port, st, prev=None):
    """Bring context c from state `prev` (None: a new context) to `st`, touching only what differs."""
    if st.net is not None and (prev is None or st.net != prev.net or st.m1p1 != prev.m1p1):
        if st.net[0] == "one":
            c.set_weights(_cfg(st.H, st.m1p1), *_weights(port, st.net))
        else:
            c.set_weights_deep(_cfg(st.H, st.m1p1), st.L, *_weights(port, st.net))
    if prev is None or st.mode != prev.mode:
        c.set_deep_mode(st.mode)
    if prev is None or st.exact != prev.exact:
        c.set_exact_residuals(bool(st.exact))
    if prev is None or st.adv != prev.adv:
        c.set_advection(bool(st.adv))


def _probe(c, st):
    """The fixed probe set of part B: {name: ("rc", status) or list of bitwise-comparable arrays}."""
    from phys_autodiff_b200 import Grid, PhysadError, PhysWeights
    g = Grid(*st.grid, 1.0, 1.0, 1.0, 2e-3, True)
    pw = PhysWeights(WS, WU)
    nz = st.grid[2]
    out = {}

    def run(name, fn):
        try:
            r = fn()
            out[name] = [x.cpu().numpy() for x in (r if isinstance(r, tuple) else (r,))]
        except PhysadError:
            out[name] = ("refused", c._lib.physad_last_error().decode())

    run("grid_infer", lambda: c.mlp_grid_infer(g, T))
    run("fused_whole", lambda: c.fused_loss_acc(g, T, DT))
    run("fused_slab", lambda: c.fused_loss_acc(g, T, DT, slab=(1, nz - 1)))
    run("fused_whole_again", lambda: c.fused_loss_acc(g, T, DT))
    run("tangent", lambda: c.tangent_loss_acc(g, T))
    run("fused_grad", lambda: c.fused_loss_grad_acc(g, pw, T, DT))
    run("deep_grad", lambda: c.deep_loss_grad_acc(g, pw, T, DT))
    run("deep_tangent_grad", lambda: c.deep_tangent_loss_grad_acc(g, pw, T))
    for mode in (0, 1):
        c.set_deep_mode(mode)
        run(f"grid_infer_deep_mode{mode}", lambda: c.mlp_grid_infer_deep(g, T))
    c.set_deep_mode(st.mode)
    return out


ONE_PROBES = ("grid_infer", "fused_whole", "fused_slab", "fused_whole_again", "tangent", "fused_grad")
DEEP_PROBES = ("deep_grad", "deep_tangent_grad", "grid_infer_deep_mode0", "grid_infer_deep_mode1")


def _compare(label, got, want, st):
    for n in want:
        a, b = got[n], want[n]
        if isinstance(b, tuple):
            assert a == b, (label, n, a, b)
        else:
            assert not isinstance(a, tuple) and _same(a, b), (label, n, a if isinstance(a, tuple) else "differs")
    # what does not apply to the state is refused
    if st.net is None:
        assert all(isinstance(got[n], tuple) for n in got), label
    elif st.L > 1:
        assert all(isinstance(got[n], tuple) for n in ONE_PROBES), label
    else:
        if st.net[0] == "one":
            assert all(isinstance(got[n], tuple) for n in DEEP_PROBES), label
        if st.adv == 0:
            assert all(not isinstance(got[n], tuple) for n in ONE_PROBES), label
    if not isinstance(got["fused_whole"], tuple):
        assert _same(got["fused_whole"], got["fused_whole_again"]), label


def _mlp_forward_action(c, f, port, st):
    """mlp_forward -> set_weights -> mlp_forward: the lazy device copy of the weights must follow the new weights."""
    import torch
    x = torch.from_numpy(np.random.default_rng(3).uniform(-1, 1, (MLP_ROWS, 4)).astype(np.float32)).cuda()
    y0 = c.mlp_forward(x).cpu().numpy()
    _apply(c, port, st, State(st.grid))                              # the new weights
    y1 = c.mlp_forward(x).cpu().numpy()
    _apply(f, port, st)
    assert _same([y1], [f.mlp_forward(x).cpu().numpy()])
    assert _same([y1.reshape(-1)], [port.mlp_forward(x.cpu().numpy(), *_weights(port, st.net), MLP_ROWS, 4, st.H, 4)])
    assert not _same([y0], [y1])


def _slab_host_action(c, f, port, st):
    """fused_loss_slab_host alternating with fused_loss_dev, and a refused slab_host before a working one: the host-result
    sequence number never waits for a launch that did not happen."""
    from phys_autodiff_b200 import Grid, PhysadError, PhysWeights
    g = Grid(*st.grid, 1.0, 1.0, 1.0, 2e-3, True)
    pw = PhysWeights(WS, WU)
    W1, b1, W2, b2 = _weights(port, st.net)
    cfg = _cfg(st.H, st.m1p1)
    nz = st.grid[2]
    _apply(f, port, st)
    res = []
    for ctx in (c, f):
        step = ctx.prepare_step_host(g, cfg, W1, b1, W2, b2, pw, T, DT, slab=(1, nz - 1))
        a = step()
        acc = ctx.fused_loss_acc(g, T, DT, slab=(1, nz - 1)).cpu().numpy()
        b = step()
        bad = ctx.prepare_step_host(g, cfg, W1, b1, W2, b2, pw, T, DT, slab=(5, 3))
        with pytest.raises(PhysadError, match="slab"):
            bad()
        d = step()
        fin = ctx.finalize(acc, pw, g.N)
        assert a == b == d and (np.float32(a[0]), np.float32(a[1])) == fin
        res.append(a)
    assert res[0] == res[1]


def _refusals_action(c, f, port, st):
    """Refused calls (bad slab, no deep weights, one-hidden-layer call on a deep network) leave nothing behind."""
    from phys_autodiff_b200 import Grid, PhysadError, PhysWeights
    g = Grid(*st.grid, 1.0, 1.0, 1.0, 2e-3, True)
    pw = PhysWeights(WS, WU)
    with pytest.raises(PhysadError, match="slab"):
        c.fused_loss_acc(g, T, DT, slab=(3, 2)) if st.L == 1 else c.deep_loss_grad_acc(g, pw, T, DT, slab=(3, 2))
    if st.L == 1:
        with pytest.raises(PhysadError, match="set_weights_deep"):
            c.deep_loss_grad_acc(g, pw, T, DT)
    else:
        with pytest.raises(PhysadError, match="one-hidden-layer"):
            c.fused_loss_grad_acc(g, pw, T, DT)
        with pytest.raises(PhysadError, match="one-hidden-layer"):
            c.mlp_grid_infer(g, T)
    _apply(f, port, st)


S0 = State((33, 18, 7), True, ("one", 64, 1))
STEPS = [
    ("one layer", S0, None),
    ("same nx+ny+nz, other extents", S0.but(grid=(20, 9, 29)), None),
    ("norm flip", S0.but(grid=(20, 9, 29), m1p1=False), None),
    ("large deep call", State((96, 64, 24), True, ("deep", 128, 6, 2)), None),
    ("small deep call", State((20, 9, 4), True, ("deep", 32, 2, 3)), None),
    ("large again", State((96, 64, 24), True, ("deep", 64, 3, 4)), None),
    ("tensor-core mode", State((96, 64, 24), True, ("deep", 64, 3, 4), mode=1), None),
    ("narrower in mode 1", State((33, 18, 7), False, ("deep", 32, 2, 3), mode=1), None),
    ("deep refusals", State((33, 18, 7), False, ("deep", 64, 3, 5)), _refusals_action),
    ("back to one layer", State((33, 18, 7), True, ("one", 32, 2)), None),
    ("exact residuals on", State((33, 18, 7), True, ("one", 32, 2), exact=1), None),
    ("exact residuals off", State((33, 18, 7), True, ("one", 32, 2)), None),
    ("upwind on", State((33, 18, 7), True, ("one", 32, 2), adv=1), None),
    ("upwind off", State((33, 18, 7), True, ("one", 32, 2)), None),
    ("mlp_forward around set_weights", State((20, 9, 4), True, ("one", 128, 3)), _mlp_forward_action),
    ("slab host form", State((33, 18, 7), True, ("one", 128, 3)), _slab_host_action),
    ("one-layer refusals", State((33, 18, 7), True, ("one", 128, 3)), _refusals_action),
    ("deep after all that", State((20, 9, 29), False, ("deep", 128, 4, 6)), None),
]


def test_state_sequence_matches_fresh_contexts(fresh, port):
    c = fresh()
    prev = None
    for label, st, action in STEPS:
        f = fresh()
        if action is None:
            _apply(c, port, st, prev)
            _apply(f, port, st)
        else:
            _apply(c, port, st.but(net=prev.net if action is _mlp_forward_action else st.net), prev)
            action(c, f, port, st)
        _compare(label, _probe(c, st), _probe(f, st), st)
        f.close()
        prev = st


# ---- part C: mlp_backward over its row limit -------------------------------------------------------------------------
def _cudart():
    """The CUDA runtime library torch loaded (stream-ordered allocations come from the device's default pool, which is
    the same for every runtime in the process)."""
    import torch
    torch.cuda.init()
    with open("/proc/self/maps") as fh:
        paths = sorted({ln.split()[-1] for ln in fh if "libcudart.so" in ln})
    return C.CDLL(paths[0] if paths else "libcudart.so.12")


def _pool_used(rt):
    import torch
    torch.cuda.synchronize()
    pool = C.c_void_p()
    assert rt.cudaDeviceGetDefaultMemPool(C.byref(pool), C.c_int(torch.cuda.current_device())) == 0
    v = C.c_uint64()
    assert rt.cudaMemPoolGetAttribute(pool, C.c_int(7), C.byref(v)) == 0    # cudaMemPoolAttrUsedMemCurrent
    return v.value


def test_mlp_backward_over_the_row_limit(fresh, port):
    """B = 65535 * 64 + 1 rows is refused before any stream-ordered allocation, in both forms, and the context then
    still gives the reference's gradients bit for bit."""
    import torch
    rt = _cudart()
    c = fresh()
    H = 8
    w = port.mlp_random_init(H, 777, 0.25)
    c.set_weights(_cfg(H, True), *w)
    B = 65535 * 64 + 1
    x = torch.zeros(B * 4, device="cuda")
    y = torch.zeros(B * 4, device="cuda")
    d = [torch.full((n,), float("nan"), device="cuda") for n in (4 * H, H, 4 * H, 4)]
    used = _pool_used(rt)
    rc = c._lib.physad_mlp_backward_dev(c._h, _p(x), _p(y), *[_p(a) for a in d], C.c_size_t(B), _stream())
    assert rc == E_UNSUPPORTED
    assert _pool_used(rt) == used
    assert all(torch.isnan(a).all() for a in d)
    del x, y
    xh = np.zeros(B * 4, np.float32)
    dh = [np.full(n, np.nan, np.float32) for n in (4 * H, H, 4 * H, 4)]
    rc = c._lib.physad_mlp_backward_host(c._h, _p(xh), _p(xh), *[_p(a) for a in dh], C.c_size_t(B))
    assert rc == E_UNSUPPORTED
    assert _pool_used(rt) == used
    assert all(np.isnan(a).all() for a in dh)
    k = _case(H, (20, 9, 4), True, True)
    want = list(port.mlp_backward(k.x, k.y, *w, MLP_ROWS, 4, H, 4))
    for fn in (_mlp_backward_dev, _mlp_backward_host):
        r = fn(c, k)
        assert r.rc == 0 and _same(r.outs, want)
