"""Analytic (forward-mode) physics loss of deeper networks and its gradient with respect to every layer's weights.

The checker is tests/deep_tangent_checker.c, compiled here into a temporary library.
CPU tier: the checker's all-double gradient against central finite differences of its all-double loss, its Jacobian
against central differences of the network, its kernel-faithful value outputs against oracle_mlp_grid_infer_deep, L = 1
against oracle_tangent_loss, and the kernels' SASS and spills.  GPU tier: k_deep_tangent against the kernel-faithful
checker (sums, residuals, gradient), the bitwise properties, slabs, L = 1, error paths, training and a torchrun
comparison across GPUs."""
import ctypes as C
import json
import os
import re
import shutil
import subprocess
import sys

import numpy as np
import pytest

from helpers import assert_grad_close
from oracle import Grid as OGrid

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
TOL_GRAD = 1e-4


def _dp(a):
    return a.ctypes.data_as(C.POINTER(C.c_double))


def _plen(H, L):
    return 9 * H + 4 + (L - 1) * (H * H + H)


class TangentChecker:
    """ctypes surface of tests/deep_tangent_checker.c (-O3 -ffp-contract=off, as the oracle port)."""

    def __init__(self, path):
        self.lib = C.CDLL(path)
        self.lib.oracle_deep_tangent_loss_grad.restype = C.c_int
        self.lib.oracle_deep_tangent_point.restype = None

    def loss_grad(self, g, H, L, theta, t, w_sigma=1.0, w_u=1.0, m1p1=True, all_double=False, grad=True):
        """theta[P] (gradient layout) -> dict(acc_sigma, acc_u, loss_sigma, loss_u, R (4 x N f32), Y (N x 4 f32), grad)."""
        theta = np.ascontiguousarray(theta, np.float64)
        assert theta.size == _plen(H, L)
        a_s, a_u = C.c_double(), C.c_double()
        R = [np.empty(g.N, np.float32) for _ in range(4)]
        Y = np.empty(g.N * 4, np.float32)
        gr = np.empty(theta.size, np.float64) if grad else None
        fp = lambda a: a.ctypes.data_as(C.POINTER(C.c_float))
        rc = self.lib.oracle_deep_tangent_loss_grad(C.byref(g.c()), C.c_int(H), C.c_int(L), C.c_int(int(m1p1)), _dp(theta),
                                                    C.c_float(t), C.c_float(w_sigma), C.c_float(w_u), C.c_int(int(all_double)),
                                                    C.byref(a_s), C.byref(a_u), *[fp(r) for r in R], fp(Y),
                                                    _dp(gr) if grad else None)
        assert rc == 0
        N = g.N
        return dict(acc_sigma=a_s.value, acc_u=a_u.value, loss_sigma=w_sigma * a_s.value / N, loss_u=w_u * a_u.value / N,
                    R=R, Y=Y.reshape(N, 4), grad=gr)

    def point(self, H, L, theta, c, all_double=True):
        theta = np.ascontiguousarray(theta, np.float64)
        c = np.ascontiguousarray(c, np.float64)
        y, J = np.empty(4), np.empty(16)
        self.lib.oracle_deep_tangent_point(C.c_int(H), C.c_int(L), _dp(theta), C.c_int(int(all_double)), _dp(c), _dp(y), _dp(J))
        return y, J.reshape(4, 4)


@pytest.fixture(scope="module")
def chk(tmp_path_factory):
    out = str(tmp_path_factory.mktemp("deep_tangent_checker") / "libdeeptangent.so")
    src = os.path.join(ROOT, "tests", "deep_tangent_checker.c")
    subprocess.run([os.environ.get("CC", "gcc"), "-std=c11", "-O3", "-ffp-contract=off", "-fPIC", "-shared", "-o", out, src, "-lm"],
                   check=True, capture_output=True)
    return TangentChecker(out)


def _deep_weights(H, L, seed=777, scale=0.25, port=None):
    import oracle
    W1, b1, W2, b2 = (port or oracle.port()).mlp_random_init(H, seed, scale)
    rng = np.random.default_rng(seed + L)
    Wh = rng.uniform(-0.2, 0.2, (L - 1) * H * H).astype(np.float32)
    bh = rng.uniform(-0.2, 0.2, (L - 1) * H).astype(np.float32)
    return W1, b1, Wh, bh, W2, b2


def _theta(w):
    return np.concatenate([np.asarray(a, np.float64).ravel() for a in w if a is not None])


# ---------------------------------------------------------------------------------------------------------------------
# CPU tier
# ---------------------------------------------------------------------------------------------------------------------
FD_CASES = [
    # (shape, H, L, m1p1, spacing)
    ((3, 4, 2), 6, 2, True, (1, 1, 1)),
    ((4, 3, 3), 6, 3, False, (0.5, 0.25, 2.0)),
    ((3, 3, 3), 4, 3, True, (0.7, 1.1, 0.9)),
    ((4, 2, 3), 6, 2, False, (0.5, 1.0, 0.25)),
    ((1, 1, 1), 6, 2, True, (1, 1, 1)),
    ((5, 1, 1), 6, 3, False, (1, 1, 1)),
    ((1, 4, 3), 4, 3, True, (1, 1, 1)),
    ((1, 4, 3), 6, 2, False, (0.5, 0.25, 2.0)),
]


@pytest.mark.parametrize("shape,H,L,m1p1,h", FD_CASES)
def test_checker_gradient_matches_finite_differences(port, chk, shape, H, L, m1p1, h):
    og = OGrid(*shape, *h, 0.05, True)
    th = _theta(_deep_weights(H, L, 11, 0.6, port))
    t, ws, wu = 0.25, 1.3, 0.7
    got = chk.loss_grad(og, H, L, th, t, ws, wu, m1p1, all_double=True)["grad"]
    assert got.size == th.size == _plen(H, L)
    rng = np.random.default_rng(sum(shape) * 31 + H + L)
    idx = rng.choice(th.size, size=min(40, th.size), replace=False)
    gmax = np.abs(got).max()
    assert gmax > 0
    for i in idx:
        eps = 1e-6 * max(1.0, abs(th[i]))
        tp, tm = th.copy(), th.copy()
        tp[i] += eps
        tm[i] -= eps
        lp = chk.loss_grad(og, H, L, tp, t, ws, wu, m1p1, all_double=True, grad=False)
        lm = chk.loss_grad(og, H, L, tm, t, ws, wu, m1p1, all_double=True, grad=False)
        fd = ((lp["loss_sigma"] + lp["loss_u"]) - (lm["loss_sigma"] + lm["loss_u"])) / (2 * eps)
        assert abs(fd - got[i]) <= 1e-6 * gmax + 1e-12, (i, fd, got[i], gmax)


@pytest.mark.parametrize("H,L", [(6, 2), (8, 3), (5, 4)])
def test_checker_jacobian_matches_central_differences(port, chk, H, L):
    """J[o][k] of the all-double network = central differences of y_o in the input coordinate c_k."""
    th = _theta(_deep_weights(H, L, 5, 0.6, port))
    rng = np.random.default_rng(H * 10 + L)
    for _ in range(20):
        c = rng.uniform(-1, 1, 4)
        _, J = chk.point(H, L, th, c)
        eps = 1e-7
        fd = np.empty((4, 4))
        for k in range(4):
            cp, cm = c.copy(), c.copy()
            cp[k] += eps
            cm[k] -= eps
            fd[:, k] = (chk.point(H, L, th, cp)[0] - chk.point(H, L, th, cm)[0]) / (2 * eps)
        assert np.abs(fd - J).max() <= 1e-6 * max(np.abs(J).max(), 1e-3), (c, fd, J)


@pytest.mark.parametrize("shape,H,L,m1p1", [((6, 5, 4), 8, 2, True), ((7, 3, 5), 16, 3, False), ((1, 4, 3), 6, 5, True),
                                            ((5, 1, 1), 6, 2, False)])
def test_checker_values_are_the_deep_forward(port, chk, shape, H, L, m1p1):
    """Kernel-faithful mode: the value row is oracle_mlp_grid_infer_deep at time t, bit for bit."""
    og = OGrid(*shape, 1.0, 0.5, 2.0, 2e-3, True)
    w = _deep_weights(H, L, 3, 0.5, port)
    r = chk.loss_grad(og, H, L, _theta(w), 0.25, m1p1=m1p1, all_double=False, grad=False)
    want = port.mlp_grid_infer_deep(og, H, L, *w, 0.25, m1p1).reshape(og.N, 4)
    assert np.array_equal(r["Y"].view(np.uint32), want.view(np.uint32))


@pytest.mark.parametrize("shape,H,m1p1,h", [((6, 5, 4), 16, True, (1, 1, 1)), ((5, 1, 1), 32, False, (0.5, 1, 1)),
                                            ((1, 4, 3), 8, True, (1, 0.25, 2.0))])
def test_checker_one_layer_is_the_tangent_oracle(port, chk, shape, H, m1p1, h):
    """L = 1: the sums equal oracle_tangent_loss's up to the fp32 rounding of J."""
    og = OGrid(*shape, *h, 2e-3, True)
    W1, b1, W2, b2 = port.mlp_random_init(H, 5, 0.5)
    want = port.tangent_loss(og, (W1, b1, W2, b2), 0.25, m1p1)
    got = chk.loss_grad(og, H, 1, _theta((W1, b1, W2, b2)), 0.25, m1p1=m1p1, all_double=False, grad=False)
    for k in ("acc_sigma", "acc_u"):
        assert abs(got[k] - want[k]) <= 1e-6 * abs(want[k]), (k, got[k], want[k])


def _sass_counts(path):
    r = subprocess.run(["cuobjdump", "-sass", path], capture_output=True, text=True)
    if r.returncode != 0:
        pytest.skip("cuobjdump unavailable")
    cur, counts = None, {}
    for line in r.stdout.splitlines():
        m = re.search(r"Function : (\S+)", line)
        if m:
            cur = m.group(1)
            counts[cur] = {"FFMA": 0, "FFMA2": 0, "FMUL2": 0, "FADD2": 0, "UTCHMMA": 0}
            continue
        m = re.match(r"\s+/\*[0-9a-f]+\*/\s+(?:@!?U?P\d+\s+)?([A-Z0-9_]+)", line)
        if m and cur and m.group(1) in counts[cur]:
            counts[cur][m.group(1)] += 1
    return counts


def test_deep_tangent_kernel_sass():
    """k_deep_tangent<H, GRAD>: the value row keeps FMUL2 / FADD2 separate, the tangent rows use scalar FFMA; no FFMA2,
    no tcgen05."""
    from phys_autodiff_b200 import capi
    p = capi.library_path()
    if not os.path.exists(p):
        capi.build_library()
    ks = {k: v for k, v in _sass_counts(p).items() if "k_deep_tangent" in k and "reduce" not in k}
    assert len(ks) == 6, ks
    for k, v in ks.items():
        assert v["FMUL2"] > 0 and v["FADD2"] >= v["FMUL2"] and v["FFMA"] > 0, (k, v)
        assert v["FFMA2"] == 0 and v["UTCHMMA"] == 0, (k, v)


def test_deep_tangent_kernel_has_no_spills(tmp_path):
    nvcc = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    if not os.path.exists(nvcc):
        pytest.skip("nvcc unavailable")
    src = os.path.join(ROOT, "phys_autodiff_b200", "csrc", "deep_tangent_kernels.cu")
    r = subprocess.run([nvcc, "-std=c++17", "-O3", "-gencode", "arch=compute_100a,code=sm_100a", "-Xptxas", "-v", "-c",
                        "-o", str(tmp_path / "k.o"), src], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr[-2000:]
    props = re.findall(r"Function properties for (\S+)\n\s+(\d+) bytes stack frame, (\d+) bytes spill stores, (\d+) bytes spill loads",
                       r.stderr)
    assert len(props) == 7, r.stderr[-2000:]
    assert all(int(st) == 0 and int(sp) == 0 and int(sl) == 0 for _, st, sp, sl in props), props


# ---------------------------------------------------------------------------------------------------------------------
# GPU tier
# ---------------------------------------------------------------------------------------------------------------------
GPU_CASES = [
    # (shape, H, L, m1p1, spacing)
    ((48, 40, 12), 32, 2, True, (1, 1, 1)),
    ((33, 18, 7), 64, 3, False, (0.5, 0.25, 2.0)),     # nx % 32 != 0, anisotropic
    ((70, 37, 5), 128, 2, True, (1, 1, 1)),
    ((20, 9, 4), 128, 6, True, (0.7, 1.1, 0.9)),       # streamed weights
    ((64, 16, 6), 64, 5, False, (1, 1, 1)),
    ((10, 3, 2), 32, 3, True, (1, 1, 1)),              # smaller than one tile
    ((1, 1, 1), 32, 3, True, (1, 1, 1)),               # degenerate extents
    ((5, 1, 1), 64, 2, False, (1, 1, 1)),
    ((1, 4, 3), 32, 5, True, (1, 1, 1)),
    ((96, 8, 3), 128, 3, False, (1, 1, 1)),
]


def _g(og):
    from phys_autodiff_b200 import Grid
    return Grid(og.nx, og.ny, og.nz, og.hx, og.hy, og.hz, og.dt, og.periodic)


def _set(ctx, H, L, w, m1p1=True):
    from phys_autodiff_b200 import MLPConfig
    ctx.set_weights_deep(MLPConfig(4, H, 4, m1p1), L, *w)


@pytest.mark.gpu
@pytest.mark.parametrize("shape,H,L,m1p1,h", GPU_CASES)
def test_loss_and_gradient_vs_checker(ctx, port, chk, shape, H, L, m1p1, h):
    import torch
    from phys_autodiff_b200 import PhysWeights
    og = OGrid(*shape, *h, 2e-3, True)
    w = _deep_weights(H, L, 777, 0.25, port)
    want = chk.loss_grad(og, H, L, _theta(w), 0.25, 1.3, 0.7, m1p1, all_double=False)
    _set(ctx, H, L, w, m1p1)
    g = _g(og)
    R = [torch.empty(og.N, dtype=torch.float32, device="cuda") for _ in range(4)]
    acc = ctx.deep_tangent_loss_acc(g, 0.25, residuals=R).cpu().numpy()
    for got, ref in zip(acc, (want["acc_sigma"], want["acc_u"])):
        assert abs(got - ref) <= 1e-6 * abs(ref), (got, ref)
    rmax = max(np.abs(r).max() for r in want["R"])
    for a, b in zip(R, want["R"]):
        assert np.abs(a.cpu().numpy() - b).max() <= 1e-5 * rmax
    out = ctx.deep_tangent_loss_grad_acc(g, PhysWeights(1.3, 0.7), 0.25).cpu().numpy()
    assert out.shape == (_plen(H, L) + 2,)
    assert np.array_equal(out[:2].view(np.uint64), acc.view(np.uint64))   # the grad call's sums are the loss call's
    assert_grad_close(out[2:], want["grad"], H, L, TOL_GRAD)


@pytest.mark.gpu
def test_repeatable_and_host_form_agrees(ctx, port):
    from phys_autodiff_b200 import MLPConfig, PhysWeights, ops
    og = OGrid(96, 80, 37, 1, 1, 1, 2e-3, True)
    H, L = 64, 3
    w = _deep_weights(H, L, 777, 0.25, port)
    pw = PhysWeights(1.3, 0.7)
    _set(ctx, H, L, w)
    g = _g(og)
    a = ctx.deep_tangent_loss_grad(g, pw, 0.25)
    acc0 = ctx.deep_tangent_loss_acc(g, 0.25).cpu().numpy()
    for _ in range(5):
        b = ctx.deep_tangent_loss_grad(g, pw, 0.25)
        assert a[0] == b[0] and a[1] == b[1] and np.array_equal(a[2].view(np.uint64), b[2].view(np.uint64))
        assert np.array_equal(ctx.deep_tangent_loss_acc(g, 0.25).cpu().numpy().view(np.uint64), acc0.view(np.uint64))
    hst = ctx.deep_tangent_loss_grad_host(g, pw, 0.25)
    assert hst[0] == a[0] and hst[1] == a[1]
    assert np.array_equal(np.concatenate(hst[2:]), a[2].astype(np.float32))
    mod = ops.mlp_phys_loss_deep_tangent_grad_cuda(g, MLPConfig(4, H, 4, True), L, w, pw, 0.25)
    assert all(np.array_equal(x, y) for x, y in zip(mod, hst))


@pytest.mark.gpu
@pytest.mark.parametrize("shape,H,L", [((40, 24, 13), 64, 3), ((33, 9, 11), 32, 2), ((128, 8, 10), 128, 4), ((20, 9, 17), 128, 2)])
def test_slabs_sum_to_the_whole(ctx, port, shape, H, L):
    """Multi-GPU decomposition on one device: the slab sums (scaled by the whole grid's N) add up to the whole grid's."""
    from phys_autodiff_b200 import PhysWeights
    from phys_autodiff_b200.ops import slab_for_rank
    og = OGrid(*shape, 1, 1, 1, 2e-3, True)
    _set(ctx, H, L, _deep_weights(H, L, 777, 0.25, port))
    pw = PhysWeights(1.3, 0.7)
    g = _g(og)
    whole = ctx.deep_tangent_loss_grad_acc(g, pw, 0.25).cpu().numpy()
    for world in (2, 3, 8):
        tot = np.zeros_like(whole)
        acc = np.zeros(2)
        for r in range(world):
            sl = slab_for_rank(og.nz, r, world)
            tot += ctx.deep_tangent_loss_grad_acc(g, pw, 0.25, sl).cpu().numpy()
            acc += ctx.deep_tangent_loss_acc(g, 0.25, sl).cpu().numpy()
        assert np.abs(tot[:2] - whole[:2]).max() <= 1e-12 * np.abs(whole[:2]).max(), world
        assert np.abs(acc - whole[:2]).max() <= 1e-12 * np.abs(whole[:2]).max(), world
        assert np.abs(tot[2:] - whole[2:]).max() <= 2e-6 * np.abs(whole[2:]).max(), world
    z = ctx.deep_tangent_loss_grad_acc(g, pw, 0.25, (og.nz // 2, og.nz // 2)).cpu().numpy()
    assert z.shape == (_plen(H, L) + 2,) and not z.any()
    assert not ctx.deep_tangent_loss_acc(g, 0.25, (og.nz // 2, og.nz // 2)).cpu().numpy().any()


@pytest.mark.gpu
@pytest.mark.parametrize("H", [32, 64, 128])
def test_one_hidden_layer_is_the_one_layer_analytic_loss(ctx, port, H):
    from phys_autodiff_b200 import MLPConfig, PhysWeights
    og = OGrid(40, 24, 13, 1, 1, 1, 2e-3, True)
    g = _g(og)
    W1, b1, W2, b2 = port.mlp_random_init(H, 777, 0.25)
    pw = PhysWeights(1.3, 0.7)
    ctx.set_weights(MLPConfig(4, H, 4, True), W1, b1, W2, b2)
    acc = ctx.tangent_loss_acc(g, 0.25).cpu().numpy()
    full = ctx.tangent_loss_grad_acc(g, pw, 0.25).cpu().numpy()
    slab = ctx.tangent_loss_grad_acc(g, pw, 0.25, (3, 9)).cpu().numpy()
    ctx.set_weights_deep(MLPConfig(4, H, 4, True), 1, W1, b1, None, None, W2, b2)
    assert np.array_equal(ctx.deep_tangent_loss_acc(g, 0.25).cpu().numpy().view(np.uint64), acc.view(np.uint64))
    assert np.array_equal(ctx.deep_tangent_loss_grad_acc(g, pw, 0.25).cpu().numpy().view(np.uint64), full.view(np.uint64))
    assert np.array_equal(ctx.deep_tangent_loss_grad_acc(g, pw, 0.25, (3, 9)).cpu().numpy().view(np.uint64), slab.view(np.uint64))


@pytest.mark.gpu
def test_training_reduces_the_analytic_deep_loss_by_90_percent(ctx, port):
    """Host-side Adam at 32^3, H = 64, L = 3, learning rate 1e-3: L_sigma + L_u must fall by at least 90 % in 120 steps.
    The kernel-faithful checker's own Adam run (12^3, same network, step size and schedule) falls by 98.5 % in 120 steps."""
    from phys_autodiff_b200 import PhysWeights
    og = OGrid(32, 32, 32, 1, 1, 1, 2e-3, True)
    H, L = 64, 3
    pw = PhysWeights(1, 1)
    w0 = _deep_weights(H, L, 777, 0.25, port)
    th = _theta(w0)
    n = [a.size for a in w0]
    m, v = np.zeros_like(th), np.zeros_like(th)
    first = last = None
    for k in range(1, 121):
        W1, b1, Wh, bh, W2, b2 = np.split(th.astype(np.float32), np.cumsum(n)[:-1])
        _set(ctx, H, L, (W1, b1, Wh, bh, W2, b2))
        ls, lu, *d = ctx.deep_tangent_loss_grad_host(_g(og), pw, 0.25)
        Lv = float(ls) + float(lu)
        first = Lv if first is None else first
        last = Lv
        gvec = np.concatenate(d).astype(np.float64)
        m = 0.9 * m + 0.1 * gvec
        v = 0.999 * v + 0.001 * gvec * gvec
        th = th - 1e-3 * (m / (1 - 0.9 ** k)) / (np.sqrt(v / (1 - 0.999 ** k)) + 1e-8)
    assert np.isfinite(last) and last <= 0.1 * first, (first, last)


@pytest.mark.gpu
def test_error_paths(port):
    """Status codes, never a silent switch: no deep weights, fast mode, bad slabs, null pointers, mixed residual pointers,
    huge slabs."""
    import torch
    from phys_autodiff_b200 import Grid, MLPConfig, PhysadError, PhysWeights, capi, ops
    c2 = ops.Context()
    try:
        g, pw = Grid(8, 8, 8, 1, 1, 1, 1e-3, True), PhysWeights(1, 1)
        c2.cfg = MLPConfig(4, 32, 4, True)
        for call in (lambda: c2.deep_tangent_loss_acc(g, 0.1), lambda: c2.deep_tangent_loss_grad_acc(g, pw, 0.1)):
            with pytest.raises(PhysadError, match="set_weights_deep"):
                call()
        w = _deep_weights(32, 3, 1, 0.1, port)
        _set(c2, 32, 3, w)
        c2.set_weights(MLPConfig(4, 32, 4, True), w[0], w[1], w[4], w[5])   # back to one hidden layer: not a deep network
        with pytest.raises(PhysadError, match="set_weights_deep"):
            c2.deep_tangent_loss_grad_acc(g, pw, 0.1)
        with pytest.raises(PhysadError, match="set_weights_deep"):
            c2.deep_tangent_loss_acc(g, 0.1)
        _set(c2, 32, 3, w)
        c2.set_deep_mode(1)
        for call in (lambda: c2.deep_tangent_loss_acc(g, 0.1), lambda: c2.deep_tangent_loss_grad_acc(g, pw, 0.1)):
            with pytest.raises(PhysadError, match="strict"):
                call()
        c2.set_deep_mode(0)
        with pytest.raises(PhysadError):
            c2.deep_tangent_loss_grad_acc(Grid(0, 8, 8), pw, 0.1)
        for sl in ((4, 12), (5, 3)):
            with pytest.raises(PhysadError, match="slab"):
                c2.deep_tangent_loss_grad_acc(g, pw, 0.1, sl)
            with pytest.raises(PhysadError, match="slab"):
                c2.deep_tangent_loss_acc(g, 0.1, sl)
        R = [torch.empty(g.N, dtype=torch.float32, device="cuda") for _ in range(3)] + [None]
        with pytest.raises(PhysadError, match="all set or all null"):
            c2.deep_tangent_loss_acc(g, 0.1, residuals=R)
        # 2^31 points or more are refused before any allocation (32-bit point indices)
        big = Grid(16384, 16384, 8, 1, 1, 1, 1e-3, True)
        with pytest.raises(PhysadError, match="2\\^31"):
            c2.deep_tangent_loss_grad_acc(big, pw, 0.1, (0, 8))
        with pytest.raises(PhysadError, match="2\\^31"):
            c2.deep_tangent_loss_acc(big, 0.1, (0, 8))
        lib = capi.lib()
        E_INVALID = lib.physad_deep_tangent_loss_grad_dev(c2._h, None, None, None, C.c_float(0), None, None, None)
        assert E_INVALID == -1
        assert lib.physad_deep_tangent_loss_dev(c2._h, None, None, C.c_float(0), None, None, None, None, None, None) == E_INVALID
        assert lib.physad_deep_tangent_loss_grad_host(None, None, None, C.c_float(0), None, None, None, None, None, None,
                                                      None, None) == E_INVALID
        # a bad call leaves the context usable
        out = c2.deep_tangent_loss_grad_acc(g, pw, 0.1).cpu().numpy()
        assert np.isfinite(out).all() and out[0] > 0
    finally:
        c2.close()


WORKER = r'''
import os, sys, json
sys.path.insert(0, %r)
import numpy as np, torch, torch.distributed as dist
from phys_autodiff_b200 import Grid, MLPConfig, PhysWeights, ops
rank, world, local = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"]), int(os.environ["LOCAL_RANK"])
torch.cuda.set_device(local)
dist.init_process_group("nccl", device_id=torch.device("cuda", local))
g = Grid(96, 80, 37, 1, 1, 1, 2e-3, True)          # 37 planes: uneven slabs
ctx = ops.Context(local)
H, L = 64, 3
W1, b1, W2, b2 = ops.mlp_random_init(H, 777, 0.25)
rng = np.random.default_rng(7)
Wh = rng.uniform(-0.2, 0.2, (L - 1) * H * H).astype(np.float32)
bh = rng.uniform(-0.2, 0.2, (L - 1) * H).astype(np.float32)
ctx.set_weights_deep(MLPConfig(4, H, 4, True), L, W1, b1, Wh, bh, W2, b2)
pw = PhysWeights(1.3, 0.7)
ls, lu, gr = ctx.deep_tangent_loss_grad(g, pw, 0.25)                     # slab per rank + one all-reduce
one = ctx.deep_tangent_loss_grad_acc(g, pw, 0.25).cpu().numpy()           # the whole grid on this rank's device
l1 = ctx.finalize(one[:2], pw, g.N)
out = dict(rank=rank, ls=float(ls), lu=float(lu), ls1=float(l1[0]), lu1=float(l1[1]),
           grad_err=float(np.abs(gr - one[2:]).max() / np.abs(one[2:]).max()))
gathered = [None] * world
dist.all_gather_object(gathered, out)
if rank == 0:
    print("RESULT " + json.dumps(gathered))
dist.destroy_process_group()
'''


@pytest.mark.gpu
def test_multi_gpu_gradient_matches_single_gpu(tmp_path):
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs >= 2 GPUs")
    script = tmp_path / "worker.py"
    script.write_text(WORKER % ROOT)
    n = min(torch.cuda.device_count(), 8)
    r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={n}",
                        "--master-addr", "127.0.0.1", "--master-port", "29736", str(script)],
                       capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-4000:]
    res = json.loads([ln for ln in r.stdout.splitlines() if ln.startswith("RESULT ")][-1][len("RESULT "):])
    assert len(res) == n
    for d in res:
        assert d["ls"] == res[0]["ls"] and d["lu"] == res[0]["lu"]
        assert abs(d["ls"] - d["ls1"]) <= 1e-6 * abs(d["ls1"]) and abs(d["lu"] - d["lu1"]) <= 1e-6 * abs(d["lu1"])
        assert d["grad_err"] <= 2e-6, d["grad_err"]
