"""Closed loop of deeper networks: d(L_sigma + L_u)/d(every layer's weights) of the finite-difference loss.

The checker is tests/deep_grad_checker.c, compiled here into a temporary library.
CPU tier: the checker (oracle_phys_loss_grad_deep) against central finite differences of its all-double loss, its
fp32-faithful losses against the pinned port, L = 1 against the one-hidden-layer checker, P(H, L), and the kernel's
SASS.  GPU tier: k_deep_grad against the fp32-faithful checker, the losses, determinism, host form, slabs, L = 1,
error paths, training and a torchrun comparison across GPUs."""
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


def _fp(a):
    if a is None or a.size == 0:
        return C.cast(None, C.POINTER(C.c_float))
    a = np.ascontiguousarray(a, np.float32)
    return a.ctypes.data_as(C.POINTER(C.c_float))


class DeepChecker:
    """ctypes surface of tests/deep_grad_checker.c (same flags as the oracle port: -O3 -ffp-contract=off)."""

    def __init__(self, path):
        self.lib = C.CDLL(path)
        self.lib.oracle_phys_loss_grad_deep.restype = C.c_int
        self.lib.oracle_phys_loss_double_deep.restype = C.c_int

    def phys_loss_grad_deep(self, g, H, L, w, t, dt, w_sigma=1.0, w_u=1.0, m1p1=True, all_double=False):
        """w = (W1, b1, Wh, bh, W2, b2) -> dict(loss_sigma, loss_u, grad[P] f64), layout dW1 | db1 | dWh | dbh | dW2 | db2."""
        w = [None if a is None else np.ascontiguousarray(a, np.float32) for a in w]
        ls, lu = C.c_double(), C.c_double()
        grad = np.empty(_plen(H, L), np.float64)
        rc = self.lib.oracle_phys_loss_grad_deep(C.byref(g.c()), C.c_int(H), C.c_int(L), C.c_int(int(m1p1)), *[_fp(a) for a in w],
                                                 C.c_float(t), C.c_float(dt), C.c_float(w_sigma), C.c_float(w_u),
                                                 C.c_int(int(all_double)), C.byref(ls), C.byref(lu),
                                                 grad.ctypes.data_as(C.POINTER(C.c_double)))
        assert rc == 0
        return dict(loss_sigma=ls.value, loss_u=lu.value, grad=grad)

    def phys_loss_double_deep(self, g, theta, H, L, t, dt, w_sigma=1.0, w_u=1.0, m1p1=True):
        """All-double (L_sigma, L_u) of double parameters theta[P] (gradient layout): what finite differences probe."""
        theta = np.ascontiguousarray(theta, np.float64)
        assert theta.size == _plen(H, L)
        ls, lu = C.c_double(), C.c_double()
        rc = self.lib.oracle_phys_loss_double_deep(C.byref(g.c()), C.c_int(H), C.c_int(L), C.c_int(int(m1p1)),
                                                   theta.ctypes.data_as(C.POINTER(C.c_double)), C.c_float(t), C.c_float(dt),
                                                   C.c_float(w_sigma), C.c_float(w_u), C.byref(ls), C.byref(lu))
        assert rc == 0
        return ls.value, lu.value


@pytest.fixture(scope="module")
def deep(tmp_path_factory):
    out = str(tmp_path_factory.mktemp("deep_checker") / "libdeepgrad.so")
    src = os.path.join(ROOT, "tests", "deep_grad_checker.c")
    subprocess.run([os.environ.get("CC", "gcc"), "-std=c11", "-O3", "-ffp-contract=off", "-fPIC", "-shared", "-o", out, src, "-lm"],
                   check=True, capture_output=True)
    return DeepChecker(out)


def _plen(H, L):
    return 9 * H + 4 + (L - 1) * (H * H + H)


def _deep_weights(H, L, seed=777, scale=0.25, port=None):
    import oracle
    W1, b1, W2, b2 = (port or oracle.port()).mlp_random_init(H, seed, scale)
    rng = np.random.default_rng(seed + L)
    Wh = rng.uniform(-0.2, 0.2, (L - 1) * H * H).astype(np.float32)
    bh = rng.uniform(-0.2, 0.2, (L - 1) * H).astype(np.float32)
    return W1, b1, Wh, bh, W2, b2


def _theta(w):
    return np.concatenate([np.asarray(a, np.float64).ravel() for a in w])


# ---------------------------------------------------------------------------------------------------------------------
# CPU tier
# ---------------------------------------------------------------------------------------------------------------------
FD_CASES = [
    # (shape, H, L, periodic, m1p1, spacing)
    ((3, 4, 2), 6, 2, True, True, (1, 1, 1)),
    ((4, 3, 3), 6, 3, False, False, (0.5, 0.25, 2.0)),
    ((3, 3, 3), 4, 3, True, False, (0.7, 1.1, 0.9)),
    ((4, 2, 3), 6, 2, False, True, (0.5, 1.0, 0.25)),
    ((1, 1, 1), 6, 2, True, True, (1, 1, 1)),
    ((5, 1, 1), 6, 3, False, False, (1, 1, 1)),
    ((1, 4, 3), 4, 3, True, True, (1, 1, 1)),
    ((1, 4, 3), 6, 2, False, False, (0.5, 0.25, 2.0)),
]


@pytest.mark.parametrize("shape,H,L,per,m1p1,h", FD_CASES)
def test_checker_gradient_matches_finite_differences(port, deep, shape, H, L, per, m1p1, h):
    og = OGrid(*shape, *h, 0.05, per)
    w = _deep_weights(H, L, 11, 0.6, port)
    t, dt, ws, wu = 0.25, 0.05, 1.3, 0.7
    got = deep.phys_loss_grad_deep(og, H, L, w, t, dt, ws, wu, m1p1, all_double=True)["grad"]
    th = _theta(w)
    assert got.size == th.size == _plen(H, L)
    rng = np.random.default_rng(sum(shape) * 31 + H + L)
    idx = rng.choice(th.size, size=min(30, th.size), replace=False)
    gmax = np.abs(got).max()
    for i in idx:
        eps = 1e-6 * max(1.0, abs(th[i]))
        tp, tm = th.copy(), th.copy()
        tp[i] += eps
        tm[i] -= eps
        lp = sum(deep.phys_loss_double_deep(og, tp, H, L, t, dt, ws, wu, m1p1))
        lm = sum(deep.phys_loss_double_deep(og, tm, H, L, t, dt, ws, wu, m1p1))
        fd = (lp - lm) / (2 * eps)
        assert abs(fd - got[i]) <= 1e-6 * gmax + 1e-12, (i, fd, got[i], gmax)


@pytest.mark.parametrize("shape,H,L,per,m1p1", [((6, 5, 4), 8, 2, True, True), ((7, 3, 5), 8, 3, False, False),
                                                ((1, 4, 3), 6, 4, True, False), ((5, 1, 1), 6, 2, False, True)])
def test_checker_fp32_losses_are_the_pinned_ports(port, deep, shape, H, L, per, m1p1):
    """fp32-faithful mode: fields = oracle_mlp_grid_infer_deep of the three slices, residuals and sums = the port's."""
    og = OGrid(*shape, 1.0, 0.5, 2.0, 2e-3, per)
    w = _deep_weights(H, L, 3, 0.5, port)
    t, dt = np.float32(0.25), np.float32(2e-3)
    r = deep.phys_loss_grad_deep(og, H, L, w, float(t), float(dt), 1.0, 1.0, m1p1, all_double=False)
    N = og.N
    s, u = [], []
    for ts in (t - dt, t, t + dt):
        f = port.mlp_grid_infer_deep(og, H, L, *w, float(np.float32(ts)), m1p1).reshape(N, 4)
        s.append(np.ascontiguousarray(f[:, 0]))
        u.append(np.ascontiguousarray(f[:, 1:].T).ravel())
    R = port.phys_residuals(og, (s[0], s[1], s[2], u[0], u[1], u[2]))
    a_s, a_u = port.sumsq(R, 0, N)
    assert abs(r["loss_sigma"] - a_s / N) <= 1e-14 * abs(a_s / N) + 1e-300
    assert abs(r["loss_u"] - a_u / N) <= 1e-14 * abs(a_u / N) + 1e-300


@pytest.mark.parametrize("all_double", [False, True])
@pytest.mark.parametrize("shape,per,m1p1", [((6, 5, 4), True, True), ((5, 1, 1), False, False), ((1, 4, 3), True, False)])
def test_checker_one_layer_equals_the_one_hidden_layer_checker(port, deep, shape, per, m1p1, all_double):
    og = OGrid(*shape, 0.5, 1.0, 0.25, 2e-3, per)
    W1, b1, W2, b2 = port.mlp_random_init(16, 5, 0.5)
    a = port.phys_loss_grad(og, (W1, b1, W2, b2), 0.25, 2e-3, 1.3, 0.7, m1p1, all_double)
    b = deep.phys_loss_grad_deep(og, 16, 1, (W1, b1, None, None, W2, b2), 0.25, 2e-3, 1.3, 0.7, m1p1, all_double)
    assert a["loss_sigma"] == b["loss_sigma"] and a["loss_u"] == b["loss_u"]
    assert np.array_equal(a["grad"].view(np.uint64), b["grad"].view(np.uint64))


def test_gradient_length():
    from phys_autodiff_b200 import capi
    lib = capi.lib()
    for H in (32, 64, 128):
        for L in (1, 2, 3, 5, 16):
            assert lib.physad_deep_grad_len(H, L) == _plen(H, L)
    assert lib.physad_deep_grad_len(128, 16) == 248836
    for H, L in ((48, 2), (256, 2), (64, 0), (64, 17)):
        assert lib.physad_deep_grad_len(H, L) == 0


def _sass_counts(path):
    r = subprocess.run(["cuobjdump", "-sass", path], capture_output=True, text=True)
    if r.returncode != 0:
        pytest.skip("cuobjdump unavailable")
    cur, counts = None, {}
    for line in r.stdout.splitlines():
        m = re.search(r"Function : (\S+)", line)
        if m:
            cur = m.group(1)
            counts[cur] = {"FFMA2": 0, "FMUL2": 0, "FADD2": 0, "UTCHMMA": 0}
            continue
        m = re.match(r"\s+/\*[0-9a-f]+\*/\s+(?:@!?U?P\d+\s+)?([A-Z0-9_]+)", line)
        if m and cur and m.group(1) in counts[cur]:
            counts[cur][m.group(1)] += 1
    return counts


def test_deep_grad_kernel_sass():
    """k_deep_grad<H>: the recomputed forward keeps FMUL2 / FADD2 separate (no FFMA2 anywhere), no tcgen05."""
    from phys_autodiff_b200 import capi
    p = capi.library_path()
    if not os.path.exists(p):
        capi.build_library()
    ks = {k: v for k, v in _sass_counts(p).items() if "k_deep_grad" in k and "reduce" not in k}
    assert len(ks) == 3, ks
    for k, v in ks.items():
        assert v["FMUL2"] > 0 and v["FADD2"] >= v["FMUL2"] and v["FFMA2"] == 0 and v["UTCHMMA"] == 0, (k, v)


def test_deep_grad_kernel_has_no_spills(tmp_path):
    nvcc = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    if not os.path.exists(nvcc):
        pytest.skip("nvcc unavailable")
    src = os.path.join(ROOT, "phys_autodiff_b200", "csrc", "deep_grad_kernels.cu")
    r = subprocess.run([nvcc, "-std=c++17", "-O3", "-gencode", "arch=compute_100a,code=sm_100a", "-Xptxas", "-v", "-c",
                        "-o", str(tmp_path / "k.o"), src], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr[-2000:]
    props = re.findall(r"Function properties for (\S+)\n\s+(\d+) bytes stack frame, (\d+) bytes spill stores, (\d+) bytes spill loads",
                       r.stderr)
    assert len(props) == 4, r.stderr[-2000:]
    assert all(int(st) == 0 and int(sp) == 0 and int(sl) == 0 for _, st, sp, sl in props), props


# ---------------------------------------------------------------------------------------------------------------------
# GPU tier
# ---------------------------------------------------------------------------------------------------------------------
GPU_CASES = [
    # (shape, H, L, periodic, m1p1, spacing)
    ((48, 40, 12), 32, 2, True, True, (1, 1, 1)),
    ((33, 18, 7), 64, 3, False, False, (0.5, 0.25, 2.0)),     # nx % 32 != 0, anisotropic, clamped
    ((70, 37, 5), 128, 2, False, True, (1, 1, 1)),
    ((20, 9, 4), 128, 6, True, True, (0.7, 1.1, 0.9)),         # streamed weights (L - 1 > 2)
    ((64, 16, 6), 64, 5, True, False, (1, 1, 1)),
    ((10, 3, 2), 32, 3, False, True, (1, 1, 1)),               # smaller than one tile
    ((1, 1, 1), 32, 3, True, True, (1, 1, 1)),                 # degenerate extents
    ((5, 1, 1), 64, 2, False, False, (1, 1, 1)),
    ((1, 4, 3), 32, 5, True, True, (1, 1, 1)),
    ((96, 8, 3), 128, 3, False, False, (1, 1, 1)),
]

# Per-tensor floors where fp32 rounding is measured to dominate.  (1, 4, 3), H = 32, L = 5: twelve points of a nearly
# constant network, so the residuals are mostly rounding of nearly equal outputs; the checker's fp32-faithful gradient
# differs from its all-double one by 0.6 - 2.6e-3 of every tensor's own scale.  dbh2 - dbh4 are 0.2 - 0.5 % of the largest
# entry, and the kernel's fp32 adjoint puts them 1.0e-3, 2.5e-3 and 1.0e-3 of their own scale (at most 7e-6 of the largest
# entry) from the faithful checker on a B200.
FP32_FLOORS = {((1, 4, 3), 32, 5): {"dbh2": 0.1, "dbh3": 0.1, "dbh4": 0.1}}


def _g(og):
    from phys_autodiff_b200 import Grid
    return Grid(og.nx, og.ny, og.nz, og.hx, og.hy, og.hz, og.dt, og.periodic)


def _set(ctx, H, L, w, m1p1=True):
    from phys_autodiff_b200 import MLPConfig
    ctx.set_weights_deep(MLPConfig(4, H, 4, m1p1), L, *w)


@pytest.mark.gpu
@pytest.mark.parametrize("shape,H,L,per,m1p1,h", GPU_CASES)
def test_gradient_vs_checker(ctx, port, deep, shape, H, L, per, m1p1, h):
    from phys_autodiff_b200 import PhysWeights
    og = OGrid(*shape, *h, 2e-3, per)
    w = _deep_weights(H, L, 777, 0.25, port)
    want = deep.phys_loss_grad_deep(og, H, L, w, 0.25, 2e-3, 1.3, 0.7, m1p1, all_double=False)
    _set(ctx, H, L, w, m1p1)
    pw = PhysWeights(1.3, 0.7)
    out = ctx.deep_loss_grad_acc(_g(og), pw, 0.25, 2e-3).cpu().numpy()
    assert out.shape == (_plen(H, L) + 2,)
    assert_grad_close(out[2:], want["grad"], H, L, TOL_GRAD, floors=FP32_FLOORS.get((shape, H, L)))
    # the losses are physad_deep_loss_host's: same fields, same residual kernel, same sums
    ls, lu = ctx.finalize(out[:2], pw, og.N)
    assert (ls, lu) == ctx.deep_loss(_g(og), pw, 0.25, 2e-3)


@pytest.mark.gpu
def test_gradient_vs_checker_when_dt_differs_from_the_grid_step(ctx, port, deep):
    """The call's dt places the slices; the residual's time derivative uses grid.dt."""
    from phys_autodiff_b200 import PhysWeights
    og = OGrid(24, 20, 9, 1, 1, 1, 2e-3, True)
    w = _deep_weights(64, 3, 5, 0.25, port)
    want = deep.phys_loss_grad_deep(og, 64, 3, w, 0.3, 5e-3, 1.0, 1.0, True, all_double=False)["grad"]
    _set(ctx, 64, 3, w)
    out = ctx.deep_loss_grad_acc(_g(og), PhysWeights(1.0, 1.0), 0.3, 5e-3).cpu().numpy()
    assert_grad_close(out[2:], want, 64, 3, TOL_GRAD)


@pytest.mark.gpu
def test_gradient_is_deterministic_and_host_form_agrees(ctx, port):
    from phys_autodiff_b200 import MLPConfig, PhysWeights, ops
    og = OGrid(96, 80, 37, 1, 1, 1, 2e-3, True)
    H, L = 64, 3
    w = _deep_weights(H, L, 777, 0.25, port)
    pw = PhysWeights(1.3, 0.7)
    _set(ctx, H, L, w)
    a = ctx.deep_loss_grad(_g(og), pw, 0.25, 2e-3)
    for _ in range(5):
        b = ctx.deep_loss_grad(_g(og), pw, 0.25, 2e-3)
        assert a[0] == b[0] and a[1] == b[1] and np.array_equal(a[2].view(np.uint64), b[2].view(np.uint64))
    hst = ctx.deep_loss_grad_host(_g(og), pw, 0.25, 2e-3)
    assert hst[0] == a[0] and hst[1] == a[1]
    assert np.array_equal(np.concatenate(hst[2:]), a[2].astype(np.float32))
    mod = ops.mlp_phys_loss_deep_grad_cuda(_g(og), MLPConfig(4, H, 4, True), L, w, pw, 0.25, 2e-3)
    assert all(np.array_equal(x, y) for x, y in zip(mod, hst))


@pytest.mark.gpu
@pytest.mark.parametrize("shape,H,L,per", [((40, 24, 13), 64, 3, True), ((33, 9, 11), 32, 2, False),
                                           ((128, 8, 10), 128, 4, True), ((20, 9, 17), 128, 2, False)])
def test_slab_gradients_sum_to_the_whole(ctx, port, shape, H, L, per):
    """Multi-GPU decomposition on one device: the slab sums (scaled by the whole grid's N) add up to the whole grid's."""
    from phys_autodiff_b200 import PhysWeights
    from phys_autodiff_b200.ops import slab_for_rank
    og = OGrid(*shape, 1, 1, 1, 2e-3, per)
    _set(ctx, H, L, _deep_weights(H, L, 777, 0.25, port))
    pw = PhysWeights(1.3, 0.7)
    whole = ctx.deep_loss_grad_acc(_g(og), pw, 0.25, 2e-3).cpu().numpy()
    for world in (2, 3, 8):
        tot = np.zeros_like(whole)
        for r in range(world):
            tot += ctx.deep_loss_grad_acc(_g(og), pw, 0.25, 2e-3, slab_for_rank(og.nz, r, world)).cpu().numpy()
        assert np.abs(tot[:2] - whole[:2]).max() <= 1e-12 * np.abs(whole[:2]).max(), world
        assert np.abs(tot[2:] - whole[2:]).max() <= 2e-6 * np.abs(whole[2:]).max(), world
    z = ctx.deep_loss_grad_acc(_g(og), pw, 0.25, 2e-3, (og.nz // 2, og.nz // 2)).cpu().numpy()
    assert z.shape == (_plen(H, L) + 2,) and not z.any()


@pytest.mark.gpu
@pytest.mark.parametrize("H,per", [(32, True), (64, False), (128, True)])
def test_one_hidden_layer_is_the_one_layer_closed_loop(ctx, port, H, per):
    from phys_autodiff_b200 import MLPConfig, PhysWeights
    og = OGrid(40, 24, 13, 1, 1, 1, 2e-3, per)
    W1, b1, W2, b2 = port.mlp_random_init(H, 777, 0.25)
    pw = PhysWeights(1.3, 0.7)
    ctx.set_weights(MLPConfig(4, H, 4, True), W1, b1, W2, b2)
    acc, grad = (x.cpu().numpy() for x in ctx.fused_loss_grad_acc(_g(og), pw, 0.25, 2e-3))
    slab = ctx.fused_loss_grad_slab_acc(_g(og), pw, 0.25, 2e-3, (3, 9)).cpu().numpy()
    ctx.set_weights_deep(MLPConfig(4, H, 4, True), 1, W1, b1, None, None, W2, b2)
    d = ctx.deep_loss_grad_acc(_g(og), pw, 0.25, 2e-3).cpu().numpy()
    assert np.array_equal(d.view(np.uint64), np.concatenate([acc, grad]).view(np.uint64))
    ds = ctx.deep_loss_grad_acc(_g(og), pw, 0.25, 2e-3, (3, 9)).cpu().numpy()
    assert np.array_equal(ds.view(np.uint64), slab.view(np.uint64))


@pytest.mark.gpu
def test_training_reduces_the_deep_loss_by_90_percent(ctx, port):
    """The closed-loop criterion of REQUIREMENT.md:164-169 for a deep network: host-side Adam, L falls >= 90 % in 120
    steps.  The CPU checker's own fp32-faithful Adam run (oracle_phys_loss_grad_deep, same size, step size and schedule,
    weights drawn the same way from another seed) falls by 99.7 % in 120 steps, so the plan's 90 % is asserted."""
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
        ls, lu, *d = ctx.deep_loss_grad_host(_g(og), pw, 0.25, 2e-3)
        Lv = float(ls) + float(lu)
        first = Lv if first is None else first
        last = Lv
        gvec = np.concatenate(d).astype(np.float64)
        m = 0.9 * m + 0.1 * gvec
        v = 0.999 * v + 0.001 * gvec * gvec
        th = th - 3e-3 * (m / (1 - 0.9 ** k)) / (np.sqrt(v / (1 - 0.999 ** k)) + 1e-8)
    assert np.isfinite(last) and last <= 0.1 * first, (first, last)


@pytest.mark.gpu
def test_gradient_error_paths(port):
    """Status codes, never a silent switch: no deep weights, fast mode, upwind, bad slabs, null pointers, huge windows."""
    from phys_autodiff_b200 import Grid, MLPConfig, PhysadError, PhysWeights, capi, ops
    c2 = ops.Context()
    try:
        g, pw = Grid(8, 8, 8, 1, 1, 1, 1e-3, True), PhysWeights(1, 1)
        c2.cfg = MLPConfig(4, 32, 4, True)
        with pytest.raises(PhysadError, match="set_weights_deep"):
            c2.deep_loss_grad_acc(g, pw, 0.1, 1e-3)
        w = _deep_weights(32, 3, 1, 0.1, port)
        _set(c2, 32, 3, w)
        c2.set_weights(MLPConfig(4, 32, 4, True), w[0], w[1], w[4], w[5])   # back to one hidden layer: not a deep network
        with pytest.raises(PhysadError, match="set_weights_deep"):
            c2.deep_loss_grad_acc(g, pw, 0.1, 1e-3)
        _set(c2, 32, 3, w)
        c2.set_deep_mode(1)
        with pytest.raises(PhysadError, match="strict"):
            c2.deep_loss_grad_acc(g, pw, 0.1, 1e-3)
        c2.set_deep_mode(0)
        c2.set_advection(True)
        with pytest.raises(PhysadError, match="central"):
            c2.deep_loss_grad_acc(g, pw, 0.1, 1e-3)
        c2.set_advection(False)
        with pytest.raises(PhysadError):
            c2.deep_loss_grad_acc(Grid(0, 8, 8), pw, 0.1, 1e-3)
        with pytest.raises(PhysadError, match="slab"):
            c2.deep_loss_grad_acc(g, pw, 0.1, 1e-3, (4, 12))
        with pytest.raises(PhysadError, match="slab"):
            c2.deep_loss_grad_acc(g, pw, 0.1, 1e-3, (5, 3))
        # a grid under 2^31 points whose slab's wrapped window of 10 planes reaches 2^31 (refused before any allocation)
        with pytest.raises(PhysadError, match="2\\^31"):
            c2.deep_loss_grad_acc(Grid(16384, 16384, 7, 1, 1, 1, 1e-3, True), pw, 0.1, 1e-3, (0, 6))
        lib = capi.lib()
        E_INVALID = lib.physad_deep_loss_grad_dev(c2._h, None, None, None, C.c_float(0), C.c_float(0), None, None, None)
        assert E_INVALID == -1
        assert lib.physad_deep_loss_grad_host(None, None, None, C.c_float(0), C.c_float(0), None, None, None, None, None,
                                              None, None, None) == E_INVALID
        # a bad call leaves the context usable
        out = c2.deep_loss_grad_acc(g, pw, 0.1, 1e-3).cpu().numpy()
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
ls, lu, gr = ctx.deep_loss_grad(g, pw, 0.25, 2e-3)                       # slab per rank + one all-reduce
one = ctx.deep_loss_grad_acc(g, pw, 0.25, 2e-3).cpu().numpy()             # the whole grid on this rank's device
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
                        "--master-addr", "127.0.0.1", "--master-port", "29735", str(script)],
                       capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-4000:]
    res = json.loads([ln for ln in r.stdout.splitlines() if ln.startswith("RESULT ")][-1][len("RESULT "):])
    assert len(res) == n
    for d in res:
        assert d["ls"] == res[0]["ls"] and d["lu"] == res[0]["lu"]
        assert abs(d["ls"] - d["ls1"]) <= 1e-6 * abs(d["ls1"]) and abs(d["lu"] - d["lu1"]) <= 1e-6 * abs(d["lu1"])
        assert d["grad_err"] <= 2e-6, d["grad_err"]
