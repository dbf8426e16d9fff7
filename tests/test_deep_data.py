"""Deeper networks at arbitrary points: the forward pass and the data-fit loss with its gradient with respect to every
layer's weights.

The checker is tests/deep_data_checker.c, compiled here into a temporary library.
CPU tier: the checker's all-double gradient against central finite differences of its all-double loss, its fp32 forward
against oracle_mlp_forward_deep, and the SASS / register report of the new kernels.  GPU tier: the forward bit for bit
against the oracle, the grid kernel and the one-hidden-layer forward; the gradient against the fp32-faithful checker and
at L = 1 against physad_mlp_backward; determinism, host / device / module forms, shards, B = 0, error paths, training with
a data term, and a torchrun comparison across GPUs."""
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


def _plen(H, L):
    return 9 * H + 4 + (L - 1) * (H * H + H)


def _theta(w):
    return np.concatenate([np.asarray(a, np.float64).ravel() for a in w if a is not None])


def _deep_weights(H, L, seed=777, scale=0.25, port=None):
    import oracle
    W1, b1, W2, b2 = (port or oracle.port()).mlp_random_init(H, seed, scale)
    rng = np.random.default_rng(seed + L)
    Wh = rng.uniform(-0.2, 0.2, (L - 1) * H * H).astype(np.float32)
    bh = rng.uniform(-0.2, 0.2, (L - 1) * H).astype(np.float32)
    return W1, b1, Wh, bh, W2, b2


def _points(B, seed, lo=-1.0, hi=1.0):
    return np.random.default_rng(seed).uniform(lo, hi, (B, 4)).astype(np.float32)


class DataChecker:
    """ctypes surface of tests/deep_data_checker.c (same flags as the oracle port: -O3 -ffp-contract=off)."""

    def __init__(self, path):
        self.lib = C.CDLL(path)
        self.lib.oracle_data_loss_grad_deep.restype = C.c_int

    def run(self, H, L, theta, x, target, lam=None, n_norm=None, all_double=False):
        """-> (acc, grad[P] f64, y [B, 4] f32 of the fp32 mode)."""
        theta = np.ascontiguousarray(theta, np.float64)
        x, target = np.ascontiguousarray(x, np.float32), np.ascontiguousarray(target, np.float32)
        B = x.size // 4
        assert theta.size == _plen(H, L)
        acc = C.c_double()
        grad = np.empty(_plen(H, L), np.float64)
        y = np.empty((B, 4), np.float32)
        lw = None if lam is None else (C.c_float * 4)(*[float(v) for v in lam])
        fp = lambda a: a.ctypes.data_as(C.c_void_p)
        rc = self.lib.oracle_data_loss_grad_deep(C.c_int(H), C.c_int(L), fp(theta), fp(x), fp(target), C.c_size_t(B), lw,
                                                 C.c_size_t(B if n_norm is None else n_norm), C.c_int(int(all_double)),
                                                 C.byref(acc), fp(grad), fp(y))
        assert rc == 0
        return acc.value, grad, y


@pytest.fixture(scope="module")
def chk(tmp_path_factory):
    out = str(tmp_path_factory.mktemp("deep_data_checker") / "libdeepdata.so")
    src = os.path.join(ROOT, "tests", "deep_data_checker.c")
    subprocess.run([os.environ.get("CC", "gcc"), "-std=c11", "-O3", "-ffp-contract=off", "-fPIC", "-shared", "-o", out, src, "-lm"],
                   check=True, capture_output=True)
    return DataChecker(out)


# ---------------------------------------------------------------------------------------------------------------------
# CPU tier
# ---------------------------------------------------------------------------------------------------------------------
LAM = (0.7, 1.9, 0.0, 0.35)
FD_CASES = [
    # (H, L, B, lam, n_norm)
    (6, 1, 5, None, 5),
    (6, 1, 37, LAM, 11),
    (6, 2, 1, None, 1),
    (6, 2, 37, LAM, 37),
    (4, 2, 5, LAM, 3),
    (6, 3, 37, None, 50),
    (6, 3, 5, LAM, 5),
    (4, 3, 1, LAM, 2),
]


@pytest.mark.parametrize("H,L,B,lam,n_norm", FD_CASES)
def test_checker_gradient_matches_finite_differences(port, chk, H, L, B, lam, n_norm):
    w = _deep_weights(H, L, 11, 0.6, port)
    th = _theta(w)
    x = _points(B, H * 100 + L * 10 + B, -1.5, 1.5)
    tgt = _points(B, B + 1, -0.5, 0.5)
    _, got, _ = chk.run(H, L, th, x, tgt, lam, n_norm, all_double=True)
    rng = np.random.default_rng(H + L + B)
    idx = rng.choice(th.size, size=min(40, th.size), replace=False)
    gmax = np.abs(got).max()
    assert gmax > 0
    for i in idx:
        eps = 1e-6 * max(1.0, abs(th[i]))
        tp, tm = th.copy(), th.copy()
        tp[i] += eps
        tm[i] -= eps
        lp = chk.run(H, L, tp, x, tgt, lam, n_norm, all_double=True)[0] / n_norm
        lm = chk.run(H, L, tm, x, tgt, lam, n_norm, all_double=True)[0] / n_norm
        fd = (lp - lm) / (2 * eps)
        assert abs(fd - got[i]) <= 1e-6 * gmax + 1e-12, (i, fd, got[i], gmax)


@pytest.mark.parametrize("H,L", [(8, 1), (8, 2), (6, 3), (16, 5)])
def test_checker_fp32_forward_is_the_oracle(port, chk, H, L):
    w = _deep_weights(H, L, 3, 0.5, port)
    x = _points(53, H + L, -2.0, 2.0)
    _, _, y = chk.run(H, L, _theta(w), x, np.zeros_like(x))
    W1, b1, Wh, bh, W2, b2 = w
    want = port.mlp_forward_deep(x, L, W1, b1, Wh, bh, W2, b2, 53, 4, H, 4)
    assert np.array_equal(y.ravel().view(np.uint32), want.view(np.uint32))


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


@pytest.fixture(scope="module")
def sass():
    from phys_autodiff_b200 import capi
    p = capi.library_path()
    if not os.path.exists(p):
        capi.build_library()
    return _sass_counts(p)


def test_forward_at_points_kernel_sass(sass):
    """k_mlp_deep's points mode (4th template argument true): strict, FMUL2 / FADD2 never contracted, no FFMA at all."""
    ks = {k: v for k, v in sass.items() if re.search(r"k_mlp_deepILi\d+ELb0ELi\d+ELb1E", k)}
    assert len(ks) == 3, ks
    for k, v in ks.items():
        assert v["FMUL2"] > 0 and v["FADD2"] >= v["FMUL2"] and v["FFMA"] == 0 and v["FFMA2"] == 0 and v["UTCHMMA"] == 0, (k, v)


def test_data_gradient_kernel_sass(sass):
    """k_deep_data_grad<H>: the recomputed forward keeps FMUL2 / FADD2 separate (no FFMA2 anywhere), no tcgen05."""
    ks = {k: v for k, v in sass.items() if "k_deep_data_grad" in k}
    assert len(ks) == 3, ks
    for k, v in ks.items():
        assert v["FMUL2"] > 0 and v["FADD2"] >= v["FMUL2"] and v["FFMA2"] == 0 and v["UTCHMMA"] == 0, (k, v)


def test_data_kernels_have_no_spills(tmp_path):
    nvcc = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    if not os.path.exists(nvcc):
        pytest.skip("nvcc unavailable")
    src = os.path.join(ROOT, "phys_autodiff_b200", "csrc", "deep_data_kernels.cu")
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
def _set(ctx, H, L, w, m1p1=True):
    from phys_autodiff_b200 import MLPConfig
    ctx.set_weights_deep(MLPConfig(4, H, 4, m1p1), L, *w)


def _dev(a):
    import torch
    return torch.from_numpy(np.ascontiguousarray(a, np.float32)).cuda()


FWD_SHAPES = [(H, L) for H in (32, 64, 128) for L in (1, 2, 3, 5)] + [(64, 4), (128, 6)]   # L - 1 > 2: streamed weights


@pytest.mark.gpu
@pytest.mark.parametrize("H,L", FWD_SHAPES)
def test_forward_at_points_is_the_oracle_bit_for_bit(ctx, port, H, L):
    w = _deep_weights(H, L, 777, 0.25, port)
    _set(ctx, H, L, w)
    sizes = [1, 191, 192, 193, 4099] + ([100007] if (H, L) in ((64, 3), (128, 6), (32, 1)) else [])
    for B in sizes:
        x = _points(B, B + H + L, -3.0, 3.0)   # inside and outside [-1, 1]
        got = ctx.mlp_forward_deep(_dev(x)).cpu().numpy()
        want = port.mlp_forward_deep(x, L, *w, B, 4, H, 4)
        assert got.shape == (B, 4)
        assert np.array_equal(got.ravel().view(np.uint32), want.view(np.uint32)), (B, np.abs(got.ravel() - want).max())
    assert ctx.mlp_forward_deep(_dev(np.zeros((0, 4)))).shape == (0, 4)


@pytest.mark.gpu
@pytest.mark.parametrize("m1p1", [True, False])
@pytest.mark.parametrize("H,L", [(32, 3), (64, 2), (128, 4)])
def test_forward_at_grid_coordinates_is_the_grid_kernel(ctx, port, H, L, m1p1):
    from phys_autodiff_b200 import Grid
    og = OGrid(33, 18, 7, 1, 1, 1, 1e-3, True)
    w = _deep_weights(H, L, 5, 0.25, port)
    _set(ctx, H, L, w, m1p1)
    t = 0.3
    x = port.make_grid_coords(og, t, m1p1).reshape(-1, 4)
    got = ctx.mlp_forward_deep(_dev(x)).cpu().numpy()
    grid = ctx.mlp_grid_infer_deep(Grid(og.nx, og.ny, og.nz), t).cpu().numpy()
    assert np.array_equal(got.view(np.uint32), grid.view(np.uint32))


@pytest.mark.gpu
@pytest.mark.parametrize("H", [32, 64, 128])
def test_forward_one_hidden_layer_is_mlp_forward(ctx, port, H):
    from phys_autodiff_b200 import MLPConfig
    W1, b1, W2, b2 = port.mlp_random_init(H, 9, 0.5)
    x = _points(5003, H, -1.5, 1.5)
    ctx.set_weights(MLPConfig(4, H, 4, True), W1, b1, W2, b2)
    one = ctx.mlp_forward(_dev(x)).cpu().numpy()
    ctx.set_weights_deep(MLPConfig(4, H, 4, True), 1, W1, b1, None, None, W2, b2)
    deep = ctx.mlp_forward_deep(_dev(x)).cpu().numpy()
    assert np.array_equal(one.view(np.uint32), deep.view(np.uint32))
    assert np.array_equal(ctx.mlp_forward_deep_host(x).view(np.uint32), deep.view(np.uint32))


GRAD_CASES = [
    # (H, L, B, lam, n_norm)
    (32, 1, 1000, None, None),
    (32, 2, 1, LAM, None),
    (32, 3, 769, None, 5000),          # H = 32 tile is 768 points: one tail row
    (64, 2, 385, LAM, None),
    (64, 3, 4096, None, None),
    (64, 5, 20011, LAM, 30000),
    (128, 2, 193, None, None),
    (128, 4, 3000, LAM, None),
    (128, 6, 1531, None, None),        # streamed weights, L = 6
    (64, 1, 191, LAM, 191),
]


@pytest.mark.gpu
@pytest.mark.parametrize("H,L,B,lam,n_norm", GRAD_CASES)
def test_gradient_vs_checker(ctx, port, chk, H, L, B, lam, n_norm):
    w = _deep_weights(H, L, 777, 0.25, port)
    x = _points(B, H + L + B, -1.2, 1.2)
    tgt = _points(B, B, -0.5, 0.5)
    n = B if n_norm is None else n_norm
    acc, want, _ = chk.run(H, L, _theta(w), x, tgt, lam, n)
    _set(ctx, H, L, w)
    out = ctx.deep_data_loss_grad_acc(_dev(x), _dev(tgt), lam, n).cpu().numpy()
    assert out.shape == (_plen(H, L) + 1,)
    assert abs(out[0] - acc) <= 1e-6 * abs(acc)
    assert_grad_close(out[1:], want, H, L, TOL_GRAD)


@pytest.mark.gpu
@pytest.mark.parametrize("H", [32, 64, 128])
def test_one_hidden_layer_matches_mlp_backward(ctx, port, H):
    """lam = NULL and n_norm = B: the reference's mean((y - target)^2) of mlp_backward."""
    from phys_autodiff_b200 import MLPConfig
    W1, b1, W2, b2 = port.mlp_random_init(H, 21, 0.5)
    B = 5000
    x = _points(B, 1, -1.0, 1.0)
    tgt = _points(B, 2, -0.5, 0.5)
    ctx.set_weights(MLPConfig(4, H, 4, True), W1, b1, W2, b2)
    ref = np.concatenate([np.asarray(a, np.float64) for a in ctx.mlp_backward_host(x, tgt)])
    ctx.set_weights_deep(MLPConfig(4, H, 4, True), 1, W1, b1, None, None, W2, b2)
    got = ctx.deep_data_loss_grad_acc(_dev(x), _dev(tgt)).cpu().numpy()[1:]
    # layouts: mlp_backward gives dW1 | db1 | dW2 | db2; with L = 1 the deep layout is the same
    assert_grad_close(got, ref, H, 1, TOL_GRAD)


@pytest.mark.gpu
def test_deterministic_and_all_forms_agree(ctx, port):
    from phys_autodiff_b200 import MLPConfig, ops
    H, L, B = 64, 3, 30011
    w = _deep_weights(H, L, 777, 0.25, port)
    x, tgt = _points(B, 3, -1, 1), _points(B, 4, -0.5, 0.5)
    _set(ctx, H, L, w)
    xd, td = _dev(x), _dev(tgt)
    a = ctx.deep_data_loss_grad_acc(xd, td, LAM).cpu().numpy()
    for _ in range(5):
        b = ctx.deep_data_loss_grad_acc(xd, td, LAM).cpu().numpy()
        assert np.array_equal(a.view(np.uint64), b.view(np.uint64))
    ld, g = ctx.deep_data_loss_grad(xd, td, LAM)
    assert ld == a[0] / B and np.array_equal(g.view(np.uint64), a[1:].view(np.uint64))
    hst = ctx.deep_data_loss_grad_host(x, tgt, LAM)
    assert hst[0] == np.float32(a[0] / B)
    assert np.array_equal(np.concatenate(hst[1:]), a[1:].astype(np.float32))
    mod = ops.mlp_data_loss_deep_grad_cuda(MLPConfig(4, H, 4, True), L, w, x, tgt, LAM)
    assert all(np.array_equal(p, q) for p, q in zip(mod, hst))
    y = ops.mlp_infer_deep_cuda(MLPConfig(4, H, 4, True), L, w, x)
    assert np.array_equal(y.view(np.uint32), port.mlp_forward_deep(x, L, *w, B, 4, H, 4).reshape(B, 4).view(np.uint32))


@pytest.mark.gpu
@pytest.mark.parametrize("H,L", [(32, 2), (64, 3), (128, 4)])
def test_shards_sum_to_the_whole(ctx, port, H, L):
    w = _deep_weights(H, L, 777, 0.25, port)
    B = 10007
    x, tgt = _points(B, 5, -1, 1), _points(B, 6, -0.5, 0.5)
    _set(ctx, H, L, w)
    whole = ctx.deep_data_loss_grad_acc(_dev(x), _dev(tgt), LAM).cpu().numpy()
    for world in (2, 3, 8):
        cuts = [0] + [(r * B) // world for r in range(1, world)] + [B]
        cuts[1] = 0   # the first shard is empty
        tot = np.zeros_like(whole)
        for r in range(world):
            lo, hi = cuts[r], cuts[r + 1]
            tot += ctx.deep_data_loss_grad_acc(_dev(x[lo:hi]), _dev(tgt[lo:hi]), LAM, B).cpu().numpy()
        assert abs(tot[0] - whole[0]) <= 1e-12 * abs(whole[0]), world
        assert np.abs(tot[1:] - whole[1:]).max() <= 1e-5 * np.abs(whole[1:]).max(), world
    z = ctx.deep_data_loss_grad_acc(_dev(np.zeros((0, 4))), _dev(np.zeros((0, 4))), LAM, B).cpu().numpy()
    assert z.shape == (_plen(H, L) + 1,) and not z.any()
    hz = ctx.deep_data_loss_grad_host(np.zeros((0, 4)), np.zeros((0, 4)))
    assert hz[0] == 0 and not any(a.any() for a in hz[1:])


@pytest.mark.gpu
def test_error_paths(port):
    """Status codes, never a silent switch; a refused call writes nothing and leaves the context usable."""
    import torch
    from phys_autodiff_b200 import MLPConfig, PhysadError, capi, ops
    c2 = ops.Context()
    try:
        H, L = 32, 3
        x, tgt = _dev(_points(100, 1)), _dev(_points(100, 2))
        out = torch.full((_plen(H, L) + 1,), 7.0, dtype=torch.float64, device="cuda")
        y = torch.full((100, 4), 7.0, device="cuda")
        lib = capi.lib()
        c2.cfg, c2.hidden_layers = MLPConfig(4, H, 4, True), L
        E_NOWEIGHTS = lib.physad_mlp_forward_deep_dev(c2._h, capi.ptr(x), capi.ptr(y), C.c_size_t(100), None)
        assert E_NOWEIGHTS == -3
        with pytest.raises(PhysadError, match="set_weights_deep"):
            c2.deep_data_loss_grad_acc(x, tgt, out=out)
        w = _deep_weights(H, L, 1, 0.1, port)
        _set(c2, H, L, w)
        c2.set_weights(MLPConfig(4, H, 4, True), w[0], w[1], w[4], w[5])   # back to one hidden layer: not a deep network
        c2.hidden_layers = L
        with pytest.raises(PhysadError, match="set_weights_deep"):
            c2.mlp_forward_deep(x)
        with pytest.raises(PhysadError, match="set_weights_deep"):
            c2.deep_data_loss_grad_acc(x, tgt, out=out)
        _set(c2, H, L, w)
        c2.set_deep_mode(1)
        with pytest.raises(PhysadError, match="strict"):
            c2.mlp_forward_deep(x)
        with pytest.raises(PhysadError, match="strict"):
            c2.deep_data_loss_grad_acc(x, tgt, out=out)
        c2.set_deep_mode(0)
        for lam in ((1, 1, -1, 1), (1, float("nan"), 1, 1), (float("inf"), 1, 1, 1)):
            with pytest.raises(PhysadError, match="lam"):
                c2.deep_data_loss_grad_acc(x, tgt, lam, out=out)
        with pytest.raises(PhysadError, match="n_norm"):
            c2.deep_data_loss_grad_acc(x, tgt, n_norm=0, out=out)
        E_INVALID = lib.physad_deep_data_loss_grad_dev(c2._h, None, capi.ptr(tgt), C.c_size_t(100), None, C.c_size_t(100),
                                                       capi.ptr(out), capi.ptr(out[1:]), None)
        assert E_INVALID == -1
        assert lib.physad_deep_data_loss_grad_dev(c2._h, C.c_void_p(x.data_ptr() + 4), capi.ptr(tgt), C.c_size_t(99), None,
                                                  C.c_size_t(100), capi.ptr(out), capi.ptr(out[1:]), None) == E_INVALID
        assert lib.physad_deep_data_loss_grad_dev(c2._h, capi.ptr(x), capi.ptr(tgt), C.c_size_t(100), None, C.c_size_t(100),
                                                  None, capi.ptr(out[1:]), None) == E_INVALID
        assert lib.physad_mlp_forward_deep_dev(c2._h, C.c_void_p(x.data_ptr() + 8), capi.ptr(y), C.c_size_t(99), None) == E_INVALID
        assert lib.physad_mlp_forward_deep_dev(c2._h, capi.ptr(x), None, C.c_size_t(100), None) == E_INVALID
        assert lib.physad_mlp_forward_deep_dev(None, None, None, C.c_size_t(0), None) == E_INVALID
        assert lib.physad_deep_data_loss_grad_host(None, None, None, C.c_size_t(0), None, None, None, None, None, None, None,
                                                   None) == E_INVALID
        torch.cuda.synchronize()
        assert bool((out == 7.0).all()) and bool((y == 7.0).all())   # nothing written by a refused call
        # a bad call leaves the context usable
        r = c2.deep_data_loss_grad_acc(x, tgt).cpu().numpy()
        assert np.isfinite(r).all() and r[0] > 0
    finally:
        c2.close()


@pytest.mark.gpu
def test_training_with_a_data_term(ctx, port):
    """Adam on L_sigma + L_u + L_d at 32^3, H = 64, L = 3, the data term at 4 096 points of a teacher network at t = 0: the
    data loss falls by >= 90 % in 200 steps and the physics loss falls too.  Measured on a B200: L_d 9.2e-2 -> 5.5e-5
    (-99.94 %), L_sigma + L_u 9.9e-3 -> 5.1e-5, so both thresholds hold with a wide margin."""
    from phys_autodiff_b200 import Grid, PhysWeights
    g = Grid(32, 32, 32, 1, 1, 1, 2e-3, True)
    H, L = 64, 3
    pw = PhysWeights(1, 1)
    x = _points(4096, 99, -1, 1)
    x[:, 3] = 0.0
    xd = _dev(x)
    _set(ctx, H, L, _deep_weights(H, L, 4242, 0.25, port))
    yd = ctx.mlp_forward_deep(xd).clone()
    w0 = _deep_weights(H, L, 777, 0.25, port)
    th = _theta(w0)
    cuts = np.cumsum([a.size for a in w0])[:-1]
    m, v = np.zeros_like(th), np.zeros_like(th)
    hist = []
    for k in range(1, 201):
        _set(ctx, H, L, np.split(th.astype(np.float32), cuts))
        ls, lu, gp = ctx.deep_loss_grad(g, pw, 0.25, 2e-3)
        ld, gd = ctx.deep_data_loss_grad(xd, yd)
        hist.append((float(ls) + float(lu), ld))
        gvec = gp + gd
        m = 0.9 * m + 0.1 * gvec
        v = 0.999 * v + 0.001 * gvec * gvec
        th = th - 3e-3 * (m / (1 - 0.9 ** k)) / (np.sqrt(v / (1 - 0.999 ** k)) + 1e-8)
    (p0, d0), (p1, d1) = hist[0], hist[-1]
    print("physics", p0, "->", p1, " data", d0, "->", d1)
    assert np.isfinite(p1) and np.isfinite(d1)
    assert d1 <= 0.1 * d0, (d0, d1)
    assert p1 < p0, (p0, p1)


WORKER = r'''
import os, sys, json
sys.path.insert(0, %r)
import numpy as np, torch, torch.distributed as dist
from phys_autodiff_b200 import MLPConfig, ops
rank, world, local = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"]), int(os.environ["LOCAL_RANK"])
torch.cuda.set_device(local)
dist.init_process_group("nccl", device_id=torch.device("cuda", local))
ctx = ops.Context(local)
H, L, N = 64, 3, 50021
W1, b1, W2, b2 = ops.mlp_random_init(H, 777, 0.25)
rng = np.random.default_rng(7)
Wh = rng.uniform(-0.2, 0.2, (L - 1) * H * H).astype(np.float32)
bh = rng.uniform(-0.2, 0.2, (L - 1) * H).astype(np.float32)
ctx.set_weights_deep(MLPConfig(4, H, 4, True), L, W1, b1, Wh, bh, W2, b2)
x = np.random.default_rng(1).uniform(-1, 1, (N, 4)).astype(np.float32)
t = np.random.default_rng(2).uniform(-1, 1, (N, 4)).astype(np.float32)
lo, hi = (rank * N) // world, ((rank + 1) * N) // world
lam = (0.7, 1.9, 0.0, 0.35)
ld, g = ctx.deep_data_loss_grad(torch.from_numpy(x[lo:hi]).cuda(), torch.from_numpy(t[lo:hi]).cuda(), lam)   # n_global found
one = ctx.deep_data_loss_grad_acc(torch.from_numpy(x).cuda(), torch.from_numpy(t).cuda(), lam).cpu().numpy()  # all points here
out = dict(rank=rank, ld=ld, ld1=float(one[0] / N), grad_err=float(np.abs(g - one[1:]).max() / np.abs(one[1:]).max()))
gathered = [None] * world
dist.all_gather_object(gathered, out)
if rank == 0:
    print("RESULT " + json.dumps(gathered))
dist.destroy_process_group()
'''


@pytest.mark.gpu
def test_multi_gpu_data_gradient_matches_single_gpu(tmp_path):
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs >= 2 GPUs")
    script = tmp_path / "worker.py"
    script.write_text(WORKER % ROOT)
    n = min(torch.cuda.device_count(), 8)
    r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={n}",
                        "--master-addr", "127.0.0.1", "--master-port", "29737", str(script)],
                       capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-4000:]
    res = json.loads([ln for ln in r.stdout.splitlines() if ln.startswith("RESULT ")][-1][len("RESULT "):])
    assert len(res) == n
    for d in res:
        assert d["ld"] == res[0]["ld"]
        assert abs(d["ld"] - d["ld1"]) <= 1e-6 * abs(d["ld1"])
        assert d["grad_err"] <= 1e-6, d["grad_err"]
