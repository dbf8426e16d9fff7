"""Analytic physics loss of deeper networks at arbitrary space-time points (collocation points) and its gradient with
respect to every layer's weights: physad_deep_tangent_points_loss_* and physad_grid_input_scales.

The checker is tests/deep_tangent_points_checker.c (it includes tests/deep_tangent_checker.c), compiled here into a
temporary library.  CPU tier: the all-double gradient against central finite differences, the kernel-faithful points
checker against the grid checker at the grid's own coordinates (bit for bit), the input scales, and k_colloc_tangent's
SASS, registers and spills.  GPU tier: k_colloc_tangent against the faithful checker, bit for bit against the grid calls at
grid coordinates, forms and repeatability, shards, errors, the C++ entry point, training, the example and a torchrun
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
E_INVALID, E_UNSUPPORTED, E_NOWEIGHTS = -1, -2, -3
TILE = {32: 128, 64: 64, 128: 32}   # points per tile of k_colloc_tangent / k_deep_tangent


def _dp(a):
    return a.ctypes.data_as(C.POINTER(C.c_double))


def _fp(a):
    return a.ctypes.data_as(C.POINTER(C.c_float))


def _plen(H, L):
    return 9 * H + 4 + (L - 1) * (H * H + H)


class PointsChecker:
    """ctypes surface of tests/deep_tangent_points_checker.c (and the grid checker it includes)."""

    def __init__(self, path):
        self.lib = C.CDLL(path)
        self.lib.oracle_deep_tangent_points_loss_grad.restype = C.c_int
        self.lib.oracle_deep_tangent_loss_grad.restype = C.c_int

    def points(self, H, L, theta, x, dcdx, w_sigma=1.0, w_u=1.0, n_norm=None, all_double=False, grad=True):
        """-> dict(acc_sigma, acc_u, loss_sigma, loss_u, R [B, 4] f32, grad)."""
        theta = np.ascontiguousarray(theta, np.float64)
        assert theta.size == _plen(H, L)
        x = np.ascontiguousarray(x, np.float32).reshape(-1, 4)
        B = x.shape[0]
        n = B if n_norm is None else n_norm
        d = np.ascontiguousarray(dcdx, np.float64)
        a_s, a_u = C.c_double(), C.c_double()
        R = np.empty((B, 4), np.float32)
        gr = np.empty(theta.size, np.float64) if grad else None
        rc = self.lib.oracle_deep_tangent_points_loss_grad(C.c_int(H), C.c_int(L), _dp(theta), C.c_size_t(B), _fp(x), _dp(d),
                                                           C.c_float(w_sigma), C.c_float(w_u), C.c_size_t(n),
                                                           C.c_int(int(all_double)), C.byref(a_s), C.byref(a_u), _fp(R),
                                                           _dp(gr) if grad else None)
        assert rc == 0
        return dict(acc_sigma=a_s.value, acc_u=a_u.value, loss_sigma=w_sigma * a_s.value / n, loss_u=w_u * a_u.value / n,
                    R=R, grad=gr)

    def grid(self, g, H, L, theta, t, w_sigma, w_u, m1p1):
        """oracle_deep_tangent_loss_grad, kernel-faithful: (acc_sigma, acc_u, R [4][N], grad)."""
        theta = np.ascontiguousarray(theta, np.float64)
        a_s, a_u = C.c_double(), C.c_double()
        R = [np.empty(g.N, np.float32) for _ in range(4)]
        gr = np.empty(theta.size, np.float64)
        rc = self.lib.oracle_deep_tangent_loss_grad(C.byref(g.c()), C.c_int(H), C.c_int(L), C.c_int(int(m1p1)), _dp(theta),
                                                    C.c_float(t), C.c_float(w_sigma), C.c_float(w_u), C.c_int(0),
                                                    C.byref(a_s), C.byref(a_u), *[_fp(r) for r in R], None, _dp(gr))
        assert rc == 0
        return a_s.value, a_u.value, R, gr


@pytest.fixture(scope="module")
def chk(tmp_path_factory):
    out = str(tmp_path_factory.mktemp("deep_tangent_points_checker") / "libdeeptangentpoints.so")
    src = os.path.join(ROOT, "tests", "deep_tangent_points_checker.c")
    subprocess.run([os.environ.get("CC", "gcc"), "-std=c11", "-O3", "-ffp-contract=off", "-fPIC", "-shared", "-o", out, src, "-lm"],
                   check=True, capture_output=True)
    return PointsChecker(out)


def _deep_weights(H, L, seed=777, scale=0.25, port=None):
    import oracle
    W1, b1, W2, b2 = (port or oracle.port()).mlp_random_init(H, seed, scale)
    rng = np.random.default_rng(seed + L)
    Wh = rng.uniform(-0.2, 0.2, (L - 1) * H * H).astype(np.float32)
    bh = rng.uniform(-0.2, 0.2, (L - 1) * H).astype(np.float32)
    return W1, b1, Wh, bh, W2, b2


def _theta(w):
    return np.concatenate([np.asarray(a, np.float64).ravel() for a in w if a is not None])


def _points(B, seed, lo=-1.5, hi=1.5):
    """B points (x, y, z, t) inside and outside [-1, 1], t varying per point."""
    return np.random.default_rng(seed).uniform(lo, hi, (B, 4)).astype(np.float32)


def _grid_scales(og, m1p1):
    """The grid checker's double s[] (deep_tangent_checker.c)."""
    f = 2.0 if m1p1 else 1.0
    n = (og.nx, og.ny, og.nz)
    h = (og.hx, og.hy, og.hz)
    return np.array([f / (float(n[k] - 1) * float(np.float32(h[k]))) if n[k] > 1 else 0.0 for k in range(3)])


# ---------------------------------------------------------------------------------------------------------------------
# CPU tier
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("L", [1, 2, 3])
@pytest.mark.parametrize("B", [1, 5, 37])
def test_checker_gradient_matches_finite_differences(port, chk, L, B):
    """All-double gradient = central differences of the all-double loss, with c_t varying per point, anisotropic dcdx with
    a zero, and n_norm != B."""
    H = 6
    th = _theta(_deep_weights(H, L, 11, 0.6, port))
    x = _points(B, 100 * L + B)
    dcdx = (0.7, 0.0, 1.9)
    ws, wu, n = 1.3, 0.7, B + 3
    got = chk.points(H, L, th, x, dcdx, ws, wu, n, all_double=True)["grad"]
    gmax = np.abs(got).max()
    assert gmax > 0
    rng = np.random.default_rng(B * 31 + L)
    for i in rng.choice(th.size, size=min(40, th.size), replace=False):
        eps = 1e-6 * max(1.0, abs(th[i]))
        tp, tm = th.copy(), th.copy()
        tp[i] += eps
        tm[i] -= eps
        lp = chk.points(H, L, tp, x, dcdx, ws, wu, n, all_double=True, grad=False)
        lm = chk.points(H, L, tm, x, dcdx, ws, wu, n, all_double=True, grad=False)
        fd = ((lp["loss_sigma"] + lp["loss_u"]) - (lm["loss_sigma"] + lm["loss_u"])) / (2 * eps)
        assert abs(fd - got[i]) <= 1e-6 * gmax + 1e-12, (i, fd, got[i], gmax)


@pytest.mark.parametrize("m1p1", [True, False])
@pytest.mark.parametrize("shape,H,L,h", [((5, 4, 3), 8, 2, (1, 1, 1)), ((4, 3, 5), 6, 3, (0.5, 0.25, 2.0)),
                                         ((1, 4, 3), 6, 1, (1, 1, 1)), ((5, 1, 1), 4, 2, (0.7, 1, 1))])
def test_faithful_checker_equals_the_grid_checker_at_grid_coordinates(port, chk, m1p1, shape, H, L, h):
    """x = the grid's points in linear order, dcdx = the grid checker's s[], n_norm = N: the same sums, residuals and
    gradient, bit for bit -- the two checkers compute one function."""
    og = OGrid(*shape, *h, 2e-3, True)
    th = _theta(_deep_weights(H, L, 3, 0.5, port))
    t = 0.25
    a_s, a_u, R, gr = chk.grid(og, H, L, th, t, 1.3, 0.7, m1p1)
    x = port.make_grid_coords(og, t, m1p1).reshape(-1, 4)
    got = chk.points(H, L, th, x, _grid_scales(og, m1p1), 1.3, 0.7, og.N)
    assert got["acc_sigma"] == a_s and got["acc_u"] == a_u
    assert np.array_equal(got["R"].view(np.uint32), np.stack(R, axis=1).view(np.uint32))
    assert np.array_equal(got["grad"].view(np.uint64), gr.view(np.uint64))


@pytest.mark.parametrize("m1p1", [True, False])
def test_grid_input_scales_are_the_checkers_rounded_to_float(m1p1):
    from phys_autodiff_b200 import Grid, PhysadError, ops
    for shape, h in (((48, 40, 12), (1, 1, 1)), ((33, 18, 7), (0.5, 0.25, 2.0)), ((1, 4, 3), (1, 1, 1)),
                     ((5, 1, 1), (0.7, 1.1, 0.9)), ((256, 256, 256), (1, 1, 1)), ((1, 1, 1), (1, 1, 1))):
        og = OGrid(*shape, *h, 2e-3, True)
        got = ops.grid_input_scales(Grid(*shape, *h, 2e-3, True), m1p1)
        assert np.array_equal(got, _grid_scales(og, m1p1).astype(np.float32)), (shape, got)
    for bad in ((Grid(0, 4, 4), 1), (Grid(4, 4, 4), 2), (Grid(4, 4, 4), -1)):
        with pytest.raises(PhysadError, match="grid_input_scales"):
            ops.grid_input_scales(*bad)


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


def test_colloc_kernel_sass():
    """k_colloc_tangent<H, GRAD>: the value row keeps FMUL2 / FADD2 separate, the tangent rows use scalar FFMA; no FFMA2,
    no tcgen05."""
    from phys_autodiff_b200 import capi
    p = capi.library_path()
    if not os.path.exists(p):
        capi.build_library()
    ks = {k: v for k, v in _sass_counts(p).items() if "k_colloc_tangent" in k}
    assert len(ks) == 6, ks
    for k, v in ks.items():
        assert v["FMUL2"] > 0 and v["FADD2"] >= v["FMUL2"] and v["FFMA"] > 0, (k, v)
        assert v["FFMA2"] == 0 and v["UTCHMMA"] == 0, (k, v)


def _ptxas(tmp_path, name):
    nvcc = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    if not os.path.exists(nvcc):
        pytest.skip("nvcc unavailable")
    src = os.path.join(ROOT, "phys_autodiff_b200", "csrc", name)
    r = subprocess.run([nvcc, "-std=c++17", "-O3", "-gencode", "arch=compute_100a,code=sm_100a", "-Xptxas", "-v", "-c",
                        "-o", str(tmp_path / (name + ".o")), src], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr[-2000:]
    props = re.findall(r"Function properties for \S*?(k_\w+?)ILi(\d+)ELb(\d)\w*\n\s+(\d+) bytes stack frame, (\d+) bytes spill stores, "
                       r"(\d+) bytes spill loads\nptxas info\s+: Used (\d+) registers", r.stderr)
    return {(int(H), g == "1"): (int(st), int(sp), int(sl), int(reg)) for _, H, g, st, sp, sl, reg in props}


def test_colloc_kernel_has_no_spills_and_no_more_registers_than_the_grid_kernel(tmp_path):
    pts = _ptxas(tmp_path, "colloc_tangent_kernels.cu")
    grid = _ptxas(tmp_path, "deep_tangent_kernels.cu")
    assert len(pts) == 6 and len(grid) == 6, (pts, grid)
    for key, (st, sp, sl, reg) in pts.items():
        assert st == 0 and sp == 0 and sl == 0, (key, pts[key])
        assert reg <= grid[key][3], (key, reg, grid[key])


# ---------------------------------------------------------------------------------------------------------------------
# GPU tier
# ---------------------------------------------------------------------------------------------------------------------
def _g(og):
    from phys_autodiff_b200 import Grid
    return Grid(og.nx, og.ny, og.nz, og.hx, og.hy, og.hz, og.dt, og.periodic)


def _set(ctx, H, L, w, m1p1=True):
    from phys_autodiff_b200 import MLPConfig
    ctx.set_weights_deep(MLPConfig(4, H, 4, m1p1), L, *w)


def _dev(a):
    import torch
    return torch.from_numpy(np.ascontiguousarray(a, np.float32)).cuda()


DCDX = np.array([0.7, 1.3, 0.25], np.float32)
GPU_CASES = [(H, L, B) for H in (32, 64, 128) for L in (1, 2, 3, 5, 6) for B in (1, TILE[H] - 1, TILE[H] + 1)]
GPU_CASES += [(32, 3, 100003), (64, 2, 100003), (128, 1, 100003)]


@pytest.mark.gpu
@pytest.mark.parametrize("H,L,B", GPU_CASES)
def test_points_loss_and_gradient_vs_checker(ctx, port, chk, H, L, B):
    import torch
    from phys_autodiff_b200 import PhysWeights
    w = _deep_weights(H, L, 777, 0.25, port)
    x = _points(B, H + 10 * L + B)
    want = chk.points(H, L, _theta(w), x, DCDX.astype(np.float64), 1.3, 0.7)
    _set(ctx, H, L, w)
    xd = _dev(x)
    R = torch.empty((B, 4), dtype=torch.float32, device="cuda")
    acc = ctx.deep_tangent_points_loss_acc(xd, DCDX, residuals=R).cpu().numpy()
    for got, ref in zip(acc, (want["acc_sigma"], want["acc_u"])):
        assert abs(got - ref) <= 1e-6 * abs(ref), (got, ref)
    rmax = np.abs(want["R"]).max()
    assert np.abs(R.cpu().numpy() - want["R"]).max() <= 1e-5 * rmax
    out = ctx.deep_tangent_points_loss_grad_acc(xd, DCDX, PhysWeights(1.3, 0.7)).cpu().numpy()
    assert out.shape == (_plen(H, L) + 2,)
    assert np.array_equal(out[:2].view(np.uint64), acc.view(np.uint64))   # the grad call's sums are the loss call's
    assert_grad_close(out[2:], want["grad"], H, L, 1e-4)


@pytest.mark.gpu
@pytest.mark.parametrize("m1p1", [True, False])
@pytest.mark.parametrize("shape,H,L,h", [((40, 24, 13), 64, 3, (1, 1, 1)), ((33, 9, 11), 32, 2, (0.5, 0.25, 2.0)),
                                         ((20, 9, 7), 128, 5, (1, 1, 1)), ((70, 37, 5), 128, 2, (0.7, 1.1, 0.9))])
def test_bit_for_bit_the_grid_calls_at_grid_coordinates(ctx, port, m1p1, shape, H, L, h):
    """x = the grid's points in linear order, dcdx from grid_input_scales: the points calls ARE the grid calls, for the
    whole grid and for a z-slab (x = the slab's points, n_norm = the whole grid's N)."""
    import torch
    from phys_autodiff_b200 import PhysWeights, ops
    og = OGrid(*shape, *h, 2e-3, True)
    g = _g(og)
    t = 0.25
    _set(ctx, H, L, _deep_weights(H, L, 777, 0.25, port), m1p1)
    pw = PhysWeights(1.3, 0.7)
    dcdx = ops.grid_input_scales(g, m1p1)
    x = port.make_grid_coords(og, t, m1p1).reshape(-1, 4)
    pln = og.nx * og.ny
    for z0, z1 in ((0, og.nz), (2, og.nz - 1)):
        xs = _dev(x[z0 * pln:z1 * pln])
        n = (z1 - z0) * pln
        Rg = [torch.empty(n, dtype=torch.float32, device="cuda") for _ in range(4)]
        acc_g = ctx.deep_tangent_loss_acc(g, t, (z0, z1), residuals=Rg).cpu().numpy()
        grad_g = ctx.deep_tangent_loss_grad_acc(g, pw, t, (z0, z1)).cpu().numpy()
        Rp = torch.empty((n, 4), dtype=torch.float32, device="cuda")
        acc_p = ctx.deep_tangent_points_loss_acc(xs, dcdx, residuals=Rp).cpu().numpy()
        grad_p = ctx.deep_tangent_points_loss_grad_acc(xs, dcdx, pw, n_norm=og.N).cpu().numpy()
        assert np.array_equal(acc_p.view(np.uint64), acc_g.view(np.uint64)), (z0, z1)
        assert np.array_equal(grad_p.view(np.uint64), grad_g.view(np.uint64)), (z0, z1)
        Rgs = torch.stack(Rg, dim=1).cpu().numpy()
        assert np.array_equal(Rp.cpu().numpy().view(np.uint32), Rgs.view(np.uint32)), (z0, z1)


@pytest.mark.gpu
def test_repeatable_and_all_forms_agree(ctx, port):
    from phys_autodiff_b200 import MLPConfig, PhysWeights, ops
    H, L, B = 64, 3, 70001
    w = _deep_weights(H, L, 777, 0.25, port)
    pw = PhysWeights(1.3, 0.7)
    _set(ctx, H, L, w)
    x = _points(B, 5)
    xd = _dev(x)
    a = ctx.deep_tangent_points_loss_grad_acc(xd, DCDX, pw).cpu().numpy()
    acc = ctx.deep_tangent_points_loss_acc(xd, DCDX).cpu().numpy()
    assert np.array_equal(a[:2].view(np.uint64), acc.view(np.uint64))
    for _ in range(2):
        assert np.array_equal(ctx.deep_tangent_points_loss_grad_acc(xd, DCDX, pw).cpu().numpy().view(np.uint64), a.view(np.uint64))
        assert np.array_equal(ctx.deep_tangent_points_loss_acc(xd, DCDX).cpu().numpy().view(np.uint64), acc.view(np.uint64))
    ls, lu, gr = ctx.deep_tangent_points_loss_grad(xd, DCDX, pw)
    assert (ls, lu) == ctx.finalize(a[:2], pw, B) and np.array_equal(gr, a[2:])
    hst = ctx.deep_tangent_points_loss_grad_host(x, DCDX, pw)
    assert hst[0] == ls and hst[1] == lu
    assert np.array_equal(np.concatenate(hst[2:]), a[2:].astype(np.float32))
    mod = ops.mlp_phys_loss_deep_tangent_points_grad_cuda(MLPConfig(4, H, 4, True), L, w, x, DCDX, pw)
    assert all(np.array_equal(p, q) for p, q in zip(mod, hst))


@pytest.mark.gpu
@pytest.mark.parametrize("H,L", [(32, 2), (64, 3), (128, 5)])
def test_shards_sum_to_the_whole(ctx, port, H, L):
    """2, 3 and 8 shards, one of them empty, n_norm = the total: cut at multiples of 128 points only the double sums across
    tiles reorder (1e-12); cut anywhere, the fp32 tile sums change too (1e-6 of the largest entry)."""
    from phys_autodiff_b200 import PhysWeights
    B = 128 * 97 + 45
    _set(ctx, H, L, _deep_weights(H, L, 777, 0.25, port))
    pw = PhysWeights(1.3, 0.7)
    x = _points(B, 17)
    whole = ctx.deep_tangent_points_loss_grad_acc(_dev(x), DCDX, pw).cpu().numpy()
    rng = np.random.default_rng(H + L)
    for world in (2, 3, 8):
        for aligned, tol in ((True, 1e-12), (False, 1e-6)):
            if aligned:
                cuts = np.sort(rng.choice(B // 128, world - 2, replace=False) * 128)
            else:
                cuts = np.sort(rng.choice(np.arange(1, B), world - 2, replace=False))
            cuts = np.concatenate([[0], cuts, [cuts[-1] if len(cuts) else 0], [B]])   # one shard empty
            tot = np.zeros_like(whole)
            for lo, hi in zip(cuts[:-1], cuts[1:]):
                part = ctx.deep_tangent_points_loss_grad_acc(_dev(x[lo:hi]), DCDX, pw, n_norm=B).cpu().numpy()
                acc = ctx.deep_tangent_points_loss_acc(_dev(x[lo:hi]), DCDX).cpu().numpy()
                assert np.array_equal(part[:2].view(np.uint64), acc.view(np.uint64))
                tot += part
            assert np.abs(tot[:2] - whole[:2]).max() <= 1e-12 * np.abs(whole[:2]).max(), (world, aligned)
            assert np.abs(tot[2:] - whole[2:]).max() <= tol * np.abs(whole[2:]).max(), (world, aligned)


@pytest.mark.gpu
def test_empty_set_gives_zeros(ctx, port):
    import torch
    from phys_autodiff_b200 import PhysWeights
    H, L = 64, 3
    _set(ctx, H, L, _deep_weights(H, L, 777, 0.25, port))
    x = torch.empty((0, 4), dtype=torch.float32, device="cuda")
    out = torch.full((_plen(H, L) + 2,), float("nan"), dtype=torch.float64, device="cuda")
    ctx.deep_tangent_points_loss_grad_acc(x, DCDX, PhysWeights(1, 1), n_norm=10, out=out)
    assert not out.cpu().numpy().any()
    acc = torch.full((2,), float("nan"), dtype=torch.float64, device="cuda")
    ctx.deep_tangent_points_loss_acc(x, DCDX, acc=acc)
    assert not acc.cpu().numpy().any()
    hst = ctx.deep_tangent_points_loss_grad_host(np.zeros((0, 4), np.float32), DCDX, PhysWeights(1, 1))
    assert all(not np.asarray(a).any() for a in hst)


@pytest.mark.gpu
def test_error_paths_write_nothing(port):
    """Every refused call returns its status and leaves its NaN-filled outputs as they were."""
    import torch
    from phys_autodiff_b200 import MLPConfig, PhysWeights, capi, ops
    lib = capi.lib()
    H, L, B = 32, 3, 300
    P = _plen(H, L)
    c2 = ops.Context()
    try:
        buf = torch.full((P + 2 + 8,), float("nan"), dtype=torch.float64, device="cuda")
        acc, grad = buf[:2], buf[2:2 + P]
        Rbuf = torch.full((4 * B + 8,), float("nan"), dtype=torch.float32, device="cuda")
        R = Rbuf[:4 * B]
        xbuf = _dev(np.concatenate([_points(B, 3).ravel(), np.zeros(8, np.float32)]))
        x = xbuf[:4 * B]
        pw = PhysWeights(1, 1)
        cw = pw.c()
        good = (C.c_float * 3)(*DCDX)
        p = lambda t, off=0: C.c_void_p(t.data_ptr() + off) if t is not None else None

        def loss(xp=p(x), dc=good, ap=p(acc), rp=p(R), n=B):
            return lib.physad_deep_tangent_points_loss_dev(c2._h, xp, C.c_size_t(n), dc, ap, rp, None)

        def lgrad(xp=p(x), dc=good, wp=C.byref(cw), nn=B, ap=p(acc), gp=p(grad), n=B):
            return lib.physad_deep_tangent_points_loss_grad_dev(c2._h, xp, C.c_size_t(n), dc, wp, C.c_size_t(nn), ap, gp, None)

        def untouched():
            torch.cuda.synchronize()
            return bool(torch.isnan(buf).all()) and bool(torch.isnan(Rbuf).all())

        assert loss() == E_NOWEIGHTS and lgrad() == E_NOWEIGHTS and untouched()
        w = _deep_weights(H, L, 1, 0.1, port)
        c2.set_weights(MLPConfig(4, H, 4, True), w[0], w[1], w[4], w[5])   # a one-hidden-layer network: not a deep one
        assert loss() == E_NOWEIGHTS and lgrad() == E_NOWEIGHTS and untouched()
        _set(c2, H, L, w)
        c2.set_deep_mode(1)
        assert loss() == E_UNSUPPORTED and lgrad() == E_UNSUPPORTED and untouched()
        c2.set_deep_mode(0)
        nan3, inf3 = (C.c_float * 3)(0.5, float("nan"), 1.0), (C.c_float * 3)(float("inf"), 0.5, 1.0)
        for rc in (loss(xp=None), loss(dc=None), loss(ap=None), loss(xp=p(x, 4)), loss(rp=p(R, 4)), loss(ap=p(acc, 4)),
                   loss(dc=nan3), loss(dc=inf3),
                   lgrad(xp=None), lgrad(dc=None), lgrad(wp=None), lgrad(ap=None), lgrad(gp=None), lgrad(xp=p(x, 8)),
                   lgrad(ap=p(acc, 4)), lgrad(gp=p(grad, 4)), lgrad(dc=nan3), lgrad(nn=0)):
            assert rc == E_INVALID
        assert untouched()
        assert lib.physad_deep_tangent_points_loss_grad_host(c2._h, None, C.c_size_t(B), good, C.byref(cw), *[None] * 8) == E_INVALID
        assert lib.physad_deep_tangent_points_loss_grad_host(None, None, C.c_size_t(0), good, C.byref(cw), *[None] * 8) == E_INVALID
        # the context is still usable, and one hidden layer set by set_weights_deep runs
        assert loss() == 0 and lgrad() == 0
        torch.cuda.synchronize()
        assert torch.isfinite(acc).all() and torch.isfinite(grad).all() and torch.isfinite(R).all()
        c2.set_weights_deep(MLPConfig(4, H, 4, True), 1, w[0], w[1], None, None, w[4], w[5])
        out = c2.deep_tangent_points_loss_grad_acc(x.view(B, 4), DCDX, pw).cpu().numpy()
        assert out.shape == (_plen(H, 1) + 2,) and np.isfinite(out).all() and out[0] > 0
    finally:
        c2.close()


CXX_PROG = r'''
#include <cmath>
#include <cstdio>
#include <vector>
#include "phys_b200.h"
int main(int argc, char** argv) {
    FILE* f = std::fopen(argv[1], "rb");
    int H, L; unsigned long long B;
    if (std::fread(&H, 4, 1, f) != 1 || std::fread(&L, 4, 1, f) != 1 || std::fread(&B, 8, 1, f) != 1) return 2;
    phys::DeepMLPWeights w;
    w.hidden_layers = L;
    auto rd = [&](std::vector<float>& v, size_t n) { v.resize(n); return std::fread(v.data(), 4, n, f) == n; };
    std::vector<float> x;
    float dcdx[3];
    if (!rd(w.W1, 4 * H) || !rd(w.b1, H) || !rd(w.Wh, size_t(L - 1) * H * H) || !rd(w.bh, size_t(L - 1) * H) ||
        !rd(w.W2, 4 * H) || !rd(w.b2, 4) || !rd(x, 4 * B) || std::fread(dcdx, 4, 3, f) != 3) return 3;
    std::fclose(f);
    phys::MLPGridConfig cfg;
    cfg.dims.In = 4; cfg.dims.H = H; cfg.dims.Out = 4;
    phys::PhysWeights pw;
    pw.w_sigma = 1.3f; pw.w_u = 0.7f;
    float ls, lu, ls2, lu2;
    phys::DeepMLPWeights g;
    std::vector<float> R(4 * B);
    phys::mlp_phys_loss_deep_tangent_points_grad_cuda(cfg, w, pw, x.data(), B, dcdx, &ls, &lu, g);
    phys::mlp_phys_loss_deep_tangent_points_cuda(cfg, w, pw, x.data(), B, dcdx, &ls2, &lu2, R.data());
    FILE* o = std::fopen(argv[2], "wb");
    std::fwrite(&ls, 4, 1, o); std::fwrite(&lu, 4, 1, o); std::fwrite(&ls2, 4, 1, o); std::fwrite(&lu2, 4, 1, o);
    for (auto* v : {&g.W1, &g.b1, &g.Wh, &g.bh, &g.W2, &g.b2}) std::fwrite(v->data(), 4, v->size(), o);
    std::fwrite(R.data(), 4, R.size(), o);
    std::fclose(o);
    return 0;
}
'''


@pytest.mark.gpu
def test_cxx_entry_points_agree_with_the_host_form(ctx, port, tmp_path):
    import torch
    from phys_autodiff_b200 import PhysWeights, capi
    H, L, B = 64, 3, 5000
    w = _deep_weights(H, L, 777, 0.25, port)
    x = _points(B, 8)
    src, exe = tmp_path / "prog.cpp", tmp_path / "prog"
    src.write_text(CXX_PROG)
    libdir = os.path.dirname(capi.library_path())
    cxx = shutil.which("g++") or shutil.which("c++")
    if cxx is None:
        pytest.skip("no C++ compiler")
    r = subprocess.run([cxx, "-std=c++17", "-O2", "-I", os.path.join(ROOT, "include"), "-I", "/usr/local/cuda/include", str(src),
                        "-o", str(exe), libdir + "/libphysad_b200.so", "-Wl,-rpath," + libdir], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr[-3000:]
    inp, outp = tmp_path / "in.bin", tmp_path / "out.bin"
    with open(inp, "wb") as f:
        f.write(np.array([H, L], np.int32).tobytes() + np.array([B], np.uint64).tobytes())
        for a in w:
            f.write(np.ascontiguousarray(a, np.float32).tobytes())
        f.write(x.tobytes() + DCDX.tobytes())
    r = subprocess.run([str(exe), str(inp), str(outp)], capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stdout + r.stderr
    got = np.fromfile(outp, np.float32)
    _set(ctx, H, L, w)
    pw = PhysWeights(1.3, 0.7)
    hst = ctx.deep_tangent_points_loss_grad_host(x, DCDX, pw)
    assert got[0] == hst[0] and got[1] == hst[1] and got[2] == hst[0] and got[3] == hst[1]
    P = _plen(H, L)
    assert np.array_equal(got[4:4 + P], np.concatenate(hst[2:]))
    R = torch.empty((B, 4), dtype=torch.float32, device="cuda")
    ctx.deep_tangent_points_loss_acc(_dev(x), DCDX, residuals=R)
    assert np.array_equal(got[4 + P:], R.cpu().numpy().ravel())


@pytest.mark.gpu
def test_training_on_collocation_points_reduces_the_loss_by_90_percent(ctx, port):
    """Host-side Adam, H = 64, L = 3, learning rate 1e-3, on a fixed set of 32 768 collocation points over t in [0, 0.5]
    (space uniform in [-1, 1]^3, the dc/dx of a 32^3 grid): L_sigma + L_u must fall by at least 90 % in 120 steps."""
    from phys_autodiff_b200 import Grid, PhysWeights, ops
    H, L, B = 64, 3, 32768
    pw = PhysWeights(1, 1)
    rng = np.random.default_rng(21)
    x = rng.uniform(-1, 1, (B, 4)).astype(np.float32)
    x[:, 3] = rng.uniform(0.0, 0.5, B).astype(np.float32)   # MinusOneToOne: the time input is t
    xd = _dev(x)
    dcdx = ops.grid_input_scales(Grid(32, 32, 32), True)
    w0 = _deep_weights(H, L, 777, 0.25, port)
    th = _theta(w0)
    cuts = np.cumsum([a.size for a in w0])[:-1]
    m, v = np.zeros_like(th), np.zeros_like(th)
    first = last = None
    for k in range(1, 121):
        _set(ctx, H, L, np.split(th.astype(np.float32), cuts))
        ls, lu, gvec = ctx.deep_tangent_points_loss_grad(xd, dcdx, pw)
        last = float(ls) + float(lu)
        first = last if first is None else first
        m = 0.9 * m + 0.1 * gvec
        v = 0.999 * v + 0.001 * gvec * gvec
        th = th - 1e-3 * (m / (1 - 0.9 ** k)) / (np.sqrt(v / (1 - 0.999 ** k)) + 1e-8)
    print("collocation training", first, "->", last)
    assert np.isfinite(last) and last <= 0.1 * first, (first, last)


@pytest.mark.gpu
def test_example_trains_initial_condition_and_dynamics():
    r = subprocess.run([sys.executable, os.path.join(ROOT, "examples", "train_closed_loop.py"), "--n", "32", "--layers", "3",
                        "--colloc", "8192", "--t-range", "0,0.5", "--data", "1024", "--steps", "5"],
                       capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-3000:]
    recs = [json.loads(ln) for ln in r.stdout.splitlines() if ln.startswith("{")]
    assert "loss_data" in recs[0] and np.isfinite(recs[-1]["loss_last"])
    assert "collocation points" in recs[-1]["summary"] and "initial condition + dynamics" in recs[-1]["summary"]


WORKER = r'''
import os, sys, json
sys.path.insert(0, %r)
import numpy as np, torch, torch.distributed as dist
from phys_autodiff_b200 import MLPConfig, PhysWeights, ops
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
lo, hi = (rank * N) // world, ((rank + 1) * N) // world
pw, dcdx = PhysWeights(1.3, 0.7), (0.7, 1.3, 0.25)
ls, lu, g = ctx.deep_tangent_points_loss_grad(torch.from_numpy(x[lo:hi]).cuda(), dcdx, pw)   # n_global found
one = ctx.deep_tangent_points_loss_grad_acc(torch.from_numpy(x).cuda(), dcdx, pw).cpu().numpy()   # all points here
l1 = ctx.finalize(one[:2], pw, N)
out = dict(rank=rank, ls=float(ls), lu=float(lu), ls1=float(l1[0]), lu1=float(l1[1]),
           grad_err=float(np.abs(g - one[2:]).max() / np.abs(one[2:]).max()))
gathered = [None] * world
dist.all_gather_object(gathered, out)
if rank == 0:
    print("RESULT " + json.dumps(gathered))
dist.destroy_process_group()
'''


@pytest.mark.gpu
def test_multi_gpu_points_gradient_matches_single_gpu(tmp_path):
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs >= 2 GPUs")
    script = tmp_path / "worker.py"
    script.write_text(WORKER % ROOT)
    n = min(torch.cuda.device_count(), 8)
    r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={n}",
                        "--master-addr", "127.0.0.1", "--master-port", "29738", str(script)],
                       capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-4000:]
    res = json.loads([ln for ln in r.stdout.splitlines() if ln.startswith("RESULT ")][-1][len("RESULT "):])
    assert len(res) == n
    for d in res:
        assert d["ls"] == res[0]["ls"] and d["lu"] == res[0]["lu"]
        assert abs(d["ls"] - d["ls1"]) <= 1e-6 * abs(d["ls1"]) and abs(d["lu"] - d["lu1"]) <= 1e-6 * abs(d["lu1"])
        assert d["grad_err"] <= 1e-6, d["grad_err"]
