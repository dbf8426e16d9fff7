"""Neumann boundaries at points: the Jacobian of deeper networks and the derivative-fit loss with its gradient with respect
to every layer's weights, L_g = (1/n_norm) sum_i sum_o lam[o] (D_io - g_io)^2 with D_io = sum_k d_ik dy_o/dc_k.

The checker is tests/deep_deriv_checker.c (which includes the points and tangent checkers), compiled here into a
temporary library.  CPU tier: the all-double gradient against central finite differences, the all-double Jacobian against
central differences of the network, the faithful forward against oracle_mlp_forward_deep, d = e_t against the Jacobian,
a zero direction, and the SASS / register report of k_deriv_tangent.  GPU tier: the Jacobian call bit for bit against
the forward and the checker, and its residuals against the points physics call; the loss call against the faithful
checker at every depth, db2 exactly +0, repeatability and all entry points, shards, the weight states of the context,
error paths, training with a Neumann term, the example, and a torchrun comparison across GPUs."""
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

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
TILE = {32: 128, 64: 64, 128: 32}   # points per tile of k_colloc_tangent / k_deriv_tangent
LAM = (0.7, 1.9, 0.0, 0.35)
E_INVALID, E_UNSUPPORTED, E_NOWEIGHTS = -1, -2, -3


def _plen(H, L):
    return 9 * H + 4 + (L - 1) * (H * H + H)


def _theta(w):
    return np.concatenate([np.asarray(a, np.float64).ravel() for a in w if a is not None])


def _deep_weights(H, L, seed=777, scale=0.25, port=None):
    """test_deep_data.py's draw: the reference initialisation for layers 1 and 2, hidden layers uniform in +-0.2."""
    import oracle
    W1, b1, W2, b2 = (port or oracle.port()).mlp_random_init(H, seed, scale)
    rng = np.random.default_rng(seed + L)
    Wh = rng.uniform(-0.2, 0.2, (L - 1) * H * H).astype(np.float32)
    bh = rng.uniform(-0.2, 0.2, (L - 1) * H).astype(np.float32)
    return W1, b1, Wh, bh, W2, b2


def _depth_weights(H, L, seed):
    """test_deep_depth.py's He-uniform draw, which keeps the signal alive through 16 hidden layers."""
    rng = np.random.default_rng(seed)
    u = lambda n, a: rng.uniform(-a, a, n).astype(np.float32)
    W1, b1 = u(4 * H, np.sqrt(6 / 4)), u(H, 0.1)
    Wh, bh = (u((L - 1) * H * H, np.sqrt(6 / H)), u((L - 1) * H, 0.1)) if L > 1 else (None, None)
    return W1, b1, Wh, bh, u(4 * H, np.sqrt(6 / H)), u(4, 0.1)


def _points(B, seed, kind="mixed", lo=-1.5, hi=1.5, targets=True):
    """(x, d, g) float32 [B, 4]: x uniform in [lo, hi]^4; d along one space axis (a grid-like scale), along t, or general;
    "mixed" cycles through the three; g uniform in +-0.5 (or zero)."""
    rng = np.random.default_rng(seed)
    x = rng.uniform(lo, hi, (B, 4)).astype(np.float32)
    d = np.zeros((B, 4), np.float32)
    for i in range(B):
        k = {"axis": 0, "t": 1, "all": 2}.get(kind, i % 3)
        if k == 0:
            d[i, i % 3] = np.float32(rng.choice([15.5, -15.5, 0.0322581, 1.0]))
        elif k == 1:
            d[i, 3] = np.float32(rng.choice([1.0, -0.75]))
        else:
            d[i] = rng.uniform(-2, 2, 4).astype(np.float32)
    g = rng.uniform(-0.5, 0.5, (B, 4)).astype(np.float32) if targets else np.zeros((B, 4), np.float32)
    return x, d, g


class DerivChecker:
    """ctypes surface of tests/deep_deriv_checker.c and the tangent checker it includes."""

    def __init__(self, path):
        self.lib = C.CDLL(path)

    @staticmethod
    def _fp(a):
        return a.ctypes.data_as(C.c_void_p)

    def run(self, H, L, theta, x, d, g, lam=None, n_norm=None, all_double=False):
        """-> (acc, grad[P] f64)."""
        theta = np.ascontiguousarray(theta, np.float64)
        x, d, g = (np.ascontiguousarray(a, np.float32) for a in (x, d, g))
        B = x.size // 4
        acc = C.c_double()
        grad = np.empty(_plen(H, L), np.float64)
        lw = None if lam is None else (C.c_float * 4)(*[float(v) for v in lam])
        fp = self._fp
        rc = self.lib.oracle_deriv_loss_grad_deep(C.c_int(H), C.c_int(L), fp(theta), fp(x), fp(d), fp(g), C.c_size_t(B), lw,
                                                  C.c_size_t(B if n_norm is None else n_norm), C.c_int(int(all_double)),
                                                  C.byref(acc), fp(grad))
        assert rc == 0
        return acc.value, grad

    def jacobian(self, H, L, theta, x):
        """oracle_jacobian_deep (faithful) -> (y [B, 4], J [B, 4, 4]) float32."""
        theta = np.ascontiguousarray(theta, np.float64)
        x = np.ascontiguousarray(x, np.float32)
        B = x.size // 4
        y, J = np.empty((B, 4), np.float32), np.empty((B, 4, 4), np.float32)
        assert self.lib.oracle_jacobian_deep(C.c_int(H), C.c_int(L), self._fp(theta), self._fp(x), C.c_size_t(B),
                                             self._fp(y), self._fp(J)) == 0
        return y, J

    def point_double(self, H, L, theta, c):
        """oracle_deep_tangent_point in all-double mode -> (y[4], J[4, 4]) float64."""
        theta = np.ascontiguousarray(theta, np.float64)
        c = np.ascontiguousarray(c, np.float64)
        y, J = np.empty(4, np.float64), np.empty(16, np.float64)
        self.lib.oracle_deep_tangent_point(C.c_int(H), C.c_int(L), self._fp(theta), C.c_int(1), self._fp(c), self._fp(y),
                                           self._fp(J))
        return y, J.reshape(4, 4)


@pytest.fixture(scope="module")
def chk(tmp_path_factory):
    out = str(tmp_path_factory.mktemp("deep_deriv_checker") / "libdeepderiv.so")
    src = os.path.join(ROOT, "tests", "deep_deriv_checker.c")
    subprocess.run([os.environ.get("CC", "gcc"), "-std=c11", "-O3", "-ffp-contract=off", "-fPIC", "-shared", "-o", out, src, "-lm"],
                   check=True, capture_output=True)
    return DerivChecker(out)


# ---------------------------------------------------------------------------------------------------------------------
# CPU tier
# ---------------------------------------------------------------------------------------------------------------------
FD_CASES = [(L, B, lam, n, kind) for (L, B), lam, n, kind in zip(
    [(L, B) for L in (1, 2, 3) for B in (1, 5, 37)],
    [None, LAM, LAM, None, LAM, None, LAM, None, LAM],
    [1, 11, 37, 3, 5, 50, 2, 5, 37],
    ["axis", "t", "all", "t", "axis", "mixed", "all", "axis", "mixed"])]


@pytest.mark.parametrize("L,B,lam,n_norm,kind", FD_CASES)
def test_checker_gradient_matches_finite_differences(port, chk, L, B, lam, n_norm, kind):
    H = 6
    th = _theta(_deep_weights(H, L, 11, 0.6, port))
    x, d, g = _points(B, 100 * L + B, kind)
    _, got = chk.run(H, L, th, x, d, g, lam, n_norm, all_double=True)
    gmax = np.abs(got).max()
    assert gmax > 0
    assert not got[-4:].any()   # db2: the value row has no seed
    rng = np.random.default_rng(L + B)
    for i in rng.choice(th.size, size=min(40, th.size), replace=False):
        eps = 1e-6 * max(1.0, abs(th[i]))
        tp, tm = th.copy(), th.copy()
        tp[i] += eps
        tm[i] -= eps
        fd = (chk.run(H, L, tp, x, d, g, lam, n_norm, True)[0] - chk.run(H, L, tm, x, d, g, lam, n_norm, True)[0]) / n_norm / (2 * eps)
        assert abs(fd - got[i]) <= 1e-6 * gmax + 1e-12, (i, fd, got[i], gmax)


@pytest.mark.parametrize("L", [1, 2, 3])
def test_checker_jacobian_matches_central_differences(port, chk, L):
    H = 8
    th = _theta(_deep_weights(H, L, 12, 0.6, port))
    x, _, _ = _points(25, 7 + L)
    for c in x.astype(np.float64):
        _, J = chk.point_double(H, L, th, c)
        for k in range(4):
            eps = 1e-7
            cp, cm = c.copy(), c.copy()
            cp[k] += eps
            cm[k] -= eps
            fd = (chk.point_double(H, L, th, cp)[0] - chk.point_double(H, L, th, cm)[0]) / (2 * eps)
            assert np.abs(fd - J[:, k]).max() <= 1e-6 * max(1.0, np.abs(J).max()), (c, k, fd, J[:, k])


@pytest.mark.parametrize("H,L", [(6, 1), (8, 2), (16, 5)])
def test_faithful_forward_is_the_deep_forward(port, chk, H, L):
    w = _deep_weights(H, L, 3, 0.5, port)
    x, _, _ = _points(41, H + L)
    y, J = chk.jacobian(H, L, _theta(w), x)
    fwd = port.mlp_forward_deep(x, L, *w, 41, 4, H, 4).reshape(41, 4)
    assert np.array_equal(y.view(np.uint32), fwd.view(np.uint32))
    assert np.isfinite(J).all() and np.abs(J).max() > 0


@pytest.mark.parametrize("H,L,lam", [(6, 1, None), (8, 3, LAM)])
def test_time_direction_gives_the_time_derivative(port, chk, H, L, lam):
    """d = e_t, g = 0: D_o = J[o][3] exactly (the other three products are zeros), so the loss is sum lam_o J[o][3]^2."""
    th = _theta(_deep_weights(H, L, 4, 0.5, port))
    x, _, _ = _points(29, 5)
    d = np.tile(np.float32([0, 0, 0, 1]), (29, 1))
    acc, _ = chk.run(H, L, th, x, d, np.zeros_like(x), lam, 29)
    _, J = chk.jacobian(H, L, th, x)
    lw = np.float32(lam if lam is not None else (0.25,) * 4).astype(np.float64)
    want = 0.0
    for i in range(29):
        for o in range(4):
            want += lw[o] * (float(J[i, o, 3]) * float(J[i, o, 3]))
    assert abs(acc - want) <= 1e-14 * abs(want) and want > 0


@pytest.mark.parametrize("all_double", [False, True])
def test_zero_direction_gives_zero(port, chk, all_double):
    x, _, g = _points(17, 4)
    acc, grad = chk.run(8, 3, _theta(_deep_weights(8, 3, 5, 0.5, port)), x, np.zeros_like(x), np.zeros_like(x), LAM, 17, all_double)
    assert acc == 0.0 and not grad.any()
    # a zero direction with non-zero targets: the seeds are zero, only the sum remains
    acc, grad = chk.run(8, 3, _theta(_deep_weights(8, 3, 5, 0.5, port)), x, np.zeros_like(x), g, LAM, 17, all_double)
    assert acc > 0 and not grad.any()


def _sass_counts(path):
    r = subprocess.run(["cuobjdump", "-sass", path], capture_output=True, text=True)
    if r.returncode != 0:
        pytest.skip("cuobjdump unavailable")
    cur, counts = None, {}
    for line in r.stdout.splitlines():
        m = re.search(r"Function : (\S+)", line)
        if m:
            cur = m.group(1)
            counts[cur] = {"FFMA": 0, "FFMA2": 0, "FMUL2": 0, "FADD2": 0, "UTCHMMA": 0, "UTCQMMA": 0, "LDTM": 0, "STTM": 0}
            continue
        m = re.match(r"\s+/\*[0-9a-f]+\*/\s+(?:@!?U?P\d+\s+)?([A-Z0-9_]+)", line)
        if m and cur and m.group(1) in counts[cur]:
            counts[cur][m.group(1)] += 1
    return counts


def test_deriv_kernel_sass():
    """k_deriv_tangent<H, GRAD>: the value row keeps FMUL2 / FADD2 separate, the tangent rows are scalar FFMA, no FFMA2
    anywhere, no tcgen05."""
    from phys_autodiff_b200 import capi
    p = capi.library_path()
    if not os.path.exists(p):
        capi.build_library()
    ks = {k: v for k, v in _sass_counts(p).items() if "k_deriv_tangent" in k}
    assert len(ks) == 6, ks
    for k, v in ks.items():
        assert v["FMUL2"] > 0 and v["FADD2"] >= v["FMUL2"] and v["FFMA"] > 0 and v["FFMA2"] == 0, (k, v)
        assert v["UTCHMMA"] == 0 and v["UTCQMMA"] == 0 and v["LDTM"] == 0 and v["STTM"] == 0, (k, v)


def _ptxas(tmp_path, name):
    nvcc = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    if not os.path.exists(nvcc):
        pytest.skip("nvcc unavailable")
    src = os.path.join(ROOT, "phys_autodiff_b200", "csrc", name)
    r = subprocess.run([nvcc, "-std=c++17", "-O3", "-gencode", "arch=compute_100a,code=sm_100a", "-Xptxas", "-v", "-c",
                        "-o", str(tmp_path / (name + ".o")), src], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr[-2000:]
    props = re.findall(r"Function properties for \S*?(k_\w+?)ILi(\d+)ELb([01])E\w*\n\s+(\d+) bytes stack frame, (\d+) bytes "
                       r"spill stores, (\d+) bytes spill loads\nptxas info\s+: Used (\d+) registers", r.stderr)
    return {(k, int(H), g == "1"): (int(st), int(sp), int(sl), int(reg)) for k, H, g, st, sp, sl, reg in props}


def test_deriv_kernel_has_no_spills_and_the_points_kernels_registers(tmp_path):
    """Measured with CUDA 12.9: k_deriv_tangent 167 / 167 / 167 registers (Jacobian) and 245 / 255 / 232 (loss) at
    H = 32 / 64 / 128; k_colloc_tangent 160 / 167 / 162 and 255 / 255 / 234; no spills."""
    mine = _ptxas(tmp_path, "deriv_tangent_kernels.cu")
    base = _ptxas(tmp_path, "colloc_tangent_kernels.cu")
    assert sorted(mine) == sorted(("k_deriv_tangent", H, g) for H in (32, 64, 128) for g in (False, True)), mine
    for (_, H, g), (st, sp, sl, reg) in mine.items():
        assert st == 0 and sp == 0 and sl == 0, (H, g, mine)
        assert reg <= base[("k_colloc_tangent", H, g)][3] + 8, (H, g, reg, base)


# ---------------------------------------------------------------------------------------------------------------------
# GPU tier
# ---------------------------------------------------------------------------------------------------------------------
def _set(ctx, H, L, w, m1p1=True):
    from phys_autodiff_b200 import MLPConfig
    ctx.set_weights_deep(MLPConfig(4, H, 4, m1p1), L, *w)


def _dev(a):
    import torch
    return torch.from_numpy(np.ascontiguousarray(a, np.float32)).cuda()


def _bits_zero(a):
    """+0.0 bit for bit (not -0.0)."""
    return not np.ascontiguousarray(a, np.float64).view(np.uint64).any()


def _weights(H, L, port):
    return _depth_weights(H, L, 100 + H + L) if L == 16 else _deep_weights(H, L, 777, 0.25, port)


@pytest.mark.gpu
@pytest.mark.parametrize("H,L,B", [(32, 1, 1), (32, 3, 129), (64, 2, 63), (64, 16, 1000), (128, 5, 33), (128, 16, 31),
                                   (64, 3, 100003)])
def test_jacobian_vs_forward_checker_and_residuals(ctx, port, chk, H, L, B):
    from phys_autodiff_b200 import Grid, ops
    w = _weights(H, L, port)
    x, _, _ = _points(B, H + L + B)
    _set(ctx, H, L, w)
    xd = _dev(x)
    y, J = ctx.mlp_jacobian_deep(xd)
    y, J = y.cpu().numpy(), J.cpu().numpy()
    assert y.shape == (B, 4) and J.shape == (B, 4, 4)
    fwd = ctx.mlp_forward_deep(xd).cpu().numpy()
    assert np.array_equal(y.view(np.uint32), fwd.view(np.uint32))
    if B <= 1000 or L < 16:
        cy, cJ = chk.jacobian(H, L, _theta(w), x)
        assert np.array_equal(y.view(np.uint32), cy.view(np.uint32))
        assert np.array_equal(J.view(np.uint32), cJ.view(np.uint32)), np.abs(J - cJ).max()
    # the residuals of the points physics call, recomputed in double from (y, J)
    dcdx = ops.grid_input_scales(Grid(32, 17, 9), True)
    R = ctx._empty(4 * B).view(B, 4)
    ctx.deep_tangent_points_loss_acc(xd, dcdx, residuals=R)
    R = R.cpu().numpy().astype(np.float64)
    yd, Jd, s = y.astype(np.float64), J.astype(np.float64), dcdx.astype(np.float64)
    gr = Jd[:, :, :3] * s            # d y_o / d x_j
    div = gr[:, 1, 0] + gr[:, 2, 1] + gr[:, 3, 2]
    want = Jd[:, :, 3] + np.einsum("bj,boj->bo", yd[:, 1:], gr)
    want[:, 0] += yd[:, 0] * div
    assert np.abs(R - want).max() <= 1e-6 * np.abs(want).max()


# B = 100 003 points only where the CPU checker stays quick
GPU_CASES = [(H, L, B) for H in (32, 64, 128) for L in (1, 2, 3, 5, 16) for B in (1, TILE[H] - 1, TILE[H] + 1)]
GPU_CASES += [(32, 1, 100003), (32, 3, 100003), (64, 2, 100003), (128, 1, 100003)]


@pytest.mark.gpu
@pytest.mark.parametrize("H,L,B", GPU_CASES)
def test_deriv_gradient_vs_checker(ctx, port, chk, H, L, B):
    w = _weights(H, L, port)
    x, d, g = _points(B, H + 10 * L + B)   # inside and outside [-1, 1]
    lam = LAM if (H + L) % 2 else None
    acc, want = chk.run(H, L, _theta(w), x, d, g, lam, B)
    _set(ctx, H, L, w)
    out = ctx.deep_deriv_loss_grad_acc(_dev(x), _dev(d), _dev(g), lam).cpu().numpy()
    assert out.shape == (_plen(H, L) + 1,)
    assert abs(out[0] - acc) <= 1e-6 * abs(acc), (out[0], acc)
    assert _bits_zero(out[-4:]), out[-4:]   # db2: every value-row seed is zero
    assert_grad_close(out[1:], want, H, L, 1e-4)


@pytest.mark.gpu
def test_repeatable_and_all_forms_agree(ctx, port, tmp_path):
    from phys_autodiff_b200 import MLPConfig, capi, ops
    H, L, B = 64, 3, 30011
    w = _deep_weights(H, L, 777, 0.25, port)
    x, d, g = _points(B, 3)
    _set(ctx, H, L, w)
    xd, dd, gd = _dev(x), _dev(d), _dev(g)
    a = ctx.deep_deriv_loss_grad_acc(xd, dd, gd, LAM).cpu().numpy()
    for _ in range(3):
        assert np.array_equal(ctx.deep_deriv_loss_grad_acc(xd, dd, gd, LAM).cpu().numpy().view(np.uint64), a.view(np.uint64))
    lg, gv = ctx.deep_deriv_loss_grad(xd, dd, gd, LAM)
    assert lg == a[0] / B and np.array_equal(gv.view(np.uint64), a[1:].view(np.uint64))
    hst = ctx.deep_deriv_loss_grad_host(x, d, g, LAM)
    assert hst[0] == np.float32(a[0] / B)
    assert np.array_equal(np.concatenate(hst[1:]), a[1:].astype(np.float32))
    mod = ops.mlp_deriv_loss_deep_grad_cuda(MLPConfig(4, H, 4, True), L, w, x, d, g, LAM)
    assert all(np.array_equal(p, q) for p, q in zip(mod, hst))
    y, J = ctx.mlp_jacobian_deep(xd)
    y, J = y.cpu().numpy(), J.cpu().numpy()
    hy, hJ = ctx.mlp_jacobian_deep_host(x)
    assert np.array_equal(hy.view(np.uint32), y.view(np.uint32)) and np.array_equal(hJ.view(np.uint32), J.view(np.uint32))
    my, mJ = ops.mlp_jacobian_deep_cuda(MLPConfig(4, H, 4, True), L, w, x)
    assert np.array_equal(my.view(np.uint32), y.view(np.uint32)) and np.array_equal(mJ.view(np.uint32), J.view(np.uint32))
    # the C++ entry points
    cxx = shutil.which("g++") or shutil.which("c++")
    if cxx is None:
        pytest.skip("no C++ compiler")
    src, exe = tmp_path / "prog.cpp", tmp_path / "prog"
    src.write_text(CXX_PROG)
    libdir = os.path.dirname(capi.library_path())
    r = subprocess.run([cxx, "-std=c++17", "-O2", "-I", os.path.join(ROOT, "include"), "-I", "/usr/local/cuda/include", str(src),
                        "-o", str(exe), libdir + "/libphysad_b200.so", "-Wl,-rpath," + libdir], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr[-3000:]
    inp, outp = tmp_path / "in.bin", tmp_path / "out.bin"
    with open(inp, "wb") as f:
        f.write(np.array([H, L], np.int32).tobytes() + np.array([B], np.uint64).tobytes())
        for arr in w:
            f.write(np.ascontiguousarray(arr, np.float32).tobytes())
        f.write(x.tobytes() + d.tobytes() + g.tobytes() + np.array(LAM, np.float32).tobytes())
    r = subprocess.run([str(exe), str(inp), str(outp)], capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stdout + r.stderr
    got = np.fromfile(outp, np.float32)
    P = _plen(H, L)
    assert got[0] == hst[0] and np.array_equal(got[1:1 + P], np.concatenate(hst[1:]))
    assert np.array_equal(got[1 + P:1 + P + 4 * B], y.ravel()) and np.array_equal(got[1 + P + 4 * B:], J.ravel())


CXX_PROG = r'''
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
    std::vector<float> x, d, g;
    float lam[4];
    if (!rd(w.W1, 4 * H) || !rd(w.b1, H) || !rd(w.Wh, size_t(L - 1) * H * H) || !rd(w.bh, size_t(L - 1) * H) ||
        !rd(w.W2, 4 * H) || !rd(w.b2, 4) || !rd(x, 4 * B) || !rd(d, 4 * B) || !rd(g, 4 * B) ||
        std::fread(lam, 4, 4, f) != 4) return 3;
    std::fclose(f);
    phys::MLPGridConfig cfg;
    cfg.dims.In = 4; cfg.dims.H = H; cfg.dims.Out = 4;
    float loss;
    phys::DeepMLPWeights gr;
    phys::mlp_deriv_loss_deep_grad_cuda(cfg, w, x.data(), d.data(), g.data(), B, lam, &loss, gr);
    std::vector<float> y(4 * B), J(16 * B);
    phys::mlp_jacobian_deep_cuda(cfg, w, x.data(), B, y.data(), J.data());
    FILE* o = std::fopen(argv[2], "wb");
    std::fwrite(&loss, 4, 1, o);
    for (auto* v : {&gr.W1, &gr.b1, &gr.Wh, &gr.bh, &gr.W2, &gr.b2, &y, &J}) std::fwrite(v->data(), 4, v->size(), o);
    std::fclose(o);
    return 0;
}
'''


@pytest.mark.gpu
@pytest.mark.parametrize("H,L", [(32, 2), (64, 3), (128, 4)])
def test_shards_sum_to_the_whole(ctx, port, H, L):
    B = 10007
    _set(ctx, H, L, _deep_weights(H, L, 777, 0.25, port))
    x, d, g = _points(B, 5)
    whole = ctx.deep_deriv_loss_grad_acc(_dev(x), _dev(d), _dev(g), LAM).cpu().numpy()
    for world in (2, 3, 8):
        cuts = [0] + [(r * B) // world for r in range(1, world)] + [B]
        cuts[1] = 0   # the first shard is empty
        tot = np.zeros_like(whole)
        for r in range(world):
            s = slice(cuts[r], cuts[r + 1])
            tot += ctx.deep_deriv_loss_grad_acc(_dev(x[s]), _dev(d[s]), _dev(g[s]), LAM, B).cpu().numpy()
        assert abs(tot[0] - whole[0]) <= 1e-12 * abs(whole[0]), world
        assert np.abs(tot[1:] - whole[1:]).max() <= 1e-5 * np.abs(whole[1:]).max(), world
    e = np.zeros((0, 4), np.float32)
    z = ctx.deep_deriv_loss_grad_acc(_dev(e), _dev(e), _dev(e), LAM, B).cpu().numpy()
    assert z.shape == (_plen(H, L) + 1,) and _bits_zero(z)
    hz = ctx.deep_deriv_loss_grad_host(e, e, e)
    assert hz[0] == 0 and not any(a.any() for a in hz[1:])
    y, J = ctx.mlp_jacobian_deep(_dev(e))
    assert y.shape == (0, 4) and J.shape == (0, 4, 4)


def _probe(c, x, B=64, n_norm=64, lam=None, xoff=0, doff=0, toff=0, aoff=0, goff=0, null=None):
    """The C-ABI device loss call on NaN-filled outputs: (status, outputs untouched)."""
    import torch
    from phys_autodiff_b200 import capi
    H = c.cfg.H if c.cfg is not None else 32
    buf = torch.full((_plen(H, 16) + 16,), float("nan"), dtype=torch.float64, device="cuda")
    args = {"x": C.c_void_p(x.data_ptr() + xoff), "dir": C.c_void_p(x.data_ptr() + doff),
            "target": C.c_void_p(x.data_ptr() + toff), "acc": C.c_void_p(buf.data_ptr() + aoff),
            "grad": C.c_void_p(buf[8:].data_ptr() + goff)}
    if null:
        args[null] = None
    torch.cuda.synchronize()
    rc = capi.lib().physad_deep_deriv_loss_grad_dev(c._h, args["x"], args["dir"], args["target"], C.c_size_t(B), lam,
                                                    C.c_size_t(n_norm), args["acc"], args["grad"], None)
    torch.cuda.synchronize()
    return rc, bool(torch.isnan(buf).all())


def _probe_jac(c, x, B=64, xoff=0, yoff=0, joff=0, null=None):
    """The C-ABI Jacobian call on NaN-filled outputs: (status, outputs untouched)."""
    import torch
    from phys_autodiff_b200 import capi
    buf = torch.full((20 * B + 16,), float("nan"), dtype=torch.float32, device="cuda")
    args = {"x": C.c_void_p(x.data_ptr() + xoff), "y": C.c_void_p(buf.data_ptr() + yoff),
            "J": C.c_void_p(buf[4 * B + 4:].data_ptr() + joff)}
    if null:
        args[null] = None
    torch.cuda.synchronize()
    rc = capi.lib().physad_mlp_jacobian_deep_dev(c._h, args["x"], args["y"], args["J"], C.c_size_t(B), None)
    torch.cuda.synchronize()
    return rc, bool(torch.isnan(buf).all())


@pytest.mark.gpu
def test_weight_states_and_error_paths(port):
    """Both calls over the context's weight states (none, set_weights, deep L = 1, deep L > 1, deep mode 1, after a
    refused set_weights*), and every error path: each refused call returns its status and writes nothing."""
    from phys_autodiff_b200 import MLPConfig, PhysadError, capi, ops
    lib = capi.lib()
    c2 = ops.Context()
    try:
        H, L, B = 32, 3, 64
        x, d, g = _points(B, 1)
        xb = _dev(np.concatenate([x.ravel(), np.zeros(8, np.float32)]))
        xv, dv, gv = _dev(x), _dev(d), _dev(g)
        w = _deep_weights(H, L, 1, 0.3, port)
        for probe in (_probe, _probe_jac):
            assert probe(c2, xb) == (E_NOWEIGHTS, True)                                  # no weights
        c2.set_weights(MLPConfig(4, H, 4, True), w[0], w[1], w[4], w[5])
        for probe in (_probe, _probe_jac):
            assert probe(c2, xb) == (E_NOWEIGHTS, True)                                  # one hidden layer, not deep
        c2.set_weights_deep(MLPConfig(4, H, 4, True), 1, w[0], w[1], None, None, w[4], w[5])
        for probe in (_probe, _probe_jac):                                               # deep, L = 1
            rc, untouched = probe(c2, xb)
            assert rc == 0 and not untouched
        one = c2.deep_deriv_loss_grad_acc(xv, dv, gv).cpu().numpy()
        assert one.shape == (_plen(H, 1) + 1,) and np.isfinite(one).all() and one[0] > 0
        _set(c2, H, L, w)                                                                # deep, L > 1
        deep = c2.deep_deriv_loss_grad_acc(xv, dv, gv).cpu().numpy()
        assert deep.shape == (_plen(H, L) + 1,) and deep[0] > 0
        jac = c2.mlp_jacobian_deep(xv)[1].cpu().numpy()
        c2.set_deep_mode(1)
        for probe in (_probe, _probe_jac):
            assert probe(c2, xb) == (E_UNSUPPORTED, True)                                # tensor-core mode
        with pytest.raises(PhysadError, match="strict"):
            c2.deep_deriv_loss_grad_acc(xv, dv, gv)
        with pytest.raises(PhysadError, match="strict"):
            c2.mlp_jacobian_deep(xv)
        c2.set_deep_mode(0)
        bad = np.zeros(4 * 64, np.float32)                                              # refused set_weights_deep: L = 0
        assert lib.physad_set_weights_deep(c2._h, C.byref(MLPConfig(4, H, 4, True).c()), C.c_int(0), *[ops.ptr(bad)] * 6) != 0
        again = c2.deep_deriv_loss_grad_acc(xv, dv, gv).cpu().numpy()
        assert np.array_equal(again.view(np.uint64), deep.view(np.uint64))              # the network is still in place
        assert np.array_equal(c2.mlp_jacobian_deep(xv)[1].cpu().numpy(), jac)
        for kw in ({"null": "x"}, {"null": "dir"}, {"null": "target"}, {"null": "acc"}, {"null": "grad"}, {"xoff": 4},
                   {"doff": 8}, {"toff": 4}, {"aoff": 4}, {"goff": 4}, {"n_norm": 0},
                   {"lam": (C.c_float * 4)(1, 1, -1, 1)}, {"lam": (C.c_float * 4)(1, float("nan"), 1, 1)},
                   {"lam": (C.c_float * 4)(float("inf"), 1, 1, 1)}):
            assert _probe(c2, xb, **kw) == (E_INVALID, True), kw
        for kw in ({"null": "x"}, {"null": "y"}, {"null": "J"}, {"xoff": 4}, {"yoff": 8}, {"joff": 4}):
            assert _probe_jac(c2, xb, **kw) == (E_INVALID, True), kw
        assert lib.physad_deep_deriv_loss_grad_dev(None, None, None, None, C.c_size_t(0), None, C.c_size_t(1), None, None,
                                                   None) == E_INVALID
        assert lib.physad_deep_deriv_loss_grad_host(c2._h, None, None, None, C.c_size_t(B), None, *[None] * 7) == E_INVALID
        assert lib.physad_deep_deriv_loss_grad_host(None, None, None, None, C.c_size_t(0), None, *[None] * 7) == E_INVALID
        assert lib.physad_mlp_jacobian_deep_dev(None, None, None, None, C.c_size_t(0), None) == E_INVALID
        assert lib.physad_mlp_jacobian_deep_host(c2._h, None, None, None, C.c_size_t(B)) == E_INVALID
        # null inputs with B = 0 are an empty shard, not an error
        assert _probe(c2, xb, B=0, null="x")[0] == 0
        assert _probe_jac(c2, xb, B=0, null="x") == (0, True)
        r = c2.deep_deriv_loss_grad_acc(xv, dv, gv).cpu().numpy()
        assert np.array_equal(r.view(np.uint64), deep.view(np.uint64))                   # a refused call changes nothing
    finally:
        c2.close()


def _face_points(n, rng, dcdx, t_range=(0.0, 0.5)):
    """(x, d) of n points on the faces of the [-1, 1]^3 domain, a third per space axis, alternating c_a = -1 and +1; the
    other space inputs uniform, t in t_range; d = dcdx[a] e_a, the physical normal derivative."""
    x = rng.uniform(-1, 1, (n, 4)).astype(np.float32)
    x[:, 3] = rng.uniform(*t_range, n).astype(np.float32)
    ax = np.arange(n) % 3
    x[np.arange(n), ax] = np.where((np.arange(n) // 3) % 2 == 0, -1.0, 1.0).astype(np.float32)
    d = np.zeros((n, 4), np.float32)
    d[np.arange(n), ax] = np.asarray(dcdx, np.float32)[ax]
    return x, d


def _train(ctx, port, neumann):
    """Adam at H = 64, L = 3: analytic loss at 32 768 collocation points over t in [0, 0.5], data at 4 096 points at t = 0
    (a teacher network), and with `neumann` 4 096 fresh face points per step with a zero normal derivative.
    -> (first total, last total, held-out mean squared normal derivative)."""
    from phys_autodiff_b200 import Grid, PhysWeights, ops
    H, L = 64, 3
    g = Grid(32, 32, 32, 1, 1, 1, 2e-3, False)
    pw = PhysWeights(1, 1)
    dcdx = ops.grid_input_scales(g, True)
    rng = np.random.default_rng(21)
    xc = rng.uniform(-1, 1, (32768, 4)).astype(np.float32)
    xc[:, 3] = rng.uniform(0.0, 0.5, 32768).astype(np.float32)
    xcd = _dev(xc)
    xdat = rng.uniform(-1, 1, (4096, 4)).astype(np.float32)
    xdat[:, 3] = 0.0
    xdd = _dev(xdat)
    _set(ctx, H, L, _deep_weights(H, L, 4242, 0.25, port))
    ydd = ctx.mlp_forward_deep(xdd).clone()
    hx, hd = _face_points(4096, np.random.default_rng(5), dcdx)
    held = (_dev(hx), _dev(hd), _dev(np.zeros_like(hx)))
    frng = np.random.default_rng(77)
    w0 = _deep_weights(H, L, 777, 0.25, port)
    th = _theta(w0)
    cuts = np.cumsum([a.size for a in w0])[:-1]
    m, v = np.zeros_like(th), np.zeros_like(th)
    first = last = None
    for k in range(1, 121):
        _set(ctx, H, L, np.split(th.astype(np.float32), cuts))
        ls, lu, gvec = ctx.deep_tangent_points_loss_grad(xcd, dcdx, pw)
        ld, gd = ctx.deep_data_loss_grad(xdd, ydd)
        total = float(ls) + float(lu) + ld
        gvec = gvec + gd
        if neumann:
            fx, fd = _face_points(4096, frng, dcdx)
            ln, gn = ctx.deep_deriv_loss_grad(_dev(fx), _dev(fd), _dev(np.zeros_like(fx)))
            total += ln
            gvec = gvec + gn
        last = total
        first = last if first is None else first
        m = 0.9 * m + 0.1 * gvec
        v = 0.999 * v + 0.001 * gvec * gvec
        th = th - 3e-3 * (m / (1 - 0.9 ** k)) / (np.sqrt(v / (1 - 0.999 ** k)) + 1e-8)
    _set(ctx, H, L, np.split(th.astype(np.float32), cuts))
    _, J = ctx.mlp_jacobian_deep(held[0])
    J = J.cpu().numpy().astype(np.float64)
    dn = np.einsum("bok,bk->bo", J, hd.astype(np.float64))
    return first, last, float(np.mean(dn * dn))


@pytest.mark.gpu
def test_training_with_a_neumann_term(ctx, port):
    """The total falls by >= 90 % in 120 steps, and the held-out mean squared normal derivative ends below that of the
    same run without the term."""
    first, last, with_term = _train(ctx, port, True)
    _, _, without = _train(ctx, port, False)
    print("neumann training", first, "->", last, "held-out mean squared normal derivative", with_term, "without the term",
          without, "ratio", with_term / without)
    assert np.isfinite(last) and last <= 0.1 * first, (first, last)
    assert with_term < without, (with_term, without)


@pytest.mark.gpu
def test_example_with_neumann_boundaries():
    r = subprocess.run([sys.executable, os.path.join(ROOT, "examples", "train_closed_loop.py"), "--n", "32", "--layers", "3",
                        "--colloc", "8192", "--t-range", "0,0.5", "--data", "1024", "--neumann", "1024", "--steps", "5"],
                       capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-3000:]
    recs = [json.loads(ln) for ln in r.stdout.splitlines() if ln.startswith("{")]
    assert "loss_neumann" in recs[0] and "loss_data" in recs[0] and np.isfinite(recs[-1]["loss_last"])
    assert "Neumann boundaries" in recs[-1]["summary"]


def test_example_refuses_neumann_with_periodic_or_without_colloc():
    for extra in (["--colloc", "64", "--periodic", "8", "--neumann", "8"], ["--neumann", "8"]):
        r = subprocess.run([sys.executable, os.path.join(ROOT, "examples", "train_closed_loop.py"), "--layers", "2", *extra],
                           capture_output=True, text=True, timeout=300)
        assert r.returncode != 0 and "--neumann" in r.stderr, (extra, r.stderr[-2000:])


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
r1 = np.random.default_rng(1)
x, d, g = (r1.uniform(-1, 1, (N, 4)).astype(np.float32) for _ in range(3))
lo, hi = (rank * N) // world, ((rank + 1) * N) // world
lam = (0.7, 1.9, 0.0, 0.35)
t = lambda a: torch.from_numpy(a).cuda()
lg, gr = ctx.deep_deriv_loss_grad(t(x[lo:hi]), t(d[lo:hi]), t(g[lo:hi]), lam)   # n_global found
one = ctx.deep_deriv_loss_grad_acc(t(x), t(d), t(g), lam).cpu().numpy()   # all points here
out = dict(rank=rank, lg=lg, lg1=float(one[0] / N), grad_err=float(np.abs(gr - one[1:]).max() / np.abs(one[1:]).max()))
gathered = [None] * world
dist.all_gather_object(gathered, out)
if rank == 0:
    print("RESULT " + json.dumps(gathered))
dist.destroy_process_group()
'''


@pytest.mark.gpu
def test_multi_gpu_deriv_gradient_matches_single_gpu(tmp_path):
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs >= 2 GPUs")
    script = tmp_path / "worker.py"
    script.write_text(WORKER % ROOT)
    n = min(torch.cuda.device_count(), 8)
    r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={n}",
                        "--master-addr", "127.0.0.1", "--master-port", "29741", str(script)],
                       capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-4000:]
    res = json.loads([ln for ln in r.stdout.splitlines() if ln.startswith("RESULT ")][-1][len("RESULT "):])
    assert len(res) == n
    for dd in res:
        assert dd["lg"] == res[0]["lg"]
        assert abs(dd["lg"] - dd["lg1"]) <= 1e-6 * abs(dd["lg1"])
        assert dd["grad_err"] <= 1e-6, dd["grad_err"]
