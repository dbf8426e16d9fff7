"""Vector-Jacobian products of deeper networks at points, and the autograd module over them.

mlp_vjp_deep(x, ybar) = sum_i ybar_i . dy_i/dtheta and mlp_jacobian_vjp_deep(x, ybar, Jbar) adds sum_i Jbar_i : dJ_i/dtheta,
both the plain sum over the points.  phys_autodiff_b200.autograd.DeepMLP runs the library's forward (or Jacobian) in its
forward and these calls in its backward, so losses written in PyTorch train the network.

The checker is tests/deep_vjp_checker.c (which includes the derivative and data checkers), compiled here into a temporary
library.  CPU tier: the all-double VJPs against central finite differences of sum ybar.y + sum Jbar:J, the faithful mode
against the data and derivative checkers, zero cotangents, SASS and registers of the two kernels, and the example's
refusals.  GPU tier: the bit-for-bit anchors against the data, pair and derivative losses; both calls against the checker;
losses written in PyTorch against the fused physics loss and against a float64 PyTorch restatement of the network; weight
states, error paths, shards, every entry point, training, the example and torchrun."""
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
TILE_DATA = {32: 768, 64: 384, 128: 192}   # rows per tile of k_deep_data_grad / k_vjp_points
TILE_TAN = {32: 128, 64: 64, 128: 32}      # points per tile of k_colloc_tangent / k_vjp_tangent
LAM = (0.7, 1.9, 0.0, 0.35)
E_INVALID, E_UNSUPPORTED, E_NOWEIGHTS = -1, -2, -3


def _plen(H, L):
    return 9 * H + 4 + (L - 1) * (H * H + H)


def _theta(w):
    return np.concatenate([np.asarray(a, np.float64).ravel() for a in w if a is not None])


def _deep_weights(H, L, seed=777, scale=0.25):
    """test_deep_data.py's draw: the reference initialisation for layers 1 and 2, hidden layers uniform in +-0.2."""
    import oracle
    W1, b1, W2, b2 = oracle.port().mlp_random_init(H, seed, scale)
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


def _weights(H, L):
    return _depth_weights(H, L, 100 + H + L) if L == 16 else _deep_weights(H, L, 777, 0.25)


def _cot(B, seed, which="both"):
    """(x [B, 4] in [-1.5, 1.5], ybar [B, 4], Jbar [B, 4, 4]) float32; which: 'y' (Jbar zero), 'J' (ybar zero) or 'both'."""
    rng = np.random.default_rng(seed)
    x = rng.uniform(-1.5, 1.5, (B, 4)).astype(np.float32)
    yb = rng.uniform(-1, 1, (B, 4)).astype(np.float32)
    Jb = rng.uniform(-1, 1, (B, 4, 4)).astype(np.float32)
    if which == "y":
        Jb[:] = 0
    if which == "J":
        yb[:] = 0
    return x, yb, Jb


class VjpChecker:
    """ctypes surface of tests/deep_vjp_checker.c and the checkers it includes."""

    def __init__(self, path):
        self.lib = C.CDLL(path)

    @staticmethod
    def _fp(a):
        return None if a is None else a.ctypes.data_as(C.c_void_p)

    def vjp(self, H, L, theta, x, yb, Jb=None, all_double=False):
        theta = np.ascontiguousarray(theta, np.float64)
        x, yb = np.ascontiguousarray(x, np.float32), np.ascontiguousarray(yb, np.float32)
        Jb = None if Jb is None else np.ascontiguousarray(Jb, np.float32)
        grad = np.empty(_plen(H, L), np.float64)
        rc = self.lib.oracle_jacobian_vjp_deep(C.c_int(H), C.c_int(L), self._fp(theta), self._fp(x), self._fp(yb), self._fp(Jb),
                                               C.c_size_t(x.size // 4), C.c_int(int(all_double)), self._fp(grad))
        assert rc == 0
        return grad

    def objective(self, H, L, theta, x, yb, Jb=None):
        out = C.c_double()
        theta = np.ascontiguousarray(theta, np.float64)
        rc = self.lib.oracle_vjp_objective(C.c_int(H), C.c_int(L), self._fp(theta), self._fp(x), self._fp(yb), self._fp(Jb),
                                           C.c_size_t(x.size // 4), C.byref(out))
        assert rc == 0
        return out.value

    def data(self, H, L, theta, x, target, lam, n_norm):
        """oracle_data_loss_grad_deep (faithful) -> (grad, y)."""
        theta = np.ascontiguousarray(theta, np.float64)
        B = x.size // 4
        acc, grad, y = C.c_double(), np.empty(_plen(H, L), np.float64), np.empty((B, 4), np.float32)
        lw = (C.c_float * 4)(*[float(v) for v in lam])
        assert self.lib.oracle_data_loss_grad_deep(C.c_int(H), C.c_int(L), self._fp(theta), self._fp(x), self._fp(target),
                                                   C.c_size_t(B), lw, C.c_size_t(n_norm), C.c_int(0), C.byref(acc),
                                                   self._fp(grad), self._fp(y)) == 0
        return grad, y

    def deriv(self, H, L, theta, x, d, g, lam, n_norm):
        theta = np.ascontiguousarray(theta, np.float64)
        acc, grad = C.c_double(), np.empty(_plen(H, L), np.float64)
        lw = (C.c_float * 4)(*[float(v) for v in lam])
        assert self.lib.oracle_deriv_loss_grad_deep(C.c_int(H), C.c_int(L), self._fp(theta), self._fp(x), self._fp(d), self._fp(g),
                                                    C.c_size_t(x.size // 4), lw, C.c_size_t(n_norm), C.c_int(0), C.byref(acc),
                                                    self._fp(grad)) == 0
        return grad

    def jacobian(self, H, L, theta, x):
        theta = np.ascontiguousarray(theta, np.float64)
        B = x.size // 4
        y, J = np.empty((B, 4), np.float32), np.empty((B, 4, 4), np.float32)
        assert self.lib.oracle_jacobian_deep(C.c_int(H), C.c_int(L), self._fp(theta), self._fp(x), C.c_size_t(B), self._fp(y),
                                             self._fp(J)) == 0
        return y, J


@pytest.fixture(scope="module")
def chk(tmp_path_factory):
    out = str(tmp_path_factory.mktemp("deep_vjp_checker") / "libdeepvjp.so")
    src = os.path.join(ROOT, "tests", "deep_vjp_checker.c")
    subprocess.run([os.environ.get("CC", "gcc"), "-std=c11", "-O3", "-ffp-contract=off", "-fPIC", "-shared", "-o", out, src, "-lm"],
                   check=True, capture_output=True)
    return VjpChecker(out)


def _deriv_seeds(J, d, g, lam, n_norm):
    """The derivative-fit loss's tangent-row seeds in fp32, in the kernel's order (DESIGN section 4.13), numpy form."""
    f = np.float32
    D = (((d[:, None, 0] * J[:, :, 0]).astype(f) + (d[:, None, 1] * J[:, :, 1]).astype(f)).astype(f)
         + (d[:, None, 2] * J[:, :, 2]).astype(f)).astype(f)
    D = (D + (d[:, None, 3] * J[:, :, 3]).astype(f)).astype(f)
    coef = np.array([np.float32(2.0 * float(np.float32(l)) / n_norm) for l in lam], f)
    ce = (coef[None, :] * (D - g).astype(f)).astype(f)
    return (ce[:, :, None] * d[:, None, :]).astype(f)


# ---------------------------------------------------------------------------------------------------------------------
# CPU tier
# ---------------------------------------------------------------------------------------------------------------------
FD_CASES = [(L, B, which) for L in (1, 2, 3) for B in (1, 5, 37) for which in ("y", "J", "both")]


@pytest.mark.parametrize("L,B,which", FD_CASES)
def test_checker_vjp_matches_finite_differences(chk, L, B, which):
    H = 6
    th = _theta(_deep_weights(H, L, 11, 0.6))
    x, yb, Jb = _cot(B, 100 * L + B + len(which), which)
    jac = which != "y"
    got = chk.vjp(H, L, th, x, yb, Jb if jac else None, all_double=True)
    if jac:   # the value-only form equals the Jacobian form with Jbar = 0
        assert np.array_equal(chk.vjp(H, L, th, x, yb, np.zeros_like(Jb), True), chk.vjp(H, L, th, x, yb, None, True))
    gmax = np.abs(got).max()
    assert gmax > 0
    rng = np.random.default_rng(L + B)
    for i in rng.choice(th.size, size=min(40, th.size), replace=False):
        eps = 1e-6 * max(1.0, abs(th[i]))
        tp, tm = th.copy(), th.copy()
        tp[i] += eps
        tm[i] -= eps
        Jx = Jb if jac else None
        fd = (chk.objective(H, L, tp, x, yb, Jx) - chk.objective(H, L, tm, x, yb, Jx)) / (2 * eps)
        assert abs(fd - got[i]) <= 1e-6 * gmax + 1e-12, (i, fd, got[i], gmax)


@pytest.mark.parametrize("H,L,B", [(6, 1, 9), (8, 2, 31), (16, 4, 17)])
def test_faithful_vjp_is_the_data_and_derivative_gradients(chk, H, L, B):
    """ybar = fl(coef) (y - target) gives the data checker's gradient; Jbar = the derivative checker's seeds its gradient."""
    th = _theta(_deep_weights(H, L, 5, 0.5))
    rng = np.random.default_rng(H + L)
    x = rng.uniform(-1.5, 1.5, (B, 4)).astype(np.float32)
    t = rng.uniform(-0.5, 0.5, (B, 4)).astype(np.float32)
    want, y = chk.data(H, L, th, x, t, LAM, B)
    coef = np.array([np.float32(2.0 * float(np.float32(l)) / B) for l in LAM], np.float32)
    yb = (coef[None, :] * (y - t).astype(np.float32)).astype(np.float32)
    got = chk.vjp(H, L, th, x, yb)
    assert np.abs(got - want).max() <= 1e-12 * np.abs(want).max()
    d = rng.uniform(-2, 2, (B, 4)).astype(np.float32)
    g = rng.uniform(-0.5, 0.5, (B, 4)).astype(np.float32)
    _, J = chk.jacobian(H, L, th, x)
    Jb = _deriv_seeds(J, d, g, LAM, B)
    want = chk.deriv(H, L, th, x, d, g, LAM, B)
    got = chk.vjp(H, L, th, x, np.zeros_like(x), Jb)
    assert np.abs(got - want).max() <= 1e-12 * np.abs(want).max()
    assert not got[-4:].any()


@pytest.mark.parametrize("all_double", [False, True])
def test_zero_cotangents_give_zero(chk, all_double):
    x, yb, Jb = _cot(23, 3)
    th = _theta(_deep_weights(8, 3, 5, 0.5))
    assert not chk.vjp(8, 3, th, x, np.zeros_like(yb), np.zeros_like(Jb), all_double).any()
    assert not chk.vjp(8, 3, th, x, np.zeros_like(yb), None, all_double).any()


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


def test_vjp_kernels_sass():
    """k_vjp_points / k_vjp_tangent: the value rows keep FMUL2 / FADD2 separate, no FFMA2 anywhere, no tcgen05."""
    from phys_autodiff_b200 import capi
    p = capi.library_path()
    if not os.path.exists(p):
        capi.build_library()
    counts = _sass_counts(p)
    for name in ("k_vjp_points", "k_vjp_tangent"):
        ks = {k: v for k, v in counts.items() if name in k}
        assert len(ks) == 3, ks
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
    props = re.findall(r"Function properties for \S*?(k_\w+?)ILi(\d+)E\w*\n\s+(\d+) bytes stack frame, (\d+) bytes "
                       r"spill stores, (\d+) bytes spill loads\nptxas info\s+: Used (\d+) registers", r.stderr)
    return {(k, int(H)): (int(st), int(sp), int(sl), int(reg)) for k, H, st, sp, sl, reg in props if k != "k_deep_data_reduce"}


def test_vjp_kernels_have_no_spills(tmp_path):
    """Measured with CUDA 12.9 (registers at H = 32 / 64 / 128): k_vjp_points 237 / 227 / 222 against k_deep_data_grad's
    243 / 255 / 224; k_vjp_tangent 249 / 255 / 255 against k_colloc_tangent<H, true>'s 255 / 255 / 234.  No spills.
    Both kernels run one 256-thread block per SM (__launch_bounds__(256, 1)), so up to 255 registers cost no occupancy;
    k_vjp_tangent<128> is the one case above its sibling + 8 (see DESIGN section 4.14)."""
    for mine_src, base_src, mine, base, over in (("vjp_points_kernels.cu", "deep_data_kernels.cu", "k_vjp_points",
                                                  "k_deep_data_grad", ()),
                                                 ("vjp_tangent_kernels.cu", "colloc_tangent_kernels.cu", "k_vjp_tangent",
                                                  "k_colloc_tangent", (128,))):
        m, b = _ptxas(tmp_path, mine_src), _ptxas(tmp_path, base_src)
        assert sorted(m) == [(mine, H) for H in (32, 64, 128)], m
        for (_, H), (st, sp, sl, reg) in m.items():
            assert st == 0 and sp == 0 and sl == 0, (mine, H, m)
            assert reg <= 255
            if H not in over:
                assert reg <= b[(base, H)][3] + 8, (mine, H, reg, b)


def test_example_refuses_torch_without_a_bridge_form():
    for extra in (["--layers", "1", "--torch"], ["--layers", "3", "--torch"], ["--layers", "1", "--colloc", "64", "--torch"]):
        r = subprocess.run([sys.executable, os.path.join(ROOT, "examples", "train_closed_loop.py"), *extra],
                           capture_output=True, text=True, timeout=300)
        assert r.returncode != 0 and "--torch" in r.stderr, (extra, r.stderr[-2000:])


# ---------------------------------------------------------------------------------------------------------------------
# GPU tier
# ---------------------------------------------------------------------------------------------------------------------
def _set(ctx, H, L, w):
    from phys_autodiff_b200 import MLPConfig
    ctx.set_weights_deep(MLPConfig(4, H, 4, True), L, *w)


def _dev(a):
    import torch
    return torch.from_numpy(np.ascontiguousarray(a, np.float32)).cuda()


def _u64(t):
    return t.cpu().numpy().view(np.uint64)


ANCHOR_CASES = [(H, L) for H in (32, 64, 128) for L in (1, 2, 3, 5, 16)]


@pytest.mark.gpu
@pytest.mark.parametrize("H,L", ANCHOR_CASES)
def test_bit_for_bit_anchors(ctx, H, L):
    """The VJPs with the data, pair and derivative losses' seeds formed in torch fp32 give those losses' gradients, bit
    for bit: one backward, one geometry, one reduction order."""
    import torch
    w = _weights(H, L)
    _set(ctx, H, L, w)
    f32 = torch.float32
    for B in sorted({1, TILE_DATA[H] - 1, TILE_DATA[H] + 1, TILE_TAN[H] - 1, TILE_TAN[H] + 1, 100003}):
        rng = np.random.default_rng(B + H + L)
        x = _dev(rng.uniform(-1.5, 1.5, (B, 4)))
        t = _dev(rng.uniform(-0.5, 0.5, (B, 4)))
        coef = torch.tensor([np.float32(2.0 * float(np.float32(l)) / B) for l in LAM], dtype=f32, device="cuda")
        # data
        y = ctx.mlp_forward_deep(x)
        g = ctx.mlp_vjp_deep(x, coef * (y - t))
        want = ctx.deep_data_loss_grad_acc(x, t, LAM)[1:]
        assert np.array_equal(_u64(g), _u64(want)), (B, np.abs(g - want).max().item())
        # pairs: rows 2i, 2i + 1 with ybar_q = -ybar_p
        pq = x[: (B // 2) * 2].reshape(-1, 2, 4) if B > 1 else torch.stack([x, x + 0.5], 1)
        n = pq.shape[0]
        cp = torch.tensor([np.float32(2.0 * float(np.float32(l)) / n) for l in LAM], dtype=f32, device="cuda")
        ypq = ctx.mlp_forward_deep(pq.reshape(-1, 4)).reshape(n, 2, 4)
        ybp = cp * (ypq[:, 0] - ypq[:, 1])
        g = ctx.mlp_vjp_deep(pq.reshape(-1, 4), torch.stack([ybp, -ybp], 1).reshape(-1, 4))
        want = ctx.deep_pair_loss_grad_acc(pq, LAM)[1:]
        assert np.array_equal(_u64(g), _u64(want)), (B, "pairs")
        # derivative fit: ybar = 0, Jbar[o][k] = (coef_o (D_o - g_o)) d_k with D_o in section 4.13's order
        d = _dev(rng.uniform(-2, 2, (B, 4)))
        _, J = ctx.mlp_jacobian_deep(x)
        D = ((d[:, None, 0] * J[:, :, 0] + d[:, None, 1] * J[:, :, 1]) + d[:, None, 2] * J[:, :, 2]) + d[:, None, 3] * J[:, :, 3]
        Jb = (coef * (D - t))[:, :, None] * d[:, None, :]
        g = ctx.mlp_jacobian_vjp_deep(x, torch.zeros_like(x), Jb)
        want = ctx.deep_deriv_loss_grad_acc(x, d, t, LAM)[1:]
        assert np.array_equal(_u64(g), _u64(want)), (B, "deriv")
        assert not _u64(g[-4:]).any()   # db2 is +0


CHK_CASES = [(H, L, B) for H in (32, 64, 128) for L in (1, 2, 3, 5, 16) for B in (1, TILE_TAN[H] - 1, TILE_DATA[H] + 1)]
CHK_CASES += [(32, 1, 100003), (64, 2, 100003), (128, 1, 100003)]   # B = 100 003 where the CPU checker stays quick


@pytest.mark.gpu
@pytest.mark.parametrize("H,L,B", CHK_CASES)
def test_vjps_vs_checker(ctx, chk, H, L, B):
    w = _weights(H, L)
    x, yb, Jb = _cot(B, H + 10 * L + B)
    _set(ctx, H, L, w)
    th = _theta(w)
    g = ctx.mlp_vjp_deep(_dev(x), _dev(yb)).cpu().numpy()
    assert_grad_close(g, chk.vjp(H, L, th, x, yb), H, L, 1e-4)
    g = ctx.mlp_jacobian_vjp_deep(_dev(x), _dev(yb), _dev(Jb)).cpu().numpy()
    assert_grad_close(g, chk.vjp(H, L, th, x, yb, Jb), H, L, 1e-4)


# ---- through autograd -------------------------------------------------------------------------------------------------
def _residuals(y, J, s):
    """k_tangent_loss's residuals in torch from (y, J) and the space scales s[3]."""
    gr = J[:, :, :3] * s
    div = (gr[:, 1, 0] + gr[:, 2, 1]) + gr[:, 3, 2]
    R = J[:, :, 3] + ((y[:, 1:2] * gr[:, :, 0] + y[:, 2:3] * gr[:, :, 1]) + y[:, 3:4] * gr[:, :, 2])
    return R[:, 0] + y[:, 0] * div, R[:, 1:]


def _model(ctx, H, L, w):
    from phys_autodiff_b200.autograd import DeepMLP
    return DeepMLP(ctx, H, L, w)


def _flat_grad(m):
    return np.concatenate([p.grad.detach().double().cpu().numpy().ravel() for p in m._params()])


@pytest.mark.gpu
@pytest.mark.parametrize("H,L", [(32, 1), (64, 3), (128, 2), (64, 16)])
def test_torch_physics_loss_equals_the_fused_points_loss(ctx, H, L):
    import torch
    from phys_autodiff_b200 import Grid, PhysWeights, ops
    w = _weights(H, L)
    B = 20011
    rng = np.random.default_rng(H + L)
    x = _dev(rng.uniform(-1, 1, (B, 4)))
    dcdx = ops.grid_input_scales(Grid(32, 17, 9), True)
    pw = PhysWeights(0.7, 1.3)
    m = _model(ctx, H, L, w)
    y, J = m(x, jacobian=True)
    Rs, Ru = _residuals(y, J, torch.tensor(dcdx, device="cuda"))
    ls, lu = pw.w_sigma * (Rs * Rs).sum() / B, pw.w_u * (Ru * Ru).sum() / B
    (ls + lu).backward()
    _set(ctx, H, L, w)
    fs, fu, fg = ctx.deep_tangent_points_loss_grad(x, dcdx, pw)
    assert abs(ls.item() - fs) <= 1e-6 * abs(fs) and abs(lu.item() - fu) <= 1e-6 * abs(fu), (ls.item(), fs, lu.item(), fu)
    assert_grad_close(_flat_grad(m), fg, H, L, 1e-4)


def _net64(params, x, L):
    """The network in float64 torch: params (W1, b1, Wh, bh, W2, b2)."""
    import torch
    W1, b1, Wh, bh, W2, b2 = params
    a = torch.relu(x @ W1.T + b1)
    for l in range(L - 1):
        a = torch.relu(a @ Wh[l].T + bh[l])
    return a @ W2.T + b2


def _losses():
    """Losses the fused calls cannot express, as functions of (x, y, J)."""
    import torch
    s = None

    def source(x, y, J):   # R - f, manufactured forcing
        Rs, Ru = _residuals(y, J, torch.ones(3, dtype=y.dtype, device=y.device))
        f = torch.sin(2 * x[:, 0]) * torch.cos(x[:, 3])
        return ((Rs - f) ** 2).mean() + (Ru ** 2).mean()

    def weighted(x, y, J):   # per-point (causal) weights
        Rs, Ru = _residuals(y, J, torch.tensor([1.5, 0.5, 2.0], dtype=y.dtype, device=y.device))
        wgt = torch.exp(-2.0 * (x[:, 3] + 1))
        return (wgt * (Rs * Rs + (Ru * Ru).sum(1))).mean()

    def huber(x, y, J):   # robust data term
        t = torch.tanh(x[:, :4] * 0.8)
        return torch.nn.functional.huber_loss(y, t, delta=0.05, reduction="mean")

    def mixed(x, y, J):   # a term mixing y and J
        return ((y[:, 0] * J[:, 1, 2] - J[:, 0, 3] * y[:, 3]) ** 2).mean() + 0.1 * (y ** 2).mean()

    del s
    return {"source": source, "weighted": weighted, "huber": huber, "mixed": mixed}


@pytest.mark.gpu
@pytest.mark.parametrize("H,L", [(32, 1), (32, 2), (64, 3), (64, 1)])
@pytest.mark.parametrize("name", ["source", "weighted", "huber", "mixed"])
def test_torch_losses_vs_float64_restatement(ctx, H, L, name):
    """A loss the fused calls cannot express: the bridge's gradient against torch.autograd of a float64 restatement of the
    network with torch.func.jacfwd for J."""
    import torch
    from torch.func import jacfwd, vmap
    w = _weights(H, L)
    B = 4099
    x = _dev(np.random.default_rng(H * L).uniform(-1.2, 1.2, (B, 4)))
    loss = _losses()[name]
    m = _model(ctx, H, L, w)
    y, J = m(x, jacobian=True)
    lb = loss(x, y, J)
    lb.backward()
    nl = L - 1
    shapes = [(H, 4), (H,), (nl, H, H), (nl, H), (4, H), (4,)]
    p64 = [torch.tensor(np.asarray(a if a is not None else np.zeros(0), np.float64).reshape(s), device="cuda",
                        requires_grad=True) for a, s in zip(w, shapes)]
    x64 = x.double()
    y64 = _net64(p64, x64, L)
    J64 = vmap(jacfwd(lambda c: _net64(p64, c[None], L)[0]))(x64)
    l64 = loss(x64, y64, J64)
    l64.backward()
    want = np.concatenate([(p.grad if p.grad is not None else torch.zeros_like(p)).cpu().numpy().ravel() for p in p64])
    assert abs(lb.item() - l64.item()) <= 1e-5 * abs(l64.item())
    assert_grad_close(_flat_grad(m), want, H, L, 1e-4)


@pytest.mark.gpu
def test_add_flat_grad_plus_a_torch_term_equals_the_bridge_doing_both(ctx):
    import torch
    from phys_autodiff_b200 import Grid, ops
    H, L, B = 64, 3, 8191
    w = _weights(H, L)
    rng = np.random.default_rng(4)
    x, xd, t = (_dev(rng.uniform(-1, 1, (B, 4))) for _ in range(3))
    s = torch.tensor(ops.grid_input_scales(Grid(32, 32, 32), True), device="cuda")

    def phys(m):
        y, J = m(x, jacobian=True)
        Rs, Ru = _residuals(y, J, s)
        return ((Rs * Rs).sum() + (Ru * Ru).sum()) / B

    both = _model(ctx, H, L, w)
    (phys(both) + 0.25 * ((both(xd) - t) ** 2).sum() / B).backward()
    mixed = _model(ctx, H, L, w)
    phys(mixed).backward()
    _set(ctx, H, L, w)
    mixed.add_flat_grad(ctx.deep_data_loss_grad_acc(xd, t)[1:])
    assert_grad_close(_flat_grad(mixed), _flat_grad(both), H, L, 1e-4)


@pytest.mark.gpu
def test_weight_states_of_modules(ctx):
    import torch
    H, L, B = 32, 3, 5003
    x = _dev(np.random.default_rng(1).uniform(-1, 1, (B, 4)))
    w1, w2 = _deep_weights(H, L, 1, 0.3), _deep_weights(H, L, 2, 0.3)

    def alone(w):
        m = _model(ctx, H, L, w)
        y, J = m(x, jacobian=True)
        ((y ** 2).sum() + (J ** 2).sum()).backward()
        return _flat_grad(m)

    a1, a2 = alone(w1), alone(w2)
    assert np.abs(a1 - a2).max() > 0
    m1, m2 = _model(ctx, H, L, w1), _model(ctx, H, L, w2)
    y1, J1 = m1(x, jacobian=True)
    y2, J2 = m2(x, jacobian=True)
    ((y1 ** 2).sum() + (J1 ** 2).sum()).backward()   # the context holds m2's weights: re-uploads m1's
    ((y2 ** 2).sum() + (J2 ** 2).sum()).backward()
    assert np.array_equal(_flat_grad(m1), a1) and np.array_equal(_flat_grad(m2), a2)
    # a set_weights_deep between forward and backward: re-upload as well
    m3 = _model(ctx, H, L, w1)
    y3 = m3(x)
    _set(ctx, H, L, w2)
    (y3 ** 2).sum().backward()
    g3 = _flat_grad(m3)
    _set(ctx, H, L, w1)
    assert np.array_equal(g3, ctx.mlp_vjp_deep(x, 2 * ctx.mlp_forward_deep(x)).float().double().cpu().numpy())
    # an optimizer step between forward and backward raises
    m4 = _model(ctx, H, L, w1)
    opt = torch.optim.SGD(m4.parameters(), lr=0.1)
    y4 = m4(x)
    for p in m4.parameters():
        p.grad = torch.ones_like(p)
    opt.step()
    with pytest.raises(RuntimeError, match="modified by an inplace operation"):
        (y4 ** 2).sum().backward()
    # gradients with respect to x are not provided
    with pytest.raises(RuntimeError, match="inputs x"):
        m4(x.clone().requires_grad_(True))


def _probe(c, x, B=64, jac=False, xoff=0, yoff=0, joff=0, goff=0, null=None):
    """A C-ABI device VJP call on a NaN-filled gradient: (status, gradient untouched)."""
    import torch
    from phys_autodiff_b200 import capi
    H = c.cfg.H if c.cfg is not None else 32
    buf = torch.full((_plen(H, 16) + 16,), float("nan"), dtype=torch.float64, device="cuda")
    args = {"x": C.c_void_p(x.data_ptr() + xoff), "ybar": C.c_void_p(x.data_ptr() + yoff),
            "Jbar": C.c_void_p(x.data_ptr() + joff), "grad": C.c_void_p(buf[8:].data_ptr() + goff)}
    if null:
        args[null] = None
    torch.cuda.synchronize()
    lib = capi.lib()
    if jac:
        rc = lib.physad_mlp_jacobian_vjp_deep_dev(c._h, args["x"], args["ybar"], args["Jbar"], C.c_size_t(B), args["grad"], None)
    else:
        rc = lib.physad_mlp_vjp_deep_dev(c._h, args["x"], args["ybar"], C.c_size_t(B), args["grad"], None)
    torch.cuda.synchronize()
    return rc, bool(torch.isnan(buf).all())


@pytest.mark.gpu
def test_error_paths_write_nothing():
    from phys_autodiff_b200 import MLPConfig, capi, ops
    lib = capi.lib()
    c2 = ops.Context()
    try:
        H, L, B = 32, 3, 64
        x = _dev(np.random.default_rng(1).uniform(-1, 1, 16 * B + 16))
        w = _deep_weights(H, L, 1, 0.3)
        for jac in (False, True):
            assert _probe(c2, x, jac=jac) == (E_NOWEIGHTS, True)                        # no weights
        c2.set_weights(MLPConfig(4, H, 4, True), w[0], w[1], w[4], w[5])
        for jac in (False, True):
            assert _probe(c2, x, jac=jac) == (E_NOWEIGHTS, True)                        # one-hidden-layer network
        _set(c2, H, L, w)
        c2.set_weights(MLPConfig(4, H, 4, True), w[0], w[1], w[4], w[5])
        for jac in (False, True):
            assert _probe(c2, x, jac=jac) == (E_NOWEIGHTS, True)                        # set_weights after deep
        _set(c2, H, L, w)
        for jac in (False, True):
            rc, untouched = _probe(c2, x, jac=jac)
            assert rc == 0 and not untouched
        c2.set_deep_mode(1)
        for jac in (False, True):
            assert _probe(c2, x, jac=jac) == (E_UNSUPPORTED, True)                      # tensor-core mode
        c2.set_deep_mode(0)
        for jac in (False, True):
            for kw in ({"null": "x"}, {"null": "ybar"}, {"null": "grad"}, {"xoff": 4}, {"yoff": 8}, {"goff": 4}):
                assert _probe(c2, x, jac=jac, **kw) == (E_INVALID, True), (jac, kw)
        for kw in ({"null": "Jbar"}, {"joff": 4}):
            assert _probe(c2, x, jac=True, **kw) == (E_INVALID, True), kw
        assert lib.physad_mlp_vjp_deep_dev(None, None, None, C.c_size_t(0), None, None) == E_INVALID
        assert lib.physad_mlp_jacobian_vjp_deep_dev(None, None, None, None, C.c_size_t(0), None, None) == E_INVALID
        assert lib.physad_mlp_vjp_deep_host(c2._h, None, None, C.c_size_t(B), *[None] * 6) == E_INVALID
        assert lib.physad_mlp_jacobian_vjp_deep_host(c2._h, None, None, None, C.c_size_t(B), *[None] * 6) == E_INVALID
        # null inputs with B = 0 are an empty shard: a zero gradient
        for jac in (False, True):
            rc, untouched = _probe(c2, x, B=0, jac=jac, null="x")
            assert rc == 0 and not untouched
    finally:
        c2.close()


@pytest.mark.gpu
def test_empty_repeatable_and_all_forms_agree(ctx, tmp_path):
    import torch
    from phys_autodiff_b200 import MLPConfig, capi, ops
    H, L, B = 64, 3, 30011
    w = _deep_weights(H, L)
    x, yb, Jb = _cot(B, 3)
    _set(ctx, H, L, w)
    xd, ybd, Jbd = _dev(x), _dev(yb), _dev(Jb)
    e = torch.zeros((0, 4), device="cuda")
    assert ctx.mlp_vjp_deep(e, e).shape == (_plen(H, L),) and not _u64(ctx.mlp_vjp_deep(e, e)).any()
    assert not _u64(ctx.mlp_jacobian_vjp_deep(e, e, torch.zeros((0, 4, 4), device="cuda"))).any()
    v = ctx.mlp_vjp_deep(xd, ybd)
    j = ctx.mlp_jacobian_vjp_deep(xd, ybd, Jbd)
    for _ in range(3):
        assert np.array_equal(_u64(ctx.mlp_vjp_deep(xd, ybd)), _u64(v))
        assert np.array_equal(_u64(ctx.mlp_jacobian_vjp_deep(xd, ybd, Jbd)), _u64(j))
    v, j = v.cpu().numpy(), j.cpu().numpy()
    hv, hj = ctx.mlp_vjp_deep_host(x, yb), ctx.mlp_jacobian_vjp_deep_host(x, yb, Jb)
    assert np.array_equal(np.concatenate(hv), v.astype(np.float32)) and np.array_equal(np.concatenate(hj), j.astype(np.float32))
    cfg = MLPConfig(4, H, 4, True)
    assert all(np.array_equal(p, q) for p, q in zip(ops.mlp_vjp_deep_cuda(cfg, L, w, x, yb), hv))
    assert all(np.array_equal(p, q) for p, q in zip(ops.mlp_jacobian_vjp_deep_cuda(cfg, L, w, x, yb, Jb), hj))
    # the module: backward of sum(ybar . y + Jbar : J) is the Jacobian VJP, of sum(ybar . y) the value VJP
    m = _model(ctx, H, L, w)
    y, J = m(xd, jacobian=True)
    ((y * ybd).sum() + (J * Jbd).sum()).backward()
    assert np.array_equal(_flat_grad(m), j.astype(np.float32).astype(np.float64))
    m = _model(ctx, H, L, w)
    (m(xd) * ybd).sum().backward()
    assert np.array_equal(_flat_grad(m), v.astype(np.float32).astype(np.float64))
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
        f.write(x.tobytes() + yb.tobytes() + Jb.tobytes())
    r = subprocess.run([str(exe), str(inp), str(outp)], capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stdout + r.stderr
    got = np.fromfile(outp, np.float32)
    P = _plen(H, L)
    assert np.array_equal(got[:P], np.concatenate(hv)) and np.array_equal(got[P:], np.concatenate(hj))


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
    std::vector<float> x, yb, Jb;
    if (!rd(w.W1, 4 * H) || !rd(w.b1, H) || !rd(w.Wh, size_t(L - 1) * H * H) || !rd(w.bh, size_t(L - 1) * H) ||
        !rd(w.W2, 4 * H) || !rd(w.b2, 4) || !rd(x, 4 * B) || !rd(yb, 4 * B) || !rd(Jb, 16 * B)) return 3;
    std::fclose(f);
    phys::MLPGridConfig cfg;
    cfg.dims.In = 4; cfg.dims.H = H; cfg.dims.Out = 4;
    phys::DeepMLPWeights gv, gj;
    phys::mlp_vjp_deep_cuda(cfg, w, x.data(), yb.data(), B, gv);
    phys::mlp_jacobian_vjp_deep_cuda(cfg, w, x.data(), yb.data(), Jb.data(), B, gj);
    FILE* o = std::fopen(argv[2], "wb");
    for (auto* v : {&gv.W1, &gv.b1, &gv.Wh, &gv.bh, &gv.W2, &gv.b2, &gj.W1, &gj.b1, &gj.Wh, &gj.bh, &gj.W2, &gj.b2})
        std::fwrite(v->data(), 4, v->size(), o);
    std::fclose(o);
    return 0;
}
'''


@pytest.mark.gpu
@pytest.mark.parametrize("H,L", [(32, 2), (64, 3), (128, 1)])
def test_shards_sum_to_the_whole(ctx, H, L):
    B = 10007
    _set(ctx, H, L, _deep_weights(H, L))
    x, yb, Jb = _cot(B, 5)
    whole_v = ctx.mlp_vjp_deep(_dev(x), _dev(yb)).cpu().numpy()
    whole_j = ctx.mlp_jacobian_vjp_deep(_dev(x), _dev(yb), _dev(Jb)).cpu().numpy()
    for world in (2, 3, 8):
        cuts = [0] + [(r * B) // world for r in range(1, world)] + [B]
        cuts[1] = 0   # the first shard is empty
        tv, tj = np.zeros_like(whole_v), np.zeros_like(whole_j)
        for r in range(world):
            s = slice(cuts[r], cuts[r + 1])
            tv += ctx.mlp_vjp_deep(_dev(x[s]), _dev(yb[s])).cpu().numpy()
            tj += ctx.mlp_jacobian_vjp_deep(_dev(x[s]), _dev(yb[s]), _dev(Jb[s])).cpu().numpy()
        assert_grad_close(tv, whole_v, H, L, 1e-5)
        assert_grad_close(tj, whole_j, H, L, 1e-5)


def _train(ctx, steps=120):
    """DeepMLP + torch.optim.Adam at H = 64, L = 3: the physics residuals in torch at 32 768 collocation points over
    t in [0, 0.5], a data term at 4 096 teacher points at t = 0 and 4 096 fresh periodic pairs per step."""
    import torch
    from phys_autodiff_b200 import Grid, ops
    H, L = 64, 3
    g = Grid(32, 32, 32, 1, 1, 1, 2e-3, True)
    s = torch.tensor(ops.grid_input_scales(g, True), device="cuda")
    period = torch.tensor(ops.grid_periods(g, True), device="cuda")
    rng = np.random.default_rng(21)
    xc = rng.uniform(-1, 1, (32768, 4)).astype(np.float32)
    xc[:, 3] = rng.uniform(0.0, 0.5, 32768).astype(np.float32)
    xc = _dev(xc)
    xd = rng.uniform(-1, 1, (4096, 4)).astype(np.float32)
    xd[:, 3] = 0.0
    xd = _dev(xd)
    _set(ctx, H, L, _deep_weights(H, L, 4242))
    yd = ctx.mlp_forward_deep(xd).clone()
    m = _model(ctx, H, L, _deep_weights(H, L))
    opt = torch.optim.Adam(m.parameters(), lr=3e-3)
    gen = torch.Generator(device="cuda")
    gen.manual_seed(5)
    rows = torch.arange(4096, device="cuda")
    ax = rows % 3
    hist = []
    for _ in range(steps):
        p = torch.rand((4096, 4), generator=gen, device="cuda") * torch.tensor([2, 2, 2, 0.5], device="cuda") \
            - torch.tensor([1, 1, 1, 0], device="cuda")
        p[rows, ax] = -1.0
        q = p.clone()
        q[rows, ax] += period[ax]
        opt.zero_grad(set_to_none=True)
        y, J = m(xc, jacobian=True)
        Rs, Ru = _residuals(y, J, s)
        ypq = m(torch.stack([p, q], 1).reshape(-1, 4)).reshape(-1, 2, 4)
        loss = (Rs * Rs).mean() + (Ru * Ru).sum(1).mean() + 0.25 * ((m(xd) - yd) ** 2).sum(1).mean() \
            + 0.25 * ((ypq[:, 0] - ypq[:, 1]) ** 2).sum(1).mean()
        loss.backward()
        opt.step()
        hist.append(loss.item())
    return hist


@pytest.mark.gpu
def test_training_through_the_module(ctx):
    hist = _train(ctx)
    print("DeepMLP + Adam", hist[0], "->", hist[-1], "reduction", 1 - hist[-1] / hist[0])
    assert np.isfinite(hist[-1]) and hist[-1] <= 0.1 * hist[0], (hist[0], hist[-1])


@pytest.mark.gpu
def test_example_torch_matches_the_fused_run(tmp_path):
    runs = {}
    for mode in ("fused", "torch"):
        gout = tmp_path / f"{mode}.bin"
        cmd = [sys.executable, os.path.join(ROOT, "examples", "train_closed_loop.py"), "--n", "32", "--layers", "3",
               "--colloc", "8192", "--t-range", "0,0.5", "--data", "1024", "--periodic", "1024", "--steps", "20",
               "--grad-out", str(gout)] + (["--torch"] if mode == "torch" else [])
        r = subprocess.run(cmd, capture_output=True, text=True, timeout=600)
        assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-3000:]
        recs = [json.loads(ln) for ln in r.stdout.splitlines() if ln.startswith("{")]
        runs[mode] = (recs, np.fromfile(gout, np.float64))
    (fr, fg), (tr, tg) = runs["fused"], runs["torch"]
    for key in ("loss_sigma", "loss_u", "loss_data", "loss_periodic"):
        assert abs(tr[0][key] - fr[0][key]) <= 1e-6 * abs(fr[0][key]), (key, tr[0][key], fr[0][key])
    assert_grad_close(tg, fg, 64, 3, 1e-4)
    assert "PyTorch" in tr[-1]["summary"] and np.isfinite(tr[-1]["loss_last"])
    assert tr[-1]["loss_last"] < tr[-1]["loss_first"]


WORKER = r'''
import os, sys, json
sys.path.insert(0, %r)
import numpy as np, torch, torch.distributed as dist
from phys_autodiff_b200 import ops
from phys_autodiff_b200.autograd import DeepMLP
rank, world, local = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"]), int(os.environ["LOCAL_RANK"])
torch.cuda.set_device(local)
dist.init_process_group("nccl", device_id=torch.device("cuda", local))
ctx = ops.Context(local)
H, L, N = 64, 3, 50021
W1, b1, W2, b2 = ops.mlp_random_init(H, 777, 0.25)
rng = np.random.default_rng(7)
Wh = rng.uniform(-0.2, 0.2, (L - 1) * H * H).astype(np.float32)
bh = rng.uniform(-0.2, 0.2, (L - 1) * H).astype(np.float32)
x = torch.from_numpy(np.random.default_rng(1).uniform(-1, 1, (N, 4)).astype(np.float32)).cuda()
lo, hi = (rank * N) // world, ((rank + 1) * N) // world

def loss(m, xs):
    y, J = m(xs, jacobian=True)
    return ((y[:, 0] * J[:, 1, 2]) ** 2).sum() / N + (J[:, :, 3] ** 2).sum() / N

m = DeepMLP(ctx, H, L, (W1, b1, Wh, bh, W2, b2))
loss(m, x[lo:hi]).backward()
for p in m.parameters():
    dist.all_reduce(p.grad)
g = np.concatenate([p.grad.double().cpu().numpy().ravel() for p in m._params()])
m1 = DeepMLP(ctx, H, L, (W1, b1, Wh, bh, W2, b2))
loss(m1, x).backward()
g1 = np.concatenate([p.grad.double().cpu().numpy().ravel() for p in m1._params()])
out = dict(rank=rank, err=float(np.abs(g - g1).max() / np.abs(g1).max()))
gathered = [None] * world
dist.all_gather_object(gathered, out)
if rank == 0:
    print("RESULT " + json.dumps(gathered))
dist.destroy_process_group()
'''


@pytest.mark.gpu
def test_multi_gpu_module_gradient_matches_single_gpu(tmp_path):
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs >= 2 GPUs")
    script = tmp_path / "worker.py"
    script.write_text(WORKER % ROOT)
    n = min(torch.cuda.device_count(), 8)
    r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={n}",
                        "--master-addr", "127.0.0.1", "--master-port", "29743", str(script)],
                       capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-4000:]
    res = json.loads([ln for ln in r.stdout.splitlines() if ln.startswith("RESULT ")][-1][len("RESULT "):])
    assert len(res) == n
    for dd in res:
        assert dd["err"] <= 1e-5, dd
