"""Closed loop of the analytic ("tangent") loss: d(L_sigma + L_u)/d(MLP weights) of the forward-mode physics loss.

There is no reference counterpart, so the chain is pinned as the finite-difference closed loop's is:
  CPU tier   a NumPy restatement of the gradient (below) == central finite differences of its own all-double loss; its
             fp32-faithful mode differentiates the same numbers port.tangent_loss (oracle.c: oracle_tangent_loss) sums;
  GPU tier   physad_tangent_loss_grad_* == the fp32-faithful restatement within TOL_GRAD of the largest gradient entry; its
             sums == physad_tangent_loss_dev's; slabs add up to the grid; the training criterion holds (L falls >= 90 %).
"""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

from helpers import assert_grad_close
from oracle import Grid as OGrid

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
TOL_GRAD = 1e-4   # max |d| / max |grad|, as the finite-difference closed loop: fp32 kernel arithmetic vs the double checker


# ---- the checker: NumPy restatement of the gradient (test infrastructure) ----------------------------------------------
def _axis(n, m1p1):
    """src/mlp_grid.cpp:25-29 in float32: u = float(i) / float(n - 1), MinusOneToOne 2u - 1."""
    if n <= 1:
        return np.zeros(1, np.float32)
    u = np.arange(n, dtype=np.float32) / np.float32(n - 1)
    return np.float32(2) * u - np.float32(1) if m1p1 else u


def _split(theta, H):
    return theta[:4 * H].reshape(H, 4), theta[4 * H:5 * H], theta[5 * H:9 * H].reshape(4, H), theta[9 * H:]


def tangent_grad_ref(g, theta, H, t, w_sigma=1.0, w_u=1.0, m1p1=True, all_double=False):
    """Loss sums and gradient (9H+4 doubles, dW1 | db1 | dW2 | db2) of the analytic loss.

    all_double=False (fp32-faithful): theta holds fp32 weights; the pre-activation z_h is formed in fp32 with the forward's
    roundings (so the ReLU masks are oracle_tangent_loss's), y and J in double, residuals rounded to float, and the VJP
    scale gb = (2w / float(N)) R formed in fp32; the adjoint then runs in double.  all_double=True: everything in double
    -- the differentiable function whose central differences pin the adjoint."""
    theta = np.asarray(theta, np.float64)
    W1, b1, W2, b2 = _split(theta, H)
    nx, ny, nz = g.nx, g.ny, g.nz
    N = nx * ny * nz
    cz, cy, cx = np.meshgrid(_axis(nz, m1p1), _axis(ny, m1p1), _axis(nx, m1p1), indexing="ij")
    c = [cx.ravel(), cy.ravel(), cz.ravel()]
    ct = np.float32(t) if m1p1 else np.float32(t) + np.float32(0.5)
    if all_double:
        z = b1[:, None] + sum(W1[:, k, None] * c[k].astype(np.float64)[None, :] for k in range(3)) + W1[:, 3, None] * float(ct)
    else:
        W1f, b1f = W1.astype(np.float32), b1.astype(np.float32)
        zf = np.broadcast_to(b1f[:, None], (H, N))
        for k in range(3):
            zf = zf + W1f[:, k, None] * c[k][None, :]
        zf = zf + W1f[:, 3, None] * ct
        z = zf.astype(np.float64)
    m = (z > 0).astype(np.float64)
    a = m * z
    y = b2[:, None] + W2 @ a                                   # [4, N]
    J = np.einsum("ohk,hn->okn", W2[:, :, None] * W1[None, :, :], m)   # [4, 4, N]
    f = 2.0 if m1p1 else 1.0
    s = [f / ((n - 1) * float(np.float32(h))) if n > 1 else 0.0 for n, h in ((nx, g.hx), (ny, g.hy), (nz, g.hz))]
    gr = J[:, :3, :] * np.array(s)[None, :, None]              # g[o][j]
    div = gr[1, 0] + gr[2, 1] + gr[3, 2]
    R = J[:, 3, :] + y[1] * gr[:, 0] + y[2] * gr[:, 1] + y[3] * gr[:, 2]
    R[0] += y[0] * div
    if all_double:
        r = R
        gb = np.array([2.0 * w_sigma / N, 2.0 * w_u / N, 2.0 * w_u / N, 2.0 * w_u / N])[:, None] * r
    else:
        r = R.astype(np.float32).astype(np.float64)
        k = np.array([np.float32(2) * np.float32(w_sigma) / np.float32(N)] + [np.float32(2) * np.float32(w_u) / np.float32(N)] * 3,
                     np.float32)
        gb = (k[:, None] * r.astype(np.float32)).astype(np.float64)
    acc_s, acc_u = float(np.sum(r[0] ** 2)), float(np.sum(r[1] ** 2 + r[2] ** 2 + r[3] ** 2))
    yb = np.empty((4, N))
    yb[0] = gb[0] * div
    for j in range(3):
        yb[j + 1] = gb[0] * gr[0, j] + gb[1] * gr[1, j] + gb[2] * gr[2, j] + gb[3] * gr[3, j]
    Jb = np.empty((4, 4, N))
    Jb[:, 3] = gb
    for o in range(4):
        for j in range(3):
            Jb[o, j] = s[j] * (gb[o] * y[j + 1] + (gb[0] * y[0] if o == j + 1 else 0.0))
    dz = m * (W2.T @ yb)                                       # [H, N]
    S = np.einsum("hn,okn->hok", m, Jb)                         # masked sums S_h[o][k]
    cc = np.stack([c[0], c[1], c[2], np.full(N, ct, np.float32)]).astype(np.float64)
    dW1 = dz @ cc.T + np.einsum("oh,hok->hk", W2, S)
    db1 = dz.sum(axis=1)
    dW2 = yb @ a.T + np.einsum("hk,hok->oh", W1, S)
    db2 = yb.sum(axis=1)
    grad = np.concatenate([dW1.ravel(), db1, dW2.ravel(), db2])
    return dict(acc_sigma=acc_s, acc_u=acc_u, loss_sigma=w_sigma * acc_s / N, loss_u=w_u * acc_u / N, grad=grad)


def _theta(w):
    return np.concatenate([np.asarray(x, np.float64).ravel() for x in w])


# ---- CPU tier -------------------------------------------------------------------------------------------------------
CPU_CASES = [
    # shape, H, m1p1, h
    ((7, 6, 5), 16, True, (0.7, 1.1, 0.9)),
    ((7, 6, 5), 16, False, (0.7, 1.1, 0.9)),
    ((9, 4, 6), 8, True, (0.5, 0.25, 2.0)),
    ((1, 1, 1), 8, True, (1, 1, 1)),
    ((5, 1, 1), 8, False, (1, 1, 1)),
    ((1, 4, 3), 8, True, (1, 1, 1)),
    ((1, 4, 3), 8, False, (0.3, 1.7, 1)),
]


@pytest.mark.parametrize("shape,H,m1p1,h", CPU_CASES)
def test_checker_adjoint_matches_finite_differences(port, shape, H, m1p1, h):
    g = OGrid(*shape, *h, 2e-3, True)
    th = _theta(port.mlp_random_init(H, seed=5, scale=0.8))
    r = tangent_grad_ref(g, th, H, 0.25, 1.3, 0.7, m1p1, all_double=True)
    gmax = max(np.abs(r["grad"]).max(), 1e-12)
    rng = np.random.default_rng(1)
    for i in rng.choice(th.size, 40, replace=False):
        e = 1e-6
        tp, tm = th.copy(), th.copy()
        tp[i] += e
        tm[i] -= e
        lp = tangent_grad_ref(g, tp, H, 0.25, 1.3, 0.7, m1p1, all_double=True)
        lm = tangent_grad_ref(g, tm, H, 0.25, 1.3, 0.7, m1p1, all_double=True)
        fd = (lp["loss_sigma"] + lp["loss_u"] - lm["loss_sigma"] - lm["loss_u"]) / (2 * e)
        assert abs(fd - r["grad"][i]) <= 1e-6 * gmax, (i, fd, r["grad"][i], gmax)


@pytest.mark.parametrize("shape,H,m1p1,h", CPU_CASES + [((20, 12, 9), 32, True, (1, 1, 1)), ((13, 7, 5), 128, False, (1, 1, 1))])
def test_checker_fp32_sums_are_the_port_tangent_loss(port, shape, H, m1p1, h):
    """The fp32-faithful mode differentiates the numbers oracle_tangent_loss sums (same masks, same float residuals)."""
    g = OGrid(*shape, *h, 2e-3, True)
    w = port.mlp_random_init(H, 777, 0.25)
    r = tangent_grad_ref(g, _theta(w), H, 0.25, 1.3, 0.7, m1p1)
    want = port.tangent_loss(g, w, 0.25, m1p1)
    assert r["acc_sigma"] == pytest.approx(want["acc_sigma"], rel=1e-14, abs=1e-300)
    assert r["acc_u"] == pytest.approx(want["acc_u"], rel=1e-14, abs=1e-300)
    # and its gradient is the all-double one up to the fp32 rounding of the forward
    rd = tangent_grad_ref(g, _theta(w), H, 0.25, 1.3, 0.7, m1p1, all_double=True)
    assert np.abs(r["grad"] - rd["grad"]).max() <= 1e-5 * np.abs(rd["grad"]).max()


# ---- GPU tier -------------------------------------------------------------------------------------------------------
GPU_CASES = [
    # shape, H, m1p1, h
    ((64, 64, 64), 64, True, (1, 1, 1)),
    ((48, 40, 12), 32, True, (1, 1, 1)),
    ((70, 37, 5), 128, False, (1, 1, 1)),
    ((20, 9, 4), 48, True, (1, 1, 1)),                # padded width
    ((33, 18, 7), 64, False, (0.5, 0.25, 2.0)),       # nx % 32 != 0, anisotropic spacing
    ((96, 64, 24), 32, False, (1, 1, 1)),
    ((132, 7, 3), 128, True, (0.7, 1.1, 0.9)),
    ((1, 1, 1), 16, True, (1, 1, 1)),                 # degenerate extents
    ((5, 1, 1), 64, False, (1, 1, 1)),
    ((1, 4, 3), 32, True, (1, 1, 1)),
]


def _g(og):
    from phys_autodiff_b200 import Grid
    return Grid(og.nx, og.ny, og.nz, og.hx, og.hy, og.hz, og.dt, og.periodic)


@pytest.mark.gpu
@pytest.mark.parametrize("shape,H,m1p1,h", GPU_CASES)
def test_gradient_vs_checker(ctx, port, shape, H, m1p1, h):
    from phys_autodiff_b200 import MLPConfig, PhysWeights
    og = OGrid(*shape, *h, 2e-3, True)
    w = port.mlp_random_init(H, 777, 0.25)
    want = tangent_grad_ref(og, _theta(w), H, 0.25, 1.3, 0.7, m1p1)
    ctx.set_weights(MLPConfig(4, H, 4, m1p1), *w)
    out = ctx.tangent_loss_grad_acc(_g(og), PhysWeights(1.3, 0.7), 0.25).cpu().numpy()
    assert_grad_close(out[2:], want["grad"], H, 1, TOL_GRAD)
    # the sums are the forward kernel's: same residual arithmetic, only the order of the double additions differs
    acc = ctx.tangent_loss_acc(_g(og), 0.25).cpu().numpy()
    assert np.abs(out[:2] - acc).max() <= 1e-12 * np.abs(acc).max() + 1e-300, (out[:2], acc)


@pytest.mark.gpu
def test_gradient_is_deterministic_and_host_form_agrees(ctx, port):
    from phys_autodiff_b200 import MLPConfig, PhysWeights, ops
    og = OGrid(96, 80, 37, 1, 1, 1, 2e-3, True)
    w = port.mlp_random_init(64, 777, 0.25)
    pw = PhysWeights(1.3, 0.7)
    ctx.set_weights(MLPConfig(4, 64, 4, True), *w)
    a = ctx.tangent_loss_grad(_g(og), pw, 0.25)
    for _ in range(5):
        b = ctx.tangent_loss_grad(_g(og), pw, 0.25)
        assert a[0] == b[0] and a[1] == b[1] and np.array_equal(a[2].view(np.uint64), b[2].view(np.uint64))
    hst = ctx.tangent_loss_grad_host(_g(og), MLPConfig(4, 64, 4, True), *w, pw, 0.25)
    assert hst[0] == a[0] and hst[1] == a[1]
    assert np.array_equal(np.concatenate(hst[2:]), a[2].astype(np.float32))
    mod = ops.mlp_phys_loss_tangent_grad_cuda(_g(og), MLPConfig(4, 64, 4, True), w, pw, 0.25)
    assert all(np.array_equal(x, y) for x, y in zip(mod, hst))
    # the losses are the analytic loss's
    lt = ops.mlp_phys_loss_tangent_cuda(_g(og), MLPConfig(4, 64, 4, True), w, pw, 0.25)
    assert abs(lt[0] - a[0]) <= 1e-6 * abs(lt[0]) and abs(lt[1] - a[1]) <= 1e-6 * abs(lt[1])


@pytest.mark.gpu
@pytest.mark.parametrize("shape,H", [((40, 24, 13), 64), ((33, 9, 3), 32), ((128, 8, 10), 128), ((20, 9, 17), 48)])
def test_slab_gradients_sum_to_the_whole(ctx, port, shape, H):
    """Multi-GPU decomposition on one device: the slab sums (scaled by the whole grid's N) add up to the whole grid's."""
    from phys_autodiff_b200 import MLPConfig, PhysWeights
    from phys_autodiff_b200.ops import slab_for_rank
    og = OGrid(*shape, 1, 1, 1, 2e-3, True)
    ctx.set_weights(MLPConfig(4, H, 4, True), *port.mlp_random_init(H, 777, 0.25))
    pw = PhysWeights(1.3, 0.7)
    whole = ctx.tangent_loss_grad_acc(_g(og), pw, 0.25).cpu().numpy()
    for world in (2, 3, 8):
        tot = np.zeros_like(whole)
        for r in range(world):
            tot += ctx.tangent_loss_grad_acc(_g(og), pw, 0.25, slab_for_rank(og.nz, r, world)).cpu().numpy()
        assert np.abs(tot[:2] - whole[:2]).max() <= 1e-12 * np.abs(whole[:2]).max()
        # the fp32 sums over 32 points fall on different points when a slab starts elsewhere
        assert np.abs(tot[2:] - whole[2:]).max() <= 2e-6 * np.abs(whole[2:]).max(), world
    z = ctx.tangent_loss_grad_acc(_g(og), pw, 0.25, (og.nz // 2, og.nz // 2)).cpu().numpy()
    assert z.shape == (9 * H + 6,) and not z.any()


@pytest.mark.gpu
def test_training_reduces_the_analytic_loss_by_90_percent(ctx, port):
    """The closed-loop criterion of REQUIREMENT.md:164-169 on the analytic loss: host-side Adam, L falls >= 90 %."""
    from phys_autodiff_b200 import MLPConfig, PhysWeights
    og = OGrid(32, 32, 32, 1, 1, 1, 2e-3, True)
    H = 64
    cfg, pw = MLPConfig(4, H, 4, True), PhysWeights(1, 1)
    th = _theta(port.mlp_random_init(H, 777, 0.25))
    m, v = np.zeros_like(th), np.zeros_like(th)
    first = last = None
    for k in range(1, 121):
        w = [th[:4 * H], th[4 * H:5 * H], th[5 * H:9 * H], th[9 * H:]]
        ls, lu, *d = ctx.tangent_loss_grad_host(_g(og), cfg, *[x.astype(np.float32) for x in w], pw, 0.25)
        L = float(ls) + float(lu)
        first = L if first is None else first
        last = L
        gvec = np.concatenate(d).astype(np.float64)
        m = 0.9 * m + 0.1 * gvec
        v = 0.999 * v + 0.001 * gvec * gvec
        th = th - 3e-3 * (m / (1 - 0.9 ** k)) / (np.sqrt(v / (1 - 0.999 ** k)) + 1e-8)
    assert np.isfinite(last) and last <= 0.1 * first, (first, last)


@pytest.mark.gpu
def test_gradient_error_paths(port):
    """Status codes, not crashes: no weights, unsupported shapes, deeper networks, bad slabs, null pointers."""
    import ctypes as C
    from phys_autodiff_b200 import Grid, MLPConfig, PhysadError, PhysWeights, capi, ops
    c2 = ops.Context()
    try:
        g, pw = Grid(8, 8, 8, 1, 1, 1, 1e-3, True), PhysWeights(1, 1)
        c2.cfg = MLPConfig(4, 16, 4, True)
        with pytest.raises(PhysadError, match="no weights"):
            c2.tangent_loss_grad_acc(g, pw, 0.1)
        c2.set_weights(MLPConfig(4, 256, 4, True), *port.mlp_random_init(256, 1, 0.1))
        with pytest.raises(PhysadError, match="H > 128"):
            c2.tangent_loss_grad_acc(g, pw, 0.1)
        w3 = port.mlp_random_init(16, 1, 0.1, In=3)
        c2.set_weights(MLPConfig(3, 16, 4, True), *w3)
        with pytest.raises(PhysadError, match="In = Out = 4"):
            c2.tangent_loss_grad_acc(g, pw, 0.1)
        w = port.mlp_random_init(32, 1, 0.1)
        rng = np.random.default_rng(0)
        c2.set_weights_deep(MLPConfig(4, 32, 4, True), 2, w[0], w[1], rng.uniform(-0.2, 0.2, 32 * 32).astype(np.float32),
                            rng.uniform(-0.2, 0.2, 32).astype(np.float32), w[2], w[3])
        with pytest.raises(PhysadError, match="one-hidden-layer"):
            c2.tangent_loss_grad_acc(g, pw, 0.1)
        c2.set_weights(MLPConfig(4, 16, 4, True), *port.mlp_random_init(16, 1, 0.1))
        with pytest.raises(PhysadError):
            c2.tangent_loss_grad_acc(Grid(0, 8, 8), pw, 0.1)
        with pytest.raises(PhysadError, match="slab"):
            c2.tangent_loss_grad_acc(g, pw, 0.1, (4, 12))
        with pytest.raises(PhysadError, match="slab"):
            c2.tangent_loss_grad_acc(g, pw, 0.1, (5, 3))
        lib = capi.lib()
        E_INVALID = lib.physad_tangent_loss_grad_dev(c2._h, None, None, None, C.c_float(0), None, None, None)
        assert E_INVALID != 0
        assert lib.physad_tangent_loss_grad_host(None, None, None, None, None, None, None, None, C.c_float(0),
                                                 None, None, None, None, None, None) == E_INVALID
        # a bad call leaves the context usable
        out = c2.tangent_loss_grad_acc(g, pw, 0.1).cpu().numpy()
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
ctx.set_weights(MLPConfig(4, 64, 4, True), *ops.mlp_random_init(64, 777, 0.25))
pw = PhysWeights(1.3, 0.7)
ls, lu, gr = ctx.tangent_loss_grad(g, pw, 0.25)                       # slab per rank + one all-reduce
one = ctx.tangent_loss_grad_acc(g, pw, 0.25).cpu().numpy()             # the whole grid on this rank's device
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
                        "--master-addr", "127.0.0.1", "--master-port", "29733", str(script)],
                       capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-4000:]
    res = json.loads([ln for ln in r.stdout.splitlines() if ln.startswith("RESULT ")][-1][len("RESULT "):])
    assert len(res) == n
    for d in res:
        assert d["ls"] == res[0]["ls"] and d["lu"] == res[0]["lu"]
        assert abs(d["ls"] - d["ls1"]) <= 1e-6 * abs(d["ls1"]) and abs(d["lu"] - d["lu1"]) <= 1e-6 * abs(d["lu1"])
        assert d["grad_err"] <= 2e-6, d["grad_err"]
