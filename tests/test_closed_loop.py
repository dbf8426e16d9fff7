"""Closed loop (SURVEY.md 8f rank 1; reference plan REQUIREMENT.md:155-169): d(L_sigma + L_u)/d(MLP weights).

The reference has no such function (its backward stops at dL/dR), so the chain is pinned differently:
  CPU tier   oracle_grad.c's adjoint == central finite differences of its own all-double loss; its fp32-faithful
             forward == the pinned port's losses (which are pinned to the reference);
  GPU tier   the CUDA kernels == oracle_grad.c (fp32-faithful mode) within TOL_GRAD of the largest gradient entry;
             losses == the fused forward path; and the acceptance test of the plan: training drives L down >= 90 %.
"""
import numpy as np
import pytest

from helpers import assert_grad_close
from oracle import Grid as OGrid

TOL_GRAD = 1e-4   # max |d| / max |grad|: fp32 adjoint arithmetic + fp32 batch sums vs the double checker
TOL_LOSS = 1e-4


def _theta(w):
    return np.concatenate([np.asarray(a, np.float64).ravel() for a in w])


CASES = [
    # shape, H, periodic, m1p1, h, dt
    ((7, 6, 5), 8, True, True, (0.7, 1.1, 0.9), 2e-3),
    ((7, 6, 5), 8, False, True, (0.7, 1.1, 0.9), 2e-3),
    ((1, 4, 3), 8, True, False, (1, 1, 1), 1e-2),
    ((2, 2, 2), 16, False, True, (1, 1, 1), 2e-3),
    ((5, 1, 1), 8, False, False, (1, 1, 1), 2e-3),
    ((1, 1, 1), 8, True, True, (1, 1, 1), 2e-3),
]


@pytest.mark.parametrize("shape,H,per,m1p1,h,dt", CASES)
def test_checker_adjoint_matches_finite_differences(port, shape, H, per, m1p1, h, dt):
    g = OGrid(*shape, *h, dt, per)
    w = port.mlp_random_init(H, seed=5, scale=0.8)
    r = port.phys_loss_grad(g, w, 0.25, dt, 1.3, 0.7, m1p1, all_double=True)
    th = _theta(w)
    ls, lu = port.phys_loss_double(g, th, H, 0.25, dt, 1.3, 0.7, m1p1)
    assert ls == pytest.approx(r["loss_sigma"], rel=1e-13, abs=1e-300) and lu == pytest.approx(r["loss_u"], rel=1e-13, abs=1e-300)
    gmax = max(np.abs(r["grad"]).max(), 1e-12)
    rng = np.random.default_rng(1)
    for i in rng.choice(th.size, 30, replace=False):
        e = 1e-6
        tp, tm = th.copy(), th.copy()
        tp[i] += e
        tm[i] -= e
        fd = (sum(port.phys_loss_double(g, tp, H, 0.25, dt, 1.3, 0.7, m1p1))
              - sum(port.phys_loss_double(g, tm, H, 0.25, dt, 1.3, 0.7, m1p1))) / (2 * e)
        assert abs(fd - r["grad"][i]) <= 1e-6 * gmax, (i, fd, r["grad"][i])


@pytest.mark.parametrize("shape,H,per,m1p1,h,dt", CASES[:4] + [((20, 12, 9), 32, True, True, (1, 1, 1), 2e-3)])
def test_checker_fp32_forward_is_the_pinned_forward(port, shape, H, per, m1p1, h, dt):
    """Mode 0 differentiates the SAME numbers the pinned port produces: losses from identical float residuals."""
    g = OGrid(*shape, *h, dt, per)
    w = port.mlp_random_init(H, seed=777, scale=0.25)
    r0 = port.phys_loss_grad(g, w, 0.25, dt, 1.3, 0.7, m1p1, all_double=False)
    ref = port.fused_loss(g, w, 0.25, dt, 1.3, 0.7, m1p1)
    assert r0["loss_sigma"] == pytest.approx(float(np.float32(1.3)) * ref["acc_sigma"] / g.N, rel=1e-14)
    assert r0["loss_u"] == pytest.approx(float(np.float32(0.7)) * ref["acc_u"] / g.N, rel=1e-14)
    # and the fp32-faithful gradient is the all-double one up to the forward's fp32 noise (amplified by 1/(2 dt))
    r1 = port.phys_loss_grad(g, w, 0.25, dt, 1.3, 0.7, m1p1, all_double=True)
    assert np.abs(r0["grad"] - r1["grad"]).max() <= 2e-3 * np.abs(r1["grad"]).max()


# ---------------------------------------------------------------------------------------------------------------
GPU_CASES = [
    ((64, 64, 64), 64, True, True, (1, 1, 1), 2e-3),
    ((48, 48, 32), 64, False, True, (1, 1, 1), 2e-3),
    ((96, 64, 24), 32, False, True, (0.5, 0.25, 2.0), 1e-2),
    ((33, 18, 7), 64, True, False, (1, 1, 1), 2e-3),
    ((70, 37, 5), 128, False, True, (1, 1, 1), 2e-3),
    ((20, 9, 4), 48, True, True, (1, 1, 1), 2e-3),      # padded width
    ((128, 20, 9), 32, True, True, (1, 1, 1), 2e-3),    # wide rows, row-aligned batches
    ((256, 6, 5), 16, False, True, (0.5, 1, 2), 2e-3),  # wide rows, clamped faces, anisotropic spacing
    ((132, 7, 3), 16, False, False, (1, 1, 1), 2e-3),   # wide rows, nx % 32 != 0
    ((5, 3, 2), 16, True, True, (1, 1, 1), 2e-3),
    ((1, 1, 1), 16, True, True, (1, 1, 1), 2e-3),
    ((2, 1, 3), 16, False, True, (1, 1, 1), 2e-3),
]


def _g(og):
    from phys_autodiff_b200 import Grid
    return Grid(og.nx, og.ny, og.nz, og.hx, og.hy, og.hz, og.dt, og.periodic)


@pytest.mark.gpu
@pytest.mark.parametrize("shape,H,per,m1p1,h,dt", GPU_CASES)
def test_gradient_vs_checker(ctx, port, shape, H, per, m1p1, h, dt):
    from phys_autodiff_b200 import MLPConfig, PhysWeights
    og = OGrid(*shape, *h, dt, per)
    w = port.mlp_random_init(H, 777, 0.25)
    want = port.phys_loss_grad(og, w, 0.25, dt, 1.3, 0.7, m1p1, all_double=False)
    ls, lu, dW1, db1, dW2, db2 = ctx.fused_loss_grad_host(_g(og), MLPConfig(4, H, 4, m1p1), *w, PhysWeights(1.3, 0.7), 0.25, dt)
    got = np.concatenate([dW1, db1, dW2, db2]).astype(np.float64)
    assert_grad_close(got, want["grad"], H, 1, TOL_GRAD)
    assert abs(ls - want["loss_sigma"]) <= TOL_LOSS * abs(want["loss_sigma"]) + 1e-30
    assert abs(lu - want["loss_u"]) <= TOL_LOSS * abs(want["loss_u"]) + 1e-30
    # the losses are the fused forward kernel's
    f = ctx.fused_loss_host(_g(og), MLPConfig(4, H, 4, m1p1), *w, PhysWeights(1.3, 0.7), 0.25, dt)
    assert abs(f[0] - ls) <= 1e-6 * abs(ls) + 1e-30 and abs(f[1] - lu) <= 1e-6 * abs(lu) + 1e-30


@pytest.mark.gpu
@pytest.mark.parametrize("shape,H,per,grid_dt,dt", [((40, 24, 13), 64, True, 2e-3, 1e-3), ((33, 18, 7), 32, False, 5e-3, 2e-2)])
def test_gradient_with_slice_offset_different_from_grid_dt(ctx, port, shape, H, per, grid_dt, dt):
    """The reference API keeps the slice offset of mlp_generate_fields(t, dt) (src/mlp_grid.cpp:87-89) independent of
    GridSpec::dt, which alone forms the residual's time derivative (src/phys_cpu.cpp:38).  Loss AND gradient must use
    1/(2 grid.dt) -- a backward scaled with the call's dt would disagree with the loss it returns."""
    from phys_autodiff_b200 import MLPConfig, PhysWeights
    og = OGrid(*shape, 1, 1, 1, grid_dt, per)
    w = port.mlp_random_init(H, 777, 0.25)
    want = port.phys_loss_grad(og, w, 0.25, dt, 1.3, 0.7, True, all_double=False)
    ls, lu, dW1, db1, dW2, db2 = ctx.fused_loss_grad_host(_g(og), MLPConfig(4, H, 4, True), *w, PhysWeights(1.3, 0.7), 0.25, dt)
    got = np.concatenate([dW1, db1, dW2, db2]).astype(np.float64)
    assert_grad_close(got, want["grad"], H, 1, TOL_GRAD)
    assert abs(ls - want["loss_sigma"]) <= TOL_LOSS * abs(want["loss_sigma"])
    assert abs(lu - want["loss_u"]) <= TOL_LOSS * abs(want["loss_u"])
    # the slab form shares grad_args_common
    from phys_autodiff_b200.ops import slab_for_rank
    ctx.set_weights(MLPConfig(4, H, 4, True), *w)
    tot = np.zeros(9 * H + 6)
    for r in range(3):
        tot += ctx.fused_loss_grad_slab_acc(_g(og), PhysWeights(1.3, 0.7), 0.25, dt, slab_for_rank(og.nz, r, 3)).cpu().numpy()
    assert_grad_close(tot[2:], want["grad"], H, 1, TOL_GRAD)


@pytest.mark.gpu
def test_gradient_is_deterministic_and_device_form_agrees(ctx, port):
    from phys_autodiff_b200 import MLPConfig, PhysWeights
    og = OGrid(96, 80, 37, 1, 1, 1, 2e-3, True)
    w = port.mlp_random_init(64, 777, 0.25)
    ctx.set_weights(MLPConfig(4, 64, 4, True), *w)
    a = ctx.fused_loss_grad(_g(og), PhysWeights(1, 1), 0.25, 2e-3)
    for _ in range(5):
        b = ctx.fused_loss_grad(_g(og), PhysWeights(1, 1), 0.25, 2e-3)
        assert a[0] == b[0] and a[1] == b[1] and np.array_equal(a[2].view(np.uint64), b[2].view(np.uint64))
    h = ctx.fused_loss_grad_host(_g(og), MLPConfig(4, 64, 4, True), *w, PhysWeights(1, 1), 0.25, 2e-3)
    assert np.array_equal(np.concatenate(h[2:]), a[2].astype(np.float32))


@pytest.mark.gpu
@pytest.mark.parametrize("shape,per,H", [((40, 24, 13), True, 64), ((40, 24, 13), False, 64), ((33, 9, 3), True, 32),
                                          ((128, 8, 10), False, 128)])
def test_slab_gradients_sum_to_the_whole(ctx, port, shape, per, H):
    """Multi-GPU decomposition on one device: the slab sums (fields two planes around each slab recomputed
    locally, window wrapped or cut at the faces) add up to the whole-grid loss sums and gradient."""
    from phys_autodiff_b200 import MLPConfig, PhysWeights
    from phys_autodiff_b200.ops import slab_for_rank
    og = OGrid(*shape, 1, 1, 1, 2e-3, per)
    ctx.set_weights(MLPConfig(4, H, 4, True), *port.mlp_random_init(H, 777, 0.25))
    pw = PhysWeights(1.3, 0.7)
    acc, grad = ctx.fused_loss_grad_acc(_g(og), pw, 0.25, 2e-3)
    whole = np.concatenate([acc.cpu().numpy(), grad.cpu().numpy()])
    for world in (2, 3, 8):
        tot = np.zeros_like(whole)
        for r in range(world):
            tot += ctx.fused_loss_grad_slab_acc(_g(og), pw, 0.25, 2e-3, slab_for_rank(og.nz, r, world)).cpu().numpy()
        assert np.abs(tot[:2] - whole[:2]).max() <= 1e-12 * np.abs(whole[:2]).max()
        # the gradient's fp32 batch sums (32 points each) fall on different points when the slabs start elsewhere
        assert np.abs(tot[2:] - whole[2:]).max() <= 2e-6 * np.abs(whole[2:]).max(), world


@pytest.mark.gpu
def test_training_reduces_the_loss_by_90_percent(ctx, port):
    """Acceptance criterion of the reference's plan (REQUIREMENT.md:164-169): within K steps L falls >= 90 %."""
    from phys_autodiff_b200 import MLPConfig, PhysWeights
    og = OGrid(32, 32, 32, 1, 1, 1, 2e-3, True)
    H = 64
    cfg, pw = MLPConfig(4, H, 4, True), PhysWeights(1, 1)
    th = np.concatenate([np.asarray(a, np.float64) for a in port.mlp_random_init(H, 777, 0.25)])
    m, v = np.zeros_like(th), np.zeros_like(th)
    first = last = None
    for k in range(1, 121):   # Adam on the host: 580 parameters
        w = [th[:4 * H], th[4 * H:5 * H], th[5 * H:9 * H], th[9 * H:]]
        ls, lu, *d = ctx.fused_loss_grad_host(_g(og), cfg, *[x.astype(np.float32) for x in w], pw, 0.25, 2e-3)
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
    """Status codes, not crashes: no weights, unsupported shapes, bad slabs, null pointers; empty slab gives zeros."""
    import ctypes as C
    from phys_autodiff_b200 import Grid, MLPConfig, PhysadError, PhysWeights, capi, ops
    c2 = ops.Context()
    try:
        g, pw = Grid(8, 8, 8, 1, 1, 1, 1e-3, True), PhysWeights(1, 1)
        c2.cfg = MLPConfig(4, 16, 4, True)
        with pytest.raises(PhysadError, match="no weights"):
            c2.fused_loss_grad_acc(g, pw, 0.1, 1e-3)
        c2.set_weights(MLPConfig(4, 256, 4, True), *port.mlp_random_init(256, 1, 0.1))
        with pytest.raises(PhysadError, match="H > 128"):
            c2.fused_loss_grad_acc(g, pw, 0.1, 1e-3)
        c2.set_weights(MLPConfig(4, 16, 4, True), *port.mlp_random_init(16, 1, 0.1))
        with pytest.raises(PhysadError):
            c2.fused_loss_grad_acc(Grid(0, 8, 8), pw, 0.1, 1e-3)
        with pytest.raises(PhysadError, match="slab"):
            c2.fused_loss_grad_slab_acc(g, pw, 0.1, 1e-3, (4, 12))
        z = c2.fused_loss_grad_slab_acc(g, pw, 0.1, 1e-3, (3, 3)).cpu().numpy()
        assert z.shape == (9 * 16 + 6,) and not z.any()
        lib = capi.lib()
        assert lib.physad_fused_loss_grad_dev(c2._h, None, None, C.c_float(0), C.c_float(0), None, None, None) != 0
        assert lib.physad_fused_loss_grad_host(None, None, None, None, None, None, None, None, C.c_float(0), C.c_float(0),
                                               None, None, None, None, None, None) != 0
    finally:
        c2.close()
