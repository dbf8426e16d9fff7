"""Deeper networks at every supported depth: L = 1 .. 16 hidden layers at H = 32, 64 and 128, with weights that keep the
signal alive, and gradients checked tensor by tensor.

The usual test weights (Wh, bh ~ U(+-0.2), first and last layers at scale 0.25) make a deep network nearly constant:
every layer shrinks how much the activations vary from point to point, so at L = 16 an error in a hidden layer barely
reaches the output or the loss.  _depth_weights is a He-uniform draw that keeps the spread over points through all 16
layers; test_depth_init_keeps_the_spread_over_points pins that property.

CPU tier: the per-tensor gradient check (helpers.assert_grad_close) against one-tensor mutations, a dropped tile and fp32
rounding of checker outputs, and the initialisation.  GPU tier, for every (H, L): the strict forward (grid, fields,
points) bit for bit against the pinned port, the tensor-core mode against an fp64 forward, the four gradient kernels
(k_deep_grad, k_deep_tangent, k_colloc_tangent, k_deep_data_grad) against their kernel-faithful checkers, and exact zeros
for dead units."""
import os
import subprocess

import numpy as np
import pytest

from helpers import assert_grad_close, bits_equal, grad_segments
from oracle import Grid as OGrid
from test_deep_data import DataChecker
from test_deep_grad import DeepChecker, _deep_weights
from test_deep_tangent import TangentChecker
from test_deep_tangent_points import DCDX, TILE, PointsChecker, _points

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
WIDTHS = (32, 64, 128)
DEPTHS = tuple(range(1, 17))
ALL = [(H, L) for H in WIDTHS for L in DEPTHS]
FD_TILE = {32: 256, 64: 128, 128: 64}        # points per tile of k_deep_grad
DATA_TILE = {32: 768, 64: 384, 128: 192}     # points per tile of k_deep_data_grad (= k_mlp_deep's infer / points tile)
LAM = (0.7, 1.9, 0.0, 0.35)


def _plen(H, L):
    return 9 * H + 4 + (L - 1) * (H * H + H)


def _depth_weights(H, L, seed):
    """He-uniform: W1 ~ U(+-sqrt(6/4)), Wh and W2 ~ U(+-sqrt(6/H)), biases ~ U(+-0.1).  (Wh, bh) are None for L = 1."""
    rng = np.random.default_rng(seed)
    u = lambda n, a: rng.uniform(-a, a, n).astype(np.float32)
    W1, b1 = u(4 * H, np.sqrt(6 / 4)), u(H, 0.1)
    Wh, bh = (u((L - 1) * H * H, np.sqrt(6 / H)), u((L - 1) * H, 0.1)) if L > 1 else (None, None)
    return W1, b1, Wh, bh, u(4 * H, np.sqrt(6 / H)), u(4, 0.1)


def _theta(w):
    return np.concatenate([np.asarray(a, np.float64).ravel() for a in w if a is not None])


def _net64(x, w, H, L):
    """fp64 forward of the network at x [B, 4] -> (every hidden layer's activations, y [B, 4])."""
    W1, b1, Wh, bh, W2, b2 = (None if a is None else np.asarray(a, np.float64) for a in w)
    a = np.maximum(np.asarray(x, np.float64) @ W1.reshape(H, 4).T + b1, 0.0)
    acts = [a]
    for l in range(L - 1):
        a = np.maximum(a @ Wh[l * H * H:(l + 1) * H * H].reshape(H, H).T + bh[l * H:(l + 1) * H], 0.0)
        acts.append(a)
    return acts, a @ W2.reshape(4, H).T + b2


def _build(tmp_path_factory, name):
    out = str(tmp_path_factory.mktemp(name) / f"lib{name}.so")
    subprocess.run([os.environ.get("CC", "gcc"), "-std=c11", "-O3", "-ffp-contract=off", "-fPIC", "-shared", "-o", out,
                    os.path.join(ROOT, "tests", name + ".c"), "-lm"], check=True, capture_output=True)
    return out


@pytest.fixture(scope="module")
def fd_chk(tmp_path_factory):
    return DeepChecker(_build(tmp_path_factory, "deep_grad_checker"))


@pytest.fixture(scope="module")
def tan_chk(tmp_path_factory):
    return TangentChecker(_build(tmp_path_factory, "deep_tangent_checker"))


@pytest.fixture(scope="module")
def pts_chk(tmp_path_factory):
    return PointsChecker(_build(tmp_path_factory, "deep_tangent_points_checker"))


@pytest.fixture(scope="module")
def data_chk(tmp_path_factory):
    return DataChecker(_build(tmp_path_factory, "deep_data_checker"))


# ---------------------------------------------------------------------------------------------------------------------
# CPU tier
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("H,L", [(4, 1), (32, 1), (6, 2), (64, 5), (128, 16)])
def test_grad_segments_tile_the_layout(H, L):
    segs = grad_segments(H, L)
    assert [n for n, _ in segs] == ["dW1", "db1"] + [f"dWh{l}" for l in range(1, L)] + [f"dbh{l}" for l in range(1, L)] + \
        ["dW2", "db2"]
    assert segs[0][1].start == 0 and segs[-1][1].stop == _plen(H, L)
    assert all(a.stop == b.start for (_, a), (_, b) in zip(segs[:-1], segs[1:]))


def _points_case(pts_chk):
    """The points case (H = 32, L = 6, B = 129) of test_deep_tangent_points' checker comparison, with its weights."""
    H, L, B = 32, 6, 129
    th = _theta(_deep_weights(H, L, 777, 0.25))
    x = _points(B, H + 10 * L + B)
    return H, L, th, x, pts_chk.points(H, L, th, x, DCDX.astype(np.float64), 1.3, 0.7)["grad"]


def _grid_case(fd_chk):
    """The finite-difference grid case ((64, 16, 6), H = 64, L = 5) of test_deep_grad's checker comparison."""
    H, L = 64, 5
    og = OGrid(64, 16, 6, 1, 1, 1, 2e-3, True)
    return H, L, fd_chk.phys_loss_grad_deep(og, H, L, _deep_weights(H, L, 777, 0.25), 0.25, 2e-3, 1.3, 0.7, False)["grad"]


def _old_criterion(got, want):
    return np.abs(got - want).max() <= 1e-4 * np.abs(want).max()


@pytest.mark.parametrize("case", ["points", "grid"])
def test_per_tensor_check_rejects_one_tensor_off_by_one_percent(pts_chk, fd_chk, case):
    """want_s x 1.01 in any single tensor s is rejected.  The whole-vector criterion max|d| <= 1e-4 max|want| accepted some
    of these: db1 and dbh1 in the points case, db2 in the grid case."""
    if case == "points":
        H, L, _, _, want = _points_case(pts_chk)
        old_blind = {"db1", "dbh1"}
    else:
        H, L, want = _grid_case(fd_chk)
        old_blind = {"db2"}
    for name, s in grad_segments(H, L):
        got = want.copy()
        got[s] *= 1.01
        with pytest.raises(AssertionError, match=name):
            assert_grad_close(got, want, H, L)
        if name in old_blind:
            assert _old_criterion(got, want), name


def test_per_tensor_check_rejects_a_dropped_tile(pts_chk):
    """The points checker on x[TILE:] with the same n_norm: one tile of points left out."""
    H, L, th, x, want = _points_case(pts_chk)
    got = pts_chk.points(H, L, th, x[TILE[H]:], DCDX.astype(np.float64), 1.3, 0.7, n_norm=x.shape[0])["grad"]
    with pytest.raises(AssertionError):
        assert_grad_close(got, want, H, L)


def test_per_tensor_check_accepts_fp32_rounding(pts_chk, fd_chk):
    H, L, _, _, want = _points_case(pts_chk)
    assert_grad_close(want.astype(np.float32), want, H, L)
    H, L, want = _grid_case(fd_chk)
    assert_grad_close(want.astype(np.float32), want, H, L)


def _spread(a):
    """Each unit's standard deviation over the points, averaged over the units."""
    return float(a.std(axis=0).mean())


@pytest.mark.parametrize("H", WIDTHS)
def test_depth_init_keeps_the_spread_over_points(port, H):
    """At L = 16 the last hidden layer's spread over 4096 points in [-1, 1]^4, relative to the first layer's, is >= 0.1 in
    the median over 8 draws of _depth_weights and >= 0.05 in each (over 20 draws: 0.09 - 0.51 at H = 32, 0.12 - 0.63 at
    H = 64, 0.17 - 0.45 at H = 128).  The usual test weights lose it: at H = 32 the ratio is below 1e-3 (their biases hold
    every unit near a constant, so the RMS alone would not show it)."""
    L = 16
    x = np.random.default_rng(H).uniform(-1, 1, (4096, 4))
    r_new = []
    for seed in range(8):
        acts, _ = _net64(x, _depth_weights(H, L, seed), H, L)
        r_new.append(_spread(acts[-1]) / _spread(acts[0]))
    old, _ = _net64(x, _deep_weights(H, L, 777, 0.25, port), H, L)
    r_old = _spread(old[-1]) / _spread(old[0])
    print(f"spread ratio H={H} L={L}: depth init {np.round(r_new, 3)}, usual test weights {r_old:.3g}")
    assert np.median(r_new) >= 0.1 and min(r_new) >= 0.05, r_new
    if H == 32:
        assert r_old < 1e-3, r_old


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


def _report(kernel, H, L, ratio):
    print(f"grad ratio {kernel} H={H} L={L}: {ratio:.3g}")


SLICES = (np.float32(0.25) - np.float32(2e-3), np.float32(0.25), np.float32(0.25) + np.float32(2e-3))


@pytest.mark.gpu
@pytest.mark.parametrize("H,L", ALL)
def test_strict_forward_is_the_port_bit_for_bit(ctx, port, H, L):
    """Grid inference, fields and points.  37 x 11 x 5 = 2035 points: a ragged last tile in the infer / points tiling
    (768, 384, 192 points) and in the fields tiling (256, 128, 64)."""
    og = OGrid(37, 11, 5, 1, 1, 1, 2e-3, True)
    w = _depth_weights(H, L, 1000 * H + L)
    _set(ctx, H, L, w)
    got = ctx.mlp_grid_infer_deep(_g(og), 0.3).cpu().numpy().reshape(-1)
    assert bits_equal(got, port.mlp_grid_infer_deep(og, H, L, *w, 0.3))
    f = ctx.mlp_generate_fields_deep(_g(og), 0.25, 2e-3)
    for k, tt in enumerate(SLICES):
        y = port.mlp_grid_infer_deep(og, H, L, *w, float(tt)).reshape(-1, 4)
        assert bits_equal(f[k].cpu().numpy(), y[:, 0]), k
        assert bits_equal(f[3 + k].cpu().numpy(), np.concatenate([y[:, 1], y[:, 2], y[:, 3]])), k
    B = 1000
    x = np.random.default_rng(H + L).uniform(-3, 3, (B, 4)).astype(np.float32)
    got = ctx.mlp_forward_deep(_dev(x)).cpu().numpy().reshape(-1)
    assert bits_equal(got, port.mlp_forward_deep(x, L, *w, B, 4, H, 4))


@pytest.mark.gpu
@pytest.mark.parametrize("L", [15, 16])
@pytest.mark.parametrize("H", WIDTHS)
def test_strict_forward_with_more_tiles_than_blocks(ctx, port, H, L):
    """About 1.5 row tiles per block: blocks that run two tiles carry the two-buffer weight streaming from one tile into the
    next, with an even (L = 15) and an odd (L = 16) number of hidden -> hidden layers.  The fields call's t slice and the
    points call at the grid's coordinates must equal the inference output, bit for bit."""
    nx, ny = 67, 37
    nz = -(-int(1.5 * ctx.sm_count * DATA_TILE[H]) // (nx * ny))
    og = OGrid(nx, ny, nz, 1, 1, 1, 2e-3, False)
    assert og.N > ctx.sm_count * DATA_TILE[H]
    w = _depth_weights(H, L, 7 * H + L)
    _set(ctx, H, L, w)
    got = ctx.mlp_grid_infer_deep(_g(og), 0.25).cpu().numpy().reshape(-1, 4)
    assert bits_equal(got.reshape(-1), port.mlp_grid_infer_deep(og, H, L, *w, 0.25))
    f = ctx.mlp_generate_fields_deep(_g(og), 0.25, 2e-3)
    assert bits_equal(f[1].cpu().numpy(), got[:, 0])
    assert bits_equal(f[4].cpu().numpy(), np.concatenate([got[:, 1], got[:, 2], got[:, 3]]))
    x = port.make_grid_coords(og, 0.25, True).reshape(-1, 4)
    assert bits_equal(ctx.mlp_forward_deep(_dev(x)).cpu().numpy(), got)


# max|fast - fp64| / max|strict - fp64| measured on a B200 (1000 W) for these weights and this grid:
#   k_mlp_deep_tc2, H = 32, L = 2 .. 16:   0.45 - 1.55
#   k_mlp_deep_tc2, H = 64, L = 2 .. 9:    0.59 - 0.87
#   k_mlp_deep_tc,  H = 64, L = 10 .. 16:  2.1 - 4.9
#   k_mlp_deep_tc,  H = 128, L = 2 .. 16:  1.4 - 6.9 (6.65 at L = 9, 6.88 at L = 16)
# The strict kernel's own error is 2e-7 - 2.4e-6 of the largest output, the fast mode's 2e-7 - 7e-6.  k_mlp_deep_tc issues
# each layer in two K halves and adds the second half's small bf16 term products onto the first half's complete sum, where
# k_mlp_deep_tc2 adds every small term product over the whole K before the large one; that is where its larger error
# comes from.
FAST_RATIO = 10.0
TC_CASES = [(H, L) for H in WIDTHS for L in DEPTHS if L >= 2]


@pytest.mark.gpu
@pytest.mark.parametrize("H,L", TC_CASES)
def test_fast_mode_error_against_fp64_is_near_the_strict_kernels(ctx, port, H, L):
    """Tensor-core mode (three-term bf16 operands, fp32 accumulation) at every supported depth: k_mlp_deep_tc2 at H = 32
    and at H = 64 up to L = 9, the streamed k_mlp_deep_tc at H = 64 from L = 10 and at H = 128 from L = 4.  Both modes are
    compared with the fp64 network at the kernels' fp32 coordinates: the fast mode's largest error must be within
    FAST_RATIO times the strict mode's, plus 1e-6 of the largest output.  67 x 37 x 9 points = 174.3 MMA tiles of 128 rows:
    more tiles than blocks and a ragged last tile.  Deterministic, and z-slabs are the whole grid's rows."""
    og = OGrid(67, 37, 9, 1, 1, 1, 2e-3, True)
    g = _g(og)
    w = _depth_weights(H, L, 11 * H + L)
    _set(ctx, H, L, w)
    _, y64 = _net64(port.make_grid_coords(og, 0.3, True).reshape(-1, 4), w, H, L)
    strict = ctx.mlp_grid_infer_deep(g, 0.3).cpu().numpy()
    fs = ctx.mlp_generate_fields_deep(g, 0.25, 2e-3)
    ctx.set_deep_mode(1)
    try:
        fast = ctx.mlp_grid_infer_deep(g, 0.3).cpu().numpy()
        scale = np.abs(y64).max()
        e_s, e_f = np.abs(strict - y64).max(), np.abs(fast - y64).max()
        print(f"fast/strict H={H} L={L}: strict {e_s / scale:.3g}, fast {e_f / scale:.3g}, ratio {e_f / e_s:.3g}")
        assert e_f <= FAST_RATIO * e_s + 1e-6 * scale, (e_s, e_f, scale)
        assert not np.array_equal(fast, strict)                # it really is the other arithmetic
        assert np.array_equal(ctx.mlp_grid_infer_deep(g, 0.3).cpu().numpy(), fast)    # deterministic
        plane = og.nx * og.ny
        for z0, z1 in [(0, 4), (4, og.nz)]:
            part = ctx.mlp_grid_infer_deep(g, 0.3, slab=(z0, z1)).cpu().numpy()
            assert np.array_equal(part, fast[z0 * plane: z1 * plane])
        ff = ctx.mlp_generate_fields_deep(g, 0.25, 2e-3)
        for x, y in zip(fs, ff):      # measured up to 7.8e-6 of the largest output
            assert float((x - y).abs().max()) <= 2e-5 * scale
        assert np.array_equal(ff[1].cpu().numpy(), ctx.mlp_grid_infer_deep(g, 0.25).cpu().numpy()[:, 0])
    finally:
        ctx.set_deep_mode(0)
    assert np.array_equal(ctx.mlp_grid_infer_deep(g, 0.3).cpu().numpy(), strict)


# ---- gradients --------------------------------------------------------------------------------------------------------
def _grid_opts(L):
    """Boundary, coordinate mapping and spacing vary with the depth."""
    return dict(per=L % 2 == 1, m1p1=L % 3 != 0, h=(1, 1, 1) if L % 4 else (0.7, 1.1, 0.9))


def _check_fd(ctx, fd_chk, og, H, L, w, m1p1):
    from phys_autodiff_b200 import PhysWeights
    pw = PhysWeights(1.3, 0.7)
    want = fd_chk.phys_loss_grad_deep(og, H, L, w, 0.25, 2e-3, 1.3, 0.7, m1p1, all_double=False)
    _set(ctx, H, L, w, m1p1)
    out = ctx.deep_loss_grad_acc(_g(og), pw, 0.25, 2e-3).cpu().numpy()
    assert out.shape == (_plen(H, L) + 2,)
    ratio = assert_grad_close(out[2:], want["grad"], H, L)
    assert ctx.finalize(out[:2], pw, og.N) == ctx.deep_loss(_g(og), pw, 0.25, 2e-3)
    return out[2:], want["grad"], ratio


def _check_tangent(ctx, tan_chk, og, H, L, w, m1p1):
    from phys_autodiff_b200 import PhysWeights
    want = tan_chk.loss_grad(og, H, L, _theta(w), 0.25, 1.3, 0.7, m1p1, all_double=False)
    _set(ctx, H, L, w, m1p1)
    acc = ctx.deep_tangent_loss_acc(_g(og), 0.25).cpu().numpy()
    for got, ref in zip(acc, (want["acc_sigma"], want["acc_u"])):
        assert abs(got - ref) <= 1e-6 * abs(ref), (got, ref)
    out = ctx.deep_tangent_loss_grad_acc(_g(og), PhysWeights(1.3, 0.7), 0.25).cpu().numpy()
    if L > 1:
        assert np.array_equal(out[:2].view(np.uint64), acc.view(np.uint64))
    else:   # the one-hidden-layer calls: same residuals, the double additions in another order (test_tangent_grad)
        assert np.abs(out[:2] - acc).max() <= 1e-12 * np.abs(acc).max() + 1e-300, (out[:2], acc)
    ratio = assert_grad_close(out[2:], want["grad"], H, L)
    return out[2:], want["grad"], ratio


def _check_points(ctx, pts_chk, H, L, w, x, copies=1):
    """The GPU runs `copies` copies of x with n_norm = copies * B; the checker runs one copy with n_norm = B: the same
    gradient, and sums `copies` times the checker's."""
    from phys_autodiff_b200 import PhysWeights
    B = x.shape[0]
    want = pts_chk.points(H, L, _theta(w), x, DCDX.astype(np.float64), 1.3, 0.7, n_norm=B)
    _set(ctx, H, L, w)
    xd = _dev(np.tile(x, (copies, 1)))
    acc = ctx.deep_tangent_points_loss_acc(xd, DCDX).cpu().numpy()
    for got, ref in zip(acc, (want["acc_sigma"], want["acc_u"])):
        assert abs(got - copies * ref) <= 1e-6 * abs(copies * ref), (got, ref, copies)
    out = ctx.deep_tangent_points_loss_grad_acc(xd, DCDX, PhysWeights(1.3, 0.7), n_norm=copies * B).cpu().numpy()
    assert np.array_equal(out[:2].view(np.uint64), acc.view(np.uint64))
    ratio = assert_grad_close(out[2:], want["grad"], H, L)
    return out[2:], want["grad"], ratio


def _check_data(ctx, data_chk, H, L, w, x, tgt, copies=1):
    B = x.shape[0]
    acc, want, _ = data_chk.run(H, L, _theta(w), x, tgt, LAM, B)
    _set(ctx, H, L, w)
    out = ctx.deep_data_loss_grad_acc(_dev(np.tile(x, (copies, 1))), _dev(np.tile(tgt, (copies, 1))), LAM,
                                      copies * B).cpu().numpy()
    assert out.shape == (_plen(H, L) + 1,)
    assert abs(out[0] - copies * acc) <= 1e-6 * abs(copies * acc), (out[0], acc, copies)
    ratio = assert_grad_close(out[1:], want, H, L)
    return out[1:], want, ratio


def _small_grid(L):
    """13 x 7 x 5 = 455 points: 1.8 / 3.6 / 7.1 tiles of k_deep_grad, 3.6 / 7.1 / 14.2 of k_deep_tangent (H = 32 / 64 /
    128), ragged at every width."""
    o = _grid_opts(L)
    return OGrid(13, 7, 5, *o["h"], 2e-3, o["per"]), o["m1p1"]


def _small_points(seed, tile):
    """2.5 tiles plus a ragged tail of 3 points."""
    B = 2 * tile + tile // 2 + 3
    return np.random.default_rng(seed).uniform(-1.2, 1.2, (B, 4)).astype(np.float32)


@pytest.mark.gpu
@pytest.mark.parametrize("H,L", ALL)
def test_fd_gradient_every_depth(ctx, fd_chk, H, L):
    og, m1p1 = _small_grid(L)
    _report("k_deep_grad", H, L, _check_fd(ctx, fd_chk, og, H, L, _depth_weights(H, L, 3 * H + L), m1p1)[2])


@pytest.mark.gpu
@pytest.mark.parametrize("H,L", ALL)
def test_tangent_gradient_every_depth(ctx, tan_chk, H, L):
    og, m1p1 = _small_grid(L)
    _report("k_deep_tangent", H, L, _check_tangent(ctx, tan_chk, og, H, L, _depth_weights(H, L, 5 * H + L), m1p1)[2])


@pytest.mark.gpu
@pytest.mark.parametrize("H,L", ALL)
def test_points_gradient_every_depth(ctx, pts_chk, H, L):
    x = _small_points(H + L, TILE[H])
    _report("k_colloc_tangent", H, L, _check_points(ctx, pts_chk, H, L, _depth_weights(H, L, 9 * H + L), x)[2])


@pytest.mark.gpu
@pytest.mark.parametrize("H,L", ALL)
def test_data_gradient_every_depth(ctx, data_chk, H, L):
    x = _small_points(H + L, DATA_TILE[H])
    tgt = np.random.default_rng(L).uniform(-1, 1, x.shape).astype(np.float32)
    _report("k_deep_data_grad", H, L, _check_data(ctx, data_chk, H, L, _depth_weights(H, L, 13 * H + L), x, tgt)[2])


# Grid kernels at L = 16 with more tiles than blocks: the CPU checker is the limit (at H = 128 about 2 ms per point for the
# finite-difference loss and 4 ms for the analytic one), so the grids are about as large as the checker runs in ~20 s,
# which is 2.5 tiles per block at H = 32, 2.3 at H = 64 and 1.1 at H = 128.
GRID_TILES_PER_BLOCK = {32: 2.5, 64: 2.3, 128: 1.1}


def _big_grid(ctx, tile, H):
    nx, ny = 45, 23
    nz = -(-int(GRID_TILES_PER_BLOCK[H] * ctx.sm_count * tile) // (nx * ny))
    og = OGrid(nx, ny, nz, 1, 1, 1, 2e-3, True)
    assert og.N > ctx.sm_count * tile
    return og


@pytest.mark.gpu
@pytest.mark.parametrize("H", WIDTHS)
def test_fd_gradient_sixteen_layers_more_tiles_than_blocks(ctx, fd_chk, H):
    L = 16
    _report("k_deep_grad(many tiles)", H, L,
            _check_fd(ctx, fd_chk, _big_grid(ctx, FD_TILE[H], H), H, L, _depth_weights(H, L, 17 * H), True)[2])


@pytest.mark.gpu
@pytest.mark.parametrize("H", WIDTHS)
def test_tangent_gradient_sixteen_layers_more_tiles_than_blocks(ctx, tan_chk, H):
    L = 16
    _report("k_deep_tangent(many tiles)", H, L,
            _check_tangent(ctx, tan_chk, _big_grid(ctx, TILE[H], H), H, L, _depth_weights(H, L, 19 * H), True)[2])


@pytest.mark.gpu
@pytest.mark.parametrize("H", WIDTHS)
def test_points_gradient_sixteen_layers_several_tiles_per_block(ctx, pts_chk, H):
    L = 16
    x = _small_points(23 * H, TILE[H])
    copies = -(-3 * ctx.sm_count * TILE[H] // x.shape[0])    # about 3 tiles per block
    _report("k_colloc_tangent(many tiles)", H, L,
            _check_points(ctx, pts_chk, H, L, _depth_weights(H, L, 29 * H), x, copies)[2])


@pytest.mark.gpu
@pytest.mark.parametrize("H", WIDTHS)
def test_data_gradient_sixteen_layers_several_tiles_per_block(ctx, data_chk, H):
    L = 16
    x = _small_points(31 * H, DATA_TILE[H])
    tgt = np.random.default_rng(H).uniform(-1, 1, x.shape).astype(np.float32)
    copies = -(-3 * ctx.sm_count * DATA_TILE[H] // x.shape[0])
    _report("k_deep_data_grad(many tiles)", H, L,
            _check_data(ctx, data_chk, H, L, _depth_weights(H, L, 37 * H), x, tgt, copies)[2])


# ---- exact zeros ------------------------------------------------------------------------------------------------------
def _dead(H, L, whole_layer):
    """L = 4 with dead units in hidden layers 1 and 3 (whole_layer: every unit of layer 3): their incoming weights and bias
    are zero, so their pre-activation is +0 at every point.  -> (weights, {tensor: flat indices that must be zero})."""
    assert L == 4
    W1, b1, Wh, bh, W2, b2 = (a.copy() for a in _depth_weights(H, L, 41 * H + int(whole_layer)))
    d1 = [0, 5, H - 1]
    d3 = list(range(H)) if whole_layer else [1, 2, H // 2]
    W1.reshape(H, 4)[d1] = 0
    b1[d1] = 0
    Wh.reshape(L - 1, H, H)[1, d3] = 0      # Wh2: layer 2 -> layer 3, [out, in]
    bh.reshape(L - 1, H)[1, d3] = 0
    z = {"dW1": (np.arange(4 * H).reshape(H, 4)[d1]).ravel(), "db1": np.array(d1),
         "dWh1": np.arange(H * H).reshape(H, H)[:, d1].ravel(),
         "dWh2": np.arange(H * H).reshape(H, H)[d3].ravel(), "dbh2": np.array(d3),
         "dWh3": np.arange(H * H).reshape(H, H)[:, d3].ravel()}
    if whole_layer:   # nothing reaches the output through layer 3: every earlier layer's gradient is zero
        z.update({n: np.arange(s.stop - s.start) for n, s in grad_segments(H, L) if n in ("dW1", "db1", "dWh1", "dbh1")})
    return (W1, b1, Wh, bh, W2, b2), z


def _assert_zeros(g, H, L, z, who):
    segs = dict(grad_segments(H, L))
    for name, idx in z.items():
        v = np.asarray(g)[segs[name]][idx]
        assert (v == 0).all(), (who, name, np.abs(v).max(), int((v != 0).sum()))


@pytest.mark.gpu
@pytest.mark.parametrize("whole_layer", [False, True])
@pytest.mark.parametrize("H", WIDTHS)
def test_dead_units_get_exactly_zero_gradients(ctx, fd_chk, tan_chk, pts_chk, data_chk, H, whole_layer):
    """A unit whose pre-activation is +0 everywhere is off (the a > 0 mask): every kernel and every checker returns exactly
    zero for its incoming weights, its bias and its outgoing weights."""
    L = 4
    w, z = _dead(H, L, whole_layer)
    og, m1p1 = _small_grid(L)
    x = _small_points(43 * H, TILE[H])
    xd = _small_points(47 * H, DATA_TILE[H])
    tgt = np.random.default_rng(H).uniform(-1, 1, xd.shape).astype(np.float32)
    for who, (got, want, _) in (("k_deep_grad", _check_fd(ctx, fd_chk, og, H, L, w, m1p1)),
                                ("k_deep_tangent", _check_tangent(ctx, tan_chk, og, H, L, w, m1p1)),
                                ("k_colloc_tangent", _check_points(ctx, pts_chk, H, L, w, x)),
                                ("k_deep_data_grad", _check_data(ctx, data_chk, H, L, w, xd, tgt))):
        _assert_zeros(got, H, L, z, who)
        _assert_zeros(want, H, L, z, who + " checker")
