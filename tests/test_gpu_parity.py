"""GPU tier: parity of the CUDA path (through the C-ABI) against the CPU checker -- the unmodified
reference library where it shipped, else the pinned C port -- and against the golden vectors.

Tolerances (BASELINE.json north_star): MLP outputs and residuals max|d|/max|ref| <= 1e-5, reduced
loss relative error <= 1e-4.  The strict MLP is expected (and asserted) to be bit-exact."""
import math

import numpy as np
import pytest

from helpers import bits_equal, manufactured_fields, max_rel_to_max, rel_l2
from oracle import Grid as OGrid

pytestmark = pytest.mark.gpu

TOL_FIELD = 1e-5
TOL_LOSS = 1e-4


def _ops():
    from phys_autodiff_b200 import ops
    return ops


def _g(og):
    from phys_autodiff_b200 import Grid
    return Grid(og.nx, og.ny, og.nz, og.hx, og.hy, og.hz, og.dt, og.periodic)


def _cfg(H, m1p1=True, In=4, Out=4):
    from phys_autodiff_b200 import MLPConfig
    return MLPConfig(In, H, Out, m1p1)


def _pw(a=1.0, b=1.0):
    from phys_autodiff_b200 import PhysWeights
    return PhysWeights(a, b)


def _t(a):
    import torch
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


# ------------------------------------------------------------------------------------------------
# MLP: bit-exact
# ------------------------------------------------------------------------------------------------
def test_library_is_loaded_and_is_cuda(ctx):
    assert ctx.sm_count >= 100  # a B200 has 148 SMs; this is not a CPU fallback
    import ctypes
    from phys_autodiff_b200 import capi
    assert isinstance(capi.lib(), ctypes.CDLL)


@pytest.mark.parametrize("shape,H,seed,t,per,m1p1", [
    ((32, 32, 24), 64, 123, 0.3, False, True),     # test/test_mlp_grid_infer.cpp:15-20
    ((64, 64, 64), 64, 123, 0.3, False, True),     # BASELINE config 2
    ((48, 48, 32), 64, 321, 0.25, True, True),     # test_mlp_phys_integration_inputs.cpp
    ((17, 9, 5), 32, 777, -0.4, True, False),      # ZeroToOne, ragged
    ((20, 20, 10), 128, 777, 0.25, True, True),
    ((13, 7, 3), 16, 42, 0.25, True, True),        # H below the smallest template (zero-padded)
    ((11, 5, 2), 100, 9, 0.1, True, True),         # H between templates
])
def test_mlp_grid_infer_bit_exact(ctx, checker, shape, H, seed, t, per, m1p1):
    og = OGrid(*shape, 1, 1, 1, 1.0, per)
    w = checker.mlp_random_init(H, seed, 0.25)
    want = checker.mlp_grid_infer(og, w, t, m1p1)
    ctx.set_weights(_cfg(H, m1p1), *w)
    got = ctx.mlp_grid_infer(_g(og), t).cpu().numpy().reshape(-1)
    assert bits_equal(got, want)
    assert rel_l2(got, want) <= 1e-6  # the reference's own criterion (test_mlp_grid_infer.cpp:24)
    # host-pointer form (what mlp_grid_infer_cuda of the reference API does)
    assert bits_equal(ctx.mlp_grid_infer_host(_g(og), t), want)


def test_mlp_grid_infer_golden_anchor(ctx, golden, checker):
    _, meta = golden
    a = meta["anchors"]["grid_infer_32x32x24"]
    w = checker.mlp_random_init(64, 123, 0.25)
    ctx.set_weights(_cfg(64), *w)
    from phys_autodiff_b200 import Grid
    y = ctx.mlp_grid_infer(Grid(32, 32, 24, 1, 1, 1, 1.0, False), 0.3).cpu().numpy().reshape(-1)
    assert [float(v) for v in y[:4]] == [float(v) for v in a["y0"]]
    assert int(np.bitwise_xor.reduce(y.view(np.uint32))) == a["crc"]


def test_mlp_forward_generic_dims_bit_exact(ctx, checker):
    rng = np.random.default_rng(1)
    for (B, In, H, Out) in [(1000, 4, 64, 4), (37, 5, 19, 3), (513, 4, 300, 4), (64, 16, 32, 8), (1, 4, 1, 4)]:
        x = rng.uniform(-1, 1, B * In).astype(np.float32)
        W1 = rng.uniform(-.5, .5, H * In).astype(np.float32); b1 = rng.uniform(-.5, .5, H).astype(np.float32)
        W2 = rng.uniform(-.5, .5, Out * H).astype(np.float32); b2 = rng.uniform(-.5, .5, Out).astype(np.float32)
        want = checker.mlp_forward(x, W1, b1, W2, b2, B, In, H, Out)
        ctx.set_weights(_cfg(H, True, In, Out), W1, b1, W2, b2)
        assert bits_equal(ctx.mlp_forward_host(x), want), (B, In, H, Out)
        got = ctx.mlp_forward(_t(x).view(B, In)).cpu().numpy().reshape(-1)
        assert bits_equal(got, want), (B, In, H, Out)


def test_mlp_backward_bit_exact(ctx, checker, golden):
    """mlp_backward<ExecCuda> (SURVEY 8f rank 1): every gradient entry equals the CPU reference bitwise,
    incl. the reference's own benchmark shape (test/test_mlp_compare.cpp:17)."""
    rng = np.random.default_rng(2)
    for (B, In, H, Out) in [(23, 5, 12, 3), (64, 4, 64, 4), (512, 256, 512, 256), (1, 4, 8, 4)]:
        x = rng.uniform(-1, 1, B * In).astype(np.float32); t = rng.uniform(-1, 1, B * Out).astype(np.float32)
        W1 = rng.uniform(-.3, .3, H * In).astype(np.float32); b1 = rng.uniform(-.3, .3, H).astype(np.float32)
        W2 = rng.uniform(-.3, .3, Out * H).astype(np.float32); b2 = rng.uniform(-.3, .3, Out).astype(np.float32)
        want = checker.mlp_backward(x, t, W1, b1, W2, b2, B, In, H, Out)
        ctx.set_weights(_cfg(H, True, In, Out), W1, b1, W2, b2)
        got = ctx.mlp_backward_host(x, t)
        for k, a, b in zip(["dW1", "db1", "dW2", "db2"], got, want):
            assert bits_equal(a, b), (B, In, H, Out, k)
    arr, meta = golden
    c = [c for c in meta["cases"] if c["kind"] == "backward"][0]
    ctx.set_weights(_cfg(c["H"], True, c["In"], c["Out"]), arr["bwd_W1"], arr["bwd_b1"], arr["bwd_W2"], arr["bwd_b2"])
    for k, a in zip(["dW1", "db1", "dW2", "db2"], ctx.mlp_backward_host(arr["bwd_x"], arr["bwd_t"])):
        assert bits_equal(a, arr["bwd_" + k]), k


@pytest.mark.parametrize("shape,H,per,m1p1", [((48, 48, 32), 64, True, True), ((19, 11, 6), 32, False, False)])
def test_generate_fields_bit_exact(ctx, checker, shape, H, per, m1p1):
    og = OGrid(*shape, 1, 1, 1, 2e-3, per)
    w = checker.mlp_random_init(H, 321, 0.25)
    want = checker.generate_fields(og, w, 0.25, 2e-3, m1p1)
    ctx.set_weights(_cfg(H, m1p1), *w)
    got = ctx.mlp_generate_fields(_g(og), 0.25, 2e-3)
    for a, b in zip(got, want):
        assert bits_equal(a.cpu().numpy(), b)
    got_h = ctx.mlp_generate_fields_host(_g(og), 0.25, 2e-3)
    for a, b in zip(got_h, want):
        assert bits_equal(a, b) and np.all(np.isfinite(a))


@pytest.mark.parametrize("H,L", [(64, 1), (64, 2), (64, 4), (32, 1), (32, 3), (32, 6), (128, 1), (128, 2), (128, 4), (64, 3)])
def test_deep_mlp_bit_exact(ctx, port, checker, H, L):
    """Deeper MLPs (additive API, BASELINE config 5): GPU == CPU restatement bitwise for every depth; with one
    hidden layer the deep entry points equal the reference-pinned one-layer path."""
    rng = np.random.default_rng(100 * H + L)
    og = OGrid(70, 9, 5, 1, 1, 1, 2e-3, True)
    g = _g(og)
    W1, b1, W2, b2 = checker.mlp_random_init(H, 777, 0.25)
    Wh = rng.uniform(-0.2, 0.2, (L - 1) * H * H).astype(np.float32)
    bh = rng.uniform(-0.2, 0.2, (L - 1) * H).astype(np.float32)
    ctx.set_weights_deep(_cfg(H), L, W1, b1, Wh, bh, W2, b2)
    got = ctx.mlp_grid_infer_deep(g, 0.3).cpu().numpy().reshape(-1)
    want = port.mlp_grid_infer_deep(og, H, L, W1, b1, Wh, bh, W2, b2, 0.3)
    assert bits_equal(got, want)
    f = ctx.mlp_generate_fields_deep(g, 0.25, 2e-3)
    for k, tt in enumerate((np.float32(0.25) - np.float32(2e-3), np.float32(0.25), np.float32(0.25) + np.float32(2e-3))):
        y = port.mlp_grid_infer_deep(og, H, L, W1, b1, Wh, bh, W2, b2, float(tt)).reshape(-1, 4)
        assert bits_equal(f[k].cpu().numpy(), y[:, 0])
        assert bits_equal(f[3 + k].cpu().numpy(), np.concatenate([y[:, 1], y[:, 2], y[:, 3]]))
    if L == 1:
        assert bits_equal(checker.mlp_grid_infer(og, (W1, b1, W2, b2), 0.3), got)   # pinned to the reference
        # L = 1 is served by the one-hidden-layer kernels; force the deep kernel once so that ITS layer-1 and output
        # phases are pinned to the reference too
        import os
        os.environ["PHYSAD_DEEP_FORCE"] = "1"
        try:
            assert bits_equal(ctx.mlp_grid_infer_deep(g, 0.3).cpu().numpy().reshape(-1), got)
            f2 = ctx.mlp_generate_fields_deep(g, 0.25, 2e-3)
            assert all(bits_equal(x.cpu().numpy(), y.cpu().numpy()) for x, y in zip(f, f2))
        finally:
            del os.environ["PHYSAD_DEEP_FORCE"]
        ctx.set_weights(_cfg(H), W1, b1, W2, b2)
        assert bits_equal(ctx.mlp_grid_infer(g, 0.3).cpu().numpy().reshape(-1), got)
    # the physics operators take the deep fields like any others
    ls, lu = ctx.phys_loss(g, _pw(), f)
    assert np.isfinite(ls) and np.isfinite(lu)


@pytest.mark.parametrize("H,L,shape", [(128, 3, (130, 37, 11)), (64, 5, (257, 19, 9)), (32, 2, (300, 41, 7))])
def test_deep_mlp_many_tiles_and_slabs(ctx, port, H, L, shape):
    """More tiles than blocks (several tiles per persistent block, streamed weight buffers for L - 1 >= 3), a ragged
    last tile, and z-slabs: slab outputs are the corresponding rows of the whole-grid outputs."""
    rng = np.random.default_rng(7 * H + L)
    og = OGrid(*shape, 1, 1, 1, 2e-3, False)
    g = _g(og)
    W1, b1, W2, b2 = port.mlp_random_init(H, 321, 0.25)
    Wh = rng.uniform(-0.2, 0.2, (L - 1) * H * H).astype(np.float32)
    bh = rng.uniform(-0.2, 0.2, (L - 1) * H).astype(np.float32)
    ctx.set_weights_deep(_cfg(H), L, W1, b1, Wh, bh, W2, b2)
    want = port.mlp_grid_infer_deep(og, H, L, W1, b1, Wh, bh, W2, b2, 0.3)
    got = ctx.mlp_grid_infer_deep(g, 0.3).cpu().numpy().reshape(-1)
    assert bits_equal(got, want)
    plane = og.nx * og.ny
    for z0, z1 in [(0, 3), (3, 4), (4, og.nz)]:
        part = ctx.mlp_grid_infer_deep(g, 0.3, slab=(z0, z1)).cpu().numpy().reshape(-1)
        assert bits_equal(part, want[z0 * plane * 4: z1 * plane * 4])
    f = ctx.mlp_generate_fields_deep(g, 0.25, 2e-3, slab=(2, 7))
    n = 5 * plane
    for k, tt in enumerate((np.float32(0.25) - np.float32(2e-3), np.float32(0.25), np.float32(0.25) + np.float32(2e-3))):
        y = port.mlp_grid_infer_deep(og, H, L, W1, b1, Wh, bh, W2, b2, float(tt)).reshape(-1, 4)[2 * plane: 7 * plane]
        assert bits_equal(f[k].cpu().numpy(), y[:, 0])
        assert bits_equal(f[3 + k].cpu().numpy(), np.concatenate([y[:, 1], y[:, 2], y[:, 3]]))
        assert f[3 + k].numel() == 3 * n


@pytest.mark.parametrize("H,L,shape", [(128, 3, (130, 37, 11)), (128, 2, (64, 64, 5)), (64, 5, (257, 19, 9)), (64, 2, (33, 7, 3)),
                                       (32, 3, (300, 41, 7)), (128, 5, (150, 33, 13)), (128, 4, (40, 9, 3)), (64, 12, (129, 65, 9))])
def test_deep_fast_mode_tracks_the_strict_kernel(ctx, port, H, L, shape):
    """Tensor-core fast mode (physad_set_deep_mode 1: three-term bf16 operands, fp32 accumulation; additive, explicitly
    NOT bit-exact): outputs within 1e-5 of the strict kernel's (measured ~1e-6, relative to the largest output), ragged
    last tile, several row tiles per block, z-slabs identical to the whole-grid rows, losses within 1e-4 relative.
    (128, 4), (128, 5) and (64, 12) do not fit in shared memory: their layer images are streamed through two buffers."""
    from phys_autodiff_b200 import PhysadError
    rng = np.random.default_rng(11 * H + L)
    og = OGrid(*shape, 1, 1, 1, 2e-3, True)
    g = _g(og)
    W1, b1, W2, b2 = port.mlp_random_init(H, 321, 0.25)
    Wh = rng.uniform(-0.2, 0.2, (L - 1) * H * H).astype(np.float32)
    bh = rng.uniform(-0.2, 0.2, (L - 1) * H).astype(np.float32)
    ctx.set_weights_deep(_cfg(H), L, W1, b1, Wh, bh, W2, b2)
    strict = ctx.mlp_grid_infer_deep(g, 0.3).cpu().numpy()
    fs = ctx.mlp_generate_fields_deep(g, 0.25, 2e-3)
    ls = ctx.phys_loss(g, _pw(), fs)
    ctx.set_deep_mode(1)
    try:
        fast = ctx.mlp_grid_infer_deep(g, 0.3).cpu().numpy()
        scale = np.abs(strict).max()
        assert np.abs(fast - strict).max() <= 1e-5 * scale
        assert not np.array_equal(fast, strict) or L == 1     # it really is the other arithmetic
        again = ctx.mlp_grid_infer_deep(g, 0.3).cpu().numpy()
        assert np.array_equal(again, fast)                     # deterministic
        plane = og.nx * og.ny
        z1 = max(1, og.nz // 2)
        for z0, z1 in [(0, z1), (z1, og.nz)]:
            part = ctx.mlp_grid_infer_deep(g, 0.3, slab=(z0, z1)).cpu().numpy()
            assert np.array_equal(part, fast[z0 * plane: z1 * plane])
        ff = ctx.mlp_generate_fields_deep(g, 0.25, 2e-3)
        for x, y in zip(fs, ff):
            assert float((x - y).abs().max()) <= 1e-5 * float(x.abs().max())
        at_t = ctx.mlp_grid_infer_deep(g, 0.25).cpu().numpy()
        assert np.array_equal(ff[1].cpu().numpy(), at_t[:, 0])                      # the t slice is the infer output
        lf = ctx.phys_loss(g, _pw(), ff)
        # (a 12-layer random network is nearly constant: losses ~1e-6, hence the absolute term)
        assert abs(lf[0] - ls[0]) <= 1e-4 * abs(ls[0]) + 1e-9 and abs(lf[1] - ls[1]) <= 1e-4 * abs(ls[1]) + 1e-9
    finally:
        ctx.set_deep_mode(0)
    assert np.array_equal(ctx.mlp_grid_infer_deep(g, 0.3).cpu().numpy(), strict)   # back to the parity mode


def test_tcgen05_layout_probe():
    """tools/tc_probe.cu: D = A B^T on exact small integers through the same descriptor / packing helpers the tensor-core
    kernels use (A in tensor memory or in shared memory, B in the K-major no-swizzle core-matrix layout).  The conventions the
    kernels rely on must give zero mismatches; the deliberately wrong variants (LBO/SBO exchanged, K pair order swapped) must not."""
    import os, re, subprocess
    exe = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tools", "_bin", "tc_probe")
    if not os.path.exists(exe):
        pytest.skip("tools/_bin/tc_probe not built (python __graft_entry__.py builds it)")
    r = subprocess.run([exe], capture_output=True, text=True, timeout=120)
    assert r.returncode == 0, r.stdout + r.stderr
    rows = re.findall(r"N=(\d+) K=(\d+) tmemA=(\d) swapLS=(\d) swapPack=(\d): (\d+) / (\d+) mismatches", r.stdout)
    assert len(rows) == 11, r.stdout
    for N, K, tm, sl, sp, bad, tot in rows:
        if sl == "0" and sp == "0":
            assert bad == "0", r.stdout
        else:
            assert int(bad) > int(tot) // 2, r.stdout


@pytest.mark.parametrize("H,L", [(128, 3), (128, 5), (64, 5), (32, 2)])
def test_deep_fast_mode_repeatability_stress(ctx, port, H, L):
    """The tensor-core kernel hands tensor-memory operands between an MMA warp and two epilogue groups through mbarriers
    (resident and streamed weights).  A missing ordering edge would show up as run-to-run differences: 25 launches over a
    grid with many row tiles per block must be bit-identical, fields and infer alike."""
    rng = np.random.default_rng(H + L)
    og = OGrid(256, 96, 12, 1, 1, 1, 2e-3, True)
    g = _g(og)
    W1, b1, W2, b2 = port.mlp_random_init(H, 11, 0.25)
    Wh = rng.uniform(-0.2, 0.2, (L - 1) * H * H).astype(np.float32)
    bh = rng.uniform(-0.2, 0.2, (L - 1) * H).astype(np.float32)
    ctx.set_weights_deep(_cfg(H), L, W1, b1, Wh, bh, W2, b2)
    ctx.set_deep_mode(1)
    try:
        import torch
        ref = [x.clone() for x in ctx.mlp_generate_fields_deep(g, 0.25, 2e-3)]
        ref_i = ctx.mlp_grid_infer_deep(g, 0.25).clone()
        for _ in range(25):
            f = ctx.mlp_generate_fields_deep(g, 0.25, 2e-3)
            assert all(torch.equal(x, y) for x, y in zip(ref, f))
            assert torch.equal(ctx.mlp_grid_infer_deep(g, 0.25), ref_i)
        assert torch.isfinite(ref_i).all()
    finally:
        ctx.set_deep_mode(0)


def test_deep_loss_one_call_equals_the_stagewise_calls(ctx, port):
    """physad_deep_loss_host = generate_fields_deep + phys_loss on context scratch: same losses as the two calls, in both
    arithmetic modes."""
    rng = np.random.default_rng(3)
    og = OGrid(48, 20, 7, 1, 1, 1, 2e-3, True)
    g = _g(og)
    H, L = 64, 3
    W1, b1, W2, b2 = port.mlp_random_init(H, 9, 0.25)
    Wh = rng.uniform(-0.2, 0.2, (L - 1) * H * H).astype(np.float32)
    bh = rng.uniform(-0.2, 0.2, (L - 1) * H).astype(np.float32)
    ctx.set_weights_deep(_cfg(H), L, W1, b1, Wh, bh, W2, b2)
    for mode in (0, 1):
        ctx.set_deep_mode(mode)
        try:
            want = ctx.phys_loss(g, _pw(1.3, 0.7), ctx.mlp_generate_fields_deep(g, 0.25, 2e-3))
            got = ctx.deep_loss(g, _pw(1.3, 0.7), 0.25, 2e-3)
            assert got[0] == want[0] and got[1] == want[1]
        finally:
            ctx.set_deep_mode(0)


def test_deep_fast_mode_one_hidden_layer_and_bad_mode(ctx, port):
    """With one hidden layer there is no hidden -> hidden contraction: the default route is the reference-pinned kernel in
    either mode (bit-identical), the forced deep kernel refuses mode 1 with PHYSAD_E_UNSUPPORTED -- never a silent switch
    of arithmetic.  Unknown modes are rejected."""
    import os
    from phys_autodiff_b200 import PhysadError
    og = OGrid(16, 8, 4, 1, 1, 1, 2e-3, True)
    g = _g(og)
    H = 64
    W1, b1, W2, b2 = port.mlp_random_init(H, 1, 0.25)
    ctx.set_weights_deep(_cfg(H), 1, W1, b1, None, None, W2, b2)
    strict = ctx.mlp_grid_infer_deep(g, 0.3).cpu().numpy()
    ctx.set_deep_mode(1)
    try:
        assert np.array_equal(ctx.mlp_grid_infer_deep(g, 0.3).cpu().numpy(), strict)
        os.environ["PHYSAD_DEEP_FORCE"] = "1"
        try:
            with pytest.raises(PhysadError, match="fast mode"):
                ctx.mlp_grid_infer_deep(g, 0.3)
            with pytest.raises(PhysadError, match="fast mode"):
                ctx.mlp_generate_fields_deep(g, 0.25, 2e-3)
        finally:
            del os.environ["PHYSAD_DEEP_FORCE"]
    finally:
        ctx.set_deep_mode(0)
    with pytest.raises(PhysadError):
        ctx.set_deep_mode(2)


def test_error_paths_and_empty_inputs(ctx, checker):
    """Status codes instead of crashes: bad arguments, unsupported shapes, missing weights, empty batches."""
    import ctypes as C
    import torch
    from phys_autodiff_b200 import Grid, PhysadError, capi, ops
    lib = capi.lib()
    c2 = ops.Context()
    try:
        g = Grid(8, 8, 8, 1, 1, 1, 1e-3, True)
        with pytest.raises(PhysadError, match="no weights"):
            c2.mlp_grid_infer(g, 0.1)                                   # PHYSAD_E_NOWEIGHTS
        w = checker.mlp_random_init(256, 1, 0.1)
        c2.set_weights(_cfg(256), *w)
        with pytest.raises(PhysadError, match="H > 128"):
            c2.fused_loss_acc(g, 0.1, 1e-3)                             # PHYSAD_E_UNSUPPORTED
        x = torch.zeros(0, 4, device="cuda")
        assert c2.mlp_forward(x).shape == (0, 4)                         # empty batch is a no-op
        w5 = [np.zeros(8 * 5, np.float32), np.zeros(8, np.float32), np.zeros(3 * 8, np.float32), np.zeros(3, np.float32)]
        c2.set_weights(_cfg(8, True, 5, 3), *w5)
        with pytest.raises(PhysadError, match="In = Out = 4"):
            c2.mlp_grid_infer(g, 0.1)
        c2.set_weights(_cfg(16), *checker.mlp_random_init(16, 1, 0.1))
        for bad in (Grid(0, 8, 8), Grid(8, -1, 8), Grid(2048, 1024, 1024)):   # empty / negative / N >= 2^31
            with pytest.raises(PhysadError):
                c2.fused_loss_acc(bad, 0.1, 1e-3)
        with pytest.raises(PhysadError, match="slab"):
            c2.fused_loss_acc(g, 0.1, 1e-3, slab=(4, 12))
        assert lib.physad_fused_loss_dev(c2._h, None, None, C.c_float(0), C.c_float(0), None, None, None, None, None, None) != 0
        assert len(lib.physad_last_error()) > 0
    finally:
        c2.close()


# ------------------------------------------------------------------------------------------------
# physics on supplied fields
# ------------------------------------------------------------------------------------------------
def test_residuals_manufactured_vs_cpu(ctx, checker):
    """test/test_phys_cuda_nonfused_vs_cpu.cpp: 64x64x32, sigma = sin(x+y+z-t), u = 1."""
    og = OGrid(64, 64, 32, 2 * math.pi / 64, 2 * math.pi / 64, 2 * math.pi / 32, 1e-3, True)
    f = manufactured_fields(og, 1.2345)
    want = checker.phys_residuals(og, f)
    got = ctx.phys_residuals_host(_g(og), f)
    assert rel_l2(got[0], want[0]) <= 3e-4 and np.max(np.abs(got[0] - want[0])) <= 1e-3     # :86-87
    for c in (1, 2, 3):
        assert np.max(np.abs(got[c] - want[c])) <= 1e-6                                      # :88-89
    # our bar is tighter than the reference's
    assert max_rel_to_max(got[0], want[0]) <= TOL_FIELD
    G = ctx.phys_backward_host(_g(og), _pw(1.7, 0.9), got)
    Gw = checker.phys_loss_backward(og, 1.7, 0.9, want)
    assert rel_l2(G[0], Gw[0]) <= 1e-7 + TOL_FIELD and np.max(np.abs(G[0] - Gw[0])) <= 1e-6  # :107


def test_fused_and_nonfused_names_agree(ctx):
    """test/test_phys_cuda_fused_vs_nonfused.cpp: 96x64x48, sigma = sin(2x+3y+4z-t), u = (sin z, cos x, sin y)."""
    ops = _ops()
    og = OGrid(96, 64, 48, 2 * math.pi / 96, 2 * math.pi / 64, 2 * math.pi / 48, 1e-3, True)
    f = manufactured_fields(og, 2.3456, 2, 3, 4, const_u=False)
    g = _g(og)
    a, b = ops.cuda_phys_residuals_fused(g, f), ops.cuda_phys_residuals_nonfused(g, f)
    for x, y in zip(a, b):
        assert rel_l2(x, y) <= 1e-7 and np.max(np.abs(x - y)) <= 1e-6                        # :74-77
    ga = ops.cuda_phys_loss_backward_fused(g, _pw(1.1, 0.8), f)
    gb = ops.cuda_phys_loss_backward_nonfused(g, _pw(1.1, 0.8), b)
    for x, y in zip(ga, gb):
        assert rel_l2(x, y) <= 1e-7 and np.max(np.abs(x - y)) <= 1e-6                        # :102-105
    (R, ms) = ops.cuda_phys_residuals_fused_timed(g, f)
    assert ms > 0 and all(bits_equal(x, y) for x, y in zip(R, a))


@pytest.mark.parametrize("shape,per", [((33, 18, 7), True), ((33, 18, 7), False), ((5, 1, 1), False), ((1, 1, 1), True),
                                       ((2, 2, 2), True), ((64, 64, 64), False),
                                       # more shapes with nx % 4 == 0 (vectorisable rows): ragged row tiles,
                                       # fewer rows than a tile, single planes, long rows,
                                       # and a mid-sized anisotropic grid
                                       ((36, 18, 7), True), ((36, 18, 7), False), ((8, 3, 5), True), ((8, 3, 1), False),
                                       ((4, 1, 2), True), ((352, 5, 3), True), ((520, 6, 2), False), ((600, 4, 2), True),
                                       ((128, 96, 40), True)])
def test_residuals_random_fields(ctx, checker, shape, per):
    """Random (non-smooth) fields, both boundary rules, degenerate extents."""
    rng = np.random.default_rng(3)
    og = OGrid(*shape, 0.7, 1.3, 0.9, 3e-3, per)
    f = [rng.standard_normal(og.N).astype(np.float32) for _ in range(3)] + \
        [rng.standard_normal(3 * og.N).astype(np.float32) for _ in range(3)]
    ls, lu, want = checker.phys_loss_forward(og, 1.1, 0.8, f, True)
    got_ls, got_lu, got = ctx.phys_loss_host(_g(og), _pw(1.1, 0.8), f, want_residuals=True)
    for a, b in zip(got, want):
        assert max_rel_to_max(a, b) <= TOL_FIELD
    assert abs(got_ls - ls) <= TOL_LOSS * abs(ls) and abs(got_lu - lu) <= TOL_LOSS * abs(lu)
    # loss-only form (no residual outputs) gives the same reduction
    l2 = ctx.phys_loss_host(_g(og), _pw(1.1, 0.8), f)
    assert l2[0] == got_ls and l2[1] == got_lu
    # device-resident form
    d = ctx.phys_loss(_g(og), _pw(1.1, 0.8), [_t(a) for a in f])
    assert d[0] == got_ls and d[1] == got_lu
    gw = checker.phys_loss_backward(og, 1.1, 0.8, want)
    gg = ctx.phys_backward_from_fields_host(_g(og), _pw(1.1, 0.8), f)
    for a, b in zip(gg, gw):
        assert max_rel_to_max(a, b) <= TOL_FIELD


@pytest.mark.parametrize("shape,per", [((128, 96, 40), True), ((128, 96, 40), False), ((33, 18, 7), True), ((36, 10, 3), False)])
def test_stagewise_slabs_with_halo_planes(ctx, shape, per):
    """Multi-GPU arithmetic of the stage-wise path on one GPU: the fields cut into 1/2/3/5 z-slabs, every slab given
    its two halo planes (wrap / clamp applied), reproduces the whole-grid residuals bitwise and the sums."""
    import torch
    from phys_autodiff_b200 import Grid
    from phys_autodiff_b200.ops import slab_for_rank
    rng = np.random.default_rng(11)
    g = Grid(*shape, 0.7, 1.3, 0.9, 3e-3, per)
    N, pln = g.N, g.nx * g.ny
    f = [_t(rng.standard_normal(N).astype(np.float32)) for _ in range(3)] + \
        [_t(rng.standard_normal(3 * N).astype(np.float32)) for _ in range(3)]
    acc_w, Rw = ctx.phys_loss_acc(g, f, want_residuals=True)
    acc_w = acc_w.cpu().numpy()

    def planes(a, z0, z1, vec):  # slab-local copy of a scalar / channel-major vector field
        if not vec:
            return a[z0 * pln:z1 * pln].contiguous()
        return torch.cat([a[c * N + z0 * pln: c * N + z1 * pln] for c in range(3)]).contiguous()

    def tplane(z):  # [4, pln] time-t plane z of the global fields
        return torch.stack([f[1][z * pln:(z + 1) * pln]] + [f[4][c * N + z * pln: c * N + (z + 1) * pln] for c in range(3)]).contiguous()
    for world in (1, 2, 3, 5):
        tot = np.zeros(2)
        for r in range(world):
            z0, z1 = slab_for_rank(g.nz, r, world)
            if z1 == z0:
                continue
            loc = [planes(f[k], z0, z1, k >= 3) for k in range(6)]
            lo_z, hi_z = ctx.halo_sources(g, (z0, z1))
            acc, R = ctx.phys_loss_slab_acc(g, (z0, z1), loc, tplane(lo_z), tplane(hi_z), want_residuals=True)
            tot += acc.cpu().numpy()
            for a, b in zip(R, Rw):
                assert torch.equal(a, b[z0 * pln:z1 * pln]), (world, r)
        assert np.allclose(tot, acc_w, rtol=1e-12)


def test_golden_path_cases(ctx, golden):
    """Committed golden vectors (generated from the reference) through every stage on the GPU."""
    from phys_autodiff_b200 import Grid
    arr, meta = golden
    for c in meta["cases"]:
        if c["kind"] != "path":
            continue
        n = c["name"]
        g = Grid(*c["g"], *c["h"], c["dt"], c["periodic"])
        key = f"w_s{c['seed']}_h{c['H']}"
        if key + "_W1" in arr:
            w = [arr[f"{key}_{k}"] for k in ("W1", "b1", "W2", "b2")]
        else:
            w = _ops().mlp_random_init(c["H"], c["seed"], c["scale"])
        ctx.set_weights(_cfg(c["H"], c["m1p1"]), *w)
        assert bits_equal(ctx.mlp_grid_infer_host(g, c["t"]), arr[n + "_y"]), n
        f = ctx.mlp_generate_fields_host(g, c["t"], c["dt"])
        for k, a in zip(["sm", "s0", "sp", "um", "u0", "up"], f):
            assert bits_equal(a, arr[f"{n}_{k}"]), (n, k)
        ls, lu, R = ctx.phys_loss_host(g, _pw(*c["w"]), f, want_residuals=True)
        fl = ctx.fused_loss_host(g, _cfg(c["H"], c["m1p1"]), *w, _pw(*c["w"]), c["t"], c["dt"], want_residuals=True)
        for k, a, b in zip(["Rs", "Rx", "Ry", "Rz"], R, fl[2]):
            assert max_rel_to_max(a, arr[f"{n}_{k}"]) <= TOL_FIELD, (n, k)
            assert max_rel_to_max(b, arr[f"{n}_{k}"]) <= TOL_FIELD, (n, k, "fused")
        for got in ((ls, lu), fl[:2]):
            assert abs(got[0] - float(c["loss_sigma"])) <= TOL_LOSS * abs(float(c["loss_sigma"])) + 1e-30, n
            assert abs(got[1] - float(c["loss_u"])) <= TOL_LOSS * abs(float(c["loss_u"])) + 1e-30, n


# ------------------------------------------------------------------------------------------------
# the metric path: fused MLP + physics loss
# ------------------------------------------------------------------------------------------------
FUSED_CASES = [
    # shape, H, periodic, m1p1, h, dt
    ((64, 64, 64), 64, True, True, (1, 1, 1), 2e-3),          # test_mlp_phys_perf shape, BASELINE anchors
    ((48, 48, 32), 64, True, True, (1, 1, 1), 2e-3),          # integration-inputs shape
    ((96, 64, 48), 32, False, True, (0.5, 0.25, 2.0), 1e-2),  # clamp, anisotropic spacing
    ((33, 18, 7), 64, True, False, (1, 1, 1), 2e-3),          # ragged tiles, ZeroToOne
    ((70, 37, 5), 128, False, True, (1, 1, 1), 2e-3),         # ragged, clamp, H=128
    ((5, 3, 2), 16, True, True, (1, 1, 1), 2e-3),             # smaller than one tile
    ((1, 1, 1), 16, True, True, (1, 1, 1), 2e-3),             # single point
    ((2, 1, 3), 16, False, True, (1, 1, 1), 2e-3),
]


@pytest.mark.parametrize("shape,H,per,m1p1,h,dt", FUSED_CASES)
def test_fused_loss_vs_cpu(ctx, checker, shape, H, per, m1p1, h, dt):
    og = OGrid(*shape, *h, dt, per)
    w = checker.mlp_random_init(H, 777, 0.25)
    f = checker.generate_fields(og, w, 0.25, dt, m1p1)
    ls, lu, R = checker.phys_loss_forward(og, 1.3, 0.7, f, True)
    got = ctx.fused_loss_host(_g(og), _cfg(H, m1p1), *w, _pw(1.3, 0.7), 0.25, dt, want_residuals=True)
    for a, b in zip(got[2], R):
        assert max_rel_to_max(a, b) <= TOL_FIELD
        assert rel_l2(a, b) <= TOL_FIELD
    assert abs(got[0] - ls) <= TOL_LOSS * abs(ls) + 1e-30 and abs(got[1] - lu) <= TOL_LOSS * abs(lu) + 1e-30
    # loss-only launch (no residual stores) reduces to the same numbers
    l2 = ctx.fused_loss_host(_g(og), _cfg(H, m1p1), *w, _pw(1.3, 0.7), 0.25, dt)
    assert l2[0] == got[0] and l2[1] == got[1]


@pytest.mark.parametrize("shape,H,per,m1p1,h,dt", FUSED_CASES[:6])
def test_exact_residual_mode_is_bit_identical_to_cpu(ctx, checker, shape, H, per, m1p1, h, dt):
    """physad_set_exact_residuals(1): stencil + residual sums in double exactly as src/phys_cpu.cpp:66-109, so
    the fused kernel's and the stage-wise kernel's residuals equal the CPU reference BITWISE."""
    og = OGrid(*shape, *h, dt, per)
    w = checker.mlp_random_init(H, 777, 0.25)
    f = checker.generate_fields(og, w, 0.25, dt, m1p1)
    ls, lu, R = checker.phys_loss_forward(og, 1.3, 0.7, f, True)
    ctx.set_exact_residuals(True)
    try:
        got = ctx.fused_loss_host(_g(og), _cfg(H, m1p1), *w, _pw(1.3, 0.7), 0.25, dt, want_residuals=True)
        staged = ctx.phys_loss_host(_g(og), _pw(1.3, 0.7), f, want_residuals=True)
    finally:
        ctx.set_exact_residuals(False)
    for a, b, c in zip(got[2], staged[2], R):
        assert bits_equal(a, c) and bits_equal(b, c)
    for out in (got, staged):  # identical residuals: only the order of the double additions differs
        assert abs(out[0] - ls) <= 1e-6 * abs(ls) + 1e-30 and abs(out[1] - lu) <= 1e-6 * abs(lu) + 1e-30


def test_fused_loss_anchors(ctx, golden, checker):
    _, meta = golden
    from phys_autodiff_b200 import Grid
    for H in (32, 64, 128):
        a = meta["anchors"][f"64c_h{H}"]
        w = checker.mlp_random_init(H, 777, 0.25)
        ls, lu = ctx.fused_loss_host(Grid(64, 64, 64, 1, 1, 1, 2e-3, True), _cfg(H), *w, _pw(), 0.25, 2e-3)
        assert abs(ls - float(a["loss_sigma"])) <= TOL_LOSS * float(a["loss_sigma"])
        assert abs(lu - float(a["loss_u"])) <= TOL_LOSS * float(a["loss_u"])


@pytest.mark.parametrize("variant", list(range(8)))
def test_fused_variants_agree(ctx, checker, variant):
    """Every launch geometry of the fused kernel gives the same residuals (bitwise) and loss."""
    og = OGrid(70, 37, 9, 1, 1, 1, 2e-3, True)
    w = checker.mlp_random_init(64, 777, 0.25)
    ctx.set_fused_variant(0)
    base = ctx.fused_loss_host(_g(og), _cfg(64), *w, _pw(), 0.25, 2e-3, want_residuals=True)
    ctx.set_fused_variant(variant)
    try:
        got = ctx.fused_loss_host(_g(og), _cfg(64), *w, _pw(), 0.25, 2e-3, want_residuals=True)
    finally:
        ctx.set_fused_variant(0)
    for a, b in zip(got[2], base[2]):
        assert bits_equal(a, b)
    assert abs(got[0] - base[0]) <= 1e-6 * abs(base[0]) and abs(got[1] - base[1]) <= 1e-6 * abs(base[1])


def test_fused_equals_staged_gpu_path(ctx, checker):
    """fused kernel == generate_fields -> phys_loss on the GPU (bitwise residuals: same fp32 stencil)."""
    og = OGrid(64, 40, 12, 1, 1, 1, 2e-3, False)
    w = checker.mlp_random_init(64, 5, 0.3)
    ctx.set_weights(_cfg(64), *w)
    f = ctx.mlp_generate_fields(_g(og), 0.25, 2e-3)
    ls, lu, R = ctx.phys_loss(_g(og), _pw(), f, want_residuals=True)
    got = ctx.fused_loss(_g(og), _pw(), 0.25, 2e-3, want_residuals=True)
    for a, b in zip(got[2], R):
        assert bits_equal(a.cpu().numpy(), b.cpu().numpy())
    assert abs(got[0] - ls) <= 1e-6 * abs(ls) and abs(got[1] - lu) <= 1e-6 * abs(lu)


def test_fused_is_deterministic(ctx, checker):
    og = OGrid(64, 64, 16, 1, 1, 1, 2e-3, True)
    w = checker.mlp_random_init(64, 777, 0.25)
    ctx.set_weights(_cfg(64), *w)
    a = ctx.fused_loss_acc(_g(og), 0.25, 2e-3).cpu().numpy()
    for _ in range(3):
        assert np.array_equal(ctx.fused_loss_acc(_g(og), 0.25, 2e-3).cpu().numpy(), a)


@pytest.mark.parametrize("shape,H,per", [((96, 80, 37), 64, True), ((70, 37, 19), 128, False), ((130, 66, 11), 32, True)])
def test_fused_repeatability_stress(ctx, checker, shape, H, per):
    """The split-phase barrier lets warps run up to one plane apart over a 4-deep ring of plane buffers; a
    missed hazard would show up as run-to-run differences.  40 launches must give bit-identical residuals
    (and they must equal the scalar, __syncthreads-based variant 3)."""
    import torch
    og = OGrid(*shape, 1, 1, 1, 2e-3, per)
    g = _g(og)
    w = checker.mlp_random_init(H, 777, 0.25)
    ctx.set_weights(_cfg(H), *w)
    ctx.set_fused_variant(3)
    ref = [torch.empty(og.N, device="cuda") for _ in range(4)]
    acc_ref = ctx.fused_loss_acc(g, 0.25, 2e-3, residuals=ref).clone()
    ctx.set_fused_variant(0)
    try:
        for it in range(40):
            R = [torch.full((og.N,), float("nan"), device="cuda") for _ in range(4)]
            acc = ctx.fused_loss_acc(g, 0.25, 2e-3, residuals=R)
            assert all(torch.equal(a, b) for a, b in zip(R, ref)), it
            assert torch.allclose(acc, acc_ref, rtol=1e-12, atol=0), it
    finally:
        ctx.set_fused_variant(0)


@pytest.mark.parametrize("shape,per,h,dt", [((40, 24, 13), True, (1, 1, 1), 2e-3), ((33, 18, 7), False, (0.5, 0.25, 2.0), 1e-2),
                                             ((256, 16, 9), True, (1, 1, 1), 1e-2), ((1, 1, 1), True, (1, 1, 1), 1e-2)])
def test_upwind_advection_switch(ctx, port, shape, per, h, dt):
    """The additive upwind switch of the stage-wise operators (physad_set_advection) against oracle.c's restatement:
    default fp32 arithmetic within the north-star tolerance, exact (double) mode to the last float bit; the loss is the
    double sum of those residuals; the fused kernel and the closed loop refuse while it is selected."""
    from phys_autodiff_b200 import PhysadError
    rng = np.random.default_rng(11)
    og = OGrid(*shape, *h, dt, per)
    g, N = _g(og), og.N
    f = [rng.uniform(-1, 1, n).astype(np.float32) for n in (N, N, N, 3 * N, 3 * N, 3 * N)]
    want = port.phys_residuals_upwind(og, f)
    central = port.phys_residuals(og, f)
    assert ctx.set_advection(True) is False
    try:
        got = ctx.phys_residuals_host(g, f)
        for a, b in zip(got, want):
            assert max_rel_to_max(a, b) <= TOL_FIELD
        if N > 1:
            assert any(max_rel_to_max(a, b) > 1e-3 for a, b in zip(got, central))     # it is a different scheme
        ls, lu, R = ctx.phys_loss_host(g, _pw(1.3, 0.7), f, want_residuals=True)
        s0 = 1.3 * np.sum(R[0].astype(np.float64) ** 2) / N
        s1 = 0.7 * sum(np.sum(r.astype(np.float64) ** 2) for r in R[1:]) / N
        assert abs(ls - s0) <= 1e-6 * s0 + 1e-30 and abs(lu - s1) <= 1e-6 * s1 + 1e-30
        ctx.set_exact_residuals(True)
        try:
            for a, b in zip(ctx.phys_residuals_host(g, f), want):
                assert bits_equal(a, b)
        finally:
            ctx.set_exact_residuals(False)
        huge = f[:3] + [(1e6 * a).astype(np.float32) for a in f[3:]]
        assert all(np.all(np.isfinite(r)) for r in ctx.phys_residuals_host(g, huge))
        w = port.mlp_random_init(32, 777, 0.25)
        with pytest.raises(PhysadError):
            ctx.fused_loss_host(g, _cfg(32), *w, _pw(), 0.25, dt)
        with pytest.raises(PhysadError):
            ctx.fused_loss_grad_host(g, _cfg(32), *w, _pw(), 0.25, dt)
    finally:
        assert ctx.set_advection(False) is True
    for a, b in zip(ctx.phys_residuals_host(g, f), central):
        assert max_rel_to_max(a, b) <= TOL_FIELD


@pytest.mark.parametrize("dtype", ["f16", "bf16"])
def test_reduced_precision_field_io(ctx, port, dtype):
    """16-bit field I/O of the stage-wise path (additive, REQUIREMENT.md:123-128): the stored fields are the strict-fp32
    MLP outputs rounded to nearest-even; the loss kernel widens them to fp32 and is then the fp32 kernel -- bitwise the
    same residuals as the fp32 kernel run on the widened values, and within the north-star tolerance of the CPU
    restatement on those values."""
    import torch
    from phys_autodiff_b200 import PhysadError
    td = {"f16": torch.float16, "bf16": torch.bfloat16}[dtype]
    og = OGrid(64, 24, 9, 1, 1, 1, 2e-3, True)
    g = _g(og)
    ctx.set_weights(_cfg(64), *port.mlp_random_init(64, 777, 0.25))
    f32 = ctx.mlp_generate_fields(g, 0.25, 2e-3)
    flp = ctx.mlp_generate_fields_lp(g, 0.25, 2e-3, dtype)
    for a, b in zip(f32, flp):
        assert b.dtype == td and torch.equal(b, a.to(td))
    wide = [x.float() for x in flp]
    acc, R = ctx.phys_loss_lp_acc(g, flp, dtype, want_residuals=True)
    acc32, R32 = ctx.phys_loss_acc(g, wide, want_residuals=True)
    assert all(torch.equal(a, b) for a, b in zip(R, R32))
    assert torch.allclose(acc, acc32, rtol=1e-12, atol=0)      # (narrow rows take the scalar fp32 kernel: another summation order)
    want = port.phys_residuals(og, [x.cpu().numpy() for x in wide])
    for a, b in zip(R, want):
        assert max_rel_to_max(a.cpu().numpy(), b) <= TOL_FIELD
    assert torch.equal(ctx.phys_loss_lp_acc(g, flp, dtype), acc)          # loss only: same sums
    s0 = float(torch.sum(R[0].double() ** 2))
    assert abs(float(acc[0]) - s0) <= 1e-9 * s0
    # a z-slab of the fields
    fs = ctx.mlp_generate_fields_lp(g, 0.25, 2e-3, dtype, slab=(2, 7))
    plane = og.nx * og.ny
    assert torch.equal(fs[1], flp[1][2 * plane: 7 * plane])
    og2 = OGrid(30, 8, 4, 1, 1, 1, 2e-3, True)                            # nx % 4 != 0: no 16-bit form
    f2 = ctx.mlp_generate_fields_lp(_g(og2), 0.25, 2e-3, dtype)
    with pytest.raises(PhysadError):
        ctx.phys_loss_lp_acc(_g(og2), f2, dtype)


@pytest.mark.parametrize("shape,H,m1p1,h", [((48, 40, 12), 64, True, (1, 1, 1)), ((33, 18, 7), 32, False, (0.5, 0.25, 2.0)),
                                              ((70, 37, 5), 128, True, (1, 1, 1)), ((1, 1, 1), 16, True, (1, 1, 1)),
                                              ((128, 64, 32), 64, True, (1, 1, 1))])
def test_tangent_loss_matches_its_checker(ctx, port, shape, H, m1p1, h):
    """The analytic forward-mode loss (additive; north_star's literal wording; NOT the parity path) against its checker
    oracle_tangent_loss (masks from the same fp32 pre-activations, the rest in double): residuals to 1e-5 of the largest,
    sums to 1e-6; z-slabs sum to the whole; repeatable."""
    import torch
    from phys_autodiff_b200.ops import slab_for_rank
    og = OGrid(*shape, *h, 2e-3, True)
    g = _g(og)
    w = port.mlp_random_init(H, 777, 0.25)
    want = port.tangent_loss(og, w, 0.25, m1p1, want_residuals=True)
    ctx.set_weights(_cfg(H, m1p1), *w)
    R = [torch.empty(og.N, device="cuda") for _ in range(4)]
    acc = ctx.tangent_loss_acc(g, 0.25, residuals=R).cpu().numpy()
    for a, b in zip(R, want["R"]):
        assert max_rel_to_max(a.cpu().numpy(), b) <= TOL_FIELD
    assert abs(acc[0] - want["acc_sigma"]) <= 1e-6 * want["acc_sigma"] + 1e-30
    assert abs(acc[1] - want["acc_u"]) <= 1e-6 * want["acc_u"] + 1e-30
    assert np.array_equal(ctx.tangent_loss_acc(g, 0.25).cpu().numpy(), acc)
    hl = _ops().mlp_phys_loss_tangent_cuda(g, _cfg(H, m1p1), w, _pw(1.3, 0.7), 0.25)      # host-buffer form
    assert hl == ctx.finalize(acc, _pw(1.3, 0.7), og.N)
    tot = np.zeros(2)
    for r in range(3):
        tot += ctx.tangent_loss_acc(g, 0.25, slab=slab_for_rank(og.nz, r, 3)).cpu().numpy()
    assert np.allclose(tot, acc, rtol=1e-12)


def test_slab_partials_sum_to_whole(ctx, checker):
    """Multi-GPU arithmetic on one GPU: slabs for world sizes 2/3/8 (halo planes recomputed, incl. the
    periodic wrap for the first/last slab) reproduce the whole-grid residuals and sums."""
    import torch
    from phys_autodiff_b200.ops import slab_for_rank
    for per in (True, False):
        og = OGrid(40, 24, 16, 1, 1, 1, 2e-3, per)
        g = _g(og)
        w = checker.mlp_random_init(32, 777, 0.25)
        ctx.set_weights(_cfg(32), *w)
        Rw = [torch.empty(og.N, device="cuda") for _ in range(4)]
        whole = ctx.fused_loss_acc(g, 0.25, 2e-3, residuals=Rw).cpu().numpy()
        for world in (2, 3, 8):
            tot = np.zeros(2)
            for r in range(world):
                z0, z1 = slab_for_rank(og.nz, r, world)
                n = (z1 - z0) * og.ny * og.nx
                Rl = [torch.empty(n, device="cuda") for _ in range(4)]
                tot += ctx.fused_loss_acc(g, 0.25, 2e-3, slab=(z0, z1), residuals=Rl).cpu().numpy()
                for a, b in zip(Rl, Rw):
                    assert torch.equal(a, b[z0 * og.ny * og.nx: z1 * og.ny * og.nx])
            assert np.allclose(tot, whole, rtol=1e-12)
        # empty slab (more ranks than planes)
        e = ctx.fused_loss_acc(g, 0.25, 2e-3, slab=(3, 3)).cpu().numpy()
        assert e[0] == 0.0 and e[1] == 0.0


def test_fused_full_size_128_properties(ctx, checker):
    """BASELINE config 3 (128^3, H=64 and 128) against the reference on all host threads where its library is built,
    and always against tests/golden/full128.npz (make_golden.py --full128): both losses and a seeded 4096-point sample
    of every residual, at the same tolerances and relative to the same whole-grid max|R|."""
    import os
    import oracle
    R = oracle.reference()
    stored = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "full128.npz"))
    og = OGrid(128, 128, 128, 1, 1, 1, 2e-3, True)
    for H in (64, 128):
        w = checker.mlp_random_init(H, 777, 0.25)
        got = ctx.fused_loss_host(_g(og), _cfg(H), *w, _pw(), 0.25, 2e-3, want_residuals=True)
        assert all(np.all(np.isfinite(r)) for r in got[2])
        ws, wu = (float(v) for v in stored[f"h{H}_loss"])
        assert abs(got[0] - ws) <= TOL_LOSS * ws and abs(got[1] - wu) <= TOL_LOSS * wu, (H, got[:2], ws, wu)
        for a, b, m in zip(got[2], stored[f"h{H}_R"], stored[f"h{H}_Rmax"]):
            assert np.max(np.abs(a[stored["idx"]].astype(np.float64) - b)) <= TOL_FIELD * m, H
        if R is not None:
            want = R.fused_loss(og, w, 0.25, 2e-3, threads=max(1, R.hardware_threads()), want_residuals=True)
            for a, b in zip(got[2], want["R"]):
                assert max_rel_to_max(a, b) <= TOL_FIELD
            assert abs(got[0] - want["loss_sigma"]) <= TOL_LOSS * want["loss_sigma"]
            assert abs(got[1] - want["loss_u"]) <= TOL_LOSS * want["loss_u"]
        else:  # size-independent property: loss == mean of squares of its own residuals
            s = np.sum(got[2][0].astype(np.float64) ** 2) / og.N
            assert abs(got[0] - s) <= 1e-6 * s


def test_fused_large_anisotropic_grid_equals_staged_path(ctx, checker):
    """A large non-cubic grid (23.6 M points, anisotropic spacing, clamp boundaries): the fused kernel's residuals
    equal the staged GPU path (fields -> vectorised stencil kernel) bitwise and its loss equals the double sum
    of its own residuals."""
    import torch
    og = OGrid(640, 384, 96, 0.5, 0.25, 2.0, 5e-3, False)
    g = _g(og)
    w = checker.mlp_random_init(32, 9, 0.3)
    ctx.set_weights(_cfg(32), *w)
    R = [torch.empty(og.N, device="cuda") for _ in range(4)]
    acc = ctx.fused_loss_acc(g, 0.1, 5e-3, residuals=R).cpu().numpy()
    f = ctx.mlp_generate_fields(g, 0.1, 5e-3)
    acc2, R2 = ctx.phys_loss_acc(g, f, want_residuals=True)
    for a, b in zip(R, R2):
        assert torch.equal(a, b)
    s0 = float(torch.sum(R[0].double() ** 2)); s1 = float(sum(torch.sum(r.double() ** 2) for r in R[1:]))
    assert abs(acc[0] - s0) <= 1e-9 * s0 and abs(acc[1] - s1) <= 1e-9 * s1
    assert np.allclose(acc2.cpu().numpy(), acc, rtol=1e-12)


@pytest.mark.parametrize("H", [64, 32, 128])
def test_fused_256_headline_losses_match_the_reference(ctx, checker, golden, H):
    """THE headline config (BASELINE.json metric: 256^3, seed 777, scale 0.25, t 0.25, dt 2e-3, periodic) and its
    width-sweep siblings against the losses the UNMODIFIED reference CPU path gives on the whole grid
    (tests/golden/make_golden.py section 3b), at the north-star's 1e-4 -- through the host-buffer C-ABI call that
    bench.py's e2e times, through the device call, and as the sum of the 8-GPU slab decomposition."""
    from phys_autodiff_b200.ops import slab_for_rank
    _, meta = golden
    want = meta["anchors"][f"256c_h{H}"]
    ws, wu = float(want["loss_sigma"]), float(want["loss_u"])
    og = OGrid(256, 256, 256, 1, 1, 1, 2e-3, True)
    g = _g(og)
    w = checker.mlp_random_init(H, 777, 0.25)
    ls, lu = ctx.fused_loss_host(g, _cfg(H), *w, _pw(), 0.25, 2e-3)
    assert abs(ls - ws) <= TOL_LOSS * ws and abs(lu - wu) <= TOL_LOSS * wu, (ls, ws, lu, wu)
    acc = ctx.fused_loss_acc(g, 0.25, 2e-3).cpu().numpy()
    l2 = ctx.finalize(acc, _pw(), og.N)
    assert l2[0] == ls and l2[1] == lu
    tot = np.zeros(2)
    for r in range(8):
        tot += ctx.fused_loss_acc(g, 0.25, 2e-3, slab=slab_for_rank(256, r, 8)).cpu().numpy()
    assert np.allclose(tot, acc, rtol=1e-12)
    l8 = ctx.finalize(tot, _pw(), og.N)
    assert abs(l8[0] - ws) <= TOL_LOSS * ws and abs(l8[1] - wu) <= TOL_LOSS * wu


def test_fused_256_matches_own_residual_sum_and_slabs(ctx, checker):
    """BASELINE config 4 size (256^3, H=64): loss equals the double sum of the kernel's own residuals;
    8 slabs (the 8-GPU decomposition) sum to the same; residual planes spot-checked against the CPU."""
    import torch
    from phys_autodiff_b200.ops import slab_for_rank
    og = OGrid(256, 256, 256, 1, 1, 1, 2e-3, True)
    g = _g(og)
    w = checker.mlp_random_init(64, 777, 0.25)
    ctx.set_weights(_cfg(64), *w)
    Rw = [torch.empty(og.N, device="cuda") for _ in range(4)]
    acc = ctx.fused_loss_acc(g, 0.25, 2e-3, residuals=Rw).cpu().numpy()
    s0 = float(torch.sum(Rw[0].double() ** 2)); s1 = float(sum(torch.sum(r.double() ** 2) for r in Rw[1:]))
    assert abs(acc[0] - s0) <= 1e-9 * s0 and abs(acc[1] - s1) <= 1e-9 * s1
    tot = np.zeros(2)
    for r in range(8):
        tot += ctx.fused_loss_acc(g, 0.25, 2e-3, slab=slab_for_rank(256, r, 8)).cpu().numpy()
    assert np.allclose(tot, acc, rtol=1e-12)
    # CPU spot check: planes 0 (wrap), 100, 255 via a 3-plane-thick evaluation of the oracle's MLP
    plane = 256 * 256
    for z in (0, 100, 255):
        zs = [(z - 1) % 256, z, (z + 1) % 256]
        sub = []
        for tt in (np.float32(0.25) - np.float32(2e-3), np.float32(0.25), np.float32(0.25) + np.float32(2e-3)):
            coords = np.empty((3, 256, 256, 4), np.float32)
            ax = (2 * (np.arange(256, dtype=np.float32) / np.float32(255)) - 1).astype(np.float32)
            coords[..., 0] = ax[None, None, :]; coords[..., 1] = ax[None, :, None]
            coords[..., 2] = ax[zs][:, None, None]; coords[..., 3] = tt
            sub.append(checker.mlp_forward(coords.reshape(-1), *w, 3 * plane, 4, 64, 4).reshape(3, plane, 4))
        # assemble 3-plane fields and evaluate the middle plane non-periodically in z is wrong at the
        # ends, so build a periodic 3-plane grid: z-neighbours of the middle plane are planes 0 and 2
        og3 = OGrid(256, 256, 3, 1, 1, 1, 2e-3, True)
        f = [np.ascontiguousarray(s[:, :, 0].reshape(-1)) for s in sub] + \
            [np.ascontiguousarray(np.concatenate([s[:, :, c].reshape(-1) for c in (1, 2, 3)])) for s in sub]
        want = checker.phys_residuals(og3, f)
        for a, b in zip(Rw, want):
            got = a[z * plane:(z + 1) * plane].cpu().numpy()
            assert max_rel_to_max(got, b[plane:2 * plane]) <= TOL_FIELD
