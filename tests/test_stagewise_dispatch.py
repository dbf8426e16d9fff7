"""GPU tier: every kernel the stage-wise physics operators can dispatch to, against the pinned C port.

launch_phys (capi.cu) picks k_phys_residual (32 x 8 tiles, any shape), k_phys_residual_v4 (quads of x, nx % 4 == 0 and
nx >= 128 or 16-bit fields, 16-byte aligned arrays) or refuses, from the shape, the pointer alignment, the dtype, the
exact-residual switch and the advection switch; phys_backward runs k_scale4 in a float4 or a scalar loop.  These tests run
each operation at shapes that land on each form, prove with torch.profiler which kernel ran, and hold it to the port:
to the last bit wherever the arithmetic is the port's (exact mode, the VJP, the fallbacks), within the north-star
tolerance otherwise.  They also run the grid shapes at the launch-geometry limits (many planes, many rows) and check that
what is still refused is refused before anything is written."""
import re
from contextlib import contextmanager

import numpy as np
import pytest

from helpers import assert_grad_close, bits_equal, max_rel_to_max
from oracle import Grid as OGrid

pytestmark = pytest.mark.gpu

TOL_FIELD = 1e-5
TOL_LOSS = 1e-4
PW = (1.1, 0.8)

# scalar kernel: ragged tiles; nx % 4 == 0 but nx < 128; nx >= 128 but nx % 4 != 0; one point; one row
SCALAR_SHAPES = [(33, 18, 7), (36, 10, 3), (130, 9, 5), (1, 1, 1), (5, 1, 1)]
# v4 kernel: many tiles; 33 quads (a block of 64 quads partly idle); a second block in x; nz = 1; ny = 1
V4_SHAPES = [(128, 96, 40), (132, 5, 9), (260, 7, 5), (512, 3, 1), (256, 1, 4)]
HOST_SHAPES = {(33, 18, 7), (130, 9, 5), (1, 1, 1), (128, 96, 40), (132, 5, 9)}
OPS = ("residuals", "loss_r", "loss", "vjp")
FLAGS = {"residuals": (1, 0, 0), "loss_r": (1, 1, 0), "loss": (0, 1, 0), "vjp": (1, 0, 1)}   # WRITE_R, REDUCE, SCALE


def _g(og):
    from phys_autodiff_b200 import Grid
    return Grid(og.nx, og.ny, og.nz, og.hx, og.hy, og.hz, og.dt, og.periodic)


def _cfg(H, m1p1=True):
    from phys_autodiff_b200 import MLPConfig
    return MLPConfig(4, H, 4, m1p1)


def _pw(a=PW[0], b=PW[1]):
    from phys_autodiff_b200 import PhysWeights
    return PhysWeights(a, b)


def _t(a):
    import torch
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def _np(x):
    return x.cpu().numpy()


def _fields(og, seed=3):
    """Random (non-smooth) fields: every stencil tap matters."""
    rng = np.random.default_rng(seed)
    return [rng.standard_normal(n).astype(np.float32) for n in (og.N,) * 3 + (3 * og.N,) * 3]


def _rel(a, b):
    return abs(float(a) - float(b)) / abs(float(b)) if b != 0 else abs(float(a))


@contextmanager
def _switches(ctx, exact, upwind):
    ctx.set_exact_residuals(exact)
    ctx.set_advection(upwind)
    try:
        yield
    finally:
        ctx.set_exact_residuals(False)
        ctx.set_advection(False)


def _b(v):
    return "true" if v else "false"


def expected_kernel(shape, op, exact=False, upwind=False, dtype="f32", aligned=True):
    """The instantiation launch_phys should pick, written as the demangled template name without spaces."""
    nx, ny, nz = shape
    w, r, s = FLAGS[op]
    v4 = (not upwind and aligned and nx % 4 == 0 and (nx >= 128 or dtype != "f32") and (nx * ny * nz) % 4 == 0
          and (ny + 1) // 2 <= 65535)
    if v4:
        e = {"f32": "float", "f16": "__half", "bf16": "__nv_bfloat16"}[dtype]
        return f"k_phys_residual_v4<{_b(w)},{_b(r)},{_b(s)},{_b(exact)},{e}>"
    return f"k_phys_residual<{_b(w)},{_b(r)},{_b(s)},{_b(exact)},{_b(upwind)}>"


def _run(ctx, g, fd, op):
    if op == "residuals":
        return ctx.phys_residuals(g, fd)
    if op == "loss_r":
        return ctx.phys_loss_acc(g, fd, want_residuals=True)
    if op == "loss":
        return ctx.phys_loss_acc(g, fd)
    return ctx.phys_backward_from_fields(g, _pw(), fd)


_KERNEL = re.compile(r"\b(k_phys_residual_v4|k_phys_residual|k_scale4)\b(<[^>]*>)?")


def _launched(fn):
    """(names of our stage-wise kernels fn launched, number of device kernels recorded), from torch.profiler."""
    import torch
    from torch.autograd import DeviceType
    from torch.profiler import ProfilerActivity, profile
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    ours, device = [], 0
    for e in prof.events():
        if e.device_type == DeviceType.CUDA:
            device += 1
        m = _KERNEL.search(e.name)
        if m:
            ours.append(re.sub(r"\s+", "", m.group(0)))
    return ours, device


def _ptr(x):
    from phys_autodiff_b200.capi import ptr
    return ptr(x)


def _offset_view(x, off):
    """A copy of device tensor x that starts `off` elements into a larger buffer (its data pointer is misaligned)."""
    import torch
    buf = torch.zeros(x.numel() + 8, dtype=x.dtype, device=x.device)
    v = buf[off:off + x.numel()]
    v.copy_(x)
    return v


# ------------------------------------------------------------------------------------------------
# a. the operator matrix
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("per", [True, False], ids=["periodic", "clamped"])
@pytest.mark.parametrize("shape", SCALAR_SHAPES + V4_SHAPES, ids=lambda s: "x".join(map(str, s)))
def test_operator_matrix(ctx, port, shape, per):
    """Residuals, loss with residuals, loss only and the VJP from fields, under both arithmetic modes and both advection
    schemes.  Exact arithmetic: residuals and VJP bitwise the port's.  Default arithmetic: within 1e-5 of the max."""
    import torch
    og = OGrid(*shape, 0.7, 1.3, 0.9, 3e-3, per)
    g, N = _g(og), og.N
    f = _fields(og)
    fd = [_t(a) for a in f]
    for exact in (False, True):
        for upwind in (False, True):
            case = (exact, upwind)
            want = port.phys_residuals_upwind(og, f) if upwind else port.phys_residuals(og, f)
            gwant = port.phys_loss_backward(og, *PW, want)
            with _switches(ctx, exact, upwind):
                R = [_np(x) for x in ctx.phys_residuals(g, fd)]
                acc, RL = ctx.phys_loss_acc(g, fd, want_residuals=True)
                acc_only = ctx.phys_loss_acc(g, fd)
                G = [_np(x) for x in ctx.phys_backward_from_fields(g, _pw(), fd)]
                host = None
                if shape in HOST_SHAPES:
                    host = (ctx.phys_residuals_host(g, f), ctx.phys_loss_host(g, _pw(), f, want_residuals=True),
                            ctx.phys_backward_from_fields_host(g, _pw(), f))
            RL = [_np(x) for x in RL]
            assert torch.equal(acc_only, acc), case                   # loss only: the same sums, bit for bit
            acc = _np(acc)
            if exact:
                for k in range(4):
                    assert bits_equal(R[k], want[k]) and bits_equal(RL[k], want[k]), (case, k)
                    assert bits_equal(G[k], gwant[k]), (case, k)
                ref = port.sumsq(want, 0, N)
                assert _rel(acc[0], ref[0]) <= 1e-12 and _rel(acc[1], ref[1]) <= 1e-12, case
            else:
                for k in range(4):
                    assert max_rel_to_max(R[k], want[k]) <= TOL_FIELD, (case, k)
                    assert max_rel_to_max(RL[k], want[k]) <= TOL_FIELD, (case, k)
                    # the VJP reference is the port's VJP of the port's residuals
                    assert max_rel_to_max(G[k], gwant[k]) <= TOL_FIELD, (case, k)
                own = port.sumsq(RL, 0, N)
                assert _rel(acc[0], own[0]) <= 1e-9 and _rel(acc[1], own[1]) <= 1e-9, case
            if host is not None:                                      # the host forms stage into scratch: same kernel
                hR, (ls, lu, hRL), hG = host
                ls_d, lu_d = ctx.finalize(acc, _pw(), N)
                assert ls == ls_d and lu == lu_d, case
                for k in range(4):
                    assert bits_equal(hR[k], R[k]) and bits_equal(hRL[k], RL[k]) and bits_equal(hG[k], G[k]), (case, k)


# ------------------------------------------------------------------------------------------------
# b. proof of dispatch
# ------------------------------------------------------------------------------------------------
def _all_instantiations():
    """Every k_phys_residual / k_phys_residual_v4 instantiation a public call can reach, and k_scale4."""
    names = set()
    for op in OPS:
        for exact in (False, True):
            for upwind in (False, True):
                names.add(expected_kernel((33, 18, 7), op, exact, upwind))
            names.add(expected_kernel((132, 5, 9), op, exact))
    for dtype in ("f16", "bf16"):
        for op in ("loss_r", "loss"):
            names.add(expected_kernel((132, 5, 9), op, dtype=dtype))
    return names | {"k_scale4"}


def test_dispatch_is_the_claimed_kernel(ctx):
    """Each case of the matrix, once, under torch.profiler: the kernel that ran is the instantiation the case claims to
    cover, and every reachable instantiation ran at least once."""
    import torch
    seen = set()

    def once(fn, want):
        got, device = _launched(fn)
        assert device > 0, "torch.profiler recorded no device kernels at all: the dispatch cannot be checked"
        assert got and set(got) == {want}, (want, got)
        seen.add(want)

    for shape, per in [(s, True) for s in SCALAR_SHAPES + V4_SHAPES] + [((132, 5, 9), False), ((33, 18, 7), False)]:
        og = OGrid(*shape, 0.7, 1.3, 0.9, 3e-3, per)
        g = _g(og)
        fd = [_t(a) for a in _fields(og)]
        for exact in (False, True):
            for upwind in (False, True):
                with _switches(ctx, exact, upwind):
                    for op in OPS:
                        once(lambda: _run(ctx, g, fd, op), expected_kernel(shape, op, exact, upwind))
        if shape[0] % 4 == 0 and shape[0] >= 128:
            # a misaligned field array takes the scalar kernel
            mis = [fd[0]] + [_offset_view(fd[1], 1)] + fd[2:]
            for exact in (False, True):
                with _switches(ctx, exact, False):
                    for op in OPS:
                        once(lambda: _run(ctx, g, mis, op), expected_kernel(shape, op, exact, aligned=False))
            for dtype, td in (("f16", torch.float16), ("bf16", torch.bfloat16)):
                flp = [x.to(td) for x in fd]
                once(lambda: ctx.phys_loss_lp_acc(g, flp, dtype, want_residuals=True), expected_kernel(shape, "loss_r", dtype=dtype))
                once(lambda: ctx.phys_loss_lp_acc(g, flp, dtype), expected_kernel(shape, "loss", dtype=dtype))
        R = ctx.phys_residuals(g, fd)
        once(lambda: ctx.phys_backward(g, _pw(), R), "k_scale4")
    missing = _all_instantiations() - seen
    assert not missing, sorted(missing)


# ------------------------------------------------------------------------------------------------
# c. alignment fallback
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("per", [True, False], ids=["periodic", "clamped"])
@pytest.mark.parametrize("shape", [(128, 96, 40), (132, 5, 9)], ids=lambda s: "x".join(map(str, s)))
def test_misaligned_fields_take_the_scalar_kernel_bitwise(ctx, port, shape, per):
    """The six fields (and then the residual outputs) as views 1, 2 and 3 floats into a larger buffer: the scalar kernel
    runs and gives the aligned v4 call's residuals and VJP bit for bit, in both arithmetic modes."""
    import torch
    og = OGrid(*shape, 0.7, 1.3, 0.9, 3e-3, per)
    g, N = _g(og), og.N
    fd = [_t(a) for a in _fields(og, 5)]
    for exact in (False, True):
        with _switches(ctx, exact, False):
            acc, R = ctx.phys_loss_acc(g, fd, want_residuals=True)
            Rr = ctx.phys_residuals(g, fd)
            G = ctx.phys_backward_from_fields(g, _pw(), fd)
            for off in (1, 2, 3):
                mis = [_offset_view(x, off) for x in fd]
                acc_m, R_m = ctx.phys_loss_acc(g, mis, want_residuals=True)
                assert all(torch.equal(a, b) for a, b in zip(R_m, R)), (exact, off)
                assert all(torch.equal(a, b) for a, b in zip(ctx.phys_residuals(g, mis), Rr)), (exact, off)
                assert all(torch.equal(a, b) for a, b in zip(ctx.phys_backward_from_fields(g, _pw(), mis), G)), (exact, off)
                assert torch.allclose(acc_m, acc, rtol=1e-12, atol=0), (exact, off)
                assert torch.equal(ctx.phys_loss_acc(g, mis), acc_m), (exact, off)
                # misaligned outputs
                outs = [_offset_view(torch.zeros(N, device="cuda"), off) for _ in range(4)]
                rc = ctx._lib.physad_phys_residuals_dev(ctx._h, _ref(g.c()), *[_ptr(x) for x in fd], *[_ptr(r) for r in outs],
                                                        ctx._stream())
                assert rc == 0
                assert all(torch.equal(a, b) for a, b in zip(outs, Rr)), (exact, off)
            if exact:
                want = port.phys_residuals(og, [_np(x) for x in fd])
                assert all(bits_equal(_np(a), b) for a, b in zip(R, want))


def _ref(c):
    import ctypes
    return ctypes.byref(c)


@pytest.mark.parametrize("shape,per", [((128, 96, 40), True), ((260, 7, 5), False)])
def test_misaligned_halo_planes(ctx, shape, per):
    """Slab mode with the two halo planes misaligned by 1, 2, 3 floats: the scalar kernel gives the aligned slab call's
    residuals bitwise and its sums to 1e-12."""
    import torch
    from phys_autodiff_b200 import Grid
    rng = np.random.default_rng(13)
    g = Grid(*shape, 0.7, 1.3, 0.9, 3e-3, per)
    N, pln = g.N, g.nx * g.ny
    f = [_t(rng.standard_normal(n).astype(np.float32)) for n in (N,) * 3 + (3 * N,) * 3]
    z0, z1 = 1, g.nz - 1
    n = (z1 - z0) * pln
    loc = [f[k][z0 * pln:z1 * pln].contiguous() if k < 3 else
           torch.cat([f[k][c * N + z0 * pln: c * N + z1 * pln] for c in range(3)]).contiguous() for k in range(6)]

    def tplane(z):
        return torch.stack([f[1][z * pln:(z + 1) * pln]] + [f[4][c * N + z * pln: c * N + (z + 1) * pln] for c in range(3)]).contiguous()
    lo, hi = ctx.halo_sources(g, (z0, z1))
    acc, R = ctx.phys_loss_slab_acc(g, (z0, z1), loc, tplane(lo), tplane(hi), want_residuals=True)
    _, Rw = ctx.phys_loss_acc(g, f, want_residuals=True)
    assert all(torch.equal(a, b[z0 * pln:z1 * pln]) for a, b in zip(R, Rw))
    assert R[0].numel() == n
    for off in (1, 2, 3):
        hl = _offset_view(tplane(lo).reshape(-1), off)
        hh = _offset_view(tplane(hi).reshape(-1), off)
        acc_m, R_m = ctx.phys_loss_slab_acc(g, (z0, z1), loc, hl, hh, want_residuals=True)
        assert all(torch.equal(a, b) for a, b in zip(R_m, R)), off
        assert torch.allclose(acc_m, acc, rtol=1e-12, atol=0), off


# ------------------------------------------------------------------------------------------------
# d. k_scale4
# ------------------------------------------------------------------------------------------------
def _special_residuals(N, seed):
    """Four residual arrays of ordinary values mixed with +-0, subnormals and +-inf (no NaN: GPU NaN payloads differ)."""
    rng = np.random.default_rng(seed)
    out = []
    tiny = np.array([0.0, -0.0, 1e-45, -1e-45, 3e-39, -3e-39, 1.1754942e-38, np.inf, -np.inf], np.float32)
    for _ in range(4):
        r = (rng.standard_normal(N) * 10.0 ** rng.integers(-30, 30, N)).astype(np.float32)
        pick = rng.random(N) < 0.2
        r[pick] = rng.choice(tiny, int(pick.sum()))
        r[:len(tiny)] = tiny[:min(N, len(tiny))]
        out.append(r)
    return out


@pytest.mark.parametrize("shape,misalign", [((16, 8, 5), 0), ((33, 18, 7), 0), ((16, 8, 5), 1), ((16, 8, 5), 3),
                                            ((160, 160, 100), 0), ((101, 101, 61), 0)],
                         ids=["vec4", "n%4!=0", "misaligned1", "misaligned3", "vec4-grid-loops", "scalar-grid-loops"])
def test_phys_backward_scale_bitwise(ctx, port, shape, misalign):
    """physad_phys_backward_dev / _host (k_scale4) against the port's g = (2 w / float(N)) R, bit for bit, on both of its
    loops, with a grid small enough that every thread visits more than one element on the two large shapes."""
    import torch
    og = OGrid(*shape, 1, 1, 1, 1e-3, True)
    N = og.N
    if shape == (160, 160, 100):
        assert N % 4 == 0 and N > ctx.sm_count * 16 * 256 * 4
    if shape == (101, 101, 61):
        assert N % 4 != 0 and N > ctx.sm_count * 16 * 256
    R = _special_residuals(N, 7)
    pw = (1.7, 0.9)
    want = port.phys_loss_backward(og, *pw, R)
    Rd = [_t(r) for r in R]
    if misalign:
        Rd = [_offset_view(r, misalign) for r in Rd]
    got = ctx.phys_backward(_g(og), _pw(*pw), Rd)
    for a, b in zip(got, want):
        assert bits_equal(_np(a), b)
    # misaligned outputs too
    outs = [_offset_view(torch.zeros(N, device="cuda"), 1) for _ in range(4)]
    cg, cw = _g(og).c(), _pw(*pw).c()
    assert ctx._lib.physad_phys_backward_dev(ctx._h, _ref(cg), _ref(cw), *[_ptr(r) for r in Rd], *[_ptr(x) for x in outs],
                                             ctx._stream()) == 0
    for a, b in zip(outs, want):
        assert bits_equal(_np(a), b)
    for a, b in zip(ctx.phys_backward_host(_g(og), _pw(*pw), R), want):
        assert bits_equal(a, b)


# ------------------------------------------------------------------------------------------------
# e. slabs under the switches
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("exact,upwind", [(True, False), (False, True), (True, True)], ids=["exact", "upwind", "exact-upwind"])
@pytest.mark.parametrize("shape,per", [((36, 10, 3), True), ((36, 10, 3), False), ((128, 96, 40), True), ((128, 96, 40), False)])
def test_slabs_with_halo_planes_under_the_switches(ctx, port, shape, per, exact, upwind):
    """The fields cut into 1/2/3/5 z-slabs, every slab given its two halo planes: each slab's residuals equal the whole
    grid's under the same switches bit for bit, the sums add up, and in exact mode the whole grid is the port's."""
    import torch
    from phys_autodiff_b200.ops import slab_for_rank
    og = OGrid(*shape, 0.7, 1.3, 0.9, 3e-3, per)
    g = _g(og)
    N, pln = g.N, g.nx * g.ny
    fh = _fields(og, 11)
    f = [_t(a) for a in fh]

    def planes(a, z0, z1, vec):
        if not vec:
            return a[z0 * pln:z1 * pln].contiguous()
        return torch.cat([a[c * N + z0 * pln: c * N + z1 * pln] for c in range(3)]).contiguous()

    def tplane(z):
        return torch.stack([f[1][z * pln:(z + 1) * pln]] + [f[4][c * N + z * pln: c * N + (z + 1) * pln] for c in range(3)]).contiguous()
    with _switches(ctx, exact, upwind):
        acc_w, Rw = ctx.phys_loss_acc(g, f, want_residuals=True)
        acc_w = _np(acc_w)
        if exact:
            want = port.phys_residuals_upwind(og, fh) if upwind else port.phys_residuals(og, fh)
            assert all(bits_equal(_np(a), b) for a, b in zip(Rw, want))
        for world in (1, 2, 3, 5):
            tot = np.zeros(2)
            for r in range(world):
                z0, z1 = slab_for_rank(g.nz, r, world)
                if z1 == z0:
                    continue
                loc = [planes(f[k], z0, z1, k >= 3) for k in range(6)]
                lo_z, hi_z = ctx.halo_sources(g, (z0, z1))
                acc, R = ctx.phys_loss_slab_acc(g, (z0, z1), loc, tplane(lo_z), tplane(hi_z), want_residuals=True)
                tot += _np(acc)
                for a, b in zip(R, Rw):
                    assert torch.equal(a, b[z0 * pln:z1 * pln]), (world, r)
            assert np.allclose(tot, acc_w, rtol=1e-12, atol=0), world


# ------------------------------------------------------------------------------------------------
# f. 16-bit fields
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("dtype", ["f16", "bf16"])
@pytest.mark.parametrize("shape,per", [((64, 24, 9), False), ((260, 7, 5), True), ((260, 7, 5), False), ((512, 3, 1), True),
                                       ((512, 3, 1), False), ((4, 3, 2), True), ((4, 3, 2), False)])
def test_reduced_precision_fields_at_more_shapes(ctx, port, shape, per, dtype):
    """k_phys_residual_v4 on 16-bit fields: bitwise the fp32 kernel on the widened fields, within 1e-5 of the port on
    them; the 16-bit MLP fields are the fp32 ones rounded.  Exact mode, or a 4-byte-misaligned array, is refused and
    writes nothing."""
    import torch
    from phys_autodiff_b200 import PhysadError
    td = {"f16": torch.float16, "bf16": torch.bfloat16}[dtype]
    og = OGrid(*shape, 0.7, 1.3, 0.9, 3e-3, per)
    g, N = _g(og), og.N
    ctx.set_weights(_cfg(64), *port.mlp_random_init(64, 777, 0.25))
    f32 = ctx.mlp_generate_fields(g, 0.25, 2e-3)
    for a, b in zip(f32, ctx.mlp_generate_fields_lp(g, 0.25, 2e-3, dtype)):
        assert b.dtype == td and torch.equal(b, a.to(td))
    flp = [_t(a).to(td) for a in _fields(og, 17)]
    wide = [x.float() for x in flp]
    acc, R = ctx.phys_loss_lp_acc(g, flp, dtype, want_residuals=True)
    acc32, R32 = ctx.phys_loss_acc(g, wide, want_residuals=True)
    assert all(torch.equal(a, b) for a, b in zip(R, R32))
    assert torch.allclose(acc, acc32, rtol=1e-12, atol=0)
    assert torch.equal(ctx.phys_loss_lp_acc(g, flp, dtype), acc)
    want = port.phys_residuals(og, [_np(x) for x in wide])
    for a, b in zip(R, want):
        assert max_rel_to_max(_np(a), b) <= TOL_FIELD
    own = port.sumsq([_np(r) for r in R], 0, N)
    assert _rel(_np(acc)[0], own[0]) <= 1e-9 and _rel(_np(acc)[1], own[1]) <= 1e-9

    def refused(fields):
        a0 = torch.full((2,), -7.0, dtype=torch.float64, device="cuda")
        outs = [torch.full((N,), -7.0, device="cuda") for _ in range(4)]
        code = {"f16": 1, "bf16": 2}[dtype]
        cg = g.c()
        import ctypes
        rc = ctx._lib.physad_phys_loss_lp_dev(ctx._h, _ref(cg), ctypes.c_int(code), *[_ptr(x) for x in fields], _ptr(a0),
                                              *[_ptr(r) for r in outs], ctx._stream())
        torch.cuda.synchronize()
        assert rc == -2, rc                                          # PHYSAD_E_UNSUPPORTED
        assert bool(torch.all(a0 == -7.0)) and all(bool(torch.all(r == -7.0)) for r in outs)

    ctx.set_exact_residuals(True)
    try:
        refused(flp)
        with pytest.raises(PhysadError, match="16-bit"):
            ctx.phys_loss_lp_acc(g, flp, dtype)
    finally:
        ctx.set_exact_residuals(False)
    refused([flp[0], _offset_view(flp[1], 2)] + flp[2:])             # 4 bytes off an 8-byte boundary


# ------------------------------------------------------------------------------------------------
# grid-shape limits
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("per", [True, False], ids=["periodic", "clamped"])
def test_more_than_65535_planes(ctx, port, per):
    """4 x 4 x 70001: the grid MLP goes out in bands of 65535 planes.  MLP outputs and fields bitwise the port's, the
    stage-wise and fused losses and the closed-loop gradient against the port, and a z-slab across plane 65535 equal to
    the whole grid's planes."""
    H, t, dt = 16, 0.25, 2e-3
    og = OGrid(4, 4, 70001, 1, 1, 1, dt, per)
    g, N, pln = _g(og), og.N, 16
    w = port.mlp_random_init(H, 777, 0.25)
    ctx.set_weights(_cfg(H), *w)
    assert bits_equal(_np(ctx.mlp_grid_infer(g, t)).ravel(), port.mlp_grid_infer(og, w, t))
    f = ctx.mlp_generate_fields(g, t, dt)
    fw = port.generate_fields(og, w, t, dt)
    for a, b in zip(f, fw):
        assert bits_equal(_np(a), b)
    ls, lu = ctx.phys_loss(g, _pw(1.3, 0.7), f)
    pls, plu = port.phys_loss_forward(og, 1.3, 0.7, fw)
    assert _rel(ls, pls) <= TOL_LOSS and _rel(lu, plu) <= TOL_LOSS
    fl = port.fused_loss(og, w, t, dt, 1.3, 0.7)
    acc = _np(ctx.fused_loss_acc(g, t, dt))
    assert _rel(acc[0], fl["acc_sigma"]) <= TOL_LOSS and _rel(acc[1], fl["acc_u"]) <= TOL_LOSS
    gl = port.phys_loss_grad(og, w, t, dt, 1.3, 0.7)
    gls, glu, grad = ctx.fused_loss_grad(g, _pw(1.3, 0.7), t, dt)
    assert_grad_close(grad, gl["grad"], H, 1, 1e-4)
    assert _rel(gls, gl["loss_sigma"]) <= TOL_LOSS and _rel(glu, gl["loss_u"]) <= TOL_LOSS
    z0, z1 = 60000, 70001
    n = (z1 - z0) * pln
    fs = ctx.mlp_generate_fields(g, t, dt, slab=(z0, z1))
    for k, (a, b) in enumerate(zip(fs, f)):
        if k < 3:
            assert bits_equal(_np(a), _np(b[z0 * pln:z1 * pln])), k
        else:
            for c in range(3):
                assert bits_equal(_np(a[c * n:(c + 1) * n]), _np(b[c * N + z0 * pln: c * N + z1 * pln])), (k, c)
    ys = ctx.mlp_grid_infer(g, t, slab=(z0, z1))
    assert bits_equal(_np(ys), _np(ctx.mlp_grid_infer(g, t))[z0 * pln:z1 * pln])


def test_v4_rows_beyond_131070_take_the_scalar_kernel(ctx, port):
    """128 x 131072 x 1: the v4 grid would need 65536 blocks in y, so fp32 fields take the scalar kernel (which it proves
    with the profiler) -- residuals, loss and VJP against the port, exact mode bitwise.  16-bit fields, which have no
    scalar form, are refused and write nothing; the closed loop on this grid now runs."""
    import torch
    from phys_autodiff_b200 import PhysadError
    shape = (128, 131072, 1)
    og = OGrid(*shape, 0.7, 1.3, 0.9, 3e-3, True)
    g, N = _g(og), og.N
    f = _fields(og, 19)
    fd = [_t(a) for a in f]
    want = port.phys_residuals(og, f)
    got, _ = _launched(lambda: ctx.phys_residuals(g, fd))
    assert got and set(got) == {expected_kernel(shape, "residuals")} and got[0].startswith("k_phys_residual<"), got
    R = [_np(x) for x in ctx.phys_residuals(g, fd)]
    for a, b in zip(R, want):
        assert max_rel_to_max(a, b) <= TOL_FIELD
    acc, RL = ctx.phys_loss_acc(g, fd, want_residuals=True)
    assert torch.equal(ctx.phys_loss_acc(g, fd), acc)
    own = port.sumsq([_np(r) for r in RL], 0, N)
    assert _rel(_np(acc)[0], own[0]) <= 1e-9 and _rel(_np(acc)[1], own[1]) <= 1e-9
    gwant = port.phys_loss_backward(og, *PW, want)
    for a, b in zip(ctx.phys_backward_from_fields(g, _pw(), fd), gwant):
        assert max_rel_to_max(_np(a), b) <= TOL_FIELD
    with _switches(ctx, True, False):
        for a, b in zip(ctx.phys_residuals(g, fd), want):
            assert bits_equal(_np(a), b)
        for a, b in zip(ctx.phys_backward_from_fields(g, _pw(), fd), gwant):
            assert bits_equal(_np(a), b)
    del fd
    flp = [_t(a).to(torch.bfloat16) for a in f]
    a0 = torch.full((2,), -7.0, dtype=torch.float64, device="cuda")
    outs = [torch.full((N,), -7.0, device="cuda") for _ in range(4)]
    import ctypes
    cg = g.c()
    rc = ctx._lib.physad_phys_loss_lp_dev(ctx._h, _ref(cg), ctypes.c_int(2), *[_ptr(x) for x in flp], _ptr(a0),
                                          *[_ptr(r) for r in outs], ctx._stream())
    torch.cuda.synchronize()
    assert rc == -2 and b"131070" in ctx._lib.physad_last_error()
    assert bool(torch.all(a0 == -7.0)) and all(bool(torch.all(r == -7.0)) for r in outs)
    with pytest.raises(PhysadError, match="131070"):
        ctx.phys_loss_lp_acc(g, flp, "bf16")
    del flp, outs
    # the closed loop's forward is the stage-wise pair: its sums equal them bit for bit
    ctx.set_weights(_cfg(16), *port.mlp_random_init(16, 777, 0.25))
    acc_g, grad = ctx.fused_loss_grad_acc(g, _pw(1.3, 0.7), 0.25, 2e-3)
    assert torch.equal(acc_g, ctx.phys_loss_acc(g, ctx.mlp_generate_fields(g, 0.25, 2e-3), want_residuals=True)[0])
    assert bool(torch.all(torch.isfinite(grad)))


def test_remaining_limits_are_refused_before_any_write(ctx, port):
    """Grid MLP with ny > 2097120 and the scalar physics kernel with ny > 524280 (also where v4 would have been eligible):
    PHYSAD_E_UNSUPPORTED with a message naming the limit, and every output left as it was."""
    import ctypes
    import torch
    from phys_autodiff_b200 import PhysadError
    ctx.set_weights(_cfg(16), *port.mlp_random_init(16, 777, 0.25))

    def untouched(*xs):
        torch.cuda.synchronize()
        return all(bool(torch.all(x == -7)) for x in xs)

    g = _g(OGrid(1, 2097121, 1, 1, 1, 1, 2e-3, True))
    N = g.N
    out = torch.full((4 * N,), -7.0, device="cuda")
    cg, cs = g.c(), ctx._slab(g, None)[0]
    assert ctx._lib.physad_mlp_grid_infer_dev(ctx._h, _ref(cg), _ref(cs), ctypes.c_float(0.25), _ptr(out), ctx._stream()) == -2
    assert b"2097120" in ctx._lib.physad_last_error() and untouched(out)
    fl = [torch.full((n,), -7.0, device="cuda") for n in (N,) * 3 + (3 * N,) * 3]
    assert ctx._lib.physad_mlp_generate_fields_dev(ctx._h, _ref(cg), _ref(cs), ctypes.c_float(0.25), ctypes.c_float(2e-3),
                                                   *[_ptr(x) for x in fl], ctx._stream()) == -2
    assert b"2097120" in ctx._lib.physad_last_error() and untouched(*fl)
    acc = torch.full((2,), -7.0, dtype=torch.float64, device="cuda")
    grad = torch.full((9 * 16 + 4,), -7.0, dtype=torch.float64, device="cuda")
    cw = _pw().c()
    assert ctx._lib.physad_fused_loss_grad_dev(ctx._h, _ref(cg), _ref(cw), ctypes.c_float(0.25), ctypes.c_float(2e-3),
                                               _ptr(acc), _ptr(grad), ctx._stream()) == -2
    assert b"2097120" in ctx._lib.physad_last_error() and untouched(acc, grad)
    with pytest.raises(PhysadError, match="2097120"):
        ctx.mlp_generate_fields(g, 0.25, 2e-3)
    del out, fl
    for shape in ((1, 524281, 1), (128, 524281, 1)):
        g = _g(OGrid(*shape, 1, 1, 1, 2e-3, True))
        N = g.N
        fields = [torch.zeros(n, device="cuda") for n in (N,) * 3 + (3 * N,) * 3]
        outs = [torch.full((N,), -7.0, device="cuda") for _ in range(4)]
        acc = torch.full((2,), -7.0, dtype=torch.float64, device="cuda")
        cg = g.c()
        assert ctx._lib.physad_phys_residuals_dev(ctx._h, _ref(cg), *[_ptr(x) for x in fields], *[_ptr(r) for r in outs],
                                                  ctx._stream()) == -2
        assert b"524280" in ctx._lib.physad_last_error() and untouched(*outs)
        assert ctx._lib.physad_phys_loss_dev(ctx._h, _ref(cg), *[_ptr(x) for x in fields], _ptr(acc),
                                             *[_ptr(r) for r in outs], ctx._stream()) == -2
        assert b"524280" in ctx._lib.physad_last_error() and untouched(acc, *outs)
        assert ctx._lib.physad_phys_backward_from_fields_dev(ctx._h, _ref(cg), _ref(cw), *[_ptr(x) for x in fields],
                                                             *[_ptr(r) for r in outs], ctx._stream()) == -2
        assert untouched(*outs)
        del fields, outs
