"""Shared test helpers: error norms in the reference's own terms and manufactured fields."""
import numpy as np


def max_rel_to_max(a, b):
    """max|a-b| / max|b| -- the per-array form of the north-star tolerance (SURVEY.md section 7:
    elementwise relative error is ill-defined where residuals cross zero)."""
    a = np.asarray(a, np.float64); b = np.asarray(b, np.float64)
    d = np.max(np.abs(a - b)) if a.size else 0.0
    m = np.max(np.abs(b)) if b.size else 0.0
    return d / m if m > 0 else d


def rel_l2(a, b):
    """The reference tests' metric (e.g. test/test_phys_cpu_ref.cpp:73-86)."""
    a = np.asarray(a, np.float64); b = np.asarray(b, np.float64)
    n = np.sqrt(np.sum(b * b))
    d = np.sqrt(np.sum((a - b) ** 2))
    return d / n if n > 0 else d


def bits_equal(a, b):
    """BIT equality of fp32 arrays: the uint32 views are compared, so +0 != -0 and NaN payloads count."""
    a = np.ascontiguousarray(a, np.float32); b = np.ascontiguousarray(b, np.float32)
    return a.shape == b.shape and bool(np.array_equal(a.view(np.uint32), b.view(np.uint32)))


def grad_segments(H, L):
    """Named slices of the weight-gradient layout dW1 | db1 | dWh1 .. dWh{L-1} | dbh1 .. dbh{L-1} | dW2 | db2 (the
    argument order of physad_set_weights_deep; with L = 1 the one-hidden-layer layout dW1 | db1 | dW2 | db2)."""
    sizes = [("dW1", 4 * H), ("db1", H)] + [(f"dWh{l}", H * H) for l in range(1, L)] + \
            [(f"dbh{l}", H) for l in range(1, L)] + [("dW2", 4 * H), ("db2", 4)]
    out, o = [], 0
    for name, n in sizes:
        out.append((name, slice(o, o + n)))
        o += n
    return out


def grad_error_ratios(got, want, H, L, floor=1e-3, floors=None):
    """Per tensor s: max|got_s - want_s| / max(max|want_s|, floor_s * max|want|), floor_s = floors.get(s, floor)."""
    got = np.asarray(got, np.float64).ravel(); want = np.asarray(want, np.float64).ravel()
    segs = grad_segments(H, L)
    assert got.shape == want.shape == (segs[-1][1].stop,), (got.shape, want.shape, segs[-1][1].stop)
    gmax = np.abs(want).max()
    out = {}
    for name, s in segs:
        err = np.abs(got[s] - want[s]).max()
        ref = max(np.abs(want[s]).max(), (floors or {}).get(name, floor) * gmax)
        out[name] = err / ref if ref > 0 else (0.0 if err == 0 else np.inf)
    return out


def assert_grad_close(got, want, H, L, tol=1e-4, floor=1e-3, floors=None):
    """Every tensor of the gradient on its own scale: max|got_s - want_s| <= tol * max(max|want_s|, floor * max|want|).
    One norm over the whole vector barely checks a tensor much smaller than the largest one.  floors = {tensor: floor}
    raises the floor of named tensors only, where a measured fp32 rounding error needs it.  Returns the largest ratio
    max|got_s - want_s| / max(...) over the tensors."""
    r = grad_error_ratios(got, want, H, L, floor, floors)
    bad = {k: v for k, v in r.items() if not v <= tol}
    assert not bad, "gradient tensors off by more than %g of their own scale: %s" % (
        tol, ", ".join(f"{k} ({v:.3g})" for k, v in bad.items()))
    return max(r.values())


def manufactured_fields(g, t, kx=1, ky=1, kz=1, const_u=True):
    """sigma = sin(kx x + ky y + kz z - t) on a 2*pi-periodic box, u = (1,1,1) or
    (sin z, cos x, sin y): the fields of test/test_phys_cpu_ref.cpp:32-48 and
    test/test_phys_cuda_fused_vs_nonfused.cpp:43-51 (float sinf/cosf like the reference)."""
    nx, ny, nz = g.nx, g.ny, g.nz
    x = (np.arange(nx, dtype=np.float32) * np.float32(g.hx))[None, None, :]
    y = (np.arange(ny, dtype=np.float32) * np.float32(g.hy))[None, :, None]
    z = (np.arange(nz, dtype=np.float32) * np.float32(g.hz))[:, None, None]
    N = g.N
    out_s, out_u = [], []
    for tt in (np.float32(t) - np.float32(g.dt), np.float32(t), np.float32(t) + np.float32(g.dt)):
        ph = (np.float32(kx) * x + np.float32(ky) * y + np.float32(kz) * z - tt).astype(np.float32)
        out_s.append(np.sin(ph).astype(np.float32).reshape(N))
        u = np.empty(3 * N, np.float32)
        if const_u:
            u[:] = 1.0
        else:
            u[0:N] = np.broadcast_to(np.sin(z), (nz, ny, nx)).reshape(N)
            u[N:2 * N] = np.broadcast_to(np.cos(x), (nz, ny, nx)).reshape(N)
            u[2 * N:] = np.broadcast_to(np.sin(y), (nz, ny, nx)).reshape(N)
        out_u.append(u)
    return out_s[0], out_s[1], out_s[2], out_u[0], out_u[1], out_u[2]
