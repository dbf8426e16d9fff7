"""Periodic boundaries at points: the matched-pair loss of deeper networks and its gradient with respect to every layer's
weights, L_p = (1/n_norm) sum_i sum_o lam[o] (y(p_i)_o - y(q_i)_o)^2.

The checker is tests/deep_pair_checker.c (which includes deep_data_checker.c), compiled here into a temporary library.
CPU tier: the all-double gradient against central finite differences, the faithful gradient against two data-checker
calls with the partners' outputs as targets, identical and swapped pairs, ops.grid_periods, and the SASS / register report
of k_deep_pair_grad.  GPU tier: the kernel against the faithful checker at every depth, db2 exactly +0, the pair call
against the composition of forwards and data calls, repeatability and all entry points, shards, the weight states of the
context, error paths, training with a periodic term, the example, and a torchrun comparison across GPUs."""
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
NROW = {32: 768, 64: 384, 128: 192}   # rows per tile of k_deep_data_grad / k_deep_pair_grad
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


def _pairs(B, seed, kind="mixed", lo=-1.5, hi=1.5):
    """[B, 2, 4] float32 pairs: p uniform in [lo, hi]^4, q = p moved along one space axis (by a period-like offset), along t,
    or in all four inputs; "mixed" cycles through the three."""
    rng = np.random.default_rng(seed)
    p = rng.uniform(lo, hi, (B, 4)).astype(np.float32)
    q = p.copy()
    for i in range(B):
        k = {"axis": 0, "t": 1, "all": 2}.get(kind, i % 3)
        if k == 0:
            q[i, i % 3] += np.float32(rng.choice([2.0625, -2.0625, 1.0322581]))
        elif k == 1:
            q[i, 3] += np.float32(rng.uniform(-0.5, 0.5))
        else:
            q[i] = rng.uniform(lo, hi, 4).astype(np.float32)
    return np.ascontiguousarray(np.stack([p, q], 1))


class PairChecker:
    """ctypes surface of tests/deep_pair_checker.c and the data checker it includes."""

    def __init__(self, path):
        self.lib = C.CDLL(path)

    def run(self, H, L, theta, x, lam=None, n_norm=None, all_double=False):
        """-> (acc, grad[P] f64, y [B, 2, 4] f32 of the fp32 mode)."""
        theta = np.ascontiguousarray(theta, np.float64)
        x = np.ascontiguousarray(x, np.float32)
        B = x.size // 8
        acc = C.c_double()
        grad = np.empty(_plen(H, L), np.float64)
        y = np.empty((B, 2, 4), np.float32)
        lw = None if lam is None else (C.c_float * 4)(*[float(v) for v in lam])
        fp = lambda a: a.ctypes.data_as(C.c_void_p)
        rc = self.lib.oracle_pair_loss_grad_deep(C.c_int(H), C.c_int(L), fp(theta), fp(x), C.c_size_t(B), lw,
                                                 C.c_size_t(B if n_norm is None else n_norm), C.c_int(int(all_double)),
                                                 C.byref(acc), fp(grad), fp(y))
        assert rc == 0
        return acc.value, grad, y

    def data(self, H, L, theta, x, target, lam=None, n_norm=None):
        """oracle_data_loss_grad_deep, fp32-faithful mode -> (acc, grad)."""
        theta = np.ascontiguousarray(theta, np.float64)
        x, target = np.ascontiguousarray(x, np.float32), np.ascontiguousarray(target, np.float32)
        B = x.size // 4
        acc = C.c_double()
        grad = np.empty(_plen(H, L), np.float64)
        lw = None if lam is None else (C.c_float * 4)(*[float(v) for v in lam])
        fp = lambda a: a.ctypes.data_as(C.c_void_p)
        rc = self.lib.oracle_data_loss_grad_deep(C.c_int(H), C.c_int(L), fp(theta), fp(x), fp(target), C.c_size_t(B), lw,
                                                 C.c_size_t(B if n_norm is None else n_norm), C.c_int(0), C.byref(acc),
                                                 fp(grad), None)
        assert rc == 0
        return acc.value, grad


@pytest.fixture(scope="module")
def chk(tmp_path_factory):
    out = str(tmp_path_factory.mktemp("deep_pair_checker") / "libdeeppair.so")
    src = os.path.join(ROOT, "tests", "deep_pair_checker.c")
    subprocess.run([os.environ.get("CC", "gcc"), "-std=c11", "-O3", "-ffp-contract=off", "-fPIC", "-shared", "-o", out, src, "-lm"],
                   check=True, capture_output=True)
    return PairChecker(out)


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
    x = _pairs(B, 100 * L + B, kind)
    _, got, _ = chk.run(H, L, th, x, lam, n_norm, all_double=True)
    gmax = np.abs(got).max()
    assert gmax > 0
    rng = np.random.default_rng(L + B)
    for i in rng.choice(th.size, size=min(40, th.size), replace=False):
        eps = 1e-6 * max(1.0, abs(th[i]))
        tp, tm = th.copy(), th.copy()
        tp[i] += eps
        tm[i] -= eps
        fd = (chk.run(H, L, tp, x, lam, n_norm, True)[0] - chk.run(H, L, tm, x, lam, n_norm, True)[0]) / n_norm / (2 * eps)
        assert abs(fd - got[i]) <= 1e-6 * gmax + 1e-12, (i, fd, got[i], gmax)


@pytest.mark.parametrize("H,L,B,lam,n_norm", [(6, 1, 37, None, 37), (8, 2, 5, LAM, 9), (6, 3, 37, LAM, 100), (16, 5, 23, None, 23)])
def test_faithful_pair_gradient_is_two_data_calls(port, chk, H, L, B, lam, n_norm):
    """The seeds are the data checker's with the partner's fp32 output as target, so the two checkers agree."""
    th = _theta(_deep_weights(H, L, 3, 0.5, port))
    x = _pairs(B, H + L + B)
    acc, got, y = chk.run(H, L, th, x, lam, n_norm)
    W1, b1, Wh, bh, W2, b2 = _deep_weights(H, L, 3, 0.5, port)
    fwd = port.mlp_forward_deep(x.reshape(-1, 4), L, W1, b1, Wh, bh, W2, b2, 2 * B, 4, H, 4).reshape(B, 2, 4)
    assert np.array_equal(y.view(np.uint32), fwd.view(np.uint32))   # the faithful forward is oracle_mlp_forward_deep
    a1, g1 = chk.data(H, L, th, x[:, 0], y[:, 1], lam, n_norm)
    a2, g2 = chk.data(H, L, th, x[:, 1], y[:, 0], lam, n_norm)
    want = g1 + g2
    assert np.abs(got - want).max() <= 1e-14 * np.abs(want).max()
    assert abs(acc - a1) <= 1e-14 * abs(a1) and abs(acc - a2) <= 1e-14 * abs(a2)


@pytest.mark.parametrize("all_double", [False, True])
@pytest.mark.parametrize("L", [1, 3])
def test_identical_pairs_give_zero(port, chk, L, all_double):
    x = _pairs(17, 4)
    x[:, 1] = x[:, 0]
    acc, grad, _ = chk.run(8, L, _theta(_deep_weights(8, L, 5, 0.5, port)), x, LAM, 17, all_double)
    assert acc == 0.0 and not grad.any()


@pytest.mark.parametrize("all_double", [False, True])
def test_swapping_p_and_q_changes_nothing_but_the_order(port, chk, all_double):
    H, L, B = 8, 3, 29
    th = _theta(_deep_weights(H, L, 6, 0.5, port))
    x = _pairs(B, 9)
    a, g, _ = chk.run(H, L, th, x, LAM, B, all_double)
    b, h, _ = chk.run(H, L, th, x[:, ::-1], LAM, B, all_double)
    assert a == b
    assert np.abs(g - h).max() <= 1e-13 * np.abs(g).max()


def test_grid_periods():
    from phys_autodiff_b200 import Grid, ops
    for shape in ((32, 17, 1), (2, 256, 5), (1, 1, 129)):
        g = Grid(*shape)
        for norm, f in ((True, 2.0), (1, 2.0), (False, 1.0), (0, 1.0)):
            got = ops.grid_periods(g, norm)
            assert got.dtype == np.float32 and got.shape == (3,)
            want = np.array([np.float32(f * n / (n - 1)) if n > 1 else 0.0 for n in shape], np.float32)
            assert np.array_equal(got, want), (shape, norm)
            # the face plus one period is the grid's coordinate formula (oracle axis_coord) at the virtual index n
            for n, T in zip(shape, got):
                if n == 1:
                    assert T == 0.0
                    continue
                u = np.float32(np.float32(n) / np.float32(n - 1))
                at_n = np.float32(np.float32(2.0) * u - np.float32(1.0)) if f == 2.0 else u
                face = np.float32(-1.0) if f == 2.0 else np.float32(0.0)
                ulp = np.spacing(np.abs(at_n))
                assert abs(np.float32(face + T) - at_n) <= 4 * ulp, (n, norm, face + T, at_n)


def _sass_counts(path):
    r = subprocess.run(["cuobjdump", "-sass", path], capture_output=True, text=True)
    if r.returncode != 0:
        pytest.skip("cuobjdump unavailable")
    cur, counts = None, {}
    for line in r.stdout.splitlines():
        m = re.search(r"Function : (\S+)", line)
        if m:
            cur = m.group(1)
            counts[cur] = {"FFMA": 0, "FFMA2": 0, "FMUL2": 0, "FADD2": 0, "UTCHMMA": 0, "LDTM": 0, "STTM": 0}
            continue
        m = re.match(r"\s+/\*[0-9a-f]+\*/\s+(?:@!?U?P\d+\s+)?([A-Z0-9_]+)", line)
        if m and cur and m.group(1) in counts[cur]:
            counts[cur][m.group(1)] += 1
    return counts


def test_pair_kernel_sass():
    """k_deep_pair_grad<H>: the recomputed forward keeps FMUL2 / FADD2 separate, no FFMA2 anywhere, no tcgen05."""
    from phys_autodiff_b200 import capi
    p = capi.library_path()
    if not os.path.exists(p):
        capi.build_library()
    ks = {k: v for k, v in _sass_counts(p).items() if "k_deep_pair_grad" in k}
    assert len(ks) == 3, ks
    for k, v in ks.items():
        assert v["FMUL2"] > 0 and v["FADD2"] >= v["FMUL2"] and v["FFMA2"] == 0, (k, v)
        assert v["UTCHMMA"] == 0 and v["LDTM"] == 0 and v["STTM"] == 0, (k, v)


def _ptxas(tmp_path, name):
    nvcc = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    if not os.path.exists(nvcc):
        pytest.skip("nvcc unavailable")
    src = os.path.join(ROOT, "phys_autodiff_b200", "csrc", name)
    r = subprocess.run([nvcc, "-std=c++17", "-O3", "-gencode", "arch=compute_100a,code=sm_100a", "-Xptxas", "-v", "-c",
                        "-o", str(tmp_path / (name + ".o")), src], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr[-2000:]
    props = re.findall(r"Function properties for \S*?(k_\w+?)(?:ILi(\d+)E\w*)?\n\s+(\d+) bytes stack frame, (\d+) bytes spill "
                       r"stores, (\d+) bytes spill loads\nptxas info\s+: Used (\d+) registers", r.stderr)
    return {(k, int(H) if H else 0): (int(st), int(sp), int(sl), int(reg)) for k, H, st, sp, sl, reg in props}


def test_pair_kernel_has_no_spills_and_the_data_kernels_registers(tmp_path):
    """Measured with CUDA 12.9: k_deep_pair_grad 243 / 213 / 224 registers at H = 32 / 64 / 128, k_deep_data_grad 243 / 255 /
    224; no spills."""
    pair = _ptxas(tmp_path, "deep_pair_kernels.cu")
    data = _ptxas(tmp_path, "deep_data_kernels.cu")
    assert sorted(pair) == [("k_deep_pair_grad", H) for H in (32, 64, 128)], pair
    for (_, H), (st, sp, sl, reg) in pair.items():
        assert st == 0 and sp == 0 and sl == 0, (H, pair)
        assert reg <= data[("k_deep_data_grad", H)][3] + 8, (H, reg, data)


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


# B = 100 003 pairs only where the CPU checker stays quick
GPU_CASES = [(H, L, B) for H in (32, 64, 128) for L in (1, 2, 3, 5, 16) for B in (1, NROW[H] // 2 - 1, NROW[H] // 2 + 1)]
GPU_CASES += [(32, 1, 100003), (32, 3, 100003), (64, 2, 100003), (128, 1, 100003)]


@pytest.mark.gpu
@pytest.mark.parametrize("H,L,B", GPU_CASES)
def test_pair_gradient_vs_checker(ctx, port, chk, H, L, B):
    w = _depth_weights(H, L, 100 + H + L) if L == 16 else _deep_weights(H, L, 777, 0.25, port)
    x = _pairs(B, H + 10 * L + B)   # inside and outside [-1, 1]
    lam = LAM if (H + L) % 2 else None
    acc, want, _ = chk.run(H, L, _theta(w), x, lam, B)
    _set(ctx, H, L, w)
    out = ctx.deep_pair_loss_grad_acc(_dev(x), lam).cpu().numpy()
    assert out.shape == (_plen(H, L) + 1,)
    assert abs(out[0] - acc) <= 1e-6 * abs(acc), (out[0], acc)
    assert _bits_zero(out[-4:]), out[-4:]   # db2: the two seeds of every pair cancel exactly
    assert_grad_close(out[1:], want, H, L, 1e-4)


@pytest.mark.gpu
@pytest.mark.parametrize("H,L,B", [(32, 3, 50021), (64, 2, 3001), (128, 5, 20011)])
def test_pair_call_is_the_composition_of_forwards_and_data_calls(ctx, port, H, L, B):
    """What a caller could write without the pair call: y(p), y(q) by two forwards, then two data calls with the partners'
    outputs as targets.  The seeds are the same fp32 numbers; only the order of the fp32 tile sums differs."""
    _set(ctx, H, L, _deep_weights(H, L, 777, 0.25, port))
    x = _pairs(B, 3 * H + L)
    xd = _dev(x)
    p, q = _dev(x[:, 0]), _dev(x[:, 1])
    yp, yq = ctx.mlp_forward_deep(p), ctx.mlp_forward_deep(q)
    d1 = ctx.deep_data_loss_grad_acc(p, yq, LAM, B).cpu().numpy()
    d2 = ctx.deep_data_loss_grad_acc(q, yp, LAM, B).cpu().numpy()
    got = ctx.deep_pair_loss_grad_acc(xd, LAM).cpu().numpy()
    assert abs(got[0] - d1[0]) <= 1e-12 * abs(d1[0]) and abs(got[0] - d2[0]) <= 1e-12 * abs(d1[0])
    want = d1[1:] + d2[1:]
    assert_grad_close(got[1:], want, H, L, 1e-6)


@pytest.mark.gpu
def test_repeatable_and_all_forms_agree(ctx, port, tmp_path):
    from phys_autodiff_b200 import MLPConfig, capi, ops
    H, L, B = 64, 3, 30011
    w = _deep_weights(H, L, 777, 0.25, port)
    x = _pairs(B, 3)
    _set(ctx, H, L, w)
    xd = _dev(x)
    a = ctx.deep_pair_loss_grad_acc(xd, LAM).cpu().numpy()
    for _ in range(3):
        assert np.array_equal(ctx.deep_pair_loss_grad_acc(xd, LAM).cpu().numpy().view(np.uint64), a.view(np.uint64))
    lp, g = ctx.deep_pair_loss_grad(xd, LAM)
    assert lp == a[0] / B and np.array_equal(g.view(np.uint64), a[1:].view(np.uint64))
    hst = ctx.deep_pair_loss_grad_host(x, LAM)
    assert hst[0] == np.float32(a[0] / B)
    assert np.array_equal(np.concatenate(hst[1:]), a[1:].astype(np.float32))
    mod = ops.mlp_pair_loss_deep_grad_cuda(MLPConfig(4, H, 4, True), L, w, x, LAM)
    assert all(np.array_equal(p, q) for p, q in zip(mod, hst))
    # the C++ entry point
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
        f.write(x.tobytes() + np.array(LAM, np.float32).tobytes())
    r = subprocess.run([str(exe), str(inp), str(outp)], capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stdout + r.stderr
    got = np.fromfile(outp, np.float32)
    assert got[0] == hst[0] and np.array_equal(got[1:], np.concatenate(hst[1:]))


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
    std::vector<float> x;
    float lam[4];
    if (!rd(w.W1, 4 * H) || !rd(w.b1, H) || !rd(w.Wh, size_t(L - 1) * H * H) || !rd(w.bh, size_t(L - 1) * H) ||
        !rd(w.W2, 4 * H) || !rd(w.b2, 4) || !rd(x, 8 * B) || std::fread(lam, 4, 4, f) != 4) return 3;
    std::fclose(f);
    phys::MLPGridConfig cfg;
    cfg.dims.In = 4; cfg.dims.H = H; cfg.dims.Out = 4;
    float loss;
    phys::DeepMLPWeights g;
    phys::mlp_pair_loss_deep_grad_cuda(cfg, w, x.data(), B, lam, &loss, g);
    FILE* o = std::fopen(argv[2], "wb");
    std::fwrite(&loss, 4, 1, o);
    for (auto* v : {&g.W1, &g.b1, &g.Wh, &g.bh, &g.W2, &g.b2}) std::fwrite(v->data(), 4, v->size(), o);
    std::fclose(o);
    return 0;
}
'''


@pytest.mark.gpu
@pytest.mark.parametrize("H,L", [(32, 2), (64, 3), (128, 4)])
def test_shards_sum_to_the_whole(ctx, port, H, L):
    B = 10007
    _set(ctx, H, L, _deep_weights(H, L, 777, 0.25, port))
    x = _pairs(B, 5)
    whole = ctx.deep_pair_loss_grad_acc(_dev(x), LAM).cpu().numpy()
    for world in (2, 3, 8):
        cuts = [0] + [(r * B) // world for r in range(1, world)] + [B]
        cuts[1] = 0   # the first shard is empty
        tot = np.zeros_like(whole)
        for r in range(world):
            tot += ctx.deep_pair_loss_grad_acc(_dev(x[cuts[r]:cuts[r + 1]]), LAM, B).cpu().numpy()
        assert abs(tot[0] - whole[0]) <= 1e-12 * abs(whole[0]), world
        assert np.abs(tot[1:] - whole[1:]).max() <= 1e-5 * np.abs(whole[1:]).max(), world
    z = ctx.deep_pair_loss_grad_acc(_dev(np.zeros((0, 2, 4))), LAM, B).cpu().numpy()
    assert z.shape == (_plen(H, L) + 1,) and not z.any()
    hz = ctx.deep_pair_loss_grad_host(np.zeros((0, 2, 4)))
    assert hz[0] == 0 and not any(a.any() for a in hz[1:])


def _probe(c, x, B=64, n_norm=64, lam=None, xoff=0, aoff=0, goff=0, null=None):
    """The C-ABI device call on NaN-filled outputs: (status, outputs untouched)."""
    import torch
    from phys_autodiff_b200 import capi
    H = c.cfg.H if c.cfg is not None else 32
    buf = torch.full((_plen(H, 16) + 16,), float("nan"), dtype=torch.float64, device="cuda")
    pa = C.c_void_p(buf.data_ptr() + aoff)
    pg = C.c_void_p(buf[8:].data_ptr() + goff)
    px = C.c_void_p(x.data_ptr() + xoff)
    args = {"x": px, "acc": pa, "grad": pg}
    if null:
        args[null] = None
    torch.cuda.synchronize()
    rc = capi.lib().physad_deep_pair_loss_grad_dev(c._h, args["x"], C.c_size_t(B), lam, C.c_size_t(n_norm), args["acc"],
                                                   args["grad"], None)
    torch.cuda.synchronize()
    return rc, bool(torch.isnan(buf).all())


@pytest.mark.gpu
def test_weight_states_and_error_paths(port):
    """The pair call over the context's weight states (none, set_weights, deep L = 1, deep L > 1, deep mode 1, after a
    refused set_weights*), and every error path: each refused call returns its status and writes nothing."""
    from phys_autodiff_b200 import MLPConfig, PhysadError, capi, ops
    lib = capi.lib()
    c2 = ops.Context()
    try:
        H, L, B = 32, 3, 64
        xb = _dev(np.concatenate([_pairs(B, 1).ravel(), np.zeros(8, np.float32)]))
        w = _deep_weights(H, L, 1, 0.3, port)
        assert _probe(c2, xb) == (E_NOWEIGHTS, True)                                     # no weights
        c2.set_weights(MLPConfig(4, H, 4, True), w[0], w[1], w[4], w[5])
        assert _probe(c2, xb) == (E_NOWEIGHTS, True)                                     # one hidden layer, not deep
        c2.set_weights_deep(MLPConfig(4, H, 4, True), 1, w[0], w[1], None, None, w[4], w[5])
        rc, untouched = _probe(c2, xb)                                                   # deep, L = 1
        assert rc == 0 and not untouched
        one = c2.deep_pair_loss_grad_acc(xb[:8 * B].view(B, 2, 4)).cpu().numpy()
        assert one.shape == (_plen(H, 1) + 1,) and np.isfinite(one).all() and one[0] > 0
        _set(c2, H, L, w)                                                                # deep, L > 1
        deep = c2.deep_pair_loss_grad_acc(xb[:8 * B].view(B, 2, 4)).cpu().numpy()
        assert deep.shape == (_plen(H, L) + 1,) and deep[0] > 0
        c2.set_deep_mode(1)
        assert _probe(c2, xb) == (E_UNSUPPORTED, True)                                   # tensor-core mode
        with pytest.raises(PhysadError, match="strict"):
            c2.deep_pair_loss_grad_acc(xb[:8 * B].view(B, 2, 4))
        c2.set_deep_mode(0)
        bad = np.zeros(4 * 64, np.float32)                                              # refused set_weights_deep: L = 0
        assert lib.physad_set_weights_deep(c2._h, C.byref(MLPConfig(4, H, 4, True).c()), C.c_int(0), *[ops.ptr(bad)] * 6) != 0
        again = c2.deep_pair_loss_grad_acc(xb[:8 * B].view(B, 2, 4)).cpu().numpy()
        assert np.array_equal(again.view(np.uint64), deep.view(np.uint64))              # the network is still in place
        for kw in ({"null": "x"}, {"null": "acc"}, {"null": "grad"}, {"xoff": 4}, {"xoff": 8}, {"aoff": 4}, {"goff": 4},
                   {"n_norm": 0}, {"lam": (C.c_float * 4)(1, 1, -1, 1)}, {"lam": (C.c_float * 4)(1, float("nan"), 1, 1)},
                   {"lam": (C.c_float * 4)(float("inf"), 1, 1, 1)}):
            assert _probe(c2, xb, **kw) == (E_INVALID, True), kw
        assert lib.physad_deep_pair_loss_grad_dev(None, None, C.c_size_t(0), None, C.c_size_t(1), None, None, None) == E_INVALID
        assert lib.physad_deep_pair_loss_grad_host(c2._h, None, C.c_size_t(B), None, *[None] * 7) == E_INVALID
        assert lib.physad_deep_pair_loss_grad_host(None, None, C.c_size_t(0), None, *[None] * 7) == E_INVALID
        # null x with B = 0 is an empty shard, not an error
        assert _probe(c2, xb, B=0, null="x")[0] == 0
        r = c2.deep_pair_loss_grad_acc(xb[:8 * B].view(B, 2, 4)).cpu().numpy()
        assert np.array_equal(r.view(np.uint64), deep.view(np.uint64))                   # a refused call changes nothing
    finally:
        c2.close()


def _periodic_pairs(n, rng, T, t_range=(0.0, 0.5)):
    """n pairs across the faces of the [-1, 1]^3 domain, a third per space axis: p_a = -1, q = p + T_a e_a."""
    p = rng.uniform(-1, 1, (n, 4)).astype(np.float32)
    p[:, 3] = rng.uniform(*t_range, n).astype(np.float32)
    ax = np.arange(n) % 3
    p[np.arange(n), ax] = -1.0
    q = p.copy()
    q[np.arange(n), ax] += T[ax]
    return np.ascontiguousarray(np.stack([p, q], 1))


def _train(ctx, port, periodic):
    """Adam at H = 64, L = 3: analytic loss at 32 768 collocation points over t in [0, 0.5], data at 4 096 points at t = 0
    (a teacher network), and with `periodic` 4 096 fresh periodic pairs per step.  -> (first total, last total, held-out
    periodic mismatch)."""
    from phys_autodiff_b200 import Grid, PhysWeights, ops
    H, L = 64, 3
    g = Grid(32, 32, 32, 1, 1, 1, 2e-3, True)
    pw = PhysWeights(1, 1)
    T = ops.grid_periods(g, True)
    rng = np.random.default_rng(21)
    xc = rng.uniform(-1, 1, (32768, 4)).astype(np.float32)
    xc[:, 3] = rng.uniform(0.0, 0.5, 32768).astype(np.float32)
    xcd = _dev(xc)
    dcdx = ops.grid_input_scales(g, True)
    xdat = rng.uniform(-1, 1, (4096, 4)).astype(np.float32)
    xdat[:, 3] = 0.0
    xdd = _dev(xdat)
    _set(ctx, H, L, _deep_weights(H, L, 4242, 0.25, port))
    ydd = ctx.mlp_forward_deep(xdd).clone()
    held = _dev(_periodic_pairs(4096, np.random.default_rng(5), T))
    prng = np.random.default_rng(77)
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
        if periodic:
            lp, gp = ctx.deep_pair_loss_grad(_dev(_periodic_pairs(4096, prng, T)))
            total += lp
            gvec = gvec + gp
        last = total
        first = last if first is None else first
        m = 0.9 * m + 0.1 * gvec
        v = 0.999 * v + 0.001 * gvec * gvec
        th = th - 3e-3 * (m / (1 - 0.9 ** k)) / (np.sqrt(v / (1 - 0.999 ** k)) + 1e-8)
    _set(ctx, H, L, np.split(th.astype(np.float32), cuts))
    mismatch = float(ctx.deep_pair_loss_grad_acc(held).cpu().numpy()[0] / 4096)
    return first, last, mismatch


@pytest.mark.gpu
def test_training_with_a_periodic_term(ctx, port):
    """The total falls by >= 90 % in 120 steps, and the periodic mismatch on held-out pairs ends at most half that of the
    same run without the term.  Measured on a B200: total 0.110 -> 9.5e-4 (-99.1 %); held-out mismatch 1.6e-4 with the
    term, 5.5e-3 without (0.029x)."""
    first, last, with_term = _train(ctx, port, True)
    _, _, without = _train(ctx, port, False)
    print("periodic training", first, "->", last, "held-out mismatch", with_term, "without the term", without)
    assert np.isfinite(last) and last <= 0.1 * first, (first, last)
    assert with_term <= 0.5 * without, (with_term, without)


@pytest.mark.gpu
def test_example_with_periodic_boundaries():
    r = subprocess.run([sys.executable, os.path.join(ROOT, "examples", "train_closed_loop.py"), "--n", "32", "--layers", "3",
                        "--colloc", "8192", "--t-range", "0,0.5", "--data", "1024", "--periodic", "1024", "--steps", "5"],
                       capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-3000:]
    recs = [json.loads(ln) for ln in r.stdout.splitlines() if ln.startswith("{")]
    assert "loss_periodic" in recs[0] and "loss_data" in recs[0] and np.isfinite(recs[-1]["loss_last"])
    assert "periodic boundaries" in recs[-1]["summary"]


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
x = np.random.default_rng(1).uniform(-1, 1, (N, 2, 4)).astype(np.float32)
lo, hi = (rank * N) // world, ((rank + 1) * N) // world
lam = (0.7, 1.9, 0.0, 0.35)
lp, g = ctx.deep_pair_loss_grad(torch.from_numpy(x[lo:hi]).cuda(), lam)   # n_global found
one = ctx.deep_pair_loss_grad_acc(torch.from_numpy(x).cuda(), lam).cpu().numpy()   # all pairs here
out = dict(rank=rank, lp=lp, lp1=float(one[0] / N), grad_err=float(np.abs(g - one[1:]).max() / np.abs(one[1:]).max()))
gathered = [None] * world
dist.all_gather_object(gathered, out)
if rank == 0:
    print("RESULT " + json.dumps(gathered))
dist.destroy_process_group()
'''


@pytest.mark.gpu
def test_multi_gpu_pair_gradient_matches_single_gpu(tmp_path):
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs >= 2 GPUs")
    script = tmp_path / "worker.py"
    script.write_text(WORKER % ROOT)
    n = min(torch.cuda.device_count(), 8)
    r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={n}",
                        "--master-addr", "127.0.0.1", "--master-port", "29739", str(script)],
                       capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-4000:]
    res = json.loads([ln for ln in r.stdout.splitlines() if ln.startswith("RESULT ")][-1][len("RESULT "):])
    assert len(res) == n
    for d in res:
        assert d["lp"] == res[0]["lp"]
        assert abs(d["lp"] - d["lp1"]) <= 1e-6 * abs(d["lp1"])
        assert d["grad_err"] <= 1e-6, d["grad_err"]
