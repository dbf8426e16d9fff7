"""Times the closed-loop step (loss + gradient w.r.t. the MLP weights): CUDA events around the launches of one
step (fields, residuals + sums, stencil adjoint, MLP backward [+ the all-reduce of 9H+6 doubles under torchrun]).
--loss tangent times the closed loop of the analytic loss instead (one kernel, physad_tangent_loss_grad_dev) and reports,
from the same process, the analytic forward alone, the finite-difference step, the counted flops and the GPU it ran on.
--loss deep times the closed loop of a deep network (physad_deep_loss_grad_dev) for every --hidden x --layers pair, in
alternation with the strict deep fields alone (generate_fields_deep) and the one-hidden-layer step; one JSON line per pair.
--loss deep-tangent times the analytic loss of a deep network (physad_deep_tangent_loss_dev) and its closed loop
(physad_deep_tangent_loss_grad_dev) for every --hidden x --layers pair, in alternation with the strict deep fields pass and
the finite-difference deep step (physad_deep_loss_grad_dev); one JSON line per pair.
--loss deep-data times the deep network at arbitrary points (physad_mlp_forward_deep_dev) and the data-fit loss + gradient
step (physad_deep_data_loss_grad_dev) at B = n^3 and B = n^2 random points for every --hidden x --layers pair, in
alternation with the strict grid forward (mlp_grid_infer_deep at n^3) and the finite-difference deep step; one JSON line per
pair and B, and with --out the whole run as one JSON document with the GPU's name and power limit.
--loss deep-tangent-points times the analytic deep loss at B uniform random space-time points
(physad_deep_tangent_points_loss_dev) and its loss + gradient step (physad_deep_tangent_points_loss_grad_dev) at B = n^3
and B = n^2, in alternation with the grid's analytic loss and loss + gradient step at n^3 (physad_deep_tangent_loss_dev /
_grad_dev); one JSON line per pair and B, and with --out the whole run as one JSON document.
  python tools/bench_grad.py [--loss fd|tangent|deep|deep-tangent|deep-data|deep-tangent-points] [--n 256] [--hidden 64]
                             [--layers 3] [--steps 20]
  python tools/bench_grad.py --loss deep --hidden 32,64,128 --layers 2,3,5
  python -m torch.distributed.run --nproc-per-node N --master-addr 127.0.0.1 tools/bench_grad.py   (z-slab per rank)"""
import argparse
import ctypes as C
import json
import subprocess
import sys, os

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch

from phys_autodiff_b200 import Grid, MLPConfig, PhysWeights, ops


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--n", type=int, default=256)
    ap.add_argument("--hidden", default="64", help="width; --loss deep takes a comma-separated list")
    ap.add_argument("--layers", default="3", help="--loss deep: hidden layers, a comma-separated list")
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--loss", choices=("fd", "tangent", "deep", "deep-tangent", "deep-data", "deep-tangent-points"), default="fd")
    ap.add_argument("--out", default=None, help="--loss deep-data / deep-tangent-points: also write the run as one JSON document here")
    a = ap.parse_args()
    if a.loss == "deep-tangent-points":
        return deep_tangent_points(a, Grid(a.n, a.n, a.n, 1, 1, 1, 2e-3, True))
    if a.loss == "deep-data":
        return deep_data(a, Grid(a.n, a.n, a.n, 1, 1, 1, 2e-3, True))
    if a.loss == "deep":
        return deep(a, Grid(a.n, a.n, a.n, 1, 1, 1, 2e-3, True))
    if a.loss == "deep-tangent":
        return deep_tangent(a, Grid(a.n, a.n, a.n, 1, 1, 1, 2e-3, True))
    a.hidden = int(a.hidden)
    g = Grid(a.n, a.n, a.n, 1, 1, 1, 2e-3, True)
    if "RANK" in os.environ and int(os.environ.get("WORLD_SIZE", "1")) > 1:
        return distributed(a, g)
    if a.loss == "tangent":
        return tangent(a, g)
    ctx = ops.Context()
    ctx.set_weights(MLPConfig(4, a.hidden, 4, True), *ops.mlp_random_init(a.hidden, 777, 0.25))
    pw = PhysWeights(1, 1)
    acc, grad = ctx.fused_loss_grad_acc(g, pw, 0.25, 2e-3)
    for _ in range(3):
        ctx.fused_loss_grad_acc(g, pw, 0.25, 2e-3, acc, grad)
    torch.cuda.synchronize()
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(a.steps)]
    for e0, e1 in ev:
        e0.record()
        ctx.fused_loss_grad_acc(g, pw, 0.25, 2e-3, acc, grad)
        e1.record()
    torch.cuda.synchronize()
    ms = sorted(e0.elapsed_time(e1) for e0, e1 in ev)
    fwd = []
    for _ in range(a.steps):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        ctx.fused_loss_acc(g, 0.25, 2e-3, acc=acc)
        e1.record()
        torch.cuda.synchronize()
        fwd.append(e0.elapsed_time(e1))
    fwd.sort()
    med = ms[len(ms) // 2]
    # backward-kernel work: per point and hidden unit 41 lane-ops (see grad_kernels.cuh) -> report the step only
    print(json.dumps({"workload": f"{a.n}^3 H={a.hidden} loss+grad", "ms_median": med, "ms_min": ms[0],
                      "gpts_per_s": g.N / med / 1e6, "forward_only_fused_ms": fwd[len(fwd) // 2],
                      "grad_norm": float(grad.norm()), "acc": acc.tolist()}))


def _times(fn, steps):
    """Sorted per-call milliseconds: CUDA events around each call, one sync at the end."""
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
    for e0, e1 in ev:
        e0.record()
        fn()
        e1.record()
    torch.cuda.synchronize()
    return sorted(e0.elapsed_time(e1) for e0, e1 in ev)


def _gpu():
    """Name and power limit of the current GPU (the limit read with nvidia-smi, None where it cannot be read)."""
    name = torch.cuda.get_device_name()
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader,nounits",
                            f"--id={torch.cuda.current_device()}"], capture_output=True, text=True, timeout=30)
        return name, float(q.stdout.strip().splitlines()[0])
    except (OSError, ValueError, IndexError, subprocess.TimeoutExpired):
        return name, None


# counted work of the analytic gradient per point and hidden unit (tangent_grad_kernels.cu): stage phase 7 (z) + 8 (y, 4 FMA)
# + 16 (the Jacobian's masked adds); backward 7 (z again) + 8 (W2^T yb) + 8 (yb a) + 6 (dz c) + 1 (dz) + 16 (the masked sums)
TANGENT_GRAD_FLOPS_PER_UNIT = 77


def tangent(a, g):
    ctx = ops.Context()
    ctx.set_weights(MLPConfig(4, a.hidden, 4, True), *ops.mlp_random_init(a.hidden, 777, 0.25))
    pw = PhysWeights(1, 1)
    out = ctx.tangent_loss_grad_acc(g, pw, 0.25)
    acc, grad = ctx.fused_loss_grad_acc(g, pw, 0.25, 2e-3)
    for _ in range(3):
        ctx.tangent_loss_grad_acc(g, pw, 0.25, out=out)
        ctx.tangent_loss_acc(g, 0.25, acc=acc)
        ctx.fused_loss_grad_acc(g, pw, 0.25, 2e-3, acc, grad)
    torch.cuda.synchronize()
    # the three are timed in alternation, so that they share whatever else the GPU is doing
    tg, tf, fd = [], [], []
    for _ in range(a.steps):
        tg += _times(lambda: ctx.tangent_loss_grad_acc(g, pw, 0.25, out=out), 1)
        tf += _times(lambda: ctx.tangent_loss_acc(g, 0.25, acc=acc), 1)
        fd += _times(lambda: ctx.fused_loss_grad_acc(g, pw, 0.25, 2e-3, acc, grad), 1)
    tg.sort(); tf.sort(); fd.sort()
    med = tg[len(tg) // 2]
    flops_pt = TANGENT_GRAD_FLOPS_PER_UNIT * a.hidden
    name, plim = _gpu()
    h = out.cpu().numpy()
    print(json.dumps({"workload": f"{a.n}^3 H={a.hidden} analytic loss+grad", "ms_median": med, "ms_min": tg[0],
                      "gpts_per_s": g.N / med / 1e6, "tangent_forward_ms": tf[len(tf) // 2],
                      "fd_loss_grad_ms": fd[len(fd) // 2], "flops_per_point": flops_pt,
                      "counted_tflops": flops_pt * g.N / (med * 1e-3) / 1e12, "gpu": name, "power_limit_w": plim,
                      "grad_norm": float(abs(h[2:]).max()), "acc": h[:2].tolist()}))


# counted work of one deep closed-loop step per row (a row = one point and time slice; 3 rows per point), 2 flops per
# multiply-add: the strict fields (hidden layers 2(L-1)H^2, layer 1 and output 16H), the recompute in k_deep_grad
# (2(L-1)H^2 + 8H), W^T delta_z and dW of every hidden layer (4(L-1)H^2), output layer and layer 1 backward (24H)
def deep_flops_per_point(H, L):
    return 3 * (8 * (L - 1) * H * H + 48 * H)


def deep(a, g):
    import numpy as np
    ctx = ops.Context()
    pw = PhysWeights(1, 1)
    name, plim = _gpu()
    for H in (int(x) for x in a.hidden.split(",")):
        w1 = ops.mlp_random_init(H, 777, 0.25)
        for L in (int(x) for x in a.layers.split(",")):
            rng = np.random.default_rng(L)
            Wh = rng.uniform(-0.2, 0.2, (L - 1) * H * H).astype(np.float32)
            bh = rng.uniform(-0.2, 0.2, (L - 1) * H).astype(np.float32)
            ctx.set_weights(MLPConfig(4, H, 4, True), *w1)
            acc, grad = ctx.fused_loss_grad_acc(g, pw, 0.25, 2e-3)
            ctx.set_weights_deep(MLPConfig(4, H, 4, True), L, w1[0], w1[1], Wh, bh, w1[2], w1[3])
            out = ctx.deep_loss_grad_acc(g, pw, 0.25, 2e-3)
            f = ctx.mlp_generate_fields_deep(g, 0.25, 2e-3)
            gen = lambda: ctx._lib.physad_mlp_generate_fields_deep_dev(ctx._h, C.byref(cg), None, C.c_float(0.25), C.c_float(2e-3),
                                                                       *[ops.ptr(x) for x in f], ctx._stream())
            cg = g.c()
            for _ in range(2):
                ctx.deep_loss_grad_acc(g, pw, 0.25, 2e-3, out=out)
                assert gen() == 0
            torch.cuda.synchronize()
            # the three are timed in alternation, so that they share whatever else the GPU is doing; the one-hidden-layer
            # step runs through the same context after set_weights (the deep weights are restored before the next deep call)
            dg, fw, fd = [], [], []
            for _ in range(a.steps):
                dg += _times(lambda: ctx.deep_loss_grad_acc(g, pw, 0.25, 2e-3, out=out), 1)
                fw += _times(gen, 1)
            ctx.set_weights(MLPConfig(4, H, 4, True), *w1)
            for _ in range(a.steps):
                fd += _times(lambda: ctx.fused_loss_grad_acc(g, pw, 0.25, 2e-3, acc, grad), 1)
            dg.sort(); fw.sort(); fd.sort()
            med = dg[len(dg) // 2]
            fl = deep_flops_per_point(H, L)
            h = out.cpu().numpy()
            print(json.dumps({"workload": f"{a.n}^3 H={H} L={L} deep loss+grad", "ms_median": med, "ms_min": dg[0],
                              "fields_deep_ms": fw[len(fw) // 2], "ratio_to_fields": med / fw[len(fw) // 2],
                              "fd_one_layer_loss_grad_ms": fd[len(fd) // 2], "flops_per_point": fl,
                              "counted_tflops": fl * g.N / (med * 1e-3) / 1e12, "gpu": name, "power_limit_w": plim,
                              "grad_absmax": float(abs(h[2:]).max()), "acc": h[:2].tolist()}), flush=True)


# counted work of the analytic deep loss per point (5 rows: value + 4 tangents), 2 flops per multiply-add: layer 1 value
# row 8H; every hidden layer 5 rows x 2H^2; output layer 8H (y) + 32H (J).  The closed loop adds, per point: dW2 and
# W2^T seed over 5 rows (80H), dW and W^T delta of every hidden layer over 5 rows (20(L-1)H^2), dW1 over 5 rows (40H).
# The strict fields pass does 3 rows per point of 2(L-1)H^2 + 16H.
def deep_tangent_flops_per_point(H, L, grad):
    fwd = 10 * (L - 1) * H * H + 48 * H
    return fwd + (20 * (L - 1) * H * H + 120 * H if grad else 0)


def deep_fields_flops_per_point(H, L):
    return 3 * (2 * (L - 1) * H * H + 16 * H)


def deep_tangent(a, g):
    import numpy as np
    ctx = ops.Context()
    pw = PhysWeights(1, 1)
    name, plim = _gpu()
    cg = g.c()
    for H in (int(x) for x in a.hidden.split(",")):
        w1 = ops.mlp_random_init(H, 777, 0.25)
        for L in (int(x) for x in a.layers.split(",")):
            rng = np.random.default_rng(L)
            Wh = rng.uniform(-0.2, 0.2, (L - 1) * H * H).astype(np.float32)
            bh = rng.uniform(-0.2, 0.2, (L - 1) * H).astype(np.float32)
            ctx.set_weights_deep(MLPConfig(4, H, 4, True), L, w1[0], w1[1], Wh, bh, w1[2], w1[3])
            acc = ctx.deep_tangent_loss_acc(g, 0.25)
            out = ctx.deep_tangent_loss_grad_acc(g, pw, 0.25)
            fdo = ctx.deep_loss_grad_acc(g, pw, 0.25, 2e-3)
            f = ctx.mlp_generate_fields_deep(g, 0.25, 2e-3)
            gen = lambda: ctx._lib.physad_mlp_generate_fields_deep_dev(ctx._h, C.byref(cg), None, C.c_float(0.25), C.c_float(2e-3),
                                                                       *[ops.ptr(x) for x in f], ctx._stream())
            loss = lambda: ctx.deep_tangent_loss_acc(g, 0.25, acc=acc)
            step = lambda: ctx.deep_tangent_loss_grad_acc(g, pw, 0.25, out=out)
            fdstep = lambda: ctx.deep_loss_grad_acc(g, pw, 0.25, 2e-3, out=fdo)
            for _ in range(2):
                loss(); step(); fdstep()
                assert gen() == 0
            torch.cuda.synchronize()
            # the four are timed in alternation, so that they share whatever else the GPU is doing
            tl, tg, fw, fd = [], [], [], []
            for _ in range(a.steps):
                tl += _times(loss, 1)
                tg += _times(step, 1)
                fw += _times(gen, 1)
                fd += _times(fdstep, 1)
            for x in (tl, tg, fw, fd):
                x.sort()
            ml, mg, mf, md = (x[len(x) // 2] for x in (tl, tg, fw, fd))
            fl, fg = deep_tangent_flops_per_point(H, L, False), deep_tangent_flops_per_point(H, L, True)
            ff, fdf = deep_fields_flops_per_point(H, L), deep_flops_per_point(H, L)
            h = out.cpu().numpy()
            print(json.dumps({"workload": f"{a.n}^3 H={H} L={L} deep analytic loss / loss+grad",
                              "loss_ms": ml, "loss_grad_ms": mg, "fields_deep_ms": mf, "fd_deep_loss_grad_ms": md,
                              "loss_ratio_to_fields": ml / mf, "loss_gpts_per_s": g.N / ml / 1e6, "loss_grad_gpts_per_s": g.N / mg / 1e6,
                              "loss_flops_per_point": fl, "loss_grad_flops_per_point": fg,
                              "loss_counted_tflops": fl * g.N / (ml * 1e-3) / 1e12,
                              "loss_grad_counted_tflops": fg * g.N / (mg * 1e-3) / 1e12,
                              "fields_counted_tflops": ff * g.N / (mf * 1e-3) / 1e12,
                              "fd_deep_loss_grad_counted_tflops": fdf * g.N / (md * 1e-3) / 1e12,
                              "gpu": name, "power_limit_w": plim,
                              "grad_absmax": float(abs(h[2:]).max()), "acc": h[:2].tolist(),
                              "acc_loss_call_equal": bool((acc.cpu().numpy() == h[:2]).all())}), flush=True)


# counted work per point of the forward at points (one row: hidden layers 2(L-1)H^2, layer 1 and output 16H) and of the data
# loss + gradient step (the forward, W^T delta and dW of every hidden layer, output layer and layer 1 backward:
# 8(L-1)H^2 + 48H, the per-row count of deep_flops_per_point)
def deep_points_flops_per_point(H, L):
    return 2 * (L - 1) * H * H + 16 * H


def deep_data_flops_per_point(H, L):
    return 8 * (L - 1) * H * H + 48 * H


def deep_data(a, g):
    import numpy as np
    ctx = ops.Context()
    pw = PhysWeights(1, 1)
    name, plim = _gpu()
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=clocks.max.sm", "--format=csv,noheader,nounits",
                            f"--id={torch.cuda.current_device()}"], capture_output=True, text=True, timeout=30)
        clk = float(q.stdout.strip().splitlines()[0])
    except (OSError, ValueError, IndexError, subprocess.TimeoutExpired):
        clk = None
    cg = g.c()
    rng = np.random.default_rng(5)
    sizes = (g.N, g.nx * g.ny)   # the point count of the grid, and one plane (the overhead regime)
    xs = {B: torch.from_numpy(rng.uniform(-1, 1, (B, 4)).astype(np.float32)).cuda() for B in sizes}
    ts = {B: torch.from_numpy(rng.uniform(-1, 1, (B, 4)).astype(np.float32)).cuda() for B in sizes}
    results = []
    for H in (int(x) for x in a.hidden.split(",")):
        w1 = ops.mlp_random_init(H, 777, 0.25)
        for L in (int(x) for x in a.layers.split(",")):
            wr = np.random.default_rng(L)
            Wh = wr.uniform(-0.2, 0.2, (L - 1) * H * H).astype(np.float32)
            bh = wr.uniform(-0.2, 0.2, (L - 1) * H).astype(np.float32)
            ctx.set_weights_deep(MLPConfig(4, H, 4, True), L, w1[0], w1[1], Wh, bh, w1[2], w1[3])
            grid_out = ctx.mlp_grid_infer_deep(g, 0.25)
            infer = lambda: ctx._lib.physad_mlp_grid_infer_deep_dev(ctx._h, C.byref(cg), None, C.c_float(0.25), ops.ptr(grid_out),
                                                                    ctx._stream())
            fdo = ctx.deep_loss_grad_acc(g, pw, 0.25, 2e-3)
            fdstep = lambda: ctx.deep_loss_grad_acc(g, pw, 0.25, 2e-3, out=fdo)
            for B in sizes:
                x, t = xs[B], ts[B]
                y = ctx.mlp_forward_deep(x)
                dout = ctx.deep_data_loss_grad_acc(x, t)
                fwd = lambda: ctx._lib.physad_mlp_forward_deep_dev(ctx._h, ops.ptr(x), ops.ptr(y), C.c_size_t(B), ctx._stream())
                step = lambda: ctx.deep_data_loss_grad_acc(x, t, out=dout)
                for _ in range(2):
                    assert fwd() == 0 and infer() == 0
                    step(); fdstep()
                torch.cuda.synchronize()
                # the four are timed in alternation, so that they share whatever else the GPU is doing
                tf, ti, td, tfd = [], [], [], []
                for _ in range(a.steps):
                    tf += _times(fwd, 1)
                    ti += _times(infer, 1)
                    td += _times(step, 1)
                    tfd += _times(fdstep, 1)
                for v in (tf, ti, td, tfd):
                    v.sort()
                mf, mi, md, mfd = (v[len(v) // 2] for v in (tf, ti, td, tfd))
                ff, fdd, fdf = deep_points_flops_per_point(H, L), deep_data_flops_per_point(H, L), deep_flops_per_point(H, L)
                dt_tf, fd_tf = fdd * B / (md * 1e-3) / 1e12, fdf * g.N / (mfd * 1e-3) / 1e12
                h = dout.cpu().numpy()
                r = {"workload": f"H={H} L={L} B={B} deep forward at points / data loss+grad", "points": B,
                     "forward_points_ms": mf, "grid_infer_deep_ms": mi, "data_loss_grad_ms": md, "fd_deep_loss_grad_ms": mfd,
                     "forward_per_point_ratio_to_grid_infer": (mf / B) / (mi / g.N),
                     "forward_points_gpts_per_s": B / mf / 1e6, "data_loss_grad_gpts_per_s": B / md / 1e6,
                     "forward_flops_per_point": ff, "data_flops_per_point": fdd, "fd_deep_flops_per_point": fdf,
                     "forward_counted_tflops": ff * B / (mf * 1e-3) / 1e12,
                     "grid_infer_counted_tflops": ff * g.N / (mi * 1e-3) / 1e12,
                     "data_counted_tflops": dt_tf, "fd_deep_counted_tflops": fd_tf, "data_to_fd_tflops_ratio": dt_tf / fd_tf,
                     "gpu": name, "power_limit_w": plim, "grad_absmax": float(abs(h[1:]).max()), "acc": float(h[0])}
                results.append(r)
                print(json.dumps(r), flush=True)
    if a.out:
        with open(a.out, "w") as fh:
            json.dump({"what": f"tools/bench_grad.py --loss deep-data --hidden {a.hidden} --layers {a.layers} --steps {a.steps} "
                               f"at {a.n}^3: the forward at B random points, mlp_grid_infer_deep on the grid, the data loss + "
                               f"gradient step at the same B points and the finite-difference deep step on the grid, timed in "
                               f"alternation (CUDA events, median of {a.steps}); B = {sizes[0]} and {sizes[1]}",
                       "gpu": name, "power_limit_w": plim, "clocks_max_sm_mhz": clk, "results": results}, fh, indent=1)


def deep_tangent_points(a, g):
    import numpy as np
    ctx = ops.Context()
    pw = PhysWeights(1, 1)
    name, plim = _gpu()
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=clocks.max.sm", "--format=csv,noheader,nounits",
                            f"--id={torch.cuda.current_device()}"], capture_output=True, text=True, timeout=30)
        clk = float(q.stdout.strip().splitlines()[0])
    except (OSError, ValueError, IndexError, subprocess.TimeoutExpired):
        clk = None
    dcdx = ops.grid_input_scales(g, True)
    rng = np.random.default_rng(5)
    sizes = (g.N, g.nx * g.ny)   # the grid's point count, and one plane (the overhead regime)
    # uniform random space-time points: space in [-1, 1]^3, the time input (MinusOneToOne: t) in [0, 0.5]
    xs = {}
    for B in sizes:
        x = rng.uniform(-1, 1, (B, 4)).astype(np.float32)
        x[:, 3] = rng.uniform(0.0, 0.5, B).astype(np.float32)
        xs[B] = torch.from_numpy(x).cuda()
    results = []
    for H in (int(v) for v in a.hidden.split(",")):
        w1 = ops.mlp_random_init(H, 777, 0.25)
        for L in (int(v) for v in a.layers.split(",")):
            wr = np.random.default_rng(L)
            Wh = wr.uniform(-0.2, 0.2, (L - 1) * H * H).astype(np.float32)
            bh = wr.uniform(-0.2, 0.2, (L - 1) * H).astype(np.float32)
            ctx.set_weights_deep(MLPConfig(4, H, 4, True), L, w1[0], w1[1], Wh, bh, w1[2], w1[3])
            gacc = ctx.deep_tangent_loss_acc(g, 0.25)
            gout = ctx.deep_tangent_loss_grad_acc(g, pw, 0.25)
            calls = {"grid_loss": lambda: ctx.deep_tangent_loss_acc(g, 0.25, acc=gacc),
                     "grid_loss_grad": lambda: ctx.deep_tangent_loss_grad_acc(g, pw, 0.25, out=gout)}
            outs = {}
            for B in sizes:
                pacc = ctx.deep_tangent_points_loss_acc(xs[B], dcdx)
                pout = ctx.deep_tangent_points_loss_grad_acc(xs[B], dcdx, pw)
                outs[B] = pout
                calls[f"points_loss_{B}"] = lambda x=xs[B], o=pacc: ctx.deep_tangent_points_loss_acc(x, dcdx, acc=o)
                calls[f"points_loss_grad_{B}"] = lambda x=xs[B], o=pout: ctx.deep_tangent_points_loss_grad_acc(x, dcdx, pw, out=o)
            for _ in range(2):
                for fn in calls.values():
                    fn()
            torch.cuda.synchronize()
            # every call is timed in alternation with the others, so that they share whatever else the GPU is doing
            ts = {k: [] for k in calls}
            for _ in range(a.steps):
                for k, fn in calls.items():
                    ts[k] += _times(fn, 1)
            med = {k: sorted(v)[len(v) // 2] for k, v in ts.items()}
            ml, mg = med["grid_loss"], med["grid_loss_grad"]
            for B in sizes:
                pl, pg = med[f"points_loss_{B}"], med[f"points_loss_grad_{B}"]
                h = outs[B].cpu().numpy()
                r = {"workload": f"H={H} L={L} B={B} deep analytic loss / loss+grad at points vs the grid at {a.n}^3", "points": B,
                     "points_loss_ms": pl, "points_loss_grad_ms": pg, "grid_loss_ms": ml, "grid_loss_grad_ms": mg,
                     "loss_per_point_ratio_to_grid": (pl / B) / (ml / g.N),
                     "loss_grad_per_point_ratio_to_grid": (pg / B) / (mg / g.N),
                     "points_loss_gpts_per_s": B / pl / 1e6, "points_loss_grad_gpts_per_s": B / pg / 1e6,
                     "loss_counted_tflops": deep_tangent_flops_per_point(H, L, False) * B / (pl * 1e-3) / 1e12,
                     "loss_grad_counted_tflops": deep_tangent_flops_per_point(H, L, True) * B / (pg * 1e-3) / 1e12,
                     "gpu": name, "power_limit_w": plim, "grad_absmax": float(abs(h[2:]).max()), "acc": h[:2].tolist()}
                results.append(r)
                print(json.dumps(r), flush=True)
    if a.out:
        with open(a.out, "w") as fh:
            json.dump({"what": f"tools/bench_grad.py --loss deep-tangent-points --hidden {a.hidden} --layers {a.layers} "
                               f"--steps {a.steps} at {a.n}^3: the analytic deep loss and its loss + gradient step at B uniform "
                               f"random space-time points (space in [-1, 1]^3, t in [0, 0.5], dc/dx of the grid) and the same two "
                               f"calls on the grid, timed in alternation (CUDA events, median of {a.steps}); B = {sizes[0]} and "
                               f"{sizes[1]}; the ratios are per point (B = n^3: the same point count as the grid)",
                       "gpu": name, "power_limit_w": plim, "clocks_max_sm_mhz": clk, "results": results}, fh, indent=1)


def distributed(a, g):
    import torch.distributed as dist
    rank, world, local = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"]), int(os.environ["LOCAL_RANK"])
    torch.cuda.set_device(local)
    dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    ctx = ops.Context(local)
    ctx.set_weights(MLPConfig(4, a.hidden, 4, True), *ops.mlp_random_init(a.hidden, 777, 0.25))
    pw = PhysWeights(1, 1)
    slab = ops.slab_for_rank(g.nz, rank, world)
    if a.loss == "tangent":
        buf = ctx.tangent_loss_grad_acc(g, pw, 0.25, slab)
    else:
        buf = ctx.fused_loss_grad_slab_acc(g, pw, 0.25, 2e-3, slab)

    def step():
        if a.loss == "tangent":
            ctx.tangent_loss_grad_acc(g, pw, 0.25, slab, buf)
        else:
            ctx.fused_loss_grad_slab_acc(g, pw, 0.25, 2e-3, slab, buf)
        dist.all_reduce(buf, op=dist.ReduceOp.SUM)

    for _ in range(5):
        step()
    torch.cuda.synchronize()
    dist.barrier()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(a.steps):
        step()
    e1.record()
    torch.cuda.synchronize()
    t = torch.tensor([e0.elapsed_time(e1) / a.steps], device="cuda")
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    if rank == 0:
        kind = "analytic loss+grad" if a.loss == "tangent" else "loss+grad"
        print(json.dumps({"workload": f"{a.n}^3 H={a.hidden} {kind}, z-slab per rank, 1 all-reduce of 9H+6 doubles",
                          "n_gpus": world, "ms_per_step_max_over_ranks": t.item(), "gpts_per_s": g.N / t.item() / 1e6,
                          "grad_norm": float(buf[2:].norm()), "acc": buf[:2].tolist()}))
    dist.destroy_process_group()


if __name__ == "__main__":
    main()
