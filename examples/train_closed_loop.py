"""Closed-loop training of the coordinate MLP against the physics loss (the reference's planned milestone M6,
REQUIREMENT.md:155-169), on 1..N GPUs:

  python examples/train_closed_loop.py [--loss fd|tangent] [--layers 1] [--data 0] [--colloc 0] [--t-range 0,0.5] [--n 128]
                                      [--hidden 64] [--steps 200]
  python -m torch.distributed.run --nproc-per-node N --master-addr 127.0.0.1 examples/train_closed_loop.py

Every rank differentiates its z-slab of the grid (physad_fused_loss_grad_slab_dev), one all-reduce of 9H+6 doubles
gives every rank the same losses and gradient, and every rank applies the same Adam update to its copy of the
580 (H=64) parameters -- no parameter broadcast is needed.  --loss tangent trains on the analytic loss instead
(derivatives propagated through the MLP, physad_tangent_loss_grad_dev): same slabs, same single all-reduce.  --layers L > 1
trains a deep network (4 -> H -> ... -> H -> 4, L hidden layers; hidden weights drawn uniform in +-0.2) on the
finite-difference loss through physad_deep_loss_grad_dev, or with --loss tangent on the analytic loss through
physad_deep_tangent_loss_grad_dev, again with one all-reduce of P+2 doubles.  --data N (with --layers L > 1) adds a data
term: a fixed "teacher" deep network (another seed) gives targets at N random points at t = 0, each rank fits its share of
the points (physad_deep_data_loss_grad_dev, mean squared error over all N points) and the student trains on
L_sigma + L_u + L_d.  --colloc N (with --layers L > 1) replaces the grid's physics term at t = 0.25 by the analytic loss at
N collocation points drawn fresh every step on the device, uniform in [-1, 1]^3 for space and in the time input of
--t-range T0,T1 (each rank draws its share from its own seeded generator; physad_deep_tangent_points_loss_grad_dev, mean
over all N points, the grid's dc/dx from physad_grid_input_scales, one all-reduce of P+2 doubles).  With --data it fits an
initial condition (the teacher at t = 0) and the dynamics that carry it over [T0, T1].  Prints one JSON line per 20 steps
and a summary."""
import argparse
import json
import os
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import torch

from phys_autodiff_b200 import Grid, MLPConfig, PhysWeights, ops


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--n", type=int, default=128)
    ap.add_argument("--hidden", type=int, default=64)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--lr", type=float, default=3e-3)
    ap.add_argument("--loss", choices=("fd", "tangent"), default="fd")
    ap.add_argument("--layers", type=int, default=1, help="hidden layers (> 1: a deep network)")
    ap.add_argument("--data", type=int, default=0, help="teacher points at t = 0 for a data term (needs --layers > 1)")
    ap.add_argument("--colloc", type=int, default=0,
                    help="collocation points per step for the physics term instead of the grid at t = 0.25 (needs --layers > 1)")
    ap.add_argument("--t-range", default="0,0.5", help="T0,T1: the time interval the collocation points cover")
    a = ap.parse_args()
    if a.data and a.layers < 2:
        ap.error("--data needs --layers > 1")
    if a.colloc and a.layers < 2:
        ap.error("--colloc needs --layers > 1")
    t0c, t1c = (float(v) for v in a.t_range.split(","))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank, local = int(os.environ.get("RANK", "0")), int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    H = a.hidden
    g = Grid(a.n, a.n, a.n, 1, 1, 1, 2e-3, True)
    cfg, pw = MLPConfig(4, H, 4, True), PhysWeights(1, 1)
    ctx = ops.Context(local)
    W1, b1, W2, b2 = ops.mlp_random_init(H, 777, 0.25)
    L = a.layers
    rng = np.random.default_rng(L)
    Wh = rng.uniform(-0.2, 0.2, (L - 1) * H * H).astype(np.float32)
    bh = rng.uniform(-0.2, 0.2, (L - 1) * H).astype(np.float32)
    parts = [W1, b1, W2, b2] if L == 1 else [W1, b1, Wh, bh, W2, b2]
    th = np.concatenate([np.asarray(x, np.float64) for x in parts])
    cuts = np.cumsum([x.size for x in parts])[:-1]
    if a.data:
        # teacher: the same construction from other seeds; this rank's share of the N points, inputs (x, y, z, t = 0)
        tW1, tb1, tW2, tb2 = ops.mlp_random_init(H, 4242, 0.25)
        trng = np.random.default_rng(4242 + L)
        tWh = trng.uniform(-0.2, 0.2, (L - 1) * H * H).astype(np.float32)
        tbh = trng.uniform(-0.2, 0.2, (L - 1) * H).astype(np.float32)
        pts = np.random.default_rng(99).uniform(-1, 1, (a.data, 4)).astype(np.float32)
        pts[:, 3] = 0.0   # network time input of t = 0 (MinusOneToOne: t itself)
        lo, hi = (rank * a.data) // world, ((rank + 1) * a.data) // world
        xd = torch.from_numpy(pts[lo:hi]).cuda()
        ctx.set_weights_deep(cfg, L, tW1, tb1, tWh, tbh, tW2, tb2)
        yd = ctx.mlp_forward_deep(xd).clone()
    if a.colloc:
        # this rank's share of the N points per step; MinusOneToOne: the network's time input is t itself
        lo_c, hi_c = (rank * a.colloc) // world, ((rank + 1) * a.colloc) // world
        gen = torch.Generator(device="cuda")
        gen.manual_seed(1000 + rank)
        lo4 = torch.tensor([-1.0, -1.0, -1.0, t0c], device="cuda")
        span4 = torch.tensor([2.0, 2.0, 2.0, t1c - t0c], device="cuda")
        dcdx = ops.grid_input_scales(g, cfg.minus_one_to_one)   # the grid's physical domain
    m, v = np.zeros_like(th), np.zeros_like(th)
    first = last = None
    t0 = time.perf_counter()
    for k in range(1, a.steps + 1):
        w = np.split(th.astype(np.float32), cuts)
        if a.colloc:
            ctx.set_weights_deep(cfg, L, *w)
            xc = lo4 + span4 * torch.rand((hi_c - lo_c, 4), generator=gen, device="cuda")
            ls, lu, grad = ctx.deep_tangent_points_loss_grad(xc, dcdx, pw, n_global=a.colloc)   # + all-reduce when world > 1
        elif L > 1 and a.loss == "tangent":
            ctx.set_weights_deep(cfg, L, *w)
            ls, lu, grad = ctx.deep_tangent_loss_grad(g, pw, 0.25)   # slab per rank + all-reduce when world > 1
        elif L > 1:
            ctx.set_weights_deep(cfg, L, *w)
            ls, lu, grad = ctx.deep_loss_grad(g, pw, 0.25, 2e-3)     # slab per rank + all-reduce when world > 1
        elif a.loss == "tangent":
            ctx.set_weights(cfg, *w)
            ls, lu, grad = ctx.tangent_loss_grad(g, pw, 0.25)      # slab per rank + all-reduce when world > 1
        else:
            ctx.set_weights(cfg, *w)
            ls, lu, grad = ctx.fused_loss_grad(g, pw, 0.25, 2e-3)
        ld = None
        if a.data:   # the network set above; all ranks' points, one all-reduce of P+1 doubles
            ld, gd = ctx.deep_data_loss_grad(xd, yd, n_global=a.data)
            grad = grad + gd
        last = float(ls) + float(lu) + (ld or 0.0)
        first = last if first is None else first
        m = 0.9 * m + 0.1 * grad
        v = 0.999 * v + 0.001 * grad * grad
        th = th - a.lr * (m / (1 - 0.9 ** k)) / (np.sqrt(v / (1 - 0.999 ** k)) + 1e-8)
        if rank == 0 and (k == 1 or k % 20 == 0):
            rec = {"step": k, "loss_sigma": float(ls), "loss_u": float(lu)}
            if ld is not None:
                rec["loss_data"] = ld
            print(json.dumps(rec), flush=True)
    dt = time.perf_counter() - t0
    if rank == 0:
        data = f" + data at {a.data} points" if a.data else ""
        summary = f"{a.n}^3 H={H} L={L} {a.loss} loss{data} on {world} GPU(s)"
        if a.colloc:
            what = " (initial condition + dynamics)" if a.data else ""
            summary = (f"H={H} L={L} analytic loss at {a.colloc} collocation points per step over t in [{t0c:g}, {t1c:g}] of the "
                       f"{a.n}^3 domain{data}{what} on {world} GPU(s)")
        print(json.dumps({"summary": summary, "steps": a.steps, "loss_first": first,
                          "loss_last": last, "reduction_pct": 100 * (1 - last / first),
                          "wall_ms_per_step_incl_host_adam": 1e3 * dt / a.steps}))
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
