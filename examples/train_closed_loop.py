"""Closed-loop training of the coordinate MLP against the physics loss (the reference's planned milestone M6,
REQUIREMENT.md:155-169), on 1..N GPUs:

  python examples/train_closed_loop.py [--loss fd|tangent] [--layers 1] [--data 0] [--colloc 0] [--periodic 0]
                                      [--neumann 0] [--t-range 0,0.5] [--n 128] [--hidden 64] [--steps 200]
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
initial condition (the teacher at t = 0) and the dynamics that carry it over [T0, T1].  --periodic N (with --colloc) adds
the periodic boundary condition of the grid's domain, which the analytic loss has no stencil to impose: N pairs drawn fresh
every step on the device, a third per space axis a, p on the face p_a = -1 (the other two space inputs uniform in [-1, 1],
the time input in [T0, T1]) and q = p + T_a e_a one period on (ops.grid_periods), fitted with the pair loss
(physad_deep_pair_loss_grad_dev, lam = 1/4 each, mean over all N pairs, one all-reduce of P+1 doubles).  --neumann M (with
--colloc, not with --periodic) makes the domain clamped instead: the grid is non-periodic, and the condition its clamped
stencil states, a zero normal derivative at the faces, is fitted at M face points drawn fresh every step on the device, a
third per space axis a alternating the faces c_a = -1 and +1 (the other space inputs uniform in [-1, 1], the time input in
[T0, T1]), with the derivative-fit loss (physad_deep_deriv_loss_grad_dev, direction dc_a/dx_a e_a, target 0, lam = 1/4
each, mean over all M points, one all-reduce of P+1 doubles).  The summary then reports the final mean squared normal
derivative at 4 096 fixed held-out face points (physad_mlp_jacobian_deep_dev).  --torch (with --layers > 1 and --colloc)
trains the same objective through phys_autodiff_b200.autograd.DeepMLP and torch.optim.Adam instead: the residuals, the
data, pair and Neumann terms are written in PyTorch from the module's (y, J) (the library's forward and Jacobian), and
.backward() runs the library's vector-Jacobian products; with several ranks every rank back-propagates its share and the
parameters' .grad are all-reduced.  The same points are drawn in the same order, so step 1's losses are the fused run's.
--grad-out FILE writes step 1's gradient (float64, the flat layout of the deep gradients) in either mode.  Prints one JSON
line per 20 steps and a summary."""
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
    ap.add_argument("--periodic", type=int, default=0,
                    help="pairs per step for the periodic boundary condition of the grid's domain (needs --colloc)")
    ap.add_argument("--neumann", type=int, default=0,
                    help="face points per step for a zero normal derivative on a clamped domain (needs --colloc)")
    ap.add_argument("--t-range", default="0,0.5", help="T0,T1: the time interval the collocation points cover")
    ap.add_argument("--torch", action="store_true",
                    help="losses written in PyTorch on DeepMLP, torch.optim.Adam (needs --layers > 1 and --colloc)")
    ap.add_argument("--grad-out", default=None, help="write step 1's gradient (float64) to this file")
    a = ap.parse_args()
    if a.torch and (a.layers < 2 or not a.colloc):
        ap.error("--torch needs --layers > 1 and --colloc: the one-hidden-layer and grid (finite-difference) objectives "
                 "have no PyTorch form here")
    if a.data and a.layers < 2:
        ap.error("--data needs --layers > 1")
    if a.colloc and a.layers < 2:
        ap.error("--colloc needs --layers > 1")
    if a.periodic and not a.colloc:
        ap.error("--periodic needs --colloc")
    if a.neumann and not a.colloc:
        ap.error("--neumann needs --colloc")
    if a.neumann and a.periodic:
        ap.error("--neumann and --periodic exclude each other: a domain is either periodic or clamped")
    t0c, t1c = (float(v) for v in a.t_range.split(","))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank, local = int(os.environ.get("RANK", "0")), int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    H = a.hidden
    g = Grid(a.n, a.n, a.n, 1, 1, 1, 2e-3, not a.neumann)
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
    if a.periodic:
        # this rank's share of the N pairs per step; pair i lies across the faces of space axis i % 3
        lo_p, hi_p = (rank * a.periodic) // world, ((rank + 1) * a.periodic) // world
        pgen = torch.Generator(device="cuda")
        pgen.manual_seed(2000 + rank)
        period = torch.from_numpy(ops.grid_periods(g, cfg.minus_one_to_one)).cuda()
        rows = torch.arange(hi_p - lo_p, device="cuda")
        axis = (rows + lo_p) % 3
    if a.neumann:
        # this rank's share of the M face points per step: point i on face c_a = -1 or +1 (alternating) of axis a = i % 3,
        # direction dc_a/dx_a e_a (the physical normal derivative), target 0
        lo_n, hi_n = (rank * a.neumann) // world, ((rank + 1) * a.neumann) // world
        ngen = torch.Generator(device="cuda")
        ngen.manual_seed(3000 + rank)
        idx = torch.arange(lo_n, hi_n, device="cuda")
        nrows, naxis = idx - lo_n, idx % 3
        nface = torch.where((idx // 3) % 2 == 0, -1.0, 1.0).to(torch.float32)
        ndir = torch.zeros((hi_n - lo_n, 4), device="cuda")
        ndir[nrows, naxis] = torch.from_numpy(dcdx).cuda()[naxis]
        nzero = torch.zeros_like(ndir)
    if a.torch:
        first, last, dt, th = _train_torch(a, ctx, cfg, pw, L, th, cuts, world, locals())
    else:
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
            lp = None
            if a.periodic:   # the network set above
                p = lo4 + span4 * torch.rand((hi_p - lo_p, 4), generator=pgen, device="cuda")
                p[rows, axis] = -1.0
                q = p.clone()
                q[rows, axis] += period[axis]
                lp, gp = ctx.deep_pair_loss_grad(torch.stack([p, q], 1), n_global=a.periodic)
                grad = grad + gp
            ln = None
            if a.neumann:   # the network set above
                xn = lo4 + span4 * torch.rand((hi_n - lo_n, 4), generator=ngen, device="cuda")
                xn[nrows, naxis] = nface
                ln, gn = ctx.deep_deriv_loss_grad(xn, ndir, nzero, n_global=a.neumann)
                grad = grad + gn
            ld = None
            if a.data:   # the network set above; all ranks' points, one all-reduce of P+1 doubles
                ld, gd = ctx.deep_data_loss_grad(xd, yd, n_global=a.data)
                grad = grad + gd
            last = float(ls) + float(lu) + (ld or 0.0) + (lp or 0.0) + (ln or 0.0)
            first = last if first is None else first
            if k == 1 and a.grad_out and rank == 0:
                np.asarray(grad, np.float64).tofile(a.grad_out)
            m = 0.9 * m + 0.1 * grad
            v = 0.999 * v + 0.001 * grad * grad
            th = th - a.lr * (m / (1 - 0.9 ** k)) / (np.sqrt(v / (1 - 0.999 ** k)) + 1e-8)
            if rank == 0 and (k == 1 or k % 20 == 0):
                rec = {"step": k, "loss_sigma": float(ls), "loss_u": float(lu)}
                if ld is not None:
                    rec["loss_data"] = ld
                if lp is not None:
                    rec["loss_periodic"] = lp
                if ln is not None:
                    rec["loss_neumann"] = ln
                print(json.dumps(rec), flush=True)
        dt = time.perf_counter() - t0
    held_dn2 = None
    if a.neumann and rank == 0:
        # the final network's mean squared normal derivative (over points and outputs) at 4 096 fixed face points
        hrng = np.random.default_rng(5)
        hx = hrng.uniform(-1, 1, (4096, 4)).astype(np.float32)
        hx[:, 3] = hrng.uniform(t0c, t1c, 4096).astype(np.float32)
        hax = np.arange(4096) % 3
        hx[np.arange(4096), hax] = np.where((np.arange(4096) // 3) % 2 == 0, -1.0, 1.0)
        ctx.set_weights_deep(cfg, L, *np.split(th.astype(np.float32), cuts))
        _, J = ctx.mlp_jacobian_deep(torch.from_numpy(hx).cuda())
        dn = J.cpu().numpy().astype(np.float64)[np.arange(4096), :, hax] * dcdx.astype(np.float64)[hax][:, None]
        held_dn2 = float(np.mean(dn * dn))
    if rank == 0:
        data = f" + data at {a.data} points" if a.data else ""
        summary = f"{a.n}^3 H={H} L={L} {a.loss} loss{data} on {world} GPU(s)"
        via = " (losses in PyTorch through DeepMLP, torch.optim.Adam)" if a.torch else ""
        if a.colloc:
            what = " (initial condition + dynamics)" if a.data else ""
            what += f" + periodic boundaries at {a.periodic} pairs per step" if a.periodic else ""
            what += f" + Neumann boundaries at {a.neumann} face points per step" if a.neumann else ""
            summary = (f"H={H} L={L} analytic loss at {a.colloc} collocation points per step over t in [{t0c:g}, {t1c:g}] of the "
                       f"{a.n}^3 domain{data}{what} on {world} GPU(s){via}")
        out = {"summary": summary, "steps": a.steps, "loss_first": first, "loss_last": last,
               "reduction_pct": 100 * (1 - last / first), "wall_ms_per_step_incl_host_adam": 1e3 * dt / a.steps}
        if held_dn2 is not None:
            out["heldout_mean_sq_normal_derivative"] = held_dn2
        print(json.dumps(out))
    if world > 1:
        dist.destroy_process_group()


def torch_objective(model, dcdx, pw, xc, n_colloc, xd=None, yd=None, n_data=1, pq=None, n_pairs=1, xn=None, ndir=None,
                    n_neumann=1):
    """The fused calls' objective written in PyTorch on DeepMLP's (y, J): the analytic residuals of k_tangent_loss at the
    collocation points xc (w / n_colloc) sum R^2), and the data, pair and Neumann terms with lam = 1/4 each.  Each term is
    this rank's share of a mean over all ranks' points.  -> (total, {name: term})."""
    y, J = model(xc, jacobian=True)
    s = torch.as_tensor(np.asarray(dcdx, np.float32), device=xc.device)
    gr = J[:, :, :3] * s                                   # d y_o / d x_j
    div = (gr[:, 1, 0] + gr[:, 2, 1]) + gr[:, 3, 2]
    R = J[:, :, 3] + ((y[:, 1:2] * gr[:, :, 0] + y[:, 2:3] * gr[:, :, 1]) + y[:, 3:4] * gr[:, :, 2])
    Rs = R[:, 0] + y[:, 0] * div
    terms = {"loss_sigma": pw.w_sigma * (Rs * Rs).sum() / n_colloc,
             "loss_u": pw.w_u * (R[:, 1:] * R[:, 1:]).sum() / n_colloc}
    if xd is not None:
        terms["loss_data"] = 0.25 * ((model(xd) - yd) ** 2).sum() / n_data
    if pq is not None:
        ypq = model(pq.reshape(-1, 4)).reshape(-1, 2, 4)
        terms["loss_periodic"] = 0.25 * ((ypq[:, 0] - ypq[:, 1]) ** 2).sum() / n_pairs
    if xn is not None:
        _, Jn = model(xn, jacobian=True)
        D = (Jn * ndir[:, None, :]).sum(-1)
        terms["loss_neumann"] = 0.25 * (D * D).sum() / n_neumann
    return sum(terms.values()), terms


def _train_torch(a, ctx, cfg, pw, L, th, cuts, world, env):
    """--torch: the loop of main() with DeepMLP and torch.optim.Adam; the same point draws in the same order."""
    from phys_autodiff_b200.autograd import DeepMLP
    rank = int(os.environ.get("RANK", "0"))
    model = DeepMLP(ctx, cfg.H, L, np.split(th.astype(np.float32), cuts), cfg.minus_one_to_one)
    opt = torch.optim.Adam(model.parameters(), lr=a.lr, betas=(0.9, 0.999), eps=1e-8)
    first = last = None
    t0 = time.perf_counter()
    for k in range(1, a.steps + 1):
        xc = env["lo4"] + env["span4"] * torch.rand((env["hi_c"] - env["lo_c"], 4), generator=env["gen"], device="cuda")
        pq = xn = None
        if a.periodic:
            p = env["lo4"] + env["span4"] * torch.rand((env["hi_p"] - env["lo_p"], 4), generator=env["pgen"], device="cuda")
            p[env["rows"], env["axis"]] = -1.0
            q = p.clone()
            q[env["rows"], env["axis"]] += env["period"][env["axis"]]
            pq = torch.stack([p, q], 1)
        if a.neumann:
            xn = env["lo4"] + env["span4"] * torch.rand((env["hi_n"] - env["lo_n"], 4), generator=env["ngen"], device="cuda")
            xn[env["nrows"], env["naxis"]] = env["nface"]
        opt.zero_grad(set_to_none=True)
        total, terms = torch_objective(model, env["dcdx"], pw, xc, a.colloc, env.get("xd"), env.get("yd"), a.data or 1, pq,
                                       a.periodic or 1, xn, env.get("ndir"), a.neumann or 1)
        total.backward()
        vals = torch.stack([t.detach().double() for t in terms.values()])
        if world > 1:
            import torch.distributed as dist
            dist.all_reduce(vals)
            for p_ in model.parameters():
                dist.all_reduce(p_.grad)
        vals = dict(zip(terms, vals.tolist()))
        last = sum(vals.values())
        first = last if first is None else first
        if k == 1 and a.grad_out and rank == 0:
            np.concatenate([p_.grad.detach().double().cpu().numpy().ravel() for p_ in model._params()]).tofile(a.grad_out)
        opt.step()
        if rank == 0 and (k == 1 or k % 20 == 0):
            print(json.dumps({"step": k, **vals}), flush=True)
    torch.cuda.synchronize()
    dt = time.perf_counter() - t0
    return first, last, dt, model.flat_parameters().astype(np.float64)


if __name__ == "__main__":
    main()
