#!/usr/bin/env python
"""Headline benchmark: grid points/sec of the fused MLP + finite-difference physics loss at 256^3.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--hidden H] [--grid n] [--impl reference] [--dump-outputs DIR]

One "step" = one pass of the hot path over the whole synthetic grid: three MLP evaluations per
point (t-dt, t, t+dt), the PDE residuals and the reduction to {L_sigma, L_u}.  Synthetic inputs as
the reference's test/test_mlp_phys_perf.cpp:21-23: GridSpec{n,n,n, h=1, dt=2e-3, periodic},
MinusOneToOne coordinates, mlp_random_init(seed 777, scale 0.25), t = 0.25, weights (1,1).
There are no input arrays: coordinates derive from the point index and the weights (2.3 KB at H=64)
ride in the kernel-parameter constant bank, so nothing needs to be (or can be) warm in L2; the L2
is flushed between timed steps anyway.  With N > 1 the grid is sharded into z-slabs (one per rank,
halo planes recomputed) and one NCCL all-reduce of two doubles combines the partial sums: total
work is fixed, i.e. strong scaling.  Prints ONE JSON line on rank 0.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

METRIC = "grid points/sec, fused MLP + finite-difference physics loss"
UNIT = "points/s"
T0, DT, SEED, SCALE = 0.25, 2e-3, 777, 0.25


def bf16_peak():
    """Dense bf16 TFLOP/s of this pool's B200s (driver-written MEASURED_PEAKS.json, burst figure); nominal 2250 otherwise."""
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as fh:
            return float(json.load(fh)["bf16_tflops"])
    except Exception:
        return 2250.0


def flops_per_point(H: int) -> int:
    """Algorithmic work, SURVEY.md section 8(d): 3 slices x 2*(4H + 4H) MLP flops + 3H ReLU + 60 stencil + 8 reduction."""
    return 51 * H + 68


def ncu_dram_traffic():
    """dram__bytes_read.sum + dram__bytes_write.sum per launch of the fused kernel from the committed
    `ncu --set full` capture of this same command (profiles/), or None."""
    try:
        with open(os.path.join(ROOT, "profiles", "r02_ncu_fused_default_summary.json")) as fh:
            d = json.load(fh)[0]
        unit = {"byte": 1.0, "Kbyte": 1e3, "Mbyte": 1e6, "Gbyte": 1e9}
        rd, wr = d["dram__bytes_read.sum"], d["dram__bytes_write.sum"]
        return float(rd[0]) * unit[rd[1]] + float(wr[0]) * unit[wr[1]]
    except Exception:
        return None


def golden_losses(H: int, n: int):
    """Losses the UNMODIFIED reference CPU path gives for this benchmark's inputs on the WHOLE n^3 grid
    (tests/golden/golden.json, written by tests/golden/make_golden.py in the dev container), or None."""
    try:
        with open(os.path.join(ROOT, "tests", "golden", "golden.json")) as fh:
            a = json.load(fh)["anchors"].get(f"{n}c_h{H}")
        return (float(a["loss_sigma"]), float(a["loss_u"])) if a else None
    except Exception:
        return None


def parity_block(H: int, n: int, ls: float, lu: float):
    """The timed path's result against the reference's, at the north-star tolerance for the reduced loss."""
    ref = golden_losses(H, n)
    if ref is None:
        return None
    es, eu = abs(ls - ref[0]) / abs(ref[0]), abs(lu - ref[1]) / abs(ref[1])
    return {"ref_sigma": ref[0], "ref_u": ref[1], "rel_err_sigma": es, "rel_err_u": eu, "tolerance": 1e-4,
            "ok": bool(es <= 1e-4 and eu <= 1e-4),
            "source": f"tests/golden/golden.json anchors[{n}c_h{H}]: unmodified reference CPU path on the whole grid"}


def executed_flops_per_point(H: int) -> float:
    """fp32 lane-operations the default kernel actually executes per point (DESIGN.md section 4.1): the three
    time slices share the layer-1 prefix and 4 columns share b1 + W1[h,0]x, so layer 1 costs 6.75 instead of 24
    ops per hidden unit; layer 2 keeps its 24; + ring (192 of 2048 columns re-evaluated at time t, 15 ops per
    hidden unit), + z-halo planes (~2 per 55), + ~55 for stencil and reduction."""
    return 30.75 * H + (192.0 / 2048.0) * 15.0 * H + (2.0 / 55.0) * 12.75 * H + 55.0


def strict_fp32_peak():
    """Measured FMUL+FADD (non-contracted) pipe peak of this pool's B200, TFLOP/s, and where it came from."""
    p = os.path.join(ROOT, "profiles", "r01_microbench_fp32_long.json")
    try:
        with open(p) as fh:
            d = json.load(fh)
        return float(d["strict"]["tflops"]), float(d["ffma"]["tflops"]), "measured: tools/microbench_fp32.cu -> " + os.path.relpath(p, ROOT)
    except Exception:
        return 37.2, 74.4, "fallback: 148 SM x 128 lanes x 1.965 GHz (SURVEY.md section 8d)"


class ClockSampler:
    """SM clock / power / throttle reasons sampled DURING the timed region (B200_PROFILING.md's clocks
    line), through NVML in-process every ~3 ms (spawning nvidia-smi is slower than the timed region)."""

    def __init__(self, index: int):
        self.index, self.rows, self.stop_flag, self.th, self.err = index, [], False, None, None

    def start(self):
        try:
            import pynvml as nv
            nv.nvmlInit()
            self.nv = nv
            # NVML enumerates physical devices; honour CUDA_VISIBLE_DEVICES when it is a list of indices
            vis = os.environ.get("CUDA_VISIBLE_DEVICES")
            idx = self.index
            if vis:
                try:
                    idx = int(vis.split(",")[self.index])
                except Exception:
                    pass
            self.h = nv.nvmlDeviceGetHandleByIndex(idx)
            self.max_sm = nv.nvmlDeviceGetMaxClockInfo(self.h, nv.NVML_CLOCK_SM)
        except Exception as e:  # pragma: no cover
            self.err = repr(e)
            return
        self.th = threading.Thread(target=self._loop, daemon=True)
        self.th.start()

    def _loop(self):
        nv = self.nv
        while not self.stop_flag:
            try:
                sm = nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM)
                pw = nv.nvmlDeviceGetPowerUsage(self.h) / 1000.0
                try:
                    rs = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
                except Exception:
                    rs = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                self.rows.append((time.perf_counter(), sm, pw, rs))
            except Exception as e:  # pragma: no cover
                self.err = repr(e)
                break
            time.sleep(0.003)

    def mark(self):
        """Start of the timed region: only samples from here on are reported (the thread itself is
        started before warm-up so NVML's first-call latencies never land inside a timed step)."""
        self.t_mark = time.perf_counter()

    def stop(self):
        if self.th is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvml unavailable: " + str(self.err)]}
        self.stop_flag = True
        self.th.join(timeout=2)
        t_mark = getattr(self, "t_mark", 0.0)
        self.rows = [r[1:] for r in self.rows if r[0] >= t_mark]
        nv = self.nv
        names = {"hw_slowdown": getattr(nv, "nvmlClocksThrottleReasonHwSlowdown", 0x8),
                 "hw_thermal_slowdown": getattr(nv, "nvmlClocksThrottleReasonHwThermalSlowdown", 0x40),
                 "sw_thermal_slowdown": getattr(nv, "nvmlClocksThrottleReasonSwThermalSlowdown", 0x20),
                 "sw_power_cap": getattr(nv, "nvmlClocksThrottleReasonSwPowerCap", 0x4)}
        sm = [r[0] for r in self.rows]
        pw = [r[1] for r in self.rows]
        reasons = sorted(n for n, bit in names.items() if any(r[2] & bit for r in self.rows))
        busy = [s for s, p in zip(sm, pw) if p >= 0.6 * max(pw)] if pw else []
        return {"sm_mhz": statistics.median(busy) if busy else None, "sm_max_mhz": float(self.max_sm),
                "power_w_max": max(pw) if pw else None, "samples": len(sm), "samples_under_load": len(busy),
                "window": "warm-up + timed steps", "reasons": reasons}


def cpu_reference_rate(H: int, nxy: int, planes: int, threads: int):
    """Reference CPU path (oracle/_ref: the unmodified reference sources; else the pinned C port) on an
    nxy x nxy x planes grid with the benchmark's weights/t/dt.  Returns (points/s, kind, cores, losses)."""
    import oracle
    from oracle import Grid
    R = oracle.reference()
    g = Grid(nxy, nxy, planes, 1.0, 1.0, 1.0, DT, True)
    if R is not None:
        w = R.mlp_random_init(H, SEED, SCALE)
        t0 = time.perf_counter()
        r = R.fused_loss(g, w, T0, DT, threads=threads)
        dt = time.perf_counter() - t0
        return g.N / dt, "reference", threads, (float(r["loss_sigma"]), float(r["loss_u"]))
    P = oracle.port()
    w = P.mlp_random_init(H, SEED, SCALE)
    t0 = time.perf_counter()
    r = P.fused_loss(g, w, T0, DT)
    dt = time.perf_counter() - t0
    return g.N / dt, "port", 1, (float(r["loss_sigma"]), float(r["loss_u"]))


def dump_outputs(out_dir: str, **arrays) -> None:
    """--dump-outputs: what the timed path returned in its last step, one <out_dir>/<name>.npy per array, so that
    two builds run with the same arguments (same seeded inputs) can be compared output for output."""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        a = np.asarray(a)
        assert a.dtype in (np.float32, np.float64), (name, a.dtype)
        np.save(os.path.join(out_dir, name + ".npy"), a)


def host_threads() -> int:
    try:
        return len(os.sched_getaffinity(0))
    except Exception:
        return os.cpu_count() or 1


def workload_name(H: int, n: int) -> str:
    return (f"fused MLP(4-{H}-4)+phys loss, {n}^3 grid, seed {SEED}, scale {SCALE}, t {T0}, dt {DT}, "
            f"h 1, periodic, MinusOneToOne (test_mlp_phys_perf.cpp:21-23 at 256^3)")


def run_reference_arm(args, rank: int, world: int):
    """--impl reference: the reference's own CPU implementation of the path on the host cores (the reference is
    single-threaded; its pointwise MLP is driven on all host threads, bit-identical results).  The FIRST timed step
    runs the WHOLE grid of the workload; the remaining steps a bounded z-sample of it (--ref-planes), so that the
    default run stays within minutes.  value = points processed / time over all timed steps."""
    if rank != 0:
        return
    H, n = args.hidden, args.grid
    threads = host_threads()
    planes = max(3, min(n, args.ref_planes))
    for _ in range(min(args.warmup, 1)):
        cpu_reference_rate(H, n, planes, threads)
    times, pts, kind, cores, whole_losses = [], 0, "port", 1, None
    for i in range(args.steps):
        p = n if i == 0 else planes
        t0 = time.perf_counter()
        rate, kind, cores, losses = cpu_reference_rate(H, n, p, threads)
        times.append(time.perf_counter() - t0)
        pts += n * n * p
        if i == 0:
            whole_losses = losses
    total = sum(times)
    value = pts / total
    sample = (f"step 1: the whole {n}^3 grid ({times[0]:.2f} s); steps 2..{args.steps}: {n}x{n}x{planes} planes of it "
              f"(same weights, t, dt, periodic); {cores} host threads")
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": 1e3 * total / len(times), "higher_is_better": True, "scaling": "strong",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": workload_name(H, n), "hidden": H, "grid": [n, n, n]},
        "loss": {"sigma": whole_losses[0], "u": whole_losses[1]},
        "parity": parity_block(H, n, whole_losses[0], whole_losses[1]),
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": kind, "sample": sample},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    if args.dump_outputs:
        import numpy as np
        dump_outputs(args.dump_outputs, loss=np.array(losses, np.float32))
    print(json.dumps(line), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--hidden", type=int, default=64)
    ap.add_argument("--grid", type=int, default=256)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--variant", type=int, default=-1, help="fused-kernel launch variant (tuning)")
    ap.add_argument("--ref-planes", type=int, default=32, help="z planes per step of the reference arm")
    ap.add_argument("--collective", default="p2p", choices=["p2p", "nccl"],
                    help="N>1: in-kernel peer-memory all-reduce (default) or kernel + NCCL all-reduce")
    ap.add_argument("--emulate-rank-of", type=int, default=0,
                    help="tuning aid: time only the kernel for rank 0's slab of an N-rank run on ONE GPU and exit")
    ap.add_argument("--emulate-planes", type=int, default=0, help="with --emulate-rank-of: slab = first P planes")
    ap.add_argument("--exact-residuals", action="store_true",
                    help="stencil/residual arithmetic in double exactly as the CPU reference (bit-identical residuals) "
                         "instead of the default fp32-with-FMA mode")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-clocks", action="store_true", help="skip the NVML clock sampler thread (diagnostics)")
    ap.add_argument("--no-extra", action="store_true", help="skip the H=32 / H=128 width sweep reported under 'extra' (N=1 only)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the timed path returned in its last step to DIR/<name>.npy: "
                         "sums (float64 [sum R_sigma^2, sum |R_u|^2] over the whole grid) and loss (float32 [L_sigma, L_u]); "
                         "the reference arm writes loss")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.emulate_rank_of > 1:
        ap.error("--dump-outputs does not apply to --emulate-rank-of (that mode times one slab only)")

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference_arm(args, rank, world)
        return

    import numpy as np
    import torch
    import torch.distributed as dist
    from phys_autodiff_b200 import Grid, MLPConfig, PhysWeights, ops
    from phys_autodiff_b200.ops import slab_for_rank

    assert torch.cuda.is_available(), "bench.py needs a B200; there is no CPU fallback"
    torch.cuda.set_device(local)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    assert world == args.gpus, f"--gpus {args.gpus} but WORLD_SIZE={world}: launch with torch.distributed.run"

    H, n = args.hidden, args.grid
    g = Grid(n, n, n, 1.0, 1.0, 1.0, DT, True)
    cfg = MLPConfig(4, H, 4, True)
    pw = PhysWeights(1.0, 1.0)
    w = ops.mlp_random_init(H, SEED, SCALE)
    ctx = ops.Context(local)
    if args.variant >= 0:
        ctx.set_fused_variant(args.variant)
    if args.exact_residuals:
        ctx.set_exact_residuals(True)
    ctx.set_weights(cfg, *w)
    slab = slab_for_rank(n, rank, world)
    acc = torch.zeros(2, dtype=torch.float64, device="cuda")
    if args.emulate_rank_of > 1:
        slab = slab_for_rank(n, 0, args.emulate_rank_of)
        if args.emulate_planes > 0:
            slab = (0, args.emulate_planes)
        launch_e = ctx.prepare_fused(g, T0, DT, slab=slab, acc=acc)
        for _ in range(5):
            launch_e()
        torch.cuda.synchronize()
        evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
        for e0, e1 in evs:       # enqueue everything, sync once: launch latency stays hidden as in the timed loop
            e0.record(); launch_e(); e1.record()
        torch.cuda.synchronize()
        ts = [e0.elapsed_time(e1) for e0, e1 in evs]
        print(json.dumps({"emulate_rank_of": args.emulate_rank_of, "slab": slab, "variant": args.variant,
                          "kernel_ms_mean": statistics.mean(ts), "kernel_ms_min": min(ts),
                          "ideal_ms_if_perfect_scaling": None}))
        return
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")  # > 126 MB L2

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize()

    # multi-GPU: the two partial sums are all-reduced inside the kernel over NVLink peer memory unless
    # --collective nccl asks for the plain kernel + one NCCL all-reduce of 2 doubles
    p2p = world > 1 and args.collective == "p2p" and ctx.connect_peers()   # False on every rank if CUDA IPC is unavailable
    if world > 1 and args.collective == "p2p" and not p2p and rank == 0:
        print("bench: peer-memory exchange unavailable; using the NCCL all-reduce", file=sys.stderr)
    launch = ctx.prepare_fused(g, T0, DT, slab=slab, acc=acc, allreduce=bool(p2p))   # pre-marshalled C-ABI call

    def step():
        launch()
        if world > 1 and not p2p:
            dist.all_reduce(acc, op=dist.ReduceOp.SUM)

    def timed(K, W, sampler=None):
        if sampler:  # sampling window = warm-up + timed steps (same kernel, same load); NVML's slow first
            sampler.start()   # calls happen before any timed step
            t_wait = time.perf_counter()
            while not sampler.rows and sampler.th is not None and time.perf_counter() - t_wait < 0.5:
                time.sleep(0.001)
            sampler.mark()
        for _ in range(W):
            step()
        barrier()
        ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(K)]
        l0 = ctx.launch_count
        wall0 = time.perf_counter()
        for e0, e1 in ev:
            flush.zero_()          # L2 flush between timed steps (outside the per-step events)
            e0.record()
            step()
            e1.record()
        barrier()
        wall = time.perf_counter() - wall0
        clocks = sampler.stop() if sampler else None
        per = [e0.elapsed_time(e1) for e0, e1 in ev]
        tot = torch.tensor([sum(per)], dtype=torch.float64, device="cuda")
        if world > 1:
            dist.all_reduce(tot, op=dist.ReduceOp.MAX)
            allper = [None] * world
            dist.all_gather_object(allper, per)
            timed.per_rank = [{"sum_ms": sum(p), "median": statistics.median(p), "max": max(p),
                               "n_over_1.2x_median": sum(1 for v in p if v > 1.2 * statistics.median(p))} for p in allper]
        return tot.item(), per, ctx.launch_count - l0, clocks, wall

    sampler = ClockSampler(local) if (rank == 0 and not args.no_clocks) else None
    total_ms, per, launches, clocks, wall = timed(args.steps, max(3, args.warmup), sampler)
    value = g.N * args.steps / (total_ms * 1e-3)
    sums = acc.cpu().numpy()     # every launch overwrites acc: these are the last timed step's global sums
    ls, lu = ctx.finalize(sums, pw, g.N)
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, sums=sums, loss=np.array([ls, lu], np.float32))

    # kernel-only duration on this rank (no all-reduce inside the events) for the roofline
    def kernel_only(K):
        for _ in range(3):
            ctx.fused_loss_acc(g, T0, DT, slab=slab, acc=acc)
        torch.cuda.synchronize()
        ts = []
        for _ in range(K):
            flush.zero_()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(); ctx.fused_loss_acc(g, T0, DT, slab=slab, acc=acc); e1.record()
            e1.synchronize()
            ts.append(e0.elapsed_time(e1))
        return statistics.mean(ts), min(ts)
    k_mean, k_min = kernel_only(min(args.steps, 20))
    slab_pts = (slab[1] - slab[0]) * n * n
    peak_strict, peak_ffma, peak_src = strict_fp32_peak()
    achieved = flops_per_point(H) * slab_pts / (k_mean * 1e-3) / 1e12

    # end to end through the host-buffer C-ABI call (physad_fused_loss_slab_host): weights from host memory ->
    # kernel (+ in-kernel all-reduce) -> 16-byte result back through pinned memory -> host finalisation,
    # one call per step.  With the NCCL collective the Python-level path (set_weights + fused_loss) is timed.
    def e2e(K):
        if world == 1 or p2p:
            host_step = ctx.prepare_step_host(g, cfg, *w, pw, T0, DT, slab=slab)
        else:
            def host_step():
                ctx.set_weights(cfg, *w)
                return ctx.fused_loss(g, pw, T0, DT)
        for _ in range(3):
            host_step()
        barrier()
        t0 = time.perf_counter()
        for _ in range(K):
            out = host_step()
        barrier()
        t = torch.tensor([time.perf_counter() - t0], dtype=torch.float64, device="cuda")
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return g.N * K / t.item(), out
    e2e_value, e2e_out = e2e(args.steps)
    h2d = sum(int(a.nbytes) for a in w)

    extra = {}
    if not args.no_extra and world == 1 and args.hidden == 64:
        for H2 in (32, 128):
            w2 = ops.mlp_random_init(H2, SEED, SCALE)
            ctx.set_weights(MLPConfig(4, H2, 4, True), *w2)
            t_ms, _, _, _, _ = timed(10, 3)
            l2s, l2u = ctx.finalize(acc.cpu().numpy(), pw, g.N)
            extra[f"H{H2}"] = {"value": g.N * 10 / (t_ms * 1e-3), "unit": UNIT, "ms_per_step": t_ms / 10,
                               "roofline_frac": flops_per_point(H2) * g.N * 10 / (t_ms * 1e-3) / 1e12 / peak_strict,
                               "loss": {"sigma": float(l2s), "u": float(l2u)}, "parity": parity_block(H2, n, float(l2s), float(l2u))}
        ctx.set_weights(cfg, *w)
        # BASELINE config 5, depth: 4 -> H -> ... -> H -> 4 with L hidden layers (additive API, parity unpinned for L > 1:
        # bit-exact against the CPU restatement in the tests), stage-wise: three slices -> six fields (k_mlp_deep), then
        # the physics loss on them.  frac = algorithmic strict-fp32 flops of the MLP / the measured FMUL+FADD peak.
        rng = np.random.default_rng(0)
        sweep = []
        for H2 in (32, 64, 128):
            wd = ops.mlp_random_init(H2, SEED, SCALE)
            for L in (2, 3, 5):
                Wh = rng.uniform(-0.2, 0.2, (L - 1) * H2 * H2).astype(np.float32)
                bh = rng.uniform(-0.2, 0.2, (L - 1) * H2).astype(np.float32)
                ctx.set_weights_deep(MLPConfig(4, H2, 4, True), L, wd[0], wd[1], Wh, bh, wd[2], wd[3])
                fields = ctx.mlp_generate_fields_deep(g, T0, DT)
                ts_f, ts_p = [], []
                for it in range(3):
                    flush.zero_()
                    e0, e1, e2 = (torch.cuda.Event(enable_timing=True) for _ in range(3))
                    e0.record(); ctx.mlp_generate_fields_deep(g, T0, DT); e1.record(); dacc = ctx.phys_loss_acc(g, fields); e2.record()
                    e2.synchronize()
                    if it:
                        ts_f.append(e0.elapsed_time(e1)); ts_p.append(e1.elapsed_time(e2))
                fl = 3 * (2 * 4 * H2 + (L - 1) * 2 * H2 * H2 + 2 * 4 * H2) + 3 * L * H2
                ms_f, ms_p = statistics.mean(ts_f), statistics.mean(ts_p)
                row = {"H": H2, "hidden_layers": L, "ms_fields": ms_f, "ms_phys_loss": ms_p,
                       "value": g.N / ((ms_f + ms_p) * 1e-3), "unit": UNIT, "mlp_flops_per_point": fl,
                       "mlp_tflops": fl * g.N / (ms_f * 1e-3) / 1e12, "frac_of_strict_fp32_peak": fl * g.N / (ms_f * 1e-3) / 1e12 / peak_strict}
                # the same network with its hidden -> hidden layers on the tensor cores (tcgen05, three-term bf16 operands, six
                # term products per layer; additive and NOT bit-exact): time, the deviation from the strict fields, and the
                # tensor-pipe rate of the 6 x 2 H^2 bf16 flops it issues per row and layer against the measured bf16 peak
                ctx.set_deep_mode(1)
                try:
                    ffast = ctx.mlp_generate_fields_deep(g, T0, DT)
                    tf = []
                    for it in range(3):
                        flush.zero_()
                        e0, e1 = (torch.cuda.Event(enable_timing=True) for _ in range(2))
                        e0.record(); ctx.mlp_generate_fields_deep(g, T0, DT); e1.record(); e1.synchronize()
                        if it:
                            tf.append(e0.elapsed_time(e1))
                    facc = ctx.phys_loss_acc(g, ffast)
                    ls_, lf_ = ctx.finalize(dacc.cpu().numpy(), pw, g.N), ctx.finalize(facc.cpu().numpy(), pw, g.N)
                    ms_fast = statistics.mean(tf)
                    tc_fl = 3 * (L - 1) * 6 * 2 * H2 * H2
                    row["tensor_core_fast_mode"] = {
                        "ms_fields": ms_fast, "speedup_vs_strict": ms_f / ms_fast,
                        "max_output_err_over_max_output": max(float((x - y).abs().max() / x.abs().max()) for x, y in zip(fields, ffast)),
                        "loss_rel_err": [abs(float(x) - float(y)) / abs(float(x)) for x, y in zip(ls_, lf_)],
                        "bf16_tflops_issued": tc_fl * g.N / (ms_fast * 1e-3) / 1e12,
                        "frac_of_bf16_peak": tc_fl * g.N / (ms_fast * 1e-3) / 1e12 / bf16_peak()}
                    del ffast
                except Exception as e:      # shapes whose layer images do not fit in shared memory: PHYSAD_E_UNSUPPORTED
                    row["tensor_core_fast_mode"] = {"unsupported": str(e)[:120]}
                finally:
                    ctx.set_deep_mode(0)
                sweep.append(row)
                del fields
        extra["depth_sweep"] = sweep
        ctx.set_weights(cfg, *w)
        # the analytic (forward-mode tangent) loss: north_star's literal wording, additive and NOT the parity path --
        # a different discretisation of the same PDE (no finite differences), FFMA arithmetic, one network evaluation
        tacc = ctx.tangent_loss_acc(g, T0)
        for _ in range(3):
            ctx.tangent_loss_acc(g, T0, acc=tacc)
        evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(10)]
        for e0, e1 in evs:
            flush.zero_()
            e0.record(); ctx.tangent_loss_acc(g, T0, acc=tacc); e1.record()
        torch.cuda.synchronize()
        tms = statistics.median(e0.elapsed_time(e1) for e0, e1 in evs)
        tl = ctx.finalize(tacc.cpu().numpy(), pw, g.N)
        extra["analytic_tangent_loss_not_parity"] = {
            "value": g.N / (tms * 1e-3), "unit": UNIT, "ms_per_step": tms, "loss": {"sigma": float(tl[0]), "u": float(tl[1])},
            "ffma_tflops": 2 * 25 * H * g.N / (tms * 1e-3) / 1e12, "frac_of_ffma_peak": 2 * 25 * H * g.N / (tms * 1e-3) / 1e12 / peak_ffma,
            "note": "forward-mode derivatives through the MLP instead of finite differences (physad_tangent_loss_dev); "
                    "different discretisation: its loss is not comparable bit-for-bit with the metric's"}
        # the closed loop (additive, SURVEY 8f rank 1): losses + d(L_sigma + L_u)/d(weights) per step, device-resident
        pwc = PhysWeights(1.0, 1.0)
        gacc, ggrad = ctx.fused_loss_grad_acc(g, pwc, T0, DT)
        for _ in range(3):
            ctx.fused_loss_grad_acc(g, pwc, T0, DT, gacc, ggrad)
        evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(10)]
        for e0, e1 in evs:
            flush.zero_()
            e0.record()
            ctx.fused_loss_grad_acc(g, pwc, T0, DT, gacc, ggrad)
            e1.record()
        torch.cuda.synchronize()
        gms = sorted(e0.elapsed_time(e1) for e0, e1 in evs)[len(evs) // 2]
        extra["closed_loop_loss_and_weight_gradient"] = {
            "value": g.N / (gms * 1e-3), "unit": UNIT, "ms_per_step": gms, "kernels_per_step": 4,
            "note": "fields (strict MLP, 3 slices) -> residuals + sums -> stencil adjoint -> MLP backward; median of 10"}

    # N > 1: every rank must hold the same losses, and the in-kernel exchange must agree with a plain NCCL all-reduce
    multi = None
    if world > 1:
        step()                                   # acc <- the global sums through the timed path (kernel_only() left the slab's there)
        barrier()
        acc2 = ctx.fused_loss_acc(g, T0, DT, slab=slab).clone()
        dist.all_reduce(acc2, op=dist.ReduceOp.SUM)
        mine = [float(ls), float(lu)] + [float(v) for v in acc2.cpu().numpy()] + [float(v) for v in acc.cpu().numpy()]
        allv = [None] * world
        dist.all_gather_object(allv, mine)
        same = all(v[:2] == allv[0][:2] for v in allv)
        rel = max(abs(v[4 + k] - v[2 + k]) / abs(v[2 + k]) for v in allv for k in range(2))
        multi = {"ranks": world, "same_loss_on_every_rank": bool(same), "in_kernel_exchange_vs_nccl_rel_diff": rel,
                 "collective": "p2p" if p2p else "nccl", "ok": bool(same and rel <= 1e-12)}

    cpu = None
    if rank == 0 and not args.no_cpu_baseline:
        threads = host_threads()
        planes = (64 if threads >= 8 else 16) if world == 1 else 16   # N > 1: a short sample, the other ranks wait for it
        rate, kind, cores, closs = cpu_reference_rate(H, n, planes, threads)
        rate1, _, _, _ = cpu_reference_rate(H, n, 4, 1)
        cpu = {"value": rate, "unit": UNIT, "cores": cores, "kind": kind,
               "sample": f"{n}x{n}x{planes} planes of the workload grid on {cores} host threads "
                         f"(reference is single-threaded: 1 thread on {n}x{n}x4 = {rate1:.4g} points/s)"}

    if rank == 0:
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": max(3, args.warmup), "ms_per_step": total_ms / args.steps, "higher_is_better": True,
            "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": workload_name(H, n),
                       "hidden": H, "grid": [n, n, n], "parallelism": f"z-slab x{world}, halo recomputed, 1 all-reduce of 2 doubles "
                                      + ("inside the kernel over NVLink peer memory" if p2p else "(NCCL)" if world > 1 else "(n/a)"),
                       "mode": "strict fp32 MLP (FMUL+FADD, bit-exact); residual arithmetic "
                               + ("in double exactly as the CPU reference (bit-identical residuals)" if args.exact_residuals
                                  else "fp32 with FMAs (as the reference's CUDA kernels; ~1e-7 of the CPU)"),
                       "l2": "no HBM-resident inputs (coordinates from index, weights in the constant bank); L2 flushed "
                             "between timed steps with a 256 MiB write outside the per-step events",
                       "fused_variant": args.variant},
            "loss": {"sigma": float(ls), "u": float(lu)},
            "parity": parity_block(H, n, float(ls), float(lu)),
            "multi_rank_parity": multi,
            "clocks": clocks,
            "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": 16,
                    "loss": [float(e2e_out[0]), float(e2e_out[1])]},
            "gpu_launches": launches,
            "roofline": {"bound": "fp32-pipe", "achieved": achieved, "peak": peak_strict, "unit": "TFLOP/s",
                         "frac": achieved / peak_strict, "frac_vs_ffma_peak": achieved / peak_ffma, "traffic": ncu_dram_traffic() if (H == 64 and n == 256 and world == 1) else None,
                         "peak_source": peak_src, "peak_ffma": peak_ffma,
                         "flops_per_point": flops_per_point(H), "kernel_ms_mean": k_mean, "kernel_ms_min": k_min,
                         "executed_flops_per_point": executed_flops_per_point(H),
                         "frac_executed": executed_flops_per_point(H) * slab_pts / (k_mean * 1e-3) / 1e12 / peak_strict,
                         "note": "achieved = ALGORITHMIC flops (51H+68)/point x slab points / CUDA-event kernel time; peak = measured "
                                 "non-contracted FMUL+FADD rate (parity mode cannot use FFMA). frac > 1 because the kernel "
                                 "executes fewer operations than the algorithmic count (shared layer-1 prefix across the three "
                                 "time slices; bit-identical results): frac_executed counts what it really executes and agrees "
                                 "with ncu's FMA-pipe utilisation. HBM traffic is ~0 by design"},
            "cpu_baseline": cpu,
            "wall_s_timed_region": wall,
            "step_ms": {"min": min(per), "median": statistics.median(per), "max": max(per)},
            "per_rank": getattr(timed, "per_rank", None),
        }
        if extra:
            line["extra"] = extra
        print(json.dumps(line), flush=True)
    ctx.close()
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
