"""Generate tests/golden/*.npz|json from the UNMODIFIED reference CPU sources.

Run in the dev container (needs /root/reference to build oracle/_ref/libphysref.so):
    python tests/golden/make_golden.py
The fixtures are small on purpose (a few hundred KB): full-size parity on the GPU box goes through
the prebuilt oracle/_ref library or the pinned C port, not through stored arrays.
"""
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
import oracle  # noqa: E402
from oracle import Grid  # noqa: E402

HERE = os.path.dirname(os.path.abspath(__file__))


def main():
    oracle.build(ref_too=True)
    R = oracle.reference()
    assert R is not None, "reference library not built (is /root/reference present?)"
    out = {}
    meta = {"cases": [], "anchors": {}}

    # 1. weight streams (libstdc++ mt19937 + uniform_real_distribution<float>)
    for seed, scale, H in [(123, 0.25, 64), (321, 0.25, 64), (777, 0.25, 32), (777, 0.25, 64), (777, 0.25, 128),
                           (42, 0.5, 16)]:
        W1, b1, W2, b2 = R.mlp_random_init(H, seed, scale)
        key = f"w_s{seed}_h{H}"
        out[key + "_W1"], out[key + "_b1"], out[key + "_W2"], out[key + "_b2"] = W1, b1, W2, b2
        meta["cases"].append({"kind": "weights", "key": key, "seed": seed, "scale": scale, "H": H})

    # 2. small full-path cases: MLP grid outputs, fields, residuals, losses, VJP
    cases = [
        dict(name="p_9x7x6_h16", g=(9, 7, 6), h=(1.0, 1.0, 1.0), dt=2e-3, periodic=True, H=16, seed=42, scale=0.5,
             t=0.25, m1p1=True, w=(1.0, 1.0)),
        dict(name="c_9x7x6_h16", g=(9, 7, 6), h=(0.5, 0.25, 2.0), dt=1e-2, periodic=False, H=16, seed=42, scale=0.5,
             t=0.25, m1p1=True, w=(1.7, 0.9)),
        dict(name="z_12x5x4_h32", g=(12, 5, 4), h=(1.0, 1.0, 1.0), dt=2e-3, periodic=True, H=32, seed=777, scale=0.25,
             t=-0.4, m1p1=False, w=(1.0, 1.0)),
        dict(name="c_33x18x3_h64", g=(33, 18, 3), h=(1.0, 1.0, 1.0), dt=2e-3, periodic=False, H=64, seed=123,
             scale=0.25, t=0.3, m1p1=True, w=(1.0, 1.0)),
        dict(name="p_1x1x1_h16", g=(1, 1, 1), h=(1.0, 1.0, 1.0), dt=2e-3, periodic=True, H=16, seed=42, scale=0.5,
             t=0.25, m1p1=True, w=(1.0, 1.0)),
        dict(name="p_2x1x3_h16", g=(2, 1, 3), h=(1.0, 1.0, 1.0), dt=2e-3, periodic=True, H=16, seed=42, scale=0.5,
             t=0.25, m1p1=True, w=(1.0, 1.0)),
    ]
    for c in cases:
        g = Grid(*c["g"], *c["h"], c["dt"], c["periodic"])
        w = R.mlp_random_init(c["H"], c["seed"], c["scale"])
        y = R.mlp_grid_infer(g, w, c["t"], c["m1p1"])
        f = R.generate_fields(g, w, c["t"], c["dt"], c["m1p1"])
        ls, lu, Rr = R.phys_loss_forward(g, c["w"][0], c["w"][1], f, want_residuals=True)
        G = R.phys_loss_backward(g, c["w"][0], c["w"][1], Rr)
        n = c["name"]
        out[n + "_y"] = y
        for k, a in zip(["sm", "s0", "sp", "um", "u0", "up"], f):
            out[f"{n}_{k}"] = a
        for k, a in zip(["Rs", "Rx", "Ry", "Rz"], Rr):
            out[f"{n}_{k}"] = a
        for k, a in zip(["gs", "gx", "gy", "gz"], G):
            out[f"{n}_{k}"] = a
        c2 = dict(c)
        c2.update(kind="path", loss_sigma=repr(float(ls)), loss_u=repr(float(lu)))
        meta["cases"].append(c2)

    # 2b. MLP backward (MSE weight gradients) on a small random batch, generic dims
    rng = np.random.default_rng(7)
    B, In, H, Out = 23, 5, 12, 3
    bw = dict(x=rng.uniform(-1, 1, B * In), t=rng.uniform(-1, 1, B * Out), W1=rng.uniform(-.4, .4, H * In),
              b1=rng.uniform(-.4, .4, H), W2=rng.uniform(-.4, .4, Out * H), b2=rng.uniform(-.4, .4, Out))
    bw = {k: v.astype(np.float32) for k, v in bw.items()}
    g4 = R.mlp_backward(bw["x"], bw["t"], bw["W1"], bw["b1"], bw["W2"], bw["b2"], B, In, H, Out)
    for k, v in bw.items():
        out["bwd_" + k] = v
    for k, v in zip(["dW1", "db1", "dW2", "db2"], g4):
        out["bwd_" + k] = v
    meta["cases"].append(dict(kind="backward", B=B, In=In, H=H, Out=Out))

    # 3. scalar anchors at the BASELINE sizes (SURVEY.md section 7 step 1 lists the same numbers)
    for H in (32, 64, 128):
        g = Grid(64, 64, 64, 1, 1, 1, 2e-3, True)
        w = R.mlp_random_init(H, 777, 0.25)
        r = R.fused_loss(g, w, 0.25, 2e-3, threads=8, want_residuals=True)
        meta["anchors"][f"64c_h{H}"] = dict(loss_sigma=repr(float(r["loss_sigma"])), loss_u=repr(float(r["loss_u"])),
                                            R_sigma0=repr(float(r["R"][0][0])), W1_0=repr(float(w[0][0])))
    # 3b. the HEADLINE config (BASELINE.json metric: 256^3, seed 777, scale 0.25, t 0.25, dt 2e-3, periodic) and its
    # width-sweep siblings, whole grid through the unmodified reference on all host threads (~10-30 s each):
    # pins what bench.py times and what tests/test_gpu_parity.py::test_fused_256_* asserts at 1e-4
    nthreads = len(os.sched_getaffinity(0))
    for H in (32, 64, 128):
        g = Grid(256, 256, 256, 1, 1, 1, 2e-3, True)
        w = R.mlp_random_init(H, 777, 0.25)
        r = R.fused_loss(g, w, 0.25, 2e-3, threads=nthreads)
        meta["anchors"][f"256c_h{H}"] = dict(loss_sigma=repr(float(r["loss_sigma"])), loss_u=repr(float(r["loss_u"])))
    g = Grid(32, 32, 24, 1, 1, 1, 1.0, False)  # test_mlp_grid_infer.cpp:15-20
    w = R.mlp_random_init(64, 123, 0.25)
    y = R.mlp_grid_infer(g, w, 0.3, True)
    meta["anchors"]["grid_infer_32x32x24"] = dict(sum=repr(float(np.sum(y.astype(np.float64)))),
                                                  y0=[repr(float(v)) for v in y[:4]],
                                                  crc=int(np.bitwise_xor.reduce(y.view(np.uint32))))
    np.savez_compressed(os.path.join(HERE, "golden.npz"), **out)
    with open(os.path.join(HERE, "golden.json"), "w") as fh:
        json.dump(meta, fh, indent=1)
    print("wrote", len(out), "arrays;", os.path.getsize(os.path.join(HERE, "golden.npz")), "bytes")


def full_size_128():
    """tests/golden/full128.npz: BASELINE config 3 (128^3, H = 64 and 128, seed 777, scale 0.25, t 0.25, dt 2e-3,
    periodic) for tests/test_gpu_parity.py::test_fused_full_size_128_properties -- both losses, the whole-grid max|R| of
    each residual and the residuals at a fixed seeded sample of 4096 points.  Computed by the reference library when it
    is built, else by the C port, which the golden vectors above pin bit for bit to the reference's CPU path.
        python tests/golden/make_golden.py --full128"""
    chk = oracle.reference() or oracle.port()
    g = Grid(128, 128, 128, 1, 1, 1, 2e-3, True)
    idx = np.sort(np.random.default_rng(128).choice(g.N, 4096, replace=False)).astype(np.int64)
    out = {"idx": idx}
    for H in (64, 128):
        w = chk.mlp_random_init(H, 777, 0.25)
        if chk.kind == "reference":
            r = chk.fused_loss(g, w, 0.25, 2e-3, threads=len(os.sched_getaffinity(0)), want_residuals=True)
        else:
            r = chk.fused_loss(g, w, 0.25, 2e-3, want_residuals=True)
        out[f"h{H}_loss"] = np.array([r["loss_sigma"], r["loss_u"]], np.float32)
        out[f"h{H}_Rmax"] = np.array([np.max(np.abs(a)) for a in r["R"]], np.float64)
        out[f"h{H}_R"] = np.stack([a[idx] for a in r["R"]])
    path = os.path.join(HERE, "full128.npz")
    np.savez_compressed(path, source=np.array(chk.kind), **out)
    print("wrote", path, os.path.getsize(path), "bytes from the", chk.kind)


if __name__ == "__main__":
    if sys.argv[1:] == ["--full128"]:
        full_size_128()
    else:
        main()
