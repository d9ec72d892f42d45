"""Parameter generation on the device (zk_groth16_generate): wall time, per-stage kernel times, fixed-base throughput against the
calibrated modmul roofline, the window-size sweep and the previous zk_scalar_mul_many kernel, and the CPU port baseline.

    python tools/setup_bench.py [--out DIR] [--exp-lib PATH] [--reps N]

Stages come from one torch.profiler run per shape (CUDA kernel activity, grouped by kernel name); wall times from a host clock
around the (synchronous) call after a warm-up, profiler off.  --exp-lib names a library built with the measurement knobs, e.g.
    make -C zero_chain_b200/csrc EXPERIMENTS=1 OBJDIR=/tmp/zkexp TARGET=/tmp/zkexp/libzkb200.so
with which the window sizes c = 6, 8, 10, 12 (ZK_FB_C) and the previous one-thread-per-point kernel (ZK_FB_OLD) are timed on the
same 2^20 G1 scalars, alternated in one process, outputs compared.  Without it those rows are reported as not measured."""
import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

STAGES = [  # (stage, kernel-name substrings)
    ("tau_powers_ifft", ("k_setup_consts", "k_tau_powers", "k_ntt_")),
    ("transpose_column_sums", ("k_col_hist", "k_col_scatter", "k_qap_")),
    ("compaction", ("k_setup_flags", "k_setup_fill", "k_scan_")),
    ("fixed_base_tables", ("k_fb_bases", "k_fb_table")),
    ("fixed_base_g1", ("k_fixed_base<Fp<FqParams>", "k_fixed_baseI2FpI8FqParams")),
    ("fixed_base_g2", ("k_fixed_base<Fq2", "k_fixed_baseI3Fq2")),
    ("window_tables_params_from_device", ("k_precompute", "k_any_inf")),
]


def card():
    try:
        return subprocess.check_output(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], text=True).strip()
    except Exception as e:          # noqa: BLE001
        return "unknown (%s)" % e


def nonzero_digits(c, samples=4000, seed=5):
    """Average non-zero signed digits of a uniform Fr scalar with c-bit windows (= mixed additions per point)."""
    import random
    from zero_chain_b200.groth16 import R_MODULUS
    rng = random.Random(seed)
    W, tot = 256 // c + 1, 0
    for _ in range(samples):
        k, carry = rng.randrange(R_MODULUS), 0
        for w in range(W):
            v = ((k >> (c * w)) & ((1 << c) - 1)) + carry
            carry = 1 if v > 1 << (c - 1) else 0
            tot += (v - (carry << c)) != 0
    return tot / samples


def stage_times(fn):
    import torch
    from torch.profiler import ProfilerActivity, profile
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    out = {s: 0.0 for s, _ in STAGES}
    other = 0.0
    for ev in prof.events():
        if ev.device_type.name != "CUDA":
            continue
        ms = ev.device_time / 1e3 if hasattr(ev, "device_time") else ev.cuda_time / 1e3
        for s, keys in STAGES:
            if any(k in ev.name for k in keys):
                out[s] += ms
                break
        else:
            other += ms
    out["other_kernels_and_copies"] = other
    return out


def sweep(exp_lib, n):
    """Child process on the experiment library: c sweep and old kernel on the same 2^20 G1 scalars, alternated."""
    import numpy as np
    from zero_chain_b200 import _lib
    _lib.SO_PATH = exp_lib
    from zero_chain_b200 import groth16 as zk
    from zero_chain_b200 import synthetic as sy
    ctx = zk.Context(0)
    sc = sy.random_fr_limbs(n, 77)
    arms = [("c%d" % c, {"ZK_FB_C": str(c)}) for c in (6, 8, 10, 12)] + [("old", {"ZK_FB_OLD": "1"})]
    res, outs = {a: [] for a, _ in arms}, {}
    for rep in range(4):
        for a, env in arms:
            for k in ("ZK_FB_C", "ZK_FB_OLD"):
                os.environ.pop(k, None)
            os.environ.update(env)
            t = time.perf_counter()
            o = zk.scalar_mul_many(ctx, 1, zk.G1_GENERATOR, sc)
            dt = time.perf_counter() - t
            if rep:                                  # rep 0 is the warm-up
                res[a].append(dt)
            outs[a] = o
    same = {a: bool(np.array_equal(outs[a], outs["old"])) for a in outs}
    ctx.close()
    return {a: dict(best_ms=1e3 * min(v), median_ms=1e3 * sorted(v)[len(v) // 2], points_per_s=n / min(v), equal_to_old=same[a]) for a, v in res.items()}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--exp-lib", default=None)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--sweep-child", default=None, help=argparse.SUPPRESS)
    a = ap.parse_args()
    if a.sweep_child:
        print(json.dumps(sweep(a.sweep_child, 1 << 20)))
        return
    from oracle import coracle as co
    from zero_chain_b200 import groth16 as zk
    from zero_chain_b200 import synthetic as sy
    rep = {"card": card()}
    print("card:", rep["card"], flush=True)
    ctx = zk.Context(0)
    fq_peak, _ = zk.bench_modmul(ctx, zk.FIELD_FQ, 148 * 4, 256, 3000)
    rep["fq_modmul_per_s"] = fq_peak
    c = 12                                          # setup.cu FB_C
    adds = nonzero_digits(c)
    rep["fixed_base"] = dict(window_bits=c, mixed_additions_per_point=adds, fq_products_per_g1_add=10, fq_products_per_g2_add=28)
    g1 = co.g1_encode(co.g1_generator(), False)
    g2 = co.g2_encode(co.g2_generator(), False)
    n20 = 1 << 20
    shapes = [("conf", sy.CONF_SHAPE), ("anon", sy.ANON_SHAPE),
              ("2p20", dict(n_constraints=n20, n_inputs=23, n_aux=n20 - 64, a_aux_density=(n20 - 64) * 4 // 5, b_density=(n20 - 64) * 5 // 8))]
    td = dict(tau=0x1234567 << 200, alpha=0x55 << 240, beta=0xABCDEF << 100, gamma=0x77 << 220, delta=3 ** 150 % zk.R_MODULUS)
    rep["shapes"] = {}
    for name, shp in shapes:
        t = time.time()
        r1cs = sy.make_r1cs(seed=1, **shp)
        cs = zk.ConstraintSystem(ctx, r1cs.n_inputs, r1cs.n_aux, r1cs.A, r1cs.B, r1cs.C)
        print("%s: circuit built in %.1fs" % (name, time.time() - t), flush=True)
        gen = lambda: zk.generate_parameters(cs, g1, g2, td["alpha"], td["beta"], td["gamma"], td["delta"], td["tau"])
        gen().free()                                                    # warm-up
        wall = []
        for _ in range(a.reps):
            t = time.perf_counter()
            p = gen()
            wall.append(time.perf_counter() - t)
            counts = (p.n_ic, p.n_h, p.n_l, p.n_a, p.n_b_g1, p.n_b_g2)
            p.free()
        st = stage_times(lambda: gen().free())
        n1 = 3 + counts[0] + (counts[1] + 1) + counts[2] + (counts[3] + 2) + (counts[4] + 2)
        n2 = counts[5] + 2 + 3
        total = sum(v for k, v in st.items() if k != "other_kernels_and_copies")
        row = dict(counts=counts, wall_ms_best=1e3 * min(wall), wall_ms_median=1e3 * sorted(wall)[len(wall) // 2], stages_ms=st,
                   kernels_ms_with_window_tables=total, kernels_ms_without_window_tables=total - st["window_tables_params_from_device"],
                   g1_points=n1, g2_points=n2)
        for grp, npts, key, per in ((1, n1, "fixed_base_g1", 10), (2, n2, "fixed_base_g2", 28)):
            ms = st[key]
            if ms > 0:
                prod = npts * adds * per
                row["g%d_points_per_s" % grp] = npts / (ms * 1e-3)
                row["g%d_roofline_share" % grp] = prod / (ms * 1e-3) / fq_peak
        rep["shapes"][name] = row
        print(name, json.dumps(row), flush=True)
        cs.free()
    ctx.close()
    # the CPU path the repository used until now: the closed-form CRS with the C oracle's fixed-base multiplication (port baseline)
    r1cs = sy.make_r1cs(seed=1, **sy.CONF_SHAPE)
    t = time.time()
    sy.make_toy_crs(r1cs, co.g1_fixed_base, co.g2_fixed_base, seed=2)
    rep["cpu_port_baseline_conf_s"] = time.time() - t
    rep["cpu_port_baseline_threads"] = co.num_threads()
    print("cpu port baseline (make_toy_crs + C oracle fixed base, CONF_SHAPE): %.2fs on %d threads" % (rep["cpu_port_baseline_conf_s"], co.num_threads()), flush=True)
    if a.exp_lib:
        out = subprocess.check_output([sys.executable, os.path.abspath(__file__), "--sweep-child", a.exp_lib], cwd=ROOT, text=True)
        rep["sweep_2p20_g1"] = json.loads(out.strip().splitlines()[-1])
    else:
        rep["sweep_2p20_g1"] = "not measured (no --exp-lib)"
    print("sweep:", json.dumps(rep["sweep_2p20_g1"]), flush=True)
    if a.out:
        os.makedirs(a.out, exist_ok=True)
        with open(os.path.join(a.out, "setup_bench.json"), "w") as f:
            json.dump(rep, f, indent=1)
    print(json.dumps(rep))


if __name__ == "__main__":
    main()
