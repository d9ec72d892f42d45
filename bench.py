#!/usr/bin/env python3
"""bench.py — headline benchmark of the B200-native Groth16 prover hot path.

Metric (BASELINE.json): G1 Pippenger MSM Mop/s at 2^20 bases (configs[1]), whole-job aggregate over
N GPUs, with proofs/sec for the confidential_transfer-shaped circuit reported in "secondary".

  python bench.py --gpus N --steps K --warmup W            # our arm (one rank per GPU under torchrun)
  python bench.py --impl reference --gpus N ...            # reference arm: the CPU restatement of the
                                                           # reference's bellman/pairing path (oracle/) on
                                                           # the box's host cores; rank 0 only

A "step" is one complete MSM of 2^20 terms per GPU: scalars -> digits -> counting sort -> bucket
accumulation -> bucket reduction -> canonical affine result (96 bytes, bit-identical to the oracle).
N > 1 is weak scaling: every rank owns a 2^20-base shard of an N*2^20-term MSM (bases partitioned by
index range, SURVEY.md §8e); the 192-byte partial results are exchanged with one NCCL all-gather and
folded on every rank.  `value` has scalars resident in HBM; `e2e` goes through the C-ABI call with
scalars in pinned HOST memory (host->device copy and the 96-byte device->host result inside the timed
region).  Only the cpu_baseline leg and --impl reference touch oracle/.

--dump-outputs DIR writes, after the timed steps, the result of the last headline step as DIR/g1_msm.npy: the 96-byte
uncompressed G1 encoding the MSM call returns, one byte per float64 element.  Inputs are generated from fixed seeds, so two
builds run with the same arguments can be compared output for output.
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

LOG_N = 20
N_SETS = 8                     # distinct scalar vectors cycled through: 8 x 32 MiB = 256 MiB > 126 MB L2
KERNELS_PER_MSM = 38           # 20-bit windows at 2^20: digits, tile_hist, col_scan, scan_block, scatter, fine_sort; 2 batched-affine rounds x
                               # (half_sizes, 2 x scan_block, scan_add, ba_forward, ba_invert, ba_backward); pick_task_len, 2 x scan_block,
                               # scan_add, len_hist, len_scan, len_place, accumulate, combine_serial, combine_warp, rowcol_stage1, 2 x seg_sums,
                               # bit_sums, sum_points, finish_bits, join_rowcol, encode_xyzz
                               # (counted from the ncu launch list profiles/r02_launches_msm_2p20.csv; N > 1 adds the fold kernel)
ALGO_MODMUL_PER_TERM = 176     # 11 (mixed add) x ceil(255/16) windows — the FIXED convention of SURVEY.md §8(d) / BASELINE.md §3,
                               # independent of the window size the library actually uses
ALGO_BYTES_PER_TERM = 128      # 96 B base + 32 B scalar


def host_cores():
    """Host threads for the CPU port: physical cores in the affinity mask, capped by the container's CPU quota."""
    try:
        cpus = os.sched_getaffinity(0)
    except Exception:
        cpus = set(range(os.cpu_count() or 1))
    n = len(cpus)
    try:        # physical cores among them: the port's OpenMP teams gain nothing from hyper-thread siblings and lose a lot in the short
        seen, cur = set(), {}          # parallel regions of create_proof (measured on the B200 box: 128 threads 25x slower than 64)
        for line in open("/proc/cpuinfo"):
            if ":" in line:
                k, v = [x.strip() for x in line.split(":", 1)]
                cur[k] = v
            elif cur:
                if int(cur.get("processor", -1)) in cpus and "core id" in cur:
                    seen.add((cur.get("physical id", "0"), cur["core id"]))
                cur = {}
        if seen:
            n = min(n, len(seen))
    except Exception:
        pass
    try:
        q, p = open("/sys/fs/cgroup/cpu.max").read().split()[:2]
        if q != "max":
            n = min(n, max(1, int(int(q) / int(p))))
    except Exception:
        try:
            q = int(open("/sys/fs/cgroup/cpu/cpu.cfs_quota_us").read()); p = int(open("/sys/fs/cgroup/cpu/cpu.cfs_period_us").read())
            if q > 0:
                n = min(n, max(1, q // p))
        except Exception:
            pass
    return n


def pick_threads(co, trial):
    """The CPU port is given the OpenMP team size it runs fastest with: `trial()` (a short sample of the workload) is timed at
    the candidate counts (all usable CPUs, then halves) and the best one stays set.  Returns (threads, {threads: seconds})."""
    top = host_cores()
    try:
        top = max(top, len(os.sched_getaffinity(0)))
    except Exception:
        pass
    cands, c = [], top
    while c >= 8 and len(cands) < 4:
        cands.append(c); c //= 2
    if not cands:
        cands = [top]
    seen = {}
    for c in cands:
        co.set_num_threads(c)
        trial()                                   # warm-up at this team size
        t = time.perf_counter(); trial(); seen[c] = time.perf_counter() - t
    best = min(seen, key=seen.get)
    co.set_num_threads(best)
    return best, {str(k): round(v, 4) for k, v in seen.items()}


def env_int(name, default):
    try:
        return int(os.environ.get(name, default))
    except ValueError:
        return default


def peaks():
    try:
        p = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        return float(p["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region."""
    Q = "index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown," \
        "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, gpu_index):
        self.f = tempfile.NamedTemporaryFile("w+", suffix=".csv", delete=False)
        self.p = None
        try:
            self.p = subprocess.Popen(["nvidia-smi", "-i", str(gpu_index), "--query-gpu=" + self.Q, "--format=csv,noheader,nounits", "-lms", "100"],
                                      stdout=self.f, stderr=subprocess.DEVNULL)
        except Exception:
            self.p = None

    def stop(self):
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        if self.p is None:
            return out
        time.sleep(0.15)
        self.p.terminate()
        try:
            self.p.wait(timeout=5)
        except Exception:
            self.p.kill()
        self.f.flush()
        rows = [l.strip().split(", ") for l in open(self.f.name) if l.strip()]
        os.unlink(self.f.name)
        sm, reasons = [], set()
        for r in rows:
            if len(r) < 9:
                continue
            try:
                sm.append(float(r[1])); out["sm_max_mhz"] = float(r[2])
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[5:9]):
                if v.strip().lower().startswith("active"):
                    reasons.add(name)
        if sm:
            out["sm_mhz"] = float(np.median(sm)); out["samples"] = len(sm)
        out["reasons"] = sorted(reasons)
        return out


R_MODULUS = 0x73eda753299d7d483339d80809a1d80553bda402fffe5bfeffffffff00000001


def dot_mod_r(s, b):
    """sum_i s_i * b_i mod r for two (n,4) uint64 limb arrays, exact, with numpy only (no curve code, nothing shared with
    the library or the oracle): 16-bit chunks, so that every partial dot product stays below 2^64 for n <= 2^24."""
    s = np.ascontiguousarray(s, np.uint64).reshape(-1, 4)
    b = np.ascontiguousarray(b, np.uint64).reshape(-1, 4)
    assert s.shape == b.shape and s.shape[0] <= (1 << 24)
    s16, b16 = s.view(np.uint16).reshape(-1, 16), b.view(np.uint16).reshape(-1, 16)
    bcols = [(k, b16[:, k].astype(np.uint64)) for k in range(16) if b16[:, k].any()]
    total = 0
    for j in range(16):
        sj = s16[:, j].astype(np.uint64)
        for k, bk in bcols:
            total += int(np.dot(sj, bk)) << (16 * (j + k))
    return total % R_MODULUS


def closed_form_g1(k):
    """Uncompressed encoding of k * G1 by the big-integer affine reference (oracle/pyref.py — used as the checker only)."""
    from oracle import pyref as pr
    return pr.g1_uncompressed(pr.ec_mul(pr.FQ, pr.G1_GEN, k % R_MODULUS))


# ---- witness factory for the proofs/sec leg: runs in worker PROCESSES (spawn), numpy / big-int only ----
_WK = {}


def _wk_init(crs_light):
    _WK["crs"] = crs_light


def _wk_witness(k):
    """Witness k of the synthetic confidential_transfer-shaped circuit: evaluations, assignment, (r, s) and the proof the
    trapdoor algebra predicts for them (closed form, oracle/pyref.py big-integer curve arithmetic: the checker)."""
    from oracle import pyref as pr
    from zero_chain_b200 import synthetic as sy
    crs = _WK["crs"]
    r = crs.r1cs
    z = sy.make_witness(r, 100 + k)
    a, b, c = sy.evaluate(r, z)
    rng = sy.SplitMix64(4242 + 7919 * k)
    rr, ss = rng.fr(), rng.fr()
    A, B, C = sy.expected_proof_scalars(crs, z, rr, ss)
    want = pr.proof_bytes(pr.ec_mul(pr.FQ, pr.G1_GEN, A), pr.ec_mul(pr.FQ2, pr.G2_GEN, B), pr.ec_mul(pr.FQ, pr.G1_GEN, C))
    arrs = [sy.ints_to_limbs(v) for v in (a, b, c, z[:r.n_inputs], z[r.n_inputs:])]
    return k, arrs, rr, ss, want


def make_witnesses(crs, count, procs):
    """`count` DISTINCT witnesses with distinct (r, s) and their closed-form proofs, generated in parallel on the host."""
    import dataclasses
    import multiprocessing as mp
    light = dataclasses.replace(crs, params_bytes=b"")
    procs = max(1, min(procs, count))
    if procs == 1:
        _wk_init(light)
        res = [_wk_witness(k) for k in range(count)]
    else:
        with mp.get_context("spawn").Pool(procs, initializer=_wk_init, initargs=(light,)) as pool:
            res = pool.map(_wk_witness, range(count), chunksize=max(1, count // (4 * procs)))
    res.sort(key=lambda t: t[0])
    return res


def make_scalars(n, rank, k):
    from zero_chain_b200 import synthetic as sy
    return sy.random_fr_limbs(n, 1000 + 97 * rank + k)


class MsmJob:
    """One sharded MSM workload on this rank: resident bases (+ window tables), N_SETS scalar vectors in HBM and in pinned
    host memory, and the two ways of running a step (blocking calls / two futures in flight on two contexts)."""

    def __init__(self, zk, torch, dist, ctxs, world, local, bases, h_sets, n):
        self.zk, self.torch, self.dist, self.world, self.n, self.bases = zk, torch, dist, world, n, bases
        self.ctx, self.ctx2 = ctxs
        self.ns = len(h_sets)
        self.dev = torch.device("cuda", local)
        self.stream = torch.cuda.ExternalStream(self.ctx.stream, device=self.dev)
        self.d_sets = [torch.from_numpy(h.view(np.int64)).cuda() for h in h_sets]
        self.pinned = [torch.from_numpy(h.view(np.int64)).pin_memory() for h in h_sets]
        psz = zk.partial_size(1)
        self.d_part = torch.zeros(psz, dtype=torch.uint8, device="cuda")
        self.d_all = torch.zeros(psz * world, dtype=torch.uint8, device="cuda")
        self.d_stage = torch.empty_like(self.d_sets[0])
        self.lanes = {}
        if world > 1:      # per context: its partial, the gathered partials, a staging buffer for the e2e arm, torch views of its two streams
            for c in ctxs:
                self.lanes[id(c)] = dict(part=torch.zeros(psz, dtype=torch.uint8, device="cuda"), all=torch.zeros(psz * world, dtype=torch.uint8, device="cuda"),
                                         stage=torch.empty_like(self.d_sets[0]), main=torch.cuda.ExternalStream(c.stream, device=self.dev),
                                         tail=torch.cuda.ExternalStream(zk.tail_stream(c), device=self.dev))
        torch.cuda.synchronize()

    # ---- blocking calls ----
    def step_device(self, k):
        zk, d = self.zk, self.d_sets[k % self.ns]
        if self.world == 1:
            return zk.multiexp_device(self.bases, d.data_ptr(), self.n)
        zk.multiexp_partial_device(self.bases, d.data_ptr(), self.n, self.d_part.data_ptr())
        with self.torch.cuda.stream(self.stream):          # NCCL all-gather enqueued on the library's stream: no host sync needed
            self.dist.all_gather_into_tensor(self.d_all, self.d_part)
        return zk.points_fold(self.ctx, 1, self.d_all.data_ptr(), self.world)

    def step_e2e(self, k):
        zk, h = self.zk, self.pinned[k % self.ns]
        if self.world == 1:
            return zk.multiexp(self.bases, h.numpy().view(np.uint64).reshape(-1, 4))    # C-ABI call with a HOST buffer
        with self.torch.cuda.stream(self.stream):
            self.d_stage.copy_(h, non_blocking=True)
        zk.multiexp_partial_device(self.bases, self.d_stage.data_ptr(), self.n, self.d_part.data_ptr())
        with self.torch.cuda.stream(self.stream):
            self.dist.all_gather_into_tensor(self.d_all, self.d_part)
        return zk.points_fold(self.ctx, 1, self.d_all.data_ptr(), self.world)

    # ---- futures ----
    def _begin_multi(self, c, d_ptr):
        L = self.lanes[id(c)]
        self.zk.multiexp_partial_device_begin(c, self.bases, d_ptr, self.n, L["part"].data_ptr())
        with self.torch.cuda.stream(L["tail"]):             # the all-gather is ordered after the partial on the context's tail stream
            self.dist.all_gather_into_tensor(L["all"], L["part"])
        self.zk.points_fold_begin(c, 1, L["all"].data_ptr(), self.world)

    def begin_device(self, c, k):
        if self.world == 1:
            return self.zk.multiexp_device_begin(c, self.bases, self.d_sets[k % self.ns].data_ptr(), self.n)
        self._begin_multi(c, self.d_sets[k % self.ns].data_ptr())

    def begin_e2e(self, c, k):
        if self.world == 1:
            return self.zk.multiexp_begin(c, self.bases, self.pinned[k % self.ns].numpy().view(np.uint64).reshape(-1, 4))
        L = self.lanes[id(c)]
        with self.torch.cuda.stream(L["main"]):
            L["stage"].copy_(self.pinned[k % self.ns], non_blocking=True)
        self._begin_multi(c, L["stage"].data_ptr())

    def barrier(self):
        if self.world > 1:
            self.dist.barrier()
        self.torch.cuda.synchronize()

    def _max_over_ranks(self, ms):
        if self.world == 1:
            return ms
        t = self.torch.tensor([ms], dtype=self.torch.float64, device="cuda")
        self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
        return float(t.item())

    def timed(self, fn, steps, warmup, profile=False):
        torch = self.torch
        for k in range(warmup):
            fn(k)
        self.barrier()
        if profile:
            self.ctx.profile(True)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(self.stream)
        last = None
        for k in range(steps):
            last = fn(warmup + k)
        e1.record(self.stream)
        self.barrier()
        ms = self._max_over_ranks(e0.elapsed_time(e1))
        if profile:
            a, ca = self.ctx.profile_read(), self.ctx.profile_counts()
            self.ctx.profile(False)
            return ms, last, (a[0], a[1], ca[0], ca[2])
        return ms, last

    def timed_pipelined(self, begin, steps, warmup, profile=False):
        """successive MSMs are independent jobs and the reference's multiexp returns a future: two of them are kept in flight on
        two contexts (zk_msm_begin / zk_msm_end), so the latency-bound tail of one MSM and the upload of the next scalars overlap
        the accumulation of the other."""
        torch, zk = self.torch, self.zk
        ctxs = [self.ctx, self.ctx2]
        res = {}

        def run(k0, k1):
            inflight = [None, None]
            for k in range(k0, k1):
                c = k % 2
                if inflight[c] is not None:
                    res[inflight[c]] = zk.multiexp_end(ctxs[c], self.bases)
                begin(ctxs[c], k)
                inflight[c] = k
            for k in sorted(x for x in inflight if x is not None):
                res[k] = zk.multiexp_end(ctxs[k % 2], self.bases)
        run(0, warmup)
        self.barrier()
        if profile:
            self.ctx.profile(True); self.ctx2.profile(True)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(self.stream)
        run(warmup, warmup + steps)
        e1.record(self.stream)                  # every MSM has been collected on the host, so this is after all of the work
        self.barrier()
        ms = self._max_over_ranks(e0.elapsed_time(e1))
        prof = None
        if profile:
            a, b_ = self.ctx.profile_read(), self.ctx2.profile_read()
            ca, cb = self.ctx.profile_counts(), self.ctx2.profile_counts()
            prof = (a[0] + b_[0], a[1] + b_[1], ca[0] + cb[0], ca[2] + cb[2])
            self.ctx.profile(False); self.ctx2.profile(False)
        return ms, res[warmup + steps - 1], prof

    def close(self):
        # ordered teardown: tensors that were used on the library's streams must be released before the streams are
        # destroyed with the contexts (their allocator blocks record events on them when freed)
        self.lanes.clear()
        self.d_sets = self.pinned = self.d_stage = self.d_part = self.d_all = None
        self.torch.cuda.synchronize()
        self.torch.cuda.empty_cache()
        self.bases.free()


def gather_ints(dist, torch, world, value):
    """all-gather one < 2^256 python integer per rank (as four 64-bit limbs over the process group)."""
    if world == 1:
        return [value]
    limbs = np.array([(value >> (64 * j)) & 0xFFFFFFFFFFFFFFFF for j in range(4)], dtype=np.uint64)
    dev = "cuda" if dist.get_backend() == "nccl" else "cpu"       # gloo in the CPU test of this plumbing
    t = torch.from_numpy(limbs.view(np.int64)).to(dev)
    out = torch.zeros(4 * world, dtype=torch.int64, device=dev)
    dist.all_gather_into_tensor(out, t)
    rows = out.cpu().numpy().view(np.uint64).reshape(world, 4)
    return [sum(int(x) << (64 * j) for j, x in enumerate(r)) for r in rows]


def strong_scaling_leg(zk, sy, torch, dist, ctxs, world, rank, local, log_total, steps):
    """BASELINE.json configs[4] / SURVEY.md §8(d) C5: ONE G1 MSM of 2^log_total terms, bases (g+1)*G over the GLOBAL index g,
    sharded by contiguous range over the ranks (2^24 over 8 GPUs = 2^21 per GPU), partial sums all-gathered over NCCL and folded.
    Fixed total work as N grows = strong scaling.  The folded result is checked against the closed form (sum s_g (g+1) mod r) * G."""
    total = 1 << log_total
    n = total // world
    g0 = rank * n
    t0 = time.time()
    idx = np.zeros((n, 4), np.uint64)
    idx[:, 0] = np.arange(g0 + 1, g0 + n + 1, dtype=np.uint64)
    bases_limbs = zk.scalar_mul_many(ctxs[0], 1, zk.G1_GENERATOR, idx)
    bases = zk.Bases(ctxs[0], 1, bases_limbs, precompute=True)
    del bases_limbs
    n_sets = 2
    h_sets = [sy.random_fr_limbs(n, 5000 + 31 * rank + k) for k in range(n_sets)]
    job = MsmJob(zk, torch, dist, ctxs, world, local, bases, h_sets, n)
    setup_s = time.time() - t0
    W = 2
    ms_p, res_p, _ = job.timed_pipelined(job.begin_device, steps, W)
    ms_b, res_b = job.timed(job.step_device, steps, W)
    last = (W + steps - 1) % n_sets
    parts = gather_ints(dist, torch, world, dot_mod_r(h_sets[last], idx))
    out = None
    if rank == 0:
        want = closed_form_g1(sum(parts))
        ok = (res_p == want) and (res_b == want)
        out = {"metric": "g1_msm_mops_2^%d_total" % log_total, "scaling": "strong", "total_terms": total, "terms_per_gpu": n, "n_gpus": world,
               "value": total * steps / (ms_p * 1e-3) / 1e6, "unit": "Mop/s", "ms_per_step": ms_p / steps, "steps": steps, "warmup": W,
               "blocking_ms_per_step": ms_b / steps, "blocking_mops": total * steps / (ms_b * 1e-3) / 1e6,
               "window_bits": bases.window_bits, "bases": "(g+1)*G over the global index g (SURVEY 8d C5)", "setup_s_untimed": round(setup_s, 2),
               "matches_closed_form": bool(ok),
               "check": "folded result == (sum_g s_g (g+1) mod r) * G; per-rank dot products in numpy, scalar multiple by oracle/pyref.py"}
        if not ok:
            raise SystemExit("PARITY FAILURE: sharded 2^%d MSM differs from the closed form" % log_total)
    job.close()
    return out


def run_ours(args):
    import torch
    import torch.distributed as dist
    from zero_chain_b200 import groth16 as zk
    from zero_chain_b200 import synthetic as sy

    world, rank, local = env_int("WORLD_SIZE", 1), env_int("RANK", 0), env_int("LOCAL_RANK", 0)
    if world != args.gpus and world > 1:
        raise SystemExit("--gpus %d but WORLD_SIZE=%d" % (args.gpus, world))
    torch.cuda.set_device(local)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        # NCCL prints its version banner to STDOUT when the first communicator is created; stdout must carry ONE JSON
        # line, so fd 1 points at stderr while the process group and its communicator come up.
        sys.stdout.flush()
        saved = os.dup(1)
        os.dup2(2, 1)
        try:
            opts = dist.ProcessGroupNCCL.Options()
            opts.is_high_priority_stream = True          # the 192-byte all-gather belongs to the latency-bound tail of an MSM
            dist.init_process_group("nccl", pg_options=opts, device_id=torch.device("cuda", local))
            warm = torch.zeros(1, device="cuda")
            dist.all_reduce(warm)
            torch.cuda.synchronize()
        finally:
            sys.stdout.flush()
            os.dup2(saved, 1)
            os.close(saved)
    n = 1 << args.log_n
    ctx, ctx2 = zk.Context(local), zk.Context(local)
    if args.affine_min_entries is not None:           # measurement switch: batched-affine bucket rounds (default: library default = off)
        for c in (ctx, ctx2):
            c.set_opt(zk.Context.OPT_AFFINE_MIN_ENTRIES, args.affine_min_entries)
            c.set_opt(zk.Context.OPT_AFFINE_LEVELS, args.affine_levels)

    # ---- setup (untimed): this rank's shard of the bases, generated on the device, + window tables ----
    t0 = time.time()
    base_scalars = sy.random_fr_limbs(n, 7 + rank)
    bases_limbs = zk.scalar_mul_many(ctx, 1, zk.G1_GENERATOR, base_scalars)      # uniform random subgroup points b_i * G
    bases = zk.Bases(ctx, 1, bases_limbs, window_bits=args.window_bits, precompute=True)
    setup_s = time.time() - t0
    h_sets = [make_scalars(n, rank, k) for k in range(N_SETS)]
    job = MsmJob(zk, torch, dist, (ctx, ctx2), world, local, bases, h_sets, n)

    # modmul roofline calibrated live on this GPU (register-resident independent Fq products)
    modmul_peak, _ = zk.bench_modmul(ctx, zk.FIELD_FQ, 148 * 4, 256, 3000)

    sampler = ClockSampler(local) if rank == 0 else None
    W = max(4, args.warmup)            # the last timed step (W + steps - 1) picks the scalar set the checks use
    ms_dev, res_dev, _ = job.timed_pipelined(job.begin_device, args.steps, W)
    clocks = sampler.stop() if sampler else None
    ms_e2e, res_e2e, _ = job.timed_pipelined(job.begin_e2e, args.steps, W)
    # the dominant stage is timed (CUDA events on the launching stream, zk_ctx_profile) during the BLOCKING loop: with two MSMs in
    # flight the interval between two events on one stream also contains the other context's kernels
    ms_b, res_b, prof = job.timed(job.step_device, args.steps, W, profile=True)
    ms_be, res_be = job.timed(job.step_e2e, args.steps, W)
    if not (res_b == res_dev == res_be == res_e2e):
        raise SystemExit("PARITY FAILURE: pipelined / blocking / host-buffer MSM results differ")
    blocking = {"device_ms_per_step": ms_b / args.steps, "device_mops": n * world * args.steps / (ms_b * 1e-3) / 1e6,
                "e2e_ms_per_step": ms_be / args.steps, "e2e_mops": n * world * args.steps / (ms_be * 1e-3) / 1e6,
                "api": "zk_msm_device / zk_msm (N > 1: zk_msm_partial_device + all-gather + zk_points_fold), one call at a time"}
    # fresh bases (bellman's multiexp takes the bases per call): no window tables, one bucket set per window + Horner tail
    fresh = None
    if world == 1 and args.secondary:
        fb = zk.Bases(ctx, 1, bases_limbs, precompute=False)
        fjob_step = lambda k: zk.multiexp_device(fb, job.d_sets[k % N_SETS].data_ptr(), n)
        ms_f, res_f = job.timed(fjob_step, max(3, args.steps // 2), 2)
        if res_f != zk.multiexp_device(bases, job.d_sets[(2 + max(3, args.steps // 2) - 1) % N_SETS].data_ptr(), n):
            raise SystemExit("PARITY FAILURE: table-free MSM differs from the table MSM")
        t1 = time.time(); tb = zk.Bases(ctx, 1, bases_limbs, window_bits=args.window_bits, precompute=True); table_s = time.time() - t1
        tb.free()
        fresh = {"device_ms_per_step": ms_f / max(3, args.steps // 2), "device_mops": n / (ms_f / max(3, args.steps // 2) * 1e-3) / 1e6, "window_bits": fb.window_bits,
                 "api": "zk_bases_upload(precompute = 0) + zk_msm_device: per-call bases, %d-bit windows, one bucket set per window" % fb.window_bits,
                 "table_build_s_incl_upload": table_s, "table_bytes": (255 // bases.window_bits + 1) * n * 96}
        fb.free()
    del bases_limbs

    # ---- closed-form check at EVERY N: bases are b_i * G, so the folded result must be (sum_ranks sum_i s_i b_i mod r) * G ----
    last_set = (W + args.steps - 1) % N_SETS
    parts = gather_ints(dist, torch, world, dot_mod_r(h_sets[last_set], base_scalars))
    closed_ok = None
    if rank == 0:
        closed_ok = closed_form_g1(sum(parts)) == res_dev
        if not closed_ok:
            raise SystemExit("PARITY FAILURE: MSM result differs from the closed form (sum s_i b_i) * G")
        if args.dump_outputs:
            os.makedirs(args.dump_outputs, exist_ok=True)
            np.save(os.path.join(args.dump_outputs, "g1_msm.npy"), np.frombuffer(res_dev, np.uint8).astype(np.float64))

    total_terms = n * world
    value = total_terms * args.steps / (ms_dev * 1e-3) / 1e6
    e2e_value = total_terms * args.steps / (ms_e2e * 1e-3) / 1e6
    hbm_peak, hbm_how = peaks()
    acc_ms, acc_launches, acc_adds, acc_xyzz = prof
    acc_avg_s = acc_ms * 1e-3 / max(1, acc_launches)
    algo_modmul = ALGO_MODMUL_PER_TERM * n            # per launch: one launch processes one rank's n terms
    # bucket additions counted on the device: 10 products for those the XYZZ pass does, 6.4 for those of the batched-affine rounds
    # (6 per addition + the warp scans of the thread totals: 13 products per 32 additions)
    exec_modmul = (10.0 * acc_xyzz + 6.4 * (acc_adds - acc_xyzz)) / max(1, acc_launches)
    roofline = {
        "kernel": "bucket accumulation stage: zkmsm::k_ba_forward / k_ba_invert / k_ba_backward rounds + zkmsm::k_accumulate<Fq>",
        "additions_per_launch": {"total": acc_adds / max(1, acc_launches), "xyzz_pass": acc_xyzz / max(1, acc_launches)},
        "bound": "int32-modmul",                       # SURVEY.md §8(d): IMAD issue rate, not HBM, not tensor
        # LEAD figure: products the kernel actually executes / time / calibrated peak = efficiency of the integer-multiply pipe
        "executed_frac": exec_modmul / acc_avg_s / modmul_peak,
        "executed_modmul_per_launch": exec_modmul,
        "achieved": algo_modmul / acc_avg_s, "peak": modmul_peak, "unit": "Fq-modmul/s",
        "frac": algo_modmul / acc_avg_s / modmul_peak,
        "peak_how": "zk_bench_modmul: register-resident independent Fq Montgomery products, measured in this run",
        "avg_launch_ms": acc_avg_s * 1e3, "launches": acc_launches, "share_of_step": acc_ms / ms_b,
        "timed_in": "the blocking-call loop (one MSM at a time): CUDA events on the launching stream around the stage, incl. the ~0.2 ms serial inversion of each batched-affine round",
        "note": "frac uses SURVEY 8(d)'s FIXED algorithmic count (176 products per term = 11 x 16 windows) and can exceed 1 because "
                "the stage executes fewer (%d table rows per term with %d-bit windows; 10 products per XYZZ mixed addition, 6.4 per "
                "batched-affine addition); executed_frac counts the additions really performed (device counters) and is the pipe efficiency"
                % (255 // bases.window_bits + 1, bases.window_bits),
        "whole_msm_frac": ALGO_MODMUL_PER_TERM * total_terms * args.steps / (ms_dev * 1e-3) / (modmul_peak * world),
        "hbm": {"bound": "hbm", "achieved": ALGO_BYTES_PER_TERM * n / acc_avg_s / 1e9, "peak": hbm_peak, "unit": "GB/s",
                "frac": ALGO_BYTES_PER_TERM * n / acc_avg_s / 1e9 / hbm_peak, "peak_how": hbm_how},
        "traffic": None,
    }
    try:
        roofline["traffic"] = json.load(open(os.path.join(ROOT, "profiles", "traffic.json")))["k_accumulate_dram_bytes_per_launch"]
    except Exception:
        pass

    cpu_baseline = None
    if rank == 0 and world == 1 and not args.no_cpu:
        from oracle import coracle as co
        co.set_num_threads(host_cores())
        bl = co.g1_fixed_base(base_scalars)           # the same bases, made by the oracle's own fixed-base code
        _, tried = pick_threads(co, lambda: co.g1_msm(bl[:1 << 17], h_sets[last_set][:1 << 17]))
        t = time.time()
        want = co.g1_msm(bl, h_sets[last_set])
        dt = time.time() - t
        ok = co.g1_encode(want, False) == res_dev == res_e2e
        cpu_baseline = {"value": n / dt / 1e6, "unit": "Mop/s", "cores": co.num_threads(), "kind": "port",
                        "threads_busy": "<= %d (bellman's multiexp runs one task per window, c = ceil(ln n))" % (255 // 14 + 1),
                        "sample": "one full 2^%d-term MSM (same bases and scalars as the last timed GPU step), oracle/zk_oracle.c "
                                  "bellman-style Pippenger, %.2f s" % (args.log_n, dt),
                        "matches_gpu_result": bool(ok), "threads_tried_s": tried}
        del bl
        if not ok:
            raise SystemExit("PARITY FAILURE: GPU MSM result differs from the oracle")
    job.close()

    # ---- BASELINE config 5: fixed-total 2^24 MSM sharded over the ranks (strong scaling), closed-form checked ----
    strong = None
    if args.strong_log_n and args.secondary:
        try:
            strong = strong_scaling_leg(zk, sy, torch, dist, (ctx, ctx2), world, rank, local, args.strong_log_n, steps=3)
        except SystemExit:
            raise
        except Exception as e:
            strong = {"error": repr(e)}

    # batched proving at N > 1 is "replicas only" (SURVEY.md §8e): every rank proves its own 256-proof batch with a resident
    # CRS, no data-path collective; aggregate = all proofs / slowest rank
    replicas = None
    if world > 1 and args.secondary:
        try:
            g = prove_metrics(ctx, zk, sy, args, batch=256, steps=2, cpu=False, procs=max(2, min(24, host_cores() // world)))
            t = torch.tensor([g["ms_per_batch"], g["from_witness"]["ms_per_batch"]], dtype=torch.float64, device="cuda")
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            replicas = {"metric": g["metric"], "scaling": "weak (replicas, no collective)", "batch_per_gpu": 256,
                        "e2e_proofs_per_sec": world * 256 / (float(t[0]) * 1e-3), "from_witness_proofs_per_sec": world * 256 / (float(t[1]) * 1e-3),
                        "ms_per_batch_max_over_ranks": float(t[0]), "proofs_checked_per_rank": g["proofs_checked"]}
        except SystemExit:
            raise
        except Exception as e:
            replicas = {"error": repr(e)}
    if rank == 0:
        line = {
            "metric": "g1_msm_mops_2^%d" % args.log_n, "value": value, "unit": "Mop/s", "n_gpus": world, "steps": args.steps,
            "warmup": W, "ms_per_step": ms_dev / args.steps, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "u32-limb Montgomery (Fq 12x32, Fr 8x32), integer", "data": "synthetic",
            "config": {"workload": "G1 Pippenger MSM, 2^%d uniform-random subgroup bases per GPU (bases sharded by index range, "
                                   "partial sums all-gathered over NCCL), uniform Fr scalars" % args.log_n,
                       "window_bits": bases.window_bits, "precomputed_window_tables": True,
                       "l2_policy": "inputs larger than L2: %d distinct 32 MiB scalar vectors cycled, %.2f GiB window tables gathered randomly" % (N_SETS, (255 // bases.window_bits + 1) * n * 96 / 2**30),
                       "setup_s_untimed": round(setup_s, 2),
                       "pipelining": "two MSMs in flight on two contexts (futures), tail kernels on a high-priority stream"},
            "e2e": {"value": e2e_value, "unit": "Mop/s", "h2d_bytes_per_step": n * 32 * world, "d2h_bytes_per_step": 96 * world,
                    "ms_per_step": ms_e2e / args.steps,
                    "api": "zk_msm_begin / zk_msm_end (C ABI futures, scalars in pinned host memory, two in flight)" if world == 1 else
                           "H2D copy of the scalars + zk_msm_partial_device_begin + NCCL all-gather + zk_points_fold_begin / zk_msm_end, two in flight"},
            "gpu_launches": (KERNELS_PER_MSM + (1 if world > 1 else 0)) * args.steps * world,
            "clocks": clocks, "roofline": roofline, "cpu_baseline": cpu_baseline,
            "matches_closed_form": closed_ok,
            "closed_form": "result == (sum over ranks and terms of s_i * b_i mod r) * G with bases b_i * G; numpy dot products + oracle/pyref.py scalar multiple",
            "blocking_call": blocking,
        }
        if fresh is not None:
            line["blocking_call"]["fresh_bases"] = fresh
        sec = {}
        if args.secondary and world == 1:
            try:
                sec = secondary_metrics(ctx, zk, sy, args)
            except SystemExit:
                raise
            except Exception as e:      # the headline line must still print
                sec = {"error": repr(e)}
        if replicas is not None:
            sec["groth16_replicas"] = replicas
        if strong is not None:
            sec["msm_strong_scaling"] = strong
        if sec:
            line["secondary"] = sec
        print(json.dumps(line), flush=True)
    ctx2.close()
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    ctx.close()


def secondary_metrics(ctx, zk, sy, args):
    """NTT 2^22 and batched proving of the confidential_transfer-shaped circuit (short runs)."""
    import torch
    import ctypes as C
    from zero_chain_b200 import _lib
    out = {}
    stream = torch.cuda.ExternalStream(ctx.stream)
    # Fr NTT 2^22, device resident
    logn = 22
    d = torch.from_numpy(sy.random_fr_limbs(1 << logn, 5).view(np.int64)).cuda()
    torch.cuda.synchronize()
    L = _lib.lib()
    for _ in range(3):
        L.zk_ntt_fr_device(ctx._h, C.c_void_p(d.data_ptr()), logn, 0)
    ctx.sync()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(stream)
    reps = 10
    for _ in range(reps):
        L.zk_ntt_fr_device(ctx._h, C.c_void_p(d.data_ptr()), logn, 0)
    e1.record(stream)
    ctx.sync(); torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / reps
    fr_peak, _ = zk.bench_modmul(ctx, zk.FIELD_FR, 148 * 4, 256, 3000)
    out["ntt_fr_2^22"] = {"ms": ms, "melem_per_s": (1 << logn) / ms / 1e3, "algo_modmul_frac": (1 << (logn - 1)) * logn / (ms * 1e-3) / fr_peak,
                          "fr_modmul_peak": fr_peak}
    out["g2_msm"] = g2_msm_metrics(ctx, zk, sy, torch)
    out["groth16"] = prove_metrics(ctx, zk, sy, args)
    return out


def g2_msm_metrics(ctx, zk, sy, torch):
    """G2 MSM roofline (SURVEY.md §8d: 528 n Fq-modmul per n-term G2 MSM = 11 Fq2 products x 3 x 16 windows): one MSM of 2^17
    uniform-random G2 bases with window tables (device-resident scalars, blocking calls), and the prover's own size (12 404 terms,
    256 scalar vectors against one table = the B-query MSM of a 256-proof batch).  Self-check without curve code on the host: the
    same MSM through tables of another window size (a different bucket structure over the same group elements) must give the same
    bytes; parity with the oracle at these sizes is in tests/test_gpu_field_msm.py and tests/test_gpu_batched_affine.py."""
    stream = torch.cuda.ExternalStream(ctx.stream)
    fq_peak, _ = zk.bench_modmul(ctx, zk.FIELD_FQ, 148 * 4, 256, 3000)
    out = {}
    for tag, n, batch in (("2^17", 1 << 17, 1), ("prover_b_query_x256", 12404, 256)):
        bl = zk.scalar_mul_many(ctx, 2, zk.G2_GENERATOR, sy.random_fr_limbs(n, 41))
        b = zk.Bases(ctx, 2, bl, precompute=True)
        d = torch.from_numpy(sy.random_fr_limbs(n * batch, 42).view(np.int64)).cuda()
        torch.cuda.synchronize()
        for _ in range(2):
            ref = zk.multiexp_device(b, d.data_ptr(), n, batch)
        ctx.profile(True)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        reps = 5
        e0.record(stream)
        for _ in range(reps):
            got = zk.multiexp_device(b, d.data_ptr(), n, batch)
        e1.record(stream)
        ctx.sync(); torch.cuda.synchronize()
        ms = e0.elapsed_time(e1) / reps
        _, g2_adds, _, g2_xyzz = ctx.profile_counts()
        ctx.profile(False)
        other = zk.Bases(ctx, 2, bl, window_bits=max(4, b.window_bits - 3), precompute=True)
        same = zk.multiexp_device(other, d.data_ptr(), n, batch) == got == ref
        other.free(); b.free()
        if not same:
            raise SystemExit("PARITY FAILURE: G2 MSM results differ between window sizes")
        terms = n * batch
        out[tag] = {"terms": terms, "ms": ms, "mops": terms / ms / 1e3, "window_bits": b.window_bits,
                    "frac": 528.0 * terms / (ms * 1e-3) / fq_peak,
                    "executed_frac": (28.0 * g2_xyzz + 17.6 * (g2_adds - g2_xyzz)) / reps / (ms * 1e-3) / fq_peak,
                    "executed_modmul": (28.0 * g2_xyzz + 17.6 * (g2_adds - g2_xyzz)) / reps, "consistent_across_window_sizes": True}
    out["unit"] = "Fq-modmul/s against the calibrated Fq peak"; out["peak"] = fq_peak
    out["note"] = "frac: SURVEY 8(d) convention 528 n; executed_frac: 28 Fq products per G2 XYZZ addition (8 Fq2 products + 2 squarings), 17.6 per batched-affine one, x additions counted on the device; bucket reduction not counted"
    return out


def prove_metrics(ctx, zk, sy, args, batch=256, steps=3, cpu=True, procs=None):
    """proofs/sec for the confidential_transfer-shaped synthetic circuit (SURVEY.md §8d C4): a batch of 256 DISTINCT witnesses
    in pinned host memory -> zk_groth16_prove_batch (one C-ABI call per step, H2D of every witness and D2H of the proofs inside
    the timed region).  EVERY proof of the batch is compared with the closed-form proof of its witness (trapdoor algebra + big-integer
    curve arithmetic, computed in host worker processes), the first 8 also with the oracle's create_proof (the CPU baseline)."""
    import torch
    r1cs = sy.make_r1cs(seed=1, **sy.CONF_SHAPE)
    dens = sy.densities(r1cs)
    g1 = lambda s: zk.scalar_mul_many(ctx, 1, zk.G1_GENERATOR, s)
    g2 = lambda s: zk.scalar_mul_many(ctx, 2, zk.G2_GENERATOR, s)
    crs = sy.make_toy_crs(r1cs, g1, g2, seed=2)                      # toy CRS (known trapdoor), exact Parameters::write bytes
    t = time.time()
    params = zk.Parameters.read(ctx, crs.params_bytes, checked=True)
    load_s = time.time() - t
    t = time.time()
    wit = make_witnesses(crs, batch, procs or min(24, host_cores()))
    wit_s = time.time() - t
    bufs = [torch.from_numpy(np.stack([w[1][j] for w in wit]).view(np.int64)).pin_memory() for j in range(5)]
    views = [t_.numpy().view(np.uint64) for t_ in bufs]
    rs = sy.ints_to_limbs([w[2] for w in wit]); ss = sy.ints_to_limbs([w[3] for w in wit])
    want_all = b"".join(w[4] for w in wit)
    h2d = sum(v.nbytes for v in views) + rs.nbytes + ss.nbytes
    zk.create_proof_batch_raw(params, batch, *views, *dens, rs, ss)          # warm-up (allocations, NTT tables)
    zk.create_proof_batch_raw(params, batch, *views, *dens, rs, ss)
    ctx.profile(True)                                                        # restarts the device-side work counters
    t = time.perf_counter()
    for _ in range(steps):
        proofs = zk.create_proof_batch_raw(params, batch, *views, *dens, rs, ss)
    dt = (time.perf_counter() - t) / steps
    g1_adds, g2_adds, g1_xyzz, g2_xyzz = ctx.profile_counts()
    acc_ms, acc_launches = ctx.profile_read()
    ctx.profile(False)
    bad = [k for k in range(batch) if proofs[192 * k:192 * (k + 1)] != want_all[192 * k:192 * (k + 1)]]
    if bad:
        raise SystemExit("PARITY FAILURE: %d of %d GPU proofs differ from the closed form (first: %d)" % (len(bad), batch, bad[0]))
    # roofline of the batch: work the kernels EXECUTE, in Fq-product equivalents, against the calibrated integer-multiply peak
    fq_peak, _ = zk.bench_modmul(ctx, zk.FIELD_FQ, 148 * 4, 256, 3000)
    fr_peak, _ = zk.bench_modmul(ctx, zk.FIELD_FR, 148 * 4, 256, 3000)
    log_m = 15
    ntt_fr = 7 * (1 << (log_m - 1)) * log_m                                   # 7 transforms of 2^15 per proof, (m/2) log m butterflies each
    per_proof = {"g1_bucket_additions": g1_adds / (steps * batch), "g2_bucket_additions": g2_adds / (steps * batch),
                 "g1_left_to_xyzz_pass": g1_xyzz / (steps * batch), "g2_left_to_xyzz_pass": g2_xyzz / (steps * batch), "ntt_fr_modmul": ntt_fr}
    g1a, g1x, g2a, g2x = (per_proof[k] for k in ("g1_bucket_additions", "g1_left_to_xyzz_pass", "g2_bucket_additions", "g2_left_to_xyzz_pass"))
    exec_fq = 10.0 * g1x + 6.4 * (g1a - g1x) + 28.0 * g2x + 17.6 * (g2a - g2x) + ntt_fr * fq_peak / fr_peak
    algo_fq = 176.0 * 80722 + 528.0 * 12402 + ntt_fr * fq_peak / fr_peak          # SURVEY 8(d): per-proof algorithmic convention
    roofline = {"bound": "int32-modmul", "unit": "Fq-modmul/s", "peak": fq_peak,
                "executed_modmul_per_proof": exec_fq, "executed_frac": exec_fq * batch / dt / fq_peak,
                "achieved": algo_fq * batch / dt, "frac": algo_fq * batch / dt / fq_peak, "per_proof": per_proof,
                "g1_accumulate_share_of_batch": acc_ms * 1e-3 / steps / dt,
                "note": "executed = 10 Fq products per G1 XYZZ addition, 6.4 per G1 batched-affine addition, 28 / 17.6 for G2 (Fq2 product = 3 Fq "
                        "products, square = 2) + NTT butterflies scaled by the Fr/Fq product cost; additions are counted on the device (non-zero digits), bucket "
                        "reductions, blinding multiplications and encodings are NOT counted (conservative).  frac uses SURVEY 8(d)'s fixed "
                        "176 n / 528 n convention, which over-counts the 0/1 witness scalars"}
    # two batches in flight: a second context (own streams and workspace, same resident CRS) driven by a second host thread, so
    # the upload of one batch and the latency-bound tails of its MSMs overlap the other's kernels (ctypes releases the GIL)
    two = None
    try:
        import threading
        ctx_b = zk.Context(ctx.device)
        params_b = zk.Parameters(ctx_b, params._h, [params.n_ic, params.n_h, params.n_l, params.n_a, params.n_b_g1, params.n_b_g2])
        outs = [None, None]

        def worker(i, prm, reps):
            for _ in range(reps):
                outs[i] = zk.create_proof_batch_raw(prm, batch, *views, *dens, rs, ss)
        worker(1, params_b, 1)                                          # warm-up of the second context (allocations, lanes)
        th = [threading.Thread(target=worker, args=(i, prm, steps)) for i, prm in enumerate((params, params_b))]
        t = time.perf_counter()
        for x in th:
            x.start()
        for x in th:
            x.join()
        dt2 = (time.perf_counter() - t) / (2 * steps)
        if outs[0] != proofs or outs[1] != proofs:
            raise SystemExit("PARITY FAILURE: proofs made with two batches in flight differ")
        two = {"e2e_proofs_per_sec": batch / dt2, "ms_per_batch": dt2 * 1e3, "batches_in_flight": 2,
               "how": "two contexts on one GPU, one host thread each, blocking zk_groth16_prove_batch calls"}
        params_b._h = None                                              # the handle belongs to `params`
        ctx_b.close()
    except SystemExit:
        raise
    except Exception as e:
        two = {"error": repr(e)}
    # same batch straight from the assignments: the fixed constraint system is resident on the device and the GPU
    # evaluates <A_j,z>, <B_j,z>, <C_j,z> itself (zk_groth16_prove_witness_batch; SURVEY.md §8 f4)
    cs = zk.ConstraintSystem(ctx, r1cs.n_inputs, r1cs.n_aux, r1cs.A, r1cs.B, r1cs.C)
    zk.create_proof_from_witness_batch(cs, params, batch, views[3], views[4], rs, ss)
    t = time.perf_counter()
    for _ in range(steps):
        proofs_w = zk.create_proof_from_witness_batch(cs, params, batch, views[3], views[4], rs, ss)
    dt_w = (time.perf_counter() - t) / steps
    if proofs_w != proofs:
        raise SystemExit("PARITY FAILURE: witness-path proofs differ from the evaluation-path proofs")
    h2d_w = views[3].nbytes + views[4].nbytes + rs.nbytes + ss.nbytes
    cs.free()
    lat = 1e9
    for _ in range(4):                   # first call loads the single-domain kernels lazily; report the steady-state latency
        t = time.perf_counter()
        single = zk.create_proof_batch_raw(params, 1, *[v[:1] for v in views], *dens, rs[:1], ss[:1])
        lat = min(lat, time.perf_counter() - t)
    assert single == proofs[:192]
    # CPU port of the reference path on the same CRS / witnesses: the first 8 proofs of the batch, each compared byte for byte
    cpu_block = None
    if cpu:
        from oracle import coracle as co
        op = co.Params(crs.params_bytes, checked=False)
        n_cpu = min(8, batch)
        to_int = lambda row: sum(int(x) << (64 * i) for i, x in enumerate(row))
        _, tried = pick_threads(co, lambda: op.prove(*[v[0] for v in views], *dens, to_int(rs[0]), to_int(ss[0])))
        t = time.perf_counter()
        cpu_proofs = [op.prove(*[v[k] for v in views], *dens, to_int(rs[k]), to_int(ss[k])) for k in range(n_cpu)]
        cpu_dt = (time.perf_counter() - t) / n_cpu
        if b"".join(cpu_proofs) != proofs[:192 * n_cpu]:
            raise SystemExit("PARITY FAILURE: GPU proof bytes differ from the oracle")
        cpu_block = {"value": 1.0 / cpu_dt, "unit": "proofs/s", "cores": co.num_threads(), "kind": "port",
                     "sample": "oracle create_proof on the first %d witnesses of the batch, one after the other, same CRS" % n_cpu,
                     "matches_gpu_proof_bytes": True, "threads_tried_s": tried}
    params.free()
    try:
        verify_block = verify_metrics(ctx, zk, crs.params_bytes, proofs, np.ascontiguousarray(views[3][:, 1:, :]), cpu)
    except SystemExit:
        raise
    except Exception as e:
        verify_block = {"error": repr(e)}
    return {"metric": "proofs_per_sec (confidential_transfer shape: 19974 constraints, 23 inputs, domain 2^15; synthetic R1CS, toy CRS)",
            "e2e_proofs_per_sec": batch / dt, "batch": batch, "steps": steps, "ms_per_batch": dt * 1e3, "h2d_bytes_per_step": int(h2d),
            "d2h_bytes_per_step": 192 * batch, "single_proof_latency_ms": lat * 1e3, "params_load_checked_s": load_s,
            "from_witness": {"e2e_proofs_per_sec": batch / dt_w, "ms_per_batch": dt_w * 1e3, "h2d_bytes_per_step": int(h2d_w),
                             "api": "zk_groth16_prove_witness_batch (constraint system resident, GPU evaluates the R1CS rows)"},
            "two_batches_in_flight": two, "cpu_baseline": cpu_block, "verify": verify_block, "roofline": roofline,
            "proofs_checked": batch, "distinct_witnesses": batch, "witness_generation_s_untimed": wit_s,
            "check": "every proof of the batch == closed-form proof of its witness (trapdoor algebra + oracle/pyref.py); first 8 == oracle create_proof",
            "timing": "host wall clock around synchronous C-ABI calls (each call ends with a stream synchronise)"}


def verify_metrics(ctx, zk, vk_bytes, proofs, inputs, cpu=True, n_v=8192):
    """verifications/sec (SURVEY.md §8 f2): the proofs the prover just made, replicated to a block-import sized batch, through
    zk_groth16_verify_batch (host buffers: H2D of proofs + public inputs, D2H of the verdicts inside the timed region) and
    zk_groth16_verify_batch_device (resident inputs, CUDA events on the library's stream); CPU: the oracle's verify_proof."""
    import torch
    import ctypes as C
    from zero_chain_b200 import _lib
    L = _lib.lib()
    t = time.perf_counter()
    pvk = zk.PreparedVerifyingKey.prepare(ctx, vk_bytes)
    prep_s = time.perf_counter() - t
    batch = len(proofs) // 192
    n_in = inputs.shape[1]
    reps = (n_v + batch - 1) // batch
    pb = np.tile(np.frombuffer(proofs, np.uint8), reps)[:192 * n_v].copy()
    inp = np.tile(inputs.reshape(batch, -1), (reps, 1))[:n_v].copy()
    hp, hi = torch.from_numpy(pb).pin_memory(), torch.from_numpy(inp.view(np.int64)).pin_memory()
    out = np.zeros(n_v, np.uint8)
    call = lambda: zk._ck(L.zk_groth16_verify_batch(ctx._h, pvk._h, n_v, C.c_void_p(hp.data_ptr()), C.c_void_p(hi.data_ptr()), n_in,
                                                    out.ctypes.data_as(C.c_void_p)))
    call()
    best = 1e9
    for _ in range(3):
        t = time.perf_counter(); call(); best = min(best, time.perf_counter() - t)
    if not (out == 1).all():
        raise SystemExit("PARITY FAILURE: the GPU verifier rejected a proof made by the GPU prover")
    dp, di = hp.cuda(), hi.cuda()
    dv = torch.zeros(n_v, dtype=torch.uint8, device="cuda")
    stream = torch.cuda.ExternalStream(ctx.stream)
    torch.cuda.synchronize()
    dev = lambda: zk.verify_proofs_device(pvk, n_v, dp.data_ptr(), di.data_ptr(), n_in, dv.data_ptr())
    dev(); ctx.sync()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(stream)
    for _ in range(3):
        dev()
    e1.record(stream)
    ctx.sync(); torch.cuda.synchronize()
    ms_dev = e0.elapsed_time(e1) / 3
    assert bool((dv == 1).all())
    # a tampered copy: one public input bumped in every 5th proof -> exactly those are rejected
    bad = inp.copy(); bad[::5, 0] ^= 1
    hb = torch.from_numpy(bad.view(np.int64))
    zk._ck(L.zk_groth16_verify_batch(ctx._h, pvk._h, n_v, C.c_void_p(hp.data_ptr()), C.c_void_p(hb.data_ptr()), n_in, out.ctypes.data_as(C.c_void_p)))
    want = np.ones(n_v, np.uint8); want[::5] = 0
    if not (out == want).all():
        raise SystemExit("PARITY FAILURE: the GPU verifier accepted a proof with a wrong public input")
    cpu_block = None
    if cpu:
        from oracle import coracle as co
        k = co.PreparedVerifyingKey.prepare(vk_bytes)
        if k.write() != pvk.write():
            raise SystemExit("PARITY FAILURE: prepared verifying key differs from the oracle's")
        n_c = 8 * co.num_threads()
        t = time.perf_counter(); v = k.verify_batch(pb[:192 * n_c].tobytes(), bad[:n_c], n_in); cpu_dt = time.perf_counter() - t
        if v != [int(x) for x in want[:n_c]]:
            raise SystemExit("PARITY FAILURE: oracle verdicts differ from the GPU's")
        cpu_block = {"value": n_c / cpu_dt, "unit": "verifications/s", "cores": co.num_threads(), "kind": "port",
                     "sample": "%d proofs (every 5th with a wrong input), oracle/pairing_oracle.inc verify_proof, %.2f s" % (n_c, cpu_dt),
                     "matches_gpu_verdicts": True}
    pvk.free()
    return {"metric": "verifications_per_sec (Proof::read + verify_proof, %d public inputs, one prepared key)" % n_in, "batch": n_v,
            "e2e_verifications_per_sec": n_v / best, "e2e_ms_per_batch": best * 1e3, "h2d_bytes_per_step": int(pb.nbytes + inp.nbytes),
            "d2h_bytes_per_step": n_v, "device_verifications_per_sec": n_v / (ms_dev * 1e-3), "device_ms_per_batch": ms_dev,
            "prepare_verifying_key_s": prep_s, "cpu_baseline": cpu_block}


def run_reference(args):
    """Reference arm: the reference's own CPU algorithm for the path — the restatement of bellman's multiexp / create_proof in
    oracle/zk_oracle.c (the reference itself is Rust and cannot be built here: no cargo/rustc, bellman un-vendored) — on ALL host
    threads of the box, on the SAME config as our arm at this N: one MSM of N * 2^log_n terms per step (weak scaling: the
    GPUs' shards together are one MSM of that size; the CPU does not get faster with more GPUs)."""
    world, rank = env_int("WORLD_SIZE", 1), env_int("RANK", 0)
    if rank != 0:
        return
    from oracle import coracle as co
    from zero_chain_b200 import synthetic as sy
    co.build()
    co.set_num_threads(host_cores())       # torchrun exports OMP_NUM_THREADS=1: the team size is set explicitly, never taken from the environment
    n = (1 << args.log_n) * max(1, args.gpus)
    bs = sy.random_fr_limbs(n, 7)
    bs[:, 1:] = 0                          # bases b_i * G with 64-bit b_i: 4x cheaper to generate on the CPU; the cost of an MSM does not depend on them
    t0 = time.time()
    bases = co.g1_fixed_base(bs)
    setup_s = time.time() - t0
    sets = [sy.random_fr_limbs(n, 1000 + k) for k in range(2)]
    cores, tried = pick_threads(co, lambda: co.g1_msm(bases[:1 << 17], sets[0][:1 << 17]))
    t0 = time.time()
    co.g1_msm(bases, sets[0])              # first warm-up step, also sizes the run
    t1 = time.time() - t0
    warmup = max(1, min(args.warmup, int(30.0 / t1)))
    steps = args.steps
    for k in range(1, warmup):
        co.g1_msm(bases, sets[k % 2])
    t0 = time.time()
    for k in range(steps):
        co.g1_msm(bases, sets[(warmup + k) % 2])
    dt = time.time() - t0
    value = n * steps / dt / 1e6
    c_win = max(3, int(np.ceil(np.log(n))))
    busy = 255 // c_win + 1
    sample = "full config: %d-term MSM per step (N * 2^%d), %d timed steps after %d warm-up (requested %d warm-up, bounded to ~30 s)" % (
        n, args.log_n, steps, warmup, args.warmup)
    line = {"impl": "reference", "metric": "g1_msm_mops_2^%d" % args.log_n, "value": value, "unit": "Mop/s", "n_gpus": args.gpus,
            "steps": steps, "warmup": warmup, "steps_requested": args.steps, "ms_per_step": dt * 1e3 / steps, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "u64-limb Montgomery, integer", "data": "synthetic",
            "config": {"workload": "G1 Pippenger MSM, 2^%d bases per GPU x %d = %d terms in one MSM on the host CPU (bellman multiexp restatement, "
                                   "c = ceil(ln n) = %d, one task per window)" % (args.log_n, max(1, args.gpus), n, c_win),
                       "threads": cores, "threads_tried_s": tried, "threads_busy": "<= %d (one task per window, as bellman's multiexp schedules it)" % busy,
                       "setup_s_untimed": round(setup_s, 2)},
            "cpu_baseline": {"value": value, "unit": "Mop/s", "cores": cores, "kind": "port", "sample": sample},
            "e2e": {"value": value, "unit": "Mop/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    if args.secondary:
        try:
            line["secondary"] = {"groth16": reference_prove_metrics(co, sy)}
        except Exception as e:
            line["secondary"] = {"error": repr(e)}
    print(json.dumps(line), flush=True)


def reference_prove_metrics(co, sy):
    """proofs/sec of the CPU restatement of create_proof on the confidential_transfer-shaped synthetic circuit (same R1CS, toy CRS
    seeds and witness seeds as our arm's secondary.groth16), all host threads, one proof after the other (zface proves one at a time)."""
    r1cs = sy.make_r1cs(seed=1, **sy.CONF_SHAPE)
    dens = sy.densities(r1cs)
    crs = sy.make_toy_crs(r1cs, co.g1_fixed_base, co.g2_fixed_base, seed=2)
    op = co.Params(crs.params_bytes, checked=False)
    _wk_init(crs)
    wit = [_wk_witness(k) for k in range(4)]
    cores, tried = pick_threads(co, lambda: op.prove(*wit[0][1], *dens, wit[0][2], wit[0][3]))
    t = time.perf_counter()
    out = [op.prove(*w[1], *dens, w[2], w[3]) for w in wit]
    dt = (time.perf_counter() - t) / len(wit)
    ok = all(o == w[4] for o, w in zip(out, wit))
    return {"metric": "proofs_per_sec (confidential_transfer shape: 19974 constraints, 23 inputs, domain 2^15; synthetic R1CS, toy CRS)",
            "e2e_proofs_per_sec": 1.0 / dt, "ms_per_proof": dt * 1e3, "cores": cores, "threads_tried_s": tried, "proofs": len(wit),
            "matches_closed_form": bool(ok)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--log-n", dest="log_n", type=int, default=LOG_N)
    ap.add_argument("--window-bits", dest="window_bits", type=int, default=0, help="0 = library default (20 bits from 2^20 terms, else <= 16)")
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline leg")
    ap.add_argument("--no-secondary", dest="secondary", action="store_false")
    ap.add_argument("--affine-min-entries", dest="affine_min_entries", type=int, default=None, help="zk_ctx_set_opt(ZK_OPT_AFFINE_MIN_ENTRIES) on the bench contexts")
    ap.add_argument("--affine-levels", dest="affine_levels", type=int, default=-1)
    ap.add_argument("--strong-log-n", dest="strong_log_n", type=int, default=24,
                    help="total terms (log2) of the fixed-total sharded MSM of secondary.msm_strong_scaling (BASELINE config 5); 0 = skip")
    ap.add_argument("--dump-outputs", dest="dump_outputs", metavar="DIR", default=None,
                    help="write the result of the last timed step as DIR/g1_msm.npy (float64)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the results of --impl ours")
    args.warmup = max(3, args.warmup)
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
