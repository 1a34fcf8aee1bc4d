#!/usr/bin/env python
"""bench.py -- MultiExp (MSM) throughput on B200, per the driver contract.

  python bench.py --gpus N --steps K --warmup W            # ours (CUDA engine through the C ABI)
  python bench.py --impl reference --gpus N --steps K ...  # the reference algorithm's CPU path (C port)
  python bench.py ... --dump-outputs DIR                   # also write the last timed result to DIR/msm_result.npy

A "step" is one bn254 G1 MultiExp over one batch of synthetic inputs.  Metric: scalar-muls/s = n_total / time.
  N = 1   BASELINE.json configs[1]: n = 2^24, window width from the engine's model.
  N > 1   BASELINE.json configs[4]: n = 2^26 in TOTAL, sharded contiguously over the N ranks ("strong"); per-rank window
          partials, one NCCL all-gather of W partial points, finalize on every rank.  The weak-scaling figure (2^24 per
          GPU) is reported beside it under "weak".
  value : inputs already resident in HBM, CUDA events, max over ranks
  e2e   : the reference-facing call with HOST buffers (pinned), H2D of points+scalars and D2H of the result inside the
          timed region (N = 1: gmsm_multiexp one-shot drop-in); e2e_pageable: the same call on ordinary (pageable) numpy
          arrays, which is what a Go caller hands over
  parity: the TIMED result is checked at full size against the closed form [sum_i (start+i) s_i] B evaluated by the
          CPU oracle (checker only) -- every curve, every N
  roofline : the accumulate kernel (bucket pass) against the measured HBM peak (the mandated yardstick) and against
          the INT32 multiplier pipe, the unit that actually binds
  cpu_baseline : the oracle's C port of the reference algorithm on the host cores
Extra sub-objects of the N = 1 line: configs[2] (bls12-381 G1 2^24), configs[3] (bn254 G2 2^22), the metric's 2^20 and
2^26 points, the reference's skewed scalar distributions, three concurrent calls.
"""
import argparse
import importlib
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

CURVE_BITS = {"bn254_g1": 254, "bn254_g2": 254, "bls12381_g1": 255, "bls12381_g2": 255, "bls12377_g1": 253, "bls12377_g2": 253,
              "secp256k1_g1": 256, "bw6761_g1": 377, "bw6761_g2": 377, "bls24315_g1": 253, "bls24317_g1": 255, "bw6633_g1": 315,
              "bw6633_g2": 315}
AFF_BYTES = {"bn254_g1": 64, "bn254_g2": 128, "bls12381_g1": 96, "bls12381_g2": 192, "bls12377_g1": 96, "bls12377_g2": 192,
             "secp256k1_g1": 64, "bw6761_g1": 192, "bw6761_g2": 192, "bls24315_g1": 80, "bls24317_g1": 80, "bw6633_g1": 160,
             "bw6633_g2": 160}
FP2_GROUPS = ("bn254_g2", "bls12381_g2", "bls12377_g2")       # coordinates in Fp2 (G2 of bw6-761 is over Fp)
FR_MOD = {
    256: 0xFFFFFFFFFFFFFFFFFFFFFFFFFFFFFFFEBAAEDCE6AF48A03BBFD25E8CD0364141,
    377: 0x1AE3A4617C510EAC63B05C06CA1493B1A22D9F300F5138F1EF3622FBA094800170B5D44300000008508C00000000001,
    254: 0x30644E72E131A029B85045B68181585D2833E84879B9709143E1F593F0000001,
    255: 0x73EDA753299D7D483339D80809A1D80553BDA402FFFE5BFEFFFFFFFF00000001,
    253: 0x12AB655E9A2CA55660B44D1E5C37B00159AA76FED00000010A11800000000001,
}
# scalar-field moduli that share a bit length with one of the above (bls24-315: 253 bits like bls12-377, bls24-317: 255 like
# bls12-381) are looked up by group first
FR_Q = {
    "bls24315_g1": 0x196DEAC24A9DA12B25FC7EC9CF927A98C8C480ECE644E36419D0C5FD00C00001,
    "bls24317_g1": 0x443F917EA68DAFC2D0B097F28D83CD491CD1E79196BF0E7AF000000000000001,
    "bw6633_g1": 0x4C23A02B586D650D3F7498BE97C5EAFDEC1D01AA27A1AE0421EE5DA52BDE5026FE802FF40300001,
    "bw6633_g2": 0x4C23A02B586D650D3F7498BE97C5EAFDEC1D01AA27A1AE0421EE5DA52BDE5026FE802FF40300001,
}


def fr_mod(g):
    """the scalar-field modulus of a group"""
    return FR_Q.get(g) or FR_MOD[CURVE_BITS[g]]


BASE_MULT = 0xC0FFEE            # the synthetic bases are [start + i] * B with B = [BASE_MULT] * generator
STAGE_NAMES = ["digits_hist", "scan", "scatter", "accumulate", "carries", "bucket_reduce", "finalize", "total"]


def ncores():
    try:
        return len(os.sched_getaffinity(0))
    except Exception:
        return os.cpu_count() or 1


def scalar_words(bits):
    """fr.Limbs: u64 words of one scalar"""
    return (bits + 63) // 64


def synth_scalars(n, bits, seed, q=None):
    """n uniform values < r as fr.Limbs x u64 limbs (mask top limb to fr.Bits, rejection-sample), read as
    the Montgomery representation -- the analogue of fr.SetRandom (fr/element.go:302-343)."""
    rng = np.random.default_rng(seed)
    q = q or FR_MOD[bits]
    nw = scalar_words(bits)
    ql = [np.uint64((q >> (64 * i)) & (2**64 - 1)) for i in range(nw)]
    out = np.empty((n, nw), dtype=np.uint64)
    todo = np.arange(n)
    top = np.uint64((1 << (bits - 64 * (nw - 1))) - 1)
    while todo.size:
        v = rng.integers(0, 2**64, size=(todo.size, nw), dtype=np.uint64)
        v[:, nw - 1] &= top
        lt = np.zeros(todo.size, dtype=bool)
        eq = np.ones(todo.size, dtype=bool)
        for k in range(nw - 1, -1, -1):
            lt |= eq & (v[:, k] < ql[k])
            eq &= v[:, k] == ql[k]
        out[todo[lt]] = v[lt]
        todo = todo[~lt]
    return out


def skew_scalars(s, kind):
    """the reference benchmark's two skewed distributions (ecc/bn254/multiexp_test.go:316-334), applied to a copy"""
    s = s.copy()
    if kind == "smallvalues":          # every 5th scalar: SetZero(); [0] = 1  -- n/5 identical scalars
        s[::5, :] = 0
        s[::5, 0] = 1
    elif kind == "redundancy":         # runs of 100 equal scalars
        n = s.shape[0]
        heads = s[::100]
        s[:] = np.repeat(heads, 100, axis=0)[:n]
    else:
        raise ValueError(kind)
    return s


def dot_index_mod(limbs, start, r):
    """sum_i (start + i) * limbs_i mod r, limbs_i read as a little-endian integer of fr.Limbs words (numpy block sums of
    14-bit x 32-bit products, Python integers only for the block totals)."""
    n = limbs.shape[0]
    nh = 2 * limbs.shape[1]
    halves = np.ascontiguousarray(limbs, dtype=np.uint64).view(np.uint32).reshape(n, nh)
    total = 0
    SUP, CH = 1 << 20, 1 << 16
    for a in range(0, n, SUP):
        b = min(n, a + SUP)
        hv = halves[a:b].astype(np.uint64)
        idx = np.arange(start + a, start + b, dtype=np.uint64)
        for shift in (0, 14, 28):
            part = (idx >> np.uint64(shift)) & np.uint64(0x3FFF)
            if not part.any():
                continue
            prod = hv * part[:, None]
            sums = np.add.reduceat(prod, np.arange(0, b - a, CH), axis=0)      # each < 2^16 * 2^14 * 2^32 = 2^62
            for k in range(nh):
                total += sum(int(x) for x in sums[:, k]) << (32 * k + shift)
    return total % r


class ClockSampler:
    """nvidia-smi clocks / throttle reasons DURING the timed region (B200_PROFILING.md recipe)"""

    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.gpu = gpu_index
        self.proc = None
        self.lines = []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "--query-gpu=" + self.Q, "--format=csv,noheader,nounits", "-lms", "50",
                                          "-i", str(self.gpu)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for ln in self.proc.stdout:
            self.lines.append(ln.strip())

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1]))
                mx.append(float(f[2]))
            except ValueError:
                continue
            for nm, val in zip(names, f[5:9]):
                if val.lower().startswith("active"):
                    reasons.add(nm)
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no samples"]}
        return {"sm_mhz": float(np.median(sm)), "sm_max_mhz": float(max(mx)), "reasons": sorted(reasons), "samples": len(sm)}


def int_pipe_fraction(g, mixed_adds_per_s, sm_mhz, wide_mads_per_mixed_add=None):
    """The binding unit of the bucket pass is the INT32 multiplier (DESIGN.md section 5): one mixed addition is 8 M + 2 S in
    the coordinate field = 10 Fp multiplications for G1, 28 for G2 (Fp2: M = 3, S = 2 Fp multiplications), each 2N^2 + N
    IMAD.WIDE (N 32-bit limbs) in the textbook count; an SM sub-partition issues one IMAD.WIDE warp-instruction every 4
    cycles: 148 SMs x 32 wide MADs per clock.  `wide_mads_per_mixed_add` overrides the textbook count with the one the
    built kernel really executes (dedicated squaring / fused products lower it).
    Returns {"wide_mads_per_s", "peak", "frac"}, or None if the clock is unknown."""
    try:
        limbs = AFF_BYTES[g] // (16 if g in FP2_GROUPS else 8)        # 32-bit limbs of one Fp element
        fp_muls = 28 if g in FP2_GROUPS else 10
        per_add = wide_mads_per_mixed_add or fp_muls * (2 * limbs * limbs + limbs)
        peak = 148 * 32 * float(sm_mhz) * 1e6
        ach = float(mixed_adds_per_s) * per_add
        return {"wide_mads_per_mixed_add": per_add, "wide_mads_per_s": ach, "peak": peak, "frac": ach / peak,
                "peak_source": "148 SMs x 32 IMAD.WIDE/clk at the sampled SM clock"}
    except Exception:
        return None


def measured_hbm_peak():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    try:
        return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json, burst copy)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md)"


def metric_name(g):
    return "bn254 G1 MultiExp scalar-muls/s" if g == "bn254_g1" else g + " MultiExp scalar-muls/s"


def workload_name(g, logn_total, world):
    tag = ""
    if g == "bn254_g1" and logn_total == 24 and world == 1:
        tag = " (BASELINE configs[1])"
    if g == "bn254_g1" and logn_total == 26 and world > 1:
        tag = " (BASELINE configs[4])"
    return "%s MultiExp n=2^%d total over %d GPU(s)%s, random scalars, on-curve bases [i]B" % (g, logn_total, world, tag)


def _generator_limbs(g):
    """group generators in Go memory layout (Montgomery limbs), precomputed from
    ecc/bn254/bn254.go:111-119 and ecc/bls12-381/bls12-381.go:107-116 by tools/gen_generators.py"""
    tab = json.load(open(os.path.join(ROOT, "gnark-crypto_b200", "generators.json")))
    return np.array([int(x, 16) for x in tab[g]], dtype=np.uint64)


# ----------------------------------------------------------------------------------------------------------------
# --impl reference
# ----------------------------------------------------------------------------------------------------------------
def run_reference(args, rank, world):
    """--impl reference: the reference's own CPU algorithm (C port in oracle/, the Go original cannot be built here) on the
    host cores, on OUR arm's workload: n = 2^logn points of the same synthetic inputs per step.  If a probe step says that
    K + W steps of the full size would not end within the time budget, each step is a bounded sample (a power of two) of it
    and the line says so."""
    if rank != 0:
        return
    from oracle import cref
    from oracle import oracle as O

    g = args.curve
    G = O.GROUPS[g]
    cores = ncores()
    logn_total = args.total_logn if args.total_logn else (args.logn if world == 1 else 26)
    base = G.encode_affine([G.scalar_mul(G.gen, BASE_MULT)])[0]
    # probe: one 2^20 step decides the per-step size (full size unless K + W steps of it would exceed the budget)
    probe_log = min(20, logn_total)
    pts = cref.generate_multiples(g, base, 1, 1 << probe_log, nthreads=cores)
    s = synth_scalars(1 << probe_log, CURVE_BITS[g], 0x5EED0000 + 2, fr_mod(g))
    cref.msm(g, pts, s, c=0, nthreads=cores)
    t0 = time.perf_counter()
    cref.msm(g, pts, s, c=0, nthreads=cores)
    probe_rate = (1 << probe_log) / (time.perf_counter() - t0)
    budget_s = float(os.environ.get("GMSM_REF_BUDGET_S", "300"))
    logs = args.sample_logn if args.sample_logn else logn_total
    while not args.sample_logn and logs > 16 and (args.steps + args.warmup) * (1 << logs) / probe_rate > budget_s:
        logs -= 1
    n = 1 << logs
    if n != (1 << probe_log):
        pts = cref.generate_multiples(g, base, 1, n, nthreads=cores)
        s = synth_scalars(n, CURVE_BITS[g], 0x5EED0000 + 2, fr_mod(g))
    for _ in range(args.warmup):
        cref.msm(g, pts, s, c=0, nthreads=cores)
    times, used_c, leaves = [], 0, 0
    t_all = time.perf_counter()
    for _ in range(args.steps):
        t0 = time.perf_counter()
        _, _, used_c, leaves = cref.msm(g, pts, s, c=0, nthreads=cores)
        times.append(time.perf_counter() - t0)
    dt = (time.perf_counter() - t_all) / args.steps
    val = n / dt
    sample = ("n=2^%d per step = the whole workload" % logs) if logs == logn_total else (
        "n=2^%d per step: a bounded sample of the 2^%d workload (K+W steps of the full size would exceed %.0f s at the probed %.1f M/s)"
        % (logs, logn_total, budget_s, probe_rate / 1e6))
    line = {
        "impl": "reference", "metric": metric_name(g),
        "value": val, "unit": "scalar-muls/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": dt * 1e3, "higher_is_better": True, "scaling": "weak" if world == 1 else "strong", "vs_baseline": None,
        "dtype": "u64", "data": "synthetic",
        "config": {"workload": workload_name(g, logn_total, world), "n_total": 1 << logn_total},
        "reference_run": {"n_per_step": n, "c": used_c, "sub_msms": leaves, "threads": cores,
                          "step_s": {"min": min(times), "median": float(np.median(times)), "max": max(times)},
                          "probe_rate_2e%d" % probe_log: probe_rate},
        "cpu_baseline": {"value": val, "unit": "scalar-muls/s", "cores": cores, "kind": "port",
                         "sample": sample + "; C port of the reference algorithm (bestC c=%d, %d sub-MSMs, batch-affine buckets as in "
                                            "getChunkProcessorG1), portable C without ADX assembly" % (used_c, leaves),
                         "best": n / min(times), "spread": (max(times) - min(times)) / float(np.median(times))},
        "e2e": {"value": val, "unit": "scalar-muls/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line))


# ----------------------------------------------------------------------------------------------------------------
# ours
# ----------------------------------------------------------------------------------------------------------------
class Ctx:
    pass


def closed_form_check(X, g, result_jac, local_dot):
    """the timed result against [sum_i (start+i) s_i * BASE_MULT] G evaluated by the CPU oracle (checker only).
    local_dot: this rank's sum_i (start+i) * mont_limbs_i mod r; all ranks' sums are combined on rank 0."""
    import torch

    r = fr_mod(g)
    dots = [local_dot]
    if X.world > 1:
        t = torch.tensor([(local_dot >> (32 * k)) & 0xFFFFFFFF for k in range(12)], dtype=torch.int64, device="cuda")
        allt = torch.empty(12 * X.world, dtype=torch.int64, device="cuda")
        X.dist.all_gather_into_tensor(allt, t)
        v = allt.cpu().numpy().reshape(X.world, 12)
        dots = [sum(int(v[q, k]) << (32 * k) for k in range(12)) for q in range(X.world)]
    if X.rank != 0:
        return None
    from oracle import oracle as O      # checker

    G = O.GROUPS[g]
    k = sum(dots) * pow(1 << (64 * scalar_words(CURVE_BITS[g])), -1, r) * BASE_MULT % r          # Montgomery limbs -> canonical scalars: * R^-1
    want = G.encode_affine([G.scalar_mul(G.gen, k)])[0] if k else None
    aw = AFF_BYTES[g] // 8               # u64 words of the affine point (X, Y); the Jacobian triple adds Z
    got = np.asarray(result_jac, dtype=np.uint64)
    if want is None:
        ok = not got[aw:].any()
    else:
        ok = bool(np.array_equal(got[:aw], np.asarray(want, dtype=np.uint64)) and got[aw:].any())
    return ok


def measure_resident(X, g, logn_local, steps, warmup, c=0, kind=None, sample_clocks=False, start_index=None):
    """One device-resident measurement of 2^logn_local points on this rank (all ranks together: 2^logn_local * world).
    Returns (dict, keep) -- keep holds the engine and the device / host inputs for follow-up legs."""
    torch, dist = X.torch, X.dist
    world, rank = X.world, X.rank
    n = 1 << logn_local
    n_total = n * world
    lo, hi = X.distmod.shard_range(n_total, rank, world)
    bits = CURVE_BITS[g]
    if c == 0 and world > 1:          # every rank runs ONE plan, that of the largest shard (dist.window_bits_for_total)
        c = X.distmod.window_bits_for_total(g, n_total, world)
    eng = X.pkg.Engine(g, n, c=c, device=X.local_rank)
    W, cc = eng.nwin, eng.c
    wds = AFF_BYTES[g] // 8
    d_B = eng.generate_multiples(_generator_limbs(g), BASE_MULT, 1)
    base = d_B.cpu().numpy().view(np.uint64).copy()
    d_points = eng.generate_multiples(base, 1 + lo, n)
    h_scalars_np = synth_scalars(n, bits, 0x5EED0000 + 2 + rank, fr_mod(g))
    if kind:
        h_scalars_np = skew_scalars(h_scalars_np, kind)
    d_scalars = eng.to_device(h_scalars_np)
    torch.cuda.synchronize()
    sharded = X.distmod.ShardedMultiExp(eng) if world > 1 else None

    def step():
        if sharded is not None:
            return sharded.msm(d_points, d_scalars, n)
        return eng.msm(d_points, d_scalars, n)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    eng.set_profiling(True)
    for _ in range(max(warmup, 3)):
        step()
    barrier()
    sampler = ClockSampler(X.local_rank) if (sample_clocks and rank == 0) else None
    if sampler:
        sampler.start()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    ev0.record()
    for _ in range(steps):
        out = step()
    ev1.record()
    barrier()
    clocks = sampler.stop() if sampler else None
    ms_total = ev0.elapsed_time(ev1)
    launches_per_step = eng.last_launches + (1 if world > 1 else 0)
    if world > 1:
        t = torch.tensor([ms_total], device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms_total = float(t.item())
    ms_step = ms_total / steps
    result_jac = out.cpu().numpy().view(np.uint64).copy()
    # parity of the TIMED result at full size
    t0 = time.perf_counter()
    ok = closed_form_check(X, g, result_jac, dot_index_mod(h_scalars_np, 1 + lo, fr_mod(g)))
    parity_s = time.perf_counter() - t0
    # stage times of the dominant kernel, averaged over a few more steps (events on the launch stream)
    acc_ms, stages = [], None
    for _ in range(3):
        step()
        torch.cuda.synchronize()
        st = eng.last_stage_ms()
        acc_ms.append(st[3])
        stages = st
    acc = float(np.mean(acc_ms))
    peak, peak_src = measured_hbm_peak()
    A = AFF_BYTES[g]
    alg_bytes = n * W * (A + 2)             # SURVEY.md 8(d): per (point, window): one affine point + one u16 digit
    achieved = alg_bytes / (acc * 1e-3) / 1e9
    try:
        traffic = json.load(open(os.path.join(ROOT, "profiles", "ncu_traffic.json"))).get("%s:%d:%d" % (g, logn_local, cc))
    except Exception:
        traffic = None
    roofline = {"bound": "hbm", "binding_unit": "INT32 multiplier pipe (IMAD.WIDE), see int_pipe -- the HBM figure is the mandated yardstick, not the limiter",
                "kernel": "k_accumulate", "achieved": achieved, "peak": peak, "unit": "GB/s",
                "frac": achieved / peak, "traffic": traffic, "peak_source": peak_src, "kernel_ms": acc,
                "alg_bytes_per_launch": alg_bytes,
                "int_pipe": {"mixed_adds_per_s": n * W / (acc * 1e-3)}}
    if clocks and clocks.get("sm_mhz"):
        roofline["int_pipe"]["multiplier_pipe"] = int_pipe_fraction(g, n * W / (acc * 1e-3), clocks["sm_mhz"], X.wide_mads.get(g))
    res = {
        "value": n_total / (ms_step * 1e-3), "unit": "scalar-muls/s", "ms_per_step": ms_step, "steps": steps,
        "n_total": n_total, "n_per_gpu": n, "c": cc, "windows": W,
        "parity": {"closed_form": ok, "n": n_total, "what": "timed result == [sum (1+i) s_i * 0x%X] G by the CPU oracle, affine limbs" % BASE_MULT,
                   "check_s": round(parity_s, 2)} if rank == 0 else None,
        "roofline": roofline, "stages_ms": dict(zip(STAGE_NAMES, [float(x) for x in stages])),
        "gpu_launches": launches_per_step * steps, "clocks": clocks,
    }
    if kind:
        res["distribution"] = kind
    keep = Ctx()
    keep.eng, keep.d_points, keep.d_scalars, keep.h_scalars_np, keep.result_jac, keep.sharded = eng, d_points, d_scalars, h_scalars_np, result_jac, sharded
    keep.n, keep.lo, keep.W, keep.c = n, lo, W, cc
    return res, keep


def release(keep):
    keep.eng.close()
    keep.d_points = keep.d_scalars = None


def fail_parity(what, res):
    if res.get("parity") is not None and not res["parity"]["closed_form"]:
        raise SystemExit("bench.py: PARITY FAILURE (%s): the timed result differs from the closed form" % what)


def dump_outputs(out_dir, result_jac):
    """--dump-outputs: the headline's last timed result, the Jacobian triple (X, Y, Z) of Montgomery limbs the engine returns,
    as msm_result.npy: one row per coordinate, each u64 limb split into its two u32 halves (low half first) so that float64
    holds every word exactly"""
    os.makedirs(out_dir, exist_ok=True)
    words = np.ascontiguousarray(result_jac, dtype=np.uint64).view(np.uint32).reshape(3, -1)
    np.save(os.path.join(out_dir, "msm_result.npy"), words.astype(np.float64))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--curve", default="bn254_g1", choices=list(CURVE_BITS))
    ap.add_argument("--logn", type=int, default=24, help="log2 of points PER GPU (N = 1, and the weak figure at N > 1)")
    ap.add_argument("--total-logn", type=int, default=0,
                    help="log2 of the TOTAL number of points sharded over the N ranks; default: 26 at N > 1 (BASELINE configs[4], "
                         "strong scaling), logn at N = 1")
    ap.add_argument("--weak", action="store_true", help="N > 1: make the weak-scaling run (2^logn per GPU) the headline instead")
    ap.add_argument("--c", type=int, default=0, help="window width (0 = engine model)")
    ap.add_argument("--sample-logn", type=int, default=0, help="cpu baseline sample size (log2)")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-tables", action="store_true", help="skip the window-table (precomputed resident bases) measurement")
    ap.add_argument("--no-extras", action="store_true", help="skip the sub-objects (configs[2], [3], 2^20, 2^26, skewed scalars, concurrent calls)")
    ap.add_argument("--table-c", type=int, default=0, help="window width of the table mode (0 = engine model)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the result of the headline's last timed step to DIR/msm_result.npy (float64), to compare two builds "
                         "output for output (the inputs are fixed by their seeds)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))

    if args.impl == "reference":
        run_reference(args, rank, world)
        return

    import torch
    import torch.distributed as dist

    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; the engine has no CPU fallback (use --impl reference for the CPU path)")
    torch.cuda.set_device(local_rank)
    if world > 1:
        # rank 0 prints ONE JSON line on stdout: keep NCCL's version banner off it
        if os.environ.get("NCCL_DEBUG", "VERSION").upper() == "VERSION":
            os.environ["NCCL_DEBUG"] = "WARN"
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    X = Ctx()
    X.torch, X.dist, X.world, X.rank, X.local_rank = torch, dist, world, rank, local_rank
    X.pkg = importlib.import_module("gnark_crypto_b200")
    X.distmod = importlib.import_module("gnark-crypto_b200.dist")
    mx = importlib.import_module("gnark-crypto_b200.multiexp")
    native = importlib.import_module("gnark-crypto_b200._native")
    try:    # IMAD.WIDE per mixed addition of the built kernels (tools/sass_count.py on the shipped objects), if recorded
        X.wide_mads = json.load(open(os.path.join(ROOT, "profiles", "wide_mads_per_mixed_add.json")))
    except Exception:
        X.wide_mads = {}

    g = args.curve
    bits = CURVE_BITS[g]
    A = AFF_BYTES[g]
    SW = scalar_words(bits)          # u64 words per scalar
    wds = A // 8
    # ---- headline configuration ----
    if world == 1:
        scaling = "weak"
        logn_local = args.total_logn if args.total_logn else args.logn
    elif args.weak:
        scaling = "weak"
        logn_local = args.logn
    else:
        scaling = "strong"
        tl = args.total_logn if args.total_logn else 26
        if (1 << tl) % world:
            raise SystemExit("--total-logn: 2^%d is not divisible by %d ranks" % (tl, world))
        logn_local = tl - (world.bit_length() - 1)
    logn_total = logn_local + (world.bit_length() - 1)
    n = 1 << logn_local
    n_total = n * world

    res, K = measure_resident(X, g, logn_local, args.steps, args.warmup, c=args.c, sample_clocks=True)
    fail_parity("headline", res)
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, K.result_jac)
    line = {
        "metric": metric_name(g),
        "value": res["value"], "unit": "scalar-muls/s", "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3),
        "ms_per_step": res["ms_per_step"], "higher_is_better": True, "scaling": scaling, "vs_baseline": None, "dtype": "u32",
        "data": "synthetic",
        "config": {"workload": workload_name(g, logn_total, world), "n_total": n_total},
        "engine": {"c": res["c"], "windows": res["windows"], "n_per_gpu": n, "parallelism": "shard%d" % world,
                   "l2": "inputs %.2f GiB per GPU > 126 MB L2 (no flush needed)" % ((n * (A + 8 * SW)) / 2**30)},
        "parity": res["parity"],
        "roofline": res["roofline"],
        "stages_ms": res["stages_ms"],
        "gpu_launches": res["gpu_launches"],
        "clocks": res["clocks"],
    }
    eng, d_points, d_scalars, h_scalars_np, result_jac, sharded = K.eng, K.d_points, K.d_scalars, K.h_scalars_np, K.result_jac, K.sharded

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---- window tables for resident bases (gmsm_bases_precompute): the static-SRS flow.  NOT the headline: the
    # headline `value` is the plain MultiExp whose bases may change on every call, like the reference's. ----
    if world == 1 and not args.no_tables:
        teng = X.pkg.Engine(g, n, c=args.table_c, device=local_rank, tables=True)
        t0 = time.perf_counter()
        d_table = teng.build_tables(d_points, n)
        torch.cuda.synchronize()
        build_s = time.perf_counter() - t0
        teng.set_profiling(True)
        for _ in range(max(args.warmup, 3)):
            tout = teng.msm_tables(d_table, n, d_scalars, n)
        torch.cuda.synchronize()
        tev0, tev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        tev0.record()
        for _ in range(args.steps):
            tout = teng.msm_tables(d_table, n, d_scalars, n)
        tev1.record()
        torch.cuda.synchronize()
        t_ms = tev0.elapsed_time(tev1) / args.steps
        if not np.array_equal(tout.cpu().numpy().view(np.uint64), result_jac):
            raise SystemExit("bench.py: window-table result differs from the plain result")
        tst = teng.last_stage_ms()
        line["resident_tables"] = {
            "value": n / (t_ms * 1e-3), "unit": "scalar-muls/s", "ms_per_step": t_ms, "c": teng.c, "windows": teng.nwin,
            "table_bytes": int(d_table.numel()) * 8, "table_build_s": build_s,
            "stages_ms": dict(zip(STAGE_NAMES, [float(x) for x in tst])),
            "accumulate_alg_GBps": n * teng.nwin * (A + 2) / (tst[3] * 1e-3) / 1e9,
            "note": "bases precomputed once as W rows 2^(c*j)*P (one shared bucket set, no Horner); result bit-identical to `value`'s",
        }
        line["gpu_launches"] += teng.last_launches * args.steps
        teng.close()
        del d_table

    # ---- end to end through the reference-facing call, host buffers ----
    if not args.no_e2e:
        h_points = torch.empty(n * wds, dtype=torch.int64).pin_memory()
        h_points.copy_(d_points.cpu())
        h_scal = torch.empty(n * SW, dtype=torch.int64).pin_memory()
        h_scal.copy_(torch.from_numpy(h_scalars_np.view(np.int64).reshape(-1)))
        hp, hs = h_points.numpy().view(np.uint64), h_scal.numpy().view(np.uint64)
        jac_words = 3 * wds // 2
        L = native.lib()
        if world == 1:
            outj = np.zeros(jac_words, dtype=np.uint64)

            def e2e_step(P=hp, S=hs):
                rc = L.gmsm_multiexp(mx.CURVES[g], P.ctypes.data, S.ctypes.data, n, 0, outj.ctypes.data)
                if rc != 0:
                    raise RuntimeError(native.last_error())
                return outj
        else:
            def e2e_step(P=hp, S=hs):
                return sharded.msm_from_host_pipelined(P, S).cpu().numpy().view(np.uint64)

        def time_e2e(fn, reps):
            for _ in range(2):
                r = fn()
            barrier()
            t0 = time.perf_counter()
            for _ in range(reps):
                r = fn()
            barrier()
            dt = (time.perf_counter() - t0) / reps
            if world > 1:
                t = torch.tensor([dt], device="cuda", dtype=torch.float64)
                dist.all_reduce(t, op=dist.ReduceOp.MAX)
                dt = float(t.item())
            if not np.array_equal(np.asarray(r), result_jac):
                raise SystemExit("bench.py: e2e result differs from the device-resident (closed-form-checked) result")
            return dt

        dt = time_e2e(e2e_step, args.steps)
        line["e2e"] = {"value": n_total / dt, "unit": "scalar-muls/s", "ms_per_step": dt * 1e3,
                       "h2d_bytes_per_step": n_total * (A + 8 * SW), "d2h_bytes_per_step": jac_words * 8 * world, "host_memory": "pinned",
                       "path": "gmsm_multiexp one-shot (points+scalars H2D every call)" if world == 1 else
                               "per rank: gmsm_multiexp_window_sums (pinned host shard, H2D pipelined under the bucket pass) -> NCCL all-gather of W partials -> finalize -> D2H"}
        # the same call on ordinary pageable memory -- what a Go caller's slices are (VERDICT r01 weak item 7)
        pp, ps = np.array(hp, copy=True), np.array(hs, copy=True)
        dtp = time_e2e(lambda: e2e_step(pp, ps), min(args.steps, 5))
        line["e2e_pageable"] = {"value": n_total / dtp, "unit": "scalar-muls/s", "ms_per_step": dtp * 1e3,
                                "h2d_bytes_per_step": n_total * (A + 8 * SW), "d2h_bytes_per_step": jac_words * 8 * world,
                                "host_memory": "pageable numpy arrays (not registered by the caller)", "vs_pinned": dtp / dt}
        del pp, ps
        if world == 1:
            launches_e2e = L.gmsm_last_oneshot_launches()
            line["gpu_launches"] += launches_e2e * args.steps
            # resident bases (prover flow: SRS static, scalars per call)
            rb = mx.ResidentBases(g, hp.reshape(n, wds), device=local_rank)
            rb.MultiExp(hs.reshape(n, SW))
            t0 = time.perf_counter()
            for _ in range(args.steps):
                rr = rb.MultiExp(hs.reshape(n, SW))
            dtr = (time.perf_counter() - t0) / args.steps
            if not np.array_equal(rr, result_jac):
                raise SystemExit("bench.py: resident-bases result differs")
            line["e2e_resident_bases"] = {"value": n / dtr, "unit": "scalar-muls/s", "ms_per_step": dtr * 1e3,
                                          "h2d_bytes_per_step": n * 8 * SW, "d2h_bytes_per_step": jac_words * 8}
            if not args.no_tables:
                tc = rb.Precompute(args.table_c)
                rb.MultiExp(hs.reshape(n, SW))
                t0 = time.perf_counter()
                for _ in range(args.steps):
                    rr = rb.MultiExp(hs.reshape(n, SW))
                dtt = (time.perf_counter() - t0) / args.steps
                if not np.array_equal(rr, result_jac):
                    raise SystemExit("bench.py: resident-bases (window tables) result differs")
                line["e2e_resident_tables"] = {"value": n / dtt, "unit": "scalar-muls/s", "ms_per_step": dtt * 1e3, "c": tc,
                                               "h2d_bytes_per_step": n * 8 * SW, "d2h_bytes_per_step": jac_words * 8}
            rb.close()
        del h_points, h_scal

    # ---- CPU baseline: the oracle's C port (rank 0, N = 1 only) on a bounded sample + parity of the GPU on that sample ----
    if rank == 0 and world == 1 and not args.no_cpu:
        from oracle import cref

        cores = ncores()
        logs = args.sample_logn if args.sample_logn else min(logn_local, 22 if cores >= 16 else 18)
        ns = 1 << logs
        sp = d_points[: ns * wds].cpu().numpy().view(np.uint64).reshape(ns, wds)
        ss = h_scalars_np[:ns]
        times = []
        for _ in range(3):
            t0 = time.perf_counter()
            want, _, used_c, leaves = cref.msm(g, sp, ss, c=0, nthreads=cores)
            times.append(time.perf_counter() - t0)
        eng_s = X.pkg.Engine(g, ns, c=0, device=local_rank)
        got = eng_s.msm_host_result(eng_s.to_device(sp), eng_s.to_device(ss), ns)
        eng_s.close()
        if not np.array_equal(got[:wds], want):
            raise SystemExit("bench.py: GPU result differs from the CPU oracle on the baseline sample")
        line["cpu_baseline"] = {"value": ns / min(times), "unit": "scalar-muls/s", "cores": cores, "kind": "port",
                                "sample": "first 2^%d points/scalars of the same workload; C port of the reference algorithm "
                                          "(bestC c=%d, %d sub-MSMs, batch-affine buckets as in getChunkProcessorG1; portable C, no ADX assembly), "
                                          "best of 3, GPU result on the sample bit-exact" % (logs, used_c, leaves),
                                "step_s": {"min": min(times), "median": float(np.median(times)), "max": max(times)}}
    release(K)
    del eng, d_points, d_scalars, K
    torch.cuda.empty_cache()

    # ---- N > 1: the weak-scaling figure beside the strong headline (or vice versa) ----
    if world > 1 and not args.no_extras:
        other_logn = args.logn if scaling == "strong" else 26 - (world.bit_length() - 1)
        if other_logn != logn_local:
            r2, K2 = measure_resident(X, g, other_logn, min(args.steps, 5), 3, c=args.c)
            fail_parity("weak" if scaling == "strong" else "strong", r2)
            release(K2)
            del K2
            torch.cuda.empty_cache()
            for k in ("roofline", "clocks"):
                r2.pop(k, None)
            line["weak" if scaling == "strong" else "strong"] = r2
            line["gpu_launches"] += r2.pop("gpu_launches")

    # ---- N = 1: the other BASELINE configs and the metric's other sizes, each closed-form checked ----
    if world == 1 and not args.no_extras and g == "bn254_g1" and logn_local == 24 and args.c == 0:
        extras = [("configs[2] bls12-381 G1 n=2^24", "bls12381_g1", 24, None), ("configs[3] bn254 G2 n=2^22", "bn254_g2", 22, None),
                  ("bn254 G1 n=2^20", "bn254_g1", 20, None), ("bn254 G1 n=2^26 on one GPU (the strong-scaling reference point)", "bn254_g1", 26, None),
                  ("bn254 G1 n=2^24 smallvalues (multiexp_test.go:316-325)", "bn254_g1", 24, "smallvalues"),
                  ("bn254 G1 n=2^24 redundancy (multiexp_test.go:327-334)", "bn254_g1", 24, "redundancy")]
        line["configs"] = {}
        for name, gg, lg, kind in extras:
            rr, KK = measure_resident(X, gg, lg, min(args.steps, 5), 3, kind=kind, sample_clocks=True)
            fail_parity(name, rr)
            release(KK)
            del KK
            torch.cuda.empty_cache()
            line["gpu_launches"] += rr.pop("gpu_launches")
            line["configs"][name] = rr
        base_ms = line["ms_per_step"]
        for name in list(line["configs"]):
            if "smallvalues" in name or "redundancy" in name:
                line["configs"][name]["vs_random_scalars"] = line["configs"][name]["ms_per_step"] / base_ms
        # three concurrent calls (BenchmarkManyMultiExpG1Reference, multiexp_test.go:385-415: three goroutines, each one MultiExp)
        line["two_in_flight"] = two_in_flight(X, g, 24, min(args.steps, 5))
        if not args.no_e2e:
            line["concurrent3"] = concurrent3(X, native, mx, g, 20)
    if rank == 0:
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


def two_in_flight(X, g, logn, steps):
    """throughput with TWO device-resident MultiExp in flight (two engine contexts on two streams, calls issued alternately): the
    latency-bound tail of one call (carry join, bucket reduction, Horner) overlaps the head and the bucket pass of the next --
    how a prover that commits to several polynomials would drive the engine.  NOT the headline (`value` times one call at a
    time); both results are compared with each other and the first with the closed form."""
    torch = X.torch
    n = 1 << logn
    engs = [X.pkg.Engine(g, n, c=0, device=X.local_rank) for _ in range(2)]
    base = engs[0].generate_multiples(_generator_limbs(g), BASE_MULT, 1).cpu().numpy().view(np.uint64).copy()
    d_points = engs[0].generate_multiples(base, 1, n)
    h_s = synth_scalars(n, CURVE_BITS[g], 0x5EED0000 + 2, fr_mod(g))
    d_s = engs[0].to_device(h_s)
    outs = [torch.zeros_like(engs[0]._out) for _ in range(2)]
    streams = [torch.cuda.Stream(device=X.local_rank) for _ in range(2)]
    L = importlib.import_module("gnark-crypto_b200._native").lib()
    import ctypes

    def issue(k):
        rc = L.gmsm_ctx_msm_device(engs[k]._h, d_points.data_ptr(), d_s.data_ptr(), n, outs[k].data_ptr(), ctypes.c_void_p(streams[k].cuda_stream))
        if rc != 0:
            raise RuntimeError("gmsm_ctx_msm_device failed")

    torch.cuda.synchronize()
    for k in (0, 1, 0, 1):
        issue(k)
    torch.cuda.synchronize()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ev0.record(torch.cuda.current_stream(X.local_rank))
    for st in streams:
        st.wait_stream(torch.cuda.current_stream(X.local_rank))
    reps = 2 * steps
    for i in range(reps):
        issue(i & 1)
    for st in streams:
        torch.cuda.current_stream(X.local_rank).wait_stream(st)
    ev1.record(torch.cuda.current_stream(X.local_rank))
    torch.cuda.synchronize()
    ms = ev0.elapsed_time(ev1) / reps
    a, b = outs[0].cpu().numpy().view(np.uint64), outs[1].cpu().numpy().view(np.uint64)
    ok = closed_form_check(X, g, a, dot_index_mod(h_s, 1, fr_mod(g)))
    for e in engs:
        e.close()
    return {"workload": "%s MultiExp n=2^%d, two calls in flight on two contexts / streams" % (g, logn), "ms_per_msm": ms,
            "value": n / (ms * 1e-3), "unit": "scalar-muls/s", "results_identical": bool(np.array_equal(a, b)), "closed_form": ok}


def concurrent3(X, native, mx, g, logn):
    """three host threads, each one gmsm_multiexp over its own host buffers, against the same three calls back to back"""
    n = 1 << logn
    wds = AFF_BYTES[g] // 8
    eng = X.pkg.Engine(g, n, c=0, device=X.local_rank)
    base = eng.generate_multiples(_generator_limbs(g), BASE_MULT, 1).cpu().numpy().view(np.uint64).copy()
    L = native.lib()
    jobs = []
    for k in range(3):
        pts = eng.generate_multiples(base, 1 + k * n, n).cpu().numpy().view(np.uint64).copy()
        sc = synth_scalars(n, CURVE_BITS[g], 0x5EED0100 + k, fr_mod(g))
        jobs.append((pts, sc, np.zeros(3 * wds // 2, dtype=np.uint64)))
    eng.close()

    def call(j):
        p, s, o = jobs[j]
        rc = L.gmsm_multiexp(mx.CURVES[g], p.ctypes.data, s.ctypes.data, n, 0, o.ctypes.data)
        if rc != 0:
            raise RuntimeError(native.last_error())

    for j in range(3):
        call(j)
    serial_out = [jobs[j][2].copy() for j in range(3)]
    th = [threading.Thread(target=call, args=(j,)) for j in range(3)]      # warm-up of the concurrent path: the pool creates its
    for t in th:                                                           # second and third session (buffers, pinned ring) here
        t.start()
    for t in th:
        t.join()
    reps = 5
    t0 = time.perf_counter()
    for _ in range(reps):
        for j in range(3):
            call(j)
    t_serial = (time.perf_counter() - t0) / reps
    t0 = time.perf_counter()
    for _ in range(reps):
        th = [threading.Thread(target=call, args=(j,)) for j in range(3)]
        for t in th:
            t.start()
        for t in th:
            t.join()
    t_conc = (time.perf_counter() - t0) / reps
    same = all(np.array_equal(jobs[j][2], serial_out[j]) for j in range(3))
    return {"workload": "3 host threads x %s MultiExp n=2^%d (pageable host buffers), gmsm_multiexp" % (g, logn),
            "serial_ms": t_serial * 1e3, "concurrent_ms": t_conc * 1e3, "speedup": t_serial / t_conc, "results_identical": bool(same)}


if __name__ == "__main__":
    main()
