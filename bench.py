#!/usr/bin/env python3
"""bench.py - BN254 G1 MSM throughput (BASELINE.json metric, configs[1]) on N B200s, plus the other BASELINE
configs as secondary legs of the same JSON line.

  python bench.py [--gpus N] [--steps K] [--warmup W]          # this repo's CUDA path
  python bench.py ... --dump-outputs DIR                        # + the last timed step's MSM point as DIR/*.npy
  python bench.py --impl reference [...]                        # CPU arm (oracle port, all host cores)
  torchrun --nproc-per-node N bench.py --gpus N ...             # one rank per GPU

One "step" = one full MSM (decompose -> sort -> bucket accumulate -> reduce) over 2^20 random scalars per GPU
against a device-resident table of 2^20 distinct bases (PinToGPU semantics of the reference,
backend/accelerated/icicle/groth16/bn254/icicle.go:185-261).  N > 1: the (scalar, base) index range is sharded
over ranks (weak scaling: 2^20 per GPU), each rank produces one partial point per step; the K partial points of
the timed region go through ONE ncclAllGather and one fold kernel on the device (b200_points_allreduce - the
multi-GPU twin of the reference's host-side sum of chunk results, icicle.go:383-411).  No .cpu() in any timed region.

Secondary legs (same line, never the headline): "strong" - ONE 2^24-point BN254 MSM sharded N ways (north_star's
target); "groth16" - prove ms at 2^20 R1CS (configs[2]); "plonk" - BLS12-381 2^22 prove (configs[3]);
"bw6" - BW6-761 G1 MSM 2^24 sharded (configs[4], N = 8 only by default).

Every loop that contains a collective runs a FIXED number of iterations on every rank (round 1's N=4/8 hang was a
rank-local wall-clock loop around all_gather); the process leaves through the normal interpreter exit after
barrier + destroy_process_group, with a watchdog that only fires if that teardown hangs.
"""

import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True    # the benchmark leaves the tree it runs from untouched (no __pycache__)

import numpy as np  # noqa: E402

METRIC = "bn254_g1_msm_scalar_muls_per_sec"
UNIT = "scalar-muls/s"
LOG_N = 20
SEED = 0x6E61726B00000002  # SURVEY.md §8d: config 2 seed
DTYPE = "u32x8 (254-bit Montgomery integers)"
# the SAME config object on both arms (the driver compares them)
CONFIG = {"workload": "BN254 G1 MSM, 2^20 uniform random scalars x 2^20 distinct known-discrete-log bases per GPU "
                      "(BASELINE configs[1]); bases resident (device table / host memory), scalars change per step",
          "curve": "bn254", "group": "G1", "points_per_gpu": 1 << LOG_N}
LEG_LIMIT_S = {"strong": 240, "groth16": 300, "plonk": 420, "bw6": 300}
WHOLE_RUN_LIMIT_S = 1500
LOAD_STEPS = 160   # fixed-count load phase (>= 0.5 s at ~3.5 ms / MSM) so that nvidia-smi's 100 ms sampler sees clocks under load
NCU_TRAFFIC_FILE = os.path.join(ROOT, "profiles", "ncu_accumulate_traffic.json")


# --------------------------------------------------------------------------------------
# workload (synthetic, seeded).  Uses the oracle ONLY to materialise known-discrete-log
# bases and to check the result before timing (checker role) and for the CPU arm.
# --------------------------------------------------------------------------------------
def rand_fr(rs, count, limbs=4, top_bits=61):
    """uniform below 2^(64*(limbs-1)+top_bits) < r; the raw limbs are used as Montgomery residues, which are
    themselves uniform field elements: no conversion needed.  rs: np.random.Generator"""
    a = rs.integers(0, 1 << 64, size=(count, limbs), dtype=np.uint64)
    a[:, limbs - 1] &= np.uint64((1 << top_bits) - 1)
    return a


def rng(seed):
    return np.random.Generator(np.random.PCG64(seed))


def make_workload(n, seed, rank=0):
    """bases: n DISTINCT known-discrete-log points k_i * G (the same on every rank); scalars: n uniform field
    elements per rank.  expected = (sum s_i k_i) * G (SURVEY.md §8c-1)."""
    from oracle import corelib, ec, ff
    from oracle.params import BN254 as C
    ks = rand_fr(rng(seed), n)
    pts = corelib.fixed_base(C, 1, ec.pack_points(C, 1, [C.g1]), ks)
    sc_m = rand_fr(rng(seed + rank + 1), n)
    dot = corelib.fr_dot(C, ks, sc_m)      # sum k_i s_i mod r
    return C, pts, sc_m, dot


def dlog_point(C, dot):
    from oracle import ec, ff
    return ec.scalar_mul(ff.Fp(C.p), dot % C.r, C.g1)


def jac_to_affine(C, jac, group=1):
    from oracle import ec, ff
    return ec.from_jac(ff.base_field(C, group), ec.unpack_points(C, group, np.ascontiguousarray(jac), ncoords=3)[0])


# --------------------------------------------------------------------------------------
class ClockSampler:
    """nvidia-smi clocks / throttle reasons DURING the timed region (B200_PROFILING.md)."""

    def __init__(self, gpu_index):
        self.rows = []
        self.proc = None
        self.idx = gpu_index

    def start(self):
        q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
             "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
             "clocks_event_reasons.sw_power_cap")
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.idx), f"--query-gpu={q}",
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([x.strip() for x in line.split(",")])

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            pass
        sm, mx, reasons = [], None, set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            try:
                sm.append(float(r[0])); mx = float(r[1])
                for k, nme in enumerate(names):
                    if r[3 + k].lower().startswith("active"):
                        reasons.add(nme)
            except Exception:
                pass
        # median over the samples taken under load (the idle samples before / after the kernels would drag it down)
        busy = [x for x in sm if mx and x >= 0.5 * mx] or sm
        return {"sm_mhz": float(np.median(busy)) if busy else None, "sm_max_mhz": mx, "reasons": sorted(reasons),
                "samples": len(sm), "samples_under_load": len(busy)}


IMAD_WIDE_LANES_PER_CLK_SM = 32   # measured issue rate of IMAD.WIDE (half-rate pipe), profiles/r01_microbench_pipes.txt
N_SMS = 148


def multiplier_roofline(entries, imad_per_entry, kernel_ms, clocks):
    mhz = (clocks or {}).get("sm_mhz") or (clocks or {}).get("sm_max_mhz") or 1965.0
    peak = N_SMS * IMAD_WIDE_LANES_PER_CLK_SM * mhz * 1e6 / 1e12
    achieved = entries * imad_per_entry / (kernel_ms / 1e3) / 1e12
    return {"bound": "int32 multiplier issue", "achieved": achieved, "peak": peak, "unit": "T IMAD.WIDE/s",
            "frac": achieved / peak, "sm_mhz": mhz, "imad_wide_per_bucket_entry": imad_per_entry,
            "model": "bucket entries x IMAD.WIDE per XYZZ mixed addition (static SASS count) / accumulate time; "
                     "peak = 148 SMs x 32 lanes/clk x SM clock under load"}


def measured_peak_gbs():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs, burst copy)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md)"


def ncu_traffic():
    """dram bytes of one k_msm_accumulate launch from the committed ncu --set full capture (profiles/), or None"""
    try:
        d = json.load(open(NCU_TRAFFIC_FILE))
        return float(d["dram_bytes_per_launch"]), d.get("source", NCU_TRAFFIC_FILE)
    except Exception:
        return None, None


# --------------------------------------------------------------------------------------
def cpu_msm(C, pts, sc, c, threads):
    """the CPU arm: signed-digit Pippenger, affine buckets with batched additions for the full windows and
    extended-Jacobian for the short top window, (window x point-range) tasks over all threads - the structure
    of gnark-crypto's MultiExp, restated in oracle/c/oracle.cpp"""
    from oracle import corelib
    return corelib.msm(C, 1, pts, sc, c=c, nthreads=threads, batch_affine=True)


def host_threads():
    """threads the CPU arm may really use: the affinity mask and the cgroup CPU quota, not just the core count"""
    t = os.cpu_count() or 1
    try:
        t = min(t, len(os.sched_getaffinity(0)))
    except Exception:
        pass
    try:
        q, per = open("/sys/fs/cgroup/cpu.max").read().split()
        if q != "max":
            t = min(t, max(1, int(float(q) / float(per) + 0.5)))
    except Exception:
        pass
    return max(1, t)


def cpu_best_config(C, pts, sc, threads):
    """pick window size and thread count the way gnark-crypto picks its window (by problem size / cores): a quick
    sweep.  On SMT hosts the integer-multiplier-bound inner loop often runs faster on one thread per core, so half
    the hardware threads is tried as well; the faster configuration is the one timed."""
    best = (None, threads, 1e9)
    cands = [threads] if threads < 16 else [threads, threads // 2]
    for th in cands:
        for c in (12, 13, 14, 15, 16, 17, 18):
            t0 = time.perf_counter()
            cpu_msm(C, pts, sc, c, th)
            dt = time.perf_counter() - t0
            if dt < best[2]:
                best = (c, th, dt)
    return best[0], best[1]


def cpu_msm_rate(C, pts, sc, sample_n, budget_s, threads):
    """oracle port (restatement of gnark-crypto's MultiExp algorithm, NOT gnark-crypto) on host cores: window and
    thread count by a sweep, then as many repetitions as fit `budget_s` seconds of wall clock (at least 3)"""
    p, s = pts[:sample_n], sc[:sample_n]
    c, th = cpu_best_config(C, p, s, threads)
    t0 = time.perf_counter()
    cpu_msm(C, p, s, c, th)
    one = time.perf_counter() - t0
    reps = max(3, min(200, int(budget_s / max(one, 1e-3))))
    t0 = time.perf_counter()
    for _ in range(reps):
        cpu_msm(C, p, s, c, th)
    dt = (time.perf_counter() - t0) / reps
    return sample_n / dt, dt, th, c, reps


def run_reference(args):
    """--impl reference: the reference's CPU implementation of this path.  gnark (Go) cannot be
    built here and its arithmetic lives in the absent gnark-crypto module, so this arm times the
    C++ restatement of the same algorithm (oracle/c/oracle.cpp) on all host cores."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    n = 1 << LOG_N
    threads = host_threads()
    sample_n = n if threads >= 16 else n >> 2
    C, pts, sc, dot = make_workload(sample_n, SEED)
    cw, threads = cpu_best_config(C, pts, sc, threads)
    assert jac_to_affine(C, cpu_msm(C, pts, sc, cw, threads)) == dlog_point(C, dot)
    for _ in range(args.warmup):
        cpu_msm(C, pts, sc, cw, threads)
    t0 = time.perf_counter()
    for _ in range(args.steps):
        cpu_msm(C, pts, sc, cw, threads)
    dt = time.perf_counter() - t0
    value = sample_n * args.steps / dt
    sample = f"{args.steps} x BN254 G1 MSM of 2^{int(np.log2(sample_n))} points per step on {threads} host threads"
    emit({
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * dt / args.steps,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": DTYPE,
        "data": "synthetic", "config": CONFIG,
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": threads, "kind": "port", "sample": sample,
                         "algorithm": f"Pippenger c={cw}, batch-affine buckets (restatement of gnark-crypto v0.21.0 MultiExp, "
                                      "not gnark-crypto itself: Go is not installed here and the module is absent)"},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    })


# --------------------------------------------------------------------------------------
class Ctx:
    """process-wide state of the CUDA arm: rank / device / stream / communicator"""

    def __init__(self, args):
        import torch
        import torch.distributed as dist
        from gnark_b200 import lib
        self.torch, self.dist, self.lib, self.args = torch, dist, lib, args
        self.world = int(os.environ.get("WORLD_SIZE", "1"))
        self.rank = int(os.environ.get("RANK", "0"))
        self.local = int(os.environ.get("LOCAL_RANK", "0"))
        if self.world != args.gpus and self.world == 1 and args.gpus > 1:
            raise SystemExit("launch with torchrun --nproc-per-node N for --gpus N")
        torch.cuda.set_device(self.local)
        if self.world > 1:
            dist.init_process_group("nccl", device_id=torch.device("cuda", self.local))
        lib.load()
        lib.init([self.local])
        self.stream = torch.cuda.Stream()          # a real (non-null) stream: kernels, events and NCCL all on it
        torch.cuda.set_stream(self.stream)
        lib.set_stream(self.local, self.stream.cuda_stream)
        if self.world > 1:
            lib.comm_init_torch(self.local)        # the library's own NCCL communicator (b200_comm_init)

    def barrier(self):
        if self.world > 1:
            self.dist.barrier()
        self.torch.cuda.synchronize()

    def max_over_ranks(self, *vals):
        if self.world == 1:
            return list(vals)
        t = self.torch.tensor(list(vals), dtype=self.torch.float64, device="cuda")
        self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
        return [float(x) for x in t]

    def sum_mod_r(self, value, r):
        """sum over ranks of a residue below r (all_gather of its 64-bit limbs)"""
        if self.world == 1:
            return value % r
        nl = (r.bit_length() + 63) // 64
        limbs = [(value >> (64 * k)) & ((1 << 64) - 1) for k in range(nl)]
        t = self.torch.tensor([x - (1 << 64) if x >= (1 << 63) else x for x in limbs], dtype=self.torch.int64, device="cuda")
        parts = [self.torch.empty_like(t) for _ in range(self.world)]
        self.dist.all_gather(parts, t)
        tot = 0
        for p in parts:
            v = [int(x) & ((1 << 64) - 1) for x in p.cpu().tolist()]
            tot += sum(x << (64 * k) for k, x in enumerate(v))
        return tot % r

    def teardown(self):
        self.barrier()
        if self.world > 1:
            self.lib.comm_destroy(self.local)
            self.dist.destroy_process_group()


def timed_region(ctx, fn):
    """barrier + synchronize, CUDA events on the launching stream around fn(), synchronize + barrier; ms, max over ranks"""
    torch = ctx.torch
    ctx.barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    res = fn()
    e1.record()
    ctx.barrier()
    return ctx.max_over_ranks(e0.elapsed_time(e1))[0], res


def msm_leg(ctx):
    """the headline: BN254 G1 MSM 2^20 per GPU (weak scaling)"""
    torch, lib, args = ctx.torch, ctx.lib, ctx.args
    world, rank, local = ctx.world, ctx.rank, ctx.local
    n = 1 << LOG_N
    K, W = args.steps, max(args.warmup, 3)
    C, pts, sc, dot = make_workload(n, SEED, rank)
    expected_local = dlog_point(C, dot)
    expected_total = dlog_point(C, ctx.sum_mod_r(dot, C.r)) if world > 1 else expected_local
    table = lib.Table(lib.BN254, 1, pts, dev=local, precomp=True)
    info = table.info()
    d_sc = torch.from_numpy(sc.view(np.int64)).cuda()
    h_sc = torch.from_numpy(sc.view(np.int64)).pin_memory()
    d_parts = torch.zeros((K, 12), dtype=torch.int64, device="cuda")
    d_tot = torch.zeros((K, 12), dtype=torch.int64, device="cuda")
    h_tot = torch.zeros((K, 12), dtype=torch.int64).pin_memory()
    torch.cuda.synchronize()

    # correctness on the timed input before timing (known-dlog oracle): this rank's partial sum
    table.msm_async(d_sc, d_parts[0], n=n)
    lib.sync(local)
    assert jac_to_affine(C, d_parts[0].cpu().numpy().view(np.uint64)) == expected_local, \
        "GPU MSM does not match the known-discrete-log oracle"

    def run_steps(k):
        """k MSMs back to back (the reduction tail of MSM i overlaps the sort / accumulate of MSM i+1), then - N > 1 -
        one gather + fold of the k partial points on the device"""
        for i in range(k):
            table.msm_pipelined(d_sc, d_parts[i], n=n)
        table.join()
        lib.points_allreduce(local, lib.BN254, 1, d_parts, k, d_tot)

    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()       # samples cover load phase + timed region + e2e region (same kernels throughout)
    for _ in range(W):
        run_steps(1)
    for _ in range(LOAD_STEPS // K + 1):     # fixed count on every rank
        run_steps(K)
    ms, _ = timed_region(ctx, lambda: run_steps(K))
    got = jac_to_affine(C, d_tot[K - 1].cpu().numpy().view(np.uint64))
    assert got == expected_total, "sum over ranks does not match the known-discrete-log oracle"
    if args.dump_outputs and rank == 0:
        # the last timed step's point in affine form, which is unique (Jacobian X, Y, Z are not): gnark-crypto's
        # uncompressed encoding, rows X and Y of 32 big-endian bytes, one exact float64 per byte
        from oracle import encoding
        raw = np.frombuffer(encoding.encode_g1(C, got, compressed=False), dtype=np.uint8)
        os.makedirs(args.dump_outputs, exist_ok=True)
        np.save(os.path.join(args.dump_outputs, "msm_point_affine.npy"), raw.reshape(2, 32).astype(np.float64))

    # ---- end to end through the C ABI with HOST buffers (e2e) -------------------------------------------
    # K x b200_msm_submit_dev (pinned host scalars: H2D on the copy stream, overlapped with the previous MSM), one
    # combine, one download of the K results; wall clock around it, synchronised on both sides
    def e2e_steps(k):
        for i in range(k):
            table.msm_submit_dev(h_sc, d_parts[i], n=n)
        table.join()
        lib.points_allreduce(local, lib.BN254, 1, d_parts, k, d_tot)
        h_tot[:k].copy_(d_tot[:k], non_blocking=True)
        lib.sync(local)
    e2e_steps(2)
    ctx.barrier()
    t0 = time.perf_counter()
    e2e_steps(K)
    e2e_s = time.perf_counter() - t0
    ctx.barrier()
    assert jac_to_affine(C, h_tot[K - 1].numpy().view(np.uint64)) == expected_total
    # the synchronous form of the same call (b200_msm_g1 / b200_msm_allreduce: upload, MSM, combine, download, return)
    table.msm_allreduce(h_sc, n=n)
    ctx.barrier()
    t0 = time.perf_counter()
    for _ in range(K):
        table.msm_allreduce(h_sc, n=n)
    sync_s = time.perf_counter() - t0
    ctx.barrier()
    clocks = sampler.stop() if rank == 0 else None
    e2e_s, sync_s = ctx.max_over_ranks(e2e_s, sync_s)

    # ---- stage profile of the dominant kernel (accumulate), live CUDA events inside the library ----------
    prof = [table.msm_profile(d_sc, d_parts[0], n=n) for _ in range(5)]
    stage_ms = {k: float(np.median([p[k] for p in prof])) for k in prof[0]}
    lib.sync(local)
    table.free()

    total = n * world
    value = total * K / (ms / 1e3)
    peak, peak_src = measured_peak_gbs()
    Wn = info["n_windows"]
    alg_bytes = n * Wn * (64 + 4)           # SURVEY.md §8d: W x (sizeof(affine) + 4 B index) per scalar-mul
    acc_ms = stage_ms["accumulate"]
    achieved = alg_bytes / (acc_ms / 1e3) / 1e9
    traffic, traffic_src = ncu_traffic()
    out = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": K, "warmup": W,
        "ms_per_step": ms / K, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": DTYPE,
        "data": "synthetic", "config": CONFIG,
        "details": {"window_bits": info["window_bits"], "windows": Wn, "precomputed_table": bool(info["precomp"]),
                    "table_bytes": info["device_bytes"],
                    "parallelism": (f"point-range shard x{world}: one ncclAllGather of K x {world} partial points + fold kernel "
                                    "on the device (b200_points_allreduce)") if world > 1 else "single GPU",
                    "l2": "no flush: per-step working set (table %.2f GiB gathered at random + scalars 32 MiB + 256 MiB sort "
                          "buffers) exceeds the 126 MB L2" % (info["device_bytes"] / 2**30)},
        "e2e": {"value": total * K / e2e_s, "unit": UNIT, "h2d_bytes_per_step": n * 32 * world, "d2h_bytes_per_step": 96 * world,
                "ms_per_step": 1e3 * e2e_s / K,
                "note": "K x b200_msm_submit_dev from pinned host scalars (upload overlapped with the previous MSM), combine, "
                        "download of the K results; bases resident (PinToGPU)",
                "synchronous_call": {"value": total * K / sync_s, "ms_per_step": 1e3 * sync_s / K,
                                     "note": "b200_msm_g1 / b200_msm_allreduce: upload, MSM, combine, download, return - per call"}},
        # own kernels per MSM: decompose, bucket_offsets, task_counts, accumulate, combine, combine_heavy,
        # reduce_chunks, set_sum, finish (the radix sort and the scans are CUB launches on top of these)
        "gpu_launches": 9 * K + (1 if world > 1 else 0),
        "roofline": {"bound": "hbm", "kernel": "k_msm_accumulate", "achieved": achieved, "peak": peak, "unit": "GB/s",
                     "frac": achieved / peak, "traffic": traffic, "peak_source": peak_src,
                     "algorithmic_bytes_per_launch": alg_bytes, "kernel_ms": acc_ms, "traffic_source": traffic_src,
                     "multiplier": multiplier_roofline(n * Wn, args.imad_per_add, acc_ms, clocks),
                     "note": "integer-multiplier bound, not HBM bound: >1000 IMAD.WIDE per gathered 68 B (DESIGN.md §3)"},
        "stage_ms": stage_ms,
        "clocks": clocks,
    }
    # the CPU arm beside it (rank 0, N = 1 only): bounded sample of the same workload
    threads = host_threads()
    if world == 1 and not args.no_cpu:
        sample_n = n if threads >= 16 else 1 << 18   # many-core hosts need the full problem to scale
        cpu_rate, cpu_dt, cpu_th, cpu_c, cpu_reps = cpu_msm_rate(C, pts, sc, sample_n, 8.0, threads)
        out["cpu_baseline"] = {"value": cpu_rate, "unit": UNIT, "cores": cpu_th, "kind": "port",
                               "sample": f"{cpu_reps} x BN254 G1 MSM of 2^{int(np.log2(sample_n))} points of the same workload "
                                         f"({cpu_dt:.3f} s each, ~{cpu_reps * cpu_dt * cpu_th:.0f} core-seconds; window c={cpu_c} and "
                                         f"thread count {cpu_th} of {threads} usable picked by a sweep)"}
    else:
        out["cpu_baseline"] = {"value": None, "unit": UNIT, "cores": threads, "kind": "port",
                               "sample": "timed on rank 0 at N=1 only (see the N=1 line)"}
    return out, pts


def strong_leg(ctx, curve_name="bn254", total_log=24, steps=5):
    """ONE MSM of 2^total_log points sharded over the ranks by point range (north_star: BN254 2^24 at 8 GPUs; BASELINE
    configs[4]: BW6-761 2^24): every rank builds ITS shard of known-discrete-log bases on its GPU
    (b200_fixed_base_batch), the result of every step is checked on the full known-dlog sum."""
    torch, lib = ctx.torch, ctx.lib
    from oracle import corelib, derive, ec, ff
    from oracle.params import CURVES
    C = CURVES[curve_name]
    world, rank, local = ctx.world, ctx.rank, ctx.local
    n_total = 1 << total_log
    n = n_total // world
    L, FL = C.fr_limbs, C.fp_limbs
    top = C.r.bit_length() - 64 * (L - 1) - 1
    rs = rng(1000 + rank)
    ks, sc = rand_fr(rs, n, L, top), rand_fr(rs, n, L, top)
    t0 = time.perf_counter()
    d_pts = torch.zeros((n, 2 * FL), dtype=torch.int64, device="cuda")
    d_ks = torch.from_numpy(ks.view(np.int64)).cuda()
    torch.cuda.synchronize()
    # the generator where the oracle holds gnark-crypto's (BN254, BLS12-381), else a derived point of order r on an
    # a = 0 curve over the same field (oracle/derive.py; BW6-761 - the group law never uses b): never the point at
    # infinity, which would make every base trivial
    base = C.g1 if C.g1 is not None else derive.subgroup_point(C, 1)
    assert base is not None
    lib.fixed_base_batch(C.curve_id, 1, ec.pack_points(C, 1, [base]), d_ks, n=n, dev=local, out=d_pts)
    table = lib.Table(C.curve_id, 1, d_pts, dev=local, precomp=True, n=n, on_device=True)
    del d_pts, d_ks
    load_s = time.perf_counter() - t0
    info = table.info()
    dot = corelib.fr_dot(C, ks, sc)
    expected = ec.scalar_mul(ff.Fp(C.p), ctx.sum_mod_r(dot, C.r), base)
    assert expected is not None
    d_sc = torch.from_numpy(sc.view(np.int64)).cuda()
    d_parts = torch.zeros((steps, 3 * FL), dtype=torch.int64, device="cuda")
    d_tot = torch.zeros((steps, 3 * FL), dtype=torch.int64, device="cuda")
    torch.cuda.synchronize()

    def run(k):
        for i in range(k):
            table.msm_pipelined(d_sc, d_parts[i], n=n)
        table.join()
        lib.points_allreduce(local, C.curve_id, 1, d_parts, k, d_tot)
    run(2)
    ms, _ = timed_region(ctx, lambda: run(steps))
    ok = jac_to_affine(C, d_tot[steps - 1].cpu().numpy().view(np.uint64)) == expected
    # latency of ONE sharded MSM, result on the host: submit, combine, download, return
    lat = []
    h_one = torch.zeros(3 * FL, dtype=torch.int64).pin_memory()
    for _ in range(4):
        ctx.barrier()
        t0 = time.perf_counter()
        table.msm_async(d_sc, d_parts[0], n=n)
        lib.points_allreduce(local, C.curve_id, 1, d_parts, 1, d_tot)
        h_one.copy_(d_tot[0], non_blocking=True)
        lib.sync(local)
        lat.append(1e3 * (time.perf_counter() - t0))
    lat_ms = ctx.max_over_ranks(float(np.median(lat[1:])))[0]
    prof = table.msm_profile(d_sc, d_parts[0], n=n)
    lib.sync(local)
    table.free()
    return {"metric": f"{curve_name}_g1_msm_2^{total_log}_sharded", "scaling": "strong", "n_gpus": world, "points_total": n_total,
            "points_per_gpu": n, "value": n_total * steps / (ms / 1e3), "unit": UNIT, "ms_per_msm": ms / steps,
            "single_msm_latency_ms": lat_ms, "steps": steps, "correct": bool(ok),
            "check": "full known-discrete-log sum over all shards, every base distinct (k_i * G built on the GPU)",
            "window_bits": info["window_bits"], "windows": info["n_windows"], "table_bytes_per_gpu": info["device_bytes"],
            "table_build_s": load_s, "stage_ms_rank0": prof,
            "combine": "one ncclAllGather + k_points_fold on the device" if world > 1 else "none (single GPU)"}


def groth16_leg(ctx):
    """Secondary BASELINE metric: Groth16 prove ms at 2^20 R1CS (configs[2]), BN254.
    From "A,B,C,W on the host" to "3 proof points on the host" (solver excluded, as in SURVEY.md §8d config 3):
    7 NTT(2^20) + 4 G1 MSM + 1 G2 MSM + host-side assembly.  The instance is a SATISFIED circuit of 2^20 - 1
    constraints with a trapdoor key (oracle/groth16_fast.py; key points built on the GPU with b200_fixed_base_batch):
    before timing, one proof with injected r, s is checked - the three proof points equal dlog * generator and the
    verifier's pairing equation holds on them (backend/groth16/bn254/verify.go:38-140)."""
    from gnark_b200 import groth16 as g16
    from oracle import ec
    from oracle import groth16_fast as gf
    from oracle.params import BN254 as C
    torch, lib = ctx.torch, ctx.lib
    dev, rank, world = ctx.local, ctx.rank, ctx.world
    t0 = time.perf_counter()
    inst = gf.satisfied_instance(C, LOG_N, seed=20)          # the same instance on every rank (each loads its shard)
    fb = lambda group, dl: lib.fixed_base_batch(C.curve_id, group, ec.pack_points(C, group, [C.g1 if group == 1 else C.g2]),
                                                np.ascontiguousarray(dl), dev=dev)
    kp = gf.key_points(inst, fb)
    pk = g16.ProvingKey.from_arrays(g16.BN254, inst.n, kp["alpha"], kp["beta"], kp["delta"], kp["A"], kp["B"], kp["Z"], kp["K"],
                                    kp["beta2"], kp["delta2"], kp["B2"], inst.inf_a, inst.inf_b, inst.nb_public)
    fixture_s = time.perf_counter() - t0
    opts = [g16.WithDeviceID(dev), g16.WithSharding(rank, world)]
    t0 = time.perf_counter()
    pk.setup_device_pointers(g16.NewConfig(*opts))
    setup_s = time.perf_counter() - t0
    a, b, c = inst.solution_abc()
    sol_pageable = g16.R1CSSolution(W=inst.wires(), A=a, B=b, C=c)
    # the solver's output vectors live in C-owned pinned buffers (b200_host_alloc, INTEGRATION.md §3)
    keep = [torch.from_numpy(v.view(np.int64)).pin_memory() for v in (sol_pageable.W, sol_pageable.A, sol_pageable.B, sol_pageable.C)]
    sol = g16.R1CSSolution(*[k.numpy().view(np.uint64) for k in keep])
    # one checked proof (r, s injected, the same on every rank)
    rs = iter([0x5EED << 200 | 1, 0xFACE << 190 | 2])
    proof = g16.ProveSolution(pk, sol, *opts, g16.WithRandomness(lambda q: next(rs)))
    verified = None
    if rank == 0:
        t0 = time.perf_counter()
        e = gf.expected(inst, 0x5EED << 200 | 1, 0xFACE << 190 | 2)
        verified = bool(gf.verify_points(inst, ec.unpack_points(C, 1, proof.Ar)[0], ec.unpack_points(C, 2, proof.Bs)[0],
                                         ec.unpack_points(C, 1, proof.Krs)[0], e, with_pairing=True))
        verify_s = time.perf_counter() - t0
    times = []
    for i in range(10):          # fixed count on every rank
        cur = sol if i < 6 else sol_pageable
        ctx.barrier()
        t0 = time.perf_counter()
        g16.ProveSolution(pk, cur, *opts)
        times.append(ctx.max_over_ranks(1e3 * (time.perf_counter() - t0))[0])
    pk.free_gpu_resources()
    out = {"metric": "groth16_prove_ms", "n_constraints": inst.m, "n_wires": inst.nb_wires, "curve": "bn254", "n_gpus": world,
           "parallelism": ("every MSM table point-range sharded x%d, computeH replicated, 5 partial points combined on the "
                           "device (ncclAllGather + fold)" % world) if world > 1 else "single GPU",
           "prove_ms_median": float(np.median(times[1:6])), "prove_ms_min": float(min(times[1:6])),
           "prove_ms_pageable_median": float(np.median(times[6:])),
           "first_call_ms": times[0], "key_load_s": setup_s, "fixture_s": fixture_s,
           "includes": "H2D of W,A,B,C (4 x 32 MiB, pinned host buffers; pageable variant reported beside it), "
                       "computeH (7 NTT), 5 MSM, combine, D2H, host assembly",
           "excludes": "R1CS solver (CPU, out of scope)",
           "data": "satisfied product-network circuit, trapdoor key with 2^20 distinct bases per table (oracle/groth16_fast.py)"}
    if rank == 0:
        out["verified"] = verified
        out["verify_s"] = verify_s
        out["check"] = ("proof points == dlog * generator (trapdoor key) and e(Ar,Bs) = e(alpha,beta) e(sum w_i K_i, gamma) "
                        "e(Krs,delta) on the proof points with a real pairing")
    return out


def plonk_leg(ctx, log2n):
    """BASELINE configs[3]: PLONK prove, BLS12-381, 2^22 gates, one b200_plonk_prove call per proof on a SATISFIED
    instance with a trapdoor SRS; the proof is checked by the verifier's equations (oracle/plonk_fast.py) before timing.
    Runs on rank 0's GPU (single-GPU prover; the sharded prover is tools/bench_plonk_multi.py)."""
    from oracle import plonk_fast
    from oracle.params import CURVES
    lib = ctx.lib
    c = CURVES["bls12-381"]
    t0 = time.perf_counter()
    inst = plonk_fast.satisfied_instance(c, log2n, seed=22)
    srs = plonk_fast.trapdoor_srs_gpu(lib, c, inst, dev=ctx.local)
    gen_s = time.perf_counter() - t0
    t0 = time.perf_counter()
    key = lib.PlonkKey(c.curve_id, log2n, inst.ql, inst.qr, inst.qm, inst.qo, inst.qk, inst.perm, srs, dev=ctx.local)
    load_s = time.perf_counter() - t0
    ch = inst.challenges_packed()
    # the solver's output columns in pinned host memory (b200_host_alloc in the Go shim; INTEGRATION.md §3), as in the
    # Groth16 leg; one run from pageable memory is reported beside it
    torch = ctx.torch
    keep = [torch.from_numpy(v.view(np.int64)).pin_memory() for v in (inst.l, inst.r, inst.o)]
    lp, rp, op = [k.numpy().view(np.uint64) for k in keep]
    times, stage_runs = [], []
    pts = vals = None
    for _ in range(5):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        pts, vals = key.prove(lp, rp, op, *ch)
        times.append(1e3 * (time.perf_counter() - t0))
        stage_runs.append(key.last_stage_ms())
    t0 = time.perf_counter()
    key.prove(inst.l, inst.r, inst.o, *ch)
    pageable_ms = 1e3 * (time.perf_counter() - t0)
    # per-stage median over the calls after the first
    stages = {k: float(np.median([r[k] for r in stage_runs[1:]])) for k in stage_runs[0]}
    key.free()
    t0 = time.perf_counter()
    ok = plonk_fast.verify(c, inst, pts, vals)
    verify_s = time.perf_counter() - t0
    return {"metric": "plonk_prove_ms", "curve": "bls12-381", "log2_gates": log2n, "n_gpus": 1,
            "prove_ms_median": float(np.median(times[1:])), "prove_ms_min": float(min(times[1:])), "first_call_ms": times[0],
            "prove_ms_pageable": pageable_ms, "verified": bool(ok), "check": "verifier's equations on the ten proof points and seven values (trapdoor SRS: "
            "openings checked as [f] - f(z)[1] + z[H] == tau [H]; oracle/plonk_fast.py), satisfied instance",
            "stage_ms": stages, "prove_ms_all": times, "key_load_s": load_s, "fixture_s": gen_s, "verify_s": verify_s,
            "includes": "H2D of L,R,O (3 x 128 MiB, pinned host buffers; pageable variant beside it), NTTs, 4 fused constraint passes, iNTT 4n, 10 KZG commitments (MSM), grand product, "
                        "evaluations, opening quotients, D2H of 10 points + 7 values",
            "excludes": "solver, Fiat-Shamir hashing (challenges injected by the caller, as the Go shim does)"}


def run_b200(args):
    ctx = Ctx(args)
    out, pts = msm_leg(ctx)

    def headline_only(name):
        def f():
            out.setdefault(name, {"error": "leg did not finish within %d s" % LEG_LIMIT_S[name]})
            if ctx.rank == 0:
                emit(out)
        return f
    legs = []
    if not args.no_strong:
        legs.append(("strong", lambda: strong_leg(ctx, "bn254", args.strong_log)))
    if not args.no_groth16:
        legs.append(("groth16", lambda: groth16_leg(ctx)))
    if args.bw6 or (args.bw6 is None and ctx.world == 8):
        legs.append(("bw6", lambda: strong_leg(ctx, "bw6-761", args.bw6_log, steps=3)))
    for name, fn in legs:
        dog = arm_watchdog(LEG_LIMIT_S[name], headline_only(name))
        try:
            out[name] = fn()
        except Exception as e:  # the headline metric must still be printed
            out[name] = {"error": repr(e)}
        dog.cancel()
        ctx.torch.cuda.empty_cache()
    if not args.no_plonk and ctx.rank == 0:     # single-GPU leg, no collective inside
        dog = arm_watchdog(LEG_LIMIT_S["plonk"], headline_only("plonk"))
        try:
            out["plonk"] = plonk_leg(ctx, args.plonk_log)
        except Exception as e:
            out["plonk"] = {"error": repr(e)}
        dog.cancel()
    if ctx.rank == 0:
        emit(out)
    dog = arm_watchdog(120)       # the line is out; a hung NCCL teardown must not turn into a driver timeout
    ctx.teardown()
    dog.cancel()


def arm_watchdog(seconds, last_words=None, code=0):
    """a stuck secondary leg (a rank lost inside a collective) must not cost the headline line: after
    `seconds` run last_words() (rank 0: print what is already measured) and leave.  Never fires on a healthy run:
    the process then ends through the normal interpreter exit."""
    def fire():
        try:
            if last_words is not None:
                last_words()
        finally:
            sys.stderr.write("bench.py: watchdog fired after %d s\n" % seconds)
            sys.stderr.flush()
            os._exit(code)
    t = threading.Timer(seconds, fire)
    t.daemon = True
    t.start()
    return t


_REAL_STDOUT = None
_EMITTED = False


def emit(obj):
    """the ONE JSON line on the real stdout (fd 1 is pointed at stderr while the bench runs, so that
    library chatter such as NCCL's version banner cannot pollute it)"""
    global _EMITTED
    if _EMITTED:
        return
    _EMITTED = True
    line = (json.dumps(obj) + "\n").encode()
    os.write(_REAL_STDOUT if _REAL_STDOUT is not None else 1, line)


def main():
    global _REAL_STDOUT
    sys.stdout.flush()
    _REAL_STDOUT = os.dup(1)
    os.dup2(2, 1)
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--no-groth16", action="store_true", help="skip the Groth16 2^20 prove-time leg (configs[2])")
    ap.add_argument("--no-strong", action="store_true", help="skip the strong-scaling leg (one 2^24 BN254 MSM over N GPUs)")
    ap.add_argument("--no-plonk", action="store_true", help="skip the PLONK BLS12-381 prove leg (configs[3])")
    ap.add_argument("--no-cpu", action="store_true", help="skip the CPU baseline beside the N=1 line")
    ap.add_argument("--strong-log", type=int, default=24)
    ap.add_argument("--plonk-log", type=int, default=22)
    ap.add_argument("--bw6", action="store_true", default=None, help="BW6-761 G1 MSM 2^24 sharded (configs[4]); default: at N=8")
    ap.add_argument("--bw6-log", type=int, default=24)
    ap.add_argument("--imad-per-add", type=int, default=1360,
                    help="IMAD.WIDE per XYZZ mixed addition of the shipped kernel (static SASS count, profiles/)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="CUDA arm: after the timed steps, write the MSM result of the last step to DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    dog = arm_watchdog(WHOLE_RUN_LIMIT_S, code=1)
    if args.impl == "reference":
        run_reference(args)
    else:
        run_b200(args)
    dog.cancel()
    sys.stdout.flush()
    sys.stderr.flush()


if __name__ == "__main__":
    main()
