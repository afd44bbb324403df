#!/usr/bin/env python3
"""Randomised parity soak ON THE GPU: random (curve, group, size, table kind, scalar pattern, sub-range) MSMs, random
NTT sizes / modes, computeH, fixed-base batches and gather-index MSMs through the C ABI, each compared bit for bit with
the C++ oracle (oracle/c/oracle.cpp) on the same seeded input.  Test infrastructure (it imports oracle/); the fixed
cases live in tests/test_gpu_*.py, this tool widens them with sizes and patterns nobody picked by hand.

    python tools/fuzz_gpu.py --seconds 300 --seed 1 > gpurun_out/fuzz_gpu.jsonl

One JSON line per case class at the end (cases run, failures with their reproducer seeds); exit code 1 on any mismatch.

    python tools/fuzz_gpu.py --field 600 --seed 1 > field_soak.jsonl

runs only the field-arithmetic soak instead (every device field template against an independent reference on
carry-hunting operands, tests/cuda/field_soak.cu; `make` builds tests/_build/libgb200_fieldsoak.so).
"""
import argparse
import json
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

from oracle import corelib, derive, ec, ff  # noqa: E402
from oracle.params import CURVES  # noqa: E402
from gnark_b200 import lib  # noqa: E402

NAMES = ["bn254", "bls12-381", "bls12-377", "bw6-761"]


def rand_fr(rs, c, count, pattern):
    """Montgomery limb arrays: uniform residues, or the skewed shapes real witnesses have (zeros, ones, small values,
    r - 1, repeated values), which stress the heavy-bucket path and the signed-digit carries"""
    L = c.fr_limbs
    a = rs.integers(0, 1 << 64, size=(count, L), dtype=np.uint64)
    a[:, L - 1] &= np.uint64((1 << (c.r.bit_length() - 64 * (L - 1) - 1)) - 1)
    if pattern == "uniform" or count == 0:
        return a
    special = ff.pack_elements([0, 1, 2, c.r - 1, c.r - 2, (c.r - 1) // 2, 1 << 16, (1 << 16) - 1, 1 << 15], c.r, L)
    pick = rs.integers(0, len(special), size=count)
    u = rs.random(count)
    if pattern == "skewed":          # half special values, half uniform
        m = u < 0.5
    elif pattern == "sparse":        # mostly zero
        m = u < 0.9
        pick[:] = 0
    else:                            # "equal": one value repeated (one bucket per window takes everything)
        m = np.ones(count, dtype=bool)
        pick[:] = int(rs.integers(0, len(special)))
        if rs.random() < 0.5:
            a[:] = a[0]
            m[:] = False
    a[m] = special[pick[m]]
    return a


def base_point(c, group):
    g = c.g1 if group == 1 else c.g2
    return g if g is not None else derive.subgroup_point(c, group)


def case_msm(rs, seed):
    c = CURVES[NAMES[int(rs.integers(0, 4))]]
    group = 1 if c.name == "bw6-761" and rs.random() < 0.5 else int(rs.integers(1, 3))
    big = rs.random() < 0.15
    n = int(rs.integers(1, 1 << 16)) if big else int(rs.integers(1, 3000))
    if c.fp_limbs > 6 or group == 2:
        n = min(n, 1 << 13)
    precomp = bool(rs.integers(0, 2))
    pattern = ["uniform", "skewed", "sparse", "equal"][int(rs.integers(0, 4))]
    ks = rand_fr(rs, c, n, "uniform")
    if rs.random() < 0.2:
        ks[int(rs.integers(0, n))] = 0                     # a base at infinity inside the table
    if rs.random() < 0.2 and n > 1:
        ks[1] = ks[0]                                       # two equal bases
    pts = corelib.fixed_base(c, group, ec.pack_points(c, group, [base_point(c, group)]), ks)
    sc = rand_fr(rs, c, n, pattern)
    t = lib.Table(c.curve_id, group, pts, precomp=precomp)
    off = int(rs.integers(0, n)) if rs.random() < 0.3 else 0
    cnt = int(rs.integers(0, n - off + 1)) if rs.random() < 0.3 else n - off
    got = t.msm(np.ascontiguousarray(sc[:cnt]), off=off, n=cnt)
    t.free()
    if cnt == 0:
        want_aff = None
    else:
        want = corelib.msm(c, group, np.ascontiguousarray(pts[off:off + cnt]), np.ascontiguousarray(sc[:cnt]))
        want_aff = aff(c, group, want)
    ok = aff(c, group, got) == want_aff
    return ok, dict(curve=c.name, group=group, n=n, off=off, cnt=cnt, precomp=precomp, pattern=pattern)


def aff(c, group, jac):
    return ec.from_jac(ff.base_field(c, group), ec.unpack_points(c, group, np.ascontiguousarray(jac), ncoords=3)[0])


def case_ntt(rs, seed):
    c = CURVES[NAMES[int(rs.integers(0, 4))]]
    logn = int(rs.integers(0, 19 if c.fr_limbs <= 4 else 17))
    inverse, dec, coset = bool(rs.integers(0, 2)), int(rs.integers(0, 2)), bool(rs.integers(0, 2))
    x = rand_fr(rs, c, 1 << logn, ["uniform", "skewed"][int(rs.integers(0, 2))])
    d = lib.Domain(c.curve_id, logn)
    got = d.ntt(x.copy(), inverse=inverse, decimation=dec, on_coset=coset)
    d.free()
    want = corelib.ntt(c, x.copy(), logn, inverse, dec, coset)
    return np.array_equal(np.asarray(got).reshape(-1), np.asarray(want).reshape(-1)), dict(
        curve=c.name, logn=logn, inverse=inverse, decimation=dec, coset=coset)


def case_compute_h(rs, seed):
    c = CURVES[NAMES[int(rs.integers(0, 4))]]
    logn = int(rs.integers(1, 17 if c.fr_limbs <= 4 else 15))
    n = 1 << logn
    length = int(rs.integers(max(1, n // 2), n + 1))
    L = c.fr_limbs
    v = [rand_fr(rs, c, length, "uniform") for _ in range(3)]
    d = lib.Domain(c.curve_id, logn)
    got = d.compute_h(v[0], v[1], v[2], length=length)
    d.free()
    pads = []
    for x in v:
        p = np.zeros((n, L), dtype=np.uint64)
        p[:length] = x
        pads.append(p)
    want = corelib.compute_h(c, pads[0], pads[1], pads[2], logn)
    return np.array_equal(np.asarray(got).reshape(-1), np.asarray(want).reshape(-1)), dict(curve=c.name, logn=logn, length=length)


def case_fixed_base(rs, seed):
    c = CURVES[NAMES[int(rs.integers(0, 4))]]
    group = int(rs.integers(1, 3))
    n = int(rs.integers(1, 4000 if c.fp_limbs <= 6 else 800))
    ks = rand_fr(rs, c, n, ["uniform", "skewed", "sparse"][int(rs.integers(0, 3))])
    base = ec.pack_points(c, group, [base_point(c, group)])
    got = lib.fixed_base_batch(c.curve_id, group, base, ks)
    want = corelib.fixed_base(c, group, base, ks)
    return np.array_equal(np.asarray(got).reshape(-1), np.asarray(want).reshape(-1)), dict(curve=c.name, group=group, n=n)


def case_gather(rs, seed):
    c = CURVES[NAMES[int(rs.integers(0, 2))]]
    n = int(rs.integers(2, 5000))
    ks = rand_fr(rs, c, n, "uniform")
    pts = corelib.fixed_base(c, 1, ec.pack_points(c, 1, [base_point(c, 1)]), ks)
    nv = int(rs.integers(n, 3 * n))
    vals = rand_fr(rs, c, nv, ["uniform", "skewed"][int(rs.integers(0, 2))])
    idx = np.sort(rs.choice(nv, size=n, replace=False)).astype(np.uint32)
    t = lib.Table(c.curve_id, 1, pts, precomp=bool(rs.integers(0, 2)))
    got = t.msm_gather(idx, vals)
    t.free()
    want = corelib.msm(c, 1, pts, np.ascontiguousarray(vals[idx]))
    return aff(c, 1, got) == aff(c, 1, want), dict(curve=c.name, n=n, nv=nv)


def case_known_dlog_big(rs, seed):
    """rare-event detector: a 2^17..2^20-point MSM over DISTINCT bases k_i * G built on the GPU (b200_fixed_base_batch),
    checked against (sum s_i k_i) * G - one dot product and one scalar multiplication on the CPU.  One such case runs
    10^8..10^10 field reductions (table build included), which is what it took to see the lost carry of round 2's first
    mont_reduce_wide (about 2^-32.5 per reduction)."""
    import torch
    c = CURVES[NAMES[int(rs.integers(0, 4))]]
    group = BIG_GROUP or int(rs.integers(1, 3))
    logn = int(rs.integers(17, 21))
    if c.fp_limbs > 6:
        logn = min(logn, 18)
    if group == 2 and c.fp_limbs > 4:
        logn = min(logn, 19)
    n = (1 << logn) - int(rs.integers(0, 1000))
    ks, sc = rand_fr(rs, c, n, "uniform"), rand_fr(rs, c, n, ["uniform", "uniform", "skewed"][int(rs.integers(0, 3))])
    G = base_point(c, group)
    deg = 1 if group == 1 or c.name == "bw6-761" else 2
    d_pts = torch.zeros((n, 2 * deg * c.fp_limbs), dtype=torch.int64, device="cuda")
    lib.fixed_base_batch(c.curve_id, group, ec.pack_points(c, group, [G]), torch.from_numpy(ks.view(np.int64)).cuda(), n=n, out=d_pts)
    precomp = bool(rs.integers(0, 2))
    t = lib.Table(c.curve_id, group, d_pts, precomp=precomp, n=n, on_device=True)
    del d_pts
    got = aff(c, group, t.msm(sc))
    t.free()
    want = ec.scalar_mul(ff.base_field(c, group), corelib.fr_dot(c, ks, sc), G)
    return got == want, dict(curve=c.name, group=group, n=n, precomp=precomp)


BIG_GROUP = 0     # --big-group: 1 / 2 pins the group of the big cases (2: the Fp2 arithmetic)


def card_info():
    """name, power limit and max SM clock of the card the soak runs on (read-only nvidia-smi query)"""
    import subprocess
    dev = os.environ.get("CUDA_VISIBLE_DEVICES", "0").split(",")[0] or "0"
    try:
        out = subprocess.run(["nvidia-smi", "-i", dev, "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=60).stdout.strip().splitlines()
        name, power, clock = (x.strip() for x in out[0].split(","))
        return {"gpu": name, "power_limit": power, "max_sm_clock": clock}
    except Exception as e:              # the numbers stay usable, the card just goes unnamed
        return {"gpu": "unknown (%r)" % e}


def field_soak(seconds, seed, lib_name="libgb200_fieldsoak.so", target=0.25):
    """--field: tests/cuda/field_soak.cu's fs_soak round-robin over every (field, op, generator) of the device field
    templates with fresh seeds, product against the independent reference in the same kernel.  Each call is sized from
    the rate of the previous one to take about `target` seconds.  Prints one header line (card, power limit), one line
    per (field, op, generator) with samples, mismatches and rate, and the recorded mismatches checked with big ints."""
    import fieldsoak as fs
    slib = fs.load(lib_name)
    head = {"kind": "field_soak", "seed": seed, "seconds": seconds, "lib": lib_name, **card_info()}
    print(json.dumps(head), flush=True)
    cases = [(f, op, gen) for f in fs.DEVICE_FIELDS for op in f.ops if op != "reduce_mutant" for gen in fs.gens_for(op)]
    count = {c: (1 << 12 if c[1] == "inverse" else 1 << 20) for c in cases}
    tot = {c: {"samples": 0, "mismatches": 0, "seconds": 0.0, "calls": 0} for c in cases}
    failures = []
    t0 = last = time.time()
    rnd = 0
    while time.time() - t0 < seconds:
        for c in cases:
            if time.time() - last >= 30:        # progress line: a long soak keeps writing
                last = time.time()
                print(json.dumps({"kind": "field_soak_progress", "elapsed": round(last - t0, 1), "round": rnd,
                                  "samples": sum(st["samples"] for st in tot.values()),
                                  "mismatches": sum(st["mismatches"] for st in tot.values())}), flush=True)
            if time.time() - t0 >= seconds:
                break
            f, op, gen = c
            s = (seed * 1_000_003 + rnd) * 4099 + f.fid
            t = time.perf_counter()
            m, recs = fs.soak(slib, f, op, gen, s, count[c])
            dt = time.perf_counter() - t
            st = tot[c]
            st["samples"] += count[c]
            st["mismatches"] += m
            st["seconds"] += dt
            st["calls"] += 1
            if m:
                msg = fs.triage(f, op, gen, s, recs, "device")
                failures.append({"field": f.name, "op": op, "gen": gen, "seed": s, "mismatches": m, "triage": msg})
                sys.stderr.write(msg + "\n")
            count[c] = int(min(max(count[c] * target / max(dt, 1e-3), 1 << 10), 1 << 34))
        rnd += 1
    for (f, op, gen), st in tot.items():
        if st["calls"]:
            print(json.dumps({"kind": "field_soak_case", "field": f.name, "op": op, "gen": gen, **st,
                              "rate_per_s": st["samples"] / st["seconds"] if st["seconds"] else None}))
    summ = {"kind": "field_soak_total", "rounds": rnd, "wall_seconds": time.time() - t0,
            "samples": sum(st["samples"] for st in tot.values()),
            "mismatches": sum(st["mismatches"] for st in tot.values()), "failures": failures}
    print(json.dumps(summ))
    return 1 if summ["mismatches"] else 0


CASES = {"msm": (case_msm, 5), "known_dlog_big": (case_known_dlog_big, 0), "ntt": (case_ntt, 3), "compute_h": (case_compute_h, 1), "fixed_base": (case_fixed_base, 1),
         "gather": (case_gather, 1)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--seconds", type=float, default=120)
    ap.add_argument("--seed", type=int, default=1)
    ap.add_argument("--only", default="")
    ap.add_argument("--big", type=float, default=0.0, help="weight of the 2^17..2^20 known-discrete-log MSM cases (0 = off)")
    ap.add_argument("--big-group", type=int, default=0, help="pin the group (1 or 2) of the big cases")
    ap.add_argument("--field", type=float, default=0.0,
                    help="run only the device field-arithmetic soak for this many seconds (tests/cuda/field_soak.cu)")
    ap.add_argument("--field-lib", default="libgb200_fieldsoak.so",
                    help="soak library under tests/_build (libgb200_hostemu.so rehearses --field on a CPU)")
    args = ap.parse_args()
    if args.field > 0:
        sys.exit(field_soak(args.field, args.seed, args.field_lib))
    global BIG_GROUP
    BIG_GROUP = args.big_group
    lib.load()
    lib.init([0])
    names = [k for k in CASES if not args.only or k in args.only.split(",")]
    weights = np.array([args.big if k == "known_dlog_big" else CASES[k][1] for k in names], dtype=float)
    weights /= weights.sum()
    top = np.random.Generator(np.random.PCG64(args.seed))
    stats = {k: {"cases": 0, "failures": []} for k in names}
    t0 = time.time()
    i = 0
    while time.time() - t0 < args.seconds:
        kind = names[int(top.choice(len(names), p=weights))]
        seed = args.seed * 1_000_003 + i
        rs = np.random.Generator(np.random.PCG64(seed))
        try:
            ok, desc = CASES[kind][0](rs, seed)
        except Exception as e:          # an error return of the library on a valid input is a failure too
            ok, desc = False, {"exception": repr(e)}
        stats[kind]["cases"] += 1
        if not ok:
            stats[kind]["failures"].append({"seed": seed, **desc})
            sys.stderr.write("MISMATCH %s %s\n" % (kind, json.dumps({"seed": seed, **desc})))
        i += 1
    bad = 0
    for k in names:
        bad += len(stats[k]["failures"])
        print(json.dumps({"kind": k, "cases": stats[k]["cases"], "failures": stats[k]["failures"], "seed": args.seed,
                          "seconds": args.seconds}))
    sys.exit(1 if bad else 0)


if __name__ == "__main__":
    main()
