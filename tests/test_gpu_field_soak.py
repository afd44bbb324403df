"""Field-arithmetic soak ON THE DEVICE (tests/_build/libgb200_fieldsoak.so: tests/cuda/field_soak.cu built by nvcc
with the product's flags): the field templates as the device runs them - carry flag live across separate asm
statements after scheduling, BW6-761 Fp's out-of-line by-value product, the out-of-line Fp2 product and square - against
Python big ints (exact evaluation) and against the independent reference of tests/cuda/field_soak.cuh computed in the
same kernel (soak).  A mismatch is counted and recorded, never trapped; every recorded one is checked again here with
big ints, and the failure message says which side is wrong and carries the operands."""
import os
import subprocess
import time

import pytest

import fieldsoak as fs

pytestmark = pytest.mark.gpu

# samples per (field, op, generator): the carry-chain cases (the product and the reduction under G1, the reduction under
# G3, the Fp2 product under G1) get BIG, inverse (a^(p-2)) gets INVERSE, everything else DEFAULT.  Sized from the rates
# measured on a B200 (DESIGN.md section 3) to keep this file at about two minutes; the palette generator G1 is the
# slowest (rejection of values >= p), so BW6-761 Fp and the 381/377-bit Fp2 products get a quarter of BIG.
BIG = 1 << 32
DEFAULT = 1 << 25
INVERSE = 1 << 16


@pytest.fixture(scope="module")
def soakdev():
    import torch
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    subprocess.check_call(["make", "-j", str(os.cpu_count() or 1), "-C", os.path.join(fs.ROOT, "gnark_b200", "csrc"),
                           "../../tests/_build/libgb200_fieldsoak.so"])
    return fs.load("libgb200_fieldsoak.so")


def seed_of(f, op, gen):
    return 7_000_003 * f.fid + 101 * fs.OPS[op] + fs.GENS[gen] + 3


def volume(f, op, gen):
    if op == "inverse":
        return INVERSE // 4 if f.N > 12 else INVERSE
    big = (op == "mul" and gen == "G1") or (op == "mont_reduce_wide" and gen in ("G1", "G3"))
    if not big:
        return DEFAULT
    return BIG // 4 if f.N > 12 or (f.beta is not None and f.N > 8) else BIG


@pytest.mark.parametrize("f", fs.DEVICE_FIELDS, ids=str)
def test_device_exact_evaluation(soakdev, f):
    """fs_eval (the product templates in a kernel) on the G1 and G2 operand sets of every op against big ints; inverse
    of 0 stays 0"""
    for op in f.ops:
        if op == "reduce_mutant":
            continue
        for gen in fs.gens_for(op):
            if gen == "G0":
                continue
            n = 200 if op == "inverse" else 3000
            a, b = fs.operands(soakdev, f, op, gen, seed_of(f, op, gen), 0, n)
            if op == "inverse":
                a[0] = (0, 0) if f.beta is not None else 0
            got = fs.evaluate(soakdev, f, op, a, b)
            bad = [i for i in range(n) if got[i] != fs.expected(f, op, a[i], b[i])]
            assert not bad, "device %s %s %s: %d wrong, first: a=%s b=%s got=%s big=%s" % (
                f, op, gen, len(bad), fs._hex(a[bad[0]]), fs._hex(b[bad[0]]), fs._hex(got[bad[0]]),
                fs._hex(fs.expected(f, op, a[bad[0]], b[bad[0]])))


@pytest.mark.parametrize("f", fs.DEVICE_FIELDS, ids=str)
def test_device_soak(soakdev, f):
    """Every op x generator of one field, product and reference in the same kernel: 0 mismatches"""
    fails = []
    for op in f.ops:
        if op == "reduce_mutant":
            continue
        for gen in fs.gens_for(op):
            seed = seed_of(f, op, gen)
            n = volume(f, op, gen)
            t0 = time.perf_counter()
            m, recs = fs.soak(soakdev, f, op, gen, seed, n)
            dt = time.perf_counter() - t0
            print("field_soak %s %s %s samples=%d mismatches=%d seconds=%.3f rate=%.3g/s" % (f, op, gen, n, m, dt, n / dt))
            if m:
                fails.append("%d mismatches in %d samples\n%s" % (m, n, fs.triage(f, op, gen, seed, recs, "device")))
    assert not fails, "\n".join(fails)


@pytest.mark.parametrize("f", [f for f in fs.DEVICE_FIELDS if f.beta is None], ids=str)
def test_device_soak_catches_the_lost_carry(soakdev, f):
    """Power on the device: round 2's first mont_reduce_wide is caught under G3 at DEFAULT samples on every field, and
    each record is confirmed by big ints as the mutant's error"""
    seed = seed_of(f, "reduce_mutant", "G3")
    m, recs = fs.soak(soakdev, f, "reduce_mutant", "G3", seed, DEFAULT)
    assert m > 0, f
    for r in recs:
        assert r["want"] == fs.expected(f, "mont_reduce_wide", r["a"], r["b"]) != r["got"], fs.triage(
            f, "reduce_mutant", "G3", seed, [r], "device")
