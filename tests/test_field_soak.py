"""Field-arithmetic soak on the CPU (tests/cuda/field_soak.cu built into the emulation library): every op of every
field template against the independent 64-bit-limb reference of tests/cuda/field_soak.cuh, on operands built to sit at
carry-chain edges, plus the host-only Montgomery code of the product (HFp, Fp2<HFp>, HostFrCtx).

Uniform operands alone have no power against a carry lost at a saturated word (round 2's first mont_reduce_wide passed
every uniform test); the palette (G1), boundary (G2) and direct reduction-input (G3) generators do, which the
reduce_mutant test shows on every field."""
import pytest

import fieldsoak as fs

VOLUME = 100_000            # samples per (field, op, generator)
INVERSE_VOLUME = 1_000      # a^(p-2): ~1.5 bits products per sample


@pytest.fixture(scope="module")
def soaklib(hostemu):
    return fs.bind(hostemu)


def seed_of(f, op, gen):
    return 1_000_003 * f.fid + 101 * fs.OPS[op] + fs.GENS[gen] + 7


def volume(f, op):
    if op == "inverse":
        return INVERSE_VOLUME // 4 if f.N > 12 else INVERSE_VOLUME
    return VOLUME


@pytest.mark.parametrize("f", fs.DEVICE_FIELDS, ids=str)
def test_reference_and_product_against_big_ints(soaklib, f):
    """The reference (fs_ref_eval) and the emulated product template (fs_eval) against Python big ints on the G1 and
    G2 operand sets of every op (G3 too for the reductions); the generated operands are inside the op's input range"""
    for op in f.ops:
        for gen in fs.gens_for(op):
            n = 20 if op == "inverse" else 400
            a, b = fs.operands(soaklib, f, op, gen, seed_of(f, op, gen), 0, n)
            if gen == "G0":
                continue
            lim = f.q * f.R if op in fs.REDUCE_OPS else f.q
            flat = [x for v in a for x in (v if f.beta is not None else (v,))]
            assert all(0 <= x < lim for x in flat), (f, op, gen)
            want = [fs.expected(f, op, x, y) for x, y in zip(a, b)]
            ref = fs.evaluate(soaklib, f, op, a, b, entry="fs_ref_eval")
            bad = [i for i in range(n) if ref[i] != want[i]]
            assert not bad, "reference %s %s %s: a=%s b=%s ref=%s big=%s" % (
                f, op, gen, fs._hex(a[bad[0]]), fs._hex(b[bad[0]]), fs._hex(ref[bad[0]]), fs._hex(want[bad[0]]))
            if op == "reduce_mutant":
                continue
            got = fs.evaluate(soaklib, f, op, a, b)
            bad = [i for i in range(n) if got[i] != want[i]]
            assert not bad, "product %s %s %s: a=%s b=%s got=%s big=%s" % (
                f, op, gen, fs._hex(a[bad[0]]), fs._hex(b[bad[0]]), fs._hex(got[bad[0]]), fs._hex(want[bad[0]]))


def test_generators_reach_the_edges(soaklib):
    """G1 draws saturated words, G2 enumerates pairs of boundary values (0, p - 1, R mod p, ...) smallest first, G3 puts
    T in [0, p R) with a full-width low half; operands depend only on (seed, index, slot)"""
    f = fs.FIELDS[0]
    a, _ = fs.operands(soaklib, f, "mul", "G1", 5, 0, 2000)
    words = [(x >> (32 * k)) & 0xFFFFFFFF for x in a for k in range(f.N)]
    assert words.count(0xFFFFFFFF) > len(words) // 20 and words.count(0) > len(words) // 20
    a, b = fs.operands(soaklib, f, "mul", "G2", 5, 0, 9)
    q, r1 = f.q, f.R % f.q
    assert list(zip(a, b)) == [(0, 0), (0, q - 1), (q - 1, 0), (q - 1, q - 1), (0, r1), (q - 1, r1), (r1, 0),
                               (r1, q - 1), (r1, r1)]
    a, _ = fs.operands(soaklib, f, "mul", "G2", 5, 0, 200 ** 2)
    assert {q // 2 - 3, q // 2 + 3, (r1 - 5) % q, r1 + 27, 1 << 20, 1 << 27, q - 12} <= set(a)
    t, _ = fs.operands(soaklib, f, "mont_reduce_wide", "G3", 5, 0, 2000)
    assert all(x < f.q * f.R for x in t)
    assert any((x & (f.R - 1)) >> (32 * f.N - 32) == 0xFFFFFFFF for x in t)
    a2, _ = fs.operands(soaklib, f, "mont_reduce_wide", "G3", 5, 1000, 1000)
    assert a2 == t[1000:]


@pytest.mark.parametrize("f", fs.DEVICE_FIELDS + fs.HOST_FIELDS, ids=str)
def test_host_soak(soaklib, f):
    """Every op x generator of one field at VOLUME samples: 0 mismatches"""
    fails = []
    for op in f.ops:
        if op == "reduce_mutant":
            continue
        for gen in fs.gens_for(op):
            seed = seed_of(f, op, gen)
            m, recs = fs.soak(soaklib, f, op, gen, seed, volume(f, op))
            if m:
                fails.append("%d mismatches\n%s" % (m, fs.triage(f, op, gen, seed, recs, "cpu")))
    assert not fails, "\n".join(fails)


@pytest.mark.parametrize("f", [f for f in fs.DEVICE_FIELDS if f.beta is None], ids=str)
def test_soak_catches_the_lost_carry(soaklib, f):
    """Power: round 2's first mont_reduce_wide (all of T preloaded) is caught under G1 products and under G3 on every
    field, and every record names the mutant, not the reference, and rebuilds from (seed, index)"""
    for gen in ("G1", "G3"):
        seed = seed_of(f, "reduce_mutant", gen)
        m, recs = fs.soak(soaklib, f, "reduce_mutant", gen, seed, VOLUME)
        assert m > 0, (f, gen)
        assert len(recs) == min(m, 16)
        for r in recs:
            assert r["want"] == fs.expected(f, "mont_reduce_wide", r["a"], r["b"]) != r["got"], (f, gen, r["index"])
            a, b = fs.operands(soaklib, f, "reduce_mutant", gen, seed, r["index"], 1)
            assert (a[0], b[0]) == (r["a"], r["b"])
