"""Helpers for the field-arithmetic soak (tests/cuda/field_soak.cu): field ids, op numbers, Python big-int semantics of
every op on raw (Montgomery) representations, packing, and the ctypes calls of the soak libraries.

Every value here is the raw integer a limb array holds, i.e. the Montgomery representation x R mod q; the big-int
semantics below are written on those representations, so that they compare directly with what the kernels store."""
import ctypes
import os

import numpy as np

from oracle.params import CURVES

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BUILD = os.path.join(ROOT, "tests", "_build")

OPS = {"add": 0, "sub": 1, "mul": 2, "inverse": 3, "neg": 4, "sqr": 5, "dbl": 6, "mul_small": 7, "from_mont": 8,
       "to_mont": 9, "wide_mul_raw": 10, "mont_reduce_wide": 11, "mul_beta": 12, "reduce_mutant": 13}
OP_NAMES = {v: k for k, v in OPS.items()}
GENS = {"G0": 0, "G1": 1, "G2": 2, "G3": 3}

FP_OPS = ["add", "sub", "mul", "inverse", "neg", "sqr", "dbl", "mul_small", "from_mont", "to_mont", "wide_mul_raw",
          "mont_reduce_wide"]
FP2_OPS = ["add", "sub", "mul", "inverse", "neg", "sqr", "dbl", "mul_beta"]
HFP_OPS = ["add", "sub", "mul", "inverse", "neg", "sqr", "dbl", "mul_small", "from_mont", "to_mont"]
HOSTFR_OPS = ["add", "sub", "mul", "inverse", "neg", "sqr"]
REDUCE_OPS = ("mont_reduce_wide", "reduce_mutant")


class Field:
    """One field id of the soak library: modulus q, N 32-bit limbs, beta (u^2 = -beta) for Fp2, supported ops"""

    def __init__(self, fid, name, q, n32, beta, ops):
        self.fid, self.name, self.q, self.N, self.beta, self.ops = fid, name, q, n32, beta, ops
        self.R = 1 << (32 * n32)
        self.Rinv = pow(self.R, -1, q)
        self.W = 2 * n32                       # padded words per element

    def __repr__(self):
        return self.name


def _fields():
    out = {}
    for c in CURVES.values():
        for which, (q, limbs) in enumerate(((c.p, c.fp_limbs), (c.r, c.fr_limbs))):
            fid = 2 * c.curve_id + which
            nm = "%s_%s" % (c.name, ("fp", "fr")[which])
            out[fid] = Field(fid, nm, q, 2 * limbs, None, FP_OPS + ["reduce_mutant"])
            out[200 + fid] = Field(200 + fid, "HFp_" + nm, q, 2 * limbs, None, HFP_OPS)
        out[300 + c.curve_id] = Field(300 + c.curve_id, "HostFrCtx_%s" % c.name, c.r, 2 * c.fr_limbs, None, HOSTFR_OPS)
        if c.fp2_nonresidue is not None:
            out[100 + 2 * c.curve_id] = Field(100 + 2 * c.curve_id, c.name + "_fp2", c.p, 2 * c.fp_limbs,
                                              -c.fp2_nonresidue, FP2_OPS)
            out[400 + 2 * c.curve_id] = Field(400 + 2 * c.curve_id, "HFp2_" + c.name, c.p, 2 * c.fp_limbs,
                                              -c.fp2_nonresidue, FP2_OPS)
    return out


FIELDS = _fields()
DEVICE_FIELDS = [FIELDS[k] for k in sorted(FIELDS) if k < 200]     # the 11 fields of the device templates
HOST_FIELDS = [FIELDS[k] for k in sorted(FIELDS) if k >= 200]      # host-only product code


def gens_for(op):
    return ["G0", "G1", "G2", "G3"] if op in REDUCE_OPS else ["G0", "G1", "G2"]


def expected(f, op, a, b):
    """Big-int result of `op` on raw representations (ints; (a0, a1) pairs for Fp2)"""
    q, R, Ri = f.q, f.R, f.Rinv
    if f.beta is not None:
        (a0, a1), (b0, b1) = a, b
        if op == "add": return ((a0 + b0) % q, (a1 + b1) % q)
        if op == "sub": return ((a0 - b0) % q, (a1 - b1) % q)
        if op == "neg": return ((-a0) % q, (-a1) % q)
        if op == "dbl": return (2 * a0 % q, 2 * a1 % q)
        if op == "mul_beta": return (f.beta * a0 % q, f.beta * a1 % q)
        if op == "sqr": b0, b1 = a0, a1
        if op in ("mul", "sqr"):
            return ((a0 * b0 - f.beta * a1 * b1) * Ri % q, (a0 * b1 + a1 * b0) * Ri % q)
        if op == "inverse":
            v0, v1 = a0 * Ri % q, a1 * Ri % q
            n = (v0 * v0 + f.beta * v1 * v1) % q
            if n == 0:
                return (0, 0)
            ni = pow(n, -1, q)
            return (v0 * ni * R % q, (-v1) * ni * R % q)
        raise ValueError(op)
    if op == "add": return (a + b) % q
    if op == "sub": return (a - b) % q
    if op == "mul": return a * b * Ri % q
    if op == "sqr": return a * a * Ri % q
    if op == "neg": return (-a) % q
    if op == "dbl": return 2 * a % q
    if op == "inverse": return 0 if a % q == 0 else pow(a * Ri % q, -1, q) * R % q
    if op == "mul_small": return (b & 0xFFFFFFFF) * a % q
    if op == "from_mont": return a * Ri % q
    if op == "to_mont": return a * R % q
    if op == "wide_mul_raw": return a * b
    if op in REDUCE_OPS: return a * Ri % q
    raise ValueError(op)


def pack(f, vals):
    """ints (or pairs) -> (n, 2N) uint32 words, each element padded to 2N words"""
    out = np.zeros((len(vals), f.W), dtype=np.uint32)
    nb = 4 * f.N
    for i, v in enumerate(vals):
        raw = (v[0].to_bytes(nb, "little") + v[1].to_bytes(nb, "little")) if f.beta is not None \
            else int(v).to_bytes(2 * nb, "little")
        out[i] = np.frombuffer(raw, dtype=np.uint32)
    return out


def unpack(f, words):
    words = np.ascontiguousarray(words, dtype=np.uint32).reshape(-1, f.W)
    out = []
    for w in words:
        raw = w.tobytes()
        if f.beta is not None:
            nb = 4 * f.N
            out.append((int.from_bytes(raw[:nb], "little"), int.from_bytes(raw[nb:], "little")))
        else:
            out.append(int.from_bytes(raw, "little"))
    return out


def _P(a):
    return a.ctypes.data_as(ctypes.c_void_p)


def bind(lib):
    u64, i32, vp = ctypes.c_uint64, ctypes.c_int, ctypes.c_void_p
    lib.fs_eval.argtypes = [i32, i32, vp, vp, vp, u64]
    lib.fs_soak.argtypes = [i32, i32, i32, u64, u64, vp]
    lib.fs_layout.argtypes = [ctypes.POINTER(i32)] * 3
    if hasattr(lib, "fs_ref_eval"):
        lib.fs_ref_eval.argtypes = [i32, i32, vp, vp, vp, u64]
        lib.fs_operands.argtypes = [i32, i32, i32, u64, u64, u64, vp, vp]
    mw, nr, sb = i32(), i32(), i32()
    lib.fs_layout(ctypes.byref(mw), ctypes.byref(nr), ctypes.byref(sb))
    lib.fs_maxw, lib.fs_nrec, lib.fs_stats_bytes = mw.value, nr.value, sb.value
    assert sb.value == 16 + nr.value * (8 + 16 * mw.value), "Stats layout"
    return lib


def load(name):
    return bind(ctypes.CDLL(os.path.join(BUILD, name)))


def evaluate(lib, f, op, a_vals, b_vals, entry="fs_eval"):
    A, B = pack(f, a_vals), pack(f, b_vals)
    O = np.zeros_like(A)
    rc = getattr(lib, entry)(f.fid, OPS[op], _P(A), _P(B), _P(O), len(a_vals))
    assert rc == 0, (entry, f, op, rc)
    return unpack(f, O)


def operands(lib, f, op, gen, seed, first, n):
    A = np.zeros((n, f.W), dtype=np.uint32)
    B = np.zeros_like(A)
    assert lib.fs_operands(f.fid, OPS[op], GENS[gen], seed, first, n, _P(A), _P(B)) == 0
    return unpack(f, A), unpack(f, B)


def soak(lib, f, op, gen, seed, count):
    """-> (mismatches, records); a record is dict(index, a, b, got, want) with ints / pairs"""
    st = np.zeros(lib.fs_stats_bytes, dtype=np.uint8)
    rc = lib.fs_soak(f.fid, OPS[op], GENS[gen], seed, count, _P(st))
    assert rc == 0, ("fs_soak", f, op, gen, rc)
    mism = int(st[:8].view(np.uint64)[0])
    claimed = int(st[8:16].view(np.uint64)[0])
    recs = []
    rb = 8 + 16 * lib.fs_maxw
    for k in range(min(claimed, lib.fs_nrec)):
        r = st[16 + k * rb: 16 + (k + 1) * rb]
        words = r[8:].view(np.uint32).reshape(4, lib.fs_maxw)[:, :f.W]
        a, b, got, want = (unpack(f, w)[0] for w in words)
        recs.append(dict(index=int(r[:8].view(np.uint64)[0]), a=a, b=b, got=got, want=want))
    return mism, recs


def _hex(v):
    return "(%s, %s)" % (hex(v[0]), hex(v[1])) if isinstance(v, tuple) else hex(v)


def triage(f, op, gen, seed, recs, where):
    """Check every recorded mismatch again with big ints; the message says which side is wrong and carries the operands"""
    lines = []
    for r in recs:
        exp = expected(f, op, r["a"], r["b"])
        side = ("the product template is wrong" if r["want"] == exp else
                "the reference is wrong" if r["got"] == exp else "both sides are wrong")
        lines.append("%s %s %s %s seed=%d index=%d: %s\n  a    = %s\n  b    = %s\n  got  = %s\n  want = %s\n  big  = %s"
                     % (where, f, op, gen, seed, r["index"], side, _hex(r["a"]), _hex(r["b"]), _hex(r["got"]),
                        _hex(r["want"]), _hex(exp)))
    return "\n".join(lines)
