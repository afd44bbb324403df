// Field-arithmetic soak (TEST ONLY): the product's field templates (field.cuh; host_field.h and host_fr.h on the host)
// against the independent reference of field_soak.cuh, on generated operands.
//
// Built twice from this one source:
//   - nvcc (tests/_build/libgb200_fieldsoak.so): the templates as the device compiles them - carry flag live across
//     separate asm statements, the out-of-line by-value Fp::mul_ni of BW6-761 Fp, the out-of-line Fp2 product / square;
//   - g++ into libgb200_hostemu.so: the same templates with the carry flag emulated (ptx.cuh), plus the host-only
//     Montgomery code that ships in the product (HFp<P>, Fp2<HFp<P>>, HostFrCtx).
//
// C entry points (extern "C" at the end):
//   fs_eval(fid, op, a, b, out, n)            product on n explicit operand pairs (device in the nvcc build)
//   fs_ref_eval(fid, op, a, b, out, n)        the reference on the same layout (host)
//   fs_operands(fid, op, gen, seed, first, n, a, b)   the generated operands of samples first .. first + n - 1 (host)
//   fs_soak(fid, op, gen, seed, count, stats)  product and reference on samples 0 .. count - 1; mismatches are counted
//                                             and the first 16 recorded, never trapped
// Operands and results are padded to 2N 32-bit words per element (N: limbs of the base field), so that a 2N-word T,
// a 2N-word product and an Fp2 element share one layout.
//
// Field ids: curve * 2 + (0: Fp, 1: Fr); 100 + 2 curve: Fp2.  Host build only: 200 + (curve * 2 + {0, 1}): HFp<P>;
// 300 + curve: HostFrCtx (Fr); 400 + 2 curve: Fp2<HFp<Fp params>>.
// Ops: 0 add, 1 sub, 2 mul, 3 inverse, 4 neg, 5 sqr, 6 dbl (tests/emu/hostemu.cpp), 7 mul_small(k = b word 0),
// 8 from_mont, 9 to_mont, 10 wide_mul_raw, 11 mont_reduce_wide (a: 2N-word T), 12 mul_beta (Fp2: both coefficients),
// 13 reduce_mutant (round 2's first mont_reduce_wide, kept here only to show that the soak catches it).
#include <algorithm>
#include <cstdint>
#include <cstring>

#include "field.cuh"
#include "field_soak.cuh"

#ifndef __CUDACC__
#include <thread>
#include <vector>

#include "host_field.h"
#include "host_fr.h"
#endif

using namespace gb200;

namespace fsoak {

enum Op {
  OP_ADD = 0, OP_SUB = 1, OP_MUL = 2, OP_INV = 3, OP_NEG = 4, OP_SQR = 5, OP_DBL = 6, OP_MUL_SMALL = 7,
  OP_FROM_MONT = 8, OP_TO_MONT = 9, OP_WIDE_MUL = 10, OP_REDUCE = 11, OP_MUL_BETA = 12, OP_REDUCE_MUTANT = 13
};

constexpr int MAXW = 48;  // 32-bit words of the widest operand: a 2N-word T of BW6-761 Fp
constexpr int NREC = 16;

struct Record {
  uint64_t index;
  uint32_t a[MAXW], b[MAXW], got[MAXW], want[MAXW];
};
struct Stats {
  unsigned long long mismatches;
  unsigned long long claimed;  // records claimed (only the first NREC are written)
  Record rec[NREC];
};

// The pre-fix mont_reduce_wide (round 2's first version): ALL of T preloaded into the accumulators, so the word a chain
// end adds its carry to may be a saturated word of T_hi, and that carry is lost.  Not product code.
template <class P>
HD void mont_reduce_wide_mutant(uint32_t* r, const uint32_t* T) {
  constexpr int N = P::N;
  uint32_t acc[2][2 * N + 3];
  uint32_t p[N];
#pragma unroll
  for (int k = 0; k < N; k++) p[k] = P::mod(k);
#pragma unroll
  for (int k = 0; k < 2 * N + 3; k++) { acc[0][k] = k < 2 * N ? T[k] : 0; acc[1][k] = 0; }
#pragma unroll
  for (int i = 0; i < N; i++) {
    uint32_t* X = acc[i & 1];
    uint32_t* Y = acc[(i & 1) ^ 1];
    const uint32_t m = (X[i] + Y[i]) * P::INV;
    if (i > 0) {
      X[i] = ptx::add_cc(X[i], Y[i]);
      mad_chain<N, 1, true>(Y, i, p, m);
    } else {
      mad_chain<N, 1, false>(Y, i, p, m);
    }
    mad_chain<N, 0, false>(X, i, p, m);
  }
  uint32_t s[N];
  s[0] = ptx::add_cc(acc[0][N], acc[1][N]);
#pragma unroll
  for (int k = 1; k < N; k++) s[k] = ptx::addc_cc(acc[0][N + k], acc[1][N + k]);
  uint32_t d[N];
  d[0] = ptx::sub_cc(s[0], p[0]);
#pragma unroll
  for (int k = 1; k < N; k++) d[k] = ptx::subc_cc(s[k], p[k]);
  const uint32_t borrow = ptx::subc(0, 0);
#pragma unroll
  for (int k = 0; k < N; k++) r[k] = borrow ? s[k] : d[k];
}

template <int W>
FS_HD void to32(uint32_t* o, const uint64_t* v) {
#pragma unroll
  for (int i = 0; i < W / 2; i++) { o[2 * i] = (uint32_t)v[i]; o[2 * i + 1] = (uint32_t)(v[i] >> 32); }
}
template <int W>
FS_HD void to64(uint64_t* o, const uint32_t* v) {
#pragma unroll
  for (int i = 0; i < W / 2; i++) o[i] = (uint64_t)v[2 * i] | ((uint64_t)v[2 * i + 1] << 32);
}

// ---------------------------------------------------------------------------------------------------------------------
// field kinds: operands, reference and product of one field id.  Buffers hold 2M 64-bit limbs (2N 32-bit words).
// ---------------------------------------------------------------------------------------------------------------------

// prime fields: operands and reference shared by the device Fp<P> and the host HFp<P> / HostFrCtx
template <class P_>
struct FpKindBase {
  using P = P_;
  static constexpr int N = P::N;
  static constexpr int M = N / 2;
  static FS_HD bool reduce_op(int op) { return op == OP_REDUCE || op == OP_REDUCE_MUTANT; }
  static FS_HD void operands(const Ref<M>& f, int op, int gen, uint64_t seed, uint64_t idx, uint64_t* a, uint64_t* b) {
#pragma unroll
    for (int i = 0; i < 2 * M; i++) { a[i] = 0; b[i] = 0; }
    if (reduce_op(op)) {
      if (gen == G_REDUCE) {
        gen_wide_T<M>(f, seed, idx, a);
      } else {  // the product of two generated values: T < p^2
        uint64_t x[M], y[M];
        gen_value<M>(f, gen, seed, idx, 0, x);
        gen_value<M>(f, gen, seed, idx, 1, y);
        wide<M>(a, x, y);
      }
      return;
    }
    gen_value<M>(f, gen, seed, idx, 0, a);
    if (op == OP_MUL_SMALL) b[0] = gen_small(seed, idx);
    else gen_value<M>(f, gen, seed, idx, 1, b);
  }
  static FS_HD void reference(const Ref<M>& f, int op, const uint64_t* a, const uint64_t* b, uint64_t* r) {
#pragma unroll
    for (int i = 0; i < 2 * M; i++) r[i] = 0;
    switch (op) {
      case OP_ADD: add<M>(f, r, a, b); break;
      case OP_SUB: sub<M>(f, r, a, b); break;
      case OP_MUL: mul<M>(f, r, a, b); break;
      case OP_INV: inverse<M>(f, r, a); break;
      case OP_NEG: neg<M>(f, r, a); break;
      case OP_SQR: mul<M>(f, r, a, a); break;
      case OP_DBL: add<M>(f, r, a, a); break;
      case OP_MUL_SMALL: mul_small<M>(f, r, a, (uint32_t)b[0]); break;
      case OP_FROM_MONT: { uint64_t T[2 * M]; for (int i = 0; i < 2 * M; i++) T[i] = i < M ? a[i] : 0; redc<M>(f, r, T); break; }
      case OP_TO_MONT: { uint64_t T[2 * M]; wide<M>(T, a, f.r2); redc<M>(f, r, T); break; }
      case OP_WIDE_MUL: wide<M>(r, a, b); break;
      case OP_REDUCE:
      case OP_REDUCE_MUTANT: redc<M>(f, r, a); break;
    }
  }
  // inverse: the product's result x is right iff x < p and x a = 1 (x = 0 for a = 0); only otherwise is a^(p-2) worth
  // computing for the record
  static FS_HD bool inverse_ok(const Ref<M>& f, const uint64_t* a, const uint64_t* x) {
    if (geq<M>(x, f.p)) return false;
    if (is_zero<M>(a)) return is_zero<M>(x);
    uint64_t t[M];
    mul<M>(f, t, x, a);
    for (int i = 0; i < M; i++) if (t[i] != f.r1[i]) return false;
    return true;
  }
};

template <class P_>
struct KFp : FpKindBase<P_> {
  using B = FpKindBase<P_>;
  using P = P_;
  using B::N;
  static FS_HD bool valid(int op, int gen) {
    if (gen < 0 || gen > G_REDUCE) return false;
    if (gen == G_REDUCE) return B::reduce_op(op);
    return (op >= OP_ADD && op <= OP_REDUCE) || op == OP_REDUCE_MUTANT;
  }
  static FS_HD void product(int op, const uint32_t* a, const uint32_t* b, uint32_t* o) {
    using F = Fp<P>;
    F x, y, r;
#pragma unroll
    for (int i = 0; i < N; i++) { x.l[i] = a[i]; y.l[i] = b[i]; }
#pragma unroll
    for (int i = 0; i < 2 * N; i++) o[i] = 0;
    switch (op) {
      case OP_ADD: r = x + y; break;
      case OP_SUB: r = x - y; break;
      case OP_MUL: r = x * y; break;
      case OP_INV: r = x.inverse(); break;
      case OP_NEG: r = x.neg(); break;
      case OP_SQR: r = x.sqr(); break;
      case OP_DBL: r = x.dbl(); break;
      case OP_MUL_SMALL: r = x.mul_small(b[0]); break;
      case OP_FROM_MONT: r = x.from_mont(); break;
      case OP_TO_MONT: r = x.to_mont(); break;
      case OP_WIDE_MUL: wide_mul_raw<N>(o, a, b); return;
      case OP_REDUCE: mont_reduce_wide<P>(o, a); return;
      case OP_REDUCE_MUTANT: mont_reduce_wide_mutant<P>(o, a); return;
      default: return;
    }
#pragma unroll
    for (int i = 0; i < N; i++) o[i] = r.l[i];
  }
};

// Fp2 = Fp[u]/(u^2 + BETA), element (a0, a1) in 2N words
template <class P_, unsigned BETA>
struct Fp2KindBase {
  using P = P_;
  static constexpr int N = P::N;
  static constexpr int M = N / 2;
  static FS_HD bool valid(int op, int gen) {
    return gen >= G_UNIFORM && gen <= G_BOUNDARY && ((op >= OP_ADD && op <= OP_DBL) || op == OP_MUL_BETA);
  }
  static FS_HD void operands(const Ref<M>& f, int op, int gen, uint64_t seed, uint64_t idx, uint64_t* a, uint64_t* b) {
    (void)op;
    gen_value<M>(f, gen, seed, idx, 0, a);
    gen_value<M>(f, gen, seed, idx, 1, a + M);
    gen_value<M>(f, gen, seed, idx, 2, b);
    gen_value<M>(f, gen, seed, idx, 3, b + M);
  }
  static FS_HD void reference(const Ref<M>& f, int op, const uint64_t* a, const uint64_t* b, uint64_t* r) {
    const uint64_t *a0 = a, *a1 = a + M, *b0 = b, *b1 = b + M;
    uint64_t *r0 = r, *r1 = r + M;
    switch (op) {
      case OP_ADD: add<M>(f, r0, a0, b0); add<M>(f, r1, a1, b1); break;
      case OP_SUB: sub<M>(f, r0, a0, b0); sub<M>(f, r1, a1, b1); break;
      case OP_MUL: fp2_mul<M>(f, BETA, r0, r1, a0, a1, b0, b1); break;
      case OP_SQR: fp2_mul<M>(f, BETA, r0, r1, a0, a1, a0, a1); break;
      case OP_NEG: neg<M>(f, r0, a0); neg<M>(f, r1, a1); break;
      case OP_DBL: add<M>(f, r0, a0, a0); add<M>(f, r1, a1, a1); break;
      case OP_MUL_BETA: mul_small<M>(f, r0, a0, BETA); mul_small<M>(f, r1, a1, BETA); break;
      case OP_INV: {  // 1 / (a0 + a1 u) = (a0 - a1 u) / (a0^2 + BETA a1^2)
        uint64_t n[M], t[M], ni[M];
        mul<M>(f, n, a0, a0);
        mul<M>(f, t, a1, a1);
        mul_small<M>(f, t, t, BETA);
        add<M>(f, n, n, t);
        inverse<M>(f, ni, n);
        mul<M>(f, r0, a0, ni);
        mul<M>(f, t, a1, ni);
        neg<M>(f, r1, t);
        break;
      }
    }
  }
  static FS_HD bool inverse_ok(const Ref<M>& f, const uint64_t* a, const uint64_t* x) {
    if (geq<M>(x, f.p) || geq<M>(x + M, f.p)) return false;
    if (is_zero<M>(a) && is_zero<M>(a + M)) return is_zero<M>(x) && is_zero<M>(x + M);
    uint64_t t0[M], t1[M];
    fp2_mul<M>(f, BETA, t0, t1, x, x + M, a, a + M);
    for (int i = 0; i < M; i++) if (t0[i] != f.r1[i] || t1[i] != 0) return false;
    return true;
  }
};

template <class P_, unsigned BETA>
struct KFp2 : Fp2KindBase<P_, BETA> {
  using P = P_;
  static constexpr int N = P::N;
  static FS_HD void product(int op, const uint32_t* a, const uint32_t* b, uint32_t* o) {
    using F2 = Fp2<Fp<P>, BETA>;
    F2 x, y, r;
#pragma unroll
    for (int i = 0; i < N; i++) { x.a0.l[i] = a[i]; x.a1.l[i] = a[N + i]; y.a0.l[i] = b[i]; y.a1.l[i] = b[N + i]; }
    switch (op) {
      case OP_ADD: r = x + y; break;
      case OP_SUB: r = x - y; break;
      case OP_MUL: r = x * y; break;
      case OP_INV: r = x.inverse(); break;
      case OP_NEG: r = x.neg(); break;
      case OP_SQR: r = x.sqr(); break;
      case OP_DBL: r = x.dbl(); break;
      case OP_MUL_BETA: r.a0 = F2::mul_beta(x.a0); r.a1 = F2::mul_beta(x.a1); break;
      default: r = F2::zero();
    }
#pragma unroll
    for (int i = 0; i < N; i++) { o[i] = r.a0.l[i]; o[N + i] = r.a1.l[i]; }
  }
};

#ifndef __CUDACC__
// host-only Montgomery code of the product: HFp<P> (Groth16 proof assembly), Fp2<HFp<P>> (its G2), HostFrCtx (PLONK)
template <class P_>
struct KHFp : FpKindBase<P_> {
  using P = P_;
  static constexpr int N = P::N;
  static bool valid(int op, int gen) { return gen >= G_UNIFORM && gen <= G_BOUNDARY && op >= OP_ADD && op <= OP_TO_MONT; }
  static void product(int op, const uint32_t* a, const uint32_t* b, uint32_t* o) {
    using F = HFp<P>;
    F x, y, r;
    memcpy(x.l, a, sizeof(x.l));
    memcpy(y.l, b, sizeof(y.l));
    memset(o, 0, 8 * N);
    switch (op) {
      case OP_ADD: r = x + y; break;
      case OP_SUB: r = x - y; break;
      case OP_MUL: r = x * y; break;
      case OP_INV: r = x.inverse(); break;
      case OP_NEG: r = x.neg(); break;
      case OP_SQR: r = x.sqr(); break;
      case OP_DBL: r = x.dbl(); break;
      case OP_MUL_SMALL: r = x.mul_small(b[0]); break;
      case OP_FROM_MONT: r = x.from_mont(); break;
      case OP_TO_MONT: r = x.to_mont(); break;
      default: return;
    }
    memcpy(o, r.l, sizeof(r.l));
  }
};

template <class P_>
struct KHostFr : FpKindBase<P_> {
  using P = P_;
  static constexpr int N = P::N;
  static bool valid(int op, int gen) { return gen >= G_UNIFORM && gen <= G_BOUNDARY && op >= OP_ADD && op <= OP_SQR; }
  static void product(int op, const uint32_t* a, const uint32_t* b, uint32_t* o) {
    static const HostFrCtx c = HostFrCtx::make<P>();
    const HostFr x = c.load(a), y = c.load(b);
    HostFr r = c.zero();
    memset(o, 0, 8 * N);
    switch (op) {
      case OP_ADD: r = c.add(x, y); break;
      case OP_SUB: r = c.sub(x, y); break;
      case OP_MUL: r = c.mul(x, y); break;
      case OP_INV: r = c.inv(x); break;
      case OP_NEG: r = c.neg(x); break;
      case OP_SQR: r = c.sqr(x); break;
      default: return;
    }
    c.store(o, r);
  }
};

template <class P_, unsigned BETA>
struct KHFp2 : Fp2KindBase<P_, BETA> {
  using P = P_;
  static constexpr int N = P::N;
  static void product(int op, const uint32_t* a, const uint32_t* b, uint32_t* o) {
    using F2 = Fp2<HFp<P>, BETA>;
    F2 x, y, r;
    memcpy(x.a0.l, a, 4 * N);
    memcpy(x.a1.l, a + N, 4 * N);
    memcpy(y.a0.l, b, 4 * N);
    memcpy(y.a1.l, b + N, 4 * N);
    switch (op) {
      case OP_ADD: r = x + y; break;
      case OP_SUB: r = x - y; break;
      case OP_MUL: r = x * y; break;
      case OP_INV: r = x.inverse(); break;
      case OP_NEG: r = x.neg(); break;
      case OP_SQR: r = x.sqr(); break;
      case OP_DBL: r = x.dbl(); break;
      case OP_MUL_BETA: r.a0 = F2::mul_beta(x.a0); r.a1 = F2::mul_beta(x.a1); break;
      default: r = F2::zero();
    }
    memcpy(o, r.a0.l, 4 * N);
    memcpy(o + N, r.a1.l, 4 * N);
  }
};
#endif

// ---------------------------------------------------------------------------------------------------------------------
// one sample: operands, product, reference, compare; a mismatch is counted and (first NREC) recorded
// ---------------------------------------------------------------------------------------------------------------------
template <class K>
FS_HD void sample(const Ref<K::M>& f, int op, int gen, uint64_t seed, uint64_t idx, Stats* st) {
  constexpr int M = K::M;
  constexpr int W = 4 * M;  // 32-bit words per padded element
  uint64_t a[2 * M], b[2 * M], want[2 * M], got64[2 * M];
  uint32_t a32[W], b32[W], got[W];
  K::operands(f, op, gen, seed, idx, a, b);
  to32<W>(a32, a);
  to32<W>(b32, b);
  K::product(op, a32, b32, got);
  to64<W>(got64, got);
  if (op == OP_INV && K::inverse_ok(f, a, got64)) return;
  K::reference(f, op, a, b, want);
  bool same = true;
#pragma unroll
  for (int i = 0; i < 2 * M; i++) same &= got64[i] == want[i];
  if (same) return;
  unsigned long long slot;
#ifdef __CUDA_ARCH__
  atomicAdd(&st->mismatches, 1ull);
  slot = atomicAdd(&st->claimed, 1ull);
#else
  st->mismatches++;
  slot = st->claimed++;
#endif
  if (slot >= NREC) return;
  Record& r = st->rec[slot];
  r.index = idx;
  for (int i = 0; i < MAXW; i++) {
    r.a[i] = i < W ? a32[i] : 0;
    r.b[i] = i < W ? b32[i] : 0;
    r.got[i] = i < W ? got[i] : 0;
    r.want[i] = 0;
  }
  to32<W>(r.want, want);
}

#ifdef __CUDACC__
template <class K>
__global__ void k_soak(Ref<K::M> f, int op, int gen, uint64_t seed, uint64_t base, uint64_t count, Stats* st) {
  const uint64_t stride = (uint64_t)gridDim.x * blockDim.x;
  for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < count; i += stride)
    sample<K>(f, op, gen, seed, base + i, st);
}

template <class K>
__global__ void k_eval(int op, const uint32_t* a, const uint32_t* b, uint32_t* out, uint64_t n) {
  constexpr int W = 2 * K::N;
  const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  uint32_t x[W], y[W], r[W];
  for (int k = 0; k < W; k++) { x[k] = a[i * W + k]; y[k] = b[i * W + k]; }
  K::product(op, x, y, r);
  for (int k = 0; k < W; k++) out[i * W + k] = r[k];
}
#endif

// field id -> kind; fn is called with a value of the kind type, returns fn's result or -1 for an unknown id
template <class Fn>
int dispatch(int fid, Fn&& fn) {
  switch (fid) {
    case 0: return fn(KFp<bn254_fp_params>());
    case 1: return fn(KFp<bn254_fr_params>());
    case 2: return fn(KFp<bls12_381_fp_params>());
    case 3: return fn(KFp<bls12_381_fr_params>());
    case 4: return fn(KFp<bls12_377_fp_params>());
    case 5: return fn(KFp<bls12_377_fr_params>());
    case 6: return fn(KFp<bw6_761_fp_params>());
    case 7: return fn(KFp<bw6_761_fr_params>());
    case 100: return fn(KFp2<bn254_fp_params, 1>());
    case 102: return fn(KFp2<bls12_381_fp_params, 1>());
    case 104: return fn(KFp2<bls12_377_fp_params, 5>());
#ifndef __CUDACC__
    case 200: return fn(KHFp<bn254_fp_params>());
    case 201: return fn(KHFp<bn254_fr_params>());
    case 202: return fn(KHFp<bls12_381_fp_params>());
    case 203: return fn(KHFp<bls12_381_fr_params>());
    case 204: return fn(KHFp<bls12_377_fp_params>());
    case 205: return fn(KHFp<bls12_377_fr_params>());
    case 206: return fn(KHFp<bw6_761_fp_params>());
    case 207: return fn(KHFp<bw6_761_fr_params>());
    case 300: return fn(KHostFr<bn254_fr_params>());
    case 301: return fn(KHostFr<bls12_381_fr_params>());
    case 302: return fn(KHostFr<bls12_377_fr_params>());
    case 303: return fn(KHostFr<bw6_761_fr_params>());
    case 400: return fn(KHFp2<bn254_fp_params, 1>());
    case 402: return fn(KHFp2<bls12_381_fp_params, 1>());
    case 404: return fn(KHFp2<bls12_377_fp_params, 5>());
#endif
  }
  return -1;
}

#ifndef __CUDACC__
// host soak: the index range cut into one contiguous piece per thread, per-thread stats merged
template <class K>
int soak_host(int op, int gen, uint64_t seed, uint64_t count, Stats* out) {
  const Ref<K::M> f = make_ref<typename K::P>();
  const unsigned nt = std::max(1u, std::min(16u, std::thread::hardware_concurrency()));
  std::vector<Stats> st(nt);
  memset(st.data(), 0, sizeof(Stats) * nt);
  std::vector<std::thread> th;
  for (unsigned t = 0; t < nt; t++)
    th.emplace_back([&, t] {
      const uint64_t lo = count * t / nt, hi = count * (t + 1) / nt;
      for (uint64_t i = lo; i < hi; i++) sample<K>(f, op, gen, seed, i, &st[t]);
    });
  for (auto& x : th) x.join();
  memset(out, 0, sizeof(Stats));
  for (unsigned t = 0; t < nt; t++) {
    out->mismatches += st[t].mismatches;
    for (unsigned long long k = 0; k < std::min<unsigned long long>(st[t].claimed, NREC); k++)
      if (out->claimed < NREC) out->rec[out->claimed++] = st[t].rec[k];
      else out->claimed++;
    if (st[t].claimed > NREC) out->claimed += st[t].claimed - NREC;
  }
  return 0;
}
#else
template <class K>
int soak_device(int op, int gen, uint64_t seed, uint64_t count, Stats* out) {
  const Ref<K::M> f = make_ref<typename K::P>();
  Stats* d = nullptr;
  if (cudaMalloc(&d, sizeof(Stats)) != cudaSuccess) return -2;
  cudaMemset(d, 0, sizeof(Stats));
  int dev = 0, sms = 0, per_sm = 0;
  cudaGetDevice(&dev);
  cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
  const int threads = 256;
  cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, k_soak<K>, threads, 0);
  const unsigned blocks = (unsigned)std::max(1, sms * std::max(1, per_sm));
  const uint64_t chunk = 1ull << 26;  // samples per launch: bounded kernel durations
  int rc = 0;
  for (uint64_t base = 0; base < count && rc == 0; base += chunk) {
    const uint64_t n = count - base < chunk ? count - base : chunk;
    k_soak<K><<<blocks, threads>>>(f, op, gen, seed, base, n, d);
    if (cudaGetLastError() != cudaSuccess) rc = -2;
  }
  if (cudaDeviceSynchronize() != cudaSuccess) rc = -2;
  if (cudaMemcpy(out, d, sizeof(Stats), cudaMemcpyDeviceToHost) != cudaSuccess) rc = -2;
  cudaFree(d);
  return rc;
}
#endif

}  // namespace fsoak

using namespace fsoak;

extern "C" {

// product on n explicit operand pairs, 2N words per element
int fs_eval(int fid, int op, const void* a, const void* b, void* out, uint64_t n) {
  return dispatch(fid, [&](auto k) -> int {
    using K = decltype(k);
    if (!K::valid(op, G_UNIFORM) && !K::valid(op, G_REDUCE)) return -1;
    constexpr int W = 2 * K::N;
#ifdef __CUDACC__
    if (n == 0) return 0;
    const size_t bytes = (size_t)n * W * 4;
    uint32_t *da = nullptr, *db = nullptr, *dout = nullptr;
    int rc = 0;
    if (cudaMalloc(&da, bytes) != cudaSuccess || cudaMalloc(&db, bytes) != cudaSuccess ||
        cudaMalloc(&dout, bytes) != cudaSuccess) rc = -2;
    if (rc == 0) {
      cudaMemcpy(da, a, bytes, cudaMemcpyHostToDevice);
      cudaMemcpy(db, b, bytes, cudaMemcpyHostToDevice);
      k_eval<K><<<(unsigned)((n + 127) / 128), 128>>>(op, da, db, dout, n);
      if (cudaGetLastError() != cudaSuccess || cudaDeviceSynchronize() != cudaSuccess) rc = -2;
      if (rc == 0 && cudaMemcpy(out, dout, bytes, cudaMemcpyDeviceToHost) != cudaSuccess) rc = -2;
    }
    cudaFree(da);
    cudaFree(db);
    cudaFree(dout);
    return rc;
#else
    for (uint64_t i = 0; i < n; i++)
      K::product(op, (const uint32_t*)a + i * W, (const uint32_t*)b + i * W, (uint32_t*)out + i * W);
    return 0;
#endif
  });
}

// the reference on the same layout (host)
int fs_ref_eval(int fid, int op, const void* a, const void* b, void* out, uint64_t n) {
  return dispatch(fid, [&](auto k) -> int {
    using K = decltype(k);
    if (!K::valid(op, G_UNIFORM) && !K::valid(op, G_REDUCE)) return -1;
    constexpr int M = K::M;
    const Ref<M> f = make_ref<typename K::P>();
    for (uint64_t i = 0; i < n; i++)
      K::reference(f, op, (const uint64_t*)a + i * 2 * M, (const uint64_t*)b + i * 2 * M, (uint64_t*)out + i * 2 * M);
    return 0;
  });
}

// the operands of samples first .. first + n - 1 (what fs_soak feeds the product), 2N words per element
int fs_operands(int fid, int op, int gen, uint64_t seed, uint64_t first, uint64_t n, void* a, void* b) {
  return dispatch(fid, [&](auto k) -> int {
    using K = decltype(k);
    if (!K::valid(op, gen)) return -1;
    constexpr int M = K::M;
    const Ref<M> f = make_ref<typename K::P>();
    for (uint64_t i = 0; i < n; i++)
      K::operands(f, op, gen, seed, first + i, (uint64_t*)a + i * 2 * M, (uint64_t*)b + i * 2 * M);
    return 0;
  });
}

// product against the reference on samples 0 .. count - 1; stats: struct Stats (mismatch count, first NREC records)
int fs_soak(int fid, int op, int gen, uint64_t seed, uint64_t count, void* stats) {
  return dispatch(fid, [&](auto k) -> int {
    using K = decltype(k);
    if (!K::valid(op, gen)) return -1;
#ifdef __CUDACC__
    return soak_device<K>(op, gen, seed, count, (Stats*)stats);
#else
    return soak_host<K>(op, gen, seed, count, (Stats*)stats);
#endif
  });
}

// layout constants for the caller: words per record operand, records kept, sizeof(Stats)
int fs_layout(int* maxw, int* nrec, int* stats_bytes) {
  *maxw = MAXW;
  *nrec = NREC;
  *stats_bytes = (int)sizeof(Stats);
  return 0;
}

}  // extern "C"
