// Field-arithmetic soak: an independent reference and the operand generators (TEST ONLY).
//
// Shared by the device build (tests/_build/libgb200_fieldsoak.so, nvcc) and the host build (compiled into
// libgb200_hostemu.so), so both soaks run the same generators against the same reference.  Nothing here comes from
// ptx.cuh or field.cuh: the reference uses 64-bit limbs on unsigned __int128 with compare-based carries, and the only
// thing it takes from the product is the modulus (params_gen.cuh).  -p^-1 mod 2^64, R mod p and R^2 mod p are derived
// here from the modulus alone.
//
// Values are raw limb arrays (the Montgomery representations the product stores); R = 2^(64 M) = 2^(32 N).
#pragma once
#include <cstdint>

#include "params_gen.cuh"

#ifdef __CUDACC__
#define FS_HD __host__ __device__ __forceinline__
#else
#define FS_HD inline
#endif

namespace fsoak {

typedef unsigned __int128 u128;

// ---------------------------------------------------------------------------------------------------------------------
// reference arithmetic, M 64-bit limbs
// ---------------------------------------------------------------------------------------------------------------------
template <int M>
struct Ref {
  uint64_t p[M];
  uint64_t half[M];   // floor(p / 2)
  uint64_t r1[M];     // R mod p
  uint64_t r2[M];     // R^2 mod p
  uint64_t ninv;      // -p^-1 mod 2^64
  int bits;           // bit length of p
};

template <int M>
FS_HD bool geq(const uint64_t* a, const uint64_t* b) {
  for (int i = M - 1; i >= 0; i--) {
    if (a[i] != b[i]) return a[i] > b[i];
  }
  return true;
}

// r = a + b, returns the carry out (compare-based)
template <int M>
FS_HD uint64_t add_raw(uint64_t* r, const uint64_t* a, const uint64_t* b) {
  uint64_t c = 0;
#pragma unroll
  for (int i = 0; i < M; i++) {
    const uint64_t s = a[i] + c;
    const uint64_t c1 = s < c;
    const uint64_t t = s + b[i];
    r[i] = t;
    c = c1 | (uint64_t)(t < s);
  }
  return c;
}

// r = a - b, returns the borrow out (compare-based)
template <int M>
FS_HD uint64_t sub_raw(uint64_t* r, const uint64_t* a, const uint64_t* b) {
  uint64_t br = 0;
#pragma unroll
  for (int i = 0; i < M; i++) {
    const uint64_t ai = a[i], bi = b[i];
    const uint64_t d = ai - bi;
    const uint64_t b1 = ai < bi;
    r[i] = d - br;
    br = b1 | (uint64_t)(d < br);
  }
  return br;
}

template <int M>
FS_HD bool is_zero(const uint64_t* a) {
  uint64_t t = 0;
#pragma unroll
  for (int i = 0; i < M; i++) t |= a[i];
  return t == 0;
}

template <int M>
FS_HD void add(const Ref<M>& f, uint64_t* r, const uint64_t* a, const uint64_t* b) {
  const uint64_t c = add_raw<M>(r, a, b);
  if (c || geq<M>(r, f.p)) sub_raw<M>(r, r, f.p);
}

template <int M>
FS_HD void sub(const Ref<M>& f, uint64_t* r, const uint64_t* a, const uint64_t* b) {
  if (sub_raw<M>(r, a, b)) add_raw<M>(r, r, f.p);
}

template <int M>
FS_HD void neg(const Ref<M>& f, uint64_t* r, const uint64_t* a) {
  if (is_zero<M>(a)) {
    for (int i = 0; i < M; i++) r[i] = 0;
  } else {
    sub_raw<M>(r, f.p, a);
  }
}

// r = a * b * R^-1 mod p, coarsely integrated operand scanning (CIOS), a, b < p
template <int M>
FS_HD void mul(const Ref<M>& f, uint64_t* r, const uint64_t* a, const uint64_t* b) {
  uint64_t t[M + 2];
#pragma unroll
  for (int i = 0; i < M + 2; i++) t[i] = 0;
#pragma unroll
  for (int i = 0; i < M; i++) {
    u128 c = 0;
#pragma unroll
    for (int j = 0; j < M; j++) {
      c += (u128)a[j] * b[i] + t[j];
      t[j] = (uint64_t)c;
      c >>= 64;
    }
    c += t[M];
    t[M] = (uint64_t)c;
    t[M + 1] = (uint64_t)(c >> 64);
    const uint64_t m = t[0] * f.ninv;
    c = ((u128)m * f.p[0] + t[0]) >> 64;
#pragma unroll
    for (int j = 1; j < M; j++) {
      c += (u128)m * f.p[j] + t[j];
      t[j - 1] = (uint64_t)c;
      c >>= 64;
    }
    c += t[M];
    t[M - 1] = (uint64_t)c;
    t[M] = t[M + 1] + (uint64_t)(c >> 64);
  }
  if (t[M] || geq<M>(t, f.p)) sub_raw<M>(t, t, f.p);
#pragma unroll
  for (int i = 0; i < M; i++) r[i] = t[i];
}

// t[0 .. 2M) = a * b exactly (schoolbook)
template <int M>
FS_HD void wide(uint64_t* t, const uint64_t* a, const uint64_t* b) {
#pragma unroll
  for (int i = 0; i < 2 * M; i++) t[i] = 0;
#pragma unroll
  for (int i = 0; i < M; i++) {
    u128 c = 0;
#pragma unroll
    for (int j = 0; j < M; j++) {
      c += (u128)a[j] * b[i] + t[i + j];
      t[i + j] = (uint64_t)c;
      c >>= 64;
    }
    t[i + M] = (uint64_t)c;
  }
}

// r = T * R^-1 mod p for T < p R: word-by-word REDC, every carry propagated to the top word
template <int M>
FS_HD void redc(const Ref<M>& f, uint64_t* r, const uint64_t* T) {
  uint64_t t[2 * M + 1];
#pragma unroll
  for (int i = 0; i < 2 * M; i++) t[i] = T[i];
  t[2 * M] = 0;
#pragma unroll
  for (int i = 0; i < M; i++) {
    const uint64_t m = t[i] * f.ninv;
    u128 c = 0;
#pragma unroll
    for (int j = 0; j < M; j++) {
      c += (u128)m * f.p[j] + t[i + j];
      t[i + j] = (uint64_t)c;
      c >>= 64;
    }
    for (int k = i + M; k <= 2 * M; k++) {
      c += t[k];
      t[k] = (uint64_t)c;
      c >>= 64;
    }
  }
  uint64_t s[M];
#pragma unroll
  for (int i = 0; i < M; i++) s[i] = t[M + i];
  if (t[2 * M] || geq<M>(s, f.p)) sub_raw<M>(s, s, f.p);
#pragma unroll
  for (int i = 0; i < M; i++) r[i] = s[i];
}

// r = k * a mod p: k to Montgomery form through R^2, then one product
template <int M>
FS_HD void mul_small(const Ref<M>& f, uint64_t* r, const uint64_t* a, uint32_t k) {
  uint64_t km[M];
#pragma unroll
  for (int i = 0; i < M; i++) km[i] = 0;
  km[0] = k;
  mul<M>(f, km, km, f.r2);
  mul<M>(f, r, a, km);
}

// a^e for an exponent of M limbs, left to right
template <int M>
FS_HD void pow(const Ref<M>& f, uint64_t* r, const uint64_t* a, const uint64_t* e) {
  uint64_t acc[M];
  for (int i = 0; i < M; i++) acc[i] = f.r1[i];
  for (int w = M - 1; w >= 0; w--)
    for (int b = 63; b >= 0; b--) {
      mul<M>(f, acc, acc, acc);
      if ((e[w] >> b) & 1) mul<M>(f, acc, acc, a);
    }
  for (int i = 0; i < M; i++) r[i] = acc[i];
}

// inverse with 0 -> 0 (a^(p-2))
template <int M>
FS_HD void inverse(const Ref<M>& f, uint64_t* r, const uint64_t* a) {
  uint64_t e[M], two[M];
  for (int i = 0; i < M; i++) two[i] = 0;
  two[0] = 2;
  sub_raw<M>(e, f.p, two);
  pow<M>(f, r, a, e);
}

// Fp2 = Fp[u]/(u^2 + beta): schoolbook, four products
//   c0 = a0 b0 - beta a1 b1,  c1 = a0 b1 + a1 b0
template <int M>
FS_HD void fp2_mul(const Ref<M>& f, unsigned beta, uint64_t* r0, uint64_t* r1, const uint64_t* a0, const uint64_t* a1,
                   const uint64_t* b0, const uint64_t* b1) {
  uint64_t v00[M], v11[M], v01[M], v10[M];
  mul<M>(f, v00, a0, b0);
  mul<M>(f, v11, a1, b1);
  mul<M>(f, v01, a0, b1);
  mul<M>(f, v10, a1, b0);
  if (beta != 1) mul_small<M>(f, v11, v11, beta);
  sub<M>(f, r0, v00, v11);
  add<M>(f, r1, v01, v10);
}

// ---------------------------------------------------------------------------------------------------------------------
// reference constants from the modulus alone (host)
// ---------------------------------------------------------------------------------------------------------------------
template <class P>
Ref<P::N / 2> make_ref() {
  constexpr int M = P::N / 2;
  Ref<M> f;
  for (int i = 0; i < M; i++) f.p[i] = (uint64_t)P::mod(2 * i) | ((uint64_t)P::mod(2 * i + 1) << 32);
  uint64_t x = 1;  // p^-1 mod 2^64 by Newton iteration: each step doubles the correct low bits (1 -> 64 in 6)
  for (int i = 0; i < 6; i++) x *= 2 - f.p[0] * x;
  f.ninv = 0 - x;
  for (int i = 0; i < M; i++) f.half[i] = (f.p[i] >> 1) | (i + 1 < M ? f.p[i + 1] << 63 : 0);
  f.bits = 0;
  for (int i = M - 1; i >= 0 && !f.bits; i--)
    if (f.p[i]) f.bits = 64 * i + 64 - __builtin_clzll(f.p[i]);
  // R mod p and R^2 mod p by doubling 1: 64 M and 128 M doublings
  uint64_t v[M];
  for (int i = 0; i < M; i++) v[i] = 0;
  v[0] = 1;
  for (int k = 0; k < 128 * M; k++) {
    add<M>(f, v, v, v);
    if (k + 1 == 64 * M)
      for (int i = 0; i < M; i++) f.r1[i] = v[i];
  }
  for (int i = 0; i < M; i++) f.r2[i] = v[i];
  return f;
}

// ---------------------------------------------------------------------------------------------------------------------
// operand generators: every operand is a function of (seed, sample index, slot) only
// ---------------------------------------------------------------------------------------------------------------------
enum Gen { G_UNIFORM = 0, G_PALETTE = 1, G_BOUNDARY = 2, G_REDUCE = 3 };

FS_HD uint64_t mix64(uint64_t z) {
  z += 0x9e3779b97f4a7c15ull;
  z = (z ^ (z >> 30)) * 0xbf58476d1ce4e5b9ull;
  z = (z ^ (z >> 27)) * 0x94d049bb133111ebull;
  return z ^ (z >> 31);
}
FS_HD uint64_t hash(uint64_t seed, uint64_t idx, uint32_t slot, uint32_t ctr) {
  return mix64(mix64(mix64(seed) ^ idx) ^ (((uint64_t)slot << 32) | ctr));
}

// 32-bit words that sit at carry-chain edges: with probability 3/4 a word is one of these (or the word of p / p - 1 at
// the same position), otherwise uniform
FS_HD uint32_t palette_word(uint64_t h, uint32_t pw, uint32_t pm1w, bool with_p) {
  const uint32_t u = (uint32_t)h;
  if (((h >> 32) & 3) == 0) return u;
  const unsigned sel = (unsigned)(h >> 34) & 7;
  switch (sel) {
    case 0: return 0u;
    case 1: return 1u;
    case 2: return 0xffffffffu;
    case 3: return 0xfffffffeu;
    case 4: return 0x80000000u;
    case 5: return 0x7fffffffu;
    case 6: return with_p ? pw : u;
    default: return with_p ? pm1w : u;
  }
}

FS_HD uint32_t word_of(const uint64_t* v, int w) { return (uint32_t)(v[w >> 1] >> (32 * (w & 1))); }

// G0 / G1: words drawn uniformly or from the palette, masked to p's bit length, rejected if >= p
template <int M>
FS_HD void gen_masked(const Ref<M>& f, bool palette, uint64_t seed, uint64_t idx, uint32_t slot, uint64_t* out) {
  const int topbits = f.bits - 64 * (M - 1);
  const uint64_t topmask = topbits >= 64 ? ~0ull : ((1ull << topbits) - 1);
  for (uint32_t attempt = 0; attempt < 64; attempt++) {
#pragma unroll
    for (int i = 0; i < M; i++) {
      uint32_t w2[2];
#pragma unroll
      for (int h = 0; h < 2; h++) {
        const int w = 2 * i + h;
        const uint64_t x = hash(seed, idx, slot, attempt * 64 + w);
        const uint32_t pw = word_of(f.p, w);
        w2[h] = palette ? palette_word(x, pw, w == 0 ? pw - 1 : pw, true) : (uint32_t)x;
      }
      out[i] = (uint64_t)w2[0] | ((uint64_t)w2[1] << 32);
    }
    out[M - 1] &= topmask;
    if (!geq<M>(out, f.p)) return;
  }
#pragma unroll
  for (int i = 0; i < M; i++) out[i] = 0;
}

// G2: the j-th boundary value.  Class j % 7, offset k = j / 7:
//   k, p-1-k, (R mod p) + k, (R mod p) - k, floor(p/2) + k, floor(p/2) - k, 2^(k mod bits) (or p - 2^(k mod bits))
template <int M>
FS_HD void boundary_value(const Ref<M>& f, uint64_t j, uint64_t* out) {
  const int cls = (int)(j % 7);
  const uint64_t k = j / 7;
  uint64_t kk[M];
#pragma unroll
  for (int i = 0; i < M; i++) kk[i] = 0;
  kk[0] = k;
  uint64_t one[M];
#pragma unroll
  for (int i = 0; i < M; i++) one[i] = 0;
  one[0] = 1;
  switch (cls) {
    case 0:
#pragma unroll
      for (int i = 0; i < M; i++) out[i] = kk[i];
      break;
    case 1:
      sub_raw<M>(out, f.p, one);
      sub_raw<M>(out, out, kk);
      break;
    case 2: add<M>(f, out, f.r1, kk); break;
    case 3: sub<M>(f, out, f.r1, kk); break;
    case 4: add_raw<M>(out, f.half, kk); break;
    case 5: sub_raw<M>(out, f.half, kk); break;
    default: {
      const uint64_t e = k % (uint64_t)f.bits;
#pragma unroll
      for (int i = 0; i < M; i++) out[i] = (uint64_t)(i == (int)(e / 64)) << (e % 64);
      if ((k / (uint64_t)f.bits) & 1) sub_raw<M>(out, f.p, out);
    }
  }
}

// the idx-th pair (ja, jb) of naturals, by square shells: all pairs with max(ja, jb) = s come before s + 1
FS_HD void shell_pair(uint64_t idx, uint64_t& ja, uint64_t& jb) {
  uint64_t s = 0;
  {
    // integer square root
    uint64_t lo = 0, hi = 1ull << 32;
    while (hi - lo > 1) {
      const uint64_t mid = (lo + hi) / 2;
      if (mid * mid <= idx) lo = mid; else hi = mid;
    }
    s = lo;
  }
  const uint64_t r = idx - s * s;
  if (r < s) { ja = r; jb = s; } else { ja = s; jb = r - s; }
}

// one field element for (gen, seed, idx, slot); slots 0, 1 enumerate the boundary pairs, higher slots pick boundary
// values by hash among the 224 with the smallest offsets
template <int M>
FS_HD void gen_value(const Ref<M>& f, int gen, uint64_t seed, uint64_t idx, uint32_t slot, uint64_t* out) {
  if (gen == G_BOUNDARY) {
    uint64_t ja, jb;
    shell_pair(idx, ja, jb);
    const uint64_t j = slot == 0 ? ja : slot == 1 ? jb : hash(seed, idx, slot, 0xb0b0) % 224;
    boundary_value<M>(f, j, out);
  } else {
    gen_masked<M>(f, gen != G_UNIFORM, seed, idx, slot, out);
  }
}

// G3: T = T_lo + R T_hi < p R; T_lo all palette words or all uniform words (any value below R), T_hi a G1 value
template <int M>
FS_HD void gen_wide_T(const Ref<M>& f, uint64_t seed, uint64_t idx, uint64_t* T) {
  const bool palette = hash(seed, idx, 0, 0xffff) & 1;
#pragma unroll
  for (int i = 0; i < M; i++) {
    uint32_t w2[2];
#pragma unroll
    for (int h = 0; h < 2; h++) {
      const uint64_t x = hash(seed, idx, 0, 2 * i + h);
      w2[h] = palette ? palette_word(x, 0, 0, false) : (uint32_t)x;
    }
    T[i] = (uint64_t)w2[0] | ((uint64_t)w2[1] << 32);
  }
  gen_masked<M>(f, true, seed, idx, 1, T + M);
}

// the small factor of mul_small: a byte with probability 3/4, a full word otherwise
FS_HD uint32_t gen_small(uint64_t seed, uint64_t idx) {
  const uint64_t h = hash(seed, idx, 7, 0);
  return ((h >> 32) & 3) ? (uint32_t)(h & 0xff) : (uint32_t)h;
}

}  // namespace fsoak
