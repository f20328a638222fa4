// GLV decomposition for BN254 G1, used where a scalar multiplication is a LATENCY chain (rejection attribution): the
// curve endomorphism phi(x, y) = (beta x, y) equals multiplication by lambda (lambda^3 = 1 mod r, beta^3 = 1 mod p), so
//   k P = k1 P + k2 phi(P)   with |k1|, |k2| < 2^128,
// which halves the dependent doublings.  The reference has no such step (its scalar multiplications are the serial
// windowed MSM of arithmetic.rs:26-108); the group element computed is the same, so nothing observable changes.
//
// Lattice basis of {(a, b): a + b lambda = 0 mod r} (extended Euclid on (r, lambda), tools checked in tests/test_host_stages.py):
//   v1 = (A1, -B1M), v2 = (A2, B2), det = r.   c1 = floor(k G1 / 2^256), c2 = floor(k G2 / 2^256) with
//   G1 = floor(2^256 B2 / r), G2 = floor(2^256 B1M / r);   k1 = k - c1 A1 - c2 A2,  k2 = c1 B1M - c2 B2.
// With floors instead of roundings the halves stay below 2^128 (checked on 2 * 10^5 random scalars and the edge cases).
#pragma once
#include "curve.cuh"
#include <algorithm>
#include <cmath>

namespace h2v {

struct GlvHalf {
  u32 l[5];  // magnitude (little-endian limbs, < 2^129)
  bool neg;
};

// schoolbook product of an na-limb by an nb-limb integer, limbs [lo, lo + n) of it
template <int NA, int NB, int LO, int N>
H2V_HD void glv_mul_limbs(const u32* a, const u32* b, u32* out) {
  u32 full[NA + NB];
#pragma unroll
  for (int i = 0; i < NA + NB; i++) full[i] = 0;
#pragma unroll
  for (int i = 0; i < NA; i++) {
    u64 cy = 0;
#pragma unroll
    for (int j = 0; j < NB; j++) {
      cy += (u64)a[i] * b[j] + full[i + j];
      full[i + j] = (u32)cy;
      cy >>= 32;
    }
    full[i + NB] = (u32)cy;
  }
#pragma unroll
  for (int i = 0; i < N; i++) out[i] = LO + i < NA + NB ? full[LO + i] : 0u;
}

// the lattice basis above, as local arrays (device code cannot read namespace-scope host arrays)
#define H2V_GLV_BASIS                                                              \
  const u32 A1[2] = {0x94d213e3u, 0x89d32568u};                                    \
  const u32 B1M[4] = {0x7d4f1128u, 0x8211bbebu, 0xeeb859fcu, 0x6f4d8248u};         \
  const u32 A2[4] = {0x1221250bu, 0x0be4e154u, 0xeeb859fdu, 0x6f4d8248u};          \
  const u32 B2[2] = {0x94d213e3u, 0x89d32568u};

// k: canonical scalar (8 limbs, < r)
H2V_HD void glv_decompose(const u32* k, GlvHalf& h1, GlvHalf& h2) {
  H2V_GLV_BASIS
  const u32 G1[3] = {0xc7e0b3d7u, 0xd91d232eu, 0x00000002u};
  const u32 G2[5] = {0x391eb18du, 0x7a7bd9d4u, 0xa773d2cfu, 0x4ccef014u, 0x00000002u};
  u32 c1[3], c2[5];
  glv_mul_limbs<8, 3, 8, 3>(k, G1, c1);
  glv_mul_limbs<8, 5, 8, 5>(k, G2, c2);
  // everything below modulo 2^192 (two's complement): the results are below 2^129 in magnitude
  u32 p11[6], p22[6], q11[6], q22[6];
  glv_mul_limbs<3, 2, 0, 6>(c1, A1, p11);
  glv_mul_limbs<5, 4, 0, 6>(c2, A2, p22);
  glv_mul_limbs<3, 4, 0, 6>(c1, B1M, q11);
  glv_mul_limbs<5, 2, 0, 6>(c2, B2, q22);
  u32 k1[6], k2[6];
  {
    long long br = 0;  // k1 = k - p11 - p22
#pragma unroll
    for (int i = 0; i < 6; i++) {
      long long d = (long long)k[i] - (long long)p11[i] - (long long)p22[i] + br;
      k1[i] = (u32)d;
      br = d >> 32;  // arithmetic shift: -2, -1 or 0
    }
    br = 0;  // k2 = q11 - q22
#pragma unroll
    for (int i = 0; i < 6; i++) {
      long long d = (long long)q11[i] - (long long)q22[i] + br;
      k2[i] = (u32)d;
      br = d >> 32;
    }
  }
  auto finish = [](const u32* v, GlvHalf& h) {
    h.neg = (v[5] >> 31) != 0;
    u64 cy = h.neg ? 1 : 0;
#pragma unroll
    for (int i = 0; i < 5; i++) {
      cy += h.neg ? (u32)~v[i] : v[i];
      h.l[i] = (u32)cy;
      cy >>= 32;
    }
  };
  finish(k1, h1);
  finish(k2, h2);
}

// Bounds of the halves for EVERY canonical k.  With u1 = k B2 / r and u2 = k B1M / r (reals), A1 B2 + B1M A2 = r gives
// k = u1 A1 + u2 A2 and u1 B1M = u2 B2.  G1, G2 are floors of 2^256 B2 / r and 2^256 B1M / r, so k G_i / 2^256 = u_i - e_i with
// 0 <= e_i < k / 2^256 < 1/4, and f_i = u_i - c_i lies in [e_i, 1 + e_i), inside [0, 5/4).  Hence
//   k1 = f1 A1 + f2 A2  in [0, 5/4 (A1 + A2)),     k2 = f2 B2 - f1 B1M  in (-5/4 B1M, 5/4 B2).
//
// Lattice lift for the bucket MSM (k_msm_digits).  The halves alone fill a window set badly: they sit in [0, ~A2) and
// (-~B1M, 0], so the top window of a 2^(W c - 1) range uses a few of its buckets, each ~20x the mean load.  Adding
// z v2 + (z' + 1) v1 (v1 = (A1, -B1M), v2 = (A2, B2) are lattice vectors: the same k) spreads them over the range:
//   a =  k1 + z A2 + (z' + 1) A1          in [0, 5/4 (A1 + A2) + (Z - 1) A2 + Z' A1)
//   b = -k2 - z B2 + (z' + 1) B1M         in (B1M - 5/4 B2 - (Z - 1) B2, (Z' + 5/4) B1M)
// for z < Z, z' < Z', with k = a - b lambda (mod r): row 2 t carries the digits of a on P, row 2 t + 1 those of -b on phi(P).
// b > 0 thanks to the + 1 on z' (k2 may be positive, up to 5/4 B2); glv_lift_ranges picks Z, Z' with both below 2^(W c - 1),
// so the top signed digit never carries out of window W - 1.
H2V_HD void glv_lift(const GlvHalf& h1, const GlvHalf& h2, u32 z, u32 z2, u32* a, u32* b) {
  H2V_GLV_BASIS
  // two's complement modulo 2^192: acc = +- half, then acc += s * v (v: nv limbs) or acc -= s * v
  auto load = [](const GlvHalf& h, bool negate, u32* acc) {
    const bool neg = h.neg != negate;
    u64 cy = neg ? 1 : 0;
#pragma unroll
    for (int i = 0; i < 6; i++) {
      const u32 m = i < 5 ? h.l[i] : 0u;
      cy += neg ? (u32)~m : m;
      acc[i] = (u32)cy;
      cy >>= 32;
    }
  };
  auto madd = [](u32* acc, const u32* v, int nv, u32 s, bool sub) {
    u32 p[6];
    u64 cy = 0;
#pragma unroll
    for (int i = 0; i < 6; i++) {
      cy += i < nv ? (u64)v[i] * s : 0;
      p[i] = (u32)cy;
      cy >>= 32;
    }
    long long br = 0;
#pragma unroll
    for (int i = 0; i < 6; i++) {
      const long long d = (long long)acc[i] + (sub ? -(long long)p[i] : (long long)p[i]) + br;
      acc[i] = (u32)d;
      br = d >> 32;
    }
  };
  u32 x[6], y[6];
  load(h1, false, x);
  madd(x, A2, 4, z, false);
  madd(x, A1, 2, z2 + 1, false);
  load(h2, true, y);
  madd(y, B2, 2, z, true);
  madd(y, B1M, 4, z2 + 1, false);
#pragma unroll
  for (int i = 0; i < 5; i++) {
    a[i] = x[i];
    b[i] = y[i];
  }
}

// The lifted halves of the scalar k (canonical) of MSM term t (k_msm_digits): z < Z and z' < Z' hashed from the term id,
// like the scalar lift k + z r of the plain windows
H2V_HD void glv_lift_term(const u32* k, u32 t, u32 Z, u32 Z2, u32* a, u32* b) {
  GlvHalf h1, h2;
  glv_decompose(k, h1, h2);
  glv_lift(h1, h2, ((t * 2654435761u) >> 8) % Z, ((t * 2246822519u) >> 8) % Z2, a, b);
}

// Lift ranges (Z, Z') of a window range 2^(W c - 1) (host, the geometry model): the largest with both bounds of glv_lift
// below it, from long-double values of the basis with a relative margin of 1e-9.  Z' >= 1 needs W c >= 130.
inline void glv_lift_ranges(u32 c, u32 W, u32& Z, u32& Z2) {
  const long double A1 = 9931322734385697763.0L;                         // 0x89d3256894d213e3 (= B2)
  const long double B1M = 147946756881789319000765030803803410728.0L;    // 0x6f4d8248eeb859fc8211bbeb7d4f1128
  const long double A2 = 147946756881789319010696353538189108491.0L;     // 0x6f4d8248eeb859fd0be4e1541221250b
  const long double cap = std::ldexp(1.0L, (int)(W * c) - 1), keep = 1.0L - 1e-9L;
  Z = Z2 = 0;
  const long double z2 = std::floor((cap / B1M - 1.25L) * keep);  // (Z' + 5/4) B1M <= cap
  if (z2 < 1.0L) return;
  const long double z = std::floor((cap - 1.25L * (A1 + A2) - z2 * A1) / A2 * keep) + 1.0L;  // 5/4 (A1 + A2) + (Z - 1) A2 + Z' A1 <= cap
  Z2 = (u32)std::min(z2, 65536.0L);
  Z = (u32)std::min(z, 65536.0L);
}

H2V_HD Fq glv_beta() {  // Montgomery form of beta = 0x59e26bcea0d48bacd4f263f1acdb5c4f5763473177fffffe
  Fq b;
  const u32 v[8] = {0xd782e155u, 0x71930c11u, 0xffbe3323u, 0xa6bb947cu, 0xd4741444u, 0xaa303344u, 0x26594943u, 0x2c3b3f0du};
#pragma unroll
  for (int i = 0; i < 8; i++) b.l[i] = v[i];
  return b;
}

// One of the FOUR summands of [k] P = k1 P + k2 phi(P):  ((k_h >> lo) mod 2^len) * 2^tail * P_h  with P_0 = P, P_1 = phi(P) and the
// sign of the half applied.  (half, lo, len, tail) = (h, 64, 65, 64) and (h, 0, 64, 0) for h = 0, 1 give four chains of at most
// 129 doublings instead of one of 254.  One half per chain on purpose: a joint double-and-add over both halves has three
// different additions (P, phi(P), P + phi(P)) and the lanes of a warp would serialise them (measured: slower than no GLV).
H2V_HDN inline G1Jac g1_mul_glv_part(const G1Affine& p, const GlvHalf& h, bool endo, u32 lo, u32 len, u32 tail) {
  G1Affine q = p;
  if (endo) q.x = Fq::mul_c(p.x, glv_beta());
  if (h.neg) q.y = q.y.neg();
  G1Jac acc = G1Jac::identity();
  for (u32 i = len; i-- > 0;) {
    const u32 bit = lo + i;
    acc = g1_double(acc);
    if (bit < 160 && ((h.l[bit >> 5] >> (bit & 31)) & 1u)) acc = g1_add_mixed(acc, q);
  }
  for (u32 i = 0; i < tail; i++) acc = g1_double(acc);
  return acc;
}

// Same with a Jacobian base (window sums and accumulators of h2v_acc_absorb, acc.cuh): phi(X, Y, Z) = (beta X, Y, Z) holds
// in Jacobian coordinates too (x = X / Z^2 scales with X), so no inversion is needed.  (A separate function rather than a
// template over the base, so that the affine callers' code stays as it was.)
H2V_HDN inline G1Jac g1_mul_glv_part(const G1Jac& p, const GlvHalf& h, bool endo, u32 lo, u32 len, u32 tail) {
  G1Jac q = p;
  if (endo) q.X = Fq::mul_c(p.X, glv_beta());
  if (h.neg) q.Y = q.Y.neg();
  G1Jac acc = G1Jac::identity();
  for (u32 i = len; i-- > 0;) {
    const u32 bit = lo + i;
    acc = g1_double(acc);
    if (bit < 160 && ((h.l[bit >> 5] >> (bit & 31)) & 1u)) acc = g1_add(acc, q);
  }
  for (u32 i = 0; i < tail; i++) acc = g1_double(acc);
  return acc;
}

}  // namespace h2v
