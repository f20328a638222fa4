// 256-bit Montgomery field arithmetic for BN254 Fr / Fq, 8 x 32-bit limbs held in registers.
//
// The reference has no such code in-tree: it calls into halo2curves (Cargo.toml:15) at
//   transcript/mod.rs:161-162,171,220-221,228,502   (from_bytes / from_repr / to_repr / from_uniform_bytes)
//   lib.rs:180,259  vanishing.rs:100  shplonk.rs:215  domain.rs:175-179,202  arithmetic.rs:169  vk.rs:583
// Everything here is written for sm_100a (CIOS on the IMAD pipe); the same source compiles for the
// host (plan compiler, host test harness) through the H2V_HD macro.
#pragma once
#include <stddef.h>
#include <stdint.h>

#if defined(__CUDACC__)
#define H2V_HD __host__ __device__ __forceinline__
#define H2V_HDN __host__ __device__ __noinline__
#else
#define H2V_HD inline
#define H2V_HDN
#endif

namespace h2v {

typedef uint32_t u32;
typedef uint64_t u64;
typedef uint8_t u8;

struct FqP {
  static constexpr bool CALL_MUL = false;  // operator* inlined: the curve / pairing kernels are tight loops around it
  static H2V_HD constexpr u32 mod(int i) {
    constexpr u32 v[8] = {0xd87cfd47u, 0x3c208c16u, 0x6871ca8du, 0x97816a91u, 0x8181585du, 0xb85045b6u, 0xe131a029u, 0x30644e72u};
    return v[i];
  }
  static H2V_HD constexpr u32 r1(int i) {
    constexpr u32 v[8] = {0xc58f0d9du, 0xd35d438du, 0xf5c70b3du, 0x0a78eb28u, 0x7879462cu, 0x666ea36fu, 0x9a07df2fu, 0x0e0a77c1u};
    return v[i];
  }
  static H2V_HD constexpr u32 r2(int i) {
    constexpr u32 v[8] = {0x538afa89u, 0xf32cfc5bu, 0xd44501fbu, 0xb5e71911u, 0x0a417ff6u, 0x47ab1effu, 0xcab8351fu, 0x06d89f71u};
    return v[i];
  }
  static H2V_HD constexpr u32 r3(int i) {
    constexpr u32 v[8] = {0xda1530dfu, 0xb1cd6dafu, 0xa7283db6u, 0x62f210e6u, 0x0ada0afbu, 0xef7f0b0cu, 0x2d592544u, 0x20fd6e90u};
    return v[i];
  }
  static constexpr u32 INV = 0xe4866389u;
};

struct FrP {
  // operator* as ONE out-of-line function per kernel (device): the scalar stage has ~100 multiplication sites, inlined they
  // were 29.5 k instructions (0.47 MB) in k_scalar and 14 % of its warp stalls were instruction fetches (ncu, r2b; now 9.3 k)
  static constexpr bool CALL_MUL = true;
  static H2V_HD constexpr u32 mod(int i) {
    constexpr u32 v[8] = {0xf0000001u, 0x43e1f593u, 0x79b97091u, 0x2833e848u, 0x8181585du, 0xb85045b6u, 0xe131a029u, 0x30644e72u};
    return v[i];
  }
  static H2V_HD constexpr u32 r1(int i) {
    constexpr u32 v[8] = {0x4ffffffbu, 0xac96341cu, 0x9f60cd29u, 0x36fc7695u, 0x7879462eu, 0x666ea36fu, 0x9a07df2fu, 0x0e0a77c1u};
    return v[i];
  }
  static H2V_HD constexpr u32 r2(int i) {
    constexpr u32 v[8] = {0xae216da7u, 0x1bb8e645u, 0xe35c59e3u, 0x53fe3ab1u, 0x53bb8085u, 0x8c49833du, 0x7f4e44a5u, 0x0216d0b1u};
    return v[i];
  }
  static H2V_HD constexpr u32 r3(int i) {
    constexpr u32 v[8] = {0xb4bf0040u, 0x5e94d8e1u, 0x1cfbb6b8u, 0x2a489cbeu, 0xa19fcfedu, 0x893cc664u, 0x7fcc657cu, 0x0cf8594bu};
    return v[i];
  }
  static constexpr u32 INV = 0xefffffffu;
};

// -------------------------------------------------------------------------------------------------
// Device Montgomery multiplication: 8-limb CIOS written against the IMAD pipe with explicit carry
// chains (mad.lo.cc / madc.hi.cc).  The portable path below is bit-identical and is what the host
// build uses; tests/test_gpu_field.py cross-checks the two on random and edge inputs.
// -------------------------------------------------------------------------------------------------
#if defined(__CUDA_ARCH__) && !defined(H2V_NO_PTX)
#define H2V_PTX 1
#endif

#ifdef H2V_PTX
__device__ __forceinline__ u32 ptx_add_cc(u32 a, u32 b) { u32 r; asm volatile("add.cc.u32 %0, %1, %2;" : "=r"(r) : "r"(a), "r"(b)); return r; }
__device__ __forceinline__ u32 ptx_addc_cc(u32 a, u32 b) { u32 r; asm volatile("addc.cc.u32 %0, %1, %2;" : "=r"(r) : "r"(a), "r"(b)); return r; }
__device__ __forceinline__ u32 ptx_addc(u32 a, u32 b) { u32 r; asm volatile("addc.u32 %0, %1, %2;" : "=r"(r) : "r"(a), "r"(b)); return r; }
__device__ __forceinline__ u32 ptx_sub_cc(u32 a, u32 b) { u32 r; asm volatile("sub.cc.u32 %0, %1, %2;" : "=r"(r) : "r"(a), "r"(b)); return r; }
__device__ __forceinline__ u32 ptx_subc_cc(u32 a, u32 b) { u32 r; asm volatile("subc.cc.u32 %0, %1, %2;" : "=r"(r) : "r"(a), "r"(b)); return r; }
__device__ __forceinline__ u32 ptx_subc(u32 a, u32 b) { u32 r; asm volatile("subc.u32 %0, %1, %2;" : "=r"(r) : "r"(a), "r"(b)); return r; }
__device__ __forceinline__ u32 ptx_mad_lo_cc(u32 a, u32 b, u32 c) { u32 r; asm volatile("mad.lo.cc.u32 %0, %1, %2, %3;" : "=r"(r) : "r"(a), "r"(b), "r"(c)); return r; }
__device__ __forceinline__ u32 ptx_madc_lo_cc(u32 a, u32 b, u32 c) { u32 r; asm volatile("madc.lo.cc.u32 %0, %1, %2, %3;" : "=r"(r) : "r"(a), "r"(b), "r"(c)); return r; }
__device__ __forceinline__ u32 ptx_mad_hi_cc(u32 a, u32 b, u32 c) { u32 r; asm volatile("mad.hi.cc.u32 %0, %1, %2, %3;" : "=r"(r) : "r"(a), "r"(b), "r"(c)); return r; }
__device__ __forceinline__ u32 ptx_madc_hi_cc(u32 a, u32 b, u32 c) { u32 r; asm volatile("madc.hi.cc.u32 %0, %1, %2, %3;" : "=r"(r) : "r"(a), "r"(b), "r"(c)); return r; }
__device__ __forceinline__ u32 ptx_madc_hi(u32 a, u32 b, u32 c) { u32 r; asm volatile("madc.hi.u32 %0, %1, %2, %3;" : "=r"(r) : "r"(a), "r"(b), "r"(c)); return r; }

// ---- building blocks of the even/odd wide multiplication (Fp::mul).  Each carry chain is ONE asm
// statement, so no carry flag is live between statements and the compiler may interleave chains.
// ptxas fuses every (mad.lo.cc, madc.hi.cc) pair into one IMAD.WIDE.U32 with carry in/out.
// acc[0..7] = (a0, a2, a4, a6) * b as four 64-bit products
__device__ __forceinline__ void wide_mul4(u32 (&acc)[8], u32 a0, u32 a2, u32 a4, u32 a6, u32 b) {
  asm("mul.lo.u32 %0, %8, %12; mul.hi.u32 %1, %8, %12;\n\t"
      "mul.lo.u32 %2, %9, %12; mul.hi.u32 %3, %9, %12;\n\t"
      "mul.lo.u32 %4, %10, %12; mul.hi.u32 %5, %10, %12;\n\t"
      "mul.lo.u32 %6, %11, %12; mul.hi.u32 %7, %11, %12;"
      : "=r"(acc[0]), "=r"(acc[1]), "=r"(acc[2]), "=r"(acc[3]), "=r"(acc[4]), "=r"(acc[5]), "=r"(acc[6]), "=r"(acc[7])
      : "r"(a0), "r"(a2), "r"(a4), "r"(a6), "r"(b));
}
// acc[0..7] += (a0, a2, a4, a6) * b along one carry chain; returns the carry out
__device__ __forceinline__ u32 wide_mad4_carry(u32 (&acc)[8], u32 a0, u32 a2, u32 a4, u32 a6, u32 b) {
  u32 cy;
  asm("mad.lo.cc.u32 %0, %9, %13, %0; madc.hi.cc.u32 %1, %9, %13, %1;\n\t"
      "madc.lo.cc.u32 %2, %10, %13, %2; madc.hi.cc.u32 %3, %10, %13, %3;\n\t"
      "madc.lo.cc.u32 %4, %11, %13, %4; madc.hi.cc.u32 %5, %11, %13, %5;\n\t"
      "madc.lo.cc.u32 %6, %12, %13, %6; madc.hi.cc.u32 %7, %12, %13, %7;\n\t"
      "addc.u32 %8, 0, 0;"
      : "+r"(acc[0]), "+r"(acc[1]), "+r"(acc[2]), "+r"(acc[3]), "+r"(acc[4]), "+r"(acc[5]), "+r"(acc[6]), "+r"(acc[7]), "=r"(cy)
      : "r"(a0), "r"(a2), "r"(a4), "r"(a6), "r"(b));
  return cy;
}
// same, carry out dropped (the caller knows the sum fits)
__device__ __forceinline__ void wide_mad4(u32 (&acc)[8], u32 a0, u32 a2, u32 a4, u32 a6, u32 b) {
  asm("mad.lo.cc.u32 %0, %8, %12, %0; madc.hi.cc.u32 %1, %8, %12, %1;\n\t"
      "madc.lo.cc.u32 %2, %9, %12, %2; madc.hi.cc.u32 %3, %9, %12, %3;\n\t"
      "madc.lo.cc.u32 %4, %10, %12, %4; madc.hi.cc.u32 %5, %10, %12, %5;\n\t"
      "madc.lo.cc.u32 %6, %11, %12, %6; madc.hi.u32 %7, %11, %12, %7;"
      : "+r"(acc[0]), "+r"(acc[1]), "+r"(acc[2]), "+r"(acc[3]), "+r"(acc[4]), "+r"(acc[5]), "+r"(acc[6]), "+r"(acc[7])
      : "r"(a0), "r"(a2), "r"(a4), "r"(a6), "r"(b));
}
// even0 += odd[1] (carry kept), then odd = (odd >> 64) + (a1, a3, a5, a7) * b with that carry folded in
__device__ __forceinline__ void wide_fold_mad4_rshift(u32& even0, u32 (&odd)[8], u32 a1, u32 a3, u32 a5, u32 a7, u32 b) {
  asm("add.cc.u32 %8, %8, %1;\n\t"
      "madc.lo.cc.u32 %0, %9, %13, %2; madc.hi.cc.u32 %1, %9, %13, %3;\n\t"
      "madc.lo.cc.u32 %2, %10, %13, %4; madc.hi.cc.u32 %3, %10, %13, %5;\n\t"
      "madc.lo.cc.u32 %4, %11, %13, %6; madc.hi.cc.u32 %5, %11, %13, %7;\n\t"
      "madc.lo.cc.u32 %6, %12, %13, 0; madc.hi.u32 %7, %12, %13, 0;"
      : "+r"(odd[0]), "+r"(odd[1]), "+r"(odd[2]), "+r"(odd[3]), "+r"(odd[4]), "+r"(odd[5]), "+r"(odd[6]), "+r"(odd[7]), "+r"(even0)
      : "r"(a1), "r"(a3), "r"(a5), "r"(a7), "r"(b));
}
// ---- shorter rows for the dedicated squaring (Fp::sqr): the multiplicand vector of row i starts with i
// zeros, so the first S products of a chain are skipped (the chain starts higher up / only shifts).
// acc[2S..7] += (terms from slot S on) * b, returns the carry out
__device__ __forceinline__ u32 wide_mad3_carry(u32 (&acc)[8], u32 a2, u32 a4, u32 a6, u32 b) {
  u32 cy;
  asm("mad.lo.cc.u32 %0, %7, %10, %0; madc.hi.cc.u32 %1, %7, %10, %1;\n\t"
      "madc.lo.cc.u32 %2, %8, %10, %2; madc.hi.cc.u32 %3, %8, %10, %3;\n\t"
      "madc.lo.cc.u32 %4, %9, %10, %4; madc.hi.cc.u32 %5, %9, %10, %5;\n\t"
      "addc.u32 %6, 0, 0;"
      : "+r"(acc[2]), "+r"(acc[3]), "+r"(acc[4]), "+r"(acc[5]), "+r"(acc[6]), "+r"(acc[7]), "=r"(cy)
      : "r"(a2), "r"(a4), "r"(a6), "r"(b));
  return cy;
}
__device__ __forceinline__ u32 wide_mad2_carry(u32 (&acc)[8], u32 a4, u32 a6, u32 b) {
  u32 cy;
  asm("mad.lo.cc.u32 %0, %5, %7, %0; madc.hi.cc.u32 %1, %5, %7, %1;\n\t"
      "madc.lo.cc.u32 %2, %6, %7, %2; madc.hi.cc.u32 %3, %6, %7, %3;\n\t"
      "addc.u32 %4, 0, 0;"
      : "+r"(acc[4]), "+r"(acc[5]), "+r"(acc[6]), "+r"(acc[7]), "=r"(cy)
      : "r"(a4), "r"(a6), "r"(b));
  return cy;
}
__device__ __forceinline__ u32 wide_mad1_carry(u32 (&acc)[8], u32 a6, u32 b) {
  u32 cy;
  asm("mad.lo.cc.u32 %0, %3, %4, %0; madc.hi.cc.u32 %1, %3, %4, %1;\n\t"
      "addc.u32 %2, 0, 0;"
      : "+r"(acc[6]), "+r"(acc[7]), "=r"(cy)
      : "r"(a6), "r"(b));
  return cy;
}
// wide_fold_mad4_rshift with the first 1 / 2 / 3 products skipped (those slots only shift down)
__device__ __forceinline__ void wide_fold_mad3_rshift(u32& even0, u32 (&odd)[8], u32 a3, u32 a5, u32 a7, u32 b) {
  asm("add.cc.u32 %8, %8, %1;\n\t"
      "addc.cc.u32 %0, %2, 0; addc.cc.u32 %1, %3, 0;\n\t"
      "madc.lo.cc.u32 %2, %9, %12, %4; madc.hi.cc.u32 %3, %9, %12, %5;\n\t"
      "madc.lo.cc.u32 %4, %10, %12, %6; madc.hi.cc.u32 %5, %10, %12, %7;\n\t"
      "madc.lo.cc.u32 %6, %11, %12, 0; madc.hi.u32 %7, %11, %12, 0;"
      : "+r"(odd[0]), "+r"(odd[1]), "+r"(odd[2]), "+r"(odd[3]), "+r"(odd[4]), "+r"(odd[5]), "+r"(odd[6]), "+r"(odd[7]), "+r"(even0)
      : "r"(a3), "r"(a5), "r"(a7), "r"(b));
}
__device__ __forceinline__ void wide_fold_mad2_rshift(u32& even0, u32 (&odd)[8], u32 a5, u32 a7, u32 b) {
  asm("add.cc.u32 %8, %8, %1;\n\t"
      "addc.cc.u32 %0, %2, 0; addc.cc.u32 %1, %3, 0;\n\t"
      "addc.cc.u32 %2, %4, 0; addc.cc.u32 %3, %5, 0;\n\t"
      "madc.lo.cc.u32 %4, %9, %11, %6; madc.hi.cc.u32 %5, %9, %11, %7;\n\t"
      "madc.lo.cc.u32 %6, %10, %11, 0; madc.hi.u32 %7, %10, %11, 0;"
      : "+r"(odd[0]), "+r"(odd[1]), "+r"(odd[2]), "+r"(odd[3]), "+r"(odd[4]), "+r"(odd[5]), "+r"(odd[6]), "+r"(odd[7]), "+r"(even0)
      : "r"(a5), "r"(a7), "r"(b));
}
__device__ __forceinline__ void wide_fold_mad1_rshift(u32& even0, u32 (&odd)[8], u32 a7, u32 b) {
  asm("add.cc.u32 %8, %8, %1;\n\t"
      "addc.cc.u32 %0, %2, 0; addc.cc.u32 %1, %3, 0;\n\t"
      "addc.cc.u32 %2, %4, 0; addc.cc.u32 %3, %5, 0;\n\t"
      "addc.cc.u32 %4, %6, 0; addc.cc.u32 %5, %7, 0;\n\t"
      "madc.lo.cc.u32 %6, %9, %10, 0; madc.hi.u32 %7, %9, %10, 0;"
      : "+r"(odd[0]), "+r"(odd[1]), "+r"(odd[2]), "+r"(odd[3]), "+r"(odd[4]), "+r"(odd[5]), "+r"(odd[6]), "+r"(odd[7]), "+r"(even0)
      : "r"(a7), "r"(b));
}
#endif

template <class P>
struct alignas(16) Fp {  // 16-byte alignment: element loads / stores vectorise to two 128-bit accesses
  u32 l[8];

  // ---- constants
  static H2V_HD Fp zero() {
    Fp r;
#pragma unroll
    for (int i = 0; i < 8; i++) r.l[i] = 0;
    return r;
  }
  static H2V_HD Fp one() {  // Montgomery form of 1
    Fp r;
#pragma unroll
    for (int i = 0; i < 8; i++) r.l[i] = P::r1(i);
    return r;
  }
  static H2V_HD Fp r2() {
    Fp r;
#pragma unroll
    for (int i = 0; i < 8; i++) r.l[i] = P::r2(i);
    return r;
  }
  static H2V_HD Fp r3() {
    Fp r;
#pragma unroll
    for (int i = 0; i < 8; i++) r.l[i] = P::r3(i);
    return r;
  }

  // ---- predicates (on the raw representation)
  H2V_HD bool is_zero() const {
    u32 a = 0;
#pragma unroll
    for (int i = 0; i < 8; i++) a |= l[i];
    return a == 0;
  }
  H2V_HD bool operator==(const Fp& o) const {
    u32 a = 0;
#pragma unroll
    for (int i = 0; i < 8; i++) a |= l[i] ^ o.l[i];
    return a == 0;
  }
  H2V_HD bool operator!=(const Fp& o) const { return !(*this == o); }
  // raw >= modulus ?
  H2V_HD bool geq_mod() const {
#pragma unroll
    for (int i = 7; i >= 0; i--) {
      if (l[i] > P::mod(i)) return true;
      if (l[i] < P::mod(i)) return false;
    }
    return true;
  }

  // ---- raw 256-bit helpers
  static H2V_HD u32 add_raw(u32* r, const u32* a, const u32* b) {  // returns carry
#ifdef H2V_PTX
    r[0] = ptx_add_cc(a[0], b[0]);
#pragma unroll
    for (int i = 1; i < 8; i++) r[i] = ptx_addc_cc(a[i], b[i]);
    return ptx_addc(0, 0);
#else
    u64 c = 0;
#pragma unroll
    for (int i = 0; i < 8; i++) {
      c += (u64)a[i] + b[i];
      r[i] = (u32)c;
      c >>= 32;
    }
    return (u32)c;
#endif
  }
  static H2V_HD u32 sub_raw(u32* r, const u32* a, const u32* b) {  // returns borrow (1 if a < b)
#ifdef H2V_PTX
    r[0] = ptx_sub_cc(a[0], b[0]);
#pragma unroll
    for (int i = 1; i < 8; i++) r[i] = ptx_subc_cc(a[i], b[i]);
    return ptx_subc(0, 0) & 1u;
#else
    u64 br = 0;
#pragma unroll
    for (int i = 0; i < 8; i++) {
      u64 t = (u64)a[i] - b[i] - br;
      r[i] = (u32)t;
      br = (t >> 32) & 1u;
    }
    return (u32)br;
#endif
  }
  H2V_HD void cond_sub_mod() {  // if raw >= p: raw -= p
    u32 m[8], t[8];
#pragma unroll
    for (int i = 0; i < 8; i++) m[i] = P::mod(i);
    u32 br = sub_raw(t, l, m);
    if (!br) {
#pragma unroll
      for (int i = 0; i < 8; i++) l[i] = t[i];
    }
  }

  // ---- field ops (Montgomery form in, Montgomery form out; inputs < p)
  friend H2V_HD Fp operator+(const Fp& a, const Fp& b) {
    Fp r;
    add_raw(r.l, a.l, b.l);  // p < 2^254: no carry out
    r.cond_sub_mod();
    return r;
  }
  friend H2V_HD Fp operator-(const Fp& a, const Fp& b) {
    Fp r;
    u32 br = sub_raw(r.l, a.l, b.l);
    if (br) {
      u32 m[8];
#pragma unroll
      for (int i = 0; i < 8; i++) m[i] = P::mod(i);
      add_raw(r.l, r.l, m);
    }
    return r;
  }
  H2V_HD Fp neg() const { return is_zero() ? *this : (zero() - *this); }
  H2V_HD Fp dbl() const { return *this + *this; }

  // Portable CIOS (bit-identical reference for the PTX path; the only path of the host build).
  static H2V_HD Fp mul_portable(const Fp& a, const Fp& b) {
    Fp r;
    u32 t[10];
#pragma unroll
    for (int i = 0; i < 10; i++) t[i] = 0;
#pragma unroll
    for (int i = 0; i < 8; i++) {
      u64 c = 0;
      const u32 bi = b.l[i];
#pragma unroll
      for (int j = 0; j < 8; j++) {
        c += (u64)a.l[j] * bi + t[j];
        t[j] = (u32)c;
        c >>= 32;
      }
      c += t[8];
      t[8] = (u32)c;
      t[9] = (u32)(c >> 32);
      const u32 m = t[0] * P::INV;
      c = (u64)m * P::mod(0) + t[0];
      c >>= 32;
#pragma unroll
      for (int j = 1; j < 8; j++) {
        c += (u64)m * P::mod(j) + t[j];
        t[j - 1] = (u32)c;
        c >>= 32;
      }
      c += t[8];
      t[7] = (u32)c;
      t[8] = t[9] + (u32)(c >> 32);
    }
#pragma unroll
    for (int i = 0; i < 8; i++) r.l[i] = t[i];
    r.cond_sub_mod();
    return r;
  }

#ifdef H2V_PTX
  // One row of the even/odd wide multiplication: acc += a * bi, then one Montgomery reduction step.
  // `even` holds the 32-bit columns 0..7 and `odd` the columns 1..8 of the running sum, each as four
  // 64-bit slots, so every 32x32->64 product lands in one slot and one IMAD.WIDE.U32 accumulates it.
  // After the reduction step column 0 is zero and the arrays swap roles (the shift by one column).
  template <bool FIRST>
  static __device__ __forceinline__ void wide_row(u32 (&even)[8], u32 (&odd)[8], const u32* a, u32 bi) {
    if (FIRST) {
      wide_mul4(odd, a[1], a[3], a[5], a[7], bi);
      wide_mul4(even, a[0], a[2], a[4], a[6], bi);
    } else {
      wide_fold_mad4_rshift(even[0], odd, a[1], a[3], a[5], a[7], bi);
      odd[7] += wide_mad4_carry(even, a[0], a[2], a[4], a[6], bi);
    }
    const u32 mi = even[0] * P::INV;
    wide_mad4(odd, P::mod(1), P::mod(3), P::mod(5), P::mod(7), mi);
    odd[7] += wide_mad4_carry(even, P::mod(0), P::mod(2), P::mod(4), P::mod(6), mi);
  }
  // Row I of the squaring: a^2 = sum_i a_i 2^(32 i) * (a_i 2^(32 i) + [2a with the bits below limb i+1 cleared]),
  // i.e. a multiplication row whose multiplicand v has v_j = 0 (j < I), v_I = a_I, v_(I+1) = a_(I+1) << 1,
  // v_j = limb j of 2a (j > I+1): 36 products instead of 64.  Column i only receives products of rows <= i/2,
  // so the interleaved reduction steps are those of `wide_row`.
  template <int I>
  static __device__ __forceinline__ void sqr_row(u32 (&even)[8], u32 (&odd)[8], const u32* a, const u32* d) {
    u32 v[8];
#pragma unroll
    for (int j = 0; j < 8; j++) v[j] = j < I ? 0u : j == I ? a[j] : j == I + 1 ? (a[j] << 1) : d[j];
    const u32 bi = a[I];
    constexpr int SO = I / 2, SE = (I + 1) / 2;  // leading zero products of the odd / even chain
    if (I == 0) {
      wide_mul4(odd, v[1], v[3], v[5], v[7], bi);
      wide_mul4(even, v[0], v[2], v[4], v[6], bi);
    } else {
      if (SO == 0) wide_fold_mad4_rshift(even[0], odd, v[1], v[3], v[5], v[7], bi);
      else if (SO == 1) wide_fold_mad3_rshift(even[0], odd, v[3], v[5], v[7], bi);
      else if (SO == 2) wide_fold_mad2_rshift(even[0], odd, v[5], v[7], bi);
      else wide_fold_mad1_rshift(even[0], odd, v[7], bi);
      if (SE == 1) odd[7] += wide_mad3_carry(even, v[2], v[4], v[6], bi);
      else if (SE == 2) odd[7] += wide_mad2_carry(even, v[4], v[6], bi);
      else if (SE == 3) odd[7] += wide_mad1_carry(even, v[6], bi);
    }
    const u32 mi = even[0] * P::INV;
    wide_mad4(odd, P::mod(1), P::mod(3), P::mod(5), P::mod(7), mi);
    odd[7] += wide_mad4_carry(even, P::mod(0), P::mod(2), P::mod(4), P::mod(6), mi);
  }
#endif

  // Montgomery product a*b*2^-256 mod p for REDUCED operands (a, b < p; exact for a < 2^255).
  // Device: 128 IMAD.WIDE.U32 + 8 IMAD on the multiply pipe (half the issue slots of a lo/hi CIOS).
  static H2V_HD Fp mul(const Fp& a, const Fp& b) {
#ifdef H2V_PTX
    u32 even[8], odd[8];
    wide_row<true>(even, odd, a.l, b.l[0]);
    wide_row<false>(odd, even, a.l, b.l[1]);
    wide_row<false>(even, odd, a.l, b.l[2]);
    wide_row<false>(odd, even, a.l, b.l[3]);
    wide_row<false>(even, odd, a.l, b.l[4]);
    wide_row<false>(odd, even, a.l, b.l[5]);
    wide_row<false>(even, odd, a.l, b.l[6]);
    wide_row<false>(odd, even, a.l, b.l[7]);
    Fp r;
    asm("add.cc.u32 %0, %8, %16; addc.cc.u32 %1, %9, %17; addc.cc.u32 %2, %10, %18; addc.cc.u32 %3, %11, %19;\n\t"
        "addc.cc.u32 %4, %12, %20; addc.cc.u32 %5, %13, %21; addc.cc.u32 %6, %14, %22; addc.u32 %7, %15, 0;"
        : "=r"(r.l[0]), "=r"(r.l[1]), "=r"(r.l[2]), "=r"(r.l[3]), "=r"(r.l[4]), "=r"(r.l[5]), "=r"(r.l[6]), "=r"(r.l[7])
        : "r"(even[0]), "r"(even[1]), "r"(even[2]), "r"(even[3]), "r"(even[4]), "r"(even[5]), "r"(even[6]), "r"(even[7]),
          "r"(odd[1]), "r"(odd[2]), "r"(odd[3]), "r"(odd[4]), "r"(odd[5]), "r"(odd[6]), "r"(odd[7]));
    r.cond_sub_mod();
    return r;
#else
    return mul_portable(a, b);
#endif
  }

  // Montgomery product for an UNREDUCED left operand: a < 2^256, b < p with no limb of b equal to 0xFFFFFFFF.  Used
  // where raw 256-bit strings enter the field (from_uniform, from_canonical), always with b = R^2 or R^3 mod p, whose
  // limbs are all below 0xFFFFFFFF (tests/test_field_vectors.py checks this).  With a close to 2^256 and a limb b_i =
  // 0xFFFFFFFF, t + a * b_i can reach 2^288, whose carry out of t[8] is lost: the result is then wrong.
  static H2V_HD Fp mul_any(const Fp& a, const Fp& b) {
#ifdef H2V_PTX
    Fp r;
    // CIOS, one row per limb of b.  t has 9 live limbs (t8 is the running top word).
    u32 t[9];
#pragma unroll
    for (int i = 0; i < 9; i++) t[i] = 0;
#pragma unroll
    for (int i = 0; i < 8; i++) {
      const u32 bi = b.l[i];
      // t += a * bi : low halves then high halves, two carry chains
      t[0] = ptx_mad_lo_cc(a.l[0], bi, t[0]);
#pragma unroll
      for (int j = 1; j < 8; j++) t[j] = ptx_madc_lo_cc(a.l[j], bi, t[j]);
      t[8] = ptx_addc(t[8], 0);
      t[1] = ptx_mad_hi_cc(a.l[0], bi, t[1]);
#pragma unroll
      for (int j = 1; j < 7; j++) t[j + 1] = ptx_madc_hi_cc(a.l[j], bi, t[j + 1]);
      t[8] = ptx_madc_hi(a.l[7], bi, t[8]);
      // m = t0 * inv ; t = (t + m * p) >> 32
      const u32 m = t[0] * P::INV;
      (void)ptx_mad_lo_cc(m, P::mod(0), t[0]);  // low word becomes 0, keep carry
#pragma unroll
      for (int j = 1; j < 8; j++) t[j - 1] = ptx_madc_lo_cc(m, P::mod(j), t[j]);
      t[7] = ptx_addc_cc(t[8], 0);
      t[8] = ptx_addc(0, 0);
      t[0] = ptx_mad_hi_cc(m, P::mod(0), t[0]);
#pragma unroll
      for (int j = 1; j < 7; j++) t[j] = ptx_madc_hi_cc(m, P::mod(j), t[j]);
      t[7] = ptx_madc_hi_cc(m, P::mod(7), t[7]);
      t[8] = ptx_addc(t[8], 0);
    }
#pragma unroll
    for (int i = 0; i < 8; i++) r.l[i] = t[i];
    r.cond_sub_mod();
    return r;
#else
    return mul_portable(a, b);
#endif
  }
#if defined(__CUDA_ARCH__)
  static __device__ __noinline__ Fp mul_call(Fp a, Fp b) { return mul(a, b); }
  static __device__ __noinline__ Fp sqr_call(Fp a) { return a.sqr(); }
#endif
  // products through ONE out-of-line copy per kernel on the device (code size, see FrP::CALL_MUL), inlined on the host
  static H2V_HD Fp mul_c(const Fp& a, const Fp& b) {
#if defined(__CUDA_ARCH__)
    return mul_call(a, b);
#else
    return mul(a, b);
#endif
  }
  static H2V_HD Fp sqr_c(const Fp& a) {
#if defined(__CUDA_ARCH__)
    return sqr_call(a);
#else
    return a.sqr();
#endif
  }
  friend H2V_HD Fp operator*(const Fp& a, const Fp& b) {
#if defined(__CUDA_ARCH__)
    if constexpr (P::CALL_MUL) return mul_call(a, b);
#endif
    return mul(a, b);
  }
  // Montgomery square (a < p): 100 IMAD.WIDE.U32 + 8 IMAD instead of 128 + 8; same integer result as mul(a, a).
  H2V_HD Fp sqr() const {
#ifdef H2V_PTX
    u32 d[8], even[8], odd[8];
    d[0] = l[0] << 1;
#pragma unroll
    for (int j = 1; j < 8; j++) d[j] = __funnelshift_l(l[j - 1], l[j], 1);  // limbs of 2a (< 2^255)
    sqr_row<0>(even, odd, l, d);
    sqr_row<1>(odd, even, l, d);
    sqr_row<2>(even, odd, l, d);
    sqr_row<3>(odd, even, l, d);
    sqr_row<4>(even, odd, l, d);
    sqr_row<5>(odd, even, l, d);
    sqr_row<6>(even, odd, l, d);
    sqr_row<7>(odd, even, l, d);
    Fp r;
    asm("add.cc.u32 %0, %8, %16; addc.cc.u32 %1, %9, %17; addc.cc.u32 %2, %10, %18; addc.cc.u32 %3, %11, %19;\n\t"
        "addc.cc.u32 %4, %12, %20; addc.cc.u32 %5, %13, %21; addc.cc.u32 %6, %14, %22; addc.u32 %7, %15, 0;"
        : "=r"(r.l[0]), "=r"(r.l[1]), "=r"(r.l[2]), "=r"(r.l[3]), "=r"(r.l[4]), "=r"(r.l[5]), "=r"(r.l[6]), "=r"(r.l[7])
        : "r"(even[0]), "r"(even[1]), "r"(even[2]), "r"(even[3]), "r"(even[4]), "r"(even[5]), "r"(even[6]), "r"(even[7]),
          "r"(odd[1]), "r"(odd[2]), "r"(odd[3]), "r"(odd[4]), "r"(odd[5]), "r"(odd[6]), "r"(odd[7]));
    r.cond_sub_mod();
    return r;
#else
    return mul_portable(*this, *this);
#endif
  }

  // ---- conversions
  // canonical integer (little-endian limbs, must be < p) -> Montgomery form
  static H2V_HD Fp from_canonical(const Fp& c) { return mul_any(c, r2()); }
  H2V_HD Fp to_canonical() const {
    Fp o = zero();
    o.l[0] = 1;
    return mul(*this, o);
  }
  static H2V_HD Fp from_u32(u32 v) {
    Fp c = zero();
    c.l[0] = v;
    return from_canonical(c);
  }
  // 32 little-endian bytes -> raw limbs (no range check, no Montgomery conversion)
  static H2V_HD Fp load_le(const u8* b) {
    Fp r;
#pragma unroll
    for (int i = 0; i < 8; i++)
      r.l[i] = (u32)b[4 * i] | ((u32)b[4 * i + 1] << 8) | ((u32)b[4 * i + 2] << 16) | ((u32)b[4 * i + 3] << 24);
    return r;
  }
  H2V_HD void store_le(u8* b) const {
#pragma unroll
    for (int i = 0; i < 8; i++) {
      b[4 * i] = (u8)l[i];
      b[4 * i + 1] = (u8)(l[i] >> 8);
      b[4 * i + 2] = (u8)(l[i] >> 16);
      b[4 * i + 3] = (u8)(l[i] >> 24);
    }
  }
  // ff::FromUniformBytes<64>: 512-bit little-endian integer mod p, result in Montgomery form.
  // lo*R^2*R^-1 + hi*R^3*R^-1 = (lo + hi*2^256)*R  (same decomposition halo2curves uses)
  static H2V_HD Fp from_uniform(const u8* b64) {
    Fp lo = load_le(b64), hi = load_le(b64 + 32);
    return mul_any(lo, r2()) + mul_any(hi, r3());
  }

  // same from 16 little-endian words (hash digests are produced as words on the device)
  static H2V_HD Fp from_uniform_words(const u32* w16) {
    Fp lo, hi;
#pragma unroll
    for (int i = 0; i < 8; i++) {
      lo.l[i] = w16[i];
      hi.l[i] = w16[8 + i];
    }
    return mul_any(lo, r2()) + mul_any(hi, r3());
  }
  // 32 little-endian bytes -> raw limbs with 32-bit loads when the address allows
  static H2V_HD Fp load_le_fast(const u8* b) {
    if (((size_t)b & 3) != 0) return load_le(b);
    Fp r;
    const u32* w = (const u32*)b;
#pragma unroll
    for (int i = 0; i < 8; i++) r.l[i] = w[i];
    return r;
  }

  // ---- exponentiation by a 256-bit exponent given as 8 limbs: sliding window of 5 bits over a table of the
  // 16 odd powers (for (p+1)/4: 250 squarings + 38 + 16 multiplications)
  H2V_HDN Fp pow_limbs(const u32* e) const {
    Fp tab[16];
    const Fp a2 = sqr();
    tab[0] = *this;
    for (int i = 1; i < 16; i++) tab[i] = tab[i - 1] * a2;
    int i = 255;
    while (i >= 0 && !((e[i >> 5] >> (i & 31)) & 1)) i--;
    Fp acc = one();
    bool started = false;
    while (i >= 0) {
      if (!((e[i >> 5] >> (i & 31)) & 1)) {
        acc = acc.sqr();
        i--;
        continue;
      }
      int j = i >= 4 ? i - 4 : 0;
      while (!((e[j >> 5] >> (j & 31)) & 1)) j++;
      u32 val = 0;
      for (int b = i; b >= j; b--) val = (val << 1) | ((e[b >> 5] >> (b & 31)) & 1);
      if (started) {
        for (int b = j; b <= i; b++) acc = acc.sqr();
        acc = acc * tab[val >> 1];
      } else {
        acc = tab[val >> 1];
        started = true;
      }
      i = j - 1;
    }
    return acc;
  }
  // small exponent, square-and-multiply (pow_vartime call sites: vk.rs:583, domain.rs:175-179)
  H2V_HDN Fp pow_u64(u64 e) const {
    Fp acc = one(), base = *this;
    while (e) {
      if (e & 1) acc = acc * base;
      base = base.sqr();
      e >>= 1;
    }
    return acc;
  }
  // inverse by Fermat (a^(p-2)); inv(0) = 0
  H2V_HDN Fp inv() const {
    u32 e[8];
    for (int i = 0; i < 8; i++) e[i] = P::mod(i);
    e[0] -= 2;  // neither modulus has low limb < 2
    return pow_limbs(e);
  }
  // The same inverse (it is unique, so the result is bit-identical to inv()) by the binary extended Euclid in Kaliski's
  // Montgomery-inverse form: shifts, additions and subtractions on 256-bit integers instead of ~310 dependent Montgomery
  // multiplications.  On the GPU that is ~35 k ALU instructions off the multiply pipe instead of ~55 k on it, and a
  // several times shorter dependent chain: it is what bounds the latency of the scalar stage (one inversion per proof).
  // Written without data-dependent branches inside an iteration so that the lanes of a warp stay converged; the
  // iteration COUNT is data dependent (254..508, then 512 - k doublings): a warp runs as long as its slowest lane.
  //   phase 1: u = p, v = a, r = 0, s = 1; while v > 0: halve the even one of (u, v) - or the larger one minus the
  //            smaller when both are odd - and double the cofactor of the other; ends with r = -a^-1 2^k mod p
  //   phase 2: a^-1 2^k  ->  a^-1 2^512 = (aR)^-1 R^2 by 512 - k modular doublings.   inv_bin(0) = 0.
  H2V_HDN Fp inv_bin() const {
    u32 u[8], v[8], r[8], s[8];
#pragma unroll
    for (int i = 0; i < 8; i++) {
      u[i] = P::mod(i);
      v[i] = l[i];
      r[i] = 0;
      s[i] = 0;
    }
    s[0] = 1;
    if (is_zero()) return zero();
    u32 k = 0;
    for (;;) {
      u32 nz = 0;
#pragma unroll
      for (int i = 0; i < 8; i++) nz |= v[i];
      if (!nz) break;
      u32 d[8], e[8];
      sub_raw(d, u, v);
      const u32 gt = sub_raw(e, v, u);  // borrow of v - u: u > v (u == v, the last step, goes to side B: v becomes 0)
      const bool u_even = !(u[0] & 1), v_even = !(v[0] & 1);
      // side A touches (u, s doubles, r grows), side B touches (v, r doubles, s grows)
      const bool side_a = u_even || (!v_even && gt);
      const bool subtract = !u_even && !v_even;  // both odd: the larger one minus the smaller one
      u32 x[8], g[8];                            // x: the value to halve; g: cofactor sum r + s
#pragma unroll
      for (int i = 0; i < 8; i++) x[i] = side_a ? (subtract ? d[i] : u[i]) : (subtract ? e[i] : v[i]);
      add_raw(g, r, s);  // r, s <= 2p - 1 < 2^255: no carry
#pragma unroll
      for (int i = 0; i < 7; i++) x[i] = (x[i] >> 1) | (x[i + 1] << 31);
      x[7] >>= 1;
      u32 grow[8], dbl[8];  // the cofactor that takes the sum (or stays), the one that doubles
#pragma unroll
      for (int i = 0; i < 8; i++) {
        grow[i] = subtract ? g[i] : (side_a ? r[i] : s[i]);
        dbl[i] = side_a ? s[i] : r[i];
      }
#pragma unroll
      for (int i = 7; i > 0; i--) dbl[i] = (dbl[i] << 1) | (dbl[i - 1] >> 31);
      dbl[0] <<= 1;
#pragma unroll
      for (int i = 0; i < 8; i++) {
        if (side_a) {
          u[i] = x[i];
          r[i] = grow[i];
          s[i] = dbl[i];
        } else {
          v[i] = x[i];
          s[i] = grow[i];
          r[i] = dbl[i];
        }
      }
      k++;
    }
    Fp m, out;
#pragma unroll
    for (int i = 0; i < 8; i++) {
      m.l[i] = P::mod(i);
      out.l[i] = r[i];
    }
    out.cond_sub_mod();                 // r < 2p
    sub_raw(out.l, m.l, out.l);         // a^-1 2^k = p - r   (r != 0 since gcd(a, p) = 1)
    for (u32 i = k; i < 512; i++) out = out.dbl();
    return out;
  }
};

typedef Fp<FqP> Fq;
typedef Fp<FrP> Fr;

// Fq square root candidate a^((p+1)/4) (p = 3 mod 4); caller checks candidate^2 == a.
H2V_HDN inline Fq fq_sqrt_candidate(const Fq& a) {
  const u32 e[8] = {0xb61f3f52u, 0x4f082305u, 0x5a1c72a3u, 0x65e05aa4u, 0xa0605617u, 0x6e14116du, 0xb84c680au, 0x0c19139cu};
  return a.pow_limbs(e);
}

}  // namespace h2v
