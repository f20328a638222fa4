// Aggregation proofs (include/h2v.h "aggregation proofs"): decoding of the KZG accumulator (lhs, rhs) that an aggregation
// circuit carries in its public instances, snark-verifier's LimbsEncoding<LIMBS, BITS>.  Every coordinate is `limbs`
// instance values, least significant limb first, x = sum_i limb_i 2^(bits i); the cells are ordered lhs.x, lhs.y, rhs.x,
// rhs.y.  A valid encoding has every limb < 2^bits, every coordinate < q, and both points on y^2 = x^3 + 3 or (0, 0), the
// identity (halo2curves from_xy).  Host-device: tests/hostlib/agg_harness.cpp checks this file against the oracle.
#pragma once
#include "curve.cuh"

namespace h2v {

static constexpr u32 AGG_MIN_LIMBS = 2, AGG_MAX_LIMBS = 8, AGG_MAX_BITS = 128;

struct AggCell {
  u32 column, row;  // column of the proof's flattened (instance-major) instance columns, row inside it
};

// One coordinate from `limbs` instance values (32-byte little-endian, least significant limb first) -> canonical Fq limbs.
// false: a limb >= 2^bits, or the coordinate >= q.
H2V_HD bool agg_coord(const u8* const* limb, u32 limbs, u32 bits, Fq& out) {
  u32 w[33];  // limbs * bits <= 1024
  for (u32 i = 0; i < 33; i++) w[i] = 0;
  bool ok = true;
  for (u32 i = 0; i < limbs; i++) {
    for (u32 k = 0; k < 32; k++) {
      const u32 b = limb[i][k];
      const u32 lo = 8 * k;
      const u32 allowed = lo + 8 <= bits ? 0xFFu : lo >= bits ? 0u : (1u << (bits - lo)) - 1u;
      if (b & ~allowed) ok = false;
      const u32 pos = bits * i + lo;
      if (!b || pos >= 32 * 33) continue;
      w[pos >> 5] |= b << (pos & 31);
      if ((pos & 31) > 24 && (pos >> 5) + 1 < 33) w[(pos >> 5) + 1] |= b >> (32 - (pos & 31));
    }
  }
  for (u32 i = 8; i < 33; i++)
    if (w[i]) ok = false;
  for (u32 i = 0; i < 8; i++) out.l[i] = w[i];
  if (out.geq_mod()) ok = false;
  return ok;
}

// One point from 2 * limbs values (x limbs, then y limbs) -> Montgomery affine, *is_id = the identity (0, 0).
// false: a coordinate fails agg_coord, or the point is off the curve.
H2V_HD bool agg_point(const u8* const* limb, u32 limbs, u32 bits, G1Affine& p, bool* is_id) {
  Fq x, y;
  const bool ok = agg_coord(limb, limbs, bits, x) & agg_coord(limb + limbs, limbs, bits, y);
  *is_id = ok && x.is_zero() && y.is_zero();
  p.x = Fq::from_canonical(x);
  p.y = Fq::from_canonical(y);
  if (!ok) return false;
  return *is_id || g1_on_curve(p);
}

}  // namespace h2v
