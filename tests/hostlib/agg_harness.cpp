// Host build of the carried-accumulator decoding (csrc/agg.cuh), for CPU-side unit tests (tests only; never shipped).
#include <string.h>
#include "agg.cuh"
using namespace h2v;

extern "C" {
// values: 4 * limbs instance values of 32 bytes (lhs.x, lhs.y, rhs.x, rhs.y limbs, least significant first).  Returns 1 when
// both points decode, 0 otherwise; out[128] = canonical lhs.x | lhs.y | rhs.x | rhs.y (valid when 1 is returned), ids[2] =
// identity flags.
int x_agg_decode(u32 limbs, u32 bits, const u8* values, u8* out, u8* ids) {
  if (limbs < AGG_MIN_LIMBS || limbs > AGG_MAX_LIMBS) return -1;
  const u8* limb[4 * AGG_MAX_LIMBS];
  for (u32 i = 0; i < 4 * limbs; i++) limb[i] = values + 32 * i;
  int ok = 1;
  for (u32 q = 0; q < 2; q++) {
    G1Affine p;
    bool id = false;
    if (!agg_point(limb + 2 * limbs * q, limbs, bits, p, &id)) ok = 0;
    ids[q] = id ? 1 : 0;
    p.x.to_canonical().store_le(out + 64 * q);
    p.y.to_canonical().store_le(out + 64 * q + 32);
  }
  return ok;
}
}
