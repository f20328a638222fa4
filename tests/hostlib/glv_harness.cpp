// Host build of the lifted GLV digits (glv.cuh), for CPU-side unit tests (tests only; never shipped).  Compiled by
// tests/test_glv_lift.py into a temporary directory.
#include "glv.cuh"
using namespace h2v;
extern "C" {
// lifted GLV halves of term t at window bits c, W windows (k_msm_digits): out12 = a (5 limbs), b (5 limbs), Z, Z'
void t_glv_lift_term(const u32* k, u32 t, u32 c, u32 W, u32* out12) {
  u32 Z, Z2;
  glv_lift_ranges(c, W, Z, Z2);
  out12[10] = Z;
  out12[11] = Z2;
  if (Z2) glv_lift_term(k, t, Z, Z2, out12, out12 + 5);
}
}
