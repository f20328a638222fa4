// Host build of the absorb arithmetic (csrc/acc.cuh), for CPU-side unit tests (tests only; never shipped).
// Points cross the boundary as 16 canonical limbs x | y (all zero = identity); `z` (canonical Fq, non-zero) picks the
// Jacobian representative (x z^2, y z^3, z) of every input point, so that the Jacobian-base code is exercised.
#include <string.h>
#include <vector>
#include "acc.cuh"
using namespace h2v;

static G1Jac load(const u32* xy, const u32* z) {
  bool zero = true;
  for (int i = 0; i < 16; i++) zero &= xy[i] == 0;
  if (zero) return G1Jac::identity();
  Fq x, y, zz;
  memcpy(x.l, xy, 32);
  memcpy(y.l, xy + 8, 32);
  memcpy(zz.l, z, 32);
  x = Fq::from_canonical(x);
  y = Fq::from_canonical(y);
  zz = Fq::from_canonical(zz);
  const Fq z2 = zz * zz;
  G1Jac r;
  r.X = x * z2;
  r.Y = y * z2 * zz;
  r.Z = zz;
  return r;
}
static void store(const G1Jac& p, u32* out) {
  G1Affine a;
  if (!g1_to_affine(p, a)) {
    memset(out, 0, 64);
    return;
  }
  const Fq x = a.x.to_canonical(), y = a.y.to_canonical();
  memcpy(out, x.l, 32);
  memcpy(out + 8, y.l, 32);
}
static Fr scalar(const u32* k) {
  Fr s;
  memcpy(s.l, k, 32);
  return s;
}

extern "C" {
void x_weight(u32 c, u32 w, u32* out8) { memcpy(out8, acc_window_weight(c, w).l, 32); }

// [k] P as the sum of the four GLV lanes of k_acc_absorb, Jacobian base
void x_mul_jac(const u32* pxy, const u32* z, const u32* k, u32* out) {
  const G1Jac p = load(pxy, z);
  G1Jac r = G1Jac::identity();
  for (u32 q = 0; q < 4; q++) r = g1_add(r, acc_mul_lane(p, scalar(k), q));
  store(r, out);
}

// One absorb as k_acc_absorb computes it, lanes and threads run as loops: wsums[(W0 + W1) x 16] (right channel first),
// acc[2 x 16] = (R, L), s canonical -> record[2 x 16] = (R_b, L_b) and acc_out[2 x 16] = s acc + (R_b, L_b).  Returns -1 for a
// geometry the kernel does not take.
int x_absorb(u32 c0, u32 W0, u32 c1, u32 W1, const u32* wsums, const u32* acc, const u32* s, const u32* z, u32* record, u32* acc_out) {
  const AccGeom g{{W0, W1}, {c0, c1}};
  if (acc_items(g) > ACC_MAX_ITEMS || W0 > ACC_TREE_SPAN || W1 > ACC_TREE_SPAN) return -1;
  std::vector<G1Jac> ws(W0 + W1), items(acc_items(g));
  G1Jac a[2] = {load(acc, z), load(acc + 16, z)};
  for (u32 i = 0; i < W0 + W1; i++) ws[i] = load(wsums + 16 * i, z);
  for (u32 it = 0; it < acc_items(g); it++) {
    G1Jac base, lane[4];
    Fr k;
    acc_item(g, it, ws.data(), a, scalar(s), base, k);
    for (u32 q = 0; q < 4; q++) lane[q] = acc_mul_lane(base, k, q);
    for (u32 q = 0; q < 2; q++) lane[q] = g1_add(lane[q], lane[q + 2]);  // the shuffles: down 2, then down 1
    items[it] = g1_add(lane[0], lane[1]);
  }
  for (u32 d = ACC_TREE_SPAN / 2; d > 0; d >>= 1)
    for (u32 t = 0; t < 4 * ACC_MAX_ITEMS; t++) acc_tree_step(g, items.data(), t, d);
  for (u32 ch = 0; ch < 2; ch++) {
    store(acc_batch_sum(g, items.data(), ch), record + 16 * ch);
    store(acc_new_value(g, items.data(), ch), acc_out + 16 * ch);
  }
  return 0;
}

// the Horner combination sum_w 2^(c w) S_w of k_fold_accum (serial doublings), for comparison
void x_horner(u32 c, u32 W, const u32* wsums, const u32* z, u32* out) {
  G1Jac acc = G1Jac::identity();
  for (u32 w = W; w-- > 0;) {
    for (u32 i = 0; i < c; i++) acc = g1_double(acc);
    acc = g1_add(acc, load(wsums + 16 * w, z));
  }
  store(acc, out);
}
}
