// Persistent accumulators (include/h2v.h "persistent accumulators"): the arithmetic of one absorb,
//   (L_b, R_b) = sum_w 2^(c w) S_w  per channel,   acc <- s_b acc + (L_b, R_b),
// written as ITEMS that k_acc_absorb runs side by side: item (channel, w) = [2^(c w) mod r] S_w, and one item per channel
// [s_b] acc.  Every item is a GLV multiplication on four lanes (glv.cuh, Jacobian base), so no chain is longer than 129
// doublings, where the Horner combination of k_fold_accum walks c W ~ 264 dependent doublings.  The items of a channel are
// then added with a tree.  Host-device: tests/hostlib/acc_harness.cpp checks this file against the oracle.
#pragma once
#include "glv.cuh"

namespace h2v {

// window geometry of the sums being absorbed: W[ch] window sums of c[ch] bits, channel 0 = right (R), 1 = left (L)
struct AccGeom {
  u32 W[2], c[2];
};
static constexpr u32 ACC_MAX_ITEMS = 136;  // >= 128 (channel, window) pairs (ensure_lines bounds a geometry) + 2
static constexpr u32 ACC_TREE_SPAN = 64;   // >= the windows of one channel (c >= 4: W <= 64)

H2V_HD u32 acc_items(const AccGeom& g) { return g.W[0] + g.W[1] + 2; }

// 2^(c w) mod r, canonical
H2V_HD Fr acc_window_weight(u32 c, u32 w) {
  Fr x = Fr::one();
  for (u32 i = 0; i < c * w; i++) x = x.dbl();
  return x.to_canonical();
}

// base and canonical scalar of item i: window sums first (wsums[W0 + W1], right channel first), then acc[0..2) scaled by s
H2V_HD void acc_item(const AccGeom& g, u32 i, const G1Jac* wsums, const G1Jac* acc, const Fr& s, G1Jac& base, Fr& k) {
  const u32 nw = g.W[0] + g.W[1];
  if (i < nw) {
    const u32 ch = i >= g.W[0] ? 1u : 0u;
    base = wsums[i];
    k = acc_window_weight(g.c[ch], i - (ch ? g.W[0] : 0u));
  } else {
    base = acc[i - nw];
    k = s;
  }
}

// lane q (0..3) of [k] P: the four lanes' results add up to [k] P
H2V_HDN inline G1Jac acc_mul_lane(const G1Jac& p, const Fr& k, u32 q) {
  GlvHalf h1, h2;
  glv_decompose(k.l, h1, h2);
  const bool endo = (q & 1) != 0, top = (q >> 1) != 0;
  return g1_mul_glv_part(p, endo ? h2 : h1, endo, top ? 64u : 0u, top ? 65u : 64u, top ? 64u : 0u);
}

// one level (span d = 32, 16, .., 1) of the tree over the window items of both channels: thread t < 2 * ACC_TREE_SPAN adds
// item i + d of channel t / ACC_TREE_SPAN onto item i.  A level writes items [0, d) and reads [d, 2d) of a channel.
H2V_HD void acc_tree_step(const AccGeom& g, G1Jac* items, u32 t, u32 d) {
  const u32 ch = t / ACC_TREE_SPAN, i = t % ACC_TREE_SPAN;
  if (ch > 1 || i >= d || i + d >= g.W[ch]) return;
  G1Jac* v = items + (ch ? g.W[0] : 0u);
  v[i] = g1_add(v[i], v[i + d]);
}

// after the tree: (L_b, R_b) of channel ch, and its new accumulator s acc + (L_b, R_b)
H2V_HD G1Jac acc_batch_sum(const AccGeom& g, const G1Jac* items, u32 ch) { return items[ch ? g.W[0] : 0u]; }
H2V_HD G1Jac acc_new_value(const AccGeom& g, const G1Jac* items, u32 ch) {
  return g1_add(items[g.W[0] + g.W[1] + ch], acc_batch_sum(g, items, ch));
}

}  // namespace h2v
