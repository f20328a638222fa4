// Host build of the grouped mixed-batch mapping (csrc/mix.cuh): the (group, member) segment table, the term lookups the MSM
// kernels make through it, and the write phase of the ragged-group coefficient scan (tests only; never shipped).
#include <vector>
#include "mix.cuh"
using namespace h2v;

static void shapes(u32 members, const u32* shape, std::vector<u32>& P, std::vector<u32>& M, std::vector<u32>& S) {
  P.resize(members);
  M.resize(members);
  S.resize(members);
  for (u32 m = 0; m < members; m++) {
    P[m] = shape[3 * m];
    M[m] = shape[3 * m + 1];
    S[m] = shape[3 * m + 2];
  }
}

extern "C" {
// Segment table of a grouped batch (counts[q * members + m], shape[3 m ..] = P, n_mo, Sh, set_of[m] among `sets`) and where every
// term goes through the kernels' lookups: out[7 t ..] = group, member, kind, proof (index in the member's arrays), index, bucket
// set, point (element offset into the member's points for kinds 0 / 1, into its shared bases for kind 2).  Returns the number of
// terms (-1 when it exceeds `capacity`).
long long x_groups_map(u32 groups, u32 members, const u32* counts, const u32* shape, const u32* set_of, u32 sets, u32* out,
                       unsigned long long capacity) {
  std::vector<u32> P, M, S;
  shapes(members, shape, P, M, S);
  std::vector<MixSeg> seg((size_t)groups * members);
  unsigned long long total = 0;
  mix_layout_groups(groups, members, counts, P.data(), M.data(), S.data(), set_of, sets, 0, seg.data(), &total);
  if (total > capacity) return -1;
  static G1Affine base[1];  // the points' and shared bases' addresses: offsets from here
  for (MixSeg& s : seg) s.pts = s.shared_pts = base;
  const u32 nseg = (u32)seg.size();
  for (u32 t = 0; t < total; t++) {
    const u32 k = mix_segment(seg.data(), nseg, t);
    const MixSeg& sg = seg[k];
    const MixTerm mt = mix_term(sg, t - sg.t0);
    const u32 row[7] = {k / members, k % members, mt.kind, mt.kind == 2 ? 0u : sg.j0 + mt.j, mt.i, sg.cls, (u32)(&mix_point(sg, mt) - base)};
    for (int q = 0; q < 7; q++) out[7 * (size_t)t + q] = row[q];
  }
  return (long long)total;
}

// One group against mix_layout (shape[4 m ..] = n, P, n_mo, Sh; set_of as above): terms whose segment member, kind, proof,
// index, bucket set or point differ, or -1 when the term counts differ
long long x_groups_vs_layout(u32 members, const u32* shape, const u32* set_of, u32 sets) {
  std::vector<u32> n(members), P(members), M(members), S(members), member_of(members + 1);
  for (u32 m = 0; m < members; m++) {
    n[m] = shape[4 * m];
    P[m] = shape[4 * m + 1];
    M[m] = shape[4 * m + 2];
    S[m] = shape[4 * m + 3];
  }
  std::vector<MixSeg> a(members + 1), b(members);
  unsigned long long ta = 0, tb = 0;
  const u32 na = mix_layout(members, n.data(), P.data(), M.data(), S.data(), a.data(), member_of.data(), &ta, set_of);
  mix_layout_groups(1, members, n.data(), P.data(), M.data(), S.data(), set_of, sets, 0, b.data(), &tb);
  if (ta != tb) return -1;
  static G1Affine base[1];
  for (MixSeg& s : a) s.pts = s.shared_pts = base;
  for (MixSeg& s : b) s.pts = s.shared_pts = base;
  long long bad = 0;
  for (u32 t = 0; t < ta; t++) {
    const u32 ka = mix_segment(a.data(), na, t), kb = mix_segment(b.data(), members, t);
    const MixTerm x = mix_term(a[ka], t - a[ka].t0), y = mix_term(b[kb], t - b[kb].t0);
    bad += member_of[ka] != kb || x.kind != y.kind || x.j != y.j || x.i != y.i || a[ka].cls != b[kb].cls ||
           &mix_point(a[ka], x) != &mix_point(b[kb], y) || a[ka].call0 + x.j != b[kb].call0 + y.j;
  }
  return bad;
}

// The ragged-group coefficient scan of k_rlc_scan_groups on the host: the same per-thread chunks of `threads` lanes, suffix
// products of the chunks, and mix_scan_chunk for every chunk.  r: N canonical little-endian scalars in call order; coef: the
// members' arrays one after the other (member m's totals, in member order), canonical little-endian out.
void x_rlc_scan_groups(u32 groups, u32 members, const u32* counts, const u8* r_bytes, u32 threads, u8* coef_bytes) {
  std::vector<u32> zero(members, 0);
  std::vector<MixSeg> seg((size_t)groups * members);
  unsigned long long total = 0, N = 0;
  std::vector<u32> set(members, 0);
  mix_layout_groups(groups, members, counts, zero.data(), zero.data(), zero.data(), set.data(), 1, 0, seg.data(), &total);
  for (u32 i = 0; i < groups * members; i++) N += counts[i];
  std::vector<Fr> r(N), coef;
  for (unsigned long long i = 0; i < N; i++) r[i] = Fr::from_canonical(Fr::load_le(r_bytes + 32 * i));
  std::vector<size_t> base(members, 0);
  size_t all = 0;
  for (u32 m = 0; m < members; m++) {
    base[m] = all;
    all += seg[m].stride;
  }
  coef.assign(all, Fr::zero());
  for (u32 i = 0; i < groups * members; i++) seg[i].coef = coef.data() + base[i % members];
  unsigned long long g0 = 0;
  for (u32 q = 0; q < groups; q++) {
    unsigned long long count = 0;
    for (u32 m = 0; m < members; m++) count += counts[(size_t)q * members + m];
    const unsigned long long per = (count + threads - 1) / threads;
    std::vector<Fr> suffix(threads + 1, Fr::one());
    std::vector<unsigned long long> lo(threads), hi(threads);
    for (u32 t = 0; t < threads; t++) {
      lo[t] = (unsigned long long)t * per < count ? g0 + (unsigned long long)t * per : g0 + count;
      hi[t] = lo[t] + per < g0 + count ? lo[t] + per : g0 + count;
    }
    for (u32 t = threads; t-- > 0;) {
      Fr p = Fr::one();
      for (unsigned long long i = lo[t]; i < hi[t]; i++) p = p * r[i];
      suffix[t] = p * suffix[t + 1];
    }
    for (u32 t = 0; t < threads; t++) mix_scan_chunk(r.data(), lo[t], hi[t], suffix[t + 1], seg.data() + (size_t)q * members, members);
    g0 += count;
  }
  for (size_t i = 0; i < all; i++) coef[i].to_canonical().store_le(coef_bytes + 32 * i);
}
}
