// Host build of the multi-params mix mapping (csrc/mix.cuh): segment -> params class -> bucket set, and the pair budget of
// the one pairing check (tests only; never shipped).
#include <vector>
#include "mix.cuh"
using namespace h2v;
extern "C" {
// Segment table of `members` members (shape[4 m ..] = n, P, n_mo, Sh) whose member m is in bucket set set_of[m] (null: every
// member in set 0), under the window geometry (c0, c1) with `sets` bucket sets, and where every (term, window) goes through
// the lookups the kernels use: out[5 t ..] = segment, member, set, first bucket, last bucket of the term (digit magnitudes
// 1 .. B of every window of its channel).  Returns the number of terms (-1 when it exceeds `capacity`); *nb = buckets per set.
long long x_class_map(u32 members, const u32* shape, const u32* set_of, u32 sets, u32 c0, u32 c1, u32* out, unsigned long long capacity, u32* nb) {
  std::vector<u32> n(members), P(members), M(members), S(members), member_of(members + 1);
  for (u32 m = 0; m < members; m++) {
    n[m] = shape[4 * m];
    P[m] = shape[4 * m + 1];
    M[m] = shape[4 * m + 2];
    S[m] = shape[4 * m + 3];
  }
  std::vector<MixSeg> seg(members + 1);
  unsigned long long total = 0;
  const u32 nseg = mix_layout(members, n.data(), P.data(), M.data(), S.data(), seg.data(), member_of.data(), &total, set_of);
  if (total > capacity) return -1;
  MsmGeom g{};
  g.G = sets;
  g.T = (u32)total;
  g.c[0] = c0;
  g.c[1] = c1;
  for (int ch = 0; ch < 2; ch++) {
    g.W[ch] = (255 + g.c[ch] - 1) / g.c[ch];
    g.B[ch] = 1u << (g.c[ch] - 1);
  }
  g.wbase[1] = g.W[0];
  g.bbase[1] = g.W[0] * g.B[0];
  *nb = g.nb();
  for (u32 t = 0; t < total; t++) {
    const MixSeg& sg = seg[mix_segment(seg.data(), nseg, t)];
    const u32 ch = mix_channel(mix_term(sg, t - sg.t0));
    const u32 row[5] = {mix_segment(seg.data(), nseg, t), member_of[mix_segment(seg.data(), nseg, t)], sg.cls, msm_bucket(g, sg.cls, ch, 0, 1),
                        msm_bucket(g, sg.cls, ch, g.W[ch] - 1, g.B[ch])};
    for (int q = 0; q < 5; q++) out[5 * (size_t)t + q] = row[q];
  }
  return (long long)total;
}
u32 x_mix_line_run(u32 sets, u32 W0, u32 W1, u32 run0) { return mix_line_run(sets, W0, W1, run0); }
}
