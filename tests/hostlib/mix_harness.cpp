// Host build of the MSM term mapping (csrc/mix.cuh), for CPU-side unit tests (tests only; never shipped).
#include <vector>
#include "mix.cuh"
using namespace h2v;
extern "C" {
// Segment table of `members` members (shape[4 m ..] = n, P, n_mo, Sh) and where every term of it goes, through the
// lookups the kernels use: out[6 t ..] = segment, member, kind, proof, index, channel.  Returns the number of terms (-1
// when it exceeds `capacity`); *nseg = segments.
long long x_map(u32 members, const u32* shape, u32* out, unsigned long long capacity, u32* nseg) {
  std::vector<u32> n(members), P(members), M(members), S(members), member_of(members + 1);
  for (u32 m = 0; m < members; m++) {
    n[m] = shape[4 * m];
    P[m] = shape[4 * m + 1];
    M[m] = shape[4 * m + 2];
    S[m] = shape[4 * m + 3];
  }
  std::vector<MixSeg> seg(members + 1);
  unsigned long long total = 0;
  *nseg = mix_layout(members, n.data(), P.data(), M.data(), S.data(), seg.data(), member_of.data(), &total);
  if (total > capacity) return -1;
  for (u32 t = 0; t < total; t++) {
    const u32 s = mix_segment(seg.data(), *nseg, t);
    const MixTerm mt = mix_term(seg[s], t - seg[s].t0);
    const u32 row[6] = {s, member_of[s], mt.kind, mt.j, mt.i, mix_channel(mt)};
    for (int q = 0; q < 6; q++) out[6 * (size_t)t + q] = row[q];
  }
  return (long long)total;
}
// One segment of shape (n, P, n_mo, Sh) against the single-VK mapping of one fold group (msm_point, channel_of_term):
// number of terms whose point or channel differ
long long x_single_mismatches(u32 n, u32 P, u32 n_mo, u32 Sh) {
  std::vector<G1Affine> pts((size_t)n * P), shared(Sh);
  MixSeg seg;
  MsmGeom g{};
  g.n = n;
  g.P = P;
  g.n_mo = n_mo;
  g.Sh = Sh;
  g.G = 1;
  g.N = n;
  g.T = n * P + n * n_mo + Sh;
  u32 member = 0;
  unsigned long long total = 0;
  if (mix_layout(1, &n, &P, &n_mo, &Sh, &seg, &member, &total) != 1 || total != g.T) return -1;
  seg.pts = pts.data();
  seg.shared_pts = shared.data();
  long long bad = 0;
  for (u32 t = 0; t < g.T; t++) {
    const MixTerm mt = mix_term(seg, t - seg.t0);
    bad += mix_segment(&seg, 1, t) != 0 || &mix_point(seg, mt) != &msm_point(g, t, pts.data(), shared.data()) ||
           mix_channel(mt) != g.channel_of_term(t);
  }
  return bad;
}
}
