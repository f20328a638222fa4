// Term spaces of the bucket MSM.  k_msm_digits, k_msm_scatter and k_msm_bucket_sum are the only kernels that map a term
// id to its scalar, its point and its channel; everything after them sees digits and bucket ids only.  Two sources:
//   single VK   (MsmGeom, msm_point): G fold groups of one plan, each n*P right-channel proof terms, n*n_mo left-channel
//               terms, Sh shared-base terms
//   mixed batch (MixSeg table): one segment per (group, member) of a grouped mix (mix_layout_groups; a plain mix is one
//               group), consecutive in term-id space; inside a segment the terms keep the single-VK order of one fold group,
//               over a window [j0, j0 + n) of the member's own arrays (per-proof stride = the member's upload).  A
//               one-segment table therefore maps every term exactly as msm_point / channel_of_term do.  The MsmGeom of a mix
//               has T = every term of the mix and G = bucket sets: groups x (params classes with proofs in the call); the
//               terms of segment (q, m) go to bucket set q * S + (set of m's class) (MixSeg::cls).
// Compiles on the host too (tests/hostlib/mix_harness.cpp checks the mapping without a GPU).
#pragma once
#include "curve.cuh"

#if defined(__CUDACC__)
#define H2V_HOST_DEVICE __host__ __device__
#else
#define H2V_HOST_DEVICE
#endif

namespace h2v {

// Fold groups: the N = G * n proofs of an upload may be G consecutive independent batches of n proofs (own fold
// coefficients, own MSM, own pairing check, own verdict) that share every kernel launch: the per-proof kernels run
// over all N proofs, the MSM kernels over G * T terms and G * nb() buckets, the pairing kernels over G blocks.
// Everything in MsmGeom is PER GROUP except G and N (the stride of the per-proof arrays).
struct MsmGeom {
  u32 n, P, n_mo, Sh;  // shape of one fold group
  u32 G, N;            // fold groups, proofs of the upload (G * n)
  u32 T;               // terms of one group = n*P (right) + n*n_mo (left) + Sh (right, shared bases)
  // per channel (0 = right, 1 = left): window bits, windows, buckets per window (2^(c-1)),
  // first global window index, first global bucket index
  u32 c[2], W[2], B[2], wbase[2], bbase[2];
  u32 Z[2];  // scalar lift range: k'' = k + z*r, z in [0, Z), keeps every window (also the top one) uniformly filled
  u32 Wmax;  // row stride of the digit table
  u32 m;     // buckets per reduction chunk
  u32 glv;   // 1: every term is split into its two GLV halves (glv.cuh), rows / entries 2 t + half; windows cover 130 bits or more
             // (the attribution sub-batches: half the windows -> half the doublings of their explicit window combination)
  u32 Z2[2]; // lattice-lift range z' of a lifted GLV geometry (glv_lift), 0 = halves unlifted (attribution).  A lifted geometry
             // reads phi(P) from the phi rows that follow the points (phi_rows)
  H2V_HOST_DEVICE bool lifted() const { return glv && Z2[0]; }
  H2V_HOST_DEVICE u32 nb() const { return W[0] * B[0] + W[1] * B[1]; }
  H2V_HOST_DEVICE u32 channel_of_term(u32 tl) const { return (tl >= n * P && tl < n * P + n * n_mo) ? 1u : 0u; }  // tl = term inside its group
};

H2V_HD const G1Affine& msm_point(const MsmGeom& g, u32 t, const G1Affine* pts, const G1Affine* shared_pts) {
  const u32 grp = t / g.T, tl = t % g.T;
  const u32 nP = g.n * g.P;
  if (tl < nP) return pts[(size_t)(tl / g.n) * g.N + grp * g.n + tl % g.n];
  const u32 nL = g.n * g.n_mo;
  if (tl < nP + nL) {
    const u32 q = (tl - nP) / g.n, jl = (tl - nP) % g.n;
    return pts[(size_t)(g.P - g.n_mo + q) * g.N + grp * g.n + jl];  // (mo_slot + q) * N + j
  }
  return shared_pts[tl - nP - nL];
}

// ---- mixed batches (h2v_mix): members of different verifying keys in one MSM
static constexpr u32 MIX_MAX_MEMBERS = 64;

// The proofs of one member in one group: proofs [j0, j0 + n) of the member's upload (its arrays have per-proof stride
// `stride`), call indices [call0, call0 + n) of the fold randomness.  Sh = the member's shared bases when it has proofs
// anywhere in the call (a group without its proofs still carries them, with zero scalars), 0 otherwise.
struct MixSeg {
  u32 t0, T;            // first term id, terms (n*P + n*n_mo + Sh)
  u32 n, P, n_mo, Sh;   // the segment's proofs and the member's plan shape
  u32 cls;              // bucket set: group * sets + set of the member's params class
  u32 j0, stride;       // first proof of the segment in the member's arrays, proofs of the member's upload
  u32 call0;            // call index of the segment's first proof (r_i, c_i)
  const Fr* right;      // [P][stride]     right-channel scalars of the proof points
  const Fr* left;       // [n_mo][stride]  left-channel scalars of the multi-open points
  const Fr* shared;     // [Sh][stride]    per-proof shared-base scalars
  Fr* coef;             // [stride]        fold coefficients c_j of the member's proofs (k_rlc_scan_groups)
  Fr* shared_sum;       // [Sh]            sum over the segment of c_j * shared scalar, canonical (k_shared_reduce_seg)
  const G1Affine* pts;  // [P][stride]     decompressed proof points
  const G1Affine* shared_pts;  // [Sh] fixed | sigma | G of the member's plan
};

// Term source of the MSM kernels (a template parameter): the kernels' own MsmGeom arguments, or a segment table.
struct SingleVkTerms {
  static constexpr bool mixed = false;
};
struct MixTerms {
  static constexpr bool mixed = true;
  const MixSeg* seg;
  u32 count;  // groups * members (empty segments included)
};

// Segment table of `members` members with n[m] proofs each (members without proofs get no segment): t0 / T / shape / cls
// fields of seg[0 .. return value), member_of[s] = member of segment s; *total = terms of all segments.  set[m] = bucket set
// of member m (null: every segment in set 0).
inline u32 mix_layout(u32 members, const u32* n, const u32* P, const u32* n_mo, const u32* Sh, MixSeg* seg, u32* member_of, unsigned long long* total,
                      const u32* set = nullptr) {
  u32 count = 0, calls = 0;
  unsigned long long t = 0;
  for (u32 m = 0; m < members; m++) {
    if (!n[m]) continue;
    MixSeg s{};
    s.t0 = (u32)t;
    s.n = n[m];
    s.P = P[m];
    s.n_mo = n_mo[m];
    s.Sh = Sh[m];
    s.cls = set ? set[m] : 0;
    s.stride = s.n;
    s.call0 = calls;
    calls += s.n;
    s.T = s.n * s.P + s.n * s.n_mo + s.Sh;
    t += s.T;
    member_of[count] = m;
    seg[count++] = s;
  }
  *total = t;
  return count;
}

// Grouped mixed batches (h2v_mix_verify_groups): groups x members segments, group-major, empty ones included (seg[q * members
// + m] = member m's counts[q * members + m] proofs of group q).  The call order is group-major, member-major inside a group,
// starting at call index call_base; a member's upload holds its proofs of every group in group order.  Members with proofs
// anywhere in the call (sum over q > 0) carry their Sh shared bases in every group, so the term count, and every launch
// shape, depends on the members' totals and `groups` only, never on the split.  set[m] = bucket set of member m's class
// among `sets` (read for members with proofs only).  *total = terms of all segments.  groups = 1 maps every term as
// mix_layout does.
inline void mix_layout_groups(u32 groups, u32 members, const u32* counts, const u32* P, const u32* n_mo, const u32* Sh, const u32* set, u32 sets,
                              unsigned long long call_base, MixSeg* seg, unsigned long long* total) {
  unsigned long long t = 0, call = call_base;
  for (u32 m = 0; m < members; m++) {  // j0 of group 0 and the member's total (stride)
    u32 sum = 0;
    for (u32 q = 0; q < groups; q++) sum += counts[(size_t)q * members + m];
    for (u32 q = 0; q < groups; q++) seg[(size_t)q * members + m].stride = sum;
  }
  for (u32 q = 0; q < groups; q++)
    for (u32 m = 0; m < members; m++) {
      MixSeg& s = seg[(size_t)q * members + m];
      const u32 stride = s.stride;
      s = MixSeg{};
      s.stride = stride;
      s.j0 = q ? seg[(size_t)(q - 1) * members + m].j0 + seg[(size_t)(q - 1) * members + m].n : 0;
      s.n = counts[(size_t)q * members + m];
      s.P = P[m];
      s.n_mo = n_mo[m];
      s.Sh = stride ? Sh[m] : 0;
      s.cls = stride ? q * sets + set[m] : q * sets;
      s.call0 = (u32)call;
      s.t0 = (u32)t;
      s.T = s.n * s.P + s.n * s.n_mo + s.Sh;
      t += s.T;
      call += s.n;
    }
  *total = t;
}

// Write phase of the ragged-group coefficient scan (k_rlc_scan_groups) for one thread's chunk [lo, hi) of group q's call
// indices: run = product of the group's r_i above hi; c_i = run * (r_i' for i < i' < hi) goes to [j0 + i - call0] of the
// member array of the segment holding i (seg = group q's `members` segments, call0 ascending; an index no segment holds, in
// a shard the other ranks' proofs, is scanned but not written).
H2V_HD void mix_scan_chunk(const Fr* r, unsigned long long lo, unsigned long long hi, Fr run, const MixSeg* seg, u32 members) {
  u32 k = 0;  // the last segment with call0 <= i: found once, then walked down as i falls
  if (hi > lo)
    while (k + 1 < members && seg[k + 1].call0 <= hi - 1) k++;
  for (unsigned long long i = hi; i-- > lo;) {
    while (k > 0 && seg[k].call0 > i) k--;
    const MixSeg& s = seg[k];
    if (i >= s.call0 && i < (unsigned long long)s.call0 + s.n) s.coef[s.j0 + (i - s.call0)] = run;
    run = run * r[i];
  }
}

// Sharded mixed batches: a rank owns proofs [base, base + n) of the member-major concatenation of global_counts[members]
// proofs.  local[m] = how many of them belong to member m (a range may start or end inside a member).  False when the range
// is empty or runs past the global batch.
inline bool mix_shard_counts(u32 members, const u32* global_counts, unsigned long long base, u32 n, u32* local) {
  unsigned long long N = 0, lo = 0;
  for (u32 m = 0; m < members; m++) N += global_counts[m];
  if (n == 0 || base + n > N) return false;
  const unsigned long long hi = base + n;
  for (u32 m = 0; m < members; m++) {
    const unsigned long long a = lo, b = lo + global_counts[m];  // member m's global range [a, b)
    const unsigned long long s = a > base ? a : base, e = b < hi ? b : hi;
    local[m] = e > s ? (u32)(e - s) : 0u;
    lo = b;
  }
  return true;
}

// Term counts per channel from which every rank of a sharded mix chooses its window geometry: a bound that depends only on
// what all ranks share (the member shapes, global_counts and the largest shard max_shard), never on the rank's own member
// composition.  right >= sum of n_m P_m + Sh_m over any rank's members with proofs (n_m summing to <= max_shard), left likewise.
inline void mix_shard_bound(u32 members, const u32* P, const u32* n_mo, const u32* Sh, const u32* global_counts, u32 max_shard,
                            unsigned long long* right, unsigned long long* left) {
  u32 maxP = 0, maxM = 0;
  unsigned long long shared = 0;
  for (u32 m = 0; m < members; m++) {
    if (P[m] > maxP) maxP = P[m];
    if (n_mo[m] > maxM) maxM = n_mo[m];
    if (global_counts[m]) shared += Sh[m];
  }
  *right = (unsigned long long)max_shard * maxP + shared;
  *left = (unsigned long long)max_shard * maxM;
}

// segment of term t: the last one whose first term is <= t (seg[0].t0 = 0, t0 ascending)
H2V_HD u32 mix_segment(const MixSeg* seg, u32 count, u32 t) {
  u32 lo = 0, hi = count;
  while (hi - lo > 1) {
    const u32 mid = (lo + hi) >> 1;
    if (seg[mid].t0 <= t) lo = mid;
    else hi = mid;
  }
  return lo;
}

// term tl of a segment: kind 0 = proof point i of proof j (right channel), 1 = multi-open point i of proof j (left
// channel), 2 = shared base i (right channel, j = 0)
struct MixTerm {
  u32 kind, j, i;
};
H2V_HD MixTerm mix_term(const MixSeg& s, u32 tl) {
  const u32 nP = s.n * s.P, nL = s.n * s.n_mo;
  if (tl < nP) return MixTerm{0, tl % s.n, tl / s.n};
  if (tl < nP + nL) return MixTerm{1, (tl - nP) % s.n, (tl - nP) / s.n};
  return MixTerm{2, 0, tl - nP - nL};
}
H2V_HD u32 mix_channel(const MixTerm& m) { return m.kind == 1 ? 1u : 0u; }
H2V_HD const G1Affine& mix_point(const MixSeg& s, const MixTerm& m) {
  if (m.kind == 0) return s.pts[(size_t)m.i * s.stride + s.j0 + m.j];
  if (m.kind == 1) return s.pts[(size_t)(s.P - s.n_mo + m.i) * s.stride + s.j0 + m.j];
  return s.shared_pts[m.i];
}
// the term's scalar, canonical: c_j times the proof's scalar, or the column sum of a shared base (0 for an identity base:
// an all-zero fixed column)
H2V_HD Fr mix_scalar(const MixSeg& s, const MixTerm& m) {
  if (m.kind == 0) return (s.right[(size_t)m.i * s.stride + s.j0 + m.j] * s.coef[s.j0 + m.j]).to_canonical();
  if (m.kind == 1) return (s.left[(size_t)m.i * s.stride + s.j0 + m.j] * s.coef[s.j0 + m.j]).to_canonical();
  const G1Affine& sp = s.shared_pts[m.i];
  return (sp.x.is_zero() && sp.y.is_zero()) ? Fr::zero() : s.shared_sum[m.i];
}

// bucket index of digit magnitude mag (1 .. B) of window w, channel ch, in bucket set `set` (fold group or params class)
H2V_HD u32 msm_bucket(const MsmGeom& g, u32 set, u32 ch, u32 w, u32 mag) { return set * g.nb() + g.bbase[ch] + w * g.B[ch] + mag - 1; }

// Run length of the partial window combination of a mix whose `sets` bucket sets share one pairing check: the smallest run
// >= run0 for which sets * (ceil(W0 / run) + ceil(W1 / run)) <= 128 pairs (LinesSmem of k_lines).  With one set every
// single-batch geometry (W <= 64 per channel) fits at run0 >= 1, so a single-params mix keeps run0; with 8 sets run = 8
// always fits (2 x 8 pairs per set).
inline u32 mix_line_run(u32 sets, u32 W0, u32 W1, u32 run0) {
  u32 run = run0 ? run0 : 1;
  while (sets * ((W0 + run - 1) / run + (W1 + run - 1) / run) > 128) run++;
  return run;
}

}  // namespace h2v
