// CUDA kernels (sm_100a) and the C ABI of the batch verifier.  See include/h2v.h for the contract and
// DESIGN.md for the data layout and per-kernel rooflines.
//
// Pipeline of one launch set = G fold groups of n proofs (G = 1: one batch), all on the context's stream and replayed as
// one CUDA graph, no host round trip until the verdicts:
//   k_init            instance-shape checks                                    lib.rs:51-55
//   k_decompress      thread per (proof, point): sqrt + curve check            transcript/mod.rs:158-166
//   k_transcript_quad four lanes per proof (Blake2b; k_transcript: thread per proof, Keccak): replay -> challenges   lib.rs:66-253
//   k_scalar          thread per proof: Lagrange, h(x), multi-open scalars     lib.rs:173-347, shplonk.rs / gwc.rs
//   k_rlc_*           r_i expansion + suffix products c_j per fold group       strategy.rs:125-136
//   k_shared_reduce   column sums of the shared-base scalars
//   k_msm_digits, k_scan_*, k_bucket_order, k_msm_scatter, k_msm_bucket_sum, k_msm_chunk_reduce, k_msm_window_reduce
//                     one signed-digit Pippenger per fold group over its proofs' points   arithmetic.rs:7-108, msm.rs:81-86
//   k_window_group    runs of consecutive windows combined (the pairing then sees one pair per run)
//   k_lines           per Miller iteration: product of the lines of every (channel, run) pair
//   k_miller_segments four blocks per group walk segments of f = f^2 M_i in parallel
//   k_pairing_check   product of the segments, division-free final exponentiation test   msm.rs:185-203
//   (k_pack_partial / k_sum_partials: shards of a multi-GPU batch; k_fold_accum: explicit (L, R), parity hook only)
//   (k_pp_*, k_window_combine: per-proof accumulators / pairings: parity hook and rejection attribution, glv.cuh)
//   (k_acc_absorb: instead of the pairing, the window sums folded into a persistent accumulator, acc.cuh)
//   (k_agg: aggregation contexts, after k_scalar: the KZG accumulator carried in the instances -> two more MSM terms, agg.cuh)
#include <cuda_runtime.h>
#include <nvtx3/nvToolsExt.h>
#include <errno.h>
#include <stdio.h>
#include <string.h>
#include <sys/random.h>
#include <time.h>
#include <unistd.h>

#include <algorithm>
#include <cmath>
#include <string>
#include <vector>

#include "h2v.h"
#include "plan_build.h"
#include "stages.cuh"
#include "tower.cuh"
#include "timeline.cuh"
#include "pairing_cta.cuh"
#include "exchange.cuh"
#include "transcript_quad.cuh"
#include "glv.cuh"
#include "mix.cuh"
#include "acc.cuh"
#include "agg.cuh"

using namespace h2v;

// Minimum resident blocks per SM of the latency-bound per-proof kernels (a register cap).  Measured on B200 with
// 16 batches in flight (round 1): capping k_scalar at 128 / 96 / 64 and k_transcript at 80 / 64 registers spills almost
// nothing but leaves the throughput unchanged (5.0 M proofs/s) and costs 5-10 % of their solo latency; measured again in
// round 2 with 4 contexts x 16 fold groups (k_transcript 128 registers, k_scalar 128): 6.08 M against 6.13 M proofs/s
// uncapped.  Left uncapped.
#ifndef H2V_TRANSCRIPT_MINB
#define H2V_TRANSCRIPT_MINB 1
#endif
#ifndef H2V_SCALAR_MINB
#define H2V_SCALAR_MINB 1
#endif

// ------------------------------------------------------------------------------------------------
// diagnostics: per-block timeline (off unless h2v_debug_timeline_start was called).  Thread 0 of every block of the
// instrumented kernels appends {kernel id, block, SM, context tag, start, end} on the global nanosecond timer; used
// to see how the kernels of many batches in flight share the SMs (bench.py, H2V_BENCH_DIAG_TIMELINE).
// ------------------------------------------------------------------------------------------------
// Programmatic dependent launch: every kernel of the batch pipeline first waits for the kernel before it in the
// stream (a no-op when it was launched without the attribute) and then lets the kernel after it be placed on the
// SMs, where that one waits in turn.  The next kernel is thus resident when its predecessor ends: with many batches
// in flight the stream-ordered hand-over cost ~350 us per kernel boundary (measured with the block timeline below).
__device__ __forceinline__ void pdl_prologue() {
  asm volatile("griddepcontrol.wait;" ::: "memory");
  asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
}

// ------------------------------------------------------------------------------------------------
// kernels
// ------------------------------------------------------------------------------------------------
__global__ void k_init(PlanView pv, u32 n, const u64* inst_off, const u32* ncols, const u32* col_len, u32* status, u32* bad) {
  pdl_prologue();
  const u32 j = blockIdx.x * blockDim.x + threadIdx.x;
  if (j >= n) return;
  const PlanHeader& hd = pv.h();
  bad[j] = H2V_NO_BAD_ITEM;
  const u64 tot = inst_off[j + 1] - inst_off[j];
  u32 st = ST_OK;
  if (ncols && ncols[j] != hd.n_inst_cols) {
    st = ST_INVALID_INSTANCES;
  } else if (col_len) {
    u64 s = 0;
    for (u32 c = 0; c < hd.n_inst_cols; c++) s += col_len[(size_t)j * hd.n_inst_cols + c];
    if (s != tot) st = ST_INVALID_INSTANCES;
  } else if (hd.n_inst_cols == 0 ? tot != 0 : (tot % hd.n_inst_cols) != 0) {
    st = ST_INVALID_INSTANCES;
  }
  status[j] = st;
}

// phi != null (a lifted GLV geometry, phi_rows): also phi(P) = (beta x, y) of every point into phi (the layout of pts), and
// every shared base b into pts[msm_points * n + b] with its phi into phi[msm_points * n + b]
__global__ void __launch_bounds__(128) k_decompress(PlanView pv, u32 n, const u8* proofs, const u64* proof_off, G1Affine* pts, G1Affine* phi, u32* ptsc, u32* bad,
                                                    u32 blk_off, u32 blk_total) {
  pdl_prologue();
  TlScope tl_(1, pts);
  const PlanHeader& hd = pv.h();
  if (phi)
    for (u32 i = (blk_off + blockIdx.x) * blockDim.x + threadIdx.x; i < hd.n_shared; i += blk_total * blockDim.x) {
      G1Affine q = pv.sec<G1Affine>(hd.off_shared_pts)[i];
      pts[(size_t)msm_points(hd) * n + i] = q;
      q.x = Fq::mul_c(q.x, glv_beta());
      phi[(size_t)msm_points(hd) * n + i] = q;
    }
  // grid-stride: the grid may be capped below the work (wide_grid) so that this multiplier-bound kernel leaves block
  // slots on every SM to the latency-bound kernels of the other contexts in flight
  for (u32 t = (blk_off + blockIdx.x) * blockDim.x + threadIdx.x; t < n * hd.n_points; t += blk_total * blockDim.x) {
    const u32 j = t % n, slot = t / n;
    const u64 off = proof_off[j];
    const u32 len = (u32)(proof_off[j + 1] - off);
    G1Affine p;
    Fq canon[2];  // canonical x | y for the quad transcript replay (ptsc == null: not wanted)
    if (!decompress_stage(pv, proofs + off, len, slot, p, ptsc ? canon : nullptr)) {
      p.x = Fq::zero();
      p.y = Fq::zero();
      canon[0] = Fq::zero();
      canon[1] = Fq::zero();
      atomicMin(&bad[j], pv.sec<u32>(hd.off_pt_item)[slot]);
    }
    pts[t] = p;
    if (phi) {
      p.x = Fq::mul_c(p.x, glv_beta());
      phi[t] = p;
    }
    if (ptsc) {
      uint4* o = (uint4*)(ptsc + 16 * (size_t)t);
      o[0] = make_uint4(canon[0].l[0], canon[0].l[1], canon[0].l[2], canon[0].l[3]);
      o[1] = make_uint4(canon[0].l[4], canon[0].l[5], canon[0].l[6], canon[0].l[7]);
      o[2] = make_uint4(canon[1].l[0], canon[1].l[1], canon[1].l[2], canon[1].l[3]);
      o[3] = make_uint4(canon[1].l[4], canon[1].l[5], canon[1].l[6], canon[1].l[7]);
    }
  }
}

template <class H>
__global__ void __launch_bounds__(64, H2V_TRANSCRIPT_MINB) k_transcript(PlanView pv, u32 n, const u8* proofs, const u64* proof_off, const u8* inst,
                                                   const u64* inst_off, const G1Affine* pts, Fr* vals, u32* status, const u32* bad) {
  pdl_prologue();
  TlScope tl_(2, pts);
  const PlanHeader& hd = pv.h();
  // grid-stride: the grid may be capped (narrow_grid) so that this latency-bound kernel shares the SMs with the
  // multiplier-bound kernels of the other contexts in flight instead of displacing them
  for (u32 j = blockIdx.x * blockDim.x + threadIdx.x; j < n; j += gridDim.x * blockDim.x) {
    if (status[j] != ST_OK) continue;
    const u64 off = proof_off[j];
    bool inst_bad;
    const u32 b = transcript_stage<H>(pv, proofs + off, (u32)(proof_off[j + 1] - off), inst + 32 * inst_off[j],
                                      (u32)(inst_off[j + 1] - inst_off[j]), pts, vals, j, n, bad[j], inst_bad);
    if (inst_bad) status[j] = ST_INVALID_INSTANCES;
    else if (b != H2V_NO_BAD_ITEM) status[j] = b < hd.first_mo_item ? ST_TRANSCRIPT : ST_OPENING;
  }
}

// Blake2b transcripts: four lanes per proof (transcript_quad.cuh)
__global__ void __launch_bounds__(4 * TQ_PROOFS_PER_BLOCK) k_transcript_quad(PlanView pv, u32 n, const u8* proofs, const u64* proof_off, const u8* inst, const u64* inst_off,
                                                                             const u32* ptsc, Fr* vals, u32* status, const u32* bad) {
  pdl_prologue();
  TlScope tl_(2, ptsc);
  __shared__ __align__(16) u8 bufs[TQ_PROOFS_PER_BLOCK][TQ_BUF_STRIDE];
  const PlanHeader& hd = pv.h();
  // grid-stride over the proofs (see k_transcript); every quad is on its own: shuffles and barriers use the quad's mask
  for (u32 j = blockIdx.x * TQ_PROOFS_PER_BLOCK + (threadIdx.x >> 2); j < n; j += gridDim.x * TQ_PROOFS_PER_BLOCK) {  // quad-uniform
    if (status[j] != ST_OK) continue;  // quad-uniform
    TqState st;
    tq_setup(st, bufs[threadIdx.x >> 2]);
    const u64 off = proof_off[j];
    bool inst_bad;
    const u32 b = transcript_quad(pv, proofs + off, (u32)(proof_off[j + 1] - off), inst + 32 * inst_off[j], (u32)(inst_off[j + 1] - inst_off[j]), ptsc, vals, j,
                                  n, bad[j], inst_bad, st);
    if (st.q == 0) {
      if (inst_bad) status[j] = ST_INVALID_INSTANCES;
      else if (b != H2V_NO_BAD_ITEM) status[j] = b < hd.first_mo_item ? ST_TRANSCRIPT : ST_OPENING;
    }
  }
}

template <int MINB>
__global__ void __launch_bounds__(64, MINB) k_scalar(PlanView pv, u32 n, const u8* inst, const u64* inst_off, const u32* col_len, Fr* vals,
                                               Fr* scratch, Fr* right, Fr* shared, Fr* left, u32* status) {
  pdl_prologue();
  TlScope tl_(3, right);
  const PlanHeader& hd = pv.h();
  for (u32 j = blockIdx.x * blockDim.x + threadIdx.x; j < n; j += gridDim.x * blockDim.x) {  // grid-stride, see k_transcript
    u32 st = status[j];
    if (st == ST_OK) {
      ScalarIO io{j, n, vals, scratch, right, shared, left};
      st = scalar_stage(pv, io, inst + 32 * inst_off[j], col_len ? col_len + (size_t)j * hd.n_inst_cols : nullptr,
                        (u32)(inst_off[j + 1] - inst_off[j]));
      if (st != ST_OK) status[j] = st;
    }
    if (st != ST_OK) {  // excluded from the fold
      for (u32 i = 0; i < hd.n_points; i++) right[(size_t)i * n + j] = Fr::zero();
      for (u32 i = 0; i < hd.n_shared; i++) shared[(size_t)i * n + j] = Fr::zero();
      for (u32 i = 0; i < hd.n_mo; i++) left[(size_t)i * n + j] = Fr::zero();
    }
  }
}

// Aggregation contexts: the KZG accumulator (lhs, rhs) carried in every proof's instances (agg.cuh), thread per proof.  In
// DualMSM orientation, e(L, [s]G2) e(R, -G2) = 1, the decider's lhs = s rhs is a right-channel term and rhs a left-channel
// one: lhs goes to slot n_points with right scalar rho, rhs to slot n_points + 1 with left scalar rho (plan.h msm_points), so
// every consumer of the per-proof terms (bucket MSM, attribution, per-proof hooks, shards, mixes) sees them.  Runs after
// k_scalar and before the shared-base sums: a proof whose encoding is invalid gets ST_INVALID_INSTANCES whatever the later
// stages found (the precedence of the instance check, lib.rs:51-55) and all its scalars are zeroed.  An identity point gets
// scalar 0 (the MSM kernels take every affine point as a curve point).
__global__ void __launch_bounds__(128) k_agg(PlanView pv, u32 n, const u8* inst, const u64* inst_off, const u32* col_len, const Fr* rho,
                                             G1Affine* pts, G1Affine* phi, Fr* right, Fr* shared, Fr* left, u32* status) {
  pdl_prologue();
  const u32 j = blockIdx.x * blockDim.x + threadIdx.x;
  if (j >= n) return;
  const PlanHeader& hd = pv.h();
  const u32 P0 = hd.n_points, M0 = hd.n_mo, L = hd.agg_limbs, C = hd.n_inst_cols;
  u32 st = status[j];
  G1Affine p[2];
  bool id[2] = {true, true};
  bool ok = st != ST_INVALID_INSTANCES;  // (k_init found the layout malformed: the cells cannot be located)
  if (ok) {
    const u64 tot = inst_off[j + 1] - inst_off[j];
    const u8* base = inst + 32 * inst_off[j];
    const AggCell* cells = pv.sec<AggCell>(hd.off_agg);
    for (u32 q = 0; q < 2 && ok; q++) {
      const u8* limb[2 * AGG_MAX_LIMBS];
      for (u32 i = 0; i < 2 * L; i++) {
        const AggCell c = cells[2 * L * q + i];
        u64 start = 0, len;
        if (col_len) {
          for (u32 k = 0; k < c.column; k++) start += col_len[(size_t)j * C + k];
          len = col_len[(size_t)j * C + c.column];
        } else {
          len = tot / C;
          start = (u64)c.column * len;
        }
        if (c.row >= len) ok = false;  // a ragged column too short for the cell
        limb[i] = base + 32 * (start + (c.row < len ? c.row : 0));
      }
      if (ok) ok = agg_point(limb, L, hd.agg_bits, p[q], &id[q]);
    }
  }
  if (!ok) {
    st = ST_INVALID_INSTANCES;
    status[j] = st;
    for (u32 i = 0; i < P0; i++) right[(size_t)i * n + j] = Fr::zero();
    for (u32 i = 0; i < hd.n_shared; i++) shared[(size_t)i * n + j] = Fr::zero();
    for (u32 i = 0; i < M0; i++) left[(size_t)i * n + j] = Fr::zero();
  }
  const bool live = st == ST_OK;
  const Fr r = *rho;
  for (u32 q = 0; q < 2; q++) {
    G1Affine a;
    a.x = ok ? p[q].x : Fq::zero();
    a.y = ok ? p[q].y : Fq::zero();
    pts[(size_t)(P0 + q) * n + j] = a;
    if (phi) {  // (as in k_decompress)
      a.x = Fq::mul_c(a.x, glv_beta());
      phi[(size_t)(P0 + q) * n + j] = a;
    }
  }
  right[(size_t)P0 * n + j] = live && !id[0] ? r : Fr::zero();
  right[(size_t)(P0 + 1) * n + j] = Fr::zero();
  left[(size_t)M0 * n + j] = Fr::zero();
  left[(size_t)(M0 + 1) * n + j] = live && !id[1] ? r : Fr::zero();
}

// fold randomness r_i: caller-supplied bytes (parity hook), a 64-bit test seed (parity hook), or the secret per-batch key
__global__ void k_rlc_expand(u64 count, u64 seed, const u8* bytes, bool keyed, RlcKey key, Fr* r) {
  const u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= count) return;
  r[i] = bytes ? Fr::from_canonical(Fr::load_le(bytes + 32 * i)) : keyed ? rlc_scalar_from_key(key, i) : rlc_scalar_from_seed(seed, i);
}

// c_j = prod_{i > j} r_i over the GLOBAL batch; one block per scan, chunked suffix scan through shared memory.
static constexpr u32 RLC_NT = 256;
// Block b scans `count` coefficients starting at r + (b / subs) * group_stride + offset + (b % subs) * count and writes
// those with index in [base, base + n) to coef + b * n.
//   fold groups (subs = 1, group_stride = count, offset = 0): block g scans the coefficients of its own global batch and
//     writes the n of this rank's shard of it
//   attribution (count = n = m, base = 0, subs = sub-batches per fold group, group_stride = proofs per group, offset = 0,
//     r = the re-fold's own scalars, one per proof of the shard): block b scans the m coefficients of sub-batch b % subs of
//     fold group b / subs: the fold restarts inside every sub-batch
__global__ void __launch_bounds__(RLC_NT) k_rlc_scan(const Fr* r, u64 count, u64 base, u32 n, Fr* coef, u32 subs, u64 group_stride, u64 offset) {
  pdl_prologue();
  TlScope tl_(14, coef);
  __shared__ Fr sh[RLC_NT];
  r += (size_t)(blockIdx.x / subs) * group_stride + offset + (size_t)(blockIdx.x % subs) * count;
  coef += (size_t)blockIdx.x * n;
  const u32 t = threadIdx.x;
  const u64 m = (count + RLC_NT - 1) / RLC_NT;
  const u64 lo = (u64)t * m < count ? (u64)t * m : count, hi = lo + m < count ? lo + m : count;
  Fr p = Fr::one();
  for (u64 i = lo; i < hi; i++) p = p * r[i];
  sh[t] = p;
  __syncthreads();
  for (u32 d = 1; d < RLC_NT; d <<= 1) {  // inclusive suffix products
    Fr v = sh[t];
    const bool act = t + d < RLC_NT;
    Fr o = act ? sh[t + d] : Fr::one();
    __syncthreads();
    if (act) sh[t] = v * o;
    __syncthreads();
  }
  Fr run = t + 1 < RLC_NT ? sh[t + 1] : Fr::one();
  for (u64 i = hi; i-- > lo;) {
    if (i >= base && i < base + n) coef[i - base] = run;
    run = run * r[i];
  }
}

// shared_sum[b] = sum_j c_j * shared[b][j]  (canonical form, ready for digit extraction)
__global__ void __launch_bounds__(256) k_shared_reduce(u32 n, u32 N, u32 Sh, const Fr* shared, const Fr* coef, Fr* shared_sum) {
  pdl_prologue();
  TlScope tl_(15, shared_sum);
  __shared__ Fr sh[256];
  const u32 b = blockIdx.x, grp = blockIdx.y, t = threadIdx.x;
  Fr acc = Fr::zero();
  for (u32 j = t; j < n; j += 256) acc = acc + shared[(size_t)b * N + grp * n + j] * coef[grp * n + j];
  sh[t] = acc;
  __syncthreads();
  for (u32 d = 128; d > 0; d >>= 1) {
    if (t < d) sh[t] = sh[t] + sh[t + d];
    __syncthreads();
  }
  if (t == 0) shared_sum[grp * Sh + b] = sh[0].to_canonical();
}

// Fold coefficients of a mixed batch, every group in one launch: block q runs the suffix scan of k_rlc_scan over group q's
// call indices [grange[q], grange[q + 1]) (the fold restarts at every group boundary, c_i = prod_{i' in group q, i' > i} r_i')
// and writes c_i into the coefficient array of the member that owns proof i: segment seg[q * members + m] holds call indices
// [call0, call0 + n) at [j0, j0 + n) of member m's arrays.  A sharded mix is one group over the global batch whose segments
// cover this rank's range only; the other indices are scanned, not written.
__global__ void __launch_bounds__(RLC_NT) k_rlc_scan_groups(const Fr* r, const u32* grange, const MixSeg* seg, u32 members) {
  pdl_prologue();
  TlScope tl_(14, r);
  __shared__ Fr sh[RLC_NT];
  const u32 q = blockIdx.x, t = threadIdx.x;
  const u64 g0 = grange[q], count = (u64)grange[q + 1] - g0;
  seg += (size_t)q * members;
  const u64 m = (count + RLC_NT - 1) / RLC_NT;
  const u64 lo = (u64)t * m < count ? g0 + (u64)t * m : g0 + count, hi = lo + m < g0 + count ? lo + m : g0 + count;
  Fr p = Fr::one();
  for (u64 i = lo; i < hi; i++) p = p * r[i];
  sh[t] = p;
  __syncthreads();
  for (u32 d = 1; d < RLC_NT; d <<= 1) {  // inclusive suffix products
    Fr v = sh[t];
    const bool act = t + d < RLC_NT;
    Fr o = act ? sh[t + d] : Fr::one();
    __syncthreads();
    if (act) sh[t] = v * o;
    __syncthreads();
  }
  mix_scan_chunk(r, lo, hi, t + 1 < RLC_NT ? sh[t + 1] : Fr::one(), seg, members);
}

// k_shared_reduce per segment of a mixed batch: block (s, b) writes seg[s].shared_sum[b] = sum over the segment's proofs of
// c_j * shared[b][j] (zero for a segment without proofs)
__global__ void __launch_bounds__(256) k_shared_reduce_seg(const MixSeg* seg) {
  pdl_prologue();
  const MixSeg& sg = seg[blockIdx.x];
  const u32 b = blockIdx.y, t = threadIdx.x;
  if (b >= sg.Sh) return;
  TlScope tl_(15, sg.shared_sum);
  __shared__ Fr sh[256];
  Fr acc = Fr::zero();
  for (u32 j = t; j < sg.n; j += 256) acc = acc + sg.shared[(size_t)b * sg.stride + sg.j0 + j] * sg.coef[sg.j0 + j];
  sh[t] = acc;
  __syncthreads();
  for (u32 d = 128; d > 0; d >>= 1) {
    if (t < d) sh[t] = sh[t] + sh[t + d];
    __syncthreads();
  }
  if (t == 0) sg.shared_sum[b] = sh[0].to_canonical();
}

// signed c-bit digits of a little-endian magnitude kk[0..NL) (bits beyond NL limbs are zero), negated when `neg`; row of
// the digit table + bucket histogram of the term's channel
template <int NL>
__device__ __forceinline__ void msm_emit_digits(const MsmGeom& g, u32 ch, u32 grp, const u32* kk, bool neg, int16_t* row, u32* hist) {
  u32 carry = 0;
  const u32 c = g.c[ch], mask = (1u << c) - 1, half = 1u << (c - 1);
  for (u32 w = 0; w < g.W[ch]; w++) {
    const u32 bit = w * c;
    const u32 li = bit >> 5, sh = bit & 31;
    u64 two = li < NL ? kk[li] : 0;
    if (li + 1 < NL) two |= (u64)kk[li + 1] << 32;
    u32 v = ((u32)(two >> sh) & mask) + carry;
    int d;
    if (v > half) {
      d = (int)v - (int)(1u << c);
      carry = 1;
    } else {
      d = (int)v;
      carry = 0;
    }
    if (neg) d = -d;
    row[w] = (int16_t)d;
    if (d != 0) atomicAdd(&hist[msm_bucket(g, grp, ch, w, (u32)(d < 0 ? -d : d))], 1u);
  }
}

// signed c-bit digits of every term's scalar (already multiplied by c_j) + bucket histogram.  Src = SingleVkTerms: the
// terms of g (the pointer arguments); MixTerms: the segment table of a mixed batch (g.T = every term, g.G = bucket sets, a
// term's set = its segment's class; the pointer arguments are unused)
template <class Src>
__global__ void __launch_bounds__(128) k_msm_digits(MsmGeom g, const Fr* right, const Fr* left, const Fr* coef, const Fr* shared_sum,
                                                    const G1Affine* shared_pts, int16_t* dig, u32* hist, const u32* parent_verdict, u32 parent_size,
                                                    Src src) {
  pdl_prologue();
  TlScope tl_(4, right);
  const u32 t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= (Src::mixed ? g.T : g.G * g.T)) return;
  u32 grp = t / g.T;
  const u32 tl = t % g.T;
  const u32 nP = g.n * g.P, nL = g.n * g.n_mo;
  const u32 rows = 1 + g.glv;  // digit rows of this term
  Fr k;
  u32 ch = 0;
  if constexpr (Src::mixed) {
    const MixSeg& sg = src.seg[mix_segment(src.seg, src.count, t)];
    const MixTerm mt = mix_term(sg, t - sg.t0);
    k = mix_scalar(sg, mt);
    ch = mix_channel(mt);
    grp = sg.cls;
  } else {
    if (parent_verdict && parent_verdict[(u32)(((u64)grp * g.n) / parent_size)]) {  // sub-batch of an accepted fold group: nothing to re-check
      ch = g.channel_of_term(tl);
      for (u32 w = 0; w < rows * g.Wmax; w++) dig[(size_t)t * rows * g.Wmax + w] = 0;
      return;
    }
    if (tl < nP) {
      const u32 j = grp * g.n + tl % g.n;
      k = (right[(size_t)(tl / g.n) * g.N + j] * coef[j]).to_canonical();
    } else if (tl < nP + nL) {
      const u32 j = grp * g.n + (tl - nP) % g.n;
      k = (left[(size_t)((tl - nP) / g.n) * g.N + j] * coef[j]).to_canonical();
      ch = 1;
    } else {
      const G1Affine& sp = shared_pts[tl - nP - nL];
      k = (sp.x.is_zero() && sp.y.is_zero()) ? Fr::zero() : shared_sum[grp * g.Sh + tl - nP - nL];  // identity base (all-zero fixed column)
    }
  }
  if (k.is_zero()) {  // excluded proof / unused slot / identity base: no bucket entries at all
    for (u32 w = 0; w < rows * g.Wmax; w++) dig[(size_t)t * rows * g.Wmax + w] = 0;
    return;
  }
  if (g.glv) {  // k = k1 + k2 lambda: row 2 t of P, row 2 t + 1 of phi(P)
    if (g.Z2[ch]) {  // lifted halves, k = a - b lambda (glv_lift)
      u32 a[5], b[5];
      glv_lift_term(k.l, t, g.Z[ch], g.Z2[ch], a, b);
      msm_emit_digits<5>(g, ch, grp, a, false, dig + (size_t)(2 * t) * g.Wmax, hist);
      msm_emit_digits<5>(g, ch, grp, b, true, dig + (size_t)(2 * t + 1) * g.Wmax, hist);
      return;
    }
    GlvHalf h1, h2;
    glv_decompose(k.l, h1, h2);
    msm_emit_digits<5>(g, ch, grp, h1.l, h1.neg, dig + (size_t)(2 * t) * g.Wmax, hist);
    msm_emit_digits<5>(g, ch, grp, h2.l, h2.neg, dig + (size_t)(2 * t + 1) * g.Wmax, hist);
    return;
  }
  // k'' = k + z*r (r*P = identity: same group element), z spread over [0, Z) so that k'' is uniform in
  // [0, Z*r) ~ [0, 2^(W*c-1)): every window, including the top one, fills its buckets evenly.
  u32 kk[9];
  {
    const u32 z = ((t * 2654435761u) >> 8) % g.Z[ch];
    u64 acc = 0;
#pragma unroll
    for (int i = 0; i < 8; i++) {
      acc += (u64)z * FrP::mod(i) + k.l[i];
      kk[i] = (u32)acc;
      acc >>= 32;
    }
    kk[8] = (u32)acc;
  }
  msm_emit_digits<9>(g, ch, grp, kk, false, dig + (size_t)t * g.Wmax, hist);
}

// exclusive scan of the bucket histogram in two launches: tiles of 1024 counters are scanned with coalesced
// loads (warp shuffles), then every tile adds the totals of the tiles before it.  off has nb + 1 entries,
// cursor is a working copy for the scatter.
// exclusive scan over the NT threads of a block (NT a multiple of 32, at most 1024)
template <int NT>
__device__ __forceinline__ u32 block_excl_scan(u32 v, u32* total) {
  __shared__ u32 wsum[32];
  const u32 lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  u32 x = v;
#pragma unroll
  for (int d = 1; d < 32; d <<= 1) {
    const u32 y = __shfl_up_sync(0xFFFFFFFFu, x, d);
    if (lane >= (u32)d) x += y;
  }
  if (lane == 31) wsum[wid] = x;
  __syncthreads();
  if (wid == 0) {
    u32 w = lane < NT / 32 ? wsum[lane] : 0;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
      const u32 y = __shfl_up_sync(0xFFFFFFFFu, w, d);
      if (lane >= (u32)d) w += y;
    }
    wsum[lane] = w;
  }
  __syncthreads();
  *total = wsum[31];
  const u32 r = x - v + (wid ? wsum[wid - 1] : 0);
  __syncthreads();  // wsum is reused by the next call
  return r;
}
// Tiles of SCAN_TILE counters are scanned by blocks of SCAN_NT threads, SCAN_PER consecutive counters per thread.
// Blocks are kept small everywhere in the pipeline: with many batches in flight a 1024-thread block has to wait
// for half an SM to drain before it can be placed.
static constexpr u32 SCAN_NT = 256, SCAN_PER = 4, SCAN_TILE = SCAN_NT * SCAN_PER;
// size_bin: bucket sizes are binned in DESCENDING order (bin 0 = 1023 entries or more) for k_bucket_order
static constexpr u32 SIZE_BINS = 1024;
__device__ __forceinline__ u32 size_bin(u32 count) { return SIZE_BINS - 1 - (count < SIZE_BINS - 1 ? count : SIZE_BINS - 1); }
__global__ void __launch_bounds__(SCAN_NT) k_scan_tiles(const u32* hist, u32 nb, u32* off, u32* tile_total, u32* size_hist) {
  pdl_prologue();
  // the bucket sizes of a uniform MSM crowd into a few dozen size bins: the per-bucket global atomics on those few
  // addresses were 100 us per launch set (ncu, 16 fold groups); the tile counts its bins in shared memory first
  __shared__ u32 bins[SIZE_BINS];
  for (u32 i = threadIdx.x; i < SIZE_BINS; i += SCAN_NT) bins[i] = 0;
  __syncthreads();
  const u32 i0 = blockIdx.x * SCAN_TILE + threadIdx.x * SCAN_PER;
  u32 v[SCAN_PER], sum = 0;
#pragma unroll
  for (u32 q = 0; q < SCAN_PER; q++) {
    v[q] = i0 + q < nb ? hist[i0 + q] : 0;
    if (i0 + q < nb) atomicAdd(&bins[size_bin(v[q])], 1u);
    sum += v[q];
  }
  u32 total;
  u32 e = block_excl_scan<SCAN_NT>(sum, &total);
#pragma unroll
  for (u32 q = 0; q < SCAN_PER; q++) {
    if (i0 + q < nb) off[i0 + q] = e;
    e += v[q];
  }
  if (threadIdx.x == 0) tile_total[blockIdx.x] = total;
  __syncthreads();
  for (u32 i = threadIdx.x; i < SIZE_BINS; i += SCAN_NT)
    if (bins[i]) atomicAdd(&size_hist[i], bins[i]);
}
__global__ void __launch_bounds__(SCAN_NT) k_scan_apply(u32 nb, u32 n_tiles, const u32* tile_total, u32* off, u32* cursor) {
  pdl_prologue();
  __shared__ u32 base_sh;
  u32 part = 0;
  for (u32 k = threadIdx.x; k < blockIdx.x; k += SCAN_NT) part += tile_total[k];
  u32 total;
  block_excl_scan<SCAN_NT>(part, &total);  // only the block total is used
  if (threadIdx.x == 0) base_sh = total;
  __syncthreads();
  const u32 base = base_sh;
#pragma unroll
  for (u32 q = 0; q < SCAN_PER; q++) {
    const u32 i = blockIdx.x * SCAN_TILE + q * SCAN_NT + threadIdx.x;
    if (i < nb) {
      const u32 o = off[i] + base;
      off[i] = o;
      cursor[i] = o;
    }
  }
  if (blockIdx.x == n_tiles - 1 && threadIdx.x == 0) off[nb] = base + tile_total[blockIdx.x];
}

// Buckets ordered by size, largest first (counting sort on the size bins): the threads of a warp of
// k_msm_bucket_sum then walk chains of (nearly) equal length, and the longest chains start first.
__global__ void __launch_bounds__(SCAN_NT) k_bucket_order(u32 nb, const u32* hist, const u32* size_hist, u32* size_cursor, u32* order) {
  pdl_prologue();
  TlScope tl_(16, order);
  static_assert(SIZE_BINS == SCAN_TILE, "one tile of size bins");
  __shared__ u32 base[SIZE_BINS];
  __shared__ u32 cnt[SIZE_BINS];  // buckets of this tile per size bin, then the tile's first slot inside the bin
  u32 v[SCAN_PER], sum = 0, total;
#pragma unroll
  for (u32 q = 0; q < SCAN_PER; q++) {
    v[q] = size_hist[threadIdx.x * SCAN_PER + q];
    sum += v[q];
    cnt[threadIdx.x * SCAN_PER + q] = 0;
  }
  u32 e = block_excl_scan<SCAN_NT>(sum, &total);
#pragma unroll
  for (u32 q = 0; q < SCAN_PER; q++) {
    base[threadIdx.x * SCAN_PER + q] = e;
    e += v[q];
  }
  __syncthreads();
  // slots inside a bin: first within the tile (shared-memory atomics), then ONE global atomic per (tile, bin) instead
  // of one per bucket (the buckets crowd into a few dozen bins: 100 us per launch set of 16 fold groups, ncu)
  u32 bin[SCAN_PER], local[SCAN_PER];
#pragma unroll
  for (u32 q = 0; q < SCAN_PER; q++) {
    const u32 i = blockIdx.x * SCAN_TILE + q * SCAN_NT + threadIdx.x;
    if (i < nb) {
      bin[q] = size_bin(hist[i]);
      local[q] = atomicAdd(&cnt[bin[q]], 1u);
    }
  }
  __syncthreads();
#pragma unroll
  for (u32 q = 0; q < SCAN_PER; q++) {
    const u32 b = threadIdx.x * SCAN_PER + q;
    if (cnt[b]) cnt[b] = atomicAdd(&size_cursor[b], cnt[b]);
  }
  __syncthreads();
#pragma unroll
  for (u32 q = 0; q < SCAN_PER; q++) {
    const u32 i = blockIdx.x * SCAN_TILE + q * SCAN_NT + threadIdx.x;
    if (i < nb) order[base[bin[q]] + cnt[bin[q]] + local[q]] = i;
  }
}

template <class Src>
__global__ void __launch_bounds__(256) k_msm_scatter(MsmGeom g, const int16_t* dig, u32* cursor, u32* sorted, Src src) {
  pdl_prologue();
  TlScope tl_(5, sorted);
  const u64 total = ((Src::mixed ? (u64)g.T : (u64)g.G * g.T) << g.glv) * g.Wmax;
  for (u64 idx = (u64)blockIdx.x * blockDim.x + threadIdx.x; idx < total; idx += (u64)gridDim.x * blockDim.x) {
    const u32 row = (u32)(idx / g.Wmax), w = (u32)(idx % g.Wmax);  // row = term, or 2 term + GLV half
    const u32 t = row >> g.glv;
    u32 ch, cls = 0;
    if constexpr (Src::mixed) {
      const MixSeg& sg = src.seg[mix_segment(src.seg, src.count, t)];
      ch = mix_channel(mix_term(sg, t - sg.t0));
      cls = sg.cls;
    } else {
      ch = g.channel_of_term(t % g.T);
    }
    if (w >= g.W[ch]) continue;
    const int d = dig[idx];
    if (d == 0) continue;
    const u32 b = msm_bucket(g, Src::mixed ? cls : t / g.T, ch, w, (u32)(d < 0 ? -d : d));
    const u32 pos = atomicAdd(&cursor[b], 1u);
    sorted[pos] = row | (d < 0 ? 0x80000000u : 0u);
  }
}

// thread per bucket: sum of its (signed) points, Jacobian += affine
__device__ __forceinline__ G1Jac shfl_down_jac(const G1Jac& p, u32 delta) {
  G1Jac r;
#pragma unroll
  for (int i = 0; i < 8; i++) {
    r.X.l[i] = __shfl_down_sync(0xFFFFFFFFu, p.X.l[i], delta);
    r.Y.l[i] = __shfl_down_sync(0xFFFFFFFFu, p.Y.l[i], delta);
    r.Z.l[i] = __shfl_down_sync(0xFFFFFFFFu, p.Z.l[i], delta);
  }
  return r;
}

// GLV = true: entry 2 t + 1 stands for phi(P_t) = (beta x, y).  LANES > 1 (attribution sub-batches): few, long buckets (56 entries
// with 4-bit windows), so GLV_BUCKET_LANES lanes share a bucket (entries e0 + q, e0 + q + LANES, ...), add their partial sums with
// shuffles and multiply x by beta themselves.  LANES = 1 (lifted GLV geometry of launch sets): many buckets, one lane each, phi(P)
// read from the phi rows after the points (one multiplication per point when they are written instead of one per entry)
#ifndef GLV_BUCKET_LANES
#define GLV_BUCKET_LANES 2
#endif
// point of term t (the source as in k_msm_digits)
template <class Src>
__device__ __forceinline__ const G1Affine& term_point(const MsmGeom& g, u32 t, const G1Affine* pts, const G1Affine* shared_pts, const Src& src) {
  if constexpr (Src::mixed) {
    const MixSeg& sg = src.seg[mix_segment(src.seg, src.count, t)];
    return mix_point(sg, mix_term(sg, t - sg.t0));
  } else {
    return msm_point(g, t, pts, shared_pts);
  }
}
template <bool GLV, int LANES, class Src>
__global__ void __launch_bounds__(128) k_msm_bucket_sum(MsmGeom g, u32 nb, const u32* off, const u32* order, const u32* sorted,
                                                        const G1Affine* pts, const G1Affine* shared_pts, G1Jac* buckets, u32 blk_off, u32 blk_total,
                                                        Src src) {
  pdl_prologue();
  TlScope tl_(6, pts);
  if constexpr (LANES > 1) {
    // LANES lanes per bucket (entries e0 + q, e0 + q + LANES, ...), partial sums added with shuffles: for launches whose bucket
    // chains are the critical path (a single batch; the attribution sub-batches)
    for (u32 t0 = (blk_off + blockIdx.x) * blockDim.x; t0 < LANES * nb; t0 += blk_total * blockDim.x) {  // block-uniform bound: every lane reaches the shuffles
      const u32 t = t0 + threadIdx.x, q = t % LANES;
      const bool live = t / LANES < nb;
      const u32 b = live ? order[t / LANES] : 0;
      G1Jac acc = G1Jac::identity();
      if (live) {
        const u32 e1 = off[b + 1];
        for (u32 e = off[b] + q; e < e1; e += LANES) {
          const u32 ent = sorted[e], row = ent & 0x7FFFFFFFu;
          if constexpr (GLV) {
            static_assert(!Src::mixed, "mixed batches have no GLV split");
            G1Affine pt = msm_point(g, row >> 1, pts, shared_pts);
            if (row & 1) pt.x = Fq::mul_c(pt.x, glv_beta());
            acc = g1_add_mixed(acc, pt, (ent >> 31) != 0);
          } else {
            acc = g1_add_mixed(acc, term_point(g, row, pts, shared_pts, src), (ent >> 31) != 0);
          }
        }
      }
#pragma unroll
      for (u32 d = LANES / 2; d >= 1; d >>= 1) acc = g1_add(acc, shfl_down_jac(acc, d));
      if (live && q == 0) buckets[b] = acc;
    }
  } else {
    for (u32 t = (blk_off + blockIdx.x) * blockDim.x + threadIdx.x; t < nb; t += blk_total * blockDim.x) {  // grid-stride, see k_decompress
      const u32 b = order[t];
      G1Jac acc = G1Jac::identity();
      const u32 e0 = off[b], e1 = off[b + 1];
      for (u32 e = e0; e < e1; e++) {
        const u32 ent = sorted[e];
        if constexpr (GLV) {  // a lifted GLV geometry (launch sets): entry 2 t + 1 reads the precomputed phi(P_t)
          static_assert(!Src::mixed, "mixed batches have no GLV split");
          const u32 row = ent & 0x7FFFFFFFu;
          const G1Affine* p = &msm_point(g, row >> 1, pts, shared_pts);  // (shared_pts: the copy after the points, phi_rows)
          if (row & 1) p += (size_t)g.P * g.N + g.Sh;
          acc = g1_add_mixed(acc, *p, (ent >> 31) != 0);
        } else {
          acc = g1_add_mixed(acc, term_point(g, ent & 0x7FFFFFFFu, pts, shared_pts, src), (ent >> 31) != 0);
        }
      }
      buckets[b] = acc;
    }
  }
}

__device__ G1Jac g1_mul_small(const G1Jac& p, u32 k) {
  G1Jac acc = G1Jac::identity();
  if (k == 0) return acc;
  for (int i = 31 - __clz(k); i >= 0; i--) {
    acc = g1_double(acc);
    if ((k >> i) & 1) acc = g1_add(acc, p);
  }
  return acc;
}

// S_w = sum_{k=1..B} k * bucket_k, in two steps.  Step A, thread per chunk of m buckets: running-sum
// trick inside the chunk plus (offset * chunk sum).  Step B, block per window: tree reduction.
__global__ void __launch_bounds__(128, 4) k_msm_chunk_reduce(MsmGeom g, u32 n_chunks, const G1Jac* buckets, G1Jac* partials) {
  pdl_prologue();
  TlScope tl_(7, buckets);
  for (u32 q = blockIdx.x * blockDim.x + threadIdx.x; q < n_chunks; q += gridDim.x * blockDim.x) {  // grid-stride, see k_transcript
    const u32 b0 = q * g.m, bl = b0 % g.nb();  // bl: inside its fold group
    const u32 ch = bl >= g.bbase[1] ? 1u : 0u;
    const u32 i0 = (bl - g.bbase[ch]) % g.B[ch];  // index of the chunk's first bucket inside its window
    G1Jac run = G1Jac::identity(), acc = G1Jac::identity();
    for (u32 i = g.m; i-- > 0;) {
      run = g1_add(run, buckets[b0 + i]);
      acc = g1_add(acc, run);
    }
    if (i0) acc = g1_add(acc, g1_mul_small(run, i0));
    partials[q] = acc;
  }
}

__global__ void __launch_bounds__(128) k_msm_window_reduce(MsmGeom g, const G1Jac* partials, G1Jac* window_sums) {
  pdl_prologue();
  TlScope tl_(8, window_sums);
  __shared__ G1Jac sh[128];
  const u32 Wt = g.W[0] + g.W[1];
  const u32 grp = blockIdx.x / Wt, wi = blockIdx.x % Wt, t = threadIdx.x;
  const u32 ch = wi >= g.wbase[1] ? 1u : 0u;
  const u32 per = g.B[ch] / g.m;  // partials of this window
  const G1Jac* p = partials + (grp * g.nb() + g.bbase[ch] + (wi - g.wbase[ch]) * g.B[ch]) / g.m;
  G1Jac total = G1Jac::identity();
  for (u32 i = t; i < per; i += 128) total = g1_add(total, p[i]);
  sh[t] = total;
  __syncthreads();
  for (u32 d = 64; d > 0; d >>= 1) {
    if (t < d) sh[t] = g1_add(sh[t], sh[t + d]);
    __syncthreads();
  }
  if (t == 0) window_sums[blockIdx.x] = sh[0];
}

struct FoldArgs {
  u32 W[2], c[2], wbase[2];  // MSM geometry per channel
};

__device__ __forceinline__ void store_affine_bytes(const G1Affine& a, bool is_id, u8* out) {
  if (is_id) {
    for (int i = 0; i < 64; i++) out[i] = 0;
    return;
  }
  a.x.to_canonical().store_le(out);
  a.y.to_canonical().store_le(out + 32);
}

// Parity hook only (the verdict path never forms these points): explicit window combination
// acc = sum_w 2^(c w) S_w of each channel (serial chain of ~W*c doublings, thread per channel) and
// conversion to affine bytes, acc_bytes = L | R  (reference msm.rs:81-95 `eval` of both MSMs).
__global__ void __launch_bounds__(32) k_fold_accum(FoldArgs fa, const G1Jac* window_sums, u8* acc_bytes) {
  pdl_prologue();
  const int t = threadIdx.x;
  if (t >= 2) return;
  // channel order in window_sums: 0 = right, 1 = left
  G1Jac acc = G1Jac::identity();
  const G1Jac* wsum = window_sums + fa.wbase[t];
  for (u32 w = fa.W[t]; w-- > 0;) {
    for (u32 i = 0; i < fa.c[t]; i++) g1_double_inl(acc);
    acc = g1_add(acc, wsum[w]);
  }
  G1Affine a;
  const bool id = !g1_to_affine_inl(acc, a);
  store_affine_bytes(a, id, acc_bytes + 64 * (t == 0 ? 1 : 0));
}

// Partial window combination before the pairing: the windows of a channel are combined in runs of `run` consecutive
// windows, T_v = sum_{i < run} 2^(c i) S_(run v + i)  ((run - 1) c dependent doublings, thread per (fold group, run)), and
// the pairing check then pairs T_v with the prepared lines of [2^(c run v)] Q.  With run = 4 the line products of
// k_lines - the stage's dominant cost: shared-memory bound Fq12 products, one per (pair, Miller line) - drop by 4x for
// ~40 doublings of latency; the full combination (one point per channel) would put ~260 dependent doublings in front of
// the pairing, no combination costs 53 pairs x 102 lines.
struct GroupArgs {
  u32 W[2], c[2], wbase[2];  // window sums per channel (in)
  u32 P[2], pbase[2];        // pairs per channel (out)
  u32 run;
};
__global__ void __launch_bounds__(64) k_window_group(GroupArgs ga, u32 groups, const G1Jac* __restrict__ wsums, G1Jac* __restrict__ out) {
  pdl_prologue();
  const u32 np = ga.P[0] + ga.P[1];
  const u32 t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= groups * np) return;
  const u32 grp = t / np, p = t % np;
  const u32 ch = p >= ga.pbase[1] ? 1u : 0u, v = p - ga.pbase[ch];
  const G1Jac* ws = wsums + (size_t)grp * (ga.W[0] + ga.W[1]) + ga.wbase[ch];
  const u32 w0 = v * ga.run, w1 = w0 + ga.run < ga.W[ch] ? w0 + ga.run : ga.W[ch];
  G1Jac acc = ws[w1 - 1];
  for (u32 w = w1 - 1; w-- > w0;) {
    for (u32 i = 0; i < ga.c[ch]; i++) g1_double_inl(acc);
    acc = g1_add(acc, ws[w]);
  }
  out[t] = acc;
}

// ---- partial accumulators of a shard: header + the Jacobian window sums (Montgomery limbs)
struct PartialHeader {
  u32 magic, cbits, windows, n_pts, rsv[4];
};
static constexpr u32 H2V_PARTIAL_MAGIC = 0x50563248u;
static_assert(sizeof(PartialHeader) == 32 && sizeof(G1Jac) == 96, "partial layout");
static_assert(sizeof(PartialHeader) + 128 * sizeof(G1Jac) == H2V_PARTIAL_BYTES, "H2V_PARTIAL_BYTES");
static_assert(XCH_PARTIAL_BYTES == H2V_PARTIAL_BYTES, "exchange.cuh partial size");

__global__ void k_pack_partial(u32 cbits, u32 windows, u32 npts, const G1Jac* wsums, u8* out) {
  pdl_prologue();
  wsums += (size_t)blockIdx.y * npts;  // fold group blockIdx.y
  out += (size_t)blockIdx.y * H2V_PARTIAL_BYTES;
  const u32 t = blockIdx.x * blockDim.x + threadIdx.x;
  u32* o = (u32*)out;
  if (t < 8) {
    const u32 hdr[8] = {H2V_PARTIAL_MAGIC, cbits, windows, npts, 0, 0, 0, 0};
    o[t] = hdr[t];
  }
  const u32* src = (const u32*)wsums;
  for (u32 i = t; i < H2V_PARTIAL_BYTES / 4 - 8; i += gridDim.x * blockDim.x) o[8 + i] = i < npts * 24 ? src[i] : 0u;
}

// window-wise sum of the shards' partials (thread per window).  *err: bit 0 = a wait timed out, bit 1 = geometry mismatch
// (fold groups: block q sums group q; partial (rank, group) lives at partials + rank * rank_stride + group * H2V_PARTIAL_BYTES).
// Exchange mode (dyn != null, exchange.cuh): the partials sit in this rank's window, stored there by the peers' pack
// kernels over NVLink; thread r first waits for rank r's sequence number of this launch set.
__global__ void __launch_bounds__(128) k_sum_partials(u32 n_partials, u32 cbits, u32 windows, u32 npts, const u8* partials, size_t rank_stride, G1Jac* out,
                                                      u32* err, const XDyn* dyn, const u64* arrive) {
  const u32 wi = threadIdx.x;
  partials += (size_t)blockIdx.x * H2V_PARTIAL_BYTES;
  out += (size_t)blockIdx.x * npts;
  if (dyn) {  // block-uniform
    __shared__ u32 timed_out;
    if (wi == 0) timed_out = 0;
    __syncthreads();
    if (wi < n_partials && !spin_until_ge(arrive + wi, dyn->seq, dyn->timeout_ns)) atomicOr(&timed_out, 1u);
    __syncthreads();
    if (timed_out) {  // never sum half-delivered data: the host turns the flag into an error, the verdicts are void
      if (wi == 0) atomicOr(err, 1u);
      if (wi < npts) out[wi] = G1Jac::identity();
      return;
    }
  }
  if (wi < n_partials) {
    const PartialHeader* h = (const PartialHeader*)(partials + (size_t)wi * rank_stride);
    if (h->magic != H2V_PARTIAL_MAGIC || h->cbits != cbits || h->windows != windows || h->n_pts != npts) atomicOr(err, 2u);
  }
  if (wi >= npts) return;
  G1Jac acc = G1Jac::identity();
  for (u32 g = 0; g < n_partials; g++) {
    const G1Jac* pts = (const G1Jac*)(partials + (size_t)g * rank_stride + sizeof(PartialHeader));
    acc = g1_add(acc, pts[wi]);
  }
  out[wi] = acc;
}

// ---- per-proof accumulators (parity hook, rejection attribution)
// thread per (base, proof): unscaled scalar * point, plain double-and-add
// (gverdict != null: proofs of fold groups whose batch check accepted are skipped; gsize = proofs per group)
__global__ void __launch_bounds__(128) k_pp_mul(PlanView pv, u32 n, const G1Affine* pts, const Fr* right, const Fr* shared, const Fr* left,
                                                const u32* status, G1Jac* out, const u32* gverdict, u32 gsize) {
  const PlanHeader& hd = pv.h();
  const u32 nP = msm_points(hd), nM = msm_mo(hd);
  const u32 nb = nP + hd.n_shared + nM;
  const u32 t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= nb * n) return;
  const u32 j = t % n, b = t / n;
  G1Jac r = G1Jac::identity();
  if ((status[j] == ST_OK || status[j] == ST_CONSTRAINT_SYSTEM_FAILURE) && !(gverdict && gverdict[j / gsize])) {
    Fr k;
    const G1Affine* p;
    if (b < nP) {
      k = right[(size_t)b * n + j];
      p = &pts[(size_t)b * n + j];
    } else if (b < nP + hd.n_shared) {
      k = shared[(size_t)(b - nP) * n + j];
      p = &pv.sec<G1Affine>(hd.off_shared_pts)[b - nP];
    } else {
      const u32 q = b - nP - hd.n_shared;
      k = left[(size_t)q * n + j];
      p = &pts[(size_t)(nP - nM + q) * n + j];
    }
    if (!k.is_zero() && !(p->x.is_zero() && p->y.is_zero())) {
      k = k.to_canonical();
      r = g1_mul_canonical(*p, k.l);
    }
  }
  out[t] = r;
}

// thread per (channel, proof): sum the per-base products; optional affine bytes out
__global__ void __launch_bounds__(128) k_pp_reduce(PlanView pv, u32 n, const G1Jac* prod, G1Jac* lr, u8* accum_bytes) {
  const PlanHeader& hd = pv.h();
  const u32 t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= 2 * n) return;
  const u32 j = t % n, ch = t / n;  // ch 0 = left, 1 = right
  G1Jac acc = G1Jac::identity();
  const u32 b0 = ch == 0 ? msm_points(hd) + hd.n_shared : 0;
  const u32 b1 = ch == 0 ? msm_points(hd) + hd.n_shared + msm_mo(hd) : msm_points(hd) + hd.n_shared;
  for (u32 b = b0; b < b1; b++) acc = g1_add(acc, prod[(size_t)b * n + j]);
  lr[(size_t)ch * n + j] = acc;
  if (accum_bytes) {
    G1Affine a;
    const bool id = !g1_to_affine(acc, a);
    store_affine_bytes(a, id, accum_bytes + (size_t)j * 128 + 64 * ch);
  }
}

// ---- attribution of a rejected fold (reference contract poly/strategy.rs:26-30: "re-process the proofs separately")
// Level 1 re-folds the rejected group in sub-batches of ATTR_SUB proofs through the bucket MSM (the fold restarts inside
// every sub-batch, so each is an AccumulatorStrategy run of its own, with coefficients drawn for the attribution and
// independent of the batch's r_i) and checks every sub-batch with one 2-pair
// pairing; level 2 forms the accumulators of the proofs of rejected sub-batches only and checks each proof alone
// (SingleStrategy semantics, strategy.rs:164-176).  With 1 % bad proofs level 2 sees ~15 % of the batch.
static constexpr u32 ATTR_SUB = 16;

// explicit window combination of a sub-batch, acc = sum_w 2^(c w) S_w  (the batch path avoids this serial chain through
// bilinearity; here one pair per window and sub-batch would cost far more line products).  FOUR lanes per (sub-batch, channel):
// lane q combines its quarter of the windows and shifts it into place, top quarter 128 doublings + 6 additions instead of
// 132 + 33 for the whole chain; the quarters are added with shuffles.
__global__ void __launch_bounds__(64) k_window_combine(u32 groups, FoldArgs fa, const G1Jac* __restrict__ wsums, G1Jac* __restrict__ pairs) {
  TlScope tl_(11, wsums);
  const u32 t = blockIdx.x * blockDim.x + threadIdx.x, item = t >> 2, q = t & 3;
  const bool live = item < 2 * groups;  // no early exit: every lane takes part in the shuffles
  G1Jac acc = G1Jac::identity();
  if (live) {
    const u32 grp = item >> 1, ch = item & 1;  // ch 0 = right, 1 = left: the pair order of the unit lines
    const G1Jac* ws = wsums + (size_t)grp * (fa.W[0] + fa.W[1]) + fa.wbase[ch];
    const u32 W = fa.W[ch], per = (W + 3) / 4, w0 = q * per < W ? q * per : W, w1 = w0 + per < W ? w0 + per : W;
    for (u32 w = w1; w-- > w0;) {
      for (u32 i = 0; i < fa.c[ch]; i++) g1_double_inl(acc);
      acc = g1_add(acc, ws[w]);
    }
    for (u32 i = 0; i < w0 * fa.c[ch]; i++) g1_double_inl(acc);
  }
  acc = g1_add(acc, shfl_down_jac(acc, 2));
  acc = g1_add(acc, shfl_down_jac(acc, 1));
  if (live && q == 0) pairs[item] = acc;
}

// suspects [base, base + cap) of the compacted list are processed per pass
__device__ __forceinline__ u32 chunk_count(u32 count, u32 base, u32 cap) { return count > base ? (count - base < cap ? count - base : cap) : 0u; }

// suspects = proofs that passed every earlier stage and sit in a rejected sub-batch (sub_verdict == null: in a rejected
// fold group; gverdict == null too: every proof): compacted list + count
__global__ void __launch_bounds__(128) k_pp_suspects(u32 n, const u32* status, const u32* sub_verdict, u32 sub_size, const u32* gverdict, u32 gsize,
                                                     u32* list, u32* count) {
  const u32 j = blockIdx.x * blockDim.x + threadIdx.x;
  if (j >= n) return;
  if (status[j] != ST_OK) return;
  if (gverdict && gverdict[j / gsize]) return;
  if (sub_verdict && sub_verdict[j / sub_size]) return;
  list[atomicAdd(count, 1u)] = j;
}

// FOUR lanes per (base, suspect): unscaled scalar * point through the GLV decomposition (glv.cuh), lane q walks half of the
// bits of one 128-bit half (129 dependent doublings instead of 254), the four summands are added with warp shuffles
// -> prod[base][slot]
__global__ void __launch_bounds__(128) k_pp_mul_list(PlanView pv, u32 n, const G1Affine* pts, const Fr* right, const Fr* shared, const Fr* left,
                                                     const u32* list, const u32* count, u32 base, u32 cap, G1Jac* out) {
  TlScope tl_(12, out);
  const PlanHeader& hd = pv.h();
  const u32 nP = msm_points(hd), nM = msm_mo(hd);
  const u32 nb = nP + hd.n_shared + nM;
  const u32 t = blockIdx.x * blockDim.x + threadIdx.x;
  const u32 cnt = chunk_count(*count, base, cap);
  const u32 item = t >> 2, q = t & 3;  // item = (base, suspect); no early exit: all lanes take part in the shuffles
  const bool live = item < nb * cnt;
  G1Jac r = G1Jac::identity();
  u32 slot = 0, b = 0;
  if (live) {
    slot = item % cnt;
    b = item / cnt;
    const u32 j = list[base + slot];
    Fr k;
    const G1Affine* p;
    if (b < nP) {
      k = right[(size_t)b * n + j];
      p = &pts[(size_t)b * n + j];
    } else if (b < nP + hd.n_shared) {
      k = shared[(size_t)(b - nP) * n + j];
      p = &pv.sec<G1Affine>(hd.off_shared_pts)[b - nP];
    } else {
      const u32 qq = b - nP - hd.n_shared;
      k = left[(size_t)qq * n + j];
      p = &pts[(size_t)(nP - nM + qq) * n + j];
    }
    if (!k.is_zero() && !(p->x.is_zero() && p->y.is_zero())) {
      k = k.to_canonical();
      GlvHalf h1, h2;
      glv_decompose(k.l, h1, h2);
      const bool endo = (q & 1) != 0, top = (q >> 1) != 0;
      r = g1_mul_glv_part(*p, endo ? h2 : h1, endo, top ? 64u : 0u, top ? 65u : 64u, top ? 64u : 0u);
    }
  }
  r = g1_add(r, shfl_down_jac(r, 2));
  r = g1_add(r, shfl_down_jac(r, 1));
  if (live && q == 0) out[(size_t)b * cap + slot] = r;
}

// thread per (channel, suspect): sum of the per-base products -> pairs[slot][0] = R_j, pairs[slot][1] = L_j
__global__ void __launch_bounds__(128) k_pp_reduce_list(PlanView pv, const u32* count, u32 base, u32 cap, const G1Jac* prod, G1Jac* pairs) {
  TlScope tl_(13, prod);
  const PlanHeader& hd = pv.h();
  const u32 t = blockIdx.x * blockDim.x + threadIdx.x;
  const u32 cnt = chunk_count(*count, base, cap);
  if (t >= 2 * cnt) return;
  const u32 slot = t >> 1, ch = t & 1;  // ch 0 = right, 1 = left
  G1Jac acc = G1Jac::identity();
  const u32 b0 = ch == 1 ? msm_points(hd) + hd.n_shared : 0;
  const u32 b1 = ch == 1 ? msm_points(hd) + hd.n_shared + msm_mo(hd) : msm_points(hd) + hd.n_shared;
  for (u32 b = b0; b < b1; b++) acc = g1_add(acc, prod[(size_t)b * cap + slot]);
  pairs[t] = acc;
}

// verdicts of the suspects' own checks -> statuses
__global__ void __launch_bounds__(128) k_pp_status(const u32* list, const u32* count, u32 base, u32 cap, const u32* verdict, u32* status) {
  const u32 t = blockIdx.x * blockDim.x + threadIdx.x;
  const u32 cnt = chunk_count(*count, base, cap);
  if (t >= cnt) return;
  if (!verdict[t]) status[list[base + t]] = ST_CONSTRAINT_SYSTEM_FAILURE;
}

// ---- persistent accumulators (acc.cuh): one block folds the window sums of a batch into the accumulator.
// acc[2] = (R, L) Jacobian; records[cap][2] = (R_b, L_b) of every absorb; *count = the next record slot, kept on the device
// so that a captured graph stays valid from one absorb to the next.  s = *r0 * *c0 = the product of the batch's r_i
// (r_1 times the coefficient c_1 = prod_{i>1} r_i that k_rlc_scan wrote).  Four lanes per item (acc_mul_lane), the items
// of a channel added by a tree in shared memory.
__global__ void __launch_bounds__(4 * ACC_MAX_ITEMS) k_acc_absorb(AccGeom ag, const G1Jac* __restrict__ wsums, const Fr* r0, const Fr* c0, G1Jac* acc,
                                                                  G1Jac* records, u32* count, u32 cap) {
  pdl_prologue();
  __shared__ G1Jac items[ACC_MAX_ITEMS];
  const u32 t = threadIdx.x, item = t >> 2, q = t & 3;
  const u32 slot = *count;
  const bool live = item < acc_items(ag);  // no early exit: every lane takes part in the shuffles
  G1Jac r = G1Jac::identity();
  if (live) {
    const Fr s = (*r0 * *c0).to_canonical();
    G1Jac base;
    Fr k;
    acc_item(ag, item, wsums, acc, s, base, k);
    r = acc_mul_lane(base, k, q);
  }
  r = g1_add(r, shfl_down_jac(r, 2));
  r = g1_add(r, shfl_down_jac(r, 1));
  if (live && q == 0) items[item] = r;
  __syncthreads();
  for (u32 d = ACC_TREE_SPAN / 2; d > 0; d >>= 1) {
    acc_tree_step(ag, items, t, d);
    __syncthreads();
  }
  if (slot >= cap) return;  // (the host refuses an absorb into a full record array)
  if (t < 2) {
    records[2 * (size_t)slot + t] = acc_batch_sum(ag, items, t);
    acc[t] = acc_new_value(ag, items, t);
  }
  if (t == 0) *count = slot + 1;
}

__global__ void k_gather_scalars(PlanView pv, u32 n, const Fr* right, const Fr* shared, const Fr* left, u8* out) {
  const PlanHeader& hd = pv.h();
  const u32 nP = msm_points(hd);
  const u32 nb = nP + hd.n_shared + msm_mo(hd);
  const u32 t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= nb * n) return;
  const u32 j = t % n, b = t / n;
  Fr k = b < nP ? right[(size_t)b * n + j] : b < nP + hd.n_shared ? shared[(size_t)(b - nP) * n + j] : left[(size_t)(b - nP - hd.n_shared) * n + j];
  k.to_canonical().store_le(out + ((size_t)j * nb + b) * 32);
}

__global__ void k_gather_challenges(PlanView pv, u32 n, const Fr* vals, u8* out) {
  const PlanHeader& hd = pv.h();
  const u32 t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= hd.n_challenges * n) return;
  const u32 j = t % n, c = t / n;
  vals[(size_t)(hd.v_chal + c) * n + j].to_canonical().store_le(out + ((size_t)j * hd.n_challenges + c) * 32);
}

// ---- self tests / calibration
template <class F>
__device__ u32 selftest_one(u64& s, bool edge) {
  F a, b;
  for (int i = 0; i < 8; i++) {
    s = s * 6364136223846793005ull + 1442695040888963407ull;
    a.l[i] = (u32)(s >> 32);
    s = s * 6364136223846793005ull + 1442695040888963407ull;
    b.l[i] = (u32)(s >> 32);
  }
  a.l[7] &= 0x1FFFFFFFu;  // < 2^253 < p
  b.l[7] &= 0x1FFFFFFFu;
  if (edge) {
    const u32 sel = (u32)(s >> 60);
    if (sel & 1) a = F::zero();
    if (sel & 2) {
      b = F::zero() - F::one();  // p - R mod p
    }
    if (sel & 4) {
      for (int i = 0; i < 8; i++) a.l[i] = 0xFFFFFFFFu;  // a may be any 256-bit value
    }
  }
  // mul_any accepts any 256-bit left operand; mul (even/odd wide form) is specified for a < 2^255
  F y = F::mul_portable(a, b);
  u32 bad = F::mul_any(a, b) != y;
  if (!(a.l[7] >> 31)) bad += F::mul(a, b) != y;
  F s1 = a.geq_mod() ? F::zero() : a;
  bad += s1.sqr() != F::mul_portable(s1, s1);  // dedicated squaring row schedule
  bad += b.sqr() != F::mul_portable(b, b);
  F u = s1 + b, v = u - b;
  bad += (v != s1);
  return bad;
}
__global__ void k_selftest_field(u32 count, u64 seed, u32* mismatches) {
  const u32 t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= count) return;
  u64 s = seed + 0x9E3779B97F4A7C15ull * (t + 1);
  u32 bad = selftest_one<Fq>(s, t % 7 == 0) + selftest_one<Fr>(s, t % 5 == 0);
  if (bad) atomicAdd(mismatches, bad);
}
// Known-answer vectors of the field operations (h2v_selftest_field_vectors): raw limbs in and out, no conversion, so that a
// test can place the operands anywhere in each operation's documented range.  op numbering: include/h2v.h.
template <class F>
__global__ void k_selftest_field_vectors(int op, u32 n, const u8* a, const u8* b, u8* out) {
  const u32 t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= n) return;
  const F x = F::load_le(a + 32 * (size_t)t), y = F::load_le(b + 32 * (size_t)t);
  F r = F::zero();
  switch (op) {
    case 0: r = F::mul(x, y); break;
    case 1: r = F::mul_c(x, y); break;
    case 2: r = x.sqr(); break;
    case 3: r = F::sqr_c(x); break;
    case 4: r = F::mul_any(x, y); break;
    case 5: r = x + y; break;
    case 6: r = x - y; break;
    case 7: r = x.neg(); break;
    case 8: r = F::from_canonical(x); break;
    case 9: r = x.to_canonical(); break;
    case 10: r = x.inv(); break;
    case 11: r = x.inv_bin(); break;
    case 12: {
      u8 w[64];
      x.store_le(w);
      y.store_le(w + 32);
      r = F::from_uniform(w);
      break;
    }
  }
  r.store_le(out + 32 * (size_t)t);
}
__global__ void k_imad(u32 iters, u32* out) {
  u32 a0 = threadIdx.x, a1 = a0 + 1, a2 = a0 + 2, a3 = a0 + 3, a4 = a0 + 4, a5 = a0 + 5, a6 = a0 + 6, a7 = a0 + 7;
  const u32 m = blockIdx.x * 2654435761u + 12345u, k = threadIdx.x | 1u;
  for (u32 i = 0; i < iters; i++) {
#pragma unroll
    for (int r = 0; r < 8; r++) {
      a0 = a0 * m + k; a1 = a1 * m + k; a2 = a2 * m + k; a3 = a3 * m + k;
      a4 = a4 * m + k; a5 = a5 * m + k; a6 = a6 * m + k; a7 = a7 * m + k;
    }
  }
  out[blockIdx.x * blockDim.x + threadIdx.x] = a0 ^ a1 ^ a2 ^ a3 ^ a4 ^ a5 ^ a6 ^ a7;
}

// ------------------------------------------------------------------------------------------------
// host side
// ------------------------------------------------------------------------------------------------
static thread_local std::string g_create_error;  // per host thread: contexts may be created concurrently

// Device buffers grow on demand.  Growth uses the stream-ordered allocator on the context's stream: cudaFree would wait
// for the whole device, i.e. also for another context's kernel that is waiting for a peer (exchange.cuh), which can close
// a cycle between two GPUs; cudaFreeAsync only orders after this context's own work.
struct DevBuf {
  void* p = nullptr;
  size_t cap = 0;
  cudaStream_t* st = nullptr;  // the owning context's stream (set at context creation)
  cudaError_t ensure(size_t bytes) {
    if (bytes <= cap) return cudaSuccess;
    if (p) {
      cudaError_t fe = st ? cudaFreeAsync(p, *st) : cudaFree(p);
      if (fe != cudaSuccess) return fe;
    }
    p = nullptr;
    cap = 0;
    size_t want = bytes + bytes / 4 + 256;
    cudaError_t e = st ? cudaMallocAsync(&p, want, *st) : cudaMalloc(&p, want);
    if (e == cudaSuccess) cap = want;
    return e;
  }
  void release() {
    if (p) {
      if (st) cudaFreeAsync(p, *st);
      else cudaFree(p);
    }
    p = nullptr;
    cap = 0;
  }
  template <class T>
  T* as() const {
    return (T*)p;
  }
};

// Pinned host staging for everything the library reads back on the data path (verdicts, statuses): a device-to-host copy
// into PAGEABLE memory keeps the calling thread inside the CUDA call until the stream reaches it - i.e., with the
// device-side exchange, until a peer rank delivered - and another thread's cudaStreamBeginCapture waits for that call
// (see ctx_sync).
struct HostBuf {
  void* p = nullptr;
  size_t cap = 0;
  cudaError_t ensure(size_t bytes) {
    if (bytes <= cap) return cudaSuccess;
    if (p) cudaFreeHost(p);
    p = nullptr;
    cap = 0;
    const size_t want = bytes + bytes / 4 + 256;
    cudaError_t e = cudaMallocHost(&p, want);
    if (e == cudaSuccess) cap = want;
    return e;
  }
  void release() {
    if (p) cudaFreeHost(p);
    p = nullptr;
    cap = 0;
  }
  template <class T>
  T* as() const {
    return (T*)p;
  }
};

// One slot of a CUDA-graph LRU (graph_lookup): the instantiated launch set of one key and the kernels it launches
struct GraphSlot {
  u64 key = 0, used = 0;
  u64 kernels = 0;
  cudaGraphExec_t exec = nullptr;
};

// LRU of prepared G2 window-line tables, one slot per (pair geometry, params classes) (ensure_lines): a service alternating
// batch shapes must not rebuild ~5,000 lines on the host at every call
struct LinesCache {
  struct Slot {
    u64 key = ~0ull, used = 0;
    DevBuf buf;
  } s[4];
  int cur = -1;  // a context's cache: the slot of its current batch's geometry
  u64 clock = 0;
};

struct h2v_ctx {
  int device = -1;  // -1 until a device was selected (h2v_ctx_destroy then frees host state only)
  cudaStream_t stream = nullptr;
  cudaStream_t stream_aux = nullptr;  // the fold-coefficient scan runs beside the per-proof stages
  cudaEvent_t ev_fork = nullptr, ev_join = nullptr, ev_done = nullptr;
  bool blocking_sync = false;
  std::vector<u8> blob;
  PlanInfo info{};
  PlanHeader hd{};
  std::string err;
  u64 launches = 0;
  cudaEvent_t ev[8]{};
  float timings[8]{};
  // options for the next batch
  const u32* opt_ncols = nullptr;
  const u32* opt_col_len = nullptr;
  u8* opt_scalar_hook = nullptr;
  // current batch
  u32 n = 0;
  u64 gbase = 0, gcount = 0;
  bool has_ncols = false, has_col_len = false;
  u32 scratch_rows = 0;
  MsmGeom geom{};
  bool ran = false;
  u32 opt_fold_groups = 0;  // next upload: that many consecutive independent fold groups (h2v_batch_set_fold_groups)
  std::vector<u32> h_verdicts;  // per fold group, of the last run (copied out of h_verd)
  bool verdicts_on_device = false;  // d_verdict holds the group verdicts of the batch in this context's buffers
  u32 opt_shard_hint = 0;   // geometry as for a shard of this many proofs (common to all ranks)
  bool opt_has_key = false;  // next upload: fold randomness expanded from this 256-bit key (h2v_batch_set_rlc_key)
  RlcKey opt_key{};
  u32 rlc_source = 0;  // of the last upload: 0 caller scalars, 1 test seed, 2 caller key, 3 key drawn from the OS
  bool opt_has_agg_scalar = false;  // next upload of an aggregation context: rho from the caller (h2v_batch_set_agg_scalar)
  Fr opt_agg_scalar{}, h_rho{};     // (Montgomery) the caller's rho; rho of the last upload, source of its copy to d_rho
  LinesCache lines;         // prepared G2 window lines, one slot per window geometry
  u64 lines_builds = 0;     // host rebuilds so far (h2v_ctx_cache_stats)
  // CUDA graphs: the ~20 kernels of a batch are captured once per (mode, shape, buffers) and replayed with one launch
  bool use_graphs = true;
  bool use_pdl = false;  // programmatic dependent launch between the kernels of a batch (pdl_prologue)
  bool capturing = false;
  bool stages_timed = false;  // ev[1..5] of the last run are valid (direct launches only)
  GraphSlot graphs[16];     // LRU over (entry point, batch shape, buffers): alternating shapes replay, never recapture
  u64 graph_clock = 0;
  u64 graph_captures = 0;   // captures so far (h2v_ctx_cache_stats)
  // accumulator of the absorb being enqueued (RUN_ABSORB, h2v_acc_absorb): its (R, L), records and record counter
  struct AbsorbTarget {
    G1Jac *acc = nullptr, *records = nullptr;
    u32* count = nullptr;
    u32 cap = 0;
  } absorb;
  // device-side exchange of sharded batches (exchange.cuh)
  struct Comm {
    bool ready = false;
    XLayout lay{};
    u8* window = nullptr;             // this context's window (cudaMalloc, exported through CUDA IPC)
    std::vector<u8*> peers;           // every rank's window as mapped here (own window at [rank])
    std::vector<void*> opened;        // cudaIpcOpenMemHandle mappings to close
    u8** d_peers = nullptr;
    XDyn* d_dyn = nullptr;
    u32* d_done = nullptr;
    XDyn* h_dyn = nullptr;            // pinned ring of per-launch parameters
    u32 ring = 0;
    u64 seq = 0;                      // launch sets run on this channel so far
    u64 timeout_ns = 30ull * 1000000000ull;
  } comm;
  // device buffers
  // buffers of one MSM run (k_shared_reduce .. k_msm_window_reduce): `mb` for the batch itself, `ab` for the regrouped MSM of the
  // attribution path (sub-batches of a rejected fold group, attribute_impl), which must not move the buffers the batch graph captured
  struct MsmBufs {
    DevBuf coef, shared_sum, dig, hist, off, cursor, order, sorted, buckets, wsums, partials_msm, tiles;
  } mb, ab;
  DevBuf d_plan, d_proofs, d_proof_off, d_inst, d_inst_off, d_ncols, d_col_len, d_pts, d_bad, d_status, d_vals, d_scratch, d_right,
      d_shared, d_left, d_rlc_bytes, d_r, d_acc_bytes, d_verdict, d_partials, d_pp_prod, d_pp_lr, d_pp_bytes, d_hook, d_chal, d_flush, d_M, d_partial_out,
      d_wsums_fin, d_sub_pairs, d_sub_verdict, d_sub_M, d_gsums, d_ptsc, d_rho, d_attr_r, d_attr_mask;
  // one-shot for the next attribute_impl (a grouped mixed batch): per proof of the upload, non-zero = its group accepted
  // (not re-checked); empty = every proof is looked at
  std::vector<u32> attr_accepted;
  const G2Line* d_lines() const { return lines.cur >= 0 ? lines.s[lines.cur].buf.as<G2Line>() : nullptr; }
  std::vector<DevBuf*> all_bufs() {
    std::vector<DevBuf*> v = {&d_plan, &d_proofs, &d_proof_off, &d_inst, &d_inst_off, &d_ncols, &d_col_len, &d_pts, &d_bad, &d_status, &d_vals, &d_scratch,
                              &d_right, &d_shared, &d_left, &d_rlc_bytes, &d_r, &d_acc_bytes, &d_verdict, &d_partials, &d_pp_prod, &d_pp_lr, &d_pp_bytes,
                              &d_hook, &d_chal, &d_flush, &d_M, &d_partial_out, &d_wsums_fin, &d_sub_pairs, &d_sub_verdict, &d_sub_M, &d_gsums, &d_ptsc, &d_rho,
                              &d_attr_r, &d_attr_mask, &lines.s[0].buf, &lines.s[1].buf, &lines.s[2].buf, &lines.s[3].buf};
    for (MsmBufs* m : {&mb, &ab})
      for (DevBuf* d : {&m->coef, &m->shared_sum, &m->dig, &m->hist, &m->off, &m->cursor, &m->order, &m->sorted, &m->buckets, &m->wsums, &m->partials_msm, &m->tiles})
        v.push_back(d);
    return v;
  }
  HostBuf h_status, h_verd;  // pinned staging of the per-proof statuses / the group verdicts + error words
  PlanView pv() const { return PlanView{d_plan.as<u8>()}; }
};

#define CKC(call)                                                                  \
  do {                                                                             \
    cudaError_t e_ = (call);                                                       \
    if (e_ != cudaSuccess) {                                                       \
      ctx->err = std::string(#call) + ": " + cudaGetErrorString(e_);               \
      return -2;                                                                   \
    }                                                                              \
  } while (0)
#define LAUNCH_CHECK()                       \
  do {                                       \
    ctx->launches++;                         \
    CKC(cudaGetLastError());                 \
  } while (0)

static inline u32 cdiv(u64 a, u32 b) { return (u32)((a + b - 1) / b); }

// NVTX ranges around the host side of every stage (header-only NVTX 3: a no-op unless a profiler is attached).  Under
// graph replay the stage ranges are seen at capture time; the replay itself shows as "h2v:launch_set".
struct NvtxRange {
  explicit NvtxRange(const char* name) { nvtxRangePushA(name); }
  ~NvtxRange() { nvtxRangePop(); }
};

// H2V_TRACE=1: host-side timestamps of the steps of a call on stderr (diagnosis of stalls between contexts)
static bool trace_on() {
  static const bool on = getenv("H2V_TRACE") != nullptr;
  return on;
}
static void trace(const h2v_ctx* ctx, const char* what) {
  if (!trace_on()) return;
  timespec ts;
  clock_gettime(CLOCK_MONOTONIC, &ts);
  fprintf(stderr, "[h2v %p %ld.%06ld] %s\n", (const void*)ctx, (long)(ts.tv_sec % 1000), ts.tv_nsec / 1000, what);
}

// Grid of a multiplier-bound kernel (k_decompress, k_msm_bucket_sum): at most H2V_WIDE_BLOCKS_PER_SM blocks per SM (0 = one
// block per 128 work items, the uncapped grid).  See the comment in k_decompress.
static u32 wide_grid(u64 items, u32 dflt_per_sm) {
  static const int sms = [] {
    int dev = 0, n = 148;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev);
    return n;
  }();
  static const int env = getenv("H2V_WIDE_BLOCKS_PER_SM") ? atoi(getenv("H2V_WIDE_BLOCKS_PER_SM")) : -1;
  const u32 per_sm = env >= 0 ? (u32)env : dflt_per_sm;
  const u32 full = cdiv(items, 128);
  return per_sm ? std::min<u32>(full, (u32)sms * per_sm) : full;
}

// H2V_WIDE_SPLIT = K > 1: a multiplier-bound kernel is launched as K consecutive grids (diagnosis of how kernels of
// several contexts interleave: the block scheduler serves the oldest grid first)
static u32 wide_split() {
  static const u32 k = [] {
    const char* e = getenv("H2V_WIDE_SPLIT");
    const int v = e ? atoi(e) : 1;
    return (u32)(v >= 1 && v <= 64 ? v : 1);
  }();
  return k;
}

// Grid of a latency-bound kernel over `units` blocks of work: H2V_NARROW_BLOCKS_PER_SM caps it (the kernels are grid-stride)
// so that, launched ahead of the multiplier-bound kernels (H2V_PRIO), it takes a slice of every SM instead of all of it.
static u32 narrow_grid(u64 units) {
  static const u32 cap = [] {
    const char* e = getenv("H2V_NARROW_BLOCKS_PER_SM");
    const int v = e ? atoi(e) : 0;
    return (u32)(v > 0 ? v * 148 : 0);
  }();
  const u32 u = (u32)std::min<u64>(units, 0x7FFFFFFFu);
  return cap ? std::min(u, cap) : u;
}

// rho of an aggregation context's upload: Blake2b-512("h2v-rla" | key[32]) mod r, or "h2v-rla" | seed_le64 for the test
// seed (the personalisation and reduction of the r_i, stages.cuh; its own tag keeps rho independent of every r_i)
static Fr agg_scalar(const RlcKey* key, u64 seed) {
  Blake2b b;
  b.init_halo2();
  const char* tag = "h2v-rla";
  for (int t = 0; t < 7; t++) b.update_byte((u8)tag[t]);
  if (key) {
    for (int t = 0; t < 32; t++) b.update_byte((u8)(key->w[t >> 2] >> (8 * (t & 3))));
  } else {
    for (int t = 0; t < 8; t++) b.update_byte((u8)(seed >> (8 * t)));
  }
  u8 d[64];
  b.digest(d);
  return Fr::from_uniform(d);
}

// `len` bytes from the kernel's CSPRNG; 0 on success
static int os_entropy(void* out, size_t len) {
  u8* p = (u8*)out;
  while (len) {
    const ssize_t got = getrandom(p, len, 0);
    if (got < 0) {
      if (errno == EINTR) continue;
      return -1;
    }
    p += got;
    len -= (size_t)got;
  }
  return 0;
}

// kernel launch with (pdl) or without the programmatic-stream-serialization attribute, and with an optional launch
// priority (H2V_PRIO, diagnosis: 0 = none; the latency-bound kernels of a launch set ahead of the multiplier-bound ones)
static int prio_mode() {
  static const int v = [] {
    const char* e = getenv("H2V_PRIO");
    return e ? atoi(e) : 0;
  }();
  return v;
}
static thread_local int tl_launch_prio = 0;  // 0 = no attribute; otherwise the priority value + 100
template <class... KArgs, class... Args>
static cudaError_t launch_k(bool pdl, void (*kern)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t st, Args&&... args) {
  cudaLaunchConfig_t cfg{};
  cfg.gridDim = grid;
  cfg.blockDim = block;
  cfg.dynamicSmemBytes = smem;
  cfg.stream = st;
  cudaLaunchAttribute at[2];
  unsigned na = 0;
  if (pdl) {
    at[na].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    at[na].val.programmaticStreamSerializationAllowed = 1;
    na++;
  }
  if (tl_launch_prio) {
    at[na].id = cudaLaunchAttributePriority;
    at[na].val.priority = tl_launch_prio - 100;
    na++;
  }
  cfg.attrs = at;
  cfg.numAttrs = na;
  return cudaLaunchKernelEx(&cfg, kern, std::forward<Args>(args)...);
}
// priority class of the launches that follow: 'W' = multiplier-bound (wide), 'M' = mid (transcript / scalar), 'N' = narrow
static void set_launch_class(char cls) {
  const int m = prio_mode();
  if (!m) return;
  static int lo = 0, hi = 0;
  static const bool init = [] { cudaDeviceGetStreamPriorityRange(&lo, &hi); return true; }();
  (void)init;
  int p = lo;  // lo = least priority (numerically largest)
  if (cls == 'N') p = hi;
  else if (cls == 'M') p = m == 1 ? hi : (m == 2 ? lo : (hi + lo) / 2);
  tl_launch_prio = p + 100;
}
#define KLAUNCH_P(pdl, kern, grid, block, smem, st, ...)                       \
  do {                                                                         \
    ctx->launches++;                                                           \
    CKC(launch_k(pdl, kern, grid, block, smem, st, __VA_ARGS__));              \
  } while (0)
#define KLAUNCH(kern, grid, block, smem, st, ...) KLAUNCH_P(ctx->use_pdl, kern, grid, block, smem, st, __VA_ARGS__)

// Host wait for everything queued on the context's stream.  Default: cudaStreamSynchronize (spins: lowest latency).
// With many contexts per host (several batches in flight on several GPUs) the spinning threads starve the cores, so
// a context can be switched to a blocking wait on an event (h2v_ctx_set_blocking_sync).
// (Everything the data path reads back lands in PINNED staging, HostBuf: a device-to-host copy into pageable memory
// keeps the caller inside the CUDA call until the stream gets there, and - measured on B200, tools/exchange_diag.py with
// H2V_TRACE - cudaStreamBeginCapture of another thread does not return while such a call is pending.  With the
// device-side exchange the stream may be waiting for a peer rank, so that stalled two contexts against each other.)
static cudaError_t ctx_sync(h2v_ctx* ctx) {
  if (!ctx->blocking_sync) return cudaStreamSynchronize(ctx->stream);
  cudaError_t e = cudaEventRecord(ctx->ev_done, ctx->stream);
  if (e != cudaSuccess) return e;
  return cudaEventSynchronize(ctx->ev_done);
}

// Graph keys: an FNV-style hash of what a captured launch set depends on (kept in memory only, never persisted)
struct KeyHash {
  u64 h = 0xcbf29ce484222325ull;
  void mix(u64 v) {
    h ^= v;
    h *= 0x100000001b3ull;
    h ^= h >> 29;
  }
};
// the window geometry: c / W / Z / Z2 per channel and the GLV split, terms and chunk, bucket sets and proofs
static void hash_geom(KeyHash& k, const MsmGeom& g) {
  for (int ch = 0; ch < 2; ch++) k.mix((u64)g.c[ch] | (u64)g.W[ch] << 8 | (u64)g.Z[ch] << 16 | (u64)g.Z2[ch] << 40 | (u64)g.glv << 63);
  k.mix((u64)g.T | (u64)g.m << 32);
  k.mix((u64)g.G | (u64)g.N << 32);
}

// The CUDA-graph LRU of a launch set: *out = the slot of `key`, captured from enqueue() on stream s (which may fork onto other
// streams) and instantiated on a miss.  During a capture every context of ctxs[0, n_ctxs) is marked capturing (no stage
// events) and gets its launch counter back afterwards: the slot counts the captured kernels, which the caller credits at each
// replay.  ctxs[0] reports the errors and counts the capture.
template <size_t N, class Enqueue>
static int graph_lookup(GraphSlot (&slots)[N], u64& clock, u64 key, h2v_ctx* const* ctxs, size_t n_ctxs, cudaStream_t s, Enqueue&& enqueue,
                        GraphSlot** out) {
  h2v_ctx* ctx = ctxs[0];
  clock++;
  GraphSlot* hit = nullptr;
  GraphSlot* victim = &slots[0];
  for (GraphSlot& sl : slots) {
    if (sl.exec && sl.key == key) hit = &sl;
    if (!sl.exec ? victim->exec != nullptr : (victim->exec && sl.used < victim->used)) victim = &sl;
  }
  GraphSlot& gs = hit ? *hit : *victim;
  gs.used = clock;
  *out = &gs;
  if (hit) return 0;
  trace(ctx, "graph capture begins");
  if (gs.exec) cudaGraphExecDestroy(gs.exec);
  gs.exec = nullptr;
  gs.key = 0;
  std::vector<u64> before(n_ctxs);
  for (size_t i = 0; i < n_ctxs; i++) before[i] = ctxs[i]->launches;
  CKC(cudaStreamBeginCapture(s, cudaStreamCaptureModeThreadLocal));
  for (size_t i = 0; i < n_ctxs; i++) ctxs[i]->capturing = true;
  const int rc = enqueue();
  for (size_t i = 0; i < n_ctxs; i++) ctxs[i]->capturing = false;
  cudaGraph_t graph = nullptr;
  const cudaError_t ce = cudaStreamEndCapture(s, &graph);
  gs.kernels = 0;
  for (size_t i = 0; i < n_ctxs; i++) {
    gs.kernels += ctxs[i]->launches - before[i];
    ctxs[i]->launches = before[i];
  }
  if (rc) {
    if (graph) cudaGraphDestroy(graph);
    return rc;
  }
  CKC(ce);
  const cudaError_t ie = cudaGraphInstantiate(&gs.exec, graph, prio_mode() ? cudaGraphInstantiateFlagUseNodePriority : 0);
  cudaGraphDestroy(graph);
  CKC(ie);
  gs.key = key;
  ctx->graph_captures++;
  trace(ctx, "graph instantiated");
  return 0;
}

// Windows of a lifted GLV geometry: W c >= 131, so that 2^(W c - 1) >= 2^130 leaves room for at least 7 lattice lifts of
// each half (glv_lift_ranges); with the bare minimum of 130 bits the top window of c = 13 stays 4x the mean load.
static u32 glv_windows(u32 c) { return (131 + c - 1) / c; }

// Window size per channel.  Thanks to the scalar lift k'' = k + z*r every window is uniformly filled, so
// the choice is a pure work trade-off: bucket additions (11 MM) against bucket reduction (2 x 16 MM
// per bucket plus the per-chunk offset multiplication), with a floor on the per-bucket serial chain.
// chain_weight: 1 = throughput (several fold groups share the launches: total work decides), 2 = latency (a single
// batch: the longest bucket chain is on the critical path).  Measured, 4096 VM proofs: c = 11 -> 5.91 M proofs/s and
// 3.08 ms alone, c = 12 -> 5.80 M and 2.92 ms.
// Returns the modelled time; chain_out = the chosen window's bucket chain.  glv: the terms are split into two lifted GLV halves
// (glv_lift): twice the entries per window, glv_windows(c) windows.
static double choose_window(u32 terms, bool glv, double chain_floor, double chain_weight, u32& c_out, u32& W_out, double& chain_out) {
  double best = 1e300;
  for (u32 c = 4; c <= 15; c++) {
    const u32 W = glv ? glv_windows(c) : (255 + c - 1) / c;
    const double B = (double)(1u << (c - 1));
    const double e = glv ? 2.0 * terms : (double)terms;  // entries per window
    const double work = (double)W * (e * 11.0 + B * 150.0);  // per bucket: measured (window sweep on B200), not just 2 additions
    const double chain = (e / B + 1.0) * 11.0;  // dependent MM per bucket thread
    // both channels share the bucket kernels: only a chain longer than the other channel's costs latency
    const double t = work / 10e9 + std::max(0.0, chain - chain_floor) * 0.4e-6 * chain_weight;
    if (t < best) {
      best = t;
      chain_out = chain;
      c_out = c;
      W_out = W;
    }
  }
  return best;
}

// Z = floor(2^(W*c-1) / r): k + z*r < 2^(W*c-1) for z < Z, so the top signed digit never carries out.
static u32 lift_range(u32 c, u32 W) {
  const int e = (int)(W * c) - 1 - 254;  // 2^(W*c-1) = 2^254 * 2^e, e in [0, 15]
  const long double ratio = 1.3225375138071345L;  // 2^254 / r
  u32 z = (u32)std::floor(ratio * (long double)(1u << e) * (1.0L - 1e-9L));
  return std::max(1u, z);
}

// n_geom >= n: the window geometry is chosen as for a batch of n_geom proofs (sharded batches: every
// rank must use the same windows so that partial window sums add up, see h2v_batch_set_shard_hint)
// window fields of g for right_terms / left_terms terms per channel and fold group (the batch size n_geom picks the chunk)
static void choose_windows(MsmGeom& g, u32 right_terms, u32 left_terms, u32 n_geom, u32 groups, u32 force_c, bool glv_ok = false) {
  const double cw = groups > 1 ? 1.0 : 2.0;
  double chain;
  double cost = choose_window(right_terms, false, 0.0, cw, g.c[0], g.W[0], chain);
  cost += choose_window(left_terms, false, chain, cw, g.c[1], g.W[1], chain);
  const char* f0 = getenv("H2V_MSM_WINDOW_RIGHT");
  const char* f1 = getenv("H2V_MSM_WINDOW_LEFT");
  const char* fg = getenv("H2V_MSM_GLV");
  g.glv = 0;
  if (glv_ok && !force_c && !f0 && !f1) {
    u32 c[2], W[2];
    double gcost = choose_window(right_terms, true, 0.0, cw, c[0], W[0], chain);
    gcost += choose_window(left_terms, true, chain, cw, c[1], W[1], chain);
    if (fg ? atoi(fg) == 1 : groups > 1 && gcost < cost) {
      g.glv = 1;
      for (int ch = 0; ch < 2; ch++) {
        g.c[ch] = c[ch];
        g.W[ch] = W[ch];
      }
    }
  }
  for (int ch = 0; ch < 2; ch++) {
    const char* f = ch == 0 ? f0 : f1;
    if (force_c) {  // attribution sub-batches: both channels with the same window size (one reduction chunk per window),
      g.c[ch] = force_c;  // GLV halves of 129 bits + the carry of the signed digits
      g.W[ch] = (130 + g.c[ch] - 1) / g.c[ch];
    } else if (f && atoi(f) >= 4 && atoi(f) <= 15) {
      g.c[ch] = (u32)atoi(f);
      g.W[ch] = (255 + g.c[ch] - 1) / g.c[ch];
    }
    g.B[ch] = 1u << (g.c[ch] - 1);
    g.Z2[ch] = 0;
    if (g.glv) glv_lift_ranges(g.c[ch], g.W[ch], g.Z[ch], g.Z2[ch]);
    else g.Z[ch] = force_c ? 1u : lift_range(g.c[ch], g.W[ch]);
  }
  g.wbase[0] = 0;
  g.wbase[1] = g.W[0];
  g.bbase[0] = 0;
  g.bbase[1] = g.W[0] * g.B[0];
  g.Wmax = std::max(g.W[0], g.W[1]);
  // buckets per reduction chunk (every B is a power of two >= 8): 8 for launch sets of several fold groups (least work), 4 for a
  // single batch, where the chunk kernel is a latency chain (measured alone: chunk + window reduction 0.236 + 0.069 ms with 8,
  // 0.153 + 0.088 with 4, 0.169 + 0.124 with 2)
  g.m = (groups == 1 && n_geom <= 8192) ? 4 : 8;
  if (const char* fm = getenv("H2V_MSM_CHUNK")) {
    const int m = atoi(fm);
    if (m == 2 || m == 4 || m == 8) g.m = (u32)m;
  }
  if (force_c) g.glv = 1;
  if (force_c) g.m = g.B[0];  // the whole window is one chunk: its weighted sum IS the window sum (enqueue_msm skips the second step)
}
static MsmGeom choose_geom(u32 n, const PlanHeader& hd, u32 n_geom, u32 groups = 1, u32 force_c = 0) {
  MsmGeom g{};
  g.n = n;
  g.G = groups;
  g.N = n * groups;
  g.P = msm_points(hd);
  g.n_mo = msm_mo(hd);
  g.Sh = hd.n_shared;
  g.T = n * g.P + n * g.n_mo + hd.n_shared;
  if (n_geom < n) n_geom = n;
  // (a GLV split doubles the term ids: 2 G T must stay inside the 31 bits of a bucket entry, k_msm_scatter)
  choose_windows(g, n_geom * g.P + hd.n_shared, n_geom * g.n_mo, n_geom, groups, force_c, 2ull * g.T * groups < (1ull << 31));
  return g;
}

static constexpr int LINES_GROUPS = 8;

// Run length of the partial window combination (k_window_group).  Measured on B200 (4096-proof VM batches): one batch alone
// 2.57 ms with runs of 1 or 2, 2.62 with 4, 2.77 with 8 (the doubling chain sits on the critical path); 4 x 16 batches in
// flight 6.15 / 6.27 / 6.33 / 6.42 M proofs/s (the line products are throughput).  Hence 2 for a single batch, 8 for launch
// sets of several fold groups; H2V_LINE_RUN / H2V_LINE_RUN_GROUPS override (1 = pair every window).
static u32 line_run(u32 groups) {
  static const int e1 = getenv("H2V_LINE_RUN") ? atoi(getenv("H2V_LINE_RUN")) : 0;
  static const int eg = getenv("H2V_LINE_RUN_GROUPS") ? atoi(getenv("H2V_LINE_RUN_GROUPS")) : 0;
  const int v = groups > 1 ? (eg ? eg : e1 ? e1 : 8) : (e1 ? e1 : 2);
  return (u32)(v >= 1 && v <= 64 ? v : 2);
}
// the (channel, run) pairs the pairing check sees for the window geometry of g: c' = c * run, P = ceil(W / run)
static MsmGeom pair_geom_run(const MsmGeom& g, u32 run) {
  MsmGeom q{};
  for (int ch = 0; ch < 2; ch++) {
    q.c[ch] = g.c[ch] * run;
    q.W[ch] = (g.W[ch] + run - 1) / run;
  }
  q.wbase[1] = q.W[0];
  return q;
}
static MsmGeom pair_geom(const MsmGeom& g, u32 groups) { return pair_geom_run(g, line_run(groups)); }
static u64 lines_key_of(const MsmGeom& g) { return (u64)g.c[0] | (u64)g.W[0] << 12 | (u64)g.c[1] << 24 | (u64)g.W[1] << 36; }

// The slot of lc that holds the prepared Miller lines of [2^(c w)] Q for pair geometry q, one table per params class of
// `classes`, concatenated in that order.  key names q and the classes.  A miss prepares them on the host (G2Prepared-style),
// uploads them on ctx's stream and counts a build in ctx->lines_builds; slot `pinned` (-1: none) is never evicted.
static int ensure_lines(h2v_ctx* ctx, LinesCache& lc, u64 key, const MsmGeom& q, const std::vector<const PlanInfo*>& classes, int pinned, int* slot_out) {
  lc.clock++;
  int victim = -1;
  for (int i = 0; i < 4; i++) {
    if (lc.s[i].key == key) {
      lc.s[i].used = lc.clock;
      *slot_out = i;
      return 0;
    }
    if (i == pinned) continue;
    if (victim < 0 || lc.s[i].used < lc.s[victim].used) victim = i;
  }
  if (classes.size() * (q.W[0] + q.W[1]) > 128) {
    ctx->err = "window geometry exceeds 128 (channel, window) pairs";
    return -1;
  }
  std::vector<u8> tab, one;
  for (const PlanInfo* info : classes) {
    build_window_lines(*info, q.c[0], q.W[0], q.c[1], q.W[1], one);
    tab.insert(tab.end(), one.begin(), one.end());
  }
  LinesCache::Slot& sl = lc.s[victim];
  CKC(ctx_sync(ctx));  // the victim's lines may still be read by queued work
  sl.key = ~0ull;
  CKC(sl.buf.ensure(tab.size()));
  CKC(cudaMemcpyAsync(sl.buf.p, tab.data(), tab.size(), cudaMemcpyHostToDevice, ctx->stream));
  CKC(ctx_sync(ctx));
  sl.key = key;
  sl.used = lc.clock;
  *slot_out = victim;
  ctx->lines_builds++;
  return 0;
}
// lines of pair geometry q from ctx's own params and cache; an auxiliary geometry (slot_out not the batch's own slot) never
// evicts the batch's geometry
static int ensure_lines(h2v_ctx* ctx, const MsmGeom& q, int* slot_out) {
  LinesCache& lc = ctx->lines;
  return ensure_lines(ctx, lc, lines_key_of(q), q, {&ctx->info}, slot_out == &lc.cur ? -1 : lc.cur, slot_out);
}
static int ensure_lines(h2v_ctx* ctx, u32 groups) { return ensure_lines(ctx, pair_geom(ctx->geom, groups), &ctx->lines.cur); }

// the batch pairing check over `wsums` (W0 + W1 Jacobian window sums per bucket set, window geometry g) -> d_verdict[group].
// Each of the `groups` checks pairs `sets` consecutive bucket sets (a multi-params mix: one per params class, 1 otherwise)
// with the prepared lines of pair_geom_run(g, run), one table per set, set-major; run 0 = line_run(groups).
static int launch_pairing(h2v_ctx* ctx, const MsmGeom& g, const G2Line* lines, const G1Jac* wsums, u32 groups, u32 run = 0, u32 sets = 1) {
  if (!run) run = line_run(groups);
  const MsmGeom q = pair_geom_run(g, run);
  cudaStream_t s = ctx->stream;
  const PairSkip none{nullptr, nullptr, 1, 0};
  const u32 np = q.W[0] + q.W[1];
  const G1Jac* pairs = wsums;
  if (run > 1) {
    GroupArgs ga{{g.W[0], g.W[1]}, {g.c[0], g.c[1]}, {0, g.W[0]}, {q.W[0], q.W[1]}, {0, q.W[0]}, run};
    KLAUNCH(k_window_group, cdiv((u64)groups * sets * np, 64), 64, 0, s, ga, groups * sets, wsums, ctx->d_gsums.as<G1Jac>());
    pairs = ctx->d_gsums.as<G1Jac>();
  }
  KLAUNCH((k_lines<LINES_GROUPS>), dim3(H2V_ATE_ITERS, groups), 64 * LINES_GROUPS, k_lines_smem<LINES_GROUPS>(), s, LinesArgs{sets * np}, pairs, lines,
                                                                                       ctx->d_M.as<E12>(), none);
  // (parallel Miller segments on four blocks per group when the launch is small, pairing_cta.cuh)
  static const bool seg_off = getenv("H2V_MILLER_SEGMENTS_OFF") != nullptr;
  if (groups * MILLER_SEGS <= 148 && !seg_off) {
    E12* seg = ctx->d_M.as<E12>() + (size_t)groups * H2V_ATE_ITERS;  // behind the iteration products (d_M holds ATE_ITERS + MILLER_SEGS per group)
    KLAUNCH(k_miller_segments, dim3(MILLER_SEGS, groups), 128, 0, s, ctx->d_M.as<E12>(), seg);
    KLAUNCH(k_pairing_check<true>, groups, 128, 0, s, seg, ctx->d_verdict.as<u32>(), none);
  } else {
    KLAUNCH(k_pairing_check<false>, groups, 128, 0, s, ctx->d_M.as<E12>(), ctx->d_verdict.as<u32>(), none);
  }
  return 0;
}

// Attribution: `count` independent 2-pair checks e(pairs[i][1], [s]G2) e(pairs[i][0], -G2) == 1 (pairs: right | left accumulator,
// Jacobian) -> verdict[i]; groups for which sk says "skip" keep their verdict word.  M: E12[count][H2V_ATE_ITERS] scratch.
static int launch_pair_checks(h2v_ctx* ctx, const G1Jac* pairs, u32 count, const G2Line* unit_lines, E12* M, u32* verdict, PairSkip sk) {
  cudaStream_t s = ctx->stream;
  KLAUNCH_P(false, (k_lines<2>), dim3(H2V_ATE_ITERS, count), 128, k_lines_smem<2>(), s, LinesArgs{2}, pairs, unit_lines, M, sk);
  KLAUNCH_P(false, k_pairing_check<false>, count, 128, 0, s, M, verdict, sk);
  return 0;
}

// verdicts of all fold groups of the last run -> ctx->h_verdicts; *all = every group accepted (waits for the stream).
// xchg: the run went through the device-side exchange; its two error words follow the verdicts.
// groups != 0: that many verdict words instead of the context's fold groups (a mixed batch's one check on its lead)
static int read_verdicts(h2v_ctx* ctx, u32* all, bool xchg = false, u32 groups = 0) {
  const u32 G = groups ? groups : ctx->geom.G ? ctx->geom.G : 1;
  CKC(ctx->h_verd.ensure(4 * (size_t)(G + 2)));
  u32* hv = ctx->h_verd.as<u32>();
  hv[G] = hv[G + 1] = 0;
  CKC(cudaMemcpyAsync(hv, ctx->d_verdict.p, 4 * (size_t)(G + (xchg ? 2 : 0)), cudaMemcpyDeviceToHost, ctx->stream));
  CKC(ctx_sync(ctx));
  ctx->h_verdicts.assign(hv, hv + G + 2);
  const u32 e_local = ctx->h_verdicts[G], e_root = ctx->h_verdicts[G + 1];
  ctx->h_verdicts.resize(G);
  if (xchg && ((e_local | e_root) & 5)) {
    ctx->err = std::string("sharded exchange timed out: ") +
               ((e_local & 1) ? "this rank is the root and a peer's partial accumulators never arrived"
                : (e_root & 1) ? "the root reports that a peer's partial accumulators never arrived"
                               : "the root's verdicts never arrived") +
               " (a rank died, or the ranks disagree on the launch-set order of this channel)";
    return -3;
  }
  if (xchg && ((e_local | e_root) & 2)) {
    ctx->err = "partial accumulators were produced with different window geometries (use h2v_batch_set_shard_hint)";
    return -1;
  }
  u32 a = 1;
  for (u32 v : ctx->h_verdicts) a &= v ? 1u : 0u;
  *all = a;
  return 0;
}

// CUDA loads kernels lazily, and loading one may wait for the device to drain.  With the device-side exchange a context
// can sit in a kernel that waits for a PEER (exchange.cuh) while another context of this process launches a kernel for
// the first time: that load would wait for the waiting kernel, whose peer may be stuck the same way on its side.  So
// every kernel of the library is loaded when a context is created (querying a function's attributes loads it).
static cudaError_t preload_kernels() {
  cudaFuncAttributes fa;
  cudaError_t e = cudaSuccess;
#define H2V_PRELOAD(k) \
  if (e == cudaSuccess) e = cudaFuncGetAttributes(&fa, k)
  H2V_PRELOAD(k_init);
  H2V_PRELOAD(k_decompress);
  H2V_PRELOAD(k_transcript<Blake2b>);
  H2V_PRELOAD(k_transcript<Keccak256>);
  H2V_PRELOAD(k_transcript_quad);
  H2V_PRELOAD(k_scalar<H2V_SCALAR_MINB>);
  H2V_PRELOAD(k_scalar<12>);
  H2V_PRELOAD(k_rlc_expand);
  H2V_PRELOAD(k_rlc_scan);
  H2V_PRELOAD(k_shared_reduce);
  H2V_PRELOAD(k_rlc_scan_groups);
  H2V_PRELOAD(k_shared_reduce_seg);
  H2V_PRELOAD(k_msm_digits<SingleVkTerms>);
  H2V_PRELOAD(k_msm_digits<MixTerms>);
  H2V_PRELOAD(k_scan_tiles);
  H2V_PRELOAD(k_scan_apply);
  H2V_PRELOAD(k_bucket_order);
  H2V_PRELOAD(k_msm_scatter<SingleVkTerms>);
  H2V_PRELOAD(k_msm_scatter<MixTerms>);
  H2V_PRELOAD((k_msm_bucket_sum<false, 1, SingleVkTerms>));
  H2V_PRELOAD((k_msm_bucket_sum<false, 2, SingleVkTerms>));
  H2V_PRELOAD((k_msm_bucket_sum<false, 4, SingleVkTerms>));
  H2V_PRELOAD((k_msm_bucket_sum<true, GLV_BUCKET_LANES, SingleVkTerms>));
  H2V_PRELOAD((k_msm_bucket_sum<true, 1, SingleVkTerms>));
  H2V_PRELOAD((k_msm_bucket_sum<false, 1, MixTerms>));
  H2V_PRELOAD((k_msm_bucket_sum<false, 2, MixTerms>));
  H2V_PRELOAD((k_msm_bucket_sum<false, 4, MixTerms>));
  H2V_PRELOAD(k_msm_chunk_reduce);
  H2V_PRELOAD(k_msm_window_reduce);
  H2V_PRELOAD(k_fold_accum);
  H2V_PRELOAD(k_window_group);
  H2V_PRELOAD(k_pack_partial);
  H2V_PRELOAD(k_sum_partials);
  H2V_PRELOAD(k_pp_mul);
  H2V_PRELOAD(k_pp_reduce);
  H2V_PRELOAD(k_window_combine);
  H2V_PRELOAD(k_pp_suspects);
  H2V_PRELOAD(k_pp_mul_list);
  H2V_PRELOAD(k_pp_reduce_list);
  H2V_PRELOAD(k_pp_status);
  H2V_PRELOAD(k_acc_absorb);
  H2V_PRELOAD(k_agg);
  H2V_PRELOAD(k_lines<2>);
  H2V_PRELOAD(k_gather_scalars);
  H2V_PRELOAD(k_gather_challenges);
  H2V_PRELOAD(k_lines<LINES_GROUPS>);
  H2V_PRELOAD(k_pairing_check<false>);
  H2V_PRELOAD(k_pairing_check<true>);
  H2V_PRELOAD(k_miller_segments);
  H2V_PRELOAD(k_pack_partial_x);
  H2V_PRELOAD(k_bcast_verdict);
  H2V_PRELOAD(k_wait_verdict);
#undef H2V_PRELOAD
  return e;
}

// ---- exchange windows (exchange.cuh): export / connect / release
struct CommHandle {  // H2V_COMM_HANDLE_BYTES, shipped between the ranks by the caller (plumbing: 128 bytes per context)
  u32 magic, rank, world, max_groups;
  u64 pid, ptr, bytes;
  int device, rsv;
  cudaIpcMemHandle_t ipc;
  u8 pad[H2V_COMM_HANDLE_BYTES - 48 - sizeof(cudaIpcMemHandle_t)];
};
static_assert(sizeof(CommHandle) == H2V_COMM_HANDLE_BYTES, "comm handle size");
static constexpr u32 H2V_COMM_MAGIC = 0x58563248u;
static constexpr u32 XDYN_RING = 64;

static void comm_release(h2v_ctx* ctx) {
  h2v_ctx::Comm& cm = ctx->comm;
  for (void* p : cm.opened) cudaIpcCloseMemHandle(p);
  cm.opened.clear();
  cm.peers.clear();
  if (cm.window) cudaFree(cm.window);
  if (cm.d_peers) cudaFree(cm.d_peers);
  if (cm.d_dyn) cudaFree(cm.d_dyn);
  if (cm.d_done) cudaFree(cm.d_done);
  if (cm.h_dyn) cudaFreeHost(cm.h_dyn);
  cm = h2v_ctx::Comm{};
}

extern "C" {

const char* h2v_last_error(const h2v_ctx* ctx) { return ctx ? ctx->err.c_str() : g_create_error.c_str(); }

int h2v_ctx_create(h2v_ctx** out, const uint8_t* params, size_t params_len, int params_format, const uint8_t* vk, size_t vk_len,
                   int vk_format, int multiopen, int hash, int device) {
  return h2v_ctx_create_multi(out, params, params_len, params_format, vk, vk_len, vk_format, multiopen, hash, device, 1);
}

}  // extern "C"

static int ctx_create(h2v_ctx** out, const uint8_t* params, size_t params_len, int params_format, const uint8_t* vk, size_t vk_len, int vk_format,
                      int multiopen, int hash, int device, uint32_t circuit_instances, const AggSpec* agg) {
  if (!out || !params || !vk) {
    g_create_error = "null argument";
    return -1;
  }
  h2v_ctx* ctx = new h2v_ctx();
  std::string err;
  if (build_plan(params, params_len, params_format, vk, vk_len, vk_format, multiopen, hash, ctx->blob, ctx->info, err, circuit_instances, agg) != 0) {
    g_create_error = err;
    h2v_ctx_destroy(ctx);
    return -1;
  }
  memcpy(&ctx->hd, ctx->blob.data(), sizeof(PlanHeader));
  int count = 0;
  cudaError_t e = cudaGetDeviceCount(&count);
  if (e != cudaSuccess || device < 0 || device >= count) {
    g_create_error = std::string("no usable CUDA device (this library has no CPU fallback): ") +
                     (e != cudaSuccess ? cudaGetErrorString(e) : "device index out of range");
    h2v_ctx_destroy(ctx);  // device still -1: nothing was created on a device
    return -2;
  }
  ctx->device = device;
  auto fail = [&](const char* what, cudaError_t ce) {
    g_create_error = std::string(what) + ": " + cudaGetErrorString(ce);
    h2v_ctx_destroy(ctx);  // frees whatever streams / events / buffers exist so far
    return -2;
  };
  if ((e = cudaSetDevice(device)) != cudaSuccess) return fail("cudaSetDevice", e);
  if ((e = cudaStreamCreateWithFlags(&ctx->stream, cudaStreamNonBlocking)) != cudaSuccess) return fail("cudaStreamCreate", e);
  for (DevBuf* b : ctx->all_bufs()) b->st = &ctx->stream;
  {  // keep freed blocks in the stream-ordered pool instead of returning them to the OS at every synchronisation
    cudaMemPool_t pool;
    uint64_t keep = ~0ull;
    if (cudaDeviceGetDefaultMemPool(&pool, device) == cudaSuccess) cudaMemPoolSetAttribute(pool, cudaMemPoolAttrReleaseThreshold, &keep);
    (void)cudaGetLastError();
  }
  if ((e = cudaStreamCreateWithFlags(&ctx->stream_aux, cudaStreamNonBlocking)) != cudaSuccess) return fail("cudaStreamCreate", e);
  if ((e = cudaEventCreateWithFlags(&ctx->ev_fork, cudaEventDisableTiming)) != cudaSuccess ||
      (e = cudaEventCreateWithFlags(&ctx->ev_join, cudaEventDisableTiming)) != cudaSuccess ||
      (e = cudaEventCreateWithFlags(&ctx->ev_done, cudaEventDisableTiming | cudaEventBlockingSync)) != cudaSuccess)
    return fail("cudaEventCreate", e);
  for (auto& ev : ctx->ev)
    if ((e = cudaEventCreate(&ev)) != cudaSuccess) return fail("cudaEventCreate", e);
  if ((e = ctx->d_plan.ensure(ctx->blob.size())) != cudaSuccess) return fail("cudaMalloc(plan)", e);
  if ((e = cudaMemcpyAsync(ctx->d_plan.p, ctx->blob.data(), ctx->blob.size(), cudaMemcpyHostToDevice, ctx->stream)) != cudaSuccess ||
      (e = cudaStreamSynchronize(ctx->stream)) != cudaSuccess)
    return fail("cudaMemcpy(plan)", e);
  if ((e = ctx->d_acc_bytes.ensure(128)) != cudaSuccess || (e = ctx->d_verdict.ensure(16)) != cudaSuccess) return fail("cudaMalloc", e);
  if (ctx->hd.n_carry && (e = ctx->d_rho.ensure(sizeof(Fr))) != cudaSuccess) return fail("cudaMalloc", e);
  if ((e = cudaFuncSetAttribute(k_lines<LINES_GROUPS>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)k_lines_smem<LINES_GROUPS>())) != cudaSuccess)
    return fail("cudaFuncSetAttribute(k_lines)", e);
  if ((e = preload_kernels()) != cudaSuccess) return fail("loading the kernels", e);
  *out = ctx;
  return 0;
}

extern "C" {

int h2v_ctx_create_multi(h2v_ctx** out, const uint8_t* params, size_t params_len, int params_format, const uint8_t* vk, size_t vk_len,
                         int vk_format, int multiopen, int hash, int device, uint32_t circuit_instances) {
  return ctx_create(out, params, params_len, params_format, vk, vk_len, vk_format, multiopen, hash, device, circuit_instances, nullptr);
}

int h2v_ctx_create_aggregation(h2v_ctx** out, const uint8_t* params, size_t params_len, int params_format, const uint8_t* vk, size_t vk_len,
                               int vk_format, int multiopen, int hash, int device, uint32_t circuit_instances, uint32_t limbs, uint32_t bits,
                               const uint32_t* cells) {
  const AggSpec spec{limbs, bits, cells};
  return ctx_create(out, params, params_len, params_format, vk, vk_len, vk_format, multiopen, hash, device, circuit_instances, &spec);
}

// Caller fold scalars (rlc_scalars, the r of h2v_acc_merge) must be canonical and non-zero: a zero r_i, or one that reduces
// to zero, makes c_j = prod_{i>j} r_i vanish for every earlier proof j, which then drops out of the batch check and out of
// the re-fold of its attribution sub-batch (an invalid proof would be accepted, or reported H2V_OK inside a rejected batch).
static const char* const FOLD_SCALARS_ERR = "fold scalars must be canonical and non-zero";
static bool fold_scalars_ok(const u8* r32, u64 count) {
  for (u64 i = 0; i < count; i++) {
    const Fr k = Fr::load_le(r32 + 32 * i);
    if (k.geq_mod() || k.is_zero()) return false;
  }
  return true;
}

int h2v_batch_set_agg_scalar(h2v_ctx* ctx, const uint8_t* rho32) {
  if (!ctx || !rho32) return -1;
  const Fr k = Fr::load_le(rho32);
  if (!ctx->hd.n_carry || k.geq_mod() || k.is_zero()) {
    ctx->err = ctx->hd.n_carry ? "the aggregation scalar must be canonical and non-zero" : "not an aggregation context";
    return -1;
  }
  ctx->opt_agg_scalar = Fr::from_canonical(k);
  ctx->opt_has_agg_scalar = true;
  return 0;
}

int h2v_ctx_create_from_bundle(h2v_ctx** out, const uint8_t* bundle, size_t bundle_len, int multiopen, int hash, int device) {
  // serialize/examples/vector_mul.rs:374-393: ParamsKZG::write (Processed, ParamsKZG::bytes_length() = 4 + 32 + 64 + 64
  // bytes, commitment.rs:209-213) immediately followed by VerifyingKey::write(RawBytes)
  const size_t plen = 4 + 32 + 64 + 64;
  if (!out || !bundle || bundle_len <= plen) {
    g_create_error = "bundle shorter than the verifier params";
    return -1;
  }
  return h2v_ctx_create(out, bundle, plen, H2V_FMT_PROCESSED, bundle + plen, bundle_len - plen, H2V_FMT_RAW_BYTES, multiopen, hash, device);
}

void h2v_ctx_destroy(h2v_ctx* ctx) {
  if (!ctx) return;
  if (ctx->device < 0) {  // failed before any device object existed
    delete ctx;
    return;
  }
  cudaSetDevice(ctx->device);
  if (ctx->stream) cudaStreamSynchronize(ctx->stream);
  if (ctx->stream_aux) cudaStreamSynchronize(ctx->stream_aux);
  comm_release(ctx);
  for (auto& gsl : ctx->graphs)
    if (gsl.exec) cudaGraphExecDestroy(gsl.exec);
  for (DevBuf* b : ctx->all_bufs()) b->release();
  ctx->h_status.release();
  ctx->h_verd.release();
  if (ctx->stream) cudaStreamSynchronize(ctx->stream);  // the stream-ordered frees
  for (auto& ev : ctx->ev)
    if (ev) cudaEventDestroy(ev);
  if (ctx->ev_fork) cudaEventDestroy(ctx->ev_fork);
  if (ctx->ev_join) cudaEventDestroy(ctx->ev_join);
  if (ctx->ev_done) cudaEventDestroy(ctx->ev_done);
  if (ctx->stream_aux) cudaStreamDestroy(ctx->stream_aux);
  if (ctx->stream) cudaStreamDestroy(ctx->stream);
  delete ctx;
}

int h2v_ctx_info(const h2v_ctx* ctx, uint32_t* out8) {
  if (!ctx || !out8) return -1;
  out8[0] = ctx->info.k;
  out8[1] = ctx->info.n_points;
  out8[2] = ctx->info.n_scalars;
  out8[3] = ctx->info.n_challenges;
  out8[4] = ctx->info.proof_len;
  out8[5] = ctx->info.n_inst_cols;
  out8[6] = ctx->info.n_shared;
  out8[7] = ctx->info.n_mo;
  return 0;
}

// Algorithmic work of scalar_stage (stages.cuh) for one proof of this plan, in Montgomery multiplications (a squaring
// counts as one): the same walk over the plan as the kernel, counting instead of multiplying.  Feeds the roofline of
// bench.py, so that the model follows the circuit instead of being fitted to one shape.
static double pow_cost(u64 e) {  // square-and-multiply, as Fp::pow_u64
  double c = 0;
  for (; e > 1; e >>= 1) c += 1 + (e & 1);
  return c;
}
static double scalar_stage_mm(const std::vector<u8>& blob, u32 rows) {
  PlanView pv{blob.data()};
  const PlanHeader& hd = pv.h();
  const RotSet* sets = pv.sec<RotSet>(hd.off_sets);
  auto poly = [&](u32 pid) {
    const PolyRange pr = pv.sec<PolyRange>(hd.off_polys)[pid];
    const PolyTerm* terms = pv.sec<PolyTerm>(hd.off_terms);
    const PolyVar* vars = pv.sec<PolyVar>(hd.off_vars);
    double c = 0;
    for (u32 t = pr.term_begin; t < pr.term_end; t++)
      for (u32 v = terms[t].var_begin; v < terms[t].var_end; v++) c += 1 + pow_cost(vars[v].pow);
    return c;
  };
  auto compress = [&](u32 b, u32 e) {
    const u32* list = pv.sec<u32>(hd.off_polylist);
    double c = 0;
    for (u32 i = b; i < e; i++) c += 1 + poly(list[i]);
    return c;
  };
  double mm = hd.k + 1;  // x^n, common
  if (hd.multiopen == MO_SHPLONK) mm += hd.n_rot + (sets[0].diff_end - sets[0].diff_begin);
  const u32 nl = hd.blinding + 2;
  const u32 li = hd.n_inst_q ? hd.inst_max_rot + rows + hd.inst_min_rot_abs : 0;
  mm += 3 + nl + pow_cost(hd.inst_max_rot) + 2.0 * li;  // prefix products
  // (the one inversion per proof runs as a binary Euclid on the ALU pipe, Fp::inv_bin: no Montgomery multiplications)
  mm += 5.0 * li + 2.0 * rows * hd.n_inst_q;            // instance Lagrange walk + inner products (from_canonical + multiply)
  mm += 4.0 * nl + 4;                                   // l_last / l_blind / l_0, the three unbatched inverses
  const ExprOp* eops = pv.sec<ExprOp>(hd.off_exprops);
  const LookupDesc* lks = pv.sec<LookupDesc>(hd.off_lookups);
  for (u32 o = 0; o < hd.n_exprops; o++) {
    const ExprOp& e = eops[o];
    switch (e.kind) {
      case E_GATE: mm += 1 + poly(e.a); break;
      case E_PERM_FIRST: mm += 2; break;
      case E_PERM_LAST: mm += 3; break;
      case E_PERM_LINK: mm += 2; break;
      case E_PERM_PROD: mm += 4.0 * (e.d - e.c) + 4; break;
      case E_LOOKUP: mm += 16 + compress(lks[e.a].in_begin, lks[e.a].in_end) + compress(lks[e.a].tab_begin, lks[e.a].tab_end); break;
      default: mm += 9 + compress(lks[e.a].in_begin, lks[e.a].in_end) + compress(lks[e.a].tab_begin, lks[e.a].tab_end); break;
    }
  }
  mm += 1;  // h / (x^n - 1)
  if (hd.multiopen == MO_SHPLONK) {
    const SetCommit* sc = pv.sec<SetCommit>(hd.off_setcms);
    for (u32 si = 0; si < hd.n_sets; si++) {
      const RotSet& S = sets[si];
      const u32 m = S.pt_end - S.pt_begin;
      mm += si == 0 ? m : (S.diff_end - S.diff_begin) + 1;
      mm += (m - 1) + (double)m * m + 1 + 1;  // x^-(m-1), Lagrange basis at u, coef_set, v power
      for (u32 c = S.cm_begin; c < S.cm_end; c++) mm += m + 3 + (sc[c].kind == CM_HMSM ? hd.n_h : 0);
    }
  } else {
    const GwcPoint* gp = pv.sec<GwcPoint>(hd.off_gwcpts);
    const GwcQuery* gq = pv.sec<GwcQuery>(hd.off_gwcq);
    for (u32 p = 0; p < hd.n_gwc_points; p++) {
      mm += 4;
      for (u32 q = gp[p].q_begin; q < gp[p].q_end; q++) mm += 3 + (gq[q].kind == CM_HMSM ? hd.n_h : 0);
    }
  }
  return mm;
}

extern "C" int h2v_ctx_work_model(const h2v_ctx* ctx, uint32_t instance_rows, double* out4) {
  if (!ctx || !out4) return -1;
  const PlanHeader& hd = ctx->hd;
  out4[0] = scalar_stage_mm(ctx->blob, instance_rows);                        // k_scalar
  out4[1] = 2.0 * hd.n_points + hd.n_scalars + 2.0 * hd.n_challenges;         // k_transcript: Montgomery conversions only (the hash is ALU work)
  out4[2] = 250 + 38 + 16 + 9;                                                // k_decompress per point: sqrt window chain + curve check + conversions
  out4[3] = (double)hd.n_inst_cols * instance_rows;                           // instance scalars per proof
  return 0;
}

int h2v_ctx_vk_lint(const h2v_ctx* ctx, char* report, size_t capacity) {
  if (!ctx) return -1;
  std::string all;
  for (const std::string& f : ctx->info.lint) all += f + "\n";
  if (report && capacity) {
    const size_t k = std::min(capacity - 1, all.size());
    memcpy(report, all.data(), k);
    report[k] = 0;
  }
  return (int)ctx->info.lint.size();
}

int h2v_batch_set_columns(h2v_ctx* ctx, const uint32_t* inst_ncols, const uint32_t* inst_col_len) {
  if (!ctx) return -1;
  ctx->opt_ncols = inst_ncols;
  ctx->opt_col_len = inst_col_len;
  return 0;
}
int h2v_batch_set_fold_groups(h2v_ctx* ctx, uint32_t groups) {
  if (!ctx) return -1;
  ctx->opt_fold_groups = groups;
  return 0;
}
int h2v_last_group_verdicts(const h2v_ctx* ctx, uint8_t* out, uint32_t capacity) {
  if (!ctx || !ctx->ran) return -1;
  const u32 G = (u32)ctx->h_verdicts.size();
  for (u32 i = 0; i < G && i < capacity; i++) out[i] = ctx->h_verdicts[i] ? 1 : 0;
  return (int)G;
}

int h2v_batch_set_rlc_key(h2v_ctx* ctx, const uint8_t* key32) {
  if (!ctx || !key32) return -1;
  memcpy(ctx->opt_key.w, key32, 32);
  ctx->opt_has_key = true;
  return 0;
}
int h2v_last_rlc_source(const h2v_ctx* ctx) { return ctx ? (int)ctx->rlc_source : -1; }

int h2v_batch_set_shard_hint(h2v_ctx* ctx, uint32_t max_shard_proofs) {
  if (!ctx) return -1;
  ctx->opt_shard_hint = max_shard_proofs;
  return 0;
}
size_t h2v_partial_bytes(void) { return H2V_PARTIAL_BYTES; }
int h2v_batch_set_scalar_hook(h2v_ctx* ctx, uint8_t* msm_scalars) {
  if (!ctx) return -1;
  ctx->opt_scalar_hook = msm_scalars;
  return 0;
}

// Column sums of the shared-base scalars of the current upload, shared_sum[grp][b] = sum_j c_j * shared[b][j] -> B.shared_sum.
static int enqueue_shared_reduce(h2v_ctx* ctx, const MsmGeom& g, h2v_ctx::MsmBufs& B, cudaStream_t s) {
  const PlanHeader& hd = ctx->hd;
  if (hd.n_shared)
    KLAUNCH(k_shared_reduce, dim3(hd.n_shared, g.G), 256, 0, s, g.n, g.N, (u32)hd.n_shared, ctx->d_shared.as<Fr>(), B.coef.as<Fr>(), B.shared_sum.as<Fr>());
  return 0;
}

// where the terms of a single-VK MSM live (a mixed batch passes nulls: its segment table points to the members' arrays)
struct TermArrays {
  const Fr *right, *left, *coef, *shared_sum;
  const G1Affine *pts, *shared_pts;
};

// The bucket MSM from the digits on: signed digits + histogram, bucket offsets, size-ordered buckets, counting sort,
// bucket sums, bucket reduction -> B.wsums[G][W0 + W1].  A zeroed B.hist must be ready on stream s.
// parent_verdict != null (attribution): group q of g is a sub-batch of fold group q * g.n / parent_size of the batch
// and is skipped (no bucket entries) when that group's batch check accepted.
extern "C++" {  // (inside the extern "C" block of the ABI)
template <class Src>
static int enqueue_buckets(h2v_ctx* ctx, const MsmGeom& g, h2v_ctx::MsmBufs& B, cudaStream_t s, const TermArrays& ta, Src src,
                           const u32* parent_verdict, u32 parent_size) {
  const u32 nb = g.nb() * g.G;
  const u64 terms = Src::mixed ? g.T : (u64)g.G * g.T;  // (a mix: g.T is every term, g.G its bucket sets)
  KLAUNCH(k_msm_digits<Src>, cdiv(terms, 128), 128, 0, s, g, ta.right, ta.left, ta.coef, ta.shared_sum, ta.shared_pts, B.dig.as<int16_t>(),
          B.hist.as<u32>(), parent_verdict, parent_size, src);
  const u32 n_tiles = cdiv(nb, SCAN_TILE);
  KLAUNCH(k_scan_tiles, n_tiles, SCAN_NT, 0, s, B.hist.as<u32>(), nb, B.off.as<u32>(), B.tiles.as<u32>(), B.hist.as<u32>() + nb);
  KLAUNCH(k_scan_apply, n_tiles, SCAN_NT, 0, s, nb, n_tiles, B.tiles.as<u32>(), B.off.as<u32>(), B.cursor.as<u32>());
  KLAUNCH(k_bucket_order, n_tiles, SCAN_NT, 0, s, nb, B.hist.as<u32>(), B.hist.as<u32>() + nb, B.hist.as<u32>() + nb + SIZE_BINS, B.order.as<u32>());
  KLAUNCH(k_msm_scatter<Src>, std::min<u32>(cdiv((terms << g.glv) * g.Wmax, 256), 148 * 16), 256, 0, s, g, B.dig.as<int16_t>(), B.cursor.as<u32>(),
          B.sorted.as<u32>(), src);
  {
    set_launch_class('W');
    // lanes per bucket: 1 for launch sets of several fold groups (throughput: no shuffle additions), 2 for a single batch and
    // for the attribution sub-batches (their bucket chains are latency)
    static const int lanes_env = getenv("H2V_BUCKET_LANES") ? atoi(getenv("H2V_BUCKET_LANES")) : 0;
    // (a lifted GLV geometry: one lane per bucket, as for the plain launch sets it replaces)
    const u32 lanes = g.lifted() ? 1u : g.glv ? GLV_BUCKET_LANES : (lanes_env ? (u32)lanes_env : (g.G == 1 && g.n <= 8192 ? 2u : 1u));
    void (*kern)(MsmGeom, u32, const u32*, const u32*, const u32*, const G1Affine*, const G1Affine*, G1Jac*, u32, u32, Src);
    kern = lanes == 2 ? k_msm_bucket_sum<false, 2, Src> : lanes == 4 ? k_msm_bucket_sum<false, 4, Src> : k_msm_bucket_sum<false, 1, Src>;
    if constexpr (!Src::mixed)  // (a mixed batch has no GLV split)
      if (g.glv) kern = g.lifted() ? k_msm_bucket_sum<true, 1, Src> : k_msm_bucket_sum<true, GLV_BUCKET_LANES, Src>;
    const u32 total = wide_grid((u64)(lanes == 2 || lanes == 4 || g.glv ? lanes : 1u) * nb, 0), K = std::min(wide_split(), total), per = cdiv(total, K);
    for (u32 off = 0; off < total; off += per)
      KLAUNCH(kern, std::min(per, total - off), 128, 0, s, g, nb, B.off.as<u32>(), B.order.as<u32>(), B.sorted.as<u32>(), ta.pts, ta.shared_pts,
              B.buckets.as<G1Jac>(), off, total, src);
  }
  set_launch_class('N');
  if (g.B[0] == g.m && g.B[1] == g.m) {
    // one chunk per window (the tiny windows of the attribution sub-batches): chunk q is window q, offset 0
    KLAUNCH(k_msm_chunk_reduce, narrow_grid(cdiv(nb / g.m, 128)), 128, 0, s, g, nb / g.m, B.buckets.as<G1Jac>(), B.wsums.as<G1Jac>());
  } else {
    KLAUNCH(k_msm_chunk_reduce, narrow_grid(cdiv(nb / g.m, 128)), 128, 0, s, g, nb / g.m, B.buckets.as<G1Jac>(), B.partials_msm.as<G1Jac>());
    KLAUNCH(k_msm_window_reduce, (g.W[0] + g.W[1]) * g.G, 128, 0, s, g, B.partials_msm.as<G1Jac>(), B.wsums.as<G1Jac>());
  }
  return 0;
}
}  // extern "C++"

// The MSM of G fold groups (geometry g) over the per-proof arrays of the current upload: column sums of the shared-base
// scalars, then the bucket MSM -> B.wsums[G][W0 + W1].  B.coef (the fold coefficients) and a zeroed B.hist must be ready on
// stream s.
static int enqueue_msm(h2v_ctx* ctx, const MsmGeom& g, h2v_ctx::MsmBufs& B, cudaStream_t s, const u32* parent_verdict, u32 parent_size) {
  int rc = enqueue_shared_reduce(ctx, g, B, s);
  if (rc) return rc;
  PlanView pv = ctx->pv();
  const G1Affine* shared_pts = g.lifted() ? ctx->d_pts.as<G1Affine>() + (size_t)g.P * g.N : pv.sec<G1Affine>(ctx->hd.off_shared_pts);  // (phi_rows)
  const TermArrays ta{ctx->d_right.as<Fr>(), ctx->d_left.as<Fr>(), B.coef.as<Fr>(), B.shared_sum.as<Fr>(), ctx->d_pts.as<G1Affine>(), shared_pts};
  return enqueue_buckets(ctx, g, B, s, ta, SingleVkTerms{}, parent_verdict, parent_size);
}

// mixed: g is a mix's geometry (g.T = every term of the mix, over all g.G bucket sets)
static cudaError_t ensure_msm_bufs(const MsmGeom& g, h2v_ctx::MsmBufs& B, u32 n_shared, bool mixed = false) {
  const size_t nb = (size_t)g.nb() * g.G, terms = mixed ? g.T : (size_t)g.G * g.T;
  cudaError_t e;
  if ((e = B.coef.ensure(32 * (size_t)g.N)) != cudaSuccess) return e;
  if ((e = B.shared_sum.ensure(32 * (size_t)n_shared * g.G + 32)) != cudaSuccess) return e;
  if ((e = B.dig.ensure(2 * (terms << g.glv) * g.Wmax)) != cudaSuccess) return e;
  if ((e = B.hist.ensure(4 * (nb + 2 * SIZE_BINS))) != cudaSuccess) return e;
  if ((e = B.order.ensure(4 * nb)) != cudaSuccess) return e;
  if ((e = B.off.ensure(4 * (nb + 1))) != cudaSuccess) return e;
  if ((e = B.cursor.ensure(4 * nb)) != cudaSuccess) return e;
  if ((e = B.tiles.ensure(4 * (nb / 1024 + 2))) != cudaSuccess) return e;
  if ((e = B.sorted.ensure(4 * (terms << g.glv) * g.Wmax)) != cudaSuccess) return e;
  if ((e = B.buckets.ensure(sizeof(G1Jac) * nb)) != cudaSuccess) return e;
  if ((e = B.wsums.ensure(sizeof(G1Jac) * (size_t)(g.W[0] + g.W[1]) * g.G)) != cudaSuccess) return e;
  return B.partials_msm.ensure(sizeof(G1Jac) * (nb / g.m));
}

// phi(P) rows of a lifted GLV geometry (k_decompress, k_agg write them; k_msm_bucket_sum<true, 1> reads them).  d_pts holds
// [points: msm_points * N | shared bases: n_shared | phi of the points | phi of the shared bases], so that phi of the base at
// d_pts[i] is d_pts[i + D], D = msm_points * N + n_shared, for proof points and shared bases alike: the MSM of a lifted
// geometry reads its shared bases from the copy.  Returns d_pts + D, null for other geometries.
static G1Affine* phi_rows(h2v_ctx* ctx) {
  return ctx->geom.lifted() ? ctx->d_pts.as<G1Affine>() + (size_t)ctx->geom.P * ctx->geom.N + ctx->geom.Sh : nullptr;
}

// Host ranges that make up a batch's proof bytes and instance bytes, in order (a member of a grouped mixed batch: its proofs
// of each group); null = the contiguous `proofs` / `instances`.
struct UploadPieces {
  std::vector<std::pair<const u8*, size_t>> proofs, instances;
};

static int upload_impl(h2v_ctx* ctx, u32 n, const u8* proofs, const u64* proof_off, const u8* instances, const u64* inst_off,
                       const u8* rlc, u64 seed, u64 gbase, u64 gcount, const UploadPieces* pieces = nullptr) {
  if (!ctx) return -1;
  NvtxRange nv_("h2v:upload");
  ctx->ran = false;
  const u32 groups = ctx->opt_fold_groups ? ctx->opt_fold_groups : 1;  // gbase / gcount describe ONE fold group (global batch)
  ctx->opt_fold_groups = 0;
  if (n == 0 || !proof_off || !inst_off || (!proofs && proof_off[n]) || groups > 1024 || n % groups != 0 || gcount < gbase + n / groups) {
    ctx->err = "bad batch arguments (with fold groups the batch must split into equal groups)";
    return -1;
  }
  if (rlc && !fold_scalars_ok(rlc, gcount * groups)) {  // every group's whole global batch
    ctx->err = FOLD_SCALARS_ERR;
    return -1;
  }
  CKC(cudaSetDevice(ctx->device));
  const PlanHeader& hd = ctx->hd;
  const size_t pbytes = proof_off[n] - proof_off[0], iscal = inst_off[n] - inst_off[0];
  if (proof_off[0] != 0 || inst_off[0] != 0 || (iscal && !instances)) {
    ctx->err = "offset arrays must start at 0";
    return -1;
  }
  // The offset arrays are caller data: a decreasing offset or an oversized proof would become an out-of-bounds device
  // read (the kernels index with 32-bit per-proof lengths), so they are validated here.
  for (u32 j = 0; j < n; j++) {
    if (proof_off[j + 1] < proof_off[j] || inst_off[j + 1] < inst_off[j] || proof_off[j + 1] - proof_off[j] > 0x7FFFFFFFull ||
        inst_off[j + 1] - inst_off[j] > 0x03FFFFFFull) {
      ctx->err = "offset arrays must be non-decreasing with per-proof sizes below 2^31 bytes / 2^26 scalars";
      return -1;
    }
  }
  {
    // 32-bit index spaces of the kernels: term ids carry the sign in bit 31 (k_msm_scatter), k_decompress indexes
    // (proof, point) pairs and the per-proof arrays with 32-bit products
    const u64 terms = (u64)n * (msm_points(hd) + msm_mo(hd)) + (u64)hd.n_shared * groups;
    const u64 widest = std::max<u64>(std::max<u64>(msm_points(hd), hd.n_vals), msm_points(hd) + hd.n_shared + msm_mo(hd));
    if (terms >= (1ull << 31) || (u64)n * widest >= (1ull << 32)) {
      ctx->err = "batch too large for the 32-bit index space of the MSM (split it into several uploads)";
      return -1;
    }
  }
  // scratch rows for the instance Lagrange range = max column length + rotation margins
  u32 max_len = 0;
  if (ctx->opt_col_len) {
    for (size_t i = 0; i < (size_t)n * hd.n_inst_cols; i++) max_len = std::max(max_len, ctx->opt_col_len[i]);
  } else if (hd.n_inst_cols) {
    for (u32 j = 0; j < n; j++) max_len = std::max<u32>(max_len, (u32)((inst_off[j + 1] - inst_off[j]) / hd.n_inst_cols));
  }
  ctx->scratch_rows = hd.inst_max_rot + max_len + hd.inst_min_rot_abs + 1;
  if ((u64)n * ctx->scratch_rows * 32 > (16ull << 30)) {  // instance columns longer than 2^k are rejected per proof; this bounds the allocation
    ctx->err = "instance columns too long for this batch size (Lagrange scratch would exceed 16 GiB)";
    return -1;
  }
  ctx->n = n;
  ctx->gbase = gbase;
  ctx->gcount = gcount;
  ctx->verdicts_on_device = false;
  ctx->geom = choose_geom(n / groups, hd, ctx->opt_shard_hint, groups);
  ctx->opt_shard_hint = 0;
  const MsmGeom& g = ctx->geom;
  const u32 nb = g.nb() * g.G;  // buckets of all fold groups
  {
    int lrc = ensure_lines(ctx, groups);
    if (lrc) return lrc;
  }
  trace(ctx, "lines ready");
  CKC(ctx->d_proofs.ensure(pbytes + 64));
  CKC(ctx->d_proof_off.ensure(8 * (size_t)(n + 1)));
  CKC(ctx->d_inst.ensure(32 * iscal + 64));
  CKC(ctx->d_inst_off.ensure(8 * (size_t)(n + 1)));
  // (a lifted GLV geometry: a copy of the shared bases and the phi rows after the points, phi_rows)
  CKC(ctx->d_pts.ensure(sizeof(G1Affine) * ((size_t)n * msm_points(hd) + (g.lifted() ? (size_t)n * msm_points(hd) + 2 * hd.n_shared : 0))));
  if (hd.hash == HASH_BLAKE2B) CKC(ctx->d_ptsc.ensure(64 * (size_t)n * hd.n_points));
  CKC(ctx->d_bad.ensure(4 * (size_t)n));
  CKC(ctx->d_status.ensure(4 * (size_t)n));
  CKC(ctx->d_vals.ensure(32 * (size_t)n * hd.n_vals));
  CKC(ctx->d_scratch.ensure(32 * (size_t)n * ctx->scratch_rows));
  CKC(ctx->d_right.ensure(32 * (size_t)n * msm_points(hd)));
  CKC(ctx->d_shared.ensure(32 * (size_t)n * hd.n_shared));
  CKC(ctx->d_left.ensure(32 * (size_t)n * msm_mo(hd)));
  CKC(ctx->d_r.ensure(32 * (size_t)gcount * groups));
  CKC(ctx->d_partial_out.ensure((size_t)H2V_PARTIAL_BYTES * groups));
  CKC(ctx->d_wsums_fin.ensure(sizeof(G1Jac) * 128 * (size_t)groups));
  CKC(ctx->d_gsums.ensure(sizeof(G1Jac) * 128 * (size_t)groups));
  CKC(ensure_msm_bufs(g, ctx->mb, hd.n_shared));
  CKC(ctx->d_M.ensure(sizeof(E12) * (H2V_ATE_ITERS + MILLER_SEGS) * (size_t)g.G));
  CKC(ctx->d_verdict.ensure(4 * (size_t)g.G + 16));
  cudaStream_t s = ctx->stream;
  if (pieces) {
    size_t o = 0;
    for (const auto& pc : pieces->proofs) {
      if (pc.second) CKC(cudaMemcpyAsync(ctx->d_proofs.as<u8>() + o, pc.first, pc.second, cudaMemcpyHostToDevice, s));
      o += pc.second;
    }
    o = 0;
    for (const auto& pc : pieces->instances) {
      if (pc.second) CKC(cudaMemcpyAsync(ctx->d_inst.as<u8>() + o, pc.first, pc.second, cudaMemcpyHostToDevice, s));
      o += pc.second;
    }
  } else {
    CKC(cudaMemcpyAsync(ctx->d_proofs.p, proofs, pbytes, cudaMemcpyHostToDevice, s));
    if (iscal) CKC(cudaMemcpyAsync(ctx->d_inst.p, instances, 32 * iscal, cudaMemcpyHostToDevice, s));
  }
  CKC(cudaMemcpyAsync(ctx->d_proof_off.p, proof_off, 8 * (size_t)(n + 1), cudaMemcpyHostToDevice, s));
  CKC(cudaMemcpyAsync(ctx->d_inst_off.p, inst_off, 8 * (size_t)(n + 1), cudaMemcpyHostToDevice, s));
  ctx->has_ncols = ctx->opt_ncols != nullptr;
  ctx->has_col_len = ctx->opt_col_len != nullptr && hd.n_inst_cols;
  if (ctx->has_ncols) {
    CKC(ctx->d_ncols.ensure(4 * (size_t)n));
    CKC(cudaMemcpyAsync(ctx->d_ncols.p, ctx->opt_ncols, 4 * (size_t)n, cudaMemcpyHostToDevice, s));
  }
  if (ctx->has_col_len) {
    CKC(ctx->d_col_len.ensure(4 * (size_t)n * hd.n_inst_cols));
    CKC(cudaMemcpyAsync(ctx->d_col_len.p, ctx->opt_col_len, 4 * (size_t)n * hd.n_inst_cols, cudaMemcpyHostToDevice, s));
  }
  ctx->opt_ncols = nullptr;
  ctx->opt_col_len = nullptr;
  const u64 n_r = gcount * groups;  // fold coefficients of every group's whole global batch
  if (rlc) {
    CKC(ctx->d_rlc_bytes.ensure(32 * (size_t)n_r));
    CKC(cudaMemcpyAsync(ctx->d_rlc_bytes.p, rlc, 32 * (size_t)n_r, cudaMemcpyHostToDevice, s));
  }
  // Fold randomness (reference strategy.rs:129 draws every r_i from the OS): explicit scalars and the 64-bit seed are
  // parity / test hooks; otherwise the r_i are expanded from a 256-bit secret key, the caller's (sharded batches: one
  // fresh key broadcast to every rank) or one drawn from the OS for this batch.
  RlcKey key{};
  bool keyed = false;
  if (rlc) {
    ctx->rlc_source = 0;
  } else if (ctx->opt_has_key) {
    key = ctx->opt_key;
    keyed = true;
    ctx->rlc_source = 2;
  } else if (seed != 0) {
    ctx->rlc_source = 1;
  } else {
    if (os_entropy(&key, sizeof(key)) != 0) {
      ctx->err = "no OS entropy for the fold coefficients (getrandom failed)";
      return -2;
    }
    keyed = true;
    ctx->rlc_source = 3;
  }
  ctx->opt_has_key = false;
  if (hd.n_carry) {  // rho of the carried accumulators (k_agg): one per upload, independent of the r_i (DESIGN.md section 6.3)
    if (!rlc) {
      ctx->h_rho = agg_scalar(keyed ? &key : nullptr, seed);
    } else if (ctx->opt_has_agg_scalar) {
      ctx->h_rho = ctx->opt_agg_scalar;
    } else {
      u8 wide[64];
      if (os_entropy(wide, sizeof(wide)) != 0) {
        ctx->err = "no OS entropy for the aggregation scalar (getrandom failed)";
        return -2;
      }
      ctx->h_rho = Fr::from_uniform(wide);
    }
    CKC(cudaMemcpyAsync(ctx->d_rho.p, &ctx->h_rho, sizeof(Fr), cudaMemcpyHostToDevice, s));
  }
  ctx->opt_has_agg_scalar = false;
  k_rlc_expand<<<cdiv(n_r, 128), 128, 0, s>>>(n_r, seed, rlc ? ctx->d_rlc_bytes.as<u8>() : nullptr, keyed, key, ctx->d_r.as<Fr>());
  LAUNCH_CHECK();
  trace(ctx, "upload enqueued");
  return 0;
}

// every kernel of the batch.  mode bits: RUN_PAIRING = batch pairing check -> d_verdict; RUN_ACCUM = explicit
// window combination -> affine (L, R) bytes in d_acc_bytes (parity hook); RUN_PARTIAL = pack the window
// sums into d_partial_out (sharded batches); RUN_ABSORB = fold the window sums into the accumulator ctx->absorb
enum : int { RUN_PAIRING = 1, RUN_ACCUM = 2, RUN_PARTIAL = 4, RUN_XCHG = 8, RUN_ROOT = 16, RUN_ABSORB = 32 };
// The per-proof stages of the current upload on the context's stream, up to the point where the MSM may start: fold
// coefficients (auxiliary stream), instance checks, decompression, transcript replay, scalar stage, and the wait for the
// coefficients.  Shared by a context's own batches (enqueue_batch) and the members of a mixed batch, whose coefficients the
// mix computes (own_coef = false: no scan and no histogram of the member's own MSM).
static int enqueue_stages(h2v_ctx* ctx, bool own_coef = true) {
  const PlanHeader& hd = ctx->hd;
  const u32 n = ctx->n;
  cudaStream_t s = ctx->stream;
  PlanView pv = ctx->pv();
  const MsmGeom& g = ctx->geom;
  const u32 nb = g.nb() * g.G;
  set_launch_class('N');
  if (!ctx->capturing) CKC(cudaEventRecord(ctx->ev[0], s));
  // c_j = prod_{i>j} r_i depends only on the coefficients: scanned on the auxiliary stream while the proofs are parsed
  if (own_coef) {
    CKC(cudaEventRecord(ctx->ev_fork, s));
    CKC(cudaStreamWaitEvent(ctx->stream_aux, ctx->ev_fork, 0));
    CKC(cudaMemsetAsync(ctx->mb.hist.p, 0, 4 * ((size_t)nb + 2 * SIZE_BINS), ctx->stream_aux));  // bucket histogram | size histogram | size cursors
    KLAUNCH_P(false, k_rlc_scan, g.G, RLC_NT, 0, ctx->stream_aux, ctx->d_r.as<Fr>(), ctx->gcount, ctx->gbase, g.n, ctx->mb.coef.as<Fr>(), 1u, ctx->gcount, (u64)0);
    CKC(cudaEventRecord(ctx->ev_join, ctx->stream_aux));
  }
  nvtxRangePushA("h2v:decompress");
  KLAUNCH(k_init, cdiv(n, 128), 128, 0, s, pv, n, ctx->d_inst_off.as<u64>(), ctx->has_ncols ? ctx->d_ncols.as<u32>() : nullptr,
                                      ctx->has_col_len ? ctx->d_col_len.as<u32>() : nullptr, ctx->d_status.as<u32>(), ctx->d_bad.as<u32>());
  // (one-warp blocks were measured for the two multiplier-bound kernels: no change, 0.300 ms / 0.364 ms alone.  A single
  // batch is 2.6 warps of decompression per SM sub-partition: the quantisation to 3 bounds the kernel at ~86 % of the pipe.)
  static const bool quad_off = getenv("H2V_TRANSCRIPT_THREAD") != nullptr;  // diagnosis: the thread-per-proof replay for Blake2b too
  const bool use_quad = hd.hash == HASH_BLAKE2B && !quad_off;
  {
    set_launch_class('W');
    const u32 total = wide_grid((u64)n * hd.n_points, 0), K = std::min(wide_split(), total), per = cdiv(total, K);
    for (u32 off = 0; off < total; off += per)
      KLAUNCH(k_decompress, std::min(per, total - off), 128, 0, s, pv, n, ctx->d_proofs.as<u8>(), ctx->d_proof_off.as<u64>(), ctx->d_pts.as<G1Affine>(),
              phi_rows(ctx), use_quad ? ctx->d_ptsc.as<u32>() : nullptr, ctx->d_bad.as<u32>(), off, total);
  }
  nvtxRangePop();
  if (!ctx->capturing) CKC(cudaEventRecord(ctx->ev[1], s));
  nvtxRangePushA("h2v:transcript");
  set_launch_class('M');
  if (use_quad)
    KLAUNCH(k_transcript_quad, narrow_grid(cdiv(n, TQ_PROOFS_PER_BLOCK)), 4 * TQ_PROOFS_PER_BLOCK, 0, s, pv, n, ctx->d_proofs.as<u8>(), ctx->d_proof_off.as<u64>(), ctx->d_inst.as<u8>(),
            ctx->d_inst_off.as<u64>(), ctx->d_ptsc.as<u32>(), ctx->d_vals.as<Fr>(), ctx->d_status.as<u32>(), ctx->d_bad.as<u32>());
  else if (hd.hash == HASH_BLAKE2B)
    KLAUNCH((k_transcript<Blake2b>), narrow_grid(cdiv(n, 64)), 64, 0, s, pv, n, ctx->d_proofs.as<u8>(), ctx->d_proof_off.as<u64>(), ctx->d_inst.as<u8>(),
                                                     ctx->d_inst_off.as<u64>(), ctx->d_pts.as<G1Affine>(), ctx->d_vals.as<Fr>(),
                                                     ctx->d_status.as<u32>(), ctx->d_bad.as<u32>());
  else
    KLAUNCH((k_transcript<Keccak256>), narrow_grid(cdiv(n, 64)), 64, 0, s, pv, n, ctx->d_proofs.as<u8>(), ctx->d_proof_off.as<u64>(), ctx->d_inst.as<u8>(),
                                                       ctx->d_inst_off.as<u64>(), ctx->d_pts.as<G1Affine>(), ctx->d_vals.as<Fr>(),
                                                       ctx->d_status.as<u32>(), ctx->d_bad.as<u32>());
  nvtxRangePop();
  if (!ctx->capturing) CKC(cudaEventRecord(ctx->ev[2], s));
  nvtxRangePushA("h2v:scalar");
  {
    // register cap of the scalar stage (see H2V_SCALAR_MINB): 80 registers = 24 warps per SM for launch sets of several fold
    // groups, uncapped for a single batch (64 blocks: the cap cannot add warps there)
    static const int cap = [] {
      const char* e = getenv("H2V_SCALAR_CAP");
      return e ? atoi(e) : 1;
    }();
    auto kern = (cap && n > 148 * 64) ? k_scalar<12> : k_scalar<H2V_SCALAR_MINB>;
    KLAUNCH(kern, narrow_grid(cdiv(n, 64)), 64, 0, s, pv, n, ctx->d_inst.as<u8>(), ctx->d_inst_off.as<u64>(),
            ctx->has_col_len ? ctx->d_col_len.as<u32>() : nullptr, ctx->d_vals.as<Fr>(), ctx->d_scratch.as<Fr>(), ctx->d_right.as<Fr>(),
            ctx->d_shared.as<Fr>(), ctx->d_left.as<Fr>(), ctx->d_status.as<u32>());
  }
  if (hd.n_carry)
    KLAUNCH(k_agg, cdiv(n, 128), 128, 0, s, pv, n, ctx->d_inst.as<u8>(), ctx->d_inst_off.as<u64>(), ctx->has_col_len ? ctx->d_col_len.as<u32>() : nullptr,
            ctx->d_rho.as<Fr>(), ctx->d_pts.as<G1Affine>(), phi_rows(ctx), ctx->d_right.as<Fr>(), ctx->d_shared.as<Fr>(), ctx->d_left.as<Fr>(), ctx->d_status.as<u32>());
  nvtxRangePop();
  set_launch_class('N');
  if (!ctx->capturing) CKC(cudaEventRecord(ctx->ev[3], s));
  if (own_coef) CKC(cudaStreamWaitEvent(s, ctx->ev_join, 0));
  return 0;
}

// k_fold_accum over `count` consecutive bucket sets of window sums (geometry g): one 128 B affine (L, R) per set at out
static int enqueue_fold_accum(h2v_ctx* ctx, const MsmGeom& g, const G1Jac* wsums, u32 count, u8* out, bool pdl) {
  const FoldArgs fa{{g.W[0], g.W[1]}, {g.c[0], g.c[1]}, {0, g.W[0]}};
  for (u32 st = 0; st < count; st++)
    KLAUNCH_P(pdl, k_fold_accum, 1, 32, 0, ctx->stream, fa, wsums + (size_t)st * (g.W[0] + g.W[1]), out + 128 * (size_t)st);
  return 0;
}

// What follows the MSM in a launch set: its window sums and how they are checked (enqueue_tail)
struct TailArgs {
  MsmGeom g;              // window geometry; g.G bucket sets
  G1Jac* wsums;           // [g.G][W0 + W1] window sums of the MSM
  const G2Line* lines;    // prepared lines of the pair geometry, one table per bucket set of a check
  u32 checks, sets, run;  // pairing checks, bucket sets per check, window-combination run (0 = line_run(checks))
  u8* partial;            // RUN_PARTIAL: one H2V_PARTIAL_BYTES blob per bucket set
};
// The kernels of a launch set after its MSM, on ctx's stream (ctx: the context, or the lead of a mixed batch), by the RUN_*
// mode bits: pairing checks -> d_verdict, packed partials, the device-side exchange over ctx's channel, the absorb into
// ctx->absorb (a context's own batch: its r_i and coefficients), the folded (L, R) of every bucket set -> d_acc_bytes.
// Stage events ev[4..6] unless capturing.
static int enqueue_tail(h2v_ctx* ctx, int mode, const TailArgs& t) {
  cudaStream_t s = ctx->stream;
  const MsmGeom& g = t.g;
  const u32 cb = g.c[0] | g.c[1] << 16, wd = g.W[0] | g.W[1] << 16, npts = g.W[0] + g.W[1];
  if (!ctx->capturing) CKC(cudaEventRecord(ctx->ev[4], s));
  if (mode & RUN_PAIRING) {
    NvtxRange nv_("h2v:pairing");
    int prc = launch_pairing(ctx, g, t.lines, t.wsums, t.checks, t.run, t.sets);
    if (prc) return prc;
  }
  if (mode & RUN_PARTIAL) KLAUNCH(k_pack_partial, dim3(8, g.G), 256, 0, s, cb, wd, npts, t.wsums, t.partial);
  if (mode & RUN_XCHG) {
    NvtxRange nv_("h2v:exchange");
    // The one exchange step of a sharded batch, device side (exchange.cuh): partials (one blob per bucket set) -> the root's
    // window over NVLink; root: wait for all ranks, sum in place, pairing checks, verdicts -> every rank's window; every rank:
    // wait for them.
    h2v_ctx::Comm& cm = ctx->comm;
    u32* vd = ctx->d_verdict.as<u32>();
    CKC(cudaMemsetAsync(vd + t.checks, 0, 8, s));  // error words of this launch set
    KLAUNCH(k_pack_partial_x, g.G, 256, 0, s, cb, wd, npts, t.wsums, cm.d_dyn, cm.d_peers, cm.lay, cm.d_done);
    if (mode & RUN_ROOT) {
      KLAUNCH_P(false, k_sum_partials, g.G, 128, 0, s, cm.lay.world, cb, wd, npts, cm.window + cm.lay.partials_off(), (size_t)cm.lay.max_groups * H2V_PARTIAL_BYTES,
                ctx->d_wsums_fin.as<G1Jac>(), vd + t.checks, cm.d_dyn, (const u64*)(cm.window + cm.lay.arrive_off()));
      int prc = launch_pairing(ctx, g, t.lines, ctx->d_wsums_fin.as<G1Jac>(), t.checks, t.run, t.sets);
      if (prc) return prc;
      KLAUNCH_P(false, k_bcast_verdict, 1, 256, 0, s, cm.d_dyn, cm.d_peers, cm.lay, t.checks, vd, vd + t.checks);
    }
    KLAUNCH_P(false, k_wait_verdict, 1, 64, 0, s, cm.d_dyn, cm.window, cm.lay, t.checks, vd);
  }
  if (mode & RUN_ABSORB) {
    const AccGeom ag{{g.W[0], g.W[1]}, {g.c[0], g.c[1]}};
    const h2v_ctx::AbsorbTarget& at = ctx->absorb;
    KLAUNCH(k_acc_absorb, 1, 32 * cdiv(4 * acc_items(ag), 32), 0, s, ag, t.wsums, ctx->d_r.as<Fr>(), ctx->mb.coef.as<Fr>(), at.acc, at.records, at.count, at.cap);
  }
  if (!ctx->capturing) CKC(cudaEventRecord(ctx->ev[5], s));
  if (mode & RUN_ACCUM) {
    int arc = enqueue_fold_accum(ctx, g, t.wsums, g.G, ctx->d_acc_bytes.as<u8>(), ctx->use_pdl);
    if (arc) return arc;
  }
  if (!ctx->capturing) CKC(cudaEventRecord(ctx->ev[6], s));
  return 0;
}

static int enqueue_batch(h2v_ctx* ctx, int mode) {
  const MsmGeom& g = ctx->geom;
  if ((mode & RUN_ACCUM) && g.G != 1) {
    ctx->err = "the folded accumulator hook is defined for a single fold group";
    return -1;
  }
  {
    int src = enqueue_stages(ctx);
    if (src) return src;
  }
  {
    NvtxRange nv_("h2v:msm");
    int mrc = enqueue_msm(ctx, g, ctx->mb, ctx->stream, nullptr, 0);
    if (mrc) return mrc;
  }
  return enqueue_tail(ctx, mode, TailArgs{g, ctx->mb.wsums.as<G1Jac>(), ctx->d_lines(), g.G, 1, 0, ctx->d_partial_out.as<u8>()});
}

static u64 graph_key(const h2v_ctx* ctx, int mode) {
  KeyHash k;
  k.mix((u64)mode);
  k.mix(ctx->n);
  k.mix(ctx->gcount);
  k.mix(ctx->gbase);
  k.mix(ctx->scratch_rows);
  k.mix((u64)ctx->has_ncols | (u64)ctx->has_col_len << 1);
  hash_geom(k, ctx->geom);
  const DevBuf* bufs[] = {&ctx->d_plan, &ctx->d_proofs, &ctx->d_proof_off, &ctx->d_inst, &ctx->d_inst_off, &ctx->d_ncols, &ctx->d_col_len,
                          &ctx->d_pts, &ctx->d_bad, &ctx->d_status, &ctx->d_vals, &ctx->d_scratch, &ctx->d_right, &ctx->d_shared, &ctx->d_left,
                          &ctx->d_r, &ctx->mb.coef, &ctx->mb.shared_sum, &ctx->mb.dig, &ctx->mb.hist, &ctx->mb.off, &ctx->mb.cursor, &ctx->mb.order,
                          &ctx->mb.sorted, &ctx->mb.buckets, &ctx->mb.wsums, &ctx->d_acc_bytes, &ctx->d_verdict, &ctx->mb.partials_msm,
                          &ctx->d_M, &ctx->d_partial_out, &ctx->mb.tiles, &ctx->d_wsums_fin, &ctx->d_ptsc};
  for (const DevBuf* b : bufs) k.mix((u64)(size_t)b->p);
  k.mix((u64)(size_t)ctx->d_lines());
  k.mix((u64)(size_t)ctx->d_gsums.p | (u64)line_run(ctx->geom.G ? ctx->geom.G : 1) << 56);
  k.mix((u64)(size_t)ctx->comm.window);
  if (ctx->hd.n_carry) k.mix((u64)(size_t)ctx->d_rho.p);
  if (mode & RUN_ABSORB) {
    k.mix((u64)(size_t)ctx->absorb.acc);
    k.mix((u64)(size_t)ctx->absorb.records);
    k.mix((u64)(size_t)ctx->absorb.count | (u64)ctx->absorb.cap << 48);
  }
  return k.h | 1;
}

// Every kernel of the batch on the context's stream: replay of the captured graph (one launch) or, with graphs
// off (per-stage event timings wanted), the direct launches.
static int run_impl(h2v_ctx* ctx, int mode) {
  if (!ctx || ctx->n == 0) return -1;
  NvtxRange nv_("h2v:launch_set");
  CKC(cudaSetDevice(ctx->device));
  cudaStream_t s = ctx->stream;
  if (!ctx->use_graphs) {
    int rc = enqueue_batch(ctx, mode);
    if (rc) return rc;
  } else {
    GraphSlot* gs = nullptr;
    int rc = graph_lookup(ctx->graphs, ctx->graph_clock, graph_key(ctx, mode), &ctx, 1, s, [&] { return enqueue_batch(ctx, mode); }, &gs);
    if (rc) return rc;
    CKC(cudaEventRecord(ctx->ev[0], s));
    CKC(cudaGraphLaunch(gs->exec, s));
    CKC(cudaEventRecord(ctx->ev[6], s));
    trace(ctx, "graph launched");
    ctx->launches += gs->kernels;
  }
  ctx->stages_timed = !ctx->use_graphs;
  ctx->verdicts_on_device = (mode & RUN_PAIRING) != 0;
  ctx->ran = true;
  return 0;
}

// parity hook: per-proof affine accumulators (L_j, R_j) of EVERY proof of the upload (reference: the DualMSM a SingleStrategy
// run would evaluate, msm.rs:81-95)
static int per_proof_accum(h2v_ctx* ctx, u8* accum_host) {
  CKC(cudaSetDevice(ctx->device));
  const PlanHeader& hd = ctx->hd;
  const u32 n = ctx->n;
  cudaStream_t s = ctx->stream;
  PlanView pv = ctx->pv();
  const u32 nbases = msm_points(hd) + hd.n_shared + msm_mo(hd);
  CKC(ctx->d_pp_prod.ensure(sizeof(G1Jac) * (size_t)n * nbases));
  CKC(ctx->d_pp_lr.ensure(sizeof(G1Jac) * (size_t)2 * n));
  CKC(ctx->d_pp_bytes.ensure(128 * (size_t)n));
  k_pp_mul<<<cdiv((u64)n * nbases, 128), 128, 0, s>>>(pv, n, ctx->d_pts.as<G1Affine>(), ctx->d_right.as<Fr>(), ctx->d_shared.as<Fr>(),
                                                       ctx->d_left.as<Fr>(), ctx->d_status.as<u32>(), ctx->d_pp_prod.as<G1Jac>(), nullptr, ctx->geom.n);
  LAUNCH_CHECK();
  k_pp_reduce<<<cdiv(2 * (u64)n, 128), 128, 0, s>>>(pv, n, ctx->d_pp_prod.as<G1Jac>(), ctx->d_pp_lr.as<G1Jac>(), ctx->d_pp_bytes.as<u8>());
  LAUNCH_CHECK();
  CKC(cudaMemcpyAsync(accum_host, ctx->d_pp_bytes.p, 128 * (size_t)n, cudaMemcpyDeviceToHost, s));
  return 0;
}

// Rejection attribution on the shard last processed by this context (see ATTR_SUB above): statuses of the proofs whose
// own check fails become ST_CONSTRAINT_SYSTEM_FAILURE.  With fold groups and the group verdicts on the device only the
// rejected groups are looked at.
static int attribute_impl(h2v_ctx* ctx) {
  NvtxRange nv_("h2v:attribution");
  CKC(cudaSetDevice(ctx->device));
  trace(ctx, "attr: begins");
  const PlanHeader& hd = ctx->hd;
  const u32 N = ctx->n;
  const MsmGeom& g = ctx->geom;
  cudaStream_t s = ctx->stream;
  PlanView pv = ctx->pv();
  const u32* gv = (ctx->verdicts_on_device && g.G > 1 && g.G * g.n == N) ? ctx->d_verdict.as<u32>() : nullptr;
  u32 gsize = g.n;  // proofs per flag of gv
  // grouped mixed batch: the per-proof flags of attr_accepted | one flag per level-1 sub-batch (accepted = all its proofs are)
  std::vector<u32> mask;
  mask.swap(ctx->attr_accepted);
  if (!mask.empty()) {
    const u32 ms = ATTR_SUB;
    for (u32 b = 0; b * ms < N; b++) {
      u32 all = 1;
      for (u32 j = b * ms; j < std::min(N, (b + 1) * ms); j++) all &= mask[j] ? 1u : 0u;
      mask.push_back(all);
    }
    CKC(ctx->d_attr_mask.ensure(4 * mask.size()));
    CKC(cudaMemcpyAsync(ctx->d_attr_mask.p, mask.data(), 4 * mask.size(), cudaMemcpyHostToDevice, s));
    gv = ctx->d_attr_mask.as<u32>();
    gsize = 1;
  }
  const u32 nbases = msm_points(hd) + hd.n_shared + msm_mo(hd);
  static constexpr u32 CHUNK = 1024;  // checks per pass: bounds the Miller scratch (E12[CHUNK][65] = 115 MB)
  MsmGeom unit{};
  unit.c[0] = unit.c[1] = 1;
  unit.W[0] = unit.W[1] = 1;
  int unit_slot = -1;
  {
    int lrc = ensure_lines(ctx, unit, &unit_slot);  // lines of -G2 (pair 0, right) and [s]G2 (pair 1, left)
    if (lrc) return lrc;
  }
  const G2Line* unit_lines = ctx->lines.s[unit_slot].buf.as<G2Line>();
  CKC(ctx->d_sub_M.ensure(sizeof(E12) * H2V_ATE_ITERS * (size_t)CHUNK));
  CKC(ctx->d_pp_lr.ensure(sizeof(G1Jac) * (size_t)2 * CHUNK));
  CKC(ctx->d_pp_prod.ensure(sizeof(G1Jac) * (size_t)CHUNK * nbases));
  CKC(ctx->d_sub_pairs.ensure(4 * ((size_t)N + 8) + 4 * (size_t)CHUNK));  // suspect list | count | verdicts of a pass
  u32* list = ctx->d_sub_pairs.as<u32>();
  u32* count = list + N;
  u32* pass_verdict = count + 8;
  const u32* sub_verdict = nullptr;
  u32 sub_size = 1;
  // ---- level 1: sub-batches of ATTR_SUB proofs through the bucket MSM, one 2-pair check each
  u32 msub = ATTR_SUB;
  if (const char* e = getenv("H2V_ATTR_SUB")) msub = (u32)atoi(e);  // (tuning: 0 = no sub-batch level)
  if (!mask.empty() && msub != ATTR_SUB) msub = 0;  // (the sub-batch flags are built for ATTR_SUB)
  // (level 1 needs twice the term ids of the batch pass - two GLV halves per term - inside the 31-bit id space)
  if (msub >= 2 && g.n >= 4 * msub && g.n % msub == 0 &&
      2 * ((u64)N * (msm_points(hd) + msm_mo(hd)) + (u64)hd.n_shared * (N / msub)) < (1ull << 31)) {
    const u32 subs = g.n / msub, SG = N / msub;
    // window bits of the re-fold: dependent chain = bucket chain (2 * 14 * msub / 2^(c-1) entries) + in-window reduction
    // (2^c additions) + window combination (130 doublings + 130 / c additions); measured (B200, sub-batches of 16): MSM + combination
    // 1.35 + 0.73 ms at c = 4, 1.73 + 0.68 at c = 5, 2.71 + 0.64 at c = 6
    u32 attr_c = 4;
    if (const char* e = getenv("H2V_ATTR_WINDOW")) attr_c = (u32)std::min(8, std::max(3, atoi(e)));
    MsmGeom sg = choose_geom(msub, hd, 0, SG, attr_c);
    CKC(ensure_msm_bufs(sg, ctx->ab, hd.n_shared));
    CKC(ctx->d_sub_verdict.ensure(4 * (size_t)SG + sizeof(G1Jac) * 2 * (size_t)SG + 64));
    u32* sv = ctx->d_sub_verdict.as<u32>();
    G1Jac* sub_pairs = (G1Jac*)(((size_t)(sv + SG) + 15) & ~(size_t)15);
    CKC(cudaMemsetAsync(ctx->ab.hist.p, 0, 4 * ((size_t)sg.nb() * sg.G + 2 * SIZE_BINS), s));
    CKC(cudaMemsetAsync(sv, 1, 4 * (size_t)SG, s));  // non-zero = accepted: sub-batches of accepted groups are never checked
    // The re-fold draws its own coefficients from a fresh key.  With the batch's r_i (caller scalars or the public test seed)
    // a cancellation the caller's scalars built into the batch fold, e.g. c_2 = -c_3 for two equal invalid proofs, would
    // repeat inside the sub-batch, which would then accept and report both proofs H2V_OK.
    RlcKey key{};
    if (os_entropy(&key, sizeof(key)) != 0) {
      ctx->err = "no OS entropy for the attribution coefficients (getrandom failed)";
      return -2;
    }
    CKC(ctx->d_attr_r.ensure(sizeof(Fr) * (size_t)N));
    KLAUNCH_P(false, k_rlc_expand, cdiv(N, 128), 128, 0, s, (u64)N, (u64)0, (const u8*)nullptr, true, key, ctx->d_attr_r.as<Fr>());
    KLAUNCH_P(false, k_rlc_scan, SG, RLC_NT, 0, s, ctx->d_attr_r.as<Fr>(), (u64)msub, (u64)0, msub, ctx->ab.coef.as<Fr>(), subs, (u64)g.n, (u64)0);
    {
      const bool pdl = ctx->use_pdl;
      ctx->use_pdl = false;
      int mrc = enqueue_msm(ctx, sg, ctx->ab, s, mask.empty() ? gv : gv + N, mask.empty() ? g.n : msub);
      ctx->use_pdl = pdl;
      if (mrc) return mrc;
    }
    if (trace_on()) { ctx_sync(ctx); trace(ctx, "attr: sub-batch msm done"); }
    FoldArgs fa{{sg.W[0], sg.W[1]}, {sg.c[0], sg.c[1]}, {sg.wbase[0], sg.wbase[1]}};
    KLAUNCH_P(false, k_window_combine, cdiv(8 * (u64)SG, 64), 64, 0, s, SG, fa, ctx->ab.wsums.as<G1Jac>(), sub_pairs);
    if (trace_on()) { ctx_sync(ctx); trace(ctx, "attr: window combine done"); }
    for (u32 base = 0; base < SG; base += CHUNK) {
      const u32 cnt = std::min(CHUNK, SG - base);
      const PairSkip sk = mask.empty() ? PairSkip{gv, nullptr, subs, base} : PairSkip{gv + N, nullptr, 1, base};
      int prc = launch_pair_checks(ctx, sub_pairs + 2 * (size_t)base, cnt, unit_lines, ctx->d_sub_M.as<E12>(), sv + base, sk);
      if (prc) return prc;
    }
    sub_verdict = sv;
    sub_size = msub;
  }
  // ---- level 2: every suspect proof alone
  CKC(cudaMemsetAsync(count, 0, 4, s));
  KLAUNCH_P(false, k_pp_suspects, cdiv(N, 128), 128, 0, s, N, ctx->d_status.as<u32>(), sub_verdict, sub_size, gv, gsize, list, count);
  CKC(ctx->h_verd.ensure(4 * 1040));
  u32* h_count = ctx->h_verd.as<u32>() + 1030;
  CKC(cudaMemcpyAsync(h_count, count, 4, cudaMemcpyDeviceToHost, s));
  CKC(ctx_sync(ctx));
  const u32 total = *h_count;
  if (trace_on()) { char b[64]; snprintf(b, sizeof b, "attr: level 1 done, %u suspects", total); trace(ctx, b); }
  for (u32 base = 0; base < total; base += CHUNK) {
    const u32 cnt = std::min(CHUNK, total - base);
    KLAUNCH_P(false, k_pp_mul_list, cdiv((u64)4 * cnt * nbases, 128), 128, 0, s, pv, N, ctx->d_pts.as<G1Affine>(), ctx->d_right.as<Fr>(), ctx->d_shared.as<Fr>(),
              ctx->d_left.as<Fr>(), list, count, base, CHUNK, ctx->d_pp_prod.as<G1Jac>());
    KLAUNCH_P(false, k_pp_reduce_list, cdiv(2 * (u64)cnt, 128), 128, 0, s, pv, count, base, CHUNK, ctx->d_pp_prod.as<G1Jac>(), ctx->d_pp_lr.as<G1Jac>());
    if (trace_on()) { ctx_sync(ctx); trace(ctx, "attr: suspects' accumulators done"); }
    int prc = launch_pair_checks(ctx, ctx->d_pp_lr.as<G1Jac>(), cnt, unit_lines, ctx->d_sub_M.as<E12>(), pass_verdict, PairSkip{nullptr, count, 1, base});
    if (prc) return prc;
    if (trace_on()) { ctx_sync(ctx); trace(ctx, "attr: suspects' checks done"); }
    KLAUNCH_P(false, k_pp_status, cdiv(cnt, 128), 128, 0, s, list, count, base, CHUNK, pass_verdict, ctx->d_status.as<u32>());
  }
  CKC(cudaEventRecord(ctx->ev[6], s));
  return 0;
}

static int download_status(h2v_ctx* ctx, u8* status) {
  CKC(ctx->h_status.ensure(4 * (size_t)ctx->n));
  const u32* hs = ctx->h_status.as<u32>();
  CKC(cudaMemcpyAsync(ctx->h_status.p, ctx->d_status.p, 4 * (size_t)ctx->n, cudaMemcpyDeviceToHost, ctx->stream));
  CKC(ctx_sync(ctx));
  if (status)
    for (u32 j = 0; j < ctx->n; j++) status[j] = (u8)hs[j];
  return 0;
}

static int hooks_impl(h2v_ctx* ctx, u8* challenges) {
  const PlanHeader& hd = ctx->hd;
  const u32 n = ctx->n;
  cudaStream_t s = ctx->stream;
  if (challenges) {
    CKC(ctx->d_chal.ensure(32 * (size_t)n * hd.n_challenges));
    k_gather_challenges<<<cdiv((u64)n * hd.n_challenges, 128), 128, 0, s>>>(ctx->pv(), n, ctx->d_vals.as<Fr>(), ctx->d_chal.as<u8>());
    LAUNCH_CHECK();
    CKC(cudaMemcpyAsync(challenges, ctx->d_chal.p, 32 * (size_t)n * hd.n_challenges, cudaMemcpyDeviceToHost, s));
  }
  if (ctx->opt_scalar_hook) {
    const u32 nbases = msm_points(hd) + hd.n_shared + msm_mo(hd);
    CKC(ctx->d_hook.ensure(32 * (size_t)n * nbases));
    k_gather_scalars<<<cdiv((u64)n * nbases, 128), 128, 0, s>>>(ctx->pv(), n, ctx->d_right.as<Fr>(), ctx->d_shared.as<Fr>(),
                                                                 ctx->d_left.as<Fr>(), ctx->d_hook.as<u8>());
    LAUNCH_CHECK();
    CKC(cudaMemcpyAsync(ctx->opt_scalar_hook, ctx->d_hook.p, 32 * (size_t)n * nbases, cudaMemcpyDeviceToHost, s));
    ctx->opt_scalar_hook = nullptr;
  }
  return 0;
}

int h2v_verify_batch(h2v_ctx* ctx, uint32_t n, const uint8_t* proofs, const uint64_t* proof_off, const uint8_t* instances,
                     const uint64_t* inst_off, const uint8_t* rlc_scalars, uint64_t seed, uint8_t* status, uint8_t* challenges,
                     uint8_t* accum, uint8_t* batch_accum) {
  int rc;
  if ((rc = upload_impl(ctx, n, proofs, proof_off, instances, inst_off, rlc_scalars, seed, 0, n / (ctx && ctx->opt_fold_groups ? ctx->opt_fold_groups : 1))) != 0) return rc;
  if ((rc = run_impl(ctx, RUN_PAIRING | (batch_accum ? RUN_ACCUM : 0))) != 0) return rc;
  if ((rc = hooks_impl(ctx, challenges)) != 0) return rc;
  u32 verdict = 0;
  if (batch_accum) CKC(cudaMemcpyAsync(batch_accum, ctx->d_acc_bytes.p, 128, cudaMemcpyDeviceToHost, ctx->stream));
  if ((rc = read_verdicts(ctx, &verdict)) != 0) return rc;
  if (accum && (rc = per_proof_accum(ctx, accum)) != 0) return rc;  // parity hook
  if (!verdict && (rc = attribute_impl(ctx)) != 0) return rc;      // rejected fold: poly/strategy.rs:26-30
  return download_status(ctx, status);
}

int h2v_verify_proof(h2v_ctx* ctx, const uint8_t* proof, size_t proof_len, const uint8_t* instances, size_t n_inst, uint8_t* status) {
  const u64 poff[2] = {0, proof_len}, ioff[2] = {0, n_inst};
  return h2v_verify_batch(ctx, 1, proof, poff, instances, ioff, nullptr, 0, status, nullptr, nullptr, nullptr);
}

int h2v_accumulate_shard(h2v_ctx* ctx, uint32_t n, const uint8_t* proofs, const uint64_t* proof_off, const uint8_t* instances,
                         const uint64_t* inst_off, const uint8_t* rlc_scalars, uint64_t seed, uint64_t global_base,
                         uint64_t global_count, uint8_t* status, uint8_t* partial) {
  int rc;
  if ((rc = upload_impl(ctx, n, proofs, proof_off, instances, inst_off, rlc_scalars, seed, global_base, global_count)) != 0) return rc;
  if ((rc = run_impl(ctx, RUN_PARTIAL)) != 0) return rc;
  if (partial) CKC(cudaMemcpyAsync(partial, ctx->d_partial_out.p, (size_t)H2V_PARTIAL_BYTES * ctx->geom.G, cudaMemcpyDefault, ctx->stream));
  return download_status(ctx, status);
}

// `bytes` of partials in this device's memory: in place when they already are (e.g. the output of a gather), else copied
static int device_partials(h2v_ctx* ctx, const u8* partials, size_t bytes, const u8** d_parts) {
  *d_parts = nullptr;
  {
    cudaPointerAttributes pa{};
    if (cudaPointerGetAttributes(&pa, partials) == cudaSuccess && pa.type == cudaMemoryTypeDevice && pa.device == ctx->device) *d_parts = partials;
    (void)cudaGetLastError();
  }
  if (!*d_parts) {
    CKC(ctx->d_partials.ensure(bytes));
    CKC(cudaMemcpyAsync(ctx->d_partials.p, partials, bytes, cudaMemcpyDefault, ctx->stream));
    *d_parts = ctx->d_partials.as<u8>();
  }
  return 0;
}

// window geometry (c, W per channel) of the partial at d_parts, from its header
static int partial_geom(h2v_ctx* ctx, const u8* d_parts, MsmGeom& g) {
  PartialHeader h;
  CKC(cudaMemcpyAsync(&h, d_parts, sizeof(h), cudaMemcpyDeviceToHost, ctx->stream));
  CKC(ctx_sync(ctx));
  g = MsmGeom{};
  g.c[0] = h.cbits & 0xFFFF;
  g.c[1] = h.cbits >> 16;
  g.W[0] = h.windows & 0xFFFF;
  g.W[1] = h.windows >> 16;
  if (h.magic != H2V_PARTIAL_MAGIC || g.c[0] < 1 || g.c[1] < 1 || g.W[0] + g.W[1] != h.n_pts || h.n_pts > 128) {
    ctx->err = "malformed partial accumulator";
    return -1;
  }
  g.wbase[1] = g.W[0];
  return 0;
}

// The final check of partials on ctx's stream: the window-wise sum of n_partials ranks' blobs ([rank][group][set], device
// memory), then `groups` pairing checks of `sets` bucket sets each (geometry g, prepared lines `lines`, run length `run`, 0 =
// line_run(groups)).  batch_accum (groups == 1): sets x 128 B folded affine (L, R), set order.  *all = every check accepted.
static int sum_and_pair(h2v_ctx* ctx, const MsmGeom& g, const G2Line* lines, u32 run, u32 n_partials, u32 groups, u32 sets, const u8* d_parts,
                        u8* batch_accum, u8* group_verdicts, u32* all) {
  cudaStream_t s = ctx->stream;
  const u32 npts = g.W[0] + g.W[1], blobs = groups * sets;
  CKC(ctx->d_verdict.ensure(4 * (size_t)groups + 16));
  CKC(ctx->d_M.ensure(sizeof(E12) * (H2V_ATE_ITERS + MILLER_SEGS) * (size_t)groups));
  CKC(ctx->d_wsums_fin.ensure(sizeof(G1Jac) * 128 * (size_t)blobs));
  CKC(ctx->d_gsums.ensure(sizeof(G1Jac) * 128 * (size_t)blobs));
  CKC(cudaMemsetAsync(ctx->d_verdict.p, 0, 4 * (size_t)groups + 16, s));
  ctx->verdicts_on_device = false;  // d_verdict now belongs to the global batches being finalized
  k_sum_partials<<<blobs, 128, 0, s>>>(n_partials, g.c[0] | g.c[1] << 16, g.W[0] | g.W[1] << 16, npts, d_parts, (size_t)blobs * H2V_PARTIAL_BYTES,
                                       ctx->d_wsums_fin.as<G1Jac>(), ctx->d_verdict.as<u32>() + groups, nullptr, nullptr);
  LAUNCH_CHECK();
  int prc = launch_pairing(ctx, g, lines, ctx->d_wsums_fin.as<G1Jac>(), groups, run, sets);
  if (prc) return prc;
  if (batch_accum) {
    CKC(ctx->d_acc_bytes.ensure(128 * (size_t)sets));
    if ((prc = enqueue_fold_accum(ctx, g, ctx->d_wsums_fin.as<G1Jac>(), sets, ctx->d_acc_bytes.as<u8>(), false)) != 0) return prc;
    CKC(cudaMemcpyAsync(batch_accum, ctx->d_acc_bytes.p, 128 * (size_t)sets, cudaMemcpyDeviceToHost, s));
  }
  CKC(ctx->h_verd.ensure(4 * (size_t)(groups + 2)));
  const u32* v = ctx->h_verd.as<u32>();
  CKC(cudaMemcpyAsync(ctx->h_verd.p, ctx->d_verdict.p, 4 * (size_t)(groups + 1), cudaMemcpyDeviceToHost, s));
  CKC(ctx_sync(ctx));
  if (v[groups]) {
    ctx->err = "partial accumulators were produced with different window geometries (use h2v_batch_set_shard_hint)";
    return -1;
  }
  *all = 1;
  for (u32 q = 0; q < groups; q++) {
    *all &= v[q] ? 1u : 0u;
    if (group_verdicts) group_verdicts[q] = v[q] ? 1 : 0;
  }
  return 0;
}

static int finalize_impl(h2v_ctx* ctx, u32 n_partials, u32 groups, const u8* partials, u8* batch_accum, int* verdict, u8* group_verdicts) {
  if (!ctx || !partials || !n_partials || n_partials > 128 || !groups || groups > 1024 || (batch_accum && groups != 1)) return -1;
  CKC(cudaSetDevice(ctx->device));
  const u8* d_parts = nullptr;
  int rc = device_partials(ctx, partials, (size_t)H2V_PARTIAL_BYTES * n_partials * groups, &d_parts);
  if (rc) return rc;
  if (ctx->n == 0 && (rc = partial_geom(ctx, d_parts, ctx->geom)) != 0) return rc;  // a context that has not processed a shard itself
  const int lines_of_batch = ctx->lines.cur;  // the resident batch of this context keeps its own line geometry (restored below)
  {
    int lrc = ensure_lines(ctx, groups);
    if (lrc) return lrc;
  }
  u32 all = 0;
  rc = sum_and_pair(ctx, ctx->geom, ctx->d_lines(), 0, n_partials, groups, 1, d_parts, batch_accum, group_verdicts, &all);
  if (lines_of_batch >= 0 && ctx->n) ctx->lines.cur = lines_of_batch;
  if (rc) return rc;
  if (verdict) *verdict = (int)all;
  return 0;
}

int h2v_finalize(h2v_ctx* ctx, uint32_t n_partials, const uint8_t* partials, uint8_t* batch_accum, int* verdict) {
  return finalize_impl(ctx, n_partials, 1, partials, batch_accum, verdict, nullptr);
}
int h2v_finalize_groups(h2v_ctx* ctx, uint32_t n_partials, uint32_t groups, const uint8_t* partials, uint8_t* group_verdicts, int* verdict) {
  return finalize_impl(ctx, n_partials, groups, partials, nullptr, verdict, group_verdicts);
}

int h2v_attribute_shard(h2v_ctx* ctx, uint8_t* status) {
  if (!ctx || !ctx->ran) return -1;
  int rc;
  if ((rc = attribute_impl(ctx)) != 0) return rc;
  return download_status(ctx, status);
}

int h2v_attribute_shard_groups(h2v_ctx* ctx, const uint8_t* group_verdicts, uint32_t groups, uint8_t* status) {
  if (!ctx || !ctx->ran || !group_verdicts || groups != ctx->geom.G) return -1;
  CKC(cudaSetDevice(ctx->device));
  std::vector<u32> v(groups);
  for (u32 q = 0; q < groups; q++) v[q] = group_verdicts[q] ? 1u : 0u;
  CKC(ctx->d_verdict.ensure(4 * (size_t)groups + 16));
  CKC(cudaMemcpyAsync(ctx->d_verdict.p, v.data(), 4 * (size_t)groups, cudaMemcpyHostToDevice, ctx->stream));
  CKC(ctx_sync(ctx));  // v is a stack buffer
  ctx->verdicts_on_device = true;  // attribute_impl skips the proofs of accepted groups
  int rc;
  if ((rc = attribute_impl(ctx)) != 0) return rc;
  return download_status(ctx, status);
}

// ---- device-side exchange (exchange.cuh) ---------------------------------------------------------
int h2v_comm_init(h2v_ctx* ctx, uint32_t rank, uint32_t world, uint32_t max_groups, uint8_t* handle_out) {
  if (!ctx || !handle_out || world == 0 || world > XCH_MAX_RANKS || rank >= world || max_groups == 0 || max_groups > 1024) {
    if (ctx) ctx->err = "h2v_comm_init: bad arguments (world <= 128, max_groups <= 1024)";
    return -1;
  }
  CKC(cudaSetDevice(ctx->device));
  CKC(ctx_sync(ctx));
  comm_release(ctx);
  for (auto& gsl : ctx->graphs) gsl.key = 0;  // graphs captured with the old window
  h2v_ctx::Comm& cm = ctx->comm;
  cm.lay = XLayout{rank, world, max_groups, 0};
  const size_t bytes = cm.lay.bytes();
  CKC(cudaMalloc((void**)&cm.window, bytes));
  CKC(cudaMemset(cm.window, 0, bytes));
  CKC(cudaMalloc((void**)&cm.d_peers, sizeof(u8*) * world));
  CKC(cudaMalloc((void**)&cm.d_dyn, sizeof(XDyn)));
  CKC(cudaMalloc((void**)&cm.d_done, 4));
  CKC(cudaMemset(cm.d_done, 0, 4));
  CKC(cudaMallocHost((void**)&cm.h_dyn, sizeof(XDyn) * XDYN_RING));
  if (const char* t = getenv("H2V_COMM_TIMEOUT_MS")) {
    const long ms = atol(t);
    if (ms > 0) cm.timeout_ns = (u64)ms * 1000000ull;
  }
  CommHandle h{};
  h.magic = H2V_COMM_MAGIC;
  h.rank = rank;
  h.world = world;
  h.max_groups = max_groups;
  h.pid = (u64)getpid();
  h.ptr = (u64)(size_t)cm.window;
  h.bytes = bytes;
  h.device = ctx->device;
  CKC(cudaIpcGetMemHandle(&h.ipc, cm.window));
  memcpy(handle_out, &h, sizeof(h));
  CKC(cudaDeviceSynchronize());
  return 0;
}

int h2v_comm_set_timeout_ms(h2v_ctx* ctx, uint32_t ms) {
  if (!ctx || !ms) return -1;
  ctx->comm.timeout_ns = (u64)ms * 1000000ull;
  return 0;
}

int h2v_comm_connect(h2v_ctx* ctx, const uint8_t* handles) {
  if (!ctx || !handles || !ctx->comm.window) {
    if (ctx) ctx->err = "h2v_comm_connect: call h2v_comm_init first";
    return -1;
  }
  CKC(cudaSetDevice(ctx->device));
  h2v_ctx::Comm& cm = ctx->comm;
  const XLayout& lay = cm.lay;
  cm.peers.assign(lay.world, nullptr);
  for (u32 r = 0; r < lay.world; r++) {
    CommHandle h;
    memcpy(&h, handles + (size_t)r * H2V_COMM_HANDLE_BYTES, sizeof(h));
    if (h.magic != H2V_COMM_MAGIC || h.rank != r || h.world != lay.world || h.max_groups != lay.max_groups || h.bytes != lay.bytes()) {
      ctx->err = "h2v_comm_connect: handle " + std::to_string(r) + " does not belong to this job (rank order, world size and max_groups must agree on every rank)";
      return -1;
    }
    if (r == lay.rank) {
      cm.peers[r] = cm.window;
    } else if (h.pid == (u64)getpid()) {  // a peer context of this very process (tests, single-process multi-GPU)
      if (h.device != ctx->device) {
        int can = 0;
        CKC(cudaDeviceCanAccessPeer(&can, ctx->device, h.device));
        if (!can) {
          ctx->err = "h2v_comm_connect: no peer access between devices " + std::to_string(ctx->device) + " and " + std::to_string(h.device);
          return -2;
        }
        const cudaError_t pe = cudaDeviceEnablePeerAccess(h.device, 0);
        if (pe != cudaSuccess && pe != cudaErrorPeerAccessAlreadyEnabled) CKC(pe);
        (void)cudaGetLastError();
      }
      cm.peers[r] = (u8*)(size_t)h.ptr;
    } else {
      void* p = nullptr;
      const cudaError_t oe = cudaIpcOpenMemHandle(&p, h.ipc, cudaIpcMemLazyEnablePeerAccess);
      if (oe != cudaSuccess) {
        (void)cudaGetLastError();
        ctx->err = std::string("h2v_comm_connect: cudaIpcOpenMemHandle of rank ") + std::to_string(r) + "'s window failed (" + cudaGetErrorString(oe) +
                   "): the ranks must be processes of one node with NVLink / PCIe peer access; otherwise exchange the partials with h2v_accumulate_shard + a gather + h2v_finalize";
        return -2;
      }
      cm.opened.push_back(p);
      cm.peers[r] = (u8*)p;
    }
  }
  CKC(cudaMemcpy(cm.d_peers, cm.peers.data(), sizeof(u8*) * lay.world, cudaMemcpyHostToDevice));
  cm.seq = 0;
  cm.ready = true;
  return 0;
}

// parameters of the next launch set on ctx's channel (sequence number, root), copied to the device on ctx's stream
static cudaError_t comm_next_launch(h2v_ctx* ctx, u32 root) {
  h2v_ctx::Comm& cm = ctx->comm;
  XDyn* d = &cm.h_dyn[cm.ring++ % XDYN_RING];
  d->seq = ++cm.seq;
  d->root = root;
  d->rsv = 0;
  d->timeout_ns = cm.timeout_ns;
  return cudaMemcpyAsync(cm.d_dyn, d, sizeof(XDyn), cudaMemcpyHostToDevice, ctx->stream);
}

// one launch set through the exchange; `status` != null: attribution inside rejected groups + status download
static int exchange_run(h2v_ctx* ctx, u32 root, u8* group_verdicts, int* verdict, bool e2e, u8* status) {
  h2v_ctx::Comm& cm = ctx->comm;
  if (!cm.ready || root >= cm.lay.world || ctx->n == 0 || ctx->geom.G > cm.lay.max_groups) {
    ctx->err = "sharded exchange: the context needs h2v_comm_init + h2v_comm_connect, an uploaded shard, root < world and fold groups <= max_groups";
    return -1;
  }
  CKC(cudaSetDevice(ctx->device));
  CKC(comm_next_launch(ctx, root));
  int rc = run_impl(ctx, RUN_XCHG | (root == cm.lay.rank ? RUN_ROOT : 0));
  if (rc) return rc;
  u32 all = 0;
  rc = read_verdicts(ctx, &all, true);
  trace(ctx, rc ? "exchange FAILED" : "verdicts read");
  if (rc) return rc;
  ctx->verdicts_on_device = true;  // d_verdict holds the verdicts of this rank's groups: attribution skips accepted groups
  if (group_verdicts)
    for (u32 q = 0; q < ctx->geom.G; q++) group_verdicts[q] = ctx->h_verdicts[q] ? 1 : 0;
  if (verdict) *verdict = (int)all;
  if (e2e) {
    if (!all && (rc = attribute_impl(ctx)) != 0) return rc;
    return download_status(ctx, status);
  }
  return 0;
}

int h2v_batch_run_shard_exchange(h2v_ctx* ctx, uint32_t root, uint8_t* group_verdicts, int* verdict) {
  if (!ctx) return -1;
  return exchange_run(ctx, root, group_verdicts, verdict, false, nullptr);
}

int h2v_verify_shard(h2v_ctx* ctx, uint32_t n, const uint8_t* proofs, const uint64_t* proof_off, const uint8_t* instances,
                     const uint64_t* inst_off, const uint8_t* rlc_scalars, uint64_t seed, uint64_t global_base, uint64_t global_count,
                     uint32_t root, uint8_t* status, uint8_t* group_verdicts, int* verdict) {
  int rc;
  if ((rc = upload_impl(ctx, n, proofs, proof_off, instances, inst_off, rlc_scalars, seed, global_base, global_count)) != 0) return rc;
  return exchange_run(ctx, root, group_verdicts, verdict, true, status);
}

int h2v_comm_last_batch_accum(h2v_ctx* ctx, uint8_t* batch_accum) {
  if (!ctx || !batch_accum || !ctx->comm.ready || ctx->geom.G != 1) return -1;
  CKC(cudaSetDevice(ctx->device));
  const int rc = enqueue_fold_accum(ctx, ctx->geom, ctx->d_wsums_fin.as<G1Jac>(), 1, ctx->d_acc_bytes.as<u8>(), false);
  if (rc) return rc;
  CKC(cudaMemcpyAsync(batch_accum, ctx->d_acc_bytes.p, 128, cudaMemcpyDeviceToHost, ctx->stream));
  CKC(ctx_sync(ctx));
  return 0;
}

int h2v_ctx_cache_stats(const h2v_ctx* ctx, uint64_t* out2) {
  if (!ctx || !out2) return -1;
  out2[0] = ctx->lines_builds;
  out2[1] = ctx->graph_captures;
  return 0;
}

int h2v_batch_upload(h2v_ctx* ctx, uint32_t n, const uint8_t* proofs, const uint64_t* proof_off, const uint8_t* instances,
                     const uint64_t* inst_off, const uint8_t* rlc_scalars, uint64_t seed) {
  int rc = upload_impl(ctx, n, proofs, proof_off, instances, inst_off, rlc_scalars, seed, 0, n / (ctx && ctx->opt_fold_groups ? ctx->opt_fold_groups : 1));
  if (rc) return rc;
  CKC(ctx_sync(ctx));
  return 0;
}

int h2v_batch_upload_shard(h2v_ctx* ctx, uint32_t n, const uint8_t* proofs, const uint64_t* proof_off, const uint8_t* instances,
                           const uint64_t* inst_off, const uint8_t* rlc_scalars, uint64_t seed, uint64_t global_base,
                           uint64_t global_count) {
  int rc = upload_impl(ctx, n, proofs, proof_off, instances, inst_off, rlc_scalars, seed, global_base, global_count);
  if (rc) return rc;
  CKC(ctx_sync(ctx));
  return 0;
}

int h2v_batch_run_shard(h2v_ctx* ctx, uint8_t* partial) {
  int rc = run_impl(ctx, RUN_PARTIAL);
  if (rc) return rc;
  if (partial) CKC(cudaMemcpyAsync(partial, ctx->d_partial_out.p, (size_t)H2V_PARTIAL_BYTES * ctx->geom.G, cudaMemcpyDefault, ctx->stream));
  CKC(ctx_sync(ctx));
  return 0;
}

int h2v_batch_run_shard_async(h2v_ctx* ctx, uint8_t* partial_device) {
  int rc = run_impl(ctx, RUN_PARTIAL);
  if (rc) return rc;
  if (partial_device) CKC(cudaMemcpyAsync(partial_device, ctx->d_partial_out.p, (size_t)H2V_PARTIAL_BYTES * ctx->geom.G, cudaMemcpyDeviceToDevice, ctx->stream));
  return 0;
}

int h2v_flush_l2(h2v_ctx* ctx, size_t bytes) {
  if (!ctx) return -1;
  CKC(cudaSetDevice(ctx->device));
  CKC(ctx->d_flush.ensure(bytes));
  CKC(cudaMemsetAsync(ctx->d_flush.p, 0x5a, bytes, ctx->stream));
  return 0;
}

int h2v_batch_run(h2v_ctx* ctx, int* verdict) {
  int rc = run_impl(ctx, RUN_PAIRING);
  if (rc) return rc;
  u32 v = 0;
  if ((rc = read_verdicts(ctx, &v)) != 0) return rc;
  if (verdict) *verdict = (int)v;
  return 0;
}

int h2v_batch_download(h2v_ctx* ctx, uint8_t* status) {
  if (!ctx || !ctx->ran) return -1;
  return download_status(ctx, status);
}

int h2v_last_timings(const h2v_ctx* cctx, float* out8) {
  h2v_ctx* ctx = (h2v_ctx*)cctx;
  if (!ctx || !ctx->ran || !out8) return -1;
  CKC(cudaSetDevice(ctx->device));
  CKC(cudaEventSynchronize(ctx->ev[6]));
  for (int i = 0; i < 8; i++) out8[i] = 0;
  CKC(cudaEventElapsedTime(&out8[0], ctx->ev[0], ctx->ev[6]));
  if (ctx->stages_timed)  // a graph replay has no events between its kernels: only the total is known
    for (int i = 1; i <= 6; i++) CKC(cudaEventElapsedTime(&out8[i], ctx->ev[i - 1], ctx->ev[i]));
  return 0;
}

uint64_t h2v_launch_count(const h2v_ctx* ctx) { return ctx ? ctx->launches : 0; }

void* h2v_ctx_stream(const h2v_ctx* ctx) { return ctx ? (void*)ctx->stream : nullptr; }

int h2v_debug_timeline_start(int device, uint32_t capacity) {
  if (cudaSetDevice(device) != cudaSuccess) return -2;
  TlRec* buf = nullptr;
  u32 zero = 0;
  if (cudaMalloc(&buf, sizeof(TlRec) * (size_t)capacity) != cudaSuccess) return -2;
  cudaDeviceSynchronize();
  cudaMemcpyToSymbol(g_tl_count, &zero, 4);
  cudaMemcpyToSymbol(g_tl_cap, &capacity, 4);
  cudaMemcpyToSymbol(g_tl_buf, &buf, sizeof(buf));
  return cudaDeviceSynchronize() == cudaSuccess ? 0 : -2;
}
/* stops recording and copies up to `capacity` 32-byte records {u32 kernel, block, sm, tag; u64 start_ns, end_ns} */
int h2v_debug_timeline_stop(int device, void* out, uint32_t capacity, uint32_t* count) {
  if (cudaSetDevice(device) != cudaSuccess) return -2;
  cudaDeviceSynchronize();
  TlRec* buf = nullptr;
  TlRec* none = nullptr;
  u32 n = 0, cap = 0;
  cudaMemcpyFromSymbol(&buf, g_tl_buf, sizeof(buf));
  cudaMemcpyFromSymbol(&n, g_tl_count, 4);
  cudaMemcpyFromSymbol(&cap, g_tl_cap, 4);
  cudaMemcpyToSymbol(g_tl_buf, &none, sizeof(none));
  if (!buf) return -1;
  if (n > cap) n = cap;
  if (n > capacity) n = capacity;
  if (out && n) cudaMemcpy(out, buf, sizeof(TlRec) * (size_t)n, cudaMemcpyDeviceToHost);
  if (count) *count = n;
  cudaFree(buf);
  return cudaDeviceSynchronize() == cudaSuccess ? 0 : -2;
}

int h2v_ctx_set_graphs(h2v_ctx* ctx, int on) {
  if (!ctx) return -1;
  ctx->use_graphs = (on & 1) != 0;
  ctx->use_pdl = (on & 2) != 0;  // bit 1 switches programmatic dependent launch ON (default off)
  for (auto& gsl : ctx->graphs) gsl.key = 0;  // (the captured graphs embed the launch attributes)
  return 0;
}

int h2v_ctx_set_blocking_sync(h2v_ctx* ctx, int blocking) {
  if (!ctx) return -1;
  ctx->blocking_sync = blocking != 0;
  return 0;
}

int h2v_last_msm_geometry(const h2v_ctx* ctx, uint32_t* out4) {
  if (!ctx || !out4) return -1;
  out4[0] = ctx->geom.c[0] | (ctx->geom.c[1] << 16);
  out4[1] = ctx->geom.W[0] | (ctx->geom.W[1] << 16);
  out4[2] = ctx->geom.T;
  out4[3] = ctx->geom.nb();
  return 0;
}

int h2v_last_msm_glv(const h2v_ctx* ctx) {
  if (!ctx) return -1;
  return ctx->geom.lifted() ? 1 : 0;
}

int h2v_selftest_field(int device, uint32_t count, uint64_t seed) {
  if (cudaSetDevice(device) != cudaSuccess) return -2;
  u32* d = nullptr;
  if (cudaMalloc(&d, 4) != cudaSuccess) return -2;
  cudaMemset(d, 0, 4);
  k_selftest_field<<<cdiv(count, 128), 128>>>(count, seed, d);
  u32 h = 0;
  cudaError_t e = cudaMemcpy(&h, d, 4, cudaMemcpyDeviceToHost);
  cudaFree(d);
  if (e != cudaSuccess || cudaGetLastError() != cudaSuccess) return -2;
  return (int)h;
}

int h2v_selftest_field_vectors(int device, int field, int op, uint32_t n, const uint8_t* a, const uint8_t* b, uint8_t* out) {
  if ((field != 0 && field != 1) || op < 0 || op > 12 || !a || !b || !out) return -1;
  if (n == 0) return 0;
  if (cudaSetDevice(device) != cudaSuccess) return -2;
  const size_t bytes = 32 * (size_t)n;
  u8* d = nullptr;
  if (cudaMalloc(&d, 3 * bytes) != cudaSuccess) return -2;
  cudaError_t e = cudaMemcpy(d, a, bytes, cudaMemcpyHostToDevice);
  if (e == cudaSuccess) e = cudaMemcpy(d + bytes, b, bytes, cudaMemcpyHostToDevice);
  if (e == cudaSuccess) {
    if (field == 0) k_selftest_field_vectors<Fq><<<cdiv(n, 128), 128>>>(op, n, d, d + bytes, d + 2 * bytes);
    else k_selftest_field_vectors<Fr><<<cdiv(n, 128), 128>>>(op, n, d, d + bytes, d + 2 * bytes);
    e = cudaGetLastError();
  }
  if (e == cudaSuccess) e = cudaMemcpy(out, d + 2 * bytes, bytes, cudaMemcpyDeviceToHost);
  cudaFree(d);
  return e == cudaSuccess ? 0 : -2;
}

double h2v_calibrate_imad(int device) {
  if (cudaSetDevice(device) != cudaSuccess) return -1.0;
  cudaDeviceProp prop;
  if (cudaGetDeviceProperties(&prop, device) != cudaSuccess) return -1.0;
  const u32 blocks = prop.multiProcessorCount * 8, threads = 256, iters = 4096;
  u32* d = nullptr;
  if (cudaMalloc(&d, 4 * (size_t)blocks * threads) != cudaSuccess) return -1.0;
  cudaEvent_t a, b;
  cudaEventCreate(&a);
  cudaEventCreate(&b);
  k_imad<<<blocks, threads>>>(64, d);  // warm-up
  double best = 0;
  for (int rep = 0; rep < 3; rep++) {
    cudaEventRecord(a);
    k_imad<<<blocks, threads>>>(iters, d);
    cudaEventRecord(b);
    cudaEventSynchronize(b);
    float ms = 0;
    cudaEventElapsedTime(&ms, a, b);
    const double ops = (double)blocks * threads * iters * 64.0;
    if (ms > 0) best = std::max(best, ops / (ms * 1e-3));
  }
  cudaEventDestroy(a);
  cudaEventDestroy(b);
  cudaFree(d);
  return cudaGetLastError() == cudaSuccess ? best : -1.0;
}

// ---- mixed batches: proofs of several contexts (verifying keys) folded into one MSM and one pairing check ----------
// The members keep their own per-proof stages; the mix owns the joint MSM's buffers, its segment table and its graphs,
// and runs the pairing check on the lead member (member 0).  In a mix of h2v_mix_create all members' params agree on
// (g, g2, s_g2) and the lead's prepared G2 lines serve every member.  In a multi-params mix (h2v_mix_create_multi_params)
// every params class with proofs gets its own bucket set and its own line table (owned by the mix), and the one pairing
// check multiplies the pairs of all classes.
struct h2v_mix {
  std::vector<h2v_ctx*> m;  // members, not owned; m[0] = lead (its stream is the mix's stream)
  std::string err;
  cudaEvent_t ev_fork = nullptr;
  std::vector<cudaEvent_t> ev_join;  // per member: its stages are done
  bool has_key = false;              // one-shot key for the next batch (h2v_mix_set_rlc_key)
  RlcKey key{};
  h2v_ctx::MsmBufs b;  // the joint MSM (coef / shared_sum unused: the segments point to the members' coefficients and d_ssum)
  DevBuf d_seg, d_grange, d_ssum;
  std::vector<MixSeg> segs;    // of the current batch: groups x members, group-major (mix_layout_groups)
  std::vector<u32> active;     // members with proofs in the current batch
  u32 groups = 1;              // fold groups of the current batch (h2v_mix_verify_groups), each with its own check
  u64 call_base = 0;           // call index of the upload's first proof (a shard: its global base)
  std::vector<u32> grange;     // call-index range of every group: [grange[q], grange[q + 1])
  MsmGeom geom{};
  int lines_slot = -1;  // slot of the lines of the joint geometry: in mlines (multi-params mix) or the lead's cache
  GraphSlot graphs[8];  // LRU over (member shapes, buffers), as for a context
  u64 graph_clock = 0;
  // params classes: members whose params agree on (g, g2, s_g2), numbered by first appearance (one class unless multi)
  bool multi = false;
  std::vector<u32> cls_of;     // per member
  std::vector<u32> class_rep;  // per class: its first member (whose params build the class's lines)
  // current batch: bucket set of each class (~0u: no proofs), bucket sets, run length of the window combination
  std::vector<u32> set_of_class;
  u32 sets = 1, run = 0;
  // multi-params mix: line tables of (pair geometry, classes with proofs), set-major; a cache of its own, so that the lead's
  // cache (keyed by geometry alone) never holds a multi-class table
  LinesCache mlines;
  // sharded mixed batches (h2v_mix_accumulate_shard / h2v_mix_verify_shard)
  DevBuf d_partial;          // this rank's partials: one H2V_PARTIAL_BYTES blob per bucket set (RUN_PARTIAL)
  u32 opt_shard_hint = 0;    // one-shot: window geometry for shards of up to this many proofs (h2v_mix_set_shard_hint)
  std::vector<u32> counts;   // proofs per member of the batch / shard last uploaded
  bool ran = false;          // a launch set ran on that upload (h2v_mix_attribute_shard)
  bool xchg_root = false;    // the last launch set went through the exchange with this rank as its root
  const G2Line* lines() const { return (multi ? mlines : m[0]->lines).s[lines_slot].buf.as<G2Line>(); }
};

static const G1Affine& plan_g(const h2v_ctx* c) {  // params.g: the last shared base of every plan
  PlanView pv{c->blob.data()};
  return pv.sec<G1Affine>(c->hd.off_shared_pts)[c->hd.n_shared - 1];
}

// the proofs of two contexts can share one pairing check: their params agree on (g, g2, s_g2)
static bool params_agree(const h2v_ctx* a, const h2v_ctx* b) {
  return !memcmp(a->info.q_left, b->info.q_left, sizeof(a->info.q_left)) && !memcmp(a->info.q_right, b->info.q_right, sizeof(a->info.q_right)) &&
         !memcmp(&plan_g(a), &plan_g(b), sizeof(G1Affine));
}

// joint window geometry: the choice for `groups` fold groups of N / groups proofs (one group: the single-batch choice) over the
// terms of each channel of the largest bucket set per group, then one bucket set per (group, params class with proofs)
// (G = sets; T stays every term of the mix)
static MsmGeom mix_geom(u32 N, u32 T, u32 right_terms, u32 left_terms, u32 sets, u32 groups) {
  MsmGeom g{};
  g.n = N;  // (picks the chunk size and bucket lanes as for a single batch of N proofs; the mixed kernels map terms through the segments)
  g.G = 1;
  g.N = N;
  g.T = T;
  choose_windows(g, right_terms, left_terms, (u32)(((u64)N + groups - 1) / groups), groups, 0);
  g.G = sets;
  return g;
}

extern "C++" {  // (inside the extern "C" block of the ABI: the mix's overloads of ensure_lines and graph_key)
// The lines of the current batch's pair geometry q -> mx->lines_slot.  A single-params mix uses the lead's lines and cache.  A
// multi-params mix uses one table per class with proofs (its (q_right, q_left)), in class order, cached in the mix under
// (geometry, classes with proofs).
static int ensure_lines(h2v_mix* mx, const MsmGeom& q) {
  h2v_ctx* lead = mx->m[0];
  if (!mx->multi) return ensure_lines(lead, q, &mx->lines_slot);
  u64 key = lines_key_of(q);
  std::vector<const PlanInfo*> classes;
  for (u32 c = 0; c < mx->set_of_class.size(); c++)
    if (mx->set_of_class[c] != ~0u) {
      key |= 1ull << (48 + c);
      classes.push_back(&mx->m[mx->class_rep[c]]->info);
    }
  return ensure_lines(lead, mx->mlines, key, q, classes, -1, &mx->lines_slot);
}

static std::vector<h2v_ctx*> mix_active(const h2v_mix* mx) {
  std::vector<h2v_ctx*> v;
  for (u32 mi : mx->active) v.push_back(mx->m[mi]);
  return v;
}

// Every kernel of a mixed batch: the members' stages forked onto their own streams, the joint MSM on the lead's stream, then,
// by the RUN_* mode bits (enqueue_tail on the lead): RUN_PAIRING the pairing check over every bucket set -> the lead's d_verdict[0];
// RUN_ACCUM (with RUN_PAIRING) one folded (L, R) per bucket set; RUN_PARTIAL one partial per bucket set -> mx->d_partial
// (sharded mixes); RUN_XCHG (+ RUN_ROOT) the device-side exchange over the lead's channel, the root's summed window sums in
// the lead's d_wsums_fin.  *fail = the context whose call failed.
static int mix_enqueue(h2v_mix* mx, int mode, h2v_ctx** fail) {
  h2v_ctx* ctx = mx->m[0];
  *fail = ctx;
  cudaStream_t s = ctx->stream;
  const MsmGeom& g = mx->geom;
  CKC(cudaMemsetAsync(mx->b.hist.p, 0, 4 * ((size_t)g.nb() * g.G + 2 * SIZE_BINS), s));
  // (direct launches: the lead's events time the joint stages, h2v_last_timings)
  if (!ctx->capturing) CKC(cudaEventRecord(ctx->ev[0], s));
  CKC(cudaEventRecord(mx->ev_fork, s));
  // fold coefficients of every group, written into the members' arrays: on the lead's auxiliary stream while the proofs are
  // parsed (every member's d_r holds the r_i of the whole call)
  CKC(cudaStreamWaitEvent(ctx->stream_aux, mx->ev_fork, 0));
  KLAUNCH_P(false, k_rlc_scan_groups, mx->groups, RLC_NT, 0, ctx->stream_aux, mx->m[mx->active[0]]->d_r.as<Fr>(), mx->d_grange.as<u32>(),
            mx->d_seg.as<MixSeg>(), (u32)mx->m.size());
  CKC(cudaEventRecord(ctx->ev_join, ctx->stream_aux));
  u32 sh_max = 0;
  for (u32 mi : mx->active) {
    h2v_ctx* mb = mx->m[mi];
    sh_max = std::max<u32>(sh_max, mb->hd.n_shared);
    *fail = mb;
    if (mb != ctx) {
      cudaError_t e = cudaStreamWaitEvent(mb->stream, mx->ev_fork, 0);
      if (e != cudaSuccess) {
        mb->err = std::string("cudaStreamWaitEvent: ") + cudaGetErrorString(e);
        return -2;
      }
    }
    int rc = enqueue_stages(mb, false);
    if (rc) return rc;
    if (mb != ctx) {
      *fail = ctx;
      CKC(cudaEventRecord(mx->ev_join[mi], mb->stream));
      CKC(cudaStreamWaitEvent(s, mx->ev_join[mi], 0));
    }
  }
  *fail = ctx;
  CKC(cudaStreamWaitEvent(s, ctx->ev_join, 0));
  if (!ctx->capturing) CKC(cudaEventRecord(ctx->ev[3], s));  // MSM = [3] -> [4], pairing = [4] -> [5]
  {
    NvtxRange nv_("h2v:mix_msm");
    if (sh_max) KLAUNCH(k_shared_reduce_seg, dim3((u32)mx->segs.size(), sh_max), 256, 0, s, mx->d_seg.as<MixSeg>());
    const MixTerms src{mx->d_seg.as<MixSeg>(), (u32)mx->segs.size()};
    int rc = enqueue_buckets(ctx, g, mx->b, s, TermArrays{}, src, nullptr, 0);
    if (rc) return rc;
  }
  // one check per group over its bucket sets; a sharded mix (one group) exchanges one blob per bucket set
  return enqueue_tail(ctx, mode, TailArgs{g, mx->b.wsums.as<G1Jac>(), mx->lines(), mx->groups, mx->sets, mx->run, mx->d_partial.as<u8>()});
}

static u64 graph_key(const h2v_mix* mx, int mode) {
  KeyHash k;
  const h2v_ctx* lead = mx->m[0];
  k.mix((mode & RUN_ACCUM) ? 1 : 0);
  // (not the split of the members' proofs over the groups: the segment table and the group ranges are device data)
  k.mix(mx->groups);
  for (u32 mi : mx->active) {
    h2v_ctx* mb = mx->m[mi];
    k.mix((u64)(size_t)mb);
    k.mix(graph_key(mb, 0));  // the member's shape, options and buffers (what enqueue_stages and the segment read)
    k.mix(mx->set_of_class[mx->cls_of[mi]]);  // the class assignment (bucket set of the member)
  }
  hash_geom(k, mx->geom);
  const DevBuf* bufs[] = {&mx->b.dig, &mx->b.hist, &mx->b.off, &mx->b.cursor, &mx->b.order, &mx->b.sorted, &mx->b.buckets, &mx->b.wsums,
                          &mx->b.partials_msm, &mx->b.tiles, &mx->d_seg, &mx->d_grange, &mx->d_ssum, &lead->d_M, &lead->d_gsums, &lead->d_verdict, &lead->d_acc_bytes};
  for (const DevBuf* b : bufs) k.mix((u64)(size_t)b->p);
  k.mix((u64)(size_t)mx->lines());
  k.mix(mx->run);
  if (mode & (RUN_PARTIAL | RUN_XCHG)) {  // sharded launch sets: the mode (root or not), the partial buffers and the lead's channel
    const h2v_ctx::Comm& cm = lead->comm;
    k.mix((u64)mode);
    k.mix((u64)(size_t)mx->d_partial.p);
    k.mix((u64)(size_t)lead->d_wsums_fin.p);
    k.mix((u64)(size_t)cm.window);
    k.mix((u64)(size_t)cm.d_peers ^ (u64)(size_t)cm.d_dyn << 1 ^ (u64)(size_t)cm.d_done << 2);
    k.mix((u64)cm.lay.rank | (u64)cm.lay.world << 32);
    k.mix(cm.lay.max_groups);
  }
  return k.h | 1;
}
}  // extern "C++"

// the launch set on the lead's stream: graph replay (capture on a miss) or, with the lead's graphs off, direct launches
static int mix_run(h2v_mix* mx, int mode, h2v_ctx** fail) {
  h2v_ctx* lead = mx->m[0];
  *fail = lead;
  h2v_ctx* ctx = lead;
  cudaStream_t s = lead->stream;
  // the members' uploads were queued on their own streams: the launch set (forked from the lead's stream) follows them
  for (u32 mi : mx->active) {
    if (mi == 0) continue;
    CKC(cudaEventRecord(mx->ev_join[mi], mx->m[mi]->stream));
    CKC(cudaStreamWaitEvent(s, mx->ev_join[mi], 0));
  }
  lead->stages_timed = !lead->use_graphs;
  if (!lead->use_graphs) return mix_enqueue(mx, mode, fail);
  // (every member is marked capturing, the lead too when it has no proofs: mix_enqueue records the lead's events)
  GraphSlot* gs = nullptr;
  int rc = graph_lookup(mx->graphs, mx->graph_clock, graph_key(mx, mode), mx->m.data(), mx->m.size(), s, [&] { return mix_enqueue(mx, mode, fail); }, &gs);
  if (rc) return rc;
  CKC(cudaGraphLaunch(gs->exec, s));
  lead->launches += gs->kernels;
  return 0;
}

// bucket sets of a batch in which member m has counts[m] proofs: one per params class with proofs, numbered in class order
static void mix_assign_sets(h2v_mix* mx, const u32* counts) {
  const u32 C = (u32)mx->class_rep.size();
  mx->set_of_class.assign(C, ~0u);
  for (u32 i = 0; i < mx->m.size(); i++)
    if (counts[i]) mx->set_of_class[mx->cls_of[i]] = 0;
  mx->sets = 0;
  for (u32 c = 0; c < C; c++)
    if (mx->set_of_class[c] != ~0u) mx->set_of_class[c] = mx->sets++;
}
static u32 mix_count_sets(const h2v_mix* mx, const u32* counts) {
  std::vector<bool> used(mx->class_rep.size(), false);
  for (u32 i = 0; i < mx->m.size(); i++)
    if (counts[i]) used[mx->cls_of[i]] = true;
  return (u32)std::count(used.begin(), used.end(), true);
}

// batch_accum in class order from one 128 B (L, R) per bucket set; a class without proofs adds nothing: all-zero bytes.
// qcounts != null: one group of a grouped batch, whose member counts these are (a class with proofs elsewhere in the call but
// none in this group is all-zero too)
static void mix_class_accum(const h2v_mix* mx, const u8* acc, u8* batch_accum, const u32* qcounts = nullptr) {
  for (u32 c = 0; c < mx->set_of_class.size(); c++) {
    bool has = mx->set_of_class[c] != ~0u;
    if (has && qcounts) {
      has = false;
      for (u32 i = 0; i < mx->m.size(); i++) has |= mx->cls_of[i] == c && qcounts[i] != 0;
    }
    if (!has) memset(batch_accum + 128 * (size_t)c, 0, 128);
    else memcpy(batch_accum + 128 * (size_t)c, acc + 128 * (size_t)mx->set_of_class[c], 128);
  }
}

// Validation and upload of a mixed batch of `groups` fold groups: qcounts[q * K + m] proofs of member m in group q, in call
// order (group-major, member-major inside a group) in proofs / offsets.  They are proofs [gbase, gbase + n) of the member-major
// concatenation of gcounts[m] proofs (a whole batch: gcounts = the members' totals, gbase = 0; a shard: one group).  The fold
// coefficients and the bucket sets are those of the global batch.  Window geometry: max_shard = 0 the mix's own choice over its
// terms, otherwise every rank's common choice for shards of up to max_shard proofs (mix_shard_bound).  Then the segment table,
// the group ranges, the joint MSM's buffers and the lines.  Everything up to the first upload_impl is host-only.
static int mix_upload(h2v_mix* mx, u32 groups, const u32* qcounts, const u32* gcounts, u64 gbase, u32 max_shard, const u8* proofs, const u64* proof_off,
                      const u8* instances, const u64* inst_off, const u8* rlc, u64 seed, h2v_ctx** fail) {
  const u32 K = (u32)mx->m.size();
  h2v_ctx* lead = mx->m[0];
  *fail = nullptr;
  u64 N = 0, n = 0;
  std::vector<u32> local(K, 0);  // the members' totals
  for (u32 q = 0; q < groups; q++)
    for (u32 i = 0; i < K; i++) local[i] += qcounts[(size_t)q * K + i];
  for (u32 i = 0; i < K; i++) {
    N += gcounts[i];
    n += local[i];
  }
  if (N == 0 || N > 0xFFFFFFFFull) {
    mx->err = "a mixed batch needs between 1 and 2^32 - 1 proofs";
    return -1;
  }
  if (rlc && !fold_scalars_ok(rlc, N)) {  // before any member is uploaded
    mx->err = FOLD_SCALARS_ERR;
    return -1;
  }
  // caller data: validated as upload_impl validates a context's batch
  if (proof_off[0] != 0 || inst_off[0] != 0 || (!proofs && proof_off[n]) || (!instances && inst_off[n])) {
    mx->err = "offset arrays must start at 0";
    return -1;
  }
  for (u64 j = 0; j < n; j++) {
    if (proof_off[j + 1] < proof_off[j] || inst_off[j + 1] < inst_off[j] || proof_off[j + 1] - proof_off[j] > 0x7FFFFFFFull ||
        inst_off[j + 1] - inst_off[j] > 0x03FFFFFFull) {
      mx->err = "offset arrays must be non-decreasing with per-proof sizes below 2^31 bytes / 2^26 scalars";
      return -1;
    }
  }
  u64 terms = 0;
  for (u32 i = 0; i < K; i++) {
    const h2v_ctx* c = mx->m[i];
    if (c->opt_fold_groups > 1 || c->opt_shard_hint) {
      mx->err = "member " + std::to_string(i) + " has a pending fold-group or shard-hint option: mixed batches do not combine with them";
      return -1;
    }
    if (local[i]) terms += (u64)local[i] * (msm_points(c->hd) + msm_mo(c->hd)) + (u64)groups * c->hd.n_shared;
  }
  // term ids carry the sign in bit 31 (k_msm_scatter): the limit of upload_impl, over the whole mix
  if (terms >= (1ull << 31)) {
    mx->err = "mixed batch too large for the 32-bit index space of the MSM (split it into several batches)";
    return -1;
  }
  // fold randomness, defined over the call indices (c_i = prod_{i' > i in the same group} r_i'): explicit scalars, the mix's
  // key, the test seed, or one key drawn from the OS for this batch; the same key is set on every member
  RlcKey key{};
  bool keyed = false;
  if (!rlc && mx->has_key) {
    key = mx->key;
    keyed = true;
  } else if (!rlc && seed == 0) {
    if (os_entropy(&key, sizeof(key)) != 0) {
      mx->err = "no OS entropy for the fold coefficients (getrandom failed)";
      return -2;
    }
    keyed = true;
  }
  mx->has_key = false;
  mx->opt_shard_hint = 0;
  mx->ran = false;
  mx->xchg_root = false;
  mx->counts = local;
  mx->groups = groups;
  mx->call_base = gbase;
  mx->active.clear();
  for (u32 i = 0; i < K; i++)
    if (local[i]) mx->active.push_back(i);
  // 1. every member's proofs of all groups, in group order, as one upload whose r_i are those of the whole call
  std::vector<u32> Pm(K), Mm(K), Sm(K);
  std::vector<u64> first(groups * (size_t)K);  // position in the call of the first proof of (group, member)
  {
    u64 at = 0;
    for (u32 q = 0; q < groups; q++)
      for (u32 i = 0; i < K; i++) {
        first[(size_t)q * K + i] = at;
        at += qcounts[(size_t)q * K + i];
      }
  }
  for (u32 i = 0; i < K; i++) {
    h2v_ctx* c = mx->m[i];
    Pm[i] = msm_points(c->hd);
    Mm[i] = msm_mo(c->hd);
    Sm[i] = c->hd.n_shared;
    if (!local[i]) continue;
    std::vector<u64> po(1, 0), io(1, 0);
    UploadPieces pcs;
    for (u32 q = 0; q < groups; q++) {
      const u32 cnt = qcounts[(size_t)q * K + i];
      const u64 f = first[(size_t)q * K + i];
      if (!cnt) continue;
      for (u32 j = 1; j <= cnt; j++) {
        po.push_back(po.back() + proof_off[f + j] - proof_off[f + j - 1]);
        io.push_back(io.back() + inst_off[f + j] - inst_off[f + j - 1]);
      }
      pcs.proofs.emplace_back(proofs ? proofs + proof_off[f] : nullptr, proof_off[f + cnt] - proof_off[f]);
      pcs.instances.emplace_back(instances ? instances + 32 * inst_off[f] : nullptr, 32 * (inst_off[f + cnt] - inst_off[f]));
    }
    if (keyed) {
      c->opt_key = key;
      c->opt_has_key = true;
    }
    *fail = c;
    // (one piece: the member's proofs are contiguous in the call and upload_impl copies them directly)
    int rc = upload_impl(c, local[i], pcs.proofs[0].first, po.data(), pcs.instances[0].first, io.data(), rlc, keyed ? 0 : seed, gbase, N,
                         pcs.proofs.size() > 1 ? &pcs : nullptr);
    if (rc) return rc;
  }
  // 2. bucket sets (group-major: one per params class with proofs in the global batch, in class order, per group), segment
  // table, group ranges, joint geometry, buffers, lines
  mix_assign_sets(mx, gcounts);
  std::vector<u32> set_of_member(K, 0);
  for (u32 i = 0; i < K; i++)
    if (mx->set_of_class[mx->cls_of[i]] != ~0u) set_of_member[i] = mx->set_of_class[mx->cls_of[i]];
  const u32 nseg = groups * K;
  mx->segs.assign(nseg, MixSeg{});
  unsigned long long total = 0;
  mix_layout_groups(groups, K, qcounts, Pm.data(), Mm.data(), Sm.data(), set_of_member.data(), mx->sets, gbase, mx->segs.data(), &total);
  u32 sh_all = 0;  // shared bases of one group over the members with proofs
  std::vector<u32> sh_off(K, 0);
  for (u32 i : mx->active) {
    sh_off[i] = sh_all;
    sh_all += Sm[i];
  }
  std::vector<u64> right_terms(mx->sets), left_terms(mx->sets);  // per params class with proofs, over all groups
  for (u32 i : mx->active) {
    right_terms[set_of_member[i]] += (u64)local[i] * Pm[i] + (u64)groups * Sm[i];
    left_terms[set_of_member[i]] += (u64)local[i] * Mm[i];
  }
  h2v_ctx* ctx = lead;
  *fail = lead;
  CKC(cudaSetDevice(lead->device));
  CKC(mx->d_ssum.ensure(32 * ((size_t)groups * sh_all + 1)));
  for (u32 sg = 0; sg < nseg; sg++) {
    MixSeg& s = mx->segs[sg];
    const u32 i = sg % K;
    if (!local[i]) continue;
    h2v_ctx* c = mx->m[i];
    s.right = c->d_right.as<Fr>();
    s.left = c->d_left.as<Fr>();
    s.shared = c->d_shared.as<Fr>();
    s.coef = c->mb.coef.as<Fr>();
    s.shared_sum = mx->d_ssum.as<Fr>() + (size_t)(sg / K) * sh_all + sh_off[i];
    s.pts = c->d_pts.as<G1Affine>();
    s.shared_pts = c->pv().sec<G1Affine>(c->hd.off_shared_pts);
  }
  mx->grange.assign(groups + 1, 0);
  if (groups == 1) {
    mx->grange[1] = (u32)N;  // (a shard scans the whole global batch and writes its own range)
  } else {
    for (u32 q = 0; q < groups; q++) {
      u64 nq = 0;
      for (u32 i = 0; i < K; i++) nq += qcounts[(size_t)q * K + i];
      mx->grange[q + 1] = mx->grange[q] + (u32)nq;
    }
  }
  if (max_shard) {  // every rank the same (c, W): the partials add up window-wise
    unsigned long long rb = 0, lb = 0;
    mix_shard_bound(K, Pm.data(), Mm.data(), Sm.data(), gcounts, max_shard, &rb, &lb);
    mx->geom = mix_geom(max_shard, (u32)total, (u32)std::min(rb, 0xFFFFFFFFull), (u32)std::min(lb, 0xFFFFFFFFull), mx->sets, 1);
  } else {
    // (per group: the largest class's terms over the groups; from the members' totals, so a new split keeps the geometry)
    const u32 big = (u32)(std::max_element(right_terms.begin(), right_terms.end()) - right_terms.begin());
    mx->geom = mix_geom((u32)N, (u32)total, (u32)((right_terms[big] + groups - 1) / groups), (u32)((left_terms[big] + groups - 1) / groups),
                        mx->sets * groups, groups);
  }
  mx->run = mix_line_run(mx->sets, mx->geom.W[0], mx->geom.W[1], line_run(groups));
  CKC(ensure_msm_bufs(mx->geom, mx->b, 0, true));
  CKC(mx->d_seg.ensure(sizeof(MixSeg) * nseg));
  CKC(cudaMemcpyAsync(mx->d_seg.p, mx->segs.data(), sizeof(MixSeg) * nseg, cudaMemcpyHostToDevice, lead->stream));
  CKC(mx->d_grange.ensure(4 * ((size_t)groups + 1)));
  CKC(cudaMemcpyAsync(mx->d_grange.p, mx->grange.data(), 4 * ((size_t)groups + 1), cudaMemcpyHostToDevice, lead->stream));
  CKC(lead->d_M.ensure(sizeof(E12) * (H2V_ATE_ITERS + MILLER_SEGS) * (size_t)groups));  // one check of up to 128 pairs per group
  CKC(lead->d_gsums.ensure(sizeof(G1Jac) * 128 * (size_t)groups));
  CKC(lead->d_verdict.ensure(4 * (size_t)groups + 16));
  CKC(lead->d_acc_bytes.ensure(128 * (size_t)mx->sets * groups));
  if (max_shard) {
    CKC(mx->d_partial.ensure((size_t)H2V_PARTIAL_BYTES * mx->sets));
    CKC(lead->d_wsums_fin.ensure(sizeof(G1Jac) * 128 * (size_t)mx->sets));
  }
  return ensure_lines(mx, pair_geom_run(mx->geom, mx->run));
}

static void mix_mark_ran(h2v_mix* mx) {
  for (h2v_ctx* c : mix_active(mx)) {
    c->verdicts_on_device = false;
    c->ran = true;
  }
  mx->ran = true;
}

// statuses of the upload's proofs in call order; attribute: the members' proofs are re-checked on their own first
// (poly/strategy.rs:26-30), with gverd (one word per group, non-zero = accepted) only those of rejected groups.
// *all_ok = every status is H2V_OK.
static int mix_statuses(h2v_mix* mx, bool attribute, const u32* gverd, u8* status, bool* all_ok, h2v_ctx** fail) {
  *all_ok = true;
  const u32 K = (u32)mx->m.size();
  for (u32 i : mx->active) {
    h2v_ctx* c = mx->m[i];
    *fail = c;
    bool attr = attribute;
    if (attr && gverd) {
      std::vector<u32> acc(mx->counts[i], 0);
      bool any_acc = false, any_rej = false;
      for (u32 q = 0; q < mx->groups; q++) {
        const MixSeg& sg = mx->segs[(size_t)q * K + i];
        for (u32 j = 0; j < sg.n; j++) acc[sg.j0 + j] = gverd[q] ? 1u : 0u;
        if (sg.n) (gverd[q] ? any_acc : any_rej) = true;
      }
      attr = any_rej;
      if (any_rej && any_acc) c->attr_accepted.swap(acc);
    }
    int rc = attr ? attribute_impl(c) : 0;
    if (!rc) rc = download_status(c, nullptr);
    if (rc) return rc;
    const u32* hs = c->h_status.as<u32>();
    for (u32 q = 0; q < mx->groups; q++) {
      const MixSeg& sg = mx->segs[(size_t)q * K + i];
      u8* out = status + (sg.call0 - mx->call_base);
      for (u32 j = 0; j < sg.n; j++) {
        out[j] = (u8)hs[sg.j0 + j];
        *all_ok &= out[j] == ST_OK;
      }
    }
  }
  return 0;
}

// The grouped mixed batch (a plain mix: one group): upload, one launch set with one pairing check per group, statuses, verdicts.
static int mix_verify_impl(h2v_mix* mx, u32 groups, const u32* counts, const u8* proofs, const u64* proof_off, const u8* instances,
                           const u64* inst_off, const u8* rlc, u64 seed, u8* status, u8* group_verdicts, u8* batch_accum, int* verdict,
                           h2v_ctx** fail) {
  h2v_ctx* lead = mx->m[0];
  *fail = nullptr;
  if (!counts || !proof_off || !inst_off || !status || !verdict) {
    mx->err = "null argument";
    return -1;
  }
  if (groups == 0 || groups > 1024) {
    mx->err = "a grouped mixed batch takes 1 .. 1024 groups";
    return -1;
  }
  const u32 K = (u32)mx->m.size();
  std::vector<u32> totals(K, 0);
  for (u32 q = 0; q < groups; q++) {
    u64 nq = 0;
    for (u32 i = 0; i < K; i++) {
      nq += counts[(size_t)q * K + i];
      totals[i] += counts[(size_t)q * K + i];  // (wraps only when the call exceeds 2^32 proofs, refused below)
    }
    if (nq == 0 && groups > 1) {
      mx->err = "group " + std::to_string(q) + " has no proofs";
      return -1;
    }
  }
  {
    u64 N = 0;
    for (u32 q = 0; q < groups; q++)
      for (u32 i = 0; i < K; i++) N += counts[(size_t)q * K + i];
    if (N == 0 || N > 0xFFFFFFFFull) {
      mx->err = "a mixed batch needs between 1 and 2^32 - 1 proofs";
      return -1;
    }
  }
  {
    int rc = mix_upload(mx, groups, counts, totals.data(), 0, 0, proofs, proof_off, instances, inst_off, rlc, seed, fail);
    if (rc) return rc;
  }
  // 3. stages + joint MSM + one pairing check per group (one graph)
  {
    int rc = mix_run(mx, RUN_PAIRING | (batch_accum ? RUN_ACCUM : 0), fail);
    if (rc) return rc;
  }
  h2v_ctx* ctx = lead;
  *fail = lead;
  CKC(lead->h_verd.ensure(4 * (size_t)groups + 16));
  CKC(cudaMemcpyAsync(lead->h_verd.p, lead->d_verdict.p, 4 * (size_t)groups, cudaMemcpyDeviceToHost, lead->stream));
  std::vector<u8> acc(batch_accum ? 128 * (size_t)mx->sets * groups : 0);
  if (batch_accum) CKC(cudaMemcpyAsync(acc.data(), lead->d_acc_bytes.p, acc.size(), cudaMemcpyDeviceToHost, lead->stream));
  CKC(ctx_sync(lead));
  const std::vector<u32> hv(lead->h_verd.as<u32>(), lead->h_verd.as<u32>() + groups);  // (attribution reuses the lead's staging)
  if (batch_accum)
    for (u32 q = 0; q < groups; q++)
      mix_class_accum(mx, acc.data() + 128 * (size_t)mx->sets * q, batch_accum + 128 * mx->class_rep.size() * q, counts + (size_t)q * K);
  bool accepted = true;
  for (u32 v : hv) accepted &= v != 0;
  // 4. statuses; after a rejected check the proofs of the rejected groups are re-checked on their own (poly/strategy.rs:26-30)
  mix_mark_ran(mx);
  bool all_ok = false;
  int rc = mix_statuses(mx, !accepted, hv.data(), status, &all_ok, fail);
  if (rc) return rc;
  int all = 1;
  for (u32 q = 0; q < groups; q++) {
    bool ok = hv[q] != 0;
    for (u32 i = mx->grange[q]; i < mx->grange[q + 1]; i++) ok &= status[i] == ST_OK;
    if (group_verdicts) group_verdicts[q] = ok ? 1 : 0;
    all &= ok ? 1 : 0;
  }
  *verdict = all;
  return 0;
}

static int mix_create(h2v_mix** out, h2v_ctx* const* members, uint32_t n_members, bool multi) {
  if (!out) {
    g_create_error = "null argument";
    return -1;
  }
  *out = nullptr;
  if (!members || n_members == 0 || n_members > MIX_MAX_MEMBERS) {
    g_create_error = "a mixed batch needs between 1 and " + std::to_string(MIX_MAX_MEMBERS) + " member contexts";
    return -1;
  }
  const h2v_ctx* lead = members[0];
  std::vector<u32> cls_of(n_members), class_rep;
  for (u32 i = 0; i < n_members; i++) {
    const h2v_ctx* c = members[i];
    if (!c || c->device < 0) {
      g_create_error = "member " + std::to_string(i) + " is not a context";
      return -1;
    }
    for (u32 j = 0; j < i; j++)
      if (members[j] == c) {
        g_create_error = "member " + std::to_string(i) + " repeats member " + std::to_string(j) + " (a context holds one batch)";
        return -1;
      }
    if (c->device != lead->device) {
      g_create_error = "member " + std::to_string(i) + " is on device " + std::to_string(c->device) + ", member 0 on device " + std::to_string(lead->device);
      return -1;
    }
    if (!multi && !params_agree(c, lead)) {
      g_create_error = "member " + std::to_string(i) + "'s params differ from member 0's in (g, g2, s_g2): their proofs cannot share one pairing check";
      return -1;
    }
    u32 k = 0;
    while (k < class_rep.size() && !params_agree(c, members[class_rep[k]])) k++;
    if (k == class_rep.size()) {
      if (k == H2V_MIX_MAX_PARAMS) {
        g_create_error = "member " + std::to_string(i) + " holds a " + std::to_string(k + 1) + "th set of KZG params: a multi-params mix takes 1 .. " +
                         std::to_string(H2V_MIX_MAX_PARAMS) + " params classes";
        return -1;
      }
      class_rep.push_back(i);
    }
    cls_of[i] = k;
  }
  h2v_mix* mx = new h2v_mix();
  mx->multi = multi;
  mx->cls_of = cls_of;
  mx->class_rep = class_rep;
  mx->m.assign(members, members + n_members);
  mx->ev_join.assign(n_members, nullptr);
  h2v_ctx* l = mx->m[0];
  for (DevBuf* d : {&mx->b.coef, &mx->b.shared_sum, &mx->b.dig, &mx->b.hist, &mx->b.off, &mx->b.cursor, &mx->b.order, &mx->b.sorted, &mx->b.buckets,
                    &mx->b.wsums, &mx->b.partials_msm, &mx->b.tiles, &mx->d_seg, &mx->d_grange, &mx->d_ssum, &mx->d_partial})
    d->st = &l->stream;
  for (auto& sl : mx->mlines.s) sl.buf.st = &l->stream;
  cudaError_t e = cudaSetDevice(l->device);
  if (e == cudaSuccess) e = cudaEventCreateWithFlags(&mx->ev_fork, cudaEventDisableTiming);
  for (u32 i = 0; i < n_members && e == cudaSuccess; i++) e = cudaEventCreateWithFlags(&mx->ev_join[i], cudaEventDisableTiming);
  if (e != cudaSuccess) {
    g_create_error = std::string("cudaEventCreate: ") + cudaGetErrorString(e);
    h2v_mix_destroy(mx);
    return -2;
  }
  *out = mx;
  return 0;
}

int h2v_mix_create(h2v_mix** out, h2v_ctx* const* members, uint32_t n_members) { return mix_create(out, members, n_members, false); }
int h2v_mix_create_multi_params(h2v_mix** out, h2v_ctx* const* members, uint32_t n_members) { return mix_create(out, members, n_members, true); }

int h2v_mix_params_classes(const h2v_mix* mx, uint32_t* class_of, uint32_t capacity) {
  if (!mx || !class_of || capacity < mx->m.size()) return -1;
  for (size_t i = 0; i < mx->m.size(); i++) class_of[i] = mx->cls_of[i];
  return (int)mx->class_rep.size();
}

void h2v_mix_destroy(h2v_mix* mx) {
  if (!mx) return;
  h2v_ctx* l = mx->m[0];
  cudaSetDevice(l->device);
  cudaStreamSynchronize(l->stream);
  for (auto& gsl : mx->graphs)
    if (gsl.exec) cudaGraphExecDestroy(gsl.exec);
  for (DevBuf* d : {&mx->b.coef, &mx->b.shared_sum, &mx->b.dig, &mx->b.hist, &mx->b.off, &mx->b.cursor, &mx->b.order, &mx->b.sorted, &mx->b.buckets,
                    &mx->b.wsums, &mx->b.partials_msm, &mx->b.tiles, &mx->d_seg, &mx->d_grange, &mx->d_ssum, &mx->d_partial})
    d->release();
  for (auto& sl : mx->mlines.s) sl.buf.release();
  cudaStreamSynchronize(l->stream);  // the stream-ordered frees
  if (mx->ev_fork) cudaEventDestroy(mx->ev_fork);
  for (cudaEvent_t ev : mx->ev_join)
    if (ev) cudaEventDestroy(ev);
  delete mx;
}

const char* h2v_mix_last_error(const h2v_mix* mx) { return mx ? mx->err.c_str() : g_create_error.c_str(); }

// rc of a mix call; a failure inside a member's call is reported as "member i: <its error>"
static int mix_report(h2v_mix* mx, int rc, h2v_ctx* fail) {
  if (rc && fail && mx->err.empty()) {
    const size_t i = std::find(mx->m.begin(), mx->m.end(), fail) - mx->m.begin();
    mx->err = "member " + std::to_string(i) + ": " + fail->err;
  }
  return rc;
}

int h2v_mix_set_rlc_key(h2v_mix* mx, const uint8_t* key32) {
  if (!mx || !key32) return -1;
  memcpy(mx->key.w, key32, 32);
  mx->has_key = true;
  return 0;
}

int h2v_mix_verify(h2v_mix* mx, const uint32_t* counts, const uint8_t* proofs, const uint64_t* proof_off, const uint8_t* instances,
                   const uint64_t* inst_off, const uint8_t* rlc_scalars, uint64_t seed, uint8_t* status, uint8_t* batch_accum, int* verdict) {
  if (!mx) return -1;
  NvtxRange nv_("h2v:mix");
  mx->err.clear();
  h2v_ctx* fail = nullptr;
  const int rc = mix_verify_impl(mx, 1, counts, proofs, proof_off, instances, inst_off, rlc_scalars, seed, status, nullptr, batch_accum, verdict, &fail);
  return mix_report(mx, rc, fail);
}

int h2v_mix_verify_groups(h2v_mix* mx, uint32_t groups, const uint32_t* counts, const uint8_t* proofs, const uint64_t* proof_off,
                          const uint8_t* instances, const uint64_t* inst_off, const uint8_t* rlc_scalars, uint64_t seed, uint8_t* status,
                          uint8_t* group_verdicts, uint8_t* batch_accum, int* verdict) {
  if (!mx) return -1;
  NvtxRange nv_("h2v:mix_groups");
  mx->err.clear();
  if (mx->opt_shard_hint) {
    mx->err = "a shard hint is pending (h2v_mix_set_shard_hint): grouped mixed batches are not sharded";
    return -1;
  }
  h2v_ctx* fail = nullptr;
  const int rc = mix_verify_impl(mx, groups, counts, proofs, proof_off, instances, inst_off, rlc_scalars, seed, status, group_verdicts, batch_accum,
                                 verdict, &fail);
  return mix_report(mx, rc, fail);
}

// ---- sharded mixed batches: one rank's share of a global mixed batch, partials per bucket set, one pairing check ----------
int h2v_mix_set_shard_hint(h2v_mix* mx, uint32_t max_shard_proofs) {
  if (!mx) return -1;
  mx->opt_shard_hint = max_shard_proofs;
  return 0;
}

size_t h2v_mix_partial_bytes(const h2v_mix* mx, const uint32_t* global_counts) {
  if (!mx || !global_counts) return 0;
  return (size_t)H2V_PARTIAL_BYTES * mix_count_sets(mx, global_counts);
}

// The checks of a shard call that need no device: local[m] = this rank's proofs of member m, *max_shard = the geometry's shard size
static int mix_shard_args(h2v_mix* mx, const uint32_t* global_counts, uint64_t global_base, uint32_t n, const uint64_t* proof_off,
                          const uint64_t* inst_off, const uint8_t* status, std::vector<u32>& local, u32* max_shard) {
  if (!global_counts || !proof_off || !inst_off || !status) {
    mx->err = "null argument";
    return -1;
  }
  u64 N = 0;
  for (u32 i = 0; i < mx->m.size(); i++) N += global_counts[i];
  if (N == 0 || N > 0xFFFFFFFFull) {
    mx->err = "a mixed batch needs between 1 and 2^32 - 1 proofs";
    return -1;
  }
  local.assign(mx->m.size(), 0);
  if (!mix_shard_counts((u32)mx->m.size(), global_counts, global_base, n, local.data())) {
    mx->err = "the shard [global_base, global_base + n) must be a non-empty range inside the global batch";
    return -1;
  }
  if (mx->opt_shard_hint && mx->opt_shard_hint < n) {
    mx->err = "the shard hint (" + std::to_string(mx->opt_shard_hint) + ") is smaller than this shard (" + std::to_string(n) + " proofs)";
    return -1;
  }
  *max_shard = mx->opt_shard_hint ? mx->opt_shard_hint : n;
  return 0;
}

static int mix_accumulate_shard_impl(h2v_mix* mx, const uint32_t* global_counts, uint64_t global_base, uint32_t n, const uint8_t* proofs,
                                     const uint64_t* proof_off, const uint8_t* instances, const uint64_t* inst_off, const uint8_t* rlc_scalars,
                                     uint64_t seed, uint8_t* status, uint8_t* partial, h2v_ctx** fail) {
  std::vector<u32> local;
  u32 max_shard = 0;
  if (!partial) {
    mx->err = "null argument";
    return -1;
  }
  int rc = mix_shard_args(mx, global_counts, global_base, n, proof_off, inst_off, status, local, &max_shard);
  if (!rc) rc = mix_upload(mx, 1, local.data(), global_counts, global_base, max_shard, proofs, proof_off, instances, inst_off, rlc_scalars, seed, fail);
  if (!rc) rc = mix_run(mx, RUN_PARTIAL, fail);
  if (rc) return rc;
  mix_mark_ran(mx);
  h2v_ctx* ctx = mx->m[0];
  *fail = ctx;
  CKC(cudaMemcpyAsync(partial, mx->d_partial.p, (size_t)H2V_PARTIAL_BYTES * mx->sets, cudaMemcpyDefault, ctx->stream));
  CKC(ctx_sync(ctx));
  bool all_ok = false;
  return mix_statuses(mx, false, nullptr, status, &all_ok, fail);
}

int h2v_mix_accumulate_shard(h2v_mix* mx, const uint32_t* global_counts, uint64_t global_base, uint32_t n, const uint8_t* proofs,
                             const uint64_t* proof_off, const uint8_t* instances, const uint64_t* inst_off, const uint8_t* rlc_scalars,
                             uint64_t seed, uint8_t* status, uint8_t* partial) {
  if (!mx) return -1;
  NvtxRange nv_("h2v:mix_shard");
  mx->err.clear();
  h2v_ctx* fail = nullptr;
  const int rc = mix_accumulate_shard_impl(mx, global_counts, global_base, n, proofs, proof_off, instances, inst_off, rlc_scalars, seed, status,
                                           partial, &fail);
  return mix_report(mx, rc, fail);
}

static int mix_finalize_impl(h2v_mix* mx, const uint32_t* global_counts, uint32_t n_partials, const uint8_t* partials, uint8_t* batch_accum,
                             int* verdict, h2v_ctx** fail) {
  if (!global_counts || !partials || !verdict) {
    mx->err = "null argument";
    return -1;
  }
  if (n_partials == 0 || n_partials > 128) {
    mx->err = "h2v_mix_finalize takes 1 .. 128 ranks' partials";
    return -1;
  }
  if (!mix_count_sets(mx, global_counts)) {
    mx->err = "a mixed batch needs between 1 and 2^32 - 1 proofs";
    return -1;
  }
  h2v_ctx* ctx = mx->m[0];
  *fail = ctx;
  CKC(cudaSetDevice(ctx->device));
  mix_assign_sets(mx, global_counts);
  const u8* d_parts = nullptr;
  MsmGeom g{};
  int rc = device_partials(ctx, partials, (size_t)H2V_PARTIAL_BYTES * n_partials * mx->sets, &d_parts);
  if (!rc) rc = partial_geom(ctx, d_parts, g);  // the geometry every rank packed with (k_sum_partials flags a rank that did not)
  if (rc) return rc;
  mx->run = mix_line_run(mx->sets, g.W[0], g.W[1], line_run(1));
  if ((rc = ensure_lines(mx, pair_geom_run(g, mx->run))) != 0) return rc;
  std::vector<u8> acc(batch_accum ? 128 * (size_t)mx->sets : 0);
  u32 all = 0;
  rc = sum_and_pair(ctx, g, mx->lines(), mx->run, n_partials, 1, mx->sets, d_parts, batch_accum ? acc.data() : nullptr, nullptr, &all);
  if (rc) return rc;
  if (batch_accum) mix_class_accum(mx, acc.data(), batch_accum);
  *verdict = (int)all;
  return 0;
}

int h2v_mix_finalize(h2v_mix* mx, const uint32_t* global_counts, uint32_t n_partials, const uint8_t* partials, uint8_t* batch_accum, int* verdict) {
  if (!mx) return -1;
  NvtxRange nv_("h2v:mix_finalize");
  mx->err.clear();
  h2v_ctx* fail = nullptr;
  const int rc = mix_finalize_impl(mx, global_counts, n_partials, partials, batch_accum, verdict, &fail);  // (before fail is read)
  return mix_report(mx, rc, fail);
}

int h2v_mix_attribute_shard(h2v_mix* mx, uint8_t* status) {
  if (!mx) return -1;
  mx->err.clear();
  if (!status || !mx->ran) {
    mx->err = status ? "no shard was processed by this mix" : "null argument";
    return -1;
  }
  h2v_ctx* fail = nullptr;
  bool all_ok = false;
  const int rc = mix_statuses(mx, true, nullptr, status, &all_ok, &fail);  // (before fail is read)
  return mix_report(mx, rc, fail);
}

static int mix_verify_shard_impl(h2v_mix* mx, const uint32_t* global_counts, uint64_t global_base, uint32_t n, const uint8_t* proofs,
                                 const uint64_t* proof_off, const uint8_t* instances, const uint64_t* inst_off, const uint8_t* rlc_scalars,
                                 uint64_t seed, uint32_t root, uint8_t* status, int* verdict, h2v_ctx** fail) {
  h2v_ctx* ctx = mx->m[0];
  const h2v_ctx::Comm& cm = ctx->comm;
  std::vector<u32> local;
  u32 max_shard = 0;
  if (!verdict) {
    mx->err = "null argument";
    return -1;
  }
  int rc = mix_shard_args(mx, global_counts, global_base, n, proof_off, inst_off, status, local, &max_shard);
  if (rc) return rc;
  if (!cm.ready || root >= cm.lay.world) {
    mx->err = "sharded exchange: the lead member (member 0) needs h2v_comm_init + h2v_comm_connect, and root < world";
    return -1;
  }
  const u32 sets = mix_count_sets(mx, global_counts);
  if (sets > cm.lay.max_groups) {
    mx->err = "sharded exchange: the lead's channel takes " + std::to_string(cm.lay.max_groups) + " partials per rank, this batch has " +
              std::to_string(sets) + " bucket sets (h2v_comm_init with max_groups >= the params classes with proofs)";
    return -1;
  }
  rc = mix_upload(mx, 1, local.data(), global_counts, global_base, max_shard, proofs, proof_off, instances, inst_off, rlc_scalars, seed, fail);
  if (rc) return rc;
  *fail = ctx;
  CKC(cudaSetDevice(ctx->device));
  CKC(comm_next_launch(ctx, root));
  if ((rc = mix_run(mx, RUN_XCHG | (root == cm.lay.rank ? RUN_ROOT : 0), fail)) != 0) return rc;
  mix_mark_ran(mx);
  *fail = ctx;
  u32 all = 0;
  if ((rc = read_verdicts(ctx, &all, true, 1)) != 0) return rc;
  mx->xchg_root = root == cm.lay.rank;
  bool all_ok = false;
  if ((rc = mix_statuses(mx, !all, nullptr, status, &all_ok, fail)) != 0) return rc;
  *verdict = (int)all;
  return 0;
}

int h2v_mix_verify_shard(h2v_mix* mx, const uint32_t* global_counts, uint64_t global_base, uint32_t n, const uint8_t* proofs, const uint64_t* proof_off,
                         const uint8_t* instances, const uint64_t* inst_off, const uint8_t* rlc_scalars, uint64_t seed, uint32_t root, uint8_t* status,
                         int* verdict) {
  if (!mx) return -1;
  NvtxRange nv_("h2v:mix_shard");
  mx->err.clear();
  h2v_ctx* fail = nullptr;
  const int rc = mix_verify_shard_impl(mx, global_counts, global_base, n, proofs, proof_off, instances, inst_off, rlc_scalars, seed, root, status,
                                       verdict, &fail);
  return mix_report(mx, rc, fail);
}

static int mix_comm_accum_impl(h2v_mix* mx, uint8_t* batch_accum) {
  if (!batch_accum || !mx->xchg_root) {
    mx->err = batch_accum ? "the last launch set of this mix was not an exchange with this rank as its root" : "null argument";
    return -1;
  }
  h2v_ctx* ctx = mx->m[0];
  std::vector<u8> acc(128 * (size_t)mx->sets);
  CKC(cudaSetDevice(ctx->device));
  // the root's summed window sums of every bucket set (lead's d_wsums_fin)
  const int rc = enqueue_fold_accum(ctx, mx->geom, ctx->d_wsums_fin.as<G1Jac>(), mx->sets, ctx->d_acc_bytes.as<u8>(), false);
  if (rc) return rc;
  CKC(cudaMemcpyAsync(acc.data(), ctx->d_acc_bytes.p, acc.size(), cudaMemcpyDeviceToHost, ctx->stream));
  CKC(ctx_sync(ctx));
  mix_class_accum(mx, acc.data(), batch_accum);
  return 0;
}

int h2v_mix_comm_last_batch_accum(h2v_mix* mx, uint8_t* batch_accum) {
  if (!mx) return -1;
  mx->err.clear();
  return mix_report(mx, mix_comm_accum_impl(mx, batch_accum), mx->m[0]);
}

// ---- persistent accumulators: the reference's AccumulatorStrategy as a value that lives across calls ---------------
// The DualMSM state (R, L) and one record (R_b, L_b) per absorb or merge live in device memory of the anchor's device.
// Absorbs from several contexts (and merges, finalize, reset) are ordered through the accumulator's event: the stream that
// works on the state waits on it first and records it afterwards.
struct h2v_acc {
  h2v_ctx* anchor = nullptr;  // not owned: params, device, stream of merge / finalize, prepared unit lines
  std::string err;
  u32 cap = 0, count = 0;  // record array: capacity, records used (host mirror of the device counter)
  bool has_key = false;    // one-shot fold key of the next absorb (h2v_acc_set_rlc_key)
  RlcKey key{};
  cudaEvent_t ev = nullptr;
  G1Jac* d_acc = nullptr;      // (R, L)
  G1Jac* d_records = nullptr;  // [cap][2] (R_b, L_b)
  u32* d_words = nullptr;      // [0] record counter, [1, 1 + ACC_CHECKS) verdicts of one pass of pair checks
  u8* d_merge = nullptr;       // merge operand: (R, L) Jacobian | r | 1 (Fr, Montgomery)
  E12* d_M = nullptr;          // Miller scratch of one pass of pair checks
  HostBuf h_buf;               // pinned staging of the read-backs and of the merge operand
};
static constexpr u32 ACC_CHECKS = 1024;  // pair checks per pass (d_M: E12[ACC_CHECKS][H2V_ATE_ITERS] = 25 MB)
static constexpr u32 ACC_MAX_RECORDS = 1u << 20;
static constexpr size_t ACC_MERGE_BYTES = 2 * sizeof(G1Jac) + 2 * sizeof(Fr);

#define CKA(call)                                                    \
  do {                                                               \
    cudaError_t e_ = (call);                                         \
    if (e_ != cudaSuccess) {                                         \
      a->err = std::string(#call) + ": " + cudaGetErrorString(e_);   \
      return -2;                                                     \
    }                                                                \
  } while (0)

static int acc_fail(h2v_acc* a, const char* who, const h2v_ctx* c, int rc) {
  a->err = std::string(who) + ": " + c->err;
  return rc;
}

// empty accumulator and record array, on stream s (which waited on a->ev)
static int acc_clear(h2v_acc* a, cudaStream_t s) {
  CKA(cudaMemsetAsync(a->d_acc, 0, 2 * sizeof(G1Jac), s));  // Z = 0: the identity
  CKA(cudaMemsetAsync(a->d_words, 0, 4, s));
  CKA(cudaEventRecord(a->ev, s));
  a->count = 0;
  return 0;
}

int h2v_acc_create(h2v_acc** out, h2v_ctx* anchor, uint32_t max_absorbs) {
  if (!out) {
    g_create_error = "null argument";
    return -1;
  }
  *out = nullptr;
  if (!anchor || anchor->device < 0) {
    g_create_error = "an accumulator needs an anchor context (it supplies the params, the device and the prepared G2 lines)";
    return -1;
  }
  if (max_absorbs == 0 || max_absorbs > ACC_MAX_RECORDS) {
    g_create_error = "max_absorbs must be between 1 and " + std::to_string(ACC_MAX_RECORDS);
    return -1;
  }
  h2v_acc* a = new h2v_acc();
  a->anchor = anchor;
  a->cap = max_absorbs;
  cudaError_t e = cudaSetDevice(anchor->device);
  if (e == cudaSuccess) e = cudaEventCreateWithFlags(&a->ev, cudaEventDisableTiming);
  if (e == cudaSuccess) e = cudaMalloc(&a->d_acc, 2 * sizeof(G1Jac));
  if (e == cudaSuccess) e = cudaMalloc(&a->d_records, 2 * sizeof(G1Jac) * (size_t)max_absorbs);
  if (e == cudaSuccess) e = cudaMalloc(&a->d_words, 4 * (size_t)(1 + ACC_CHECKS));
  if (e == cudaSuccess) e = cudaMalloc(&a->d_merge, ACC_MERGE_BYTES);
  if (e == cudaSuccess) e = cudaMalloc(&a->d_M, sizeof(E12) * H2V_ATE_ITERS * (size_t)std::min(max_absorbs, ACC_CHECKS));
  if (e == cudaSuccess) e = a->h_buf.ensure(std::max<size_t>(4 * (size_t)(1 + ACC_CHECKS), ACC_MERGE_BYTES));
  if (e == cudaSuccess && acc_clear(a, anchor->stream) == 0) e = cudaStreamSynchronize(anchor->stream);
  else if (e == cudaSuccess) e = cudaErrorUnknown;  // (a->err names the call)
  if (e != cudaSuccess) {
    g_create_error = "creating the accumulator: " + (a->err.empty() ? std::string(cudaGetErrorString(e)) : a->err);
    h2v_acc_destroy(a);
    return -2;
  }
  *out = a;
  return 0;
}

void h2v_acc_destroy(h2v_acc* a) {
  if (!a) return;
  cudaSetDevice(a->anchor->device);
  if (a->ev) cudaEventSynchronize(a->ev);
  for (void* p : {(void*)a->d_acc, (void*)a->d_records, (void*)a->d_words, (void*)a->d_merge, (void*)a->d_M})
    if (p) cudaFree(p);
  a->h_buf.release();
  if (a->ev) cudaEventDestroy(a->ev);
  delete a;
}

const char* h2v_acc_last_error(const h2v_acc* a) { return a ? a->err.c_str() : g_create_error.c_str(); }

int h2v_acc_set_rlc_key(h2v_acc* a, const uint8_t* key32) {
  if (!a || !key32) return -1;
  memcpy(a->key.w, key32, 32);
  a->has_key = true;
  return 0;
}

int h2v_acc_reset(h2v_acc* a) {
  if (!a) return -1;
  a->err.clear();
  CKA(cudaSetDevice(a->anchor->device));
  CKA(cudaStreamWaitEvent(a->anchor->stream, a->ev, 0));
  return acc_clear(a, a->anchor->stream);
}

int h2v_acc_absorb(h2v_acc* a, h2v_ctx* ctx, uint32_t n, const uint8_t* proofs, const uint64_t* proof_off, const uint8_t* instances,
                   const uint64_t* inst_off, const uint8_t* rlc_scalars, uint64_t seed, uint8_t* status, uint32_t* index) {
  if (!a) return -1;
  NvtxRange nv_("h2v:absorb");
  a->err.clear();
  // refusals before any device call: the accumulator and the context stay as they are
  if (!ctx || ctx->device < 0 || !status) {
    a->err = "null argument";
    return -1;
  }
  if (ctx->device != a->anchor->device) {
    a->err = "the context is on device " + std::to_string(ctx->device) + ", the accumulator's anchor on device " + std::to_string(a->anchor->device);
    return -1;
  }
  if (!params_agree(ctx, a->anchor)) {
    a->err = "the context's params differ from the anchor's in (g, g2, s_g2): its proofs cannot share the accumulator's pairing check";
    return -1;
  }
  if (n == 0) {
    a->err = "an absorb needs at least one proof";
    return -1;
  }
  if (a->count >= a->cap) {
    a->err = "the record array is full (max_absorbs = " + std::to_string(a->cap) + "): finalize or reset the accumulator first";
    return -1;
  }
  if (ctx->opt_fold_groups > 1 || ctx->opt_shard_hint) {
    a->err = "the context has a pending fold-group or shard-hint option: absorbs do not combine with them";
    return -1;
  }
  const bool set_key = !rlc_scalars && a->has_key;
  if (set_key) {
    ctx->opt_key = a->key;
    ctx->opt_has_key = true;
  }
  int rc = upload_impl(ctx, n, proofs, proof_off, instances, inst_off, rlc_scalars, seed, 0, n);
  if (rc) {
    if (set_key) ctx->opt_has_key = false;
    return acc_fail(a, "context", ctx, rc);
  }
  a->has_key = false;
  const MsmGeom& g = ctx->geom;
  if (g.W[0] > ACC_TREE_SPAN || g.W[1] > ACC_TREE_SPAN) {
    a->err = "window geometry with more than " + std::to_string(ACC_TREE_SPAN) + " windows per channel";
    return -1;
  }
  CKA(cudaStreamWaitEvent(ctx->stream, a->ev, 0));  // outside any capture: the previous absorb, merge or reset first
  ctx->absorb = h2v_ctx::AbsorbTarget{a->d_acc, a->d_records, a->d_words, a->cap};
  rc = run_impl(ctx, RUN_ABSORB);
  ctx->absorb = h2v_ctx::AbsorbTarget{};
  if (rc) return acc_fail(a, "context", ctx, rc);
  CKA(cudaEventRecord(a->ev, ctx->stream));
  if (index) *index = a->count;
  a->count++;
  rc = download_status(ctx, status);
  return rc ? acc_fail(a, "context", ctx, rc) : 0;
}

// 64 bytes x | y, little-endian canonical, all-zero = identity -> Jacobian (Montgomery); false if not a point
static bool acc_read_point(const u8* b, G1Jac& out) {
  bool zero = true;
  for (int i = 0; i < 64; i++) zero &= b[i] == 0;
  out = G1Jac::identity();
  if (zero) return true;
  const Fq x = Fq::load_le(b), y = Fq::load_le(b + 32);
  if (x.geq_mod() || y.geq_mod()) return false;
  const G1Affine p{Fq::from_canonical(x), Fq::from_canonical(y)};
  if (!g1_on_curve(p)) return false;
  out = G1Jac::from_affine(p);
  return true;
}

int h2v_acc_merge(h2v_acc* a, const uint8_t* in128, const uint8_t* r32) {
  if (!a) return -1;
  a->err.clear();
  if (!in128) {
    a->err = "null argument";
    return -1;
  }
  G1Jac rl[2];  // (R, L): the bytes are L | R
  if (!acc_read_point(in128 + 64, rl[0]) || !acc_read_point(in128, rl[1])) {
    a->err = "merge operand is not two canonical G1 points (x | y little-endian, coordinates below p, on the curve)";
    return -1;
  }
  Fr sc[2] = {Fr::zero(), Fr::one()};
  if (r32) {
    if (!fold_scalars_ok(r32, 1)) {  // r = 0 would drop every earlier absorb out of the final check
      a->err = FOLD_SCALARS_ERR;
      return -1;
    }
    sc[0] = Fr::from_canonical(Fr::load_le(r32));
  } else {
    u8 wide[64];
    if (os_entropy(wide, sizeof(wide)) != 0) {
      a->err = "no OS entropy for the merge scalar (getrandom failed)";
      return -1;
    }
    sc[0] = Fr::from_uniform(wide);
  }
  if (a->count >= a->cap) {
    a->err = "the record array is full (max_absorbs = " + std::to_string(a->cap) + "): finalize or reset the accumulator first";
    return -1;
  }
  h2v_ctx* ctx = a->anchor;
  cudaStream_t s = ctx->stream;
  CKA(cudaSetDevice(ctx->device));
  CKA(cudaStreamWaitEvent(s, a->ev, 0));
  u8* hb = a->h_buf.as<u8>();
  memcpy(hb, rl, sizeof(rl));
  memcpy(hb + sizeof(rl), sc, sizeof(sc));
  CKA(cudaMemcpyAsync(a->d_merge, hb, ACC_MERGE_BYTES, cudaMemcpyHostToDevice, s));
  // the absorb kernel on one window per channel of weight 2^0: acc <- r acc + P, record P
  const AccGeom ag{{1, 1}, {0, 0}};
  const Fr* dr = (const Fr*)(a->d_merge + sizeof(rl));
  KLAUNCH_P(false, k_acc_absorb, 1, 32 * cdiv(4 * acc_items(ag), 32), 0, s, ag, (const G1Jac*)a->d_merge, dr, dr + 1, a->d_acc, a->d_records, a->d_words, a->cap);
  CKA(cudaEventRecord(a->ev, s));
  a->count++;
  CKA(ctx_sync(ctx));  // (the staging buffer is reused by the next call)
  return 0;
}

int h2v_acc_get(const h2v_acc* ca, uint8_t* out128) {
  h2v_acc* a = (h2v_acc*)ca;
  if (!a || !out128) return -1;
  a->err.clear();
  h2v_ctx* ctx = a->anchor;
  CKA(cudaSetDevice(ctx->device));
  CKA(cudaStreamWaitEvent(ctx->stream, a->ev, 0));
  CKA(cudaMemcpyAsync(a->h_buf.p, a->d_acc, 2 * sizeof(G1Jac), cudaMemcpyDeviceToHost, ctx->stream));
  CKA(ctx_sync(ctx));
  const G1Jac* rl = a->h_buf.as<G1Jac>();
  for (int ch = 0; ch < 2; ch++) {  // bytes L | R, the batch_accum layout
    u8* o = out128 + (ch == 0 ? 64 : 0);
    G1Affine p;
    if (!g1_to_affine(rl[ch], p)) {
      memset(o, 0, 64);
      continue;
    }
    p.x.to_canonical().store_le(o);
    p.y.to_canonical().store_le(o + 32);
  }
  return 0;
}

int h2v_acc_finalize(h2v_acc* a, int* verdict, uint8_t* absorb_verdicts, uint32_t capacity) {
  if (!a) return -1;
  NvtxRange nv_("h2v:acc_finalize");
  a->err.clear();
  if (!verdict) {
    a->err = "null argument";
    return -1;
  }
  h2v_ctx* ctx = a->anchor;
  cudaStream_t s = ctx->stream;
  CKA(cudaSetDevice(ctx->device));
  MsmGeom unit{};
  unit.c[0] = unit.c[1] = 1;
  unit.W[0] = unit.W[1] = 1;
  int unit_slot = -1;
  int rc = ensure_lines(ctx, unit, &unit_slot);  // lines of -G2 (pair 0, right) and [s]G2 (pair 1, left)
  if (rc) return acc_fail(a, "anchor", ctx, rc);
  const G2Line* unit_lines = ctx->lines.s[unit_slot].buf.as<G2Line>();
  const PairSkip none{nullptr, nullptr, 1, 0};
  u32* hv = a->h_buf.as<u32>();
  CKA(cudaStreamWaitEvent(s, a->ev, 0));
  // DualMSM::check (msm.rs:185-203) on the accumulator: e(L, [s]G2) e(R, -G2) == 1
  if ((rc = launch_pair_checks(ctx, a->d_acc, 1, unit_lines, a->d_M, a->d_words + 1, none)) != 0) return acc_fail(a, "anchor", ctx, rc);
  CKA(cudaMemcpyAsync(hv, a->d_words + 1, 4, cudaMemcpyDeviceToHost, s));
  CKA(ctx_sync(ctx));
  const bool ok = hv[0] != 0;
  if (absorb_verdicts)
    for (u32 i = 0; i < a->count && i < capacity; i++) absorb_verdicts[i] = 1;
  // rejected: one check per record names the absorbs (and merges) that fail; the caller re-verifies those batches
  for (u32 base = 0; !ok && base < a->count; base += ACC_CHECKS) {
    const u32 cnt = std::min(ACC_CHECKS, a->count - base);
    if ((rc = launch_pair_checks(ctx, a->d_records + 2 * (size_t)base, cnt, unit_lines, a->d_M, a->d_words + 1, none)) != 0) return acc_fail(a, "anchor", ctx, rc);
    CKA(cudaMemcpyAsync(hv, a->d_words + 1, 4 * (size_t)cnt, cudaMemcpyDeviceToHost, s));
    CKA(ctx_sync(ctx));
    if (absorb_verdicts)
      for (u32 i = 0; i < cnt && base + i < capacity; i++) absorb_verdicts[base + i] = hv[i] ? 1 : 0;
  }
  *verdict = ok ? 1 : 0;
  return acc_clear(a, s);  // finalize(self) consumes the strategy
}

}  // extern "C"
