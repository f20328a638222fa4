// The "verification plan": everything `verify_proof` derives from (params, vk) alone, compiled once
// on the host (plan_build.cpp) into one flat blob that the kernels interpret per proof.
//
// It encodes, for one VerifyingKey:
//   * the transcript schedule          reference lib.rs:66-253 (+ shplonk.rs:195-200 / gwc.rs:68-76)
//   * the expression list for h(x)     lib.rs:273-344, permutation.rs:189-288, lookup.rs:159-230, shuffle.rs:148-203
//   * the query list, folded into rotation sets (SHPLONK, shplonk.rs:58-149) or point groups (GWC, gwc.rs:138-163)
//   * domain constants                 domain.rs:34-140 (omega powers, 1/n), permutation.rs:268 (DELTA powers)
//   * the shared MSM bases (fixed / sigma commitments, G) and the prepared G2 lines of msm.rs:186-187
// Commitment identity in the reference is pointer equality (query.rs:63-74); here it is (kind, index).
#pragma once
#include "field.cuh"

namespace h2v {

enum : u32 { MO_SHPLONK = 0, MO_GWC = 1 };
enum : u32 { HASH_BLAKE2B = 0, HASH_KECCAK = 1 };

// per-proof status codes (plonk/mod.rs:19-32 error classes)
enum : u32 {
  ST_OK = 0,
  ST_INVALID_INSTANCES = 1,
  ST_TRANSCRIPT = 2,
  ST_OPENING = 3,
  ST_CONSTRAINT_SYSTEM_FAILURE = 4,
  ST_WOULD_PANIC = 5,  // x^n = 1 (vanishing.rs:100), z_diff = 0 (shplonk.rs:215), x = 0
};

enum : u32 { T_ABS_VK = 0, T_ABS_INST = 1, T_POINTS = 2, T_SCALARS = 3, T_SQUEEZE = 4 };
struct TranscriptOp {
  u32 kind, count;
};

enum : u32 { E_GATE = 0, E_PERM_FIRST, E_PERM_LAST, E_PERM_LINK, E_PERM_PROD, E_LOOKUP, E_SHUFFLE };
struct ExprOp {
  u32 kind, a, b, c, d, e;
};
struct PolyRange {
  u32 term_begin, term_end;
};
struct PolyTerm {
  u32 coeff, var_begin, var_end;  // coeff: index into fr_consts
};
struct PolyVar {
  u32 val, pow;  // val: value-table index
};
struct PermCol {
  u32 col_val, sigma_val;
};
struct LookupDesc {  // also used for shuffles (v_in, v_in_inv, v_tab unused there)
  u32 in_begin, in_end, tab_begin, tab_end;  // ranges into polylist[]
  u32 v_prod, v_prod_next, v_in, v_in_inv, v_tab;
};

enum : u32 { CM_PROOF = 0, CM_FIXED = 1, CM_SIGMA = 2, CM_HMSM = 3 };
struct SetPoint {
  u32 rot_id;  // index into the distinct-rotation table
  u32 invden;  // fr_consts index: prod_{m != k} (omega^{r_k} - omega^{r_m})^-1
};
struct SetCommit {
  u32 kind, idx, eval_begin;  // setevals[eval_begin + k] = value index of the eval at set point k
};
struct RotSet {
  u32 pt_begin, pt_end, cm_begin, cm_end, diff_begin, diff_end;
};
struct GwcPoint {
  u32 rot_id, q_begin, q_end;
};
struct GwcQuery {
  u32 kind, idx, eval_val;
};
struct InstQuery {
  u32 column, offset;  // offset = max_rotation - rotation (lib.rs:212)
};

static constexpr u32 H2V_MAX_ROT = 32;        // distinct opening rotations
static constexpr u32 H2V_MAX_LEVALS = 64;     // blinding_factors + 2
static constexpr u32 H2V_MAX_INST_Q = 16;     // instance queries
static constexpr u32 H2V_MAX_SET_POINTS = 8;  // points per rotation set
static constexpr u32 H2V_PLAN_MAGIC = 0x48325631u;

struct PlanHeader {
  u32 magic, total_bytes;
  u32 k, multiopen, hash;
  u32 n_points, n_scalars, n_items, first_mo_item, n_mo, proof_len;
  u32 n_challenges;  // number of squeezes C
  u32 n_inst_cols, n_inst_q, inst_max_rot, inst_min_rot_abs;
  u32 n_vals, v_chal, v_inst, v_expected_h;  // value table: [0,S) scalars | challenges | instance evals | expected_h
  u32 ch_theta, ch_beta, ch_gamma, ch_y, ch_x, ch_mo0, ch_mo1, ch_mo2;  // squeeze-order indices
  u32 blinding;  // blinding_factors() (vk.rs:396-401)
  u32 c_vk_repr, c_one_over_n, c_omega, c_omega_inv, c_delta, c_lrot;  // fr_consts indices; c_lrot..: omega^rot, rot=-(bf+1)..0
  u32 h_slot, n_h;             // point slots of the h pieces
  u32 n_fixed, n_sigma, n_shared;  // shared bases: fixed | sigma | G
  u32 n_rot, n_sets, n_gwc_points;
  u32 n_tops, n_exprops, n_consts;
  // section offsets (bytes from the start of the blob)
  u32 off_tops, off_exprops, off_polys, off_terms, off_vars, off_polylist, off_permcols, off_lookups;
  u32 off_consts, off_pt_item, off_sc_item, off_rot, off_sets, off_setpts, off_setcms, off_setevals, off_diffs;
  u32 off_gwcpts, off_gwcq, off_instq, off_shared_pts, off_lines0, off_lines1;
  // aggregation contexts (agg.cuh): the carried accumulator's two points (lhs, rhs) follow the proof points in the per-proof
  // MSM layout; n_carry = 2 there, 0 for every other context.  off_agg: 4 * agg_limbs AggCell.
  u32 n_carry, agg_limbs, agg_bits, off_agg;
};

// Per-proof point slots of the MSM: the proof points, then the carried lhs and rhs.  The last msm_mo() slots are the left
// channel's points: the multi-open points, then lhs (left scalar 0) and rhs (left scalar rho); the right channel covers every
// slot (lhs: rho, rhs: 0).  n_points / n_mo themselves count what is read from the proof.
H2V_HD u32 msm_points(const PlanHeader& h) { return h.n_points + h.n_carry; }
H2V_HD u32 msm_mo(const PlanHeader& h) { return h.n_mo + h.n_carry; }

struct PlanView {
  const u8* base;
  H2V_HD const PlanHeader& h() const { return *(const PlanHeader*)base; }
  template <class T>
  H2V_HD const T* sec(u32 off) const {
    return (const T*)(base + off);
  }
  H2V_HD const Fr& cst(u32 i) const { return sec<Fr>(h().off_consts)[i]; }
};

}  // namespace h2v
