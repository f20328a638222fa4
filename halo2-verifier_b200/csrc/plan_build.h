// Host-side plan compiler interface (see plan_build.cpp).
#pragma once
#include <stddef.h>

#include <string>
#include <vector>

#include "plan.h"

// SerdeFormat of the reference (helpers.rs:7-19)
#define H2V_FMT_PROCESSED 0
#define H2V_FMT_RAW_BYTES 1
#define H2V_FMT_RAW_BYTES_UNCHECKED 2

namespace h2v {

struct PlanInfo {
  u32 k, n_points, n_scalars, n_challenges, proof_len, n_inst_cols, n_shared, n_mo;
  // G2 arguments of the pairing check as raw Montgomery limbs (x.c0 | x.c1 | y.c0 | y.c1):
  // q_left = [s]G2 (pairs with the left accumulator), q_right = -G2   (msm.rs:186-199)
  u32 q_left[32], q_right[32];
  // VK lint (h2v_ctx_vk_lint): places where the reference's own VerifyingKey::write and ::read disagree, so that bytes
  // produced by `write` would be read into a DIFFERENT constraint system than the one written (SURVEY.md section 4)
  std::vector<std::string> lint;
};

// The KZG accumulator an aggregation circuit carries in its instances (agg.cuh): LimbsEncoding<limbs, bits> and the
// 4 * limbs (column, row) cells of lhs.x, lhs.y, rhs.x, rhs.y
struct AggSpec {
  u32 limbs, bits;
  const u32* cells;
};

// circuit_instances: how many circuit instances one proof transcript carries (`instances.len()` of verify_proof; 1 in
// every reference test).  agg != null: an aggregation context; the spec is validated here (before any device call).
int build_plan(const u8* params, size_t params_len, int params_fmt, const u8* vk, size_t vk_len, int vk_fmt, int multiopen,
               int hash, std::vector<u8>& blob, PlanInfo& info, std::string& err, u32 circuit_instances = 1, const AggSpec* agg = nullptr);

// Miller-line tables of the G2 multiples [2^(c w)] Q used by the window-decomposed pairing check
// (pairing_cta.cuh): pairs 0..W0-1 = right channel (Q = -G2, c = c0), then W1 pairs of the left
// channel (Q = [s]G2, c = c1); H2V_ATE_LINES G2Line entries per pair.
void build_window_lines(const PlanInfo& info, u32 c0, u32 W0, u32 c1, u32 W1, std::vector<u8>& out);

}  // namespace h2v
