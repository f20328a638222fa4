// Host side: parse ParamsKZG / VerifyingKey bytes and compile the verification plan (plan.h).
//
// Formats restated from the reference (paths under halo2_verifier/src):
//   helpers.rs:7-19,40-98,120-164        SerdeFormat; BE integers; curve / field (de)serialisation
//   poly/kzg/commitment.rs:155-207       ParamsKZG::read_custom (k little-endian)
//   plonk/vk.rs:76-115,274-365,514-546   VerifyingKey / ConstraintSystem / IndexedExpressionPoly readers
//   plonk/circuit.rs:53-65               Column<Any> codec;  permutation.rs:37-44,164-176;  lookup.rs:51-68; shuffle.rs:85-102
// Structure derived from the VK follows lib.rs:86-253 (transcript order), lib.rs:273-344 (expressions),
// lib.rs:349-414 (queries), shplonk.rs:58-149 (rotation sets), gwc.rs:138-163 (point groups).
// A VK on which the reference would panic at verify time (missing permutation query, empty polynomial,
// out-of-range variable) is rejected here with an error instead.
#include "plan_build.h"

#include <string.h>

#include <algorithm>
#include <map>

#include "agg.cuh"
#include "tower.cuh"

namespace h2v {

namespace {

struct Rd {
  const u8* p;
  size_t n, pos = 0;
  bool fail = false;
  Rd(const u8* p_, size_t n_) : p(p_), n(n_) {}
  const u8* take(size_t k) {
    if (fail || pos + k > n) {
      fail = true;
      return nullptr;
    }
    const u8* r = p + pos;
    pos += k;
    return r;
  }
  u32 u8_() {
    const u8* b = take(1);
    return b ? b[0] : 0;
  }
  u32 u16() {
    const u8* b = take(2);
    return b ? ((u32)b[0] << 8) | b[1] : 0;
  }
  u32 u32_() {
    const u8* b = take(4);
    return b ? ((u32)b[0] << 24) | ((u32)b[1] << 16) | ((u32)b[2] << 8) | b[3] : 0;
  }
  int32_t i32() { return (int32_t)u32_(); }
};

struct Err {
  std::string msg;
};
#define H2V_REQUIRE(cond, text) \
  do {                          \
    if (!(cond)) throw Err{text}; \
  } while (0)

bool is_all_zero(const u8* b, size_t n) {
  for (size_t i = 0; i < n; i++)
    if (b[i]) return false;
  return true;
}

// identity is represented as (0, 0), which is not on the curve
G1Affine read_g1(Rd& r, int fmt) {
  G1Affine out;
  out.x = Fq::zero();
  out.y = Fq::zero();
  if (fmt == H2V_FMT_PROCESSED) {
    const u8* b = r.take(32);
    H2V_REQUIRE(b, "truncated G1 point");
    u8 tmp[32];
    memcpy(tmp, b, 32);
    if (is_all_zero(tmp, 32)) return out;
    H2V_REQUIRE(g1_decompress(tmp, out), "invalid G1 point encoding");
    return out;
  }
  const u8* b = r.take(64);
  H2V_REQUIRE(b, "truncated G1 point");
  out.x = Fq::load_le(b);
  out.y = Fq::load_le(b + 32);
  if (fmt == H2V_FMT_RAW_BYTES) {
    H2V_REQUIRE(!out.x.geq_mod() && !out.y.geq_mod(), "G1 coordinate not reduced");
    if (!(out.x.is_zero() && out.y.is_zero())) H2V_REQUIRE(g1_on_curve(out), "G1 point not on curve");
  }
  return out;
}

Fr read_fr(Rd& r, int fmt) {
  const u8* b = r.take(32);
  H2V_REQUIRE(b, "truncated field element");
  Fr v = Fr::load_le(b);
  if (fmt != H2V_FMT_RAW_BYTES_UNCHECKED) H2V_REQUIRE(!v.geq_mod(), "field element not reduced");
  return fmt == H2V_FMT_PROCESSED ? Fr::from_canonical(v) : v;
}

Fq2 fq2_pow(const Fq2& a, const u32* e, int nlimbs) {
  Fq2 r = Fq2::one();
  for (int i = nlimbs * 32 - 1; i >= 0; i--) {
    r = r.sqr();
    if ((e[i >> 5] >> (i & 31)) & 1) r = r * a;
  }
  return r;
}

// sqrt in Fq2 for p = 3 mod 4 (Adj & Rodriguez-Henriquez, Alg. 9); false if non-residue
bool fq2_sqrt(const Fq2& a, Fq2& out) {
  if (a.is_zero()) {
    out = a;
    return true;
  }
  u32 pm3d4[8], pm1d2[8];  // (p-3)/4, (p-1)/2
  u32 p[8];
  for (int i = 0; i < 8; i++) p[i] = FqP::mod(i);
  u32 t[8];
  memcpy(t, p, 32);
  t[0] -= 3;
  for (int i = 0; i < 8; i++) pm3d4[i] = (t[i] >> 2) | (i < 7 ? t[i + 1] << 30 : 0);
  memcpy(t, p, 32);
  t[0] -= 1;
  for (int i = 0; i < 8; i++) pm1d2[i] = (t[i] >> 1) | (i < 7 ? t[i + 1] << 31 : 0);
  Fq2 a1 = fq2_pow(a, pm3d4, 8);
  Fq2 alpha = a1.sqr() * a;
  Fq2 a0 = alpha.conj() * alpha;
  Fq2 minus_one = Fq2::one().neg();
  if (a0 == minus_one) return false;
  Fq2 x0 = a1 * a;
  if (alpha == minus_one) {
    Fq2 i_ = {Fq::zero(), Fq::one()};
    out = i_ * x0;
  } else {
    Fq2 b = fq2_pow(Fq2::one() + alpha, pm1d2, 8);
    out = b * x0;
  }
  return out.sqr() == a;
}

// G2 compressed convention: see oracle/bn254.py (g2_to_bytes) and DESIGN.md -- unpinned dependency detail.
G2Affine read_g2(Rd& r, int fmt) {
  G2Affine q;
  if (fmt == H2V_FMT_PROCESSED) {
    const u8* b = r.take(64);
    H2V_REQUIRE(b, "truncated G2 point");
    u8 tmp[64];
    memcpy(tmp, b, 64);
    const bool sign = tmp[63] & 0x80;
    H2V_REQUIRE(!(tmp[63] & 0x40) && !is_all_zero(tmp, 64), "G2 identity / flagged encoding not accepted in params");
    tmp[63] &= 0x3F;
    Fq x0 = Fq::load_le(tmp), x1 = Fq::load_le(tmp + 32);
    H2V_REQUIRE(!x0.geq_mod() && !x1.geq_mod(), "G2 coordinate not reduced");
    q.x = {Fq::from_canonical(x0), Fq::from_canonical(x1)};
    Fq2 rhs = q.x.sqr() * q.x + twist_b();
    H2V_REQUIRE(fq2_sqrt(rhs, q.y), "invalid G2 point encoding");
    if ((bool)(q.y.c0.to_canonical().l[0] & 1) != sign) q.y = q.y.neg();
    return q;
  }
  const u8* b = r.take(128);
  H2V_REQUIRE(b, "truncated G2 point");
  q.x = {Fq::load_le(b), Fq::load_le(b + 32)};
  q.y = {Fq::load_le(b + 64), Fq::load_le(b + 96)};
  if (fmt == H2V_FMT_RAW_BYTES) {
    H2V_REQUIRE(!q.x.c0.geq_mod() && !q.x.c1.geq_mod() && !q.y.c0.geq_mod() && !q.y.c1.geq_mod(), "G2 coordinate not reduced");
    H2V_REQUIRE(g2_on_curve(q), "G2 point not on curve");
  }
  return q;
}

struct Poly {
  std::vector<std::pair<u32, std::vector<std::pair<u32, u32>>>> terms;
};
Poly read_poly(Rd& r) {
  Poly p;
  (void)r.u32_();  // num_vars
  u32 nt = r.u32_();
  H2V_REQUIRE(!r.fail && nt < (1u << 24), "bad polynomial");
  for (u32 t = 0; t < nt; t++) {
    u32 coeff = r.u16();
    u32 nv = r.u32_();
    H2V_REQUIRE(!r.fail && nv < (1u << 20), "bad polynomial term");
    std::vector<std::pair<u32, u32>> vars;
    for (u32 v = 0; v < nv; v++) {
      u32 var = r.u32_(), pw = r.u32_();
      vars.push_back({var, pw});
    }
    p.terms.push_back({coeff, vars});
  }
  H2V_REQUIRE(!r.fail, "truncated polynomial");
  return p;
}

struct Query {
  u32 kind, idx;
  int32_t rot;
  u32 eval_val;
};

template <class T>
u32 append(std::vector<u8>& blob, const std::vector<T>& v) {
  while (blob.size() % 16) blob.push_back(0);
  u32 off = (u32)blob.size();
  const u8* p = (const u8*)v.data();
  blob.insert(blob.end(), p, p + v.size() * sizeof(T));
  return off;
}

}  // namespace

// `m` = circuit instances carried by ONE proof transcript (`instances.len()` of verify_proof, lib.rs:63,92,117,134):
// advice / lookup / permutation / shuffle commitments and evaluations, the instance columns, the expressions and the
// queries repeat per instance in the reference's interleaving; fixed columns, sigma, the random polynomial and h are shared.
int build_plan(const u8* params, size_t params_len, int params_fmt, const u8* vkb, size_t vk_len, int vk_fmt,
               int multiopen, int hash, std::vector<u8>& blob, PlanInfo& info, std::string& err, u32 m, const AggSpec* agg) {
  // write emits len() of the instance / fixed query lists but read takes exactly one query per column
  // (plonk/vk.rs:243-251 vs 310-322): with more queries than columns everything after them is read misaligned
  static const char* const query_hint =
      "VerifyingKey::write emits every instance / fixed query but ::read takes one per column (plonk/vk.rs:243-251 vs 310-322): "
      "a constraint system that queries an instance or fixed column at more than one rotation does not survive its own write/read round trip";
  bool in_vk = false;
  try {
    H2V_REQUIRE(m >= 1 && m <= 16, "circuit instances per proof out of range (1..16)");
    H2V_REQUIRE(multiopen == MO_SHPLONK || multiopen == MO_GWC, "unknown multiopen scheme");
    H2V_REQUIRE(hash == HASH_BLAKE2B || hash == HASH_KECCAK, "unknown transcript hash");
    // ---------------- params (kzg/commitment.rs:155-207)
    Rd pr(params, params_len);
    const u8* kb = pr.take(4);
    H2V_REQUIRE(kb, "truncated params");
    const u32 pk = (u32)kb[0] | ((u32)kb[1] << 8) | ((u32)kb[2] << 16) | ((u32)kb[3] << 24);
    G1Affine g = read_g1(pr, params_fmt);
    H2V_REQUIRE(!(g.x.is_zero() && g.y.is_zero()), "params: g is the identity");
    G2Affine g2 = read_g2(pr, params_fmt);
    G2Affine s_g2 = read_g2(pr, params_fmt);

    // ---------------- verifying key (vk.rs:76-115)
    Rd r(vkb, vk_len);
    in_vk = true;
    const u32 k = r.u32_();
    H2V_REQUIRE(!r.fail && k >= 1 && k <= 28, "vk: k out of range");
    H2V_REQUIRE(k == pk, "params.k != vk.k");
    const u32 n_fixed_commit = r.u32_();
    H2V_REQUIRE(!r.fail && n_fixed_commit < (1u << 20), "vk: bad fixed commitment count");
    std::vector<G1Affine> fixed_commitments;
    for (u32 i = 0; i < n_fixed_commit; i++) fixed_commitments.push_back(read_g1(r, vk_fmt));
    const u32 cs_degree = r.u32_();
    const u32 num_fixed_columns = r.u32_(), num_advice_columns = r.u32_(), num_instance_columns = r.u32_();
    const u32 num_selectors = r.u32_(), num_challenges = r.u32_(), num_gates = r.u32_(), num_lookups = r.u32_();
    const u32 num_shuffles = r.u32_(), num_coeff = r.u32_();
    H2V_REQUIRE(!r.fail, "truncated vk header");
    H2V_REQUIRE(cs_degree >= 3 && cs_degree < 64, "vk: cs_degree out of range");  // chunk_len = cs_degree - 2 >= 1
    H2V_REQUIRE((num_fixed_columns | num_advice_columns | num_instance_columns | num_selectors | num_challenges | num_gates |
                 num_lookups | num_shuffles) < (1u << 20) && num_coeff <= 65536, "vk: implausible counts");
    {  // extended_k <= S (domain.rs:46-52)
      u32 ek = k;
      while ((1ull << ek) < (1ull << k) * (u64)(cs_degree - 1)) ek++;
      H2V_REQUIRE(ek <= 28, "vk: extended domain exceeds 2-adicity");
    }
    std::vector<u32> advice_phase(num_advice_columns), challenge_phase(num_challenges), num_advice_queries(num_advice_columns);
    for (auto& p : advice_phase) p = r.u8_();
    for (auto& p : challenge_phase) p = r.u8_();
    u64 total_aq = 0;
    for (auto& c : num_advice_queries) {
      c = r.u32_();
      total_aq += c;
    }
    H2V_REQUIRE(!r.fail && total_aq < (1u << 20), "vk: bad advice query counts");
    struct AQ {
      u32 col, phase;
      int32_t rot;
    };
    std::vector<AQ> advice_queries;
    for (u64 i = 0; i < total_aq; i++) {
      AQ q;
      q.col = r.u32_();
      q.phase = r.u8_();
      q.rot = r.i32();
      advice_queries.push_back(q);
    }
    std::vector<std::pair<u32, int32_t>> instance_queries, fixed_queries;
    for (u32 i = 0; i < num_instance_columns; i++) {
      u32 c = r.u32_();
      instance_queries.push_back({c, r.i32()});
    }
    for (u32 i = 0; i < num_fixed_columns; i++) {
      u32 c = r.u32_();
      fixed_queries.push_back({c, r.i32()});
    }
    const u32 n_perm = r.u32_();
    H2V_REQUIRE(!r.fail && n_perm < (1u << 20), "vk: bad permutation column count");
    std::vector<std::pair<u32, u32>> perm_cols;
    for (u32 i = 0; i < n_perm; i++) {
      u32 idx = r.u32_(), typ = r.u8_();
      H2V_REQUIRE(typ == 255 || typ == 254 || typ <= 2, "Invalid phase for advice column");
      perm_cols.push_back({idx, typ});
    }
    std::vector<Poly> gates;
    for (u32 i = 0; i < num_gates; i++) gates.push_back(read_poly(r));
    struct Arg {
      std::vector<Poly> in, tab;
    };
    std::vector<Arg> lookups, shuffles;
    for (int pass = 0; pass < 2; pass++) {
      for (u32 i = 0; i < (pass == 0 ? num_lookups : num_shuffles); i++) {
        u32 m = r.u32_();
        H2V_REQUIRE(!r.fail && m < (1u << 16), "vk: bad argument expression count");
        Arg a;
        for (u32 e = 0; e < m; e++) {  // READ side: interleaved pairs (lookup.rs:58-61, shuffle.rs:92-95)
          a.in.push_back(read_poly(r));
          a.tab.push_back(read_poly(r));
        }
        if (m > 1)  // the reference's write emits all inputs, then all tables (lookup.rs:42-47, shuffle.rs:76-81)
          info.lint.push_back(std::string(pass == 0 ? "lookup " : "shuffle ") + std::to_string(i) + " has " + std::to_string(m) +
                              " expression pairs: VerifyingKey::write emits [inputs..., tables...] but VerifyingKey::read takes (input, table) pairs interleaved (" +
                              (pass == 0 ? "plonk/lookup.rs:42-47 vs 58-61" : "plonk/shuffle.rs:76-81 vs 92-95") +
                              "); this plan follows `read`, so bytes that came from `write` pair the wrong expressions");
        (pass == 0 ? lookups : shuffles).push_back(a);
      }
    }
    std::vector<Fr> coeff_vals;
    for (u32 i = 0; i < num_coeff; i++) coeff_vals.push_back(read_fr(r, vk_fmt));
    std::vector<G1Affine> sigma_commitments;
    for (u32 i = 0; i < n_perm; i++) sigma_commitments.push_back(read_g1(r, vk_fmt));
    if (num_selectors)  // bit-packed selector columns, unused by verification (vk.rs:92-102)
      H2V_REQUIRE(r.take((size_t)num_selectors * ((((size_t)1 << k) + 7) / 8)), "truncated selectors");
    Fr transcript_repr = read_fr(r, vk_fmt);
    H2V_REQUIRE(!r.fail, "truncated vk");
    {
      // symptoms of that misalignment that survive as a "successful" parse: a column queried twice among the first
      // `columns` entries, bytes left over after transcript_repr (a failed parse gets the hint appended to its message)
      auto dup = [](const std::vector<std::pair<u32, int32_t>>& q) {
        for (size_t a = 0; a < q.size(); a++)
          for (size_t b = a + 1; b < q.size(); b++)
            if (q[a].first == q[b].first) return true;
        return false;
      };
      if (dup(instance_queries) || dup(fixed_queries))
        info.lint.push_back(std::string("an instance / fixed column appears twice among the per-column queries: ") + query_hint);
      if (r.pos < vk_len) info.lint.push_back(std::to_string(vk_len - r.pos) + " bytes follow transcript_repr: " + query_hint);
    }
    in_vk = false;

    // ---------------- validation of what verify_proof would index
    const u32 A = (u32)advice_queries.size(), F = (u32)fixed_queries.size(), I = (u32)instance_queries.size();
    for (auto& q : advice_queries) H2V_REQUIRE(q.col < num_advice_columns, "advice query column out of range");
    for (auto& q : fixed_queries) H2V_REQUIRE(q.first < n_fixed_commit, "fixed query column out of range");
    for (auto& q : instance_queries) H2V_REQUIRE(q.first < num_instance_columns, "instance query column out of range");
    H2V_REQUIRE((u64)I * m <= H2V_MAX_INST_Q, "too many instance queries for this build");

    // blinding_factors (vk.rs:396-401), phases (vk.rs:403-411)
    u32 bf = 1;
    if (!num_advice_queries.empty()) bf = *std::max_element(num_advice_queries.begin(), num_advice_queries.end());
    bf = std::max(3u, bf) + 2;
    H2V_REQUIRE(bf + 2 <= H2V_MAX_LEVALS, "too many blinding factors for this build");
    u32 max_phase = 0;
    for (u32 p : advice_phase) max_phase = std::max(max_phase, p);
    const u32 chunk_len = cs_degree - 2;
    const u32 n_sets = n_perm ? (n_perm + chunk_len - 1) / chunk_len : 0;
    const u32 n_h = cs_degree - 1;
    const u32 L = num_lookups, SH = num_shuffles;

    // ---------------- constants table
    std::vector<Fr> consts;
    auto add_const = [&](const Fr& v) {
      consts.push_back(v);
      return (u32)consts.size() - 1;
    };
    Fr omega;
    {
      const u32 root_mont[8] = {0xb639feb8u, 0x9632c7c5u, 0x0d0ff299u, 0x985ce340u, 0x01b0ecd8u, 0xb2dd8800u, 0x6d98ce29u, 0x1d69070du};
      for (int i = 0; i < 8; i++) omega.l[i] = root_mont[i];
      for (u32 i = k; i < 28; i++) omega = omega.sqr();  // ROOT_OF_UNITY^(2^(S-k)), domain.rs:50-72
    }
    const Fr omega_inv = omega.inv();
    Fr delta;
    {
      const u32 delta_mont[8] = {0xefd78855u, 0x9a0c322bu, 0x249b563cu, 0x46e82d14u, 0xe0b0b7a7u, 0x5983a663u, 0xaaa111adu, 0x22ab452bu};
      for (int i = 0; i < 8; i++) delta.l[i] = delta_mont[i];
    }
    auto omega_pow = [&](int64_t rot) { return rot >= 0 ? omega.pow_u64((u64)rot) : omega_inv.pow_u64((u64)(-rot)); };

    PlanHeader hd;
    memset(&hd, 0, sizeof(hd));
    hd.magic = H2V_PLAN_MAGIC;
    hd.k = k;
    hd.multiopen = multiopen;
    hd.hash = hash;
    hd.blinding = bf;
    hd.c_vk_repr = add_const(transcript_repr);
    {
      Fr nn = Fr::from_u32(1);
      Fr two = Fr::from_u32(2);
      for (u32 i = 0; i < k; i++) nn = nn * two;
      hd.c_one_over_n = add_const(nn.inv());
    }
    hd.c_omega = add_const(omega);
    hd.c_omega_inv = add_const(omega_inv);
    hd.c_delta = add_const(delta);
    hd.c_lrot = (u32)consts.size();
    for (int32_t rot = -(int32_t)(bf + 1); rot <= 0; rot++) add_const(omega_pow(rot));
    const u32 c_coeff = (u32)consts.size();
    for (auto& c : coeff_vals) add_const(c);

    // ---------------- transcript schedule + slot maps (lib.rs:86-253)
    std::vector<TranscriptOp> tops;
    std::vector<u32> pt_item, sc_item;
    u32 item = 0, n_squeeze = 0;
    auto op = [&](u32 kind, u32 count) {
      if (count == 0 && kind != T_ABS_VK && kind != T_ABS_INST) return;
      tops.push_back({kind, count});
      if (kind == T_POINTS)
        for (u32 i = 0; i < count; i++) pt_item.push_back(item++);
      if (kind == T_SCALARS)
        for (u32 i = 0; i < count; i++) sc_item.push_back(item++);
      if (kind == T_SQUEEZE) n_squeeze += count;
    };
    op(T_ABS_VK, 0);
    op(T_ABS_INST, 0);
    std::vector<u32> advice_slot((size_t)m * num_advice_columns, 0xFFFFFFFFu), user_ch_sq(num_challenges, 0xFFFFFFFFu);  // [pi][column]
    for (u32 phase = 0; phase <= max_phase; phase++) {
      u32 cnt = 0;
      for (u32 pi = 0; pi < m; pi++)  // lib.rs:91-103: every instance's advice commitments of this phase
        for (u32 c = 0; c < num_advice_columns; c++)
          if (advice_phase[c] == phase) advice_slot[(size_t)pi * num_advice_columns + c] = (u32)pt_item.size() + cnt++;
      op(T_POINTS, cnt);
      cnt = 0;
      for (u32 c = 0; c < num_challenges; c++)
        if (challenge_phase[c] == phase) user_ch_sq[c] = n_squeeze + cnt++;
      op(T_SQUEEZE, cnt);
    }
    hd.ch_theta = n_squeeze;
    op(T_SQUEEZE, 1);
    const u32 slot_lookup_permuted = (u32)pt_item.size();  // per instance, 2 per lookup: input, table
    op(T_POINTS, 2 * L * m);
    hd.ch_beta = n_squeeze;
    hd.ch_gamma = n_squeeze + 1;
    op(T_SQUEEZE, 2);
    const u32 slot_perm = (u32)pt_item.size();              // [pi][set]
    const u32 slot_lookup_prod = slot_perm + n_sets * m;    // [pi][lookup]
    const u32 slot_shuffle_prod = slot_lookup_prod + L * m; // [pi][shuffle]
    const u32 slot_random = slot_shuffle_prod + SH * m;
    op(T_POINTS, (n_sets + L + SH) * m + 1);
    hd.ch_y = n_squeeze;
    op(T_SQUEEZE, 1);
    hd.h_slot = (u32)pt_item.size();
    hd.n_h = n_h;
    op(T_POINTS, n_h);
    hd.ch_x = n_squeeze;
    op(T_SQUEEZE, 1);
    // scalar slots
    // (lib.rs:219-253: advice evals per instance, fixed, random, sigma, then per instance permutation / lookup / shuffle evals)
    const u32 s_advice = 0, s_fixed = A * m, s_random = s_fixed + F, s_sigma = s_random + 1, s_perm = s_sigma + n_perm;
    const u32 n_perm_evals = n_sets ? 3 * n_sets - 1 : 0;
    const u32 s_lookup = s_perm + n_perm_evals * m, s_shuffle = s_lookup + 5 * L * m;
    const u32 S = s_shuffle + 2 * SH * m;
    op(T_SCALARS, S);
    hd.first_mo_item = item;

    // ---------------- query list (lib.rs:349-414)
    auto perm_eval = [&](u32 pi, u32 set, u32 which) { return s_perm + pi * n_perm_evals + 3 * set + which; };  // eval, next, last
    std::vector<Query> queries;
    const u32 V_EXPECTED_H_TMP = 0xFFFFFFF0u;
    for (u32 pi = 0; pi < m; pi++) {
      for (u32 qi = 0; qi < A; qi++) {
        const AQ& q = advice_queries[qi];
        const u32 slot = advice_slot[(size_t)pi * num_advice_columns + q.col];
        H2V_REQUIRE(slot != 0xFFFFFFFFu, "advice column without commitment");
        queries.push_back({CM_PROOF, slot, q.rot, s_advice + pi * A + qi});
      }
      for (u32 s = 0; s < n_sets; s++) {
        queries.push_back({CM_PROOF, slot_perm + pi * n_sets + s, 0, perm_eval(pi, s, 0)});
        queries.push_back({CM_PROOF, slot_perm + pi * n_sets + s, 1, perm_eval(pi, s, 1)});
      }
      for (u32 s = n_sets; s-- > 0;) {
        if (s == n_sets - 1) continue;  // all but the last set, in reverse (permutation.rs:318)
        queries.push_back({CM_PROOF, slot_perm + pi * n_sets + s, -(int32_t)(bf + 1), perm_eval(pi, s, 2)});
      }
      for (u32 l = 0; l < L; l++) {  // lookup.rs:232-271
        const u32 e = s_lookup + 5 * (pi * L + l), pin = slot_lookup_permuted + 2 * (pi * L + l), ptab = pin + 1, pprod = slot_lookup_prod + pi * L + l;
        queries.push_back({CM_PROOF, pprod, 0, e + 0});
        queries.push_back({CM_PROOF, pin, 0, e + 2});
        queries.push_back({CM_PROOF, ptab, 0, e + 4});
        queries.push_back({CM_PROOF, pin, -1, e + 3});
        queries.push_back({CM_PROOF, pprod, 1, e + 1});
      }
      for (u32 s = 0; s < SH; s++) {  // shuffle.rs:205-225
        const u32 e = s_shuffle + 2 * (pi * SH + s);
        queries.push_back({CM_PROOF, slot_shuffle_prod + pi * SH + s, 0, e});
        queries.push_back({CM_PROOF, slot_shuffle_prod + pi * SH + s, 1, e + 1});
      }
    }
    for (u32 qi = 0; qi < F; qi++) queries.push_back({CM_FIXED, fixed_queries[qi].first, fixed_queries[qi].second, s_fixed + qi});
    for (u32 i = 0; i < n_perm; i++) queries.push_back({CM_SIGMA, i, 0, s_sigma + i});
    queries.push_back({CM_HMSM, 0, 0, V_EXPECTED_H_TMP});
    queries.push_back({CM_PROOF, slot_random, 0, s_random});

    // distinct rotations (points are x*omega^rot: equal iff rotations agree mod n)
    const int64_t nn = (int64_t)1 << k;
    auto rot_key = [&](int32_t rot) { return (u32)((((int64_t)rot % nn) + nn) % nn); };
    std::vector<u32> rot_keys;      // first-appearance order
    std::vector<int32_t> rot_repr;  // a representative rotation
    auto rot_id = [&](int32_t rot) {
      u32 key = rot_key(rot);
      for (u32 i = 0; i < rot_keys.size(); i++)
        if (rot_keys[i] == key) return i;
      rot_keys.push_back(key);
      rot_repr.push_back(rot);
      return (u32)rot_keys.size() - 1;
    };
    for (auto& q : queries) rot_id(q.rot);
    const u32 n_rot = (u32)rot_keys.size();
    H2V_REQUIRE(n_rot <= H2V_MAX_ROT, "too many distinct rotations for this build");

    // ---------------- multiopen part of the schedule
    u32 n_mo;
    if (multiopen == MO_SHPLONK) {
      hd.ch_mo0 = n_squeeze;
      hd.ch_mo1 = n_squeeze + 1;
      op(T_SQUEEZE, 2);
      op(T_POINTS, 1);
      hd.ch_mo2 = n_squeeze;
      op(T_SQUEEZE, 1);
      op(T_POINTS, 1);
      n_mo = 2;
    } else {
      hd.ch_mo0 = n_squeeze;
      op(T_SQUEEZE, 1);
      op(T_POINTS, n_rot);
      hd.ch_mo1 = n_squeeze;
      op(T_SQUEEZE, 1);
      n_mo = n_rot;
    }
    hd.n_mo = n_mo;
    hd.n_points = (u32)pt_item.size();
    hd.n_scalars = S;
    hd.n_items = item;
    hd.proof_len = 32 * item;
    hd.n_challenges = n_squeeze;
    hd.n_inst_cols = num_instance_columns * m;  // instance-major "virtual" columns: the layout of lib.rs:76-82
    hd.n_inst_q = I * m;
    hd.v_chal = S;
    hd.v_inst = S + n_squeeze;
    hd.v_expected_h = S + n_squeeze + I * m;
    hd.n_vals = hd.v_expected_h + 1;
    for (auto& q : queries)
      if (q.eval_val == V_EXPECTED_H_TMP) q.eval_val = hd.v_expected_h;

    // instance query offsets (lib.rs:181-213)
    int32_t min_rot = 0, max_rot = 0;
    for (auto& q : instance_queries) {
      if (q.second < min_rot) min_rot = q.second;
      else if (q.second > max_rot) max_rot = q.second;
    }
    hd.inst_max_rot = (u32)max_rot;
    hd.inst_min_rot_abs = (u32)(-(int64_t)min_rot);
    std::vector<InstQuery> instq;
    for (u32 pi = 0; pi < m; pi++)
      for (auto& q : instance_queries) instq.push_back({pi * num_instance_columns + q.first, (u32)(max_rot - q.second)});

    // ---------------- expressions (lib.rs:273-344)
    std::vector<PolyRange> polys;
    std::vector<PolyTerm> terms;
    std::vector<PolyVar> vars;
    std::vector<u32> polylist;
    auto var_val = [&](u32 pi, u32 var) -> u32 {
      if (var < A) return s_advice + pi * A + var;  // this instance's advice evals
      if (var < A + F) return s_fixed + (var - A);
      if (var < A + F + I) return hd.v_inst + pi * I + (var - A - F);
      H2V_REQUIRE(var < A + F + I + num_challenges, "polynomial variable index out of range");
      u32 sq = user_ch_sq[var - A - F - I];
      H2V_REQUIRE(sq != 0xFFFFFFFFu, "challenge is never squeezed");
      return hd.v_chal + sq;
    };
    auto add_poly = [&](u32 pi, const Poly& p) -> u32 {
      H2V_REQUIRE(!p.terms.empty(), "empty polynomial (reference unwraps the first term)");
      PolyRange pr2;
      pr2.term_begin = (u32)terms.size();
      for (auto& t : p.terms) {
        H2V_REQUIRE(t.first < num_coeff, "coefficient index out of range");
        PolyTerm pt;
        pt.coeff = c_coeff + t.first;
        pt.var_begin = (u32)vars.size();
        for (auto& v : t.second) vars.push_back({var_val(pi, v.first), v.second});
        pt.var_end = (u32)vars.size();
        terms.push_back(pt);
      }
      pr2.term_end = (u32)terms.size();
      polys.push_back(pr2);
      return (u32)polys.size() - 1;
    };
    std::vector<ExprOp> eops;
    std::vector<PermCol> permcols;
    std::vector<LookupDesc> lks;
    for (u32 pi = 0; pi < m; pi++) {  // lib.rs:273-344: gates, permutation, lookups, shuffles of instance pi, then the next instance
      for (auto& g_ : gates) eops.push_back({E_GATE, add_poly(pi, g_), 0, 0, 0, 0});
      if (n_sets) {
        eops.push_back({E_PERM_FIRST, perm_eval(pi, 0, 0), 0, 0, 0, 0});
        eops.push_back({E_PERM_LAST, perm_eval(pi, n_sets - 1, 0), 0, 0, 0, 0});
        for (u32 s = 1; s < n_sets; s++) eops.push_back({E_PERM_LINK, perm_eval(pi, s, 0), perm_eval(pi, s - 1, 2), 0, 0, 0});
        const u32 pc0 = (u32)permcols.size();
        for (u32 i = 0; i < n_perm; i++) {  // get_any_query_index(column, Rotation::cur()), vk.rs:413-455
          u32 idx = perm_cols[i].first, typ = perm_cols[i].second, val = 0xFFFFFFFFu;
          if (typ == 255) {
            for (u32 q = 0; q < F && val == 0xFFFFFFFFu; q++)
              if (fixed_queries[q].first == idx && fixed_queries[q].second == 0) val = s_fixed + q;
          } else if (typ == 254) {
            for (u32 q = 0; q < I && val == 0xFFFFFFFFu; q++)
              if (instance_queries[q].first == idx && instance_queries[q].second == 0) val = hd.v_inst + pi * I + q;
          } else {
            for (u32 q = 0; q < A && val == 0xFFFFFFFFu; q++)
              if (advice_queries[q].col == idx && advice_queries[q].phase == typ && advice_queries[q].rot == 0) val = s_advice + pi * A + q;
          }
          H2V_REQUIRE(val != 0xFFFFFFFFu, "permutation column has no query at the current rotation (reference panics)");
          permcols.push_back({val, s_sigma + i});
        }
        for (u32 s = 0; s < n_sets; s++) {
          u32 b = s * chunk_len, e = std::min(n_perm, b + chunk_len);
          eops.push_back({E_PERM_PROD, perm_eval(pi, s, 0), perm_eval(pi, s, 1), pc0 + b, pc0 + e, add_const(delta.pow_u64((u64)s * chunk_len))});
        }
      }
      for (int pass = 0; pass < 2; pass++) {
        auto& args = pass == 0 ? lookups : shuffles;
        for (u32 a = 0; a < args.size(); a++) {
          LookupDesc d;
          memset(&d, 0, sizeof(d));
          d.in_begin = (u32)polylist.size();
          for (auto& p : args[a].in) polylist.push_back(add_poly(pi, p));
          d.in_end = d.tab_begin = (u32)polylist.size();
          for (auto& p : args[a].tab) polylist.push_back(add_poly(pi, p));
          d.tab_end = (u32)polylist.size();
          if (pass == 0) {
            const u32 e = s_lookup + 5 * (pi * L + a);
            d.v_prod = e; d.v_prod_next = e + 1; d.v_in = e + 2; d.v_in_inv = e + 3; d.v_tab = e + 4;
          } else {
            const u32 e = s_shuffle + 2 * (pi * SH + a);
            d.v_prod = e; d.v_prod_next = e + 1;
          }
          lks.push_back(d);
          eops.push_back({pass == 0 ? (u32)E_LOOKUP : (u32)E_SHUFFLE, (u32)lks.size() - 1, 0, 0, 0, 0});
        }
      }
    }

    // ---------------- rotation table and SHPLONK sets / GWC groups
    std::vector<u32> rot_consts;
    for (u32 i = 0; i < n_rot; i++) rot_consts.push_back(add_const(omega_pow(rot_repr[i])));
    std::vector<RotSet> sets;
    std::vector<SetPoint> setpts;
    std::vector<SetCommit> setcms;
    std::vector<u32> setevals, diffs;
    std::vector<GwcPoint> gwcpts;
    std::vector<GwcQuery> gwcq;
    if (multiopen == MO_SHPLONK) {
      // commitment -> set of rotation ids, first-appearance order (shplonk.rs:85-101)
      struct CR {
        u32 kind, idx;
        std::vector<u32> rids;
      };
      std::vector<CR> cmap;
      for (auto& q : queries) {
        u32 rid = rot_id(q.rot);
        CR* f = nullptr;
        for (auto& c : cmap)
          if (c.kind == q.kind && c.idx == q.idx) f = &c;
        if (!f) {
          cmap.push_back({q.kind, q.idx, {}});
          f = &cmap.back();
        }
        if (std::find(f->rids.begin(), f->rids.end(), rid) == f->rids.end()) f->rids.push_back(rid);
      }
      // set equality is on the SET of points (BTreeSet), shplonk.rs:110-121
      struct SetB {
        std::vector<u32> rids_sorted, rids;
        std::vector<u32> members;
      };
      std::vector<SetB> sb;
      for (u32 ci = 0; ci < cmap.size(); ci++) {
        std::vector<u32> sorted = cmap[ci].rids;
        std::sort(sorted.begin(), sorted.end());
        SetB* f = nullptr;
        for (auto& s : sb)
          if (s.rids_sorted == sorted) f = &s;
        if (!f) {
          sb.push_back({sorted, cmap[ci].rids, {}});
          f = &sb.back();
        }
        f->members.push_back(ci);
      }
      for (auto& s : sb) {
        H2V_REQUIRE(s.rids.size() <= H2V_MAX_SET_POINTS, "rotation set too large for this build");
        RotSet rs;
        rs.pt_begin = (u32)setpts.size();
        for (u32 k2 = 0; k2 < s.rids.size(); k2++) {
          Fr den = Fr::one();
          for (u32 m = 0; m < s.rids.size(); m++)
            if (m != k2) den = den * (consts[rot_consts[s.rids[k2]]] - consts[rot_consts[s.rids[m]]]);
          setpts.push_back({s.rids[k2], add_const(den.inv())});
        }
        rs.pt_end = (u32)setpts.size();
        rs.cm_begin = (u32)setcms.size();
        for (u32 ci : s.members) {
          SetCommit sc;
          sc.kind = cmap[ci].kind;
          sc.idx = cmap[ci].idx;
          sc.eval_begin = (u32)setevals.size();
          for (u32 rid : s.rids) {  // get_eval: first query matching (commitment, point), shplonk.rs:67-73
            u32 ev = 0xFFFFFFFFu;
            for (auto& q : queries)
              if (q.kind == sc.kind && q.idx == sc.idx && rot_id(q.rot) == rid) {
                ev = q.eval_val;
                break;
              }
            setevals.push_back(ev);
          }
          setcms.push_back(sc);
        }
        rs.cm_end = (u32)setcms.size();
        rs.diff_begin = (u32)diffs.size();
        for (u32 rid = 0; rid < n_rot; rid++)
          if (std::find(s.rids.begin(), s.rids.end(), rid) == s.rids.end()) diffs.push_back(rid);
        rs.diff_end = (u32)diffs.size();
        sets.push_back(rs);
      }
    } else {
      for (u32 rid = 0; rid < n_rot; rid++) {  // first-appearance order of points == rid order (gwc.rs:138-163)
        GwcPoint gp;
        gp.rot_id = rid;
        gp.q_begin = (u32)gwcq.size();
        for (auto& q : queries)
          if (rot_id(q.rot) == rid) gwcq.push_back({q.kind, q.idx, q.eval_val});
        gp.q_end = (u32)gwcq.size();
        gwcpts.push_back(gp);
      }
    }
    hd.n_rot = n_rot;
    hd.n_sets = (u32)sets.size();
    hd.n_gwc_points = (u32)gwcpts.size();

    // ---------------- shared bases and G2 lines
    hd.n_fixed = n_fixed_commit;
    hd.n_sigma = n_perm;
    hd.n_shared = n_fixed_commit + n_perm + 1;
    std::vector<G1Affine> shared_pts = fixed_commitments;
    shared_pts.insert(shared_pts.end(), sigma_commitments.begin(), sigma_commitments.end());
    shared_pts.push_back(g);
    std::vector<G2Line> lines0(H2V_ATE_LINES), lines1(H2V_ATE_LINES);
    g2_prepare(s_g2, lines0.data());  // e(left, [s]G2)
    G2Affine ng2 = g2;
    ng2.y = ng2.y.neg();
    g2_prepare(ng2, lines1.data());  // e(right, -G2)

    // ---------------- carried accumulator of an aggregation circuit (agg.cuh)
    std::vector<AggCell> agg_cells;
    if (agg) {
      H2V_REQUIRE(agg->limbs >= AGG_MIN_LIMBS && agg->limbs <= AGG_MAX_LIMBS, "aggregation spec: limbs must be in [2, 8]");
      H2V_REQUIRE(agg->bits >= 1 && agg->bits <= AGG_MAX_BITS, "aggregation spec: bits must be in [1, 128]");
      H2V_REQUIRE(agg->limbs * agg->bits >= 254, "aggregation spec: limbs * bits must be >= 254 (a coordinate of q)");
      H2V_REQUIRE(agg->cells != nullptr, "aggregation spec: cells is null");
      for (u32 i = 0; i < 4 * agg->limbs; i++) {
        const AggCell c{agg->cells[2 * i], agg->cells[2 * i + 1]};
        H2V_REQUIRE(c.column < hd.n_inst_cols, "aggregation spec: cell " + std::to_string(i) + " names column " + std::to_string(c.column) +
                                                   " of a proof with " + std::to_string(hd.n_inst_cols) + " instance columns");
        agg_cells.push_back(c);
      }
      hd.n_carry = 2;
      hd.agg_limbs = agg->limbs;
      hd.agg_bits = agg->bits;
    }

    // ---------------- assemble the blob
    hd.n_tops = (u32)tops.size();
    hd.n_exprops = (u32)eops.size();
    hd.n_consts = (u32)consts.size();
    blob.assign(sizeof(PlanHeader), 0);
    hd.off_tops = append(blob, tops);
    hd.off_exprops = append(blob, eops);
    hd.off_polys = append(blob, polys);
    hd.off_terms = append(blob, terms);
    hd.off_vars = append(blob, vars);
    hd.off_polylist = append(blob, polylist);
    hd.off_permcols = append(blob, permcols);
    hd.off_lookups = append(blob, lks);
    hd.off_consts = append(blob, consts);
    hd.off_pt_item = append(blob, pt_item);
    hd.off_sc_item = append(blob, sc_item);
    hd.off_rot = append(blob, rot_consts);
    hd.off_sets = append(blob, sets);
    hd.off_setpts = append(blob, setpts);
    hd.off_setcms = append(blob, setcms);
    hd.off_setevals = append(blob, setevals);
    hd.off_diffs = append(blob, diffs);
    hd.off_gwcpts = append(blob, gwcpts);
    hd.off_gwcq = append(blob, gwcq);
    hd.off_instq = append(blob, instq);
    hd.off_shared_pts = append(blob, shared_pts);
    hd.off_lines0 = append(blob, lines0);
    hd.off_lines1 = append(blob, lines1);
    hd.off_agg = append(blob, agg_cells);
    while (blob.size() % 16) blob.push_back(0);
    hd.total_bytes = (u32)blob.size();
    memcpy(blob.data(), &hd, sizeof(hd));

    info.k = k;
    memcpy(info.q_left, &s_g2, sizeof(info.q_left));
    memcpy(info.q_right, &ng2, sizeof(info.q_right));
    info.n_points = hd.n_points;
    info.n_scalars = S;
    info.n_challenges = n_squeeze;
    info.proof_len = hd.proof_len;
    info.n_inst_cols = num_instance_columns * m;
    info.n_shared = hd.n_shared;
    info.n_mo = n_mo;
    return 0;
  } catch (const Err& e) {
    err = e.msg;
    if (in_vk) err += std::string(" (if these bytes came from VerifyingKey::write: ") + query_hint + ")";
    return -1;
  }
}

void build_window_lines(const PlanInfo& info, u32 c0, u32 W0, u32 c1, u32 W1, std::vector<u8>& out) {
  const u32 np = W0 + W1;
  std::vector<G2Affine> q(np);
  for (int ch = 0; ch < 2; ch++) {
    G2Affine cur;
    memcpy(&cur, ch == 0 ? info.q_right : info.q_left, sizeof(cur));
    const u32 W = ch == 0 ? W0 : W1, c = ch == 0 ? c0 : c1, base = ch == 0 ? 0 : W0;
    for (u32 w = 0; w < W; w++) {
      q[base + w] = cur;
      if (w + 1 < W)
        for (u32 i = 0; i < c; i++) cur = g2_double_affine(cur);  // order r is prime: never the identity
    }
  }
  out.resize((size_t)np * H2V_ATE_LINES * sizeof(G2Line));
  g2_prepare_many(q.data(), (int)np, (G2Line*)out.data());
}

}  // namespace h2v
