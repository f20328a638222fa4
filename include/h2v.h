/* C ABI of the B200 batch verifier for Halo2 KZG proofs (BN254; SHPLONK / GWC; Blake2b / Keccak).
 *
 * The reference (ChainSafe/halo2-verifier) has no FFI: its boundary is the Rust API.  Each entry
 * point below names the reference interface it stands behind; a `cuda`-feature Rust shim (see
 * INTEGRATION.md) binds exactly these symbols.
 *
 * Conventions: every buffer is caller-owned host memory (pinned preferred); the library copies what
 * it keeps.  Return value: 0 ok, <0 infrastructure failure (CUDA error, malformed VK/params, bad
 * argument) with text in h2v_last_error(); per-proof verdicts only through `status`.  A context is
 * single-owner (one in-flight batch); distinct contexts / devices may be driven from distinct host
 * threads.  There is no CPU fallback: without a CUDA device h2v_ctx_create fails.
 */
#ifndef H2V_H
#define H2V_H
#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

/* SerdeFormat (reference helpers.rs:7-19) */
#define H2V_FORMAT_PROCESSED 0
#define H2V_FORMAT_RAW_BYTES 1
#define H2V_FORMAT_RAW_BYTES_UNCHECKED 2
/* generic parameter V of verify_proof (reference lib.rs:36): VerifierSHPLONK / VerifierGWC */
#define H2V_MULTIOPEN_SHPLONK 0
#define H2V_MULTIOPEN_GWC 1
/* generic parameter T of verify_proof (lib.rs:38): Blake2bRead / Keccak256Read (+ Challenge255) */
#define H2V_HASH_BLAKE2B 0
#define H2V_HASH_KECCAK256 1

/* per-proof status: plonk::Error classes (reference plonk/mod.rs:19-32) */
#define H2V_OK 0
#define H2V_INVALID_INSTANCES 1          /* lib.rs:51-55 */
#define H2V_TRANSCRIPT 2                 /* Error::Transcript: any read before the multi-open part fails */
#define H2V_OPENING 3                    /* Error::Opening: lib.rs:420-424 (h1/h2 or W_i unreadable) */
#define H2V_CONSTRAINT_SYSTEM_FAILURE 4  /* strategy.rs:164-176: pairing check fails */
#define H2V_WOULD_PANIC 5                /* reference unwraps None: vanishing.rs:100 (x^n = 1), shplonk.rs:215 (z_diff = 0).
                                          * One deviation: the evaluation challenge x = 0 is also reported as H2V_WOULD_PANIC although the
                                          * reference would not panic on it (the Lagrange-basis shortcut used here divides by x; the
                                          * reference's l_i_range, poly/domain.rs:187-212, does not).  x is a transcript hash output, so
                                          * the case has probability 2^-254 and cannot be steered by a prover. */

typedef struct h2v_ctx h2v_ctx;

/* ParamsKZG::read_custom (poly/kzg/commitment.rs:155-207) + VerifyingKey::read (plonk/vk.rs:76-115)
 * + EvaluationDomain::new (poly/domain.rs:34-140) + G2Prepared::from (poly/kzg/msm.rs:186-187):
 * parses both byte strings, compiles the device plan, uploads it to `device`. */
int h2v_ctx_create(h2v_ctx** out, const uint8_t* params, size_t params_len, int params_format,
                   const uint8_t* vk, size_t vk_len, int vk_format, int multiopen, int hash, int device);
/* Same for proofs that carry `circuit_instances` circuit instances in ONE transcript (`instances.len()` of the
 * reference's verify_proof, lib.rs:63,92,117,134; h2v_ctx_create = 1): the per-instance commitments, evaluations,
 * expressions and queries repeat in the reference's interleaving.  The instance scalars of a proof are then laid out
 * instance-major (instance 0: column 0, column 1, ...; instance 1: ...), i.e. as circuit_instances x columns "columns":
 * h2v_ctx_info reports that product as the column count and h2v_batch_set_columns takes that many lengths per proof. */
int h2v_ctx_create_multi(h2v_ctx** out, const uint8_t* params, size_t params_len, int params_format,
                         const uint8_t* vk, size_t vk_len, int vk_format,
                         int multiopen, int hash, int device, uint32_t circuit_instances);
/* Same from the `VALID_VK.bin` bundle the reference's tooling writes (serialize/examples/vector_mul.rs:374-393):
 * ParamsKZG::write (Processed form, 164 bytes) immediately followed by VerifyingKey::write(SerdeFormat::RawBytes). */
int h2v_ctx_create_from_bundle(h2v_ctx** out, const uint8_t* bundle, size_t bundle_len, int multiopen, int hash, int device);
/* ---- aggregation proofs: the KZG accumulator carried in the public instances ----------------------------------------
 * An aggregation circuit (snark-verifier with halo2-lib or halo2wrong) verifies inner proofs in-circuit and defers their
 * pairing: it exposes a KZG accumulator (lhs, rhs) as limbs of its public instances, and the proof is only sound if the
 * verifier also checks e(lhs, g2) e(rhs, -[s]g2) = 1, i.e. lhs = s rhs.  An aggregation context checks it inside the batch
 * fold.  The spec is a property of the circuit (snark-verifier's accumulator_indices + LimbsEncoding<limbs, bits>):
 *   limbs, bits   2 <= limbs <= 8, 1 <= bits <= 128, limbs * bits >= 254; (3, 88) is halo2-lib, (4, 68) halo2wrong
 *   cells         4 * limbs (column, row) pairs, 8 * limbs uint32: lhs.x, lhs.y, rhs.x, rhs.y, least significant limb
 *                 first; `column` indexes the proof's flattened instance columns (instance-major when circuit_instances > 1,
 *                 as h2v_ctx_create_multi lays them out)
 * Exactly one carried accumulator per proof.  A malformed spec (limits above, a column beyond the flattened columns, NULL
 * cells) is refused before any device call, text in h2v_last_error(NULL).
 * Per proof, on the device: every limb must be < 2^bits, each coordinate sum_i limb_i 2^(bits i) < q, each point on
 * y^2 = x^3 + 3 or (0, 0) (the identity, halo2curves from_xy); a cell whose row lies beyond its column's length (ragged
 * layouts, h2v_batch_set_columns) fails too.  A failure is H2V_INVALID_INSTANCES for that proof only, whatever the later
 * stages found (the precedence of lib.rs:51-55), and the proof adds nothing to the fold.
 * Fold: proof j adds rho rhs to its L_j and rho lhs to its R_j (DualMSM orientation e(L, [s]G2) e(R, -G2) = 1), then (L_j, R_j)
 * is folded with c_j as for any proof: two more MSM terms per proof, no extra pairing.  One rho per upload, independent of
 * the r_i: from the upload's key (caller's or OS), Blake2b-512("h2v-rla" | key) mod r, or from the test seed likewise; with
 * caller rlc_scalars from h2v_batch_set_agg_scalar (one-shot, 32 B canonical, non-zero), or drawn from the OS when that was
 * not called (verdicts are unaffected; bit-exact accumulators need the setter).
 * Every entry point covers the carried terms: h2v_verify_proof and every per-proof check (attribution after a rejected
 * fold, the `accum` hook) include them, so a valid outer proof whose carried accumulator is false is
 * H2V_CONSTRAINT_SYSTEM_FAILURE; fold groups, shards + h2v_finalize, the device-side exchange, mixed batches with
 * aggregation members and h2v_acc_absorb fold them like any other term.
 * h2v_ctx_info reports the proof's own counts (points and multi-open points read from the proof).  The scalar hook
 * (h2v_batch_set_scalar_hook) has points + 2 right-channel and multi-open + 2 left-channel entries per proof: the carried
 * lhs, rhs follow the proof points in both channels (right: rho, 0; left: 0, rho; 0 for an identity point). */
int h2v_ctx_create_aggregation(h2v_ctx** out, const uint8_t* params, size_t params_len, int params_format, const uint8_t* vk, size_t vk_len,
                               int vk_format, int multiopen, int hash, int device, uint32_t circuit_instances, uint32_t limbs, uint32_t bits,
                               const uint32_t* cells);
int h2v_batch_set_agg_scalar(h2v_ctx* ctx, const uint8_t* rho32);
void h2v_ctx_destroy(h2v_ctx* ctx);
/* error text of the last failing call on this context (ctx == NULL: of the last failed h2v_ctx_create) */
const char* h2v_last_error(const h2v_ctx* ctx);
/* out[8] = k, points per proof, scalars per proof, challenges per proof, proof length in bytes,
 * instance columns, shared MSM bases (fixed | sigma | G), multi-open points */
int h2v_ctx_info(const h2v_ctx* ctx, uint32_t* out8);

/* VK lint.  The reference's VerifyingKey::write and ::read disagree in three places (SURVEY.md section 4): lookups and
 * shuffles with more than one expression pair are written [inputs..., tables...] but read as interleaved pairs
 * (plonk/lookup.rs:42-47 vs 58-61, plonk/shuffle.rs:76-81 vs 92-95), and `write` emits every instance / fixed query while
 * `read` takes exactly one per column (plonk/vk.rs:243-251 vs 310-322).  This library parses what `read` reads, i.e. it
 * builds the constraint system the reference's verifier would verify against; bytes that came out of `write` for such a
 * circuit describe a different one.  The lint reports every place of the VK of this context where that can have happened
 * (one line per finding, NUL-terminated, truncated to `capacity`); returns the number of findings. */
int h2v_ctx_vk_lint(const h2v_ctx* ctx, char* report, size_t capacity);

/* verify_proof with SingleStrategy (lib.rs:33-46, strategy.rs:164-176) for one proof.
 * instances: n_inst 32-byte little-endian canonical Fr values, columns concatenated (a value >= r: H2V_INVALID_INSTANCES). */
int h2v_verify_proof(h2v_ctx* ctx, const uint8_t* proof, size_t proof_len, const uint8_t* instances,
                     size_t n_inst, uint8_t* status);

/* verify_proofs_batch: AccumulatorStrategy::process per proof + finalize (strategy.rs:125-140), and on
 * a failed batch the per-proof re-check the reference prescribes (poly/strategy.rs:26-30).  The statuses after a
 * rejected fold are those of that separate re-check of every proof: they do not depend on the fold scalars (the
 * re-check draws its own coefficients from the OS), so no choice of rlc_scalars can hide an invalid proof from it.
 * The same holds for every entry point that attributes a rejection (fold groups, shards, mixed batches).
 *   proofs / proof_off    concatenated proof bytes, n+1 byte offsets
 *   instances / inst_off  concatenated 32-byte LE canonical Fr, n+1 offsets in units of scalars;
 *                         per proof: columns concatenated, equal length (see h2v_batch_set_columns).  A value >= r
 *                         fails its proof alone with H2V_INVALID_INSTANCES, ahead of any transcript or opening error.
 *   rlc_scalars           n x 32 B canonical non-zero r_i, or NULL to expand them from `seed`; proof j is folded
 *                         with c_j = prod_{i>j} r_i, the reference's convention (SURVEY.md 3.2).  A zero or
 *                         non-canonical r_i (it would zero c_j of every earlier proof) is refused before any
 *                         device call: -1, "fold scalars must be canonical and non-zero".  The same holds for
 *                         every entry point that takes rlc_scalars.  They define the batch fold and the folded
 *                         (L, R) only: per-proof statuses never depend on them.
 *   status                n bytes out
 *   challenges            optional out, n x C x 32 B canonical, squeeze order            (parity hook)
 *   accum                 optional out, n x 2 x 64 B per-proof affine (L_j, R_j), x|y LE canonical,
 *                         all-zero = identity                                            (parity hook)
 *   batch_accum           optional out, 2 x 64 B folded (L, R) */
int h2v_verify_batch(h2v_ctx* ctx, uint32_t n, const uint8_t* proofs, const uint64_t* proof_off,
                     const uint8_t* instances, const uint64_t* inst_off, const uint8_t* rlc_scalars,
                     uint64_t seed, uint8_t* status, uint8_t* challenges, uint8_t* accum,
                     uint8_t* batch_accum);

/* Fold randomness (reference strategy.rs:129: the accumulator is scaled by Fr::random(OsRng) before every proof; the
 * soundness of the batch check rests on r_i the prover cannot predict).  Precedence for a batch:
 *   rlc_scalars != NULL            the caller's r_i                                   (parity hook: bit-exact accumulators)
 *   h2v_batch_set_rlc_key(key)     r_i = Blake2b-512("h2v-rlk" | key | i) mod r, key = 32 SECRET bytes; one-shot option for
 *                                  the next upload.  Sharded batches: draw one fresh key per global batch and give it to
 *                                  every rank (the c_j are then defined globally, independent of the shard count)
 *   seed != 0                      r_i = Blake2b-512("h2v-rlc" | seed | i) mod r      (test hook: public, reproducible)
 *   otherwise (NULL, no key, 0)    the library draws a fresh 256-bit key from the OS (getrandom) for this upload; a shard
 *                                  drawing its own key is sound too (its proofs get unpredictable coefficients), only the
 *                                  folded (L, R) then depend on the sharding
 * h2v_last_rlc_source: 0 caller scalars, 1 test seed, 2 caller key, 3 OS entropy (of the last upload). */
int h2v_batch_set_rlc_key(h2v_ctx* ctx, const uint8_t* key32);
int h2v_last_rlc_source(const h2v_ctx* ctx);

/* Optional ragged instance layout for the NEXT batch call: inst_ncols[n] = columns supplied per proof
 * (a mismatch with the VK gives H2V_INVALID_INSTANCES, lib.rs:51-55) and inst_col_len[n * columns]
 * = length of each column.  Either may be NULL (equal split).  Cleared after one batch. */
int h2v_batch_set_columns(h2v_ctx* ctx, const uint32_t* inst_ncols, const uint32_t* inst_col_len);

/* Optional extra parity hook for the NEXT batch call: per-proof MSM scalars before RLC folding,
 * n x (points + shared + multi-open) x 32 B canonical: right-channel scalar of every proof point,
 * then of every shared base, then left-channel scalar of every multi-open point. */
int h2v_batch_set_scalar_hook(h2v_ctx* ctx, uint8_t* msm_scalars);

/* ---- sharded batches (one context per GPU; SURVEY.md 8e) -------------------------------------
 * h2v_accumulate_shard processes proofs [global_base, global_base + n) of a global batch of
 * global_count proofs with GLOBALLY defined coefficients c_j (rlc_scalars, if given, has
 * global_count entries) and returns this shard's partial accumulators without running a pairing.
 * A partial is an opaque blob of H2V_PARTIAL_BYTES: a 32-byte header (window geometry) and the
 * shard's per-window Jacobian bucket sums S_w of both MSM channels, L_g = sum_w 2^(c w) S_w^left,
 * R_g likewise; the partials of all shards add up window-wise, and the final check pairs each
 * summed S_w with the prepared multiple [2^(c w)] of its G2 argument, so the explicit (L, R) are
 * only formed when `batch_accum` is requested.  Every shard of one global batch must use the same
 * window geometry: shards of equal size do; otherwise call h2v_batch_set_shard_hint with the
 * largest shard size on every rank.  Proof statuses are final except that H2V_OK means
 * "accumulated".  `partial` (and `partials` of h2v_finalize) may be host or device pointers. */
#define H2V_PARTIAL_BYTES 12320
size_t h2v_partial_bytes(void);
/* Fold groups (one-shot option for the next upload; default 1).  With groups = G the n proofs of the upload are G
 * consecutive INDEPENDENT batches of n / G proofs: each has its own fold coefficients (the reference's
 * AccumulatorStrategy run once per group, strategy.rs:125-136), its own MSM and its own pairing check, and all of
 * them share every kernel launch.  This is how several 4096-proof batches fill the GPU together: the per-proof
 * kernels run over all n proofs, the bucket kernels over G bucket sets, the pairing kernels over G blocks.
 * h2v_verify_batch / h2v_batch_run report the AND of the group verdicts, per-proof statuses are unchanged
 * (attribution runs only inside rejected groups); h2v_last_group_verdicts copies the G verdicts (1 = accepted) and
 * returns G.  n must be a multiple of G; not combinable with the folded-accumulator hook.
 * With shards (h2v_accumulate_shard / h2v_batch_upload_shard) group q is this rank's shard of global batch q:
 * global_base / global_count describe ONE global batch, rlc_scalars holds G x global_count coefficients, the partial
 * output is G consecutive H2V_PARTIAL_BYTES blobs, and h2v_finalize_groups takes the ranks' outputs concatenated
 * ([rank][group]) and runs the G pairing checks in one set of launches (group_verdicts: G bytes, may be NULL). */
int h2v_batch_set_fold_groups(h2v_ctx* ctx, uint32_t groups);
int h2v_last_group_verdicts(const h2v_ctx* ctx, uint8_t* out, uint32_t capacity);
int h2v_finalize_groups(h2v_ctx* ctx, uint32_t n_partials, uint32_t groups, const uint8_t* partials, uint8_t* group_verdicts, int* verdict);
/* window geometry of the NEXT batch call as for a shard of `max_shard_proofs` proofs; cleared after one batch */
int h2v_batch_set_shard_hint(h2v_ctx* ctx, uint32_t max_shard_proofs);
int h2v_accumulate_shard(h2v_ctx* ctx, uint32_t n, const uint8_t* proofs, const uint64_t* proof_off,
                         const uint8_t* instances, const uint64_t* inst_off, const uint8_t* rlc_scalars,
                         uint64_t seed, uint64_t global_base, uint64_t global_count, uint8_t* status,
                         uint8_t* partial);
/* Adds n_partials (<= 128) partial accumulators (gathered over NCCL; n_partials x H2V_PARTIAL_BYTES) and
 * runs the single pairing check DualMSM::check (msm.rs:185-203).  verdict: 1 accept, 0 reject.
 * batch_accum: optional 2 x 64 B folded affine (L, R) (parity hook; costs the serial window combination). */
int h2v_finalize(h2v_ctx* ctx, uint32_t n_partials, const uint8_t* partials, uint8_t* batch_accum,
                 int* verdict);
/* After a rejected h2v_finalize: per-proof pairing checks on the shard last processed by this
 * context; proofs that fail get H2V_CONSTRAINT_SYSTEM_FAILURE in status (n bytes, in/out). */
int h2v_attribute_shard(h2v_ctx* ctx, uint8_t* status);

/* Same for a launch set with fold groups: only the proofs of groups whose verdict (group_verdicts[q] = 0) was a
 * rejection are re-checked; `groups` must equal the fold groups of the shard last processed by this context. */
int h2v_attribute_shard_groups(h2v_ctx* ctx, const uint8_t* group_verdicts, uint32_t groups, uint8_t* status);

/* ---- device-side exchange of sharded batches (one process per GPU of one node; NVLink peer memory) ------------
 * The product path of SURVEY.md 8e / north_star "the 8 partial accumulators are gathered for the single final pairing":
 * every rank's context owns a window in its HBM which the peers map through CUDA IPC.  A launch set then runs WITHOUT
 * the host or a library collective in its data path, as part of the captured CUDA graph: the kernel that packs a
 * shard's per-window sums stores them into the ROOT rank's window over NVLink and publishes a sequence number; the
 * root's summing kernel waits for all ranks, adds the partials in place, runs the pairing check of every fold group and
 * stores the verdicts into every rank's window; every rank's last kernel waits for them (a gather to the root plus a
 * verdict broadcast, not an all-gather).  The contexts that share a window set form a CHANNEL: every rank must run the
 * same sequence of launch sets on it, with the same `root` per launch set (e.g. launch set i on rank i mod world, which
 * spreads the pairing checks).  Several channels (contexts) per rank run independently.  Every device-side wait is bounded
 * (H2V_COMM_TIMEOUT_MS, default 30000): a missing peer yields return code -3, never a hung GPU or an "accepted".
 *   h2v_comm_init     allocates the window for `world` ranks and up to `max_groups` fold groups per launch set; writes an
 *                     opaque handle (H2V_COMM_HANDLE_BYTES) that the caller ships to every rank (plumbing: e.g. one
 *                     torch.distributed all_gather of 128 bytes per context at start-up)
 *   h2v_comm_connect  handles: world x H2V_COMM_HANDLE_BYTES in rank order (own handle included)
 *   h2v_batch_run_shard_exchange   on a shard resident in HBM (h2v_batch_upload_shard): the launch set described above;
 *                     group_verdicts: G bytes out (may be NULL), verdict: AND of them
 *   h2v_verify_shard  the end-to-end call of a rank: upload of its shard (arguments as h2v_accumulate_shard), the launch
 *                     set, per-proof attribution inside the rejected groups of this rank's shard (poly/strategy.rs:26-30),
 *                     status download.  Reference: AccumulatorStrategy::process per proof + finalize (strategy.rs:125-140)
 *                     with the MSM split over the ranks.
 *   h2v_comm_last_batch_accum      root only, one fold group: the folded affine (L, R) of the last launch set, 2 x 64 B
 *                     (parity hook: identical for every shard count when the fold randomness is defined globally) */
#define H2V_COMM_HANDLE_BYTES 128
int h2v_comm_init(h2v_ctx* ctx, uint32_t rank, uint32_t world, uint32_t max_groups, uint8_t* handle_out);
int h2v_comm_connect(h2v_ctx* ctx, const uint8_t* handles);
/* bound of every device-side wait of this context's launch sets from now on (default 30 s, or H2V_COMM_TIMEOUT_MS at h2v_comm_init) */
int h2v_comm_set_timeout_ms(h2v_ctx* ctx, uint32_t ms);
int h2v_batch_run_shard_exchange(h2v_ctx* ctx, uint32_t root, uint8_t* group_verdicts, int* verdict);
int h2v_verify_shard(h2v_ctx* ctx, uint32_t n, const uint8_t* proofs, const uint64_t* proof_off, const uint8_t* instances,
                     const uint64_t* inst_off, const uint8_t* rlc_scalars, uint64_t seed, uint64_t global_base,
                     uint64_t global_count, uint32_t root, uint8_t* status, uint8_t* group_verdicts, int* verdict);
int h2v_comm_last_batch_accum(h2v_ctx* ctx, uint8_t* batch_accum);

/* ---- mixed batches: proofs of several verifying keys in ONE fold ---------------------------------------------------
 * The reference's AccumulatorStrategy carries only the DualMSM of the params (poly/kzg/strategy.rs:125-140): a caller may
 * loop verify_proof(params, vk_i, strategy, instances_i, transcript_i) over proofs of different VKs, and even of
 * VerifierSHPLONK and VerifierGWC, as long as the KZG params agree, and `finalize` then runs ONE DualMSM::check
 * (msm.rs:185-203).  A mix is that use: it is defined over existing contexts, the "members", whose params agree on
 * (g, g2, s_g2) (k, VK, multiopen, hash and circuit_instances may differ).  Each member runs its own per-proof stages on
 * its slice; the fold is ONE bucket MSM over the members' terms (segmented term space, csrc/mix.cuh) and one pairing check,
 * on member 0 ("the lead", whose stream runs the batch and whose prepared G2 lines serve every member).  The whole launch
 * set is one CUDA graph (an LRU keyed by the members' shapes and buffers; the lead's h2v_ctx_set_graphs(0) selects direct
 * launches, h2v_ctx_cache_stats of the lead counts the captures).
 *   h2v_mix_create  members on ONE device, 1 .. 64 distinct contexts.  The mix keeps the pointers: members must outlive it
 *                   and must not run their own batches while a mixed batch is in flight.  Bad member sets (none, more than
 *                   64, repeated, on different devices, params differing in (g, g2, s_g2)) are refused before any device
 *                   call; the text is in h2v_mix_last_error(NULL).
 *   h2v_mix_set_rlc_key   one-shot fold key of the next batch, as h2v_batch_set_rlc_key
 *   h2v_mix_verify  counts[m] proofs of member m (0 allowed: the member takes no part); proofs / proof_off / instances /
 *                   inst_off as h2v_verify_batch over the concatenation, member-major (member 0's proofs first).  Fold order =
 *                   that order: proof j of the concatenation gets c_j = prod_{i>j} r_i over all N = sum counts proofs, i.e. the
 *                   reference's AccumulatorStrategy fed member 0's proofs, then member 1's, ...  rlc_scalars (N x 32 B) / key /
 *                   seed / OS entropy: the precedence of h2v_verify_batch, the r_i defined over the whole concatenation.
 *                   Ragged instances: h2v_batch_set_columns on the member before the call.  status: N bytes out;
 *                   batch_accum: optional 2 x 64 B folded affine (L, R); verdict: 1 = every proof accepted.  On a rejected
 *                   fold every member's proofs are re-checked on their own (poly/strategy.rs:26-30), as in h2v_verify_batch.
 *                   A member with a pending fold-group or shard-hint option is refused: mixes do not combine with them. */
typedef struct h2v_mix h2v_mix;
int h2v_mix_create(h2v_mix** out, h2v_ctx* const* members, uint32_t n_members);
void h2v_mix_destroy(h2v_mix* mx);
const char* h2v_mix_last_error(const h2v_mix* mx);
int h2v_mix_set_rlc_key(h2v_mix* mx, const uint8_t* key32);
int h2v_mix_verify(h2v_mix* mx, const uint32_t* counts, const uint8_t* proofs, const uint64_t* proof_off, const uint8_t* instances,
                   const uint64_t* inst_off, const uint8_t* rlc_scalars, uint64_t seed, uint8_t* status, uint8_t* batch_accum,
                   int* verdict);
/* Multi-params mixes: proofs under several KZG params in ONE fold.  For params classes p with G2 arguments
 * ([s_p]g2_p, -g2_p) the check is prod_p e(L_p, [s_p]g2_p) e(R_p, -g2_p) = 1, L_p / R_p = the fold of class p's proofs with
 * the c_j of the whole member-major concatenation: one Miller product over every class's pairs and one final
 * exponentiation.  Each class with proofs gets its own bucket set of the joint MSM and its own prepared lines (owned by the
 * mix); all classes together take at most 128 (channel, window-run) pairs, so more classes pair longer window runs.
 * h2v_mix_verify keeps its signature and semantics (statuses, attribution under each member's own params, fold
 * randomness) except batch_accum: classes x 128 B, the folded affine (L_p, R_p) of every class in class order; a class
 * with no proofs in the call gets all-zero bytes and adds nothing to the check.  Not combinable with fold groups, as for
 * every mix; shards and the device-side exchange: see "sharded mixed batches" below. */
#define H2V_MIX_MAX_PARAMS 8
/* As h2v_mix_create, but members may hold different KZG params.  Members whose params agree on (g, g2, s_g2) (the comparison
 * h2v_mix_create makes) form one params class; classes are numbered by first appearance in member order (member 0 is in
 * class 0).  1 .. H2V_MIX_MAX_PARAMS classes; more are refused before any device call, with the text in
 * h2v_mix_last_error(NULL).  The other refusals are those of h2v_mix_create. */
int h2v_mix_create_multi_params(h2v_mix** out, h2v_ctx* const* members, uint32_t n_members);
/* class_of[m] = params class of member m (capacity >= n_members); returns the number of classes (1 for a mix of
 * h2v_mix_create), -1 on a null argument or a short array */
int h2v_mix_params_classes(const h2v_mix* mx, uint32_t* class_of, uint32_t capacity);

/* ---- sharded mixed batches: one mixed batch split over the GPUs of a box, one pairing check -------------------------------
 * Every rank holds a mix of its own member contexts (on its own GPU) with the SAME member list on every rank: the same VKs,
 * options and params classes in the same order.  The global batch is what h2v_mix_verify would take: the member-major
 * concatenation of global_counts[m] proofs, N = sum global_counts.  A rank owns the contiguous range [global_base, global_base
 * + n) of it (a range may start or end inside a member, or lie inside one member) and passes only its proofs, member-major,
 * as for h2v_mix_verify; the library derives its per-member counts.  Fold randomness as h2v_mix_verify over the GLOBAL
 * indices: rlc_scalars has N entries, the mix's key (h2v_mix_set_rlc_key) and the test seed expand by global index; with
 * neither, each rank draws its own key from the OS (sound, but the folded (L, R) then depend on the sharding).  With caller
 * scalars or a shared key the folded (L, R) equal, bit for bit, those of one h2v_mix_verify over the concatenation, for
 * every world size and split.
 * Bucket sets: one per params class with proofs in global_counts, in class order.  Every rank emits one partial
 * (H2V_PARTIAL_BYTES, as h2v_accumulate_shard's) per bucket set, also for a class without proofs on that rank (its window
 * sums are the identity), so that partials line up [rank][set].  Window geometry: every rank chooses it from a bound all
 * ranks share (the member shapes, global_counts and the largest shard), never from its own member composition; shards of
 * unequal size need h2v_mix_set_shard_hint(largest shard) on every rank.
 * Statuses (n bytes, this rank's proofs in member-major order) are final at accumulate time except that H2V_OK means
 * "accumulated".  Refused before any device call, text in h2v_mix_last_error(mx), state unchanged: a null argument, N = 0,
 * n = 0, global_base + n > N, a hint smaller than n, non-canonical or zero rlc_scalars, a member with a pending fold-group or
 * shard-hint option; on the exchange also a lead without a connected channel, root >= world or max_groups < sets.  Partials
 * of different window geometries give the "different window geometries" error of h2v_finalize.
 *   h2v_mix_set_shard_hint      one-shot: window geometry of the next shard call as for shards of max_shard_proofs proofs
 *   h2v_mix_partial_bytes       sets x H2V_PARTIAL_BYTES for this global batch (0 on a null argument)
 *   h2v_mix_accumulate_shard    upload + every kernel up to the partials (host or device pointer) + statuses
 *   h2v_mix_finalize            partials: n_partials ranks x sets blobs, [rank][set], host or device pointer; sums them and runs
 *                               ONE multi-pairing check over all sets (one set: the plain 2-pair check).  Works on a mix that
 *                               processed no shard itself (geometry from the partials' headers, sets from global_counts).
 *                               verdict: 1 = the check accepts; batch_accum: optional, classes x 128 B as h2v_mix_verify's
 *   h2v_mix_attribute_shard     after a rejection: every member's proofs of the shard this mix last processed are re-checked
 *                               on their own (poly/strategy.rs:26-30); status (n bytes) out
 *   h2v_mix_verify_shard        the end-to-end call of one rank through the device-side exchange over the LEAD member's
 *                               channel (h2v_comm_init with max_groups >= sets + h2v_comm_connect on member 0): upload, the
 *                               launch set (one CUDA graph: partials -> the root's window, the root's sum and one check,
 *                               verdict -> every rank), attribution on rejection, statuses.  verdict: the global check
 *   h2v_mix_comm_last_batch_accum   root only: classes x 128 B folded (L_p, R_p) of the last exchange launch set */
int h2v_mix_set_shard_hint(h2v_mix* mx, uint32_t max_shard_proofs);
size_t h2v_mix_partial_bytes(const h2v_mix* mx, const uint32_t* global_counts);
int h2v_mix_accumulate_shard(h2v_mix* mx, const uint32_t* global_counts, uint64_t global_base, uint32_t n, const uint8_t* proofs,
                             const uint64_t* proof_off, const uint8_t* instances, const uint64_t* inst_off, const uint8_t* rlc_scalars,
                             uint64_t seed, uint8_t* status, uint8_t* partial);
int h2v_mix_finalize(h2v_mix* mx, const uint32_t* global_counts, uint32_t n_partials, const uint8_t* partials, uint8_t* batch_accum, int* verdict);
int h2v_mix_attribute_shard(h2v_mix* mx, uint8_t* status);
int h2v_mix_verify_shard(h2v_mix* mx, const uint32_t* global_counts, uint64_t global_base, uint32_t n, const uint8_t* proofs, const uint64_t* proof_off,
                         const uint8_t* instances, const uint64_t* inst_off, const uint8_t* rlc_scalars, uint64_t seed, uint32_t root, uint8_t* status,
                         int* verdict);

/* ---- grouped mixed batches: many independent mixed batches in one launch set, one pairing check and verdict each ------------
 * `groups` (1 .. 1024) independent batches of the mix's members, each what h2v_mix_verify would take: counts[q * M + m] =
 * proofs of member m in group q (M = members; 0 allowed), every group with at least one proof, N = sum counts.  proofs /
 * offsets / instances follow the call order: group 0's member-major concatenation, then group 1's, ...  The r_i are indexed
 * by call index i in [0, N); group q covers [o_q, o_q + N_q) and proof j of it is folded with c_j = prod_{i in group q, i > j}
 * r_i: the fold restarts at every group boundary.  rlc_scalars (N x 32 B; group q's slice = what h2v_mix_verify takes for
 * group q alone), the mix's one-shot key, the test seed and OS entropy (one fresh key per call) follow the precedence of
 * h2v_mix_verify and expand by call index; aggregation members: one rho per member upload.
 * Group q passes when prod_p e(L_{q,p}, [s_p]g2_p) e(R_{q,p}, -g2_p) = 1 over the params classes with proofs anywhere in
 * the call (a class without proofs in group q contributes the identity); the 128-pair budget of the check applies per group.
 * Every member uploads once (its proofs of all groups, in group order: h2v_batch_set_columns on a member describes them in
 * that order) and runs its per-proof stages once; the joint bucket MSM has one bucket set per (group, class) and the pairing
 * kernels one check per group, all in one CUDA graph whose key depends on the members' totals and `groups`, not on the split.
 *   status          N bytes, call order
 *   group_verdicts  optional, `groups` bytes: 1 exactly when h2v_mix_verify on group q alone would return verdict 1 (the
 *                   group's check accepted and every proof of it is H2V_OK)
 *   batch_accum     optional, groups x classes x 128 B: per group the class layout of h2v_mix_verify (all-zero bytes for a
 *                   class without proofs in that group)
 *   verdict         the AND of the group verdicts
 * After a rejected check only the proofs of the rejected groups are re-checked on their own (poly/strategy.rs:26-30), with
 * coefficients of their own as in h2v_verify_batch; proofs of accepted groups keep their accumulate-time statuses.
 * Refused before any device call, text in h2v_mix_last_error(mx), state unchanged (the one-shot key stays set): groups = 0 or
 * > 1024, a group without proofs, a null counts / proof_off / inst_off / status / verdict, N = 0 or N >= 2^32, more terms
 * than the 31-bit term ids hold, zero or non-canonical rlc_scalars, a member with a pending fold-group or shard-hint option,
 * a pending h2v_mix_set_shard_hint.  h2v_mix_verify is this call with groups = 1. */
int h2v_mix_verify_groups(h2v_mix* mx, uint32_t groups, const uint32_t* counts, const uint8_t* proofs, const uint64_t* proof_off,
                          const uint8_t* instances, const uint64_t* inst_off, const uint8_t* rlc_scalars, uint64_t seed, uint8_t* status,
                          uint8_t* group_verdicts, uint8_t* batch_accum, int* verdict);
int h2v_mix_comm_last_batch_accum(h2v_mix* mx, uint8_t* batch_accum);

/* ---- persistent accumulators: AccumulatorStrategy as a value that lives across calls ------------------------------------
 * The reference's AccumulatorStrategy (poly/kzg/strategy.rs:125-140) is fed proofs through any number of verify_proof calls,
 * possibly for different VKs, and runs ONE DualMSM::check (msm.rs:185-203) at `finalize`.  An accumulator is that value: its
 * DualMSM (L, R) lives in device memory, batches from any context whose params agree with the anchor's are absorbed into
 * it, and h2v_acc_finalize runs one 2-pair check.
 *   Absorb b of n proofs with fold randomness r_1..r_n (precedence of h2v_verify_batch: rlc_scalars > h2v_acc_set_rlc_key >
 *   seed > OS entropy): proof j gets c_j = prod_{i>j} r_i, and  acc <- s_b acc + (L_b, R_b)  with s_b = prod_i r_i.  Absorbing a
 *   sequence in chunks therefore gives bit for bit the folded (L, R) of ONE h2v_verify_batch over the concatenation with the
 *   concatenated r_i.  Statuses are final at absorb time, except that H2V_OK means "accumulated"; failed proofs add nothing.
 *   Every absorb and every merge appends its own (R_b, L_b) to a record array of max_absorbs entries (index: its slot).
 *   h2v_acc_create    anchor: supplies the params (g, g2, s_g2), the device and the prepared G2 lines; not owned, must outlive
 *                     the accumulator.  Errors of creation: h2v_acc_last_error(NULL).
 *   h2v_acc_absorb    ctx: any context on the anchor's device whose params agree with the anchor's in (g, g2, s_g2).  Arguments
 *                     as h2v_verify_batch.  Refused before any device call, state unchanged: such a mismatch, n = 0, a full
 *                     record array, a pending fold-group or shard-hint option on ctx.  The launch set is the context's batch up
 *                     to the window sums, then one kernel that folds them into the accumulator (one CUDA graph, the context's
 *                     LRU; h2v_ctx_set_graphs(0): direct launches).  Absorbs from different contexts are ordered through an
 *                     event the accumulator owns.
 *   h2v_acc_finalize  verdict: 1 = the 2-pair check on (L, R) accepts (an empty accumulator accepts).  On a rejection one check
 *                     per record: absorb_verdicts[i] (capacity bytes) = 0 for the absorbs / merges that fail on their own, and
 *                     the caller re-verifies those batches with h2v_verify_batch for per-proof statuses (poly/strategy.rs:26-30).
 *                     Resets the accumulator afterwards (finalize(self) consumes the strategy).
 *   h2v_acc_get       the affine L | R, 2 x 64 B in the batch_accum layout (all-zero = identity)
 *   h2v_acc_merge     acc <- r acc + P with P = L | R in the same layout: the DualMSM scale followed by adding another
 *                     accumulator (of another GPU or process; into an empty accumulator: restore from a checkpoint).  r32: 32 B
 *                     canonical and non-zero (r = 0 would drop every earlier absorb out of the check), or NULL to draw r from
 *                     the OS.  A zero or non-canonical r, non-canonical or off-curve bytes are refused, state unchanged.
 *                     A merge is one record.
 *   h2v_acc_reset     empty accumulator and record array
 * Not combinable with mixed batches, fold groups, shards or the device-side exchange. */
typedef struct h2v_acc h2v_acc;
int h2v_acc_create(h2v_acc** out, h2v_ctx* anchor, uint32_t max_absorbs);
void h2v_acc_destroy(h2v_acc* acc);
const char* h2v_acc_last_error(const h2v_acc* acc);
int h2v_acc_set_rlc_key(h2v_acc* acc, const uint8_t* key32);
int h2v_acc_absorb(h2v_acc* acc, h2v_ctx* ctx, uint32_t n, const uint8_t* proofs, const uint64_t* proof_off, const uint8_t* instances,
                   const uint64_t* inst_off, const uint8_t* rlc_scalars, uint64_t seed, uint8_t* status, uint32_t* index);
int h2v_acc_finalize(h2v_acc* acc, int* verdict, uint8_t* absorb_verdicts, uint32_t capacity);
int h2v_acc_get(const h2v_acc* acc, uint8_t* out128);
int h2v_acc_merge(h2v_acc* acc, const uint8_t* in128, const uint8_t* r32);
int h2v_acc_reset(h2v_acc* acc);

/* ---- staged execution for measurement (bench.py): upload, run (device-resident), download ---- */
int h2v_batch_upload(h2v_ctx* ctx, uint32_t n, const uint8_t* proofs, const uint64_t* proof_off,
                     const uint8_t* instances, const uint64_t* inst_off, const uint8_t* rlc_scalars,
                     uint64_t seed);
/* same, for one shard of a global batch (see h2v_accumulate_shard) */
int h2v_batch_upload_shard(h2v_ctx* ctx, uint32_t n, const uint8_t* proofs, const uint64_t* proof_off,
                           const uint8_t* instances, const uint64_t* inst_off, const uint8_t* rlc_scalars,
                           uint64_t seed, uint64_t global_base, uint64_t global_count);
/* runs every kernel of the shard except the pairing; partial: H2V_PARTIAL_BYTES out, host OR device pointer */
int h2v_batch_run_shard(h2v_ctx* ctx, uint8_t* partial);
/* same, enqueue only: returns without waiting; `partial_device` must be device memory and is valid for work
 * ordered after this call on the context's stream (h2v_ctx_stream), e.g. an NCCL all-gather issued on it */
int h2v_batch_run_shard_async(h2v_ctx* ctx, uint8_t* partial_device);
/* overwrites `bytes` of scratch HBM on the context's stream (L2 flush between timed iterations) */
int h2v_flush_l2(h2v_ctx* ctx, size_t bytes);
/* runs every kernel of the batch on data already resident in HBM; verdict of the batch pairing out */
int h2v_batch_run(h2v_ctx* ctx, int* verdict);
int h2v_batch_download(h2v_ctx* ctx, uint8_t* status);
/* CUDA-event timings (ms) of the last run, on the context's stream:
 * out[0] total, [1] decompress, [2] transcript, [3] scalar stage, [4] rlc + msm, [5] pairing, [6] attribution */
int h2v_last_timings(const h2v_ctx* ctx, float* out8);
/* number of kernel launches issued by this context so far */
uint64_t h2v_launch_count(const h2v_ctx* ctx);
/* the context's cudaStream_t (every kernel and copy of the context is issued on it), so that a caller
 * can record its own CUDA events around calls or order other work after them */
void* h2v_ctx_stream(const h2v_ctx* ctx);
/* host waits of this context: 0 (default) spin on the stream (lowest latency), 1 block on an event (use when many
 * contexts share few host cores, e.g. several batches in flight on every GPU of a box) */
int h2v_ctx_set_blocking_sync(h2v_ctx* ctx, int blocking);
/* CUDA graphs (bit 0, default 1): the kernels of a batch are captured once per (entry point, batch shape, buffers) and
 * replayed with ONE launch per batch, which removes ~40 driver calls per batch from the host threads (with many
 * batches in flight those calls, serialised by the driver, bounded the throughput).  The context keeps the last 16
 * graphs and the prepared window lines of the last 4 MSM geometries, so a service that alternates batch shapes replays.
 * Bit 0 = 0: direct launches with a CUDA event after every stage: required for the per-stage values of
 * h2v_last_timings (a replay only yields the total).  Bit 1 (default 0): programmatic dependent launch between the
 * kernels of a batch (measured: no gain, kept for diagnosis). */
int h2v_ctx_set_graphs(h2v_ctx* ctx, int on);
/* out[0] = host rebuilds of prepared window lines, out[1] = graph captures, since the context was created */
int h2v_ctx_cache_stats(const h2v_ctx* ctx, uint64_t* out2);
/* diagnostics: per-block timeline of the per-proof and MSM kernels on `device` (all contexts).  start allocates a
 * log of `capacity` records and switches recording on; stop switches it off and copies up to `capacity` 32-byte
 * records {u32 kernel id, block, SM, context tag; u64 start_ns, end_ns} (global nanosecond timer) into `out`. */
int h2v_debug_timeline_start(int device, uint32_t capacity);
int h2v_debug_timeline_stop(int device, void* out, uint32_t capacity, uint32_t* count);
/* Algorithmic work model of this plan (bench.py roofline), per proof with `instance_rows` values per instance column:
 * out[0] Montgomery multiplications of the scalar stage (a walk over the plan that counts what scalar_stage multiplies),
 * out[1] of the transcript stage (Montgomery conversions), out[2] of one point decompression, out[3] instance scalars. */
int h2v_ctx_work_model(const h2v_ctx* ctx, uint32_t instance_rows, double* out4);
/* MSM geometry of the last run: out[0] window bits, [1] windows, [2] terms, [3] buckets */
int h2v_last_msm_geometry(const h2v_ctx* ctx, uint32_t* out4);
/* GLV split of the last run's MSM: 1 when every scalar was split as k = a - b lambda into lifted half-length digit rows
 * (window geometry of h2v_last_msm_geometry then covers ~131 bits), 0 for plain windows */
int h2v_last_msm_glv(const h2v_ctx* ctx);

/* ---- device self tests (used by tests/ only) ---------------------------------------------------
 * Runs the PTX field multiplication against the portable one on `count` pseudo-random and edge
 * operands for both fields; returns the number of mismatches (0 = pass), <0 on CUDA error. */
int h2v_selftest_field(int device, uint32_t count, uint64_t seed);
/* Known-answer vectors: one field operation on n operand pairs, raw 32-byte little-endian limbs in and out (no conversion:
 * the caller places operands anywhere in the operation's documented range and compares with exact integers).
 * field: 0 = Fq, 1 = Fr.  op: 0 mul (a < 2^255, b < p), 1 mul_c, 2 sqr, 3 sqr_c, 4 mul_any (a < 2^256), 5 a + b, 6 a - b,
 * 7 neg, 8 from_canonical, 9 to_canonical, 10 inv (Fermat), 11 inv_bin, 12 from_uniform of the 64 bytes a | b.
 * Returns 0, -1 on a bad argument, -2 on a CUDA error. */
int h2v_selftest_field_vectors(int device, int field, int op, uint32_t n, const uint8_t* a, const uint8_t* b, uint8_t* out);
/* integer multiply-add peak calibration: returns achieved 32-bit IMAD operations per second */
double h2v_calibrate_imad(int device);

#ifdef __cplusplus
}
#endif
#endif
