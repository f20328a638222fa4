"""GPU parity tests (run on the B200 box: pytest -m gpu).  Every call goes through the C ABI
(include/h2v.h) of libh2v_b200.so; the checker is the CPU oracle (oracle/), on the same seeded inputs,
plus the committed golden vectors, plus size-independent properties at the full batch size."""
import ctypes
import json
import os
import random

import pytest

import bn254 as bn
import formats as F
import prover_sim as sim
import verifier as orc
from workloads import enc_point, make_batch, oracle_scalars, setup, split32

pytestmark = pytest.mark.gpu
HERE = os.path.dirname(os.path.abspath(__file__))


def make_bv(pkg, params, vk, mo, hk, vkfmt=F.RAW_BYTES):
    return pkg.BatchVerifier(pkg.ParamsKZG.from_bytes(params.to_bytes()), pkg.VerifyingKey.from_bytes(vk.to_bytes(vkfmt), vkfmt),
                             mo, "keccak256" if hk == "keccak" else hk, device=0)


def test_field_ptx_matches_portable(pkg):
    lib = pkg.load_library()
    assert lib.h2v_selftest_field(0, 1 << 20, 20261018) == 0
    assert lib.h2v_calibrate_imad(0) > 1e12


def check_against_oracle(bv, params, vk, instances, proofs, mo, hk, rs):
    """instances: the oracle's [circuit instance][column][row] per proof"""
    api = [i[0] for i in instances] if bv.circuit_instances == 1 else instances
    res = bv.verify_batch(proofs, api, rlc_scalars=rs, want_challenges=True, want_accum=True,
                          want_batch_accum=True, want_scalars=True)
    want = [orc.verify_proof(params, vk, inst, p, mo, hk) for inst, p in zip(instances, proofs)]
    assert res.status == [w.status for w in want]
    C, nb = bv.n_challenges, bv.n_bases
    for j, w in enumerate(want):
        if w.status in (orc.OK, orc.CONSTRAINT_SYSTEM_FAILURE):
            assert split32(res.challenges[32 * C * j:], C) == w.challenges, f"challenges of proof {j}"
            assert split32(res.msm_scalars[32 * nb * j:], nb) == oracle_scalars(vk, w, bv.n_points, bv.n_mo), f"scalars of proof {j}"
            assert res.accum[128 * j: 128 * j + 128] == enc_point(w.L) + enc_point(w.R), f"accumulators of proof {j}"
    L, R_, ok = orc.accumulate(params, want, rs)
    assert res.batch_accum == enc_point(L) + enc_point(R_)
    assert ok == all(w.status != orc.CONSTRAINT_SYSTEM_FAILURE for w in want)
    return res, want


@pytest.mark.parametrize("shape,k", [("vm", 8), ("vm", 10), ("sh", 8), ("mix", 6)])
@pytest.mark.parametrize("mo", ["shplonk", "gwc"])
@pytest.mark.parametrize("hk", ["blake2b", "keccak"])
def test_batch_parity_small(pkg, shape, k, mo, hk):
    params, vk, instances, proofs, rng = make_batch(shape, k, 6, mo, hk)
    rs = [rng.randrange(1, bn.R) for _ in proofs]
    with make_bv(pkg, params, vk, mo, hk, F.RAW_BYTES if mo == "shplonk" else F.PROCESSED) as bv:
        assert bv.proof_len == len(proofs[0])
        check_against_oracle(bv, params, vk, instances, proofs, mo, hk, rs)
        # every rejection class, attributed inside a batch (SURVEY.md section 7)
        bad = list(proofs)
        kinds = list(sim.CORRUPTIONS)[: len(bad) - 1]
        for i, kind in enumerate(kinds):
            bad[i], _ = sim.corrupt(proofs[i], vk, kind, rng, mo)
        check_against_oracle(bv, params, vk, instances, bad, mo, hk, rs)


def test_all_corruption_classes_and_instances(pkg):
    params, vk, instances, proofs, rng = make_batch("vm", 8, len(sim.CORRUPTIONS) + 3, "shplonk", "blake2b", seed=5)
    rs = [rng.randrange(1, bn.R) for _ in proofs]
    bad, insts = list(proofs), [[list(map(list, i[0]))] for i in instances]
    for i, kind in enumerate(sim.CORRUPTIONS):
        bad[i], _ = sim.corrupt(proofs[i], vk, kind, rng)
    j = len(sim.CORRUPTIONS)
    insts[j][0][0][0] = (insts[j][0][0][0] + 1) % bn.R  # the reference's negative test (vector_mul.rs:327-330)
    insts[j + 1] = [[]]  # wrong number of instance columns -> InvalidInstances
    with make_bv(pkg, params, vk, "shplonk", "blake2b") as bv:
        res, want = check_against_oracle(bv, params, vk, insts, bad, "shplonk", "blake2b", rs)
        assert res.status[j] == 4 and res.status[j + 1] == 1 and res.status[j + 2] == 0
        assert sorted(set(res.status)) == [0, 1, 2, 3, 4]
        # ragged public inputs: different lengths per proof
        insts2 = [sim.random_instances(vk, rng, 3 + 5 * t) for t in range(4)]
        _p, _v, dl, s = setup("vm", 8)
        proofs2 = [sim.simulate_proof(params, vk, dl, s, inst, rng) for inst in insts2]
        check_against_oracle(bv, params, vk, insts2, proofs2, "shplonk", "blake2b", rs[:4])
        # single-proof entry point (SingleStrategy)
        st = ctypes.c_uint8(9)
        ib = b"".join(bn.fr_to_repr(v) for col in insts2[0][0] for v in col)
        assert bv.lib.h2v_verify_proof(bv._ctx, proofs2[0], len(proofs2[0]), ib, len(ib) // 32, ctypes.byref(st)) == 0 and st.value == 0
        assert bv.lib.h2v_verify_proof(bv._ctx, proofs2[1], len(proofs2[1]), ib, len(ib) // 32, ctypes.byref(st)) == 0 and st.value == 4


def test_python_api_mirrors_reference(pkg):
    params, vk, instances, proofs, rng = make_batch("vm", 8, 3, "gwc", "blake2b", seed=9)
    P, V = pkg.ParamsKZG.from_bytes(params.to_bytes()), pkg.VerifyingKey.from_bytes(vk.to_bytes(F.PROCESSED), pkg.SerdeFormat.Processed)
    assert pkg.verify_proof(P, V, proofs[0], instances[0][0], multiopen="gwc") is None
    bad, _ = sim.corrupt(proofs[1], vk, "eval_flip", rng, "gwc")
    with pytest.raises(pkg.ConstraintSystemFailure):
        pkg.verify_proof(P, V, bad, instances[1][0], multiopen="gwc")
    errs = pkg.verify_proofs_batch(P, V, [proofs[0], bad, proofs[2][:100]], [i[0] for i in instances], multiopen="gwc")
    assert errs[0] is None and isinstance(errs[1], pkg.ConstraintSystemFailure) and isinstance(errs[2], pkg.TranscriptError)


def test_golden_vectors(pkg):
    for fn in sorted(os.listdir(os.path.join(HERE, "golden"))):
        if not fn.endswith(".json") or fn == "srs_kat.json":
            continue
        g = json.load(open(os.path.join(HERE, "golden", fn)))
        bv = pkg.BatchVerifier(pkg.ParamsKZG.from_bytes(bytes.fromhex(g["params"])),
                               pkg.VerifyingKey.from_bytes(bytes.fromhex(g["vk"]), pkg.SerdeFormat(g["vk_format"])),
                               g["multiopen"], "keccak256" if g["hash"] == "keccak" else g["hash"], device=0,
                               circuit_instances=g.get("circuit_instances", 1))
        proofs = [bytes.fromhex(e["proof"]) for e in g["proofs"]]
        if "circuit_instances" in g:  # [circuit instance][column][row]
            insts = [[[[int(v, 16) for v in col] for col in ci] for ci in e["instances"]] for e in g["proofs"]]
        else:
            insts = [[[int(v, 16) for v in col] for col in e["instances"]] for e in g["proofs"]]
        res = bv.verify_batch(proofs, insts, rlc_scalars=[int(r, 16) for r in g["rlc_scalars"]], want_challenges=True,
                              want_accum=True, want_batch_accum=True, want_scalars=True)
        C, nb = bv.n_challenges, bv.n_bases
        assert res.status == [e["status"] for e in g["proofs"]], fn
        assert res.batch_accum.hex() == g["folded"], fn
        for j, e in enumerate(g["proofs"]):
            if "accum" in e:
                assert [hex(c) for c in split32(res.challenges[32 * C * j:], C)] == e["challenges"], fn
                assert res.accum[128 * j: 128 * j + 128].hex() == e["accum"], fn
                assert [hex(c) for c in split32(res.msm_scalars[32 * nb * j:], nb)] == e["msm_scalars"], fn
        bv.close()


def test_k18_lookup_heavy(pkg):
    params, vk, instances, proofs, rng = make_batch("k18", 18, 3, "shplonk", "blake2b")
    proofs[1], _ = sim.corrupt(proofs[1], vk, "eval_flip", rng)
    with make_bv(pkg, params, vk, "shplonk", "blake2b") as bv:
        assert bv.proof_len == 12960  # SURVEY.md section 8 (K18)
        check_against_oracle(bv, params, vk, instances, proofs, "shplonk", "blake2b", [rng.randrange(1, bn.R) for _ in proofs])


def _big_batch(n, mo):
    """Full-size batch: 64 distinct oracle-simulated proofs tiled to n (bounded CPU generation time)."""
    params, vk, instances, proofs, rng = make_batch("vm", 10, 64, mo, "blake2b", seed=77)
    reps = n // 64
    return params, vk, instances * reps, proofs * reps, rng


@pytest.mark.parametrize("mo", ["shplonk", "gwc"])
def test_full_batch_4096_properties(pkg, mo):
    """BASELINE.json configs[1] / [2] size.  Size-independent properties:
    (1) an all-valid batch is accepted and the fold is linear: fold(A || B) = c * fold(A) + fold(B);
    (2) the fold over tiled copies equals the oracle fold computed from 64 per-proof accumulators;
    (3) 1% corrupted proofs -> batch rejected -> attribution flags exactly the injected indices."""
    n = 4096
    params, vk, instances, proofs, rng = _big_batch(n, mo)
    insts = [i[0] for i in instances]
    rs = [rng.randrange(1, bn.R) for _ in range(n)]
    with make_bv(pkg, params, vk, mo, "blake2b") as bv:
        res = bv.verify_batch(proofs, insts, rlc_scalars=rs, want_batch_accum=True)
        assert res.verdict and res.status == [0] * n
        # (2) oracle fold from the 64 distinct accumulators
        want = [orc.verify_proof(params, vk, instances[j], proofs[j], mo, "blake2b", check_pairing=False) for j in range(64)]
        cs = orc.rlc_coefficients(rs)
        coef = [sum(cs[j + 64 * t] for t in range(n // 64)) % bn.R for j in range(64)]
        L = R_ = None
        for w, c in zip(want, coef):
            L, R_ = bn.g1_add(L, bn.g1_mul(w.L, c)), bn.g1_add(R_, bn.g1_mul(w.R, c))
        assert res.batch_accum == enc_point(L) + enc_point(R_)
        # (1) linearity across a split
        h = n // 2
        a = bv.verify_batch(proofs[:h], insts[:h], rlc_scalars=rs[:h], want_batch_accum=True).batch_accum
        b = bv.verify_batch(proofs[h:], insts[h:], rlc_scalars=rs[h:], want_batch_accum=True).batch_accum
        dec = lambda e: None if e == bytes(64) else (int.from_bytes(e[:32], "little"), int.from_bytes(e[32:], "little"))
        c_split = cs[h - 1]  # = prod_{i >= h} r_i: what the first half's last coefficient (1) becomes in the whole batch
        for off in (0, 64):
            whole = dec(res.batch_accum[off: off + 64])
            assert whole == bn.g1_add(bn.g1_mul(dec(a[off: off + 64]), c_split), dec(b[off: off + 64]))
        # (3) attribution
        bad_idx = sorted(rng.sample(range(n), n // 100))
        bad = list(proofs)
        expect = [0] * n
        kinds = ["eval_flip", "point_swap", "scalar_ge_r", "point_offcurve", "opening_offcurve", "truncate_body"]
        for t, i in enumerate(bad_idx):
            bad[i], expect[i] = sim.corrupt(proofs[i], vk, kinds[t % len(kinds)], rng, mo)
        res = bv.verify_batch(bad, insts, rlc_scalars=rs)
        assert not res.verdict and res.status == expect


def test_sharded_accumulation_matches_whole_batch(pkg):
    """SURVEY.md 8e on one GPU: two contexts play two ranks; the folded (L, R) must be identical for
    every shard count, and a corrupted shard is attributed locally."""
    n = 256
    params, vk, instances, proofs, rng = make_batch("vm", 10, 32, "shplonk", "blake2b", seed=3)
    instances, proofs = instances * 8, proofs * 8
    insts = [i[0] for i in instances]
    rs = [rng.randrange(1, bn.R) for _ in range(n)]
    with make_bv(pkg, params, vk, "shplonk", "blake2b") as b0, make_bv(pkg, params, vk, "shplonk", "blake2b") as b1:
        whole = b0.verify_batch(proofs, insts, rlc_scalars=rs, want_batch_accum=True)
        for shards in (2, 4):
            per = n // shards
            parts = []
            for g in range(shards):
                bv = (b0, b1)[g % 2]
                st, partial = bv.accumulate_shard(proofs[g * per:(g + 1) * per], insts[g * per:(g + 1) * per], g * per, n, rlc_scalars=rs)
                assert st == [0] * per
                parts.append(partial)
            ok, folded = b0.finalize(parts)
            assert ok and folded == whole.batch_accum
        # seed-derived coefficients agree between whole and sharded runs too
        w2 = b0.verify_batch(proofs, insts, seed=99, want_batch_accum=True)
        parts = [bv.accumulate_shard(proofs[g * 128:(g + 1) * 128], insts[g * 128:(g + 1) * 128], g * 128, n, seed=99)[1] for g, bv in ((0, b0), (1, b1))]
        assert b1.finalize(parts) == (True, w2.batch_accum)
        # uneven shards (86 / 85 / 85): the shard hint gives every rank the same window geometry
        cuts = [0, 86, 171, 256]
        parts = [(b0, b1)[g % 2].accumulate_shard(proofs[cuts[g]:cuts[g + 1]], insts[cuts[g]:cuts[g + 1]], cuts[g], n, rlc_scalars=rs, shard_hint=86)[1]
                 for g in range(3)]
        assert b0.finalize(parts) == (True, whole.batch_accum)
        # corrupted proof in shard 1
        bad = list(proofs)
        bad[200], _ = sim.corrupt(proofs[200], vk, "eval_flip", rng)
        st0, p0 = b0.accumulate_shard(bad[:128], insts[:128], 0, n, rlc_scalars=rs)
        st1, p1 = b1.accumulate_shard(bad[128:], insts[128:], 128, n, rlc_scalars=rs)
        ok, _ = b0.finalize([p0, p1])
        assert not ok
        assert b0.attribute_shard(st0) == [0] * 128
        st1 = b1.attribute_shard(st1)
        assert st1[72] == 4 and sum(st1) == 4


# ---- BASELINE.json full sizes, every proof checked against the C oracle (oracle/c)
def _pack(proofs, insts):
    import numpy as np

    pb = np.frombuffer(b"".join(proofs), dtype=np.uint8)
    poff = np.cumsum([0] + [len(p) for p in proofs]).astype(np.uint64)
    ib = np.frombuffer(b"".join(v if isinstance(v, (bytes, bytearray)) else int(v).to_bytes(32, "little") for inst in insts for col in inst for v in col),
                       dtype=np.uint8)
    ioff = np.cumsum([0] + [sum(len(c) for c in inst) for inst in insts]).astype(np.uint64)
    return pb, poff, ib, ioff


def test_config2_4096_shplonk_every_proof_against_c_oracle(pkg):
    """BASELINE.json configs[1] (+ the corruption mix of configs[2]): 4096 SHPLONK proofs, k = 10; statuses, challenges,
    per-proof accumulators and the folded (L, R) of ALL proofs bit-exact against the C restatement."""
    import c_oracle
    from importlib import import_module

    synth = import_module("halo2_verifier_b200.synth")
    n, k = 4096, 10
    rng = random.Random(4096)
    s = rng.randrange(1, bn.R)
    vk_bytes, shared_dlogs = synth.make_vk_bytes("vm", k)
    pbytes = synth.params_bytes_raw(k, s)
    vk = F.VerifyingKey.from_bytes(vk_bytes, F.RAW_BYTES)
    co = c_oracle.COracle(pbytes, 1, vk_bytes, 1)
    with pkg.BatchVerifier(pkg.ParamsKZG.from_bytes(pbytes, pkg.SerdeFormat.RawBytes), pkg.VerifyingKey.from_bytes(vk_bytes)) as bv:
        proofs, insts = synth.synthesize_shplonk_batch(bv, shared_dlogs, s, n, seed=("t", 1))
        C = bv.n_challenges
        rs = [rng.randrange(1, bn.R) for _ in range(n)]
        for rnd in range(2):
            if rnd == 1:  # 1 % corrupted, every rejection class
                kinds = list(sim.CORRUPTIONS)
                for t, i in enumerate(sorted(rng.sample(range(n), n // 100))):
                    proofs[i], _ = sim.corrupt(proofs[i], vk, kinds[t % len(kinds)], rng)
            res = bv.verify_batch(proofs, insts, rlc_scalars=rs, want_challenges=True, want_accum=True, want_batch_accum=True)
            st, _secs, lr, ch = co.verify_many(*_pack(proofs, insts), n, threads=os.cpu_count() or 1, want_lr=True, chal_cap=C)
            assert res.status == [int(x) for x in st]
            live = [x in (0, 4) for x in res.status]
            for j in range(n):
                if live[j]:
                    assert res.challenges[32 * C * j: 32 * C * (j + 1)] == ch[32 * C * j: 32 * C * (j + 1)], f"challenges of proof {j}"
                    assert res.accum[128 * j: 128 * (j + 1)] == lr[128 * j: 128 * (j + 1)], f"accumulators of proof {j}"
            folded, ok = co.fold(lr, rs, live)
            assert res.batch_accum == folded
            assert ok == res.verdict or (not ok and not res.verdict)
            assert (rnd == 0) == res.verdict
            if rnd == 1:
                assert sorted(set(res.status)) == [0, 2, 3, 4]
    co.close()


def test_config3_gwc_batch_with_attribution_against_c_oracle(pkg):
    """BASELINE.json configs[2]: GWC multi-open, corrupted proofs attributed inside the batch (1024 proofs: oracle-simulated
    proofs are slow to manufacture; 64 distinct proofs tiled, then 1 % corrupted)."""
    import c_oracle

    n = 1024
    params, vk, instances, proofs, rng = make_batch("vm", 10, 64, "gwc", "blake2b", seed=31)
    proofs, insts = (proofs * (n // 64)), [i[0] for i in instances] * (n // 64)
    kinds = list(sim.CORRUPTIONS)
    for t, i in enumerate(sorted(rng.sample(range(n), n // 100))):
        proofs[i], _ = sim.corrupt(proofs[i], vk, kinds[t % len(kinds)], rng, "gwc")
    rs = [rng.randrange(1, bn.R) for _ in range(n)]
    co = c_oracle.COracle(params.to_bytes(1), 1, vk.to_bytes(1), 1)
    with make_bv(pkg, params, vk, "gwc", "blake2b") as bv:
        C = bv.n_challenges
        res = bv.verify_batch(proofs, insts, rlc_scalars=rs, want_challenges=True, want_accum=True, want_batch_accum=True)
        st, _secs, lr, ch = co.verify_many(*_pack(proofs, insts), n, "gwc", "blake2b", threads=os.cpu_count() or 1, want_lr=True, chal_cap=C)
        assert res.status == [int(x) for x in st] and not res.verdict and res.status.count(0) >= n - n // 100
        live = [x in (0, 4) for x in res.status]
        for j in range(n):
            if live[j]:
                assert res.challenges[32 * C * j: 32 * C * (j + 1)] == ch[32 * C * j: 32 * C * (j + 1)]
                assert res.accum[128 * j: 128 * (j + 1)] == lr[128 * j: 128 * (j + 1)]
        assert res.batch_accum == co.fold(lr, rs, live)[0]
    co.close()


def test_config4_k18_lookup_heavy_batch_against_c_oracle(pkg):
    """BASELINE.json configs[3] shape: k = 18, 64 advice columns, degree-5 gates, 8 lookups, 66-column permutation
    (batch of 64: 4 distinct oracle-simulated proofs tiled; the full 1024 only repeats them)."""
    import c_oracle

    n = 64
    params, vk, instances, proofs, rng = make_batch("k18", 18, 4, "shplonk", "blake2b", seed=41)
    proofs, insts = proofs * (n // 4), [i[0] for i in instances] * (n // 4)
    proofs[7], _ = sim.corrupt(proofs[7], vk, "eval_flip", rng)
    rs = [rng.randrange(1, bn.R) for _ in range(n)]
    co = c_oracle.COracle(params.to_bytes(1), 1, vk.to_bytes(1), 1)
    with make_bv(pkg, params, vk, "shplonk", "blake2b") as bv:
        C = bv.n_challenges
        res = bv.verify_batch(proofs, insts, rlc_scalars=rs, want_challenges=True, want_accum=True, want_batch_accum=True)
        st, _secs, lr, ch = co.verify_many(*_pack(proofs, insts), n, threads=os.cpu_count() or 1, want_lr=True, chal_cap=C)
        assert res.status == [int(x) for x in st] == [4 if j == 7 else 0 for j in range(n)]
        assert res.challenges == ch and res.accum == lr
        assert res.batch_accum == co.fold(lr, rs, [True] * n)[0]
    co.close()


def test_vk_bundle_and_honest_proof_through_the_c_abi(pkg):
    """The reference tooling's artefacts (serialize/examples/vector_mul.rs:363-393): VALID_VK.bin = params (Processed) | VK
    (RawBytes), VALID_PROOF.bin, VALID_PUBS.bin -- here produced by the honest mini-prover -- verified like `verify_proof`."""
    import honest_prover as hp

    rng = random.Random(77)
    s = sim.FIXTURE_SRS_SECRET
    params, vk, pk = hp.keygen_vm(8, s, 10)
    lhs, rhs = [rng.randrange(bn.R) for _ in range(10)], [rng.randrange(bn.R) for _ in range(10)]
    proof, inst = hp.prove_vm(params, vk, pk, s, lhs, rhs, rng)
    bundle = params.to_bytes(F.PROCESSED) + vk.to_bytes(F.RAW_BYTES)
    pubs = b"".join(bn.fr_to_repr(v) for v in inst[0][0])
    P, V = pkg.read_vk_bundle(bundle)
    assert pkg.verify_proof(P, V, proof, pkg.instances_from_pubs(pubs)) is None
    wrong = pkg.instances_from_pubs(pubs)
    wrong[0][2] = (wrong[0][2] + 1) % bn.R
    with pytest.raises(pkg.ConstraintSystemFailure):  # tests/vector_mul.rs:327-330
        pkg.verify_proof(P, V, proof, wrong)
    lib = pkg.load_library()
    ctx = ctypes.c_void_p()
    assert lib.h2v_ctx_create_from_bundle(ctypes.byref(ctx), bundle, len(bundle), 0, 0, 0) == 0
    st = ctypes.c_uint8(9)
    assert lib.h2v_verify_proof(ctx, proof, len(proof), pubs, len(pubs) // 32, ctypes.byref(st)) == 0 and st.value == 0
    lib.h2v_ctx_destroy(ctx)
    assert lib.h2v_ctx_create_from_bundle(ctypes.byref(ctx), bundle[:100], 100, 0, 0, 0) != 0


def test_edge_cases_empty_inputs_single_proof_all_invalid(pkg):
    """Edge cases of the batch API: no public inputs at all, a batch of one, a batch in which every proof is unreadable
    (nothing to fold: the pairing check of two identities accepts, the statuses carry the errors), empty proof bytes."""
    import honest_prover as hp

    rng = random.Random(5150)
    s = rng.randrange(1, bn.R)
    params, vk, pk = hp.keygen_vm(6, s, 0)  # zero multiplications: empty instance column
    proof, inst = hp.prove_vm(params, vk, pk, s, [], [], rng)
    assert inst == [[[]]] and orc.verify_proof(params, vk, inst, proof).status == 0
    with make_bv(pkg, params, vk, "shplonk", "blake2b") as bv:
        assert bv.verify_batch([proof], [inst[0]]).status == [0]
        assert bv.verify_batch([proof] * 3, [inst[0]] * 3).status == [0, 0, 0]
        bad = bv.verify_batch([proof[:40], b"", proof[:-1]], [inst[0]] * 3, want_batch_accum=True)
        assert bad.status == [2, 2, 3] and bad.batch_accum == bytes(128)
        mixed = bv.verify_batch([b"", proof], [inst[0]] * 2)
        assert mixed.status == [2, 0]
        with pytest.raises(AssertionError):
            bv.verify_batch([], [])
        v = ctypes.c_int(7)
        assert bv.lib.h2v_verify_batch(bv._ctx, 0, None, None, None, None, None, 0, None, None, None, None) != 0  # n = 0 is an argument error


def test_config5_shard_sizes_large_batch_tiled(pkg):
    """BASELINE.json configs[4] shard sizes: 16384 proofs on one GPU (what one of 4 GPUs gets of a 65,536-proof batch),
    4096 distinct proofs tiled; verdict, statuses and the folded accumulators against the C oracle's fold."""
    import c_oracle
    from importlib import import_module

    synth = import_module("halo2_verifier_b200.synth")
    n0, reps, k = 4096, 4, 10
    rng = random.Random(16384)
    s = rng.randrange(1, bn.R)
    vk_bytes, shared_dlogs = synth.make_vk_bytes("vm", k)
    pbytes = synth.params_bytes_raw(k, s)
    co = c_oracle.COracle(pbytes, 1, vk_bytes, 1)
    with pkg.BatchVerifier(pkg.ParamsKZG.from_bytes(pbytes, pkg.SerdeFormat.RawBytes), pkg.VerifyingKey.from_bytes(vk_bytes)) as bv:
        proofs, insts = synth.synthesize_shplonk_batch(bv, shared_dlogs, s, n0, seed=("t", 5))
        st, _secs, lr, _ch = co.verify_many(*_pack(proofs, insts), n0, check_pairing=False, threads=os.cpu_count() or 1, want_lr=True)
        assert int(st.max()) == 0
        n = n0 * reps
        rs = [rng.randrange(1, bn.R) for _ in range(n)]
        res = bv.verify_batch(proofs * reps, insts * reps, rlc_scalars=rs, want_batch_accum=True)
        assert res.verdict and res.status == [0] * n
        assert bv.msm_geometry()["terms"] == n * (bv.n_points + bv.n_mo) + bv.n_shared
        folded, ok = co.fold(lr * reps, rs, [True] * n)
        assert ok and res.batch_accum == folded
    co.close()


def test_graph_replay_equals_direct_launches(pkg):
    """The batch kernels run as a replayed CUDA graph by default.  Same results as the direct launches (statuses,
    challenges, accumulators, folded pair), re-capture when the batch shape changes, and repeated replays over new
    proof bytes in the same buffers; only the direct launches carry per-stage event timings."""
    params, vk, instances, proofs, rng = make_batch("vm", 8, 9, "shplonk", "blake2b")
    rs = [rng.randrange(1, bn.R) for _ in proofs]
    bad = list(proofs)
    bad[2], _ = sim.corrupt(proofs[2], vk, list(sim.CORRUPTIONS)[0], rng, "shplonk")
    with make_bv(pkg, params, vk, "shplonk", "blake2b") as bv:
        runs = {}
        # mode word of h2v_ctx_set_graphs: bit 0 = graph replay, bit 1 = programmatic dependent launch (default off, ADVICE r1)
        for mode in (1, 0, 1, 3, 2):
            graphs = bool(mode & 1)
            bv._check(bv.lib.h2v_ctx_set_graphs(bv._ctx, mode))
            for name, pr, n in (("all", proofs, 9), ("bad", bad, 9), ("short", proofs, 5), ("all2", proofs, 9)):
                res = bv.verify_batch(pr[:n], [i[0] for i in instances[:n]], rlc_scalars=rs[:n], want_challenges=True, want_accum=True, want_batch_accum=True)
                got = (res.verdict, tuple(res.status), bytes(res.challenges), bytes(res.accum), bytes(res.batch_accum))
                assert runs.setdefault(name, got) == got, (name, mode)
                t = bv.timings()
                assert t["total"] > 0 and (t["scalar"] > 0) == (not graphs)
        assert runs["all"][0] and not runs["bad"][0] and runs["bad"][1][2] != 0 and runs["all"] == runs["all2"]
        check_against_oracle(bv, params, vk, instances, bad, "shplonk", "blake2b", rs)


@pytest.mark.parametrize("mo", ["shplonk", "gwc"])
def test_fold_groups_equal_separate_batches(pkg, mo):
    """G independent batches in ONE set of kernel launches (h2v_batch_set_fold_groups): per-proof statuses, challenges
    and accumulators equal those of G separate calls, every group gets the verdict of its own fold (a bad proof only
    rejects its own group, attribution stays inside it), fold coefficients restart in every group."""
    G, n = 3, 5
    params, vk, instances, proofs, rng = make_batch("vm", 8, G * n, mo, "blake2b")
    insts = [i[0] for i in instances]
    rs = [rng.randrange(1, bn.R) for _ in proofs]
    bad = list(proofs)
    bad[n + 2], _ = sim.corrupt(proofs[n + 2], vk, "eval_flip", rng, mo)  # only the pairing check of its group can see it
    with make_bv(pkg, params, vk, mo, "blake2b") as bv:
        for pr in (proofs, bad):
            whole = bv.verify_batch(pr, insts, rlc_scalars=rs, want_challenges=True, want_accum=True, fold_groups=G)
            C = bv.n_challenges
            want_gv = []
            for g_ in range(G):
                sl = slice(g_ * n, (g_ + 1) * n)
                part = bv.verify_batch(pr[sl], insts[sl], rlc_scalars=rs[sl], want_challenges=True, want_accum=True, want_batch_accum=True)
                assert whole.status[sl] == part.status
                assert whole.challenges[32 * C * g_ * n: 32 * C * (g_ + 1) * n] == part.challenges
                assert whole.accum[128 * g_ * n: 128 * (g_ + 1) * n] == part.accum
                want_gv.append(part.verdict)
            assert whole.group_verdicts == want_gv and whole.verdict == all(want_gv)
        assert want_gv == [True, False, True]
        # the grouped run without the accumulator hook: attribution restricted to the rejected group
        res = bv.verify_batch(bad, insts, rlc_scalars=rs, fold_groups=G)
        assert res.group_verdicts == [True, False, True] and [i for i, s_ in enumerate(res.status) if s_] == [n + 2]
        want = [orc.verify_proof(params, vk, inst, p, mo, "blake2b").status for inst, p in zip(instances, bad)]
        assert res.status == want
        with pytest.raises(Exception):
            bv.verify_batch(proofs, insts, fold_groups=4)  # 15 proofs do not split into 4 groups


def test_sharded_fold_groups(pkg):
    """Fold groups across shards: G global batches, every rank holds its shard of each and processes all of them in one
    set of launches; the G partials per rank are concatenated ([rank][group]) and finalized together.  Verdicts equal
    those of the unsharded grouped run and of the separate batches; a corrupted proof rejects only its global batch."""
    G, n, shards = 3, 64, 2
    per = n // shards
    params, vk, instances, proofs, rng = make_batch("vm", 10, 32, "shplonk", "blake2b", seed=5)
    proofs, insts = proofs * 6, [i[0] for i in instances] * 6  # G * n = 192 proofs, global batch q = proofs[q*n:(q+1)*n]
    rs = [rng.randrange(1, bn.R) for _ in range(G * n)]
    bad = list(proofs)
    bad[n + 40], _ = sim.corrupt(proofs[n + 40], vk, "eval_flip", rng)
    with make_bv(pkg, params, vk, "shplonk", "blake2b") as b0, make_bv(pkg, params, vk, "shplonk", "blake2b") as b1:
        for pr, want in ((proofs, [True, True, True]), (bad, [True, False, True])):
            whole = b0.verify_batch(pr, insts, rlc_scalars=rs, fold_groups=G)
            assert whole.group_verdicts == want
            parts = []
            for rank, bv in ((0, b0), (1, b1)):
                sel = [q * n + rank * per + j for q in range(G) for j in range(per)]  # this rank's shard of every global batch
                st, partial = bv.accumulate_shard([pr[i] for i in sel], [insts[i] for i in sel], rank * per, n, rlc_scalars=rs, fold_groups=G)
                assert st == [0] * len(sel) and len(partial) == G * pkg.load_library().h2v_partial_bytes()
                parts.append(partial)
            assert b1.finalize_groups(parts, G) == want
            # the same global batches one at a time through the single-group shard API
            for q in range(G):
                single = [bv.accumulate_shard(pr[q * n + r_ * per: q * n + (r_ + 1) * per], insts[q * n + r_ * per: q * n + (r_ + 1) * per], r_ * per, n,
                                              rlc_scalars=rs[q * n:(q + 1) * n])[1] for r_, bv in ((0, b0), (1, b1))]
                assert b0.finalize(single)[0] == want[q]


def test_verify_batches_sharded_world1(pkg):
    """sharding.verify_batches_sharded (the reference-facing helper for G global batches per launch set) at world size 1"""
    from importlib import import_module

    sharding = import_module("halo2_verifier_b200.sharding")
    G, n = 2, 8
    params, vk, instances, proofs, rng = make_batch("vm", 8, G * n, "gwc", "keccak")
    insts = [i[0] for i in instances]
    bad = list(proofs)
    bad[3], _ = sim.corrupt(proofs[3], vk, "eval_flip", rng, "gwc")
    with make_bv(pkg, params, vk, "gwc", "keccak", F.PROCESSED) as bv:
        batches = [(bad[q * n:(q + 1) * n], insts[q * n:(q + 1) * n]) for q in range(G)]
        verdicts, status = sharding.verify_batches_sharded(bv, batches, 0, 1, seed=5)
        assert verdicts == [False, True]
        want = [orc.verify_proof(params, vk, inst, p, "gwc", "keccak").status for inst, p in zip(instances, bad)]
        assert status[0] + status[1] == want and status[0][3] == orc.CONSTRAINT_SYSTEM_FAILURE


@pytest.mark.parametrize("shape,k,m,mo", [("mix", 6, 3, "shplonk"), ("vm", 8, 2, "gwc")])
def test_multi_instance_proofs(pkg, shape, k, m, mo):
    """Proofs carrying m circuit instances in one transcript (h2v_ctx_create_multi; `instances.len() = m` in the reference's
    verify_proof): statuses, challenges, MSM scalars, per-proof and folded accumulators against the oracle, with one
    corrupted proof and one proof whose LAST instance has a wrong public input."""
    from workloads import setup

    params, vk, dl, s = setup(shape, k)
    rng = random.Random(f"gpu-multi-{shape}{k}{m}{mo}")
    n = 5
    insts = [[sim.random_instances(vk, rng, 6)[0] for _ in range(m)] for _ in range(n)]
    proofs = [sim.simulate_proof(params, vk, dl, s, inst, rng, mo, "blake2b") for inst in insts]
    proofs[1], _ = sim.corrupt(proofs[1], vk, "eval_flip", rng, mo, m)
    if vk.cs.num_instance_columns:
        insts[3] = [[list(c) for c in inst] for inst in insts[3]]
        insts[3][-1][0][0] = (insts[3][-1][0][0] + 1) % bn.R
    rs = [rng.randrange(1, bn.R) for _ in range(n)]
    bv = pkg.BatchVerifier(pkg.ParamsKZG.from_bytes(params.to_bytes()), pkg.VerifyingKey.from_bytes(vk.to_bytes(F.RAW_BYTES), F.RAW_BYTES),
                           mo, "blake2b", device=0, circuit_instances=m)
    with bv:
        assert bv.proof_len == len(proofs[0]) and bv.n_inst_cols == m * vk.cs.num_instance_columns
        res = bv.verify_batch(proofs, insts, rlc_scalars=rs, want_challenges=True, want_accum=True, want_batch_accum=True, want_scalars=True)
        want = [orc.verify_proof(params, vk, inst, p, mo, "blake2b") for inst, p in zip(insts, proofs)]
        assert res.status == [w.status for w in want] and res.status[1] == 4 and res.status[0] == 0
        C, nb = bv.n_challenges, bv.n_bases
        for j, w in enumerate(want):
            assert split32(res.challenges[32 * C * j:], C) == w.challenges
            assert split32(res.msm_scalars[32 * nb * j:], nb) == oracle_scalars(vk, w, bv.n_points, bv.n_mo)
            assert res.accum[128 * j: 128 * j + 128] == enc_point(w.L) + enc_point(w.R)
        L, R_, ok = orc.accumulate(params, want, rs)
        assert res.batch_accum == enc_point(L) + enc_point(R_) and not ok and not res.verdict


def test_honest_multi_instance_proof_through_the_c_abi(pkg):
    """An honest proof for 3 circuit instances of the vector_mul circuit (oracle/honest_prover.prove_multi: real witnesses,
    real polynomials) is accepted by the CUDA path; swapped public inputs and a cheat in one instance are rejected."""
    import honest_prover as hp

    rng = random.Random("gpu-honest-multi")
    s = rng.randrange(1, bn.R)
    params, vk, pk = hp.keygen_vm(6, s, 4)
    m = 3
    wit = [([rng.randrange(bn.R) for _ in range(4)], [rng.randrange(bn.R) for _ in range(4)]) for _ in range(m)]
    asg = [hp.vm_assignment(l, r) for l, r in wit]
    proof = hp.prove_multi(params, vk, pk, s, [a for a, _ in asg], [i for _, i in asg], rng)
    insts = [i for _, i in asg]
    asg_bad = list(asg)
    asg_bad[2] = hp.vm_assignment(*wit[2], cheat_row=1)
    bad = hp.prove_multi(params, vk, pk, s, [a for a, _ in asg_bad], [i for _, i in asg_bad], rng, expect_honest=False)
    bv = pkg.BatchVerifier(pkg.ParamsKZG.from_bytes(params.to_bytes()), pkg.VerifyingKey.from_bytes(vk.to_bytes(F.RAW_BYTES), F.RAW_BYTES),
                           "shplonk", "blake2b", device=0, circuit_instances=m)
    with bv:
        res = bv.verify_batch([proof, proof, bad], [insts, [insts[1], insts[0], insts[2]], [i for _, i in asg_bad]],
                              want_challenges=True, want_accum=True)
        assert res.status == [0, 4, 4]
        w = orc.verify_proof(params, vk, insts, proof)
        assert w.status == 0 and split32(res.challenges, bv.n_challenges) == w.challenges
        assert res.accum[:128] == enc_point(w.L) + enc_point(w.R)


def test_honest_gwc_proof_through_the_c_abi(pkg):
    """Honest proofs opened with GWC (oracle/honest_prover, multiopen="gwc"): the lookup + shuffle + rotated-gate circuit and a
    two-instance vector_mul proof through the CUDA path, with one cheating witness each."""
    import honest_prover as hp

    rng = random.Random("gpu-honest-gwc")
    s = rng.randrange(1, bn.R)
    circ = hp.lookup_shuffle_circuit(6, 16)
    params, vk, pk = hp.keygen(circ, s)
    adv, ins = hp.lookup_shuffle_assignment(circ, 16, rng)
    good = hp.prove(params, vk, pk, s, adv, ins, rng, multiopen="gwc")
    adv_b, ins_b = hp.lookup_shuffle_assignment(circ, 16, rng, "lookup")
    bad = hp.prove(params, vk, pk, s, adv_b, ins_b, rng, expect_honest=False, multiopen="gwc")
    with make_bv(pkg, params, vk, "gwc", "blake2b") as bv:
        res = bv.verify_batch([good, bad], [ins, ins_b], want_accum=True)
        w = orc.verify_proof(params, vk, [ins], good, "gwc")
        assert res.status == [0, 4] and w.status == 0 and res.accum[:128] == enc_point(w.L) + enc_point(w.R)
    params, vk, pk = hp.keygen_vm(6, s, 4)
    wit = [([rng.randrange(bn.R) for _ in range(4)], [rng.randrange(bn.R) for _ in range(4)]) for _ in range(2)]
    asg = [hp.vm_assignment(l, r) for l, r in wit]
    proof = hp.prove_multi(params, vk, pk, s, [a for a, _ in asg], [i for _, i in asg], rng, multiopen="gwc")
    insts = [i for _, i in asg]
    bv = pkg.BatchVerifier(pkg.ParamsKZG.from_bytes(params.to_bytes()), pkg.VerifyingKey.from_bytes(vk.to_bytes(F.RAW_BYTES), F.RAW_BYTES),
                           "gwc", "blake2b", device=0, circuit_instances=2)
    with bv:
        assert bv.verify_batch([proof, proof], [insts, insts[::-1]]).status == [0, 4]


def test_honest_two_phase_proof_through_the_c_abi(pkg):
    """The two-phase circuit with a user challenge (oracle/honest_prover.two_phase_circuit): honest proof accepted, phase-1
    cheat and wrong public input rejected by the CUDA path; challenges equal the oracle's."""
    import honest_prover as hp

    rng = random.Random("gpu-honest-phases")
    s = rng.randrange(1, bn.R)
    circ = hp.two_phase_circuit(5, 6)
    params, vk, pk = hp.keygen(circ, s)
    adv, ins = hp.two_phase_assignment([rng.randrange(bn.R) for _ in range(6)])
    good = hp.prove_multi(params, vk, pk, s, [adv], [ins], rng)
    adv_b, ins_b = hp.two_phase_assignment(ins[0], cheat=True)
    bad = hp.prove_multi(params, vk, pk, s, [adv_b], [ins_b], rng, expect_honest=False)
    wrong = [list(ins[0])]
    wrong[0][1] = (wrong[0][1] + 1) % bn.R
    with make_bv(pkg, params, vk, "shplonk", "blake2b") as bv:
        res = bv.verify_batch([good, bad, good], [ins, ins_b, wrong], want_challenges=True)
        w = orc.verify_proof(params, vk, [ins], good)
        assert res.status == [0, 4, 4] and w.status == 0 and split32(res.challenges, bv.n_challenges) == w.challenges
