"""Aggregation proofs (include/h2v.h "aggregation proofs"): the KZG accumulator (lhs, rhs) an aggregation circuit carries in
its public instances is decoded on the device and folded as two more MSM terms, rho * rhs on the left and rho * lhs on the
right.  The checker is the CPU oracle extended by tests/agg_oracle.py (ao.verify_proof(..., accumulator=, rho=)).  Fixtures are
synthetic: prover_sim yields accepting outer proofs for any instances and the SRS trapdoor s is known, so a valid carried
pair is (lhs, rhs) = (s P, P) for a random P."""
import ctypes
import functools
import os
import random

import pytest

import bn254 as bn
import formats as F
import prover_sim as sim
import agg_oracle as ao
import verifier as orc
from test_mixed_batch import Circ, S
from workloads import enc_point

HERE = os.path.dirname(os.path.abspath(__file__))
ENCODINGS = ((3, 88), (4, 68))  # halo2-lib, halo2wrong


class Spec:
    """the oracle's view of an InstanceAccumulator"""

    def __init__(self, limbs, bits, cells):
        self.limbs, self.bits, self.cells = limbs, bits, tuple(cells)

    def api(self, pkg):
        return pkg.InstanceAccumulator(self.limbs, self.bits, self.cells)


def _pair(rng, valid=True):
    P = bn.g1_mul_gen(rng.randrange(1, bn.R))
    return (bn.g1_mul(P, S if valid else S + 1), P)


def _place(insts, spec, lhs, rhs):
    """writes the encoded pair into the [circuit][column][row] instances at spec.cells (columns flattened instance-major)"""
    cols = [col for inst in insts for col in inst]
    for (c, r), v in zip(spec.cells, ao.encode_accumulator(lhs, rhs, spec.limbs, spec.bits)):
        cols[c][r] = v
    return insts


# ---------------------------------------------------------------- CPU: decoding (csrc/agg.cuh) against the oracle
@functools.lru_cache(maxsize=None)
def _agglib():
    return ctypes.CDLL(os.path.join(HERE, "hostlib", "libagg.so"))


def _host_decode(limbs, bits, values):
    out, ids = ctypes.create_string_buffer(128), ctypes.create_string_buffer(2)
    buf = b"".join(int(v).to_bytes(32, "little") for v in values)
    ok = _agglib().x_agg_decode(limbs, bits, buf, out, ids)
    if ok != 1:
        return None
    pts = []
    for q in range(2):
        x, y = (int.from_bytes(out.raw[64 * q + 32 * i: 64 * q + 32 * i + 32], "little") for i in range(2))
        assert (x, y) == (0, 0) if ids.raw[q] else True
        pts.append(None if ids.raw[q] else (x, y))
    return tuple(pts)


def _py_decode(limbs, bits, values):
    spec = Spec(limbs, bits, [(0, i) for i in range(4 * limbs)])
    return ao.decode_accumulator([[list(values)]], spec)


def test_host_decoding_matches_the_oracle(built):
    rng = random.Random("agg-decode")
    for limbs, bits in ENCODINGS + ((2, 128), (8, 32)):
        cases = []
        for _ in range(6):
            lhs, rhs = _pair(rng, rng.random() < 0.5)
            cases.append(ao.encode_accumulator(lhs, rhs, limbs, bits))
        cases.append(ao.encode_accumulator(None, _pair(rng)[1], limbs, bits))  # the identity
        cases.append(ao.encode_accumulator(None, None, limbs, bits))
        good = ao.encode_accumulator(*_pair(rng), limbs, bits)
        v = list(good)
        v[0] += 1 << bits  # a limb of exactly 2^bits more: the same coordinate mod 2^(limbs bits) would be hidden
        cases.append(v)
        v = list(good)
        v[limbs - 1] = 1 << bits  # a limb of exactly 2^bits
        cases.append(v)
        for x in (bn.P, bn.P - 1):  # coordinate = q (not canonical), q - 1 (canonical; on the curve or not)
            cases.append(ao.encode_accumulator((x, 2), _pair(rng)[1], limbs, bits) if x < (1 << (limbs * bits)) else good)
        v = list(good)
        v[0] ^= 1  # off-curve x
        cases.append(v)
        for _ in range(4):  # random limbs: mostly off-curve
            cases.append([rng.randrange(1 << bits) for _ in range(4 * limbs)])
        for values in cases:
            want = _py_decode(limbs, bits, values)
            assert _host_decode(limbs, bits, values) == want, (limbs, bits, values)
        assert _host_decode(limbs, bits, good) is not None
    # (q, 2) is rejected as non-canonical, a limb of 2^bits as out of range, the identity accepted
    assert _py_decode(3, 88, ao.encode_accumulator((bn.P, 2), None, 3, 88)) is None
    assert _py_decode(3, 88, ao.encode_accumulator(None, None, 3, 88)) == (None, None)


def test_oracle_accepts_valid_pairs_and_rejects_false_ones():
    C = _circ("vm8")
    rng = random.Random("agg-oracle")
    spec = _spec(C, 3, 88)
    rho = rng.randrange(1, bn.R)
    for how, ok in (("valid", True), ("false", False), ("swapped", False)):
        lhs, rhs = _pair(rng, how != "false")
        if how == "swapped":
            lhs, rhs = rhs, lhs
        insts = _place(C.instances(rng, 16), spec, lhs, rhs)
        proof = sim.simulate_proof(C.params, C.vk, C.dl, S, insts, rng, C.mo, C.hk)
        assert orc.verify_proof(C.params, C.vk, insts, proof, C.mo, C.hk).status == orc.OK  # the outer proof is valid
        got = ao.verify_proof(C.params, C.vk, insts, proof, C.mo, C.hk, accumulator=spec, rho=rho).status
        assert got == (orc.OK if ok else orc.CONSTRAINT_SYSTEM_FAILURE), how


def test_malformed_specs_are_refused_at_creation(built, pkg):
    C = _circ("vm8")
    params, vk = pkg.ParamsKZG.from_bytes(C.params.to_bytes()), pkg.VerifyingKey.from_bytes(C.vk.to_bytes(F.RAW_BYTES), F.RAW_BYTES)
    bad = [
        (pkg.InstanceAccumulator.rows(1, 254), "limbs"),
        (pkg.InstanceAccumulator.rows(9, 32), "limbs"),
        (pkg.InstanceAccumulator.rows(2, 129), "bits"),
        (pkg.InstanceAccumulator.rows(3, 84), "limbs \\* bits"),
        (pkg.InstanceAccumulator.rows(3, 88, column=1), "column 1"),
        (pkg.InstanceAccumulator(3, 88, ()), "cells is null"),
    ]
    for spec, msg in bad:
        with pytest.raises(pkg.BackendError, match="aggregation spec: .*" + msg):
            pkg.BatchVerifier(params, vk, accumulator=spec)


# ---------------------------------------------------------------- GPU
@functools.lru_cache(maxsize=None)
def _circ(name):
    return {"vm8": Circ("vm", 8, "shplonk", "blake2b"), "gwc": Circ("vm", 8, "gwc", "keccak"),
            "multi": Circ("mix", 6, "shplonk", "blake2b", m=3)}[name]


def _spec(C, limbs, bits):
    """the carried limbs in rows 2.. of column 0; on the multi-instance circuit spread over two flattened columns"""
    n = 4 * limbs
    if C.m == 1:
        return Spec(limbs, bits, [(0, 2 + i) for i in range(n)])
    ncols = C.vk.cs.num_instance_columns
    return Spec(limbs, bits, [(1, 1 + i) if i < n // 2 else (2 * ncols, i - n // 2) for i in range(n)])


def _make(C, spec, rng, n, valid=None, rows=20):
    """n accepting outer proofs whose instances carry a pair; valid[j] = False: lhs != s rhs"""
    insts, proofs = [], []
    for j in range(n):
        lhs, rhs = _pair(rng, True if valid is None else valid[j])
        i = _place(C.instances(rng, rows), spec, lhs, rhs)
        insts.append(i)
        proofs.append(sim.simulate_proof(C.params, C.vk, C.dl, S, i, rng, C.mo, C.hk))
    return insts, proofs


def _bv(pkg, C, spec):
    return pkg.BatchVerifier(pkg.ParamsKZG.from_bytes(C.params.to_bytes()), pkg.VerifyingKey.from_bytes(C.vk.to_bytes(F.RAW_BYTES), F.RAW_BYTES),
                             C.mo, "keccak256" if C.hk == "keccak" else C.hk, device=0, circuit_instances=C.m,
                             accumulator=None if spec is None else spec.api(pkg))


def _oracle(C, insts, proofs, spec, rho):
    return [ao.verify_proof(C.params, C.vk, i, p, C.mo, C.hk, accumulator=spec, rho=rho) for i, p in zip(insts, proofs)]


def _check(bv, C, insts, proofs, spec, rng, **kw):
    """statuses, per-proof (L_j, R_j) and folded (L, R) bit-exact with the oracle under caller rlc_scalars + agg_scalar"""
    rs = [rng.randrange(1, bn.R) for _ in proofs]
    rho = rng.randrange(1, bn.R)
    res = bv.verify_batch(proofs, C.api(insts), rlc_scalars=rs, agg_scalar=rho if spec else None, want_accum=True, want_batch_accum=True, **kw)
    want = _oracle(C, insts, proofs, spec, rho)
    assert res.status == [w.status for w in want]
    for j, w in enumerate(want):
        if w.status in (orc.OK, orc.CONSTRAINT_SYSTEM_FAILURE):
            assert res.accum[128 * j: 128 * j + 128] == enc_point(w.L) + enc_point(w.R), f"per-proof accumulator of proof {j}"
    L, R_, ok = orc.accumulate(C.params, want, rs)
    assert res.batch_accum == enc_point(L) + enc_point(R_)
    assert res.verdict == (ok and all(w.status == orc.OK for w in want))
    return res, want


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["vm8", "gwc", "multi"])
@pytest.mark.parametrize("enc", ENCODINGS)
def test_valid_aggregation_proofs_parity(pkg, name, enc):
    C = _circ(name)
    spec = _spec(C, *enc)
    rng = random.Random(("agg-parity", name, enc).__repr__())
    insts, proofs = _make(C, spec, rng, 5)
    with _bv(pkg, C, spec) as bv:
        res, _ = _check(bv, C, insts, proofs, spec, rng)
        assert res.verdict and res.status == [0] * 5


@pytest.mark.gpu
def test_false_accumulators_are_attributed_and_plain_context_does_not_check(pkg):
    C = _circ("vm8")
    spec = _spec(C, 3, 88)
    rng = random.Random("agg-false")
    valid = [True, False, True, True, True, True, False, True]
    insts, proofs = _make(C, spec, rng, 8, valid)
    lhs, rhs = _pair(rng)
    _place(insts[4], spec, rhs, lhs)  # swapped pair
    proofs[4] = sim.simulate_proof(C.params, C.vk, C.dl, S, insts[4], rng, C.mo, C.hk)
    proofs[2], _ = sim.corrupt(proofs[2], C.vk, "eval_flip", rng, C.mo)
    proofs[5], _ = sim.corrupt(proofs[5], C.vk, "scalar_ge_r", rng, C.mo)
    with _bv(pkg, C, spec) as bv:
        res, want = _check(bv, C, insts, proofs, spec, rng)
    assert not res.verdict
    assert res.status == [0, orc.CONSTRAINT_SYSTEM_FAILURE, orc.CONSTRAINT_SYSTEM_FAILURE, 0, orc.CONSTRAINT_SYSTEM_FAILURE, orc.TRANSCRIPT,
                          orc.CONSTRAINT_SYSTEM_FAILURE, 0]
    with _bv(pkg, C, None) as plain:  # the same proofs on a plain context: the carried accumulator is not checked
        res, _ = _check(plain, C, insts, proofs, None, rng)
    assert res.status == [0, 0, orc.CONSTRAINT_SYSTEM_FAILURE, 0, 0, orc.TRANSCRIPT, 0, 0]


@pytest.mark.gpu
def test_malformed_encodings_are_invalid_instances_per_proof(pkg):
    C = _circ("vm8")
    spec = _spec(C, 4, 68)
    rng = random.Random("agg-malformed")
    insts, proofs = _make(C, spec, rng, 7)
    col = lambda j: insts[j][0][0]
    col(1)[spec.cells[0][1]] = 1 << 68  # a limb of 2^bits
    x = ao.encode_accumulator((bn.P, 2), None, 4, 68)  # lhs.x = q
    for (c, r), v in zip(spec.cells[:4], x[:4]):
        col(2)[r] = v
    col(3)[spec.cells[5][1]] ^= 1  # lhs.y changed: off the curve
    col(4)[spec.cells[12][1]] ^= 1  # rhs.x changed: off the curve
    for j in (1, 2, 3, 4):
        proofs[j] = sim.simulate_proof(C.params, C.vk, C.dl, S, insts[j], rng, C.mo, C.hk)
    del insts[5][0][0][spec.cells[-1][1]:]  # a ragged column too short for the last cell
    proofs[5] = sim.simulate_proof(C.params, C.vk, C.dl, S, insts[5], rng, C.mo, C.hk)
    proofs[6], _ = sim.corrupt(proofs[6], C.vk, "truncate_body", rng, C.mo)
    col(6)[spec.cells[0][1]] = 1 << 68  # invalid encoding AND a transcript failure: the instance status wins
    with _bv(pkg, C, spec) as bv:
        res, _ = _check(bv, C, insts, proofs, spec, rng)
    assert res.status == [0] + [orc.INVALID_INSTANCES] * 6 and not res.verdict


@pytest.mark.gpu
def test_verify_proof_single(pkg):
    C = _circ("vm8")
    spec = _spec(C, 3, 88)
    rng = random.Random("agg-single")
    insts, proofs = _make(C, spec, rng, 2, [True, False])
    params, vk = pkg.ParamsKZG.from_bytes(C.params.to_bytes()), pkg.VerifyingKey.from_bytes(C.vk.to_bytes(F.RAW_BYTES), F.RAW_BYTES)
    assert pkg.verify_proof(params, vk, proofs[0], insts[0][0], accumulator=spec.api(pkg)) is None
    with pytest.raises(pkg.ConstraintSystemFailure):
        pkg.verify_proof(params, vk, proofs[1], insts[1][0], accumulator=spec.api(pkg))
    pkg.verify_proof(params, vk, proofs[1], insts[1][0])  # a plain context accepts it
    errs = pkg.verify_proofs_batch(params, vk, proofs, [i[0] for i in insts], accumulator=spec.api(pkg))
    assert errs[0] is None and isinstance(errs[1], pkg.ConstraintSystemFailure)


@pytest.mark.gpu
def test_fold_groups_graphs_and_randomness_sources(pkg):
    C = _circ("vm8")
    spec = _spec(C, 4, 68)
    rng = random.Random("agg-groups")
    valid = [True] * 16
    valid[11] = False
    insts, proofs = _make(C, spec, rng, 16, valid)
    want = [orc.CONSTRAINT_SYSTEM_FAILURE if not v else orc.OK for v in valid]
    with _bv(pkg, C, spec) as bv:
        res = bv.verify_batch(proofs, C.api(insts), fold_groups=4)
        assert res.group_verdicts == [True, True, False, True] and res.status == want
        rs, rho = [rng.randrange(1, bn.R) for _ in proofs], rng.randrange(1, bn.R)
        outs = []
        for graphs in (1, 0, 1):
            bv.set_graphs(graphs)
            r = bv.verify_batch(proofs, C.api(insts), rlc_scalars=rs, agg_scalar=rho, want_batch_accum=True)
            outs.append((r.status, r.batch_accum))
        assert outs[0] == outs[1] == outs[2] and outs[0][0] == want
        for kw, src in (({"rlc_scalars": rs}, "scalars"), ({"seed": 7}, "seed"), ({"key": bytes(range(32))}, "key"), ({}, "os")):
            r = bv.verify_batch(proofs, C.api(insts), **kw)
            assert r.status == want and not r.verdict and bv.rlc_source() == src
        assert bv.verify_batch(proofs[:11], C.api(insts[:11]), seed=9).verdict


@pytest.mark.gpu
def test_mixed_batch_with_an_aggregation_member(pkg):
    A, B = _circ("vm8"), _circ("gwc")
    spec = _spec(A, 3, 88)
    rng = random.Random("agg-mix")
    ia, pa = _make(A, spec, rng, 4, [True, True, False, True])
    ib, pb = B.proofs(rng, 3)
    rs, rho = [rng.randrange(1, bn.R) for _ in range(7)], rng.randrange(1, bn.R)
    ba, bb = _bv(pkg, A, spec), _bv(pkg, B, None)
    try:
        with pkg.MixedBatchVerifier([ba, bb]) as mx:
            res = mx.verify_batch([pa, pb], [A.api(ia), B.api(ib)], rlc_scalars=rs, agg_scalar=rho, want_batch_accum=True)
            want = _oracle(A, ia, pa, spec, rho) + B.oracle(ib, pb)
            assert res.status == [[w.status for w in want[:4]], [w.status for w in want[4:]]]
            assert res.status[0][2] == orc.CONSTRAINT_SYSTEM_FAILURE and not res.verdict
            L, R_, _ok = orc.accumulate(A.params, want, rs)
            assert res.batch_accum == enc_point(L) + enc_point(R_)
    finally:
        ba.close()
        bb.close()


@pytest.mark.gpu
def test_chunked_absorbs_and_shards_equal_one_batch(pkg):
    C = _circ("vm8")
    spec = _spec(C, 3, 88)
    rng = random.Random("agg-absorb")
    insts, proofs = _make(C, spec, rng, 12)
    rs, rho = [rng.randrange(1, bn.R) for _ in proofs], rng.randrange(1, bn.R)
    bv, bv2 = _bv(pkg, C, spec), _bv(pkg, C, spec)
    try:
        one = bv.verify_batch(proofs, C.api(insts), rlc_scalars=rs, agg_scalar=rho, want_batch_accum=True)
        L, R_, ok = orc.accumulate(C.params, _oracle(C, insts, proofs, spec, rho), rs)
        assert one.verdict and ok and one.batch_accum == enc_point(L) + enc_point(R_)
        with pkg.Accumulator(bv) as acc:
            for a, b in ((0, 5), (5, 12)):
                r = acc.absorb(bv, proofs[a:b], C.api(insts[a:b]), rlc_scalars=rs[a:b], agg_scalar=rho)
                assert r.statuses == [0] * (b - a)
            assert acc.to_bytes() == one.batch_accum
            assert acc.finalize().verdict
        # two shards of one global batch on two contexts, one pairing check at finalize
        st0, p0 = bv.accumulate_shard(proofs[:6], C.api(insts[:6]), 0, 12, rlc_scalars=rs, agg_scalar=rho)
        st1, p1 = bv2.accumulate_shard(proofs[6:], C.api(insts[6:]), 6, 12, rlc_scalars=rs, agg_scalar=rho)
        verdict, bacc = bv.finalize([p0, p1])
        assert st0 + st1 == [0] * 12 and verdict and bacc == one.batch_accum
        bad = list(insts)
        lhs, rhs = _pair(rng, False)
        bad[8] = _place(C.instances(rng, 20), spec, lhs, rhs)
        bproofs = list(proofs)
        bproofs[8] = sim.simulate_proof(C.params, C.vk, C.dl, S, bad[8], rng, C.mo, C.hk)
        _st0, p0 = bv.accumulate_shard(bproofs[:6], C.api(bad[:6]), 0, 12, seed=3)
        st1, p1 = bv2.accumulate_shard(bproofs[6:], C.api(bad[6:]), 6, 12, seed=3)
        verdict, _ = bv.finalize([p0, p1])
        assert not verdict and bv2.attribute_shard(st1) == [0, 0, orc.CONSTRAINT_SYSTEM_FAILURE, 0, 0, 0]
    finally:
        bv.close()
        bv2.close()
