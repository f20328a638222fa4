"""Mixed batches (include/h2v.h "mixed batches"): proofs of several verifying keys folded into one MSM and one pairing
check.  The checker is the CPU oracle: orc.accumulate over the member-major concatenation of the per-proof oracle results
IS the reference's AccumulatorStrategy fed proofs of several VKs under one set of KZG params."""
import ctypes
import functools
import hashlib
import os
import random

import pytest

import bn254 as bn
import formats as F
import prover_sim as sim
import verifier as orc
from workloads import enc_point

HERE = os.path.dirname(os.path.abspath(__file__))
S = sim.FIXTURE_SRS_SECRET  # one trapdoor for every circuit: the params agree on (g, g2, s_g2)


# ---------------------------------------------------------------- CPU: the segment mapping (csrc/mix.cuh)
@functools.lru_cache(maxsize=None)
def _mixlib():
    return ctypes.CDLL(os.path.join(HERE, "hostlib", "libmix.so"))


def _map(shapes):
    lib = _mixlib()
    flat = (ctypes.c_uint32 * (4 * len(shapes)))(*[v for sh in shapes for v in sh])
    cap = sum(n * (P + M) + Sh for n, P, M, Sh in shapes if n)
    out = (ctypes.c_uint32 * max(1, 6 * cap))()
    nseg = ctypes.c_uint32(0)
    lib.x_map.restype = ctypes.c_longlong
    total = lib.x_map(len(shapes), flat, out, ctypes.c_ulonglong(cap), ctypes.byref(nseg))
    assert total == cap
    return nseg.value, [tuple(out[6 * t: 6 * t + 6]) for t in range(total)]


def test_segment_mapping_is_a_bijection(built):
    rng = random.Random("mix-map")
    tables = [[(0, 5, 2, 3), (7, 5, 2, 3)], [(3, 4, 1, 2)], [(0, 1, 1, 1), (0, 2, 2, 2)] + [(1, 1, 0, 1)]]
    for _ in range(40):
        tables.append([(rng.choice([0, 0, 1, 2, 5, 17]), rng.randint(1, 20), rng.randint(0, 4), rng.randint(1, 9)) for _ in range(rng.randint(1, 64))])
    for shapes in tables:
        if not any(n for n, *_ in shapes):
            continue
        nseg, rows = _map(shapes)
        assert nseg == sum(1 for n, *_ in shapes if n)
        want = set()
        for m, (n, P, M, Sh) in enumerate(shapes):
            if not n:
                continue
            want |= {(m, 0, j, i) for j in range(n) for i in range(P)}
            want |= {(m, 1, j, i) for j in range(n) for i in range(M)}
            want |= {(m, 2, 0, i) for i in range(Sh)}
        got = [(m, kind, j, i) for _s, m, kind, j, i, _ch in rows]
        assert len(got) == len(set(got)) and set(got) == want  # every (member, proof, base) exactly once
        assert all(ch == (kind == 1) for _s, _m, kind, _j, _i, ch in rows)  # left channel = the multi-open terms
        members = [m for m, (n, *_r) in enumerate(shapes) if n]
        assert all(members[s] == m for s, m, *_r in rows)
        firsts = [s for s, *_r in rows]
        assert firsts == sorted(firsts)  # segments are consecutive in term-id space


def test_single_segment_matches_single_vk_mapping(built):
    lib = _mixlib()
    lib.x_single_mismatches.restype = ctypes.c_longlong
    for n, P, M, Sh in [(1, 1, 0, 1), (4, 12, 2, 5), (37, 9, 3, 11), (256, 20, 4, 9)]:
        assert lib.x_single_mismatches(n, P, M, Sh) == 0


def test_mix_create_rejects_an_empty_member_list(built, pkg):
    with pytest.raises(pkg.BackendError, match="between 1 and 64"):
        pkg.MixedBatchVerifier([])


# ---------------------------------------------------------------- GPU
class Circ:
    """one circuit of the fixture: (shape, k, multiopen, hash, circuit instances, vk seed, trapdoor)"""

    def __init__(self, shape, k, mo, hk, m=1, vk_seed=0, s=S):
        self.shape, self.k, self.mo, self.hk, self.m, self.s = shape, k, mo, hk, m, s
        self.params = sim.make_params(k, s)
        self.vk, self.dl = sim.make_vk(shape, k, vk_seed)

    def bv(self, pkg):
        return pkg.BatchVerifier(pkg.ParamsKZG.from_bytes(self.params.to_bytes()), pkg.VerifyingKey.from_bytes(self.vk.to_bytes(F.RAW_BYTES), F.RAW_BYTES),
                                 self.mo, "keccak256" if self.hk == "keccak" else self.hk, device=0, circuit_instances=self.m)

    def instances(self, rng, rows=6):
        return [sim.random_instances(self.vk, rng, rows)[0] for _ in range(self.m)]

    def proofs(self, rng, n, rows=6):
        """(oracle instances [circuit][column][row], proofs); the API takes the same lists for m > 1 and inst[0] for m = 1"""
        insts = [self.instances(rng, rows) for _ in range(n)]
        return insts, [sim.simulate_proof(self.params, self.vk, self.dl, self.s, i, rng, self.mo, self.hk) for i in insts]

    def api(self, insts):
        return [i if self.m > 1 else i[0] for i in insts]

    def oracle(self, insts, proofs):
        return [orc.verify_proof(self.params, self.vk, i, p, self.mo, self.hk) for i, p in zip(insts, proofs)]


@functools.lru_cache(maxsize=None)
def circuits():
    return (Circ("vm", 8, "shplonk", "blake2b"), Circ("sh", 8, "gwc", "keccak"), Circ("mix", 6, "shplonk", "blake2b", m=3),
            Circ("vm", 10, "gwc", "blake2b"))


def _expand(tag, material, n):
    """r_i of the seed / key expansion (stages.cuh rlc_scalar_from_seed / _from_key)"""
    return [int.from_bytes(hashlib.blake2b(tag + material + i.to_bytes(8, "little"), digest_size=64, person=b"Halo2-Transcript").digest(),
                           "little") % bn.R for i in range(n)]


def _dec(e):
    return None if e == bytes(64) else (int.from_bytes(e[:32], "little"), int.from_bytes(e[32:], "little"))


def _check(mx, circs, insts, proofs, rs):
    """mixed batch against the oracle's AccumulatorStrategy over the member-major concatenation"""
    res = mx.verify_batch(proofs, [c.api(i) for c, i in zip(circs, insts)], rlc_scalars=rs, want_batch_accum=True)
    want = [c.oracle(i, p) for c, i, p in zip(circs, insts, proofs)]
    assert res.status == [[w.status for w in ws] for ws in want]
    L, R_, ok = orc.accumulate(circs[0].params, [w for ws in want for w in ws], rs)
    assert res.batch_accum == enc_point(L) + enc_point(R_)
    assert res.verdict == (ok and all(w.status == orc.OK for ws in want for w in ws))
    return res, want


@pytest.mark.gpu
def test_mixed_parity_against_oracle(pkg):
    """SHPLONK + GWC, Blake2b + Keccak, 3 circuit instances per proof, ragged instances on one member, a member with no
    proofs; and a one-member mix equals that member's own batch"""
    A, B, C, D = circuits()
    rng = random.Random("mix-parity")
    ia = [sim.random_instances(A.vk, rng, 3 + 5 * t) for t in range(4)]  # ragged public inputs: lengths differ per proof
    pa = [sim.simulate_proof(A.params, A.vk, A.dl, S, i, rng) for i in ia]
    ia.append([[]])  # wrong column count -> InvalidInstances, through the member's column layout
    pa.append(pa[0])
    ib, pb = B.proofs(rng, 3)
    ic, pc = C.proofs(rng, 3)
    bvs = [c.bv(pkg) for c in (A, B, C, D)]
    try:
        with pkg.MixedBatchVerifier(bvs) as mx:
            rs = [rng.randrange(1, bn.R) for _ in range(11)]
            res, want = _check(mx, (A, B, C, D), [ia, ib, ic, []], [pa, pb, pc, []], rs)
            assert res.status[0][4] == orc.INVALID_INSTANCES and res.status[3] == [] and not res.verdict
            res, _ = _check(mx, (A, B, C, D), [ia[:4], ib, ic, []], [pa[:4], pb, pc, []], rs[:10])
            assert res.verdict
        with pkg.MixedBatchVerifier(bvs[1:2]) as one:
            rs = rs[:3]
            res, _ = _check(one, (B,), [ib], [pb], rs)
            own = bvs[1].verify_batch(pb, B.api(ib), rlc_scalars=rs, want_batch_accum=True)
            assert res.batch_accum == own.batch_accum and res.status == [own.status] and res.verdict
    finally:
        [bv.close() for bv in bvs]


@pytest.mark.gpu
def test_mixed_rejection_attributed_per_member(pkg):
    """one proof of every corruption class, spread over the members: statuses as the oracle's, and only the corrupted
    proofs are flagged"""
    A, B, C, _D = circuits()
    rng = random.Random("mix-reject")
    circs = (A, B, C)
    insts, proofs = zip(*[c.proofs(rng, n) for c, n in zip(circs, (6, 5, 4))])
    proofs = [list(p) for p in proofs]
    slots = [(0, 0), (0, 2), (0, 3), (0, 5), (1, 0), (1, 1), (1, 4), (2, 1), (2, 2)]
    for kind, (m, j) in zip(sim.CORRUPTIONS, slots):
        proofs[m][j], _ = sim.corrupt(proofs[m][j], circs[m].vk, kind, rng, circs[m].mo, circs[m].m)
    bvs = [c.bv(pkg) for c in circs]
    try:
        with pkg.MixedBatchVerifier(bvs) as mx:
            res, _ = _check(mx, circs, list(insts), proofs, [rng.randrange(1, bn.R) for _ in range(15)])
            assert not res.verdict
            flagged = {(m, j) for m, st in enumerate(res.status) for j, v in enumerate(st) if v}
            assert flagged == set(slots)
            assert sum(v == orc.CONSTRAINT_SYSTEM_FAILURE for st in res.status for v in st) >= 2
    finally:
        [bv.close() for bv in bvs]


@pytest.mark.gpu
def test_cross_vk_proof_is_rejected_and_foreign_params_refused(pkg):
    A = circuits()[0]
    A2 = Circ("vm", 8, "shplonk", "blake2b", vk_seed=1)  # same layout, another verifying key
    rng = random.Random("mix-cross")
    ia, pa = A.proofs(rng, 3)
    i2, p2 = A2.proofs(rng, 4)
    i2[2], p2[2] = ia[0], pa[0]  # a proof of circuit A submitted under member A2
    bvs = [A.bv(pkg), A2.bv(pkg)]
    try:
        with pkg.MixedBatchVerifier(bvs) as mx:
            res, want = _check(mx, (A, A2), [ia, i2], [pa, p2], [rng.randrange(1, bn.R) for _ in range(7)])
            assert not res.verdict and res.status == [[0, 0, 0], [0, 0, want[1][2].status, 0]] and want[1][2].status != orc.OK
        X = Circ("vm", 8, "shplonk", "blake2b", s=S + 1)  # params of another trapdoor
        with X.bv(pkg) as bx:
            with pytest.raises(pkg.BackendError, match="differ"):
                pkg.MixedBatchVerifier([bvs[0], bx])
    finally:
        [bv.close() for bv in bvs]


@pytest.mark.gpu
def test_mixed_graph_replay_equals_direct_launches(pkg):
    A, B, C, _D = circuits()
    rng = random.Random("mix-graph")
    circs = (A, B, C)
    insts, proofs = zip(*[c.proofs(rng, n) for c, n in zip(circs, (5, 4, 3))])
    api = [c.api(i) for c, i in zip(circs, insts)]
    rs = [rng.randrange(1, bn.R) for _ in range(12)]
    bvs = [c.bv(pkg) for c in circs]
    try:
        with pkg.MixedBatchVerifier(bvs) as mx:
            a = mx.verify_batch(proofs, api, rlc_scalars=rs, want_batch_accum=True)
            caps = mx.cache_stats()["graph_captures"]
            b = mx.verify_batch(proofs, api, rlc_scalars=rs, want_batch_accum=True)
            assert mx.cache_stats()["graph_captures"] == caps and a == b and a.verdict  # same shapes: replay
            bad = [list(p) for p in proofs]
            bad[1][2], _ = sim.corrupt(bad[1][2], B.vk, "eval_flip", rng, B.mo)
            g = mx.verify_batch(bad, api, rlc_scalars=rs, want_batch_accum=True)
            bvs[0].set_graphs(False)
            d = mx.verify_batch(bad, api, rlc_scalars=rs, want_batch_accum=True)
            assert d == g and not d.verdict and d.status[1][2] == orc.CONSTRAINT_SYSTEM_FAILURE
            d2 = mx.verify_batch(proofs, api, rlc_scalars=rs, want_batch_accum=True)
            assert d2 == a
    finally:
        [bv.close() for bv in bvs]


@pytest.mark.gpu
def test_mixed_fold_randomness_sources(pkg):
    A, B, C, _D = circuits()
    rng = random.Random("mix-rand")
    circs = (A, B, C)
    insts, proofs = zip(*[c.proofs(rng, n) for c, n in zip(circs, (3, 2, 2))])
    api = [c.api(i) for c, i in zip(circs, insts)]
    bvs = [c.bv(pkg) for c in circs]
    try:
        with pkg.MixedBatchVerifier(bvs) as mx:
            seed = 0x5EED
            a = mx.verify_batch(proofs, api, seed=seed, want_batch_accum=True)
            assert bvs[0].rlc_source() == "seed"
            b = mx.verify_batch(proofs, api, rlc_scalars=_expand(b"h2v-rlc", seed.to_bytes(8, "little"), 7), want_batch_accum=True)
            assert a == b and a.verdict
            key = bytes(rng.getrandbits(8) for _ in range(32))
            c = mx.verify_batch(proofs, api, key=key, want_batch_accum=True)
            d = mx.verify_batch(proofs, api, rlc_scalars=_expand(b"h2v-rlk", key, 7), want_batch_accum=True)
            assert c == d and c.verdict and c.batch_accum != a.batch_accum
            e = mx.verify_batch(proofs, api, want_batch_accum=True)  # OS entropy
            f = mx.verify_batch(proofs, api, want_batch_accum=True)
            assert e.verdict and f.verdict and e.batch_accum != f.batch_accum and bvs[2].rlc_source() == "key"
        errs = pkg.verify_proofs_mixed([(pkg.ParamsKZG.from_bytes(c.params.to_bytes()), pkg.VerifyingKey.from_bytes(c.vk.to_bytes(F.RAW_BYTES)),
                                         p, a_, c.mo, "keccak256" if c.hk == "keccak" else c.hk) for c, p, a_ in zip((A, B), proofs[:2], api[:2])])
        assert errs == [[None] * 3, [None] * 2]
    finally:
        [bv.close() for bv in bvs]


@pytest.mark.gpu
def test_full_size_mix_properties(pkg):
    """vm k=10 x 4096 + sh k=8 x 1024 (64 / 32 distinct proofs tiled): all accepted; the mixed fold equals
    sum_m t_m A_m, A_m = member m's own folded accumulator under its slice of the r_i and t_m = the product of the r_i of
    every later member's slice; one corrupted proof is found"""
    V = Circ("vm", 10, "shplonk", "blake2b")
    B = circuits()[1]
    rng = random.Random("mix-full")
    iv, pv_ = V.proofs(rng, 64)
    ib, pb = B.proofs(rng, 32)
    iv, pv_, ib, pb = iv * 64, pv_ * 64, ib * 32, pb * 32
    nv, nb_ = len(pv_), len(pb)
    rs = [rng.randrange(1, bn.R) for _ in range(nv + nb_)]
    bvs = [V.bv(pkg), B.bv(pkg)]
    try:
        with pkg.MixedBatchVerifier(bvs) as mx:
            api = [V.api(iv), B.api(ib)]
            res = mx.verify_batch([pv_, pb], api, rlc_scalars=rs, want_batch_accum=True)
            assert res.verdict and res.status == [[0] * nv, [0] * nb_]
            own = [bvs[0].verify_batch(pv_, api[0], rlc_scalars=rs[:nv], want_batch_accum=True).batch_accum,
                   bvs[1].verify_batch(pb, api[1], rlc_scalars=rs[nv:], want_batch_accum=True).batch_accum]
            t0 = 1
            for r in rs[nv:]:
                t0 = t0 * r % bn.R
            for off in (0, 64):
                want = bn.g1_add(bn.g1_mul(_dec(own[0][off: off + 64]), t0), _dec(own[1][off: off + 64]))
                assert _dec(res.batch_accum[off: off + 64]) == want
            j = rng.randrange(nb_)
            bad = list(pb)
            bad[j], expect = sim.corrupt(pb[j], B.vk, "point_swap", rng, B.mo)
            res = mx.verify_batch([pv_, bad], api, rlc_scalars=rs)
            assert not res.verdict and res.status[0] == [0] * nv and res.status[1] == [expect if i == j else 0 for i in range(nb_)]
    finally:
        [bv.close() for bv in bvs]
