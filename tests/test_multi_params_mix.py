"""Multi-params mixes (include/h2v.h "multi-params mixes"): proofs under several KZG params folded into one MSM and one
pairing check, prod_p e(L_p, [s_p]g2_p) e(R_p, -g2_p) = 1.  The checker is the CPU oracle: the per-proof orc.verify_proof
results under each member's own params, orc.rlc_coefficients over the member-major concatenation, per-class sums, and
bn.pairing_check over all 2K pairs (mp_oracle below)."""
import ctypes
import functools
import hashlib
import os
import random

import pytest

import agg_oracle as ao
import bn254 as bn
import formats as F
import prover_sim as sim
import verifier as orc
from test_mixed_batch import Circ, S
from workloads import enc_point

HERE = os.path.dirname(os.path.abspath(__file__))
T2 = 7  # g2 = [T2] G2 for the class that differs from the standard params only in g2


# ---------------------------------------------------------------- the oracle of a multi-params mix
def g2_params(k, s, t):
    """params whose g2 is [t] G2 (s_g2 = [s t] G2): proofs simulated with trapdoor s verify under them"""
    return F.ParamsKZG(k, bn.G1_GEN, bn.g2_mul(bn.G2_GEN, t), bn.g2_mul(bn.G2_GEN, s * t % bn.R))


def params_key(p):
    return (p.g, p.g2, p.s_g2)


def classes_of(params_list):
    """params class of each member: equal (g, g2, s_g2), numbered by first appearance"""
    seen, out = {}, []
    for p in params_list:
        out.append(seen.setdefault(params_key(p), len(seen)))
    return out


def class_folds(results, member_of, class_of, n_classes, rs):
    """per class: (L_p, R_p) = sum over its proofs of c_j (L_j, R_j), c_j over the whole concatenation (orc.accumulate's sums)"""
    folds = [[None, None] for _ in range(n_classes)]
    for res, m, c in zip(results, member_of, orc.rlc_coefficients(rs)):
        f = folds[class_of[m]]
        f[0] = bn.g1_add(f[0], bn.g1_mul(res.L, c))
        f[1] = bn.g1_add(f[1], bn.g1_mul(res.R, c))
    return folds


def multi_check(class_params, folds):
    """the one pairing check over all 2K pairs"""
    pairs = []
    for p, (L, R_) in zip(class_params, folds):
        pairs += [(L, p.s_g2), (R_, bn.g2_neg(p.g2))]
    return bn.pairing_check(pairs)


def mp_oracle(params_list, want):
    """want[m] = member m's oracle results; returns (class_of, per-class folds as a function of rs, verdict function)"""
    class_of = classes_of(params_list)
    reps = {}
    for m, c in enumerate(class_of):
        reps.setdefault(c, params_list[m])
    class_params = [reps[c] for c in range(len(reps))]
    flat = [w for ws in want for w in ws]
    member_of = [m for m, ws in enumerate(want) for _ in ws]

    def run(rs):
        folds = class_folds(flat, member_of, class_of, len(class_params), rs)
        return folds, multi_check(class_params, folds) and all(w.status == orc.OK for w in flat)
    return class_of, run


# ---------------------------------------------------------------- CPU: mapping, pair budget, oracle helper
@functools.lru_cache(maxsize=None)
def _lib():
    return ctypes.CDLL(os.path.join(HERE, "hostlib", "libmixparams.so"))


def _class_map(shapes, set_of, sets, c0, c1):
    lib = _lib()
    flat = (ctypes.c_uint32 * (4 * len(shapes)))(*[v for sh in shapes for v in sh])
    so = (ctypes.c_uint32 * len(shapes))(*set_of) if set_of is not None else None
    cap = sum(n * (P + M) + Sh for n, P, M, Sh in shapes if n)
    out = (ctypes.c_uint32 * max(1, 5 * cap))()
    nb = ctypes.c_uint32(0)
    lib.x_class_map.restype = ctypes.c_longlong
    total = lib.x_class_map(len(shapes), flat, so, sets, c0, c1, out, ctypes.c_ulonglong(cap), ctypes.byref(nb))
    assert total == cap
    return nb.value, [tuple(out[5 * t: 5 * t + 5]) for t in range(total)]


def test_class_mapping_is_a_bijection_onto_disjoint_bucket_sets(built):
    rng = random.Random("mparams-map")
    for _ in range(60):
        members = rng.randint(1, 24)
        shapes = [(rng.choice([0, 1, 2, 5, 9]), rng.randint(1, 12), rng.randint(0, 3), rng.randint(1, 6)) for _ in range(members)]
        if not any(n for n, *_ in shapes):
            continue
        cls = [rng.randrange(rng.randint(1, 8)) for _ in range(members)]
        active = sorted({c for c, (n, *_r) in zip(cls, shapes) if n})
        set_of = [active.index(c) if c in active else 0xFFFFFFFF for c in cls]  # dense bucket sets, as mix_verify_impl numbers them
        c0, c1 = rng.randint(4, 15), rng.randint(4, 15)
        nb, rows = _class_map(shapes, set_of, len(active), c0, c1)
        assert nb == -(-255 // c0) * (1 << (c0 - 1)) + -(-255 // c1) * (1 << (c1 - 1))
        seen_sets = {}
        for seg, m, st, lo, hi in rows:
            assert st == set_of[m] and st < len(active)
            assert st * nb <= lo <= hi < (st + 1) * nb  # every bucket of the term inside its class's set
            seen_sets.setdefault(st, set()).add(cls[m])
        # class <-> bucket set is a bijection: each set holds exactly one class, each class with proofs has one set
        assert sorted(seen_sets) == list(range(len(active)))
        assert all(len(v) == 1 for v in seen_sets.values()) and sorted(c for v in seen_sets.values() for c in v) == active


def test_single_class_maps_as_the_one_segment_table(built):
    from test_mixed_batch import _map
    rng = random.Random("mparams-one")
    for shapes in ([(4, 12, 2, 5)], [(0, 3, 1, 2), (7, 5, 2, 3), (3, 4, 1, 2)], [(rng.randint(0, 6), rng.randint(1, 9), rng.randint(0, 3), rng.randint(1, 5)) for _ in range(20)]):
        if not any(n for n, *_ in shapes):
            continue
        for set_of in (None, [0] * len(shapes)):
            nb, rows = _class_map(shapes, set_of, 1, 9, 7)
            _nseg, plain = _map(shapes)
            assert [(s, m) for s, m, *_r in rows] == [(s, m) for s, m, *_r in plain]
            for (_s, _m, st, lo, hi), (_s2, _m2, kind, _j, _i, ch) in zip(rows, plain):
                W, B = (-(-255 // 9), 256) if ch == 0 else (-(-255 // 7), 64)
                base = 0 if ch == 0 else -(-255 // 9) * 256
                assert st == 0 and (lo, hi) == (base, base + W * B - 1)  # the single-VK bucket range of the term's channel


def _run(sets, W0, W1, run0):
    return _lib().x_mix_line_run(sets, W0, W1, run0)


@pytest.mark.parametrize("run0", [1, 2])
def test_pair_budget(built, run0):
    """every single-batch window geometry (c = 4 .. 15 per channel, W = ceil(255 / c)), 1 .. 8 classes"""
    for c0 in range(4, 16):
        for c1 in range(4, 16):
            W0, W1 = -(-255 // c0), -(-255 // c1)
            pairs = lambda K, r: K * (-(-W0 // r) + -(-W1 // r))
            assert _run(1, W0, W1, run0) == run0  # one class: today's run
            for K in range(1, 9):
                r = _run(K, W0, W1, run0)
                assert r >= run0 and pairs(K, r) <= 128
                assert r == run0 or pairs(K, r - 1) > 128  # minimal


def _pts(rng, s, valid=True):
    """(L, R) of a proof under trapdoor s: e(L, [s t] G2) e(R, -[t] G2) = 1 iff R = s L"""
    a = rng.randrange(1, bn.R)
    return bn.g1_mul_gen(a), bn.g1_mul_gen(a * s % bn.R if valid else (a * s + 1) % bn.R), a


class _Res:
    def __init__(self, L, R_):
        self.L, self.R, self.status = L, R_, orc.OK


def test_oracle_helper_against_direct_evaluation():
    """the multi-class check equals the exponent identity sum_p t_p (s_p l_p - r_p) = 0, and, on accepting inputs, the
    product of the per-class two-pair checks; classes that differ only in g2 are distinct classes"""
    rng = random.Random("mparams-oracle")
    params = [sim.make_params(4, S), sim.make_params(4, S + 1), g2_params(4, S, T2), sim.make_params(4, S + 1)]
    ts = [1, 1, T2, 1]
    ss = [S, S + 1, S, S + 1]
    assert classes_of(params) == [0, 1, 2, 1]
    for case in range(6):
        valid = [[True, True], [True], [True, True], [True]]
        if case >= 2:
            m = case % 4
            valid[m][0] = False
        pts = [[_pts(rng, ss[m], v) for v in vs] for m, vs in enumerate(valid)]
        want = [[_Res(L, R_) for L, R_, _a in ps] for ps in pts]
        class_of, run = mp_oracle(params, want)
        rs = [rng.randrange(1, bn.R) for _ in range(6)]
        folds, ok = run(rs)
        cs = orc.rlc_coefficients(rs)
        expo = [0, 0, 0]
        j = 0
        for m, ps in enumerate(pts):
            for (_L, _R, a), v in zip(ps, valid[m]):
                r_exp = a * ss[m] if v else a * ss[m] + 1
                expo[class_of[m]] += ts[m] * (ss[m] * a - r_exp) * cs[j]
                j += 1
        assert ok == all(e % bn.R == 0 for e in expo) == (case < 2)
        if case < 2:
            reps = [params[0], params[1], params[2]]
            assert all(bn.pairing_check([(L, p.s_g2), (R_, bn.g2_neg(p.g2))]) for p, (L, R_) in zip(reps, folds))
    # differ only in g2: a proof of trapdoor S checked as class 0 (g2) passes, and its pair under class 2 also passes;
    # mixing the folds (class 0's sums against class 2's G2 arguments) fails unless t = 1
    L, R_, _a = _pts(rng, S)
    assert multi_check([params[2]], [[L, R_]]) and multi_check([params[0]], [[L, R_]])
    assert not multi_check([params[0], params[2]], [[L, R_], [bn.g1_mul(L, 2), R_]])


# ---------------------------------------------------------------- GPU
class PCirc(Circ):
    """a circuit of the fixture under its own params: trapdoor s, and g2 = [t] G2 when t != 1"""

    def __init__(self, shape, k, mo, hk, m=1, vk_seed=0, s=S, t=1):
        super().__init__(shape, k, mo, hk, m=m, vk_seed=vk_seed, s=s)
        if t != 1:
            self.params = g2_params(k, s, t)


@functools.lru_cache(maxsize=None)
def pcircuits():
    """A: class S (vm k=8 SHPLONK/Blake2b), B: class S+1 (sh k=8 GWC/Keccak), C: class S+2 (3 instances), D: S with
    g2 = [T2] G2 (vm k=10 GWC/Blake2b), E: a second member of class S+1 (vm k=8, another VK), F: class S+2 (takes no proofs)"""
    return (PCirc("vm", 8, "shplonk", "blake2b"), PCirc("sh", 8, "gwc", "keccak", s=S + 1), PCirc("mix", 6, "shplonk", "blake2b", m=3, s=S + 2),
            PCirc("vm", 10, "gwc", "blake2b", t=T2), PCirc("vm", 8, "shplonk", "blake2b", vk_seed=1, s=S + 1),
            PCirc("sh", 8, "gwc", "keccak", s=S + 2))


def _check(mx, circs, insts, proofs, rs, want=None, **kw):
    """multi-params mix against the oracle: statuses, per-class batch_accum and verdict, bit for bit"""
    res = mx.verify_batch(proofs, [c.api(i) for c, i in zip(circs, insts)], rlc_scalars=rs, want_batch_accum=True, **kw)
    if want is None:
        want = [c.oracle(i, p) for c, i, p in zip(circs, insts, proofs)]
    class_of, run = mp_oracle([c.params for c in circs], want)
    assert mx.params_classes == class_of
    folds, ok = run(rs)
    assert res.status == [[w.status for w in ws] for ws in want]
    active = {class_of[m] for m, ws in enumerate(want) if ws}
    assert res.batch_accum == b"".join(enc_point(L) + enc_point(R_) if c in active else bytes(128) for c, (L, R_) in enumerate(folds))
    assert res.verdict == ok
    return res, want


def _bvs(pkg, circs):
    return [c.bv(pkg) for c in circs]


@pytest.mark.gpu
def test_multi_params_parity_against_oracle(pkg):
    A, B, C, D, E, Fc = pcircuits()
    circs = (A, B, C, D, E, Fc)
    rng = random.Random("mparams-parity")
    ia = [sim.random_instances(A.vk, rng, 3 + 5 * t) for t in range(3)]  # ragged public inputs
    pa = [sim.simulate_proof(A.params, A.vk, A.dl, S, i, rng) for i in ia]
    ib, pb = B.proofs(rng, 3)
    ic, pc = C.proofs(rng, 2)
    id_, pd = D.proofs(rng, 2)
    ie, pe = E.proofs(rng, 2)
    bvs = _bvs(pkg, circs)
    try:
        with pkg.MixedBatchVerifier(bvs, multi_params=True) as mx:
            assert mx.params_classes == [0, 1, 2, 3, 1, 2] and mx.n_classes == 4
            n = 12
            rs = [rng.randrange(1, bn.R) for _ in range(n)]
            res, _ = _check(mx, circs, [ia, ib, ic, id_, ie, []], [pa, pb, pc, pd, pe, []], rs)
            assert res.verdict and res.status[5] == []
            bad = list(pd)
            bad[1], _ = sim.corrupt(pd[1], D.vk, "eval_flip", rng, D.mo)
            res, _ = _check(mx, circs, [ia, ib, ic, id_, ie, []], [pa, pb, pc, bad, pe, []], rs)
            assert not res.verdict and res.status[3][1] != orc.OK
            # a class without proofs in the call: all-zero bytes
            res, _ = _check(mx, circs, [ia, [], ic, id_, [], []], [pa, [], pc, pd, [], []], rs[:7])
            assert res.verdict and res.batch_accum[128:256] == bytes(128)
    finally:
        [bv.close() for bv in bvs]


@pytest.mark.gpu
def test_one_class_equals_the_plain_mix(pkg):
    A = pcircuits()[0]
    A2 = PCirc("sh", 8, "gwc", "keccak")
    A3 = PCirc("mix", 6, "shplonk", "blake2b", m=3)
    circs = (A, A2, A3)
    rng = random.Random("mparams-one-class")
    insts, proofs = zip(*[c.proofs(rng, n) for c, n in zip(circs, (4, 3, 2))])
    proofs = [list(p) for p in proofs]
    api = [c.api(i) for c, i in zip(circs, insts)]
    bvs = _bvs(pkg, circs)
    try:
        with pkg.MixedBatchVerifier(bvs) as plain, pkg.MixedBatchVerifier(bvs, multi_params=True) as multi:
            assert multi.params_classes == [0, 0, 0] and plain.params_classes == [0, 0, 0]
            for corrupt in (False, True):
                if corrupt:
                    proofs[1][1], _ = sim.corrupt(proofs[1][1], A2.vk, "point_swap", rng, A2.mo)
                rs = [rng.randrange(1, bn.R) for _ in range(9)]
                a = plain.verify_batch(proofs, api, rlc_scalars=rs, want_batch_accum=True)
                b = multi.verify_batch(proofs, api, rlc_scalars=rs, want_batch_accum=True)
                assert a == b and a.verdict == (not corrupt)
                _check(multi, circs, insts, proofs, rs)
    finally:
        [bv.close() for bv in bvs]


@pytest.mark.gpu
def test_each_class_meets_its_own_lines(pkg):
    """a proof of trapdoor S+1 submitted to a class-S member (same VK) is flagged, and only it; so is a whole proof list
    swapped between the classes.  Both would pass if a class's terms met the other class's lines."""
    X0 = PCirc("vm", 8, "shplonk", "blake2b")
    X1 = PCirc("vm", 8, "shplonk", "blake2b", s=S + 1)
    circs = (X0, X1)
    rng = random.Random("mparams-lines")
    i0, p0 = X0.proofs(rng, 4)
    i1, p1 = X1.proofs(rng, 3)
    bvs = _bvs(pkg, circs)
    try:
        with pkg.MixedBatchVerifier(bvs, multi_params=True) as mx:
            q0, j0 = list(p0), list(i0)
            j0[2], q0[2] = i1[0], p1[0]  # made under S+1, submitted under S
            res, want = _check(mx, circs, [j0, i1], [q0, p1], [rng.randrange(1, bn.R) for _ in range(7)])
            assert want[0][2].status != orc.OK and not res.verdict
            assert res.status == [[0, 0, want[0][2].status, 0], [0, 0, 0]]
            res, want = _check(mx, circs, [i1, i0[:3]], [p1, p0[:3]], [rng.randrange(1, bn.R) for _ in range(6)])  # lists swapped
            assert not res.verdict and all(s != orc.OK for st in res.status for s in st)
            assert res.status == [[w.status for w in ws] for ws in want]
    finally:
        [bv.close() for bv in bvs]


@pytest.mark.gpu
def test_rejections_spread_over_the_classes(pkg):
    A, B, C, D, E, _F = pcircuits()
    circs = (A, B, C, D, E)
    rng = random.Random("mparams-reject")
    insts, proofs = zip(*[c.proofs(rng, n) for c, n in zip(circs, (3, 3, 2, 2, 2))])
    proofs = [list(p) for p in proofs]
    slots = [(0, 0), (0, 2), (1, 0), (1, 1), (2, 1), (3, 0), (3, 1), (4, 0), (4, 1)]
    for kind, (m, j) in zip(sim.CORRUPTIONS, slots):
        proofs[m][j], _ = sim.corrupt(proofs[m][j], circs[m].vk, kind, rng, circs[m].mo, circs[m].m)
    bvs = _bvs(pkg, circs)
    try:
        with pkg.MixedBatchVerifier(bvs, multi_params=True) as mx:
            res, _ = _check(mx, circs, list(insts), proofs, [rng.randrange(1, bn.R) for _ in range(12)])
            assert not res.verdict
            flagged = {(m, j) for m, st in enumerate(res.status) for j, v in enumerate(st) if v}
            assert flagged == set(slots[:len(sim.CORRUPTIONS)])
    finally:
        [bv.close() for bv in bvs]


@pytest.mark.gpu
def test_aggregation_member_in_a_non_lead_class(pkg):
    from test_instance_accumulator import Spec, _place
    A = pcircuits()[0]
    G = PCirc("vm", 8, "shplonk", "blake2b", s=S + 1)
    spec = Spec(3, 88, [(0, 2 + i) for i in range(12)])
    rng = random.Random("mparams-agg")
    ia, pa = A.proofs(rng, 2)
    ig, pg = [], []
    for j in range(3):
        P = bn.g1_mul_gen(rng.randrange(1, bn.R))
        lhs = bn.g1_mul(P, S if j == 1 else S + 1)  # proof 1 carries a pair valid only under the lead's s
        i = _place(G.instances(rng, 20), spec, lhs, P)
        ig.append(i)
        pg.append(sim.simulate_proof(G.params, G.vk, G.dl, G.s, i, rng, G.mo, G.hk))
    ba = A.bv(pkg)
    bg = pkg.BatchVerifier(pkg.ParamsKZG.from_bytes(G.params.to_bytes()), pkg.VerifyingKey.from_bytes(G.vk.to_bytes(F.RAW_BYTES), F.RAW_BYTES),
                           G.mo, G.hk, device=0, accumulator=spec.api(pkg))
    try:
        with pkg.MixedBatchVerifier([ba, bg], multi_params=True) as mx:
            rho = rng.randrange(1, bn.R)
            want = [A.oracle(ia, pa), [ao.verify_proof(G.params, G.vk, i, p, G.mo, G.hk, accumulator=spec, rho=rho) for i, p in zip(ig, pg)]]
            assert [w.status for w in want[1]] == [orc.OK, orc.CONSTRAINT_SYSTEM_FAILURE, orc.OK]
            res, _ = _check(mx, (A, G), [ia, ig], [pa, pg], [rng.randrange(1, bn.R) for _ in range(5)], want=want, agg_scalar=rho)
            assert not res.verdict and res.status == [[0, 0], [0, orc.CONSTRAINT_SYSTEM_FAILURE, 0]]
            want = [want[0], [want[1][0], want[1][2]]]
            res, _ = _check(mx, (A, G), [ia, [ig[0], ig[2]]], [pa, [pg[0], pg[2]]], [rng.randrange(1, bn.R) for _ in range(4)], want=want, agg_scalar=rho)
            assert res.verdict
    finally:
        ba.close()
        bg.close()


@pytest.mark.gpu
def test_limits_eight_classes_and_numbering(pkg):
    circs = [PCirc("vm", 8, "shplonk", "blake2b", s=S + d) for d in range(8)]
    rng = random.Random("mparams-limits")
    insts, proofs = zip(*[c.proofs(rng, 1 + (d % 2)) for d, c in enumerate(circs)])
    bvs = _bvs(pkg, circs)
    ninth = PCirc("vm", 8, "shplonk", "blake2b", s=S + 8).bv(pkg)
    try:
        with pkg.MixedBatchVerifier(bvs, multi_params=True) as mx:
            assert mx.params_classes == list(range(8))
            n = sum(len(p) for p in proofs)
            res, _ = _check(mx, circs, list(insts), list(proofs), [rng.randrange(1, bn.R) for _ in range(n)])
            assert res.verdict
        with pytest.raises(pkg.BackendError, match="1 .. 8 params classes"):
            pkg.MixedBatchVerifier(bvs + [ninth], multi_params=True)
        with pkg.MixedBatchVerifier([bvs[3], bvs[0], bvs[4]], multi_params=True) as mx:
            assert mx.params_classes == [0, 1, 2]
        A, B = pcircuits()[0], pcircuits()[4]
        b_a, b_b, b_s = A.bv(pkg), B.bv(pkg), PCirc("sh", 8, "gwc", "keccak").bv(pkg)  # classes S, S+1, S
        try:
            with pkg.MixedBatchVerifier([b_b, b_a, b_s], multi_params=True) as mx:
                assert mx.params_classes == [0, 1, 1] and mx.n_classes == 2
            with pytest.raises(pkg.BackendError, match="differ"):
                pkg.MixedBatchVerifier([b_a, b_b])
        finally:
            [b.close() for b in (b_a, b_b, b_s)]
    finally:
        [bv.close() for bv in bvs]
        ninth.close()


@pytest.mark.gpu
def test_graphs_and_line_caches(pkg):
    A, B, C, D, _E, _F = pcircuits()
    A2 = PCirc("sh", 8, "gwc", "keccak")  # class S: a plain mix with the same lead
    circs = (A, B, C, D)
    rng = random.Random("mparams-graphs")
    insts, proofs = zip(*[c.proofs(rng, n) for c, n in zip(circs, (3, 2, 2, 2))])
    api = [c.api(i) for c, i in zip(circs, insts)]
    i2, p2 = A2.proofs(rng, 2)
    rs = [rng.randrange(1, bn.R) for _ in range(9)]
    bvs = _bvs(pkg, circs)
    b2 = A2.bv(pkg)
    try:
        with pkg.MixedBatchVerifier(bvs, multi_params=True) as mx, pkg.MixedBatchVerifier([bvs[0], b2]) as plain:
            a = mx.verify_batch(proofs, api, rlc_scalars=rs, want_batch_accum=True)
            p = plain.verify_batch([proofs[0], p2], [api[0], A2.api(i2)], rlc_scalars=rs[:5], want_batch_accum=True)
            assert a.verdict and p.verdict
            st = mx.cache_stats()
            for _ in range(2):  # alternate: neither rebuilds its lines, neither recaptures
                assert mx.verify_batch(proofs, api, rlc_scalars=rs, want_batch_accum=True) == a
                assert plain.verify_batch([proofs[0], p2], [api[0], A2.api(i2)], rlc_scalars=rs[:5], want_batch_accum=True) == p
            assert mx.cache_stats() == st
            bad = [list(q) for q in proofs]
            bad[2][1], _ = sim.corrupt(bad[2][1], C.vk, "eval_flip", rng, C.mo, C.m)
            g = mx.verify_batch(bad, api, rlc_scalars=rs, want_batch_accum=True)
            bvs[0].set_graphs(False)
            d = mx.verify_batch(bad, api, rlc_scalars=rs, want_batch_accum=True)
            assert d == g and not d.verdict and d.status[2][1] == orc.CONSTRAINT_SYSTEM_FAILURE
            assert mx.verify_batch(proofs, api, rlc_scalars=rs, want_batch_accum=True) == a
            t = bvs[0].timings()
            assert t["rlc_msm"] > 0 and t["pairing"] > 0
    finally:
        [bv.close() for bv in bvs]
        b2.close()


def _expand(tag, material, n):
    """r_i of the seed / key expansion (stages.cuh rlc_scalar_from_seed / _from_key)"""
    return [int.from_bytes(hashlib.blake2b(tag + material + i.to_bytes(8, "little"), digest_size=64, person=b"Halo2-Transcript").digest(),
                           "little") % bn.R for i in range(n)]


@pytest.mark.gpu
def test_fold_randomness_sources(pkg):
    A, B, _C, D, _E, _F = pcircuits()
    circs = (A, B, D)
    rng = random.Random("mparams-rand")
    insts, proofs = zip(*[c.proofs(rng, n) for c, n in zip(circs, (3, 2, 2))])
    api = [c.api(i) for c, i in zip(circs, insts)]
    bvs = _bvs(pkg, circs)
    try:
        with pkg.MixedBatchVerifier(bvs, multi_params=True) as mx:
            seed = 0x5EED
            a = mx.verify_batch(proofs, api, seed=seed, want_batch_accum=True)
            assert bvs[0].rlc_source() == "seed"
            b = mx.verify_batch(proofs, api, rlc_scalars=_expand(b"h2v-rlc", seed.to_bytes(8, "little"), 7), want_batch_accum=True)
            assert a == b and a.verdict and len(a.batch_accum) == 3 * 128
            key = bytes(rng.getrandbits(8) for _ in range(32))
            c = mx.verify_batch(proofs, api, key=key, want_batch_accum=True)
            d = mx.verify_batch(proofs, api, rlc_scalars=_expand(b"h2v-rlk", key, 7), want_batch_accum=True)
            assert c == d and c.verdict and c.batch_accum != a.batch_accum
            e = mx.verify_batch(proofs, api, want_batch_accum=True)  # OS entropy
            f = mx.verify_batch(proofs, api, want_batch_accum=True)
            assert e.verdict and f.verdict and e.batch_accum != f.batch_accum and bvs[2].rlc_source() == "key"
        errs = pkg.verify_proofs_mixed([(pkg.ParamsKZG.from_bytes(c.params.to_bytes()), pkg.VerifyingKey.from_bytes(c.vk.to_bytes(F.RAW_BYTES)),
                                         p, a_, c.mo, "keccak256" if c.hk == "keccak" else c.hk) for c, p, a_ in zip(circs, proofs, api)],
                                       multi_params=True)
        assert errs == [[None] * 3, [None] * 2, [None] * 2]
    finally:
        [bv.close() for bv in bvs]
