"""Grouped mixed batches (include/h2v.h "grouped mixed batches"): independent mixed batches in one launch set, each with its
own fold, pairing check and verdict.  Every group is checked against h2v_mix_verify on that group alone and against the
oracle's AccumulatorStrategy over the group's proofs."""
import ctypes
import functools
import os
import random

import pytest

import bn254 as bn
import prover_sim as sim
import verifier as orc
from test_mixed_batch import Circ, _expand, circuits
from test_multi_params_mix import mp_oracle, pcircuits
from workloads import enc_point

HERE = os.path.dirname(os.path.abspath(__file__))


# ---------------------------------------------------------------- CPU: grouped segment table and the ragged scan (csrc/mix.cuh)
@functools.lru_cache(maxsize=None)
def _lib():
    lib = ctypes.CDLL(os.path.join(HERE, "hostlib", "libmixgroups.so"))
    lib.x_groups_map.restype = ctypes.c_longlong
    lib.x_groups_vs_layout.restype = ctypes.c_longlong
    return lib


def _u32(v):
    return (ctypes.c_uint32 * max(1, len(v)))(*v)


def _enumerate(counts, shapes, set_of, sets):
    """the terms of a grouped batch in term-id order, written out: (group, member, kind, proof in the member's arrays, index,
    bucket set, point offset)"""
    G, M = len(counts), len(shapes)
    total = [sum(counts[q][m] for q in range(G)) for m in range(M)]
    out = []
    for q in range(G):
        for m, (P, Mo, Sh) in enumerate(shapes):
            n, j0, st = counts[q][m], sum(counts[p][m] for p in range(q)), total[m]
            bset = q * sets + (set_of[m] if st else 0)
            out += [(q, m, 0, j0 + j, i, bset, i * st + j0 + j) for i in range(P) for j in range(n)]
            out += [(q, m, 1, j0 + j, i, bset, (P - Mo + i) * st + j0 + j) for i in range(Mo) for j in range(n)]
            if st:
                out += [(q, m, 2, 0, i, bset, i) for i in range(Sh)]
    return out


def _gmap(counts, shapes, set_of, sets):
    G, M = len(counts), len(shapes)
    cap = len(_enumerate(counts, shapes, set_of, sets))
    out = (ctypes.c_uint32 * max(1, 7 * cap))()
    flat = [counts[q][m] for q in range(G) for m in range(M)]
    total = _lib().x_groups_map(G, M, _u32(flat), _u32([v for sh in shapes for v in sh]), _u32(set_of), sets, out, ctypes.c_ulonglong(cap))
    assert total == cap
    return [tuple(out[7 * t: 7 * t + 7]) for t in range(total)]


def test_grouped_mapping_is_a_bijection_onto_the_enumeration(built):
    rng = random.Random("mix-groups-map")
    cases = [([[1, 0], [0, 3]], [(5, 2, 3), (4, 1, 2)], [0, 0], 1),  # every member absent from one group
             ([[0, 2, 0], [1, 0, 0], [0, 0, 0]], [(3, 1, 2), (2, 2, 1), (6, 0, 4)], [0, 1, 0], 2)]  # member 2 in no group
    for _ in range(40):
        G, M = rng.randint(1, 9), rng.randint(1, 7)
        counts = [[rng.choice([0, 0, 1, 2, 5, 13]) for _ in range(M)] for _ in range(G)]
        counts[rng.randrange(G)] = [0] * M
        counts[rng.randrange(G)][rng.randrange(M)] = 1
        only = rng.randrange(M)  # a member present in one group only
        for q in range(G):
            counts[q][only] = 0
        counts[rng.randrange(G)][only] = rng.randint(1, 4)
        sets = rng.randint(1, 3)
        shapes = []
        for _m in range(M):
            P = rng.randint(1, 12)
            shapes.append((P, rng.randint(0, min(3, P)), rng.randint(1, 6)))  # the multi-open points are proof points
        cases.append((counts, shapes, [rng.randrange(sets) for _ in range(M)], sets))
    for counts, shapes, set_of, sets in cases:
        got = _gmap(counts, shapes, set_of, sets)
        want = _enumerate(counts, shapes, set_of, sets)
        assert got == want  # the same terms in the same order: every (group, member, kind, proof, index) exactly once
        assert all(b == q * sets + set_of[m] for q, m, _k, _j, _i, b, _p in got)  # bucket set q * S + class


def test_one_group_maps_as_the_mix_layout(built):
    rng = random.Random("mix-groups-one")
    tables = [[(3, 5, 2, 3), (0, 4, 1, 2), (7, 2, 2, 1)], [(1, 1, 0, 1)]]
    for _ in range(30):
        tables.append([(rng.choice([0, 1, 2, 9]), P, rng.randint(0, min(4, P)), rng.randint(1, 8)) for P in [rng.randint(1, 16) for _ in range(rng.randint(1, 64))]])
    for shapes in tables:
        if not any(s[0] for s in shapes):
            continue
        sets = rng.randint(1, 4)
        set_of = [rng.randrange(sets) for _ in shapes]
        assert _lib().x_groups_vs_layout(len(shapes), _u32([v for s in shapes for v in s]), _u32(set_of), sets) == 0


def test_ragged_scan_matches_the_oracle_per_group(built):
    """the host restatement of k_rlc_scan_groups (same chunks, same write phase) gives every proof of group q the coefficient
    orc.rlc_coefficients gives it over group q's r_i alone"""
    rng = random.Random("mix-groups-scan")
    lib = _lib()
    for G, M, threads in [(1, 1, 256), (3, 2, 4), (6, 4, 256), (5, 3, 7), (2, 5, 1)]:
        counts = [[rng.choice([0, 1, 3, 40]) for _ in range(M)] for _ in range(G)]
        for q in range(G):
            if not any(counts[q]):
                counts[q][rng.randrange(M)] = 1
        N = sum(map(sum, counts))
        rs = [rng.randrange(1, bn.R) for _ in range(N)]
        total = [sum(counts[q][m] for q in range(G)) for m in range(M)]
        out = ctypes.create_string_buffer(32 * max(1, sum(total)))
        lib.x_rlc_scan_groups(G, M, _u32([c for row in counts for c in row]), b"".join(r.to_bytes(32, "little") for r in rs), threads, out)
        got = [int.from_bytes(out.raw[32 * i: 32 * i + 32], "little") for i in range(sum(total))]
        want = [[] for _ in range(M)]  # member-major in the members' arrays, group order inside a member
        i = 0
        for q in range(G):
            Nq = sum(counts[q])
            cq = orc.rlc_coefficients(rs[i:i + Nq])
            o = 0
            for m in range(M):
                want[m] += cq[o:o + counts[q][m]]
                o += counts[q][m]
            i += Nq
        assert got == [c for w in want for c in w]


# ---------------------------------------------------------------- GPU
def _slices(groups, M):
    """call-order offsets of every group"""
    offs, o = [], 0
    for _insts, proofs in groups:
        offs.append(o)
        o += sum(len(proofs[m]) for m in range(M))
    return offs, o


def _check_groups(mx, circs, groups, rs, want=None, agg_scalar=None, alone=True):
    """grouped call against the oracle per group (statuses, per-class batch_accum, verdict) and against verify_batch on each
    group alone with its slice of the scalars; groups[q] = (oracle instances per member, proofs per member)"""
    M = len(circs)
    kw = {} if agg_scalar is None else {"agg_scalar": agg_scalar}
    res = mx.verify_groups([(proofs, [c.api(i) for c, i in zip(circs, insts)]) for insts, proofs in groups], rlc_scalars=rs, want_batch_accum=True, **kw)
    offs, N = _slices(groups, M)
    assert len(rs) == N and len(res.group_verdicts) == len(groups)
    for q, (insts, proofs) in enumerate(groups):
        wq = want[q] if want is not None else [c.oracle(i, p) for c, i, p in zip(circs, insts, proofs)]
        rq = rs[offs[q]:offs[q] + sum(len(p) for p in proofs)]
        class_of, run = mp_oracle([c.params for c in circs], wq)
        folds, ok = run(rq)
        assert res.status[q] == [[w.status for w in ws] for ws in wq]
        active = {class_of[m] for m, ws in enumerate(wq) if ws}
        assert res.batch_accum[q] == b"".join(enc_point(L) + enc_point(R_) if c in active else bytes(128) for c, (L, R_) in enumerate(folds))
        assert res.group_verdicts[q] == ok
        if alone:
            one = mx.verify_batch(proofs, [c.api(i) for c, i in zip(circs, insts)], rlc_scalars=rq, want_batch_accum=True, **kw)
            assert one.status == res.status[q] and one.batch_accum == res.batch_accum[q] and one.verdict == res.group_verdicts[q]
    assert res.verdict == all(res.group_verdicts)
    return res


def _groups(rng, circs, layout):
    """layout[q][m] = proofs of member m in group q"""
    return [tuple(map(list, zip(*[c.proofs(rng, n) if n else ([], []) for c, n in zip(circs, row)]))) for row in layout]


@pytest.mark.gpu
def test_one_group_equals_the_mix(pkg):
    rng = random.Random("mix-groups-g1")
    for circs, multi in ((circuits()[:3], False), (pcircuits()[:4], True)):
        bvs = [c.bv(pkg) for c in circs]
        try:
            with pkg.MixedBatchVerifier(bvs, multi_params=multi) as mx:
                groups = _groups(rng, circs, [[3, 2, 0] + [2] * (len(circs) - 3)])
                insts, proofs = groups[0]
                proofs[1][1], _ = sim.corrupt(proofs[1][1], circs[1].vk, "eval_flip", rng, circs[1].mo, circs[1].m)
                rs = [rng.randrange(1, bn.R) for _ in range(sum(map(len, proofs)))]
                res = _check_groups(mx, circs, groups, rs)
                assert not res.verdict and res.status[0][1][1] == orc.CONSTRAINT_SYSTEM_FAILURE
        finally:
            [bv.close() for bv in bvs]


@pytest.mark.gpu
def test_ragged_groups_with_caller_scalars(pkg):
    """G = 5: a one-proof group, members absent from groups, SHPLONK + GWC, Blake2b + Keccak, a 3-instance member"""
    A, B, C, D = circuits()
    circs = (A, B, C, D)
    rng = random.Random("mix-groups-ragged")
    groups = _groups(rng, circs, [[2, 1, 1, 0], [0, 0, 1, 0], [3, 0, 0, 2], [1, 2, 2, 1], [0, 4, 0, 0]])
    N = _slices(groups, 4)[1]
    bvs = [c.bv(pkg) for c in circs]
    try:
        with pkg.MixedBatchVerifier(bvs) as mx:
            res = _check_groups(mx, circs, groups, [rng.randrange(1, bn.R) for _ in range(N)])
            assert res.verdict and res.group_verdicts == [True] * 5
    finally:
        [bv.close() for bv in bvs]


@pytest.mark.gpu
def test_one_member_ragged_groups_equal_its_own_batches(pkg):
    A = circuits()[0]
    rng = random.Random("mix-groups-one-member")
    insts, proofs = A.proofs(rng, 24)
    sizes = (1, 7, 300)
    groups, k = [], 0
    for n in sizes:
        idx = [(k + j) % 24 for j in range(n)]
        groups.append(([[insts[i] for i in idx]], [[proofs[i] for i in idx]]))
        k += n
    rs = [rng.randrange(1, bn.R) for _ in range(sum(sizes))]
    with A.bv(pkg) as bv:
        with pkg.MixedBatchVerifier([bv]) as mx:
            res = mx.verify_groups([(p, [A.api(i[0])]) for i, p in groups], rlc_scalars=rs, want_batch_accum=True)
            assert res.verdict and res.group_verdicts == [True] * 3
            o = 0
            for q, (i, p) in enumerate(groups):
                own = bv.verify_batch(p[0], A.api(i[0]), rlc_scalars=rs[o:o + sizes[q]], want_batch_accum=True)
                assert res.batch_accum[q] == own.batch_accum and res.status[q] == [own.status]
                o += sizes[q]


@pytest.mark.gpu
def test_corrupted_proofs_reject_only_their_groups(pkg):
    A, B, C, _D = circuits()
    circs = (A, B, C)
    rng = random.Random("mix-groups-reject")
    groups = _groups(rng, circs, [[3, 2, 1]] * 6)
    slots = [(1, 0, 0), (1, 0, 2), (1, 1, 1), (1, 2, 0), (3, 0, 1), (3, 1, 0), (3, 1, 1), (3, 2, 0), (3, 0, 2)]
    for kind, (q, m, j) in zip(sim.CORRUPTIONS, slots):
        groups[q][1][m][j], _ = sim.corrupt(groups[q][1][m][j], circs[m].vk, kind, rng, circs[m].mo, circs[m].m)
    N = _slices(groups, 3)[1]
    bvs = [c.bv(pkg) for c in circs]
    try:
        with pkg.MixedBatchVerifier(bvs) as mx:
            res = _check_groups(mx, circs, groups, [rng.randrange(1, bn.R) for _ in range(N)], alone=False)
            assert res.group_verdicts == [q not in (1, 3) for q in range(6)] and not res.verdict
            flagged = {(q, m, j) for q, sq in enumerate(res.status) for m, st in enumerate(sq) for j, v in enumerate(st) if v}
            assert flagged == set(slots)
            # every status is the C oracle's too (the per-proof oracle run above is the Python one)
            import c_oracle
            import formats as F
            cos = [c_oracle.COracle(c.params.to_bytes(), 0, c.vk.to_bytes(F.RAW_BYTES), F.RAW_BYTES) for c in circs]
            for q, (insts, proofs) in enumerate(groups):
                for m, c in enumerate(circs):
                    for j, (i, pr) in enumerate(zip(insts[m], proofs[m])):
                        assert res.status[q][m][j] == cos[m].verify_multi(pr, i, c.mo, c.hk)[0]
            [co.close() for co in cos]
    finally:
        [bv.close() for bv in bvs]


@pytest.mark.gpu
def test_multi_params_with_absent_classes(pkg):
    """class of B/E absent from group 1 (identity set there), class of F absent from every group (no set)"""
    A, B, C, D, E, F_ = pcircuits()
    circs = (A, B, C, D, E, F_)
    rng = random.Random("mix-groups-mparams")
    groups = _groups(rng, circs, [[2, 1, 1, 1, 1, 0], [1, 0, 2, 0, 0, 0], [0, 2, 0, 1, 1, 0]])
    N = _slices(groups, 6)[1]
    bvs = [c.bv(pkg) for c in circs]
    try:
        with pkg.MixedBatchVerifier(bvs, multi_params=True) as mx:
            res = _check_groups(mx, circs, groups, [rng.randrange(1, bn.R) for _ in range(N)])
            assert res.verdict
            groups[2][1][3][0], _ = sim.corrupt(groups[2][1][3][0], D.vk, "eval_flip", rng, D.mo)
            res = _check_groups(mx, circs, groups, [rng.randrange(1, bn.R) for _ in range(N)], alone=False)
            assert res.group_verdicts == [True, True, False]
    finally:
        [bv.close() for bv in bvs]


@pytest.mark.gpu
def test_aggregation_member_rejects_only_its_group(pkg):
    import agg_oracle as ao
    from test_instance_accumulator import Spec, _place
    import formats as F
    A = circuits()[0]
    Gc = Circ("vm", 8, "shplonk", "blake2b", vk_seed=2)
    spec = Spec(3, 88, [(0, 2 + i) for i in range(12)])
    rng = random.Random("mix-groups-agg")
    rho = rng.randrange(1, bn.R)

    def agg(valid):
        P = bn.g1_mul_gen(rng.randrange(1, bn.R))
        i = _place(Gc.instances(rng, 20), spec, bn.g1_mul(P, Gc.s if valid else Gc.s + 1), P)
        return i, sim.simulate_proof(Gc.params, Gc.vk, Gc.dl, Gc.s, i, rng, Gc.mo, Gc.hk)

    ia, pa = A.proofs(rng, 4)
    g_items = [agg(True), agg(True), agg(False), agg(True)]
    groups = [([ia[:2], [g_items[0][0]]], [pa[:2], [g_items[0][1]]]), ([ia[2:], [x[0] for x in g_items[1:3]]], [pa[2:], [x[1] for x in g_items[1:3]]]),
              ([[], [g_items[3][0]]], [[], [g_items[3][1]]])]
    ba = A.bv(pkg)
    bg = pkg.BatchVerifier(pkg.ParamsKZG.from_bytes(Gc.params.to_bytes()), pkg.VerifyingKey.from_bytes(Gc.vk.to_bytes(F.RAW_BYTES), F.RAW_BYTES),
                           Gc.mo, Gc.hk, device=0, accumulator=spec.api(pkg))
    try:
        with pkg.MixedBatchVerifier([ba, bg]) as mx:
            def want_of(gs):
                return [[A.oracle(i[0], p[0]), [ao.verify_proof(Gc.params, Gc.vk, x, y, Gc.mo, Gc.hk, accumulator=spec, rho=rho) for x, y in zip(i[1], p[1])]]
                        for i, p in gs]
            res = _check_groups(mx, (A, Gc), groups, [rng.randrange(1, bn.R) for _ in range(8)], want=want_of(groups), agg_scalar=rho, alone=False)
            assert res.group_verdicts == [True, False, True] and res.status[1][1] == [0, orc.CONSTRAINT_SYSTEM_FAILURE]
            # a malformed accumulator encoding (a limb out of range) in group 0: InvalidInstances there only
            i_bad, _ = agg(True)
            cols = [col for inst in i_bad for col in inst]
            cols[spec.cells[0][0]][spec.cells[0][1]] = 1 << 68
            p_bad = sim.simulate_proof(Gc.params, Gc.vk, Gc.dl, Gc.s, i_bad, rng, Gc.mo, Gc.hk)
            g2 = [([ia[:1], [i_bad]], [pa[:1], [p_bad]]), groups[2]]
            res = _check_groups(mx, (A, Gc), g2, [rng.randrange(1, bn.R) for _ in range(3)], want=want_of(g2), agg_scalar=rho, alone=False)
            assert res.status[0][1] == [orc.INVALID_INSTANCES] and res.group_verdicts == [False, True]
    finally:
        ba.close()
        bg.close()


@pytest.mark.gpu
def test_fold_randomness_sources(pkg):
    A, B, C, _D = circuits()
    circs = (A, B, C)
    rng = random.Random("mix-groups-rand")
    groups = _groups(rng, circs, [[2, 1, 0], [0, 1, 1], [1, 0, 2]])
    api = [(p, [c.api(i) for c, i in zip(circs, ins)]) for ins, p in groups]
    bvs = [c.bv(pkg) for c in circs]
    try:
        with pkg.MixedBatchVerifier(bvs) as mx:
            a = mx.verify_groups(api, seed=0x5EED, want_batch_accum=True)
            b = mx.verify_groups(api, rlc_scalars=_expand(b"h2v-rlc", (0x5EED).to_bytes(8, "little"), 8), want_batch_accum=True)
            assert a == b and a.verdict
            key = bytes(rng.getrandbits(8) for _ in range(32))
            c = mx.verify_groups(api, key=key, want_batch_accum=True)
            d = mx.verify_groups(api, key=key, want_batch_accum=True)
            e = mx.verify_groups(api, rlc_scalars=_expand(b"h2v-rlk", key, 8), want_batch_accum=True)
            assert c == d == e and c.verdict and c.batch_accum != a.batch_accum
            f = mx.verify_groups(api, want_batch_accum=True)  # OS entropy: one fresh key per call
            g = mx.verify_groups(api, want_batch_accum=True)
            assert f.verdict and g.verdict and f.batch_accum != g.batch_accum
    finally:
        [bv.close() for bv in bvs]


@pytest.mark.gpu
def test_graphs_replay_across_splits(pkg):
    A, B, C, _D = circuits()
    circs = (A, B, C)
    rng = random.Random("mix-groups-graph")
    insts, proofs = zip(*[c.proofs(rng, n) for c, n in zip(circs, (6, 4, 3))])

    def split(layout):  # the same member totals (6, 4, 3) over 3 groups
        out, k = [], [0, 0, 0]
        for row in layout:
            out.append((tuple(list(proofs[m][k[m]:k[m] + n]) for m, n in enumerate(row)),
                        [circs[m].api(insts[m][k[m]:k[m] + n]) for m, n in enumerate(row)]))
            k = [k[m] + n for m, n in enumerate(row)]
        return [(list(p), a) for p, a in out]

    rs = [rng.randrange(1, bn.R) for _ in range(13)]
    bvs = [c.bv(pkg) for c in circs]
    try:
        with pkg.MixedBatchVerifier(bvs) as mx:
            s1, s2 = split([[2, 1, 1], [2, 2, 0], [2, 1, 2]]), split([[5, 0, 0], [1, 4, 0], [0, 0, 3]])
            a = mx.verify_groups(s1, rlc_scalars=rs, want_batch_accum=True)
            caps = mx.cache_stats()["graph_captures"]
            b = mx.verify_groups(s2, rlc_scalars=rs, want_batch_accum=True)
            assert mx.cache_stats()["graph_captures"] == caps  # another split, the same totals and G: replay
            assert a.verdict and b.verdict
            bad = [(list(map(list, p)), x) for p, x in s2]
            bad[1][0][1][2], _ = sim.corrupt(bad[1][0][1][2], B.vk, "eval_flip", rng, B.mo)
            g = mx.verify_groups(bad, rlc_scalars=rs, want_batch_accum=True)
            bvs[0].set_graphs(False)
            d = mx.verify_groups(bad, rlc_scalars=rs, want_batch_accum=True)
            assert d == g and d.group_verdicts == [True, False, True] and d.status[1][1][2] == orc.CONSTRAINT_SYSTEM_FAILURE
            assert mx.verify_groups(s2, rlc_scalars=rs, want_batch_accum=True) == b
    finally:
        [bv.close() for bv in bvs]


@pytest.mark.gpu
def test_refusals_leave_the_state_unchanged(pkg):
    A, B, _C, _D = circuits()
    circs = (A, B)
    rng = random.Random("mix-groups-refuse")
    groups = _groups(rng, circs, [[1, 1], [2, 0]])
    api = [(p, [c.api(i) for c, i in zip(circs, ins)]) for ins, p in groups]
    bvs = [c.bv(pkg) for c in circs]
    lib = bvs[0].lib
    try:
        with pkg.MixedBatchVerifier(bvs) as mx:
            key = bytes(range(32))
            want = mx.verify_groups(api, key=key, want_batch_accum=True)
            st, gv, verdict = (ctypes.c_uint8 * 8)(), (ctypes.c_uint8 * 8)(), ctypes.c_int(0)
            off = (ctypes.c_uint64 * 8)()

            def call(groups_, counts, **kw):
                args = dict(proofs=b"\0", poff=off, inst=b"\0", ioff=off, rlc=None, status=st, verdict=ctypes.byref(verdict))
                args.update(kw)
                return lib.h2v_mix_verify_groups(mx._mx, groups_, counts, args["proofs"], args["poff"], args["inst"], args["ioff"], args["rlc"], 0,
                                                 args["status"], gv, None, args["verdict"])

            refusals = [
                (lambda: call(0, mx._u32([1, 0])), "1 .. 1024 groups"),
                (lambda: call(1025, mx._u32([1, 0] * 1025)), "1 .. 1024 groups"),
                (lambda: call(2, mx._u32([1, 0, 0, 0])), "group 1 has no proofs"),
                (lambda: call(1, None), "null argument"),
                (lambda: call(1, mx._u32([1, 0]), poff=None), "null argument"),
                (lambda: call(1, mx._u32([1, 0]), ioff=None), "null argument"),
                (lambda: call(1, mx._u32([1, 0]), status=None), "null argument"),
                (lambda: call(1, mx._u32([1, 0]), verdict=None), "null argument"),
                (lambda: call(1, mx._u32([0, 0])), "between 1 and 2\\^32 - 1"),
                (lambda: call(2, mx._u32([0xFFFFFFFF, 0, 1, 0])), "between 1 and 2\\^32 - 1"),
                (lambda: call(1, mx._u32([1, 0]), rlc=bytes(32)), "canonical and non-zero"),
                (lambda: call(1, mx._u32([1, 0]), rlc=b"\xff" * 32), "canonical and non-zero"),
            ]
            for fn, msg in refusals:
                mx._check(lib.h2v_mix_set_rlc_key(mx._mx, key))
                with pytest.raises(pkg.BackendError, match=msg):
                    mx._check(fn())
                assert mx.verify_groups(api, want_batch_accum=True) == want  # the key was not consumed
            # options that make the call refuse: a member's fold groups or shard hint, the mix's shard hint
            for set_opt, msg in ((lambda: bvs[1]._check(lib.h2v_batch_set_fold_groups(bvs[1]._ctx, 2)), "fold-group or shard-hint"),
                                 (lambda: mx._check(lib.h2v_mix_set_shard_hint(mx._mx, 8)), "shard hint is pending")):
                set_opt()
                mx._check(lib.h2v_mix_set_rlc_key(mx._mx, key))
                with pytest.raises(pkg.BackendError, match=msg):
                    mx.verify_groups(api, want_batch_accum=True)
                lib.h2v_batch_set_fold_groups(bvs[1]._ctx, 0)
                lib.h2v_mix_set_shard_hint(mx._mx, 0)
                assert mx.verify_groups(api, want_batch_accum=True) == want
    finally:
        [bv.close() for bv in bvs]
