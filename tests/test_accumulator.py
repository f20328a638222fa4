"""Persistent accumulators (include/h2v.h "persistent accumulators"): batches absorbed across calls into one device-resident
DualMSM, one pairing check at finalize.  The checker is the CPU oracle: orc.accumulate over the concatenation of the absorbed
proofs, in absorb order, IS the reference's AccumulatorStrategy fed the same proofs."""
import ctypes
import functools
import os
import random

import pytest

import bn254 as bn
import prover_sim as sim
import verifier as orc
from test_mixed_batch import Circ, S, _dec, _expand, circuits
from workloads import enc_point

HERE = os.path.dirname(os.path.abspath(__file__))


# ---------------------------------------------------------------- CPU: the absorb arithmetic (csrc/acc.cuh)
@functools.lru_cache(maxsize=None)
def _acclib():
    return ctypes.CDLL(os.path.join(HERE, "hostlib", "libacc.so"))


def _limbs(v, n=8):
    return (ctypes.c_uint32 * n)(*[(v >> (32 * i)) & 0xFFFFFFFF for i in range(n)])


def _int(arr, lo=0, n=8):
    return sum(int(arr[lo + i]) << (32 * i) for i in range(n))


def _pts(points):
    """affine points (None = identity) -> 16 limbs each"""
    flat = []
    for p in points:
        x, y = (0, 0) if p is None else p
        flat += list(_limbs(x)) + list(_limbs(y))
    return (ctypes.c_uint32 * max(16, len(flat)))(*flat)


def _pt(arr, i=0):
    x, y = _int(arr, 16 * i), _int(arr, 16 * i + 8)
    return None if x == 0 and y == 0 else (x, y)


def _rand_point(rng):
    return bn.g1_mul_gen(rng.randrange(1, bn.R))


def test_window_weights(built):
    lib = _acclib()
    out = (ctypes.c_uint32 * 8)()
    for c, w in [(0, 0), (0, 5), (1, 0), (4, 63), (12, 21), (15, 16), (13, 20), (16, 16), (17, 15)]:
        lib.x_weight(c, w, out)
        assert _int(out) == pow(2, c * w, bn.R), (c, w)


def test_glv_mul_with_jacobian_base(built):
    lib = _acclib()
    rng = random.Random("acc-glv")
    out = (ctypes.c_uint32 * 16)()
    lam = 0xB3C4D79D41A917585BFC41088D8DAAA78B17EA66B99C90DD  # the GLV eigenvalue: phi(P) = [lambda] P
    edge = [0, 1, 2, bn.R - 1, bn.R - 2, 1 << 128, (1 << 128) - 1, 1 << 252, lam, bn.R - lam]
    for k in edge + [rng.randrange(bn.R) for _ in range(30)]:
        p = _rand_point(rng)
        z = rng.randrange(1, bn.P)
        lib.x_mul_jac(_pts([p]), _limbs(z), _limbs(k), out)
        assert _pt(out) == bn.g1_mul(p, k), k
    lib.x_mul_jac(_pts([None]), _limbs(5), _limbs(rng.randrange(bn.R)), out)
    assert _pt(out) is None


def _absorb(c, W, wsums, acc, s, z):
    lib = _acclib()
    rec, new = (ctypes.c_uint32 * 32)(), (ctypes.c_uint32 * 32)()
    assert lib.x_absorb(c[0], W[0], c[1], W[1], _pts(wsums), _pts(acc), _limbs(s), _limbs(z), rec, new) == 0
    return (_pt(rec, 0), _pt(rec, 1)), (_pt(new, 0), _pt(new, 1))


def _combine(c, ws):
    out = None
    for w, p in enumerate(ws):
        out = bn.g1_add(out, bn.g1_mul(p, pow(2, c * w, bn.R)) if p is not None else None)
    return out


def test_tree_sum_equals_horner_combination(built):
    lib = _acclib()
    rng = random.Random("acc-tree")
    out = (ctypes.c_uint32 * 16)()
    geoms = [((12, 12), (22, 22)), ((4, 4), (64, 64)), ((15, 9), (17, 29)), ((7, 5), (37, 51)), ((13, 11), (1, 2)), ((0, 0), (1, 1))]
    for c, W in geoms:
        base = _rand_point(rng)
        ws = []
        for ch in range(2):
            row = [_rand_point(rng) for _ in range(W[ch])]
            for w in rng.sample(range(W[ch]), min(W[ch], 3)):  # empty windows, and equal sums meeting in the tree
                row[w] = rng.choice([None, base])
            ws.append(row)
        z = rng.randrange(1, bn.P)
        rec, _ = _absorb(c, W, ws[0] + ws[1], [None, None], rng.randrange(1, bn.R), z)
        for ch in range(2):
            want = _combine(c[ch], ws[ch])
            assert rec[ch] == want, (c, W, ch)
            lib.x_horner(c[ch], W[ch], _pts(ws[ch]), _limbs(z), out)
            assert _pt(out) == want


def test_scale_and_add(built):
    rng = random.Random("acc-scale")
    for _ in range(6):
        acc = [_rand_point(rng), _rand_point(rng)]
        ws = [_rand_point(rng) for _ in range(5)] + [_rand_point(rng) for _ in range(7)]
        s = rng.randrange(1, bn.R)
        rec, new = _absorb((9, 11), (5, 7), ws, acc, s, rng.randrange(1, bn.P))
        for ch in range(2):
            assert new[ch] == bn.g1_add(bn.g1_mul(acc[ch], s), rec[ch])
    # edge cases on one window of weight 1 (the merge geometry): empty accumulator, empty batch, s = 1, a sum of zero
    p, q = _rand_point(rng), _rand_point(rng)
    s = rng.randrange(2, bn.R)
    for acc, ws, sc, want in [([None, None], [p, q], s, (p, q)), ([p, q], [None, None], s, (bn.g1_mul(p, s), bn.g1_mul(q, s))),
                              ([p, q], [q, p], 1, (bn.g1_add(p, q), bn.g1_add(p, q))),
                              ([p, q], [bn.g1_neg(bn.g1_mul(p, s)), bn.g1_mul(q, s)], s, (None, bn.g1_mul(q, 2 * s)))]:
        _rec, new = _absorb((0, 0), (1, 1), ws, acc, sc, rng.randrange(1, bn.P))
        assert new == want


def test_create_refuses_a_null_anchor(built, pkg):
    with pytest.raises(pkg.BackendError, match="anchor"):
        pkg.Accumulator(None)


# ---------------------------------------------------------------- GPU
def _enc(L, R_):
    return enc_point(L) + enc_point(R_)


def _rs(rng, n):
    return [rng.randrange(1, bn.R) for _ in range(n)]


@pytest.mark.gpu
def test_chunks_equal_the_concatenated_batch(pkg):
    """uneven chunks, one of a single proof, one whose proofs all fail, ragged instances: the accumulator equals one
    verify_batch over the concatenation and the oracle's AccumulatorStrategy"""
    A = circuits()[0]
    rng = random.Random("acc-chunks")
    insts = [sim.random_instances(A.vk, rng, 3 + 4 * (t % 3)) for t in range(13)]  # ragged: lengths differ per proof
    proofs = [sim.simulate_proof(A.params, A.vk, A.dl, S, i, rng) for i in insts]
    api = [i[0] for i in insts]
    for j in (4, 5, 6):  # the chunk [4, 7) fails entirely: transcript-class corruptions
        proofs[j], _ = sim.corrupt(proofs[j], A.vk, ("truncate_body", "point_offcurve", "scalar_ge_r")[j - 4], rng)
    want = [orc.verify_proof(A.params, A.vk, i, p) for i, p in zip(insts, proofs)]
    assert all(w.status != orc.OK for w in want[4:7])
    rs = _rs(rng, len(proofs))
    with A.bv(pkg) as bv, pkg.Accumulator(bv, max_absorbs=8) as acc:
        st = []
        for k, (lo, hi) in enumerate([(0, 3), (3, 4), (4, 7), (7, 13)]):
            res = acc.absorb(bv, proofs[lo:hi], api[lo:hi], rlc_scalars=rs[lo:hi])
            assert res.index == k
            st += res.statuses
        assert st == [w.status for w in want]
        L, R_, ok = orc.accumulate(A.params, want, rs)
        assert ok and acc.to_bytes() == _enc(L, R_)
        assert acc.to_bytes() == bv.verify_batch(proofs, api, rlc_scalars=rs, want_batch_accum=True).batch_accum
        fin = acc.finalize()
        assert fin.verdict and fin.absorb_verdicts == [True] * 4
        assert acc.to_bytes() == bytes(128)  # finalize consumed the accumulator


@pytest.mark.gpu
def test_absorbs_across_contexts(pkg):
    """SHPLONK/Blake2b, GWC/Keccak, 3 circuit instances per proof and another k under one trapdoor: the accumulator
    equals the mixed batch over the same member-major order; params of another trapdoor are refused"""
    circs = circuits()
    rng = random.Random("acc-ctx")
    insts, proofs = zip(*[c.proofs(rng, n) for c, n in zip(circs, (4, 3, 2, 5))])
    api = [c.api(i) for c, i in zip(circs, insts)]
    rs = _rs(rng, 14)
    bvs = [c.bv(pkg) for c in circs]
    try:
        with pkg.Accumulator(bvs[0]) as acc:
            off = 0
            for bv, p, a in zip(bvs, proofs, api):
                assert acc.absorb(bv, p, a, rlc_scalars=rs[off: off + len(p)]).statuses == [0] * len(p)
                off += len(p)
            want = [w for c, i, p in zip(circs, insts, proofs) for w in c.oracle(i, p)]
            L, R_, ok = orc.accumulate(circs[0].params, want, rs)
            with pkg.MixedBatchVerifier(bvs) as mx:
                mixed = mx.verify_batch(list(proofs), api, rlc_scalars=rs, want_batch_accum=True)
            assert ok and acc.to_bytes() == _enc(L, R_) == mixed.batch_accum
            X = Circ("vm", 8, "shplonk", "blake2b", s=S + 1)
            ix, px = X.proofs(rng, 2)
            with X.bv(pkg) as bx:
                with pytest.raises(pkg.BackendError, match="differ"):
                    acc.absorb(bx, px, X.api(ix))
            assert acc.to_bytes() == _enc(L, R_)
            assert acc.finalize() == pkg.FinalizeResult(True, [True] * 4)
    finally:
        [bv.close() for bv in bvs]


@pytest.mark.gpu
def test_rejection_names_the_absorb(pkg):
    A = circuits()[0]
    rng = random.Random("acc-reject")
    with A.bv(pkg) as bv, pkg.Accumulator(bv) as acc:
        batches = [A.proofs(rng, n) for n in (3, 4, 2, 3)]
        bi, bp = batches[2]
        bp = list(bp)
        bp[1], expect = sim.corrupt(bp[1], A.vk, "eval_flip", rng)
        batches[2] = (bi, bp)
        for k, (i, p) in enumerate(batches):
            assert acc.absorb(bv, p, A.api(i)).statuses == [0] * len(p)  # a pairing failure shows at finalize only
        fin = acc.finalize()
        assert not fin.verdict and fin.absorb_verdicts == [True, True, False, True]
        re = bv.verify_batch(bp, A.api(bi))  # the caller re-verifies the named batch
        assert re.status == [w.status for w in A.oracle(bi, bp)] and re.status[1] == expect
        # transcript-class corruptions: their statuses at absorb time, the rest of the sequence accepted
        i, p = A.proofs(rng, 6)
        p = list(p)
        kinds = ["scalar_ge_r", "point_offcurve", "truncate_opening"]
        exp = [0] * 6
        for j, kind in zip((0, 2, 5), kinds):
            p[j], exp[j] = sim.corrupt(p[j], A.vk, kind, rng)
        assert acc.absorb(bv, p, A.api(i)).statuses == exp == [w.status for w in A.oracle(i, p)]
        i2, p2 = A.proofs(rng, 2)
        acc.absorb(bv, p2, A.api(i2))
        assert acc.finalize() == pkg.FinalizeResult(True, [True, True])


@pytest.mark.gpu
def test_export_merge_restore(pkg):
    A = circuits()[0]
    rng = random.Random("acc-merge")
    with A.bv(pkg) as bv, pkg.Accumulator(bv) as a, pkg.Accumulator(bv) as b, pkg.Accumulator(bv, max_absorbs=1) as c:
        i, p = A.proofs(rng, 5)
        a.absorb(bv, p[:2], A.api(i[:2]))
        b.absorb(bv, p[2:], A.api(i[2:]))
        xa, xb = a.to_bytes(), b.to_bytes()
        c.merge(xa, r=12345)  # restore a checkpoint
        assert c.to_bytes() == xa and c.finalize().verdict and a.to_bytes() == xa
        r = rng.randrange(1, bn.R)
        a.merge(xb, r=r)
        for off in (0, 64):
            assert _dec(a.to_bytes()[off: off + 64]) == bn.g1_add(bn.g1_mul(_dec(xa[off: off + 64]), r), _dec(xb[off: off + 64]))
        xm = a.to_bytes()
        x, y = _dec(xb[:64])
        for bad in (enc_point((x, (y + 1) % bn.P)) + xb[64:], xb[:64] + (x + bn.P).to_bytes(32, "little") + xb[96:],
                    xb[:64] + xb[64:96] + (y + bn.P).to_bytes(32, "little")):
            with pytest.raises(pkg.BackendError, match="canonical"):
                a.merge(bad, r=3)
        with pytest.raises(pkg.BackendError, match="scalar"):
            a.merge(xb, r=bn.R)
        assert a.to_bytes() == xm
        fin = a.finalize()
        assert fin.verdict and fin.absorb_verdicts == [True, True]
        # a rejected state survives export and restore
        bp = list(p)
        bp[0], _ = sim.corrupt(bp[0], A.vk, "point_swap", rng)
        b.absorb(bv, bp, A.api(i))
        xr = b.to_bytes()
        c.merge(xr)  # r from the OS: into an empty accumulator it does not matter
        assert c.to_bytes() == xr
        with pytest.raises(pkg.BackendError, match="full"):
            c.merge(xr)
        assert not c.finalize().verdict and not b.finalize().verdict


@pytest.mark.gpu
def test_graph_replay_equals_direct_launches(pkg):
    A = circuits()[0]
    rng = random.Random("acc-graph")
    shapes = [A.proofs(rng, n) for n in (3, 5)]
    rs = {n: _rs(rng, n) for n in (3, 5)}
    with A.bv(pkg) as bv:
        out = []
        for graphs in (True, False):
            bv.set_graphs(graphs)
            with pkg.Accumulator(bv, max_absorbs=64) as acc:
                for t in range(4):  # warm-up: every shape's buffers and graph
                    i, p = shapes[t % 2]
                    acc.absorb(bv, p, A.api(i), rlc_scalars=rs[len(p)])
                caps = bv.cache_stats()["graph_captures"]
                for t in range(50):
                    i, p = shapes[t % 2]
                    assert acc.absorb(bv, p, A.api(i), rlc_scalars=rs[len(p)]).index == 4 + t
                if graphs:
                    assert bv.cache_stats()["graph_captures"] == caps
                out.append(acc.to_bytes())
                assert acc.finalize() == pkg.FinalizeResult(True, [True] * 54)
        assert out[0] == out[1] and out[0] != bytes(128)


@pytest.mark.gpu
def test_fold_randomness_and_refusals(pkg):
    A = circuits()[0]
    rng = random.Random("acc-rand")
    i, p = A.proofs(rng, 4)
    api = A.api(i)
    with A.bv(pkg) as bv:
        seed = 0x5EED
        key = bytes(rng.getrandbits(8) for _ in range(32))
        got = {}
        for name, kw in [("seed", dict(seed=seed)), ("seed_rs", dict(rlc_scalars=_expand(b"h2v-rlc", seed.to_bytes(8, "little"), 4))),
                         ("key", dict(key=key)), ("key_rs", dict(rlc_scalars=_expand(b"h2v-rlk", key, 4))), ("os1", {}), ("os2", {})]:
            with pkg.Accumulator(bv) as acc:
                acc.absorb(bv, p, api, **kw)
                got[name] = (acc.to_bytes(), bv.rlc_source())
                assert acc.finalize().verdict
        assert got["seed"][0] == got["seed_rs"][0] and got["seed"][1] == "seed"
        assert got["key"][0] == got["key_rs"][0] and got["key"][1] == "key"
        assert got["os1"][1] == got["os2"][1] == "os" and got["os1"][0] != got["os2"][0]
        with pkg.Accumulator(bv, max_absorbs=2) as acc:
            acc.absorb(bv, p[:1], api[:1])
            x = acc.to_bytes()
            with pytest.raises(pkg.BackendError, match="at least one proof"):
                acc.absorb(bv, [], [])
            assert acc.to_bytes() == x
            bv.lib.h2v_batch_set_fold_groups(bv._ctx, 2)
            with pytest.raises(pkg.BackendError, match="fold-group"):
                acc.absorb(bv, p[:2], api[:2])
            bv.lib.h2v_batch_set_fold_groups(bv._ctx, 1)
            acc.absorb(bv, p[1:], api[1:])
            x = acc.to_bytes()
            with pytest.raises(pkg.BackendError, match="full"):
                acc.absorb(bv, p[:1], api[:1])
            assert acc.to_bytes() == x
            acc.reset()
            assert acc.to_bytes() == bytes(128)
            assert acc.finalize() == pkg.FinalizeResult(True, [])
            assert acc.finalize() == pkg.FinalizeResult(True, [])  # empty: the identity DualMSM accepts
