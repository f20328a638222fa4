"""Sharded mixed batches (include/h2v.h "sharded mixed batches"): one mixed batch split over ranks, each rank folding its
share with globally defined coefficients, one pairing check over the ranks' partials.  The checkers are the unsharded
h2v_mix_verify over the concatenation and the CPU oracle's AccumulatorStrategy over it.

CPU: the range -> per-member counts split and the window-geometry bound (csrc/mix.cuh, through tests/hostlib), and
sharding.mixed_shard.  GPU (one B200): the ranks are mixes of distinct member contexts on one device; the exchange tests
drive each rank from its own host thread, as two processes would.  Multi-GPU: one process per GPU (self-skips below 2)."""
import ctypes
import functools
import os
import random
import sys

import pytest

import bn254 as bn
import formats as F
import prover_sim as sim
import verifier as orc
from test_mixed_batch import S, circuits
from test_multi_params_mix import PCirc, mp_oracle
from workloads import enc_point

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)


# ---------------------------------------------------------------- CPU: split helper and geometry bound
@functools.lru_cache(maxsize=None)
def _lib():
    return ctypes.CDLL(os.path.join(HERE, "hostlib", "libmixshard.so"))


def _u32(v):
    return (ctypes.c_uint32 * max(1, len(v)))(*v)


def shard_counts(gc, base, n):
    out = (ctypes.c_uint32 * len(gc))()
    ok = _lib().x_shard_counts(len(gc), _u32(gc), ctypes.c_ulonglong(base), n, out)
    return list(out) if ok else None


def shard_bound(P, M, Sh, gc, max_shard):
    out = (ctypes.c_ulonglong * 2)()
    _lib().x_shard_bound(len(P), _u32(P), _u32(M), _u32(Sh), _u32(gc), max_shard, out)
    return tuple(out)


def _sharding(pkg):
    import importlib

    return importlib.import_module("halo2_verifier_b200.sharding")


def _splits(rng, N, world):
    """uneven contiguous ranges covering [0, N), each non-empty"""
    cuts = sorted(rng.sample(range(1, N), world - 1)) if world > 1 else []
    return [0] + cuts + [N]


def test_shard_counts_split_the_global_order(built, pkg):
    sharding = _sharding(pkg)
    rng = random.Random("mixshard-split")
    for _ in range(300):
        K = rng.randint(1, 12)
        gc = [rng.choice([0, 0, 1, 2, 3, 7, 20]) for _ in range(K)]
        N = sum(gc)
        if N == 0:
            assert shard_counts(gc, 0, 1) is None
            continue
        order = [(m, j) for m, c in enumerate(gc) for j in range(c)]  # the global member-major order
        for world in range(1, min(8, N) + 1):
            for b in (_splits(rng, N, world), [sharding.shard_range(N, r, world)[0] for r in range(world)] + [N]):
                got = []
                for r in range(world):
                    lo, hi = b[r], b[r + 1]
                    loc = shard_counts(gc, lo, hi - lo)
                    assert sum(loc) == hi - lo and loc == sharding.mixed_shard_counts(gc, lo, hi - lo)
                    # this rank's portion, member-major: member m's proofs from its first global index inside the range
                    for m, k in enumerate(loc):
                        first = max(lo - sum(gc[:m]), 0)
                        got += [(m, first + j) for j in range(k)]
                assert got == order
            for r in range(world):  # mixed_shard = shard_range + per-member [lo, hi)
                (lo, hi), per = sharding.mixed_shard(gc, r, world)
                assert (lo, hi) == sharding.shard_range(N, r, world)
                assert [b - a for a, b in per] == shard_counts(gc, lo, hi - lo)
                assert [order.index((m, a)) for m, (a, b) in enumerate(per) if b > a] == sorted(
                    order.index((m, a)) for m, (a, b) in enumerate(per) if b > a)
        assert shard_counts(gc, 0, 0) is None and shard_counts(gc, N, 1) is None and shard_counts(gc, 1, N) is None


def test_geometry_bound_is_common_and_covers_every_rank(built):
    rng = random.Random("mixshard-bound")
    for _ in range(200):
        K = rng.randint(1, 10)
        gc = [rng.choice([0, 1, 3, 9, 40]) for _ in range(K)]
        N = sum(gc)
        if N == 0:
            continue
        P = [rng.randint(1, 40) for _ in range(K)]
        M = [rng.randint(0, 6) for _ in range(K)]
        Sh = [rng.randint(1, 30) for _ in range(K)]
        world = rng.randint(1, min(8, N))
        b = _splits(rng, N, world)
        hint = max(b[r + 1] - b[r] for r in range(world))
        bound = shard_bound(P, M, Sh, gc, hint)
        for r in range(world):
            loc = shard_counts(gc, b[r], b[r + 1] - b[r])
            # the bound is a function of what the ranks share: the same whatever the rank's composition
            assert shard_bound(P, M, Sh, gc, hint) == bound
            right = sum(n * p + s for n, p, s in zip(loc, P, Sh) if n)
            left = sum(n * m for n, m in zip(loc, M))
            assert bound[0] >= right and bound[1] >= left


# ---------------------------------------------------------------- GPU helpers
def _portions(gc, lo, hi):
    """per member [a, b) of its own proof list inside the global range [lo, hi)"""
    out, start = [], 0
    for c in gc:
        a, b = min(max(lo - start, 0), c), min(max(hi - start, 0), c)
        out.append((a, b))
        start += c
    return out


class Ranks:
    """`world` mixes over distinct member contexts of the same circuits on one device"""

    def __init__(self, pkg, circs, world, multi_params=False):
        self.bvs = [[c.bv(pkg) for c in circs] for _ in range(world)]
        self.mixes = [pkg.MixedBatchVerifier(b, multi_params=multi_params) for b in self.bvs]

    def close(self):
        [mx.close() for mx in self.mixes]
        [bv.close() for b in self.bvs for bv in b]


def _share(proofs, api, b, r):
    gc = [len(p) for p in proofs]
    per = _portions(gc, b[r], b[r + 1])
    return [p[x:y] for p, (x, y) in zip(proofs, per)], [i[x:y] for i, (x, y) in zip(api, per)]


def gather_run(ranks, proofs, api, b, root=0, finalizer=None, **fold):
    """every rank's accumulate_shard, `finalizer` (default: the root rank's mix) sums and checks, attribution on rejection.
    Returns (verdict, statuses per member of the concatenation, batch_accum)."""
    gc = [len(p) for p in proofs]
    world = len(b) - 1
    hint = max(b[r + 1] - b[r] for r in range(world))
    parts, sts = [], []
    for r in range(world):
        p, i = _share(proofs, api, b, r)
        st, part = ranks.mixes[r].accumulate_shard(p, i, gc, b[r], shard_hint=hint, **fold)
        assert len(part) == ranks.mixes[r].partial_bytes(gc)
        parts.append(part)
        sts.append(st)
    ok, bacc = (finalizer or ranks.mixes[root]).finalize(parts, gc)
    if not ok:
        sts = [ranks.mixes[r].attribute_shard(sts[r]) for r in range(world)]
    return ok, [sum((st[m] for st in sts), []) for m in range(len(gc))], bacc


def _parity_batch(rng):
    A, B, C, D = circuits()
    ia = [sim.random_instances(A.vk, rng, 3 + 4 * (t % 3)) for t in range(7)]  # ragged public inputs
    pa = [sim.simulate_proof(A.params, A.vk, A.dl, S, i, rng) for i in ia]
    ib, pb = B.proofs(rng, 6)
    ic, pc = C.proofs(rng, 4)
    circs = (A, B, C, D)
    return circs, [ia, ib, ic, []], [pa, pb, pc, []]


# ---------------------------------------------------------------- GPU
@pytest.mark.gpu
def test_world_one_equals_mix_verify(pkg):
    rng = random.Random("mixshard-w1")
    circs, insts, proofs = _parity_batch(rng)
    api = [c.api(i) for c, i in zip(circs, insts)]
    proofs[1][2], _ = sim.corrupt(proofs[1][2], circs[1].vk, "scalar_ge_r", rng, circs[1].mo)  # a transcript error: excluded from the fold
    n = sum(len(p) for p in proofs)
    ranks = Ranks(pkg, circs, 1)
    try:
        for corrupt in (False, True):
            if corrupt:
                proofs[2][1], _ = sim.corrupt(proofs[2][1], circs[2].vk, "eval_flip", rng, circs[2].mo, circs[2].m)
            rs = [rng.randrange(1, bn.R) for _ in range(n)]
            want = ranks.mixes[0].verify_batch(proofs, api, rlc_scalars=rs, want_batch_accum=True)
            ok, st, bacc = gather_run(ranks, proofs, api, [0, n], rlc_scalars=rs)
            assert st == want.status and bacc == want.batch_accum
            assert (ok and all(v == 0 for s in st for v in s)) == want.verdict and ok == (not corrupt)
    finally:
        ranks.close()


# uneven splits of the 17-proof parity batch (members at [0, 7), [7, 13), [13, 17)) with cuts inside members
SPLITS = {2: [0, 10, 17], 3: [0, 3, 12, 17], 5: [0, 2, 8, 9, 15, 17]}


@pytest.mark.gpu
@pytest.mark.parametrize("world", [2, 3, 5])
def test_sharded_parity(pkg, world):
    rng = random.Random(f"mixshard-parity-{world}")
    circs, insts, proofs = _parity_batch(rng)
    api = [c.api(i) for c, i in zip(circs, insts)]
    n = sum(len(p) for p in proofs)
    want = [c.oracle(i, p) for c, i, p in zip(circs, insts, proofs)]
    ranks = Ranks(pkg, circs, world)
    try:
        for trial in range(2):
            b = SPLITS[world] if trial == 0 else _splits(rng, n, world)
            rs = [rng.randrange(1, bn.R) for _ in range(n)]
            L, R_, okk = orc.accumulate(circs[0].params, [w for ws in want for w in ws], rs)
            whole = ranks.mixes[0].verify_batch(proofs, api, rlc_scalars=rs, want_batch_accum=True)
            assert whole.batch_accum == enc_point(L) + enc_point(R_) and whole.verdict and okk
            ok, st, bacc = gather_run(ranks, proofs, api, b, root=trial % world, rlc_scalars=rs)
            assert ok and bacc == whole.batch_accum and st == whole.status == [[w.status for w in ws] for ws in want]
            key = bytes(rng.getrandbits(8) for _ in range(32))
            ok, st, bacc = gather_run(ranks, proofs, api, b, key=key)
            whole_key = ranks.mixes[0].verify_batch(proofs, api, key=key, want_batch_accum=True)
            assert ok and st == whole_key.status and bacc == whole_key.batch_accum != whole.batch_accum
    finally:
        ranks.close()


@pytest.mark.gpu
def test_rejections_attributed_on_every_rank(pkg):
    A, B, C, _D = circuits()
    circs = (A, B, C)
    rng = random.Random("mixshard-reject")
    insts, proofs = zip(*[c.proofs(rng, n) for c, n in zip(circs, (6, 5, 4))])
    proofs = [list(p) for p in proofs]
    slots = [(0, 0), (0, 2), (0, 3), (0, 5), (1, 0), (1, 1), (1, 4), (2, 1), (2, 2)]
    for kind, (m, j) in zip(sim.CORRUPTIONS, slots):
        proofs[m][j], _ = sim.corrupt(proofs[m][j], circs[m].vk, kind, rng, circs[m].mo, circs[m].m)
    api = [c.api(i) for c, i in zip(circs, insts)]
    want = [[w.status for w in c.oracle(i, p)] for c, i, p in zip(circs, insts, proofs)]
    ranks = Ranks(pkg, circs, 3)
    try:
        rs = [rng.randrange(1, bn.R) for _ in range(15)]
        whole = ranks.mixes[0].verify_batch(proofs, api, rlc_scalars=rs)
        ok, st, _ = gather_run(ranks, proofs, api, [0, 4, 9, 15], rlc_scalars=rs)
        assert not ok and st == whole.status == want
    finally:
        ranks.close()


@pytest.mark.gpu
def test_multi_params_every_rank_emits_every_set(pkg):
    X0 = PCirc("vm", 8, "shplonk", "blake2b")
    X1 = PCirc("sh", 8, "gwc", "keccak", s=S + 1)
    X2 = PCirc("vm", 10, "gwc", "blake2b", t=7)
    circs = (X0, X1, X2)
    rng = random.Random("mixshard-mparams")
    insts, proofs = zip(*[c.proofs(rng, n) for c, n in zip(circs, (5, 2, 4))])
    proofs = [list(p) for p in proofs]
    api = [c.api(i) for c, i in zip(circs, insts)]
    ranks = Ranks(pkg, circs, 2, multi_params=True)
    try:
        gc = [5, 2, 4]
        assert ranks.mixes[0].n_classes == 3 and ranks.mixes[0].partial_bytes(gc) == 3 * pkg.load_library().h2v_partial_bytes()
        b = [0, 4, 11]  # rank 0: member 0 only (no proof of class 1); rank 1: the rest
        for corrupt in (False, True):
            if corrupt:
                proofs[2][3], _ = sim.corrupt(proofs[2][3], X2.vk, "eval_flip", rng, X2.mo)
            rs = [rng.randrange(1, bn.R) for _ in range(11)]
            whole = ranks.mixes[1].verify_batch(proofs, api, rlc_scalars=rs, want_batch_accum=True)
            _class_of, run = mp_oracle([c.params for c in circs], [c.oracle(i, p) for c, i, p in zip(circs, insts, proofs)])
            folds, okk = run(rs)
            assert whole.batch_accum == b"".join(enc_point(L) + enc_point(R_) for L, R_ in folds)
            ok, st, bacc = gather_run(ranks, proofs, api, b, rlc_scalars=rs)
            assert ok == okk == (not corrupt) and bacc == whole.batch_accum and st == whole.status
    finally:
        ranks.close()


def _run_threads(fns):
    from test_exchange import run_ranks

    return run_ranks(fns)


@pytest.mark.gpu
def test_exchange_two_ranks(pkg):
    os.environ.setdefault("H2V_COMM_TIMEOUT_MS", "5000")
    rng = random.Random("mixshard-xchg")
    circs, insts, proofs = _parity_batch(rng)
    api = [c.api(i) for c, i in zip(circs, insts)]
    gc = [len(p) for p in proofs]
    n, b = sum(gc), [0, 9, sum(gc)]
    ranks = Ranks(pkg, circs, 2)
    try:
        handles = [mx.comm_init(r, 2) for r, mx in enumerate(ranks.mixes)]
        [mx.comm_connect(handles) for mx in ranks.mixes]
        assert all(mx.comm_ready for mx in ranks.mixes)
        rs = [rng.randrange(1, bn.R) for _ in range(n)]
        ok, st, bacc = gather_run(ranks, proofs, api, b, rlc_scalars=rs)

        def rank_call(r, root, prf):
            p, i = _share(prf, api, b, r)
            return ranks.mixes[r].verify_shard(p, i, gc, b[r], root, rlc_scalars=rs, shard_hint=9)
        for root in (0, 1, 1, 0, 0, 1):
            res = _run_threads([lambda r=r: rank_call(r, root, proofs) for r in range(2)])
            assert all(v == ok for v, _ in res) and ok
            assert [sum((x[1][m] for x in res), []) for m in range(len(gc))] == st
            assert ranks.mixes[root].comm_last_batch_accum() == bacc
            with pytest.raises(pkg.BackendError, match="root"):
                ranks.mixes[1 - root].comm_last_batch_accum()
        caps = [mx.cache_stats()["graph_captures"] for mx in ranks.mixes]
        for root in (1, 0):  # replays: no recapture after the first launch set of each kind
            _run_threads([lambda r=r: rank_call(r, root, proofs) for r in range(2)])
        assert [mx.cache_stats()["graph_captures"] for mx in ranks.mixes] == caps
        # a corrupted proof on the non-root rank (rank 1 holds member 1's last proofs)
        bad = [list(p) for p in proofs]
        bad[1][5], _ = sim.corrupt(bad[1][5], circs[1].vk, "eval_flip", rng, circs[1].mo)
        want = [[w.status for w in c.oracle(i, p)] for c, i, p in zip(circs, insts, bad)]
        res = _run_threads([lambda r=r: rank_call(r, 0, bad) for r in range(2)])
        assert [v for v, _ in res] == [False, False]
        assert res[0][1] == [[0] * len(x) for x in res[0][1]]
        assert [sum((x[1][m] for x in res), []) for m in range(len(gc))] == want and orc.CONSTRAINT_SYSTEM_FAILURE in res[1][1][1]
    finally:
        ranks.close()


@pytest.mark.gpu
def test_graphs_off_equals_replay(pkg):
    rng = random.Random("mixshard-graphs")
    circs, insts, proofs = _parity_batch(rng)
    api = [c.api(i) for c, i in zip(circs, insts)]
    n = sum(len(p) for p in proofs)
    proofs[0][1], _ = sim.corrupt(proofs[0][1], circs[0].vk, "point_swap", rng)
    ranks = Ranks(pkg, circs, 2)
    try:
        rs = [rng.randrange(1, bn.R) for _ in range(n)]
        b = [0, 5, n]
        g = gather_run(ranks, proofs, api, b, rlc_scalars=rs)
        [bvs[0].set_graphs(False) for bvs in ranks.bvs]
        d = gather_run(ranks, proofs, api, b, rlc_scalars=rs)
        assert g == d and not g[0] and g[1][0][1] == orc.CONSTRAINT_SYSTEM_FAILURE
        t = ranks.bvs[1][0].timings()
        assert t["rlc_msm"] > 0
    finally:
        ranks.close()


@pytest.mark.gpu
def test_refusals_leave_the_state_unchanged(pkg):
    rng = random.Random("mixshard-refuse")
    A, B, C, D = circuits()
    circs = (A, B)
    insts, proofs = zip(*[c.proofs(rng, n) for c, n in zip(circs, (3, 3))])
    proofs = [list(p) for p in proofs]
    api = [c.api(i) for c, i in zip(circs, insts)]
    gc = [3, 3]
    ranks = Ranks(pkg, circs, 2)
    mx = ranks.mixes[0]
    lib = mx.lib
    try:
        rs = [rng.randrange(1, bn.R) for _ in range(6)]
        ref = gather_run(ranks, proofs, api, [0, 3, 6], rlc_scalars=rs)
        launches = [bv.launch_count() for bv in ranks.bvs[0]]
        p0, i0 = _share(proofs, api, [0, 3, 6], 0)
        counts, packed = mx._pack(p0, i0)
        st = (ctypes.c_uint8 * 3)()
        part = ctypes.create_string_buffer(2 * 12320)
        rsb = b"".join(r.to_bytes(32, "little") for r in rs)

        def acc(gcounts=gc, base=0, n=3, rlc=rsb, status=st, partial=part, packed_=packed):
            return lib.h2v_mix_accumulate_shard(mx._mx, None if gcounts is None else mx._u32(gcounts), base, n, *packed_[:4], rlc, 0,
                                                status, None if partial is None else ctypes.cast(partial, ctypes.c_void_p))
        cases = [(dict(gcounts=None), "null"), (dict(status=None), "null"), (dict(partial=None), "null"), (dict(gcounts=[0, 0]), "between 1"),
                 (dict(n=0), "non-empty range"), (dict(base=4), "non-empty range"),
                 (dict(rlc=bytes(32) + rsb[32:]), "canonical and non-zero"), (dict(rlc=bn.R.to_bytes(32, "little") + rsb[32:]), "canonical")]
        for kw, msg in cases:
            assert acc(**kw) == -1 and msg in lib.h2v_mix_last_error(mx._mx).decode(), (kw, lib.h2v_mix_last_error(mx._mx))
        assert lib.h2v_mix_set_shard_hint(mx._mx, 2) == 0
        assert acc() == -1 and "smaller than this shard" in lib.h2v_mix_last_error(mx._mx).decode()
        assert lib.h2v_mix_set_shard_hint(mx._mx, 0) == 0
        lib.h2v_batch_set_fold_groups(ranks.bvs[0][1]._ctx, 2)
        assert acc() == -1 and "pending fold-group" in lib.h2v_mix_last_error(mx._mx).decode()
        lib.h2v_batch_set_fold_groups(ranks.bvs[0][1]._ctx, 1)
        ok = ctypes.c_int(0)
        assert lib.h2v_mix_finalize(mx._mx, mx._u32(gc), 0, ctypes.cast(part, ctypes.c_void_p), None, ctypes.byref(ok)) == -1
        assert lib.h2v_mix_attribute_shard(mx._mx, None) == -1
        # exchange refusals: no channel; then max_groups < sets on a multi-class mix is covered by comm_init's floor
        vr = ctypes.c_int(0)
        assert lib.h2v_mix_verify_shard(mx._mx, mx._u32(gc), 0, 3, *packed[:4], rsb, 0, 0, st, ctypes.byref(vr)) == -1
        assert "h2v_comm_init" in lib.h2v_mix_last_error(mx._mx).decode()
        assert [bv.launch_count() for bv in ranks.bvs[0]] == launches
        assert gather_run(ranks, proofs, api, [0, 3, 6], rlc_scalars=rs) == ref  # nothing pending, nothing changed
        # different hints on the ranks: the partials' geometries differ
        parts = []
        for r, hint in ((0, 3), (1, 4000)):
            p, i = _share(proofs, api, [0, 3, 6], r)
            parts.append(ranks.mixes[r].accumulate_shard(p, i, gc, 3 * r, rlc_scalars=rs, shard_hint=hint)[1])
        assert parts[0][4:12] != parts[1][4:12]
        with pytest.raises(pkg.BackendError, match="different window geometries"):
            mx.finalize(parts, gc)
        with pytest.raises(ValueError):
            mx.accumulate_shard([proofs[0][:2], []], [api[0][:2], []], gc, 2)  # the share of [2, 4) is one proof of each member
    finally:
        ranks.close()


@pytest.mark.gpu
def test_exchange_refuses_a_small_channel(pkg):
    X0 = PCirc("vm", 8, "shplonk", "blake2b")
    X1 = PCirc("vm", 8, "shplonk", "blake2b", s=S + 1)
    rng = random.Random("mixshard-small")
    insts, proofs = zip(*[c.proofs(rng, 2) for c in (X0, X1)])
    api = [c.api(i) for c, i in zip((X0, X1), insts)]
    ranks = Ranks(pkg, (X0, X1), 1, multi_params=True)
    try:
        mx = ranks.mixes[0]
        h = ranks.bvs[0][0].comm_init(0, 1, 1)  # max_groups 1 < 2 sets, bypassing the mix's floor
        ranks.bvs[0][0].comm_connect([h])
        mx.comm_ready = True
        with pytest.raises(pkg.BackendError, match="bucket sets"):
            mx.verify_shard([list(p) for p in proofs], api, [2, 2], 0, 0, seed=5)
        assert mx.verify_shard([list(proofs[0]), []], [api[0], []], [2, 0], 0, 0, seed=5)[0]  # one set fits
    finally:
        ranks.close()


# ---------------------------------------------------------------- one process per GPU
def _rank_main(rank, world, port, q, use_exchange):
    for p in (ROOT, os.path.join(ROOT, "oracle"), HERE):
        sys.path.insert(0, p)
    import hashlib

    import torch
    import torch.distributed as dist

    import __graft_entry__ as g

    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), H2V_COMM_TIMEOUT_MS="20000")
    torch.cuda.set_device(rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=torch.device("cuda", rank))
    pkg = g.load_package()
    sharding = __import__("importlib").import_module("halo2_verifier_b200.sharding")
    try:
        rng = random.Random("mixshard-procs")
        circs, insts, proofs = _parity_batch(rng)
        api = [c.api(i) for c, i in zip(circs, insts)]
        n = sum(len(p) for p in proofs)
        rs = [rng.randrange(1, bn.R) for _ in range(n)]
        bvs = [pkg.BatchVerifier(pkg.ParamsKZG.from_bytes(c.params.to_bytes()), pkg.VerifyingKey.from_bytes(c.vk.to_bytes(F.RAW_BYTES), F.RAW_BYTES), c.mo,
                                 "keccak256" if c.hk == "keccak" else c.hk, device=rank, circuit_instances=c.m) for c in circs]
        mx = pkg.MixedBatchVerifier(bvs)
        if use_exchange:
            assert sharding.connect_channel(mx, rank, world), "CUDA IPC mapping of the peers' windows failed"
        for root in range(world):
            ok, st = sharding.verify_mixed_batch_sharded(mx, proofs, api, rank, world, rlc_scalars=rs, root=root)
            assert ok and all(v == 0 for s in st for v in s)
            if use_exchange and rank == root:
                acc = mx.comm_last_batch_accum()
                q.put((rank, "acc", hashlib.sha256(acc).hexdigest()))
        bad = [list(p) for p in proofs]
        bad[2][3], _ = sim.corrupt(bad[2][3], circs[2].vk, "eval_flip", rng, circs[2].mo, circs[2].m)
        ok, st = sharding.verify_mixed_batch_sharded(mx, bad, api, rank, world, rlc_scalars=rs, root=0)
        (_lo, _hi), per = sharding.mixed_shard([len(p) for p in proofs], rank, world)
        want = [[w.status for w in c.oracle(i[a:b], p[a:b])] for c, i, p, (a, b) in zip(circs, insts, bad, per)]
        assert not ok and st == want
        mx.close()
        [bv.close() for bv in bvs]
        q.put((rank, "ok", None))
    except Exception:  # noqa: BLE001
        import traceback

        q.put((rank, "FAIL: " + traceback.format_exc(), None))
    finally:
        dist.barrier()
        dist.destroy_process_group()


@pytest.mark.gpu
@pytest.mark.parametrize("use_exchange", [True, False], ids=["device_exchange", "library_gather"])
def test_sharded_mix_processes_multi_gpu(pkg, use_exchange):
    import hashlib

    import torch
    import torch.multiprocessing as mp

    world = min(torch.cuda.device_count(), 4)
    if world < 2:
        pytest.skip("needs >= 2 GPUs")
    rng = random.Random("mixshard-procs")
    circs, insts, proofs = _parity_batch(rng)
    n = sum(len(p) for p in proofs)
    rs = [rng.randrange(1, bn.R) for _ in range(n)]
    L, R_, _ok = orc.accumulate(circs[0].params, [w for c, i, p in zip(circs, insts, proofs) for w in c.oracle(i, p)], rs)
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = 29600 + os.getpid() % 200 + (7 if use_exchange else 0)
    procs = [ctx.Process(target=_rank_main, args=(r, world, port, q, use_exchange)) for r in range(world)]
    [p.start() for p in procs]
    res = []
    while sum(1 for r in res if r[1] != "acc") < world:
        res.append(q.get(timeout=900))
    [p.join(timeout=120) for p in procs]
    assert all(r[1] in ("ok", "acc") for r in res), res
    accs = {r[2] for r in res if r[1] == "acc"}
    assert accs == ({hashlib.sha256(enc_point(L) + enc_point(R_)).hexdigest()} if use_exchange else set())
