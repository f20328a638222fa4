"""Rejection attribution against the per-proof oracle, at every level and pass boundary of attribute_impl.

When a fold is rejected, every per-proof status a caller acts on comes from attribute_impl (csrc/kernels.cu).  Its contract
is the reference's (poly/strategy.rs:26-30): re-process every proof separately, so a proof that fails on its own never
comes back H2V_OK, whatever the fold scalars were.  It works in two levels, each in passes of CHUNK checks:
  level 1  sub-batches of H2V_ATTR_SUB proofs (default 16) re-folded through the bucket MSM with coefficients of their own,
           one 2-pair check each; it runs when sub >= 2 and a fold group holds at least 4 sub-batches and splits into them
           evenly
  level 2  every suspect - a proof that passed the earlier stages and sits in a rejected sub-batch (in a rejected fold
           group when level 1 is off) - accumulated and checked alone
Every case compares the statuses with the Python oracle's verify_proof of each proof on its own and, through
h2v_launch_count, which levels ran and how many passes each took, so that a case cannot pass by skipping a level or a
pass.  The inputs tile a few dozen distinct oracle-simulated proofs (vector_mul shape, k = 8) to the batch size, with
corruptions injected at chosen positions; the oracle's results are cached by proof bytes and instances."""
import random

import pytest

import bn254 as bn
import formats as F
import prover_sim as sim
import verifier as orc
from workloads import make_batch

gpu = pytest.mark.gpu
MO, HK = "shplonk", "blake2b"
N_BASE = 32
SEED = 2080
OK, CSF = orc.OK, orc.CONSTRAINT_SYSTEM_FAILURE
CSF_KINDS = ("eval_flip", "point_swap", "wrong_input")
EARLY_KINDS = ("scalar_ge_r", "point_offcurve", "truncate_body", "opening_offcurve", "truncate_opening", "no_instances")

# Launches of attribute_impl, from its code.  Checks per pass of either level:
CHUNK = 1024
# level 2: k_pp_suspects once; per pass k_pp_mul_list, k_pp_reduce_list, k_lines, k_pairing_check, k_pp_status
L2_FIXED, L2_PASS = 1, 5
# level 1: k_rlc_expand, k_rlc_scan, the bucket MSM of the sub-batches (k_shared_reduce, k_msm_digits, k_scan_tiles,
# k_scan_apply, k_bucket_order, k_msm_scatter, k_msm_bucket_sum, k_msm_chunk_reduce: one chunk per window), k_window_combine;
# per pass k_lines, k_pairing_check
L1_FIXED, L1_PASS = 11, 2
DEFAULT_SUB = 16


def cdiv(a, b):
    return -(-a // b)


class Pool:
    """N_BASE accepting proofs and their corrupted variants; entry = (proof bytes, instance columns)"""

    def __init__(self):
        self.params, self.vk, instances, proofs, _rng = make_batch("vm", 8, N_BASE, MO, HK, seed=SEED)
        self.good = [(p, i[0]) for p, i in zip(proofs, instances)]
        self._bad, self._res = {}, {}

    def bad(self, kind, j):
        """proof j % N_BASE made invalid by `kind` (a sim.corrupt kind, a wrong public input, or no instance columns)"""
        key = (kind, j % N_BASE)
        if key not in self._bad:
            proof, cols = self.good[key[1]]
            if kind == "wrong_input":
                cols = [[(cols[0][0] + 1) % bn.R] + list(cols[0][1:])]
            elif kind == "no_instances":
                cols = []
            else:
                proof, _ = sim.corrupt(proof, self.vk, kind, random.Random(f"attr-{kind}-{key[1]}"), MO)
            self._bad[key] = (proof, cols)
        return self._bad[key]

    def result(self, entry):
        key = (entry[0], repr(entry[1]))
        if key not in self._res:
            self._res[key] = orc.verify_proof(self.params, self.vk, [entry[1]], entry[0], MO, HK)
        return self._res[key]

    def statuses(self, entries):
        return [self.result(e).status for e in entries]

    def tile(self, n, inject=(), offset=0):
        """n positions holding good proof (offset + j) % N_BASE, then the (position, kind) injections"""
        out = [self.good[(offset + j) % N_BASE] for j in range(n)]
        for pos, kind in inject:
            out[pos] = self.bad(kind, offset + pos)
        return out


@pytest.fixture(scope="module")
def pool():
    return Pool()


@pytest.fixture(scope="module")
def bvs(pkg, pool):
    """two contexts of the same circuit: two ranks of a sharded batch, or two members of a mixed one"""
    mk = lambda: pkg.BatchVerifier(pkg.ParamsKZG.from_bytes(pool.params.to_bytes()),
                                   pkg.VerifyingKey.from_bytes(pool.vk.to_bytes(F.RAW_BYTES), F.RAW_BYTES), MO, HK, device=0)
    a, b = mk(), mk()
    yield a, b
    a.close()
    b.close()


@pytest.fixture(autouse=True)
def default_knobs(monkeypatch):
    monkeypatch.delenv("H2V_ATTR_SUB", raising=False)
    monkeypatch.delenv("H2V_ATTR_WINDOW", raising=False)


def split(entries):
    return [e[0] for e in entries], [e[1] for e in entries]


class Model:
    """What attribute_impl does with the oracle statuses `want` of one upload of `groups` fold groups (the per-group check
    rejects exactly when the group holds a ConstraintSystemFailure; a sub-batch re-fold likewise)"""

    def __init__(self, want, groups=1, sub=DEFAULT_SUB, accepted=None):
        n = len(want)
        gn = n // groups
        self.accepted = accepted or [CSF not in want[q * gn:(q + 1) * gn] for q in range(groups)]
        looked_at = lambda j: groups == 1 or not self.accepted[j // gn]  # group verdicts gate it only with fold groups
        self.level1 = sub >= 2 and gn >= 4 * sub and gn % sub == 0
        if self.level1:
            self.rejected_subs = sorted({j // sub for j in range(n) if want[j] == CSF and looked_at(j)})
            rej = set(self.rejected_subs)
            self.suspects = sum(1 for j in range(n) if want[j] in (OK, CSF) and j // sub in rej)
            self.passes1 = cdiv(n // sub, CHUNK)
        else:
            self.rejected_subs = []
            self.suspects = sum(1 for j in range(n) if want[j] in (OK, CSF) and looked_at(j))
            self.passes1 = 0
        self.passes2 = cdiv(self.suspects, CHUNK)
        self.launches = (L1_FIXED + L1_PASS * self.passes1 if self.level1 else 0) + L2_FIXED + L2_PASS * self.passes2

    def __repr__(self):
        return (f"level 1 {'on' if self.level1 else 'off'} ({self.passes1} passes, {len(self.rejected_subs)} rejected sub-batches), "
                f"{self.suspects} suspects ({self.passes2} passes), {self.launches} launches")


def check(pool, status, entries, attr_launches, groups=1, sub=DEFAULT_SUB, attributed=True, accepted=None):
    """statuses equal the oracle's; attribute_impl ran (attributed) with the levels and passes of the Model"""
    want = pool.statuses(entries)
    assert status == want, f"statuses differ from the oracle's at {[j for j, (a, b) in enumerate(zip(status, want)) if a != b][:20]}"
    m = Model(want, groups, sub, accepted)
    expect = m.launches if attributed else 0
    assert attr_launches == expect, f"attribution launched {attr_launches} kernels, expected {expect}: {m}"
    return m


_BATCH_LAUNCHES = {}


def run_batch(bv, pool, entries, groups=1, rlc_scalars=None):
    """verify_batch; returns (result, kernels launched by its attribution): the call's launches minus those of an accepted
    batch of the same size and fold groups"""
    n = len(entries)
    key = (id(bv), n, groups)
    if key not in _BATCH_LAUNCHES:
        before = bv.launch_count()
        assert bv.verify_batch(*split(pool.tile(n)), seed=SEED, fold_groups=groups).verdict
        _BATCH_LAUNCHES[key] = bv.launch_count() - before
    before = bv.launch_count()
    res = bv.verify_batch(*split(entries), rlc_scalars=rlc_scalars, seed=None if rlc_scalars else SEED, fold_groups=groups)
    return res, bv.launch_count() - before - _BATCH_LAUNCHES[key]


def run_and_check(bv, pool, entries, groups=1, sub=DEFAULT_SUB, rlc_scalars=None):
    res, attr = run_batch(bv, pool, entries, groups, rlc_scalars)
    want = pool.statuses(entries)
    m = Model(want, groups, sub)
    assert res.group_verdicts == m.accepted and res.verdict == all(m.accepted)
    check(pool, res.status, entries, attr, groups, sub, attributed=not all(m.accepted))
    return m


# ---- (a) fold scalars that cancel two invalid proofs: the re-fold must not inherit the cancellation
def cancellation(pool, n=64, at=0):
    """n copies of proof 0; the same eval_flip of proof 0 at at + 2 and at + 3 with r_(at+3) = r - 1, so that
    c_(at+2) = -c_(at+3) cancels the pair in the batch fold and in a re-fold of its sub-batch [at, at + 16) with the same
    r_i; an eval_flip of proof 1 at at + 40 makes the batch reject"""
    entries = [pool.good[0]] * n
    entries[at + 2] = entries[at + 3] = pool.bad("eval_flip", 0)
    entries[at + 40] = pool.bad("eval_flip", 1)
    rng = random.Random("attr-cancel")
    rs = [rng.randrange(1, bn.R) for _ in range(n)]
    rs[at + 3] = bn.R - 1
    return entries, rs


@pytest.mark.parametrize("at", [0, 40])
def test_cancellation_premise(pool, at):
    """(oracle only) the cases below are meaningful: the batch fold rejects, but the fold of the pair's sub-batch with the
    batch's own r_i accepts, so only a re-fold with independent coefficients finds the pair"""
    entries, rs = cancellation(pool, at + 64, at)
    res = [pool.result(e) for e in entries]
    assert [j for j, r in enumerate(res) if r.status] == [at + 2, at + 3, at + 40]
    assert {r.status for r in res if r.status} == {CSF}
    assert not orc.accumulate(pool.params, res, rs)[2]
    assert orc.accumulate(pool.params, res[at:at + 16], rs[at:at + 16])[2]


@gpu
def test_cancellation_batch(bvs, pool):
    entries, rs = cancellation(pool)
    m = run_and_check(bvs[0], pool, entries, rlc_scalars=rs)
    assert m.level1 and m.rejected_subs == [0, 2]


@gpu
def test_cancellation_in_fold_group(bvs, pool):
    """the pattern in group 1 of G = 2 (r_67 = r - 1); group 0 accepts"""
    entries, rs = cancellation(pool)
    rng = random.Random("attr-cancel-g0")
    m = run_and_check(bvs[0], pool, [pool.good[0]] * 64 + entries, groups=2, rlc_scalars=[rng.randrange(1, bn.R) for _ in range(64)] + rs)
    assert m.accepted == [True, False] and m.rejected_subs == [4, 6]


@gpu
def test_cancellation_in_shard(bvs, pool):
    """global batch of 104 in shards [0, 40) and [40, 104) (hint 64): the pattern at global 42, 43 (r_43 = r - 1) and 80,
    in the second shard, whose sub-batches start at global 40, 56, ..."""
    a, b = bvs
    entries, rs = cancellation(pool, 104, 40)
    proofs, insts = split(entries)
    st0, p0 = a.accumulate_shard(proofs[:40], insts[:40], 0, 104, rlc_scalars=rs, shard_hint=64)
    st1, p1 = b.accumulate_shard(proofs[40:], insts[40:], 40, 104, rlc_scalars=rs, shard_hint=64)
    ok, _ = a.finalize([p0, p1], want_batch_accum=False)
    assert not ok
    for bv, st, sl in ((a, st0, slice(0, 40)), (b, st1, slice(40, 104))):
        before = bv.launch_count()
        got = bv.attribute_shard(st)
        m = check(pool, got, entries[sl], bv.launch_count() - before)
    assert m.level1 and m.rejected_subs == [0, 2]


@gpu
def test_cancellation_in_mixed_member(pkg, bvs, pool):
    """the pattern in member 0 of a two-member mix (the fold runs over the concatenation, r_3 = r - 1)"""
    entries, rs = cancellation(pool)
    rng = random.Random("attr-cancel-mix")
    with pkg.MixedBatchVerifier(list(bvs)) as mx:
        p0, i0 = split(entries)
        p1, i1 = split(pool.tile(16))
        res = mx.verify_batch([p0, p1], [i0, i1], rlc_scalars=rs + [rng.randrange(1, bn.R) for _ in range(16)])
    assert not res.verdict
    assert res.status == [pool.statuses(entries), [OK] * 16]


# ---- (b) positions, default sub-batches of 16
POSITIONS = {
    "first_and_last": lambda n: [(0, "eval_flip"), (n - 1, "point_swap")],
    "sub_batch_boundary": lambda n: [(15, "eval_flip"), (16, "wrong_input")],
    "two_in_one_sub_batch": lambda n: [(33, "eval_flip"), (38, "point_swap")],
    "whole_sub_batch": lambda n: [(16 + i, CSF_KINDS[i % 3]) for i in range(16)],
    "one_in_every_sub_batch": lambda n: [(16 * b + (5 * b) % 16, CSF_KINDS[b % 3]) for b in range(n // 16)],
    "every_proof": lambda n: [(j, (CSF_KINDS + EARLY_KINDS)[j % 9]) for j in range(n)],
    "every_class_in_one_sub_batch": lambda n: [(35 + i, k) for i, k in enumerate(CSF_KINDS + EARLY_KINDS)],
    "earlier_stage_only_sub_batch": lambda n: [(16 + 2 * i, k) for i, k in enumerate(EARLY_KINDS)] + [(n - 10, "eval_flip")],
}


@gpu
@pytest.mark.parametrize("n", [64, 256])
@pytest.mark.parametrize("case", list(POSITIONS))
def test_positions(bvs, pool, n, case):
    entries = pool.tile(n, POSITIONS[case](n))
    want = pool.statuses(entries)
    if case == "every_class_in_one_sub_batch":
        assert sorted(set(want[32:48])) == [0, 1, 2, 3, 4]
    if case == "earlier_stage_only_sub_batch":  # its failures carry no fold terms: the sub-batch accepts, no suspects there
        assert CSF not in want[16:32] and sorted(set(want[16:32])) == [0, 1, 2, 3]
    m = run_and_check(bvs[0], pool, entries)
    assert m.level1
    if case == "earlier_stage_only_sub_batch":
        assert m.rejected_subs == [(n - 10) // 16] and m.suspects == 16


# ---- (c) level-1 eligibility: it runs exactly when the rule says, and the statuses are the oracle's either way
@gpu
@pytest.mark.parametrize("sub", [0, 2, 16, 32])
@pytest.mark.parametrize("n", [48, 63, 64, 65, 80, 128, 1000])
def test_level1_eligibility(bvs, pool, monkeypatch, n, sub):
    monkeypatch.setenv("H2V_ATTR_SUB", str(sub))
    entries = pool.tile(n, [(1, "eval_flip"), (n // 3, "truncate_body"), (n // 2, "point_swap"), (n - 1, "wrong_input")])
    m = run_and_check(bvs[0], pool, entries, sub=sub)
    runs = {0: (), 2: (48, 64, 80, 128, 1000), 16: (64, 80, 128), 32: (128,)}[sub]
    assert m.level1 == (n in runs)


# ---- (d) level-2 pass boundary: 1024 suspects are one pass, 1025 two
SPREAD_64 = list(range(0, 128, 2))  # 64 of the 128 sub-batches of 2048 proofs
SPREAD_65 = [round(t * 127 / 64) for t in range(65)]  # 65 distinct ones, first and last included
LEVEL2 = {
    # (n, H2V_ATTR_SUB, injections, suspects, level-2 passes)
    "1024_suspects": (1024, 0, [(0, "eval_flip"), (511, "point_swap"), (1023, "wrong_input")], 1024, 1),
    "1025_suspects": (1025, 0, [(0, "eval_flip"), (512, "point_swap"), (1024, "wrong_input")], 1025, 2),
    "1025_suspects_all_invalid": (1025, 0, [(j, CSF_KINDS[j % 3]) for j in range(1025)], 1025, 2),
    "64_rejected_sub_batches": (2048, 16, [(16 * b + b % 16, CSF_KINDS[b % 3]) for b in SPREAD_64], 1024, 1),
    "65_rejected_sub_batches": (2048, 16, [(16 * b + b % 16, CSF_KINDS[b % 3]) for b in SPREAD_65], 1040, 2),
    "65_rejected_sub_batches_half_invalid": (2048, 16, [(16 * b + i, CSF_KINDS[i % 3]) for b in SPREAD_65 for i in range(0, 16, 2)], 1040, 2),
    "65_rejected_sub_batches_all_invalid": (2048, 16, [(16 * b + i, CSF_KINDS[i % 3]) for b in SPREAD_65 for i in range(16)], 1040, 2),
}


@gpu
@pytest.mark.parametrize("case", list(LEVEL2))
def test_level2_pass_boundary(bvs, pool, monkeypatch, case):
    """the suspect list is filled through atomics, so which suspects land in the second pass is not known: the invalid
    proofs are spread over the list (in the all_invalid cases every suspect of the second pass is invalid)"""
    n, sub, inject, suspects, passes = LEVEL2[case]
    monkeypatch.setenv("H2V_ATTR_SUB", str(sub))
    m = run_and_check(bvs[0], pool, pool.tile(n, inject), sub=sub)
    assert (m.suspects, m.passes2) == (suspects, passes)


# ---- (e) level-1 pass boundary: sub-batches of 2 over 2080 proofs are 1040 checks, two passes
L1_BOUNDARY_SUBS = {"group1": [1023, 1024, 1039], "group0": [0, 519], "both": [0, 519, 1023, 1024, 1039]}


@gpu
@pytest.mark.parametrize("groups,which", [(1, "both"), (2, "group1"), (2, "group0"), (2, "both")])
def test_level1_pass_boundary(bvs, pool, monkeypatch, groups, which):
    """with G = 2 every group holds 520 sub-batches, so the second pass (sub-batches 1024..1039) reads the verdict of
    group 1; proofs of an accepted group stay OK"""
    monkeypatch.setenv("H2V_ATTR_SUB", "2")
    n = 2080
    inject = [(2 * b + (b % 2), CSF_KINDS[t % 3]) for t, b in enumerate(L1_BOUNDARY_SUBS[which])]
    inject += [(2 * 1030, "opening_offcurve"), (2 * 10 + 1, "scalar_ge_r")]  # earlier-stage failures in both groups
    m = run_and_check(bvs[0], pool, pool.tile(n, inject), groups=groups, sub=2)
    assert m.level1 and m.passes1 == 2 and m.rejected_subs == L1_BOUNDARY_SUBS[which]
    if groups == 2:
        assert m.accepted == {"group1": [True, False], "group0": [False, True], "both": [False, False]}[which]


# ---- (f) fold groups and shards
@gpu
@pytest.mark.parametrize("groups", [2, 4, 8])
def test_fold_group_boundaries(bvs, pool, groups):
    """G groups of 64: invalid proofs on both sides of group boundaries, an earlier-stage failure in an accepted group"""
    gn = 64
    cuts = {2: [1], 4: [2], 8: [3, 7]}[groups]
    inject = [(q * gn + d, k) for q in cuts for d, k in ((-1, "eval_flip"), (0, "point_swap"))]
    inject.append((5, "truncate_opening"))
    m = run_and_check(bvs[0], pool, pool.tile(groups * gn, inject), groups=groups)
    assert not all(m.accepted) and m.accepted.count(False) == 2 * len(cuts)


@gpu
@pytest.mark.parametrize("groups", [2, 4, 8])
def test_uneven_shards_with_fold_groups(bvs, pool, groups):
    """G global batches of 160 in shards [0, 96) and [96, 160) (shard hint 96, global bases 0 and 96): group verdicts from
    finalize_groups, then attribute_shard with them on both ranks; invalid proofs on both sides of the shard boundary of
    every odd global batch, at the last proof of the last one, an earlier-stage failure in global batch 0 (accepted)"""
    a, b = bvs
    gcount, cut = 160, 96
    batches = []
    for q in range(groups):
        inject = [(3, "scalar_ge_r")] if q == 0 else []
        if q % 2:
            inject += [(cut - 1, "eval_flip"), (cut, "wrong_input")]
        if q == groups - 1:
            inject.append((gcount - 1, "point_swap"))
        batches.append(pool.tile(gcount, inject, offset=q))
    want_gv = [CSF not in pool.statuses(e) for e in batches]
    assert want_gv == [q % 2 == 0 and q != groups - 1 for q in range(groups)]
    parts, shards = [], []
    for bv, lo, hi in ((a, 0, cut), (b, cut, gcount)):
        entries = [e for batch in batches for e in batch[lo:hi]]
        st, partial = bv.accumulate_shard(*split(entries), lo, gcount, seed=SEED, shard_hint=cut, fold_groups=groups)
        parts.append(partial)
        shards.append((bv, st, entries))
    gv = a.finalize_groups(parts, groups)
    assert gv == want_gv
    for bv, st, entries in shards:
        before = bv.launch_count()
        got = bv.attribute_shard(st, group_verdicts=gv)
        m = check(pool, got, entries, bv.launch_count() - before, groups=groups, accepted=gv)
        assert m.level1
