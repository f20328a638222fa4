"""The per-proof stages (decompression, transcript replay, scalar stage) and the plan compiler on random constraint systems
(tests/random_cs.py), at the device code's build limits, and at every byte-level encoding boundary of proof scalars,
instance values and compressed points.  The checker is the Python oracle; the CPU tests run the stages through the host
build (tests/hostlib/libstage.so), the GPU tests through the C ABI."""
import ctypes
import functools
import os
import random

import pytest

import bn254 as bn
import formats as F
import prover_sim as sim
import verifier as orc
from random_cs import LIMIT_ERRORS, limit_vk, random_vk, usable_rows
from workloads import enc_point, oracle_scalars, setup, split32

HERE = os.path.dirname(os.path.abspath(__file__))
MO = {"shplonk": 0, "gwc": 1}
HK = {"blake2b": 0, "keccak": 1}
COMBOS = [(mo, hk) for mo in MO for hk in HK]
SEEDS = range(64)


@pytest.fixture(scope="module")
def stage(built):
    lib = ctypes.CDLL(os.path.join(HERE, "hostlib", "libstage.so"))
    lib.s_err.restype = ctypes.c_char_p
    return lib


# ---------------------------------------------------------------- host harness
class HostPlan:
    """one plan compiled by the host build of plan_build.cpp; verify() runs one proof through the host stages"""

    def __init__(self, stage, params, vk, mo, hk, m=1):
        self.stage = stage
        pb, vb = params.to_bytes(), vk.to_bytes(F.RAW_BYTES)
        self.rc = stage.s_build_m(pb, len(pb), 0, vb, len(vb), F.RAW_BYTES, MO[mo], HK[hk], m)
        self.err = stage.s_err().decode()
        info = (ctypes.c_uint32 * 8)()
        stage.s_info(info)
        _k, self.P, _S, self.C, self.proof_len, self.n_inst_cols, self.nsh, self.nmo = list(info)

    def verify(self, proof, insts, ragged=True):
        """insts [circuit instance][column][row] of ints below 2^256 (not reduced); ragged: pass the column lengths
        (col_len), else the equal split of the values.  Returns (status, challenges, MSM scalars in hook order, (L, R))."""
        cols = [c for inst in insts for c in inst]
        ib = b"".join(int(v).to_bytes(32, "little") for c in cols for v in c)
        tot = sum(len(c) for c in cols)
        col_len = (ctypes.c_uint32 * max(1, len(cols)))(*[len(c) for c in cols]) if ragged else None
        C, P, nsh, nmo = self.C, self.P, self.nsh, self.nmo
        ch = (ctypes.c_uint8 * (32 * C))(); rt = (ctypes.c_uint8 * (32 * P))(); sh = (ctypes.c_uint8 * (32 * nsh))()
        lf = (ctypes.c_uint8 * (32 * nmo))(); LR = (ctypes.c_uint8 * 128)(); ok = ctypes.c_int(0)
        st = self.stage.s_verify_one(proof, len(proof), ib, tot, col_len, len(cols) if ragged else -1, ch, rt, sh, lf, LR, ctypes.byref(ok))
        g = lambda a, i: int.from_bytes(bytes(a[32 * i: 32 * i + 32]), "little")
        pt = lambda i: None if not (g(LR, i) or g(LR, i + 1)) else (g(LR, i), g(LR, i + 1))
        return (st, [g(ch, i) for i in range(C)], [g(rt, i) for i in range(P)] + [g(sh, i) for i in range(nsh)] + [g(lf, i) for i in range(nmo)],
                (pt(0), pt(2)))


def assert_matches_oracle(plan, params, vk, proof, insts, mo, hk, ragged=True, expect=None):
    got = plan.verify(proof, insts, ragged)
    res = orc.verify_proof(params, vk, insts, proof, mo, hk)
    assert got[0] == res.status, res.error
    if expect is not None:
        assert res.status == expect, res.error
    if res.status in (orc.OK, orc.CONSTRAINT_SYSTEM_FAILURE):
        assert got[1] == res.challenges
        assert got[2] == oracle_scalars(vk, res, plan.P, plan.nmo)
        assert got[3] == (res.L, res.R)
    return got, res


# ---------------------------------------------------------------- random constraint systems
@functools.lru_cache(maxsize=None)
def random_case(seed):
    """(params, vk, dlogs, s, m) of seed: k cycles through 4..8, circuit instances per proof m through 1, 2, 3"""
    rng = random.Random(repr(("random-cs", seed)))
    k = 4 + seed % 5
    vk, dl = random_vk(rng, k)
    s = rng.randrange(1, bn.R)
    return sim.make_params(k, s), vk, dl, s, 1 + seed % 3


def ragged_instances(vk, rng, m):
    """per column: empty, the usable maximum n - (blinding_factors + 1), or a length in between"""
    top = usable_rows(vk)
    return [[[rng.randrange(bn.R) for _ in range(rng.choice((0, top, rng.randint(1, top))))] for _ in range(vk.cs.num_instance_columns)]
            for _ in range(m)]


def test_generator_reaches_the_listed_structures():
    """aggregate coverage of the seeds the random tests run"""
    seen = set()
    for seed in SEEDS:
        _p, vk, _dl, _s, _m = random_case(seed)
        cs, n = vk.cs, vk.n
        rots = sim.query_rotations(vk)
        if len(set(rots)) > len({r % n for r in rots}):
            seen.add("collision mod n")
        if -(cs.blinding_factors() + 1) in [r for _c, _p, r in cs.advice_queries]:
            seen.add("user rotation -(bf + 1)")
        chunk, npc = vk.cs_degree - 2, len(cs.permutation_columns)
        if not npc:
            seen.add("no permutation")
        elif chunk > 2:
            seen.add({0: "chunk multiple", 1: "chunk + 1", chunk - 1: "chunk - 1"}.get(npc % chunk, "other"))
        if max(cs.advice_column_phase) == 2:
            seen.add("three phases")
        if len(set(cs.advice_column_phase)) <= max(cs.advice_column_phase):
            seen.add("empty phase")
        ch0 = len(cs.advice_queries) + cs.num_fixed_columns + cs.num_instance_columns
        if any(v >= ch0 for ins, tabs in cs.lookups for p in ins + tabs for _c, vs in p[1] for v, _pw in vs):
            seen.add("challenge in a lookup")
        if any(len(ins) > 1 for ins, _t in cs.lookups):
            seen.add("lookup with several pairs")
        if cs.shuffles:
            seen.add("shuffle")
        seen.add(f"degree {vk.cs_degree}")
        seen.add(f"instance columns {cs.num_instance_columns}")
    want = {"collision mod n", "user rotation -(bf + 1)", "no permutation", "chunk multiple", "chunk + 1", "chunk - 1", "three phases",
            "empty phase", "challenge in a lookup", "lookup with several pairs", "shuffle"}
    want |= {f"degree {d}" for d in range(3, 10)} | {f"instance columns {i}" for i in range(4)}
    assert want <= seen, want - seen


@pytest.mark.parametrize("seed", SEEDS)
def test_random_circuit_stages_match_oracle(stage, seed):
    """statuses, challenges, MSM scalars and (L, R) of the host stages against the oracle under both multi-open schemes
    and both transcript hashes, with ragged instance columns (equal lengths in one combination, given with and without
    the column lengths); every corruption class in one combination of every eighth seed"""
    params, vk, dl, s, m = random_case(seed)
    rng = random.Random(repr(("random-cs-proofs", seed)))
    for c, (mo, hk) in enumerate(COMBOS):
        plan = HostPlan(stage, params, vk, mo, hk, m)
        assert plan.rc == 0, plan.err
        equal = c == seed % 4
        if equal:
            rows = rng.randint(0, usable_rows(vk))
            insts = [sim.random_instances(vk, rng, rows)[0] for _ in range(m)]
        else:
            insts = ragged_instances(vk, rng, m)
        proof = sim.simulate_proof(params, vk, dl, s, insts, rng, mo, hk)
        assert plan.proof_len == len(proof) and plan.n_inst_cols == m * vk.cs.num_instance_columns
        got, _res = assert_matches_oracle(plan, params, vk, proof, insts, mo, hk, expect=orc.OK)
        if equal:
            assert plan.verify(proof, insts, ragged=False) == got
        if seed % 8 == 0 and c == (seed // 8) % 4:
            for kind in sim.CORRUPTIONS:
                bad, exp = sim.corrupt(proof, vk, kind, rng, mo, m)
                assert_matches_oracle(plan, params, vk, bad, insts, mo, hk, expect=exp)


# ---------------------------------------------------------------- build limits
LIMIT_CASES = [("set_points", 1, ("shplonk",)), ("rot", 1, ("gwc", "shplonk")), ("inst_q", 1, ("shplonk", "gwc")),
               ("inst_q", 2, ("shplonk", "gwc")), ("levals", 1, ("shplonk", "gwc"))]


@functools.lru_cache(maxsize=None)
def limit_case(which, at_limit, m):
    vk, dl = limit_vk(which, at_limit, m)
    s = random.Random(repr(("limit-s", which, m))).randrange(1, bn.R)
    return sim.make_params(vk.k, s), vk, dl, s


@pytest.mark.parametrize("which,m,schemes", LIMIT_CASES)
def test_plan_at_and_past_each_build_limit(stage, which, m, schemes):
    """at the limit the plan verifies like the oracle; one past it the plan compiler refuses the VK"""
    params, vk, dl, s = limit_case(which, True, m)
    rng = random.Random(repr(("limit-proofs", which, m)))
    for mo in schemes:
        plan = HostPlan(stage, params, vk, mo, "blake2b", m)
        assert plan.rc == 0, plan.err
        insts = [sim.random_instances(vk, rng, 2)[0] for _ in range(m)]
        proof = sim.simulate_proof(params, vk, dl, s, insts, rng, mo, "blake2b")
        assert_matches_oracle(plan, params, vk, proof, insts, mo, "blake2b", expect=orc.OK)
        bad, exp = sim.corrupt(proof, vk, "eval_flip", rng, mo, m)
        assert_matches_oracle(plan, params, vk, bad, insts, mo, "blake2b", expect=exp)
    params, vk, _dl, _s = limit_case(which, False, m)
    for mo in schemes:
        plan = HostPlan(stage, params, vk, mo, "blake2b", m)
        assert plan.rc != 0 and plan.err.startswith(LIMIT_ERRORS[which]), plan.err


def test_limit_vks_sit_on_the_limits():
    """the structure each limit VK claims: counted with the oracle's own definitions"""
    for at in (True, False):
        d = 0 if at else 1
        _p, vk, _dl, _s = limit_case("set_points", at, 1)
        assert max(len({r % vk.n for c, _ph, r in vk.cs.advice_queries if c == col}) for col in range(vk.cs.num_advice_columns)) == 8 + d
        _p, vk, _dl, _s = limit_case("rot", at, 1)
        assert len({r % vk.n for r in sim.query_rotations(vk)}) == 32 + d
        for m in (1, 2):
            _p, vk, _dl, _s = limit_case("inst_q", at, m)
            assert vk.cs.num_instance_columns * m == 16 + d * m
        _p, vk, _dl, _s = limit_case("levals", at, 1)
        assert vk.cs.blinding_factors() + 2 == 64 + d and len({r % vk.n for r in sim.query_rotations(vk)}) <= 8


# ---------------------------------------------------------------- encoding boundaries
R_, P_ = bn.R, bn.P
SCALAR_EDGES = ([("r-1", R_ - 1), ("r", R_), ("r+1", R_ + 1)] + [(f"r+limb{i}", R_ + (1 << (32 * i))) for i in range(8)] +
                [(f"r-limb{i}", R_ - (1 << (32 * i))) for i in range(8)] + [("2^254", 1 << 254), ("2^255", 1 << 255), ("2^256-1", (1 << 256) - 1)])
FLAGS = {"none": 0, "sign": 0x80, "inf": 0x40, "both": 0xC0}


def _point_edges(valid):
    """(label, 32 bytes) for every x boundary x flag combination, plus variants of the valid encoding `valid`"""
    xs = [("p-1", P_ - 1), ("p", P_), ("p+1", P_ + 1), ("2^254-1", (1 << 254) - 1), ("non-residue", sim._offcurve_x())]
    out = []
    for xn, x in xs:
        for fn, f in FLAGS.items():
            b = bytearray(x.to_bytes(32, "little"))
            b[31] |= f
            out.append((f"x={xn} {fn}", bytes(b)))
    inf = bytearray(valid); inf[31] |= 0x40
    flip = bytearray(valid); flip[31] ^= 0x80
    return out + [("valid x, inf", bytes(inf)), ("valid, sign flipped", bytes(flip)), ("zeros", bytes(32))]


BOUNDARY_SETS = {"blake2b": ("mix", 6, "shplonk"), "keccak": ("mix", 6, "gwc")}


@functools.lru_cache(maxsize=None)
def boundary_cases(hk):
    """(params, vk, mo, [(label, instances, proof, invalid_instances)]) for one transcript hash: the base proof, every
    scalar edge in a pre-multi-open scalar slot and as an instance value, every point edge in a pre-multi-open point slot
    and in an opening slot.  invalid_instances: an instance value >= r, which the oracle (it reduces mod r) has no
    counterpart for: the proof must fail with InvalidInstances whatever else is wrong with it."""
    shape, k, mo = BOUNDARY_SETS[hk]
    params, vk, dl, s = setup(shape, k)
    rng = random.Random(repr(("boundary", hk)))
    inst = sim.random_instances(vk, rng, 5)
    proof = sim.simulate_proof(params, vk, dl, s, inst, rng, mo, hk)
    items, first_mo = sim.proof_layout(vk, mo)
    si, pi = items.index("S"), items.index("P")

    def put(i, b):
        return proof[:32 * i] + b + proof[32 * i + 32:]

    cases = [("base", inst, proof, False)]
    for name, v in SCALAR_EDGES:
        cases.append((f"scalar {name}", inst, put(si, v.to_bytes(32, "little")), False))
        bad_inst = [[list(c) for c in inst[0]]]
        bad_inst[0][0][0] = v
        if v < R_:  # canonical: an accepting proof for these instances
            cases.append((f"instance {name}", bad_inst, sim.simulate_proof(params, vk, dl, s, bad_inst, rng, mo, hk), False))
        else:
            cases.append((f"instance {name}", bad_inst, proof, True))
    nc = [[list(c) for c in inst[0]]]
    nc[0][1][-1] = R_
    cases.append(("instance r (last value) + truncated proof", nc, proof[:100], True))
    cases.append(("instance r (last value) + scalar r", nc, put(si, R_.to_bytes(32, "little")), True))
    cases.append(("instance r (last value) + opening point off-curve", nc, put(first_mo, sim._offcurve_x().to_bytes(32, "little")), True))
    for where, slot in (("pre-multi-open", pi), ("opening", first_mo)):
        for name, b in _point_edges(proof[32 * slot: 32 * slot + 32]):
            cases.append((f"{where} point {name}", inst, put(slot, b), False))
    return params, vk, mo, cases


@pytest.mark.parametrize("hk", list(HK))
def test_encoding_boundaries_on_the_host(stage, hk):
    """scalars at and around r (and with r's top words), every x / flag combination of a compressed point, in transcript
    and opening slots: statuses as the oracle's, values bit-exact where a proof is accepted or reaches the pairing; a
    non-canonical instance value is InvalidInstances, ahead of any transcript or opening error"""
    params, vk, mo, cases = boundary_cases(hk)
    plan = HostPlan(stage, params, vk, mo, hk)
    assert plan.rc == 0, plan.err
    _items, first_mo = sim.proof_layout(vk, mo)
    base = cases[0][2]
    for label, insts, proof, invalid_instances in cases:
        if invalid_instances:
            assert plan.verify(proof, insts)[0] == orc.INVALID_INSTANCES, label
            assert plan.verify(proof, insts, ragged=False)[0] == orc.INVALID_INSTANCES, label
            continue
        (st, *_), _res = assert_matches_oracle(plan, params, vk, proof, insts, mo, hk)
        # the status each edge must produce, from the oracle's decoders
        if label.startswith("scalar"):
            v = dict(SCALAR_EDGES)[label.split()[1]]
            assert st == (orc.TRANSCRIPT if v >= R_ else orc.CONSTRAINT_SYSTEM_FAILURE), label
        elif label.startswith("instance"):
            assert st == orc.OK, label
        elif "point" in label:
            slot = next(i for i in range(len(base) // 32) if proof[32 * i: 32 * i + 32] != base[32 * i: 32 * i + 32])
            ok, pt = bn.g1_from_bytes(proof[32 * slot: 32 * slot + 32])
            if ok and pt is not None:
                assert st == orc.CONSTRAINT_SYSTEM_FAILURE, label
            else:
                assert st == (orc.TRANSCRIPT if slot < first_mo else orc.OPENING), label
        else:
            assert st == orc.OK, label


# ---------------------------------------------------------------- GPU
def _bv(pkg, params, vk, mo, hk, m=1):
    return pkg.BatchVerifier(pkg.ParamsKZG.from_bytes(params.to_bytes()), pkg.VerifyingKey.from_bytes(vk.to_bytes(F.RAW_BYTES), F.RAW_BYTES),
                             mo, "keccak256" if hk == "keccak" else hk, device=0, circuit_instances=m)


@pytest.mark.gpu
@pytest.mark.parametrize("seed", range(16))
def test_random_circuits_on_the_device(pkg, seed):
    """8 proofs with ragged instance columns and two corruptions per batch; the four (multi-open, hash) combinations
    rotate over the seeds, so both transcript kernels (the Blake2b quad replay, the Keccak replay) and both reductions run"""
    from test_gpu_parity import check_against_oracle

    params, vk, dl, s, m = random_case(seed)
    mo, hk = COMBOS[seed % 4]
    rng = random.Random(repr(("random-cs-gpu", seed)))
    insts = [ragged_instances(vk, rng, m) for _ in range(8)]
    proofs = [sim.simulate_proof(params, vk, dl, s, i, rng, mo, hk) for i in insts]
    for j, kind in ((2, sim.CORRUPTIONS[seed % len(sim.CORRUPTIONS)]), (5, "eval_flip")):
        proofs[j], _ = sim.corrupt(proofs[j], vk, kind, rng, mo, m)
    rs = [rng.randrange(1, bn.R) for _ in proofs]
    with _bv(pkg, params, vk, mo, hk, m) as bv:
        res, want = check_against_oracle(bv, params, vk, insts, proofs, mo, hk, rs)
        assert res.status[5] == orc.CONSTRAINT_SYSTEM_FAILURE and res.status.count(orc.OK) >= 6


@pytest.mark.gpu
@pytest.mark.parametrize("which,m,schemes", LIMIT_CASES)
def test_build_limits_on_the_device(pkg, which, m, schemes):
    from test_gpu_parity import check_against_oracle

    params, vk, dl, s = limit_case(which, True, m)
    rng = random.Random(repr(("limit-gpu", which, m)))
    for mo in schemes:
        for hk in HK:
            insts = [[sim.random_instances(vk, rng, 2)[0] for _ in range(m)] for _ in range(4)]
            proofs = [sim.simulate_proof(params, vk, dl, s, i, rng, mo, hk) for i in insts]
            proofs[1], _ = sim.corrupt(proofs[1], vk, "eval_flip", rng, mo, m)
            with _bv(pkg, params, vk, mo, hk, m) as bv:
                res, _ = check_against_oracle(bv, params, vk, insts, proofs, mo, hk, [rng.randrange(1, bn.R) for _ in proofs])
                assert res.status == [0, 4, 0, 0]
    params, vk, _dl, _s = limit_case(which, False, m)
    for mo in schemes:
        with pytest.raises(pkg.BackendError, match=LIMIT_ERRORS[which]):
            _bv(pkg, params, vk, mo, "blake2b", m)


@pytest.mark.gpu
def test_mixed_batch_of_random_circuits(pkg):
    """one mixed batch over 4 random VKs under one params (different point and multi-open counts share the segmented term
    space): statuses and the folded (L, R) against the oracle's AccumulatorStrategy"""
    k, s = 6, sim.FIXTURE_SRS_SECRET
    params = sim.make_params(k, s)
    rng = random.Random("random-cs-mix")
    members = []
    for t, (mo, hk) in enumerate(COMBOS):
        vk, dl = random_vk(random.Random(repr(("random-cs-mix-vk", t))), k)
        insts = [ragged_instances(vk, rng, 1) for _ in range(2 + t)]
        proofs = [sim.simulate_proof(params, vk, dl, s, i, rng, mo, hk) for i in insts]
        members.append((vk, mo, hk, insts, proofs))
    members[1][4][0], _ = sim.corrupt(members[1][4][0], members[1][0], "eval_flip", rng, members[1][1])
    bvs = [_bv(pkg, params, vk, mo, hk) for vk, mo, hk, _i, _p in members]
    try:
        assert len({(bv.n_points, bv.n_mo) for bv in bvs}) > 1
        with pkg.MixedBatchVerifier(bvs) as mx:
            n = sum(len(p) for *_r, p in members)
            rs = [rng.randrange(1, bn.R) for _ in range(n)]
            res = mx.verify_batch([p for *_r, p in members], [[i[0] for i in insts] for *_r, insts, _p in members], rlc_scalars=rs,
                                  want_batch_accum=True)
            want = [[orc.verify_proof(params, vk, i, p, mo, hk) for i, p in zip(insts, proofs)] for vk, mo, hk, insts, proofs in members]
            assert res.status == [[w.status for w in ws] for ws in want] and res.status[1][0] == orc.CONSTRAINT_SYSTEM_FAILURE
            L, R, ok = orc.accumulate(params, [w for ws in want for w in ws], rs)
            assert res.batch_accum == enc_point(L) + enc_point(R) and not ok and not res.verdict
    finally:
        [bv.close() for bv in bvs]


@pytest.mark.gpu
@pytest.mark.parametrize("hk", list(HK))
def test_encoding_boundaries_on_the_device(stage, pkg, hk):
    """every boundary case of test_encoding_boundaries_on_the_host in one batch: statuses equal the host stages', values of
    the proofs that reach the pairing equal the oracle's, and the fold skips every rejected proof"""
    params, vk, mo, cases = boundary_cases(hk)
    plan = HostPlan(stage, params, vk, mo, hk)
    host = [plan.verify(proof, insts)[0] for _l, insts, proof, _b in cases]
    want = [orc.Result(status=orc.INVALID_INSTANCES) if invalid else orc.verify_proof(params, vk, insts, proof, mo, hk)
            for _l, insts, proof, invalid in cases]
    rng = random.Random(repr(("boundary-gpu", hk)))
    rs = [rng.randrange(1, bn.R) for _ in cases]
    with _bv(pkg, params, vk, mo, hk) as bv:
        res = bv.verify_batch([c[2] for c in cases], [c[1][0] for c in cases], rlc_scalars=rs, want_challenges=True, want_accum=True,
                              want_batch_accum=True)
        assert res.status == host, [(c[0], a, b) for c, a, b in zip(cases, res.status, host) if a != b]
        assert res.status == [w.status for w in want]
        C = bv.n_challenges
        for j, w in enumerate(want):
            if w.status in (orc.OK, orc.CONSTRAINT_SYSTEM_FAILURE):
                assert split32(res.challenges[32 * C * j:], C) == w.challenges, cases[j][0]
                assert res.accum[128 * j: 128 * j + 128] == enc_point(w.L) + enc_point(w.R), cases[j][0]
        L, R, _ok = orc.accumulate(params, want, rs)
        assert res.batch_accum == enc_point(L) + enc_point(R)
