"""The lifted GLV geometry of the batch MSM (H2V_MSM_GLV, glv_lift, the phi rows written by the decompression) against the
CPU oracle: statuses, verdicts, group verdicts and batch accumulators bit for bit, with the split forced on and off, with
corrupted proofs so that rejection attribution runs after a GLV pass, and under degenerate bucket loads."""
import pytest

import bn254 as bn
import prover_sim as sim
import verifier as orc
from workloads import enc_point
from test_msm_geometry import Workload, force, times

pytestmark = pytest.mark.gpu
N_COPIES = 1104


@pytest.fixture(scope="module")
def wls(pkg):
    out = {"shplonk-blake2b": Workload(pkg, "shplonk", "blake2b"), "gwc-keccak": Workload(pkg, "gwc", "keccak")}
    yield out
    for wl in out.values():
        wl.bv.close()


def glv(monkeypatch, on):
    force(monkeypatch)
    if on is None:
        monkeypatch.delenv("H2V_MSM_GLV", raising=False)
    else:
        monkeypatch.setenv("H2V_MSM_GLV", str(on))


@pytest.mark.parametrize("name", ["shplonk-blake2b", "gwc-keccak"])
@pytest.mark.parametrize("on", [0, 1])
def test_single_batch_against_oracle(wls, monkeypatch, name, on):
    """batch_accum, verdict, statuses and per-proof accumulators, clean and with a corrupted proof (attribution)"""
    wl = wls[name]
    glv(monkeypatch, on)
    for bad in (False, True):
        wl.check(bad)
        assert wl.bv.msm_glv() == bool(on)


@pytest.mark.parametrize("name", ["shplonk-blake2b", "gwc-keccak"])
@pytest.mark.parametrize("on", [None, 0, 1])
def test_fold_groups_against_oracle(wls, monkeypatch, name, on):
    """three fold groups, some holding the corrupted proof: each group's verdict and statuses equal its own oracle batch"""
    wl = wls[name]
    glv(monkeypatch, on)
    for pattern in ((False, True, False), (True, False, True), (False, False, False)):
        pr = sum(((wl.bad if b else wl.proofs) for b in pattern), [])
        res = wl.bv.verify_batch(pr, wl.insts * 3, rlc_scalars=wl.rs * 3, fold_groups=3)
        if on is not None:
            assert wl.bv.msm_glv() == bool(on)
        assert res.group_verdicts == [wl.ok[b] for b in pattern]
        assert res.status == sum(([w.status for w in wl.want[b]] for b in pattern), [])


def test_model_choice(wls, monkeypatch):
    """the model: plain windows for a single batch and under forced windows; the launch-set choice is the same on every
    call (sharded ranks derive it from the same shape)"""
    wl = wls["shplonk-blake2b"]
    glv(monkeypatch, None)
    wl.check(False)
    assert not wl.bv.msm_glv()
    res = [wl.bv.verify_batch(wl.proofs * 2, wl.insts * 2, rlc_scalars=wl.rs * 2, fold_groups=2) for _ in range(2)]
    first = wl.bv.msm_glv(), wl.bv.msm_geometry()
    wl.bv.verify_batch(wl.proofs * 2, wl.insts * 2, rlc_scalars=wl.rs * 2, fold_groups=2)
    assert (wl.bv.msm_glv(), wl.bv.msm_geometry()) == first
    assert all(r.group_verdicts == [True, True] for r in res)
    monkeypatch.setenv("H2V_MSM_GLV", "1")
    monkeypatch.setenv("H2V_MSM_WINDOW_RIGHT", "9")
    wl.bv.verify_batch(wl.proofs * 2, wl.insts * 2, rlc_scalars=wl.rs * 2, fold_groups=2)
    assert not wl.bv.msm_glv()


def test_graph_replay_matches_direct_launches(wls, monkeypatch):
    wl = wls["gwc-keccak"]
    glv(monkeypatch, 1)
    try:
        for graphs in (True, False, True):
            wl.bv.set_graphs(graphs)
            for bad in (False, True):
                wl.check(bad)
                assert wl.bv.msm_glv()
    finally:
        wl.bv.set_graphs(True)


@pytest.fixture(scope="module")
def one_proof(wls):
    wl = wls["shplonk-blake2b"]
    w1 = wl.want[False][0]
    assert w1.status == orc.OK
    return wl, w1


def test_identical_proofs_fill_single_buckets(one_proof, monkeypatch):
    """r_i = 1: every copy of a term has the same scalar; the lift (hashed from the term id) spreads the copies, and P and
    phi(P) of one term can meet in one bucket.  Then one copy flipped: rejected and attributed to exactly that copy."""
    wl, w1 = one_proof
    glv(monkeypatch, 1)
    n = N_COPIES
    proofs, insts = [wl.proofs[0]] * n, [wl.insts[0]] * n
    res = wl.bv.verify_batch(proofs, insts, rlc_scalars=[1] * n, want_batch_accum=True)
    assert wl.bv.msm_glv()
    assert res.verdict and res.status == [0] * n
    assert res.batch_accum == times(w1.L, n) + times(w1.R, n)
    bad, bad_insts = list(proofs), list(insts)
    bad[700], bad_insts[700] = wl.bad[2], wl.insts[2]
    res = wl.bv.verify_batch(bad, bad_insts, rlc_scalars=[1] * n)
    assert not res.verdict and [j for j, s in enumerate(res.status) if s] == [700]


def test_alternating_fold_scalars_cancel(one_proof, monkeypatch):
    wl, w1 = one_proof
    glv(monkeypatch, 1)
    for n in (N_COPIES, N_COPIES - 1):
        res = wl.bv.verify_batch([wl.proofs[0]] * n, [wl.insts[0]] * n, rlc_scalars=[bn.R - 1] * n, want_batch_accum=True)
        assert wl.bv.msm_glv()
        assert res.verdict and res.status == [0] * n
        assert res.batch_accum == (bytes(128) if n % 2 == 0 else enc_point(w1.L) + enc_point(w1.R))
