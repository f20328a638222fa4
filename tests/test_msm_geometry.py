"""The bucket MSM at every window geometry, under degenerate bucket loads, and with degenerate caller fold scalars.

The verdict of every batch path rests on one device pipeline (digits, scan / order / scatter into buckets, bucket sums with
1, 2 or 4 lanes or the GLV variant, chunk and window reduction, window grouping before the pairing) whose shape is chosen at
run time from the batch size: c in 4..15 per channel, chunk m in {2, 4, 8}, the lanes per bucket, the line run.  A bug that
shows at one geometry only would pass tests that run the default geometry of a few batch sizes, so here the geometry is
forced through the tuning knobs and every configuration is compared bit for bit with the CPU oracle.  Knobs read at call
time are set per test; knobs a process reads once run in child processes.  Every test that forces windows checks through
msm_geometry() that they took effect."""
import ctypes
import json
import os
import subprocess
import sys

import pytest

import bn254 as bn
import formats as F
import prover_sim as sim
import verifier as orc
from workloads import enc_point, make_batch

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
FOLD_ERR = "fold scalars must be canonical and non-zero"


def windows(c):
    return (255 + c - 1) // c


def geometry(bv):
    g = bv.msm_geometry()
    return (g["window_bits"] & 0xFFFF, g["window_bits"] >> 16), (g["windows"] & 0xFFFF, g["windows"] >> 16)


def assert_geometry(bv, c0, c1):
    assert geometry(bv) == ((c0, c1), (windows(c0), windows(c1))), "a forced window size did not take effect"


def force(monkeypatch, right=None, left=None, chunk=None):
    for name, v in (("H2V_MSM_WINDOW_RIGHT", right), ("H2V_MSM_WINDOW_LEFT", left), ("H2V_MSM_CHUNK", chunk)):
        if v is None:
            monkeypatch.delenv(name, raising=False)
        else:
            monkeypatch.setenv(name, str(v))


class Workload:
    """n seeded VM k = 8 proofs with their oracle results, and the same batch with one eval_flip proof; the oracle results
    do not depend on the geometry, so every configuration is checked against the same expected bytes"""

    def __init__(self, pkg, mo, hk, n=6, seed=1, flip=(2,)):
        self.mo, self.hk = mo, hk
        self.params, self.vk, instances, self.proofs, rng = make_batch("vm", 8, n, mo, hk, seed=seed)
        self.insts = [i[0] for i in instances]
        self.rs = [rng.randrange(1, bn.R) for _ in range(n)]
        self.bad = list(self.proofs)
        for j in flip:
            self.bad[j], _ = sim.corrupt(self.proofs[j], self.vk, "eval_flip", rng, mo)
        self.want, self.folded, self.ok = {}, {}, {}
        for key, pr in ((False, self.proofs), (True, self.bad)):
            w = [orc.verify_proof(self.params, self.vk, inst, p, mo, hk) for inst, p in zip(instances, pr)]
            L, R_, ok = orc.accumulate(self.params, w, self.rs)
            self.want[key], self.folded[key], self.ok[key] = w, enc_point(L) + enc_point(R_), ok
        assert self.ok[False] and not self.ok[True]
        vkfmt = F.RAW_BYTES if mo == "shplonk" else F.PROCESSED
        self.bv = pkg.BatchVerifier(pkg.ParamsKZG.from_bytes(self.params.to_bytes()), pkg.VerifyingKey.from_bytes(self.vk.to_bytes(vkfmt), vkfmt),
                                    mo, "keccak256" if hk == "keccak" else hk, device=0)

    def check(self, bad):
        """batch_accum, verdict, statuses and per-proof accumulators bit-exact against the oracle"""
        res = self.bv.verify_batch(self.bad if bad else self.proofs, self.insts, rlc_scalars=self.rs, want_accum=True, want_batch_accum=True)
        want = self.want[bad]
        assert res.status == [w.status for w in want]
        for j, w in enumerate(want):
            if w.status in (orc.OK, orc.CONSTRAINT_SYSTEM_FAILURE):
                assert res.accum[128 * j: 128 * j + 128] == enc_point(w.L) + enc_point(w.R), f"accumulators of proof {j}"
        assert res.batch_accum == self.folded[bad]
        assert res.verdict == self.ok[bad] and res.group_verdicts == [self.ok[bad]]
        return res


@pytest.fixture(scope="module")
def workloads(pkg):
    wls = {"shplonk-blake2b": Workload(pkg, "shplonk", "blake2b"), "gwc-keccak": Workload(pkg, "gwc", "keccak")}
    yield wls
    for wl in wls.values():
        wl.bv.close()


@pytest.fixture(scope="module")
def default_windows(workloads):
    """the window sizes the model picks for these batches when nothing is forced"""
    out = {}
    saved = {k: os.environ.pop(k) for k in ("H2V_MSM_WINDOW_RIGHT", "H2V_MSM_WINDOW_LEFT", "H2V_MSM_CHUNK") if k in os.environ}
    try:
        for name, wl in workloads.items():
            wl.check(False)
            out[name] = geometry(wl.bv)[0]
    finally:
        os.environ.update(saved)
    return out


# ---- (a) window sweep: each channel over c = 4..15 with the other at its default, equal pairs, every chunk size
SWEEP = ([("right", c, None) for c in range(4, 16)] + [("left", c, None) for c in range(4, 16)] + [("both", c, None) for c in (4, 5, 15)]
         + [("both", c, m) for c in (4, 9, 15) for m in (2, 4, 8)])


@pytest.mark.parametrize("name", ["shplonk-blake2b", "gwc-keccak"])
@pytest.mark.parametrize("chan,c,m", SWEEP, ids=[f"{ch}{c}" + (f"-m{m}" if m else "") for ch, c, m in SWEEP])
def test_window_sweep(workloads, default_windows, monkeypatch, name, chan, c, m):
    wl = workloads[name]
    d0, d1 = default_windows[name]
    c0, c1 = (c if chan in ("right", "both") else d0), (c if chan in ("left", "both") else d1)
    force(monkeypatch, right=c if chan != "left" else None, left=c if chan != "right" else None, chunk=m)
    for bad in (False, True):
        wl.check(bad)
        assert_geometry(wl.bv, c0, c1)


# ---- (b) geometry-dependent paths at forced windows
@pytest.mark.parametrize("c0,c1", [(4, 15), (13, 6)])
def test_fold_groups_at_forced_windows(workloads, monkeypatch, c0, c1):
    """two fold groups in one launch set (line run 8): each group's verdict and statuses equal its own oracle batch"""
    wl = workloads["shplonk-blake2b"]
    force(monkeypatch, right=c0, left=c1)
    for first, second in ((False, True), (True, False)):
        pr = (wl.bad if first else wl.proofs) + (wl.bad if second else wl.proofs)
        res = wl.bv.verify_batch(pr, wl.insts * 2, rlc_scalars=wl.rs * 2, fold_groups=2)
        assert_geometry(wl.bv, c0, c1)
        assert res.group_verdicts == [wl.ok[first], wl.ok[second]]
        assert res.status == [w.status for w in wl.want[first] + wl.want[second]]


def test_two_shards_fill_every_window_slot(pkg, workloads, monkeypatch):
    """c = 4 on both channels is 64 + 64 windows: the whole H2V_PARTIAL_BYTES blob.  Two shards finalized together equal the
    whole batch and the oracle, accepted and rejected"""
    wl = workloads["shplonk-blake2b"]
    force(monkeypatch, right=4, left=4)
    n = len(wl.proofs)
    for bad in (False, True):
        pr = wl.bad if bad else wl.proofs
        whole = wl.check(bad)
        assert_geometry(wl.bv, 4, 4)
        parts = []
        for lo, hi in ((0, n // 2), (n // 2, n)):
            st, part = wl.bv.accumulate_shard(pr[lo:hi], wl.insts[lo:hi], lo, n, rlc_scalars=wl.rs)
            assert_geometry(wl.bv, 4, 4)
            assert len(part) == pkg.load_library().h2v_partial_bytes()
            parts.append(part)
        ok, folded = wl.bv.finalize(parts)
        assert folded == whole.batch_accum == wl.folded[bad] and ok == wl.ok[bad]


@pytest.mark.parametrize("c", [4, 15])
def test_single_proof_at_forced_windows(workloads, monkeypatch, c):
    wl = workloads["gwc-keccak"]
    force(monkeypatch, right=c, left=c)
    for pr, inst, want in ((wl.proofs[0], wl.insts[0], wl.want[False][0]), (wl.bad[2], wl.insts[2], wl.want[True][2])):
        st = ctypes.c_uint8(9)
        ib = b"".join(bn.fr_to_repr(v) for col in inst for v in col)
        assert wl.bv.lib.h2v_verify_proof(wl.bv._ctx, pr, len(pr), ib, len(ib) // 32, ctypes.byref(st)) == 0
        assert st.value == want.status
        assert_geometry(wl.bv, c, c)


# ---- (c) attribution level 1 (sub-batches through the GLV bucket MSM) at small n
@pytest.fixture(scope="module")
def attribution_batch(pkg):
    wl = Workload(pkg, "shplonk", "blake2b", n=16, seed=7, flip=(4, 5, 13))  # two in one sub-batch, one in another
    yield wl
    wl.bv.close()


@pytest.mark.parametrize("sub", [2, 4])
@pytest.mark.parametrize("attr_c", range(3, 9))
def test_attribution_sub_batches(attribution_batch, monkeypatch, sub, attr_c):
    wl = attribution_batch
    force(monkeypatch, right=7, left=10)
    monkeypatch.setenv("H2V_ATTR_SUB", str(sub))
    monkeypatch.setenv("H2V_ATTR_WINDOW", str(attr_c))
    res = wl.check(True)
    assert_geometry(wl.bv, 7, 10)
    assert [j for j, s in enumerate(res.status) if s] == [4, 5, 13]


# ---- (d) knobs a process reads once: a child process per combination runs the check of (a) at two geometries
CHILD = r"""
import json, os, sys
sys.path.insert(0, sys.argv[1])
import __graft_entry__ as g
pkg = g.load_package()
job = json.load(open(sys.argv[2]))
with pkg.BatchVerifier(pkg.ParamsKZG.from_bytes(bytes.fromhex(job["params"])), pkg.VerifyingKey.from_bytes(bytes.fromhex(job["vk"])), device=0) as bv:
    for c0, c1 in job["geometries"]:
        os.environ["H2V_MSM_WINDOW_RIGHT"], os.environ["H2V_MSM_WINDOW_LEFT"] = str(c0), str(c1)
        for run in job["runs"]:
            res = bv.verify_batch([bytes.fromhex(p) for p in run["proofs"]], job["insts"], rlc_scalars=job["rs"], want_accum=True,
                                  want_batch_accum=True)
            gm = bv.msm_geometry()
            assert (gm["window_bits"] & 0xFFFF, gm["window_bits"] >> 16) == (c0, c1), gm
            assert res.status == run["status"], (c0, c1, res.status)
            assert res.batch_accum.hex() == run["folded"], (c0, c1)
            for j, a in enumerate(run["accum"]):
                assert a is None or res.accum[128 * j: 128 * j + 128].hex() == a, (c0, c1, j)
            assert res.verdict == run["ok"]
print("child ok")
"""
ONCE = [(lanes, run, seg) for lanes in (1, 4) for run in (1, 3) for seg in (False, True)]


@pytest.fixture(scope="module")
def child_job(workloads, tmp_path_factory):
    wl = workloads["shplonk-blake2b"]
    runs = []
    for bad in (False, True):
        acc = [enc_point(w.L).hex() + enc_point(w.R).hex() if w.status in (orc.OK, orc.CONSTRAINT_SYSTEM_FAILURE) else None for w in wl.want[bad]]
        runs.append({"proofs": [p.hex() for p in (wl.bad if bad else wl.proofs)], "status": [w.status for w in wl.want[bad]],
                     "folded": wl.folded[bad].hex(), "accum": acc, "ok": wl.ok[bad]})
    job = {"params": wl.params.to_bytes().hex(), "vk": wl.vk.to_bytes(F.RAW_BYTES).hex(), "insts": wl.insts, "rs": wl.rs,
           "geometries": [[4, 4], [15, 11]], "runs": runs}
    path = tmp_path_factory.mktemp("msm-once") / "job.json"
    path.write_text(json.dumps(job))
    return str(path)


@pytest.mark.parametrize("lanes,run,seg_off", ONCE, ids=[f"lanes{a}-run{b}" + ("-segoff" if s else "") for a, b, s in ONCE])
def test_process_knobs_in_child(child_job, lanes, run, seg_off):
    env = {k: v for k, v in os.environ.items() if not k.startswith("H2V_")}
    env.update(H2V_BUCKET_LANES=str(lanes), H2V_LINE_RUN=str(run))
    if seg_off:
        env["H2V_MILLER_SEGMENTS_OFF"] = "1"
    out = subprocess.run([sys.executable, "-c", CHILD, ROOT, child_job], env=env, cwd=ROOT, capture_output=True, text=True, timeout=300)
    assert out.returncode == 0 and "child ok" in out.stdout, out.stdout[-2000:] + out.stderr[-4000:]


# ---- (e) degenerate bucket loads through caller fold scalars: n copies of one proof, expected values in closed form
N_COPIES = 1104  # 69 attribution sub-batches of 16


@pytest.fixture(scope="module")
def one_proof(workloads):
    wl = workloads["shplonk-blake2b"]
    w1, wbad = wl.want[False][0], wl.want[True][2]
    assert w1.status == orc.OK and wbad.status == orc.CONSTRAINT_SYSTEM_FAILURE
    return wl, w1


def times(pt, k):
    return enc_point(bn.g1_mul(pt, k % bn.R) if pt is not None else None)


@pytest.mark.parametrize("c", [5, 15, 4, 8])
def test_identical_proofs_fill_single_buckets(one_proof, monkeypatch, c):
    """r_i = 1: every c_j = 1, so at Z = 1 (c = 5, 15) every copy of a term has the same digits and each used bucket holds n
    copies of one point (P + P in the bucket sums, equal halves in the 2-lane combine, the size bins saturate at 1023); at
    c = 4, 8 (Z = 2) two digit patterns.  Then one copy flipped: rejected, and level 1 of attribution runs GLV buckets of
    equal points and must name exactly that copy."""
    wl, w1 = one_proof
    force(monkeypatch, right=c, left=c)
    n = N_COPIES
    proofs, insts = [wl.proofs[0]] * n, [wl.insts[0]] * n
    res = wl.bv.verify_batch(proofs, insts, rlc_scalars=[1] * n, want_batch_accum=True)
    assert_geometry(wl.bv, c, c)
    assert res.verdict and res.status == [0] * n
    assert res.batch_accum == times(w1.L, n) + times(w1.R, n)
    bad = list(proofs)
    bad[700] = wl.bad[2]
    bad_insts = list(insts)
    bad_insts[700] = wl.insts[2]
    res = wl.bv.verify_batch(bad, bad_insts, rlc_scalars=[1] * n)
    assert not res.verdict and [j for j, s in enumerate(res.status) if s] == [700] and res.status[700] == orc.CONSTRAINT_SYSTEM_FAILURE


@pytest.mark.parametrize("c", [5, 15])
def test_alternating_fold_scalars_cancel(one_proof, monkeypatch, c):
    """r_i = r - 1 = -1: c_j = (-1)^(n-1-j), so n copies fold to the identity for n even (accepted) and to (L_1, R_1) for n odd"""
    wl, w1 = one_proof
    force(monkeypatch, right=c, left=c)
    for n in (N_COPIES, N_COPIES - 1):
        res = wl.bv.verify_batch([wl.proofs[0]] * n, [wl.insts[0]] * n, rlc_scalars=[bn.R - 1] * n, want_batch_accum=True)
        assert_geometry(wl.bv, c, c)
        assert res.verdict and res.status == [0] * n
        assert res.batch_accum == (bytes(128) if n % 2 == 0 else enc_point(w1.L) + enc_point(w1.R))


# ---- caller fold scalars must be canonical and non-zero
BAD_SCALARS = {"zero": 0, "r": bn.R, "r+5": bn.R + 5}


@pytest.mark.parametrize("what", list(BAD_SCALARS))
def test_bad_fold_scalars_refused_everywhere(pkg, workloads, what):
    """every entry point that takes caller fold scalars refuses a list with one zero or non-canonical entry before any device
    call (the launch count does not move), and the contexts then verify a good batch normally"""
    wl, wg = workloads["shplonk-blake2b"], workloads["gwc-keccak"]
    bv, n = wl.bv, len(wl.proofs)
    rs = list(wl.rs)
    rs[3] = BAD_SCALARS[what]
    before = (bv.launch_count(), wg.bv.launch_count())
    # C ABI
    pbytes, poff, ibytes, ioff, _keep = bv._pack(wl.proofs, wl.insts)
    rb = b"".join(r.to_bytes(32, "little") for r in rs)
    st = (ctypes.c_uint8 * n)()
    assert bv.lib.h2v_verify_batch(bv._ctx, n, pbytes, poff, ibytes, ioff, rb, 0, st, None, None, None) == -1
    assert bv.lib.h2v_last_error(bv._ctx).decode() == FOLD_ERR
    # Python: batch, fold groups (the bad scalar in the second group), shard (scalars of the whole global batch)
    with pytest.raises(pkg.BackendError, match=FOLD_ERR):
        bv.verify_batch(wl.proofs, wl.insts, rlc_scalars=rs)
    with pytest.raises(pkg.BackendError, match=FOLD_ERR):
        bv.verify_batch(wl.proofs * 2, wl.insts * 2, rlc_scalars=wl.rs + rs, fold_groups=2)
    with pytest.raises(pkg.BackendError, match=FOLD_ERR):
        bv.accumulate_shard(wl.proofs[:3], wl.insts[:3], 0, n, rlc_scalars=rs)
    # mixed batch: the scalars of the whole concatenation, refused before any member is uploaded
    with pkg.MixedBatchVerifier([bv, wg.bv]) as mx:
        with pytest.raises(pkg.BackendError, match=FOLD_ERR):
            mx.verify_batch([wl.proofs, wg.proofs], [wl.insts, wg.insts], rlc_scalars=wl.rs + rs[::-1])
        assert (bv.launch_count(), wg.bv.launch_count()) == before
        good = mx.verify_batch([wl.proofs, wg.proofs], [wl.insts, wg.insts], rlc_scalars=wl.rs + wg.rs)
        assert good.verdict
    # accumulator: absorb (upload) and merge, through Python and the C ABI
    with pkg.Accumulator(bv) as acc:
        before = bv.launch_count()
        with pytest.raises(pkg.BackendError, match=FOLD_ERR):
            acc.absorb(bv, wl.proofs, wl.insts, rlc_scalars=rs)
        with pytest.raises(pkg.BackendError, match=FOLD_ERR):
            acc.merge(bytes(128), r=BAD_SCALARS[what])
        assert acc.lib.h2v_acc_merge(acc._acc, bytes(128), BAD_SCALARS[what].to_bytes(32, "little")) == -1
        assert acc.lib.h2v_acc_last_error(acc._acc).decode() == FOLD_ERR
        assert bv.launch_count() == before
        assert acc.absorb(bv, wl.proofs, wl.insts, rlc_scalars=wl.rs).statuses == [0] * n
        acc.merge(acc.to_bytes(), r=5)
        assert acc.finalize().verdict
    before = bv.launch_count()
    with pytest.raises(pkg.BackendError, match=FOLD_ERR):
        bv.verify_batch(wl.proofs, wl.insts, rlc_scalars=rs)
    assert bv.launch_count() == before
    wl.check(True)


def test_zero_fold_scalar_cannot_mask_an_invalid_proof(pkg):
    """64 proofs, ConstraintSystemFailure at 2 and 40, r_5 = 0: c_j = 0 for every j < 5, so proof 2 would drop out of the
    batch fold and out of the re-fold of its attribution sub-batch and be reported OK.  Such scalars are refused; with
    valid scalars the statuses are the oracle's"""
    wl = Workload(pkg, "shplonk", "blake2b", n=64, seed=11, flip=(2, 40))
    try:
        expect = [w.status for w in wl.want[True]]
        assert expect[2] == expect[40] == orc.CONSTRAINT_SYSTEM_FAILURE and expect.count(0) == 62
        rs = list(wl.rs)
        rs[5] = 0
        before = wl.bv.launch_count()
        with pytest.raises(pkg.BackendError, match=FOLD_ERR):
            wl.bv.verify_batch(wl.bad, wl.insts, rlc_scalars=rs)
        assert wl.bv.launch_count() == before
        assert wl.bv.verify_batch(wl.bad, wl.insts, rlc_scalars=wl.rs).status == expect
    finally:
        wl.bv.close()
