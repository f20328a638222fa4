"""Multi-params mix against one plain mix per params class, on the same inputs (include/h2v.h "multi-params mixes").

Three arms, alternated pass by pass, the L2 overwritten (h2v_flush_l2 through the lead context) before every timed pass:
  multi       one h2v_mix_verify of a multi-params mix over every class's proofs: one MSM, one pairing check
  sequential  one plain mix (h2v_mix_create) per class, one after the other
  threads     the same plain mixes from one host thread each, concurrently
Every call is timed on the host around the C calls, which return after the statuses are downloaded.  Inputs are pre-packed.
Each circuit is its own params class (its own trapdoor), so a plain mix per class holds one member.  Then, with graphs
off, the device time of the joint MSM and of the pairing stage of one multi call and of each plain mix (h2v_last_timings
of the lead: MSM = rlc_msm, pairing).  Workloads (SHPLONK / Blake2b unless noted, synth.py):
  k2  vm k=10 x 2048 under s, vm k=12 x 2048 under s + 1
  k4  4 x 1024: vm k=10, vm k=12, sh k=8 GWC / Keccak, k18, each under its own trapdoor
The fold key is fixed, so every arm folds with the same coefficients.
Usage: python tools/multi_params_bench.py [--reps 30] [--warmup 3] [--distinct 256] [--out profiles/mparams_bench.jsonl]"""
import argparse
import ctypes
import json
import os
import random
import sys
import time
from concurrent.futures import ThreadPoolExecutor
from importlib import import_module

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))
import __graft_entry__ as entry  # noqa: E402
from mixed_bench import FLUSH_BYTES, FOLD_KEY, Packed, card, pct  # noqa: E402

# (shape, k, n, multiopen, transcript)
WORKLOADS = {
    "k2": [("vm", 10, 2048, "shplonk", "blake2b"), ("vm", 12, 2048, "shplonk", "blake2b")],
    "k4": [("vm", 10, 1024, "shplonk", "blake2b"), ("vm", 12, 1024, "shplonk", "blake2b"), ("sh", 8, 1024, "gwc", "keccak"),
           ("k18", 18, 1024, "shplonk", "blake2b")],
}


def packed_mix(lib, mx, packs):
    counts = (ctypes.c_uint32 * len(packs))(*[p.n for p in packs])
    allp = b"".join(p.pbytes for p in packs)
    alli = b"".join(p.ibytes for p in packs)
    po, io = [0], [0]
    for p in packs:
        po += [po[-1] + v for v in p.po[1:]]
        io += [io[-1] + v for v in p.io[1:]]
    mpo, mio = (ctypes.c_uint64 * len(po))(*po), (ctypes.c_uint64 * len(io))(*io)
    status = (ctypes.c_uint8 * sum(p.n for p in packs))()
    verdict = ctypes.c_int(0)

    def run():
        mx._check(lib.h2v_mix_set_rlc_key(mx._mx, FOLD_KEY))
        mx._check(lib.h2v_mix_verify(mx._mx, counts, allp, mpo, alli, mio, None, 0, status, None, ctypes.byref(verdict)))
        return bool(verdict.value)
    return run


def run_workload(pkg, synth, name, spec, args):
    lib = pkg.load_library()
    s0 = random.Random("mparams-bench-srs").randrange(1, synth.R)
    bvs, packs = [], []
    for i, (shape, k, n, mo, tr) in enumerate(spec):
        s = (s0 + i) % synth.R  # every circuit its own trapdoor: its own params class
        d = min(n, args.distinct)
        if mo == "shplonk" and tr == "blake2b":
            vk_bytes, dlogs = synth.make_vk_bytes(shape, k)
            bv = pkg.BatchVerifier(pkg.ParamsKZG.from_bytes(synth.params_bytes_raw(k, s), pkg.SerdeFormat.RawBytes),
                                   pkg.VerifyingKey.from_bytes(vk_bytes, pkg.SerdeFormat.RawBytes), mo, tr, device=0)
            proofs, insts = synth.synthesize_shplonk_batch(bv, dlogs, s, d, seed=(name, shape, k))
        else:  # (synth.py makes SHPLONK / Blake2b proofs only: the CPU oracle's simulated prover, fewer distinct proofs)
            sys.path.insert(0, os.path.join(ROOT, "oracle"))
            F, sim = import_module("formats"), import_module("prover_sim")
            params, (vk, dl) = sim.make_params(k, s), sim.make_vk(shape, k)
            bv = pkg.BatchVerifier(pkg.ParamsKZG.from_bytes(params.to_bytes()), pkg.VerifyingKey.from_bytes(vk.to_bytes(F.RAW_BYTES), F.RAW_BYTES),
                                   mo, "keccak256" if tr == "keccak" else tr, device=0)
            rng = random.Random(f"{name}-{shape}-{k}")
            d = min(d, 32)
            ints = [sim.random_instances(vk, rng, 10) for _ in range(d)]
            proofs = [sim.simulate_proof(params, vk, dl, s, i, rng, mo, tr) for i in ints]
            insts = [[[v.to_bytes(32, "little") for v in col] for col in i[0]] for i in ints]
        reps = -(-n // d)
        bvs.append(bv)
        packs.append(Packed((proofs * reps)[:n], (insts * reps)[:n]))
    N = sum(p.n for p in packs)
    multi = pkg.MixedBatchVerifier(bvs, multi_params=True)
    assert multi.n_classes == len(bvs)
    plains = [pkg.MixedBatchVerifier([bv]) for bv in bvs]
    run_multi = packed_mix(lib, multi, packs)
    run_plain = [packed_mix(lib, mx, [p]) for mx, p in zip(plains, packs)]
    pool = ThreadPoolExecutor(len(bvs))
    arms = {
        "multi": run_multi,
        "sequential": lambda: all([f() for f in run_plain]),
        "threads": lambda: all(pool.map(lambda f: f(), run_plain)),
    }
    times = {a: [] for a in arms}
    ok = {a: True for a in arms}
    for rep in range(args.warmup + args.reps):
        for a, f in arms.items():
            bvs[0]._check(lib.h2v_flush_l2(bvs[0]._ctx, FLUSH_BYTES))
            bvs[0]._check(lib.h2v_batch_download(bvs[0]._ctx, None))  # waits for the flush
            t0 = time.perf_counter()
            good = f()
            dt = time.perf_counter() - t0
            ok[a] &= good
            if rep >= args.warmup:
                times[a].append(dt)
    pool.shutdown()
    out = {"workload": name, "circuits": [f"{sh} k={k} x {n} {mo}/{tr} (class {i})" for i, (sh, k, n, mo, tr) in enumerate(spec)], "proofs": N,
           "reps": args.reps}
    for a in arms:
        p50, p90 = pct(times[a], 0.5), pct(times[a], 0.9)
        out[a] = {"p50_ms": round(1e3 * p50, 3), "p90_ms": round(1e3 * p90, 3), "proofs_per_s": round(N / p50), "all_accepted": ok[a]}
    # device time per stage, direct launches (median of 5 calls after one warm call)
    for bv in bvs:
        bv.set_graphs(False)

    def stages(f, lead):
        f()
        msm, pair = [], []
        for _ in range(5):
            f()
            t = lead.timings()
            msm.append(t["rlc_msm"])
            pair.append(t["pairing"])
        return round(sorted(msm)[2], 4), round(sorted(pair)[2], 4)
    m_msm, m_pair = stages(run_multi, bvs[0])
    out["multi_stages_ms"] = {"msm": m_msm, "pairing": m_pair}
    per = [stages(f, bv) for f, bv in zip(run_plain, bvs)]
    out["plain_stages_ms"] = {"msm": [m for m, _ in per], "pairing": [p for _, p in per], "msm_sum": round(sum(m for m, _ in per), 4),
                              "pairing_sum": round(sum(p for _, p in per), 4)}
    for mx in plains + [multi]:
        mx.close()
    [bv.close() for bv in bvs]
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=30)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--distinct", type=int, default=256, help="distinct synthesised proofs per circuit (tiled to the batch size)")
    ap.add_argument("--workloads", default="k2,k4")
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    pkg = entry.load_package()
    synth = import_module("halo2_verifier_b200.synth")
    head = card()
    lines = []
    for name in args.workloads.split(","):
        res = {**head, **run_workload(pkg, synth, name, WORKLOADS[name], args)}
        print(json.dumps(res), flush=True)
        lines.append(json.dumps(res))
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
