"""Grouped mixed batches against the same mixes one call each (include/h2v.h "grouped mixed batches").

Two arms, alternated pass by pass, the L2 overwritten (h2v_flush_l2 through the lead context) before every timed pass:
  groups      one h2v_mix_verify_groups over G groups: every member uploads once, one launch set, G pairing checks
  separate    the same G mixes through G successive h2v_mix_verify calls
Each group is the workload of tools/mixed_bench.py ("small" = 4 circuits x 256, "large" = vm k=10 x 2048 + vm k=12 x 1024
+ k18 x 1024).  Calls are timed on the host around the C call, which returns after the statuses are downloaded; inputs are
pre-packed.  The fold key is fixed.  The "corrupt" line puts one invalid proof (another proof's instances) into group 5 of
16 small groups: attribution then re-checks that group's proofs only.
Usage: python tools/mixed_groups_bench.py [--reps 20] [--warmup 3] [--out FILE]"""
import argparse
import ctypes
import json
import os
import random
import sys
import time
from importlib import import_module

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))
import __graft_entry__ as entry  # noqa: E402
from mixed_bench import FLUSH_BYTES, FOLD_KEY, WORKLOADS, Packed, card, pct  # noqa: E402


def concat(packs):
    """one call's buffers over several Packed, in order"""
    pb = b"".join(p.pbytes for p in packs)
    ib = b"".join(p.ibytes for p in packs)
    po, io = [0], [0]
    for p in packs:
        po += [po[-1] + v for v in p.po[1:]]
        io += [io[-1] + v for v in p.io[1:]]
    return pb, (ctypes.c_uint64 * len(po))(*po), ib, (ctypes.c_uint64 * len(io))(*io), len(po) - 1


def run(pkg, synth, name, G, args, corrupt_group=None):
    lib = pkg.load_library()
    spec = WORKLOADS[name]
    s = random.Random("mixed-bench-srs").randrange(1, synth.R)
    bvs, members = [], []
    for shape, k, n in spec:
        vk_bytes, dlogs = synth.make_vk_bytes(shape, k)
        bv = pkg.BatchVerifier(pkg.ParamsKZG.from_bytes(synth.params_bytes_raw(k, s), pkg.SerdeFormat.RawBytes),
                               pkg.VerifyingKey.from_bytes(vk_bytes, pkg.SerdeFormat.RawBytes), "shplonk", "blake2b", device=0)
        d = min(n, args.distinct)
        proofs, insts = synth.synthesize_shplonk_batch(bv, dlogs, s, d, seed=(name, shape, k))
        reps = -(-n // d)
        bvs.append(bv)
        members.append(((proofs * reps)[:n], (insts * reps)[:n]))
    M = len(spec)
    per_group = []
    for q in range(G):
        packs = []
        for m, (proofs, insts) in enumerate(members):
            insts = list(insts)
            if q == corrupt_group and m == 0:
                insts[0] = insts[1]  # a valid proof under another proof's instances: passes the stages, fails the fold
            packs.append(Packed(proofs, insts))
        per_group.append(packs)
    mx = pkg.MixedBatchVerifier(bvs)
    counts1 = (ctypes.c_uint32 * M)(*[len(p[0]) for p in members])
    calls1 = [concat(packs) for packs in per_group]
    countsG = (ctypes.c_uint32 * (G * M))(*([len(p[0]) for p in members] * G))
    allp = concat([p for packs in per_group for p in packs])
    N = allp[4]
    status = (ctypes.c_uint8 * N)()
    gverd = (ctypes.c_uint8 * G)()
    verdict = ctypes.c_int(0)

    def grouped():
        mx._check(lib.h2v_mix_set_rlc_key(mx._mx, FOLD_KEY))
        mx._check(lib.h2v_mix_verify_groups(mx._mx, G, countsG, allp[0], allp[1], allp[2], allp[3], None, 0, status, gverd, None, ctypes.byref(verdict)))
        return [bool(v) for v in gverd]

    def separate():
        out = []
        for pb, po, ib, io, n in calls1:
            mx._check(lib.h2v_mix_set_rlc_key(mx._mx, FOLD_KEY))
            mx._check(lib.h2v_mix_verify(mx._mx, counts1, pb, po, ib, io, None, 0, status, None, ctypes.byref(verdict)))
            out.append(bool(verdict.value))
        return out

    arms = {"groups": grouped, "separate": separate}
    times = {a: [] for a in arms}
    verdicts = {}
    for rep in range(args.warmup + args.reps):
        for a, f in arms.items():
            bvs[0]._check(lib.h2v_flush_l2(bvs[0]._ctx, FLUSH_BYTES))
            bvs[0]._check(lib.h2v_batch_download(bvs[0]._ctx, None))
            t0 = time.perf_counter()
            v = f()
            dt = time.perf_counter() - t0
            verdicts.setdefault(a, v)
            assert verdicts[a] == v
            if rep >= args.warmup:
                times[a].append(dt)
    mx.close()
    [bv.close() for bv in bvs]
    want = [q != corrupt_group for q in range(G)]
    out = {"workload": name, "groups": G, "per_group": [f"{sh} k={k} x {n}" for sh, k, n in spec], "proofs": N, "reps": args.reps,
           "corrupt_group": corrupt_group}
    for a in arms:
        p50, p90 = pct(times[a], 0.5), pct(times[a], 0.9)
        out[a] = {"p50_ms": round(1e3 * p50, 3), "p90_ms": round(1e3 * p90, 3), "proofs_per_s": round(N / p50),
                  "group_verdicts_as_expected": verdicts[a] == want}
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--distinct", type=int, default=256)
    ap.add_argument("--cases", default="small:1,small:4,small:16,large:1,large:4,small:16:corrupt")
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    pkg = entry.load_package()
    synth = import_module("halo2_verifier_b200.synth")
    head = card()
    lines = []
    for case in args.cases.split(","):
        parts = case.split(":")
        res = {**head, **run(pkg, synth, parts[0], int(parts[1]), args, corrupt_group=5 if len(parts) > 2 else None)}
        print(json.dumps(res), flush=True)
        lines.append(json.dumps(res))
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
