"""Mixed batch against separate batches, on the same inputs (include/h2v.h "mixed batches").

Three arms, alternated pass by pass, the L2 overwritten (h2v_flush_l2 through the lead context) before every timed pass:
  mixed       one h2v_mix_verify over every circuit's proofs: one MSM, one pairing check
  sequential  one h2v_verify_batch per circuit, one after the other, one context each
  threads     the same calls from one host thread per context, concurrently
Every call is timed on the host around the C call, which returns after the statuses are downloaded.  Inputs are
pre-packed, so the times are the library's, not the Python packing.  Workloads (SHPLONK / Blake2b, synth.py, one trapdoor
for every circuit so that the params agree): "large" = vm k=10 x 2048 + vm k=12 x 1024 + k18 x 1024, "small" = 4 circuits
x 256 (fixed costs dominate).  The fold key is fixed, so every arm folds with the same coefficients.
Usage: python tools/mixed_bench.py [--reps 30] [--warmup 3] [--distinct 256] [--out FILE]"""
import argparse
import ctypes
import json
import os
import random
import subprocess
import sys
import time
from concurrent.futures import ThreadPoolExecutor
from importlib import import_module

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import __graft_entry__ as entry  # noqa: E402

WORKLOADS = {
    "large": [("vm", 10, 2048), ("vm", 12, 1024), ("k18", 18, 1024)],
    "small": [("vm", 10, 256), ("vm", 12, 256), ("vm", 14, 256), ("k18", 18, 256)],
}
FOLD_KEY = bytes(range(7, 39))
FLUSH_BYTES = 256 << 20  # twice the 126 MB L2


def card():
    q = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True)
    name, _, power = q.stdout.strip().partition(",")
    return {"card": name.strip(), "power_limit": power.strip()}


class Packed:
    def __init__(self, proofs, instances):
        self.n = len(proofs)
        self.pbytes = b"".join(proofs)
        self.ibytes = b"".join(v for inst in instances for col in inst for v in col)
        po, io = [0], [0]
        for p, inst in zip(proofs, instances):
            po.append(po[-1] + len(p))
            io.append(io[-1] + sum(len(c) for c in inst))
        self.po, self.io = po, io
        self.poff = (ctypes.c_uint64 * len(po))(*po)
        self.ioff = (ctypes.c_uint64 * len(io))(*io)
        self.status = (ctypes.c_uint8 * self.n)()


def pct(xs, q):
    xs = sorted(xs)
    return xs[min(len(xs) - 1, int(round(q * (len(xs) - 1))))]


def run_workload(pkg, synth, name, spec, args):
    lib = pkg.load_library()
    s = random.Random("mixed-bench-srs").randrange(1, synth.R)  # one trapdoor: (g, g2, s_g2) agree for every k
    bvs, packs = [], []
    for shape, k, n in spec:
        vk_bytes, dlogs = synth.make_vk_bytes(shape, k)
        bv = pkg.BatchVerifier(pkg.ParamsKZG.from_bytes(synth.params_bytes_raw(k, s), pkg.SerdeFormat.RawBytes),
                               pkg.VerifyingKey.from_bytes(vk_bytes, pkg.SerdeFormat.RawBytes), "shplonk", "blake2b", device=0)
        d = min(n, args.distinct)
        proofs, insts = synth.synthesize_shplonk_batch(bv, dlogs, s, d, seed=(name, shape, k))
        reps = -(-n // d)
        bvs.append(bv)
        packs.append(Packed((proofs * reps)[:n], (insts * reps)[:n]))
    N = sum(p.n for p in packs)
    mx = pkg.MixedBatchVerifier(bvs)
    counts = (ctypes.c_uint32 * len(packs))(*[p.n for p in packs])
    allp = b"".join(p.pbytes for p in packs)
    alli = b"".join(p.ibytes for p in packs)
    po, io = [0], [0]
    for p in packs:
        po += [po[-1] + v for v in p.po[1:]]
        io += [io[-1] + v for v in p.io[1:]]
    mpo, mio = (ctypes.c_uint64 * len(po))(*po), (ctypes.c_uint64 * len(io))(*io)
    mstatus = (ctypes.c_uint8 * N)()
    verdict = ctypes.c_int(0)

    def one(i):
        bv, p = bvs[i], packs[i]
        bv._check(lib.h2v_batch_set_rlc_key(bv._ctx, FOLD_KEY))
        bv._check(lib.h2v_verify_batch(bv._ctx, p.n, p.pbytes, p.poff, p.ibytes, p.ioff, None, 0, p.status, None, None, None))
        return all(v == 0 for v in p.status)

    def mixed():
        mx._check(lib.h2v_mix_set_rlc_key(mx._mx, FOLD_KEY))
        mx._check(lib.h2v_mix_verify(mx._mx, counts, allp, mpo, alli, mio, None, 0, mstatus, None, ctypes.byref(verdict)))
        return bool(verdict.value)

    pool = ThreadPoolExecutor(len(bvs))
    arms = {
        "mixed": mixed,
        "sequential": lambda: all([one(i) for i in range(len(bvs))]),
        "threads": lambda: all(pool.map(one, range(len(bvs)))),
    }
    times = {a: [] for a in arms}
    ok = {a: True for a in arms}
    for rep in range(args.warmup + args.reps):
        for a, f in arms.items():
            bvs[0]._check(lib.h2v_flush_l2(bvs[0]._ctx, FLUSH_BYTES))
            bvs[0]._check(lib.h2v_batch_download(bvs[0]._ctx, None))  # waits for the flush (h2v_batch_download syncs the stream)
            t0 = time.perf_counter()
            good = f()
            dt = time.perf_counter() - t0
            ok[a] &= good
            if rep >= args.warmup:
                times[a].append(dt)
    pool.shutdown()
    mx.close()
    [bv.close() for bv in bvs]
    out = {"workload": name, "circuits": [f"{sh} k={k} x {n}" for sh, k, n in spec], "proofs": N, "reps": args.reps}
    for a in arms:
        p50, p90 = pct(times[a], 0.5), pct(times[a], 0.9)
        out[a] = {"p50_ms": round(1e3 * p50, 3), "p90_ms": round(1e3 * p90, 3), "proofs_per_s": round(N / p50), "all_accepted": ok[a]}
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=30)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--distinct", type=int, default=256, help="distinct synthesised proofs per circuit (tiled to the batch size)")
    ap.add_argument("--workloads", default="large,small")
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
