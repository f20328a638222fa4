"""Aggregation proofs: the carried KZG accumulator checked inside the batch fold, against not checking it and against the
in-library alternative (include/h2v.h "aggregation proofs").

4096 VM k=10 SHPLONK / Blake2b proofs (64 distinct synthesised proofs tiled, synth.py) whose instances carry a valid accumulator
(lhs, rhs) = (s P, P) in LimbsEncoding<3, 88> (rows 0..11 of the instance column, 16 rows).  Three arms, alternated pass by pass
for --reps passes, the L2 overwritten (h2v_flush_l2, 256 MB) before every pass:
  (a) plain        h2v_verify_batch on a plain context: the carried accumulator is NOT checked
  (b) aggregation  h2v_verify_batch on an aggregation context: checked inside the fold (two more MSM terms per proof)
  (c) merge        (a) plus one h2v_acc_merge per carried pair (acc <- r acc + (rhs, lhs), r from the OS) and one
                   h2v_acc_finalize: today's in-library route.  The pairs are decoded from the limbs before the timed region.
Every call is timed on the host around the C call, which returns after the statuses (or the verdict) are downloaded; inputs
are pre-packed.  Every arm expands its fold coefficients from the same fixed key.  Afterwards, with graphs off (direct
launches, per-stage CUDA events), the per-stage device times of (a) and (b) (h2v_last_timings).
Usage: python tools/aggregation_bench.py [--reps 30] [--warmup 3] [--n 4096] [--out FILE]"""
import argparse
import ctypes
import json
import os
import random
import statistics
import subprocess
import sys
import time
from importlib import import_module

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import __graft_entry__ as entry  # noqa: E402

FOLD_KEY = bytes(range(11, 43))
FLUSH_BYTES = 256 << 20  # twice the 126 MB L2
LIMBS, BITS, ROWS = 3, 88, 16


def card():
    q = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True)
    name, _, power = q.stdout.strip().partition(",")
    return {"card": name.strip(), "power_limit": power.strip()}


def pct(xs, q):
    xs = sorted(xs)
    return xs[min(len(xs) - 1, int(round(q * (len(xs) - 1))))]


def limbs_of(pt):
    out = []
    for v in ((0, 0) if pt is None else pt):
        out += [(v >> (BITS * i)) & ((1 << BITS) - 1) for i in range(LIMBS)]
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=30)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--n", type=int, default=4096)
    ap.add_argument("--distinct", type=int, default=64, help="distinct synthesised proofs (tiled to the batch size)")
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    pkg = entry.load_package()
    synth = import_module("halo2_verifier_b200.synth")
    lib = pkg.load_library()
    head = card()
    s = random.Random("agg-bench-srs").randrange(1, synth.R)
    vk_bytes, dlogs = synth.make_vk_bytes("vm", 10)
    params = pkg.ParamsKZG.from_bytes(synth.params_bytes_raw(10, s), pkg.SerdeFormat.RawBytes)
    vk = pkg.VerifyingKey.from_bytes(vk_bytes, pkg.SerdeFormat.RawBytes)
    spec = pkg.InstanceAccumulator.rows(LIMBS, BITS)
    plain = pkg.BatchVerifier(params, vk, "shplonk", "blake2b", device=0)
    agg = pkg.BatchVerifier(params, vk, "shplonk", "blake2b", device=0, accumulator=spec)
    pairs = []

    def instances_of(j, rng):
        d = rng.randrange(1, synth.R)
        lhs, rhs = synth.g1_mul_gen(d * s % synth.R), synth.g1_mul_gen(d)
        pairs.append((lhs, rhs))
        col = limbs_of(lhs) + limbs_of(rhs) + [rng.randrange(synth.R) for _ in range(ROWS - 4 * LIMBS)]
        return [[v.to_bytes(32, "little") for v in col]]

    proofs, insts = synth.synthesize_shplonk_batch(plain, dlogs, s, args.distinct, seed="agg-bench", rows=ROWS, instances_of=instances_of)
    n = args.n
    tile = lambda xs: (xs * (-(-n // len(xs))))[:n]
    proofs, insts, pairs = tile(proofs), tile(insts), tile(pairs)
    pbytes = b"".join(proofs)
    ibytes = b"".join(v for inst in insts for col in inst for v in col)
    po, io = [0], [0]
    for p, inst in zip(proofs, insts):
        po.append(po[-1] + len(p))
        io.append(io[-1] + sum(len(c) for c in inst))
    poff, ioff = (ctypes.c_uint64 * len(po))(*po), (ctypes.c_uint64 * len(io))(*io)
    status = (ctypes.c_uint8 * n)()
    enc = lambda p: bytes(64) if p is None else p[0].to_bytes(32, "little") + p[1].to_bytes(32, "little")
    merge_ops = [enc(rhs) + enc(lhs) for lhs, rhs in pairs]  # (L, R) layout: rhs pairs with [s]G2, lhs with -G2
    acc = pkg.Accumulator(plain, max_absorbs=n)
    verdict = ctypes.c_int(0)
    av = (ctypes.c_uint8 * n)()

    def batch(bv):
        bv._check(lib.h2v_batch_set_rlc_key(bv._ctx, FOLD_KEY))
        bv._check(lib.h2v_verify_batch(bv._ctx, n, pbytes, poff, ibytes, ioff, None, 0, status, None, None, None))
        return all(v == 0 for v in status)

    def arm_plain():
        return batch(plain)

    def arm_agg():
        return batch(agg)

    def arm_merge():
        ok = batch(plain)
        for op in merge_ops:
            acc._check(lib.h2v_acc_merge(acc._acc, op, None))
        acc._check(lib.h2v_acc_finalize(acc._acc, ctypes.byref(verdict), av, n))
        return ok and bool(verdict.value)

    arms = {"plain": arm_plain, "aggregation": arm_agg, "merge": arm_merge}
    times = {a: [] for a in arms}
    ok = {a: True for a in arms}
    for rep in range(args.warmup + args.reps):
        for a, f in arms.items():
            plain._check(lib.h2v_flush_l2(plain._ctx, FLUSH_BYTES))
            plain._check(lib.h2v_batch_download(plain._ctx, None))  # waits for the flush
            t0 = time.perf_counter()
            ok[a] &= f()
            dt = time.perf_counter() - t0
            if rep >= args.warmup:
                times[a].append(dt)
    res = {**head, "workload": f"vm k=10 shplonk blake2b, {n} proofs, LimbsEncoding<{LIMBS}, {BITS}>", "reps": args.reps}
    for a in arms:
        res[a] = {"p50_ms": round(1e3 * pct(times[a], 0.5), 3), "p90_ms": round(1e3 * pct(times[a], 0.9), 3), "all_accepted": ok[a]}
    stages = {}
    for name, bv in (("plain", plain), ("aggregation", agg)):
        bv.set_graphs(False)
        rows = []
        for r in range(12):
            batch(bv)
            if r >= 2:
                rows.append(bv.timings())
        bv.set_graphs(True)
        stages[name] = {k: round(statistics.median(t[k] for t in rows), 4) for k in rows[0] if k != "attribution"}
    res["stage_device_ms_graphs_off"] = stages
    print(json.dumps(res), flush=True)
    acc.close()
    agg.close()
    plain.close()
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(json.dumps(res) + "\n")


if __name__ == "__main__":
    main()
