"""Persistent accumulator against one batch check per batch, on the same proof stream (include/h2v.h "persistent accumulators").

Two arms over a stream of K batches of n proofs, alternated pass by pass, the L2 overwritten (h2v_flush_l2) before every pass:
  verify_batch  K x h2v_verify_batch: one pairing check per batch
  accumulator   K x h2v_acc_absorb + 1 h2v_acc_finalize: one pairing check for the stream
Every call is timed on the host around the C call, which returns after the statuses (or the verdict) are downloaded; the
stream time is the sum of its calls.  Inputs are pre-packed, so the times are the library's, not the Python packing.  Both
arms expand their fold coefficients from the same fixed key.  Workload: VM k=10 SHPLONK / Blake2b (synth.py), streams of
64 x 64 and 16 x 256 proofs.  Afterwards, with graphs off (direct launches, per-stage events): the device time of
k_acc_absorb (h2v_last_timings slot [5], events around the kernel) against that of the batch pairing of verify_batch (same
slot), and the device time of h2v_acc_finalize (CUDA events around the call on the anchor's stream).
Usage: python tools/accumulator_bench.py [--reps 20] [--warmup 3] [--out FILE]"""
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

STREAMS = [(64, 64), (16, 256)]  # (batches K, proofs per batch n)
FOLD_KEY = bytes(range(11, 43))
FLUSH_BYTES = 256 << 20  # twice the 126 MB L2


def card():
    q = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True)
    name, _, power = q.stdout.strip().partition(",")
    return {"card": name.strip(), "power_limit": power.strip()}


def pct(xs, q):
    xs = sorted(xs)
    return xs[min(len(xs) - 1, int(round(q * (len(xs) - 1))))]


class Packed:
    def __init__(self, proofs, instances):
        self.n = len(proofs)
        self.pbytes = b"".join(proofs)
        self.ibytes = b"".join(v for inst in instances for col in inst for v in col)
        po, io = [0], [0]
        for p, inst in zip(proofs, instances):
            po.append(po[-1] + len(p))
            io.append(io[-1] + sum(len(c) for c in inst))
        self.poff = (ctypes.c_uint64 * len(po))(*po)
        self.ioff = (ctypes.c_uint64 * len(io))(*io)
        self.status = (ctypes.c_uint8 * self.n)()


def run_stream(pkg, lib, bv, acc, proofs, insts, K, n, args):
    batches = []
    for b in range(K):  # every batch a different rotation of the distinct proofs
        o = (b * 7) % len(proofs)
        rot = lambda xs: (xs[o:] + xs[:o]) * (-(-n // len(xs)))
        batches.append(Packed(rot(proofs)[:n], rot(insts)[:n]))
    index, verdict = ctypes.c_uint32(0), ctypes.c_int(0)
    av = (ctypes.c_uint8 * K)()

    def verify_stream(calls):
        ok = True
        for p in batches:
            t0 = time.perf_counter()
            bv._check(lib.h2v_batch_set_rlc_key(bv._ctx, FOLD_KEY))
            bv._check(lib.h2v_verify_batch(bv._ctx, n, p.pbytes, p.poff, p.ibytes, p.ioff, None, 0, p.status, None, None, None))
            calls.append(time.perf_counter() - t0)
            ok &= all(v == 0 for v in p.status)
        return ok

    def acc_stream(calls):
        for p in batches:
            t0 = time.perf_counter()
            acc._check(lib.h2v_acc_set_rlc_key(acc._acc, FOLD_KEY))
            acc._check(lib.h2v_acc_absorb(acc._acc, bv._ctx, n, p.pbytes, p.poff, p.ibytes, p.ioff, None, 0, p.status, ctypes.byref(index)))
            calls.append(time.perf_counter() - t0)
        t0 = time.perf_counter()
        acc._check(lib.h2v_acc_finalize(acc._acc, ctypes.byref(verdict), av, K))
        calls.append(time.perf_counter() - t0)
        return bool(verdict.value)

    arms = {"verify_batch": verify_stream, "accumulator": acc_stream}
    stream_t = {a: [] for a in arms}
    call_t = {a: [] for a in arms}
    finalize_t = []
    ok = {a: True for a in arms}
    for rep in range(args.warmup + args.reps):
        for a, f in arms.items():
            bv._check(lib.h2v_flush_l2(bv._ctx, FLUSH_BYTES))
            bv._check(lib.h2v_batch_download(bv._ctx, None))  # waits for the flush
            calls = []
            ok[a] &= f(calls)
            if rep >= args.warmup:
                stream_t[a].append(sum(calls))
                if a == "accumulator":
                    finalize_t.append(calls.pop())
                call_t[a] += calls
    out = {"stream": f"{K} x {n}", "proofs": K * n, "reps": args.reps}
    for a in arms:
        p50, p90 = pct(stream_t[a], 0.5), pct(stream_t[a], 0.9)
        out[a] = {"stream_p50_ms": round(1e3 * p50, 3), "stream_p90_ms": round(1e3 * p90, 3), "proofs_per_s": round(K * n / p50),
                  "call_p50_ms": round(1e3 * pct(call_t[a], 0.5), 3), "call_p90_ms": round(1e3 * pct(call_t[a], 0.9), 3), "all_accepted": ok[a]}
    out["accumulator"]["finalize_host_p50_ms"] = round(1e3 * pct(finalize_t, 0.5), 3)
    return out, batches


def device_times(pkg, lib, bv, acc, batches, n, reps=30):
    """graphs off: per-stage events; the slot [5] span holds the batch pairing (verify_batch) or k_acc_absorb (absorb)"""
    import torch

    bv.set_graphs(False)
    index, verdict = ctypes.c_uint32(0), ctypes.c_int(0)
    av = (ctypes.c_uint8 * 1)()
    pairing, absorb, fin = [], [], []
    stream = torch.cuda.ExternalStream(bv.stream_handle(), device=0)
    for r in range(reps + 2):
        p = batches[r % len(batches)]
        bv._check(lib.h2v_verify_batch(bv._ctx, n, p.pbytes, p.poff, p.ibytes, p.ioff, None, 0, p.status, None, None, None))
        t_pair = bv.timings()["pairing"]
        acc._check(lib.h2v_acc_absorb(acc._acc, bv._ctx, n, p.pbytes, p.poff, p.ibytes, p.ioff, None, 0, p.status, ctypes.byref(index)))
        t_abs = bv.timings()["pairing"]
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        acc._check(lib.h2v_acc_finalize(acc._acc, ctypes.byref(verdict), av, 1))
        e1.record(stream)
        e1.synchronize()
        if r >= 2:
            pairing.append(t_pair)
            absorb.append(t_abs)
            fin.append(e0.elapsed_time(e1))
    bv.set_graphs(True)
    return {"k_acc_absorb_ms": round(statistics.median(absorb), 4), "batch_pairing_ms": round(statistics.median(pairing), 4),
            "finalize_device_ms": round(statistics.median(fin), 4)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--distinct", type=int, default=64, help="distinct synthesised proofs (tiled to the batch size)")
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    pkg = entry.load_package()
    synth = import_module("halo2_verifier_b200.synth")
    lib = pkg.load_library()
    head = card()
    s = random.Random("acc-bench-srs").randrange(1, synth.R)
    vk_bytes, dlogs = synth.make_vk_bytes("vm", 10)
    bv = pkg.BatchVerifier(pkg.ParamsKZG.from_bytes(synth.params_bytes_raw(10, s), pkg.SerdeFormat.RawBytes),
                           pkg.VerifyingKey.from_bytes(vk_bytes, pkg.SerdeFormat.RawBytes), "shplonk", "blake2b", device=0)
    proofs, insts = synth.synthesize_shplonk_batch(bv, dlogs, s, args.distinct, seed="acc-bench")
    lines = []
    with pkg.Accumulator(bv, max_absorbs=max(K for K, _ in STREAMS)) as acc:
        first = Packed(proofs[:1], insts[:1])
        bv._check(lib.h2v_verify_batch(bv._ctx, 1, first.pbytes, first.poff, first.ibytes, first.ioff, None, 7, first.status, None, None, None))
        for K, n in STREAMS:
            res, batches = run_stream(pkg, lib, bv, acc, proofs, insts, K, n, args)
            res.update(device_times(pkg, lib, bv, acc, batches, n))
            res = {**head, "workload": "vm k=10 shplonk blake2b", **res}
            print(json.dumps(res), flush=True)
            lines.append(json.dumps(res))
    bv.close()
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
