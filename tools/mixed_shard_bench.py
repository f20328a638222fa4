"""Sharded mixed batch (include/h2v.h "sharded mixed batches"): one global mix split over the GPUs of a box.

Run under torch.distributed.run, one process per GPU:
    python -m torch.distributed.run --nproc_per_node N tools/mixed_shard_bench.py [--reps 30] [--warmup 3] [--out FILE]
Workload: one 16,384-proof global mix of vm k=10 x 6144, vm k=12 x 4096, sh k=8 GWC/Keccak x 2048 and k18 x 4096 (one
trapdoor, so one params class; SHPLONK / Blake2b from synth.py, the GWC / Keccak member from the oracle's simulated prover with
fewer distinct proofs, tiled).  Every rank takes its shard_range of the member-major concatenation.  Arms, alternated pass by
pass, the L2 overwritten (h2v_flush_l2 through the lead) before every timed pass, every pass one fold key for all ranks:
  exchange   h2v_mix_verify_shard, the device-side exchange inside the mix's graph (root 0)
  gather     h2v_mix_accumulate_shard into device memory, NCCL gather to rank 0, h2v_mix_finalize there, verdict broadcast
  whole      (N = 1 only) h2v_mix_verify over the same batch
The time is the host clock around the per-rank call, which returns after the statuses are on the host; gather includes its
collectives.  Inputs are pre-packed.  Rank 0 writes one JSON line with p50 / p90 per arm and the sha256 of the folded (L, R),
which is the same for every process count."""
import argparse
import ctypes
import hashlib
import json
import os
import random
import subprocess
import sys
import time
from importlib import import_module

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import __graft_entry__ as entry  # noqa: E402

SPEC = [("vm", 10, 6144, "shplonk", "blake2b"), ("vm", 12, 4096, "shplonk", "blake2b"), ("sh", 8, 2048, "gwc", "keccak"),
        ("k18", 18, 4096, "shplonk", "blake2b")]
FOLD_KEY = bytes(range(11, 43))
FLUSH_BYTES = 256 << 20  # twice the 126 MB L2


def card(dev):
    q = subprocess.run(["nvidia-smi", "-i", str(dev), "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True)
    name, _, power = q.stdout.strip().partition(",")
    return {"card": name.strip(), "power_limit": power.strip()}


def pct(xs, q):
    xs = sorted(xs)
    return xs[min(len(xs) - 1, int(round(q * (len(xs) - 1))))]


def members(pkg, synth, dev, distinct):
    s = random.Random("mixshard-bench-srs").randrange(1, synth.R)
    bvs, proofs, insts = [], [], []
    for shape, k, n, mo, tr in SPEC:
        if mo == "shplonk" and tr == "blake2b":
            vk_bytes, dlogs = synth.make_vk_bytes(shape, k)
            bv = pkg.BatchVerifier(pkg.ParamsKZG.from_bytes(synth.params_bytes_raw(k, s), pkg.SerdeFormat.RawBytes),
                                   pkg.VerifyingKey.from_bytes(vk_bytes, pkg.SerdeFormat.RawBytes), mo, tr, device=dev)
            p, i = synth.synthesize_shplonk_batch(bv, dlogs, s, min(n, distinct), seed=("mixshard", shape, k))
        else:
            sys.path.insert(0, os.path.join(ROOT, "oracle"))
            F, sim = import_module("formats"), import_module("prover_sim")
            params, (vk, dl) = sim.make_params(k, s), sim.make_vk(shape, k)
            bv = pkg.BatchVerifier(pkg.ParamsKZG.from_bytes(params.to_bytes()), pkg.VerifyingKey.from_bytes(vk.to_bytes(F.RAW_BYTES), F.RAW_BYTES),
                                   mo, "keccak256" if tr == "keccak" else tr, device=dev)
            rng = random.Random(f"mixshard-{shape}-{k}")
            ints = [sim.random_instances(vk, rng, 10) for _ in range(32)]
            p = [sim.simulate_proof(params, vk, dl, s, i, rng, mo, tr) for i in ints]
            i = [[[v.to_bytes(32, "little") for v in col] for col in x[0]] for x in ints]
        reps = -(-n // len(p))
        bvs.append(bv)
        proofs.append((p * reps)[:n])
        insts.append((i * reps)[:n])
    return bvs, proofs, insts


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=30)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--distinct", type=int, default=256)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import torch
    import torch.distributed as dist

    rank, world = int(os.environ.get("RANK", 0)), int(os.environ.get("WORLD_SIZE", 1))
    dev = int(os.environ.get("LOCAL_RANK", 0))
    torch.cuda.set_device(dev)
    if world > 1:
        dist.init_process_group("nccl", rank=rank, world_size=world, device_id=torch.device("cuda", dev))
    pkg = entry.load_package()
    synth = import_module("halo2_verifier_b200.synth")
    sharding = import_module("halo2_verifier_b200.sharding")
    lib = pkg.load_library()
    head = card(dev)
    bvs, proofs, insts = members(pkg, synth, dev, args.distinct)
    mx = pkg.MixedBatchVerifier(bvs)
    gc = [len(p) for p in proofs]
    N = sum(gc)
    (lo, hi), per = sharding.mixed_shard(gc, rank, world)
    hint = max(b - a for a, b in (sharding.shard_range(N, r, world) for r in range(world)))
    n, counts, packed = mx._shard_args([p[a:b] for p, (a, b) in zip(proofs, per)], [i[a:b] for i, (a, b) in zip(insts, per)], gc, lo, None, 0)
    ucounts = mx._u32(gc)
    status = (ctypes.c_uint8 * n)()
    verdict = ctypes.c_int(0)
    exchange = sharding.connect_channel(mx, rank, world)
    part = torch.empty(mx.partial_bytes(gc), dtype=torch.uint8, device=f"cuda:{dev}")
    digests = {}

    def run_exchange():
        lib.h2v_mix_set_rlc_key(mx._mx, FOLD_KEY)
        lib.h2v_mix_set_shard_hint(mx._mx, hint)
        mx._check(lib.h2v_mix_verify_shard(mx._mx, ucounts, lo, n, *packed[:4], None, 0, 0, status, ctypes.byref(verdict)))
        return bool(verdict.value)

    def run_gather(accum=False):
        lib.h2v_mix_set_rlc_key(mx._mx, FOLD_KEY)
        lib.h2v_mix_set_shard_hint(mx._mx, hint)
        mx._check(lib.h2v_mix_accumulate_shard(mx._mx, ucounts, lo, n, *packed[:4], None, 0, status, ctypes.c_void_p(part.data_ptr())))
        parts = sharding._gather_to_root(part, 0, rank, world)
        flag = torch.zeros(1, dtype=torch.int32, device=f"cuda:{dev}")
        if rank == 0:
            ok, acc = mx.finalize(parts.data_ptr(), gc, want_batch_accum=accum, n_partials=world)
            if accum:
                digests["gather"] = hashlib.sha256(acc).hexdigest()
            flag[0] = int(ok)
        if world > 1:
            dist.broadcast(flag, src=0)
        return bool(flag.item())

    arms = {"gather": run_gather}
    if exchange:
        arms["exchange"] = run_exchange
    if world == 1:
        allp = packed  # the whole batch is this rank's share
        wst = (ctypes.c_uint8 * N)()

        def run_whole(accum=False):
            lib.h2v_mix_set_rlc_key(mx._mx, FOLD_KEY)
            acc = ctypes.create_string_buffer(128) if accum else None
            mx._check(lib.h2v_mix_verify(mx._mx, ucounts, *allp[:4], None, 0, wst, acc, ctypes.byref(verdict)))
            if accum:
                digests["whole"] = hashlib.sha256(acc.raw).hexdigest()
            return bool(verdict.value)
        arms["whole"] = run_whole
    times = {a: [] for a in arms}
    ok = {a: True for a in arms}
    for rep in range(args.warmup + args.reps):
        for a, f in arms.items():
            bvs[0]._check(lib.h2v_flush_l2(bvs[0]._ctx, FLUSH_BYTES))
            bvs[0]._check(lib.h2v_batch_download(bvs[0]._ctx, None))
            if world > 1:
                dist.barrier()
            t0 = time.perf_counter()
            good = f()
            dt = time.perf_counter() - t0
            ok[a] &= good
            if rep >= args.warmup:
                times[a].append(dt)
    if world == 1:
        ok["whole"] &= run_whole(accum=True)
    ok["gather"] &= run_gather(accum=True)  # untimed: the explicit (L, R) costs a serial window combination the timed arms skip
    if exchange:  # one more exchange launch set (untimed): its root holds the folded (L, R) until the mix's next call
        ok["exchange"] &= run_exchange()
        if rank == 0:
            digests["exchange"] = hashlib.sha256(mx.comm_last_batch_accum()).hexdigest()
    if rank == 0:
        out = {**head, "world": world, "proofs": N, "circuits": [f"{sh} k={k} x {c} {mo}/{tr}" for sh, k, c, mo, tr in SPEC], "reps": args.reps,
               "shard_proofs": n, "fold_LR_sha256": digests}
        for a in arms:
            out[a] = {"p50_ms": round(1e3 * pct(times[a], 0.5), 3), "p90_ms": round(1e3 * pct(times[a], 0.9), 3), "all_accepted": ok[a]}
        print(json.dumps(out), flush=True)
        if args.out:
            os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
            with open(args.out, "a") as f:
                f.write(json.dumps(out) + "\n")
    mx.close()
    [bv.close() for bv in bvs]
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
