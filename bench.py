#!/usr/bin/env python
"""Benchmark of the hot path: verified proofs/sec on batches of 4096 SHPLONK proofs (BN254, Blake2b
transcript) of the reference's vector_mul test-circuit shape at k = 10 (BASELINE.json configs[1]).

    python bench.py --gpus N --steps K --warmup W          this repo's CUDA path (one rank per GPU)
    python bench.py --impl reference ...                    CPU restatement of the reference algorithm
                                                            (oracle/), all host threads, rank 0 only
    python bench.py --config 5 [--gpus N]                   ONE 65,536-proof global batch sharded over N GPUs (configs[4])
    python bench.py --config 4                              the k = 18 lookup-heavy shape, batch 1024 (configs[3])
    python bench.py --selfcheck ...                         additionally: the (sharded) path against the C oracle on the
                                                            bench's own inputs, incl. a corrupted proof on a non-root rank
    python bench.py --dump-outputs DIR ...                  additionally: what the last timed step returned (rank 0), as
                                                            DIR/{status,group_verdicts,verdict}.npy (float32)

A step = ONE launch set: `--fold-groups` complete, independent batch verifications (each: transcript replay,
expression / multi-open scalars, one folded MSM, one pairing check, one verdict) of `--batch` proofs per GPU that
share one set of kernel launches.  `value` times `--steps` steps on inputs already resident in HBM (L2 flushed between
steps; `--blocks R`: R such blocks, the median block is reported); `e2e` times the C-ABI call a user makes
(`h2v_verify_batch` at N=1, `h2v_verify_shard` at N>1) from pinned host buffers, host<->device copies included.
Inputs are the same in every run with the same arguments: seeded proofs and, on the resident path, fold coefficients
expanded from a fixed key.
At N>1 the one exchange step runs device-side over NVLink inside the CUDA graph (csrc/exchange.cuh); torch.distributed
is plumbing (barriers, start-up handle exchange).  Prints ONE JSON line on rank 0.
"""
import argparse
import ctypes
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
# one hardware work queue per stream in flight (default 8): batches of different contexts must not serialise behind
# each other (read at CUDA initialisation)
os.environ.setdefault("CUDA_DEVICE_MAX_CONNECTIONS", "32")

METRIC = "verified proofs/sec (BN254 SHPLONK, batch 4096)"
UNIT = "proofs/s"
SRS_SEED = 2  # BASELINE.md config 2: SRS secret from seed 2
# fold-coefficient key of the resident uploads (h2v_batch_set_rlc_key: the keyed expansion that OS entropy also feeds),
# fixed so that every run verifies the same batches with the same coefficients
FOLD_KEY = bytes(range(1, 33))
R_MOD = 0x30644E72E131A029B85045B68181585D2833E84879B9709143E1F593F0000001
IMAD_SLOTS_PER_MM = 272  # 8-limb CIOS: 136 32x32->64 multiply-adds = 272 lo/hi IMAD issue slots (DESIGN.md section 5)


def srs_secret(k):
    import random

    return random.Random(repr(("srs", k, SRS_SEED))).randrange(1, R_MOD)


# ------------------------------------------------------------------------------------------------
class ClockSampler(threading.Thread):
    """nvidia-smi clocks / throttle reasons DURING the timed region (B200_PROFILING.md recipe)."""

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.samples, self.stop_flag = index, [], threading.Event()

    def run(self):
        q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        while not self.stop_flag.is_set():
            try:
                out = subprocess.run(["nvidia-smi", "-i", str(self.index), f"--query-gpu={q}", "--format=csv,noheader,nounits"],
                                     capture_output=True, text=True, timeout=5).stdout.strip()
                if out:
                    self.samples.append([x.strip() for x in out.split(",")])
            except Exception:
                pass
            self.stop_flag.wait(0.3)

    def summary(self):
        self.stop_flag.set()
        self.join(timeout=6)
        sm = [int(s[0]) for s in self.samples if s[0].isdigit()]
        mx = [int(s[1]) for s in self.samples if s[1].isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = sorted({n for s in self.samples for n, v in zip(names, s[2:6]) if v.lower().startswith("active")})
        return {"sm_mhz": int(statistics.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": reasons, "samples": len(sm)}


def pinned_bytes(torch, data: bytes):
    t = torch.empty(max(1, len(data)), dtype=torch.uint8).pin_memory()
    if data:
        t[: len(data)] = torch.frombuffer(bytearray(data), dtype=torch.uint8)
    return t


class PackedBatch:
    """One batch packed exactly as the Rust host would: pinned buffers + offset arrays."""

    def __init__(self, torch, proofs, instances):
        import numpy as np

        self.n = len(proofs)
        self.src = (proofs, instances)
        self.proofs = pinned_bytes(torch, b"".join(proofs))
        inst = b"".join(v for inst in instances for col in inst for v in col)
        self.inst = pinned_bytes(torch, inst)
        poff = np.zeros(self.n + 1, dtype=np.uint64)
        poff[1:] = np.cumsum([len(p) for p in proofs])
        ioff = np.zeros(self.n + 1, dtype=np.uint64)
        ioff[1:] = np.cumsum([sum(len(col) for col in i) for i in instances])
        self.poff = torch.from_numpy(poff.view(np.int64)).pin_memory()
        self.ioff = torch.from_numpy(ioff.view(np.int64)).pin_memory()
        self.status = torch.zeros(self.n, dtype=torch.uint8).pin_memory()
        self.h2d_bytes = len(b"".join(proofs)) + len(inst) + 2 * 8 * (self.n + 1)
        self.d2h_bytes = 4 * self.n + 4

    def args(self):
        return (self.n, self.proofs.data_ptr(), self.poff.data_ptr(), self.inst.data_ptr(), self.ioff.data_ptr())


def algorithmic_mm(bv, n, geom, rows=10):
    """Algorithmic 256-bit Montgomery multiplications per stage of ONE batch of n proofs (DESIGN.md section 5);
    1 MM = 136 32x32->64 multiply-adds (8-limb CIOS: 64 for a*b, 64 for m*p, 8 for m_i); a squaring counts as one MM.
    The per-proof stages come from the plan itself (h2v_ctx_work_model walks the plan like scalar_stage does), the MSM and
    pairing terms from the window geometry of the run."""
    wm = bv.work_model(rows)
    P = bv.n_points
    c0, c1 = geom["window_bits"] & 0xFFFF, geom["window_bits"] >> 16
    W0, W1 = geom["windows"] & 0xFFFF, geom["windows"] >> 16
    left_live = bv.n_mo if getattr(bv, "multiopen", "shplonk") == "gwc" else bv.n_mo // 2  # SHPLONK: h1 has left scalar 0
    t_right, t_left = n * P + bv.n_shared, n * left_live
    return {
        "decompress": n * P * wm["decompress_per_point"],
        "transcript": n * wm["transcript"],
        "scalar": n * wm["scalar"],
        # fold coefficients (scalar x c_j per term) + bucket accumulation (mixed addition 7 M + 4 S) + bucket reduction (2 full additions per bucket)
        "rlc_msm": n * (P + bv.n_mo) * 2 + (W0 * t_right + W1 * t_left) * 11 + (W0 * (1 << (c0 - 1)) + W1 * (1 << (c1 - 1))) * 32,
        "pairing": 65 * (W0 + W1) * 58 + 430 * 54,  # k_lines: line value (4) + sparse product (54) per pair and step; check: ~430 Fq12 products
    }


def bucket_sum_mm(bv, n, geom):
    """k_msm_bucket_sum alone: one mixed addition (7 MM + 4 S, counted as 11 MM) per bucket entry"""
    W0, W1 = geom["windows"] & 0xFFFF, geom["windows"] >> 16
    left_live = bv.n_mo if getattr(bv, "multiopen", "shplonk") == "gwc" else bv.n_mo // 2
    return (W0 * (n * bv.n_points + bv.n_shared) + W1 * (n * left_live)) * 11


def plan_launch_sets(steps, n_ctx):
    """A step is ONE launch set (fold_groups independent batches through one set of kernel launches on one context).
    The `steps` launch sets of a timed block go round-robin over the contexts; launch set i is rooted at rank i mod N.
    Returns assign[i] = context of launch set i (identical on every rank: the contexts of equal index form a channel and
    must see the same sequence of launch sets)."""
    return [i % n_ctx for i in range(steps)]


CONFIGS = {
    # BASELINE.json configs[1]: the headline
    2: dict(shape="vm", k=10, batch=4096, multiopen="shplonk", scaling="weak",
            name="BASELINE.json configs[1]: 4096-proof SHPLONK batches, vector_mul test-circuit shape, k=10"),
    # configs[3]: lookup + permutation heavy
    4: dict(shape="k18", k=18, batch=1024, multiopen="shplonk", scaling="weak",
            name="BASELINE.json configs[3]: 1024-proof batches of the lookup+permutation-heavy shape (k=18, degree 5, 64 advice columns, 12,960-byte proofs)"),
    # configs[4]: ONE 65,536-proof global batch sharded over the ranks
    5: dict(shape="vm", k=10, batch=65536, multiopen="shplonk", scaling="strong",
            name="BASELINE.json configs[4]: ONE 65,536-proof SHPLONK global batch sharded over the GPUs, partial accumulators gathered over NVLink, one final pairing"),
}


def run_ours(args):
    import numpy as np
    import torch
    import __graft_entry__ as g

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world != args.gpus:
        raise SystemExit(f"--gpus {args.gpus} but WORLD_SIZE={world}: launch with torch.distributed.run --nproc-per-node {args.gpus}")
    torch.cuda.set_device(local)
    dist = None
    if world > 1:  # torch.distributed = plumbing only: barriers, the start-up exchange of window handles, max over ranks
        import torch.distributed as dist

        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    pkg = g.load_package()
    from importlib import import_module

    synth = import_module("halo2_verifier_b200.synth")
    sharding = import_module("halo2_verifier_b200.sharding")
    lib = pkg.load_library()
    cfg = CONFIGS[args.config]
    k, shape = args.k, args.shape
    strong = cfg["scaling"] == "strong"
    if strong:  # one global batch per fold group, every rank holds 1 / world of it
        assert args.batch % world == 0
        n = args.batch // world
        # small shards (8 GPUs: 8192 proofs) do not fill a GPU: several global batches then share a launch set
        G = args.fold_groups if args.fold_groups > 1 else max(1, min(8, 32768 // n))
    else:
        n, G = args.batch, max(1, args.fold_groups)
    gcount, gbase = n * world, n * rank  # of ONE global batch
    s = srs_secret(k)
    vk_bytes, shared_dlogs = synth.make_vk_bytes(shape, k)
    params = pkg.ParamsKZG.from_bytes(synth.params_bytes_raw(k, s), pkg.SerdeFormat.RawBytes)
    vk = pkg.VerifyingKey.from_bytes(vk_bytes, pkg.SerdeFormat.RawBytes)
    n_ctx = max(1, args.streams)
    bvs = [pkg.BatchVerifier(params, vk, "shplonk", "blake2b", device=local) for _ in range(n_ctx)]
    bv = bvs[0]
    if os.environ.get("H2V_BENCH_DIAG_NOGRAPH"):
        [b.set_graphs(False) for b in bvs]
    # host threads: one per context and rank; when they outnumber the cores, waits must block instead of spin
    blocking = n_ctx * world > max(1, (os.cpu_count() or 1) // 2)
    for b in bvs:
        lib.h2v_ctx_set_blocking_sync(b._ctx, 1 if blocking else 0)
    for ci, ctx in enumerate(bvs):
        ctx.ci = ci
    if world > 1:  # one exchange channel per context index (include/h2v.h): windows mapped once, at start-up
        for ctx in bvs:
            if not sharding.connect_channel(ctx, rank, world, max_groups=G):
                raise SystemExit("the ranks cannot map each other's exchange windows (CUDA IPC / peer access): " + lib.h2v_last_error(ctx._ctx).decode())
    # ---------------- inputs: two distinct accepting batches per rank (seeded), alternated between fold groups
    t0 = time.time()
    n_dist = min(n, 4096)
    batches = []
    for b in range(2):
        if strong:  # the SAME global batch for every N (4096 distinct proofs, tiled): rank r holds positions [gbase, gbase + n)
            proofs, instances = synth.synthesize_shplonk_batch(bv, shared_dlogs, s, 4096, seed=("global", b))
            reps = -(-(gbase + n) // 4096)
            batches.append(PackedBatch(torch, (proofs * reps)[gbase:gbase + n], (instances * reps)[gbase:gbase + n]))
            continue
        proofs, instances = synth.synthesize_shplonk_batch(bv, shared_dlogs, s, n_dist, seed=(rank, b))
        reps = -(-n // n_dist)
        batches.append(PackedBatch(torch, (proofs * reps)[:n], (instances * reps)[:n]))
    gen_s = time.time() - t0

    def packed_groups(first, count):
        pr, ins = [], []
        for q in range(count):
            pr += batches[(first + q) % 2].src[0]
            ins += batches[(first + q) % 2].src[1]
        return PackedBatch(torch, pr, ins)

    gbatches = [packed_groups(b, G) for b in range(2)] if G > 1 else batches
    chk = lambda ctx, rc: ctx._check(rc)
    ext_streams = [torch.cuda.ExternalStream(b.stream_handle(), device=torch.device("cuda", local)) for b in bvs]
    NULL = None

    def set_groups(ctx, pb):
        if pb.n > n:
            chk(ctx, lib.h2v_batch_set_fold_groups(ctx._ctx, pb.n // n))

    def upload(ctx, pb):
        set_groups(ctx, pb)
        chk(ctx, lib.h2v_batch_set_rlc_key(ctx._ctx, FOLD_KEY))
        if world == 1:
            chk(ctx, lib.h2v_batch_upload(ctx._ctx, *pb.args(), NULL, 0))
        else:
            chk(ctx, lib.h2v_batch_upload_shard(ctx._ctx, *pb.args(), NULL, 0, gbase, gcount))

    def step_resident(ctx, i=0):
        """one launch set on data resident in HBM; N > 1: through the device-side exchange, rooted at rank i mod N"""
        v = ctypes.c_int(0)
        if not os.environ.get("H2V_BENCH_DIAG_NOFLUSH"):  # (diagnosis only; reported numbers always flush)
            chk(ctx, lib.h2v_flush_l2(ctx._ctx, 256 << 20))
        if world == 1:
            chk(ctx, lib.h2v_batch_run(ctx._ctx, ctypes.byref(v)))
        else:
            chk(ctx, lib.h2v_batch_run_shard_exchange(ctx._ctx, i % world, NULL, ctypes.byref(v)))
        return v.value

    def step_e2e(ctx, pb, i=0):
        """the call a user makes: host buffers in, statuses out (fold randomness from the OS: seed 0, no scalars)"""
        set_groups(ctx, pb)
        if world == 1:
            chk(ctx, lib.h2v_verify_batch(ctx._ctx, *pb.args(), NULL, 0, pb.status.data_ptr(), NULL, NULL, NULL))
            return int(pb.status.max()) == 0
        v = ctypes.c_int(0)
        chk(ctx, lib.h2v_verify_shard(ctx._ctx, *pb.args(), NULL, 0, gbase, gcount, i % world, pb.status.data_ptr(), NULL, ctypes.byref(v)))
        return v.value == 1 and int(pb.status.max()) == 0

    def sync_all():
        torch.cuda.synchronize()
        if dist is not None:
            dist.barrier()
            torch.cuda.synchronize()

    def run_steps(fn, count, ctxs, before=None):
        """`count` launch sets round-robin over the contexts; each context is driven by its own host thread (ctypes
        releases the GIL), so the launch sets of different contexts overlap on the device.  `before` runs on the
        main thread once every worker stands at the start line."""
        out = [None] * count
        assign = plan_launch_sets(count, len(ctxs))
        start = threading.Barrier(len(ctxs) + 1)
        errs = []

        def worker(ci):
            torch.cuda.set_device(local)
            start.wait()
            try:
                for i in range(count):
                    if assign[i] == ci:
                        out[i] = fn(ctxs[ci], i)
            except Exception as e:  # noqa: BLE001
                errs.append(e)

        ths = [threading.Thread(target=worker, args=(ci,)) for ci in range(len(ctxs))]
        [t.start() for t in ths]
        if before is not None:
            before()
        start.wait()
        [t.join() for t in ths]
        if errs:
            raise errs[0]
        return out

    def timed_block(fn, count, ctxs):
        """`count` launch sets between barrier + synchronize on both sides; returns (results, seconds on the DEVICE clock:
        CUDA events on the contexts' streams, first start -> last end; seconds on the host clock)."""
        sync_all()
        ev0 = torch.cuda.Event(enable_timing=True)
        w0 = [0.0]

        def before():
            ev0.record(ext_streams[ctxs[0].ci])
            w0[0] = time.perf_counter()

        res_ = run_steps(fn, count, ctxs, before)
        ends = []
        for c in ctxs:
            e = torch.cuda.Event(enable_timing=True)
            e.record(ext_streams[c.ci])
            ends.append(e)
        sync_all()
        wall = time.perf_counter() - w0[0]
        return res_, max(ev0.elapsed_time(e) for e in ends) * 1e-3, wall

    def reduce_max(vals):
        t = torch.tensor(vals, dtype=torch.float64, device="cuda")
        if dist is not None:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return [float(x) for x in t]

    W = max(args.warmup, 3)
    R = max(1, args.blocks)
    steps = args.steps
    proofs_per_step = n * G * world  # one launch set on every rank
    # ---------------- one batch in flight: latency view (single batches, one context, spinning waits)
    upload(bv, batches[0])
    ok = run_steps(lambda ctx, i: step_resident(ctx, i), W, bvs[:1])
    assert all(v == 1 for v in ok), "warm-up batch was rejected"
    geom = geom_tp = bv.msm_geometry()
    # clocks DURING the timed region: rank 0 samples its own GPU, a few times per second (every rank polling nvidia-smi ten
    # times per second measurably disturbed the timed blocks at N = 8: the query takes driver locks and host cores)
    sampler = ClockSampler(local) if rank == 0 else None
    if sampler is not None:
        sampler.start()
    lib.h2v_ctx_set_blocking_sync(bv._ctx, 0)
    res, dt1, _ = timed_block(lambda ctx, i: step_resident(ctx, i), steps, bvs[:1])
    lib.h2v_ctx_set_blocking_sync(bv._ctx, 1 if blocking else 0)
    assert all(v == 1 for v in res), "a timed batch was rejected"
    # ---------------- device-resident throughput (`value`): R timed blocks of `steps` launch sets, median block
    for ci, ctx in enumerate(bvs):
        upload(ctx, gbatches[ci % 2])
    ok = run_steps(lambda ctx, i: step_resident(ctx, i), W * n_ctx, bvs)
    assert all(v == 1 for v in ok), "warm-up launch set was rejected"
    geom_tp = bv.msm_geometry()
    block_dt = []
    launches = 0
    for _ in range(R):
        launches0 = sum(b.launch_count() for b in bvs)
        res, dtb, _ = timed_block(lambda ctx, i: step_resident(ctx, i), steps, bvs)
        assert all(v == 1 for v in res), "a timed launch set was rejected"
        launches = sum(b.launch_count() for b in bvs) - launches0
        block_dt.append(dtb)
    if args.dump_outputs and rank == 0:  # what the last timed step's caller receives: its verdicts and per-proof statuses
        last = bvs[plan_launch_sets(steps, n_ctx)[-1]]
        status = np.zeros(n * G, dtype=np.uint8)
        chk(last, lib.h2v_batch_download(last._ctx, status.ctypes.data))
        group_verdicts = np.zeros(G, dtype=np.uint8)
        assert lib.h2v_last_group_verdicts(last._ctx, group_verdicts.ctypes.data, G) == G
        os.makedirs(args.dump_outputs, exist_ok=True)
        for name, a in (("status", status), ("group_verdicts", group_verdicts), ("verdict", np.array([res[-1]]))):
            np.save(os.path.join(args.dump_outputs, name + ".npy"), a.astype(np.float32))
    clocks = sampler.summary() if sampler is not None else None
    if os.environ.get("H2V_BENCH_DIAG_TIMELINE") and rank == 0 and world == 1:  # (diagnosis only) per-block timeline of 3 sets per context
        cap = 1 << 20
        chk(bv, lib.h2v_debug_timeline_start(local, cap))
        run_steps(lambda ctx, i: step_resident(ctx, i), 3 * n_ctx, bvs)
        buf = np.zeros(cap * 8, dtype=np.uint32)
        cnt = ctypes.c_uint32(0)
        chk(bv, lib.h2v_debug_timeline_stop(local, buf.ctypes.data, cap, ctypes.byref(cnt)))
        np.save(os.environ["H2V_BENCH_DIAG_TIMELINE"], buf[: cnt.value * 8].reshape(-1, 8))
    # ---------------- per-stage / per-kernel device times of serial single batches under graph replay, from the on-device
    # block timeline (global nanosecond timer: first block start -> last block end of every kernel; no host in the loop)
    stage_ms, kern_ms = {}, {}
    if world == 1:
        upload(bv, batches[0])
        run_steps(lambda ctx, i_: step_resident(ctx, i_), 2, bvs[:1])
        stage_acc, kern_acc = {}, {}
        cap = 1 << 18
        tlbuf = np.zeros(cap * 8, dtype=np.uint32)
        for _ in range(5):
            chk(bv, lib.h2v_debug_timeline_start(local, cap))
            run_steps(lambda ctx, i_: step_resident(ctx, i_), 1, bvs[:1])
            cnt = ctypes.c_uint32(0)
            chk(bv, lib.h2v_debug_timeline_stop(local, tlbuf.ctypes.data, cap, ctypes.byref(cnt)))
            rec = tlbuf[: cnt.value * 8].reshape(-1, 8).astype(np.uint64)
            kid, t0_, t1_ = rec[:, 0], rec[:, 4] | (rec[:, 5] << np.uint64(32)), rec[:, 6] | (rec[:, 7] << np.uint64(32))
            span = {int(k_): (int(t0_[kid == k_].min()), int(t1_[kid == k_].max())) for k_ in np.unique(kid)}
            if not all(k_ in span for k_ in range(1, 11)):
                continue
            ms = lambda a, b: (b - a) * 1e-6
            for name, v in (("total", ms(span[1][0], span[10][1])), ("decompress", ms(*span[1])), ("transcript", ms(span[1][1], span[2][1])),
                            ("scalar", ms(span[2][1], span[3][1])), ("rlc_msm", ms(span[3][1], span[8][1])), ("pairing", ms(span[8][1], span[10][1]))):
                stage_acc.setdefault(name, []).append(v)
            for name, k_ in (("k_decompress", 1), ("k_transcript", 2), ("k_scalar", 3), ("k_msm_digits", 4), ("k_msm_scatter", 5), ("k_msm_bucket_sum", 6),
                             ("k_msm_chunk_reduce", 7), ("k_msm_window_reduce", 8), ("k_lines", 9), ("k_pairing_check", 10)):
                kern_acc.setdefault(name, []).append(ms(*span[k_]))
        stage_ms = {k_: statistics.median(v) for k_, v in stage_acc.items()}
        kern_ms = {k_: statistics.median(v) for k_, v in kern_acc.items()}
    # ---------------- end to end through the C ABI from pinned host memory
    run_steps(lambda ctx, i: step_e2e(ctx, batches[i % 2], i), W, bvs[:1])
    lat = []

    def timed_e2e(ctx, i, pbs):
        a = time.perf_counter()
        okk = step_e2e(ctx, pbs[i % 2], i)
        lat.append(time.perf_counter() - a)
        return okk

    lib.h2v_ctx_set_blocking_sync(bv._ctx, 0)
    res, _, dt_e2e1 = timed_block(lambda ctx, i: timed_e2e(ctx, i, batches), steps, bvs[:1])  # e2e is what the caller sees: host clock around the calls
    lib.h2v_ctx_set_blocking_sync(bv._ctx, 1 if blocking else 0)
    assert all(res), "an end-to-end batch was rejected"
    p50 = statistics.median(lat) * 1e3
    run_steps(lambda ctx, i: step_e2e(ctx, gbatches[i % 2], i), W * n_ctx, bvs)
    block_e2e = []
    for _ in range(R):
        res, _, dte = timed_block(lambda ctx, i: timed_e2e(ctx, i, gbatches), steps, bvs)
        assert all(res), "an end-to-end launch set was rejected"
        block_e2e.append(dte)
    red = reduce_max(block_dt + block_e2e + [dt1, dt_e2e1])  # every block: max over ranks
    block_dt, block_e2e, dt1, dt_e2e1 = red[:R], red[R:2 * R], red[2 * R], red[2 * R + 1]
    dt, dt_e2e = statistics.median(block_dt), statistics.median(block_e2e)

    selfcheck = run_selfcheck(args, pkg, lib, torch, dist, synth, sharding, bv, batches[0], rank, world, n, gbase, gcount, synth.params_bytes_raw(k, s), vk_bytes) if args.selfcheck else None

    out = None
    if rank == 0:
        rows = 10
        mm = algorithmic_mm(bv, n, geom, rows)  # one batch alone (the stage / kernel times below)
        mm_tp = algorithmic_mm(bv, n, geom_tp, rows)  # one batch of a launch set of the timed region
        imad_peak = lib.h2v_calibrate_imad(local)
        slots = lambda m: m * IMAD_SLOTS_PER_MM
        # whole timed step: the work of one launch set on this GPU (G batches) / the median block time per launch set
        achieved_all = slots(sum(mm_tp.values()) * G) / (dt / steps)
        if world > 1:  # the pairing checks of a global batch run once, on its root: 1 / world of them per rank
            achieved_all = slots((sum(mm_tp.values()) - mm_tp["pairing"] * (1 - 1 / world)) * G) / (dt / steps)
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json"))) if os.path.exists(os.path.join(ROOT, "MEASURED_PEAKS.json")) else {}
        hbm_peak, hbm_src = (peaks["hbm_gbs"], "measured") if "hbm_gbs" in peaks else (6650.0, "fallback")
        pipe = {}
        ppath = os.path.join(ROOT, "profiles", "ncu_pipe.json")  # sm__pipe_fmaheavy_cycles_active of the stage kernels from the committed ncu --set full capture
        if os.path.exists(ppath):
            pipe = json.load(open(ppath))
        traffic = None
        tpath = os.path.join(ROOT, "profiles", "dram_traffic.json")  # per-launch dram bytes of the stage kernels from one ncu --set full capture
        kern_mm = {"k_decompress": mm["decompress"], "k_msm_bucket_sum": bucket_sum_mm(bv, n, geom), "k_scalar": mm["scalar"]}
        roof = {"bound": "imad", "kernel": "whole timed step (every kernel of a launch set; no single kernel holds more than 40 % of it)",
                "achieved": achieved_all / 1e12, "peak": imad_peak / 1e12, "unit": "T IMAD/s", "frac": achieved_all / imad_peak,
                "mm_per_proof": sum(mm_tp.values()) / n, "traffic": None,
                "note": "integer-multiply bound (no HBM/tensor roofline applies, DESIGN.md section 5): algorithmic 256-bit Montgomery multiplications (a squaring "
                        "counted as one, so squaring-heavy kernels read up to 23 % high) x 272 IMAD issue slots (136 32x32->64 multiply-adds, lo + hi) of ALL stages of a "
                        "launch set / the median timed block (CUDA events) per launch set; peak = 32-bit IMAD issue rate measured by the calibration kernel in this run. "
                        "`kernels` / `stages`: one 4096-proof batch ALONE under graph replay, durations from the on-device global timer (first block start -> last block "
                        "end, h2v_debug_timeline); `pipe_fmaheavy_pct` = sm__pipe_fmaheavy_cycles_active of that kernel in the committed ncu --set full capture"}
        if kern_ms:
            if os.path.exists(tpath):
                roof["traffic"] = json.load(open(tpath)).get("k_decompress")
            roof["kernels"] = {k_: {"ms_one_in_flight": round(kern_ms[k_], 4), "mm": int(kern_mm[k_]), "frac": slots(kern_mm[k_]) / (kern_ms[k_] * 1e-3) / imad_peak,
                                    "pipe_fmaheavy_pct": pipe.get(k_)} for k_ in kern_mm if k_ in kern_ms}
            roof["stages"] = {k_: {"ms_one_in_flight": round(stage_ms[k_], 4), "mm": int(mm[k_]), "frac": slots(mm[k_]) / (stage_ms[k_] * 1e-3) / imad_peak}
                              for k_ in mm if k_ in stage_ms}
        eval_bytes = n * (bv.proof_len + 32 * bv.n_inst_cols * rows + 64 * bv.n_points + 32 * (bv.n_scalars + bv.n_challenges))
        out = {
            "metric": METRIC, "value": proofs_per_step * steps / dt, "unit": UNIT, "n_gpus": world, "steps": steps, "warmup": W,
            "ms_per_step": dt / steps * 1e3, "higher_is_better": True, "scaling": cfg["scaling"], "vs_baseline": None,
            "dtype": "u32x8 (256-bit Montgomery integers)",
            "data": ("synthetic (trapdoor-simulated accepting proofs, seeded; the same two 65,536-proof global batches for every N: 4096 distinct proofs, tiled)" if strong else
                     "synthetic (trapdoor-simulated accepting proofs, seeded; two distinct 4096-proof batches per rank)"),
            "config": {"workload": f"{cfg['name']}; shape '{shape}', k={k}, Blake2b transcript, {rows} public inputs, {bv.proof_len}-byte proofs",
                       "batch": args.batch, "proofs_per_gpu_and_batch": n, "global_batch": n * world,
                       "step": f"one launch set = {G} independent global batch(es) of {n * world} proofs ({n} per GPU): every batch has its own fold coefficients, "
                               f"its own MSM, its own pairing check and its own verdict; they share one set of kernel launches (h2v_batch_set_fold_groups)",
                       "proofs_per_step": proofs_per_step, "fold_groups_per_launch_set": G, "contexts_in_flight": n_ctx,
                       "timed_blocks": R, "block_ms": [round(x * 1e3, 3) for x in block_dt],
                       "timing": f"{R} timed blocks of {steps} steps, each between barrier + synchronize on both sides; a block's time = CUDA events on the contexts' "
                                 f"streams (first start -> last end), max over ranks; `value` = proofs of a block / MEDIAN block time; e2e on the host clock around the C-ABI calls",
                       "host_waits": "blocking" if blocking else "spinning",
                       "l2": "flushed before every step (256 MiB overwrite on the step's stream, inside the timed region)",
                       "fold_randomness": "resident path: fixed key (h2v_batch_set_rlc_key); e2e: OS entropy per call (h2v.h: no scalars, no key, seed 0)",
                       "parallelism": (f"proof-sharded x{world}: device-side exchange (csrc/exchange.cuh) - each rank's pack kernel stores its per-window partial accumulators "
                                       f"(12,320 B per global batch) into the root's HBM window over NVLink, the root (rank i mod N for launch set i) sums them in place, runs the "
                                       f"pairing check(s) and stores the verdicts into every rank's window; all inside the CUDA graph, no host or NCCL call per step")
                       if world > 1 else "one GPU"},
            "e2e": {"value": proofs_per_step * steps / dt_e2e, "unit": UNIT, "h2d_bytes_per_step": gbatches[0].h2d_bytes, "d2h_bytes_per_step": gbatches[0].d2h_bytes,
                    "ms_per_step": dt_e2e / steps * 1e3, "block_ms": [round(x * 1e3, 3) for x in block_e2e], "p50_latency_ms_one_batch": p50},
            "one_in_flight": {"value": n * world * steps / dt1, "ms_per_batch": dt1 / steps * 1e3, "e2e_value": n * world * steps / dt_e2e1,
                              "e2e_p50_latency_ms": p50, "note": f"strictly serial single batches of {n * world} proofs on one context"},
            "gpu_launches": int(launches),
            "clocks": clocks,
            "stage_ms": {k_: round(v, 4) for k_, v in stage_ms.items()},
            "kernel_ms": {k_: round(v, 4) for k_, v in kern_ms.items()},
            "msm": {"window_bits": [geom_tp["window_bits"] & 0xFFFF, geom_tp["window_bits"] >> 16], "windows": [geom_tp["windows"] & 0xFFFF, geom_tp["windows"] >> 16],
                    "terms": geom_tp["terms"], "buckets": geom_tp["buckets"],
                    "one_in_flight": {"window_bits": [geom["window_bits"] & 0xFFFF, geom["window_bits"] >> 16], "buckets": geom["buckets"]}},
            "roofline": roof,
            "input_generation_s": round(gen_s, 2),
        }
        if stage_ms:
            t_eval = (stage_ms["transcript"] + stage_ms["scalar"]) * 1e-3
            out["roofline_hbm"] = {"bound": "hbm", "kernel": "transcript+scalar (evaluation loads)", "achieved": eval_bytes / t_eval / 1e9, "peak": hbm_peak,
                                   "peak_source": hbm_src, "unit": "GB/s", "frac": eval_bytes / t_eval / 1e9 / hbm_peak, "traffic": None}
        if selfcheck is not None:
            out["selfcheck"] = selfcheck
    if world == 1 and args.config == 2 and not args.no_config3:
        c3 = config3_leg(args, pkg, torch)
        if out is not None:
            out["config3_gwc_attribution"] = c3
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        out["cpu_baseline"] = cpu_baseline_from_batch(synth.params_bytes_raw(k, s), vk_bytes, batches[0], budget_s=args.cpu_budget)
    if dist is not None:
        dist.barrier()
        dist.destroy_process_group()
    for b in bvs:
        b.close()
    return out


# ------------------------------------------------------------------------------------------------
# --selfcheck: the sharded product path against the C oracle (checker only), on the bench's own inputs
# ------------------------------------------------------------------------------------------------
def run_selfcheck(args, pkg, lib, torch, dist, synth, sharding, bv, pb, rank, world, n, gbase, gcount, params_bytes, vk_bytes):
    """(1) clean global batch with GLOBAL explicit coefficients: the folded (L, R) the root computed from the gathered
    partials == the C oracle's fold of every proof's accumulators (so they are identical for every shard count);
    (2) one corrupted proof on the LAST rank (not the root): every rank learns the rejection, the statuses of every
    shard == the C oracle's per-proof verdicts."""
    import random

    import numpy as np

    cores = max(1, (os.cpu_count() or 1) // world)
    co = _load_c_oracle(params_bytes, vk_bytes)
    proofs, insts = pb.src
    rng = random.Random(20261018)
    rs = [rng.randrange(1, R_MOD) for _ in range(gcount)]  # the same on every rank
    root = 0
    if world == 1:
        res = bv.verify_batch(proofs, insts, rlc_scalars=rs, want_batch_accum=True)
        ok, status, folded = res.verdict, res.status, res.batch_accum
    else:
        verdicts, status = bv.verify_shard(proofs, insts, gbase, gcount, root, rlc_scalars=rs)
        ok = verdicts[0]
        folded = bv.comm_last_batch_accum() if rank == root else None
    assert ok and status == [0] * n, "selfcheck: clean batch rejected"
    # C oracle: per-proof accumulators of this shard, folded with the global coefficients of the shard
    proofs_np, inst_np = pb.proofs.numpy(), pb.inst.numpy()
    poff, ioff = pb.poff.numpy().view(np.uint64), pb.ioff.numpy().view(np.uint64)
    st, _, lr, _ = co.verify_many(proofs_np, poff, inst_np, ioff, n, "shplonk", "blake2b", False, cores, want_lr=True)
    assert int(st.max()) == 0
    tail = 1
    for r_ in rs[gbase + n:]:
        tail = tail * r_ % R_MOD
    part, _ = co.fold(lr + bytes(128), rs[gbase:gbase + n] + [tail], [1] * n + [0])  # the dummy last entry carries the product of the later ranks' r_i
    parts = sharding.all_gather_bytes(part, world)
    match = None
    if rank == root:
        dec = lambda e: None if e == bytes(64) else (int.from_bytes(e[:32], "little"), int.from_bytes(e[32:], "little"))
        enc = lambda p: bytes(64) if p is None else p[0].to_bytes(32, "little") + p[1].to_bytes(32, "little")
        L = R_ = None
        for p in parts:
            L, R_ = synth.g1_add(L, dec(p[:64])), synth.g1_add(R_, dec(p[64:]))
        match = folded == enc(L) + enc(R_)
        assert match, "selfcheck: folded (L, R) differ from the C oracle's"
    # corrupted proof on the last rank
    bad_rank, j_bad = world - 1, 17 % n
    bad = list(proofs)
    if rank == bad_rank:
        b = bytearray(bad[j_bad])
        b[(bv.n_points - bv.n_mo) * 32 + 1] ^= 0x40  # an evaluation scalar: still canonical, wrong value
        bad[j_bad] = bytes(b)
    pbb = PackedBatch(torch, bad, insts)
    if world == 1:
        res = bv.verify_batch(bad, insts, rlc_scalars=rs)
        ok2, status2 = res.verdict, res.status
    else:
        verdicts, status2 = bv.verify_shard(bad, insts, gbase, gcount, root, rlc_scalars=rs)
        ok2 = verdicts[0]
    st2, _, _, _ = co.verify_many(pbb.proofs.numpy(), pbb.poff.numpy().view(np.uint64), pbb.inst.numpy(), pbb.ioff.numpy().view(np.uint64), n,
                                  "shplonk", "blake2b", True, cores)
    assert not ok2, "selfcheck: the corrupted global batch was accepted"
    assert status2 == [int(x) for x in st2], "selfcheck: statuses differ from the C oracle's"
    assert (sum(1 for x in status2 if x) == 1 and status2[j_bad] == 4) if rank == bad_rank else not any(status2)
    co.close()
    flag = torch.ones(1, dtype=torch.int32, device="cuda")
    if dist is not None:
        dist.all_reduce(flag, op=dist.ReduceOp.MIN)
    folded_hex = None
    if rank == root:
        import hashlib

        folded_hex = hashlib.sha256(folded).hexdigest()
    return {"ranks_ok": int(flag.item()) == 1, "global_batch": gcount, "folded_LR_equals_c_oracle": match, "folded_LR_sha256": folded_hex,
            "corrupted_proof": {"rank": bad_rank, "index_in_shard": j_bad, "root": root, "global_verdict": "rejected", "statuses_equal_c_oracle": True},
            "note": "explicit global fold coefficients (seeded) so that the folded (L, R) are comparable across shard counts; checker = oracle/c"}


# ------------------------------------------------------------------------------------------------
# BASELINE.json configs[2]: GWC, 4096-proof batch, 1 % corrupted proofs -> the fold is rejected and attributed per proof
# ------------------------------------------------------------------------------------------------
def _gwc_gen_worker(job):
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import random

    import prover_sim as sim

    shape, k, s, seed = job
    params = sim.make_params(k, s)
    vk, dl = sim.make_vk(shape, k)
    rng = random.Random(seed)
    inst = sim.random_instances(vk, rng, 10)
    return inst[0], sim.simulate_proof(params, vk, dl, s, inst, rng, "gwc", "blake2b")


def config3_leg(args, pkg, torch):
    """Clean and 1 %-corrupted 4096-proof GWC batches end to end through h2v_verify_batch (host clock, median of 7);
    statuses of the corrupted batch against the C oracle.  The GWC inputs come from the oracle's proof simulator
    (64 distinct proofs, tiled) and its corruption injector: input generation and checking only, not the measured path."""
    import random
    from multiprocessing import get_context

    import numpy as np

    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import formats as F
    import prover_sim as sim

    n, distinct, k, shape = 4096, 64, args.k, "vm"
    s = srs_secret(k)
    params = sim.make_params(k, s)
    vk, _dl = sim.make_vk(shape, k)
    with get_context("spawn").Pool(min(os.cpu_count() or 1, 16)) as pool:
        items = pool.map(_gwc_gen_worker, [(shape, k, s, 3000003 + i) for i in range(distinct)])
    proofs = [it[1] for it in items] * (n // distinct)
    insts = [[[int(v).to_bytes(32, "little") for v in col] for col in it[0]] for it in items] * (n // distinct)
    rng = random.Random(3)
    idx = sorted(rng.sample(range(n), n // 100))
    kinds = list(sim.CORRUPTIONS)
    bad = list(proofs)
    for t, i in enumerate(idx):
        bad[i], _ = sim.corrupt(proofs[i], vk, kinds[t % len(kinds)], rng, "gwc")
    pvk = pkg.VerifyingKey.from_bytes(vk.to_bytes(F.RAW_BYTES), pkg.SerdeFormat.RawBytes)
    bv = pkg.BatchVerifier(pkg.ParamsKZG.from_bytes(params.to_bytes(F.RAW_BYTES), pkg.SerdeFormat.RawBytes), pvk, "gwc", "blake2b", device=0)
    lib = bv.lib
    clean, dirty = PackedBatch(torch, proofs, insts), PackedBatch(torch, bad, insts)

    def timed(pb):
        ts = []
        for _ in range(9):
            a = time.perf_counter()
            bv._check(lib.h2v_verify_batch(bv._ctx, *pb.args(), None, 0, pb.status.data_ptr(), None, None, None))
            ts.append(time.perf_counter() - a)
        return statistics.median(ts[2:]) * 1e3

    ms_clean = timed(clean)
    assert int(clean.status.max()) == 0
    ms_bad = timed(dirty)
    att = bv.timings()
    got = [int(x) for x in dirty.status]
    co = _load_c_oracle(params.to_bytes(F.RAW_BYTES), vk.to_bytes(F.RAW_BYTES))
    st, _, _, _ = co.verify_many(dirty.proofs.numpy(), dirty.poff.numpy().view(np.uint64), dirty.inst.numpy(), dirty.ioff.numpy().view(np.uint64), n,
                                 "gwc", "blake2b", True, os.cpu_count() or 1)
    co.close()
    same = got == [int(x) for x in st]
    assert same and [i for i, x in enumerate(got) if x] == idx, "config 3: statuses differ from the C oracle's"
    bv.close()
    return {"workload": "BASELINE.json configs[2]: 4096 GWC proofs (vector_mul shape, k=10, 1,056-byte proofs), h2v_verify_batch from pinned host buffers, median of 7",
            "clean_ms": round(ms_clean, 3), "corrupted_1pct_ms": round(ms_bad, 3), "ratio": round(ms_bad / ms_clean, 3),
            "clean_proofs_per_s": n / (ms_clean * 1e-3), "corrupted_1pct_proofs_per_s": n / (ms_bad * 1e-3),
            "corrupted_proofs": len(idx), "statuses_equal_c_oracle": same, "last_call_ms": {k_: round(v, 3) for k_, v in att.items() if v}}


# ------------------------------------------------------------------------------------------------
# CPU arm: the C oracle (oracle/c: restatement of the reference's algorithm, SingleStrategy = one
# windowed serial MSM pair + one 2-pair pairing per proof), one thread per host core
# ------------------------------------------------------------------------------------------------
def _load_c_oracle(params_bytes, vk_bytes):
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import c_oracle

    return c_oracle.COracle(params_bytes, 1, vk_bytes, 1)


def _cpu_rate(co, proofs_np, poff, inst_np, ioff, n, threads):
    st, secs, _, _ = co.verify_many(proofs_np, poff, inst_np, ioff, n, "shplonk", "blake2b", True, threads)
    assert int(st.max()) == 0, "the CPU oracle rejected a valid proof"
    return n / secs, secs


CPU_KIND_NOTE = ("C restatement of the reference algorithm (oracle/c: verify_proof with SingleStrategy, i.e. the reference's serial windowed "
                 "MSM and one 2-pair pairing per proof; 4x64-bit Montgomery arithmetic like halo2curves without asm; G2 lines prepared once "
                 "per VK, which favours the CPU), pthreads over proofs; NOT the Rust binary (no Rust toolchain / network in this image)")


def cpu_baseline_from_batch(params_bytes, vk_bytes, pb, budget_s=12.0):
    """Times the C oracle on a bounded prefix of the batch the GPU just verified."""
    import numpy as np

    cores = os.cpu_count() or 1
    co = _load_c_oracle(params_bytes, vk_bytes)
    proofs_np, inst_np = pb.proofs.numpy(), pb.inst.numpy()
    poff, ioff = pb.poff.numpy().view(np.uint64), pb.ioff.numpy().view(np.uint64)
    n0 = min(pb.n, 4 * cores)
    rate, _ = _cpu_rate(co, proofs_np, poff, inst_np, ioff, n0, cores)
    n1 = int(max(n0, min(pb.n, rate * budget_s)))
    rate, secs = _cpu_rate(co, proofs_np, poff, inst_np, ioff, n1, cores)
    # latency of ONE verify_proof on one core (the shape of BASELINE.json configs[0]; the exact k = 8 fixture case: tools/config1_cpu_latency.py)
    one = []
    for _ in range(200):
        _, s1, _, _ = co.verify_many(proofs_np, poff, inst_np, ioff, 1, "shplonk", "blake2b", True, 1)
        one.append(s1 * 1e3)
    co.close()
    return {"value": rate, "unit": UNIT, "cores": cores, "kind": "port", "single_verify_proof_p50_ms_one_core": round(statistics.median(one), 4),
            "sample": f"first {n1} proofs of the timed 4096-proof batch, {secs:.1f} s on {cores} threads; " + CPU_KIND_NOTE}


def _gen_worker(job):
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import random

    import prover_sim as sim

    shape, k, s, seed = job
    params = sim.make_params(k, s)
    vk, dl = sim.make_vk(shape, k)
    rng = random.Random(seed)
    inst = sim.random_instances(vk, rng, 10)
    return inst[0], sim.simulate_proof(params, vk, dl, s, inst, rng)


def run_reference(args):
    """The reference arm: CPU only, no CUDA code of this repository on the path.  Inputs come from the oracle's own
    proof simulator (a few distinct proofs, tiled: the verifier's cost does not depend on the witness)."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return None
    import numpy as np
    from multiprocessing import get_context

    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import formats as F
    import prover_sim as sim

    cores = os.cpu_count() or 1
    s = srs_secret(args.k)
    params = sim.make_params(args.k, s)
    vk, _dl = sim.make_vk(args.shape, args.k)
    distinct = max(8, min(64, cores))
    with get_context("spawn").Pool(min(cores, distinct)) as pool:
        items = pool.map(_gen_worker, [(args.shape, args.k, s, 1000003 + i) for i in range(distinct)])
    co = _load_c_oracle(params.to_bytes(F.RAW_BYTES), vk.to_bytes(F.RAW_BYTES))
    per_step = max(distinct, args.ref_proofs_per_core * cores)
    reps = -(-per_step // distinct)
    proofs = [it[1] for it in items] * reps
    insts = [it[0] for it in items] * reps
    n = len(proofs)
    proofs_np = np.frombuffer(b"".join(proofs), dtype=np.uint8)
    poff = np.cumsum([0] + [len(p) for p in proofs]).astype(np.uint64)
    inst_np = np.frombuffer(b"".join(int(v).to_bytes(32, "little") for inst in insts for col in inst for v in col), dtype=np.uint8)
    ioff = np.cumsum([0] + [sum(len(c) for c in inst) for inst in insts]).astype(np.uint64)
    for _ in range(max(args.warmup, 0)):
        _cpu_rate(co, proofs_np, poff, inst_np, ioff, min(n, 2 * cores), cores)
    vals, t_all = [], time.perf_counter()
    for _ in range(args.steps):
        vals.append(_cpu_rate(co, proofs_np, poff, inst_np, ioff, n, cores)[0])
    wall_all = time.perf_counter() - t_all
    v = statistics.median(vals)
    sample = f"each step verifies {n} proofs of the workload ({distinct} distinct, tiled) on {cores} threads; " + CPU_KIND_NOTE
    return {
        "impl": "reference", "metric": METRIC, "value": v, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": wall_all / max(1, args.steps) * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "u64x4 (256-bit Montgomery integers, CPU)", "data": "synthetic (trapdoor-simulated accepting proofs, seeded)",
        "config": {"workload": f"bounded sample of: {args.batch} SHPLONK proofs per GPU, vector_mul test-circuit shape ('{args.shape}'), k={args.k}, "
                               f"Blake2b transcript, 10 public inputs, 1,024-byte proofs; BASELINE.json configs[1]"},
        "cpu_baseline": {"value": v, "unit": UNIT, "cores": cores, "kind": "port", "sample": sample},
        "e2e": {"value": v, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }


def main():
    # stdout must carry exactly one JSON line: libraries (e.g. NCCL with NCCL_DEBUG set) print there too, so
    # everything else goes to stderr and the JSON is written to the saved descriptor at the end
    real_stdout = os.dup(1)
    os.dup2(2, 1)
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20, help="timed launch sets (of each timed block)")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--blocks", type=int, default=1, help="timed blocks of --steps steps; the median block is reported")
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", type=int, default=2, choices=sorted(CONFIGS), help="BASELINE.json configuration (2 = configs[1], the headline)")
    ap.add_argument("--batch", type=int, default=0)
    ap.add_argument("--shape", default="")
    ap.add_argument("--k", type=int, default=0)
    ap.add_argument("--streams", type=int, default=int(os.environ.get("H2V_BENCH_STREAMS", "0")),
                    help="contexts (CUDA stream + host thread each) per GPU; default 4")
    ap.add_argument("--fold-groups", type=int, default=int(os.environ.get("H2V_BENCH_FOLD_GROUPS", "0")),
                    help="independent batches (own fold + pairing check each) per launch set of a context; default 16")
    ap.add_argument("--selfcheck", action="store_true", help="also check the (sharded) path against the C oracle, incl. a corrupted proof on a non-root rank")
    ap.add_argument("--no-config3", action="store_true", help="skip the GWC attribution leg (BASELINE.json configs[2]) of the N=1 line")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--cpu-budget", type=float, default=12.0)
    ap.add_argument("--ref-proofs-per-core", type=int, default=64)
    ap.add_argument("--dump-outputs", metavar="DIR", help="write what the last timed step returned to DIR/<name>.npy (float32)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    cfg = CONFIGS[args.config]
    args.batch = args.batch or cfg["batch"]
    args.shape = args.shape or cfg["shape"]
    args.k = args.k or cfg["k"]
    # 64 batches in flight per GPU: 4 contexts x 16 fold groups (the driver's --steps 20 then spreads evenly over the contexts; fewer host
    # threads and fewer, larger launch sets also measured better at 8 ranks on one host)
    if args.streams <= 0:
        args.streams = 4
    if args.fold_groups <= 0:
        args.fold_groups = 16 if args.config == 2 else (8 if args.config == 4 else 0)
    out = run_reference(args) if args.impl == "reference" else run_ours(args)
    sys.stdout.flush()
    if out is not None:
        os.write(real_stdout, (json.dumps(out) + "\n").encode())


if __name__ == "__main__":
    main()
