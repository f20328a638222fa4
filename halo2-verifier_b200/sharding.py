"""Multi-GPU plumbing (one process per GPU): contiguous proof shards, globally defined fold
coefficients, one exchange step per global batch (SURVEY.md section 8(e)).

Data plane, in order of preference:

* **device-side exchange** (`connect_channel` succeeded; `include/h2v.h`, `csrc/exchange.cuh`): every rank's
  context owns a window in HBM that the peers map through CUDA IPC.  The shard's packing kernel stores its
  per-window partial sums into the ROOT rank's window over NVLink, the root waits on sequence numbers, sums
  in place, runs the single pairing check and stores the verdict into every rank's window - all inside the
  captured CUDA graph, no host thread, no library collective, and only the root receives data (a gather).
  `torch.distributed` is used ONCE, at start-up, to ship the 128-byte window handles (and, per batch, 32
  bytes of fold key).
* **library gather** (ranks that cannot map each other's memory, e.g. several nodes): `h2v_accumulate_shard`
  leaves the partial in device memory, `torch.distributed.gather` (NCCL) moves it to the root only, the root
  sums it in place (`h2v_finalize*` on the device pointer) and broadcasts the verdicts.

NCCL cannot reduce with an elliptic-curve addition, hence gather-then-add in both.  On rejection every rank
attributes inside its own shard, and only inside rejected fold groups (reference contract poly/strategy.rs:26-30).
"""
import os
from typing import List, Optional, Tuple

import torch
import torch.distributed as dist


def shard_range(n: int, rank: int, world: int) -> Tuple[int, int]:
    """Contiguous range [lo, hi) of global proof indices owned by `rank`."""
    base, rem = divmod(n, world)
    lo = rank * base + min(rank, rem)
    return lo, lo + base + (1 if rank < rem else 0)


def _pg_device(group=None):
    """device the process group's backend moves tensors on (NCCL: the current CUDA device; gloo: the host)"""
    return torch.device("cuda", torch.cuda.current_device()) if dist.get_backend(group) == "nccl" else torch.device("cpu")


def all_gather_bytes(blob: bytes, world: int, group=None) -> List[bytes]:
    """Every rank's `blob` (equal length), rank order: the start-up plumbing of the exchange (window handles)."""
    if world == 1:
        return [bytes(blob)]
    dev = _pg_device(group)
    t = torch.frombuffer(bytearray(blob), dtype=torch.uint8).to(dev)
    out = [torch.empty_like(t) for _ in range(world)]
    dist.all_gather(out, t, group=group)
    return [bytes(o.cpu().numpy().tobytes()) for o in out]


def all_gather_partials(partial: torch.Tensor, world: int) -> List[bytes]:
    """partial: uint8[...] of this rank, on the device of the process group's backend.  Returns every rank's
    partial as bytes, rank order (kept for the host-logic tests; the product paths below gather to the root only)."""
    assert partial.dtype == torch.uint8 and partial.dim() == 1
    if world == 1:
        return [bytes(partial.cpu().numpy().tobytes())]
    out = [torch.empty_like(partial) for _ in range(world)]
    dist.all_gather(out, partial)
    return [bytes(t.cpu().numpy().tobytes()) for t in out]


def connect_channel(bv, rank: int, world: int, max_groups: int = 1, group=None) -> bool:
    """Builds the device-side exchange channel of `bv` (one context per rank, called by every rank in the same
    order): allocates the window, ships the handles, maps the peers.  Returns False (and leaves `bv` on the
    library-gather path) when the peers cannot be mapped."""
    from . import BackendError

    handle = bv.comm_init(rank, world, max_groups)
    handles = all_gather_bytes(handle, world, group)
    ok = 1
    try:
        bv.comm_connect(handles)
    except BackendError:
        ok = 0
    if world > 1:  # all or nothing: a channel works only if every rank mapped every peer
        flag = torch.tensor([ok], dtype=torch.int32, device=_pg_device(group))
        dist.all_reduce(flag, op=dist.ReduceOp.MIN, group=group)
        ok = int(flag.item())
    bv.comm_ready = bool(ok)
    return bool(ok)


def fresh_fold_key(world: int, group=None, src: int = 0) -> bytes:
    """One 256-bit secret per global batch, drawn from the OS on `src` and given to every rank, so that the fold
    coefficients c_j are defined globally (the folded (L, R) do not depend on the shard count).  The reference draws
    its r_i from the OS too (strategy.rs:129)."""
    if world == 1:
        return os.urandom(32)
    dev = _pg_device(group)
    t = torch.frombuffer(bytearray(os.urandom(32)), dtype=torch.uint8).to(dev)
    dist.broadcast(t, src=src, group=group)
    return bytes(t.cpu().numpy().tobytes())


def _gather_to_root(part: torch.Tensor, root: int, rank: int, world: int, group=None) -> Optional[torch.Tensor]:
    """library gather of the device-resident partial blobs to `root` only ([rank][...] order); None elsewhere"""
    if world == 1:
        return part
    if rank == root:
        out = torch.empty(world * part.numel(), dtype=torch.uint8, device=part.device)
        dist.gather(part, list(out.chunk(world)), dst=root, group=group)
        # The collective is asynchronous to the host and ordered only against torch's current stream; the context's own stream
        # (cudaStreamNonBlocking) reads `out` next (h2v_finalize*), so the host waits for the gather here.  Without this wait the
        # finalize raced the incoming partials (2-GPU test: a rejected / accepted pair of fold groups came out wrong once the
        # root's kernels got faster than the peer's send).
        if out.is_cuda:
            torch.cuda.current_stream(out.device).synchronize()
        return out
    dist.gather(part, None, dst=root, group=group)
    return None


def _randomness(rlc_scalars, seed, key, world, group):
    """explicit scalars / explicit key / test seed pass through; otherwise a fresh global key"""
    if rlc_scalars is None and seed is None and key is None:
        key = fresh_fold_key(world, group)
    return rlc_scalars, seed, key


def verify_batches_sharded(bv, batches, rank: int, world: int, rlc_scalars=None, seed=None, key=None, root: int = 0, group=None):
    """`batches`: G global batches [(proofs, instances), ...] of EQUAL size n, each sharded over the ranks; every rank
    processes its shard of all G batches in ONE set of kernel launches (fold groups, include/h2v.h); the G partials of a
    rank reach `root`, which runs the G pairing checks together.  `rlc_scalars`: G * n coefficients (batch-major) or
    None (then `seed`, a test seed, or `key`, or - default - a fresh secret key drawn on rank 0 for this call).
    Returns (G verdicts, statuses of this rank's shard of every batch)."""
    G, n = len(batches), len(batches[0][0])
    assert all(len(p) == n and len(i) == n for p, i in batches) and n % world == 0, "equal batches, equal shards"
    lo, hi = shard_range(n, rank, world)
    proofs = [p for pr, _ in batches for p in pr[lo:hi]]
    insts = [i for _, ins in batches for i in ins[lo:hi]]
    rlc_scalars, seed, key = _randomness(rlc_scalars, seed, key, world, group)
    if getattr(bv, "comm_ready", False):  # device-side exchange
        verdicts, status = bv.verify_shard(proofs, insts, lo, n, root, rlc_scalars=rlc_scalars, seed=seed, key=key, fold_groups=G)
    else:  # library gather of device-resident partials to the root
        dev = _pg_device(group) if world > 1 else torch.device("cuda", torch.cuda.current_device())
        part = torch.empty(G * bv.lib.h2v_partial_bytes(), dtype=torch.uint8, device=dev)
        status, _ = bv.accumulate_shard(proofs, insts, lo, n, rlc_scalars=rlc_scalars, seed=seed, key=key, fold_groups=G, partial_out=part.data_ptr())
        parts = _gather_to_root(part, root, rank, world, group)
        flags = torch.zeros(G, dtype=torch.int32, device=dev)
        if rank == root:
            flags[:] = torch.tensor([1 if v else 0 for v in bv.finalize_groups(parts.data_ptr(), G, n_partials=world)], dtype=torch.int32)
        if world > 1:
            dist.broadcast(flags, src=root, group=group)
        verdicts = [bool(v) for v in flags.tolist()]
        if not all(verdicts):  # attribution inside this rank's shards of the REJECTED batches only
            status = bv.attribute_shard(status, group_verdicts=verdicts)
    per = hi - lo
    return verdicts, [status[q * per:(q + 1) * per] for q in range(G)]


def verify_batch_sharded(bv, proofs, instances, rank: int, world: int, rlc_scalars=None, seed=None, key=None, root: int = 0, group=None):
    """Every rank calls this with the WHOLE batch description (or at least its own shard's data at
    the right indices); returns (global verdict, statuses of this rank's shard).  Shards may differ in size by one."""
    n = len(proofs)
    lo, hi = shard_range(n, rank, world)
    hint = shard_range(n, 0, world)[1]  # largest shard: common window geometry on every rank
    rlc_scalars, seed, key = _randomness(rlc_scalars, seed, key, world, group)
    if getattr(bv, "comm_ready", False):
        verdicts, status = bv.verify_shard(proofs[lo:hi], instances[lo:hi], lo, n, root, rlc_scalars=rlc_scalars, seed=seed, key=key, shard_hint=hint)
        return verdicts[0], status
    dev = _pg_device(group) if world > 1 else torch.device("cuda", torch.cuda.current_device())
    part = torch.empty(bv.lib.h2v_partial_bytes(), dtype=torch.uint8, device=dev)
    status, _ = bv.accumulate_shard(proofs[lo:hi], instances[lo:hi], lo, n, rlc_scalars=rlc_scalars, seed=seed, key=key, shard_hint=hint,
                                    partial_out=part.data_ptr())
    parts = _gather_to_root(part, root, rank, world, group)
    flag = torch.zeros(1, dtype=torch.int32, device=dev)
    if rank == root:
        ok, _ = bv.finalize(parts.data_ptr(), want_batch_accum=False, n_partials=world)
        flag[0] = 1 if ok else 0
    if world > 1:
        dist.broadcast(flag, src=root, group=group)
    ok = bool(flag.item())
    if not ok:  # rejected fold: every rank attributes inside its own shard, no further exchange
        status = bv.attribute_shard(status)
    return ok, status


def mixed_shard_counts(global_counts, base: int, n: int) -> List[int]:
    """proofs per member of the range [base, base + n) of the member-major concatenation of global_counts proofs"""
    out, lo = [], 0
    for c in global_counts:
        out.append(max(0, min(lo + c, base + n) - max(lo, base)))
        lo += c
    return out


def mixed_shard(global_counts, rank: int, world: int):
    """`rank`'s share of a mixed batch of global_counts[m] proofs per member: (lo, hi) of the member-major concatenation
    (shard_range over its N proofs) and, per member, the [lo_m, hi_m) indices into that member's own proof list."""
    lo, hi = shard_range(sum(global_counts), rank, world)
    per, start = [], 0
    for c, k in zip(global_counts, mixed_shard_counts(global_counts, lo, hi - lo)):
        first = min(max(lo - start, 0), c)
        per.append((first, first + k))
        start += c
    return (lo, hi), per


def verify_mixed_batch_sharded(mix, proofs_per_member, instances_per_member, rank: int, world: int, rlc_scalars=None, seed=None, key=None,
                               root: int = 0, group=None):
    """A mixed batch (the whole description on every rank, or at least this rank's share at the right indices) split over the
    ranks as mixed_shard does: each rank folds its share with globally defined coefficients, `root` runs the one pairing check
    (through the device-side exchange when mix.comm_ready, otherwise a library gather of the device-resident partials), and
    a rejection is attributed per proof by every rank inside its share.  Returns (global verdict, this rank's statuses per member)."""
    global_counts = [len(p) for p in proofs_per_member]
    (lo, hi), per = mixed_shard(global_counts, rank, world)
    hint = max(b - a for a, b in (shard_range(sum(global_counts), r, world) for r in range(world)))  # common window geometry
    proofs = [p[a:b] for p, (a, b) in zip(proofs_per_member, per)]
    insts = [i[a:b] for i, (a, b) in zip(instances_per_member, per)]
    rlc_scalars, seed, key = _randomness(rlc_scalars, seed, key, world, group)
    if getattr(mix, "comm_ready", False):
        return mix.verify_shard(proofs, insts, global_counts, lo, root, rlc_scalars=rlc_scalars, seed=seed, key=key, shard_hint=hint)
    dev = _pg_device(group) if world > 1 else torch.device("cuda", torch.cuda.current_device())
    part = torch.empty(mix.partial_bytes(global_counts), dtype=torch.uint8, device=dev)
    status, _ = mix.accumulate_shard(proofs, insts, global_counts, lo, rlc_scalars=rlc_scalars, seed=seed, key=key, shard_hint=hint,
                                     partial_out=part.data_ptr())
    parts = _gather_to_root(part, root, rank, world, group)
    flag = torch.zeros(1, dtype=torch.int32, device=dev)
    if rank == root:
        ok, _ = mix.finalize(parts.data_ptr(), global_counts, want_batch_accum=False, n_partials=world)
        flag[0] = 1 if ok else 0
    if world > 1:
        dist.broadcast(flag, src=root, group=group)
    ok = bool(flag.item())
    if not ok:
        status = mix.attribute_shard(status)
    return ok, status


def split_group_partials(rank_blob: bytes, groups: int) -> List[bytes]:
    """One rank's output of a launch set with `groups` fold groups = `groups` consecutive partials."""
    assert len(rank_blob) % groups == 0
    step = len(rank_blob) // groups
    return [rank_blob[q * step:(q + 1) * step] for q in range(groups)]
