"""halo2-verifier_b200: B200-native batch verifier for Halo2 KZG proofs (BN254).

Host-side mirror of the reference's verification surface (ChainSafe/halo2-verifier):

    reference (Rust)                                   here
    -------------------------------------------------  ------------------------------------------
    ParamsKZG::{read, from_bytes, read_custom}         ParamsKZG.{read, from_bytes}
      poly/kzg/commitment.rs:133-232
    VerifyingKey::{read, from_bytes}                   VerifyingKey.{read, from_bytes}
      plonk/vk.rs:76-127
    SerdeFormat  helpers.rs:7-19                       SerdeFormat
    verify_proof::<Scheme, V, E, T, Strategy>(..)      verify_proof(params, vk, proof, instances,
      lib.rs:33-46                                                  multiopen=, transcript=)
    VerifierSHPLONK | VerifierGWC                      multiopen="shplonk" | "gwc"
    Blake2bRead | Keccak256Read (+Challenge255)        transcript="blake2b" | "keccak256"
    plonk::Error  plonk/mod.rs:19-32                   Error subclasses
    (added) verify_proofs_batch                        verify_proofs_batch(..) / BatchVerifier
    AccumulatorStrategy over proofs of several VKs     verify_proofs_mixed(..) / MixedBatchVerifier
      poly/kzg/strategy.rs:125-140
    (added) one pairing check over several params     verify_proofs_mixed(.., multi_params=True) / MixedBatchVerifier
    AccumulatorStrategy across calls: process, finalize  Accumulator.{absorb, finalize, to_bytes, merge}
      poly/kzg/strategy.rs:125-140
    (snark-verifier) KZG accumulator in the instances    accumulator=InstanceAccumulator(limbs, bits, cells)
      of an aggregation proof, its deferred decider

All arithmetic runs in the CUDA library `libh2v_b200.so` behind the C ABI in include/h2v.h.
There is NO CPU fallback: importing works anywhere, but creating a verifier without the built
library or without a CUDA device raises.
"""
import ctypes
import enum
import os
from dataclasses import dataclass
from typing import List, Optional, Sequence, Tuple

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libh2v_b200.so")

R_MODULUS = 0x30644E72E131A029B85045B68181585D2833E84879B9709143E1F593F0000001


class SerdeFormat(enum.IntEnum):
    Processed = 0
    RawBytes = 1
    RawBytesUnchecked = 2


class Error(Exception):
    """plonk::Error (reference plonk/mod.rs:19-32)."""


class InvalidInstances(Error):
    pass


class TranscriptError(Error):
    pass


class OpeningError(Error):
    pass


class ConstraintSystemFailure(Error):
    pass


class ReferenceWouldPanic(Error):
    """Inputs on which the reference unwraps None (vanishing.rs:100, shplonk.rs:215)."""


class BackendError(RuntimeError):
    """Infrastructure failure: library missing, CUDA error, malformed VK / params."""


STATUS_ERRORS = {
    1: InvalidInstances,
    2: TranscriptError,
    3: OpeningError,
    4: ConstraintSystemFailure,
    5: ReferenceWouldPanic,
}

_MULTIOPEN = {"shplonk": 0, "gwc": 1}
_HASH = {"blake2b": 0, "keccak256": 1, "keccak": 1}

_lib = None


def load_library():
    """Loads the CUDA library; fails loudly if it has not been built (see __graft_entry__.build)."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise BackendError(f"{LIB_PATH} is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'`")
    lib = ctypes.CDLL(LIB_PATH)
    u8p, u32p, u64p = ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p
    lib.h2v_ctx_create.argtypes = [ctypes.POINTER(ctypes.c_void_p), ctypes.c_char_p, ctypes.c_size_t, ctypes.c_int,
                                   ctypes.c_char_p, ctypes.c_size_t, ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_int]
    lib.h2v_ctx_create_multi.argtypes = [ctypes.POINTER(ctypes.c_void_p), ctypes.c_char_p, ctypes.c_size_t, ctypes.c_int,
                                         ctypes.c_char_p, ctypes.c_size_t, ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_uint32]
    lib.h2v_ctx_create_aggregation.argtypes = [ctypes.POINTER(ctypes.c_void_p), ctypes.c_char_p, ctypes.c_size_t, ctypes.c_int,
                                               ctypes.c_char_p, ctypes.c_size_t, ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_int,
                                               ctypes.c_uint32, ctypes.c_uint32, ctypes.c_uint32, u32p]
    lib.h2v_batch_set_agg_scalar.argtypes = [ctypes.c_void_p, ctypes.c_char_p]
    lib.h2v_ctx_create_from_bundle.argtypes = [ctypes.POINTER(ctypes.c_void_p), ctypes.c_char_p, ctypes.c_size_t, ctypes.c_int, ctypes.c_int,
                                               ctypes.c_int]
    lib.h2v_ctx_destroy.argtypes = [ctypes.c_void_p]
    lib.h2v_ctx_destroy.restype = None
    lib.h2v_last_error.argtypes = [ctypes.c_void_p]
    lib.h2v_last_error.restype = ctypes.c_char_p
    lib.h2v_ctx_info.argtypes = [ctypes.c_void_p, u32p]
    lib.h2v_verify_proof.argtypes = [ctypes.c_void_p, u8p, ctypes.c_size_t, u8p, ctypes.c_size_t, u8p]
    lib.h2v_verify_batch.argtypes = [ctypes.c_void_p, ctypes.c_uint32, u8p, u64p, u8p, u64p, u8p, ctypes.c_uint64,
                                     u8p, u8p, u8p, u8p]
    lib.h2v_batch_set_columns.argtypes = [ctypes.c_void_p, u32p, u32p]
    lib.h2v_batch_set_scalar_hook.argtypes = [ctypes.c_void_p, u8p]
    lib.h2v_batch_set_shard_hint.argtypes = [ctypes.c_void_p, ctypes.c_uint32]
    lib.h2v_batch_set_fold_groups.argtypes = [ctypes.c_void_p, ctypes.c_uint32]
    lib.h2v_last_group_verdicts.argtypes = [ctypes.c_void_p, u8p, ctypes.c_uint32]
    lib.h2v_finalize_groups.argtypes = [ctypes.c_void_p, ctypes.c_uint32, ctypes.c_uint32, u8p, u8p, ctypes.POINTER(ctypes.c_int)]
    lib.h2v_partial_bytes.argtypes = []
    lib.h2v_partial_bytes.restype = ctypes.c_size_t
    lib.h2v_accumulate_shard.argtypes = [ctypes.c_void_p, ctypes.c_uint32, u8p, u64p, u8p, u64p, u8p, ctypes.c_uint64,
                                         ctypes.c_uint64, ctypes.c_uint64, u8p, u8p]
    lib.h2v_finalize.argtypes = [ctypes.c_void_p, ctypes.c_uint32, u8p, u8p, ctypes.POINTER(ctypes.c_int)]
    lib.h2v_attribute_shard.argtypes = [ctypes.c_void_p, u8p]
    lib.h2v_attribute_shard_groups.argtypes = [ctypes.c_void_p, u8p, ctypes.c_uint32, u8p]
    lib.h2v_batch_set_rlc_key.argtypes = [ctypes.c_void_p, ctypes.c_char_p]
    lib.h2v_last_rlc_source.argtypes = [ctypes.c_void_p]
    lib.h2v_comm_init.argtypes = [ctypes.c_void_p, ctypes.c_uint32, ctypes.c_uint32, ctypes.c_uint32, u8p]
    lib.h2v_comm_connect.argtypes = [ctypes.c_void_p, ctypes.c_char_p]
    lib.h2v_comm_set_timeout_ms.argtypes = [ctypes.c_void_p, ctypes.c_uint32]
    lib.h2v_batch_run_shard_exchange.argtypes = [ctypes.c_void_p, ctypes.c_uint32, u8p, ctypes.POINTER(ctypes.c_int)]
    lib.h2v_verify_shard.argtypes = [ctypes.c_void_p, ctypes.c_uint32, u8p, u64p, u8p, u64p, u8p, ctypes.c_uint64, ctypes.c_uint64,
                                     ctypes.c_uint64, ctypes.c_uint32, u8p, u8p, ctypes.POINTER(ctypes.c_int)]
    lib.h2v_comm_last_batch_accum.argtypes = [ctypes.c_void_p, u8p]
    lib.h2v_ctx_cache_stats.argtypes = [ctypes.c_void_p, ctypes.c_void_p]
    lib.h2v_ctx_vk_lint.argtypes = [ctypes.c_void_p, ctypes.c_char_p, ctypes.c_size_t]
    lib.h2v_ctx_work_model.argtypes = [ctypes.c_void_p, ctypes.c_uint32, ctypes.c_void_p]
    lib.h2v_batch_upload.argtypes = [ctypes.c_void_p, ctypes.c_uint32, u8p, u64p, u8p, u64p, u8p, ctypes.c_uint64]
    lib.h2v_batch_upload_shard.argtypes = [ctypes.c_void_p, ctypes.c_uint32, u8p, u64p, u8p, u64p, u8p, ctypes.c_uint64,
                                           ctypes.c_uint64, ctypes.c_uint64]
    lib.h2v_batch_run_shard.argtypes = [ctypes.c_void_p, u8p]
    lib.h2v_batch_run_shard_async.argtypes = [ctypes.c_void_p, u8p]
    lib.h2v_flush_l2.argtypes = [ctypes.c_void_p, ctypes.c_size_t]
    lib.h2v_batch_run.argtypes = [ctypes.c_void_p, ctypes.POINTER(ctypes.c_int)]
    lib.h2v_batch_download.argtypes = [ctypes.c_void_p, u8p]
    lib.h2v_last_timings.argtypes = [ctypes.c_void_p, ctypes.c_void_p]
    lib.h2v_launch_count.argtypes = [ctypes.c_void_p]
    lib.h2v_launch_count.restype = ctypes.c_uint64
    lib.h2v_ctx_stream.argtypes = [ctypes.c_void_p]
    lib.h2v_ctx_stream.restype = ctypes.c_void_p
    lib.h2v_ctx_set_blocking_sync.argtypes = [ctypes.c_void_p, ctypes.c_int]
    lib.h2v_ctx_set_graphs.argtypes = [ctypes.c_void_p, ctypes.c_int]
    lib.h2v_debug_timeline_start.argtypes = [ctypes.c_int, ctypes.c_uint32]
    lib.h2v_debug_timeline_stop.argtypes = [ctypes.c_int, ctypes.c_void_p, ctypes.c_uint32, u32p]
    lib.h2v_last_msm_geometry.argtypes = [ctypes.c_void_p, u32p]
    lib.h2v_last_msm_glv.argtypes = [ctypes.c_void_p]
    lib.h2v_selftest_field.argtypes = [ctypes.c_int, ctypes.c_uint32, ctypes.c_uint64]
    lib.h2v_selftest_field_vectors.argtypes = [ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_uint32, ctypes.c_char_p, ctypes.c_char_p, u8p]
    lib.h2v_calibrate_imad.argtypes = [ctypes.c_int]
    lib.h2v_calibrate_imad.restype = ctypes.c_double
    lib.h2v_mix_create.argtypes = [ctypes.POINTER(ctypes.c_void_p), ctypes.c_void_p, ctypes.c_uint32]
    lib.h2v_mix_create_multi_params.argtypes = [ctypes.POINTER(ctypes.c_void_p), ctypes.c_void_p, ctypes.c_uint32]
    lib.h2v_mix_params_classes.argtypes = [ctypes.c_void_p, ctypes.POINTER(ctypes.c_uint32), ctypes.c_uint32]
    lib.h2v_mix_destroy.argtypes = [ctypes.c_void_p]
    lib.h2v_mix_destroy.restype = None
    lib.h2v_mix_last_error.argtypes = [ctypes.c_void_p]
    lib.h2v_mix_last_error.restype = ctypes.c_char_p
    lib.h2v_mix_set_rlc_key.argtypes = [ctypes.c_void_p, ctypes.c_char_p]
    lib.h2v_mix_verify.argtypes = [ctypes.c_void_p, u32p, u8p, u64p, u8p, u64p, u8p, ctypes.c_uint64, u8p, u8p, ctypes.POINTER(ctypes.c_int)]
    lib.h2v_mix_set_shard_hint.argtypes = [ctypes.c_void_p, ctypes.c_uint32]
    lib.h2v_mix_partial_bytes.argtypes = [ctypes.c_void_p, u32p]
    lib.h2v_mix_partial_bytes.restype = ctypes.c_size_t
    lib.h2v_mix_accumulate_shard.argtypes = [ctypes.c_void_p, u32p, ctypes.c_uint64, ctypes.c_uint32, u8p, u64p, u8p, u64p, u8p, ctypes.c_uint64, u8p,
                                             ctypes.c_void_p]
    lib.h2v_mix_finalize.argtypes = [ctypes.c_void_p, u32p, ctypes.c_uint32, ctypes.c_void_p, u8p, ctypes.POINTER(ctypes.c_int)]
    lib.h2v_mix_attribute_shard.argtypes = [ctypes.c_void_p, u8p]
    lib.h2v_mix_verify_shard.argtypes = [ctypes.c_void_p, u32p, ctypes.c_uint64, ctypes.c_uint32, u8p, u64p, u8p, u64p, u8p, ctypes.c_uint64,
                                         ctypes.c_uint32, u8p, ctypes.POINTER(ctypes.c_int)]
    lib.h2v_mix_comm_last_batch_accum.argtypes = [ctypes.c_void_p, u8p]
    lib.h2v_mix_verify_groups.argtypes = [ctypes.c_void_p, ctypes.c_uint32, u32p, u8p, u64p, u8p, u64p, u8p, ctypes.c_uint64, u8p, u8p, u8p,
                                          ctypes.POINTER(ctypes.c_int)]
    lib.h2v_acc_create.argtypes = [ctypes.POINTER(ctypes.c_void_p), ctypes.c_void_p, ctypes.c_uint32]
    lib.h2v_acc_destroy.argtypes = [ctypes.c_void_p]
    lib.h2v_acc_destroy.restype = None
    lib.h2v_acc_last_error.argtypes = [ctypes.c_void_p]
    lib.h2v_acc_last_error.restype = ctypes.c_char_p
    lib.h2v_acc_set_rlc_key.argtypes = [ctypes.c_void_p, ctypes.c_char_p]
    lib.h2v_acc_absorb.argtypes = [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_uint32, u8p, u64p, u8p, u64p, u8p, ctypes.c_uint64, u8p,
                                   ctypes.POINTER(ctypes.c_uint32)]
    lib.h2v_acc_finalize.argtypes = [ctypes.c_void_p, ctypes.POINTER(ctypes.c_int), u8p, ctypes.c_uint32]
    lib.h2v_acc_get.argtypes = [ctypes.c_void_p, u8p]
    lib.h2v_acc_merge.argtypes = [ctypes.c_void_p, ctypes.c_char_p, ctypes.c_char_p]
    lib.h2v_acc_reset.argtypes = [ctypes.c_void_p]
    _lib = lib
    return lib


EXPORTED_SYMBOLS = (
    "h2v_ctx_create", "h2v_ctx_create_from_bundle", "h2v_ctx_destroy", "h2v_last_error", "h2v_ctx_info", "h2v_verify_proof", "h2v_verify_batch",
    "h2v_batch_set_columns", "h2v_batch_set_scalar_hook", "h2v_batch_set_shard_hint", "h2v_partial_bytes", "h2v_accumulate_shard", "h2v_finalize", "h2v_attribute_shard",
    "h2v_batch_upload", "h2v_batch_upload_shard", "h2v_batch_run", "h2v_batch_run_shard", "h2v_batch_run_shard_async", "h2v_flush_l2", "h2v_batch_download", "h2v_last_timings", "h2v_launch_count", "h2v_ctx_stream", "h2v_ctx_set_blocking_sync", "h2v_ctx_set_graphs", "h2v_ctx_create_multi", "h2v_batch_set_fold_groups", "h2v_last_group_verdicts", "h2v_finalize_groups", "h2v_debug_timeline_start", "h2v_debug_timeline_stop",
    "h2v_last_msm_geometry", "h2v_last_msm_glv", "h2v_selftest_field", "h2v_selftest_field_vectors", "h2v_calibrate_imad",
    "h2v_attribute_shard_groups", "h2v_batch_set_rlc_key", "h2v_last_rlc_source", "h2v_comm_init", "h2v_comm_connect", "h2v_comm_set_timeout_ms",
    "h2v_batch_run_shard_exchange", "h2v_verify_shard", "h2v_comm_last_batch_accum", "h2v_ctx_cache_stats", "h2v_ctx_work_model", "h2v_ctx_vk_lint",
    "h2v_mix_create", "h2v_mix_destroy", "h2v_mix_last_error", "h2v_mix_set_rlc_key", "h2v_mix_verify",
    "h2v_mix_create_multi_params", "h2v_mix_params_classes",
    "h2v_mix_set_shard_hint", "h2v_mix_partial_bytes", "h2v_mix_accumulate_shard", "h2v_mix_finalize", "h2v_mix_attribute_shard",
    "h2v_mix_verify_shard", "h2v_mix_comm_last_batch_accum", "h2v_mix_verify_groups",
    "h2v_acc_create", "h2v_acc_destroy", "h2v_acc_last_error", "h2v_acc_set_rlc_key", "h2v_acc_absorb", "h2v_acc_finalize", "h2v_acc_get",
    "h2v_acc_merge", "h2v_acc_reset", "h2v_ctx_create_aggregation", "h2v_batch_set_agg_scalar",
)

COMM_HANDLE_BYTES = 128


@dataclass
class ParamsKZG:
    """Verifier-side KZG parameters (reference poly/kzg/commitment.rs:22-29), kept as bytes."""

    data: bytes
    format: SerdeFormat = SerdeFormat.Processed

    @classmethod
    def from_bytes(cls, data: bytes, format: SerdeFormat = SerdeFormat.Processed):
        return cls(bytes(data), SerdeFormat(format))

    @classmethod
    def read(cls, reader, format: SerdeFormat = SerdeFormat.Processed):
        size = 4 + (32 + 64 + 64 if format == SerdeFormat.Processed else 64 + 128 + 128)
        return cls(reader.read(size), SerdeFormat(format))

    @property
    def k(self):
        return int.from_bytes(self.data[:4], "little")  # little-endian, commitment.rs:147


@dataclass
class VerifyingKey:
    """Serialized verifying key (reference plonk/vk.rs:16-26), kept as bytes; parsed by the library."""

    data: bytes
    format: SerdeFormat = SerdeFormat.RawBytes

    @classmethod
    def from_bytes(cls, data: bytes, format: SerdeFormat = SerdeFormat.RawBytes):
        return cls(bytes(data), SerdeFormat(format))

    @classmethod
    def read(cls, reader, format: SerdeFormat = SerdeFormat.RawBytes):
        return cls(reader.read(), SerdeFormat(format))


PARAMS_BYTES_LENGTH = 4 + 32 + 64 + 64  # ParamsKZG::bytes_length() (poly/kzg/commitment.rs:209-213)


def read_vk_bundle(data: bytes):
    """Splits a `VALID_VK.bin` bundle (reference serialize/examples/vector_mul.rs:374-393: verifier params in
    Processed form followed by the VK in RawBytes form) into (ParamsKZG, VerifyingKey)."""
    if len(data) <= PARAMS_BYTES_LENGTH:
        raise BackendError("bundle shorter than the verifier params")
    return (ParamsKZG(bytes(data[:PARAMS_BYTES_LENGTH]), SerdeFormat.Processed),
            VerifyingKey(bytes(data[PARAMS_BYTES_LENGTH:]), SerdeFormat.RawBytes))


def instances_from_pubs(data: bytes):
    """`VALID_PUBS.bin` of the same example (public inputs as consecutive 32-byte `to_bytes()` values) -> one
    instance column of ints."""
    if len(data) % 32:
        raise BackendError("public-input file is not a multiple of 32 bytes")
    return [[int.from_bytes(data[i: i + 32], "little") for i in range(0, len(data), 32)]]


def pack_instances(instances) -> (bytes, List[int], Optional[List[int]], Optional[List[int]]):
    """instances[proof][column][row] of ints (or 32-byte strings) -> (bytes, per-proof scalar counts,
    per-proof column counts, per-proof per-column lengths)."""
    out = bytearray()
    counts, ncols, col_len = [], [], []
    for proof_inst in instances:
        c = 0
        ncols.append(len(proof_inst))
        for col in proof_inst:
            col_len.append(len(col))
            for v in col:
                out += v if isinstance(v, (bytes, bytearray)) else int(v).to_bytes(32, "little")
                c += 1
        counts.append(c)
    return bytes(out), counts, ncols, col_len


@dataclass(frozen=True)
class InstanceAccumulator:
    """The KZG accumulator (lhs, rhs) an aggregation circuit (snark-verifier with halo2-lib or halo2wrong) carries in its
    public instances, whose deferred check lhs = s * rhs the verifier must run (include/h2v.h "aggregation proofs").
    limbs, bits: snark-verifier's LimbsEncoding<LIMBS, BITS>, (3, 88) for halo2-lib, (4, 68) for halo2wrong.  cells: 4 * limbs
    (column, row) pairs of lhs.x, lhs.y, rhs.x, rhs.y, least significant limb first; column indexes the proof's flattened
    instance columns (instance-major with circuit_instances > 1)."""

    limbs: int
    bits: int
    cells: Tuple[Tuple[int, int], ...]

    @classmethod
    def rows(cls, limbs, bits, column=0, first_row=0):
        """the common layout: the 4 * limbs values in consecutive rows of one column"""
        return cls(int(limbs), int(bits), tuple((int(column), int(first_row) + i) for i in range(4 * int(limbs))))


@dataclass
class BatchResult:
    status: List[int]
    verdict: bool  # every proof accepted
    challenges: Optional[bytes] = None
    accum: Optional[bytes] = None
    batch_accum: Optional[bytes] = None
    msm_scalars: Optional[bytes] = None
    group_verdicts: Optional[List[bool]] = None  # one per fold group (fold_groups > 1)

    def errors(self):
        return [None if s == 0 else STATUS_ERRORS[s]() for s in self.status]


class BatchVerifier:
    """One (params, vk, multiopen, transcript, device) context: owns the device plan and buffers."""

    def __init__(self, params: ParamsKZG, vk: VerifyingKey, multiopen="shplonk", transcript="blake2b", device=0, circuit_instances=1,
                 accumulator: Optional[InstanceAccumulator] = None):
        """circuit_instances = m > 1: every proof carries m circuit instances in one transcript (`instances.len()` of the
        reference's verify_proof); the `instances` entry of a proof is then a list of m column lists.
        accumulator: the proofs are aggregation proofs carrying this KZG accumulator, which is checked inside the fold
        (a proof whose carried accumulator is false fails with ConstraintSystemFailure, a malformed encoding with
        InvalidInstances).  A malformed spec raises BackendError here, before any device work."""
        self.lib = load_library()
        self._ctx = ctypes.c_void_p()
        self.circuit_instances = int(circuit_instances)
        self.multiopen, self.transcript = multiopen, transcript
        self.accumulator = accumulator
        if accumulator is None:
            rc = self.lib.h2v_ctx_create_multi(ctypes.byref(self._ctx), params.data, len(params.data), int(params.format), vk.data,
                                               len(vk.data), int(vk.format), _MULTIOPEN[multiopen], _HASH[transcript], int(device),
                                               self.circuit_instances)
        else:
            flat = [int(v) for cell in accumulator.cells for v in cell]
            cells = (ctypes.c_uint32 * max(1, len(flat)))(*flat) if len(flat) == 8 * int(accumulator.limbs) else None
            if cells is None and flat:
                raise BackendError(f"aggregation spec: {len(flat) // 2} cells given, 4 * limbs = {4 * int(accumulator.limbs)} needed")
            rc = self.lib.h2v_ctx_create_aggregation(ctypes.byref(self._ctx), params.data, len(params.data), int(params.format), vk.data,
                                                     len(vk.data), int(vk.format), _MULTIOPEN[multiopen], _HASH[transcript], int(device),
                                                     self.circuit_instances, int(accumulator.limbs), int(accumulator.bits), cells)
        if rc != 0:
            self._ctx = None
            raise BackendError(self.lib.h2v_last_error(None).decode())
        info = (ctypes.c_uint32 * 8)()
        self.lib.h2v_ctx_info(self._ctx, info)
        (self.k, self.n_points, self.n_scalars, self.n_challenges, self.proof_len, self.n_inst_cols, self.n_shared,
         self.n_mo) = list(info)
        # scalar hook layout: on an aggregation context the carried lhs, rhs follow the proof points in both channels
        self.n_carry = 0 if accumulator is None else 2
        self.n_bases = self.n_points + self.n_shared + self.n_mo + 2 * self.n_carry

    def close(self):
        if getattr(self, "_ctx", None):
            self.lib.h2v_ctx_destroy(self._ctx)
            self._ctx = None

    __del__ = close

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()

    def _check(self, rc):
        if rc != 0:
            raise BackendError(self.lib.h2v_last_error(self._ctx).decode())

    @staticmethod
    def _offsets(sizes):
        arr = (ctypes.c_uint64 * (len(sizes) + 1))()
        t = 0
        for i, s in enumerate(sizes):
            arr[i] = t
            t += s
        arr[len(sizes)] = t
        return arr

    def _pack(self, proofs, instances):
        if self.circuit_instances > 1:  # instance-major "virtual" columns (lib.rs:76-82)
            instances = [[col for inst in proof_insts for col in inst] for proof_insts in instances]
        pbytes = b"".join(proofs)
        poff = self._offsets([len(p) for p in proofs])
        ibytes, counts, ncols, col_len = pack_instances(instances)
        ioff = self._offsets(counts)
        ragged = any(c != self.n_inst_cols for c in ncols) or any(
            len({len(col) for col in inst}) > 1 for inst in instances
        )
        keep = []
        if ragged:
            a = (ctypes.c_uint32 * len(ncols))(*ncols)
            # column lengths are laid out with exactly n_inst_cols entries per proof
            flat = []
            for inst in instances:
                lens = [len(c) for c in inst][: self.n_inst_cols]
                flat += lens + [0] * (self.n_inst_cols - len(lens))
            b = (ctypes.c_uint32 * max(1, len(flat)))(*flat)
            self._check(self.lib.h2v_batch_set_columns(self._ctx, a, b if self.n_inst_cols else None))
            keep = [a, b]
        return pbytes, poff, ibytes, ioff, keep

    def _fold_randomness(self, rlc_scalars, seed, key):
        """Fold randomness of the next upload (include/h2v.h): explicit scalars (parity hook) > `key` (32 secret bytes) >
        `seed` (a non-zero test seed: public, reproducible) > None: the library draws a fresh key from the OS, which is
        what the reference does (strategy.rs:129) and what production callers want.  Returns (scalar bytes, seed)."""
        if rlc_scalars is not None:
            return b"".join(int(r).to_bytes(32, "little") for r in rlc_scalars), 0
        if key is not None:
            if len(key) != 32:
                raise ValueError("the fold key is 32 bytes")
            self._check(self.lib.h2v_batch_set_rlc_key(self._ctx, bytes(key)))
            return None, 0
        if seed is None:
            return None, 0
        if int(seed) == 0:
            raise ValueError("seed 0 is reserved (the C ABI reads it as 'draw from the OS'): pass seed=None for OS entropy")
        return None, int(seed)

    def _set_agg_scalar(self, agg_scalar):
        """rho of the carried accumulators for the next upload (needed for bit-exact accumulators with rlc_scalars)"""
        if agg_scalar is not None:
            self._check(self.lib.h2v_batch_set_agg_scalar(self._ctx, int(agg_scalar).to_bytes(32, "little")))

    def rlc_source(self):
        """of the last upload: 'scalars' | 'seed' | 'key' | 'os'"""
        return ("scalars", "seed", "key", "os")[self.lib.h2v_last_rlc_source(self._ctx)]

    def verify_batch(self, proofs: Sequence[bytes], instances, rlc_scalars: Optional[Sequence[int]] = None, seed=None,
                     want_challenges=False, want_accum=False, want_batch_accum=False, want_scalars=False, fold_groups=1, key=None,
                     agg_scalar=None) -> BatchResult:
        """`fold_groups` = G: the proofs are G consecutive independent batches of len(proofs) / G proofs (own fold, own
        pairing check) that share every kernel launch; `group_verdicts` holds their G batch verdicts.
        Fold randomness: OS entropy unless `rlc_scalars` / `key` / `seed` say otherwise (_fold_randomness).
        agg_scalar (aggregation contexts, with rlc_scalars): the fold scalar rho of the carried accumulators; without it
        rho comes from the key / seed, or from the OS next to rlc_scalars."""
        n = len(proofs)
        assert n == len(instances) and n > 0
        self._set_agg_scalar(agg_scalar)
        if fold_groups > 1:
            self._check(self.lib.h2v_batch_set_fold_groups(self._ctx, int(fold_groups)))
        pbytes, poff, ibytes, ioff, keep = self._pack(proofs, instances)
        rlc, seed = self._fold_randomness(rlc_scalars, seed, key)
        status = (ctypes.c_uint8 * n)()
        ch = ctypes.create_string_buffer(32 * n * self.n_challenges) if want_challenges else None
        acc = ctypes.create_string_buffer(128 * n) if want_accum else None
        bacc = ctypes.create_string_buffer(128) if want_batch_accum else None
        sc = ctypes.create_string_buffer(32 * n * self.n_bases) if want_scalars else None
        if sc is not None:
            self._check(self.lib.h2v_batch_set_scalar_hook(self._ctx, sc))
        self._check(self.lib.h2v_verify_batch(self._ctx, n, pbytes, poff, ibytes, ioff, rlc, seed, status, ch, acc, bacc))
        st = list(status)
        gv = (ctypes.c_uint8 * max(1, int(fold_groups)))()
        ng = self.lib.h2v_last_group_verdicts(self._ctx, gv, len(gv))
        return BatchResult(st, all(s == 0 for s in st), ch.raw if ch else None, acc.raw if acc else None,
                           bacc.raw if bacc else None, sc.raw if sc else None, [bool(v) for v in gv[:ng]])

    def accumulate_shard(self, proofs, instances, global_base, global_count, rlc_scalars=None, seed=None, shard_hint=0, fold_groups=1, key=None,
                         partial_out=None, agg_scalar=None):
        """Returns (statuses, partial): `partial` is the opaque H2V_PARTIAL_BYTES blob of this shard's
        per-window bucket sums (bytes; or None when `partial_out`, a device or host pointer, receives it).
        `shard_hint` = size of the largest shard of the global batch when the
        shards are not all of the same size (every rank must use the same window geometry)."""
        n = len(proofs)
        self._set_agg_scalar(agg_scalar)
        pbytes, poff, ibytes, ioff, keep = self._pack(proofs, instances)
        rlc, seed = self._fold_randomness(rlc_scalars, seed, key)
        status = (ctypes.c_uint8 * n)()
        partial = ctypes.create_string_buffer(self.lib.h2v_partial_bytes() * max(1, int(fold_groups))) if partial_out is None else None
        if fold_groups > 1:  # group q = this rank's shard of global batch q; rlc_scalars: fold_groups x global_count values
            self._check(self.lib.h2v_batch_set_fold_groups(self._ctx, int(fold_groups)))
        if shard_hint:
            self._check(self.lib.h2v_batch_set_shard_hint(self._ctx, int(shard_hint)))
        self._check(self.lib.h2v_accumulate_shard(self._ctx, n, pbytes, poff, ibytes, ioff, rlc, seed, global_base,
                                                  global_count, status, partial if partial_out is None else ctypes.c_void_p(int(partial_out))))
        return list(status), (partial.raw if partial is not None else None)

    # ---- device-side exchange (include/h2v.h "device-side exchange of sharded batches")
    def comm_init(self, rank, world, max_groups=1) -> bytes:
        """allocates this context's exchange window; returns the opaque handle to ship to every rank"""
        h = ctypes.create_string_buffer(COMM_HANDLE_BYTES)
        self._check(self.lib.h2v_comm_init(self._ctx, int(rank), int(world), int(max_groups), h))
        self.comm_rank, self.comm_world, self.comm_ready = int(rank), int(world), False
        return h.raw

    def comm_connect(self, handles: Sequence[bytes]):
        """handles of all ranks' contexts of this channel, rank order (own included)"""
        self._check(self.lib.h2v_comm_connect(self._ctx, b"".join(handles)))
        self.comm_ready = True

    def verify_shard(self, proofs, instances, global_base, global_count, root, rlc_scalars=None, seed=None, key=None, shard_hint=0, fold_groups=1):
        """This rank's part of a sharded batch through the device-side exchange: returns (group verdicts, statuses of
        this shard); rejected groups are attributed per proof inside the shard."""
        n = len(proofs)
        pbytes, poff, ibytes, ioff, keep = self._pack(proofs, instances)
        rlc, seed = self._fold_randomness(rlc_scalars, seed, key)
        status = (ctypes.c_uint8 * n)()
        G = max(1, int(fold_groups))
        gv = (ctypes.c_uint8 * G)()
        verdict = ctypes.c_int(0)
        if G > 1:
            self._check(self.lib.h2v_batch_set_fold_groups(self._ctx, G))
        if shard_hint:
            self._check(self.lib.h2v_batch_set_shard_hint(self._ctx, int(shard_hint)))
        self._check(self.lib.h2v_verify_shard(self._ctx, n, pbytes, poff, ibytes, ioff, rlc, seed, global_base, global_count, int(root),
                                              status, gv, ctypes.byref(verdict)))
        return [bool(v) for v in gv], list(status)

    def comm_last_batch_accum(self) -> bytes:
        out = ctypes.create_string_buffer(128)
        self._check(self.lib.h2v_comm_last_batch_accum(self._ctx, out))
        return out.raw

    def vk_lint(self) -> List[str]:
        """places where this VK may have been mangled by the reference's own write/read asymmetry (include/h2v.h)"""
        buf = ctypes.create_string_buffer(1 << 16)
        n = self.lib.h2v_ctx_vk_lint(self._ctx, buf, len(buf))
        return [l for l in buf.value.decode().split("\n") if l][:max(n, 0)]

    def work_model(self, instance_rows):
        """algorithmic Montgomery multiplications per proof of this plan (include/h2v.h h2v_ctx_work_model)"""
        out = (ctypes.c_double * 4)()
        self._check(self.lib.h2v_ctx_work_model(self._ctx, int(instance_rows), out))
        return dict(zip(("scalar", "transcript", "decompress_per_point", "instance_scalars"), list(out)))

    def cache_stats(self):
        out = (ctypes.c_uint64 * 2)()
        self._check(self.lib.h2v_ctx_cache_stats(self._ctx, out))
        return {"lines_builds": int(out[0]), "graph_captures": int(out[1])}

    def finalize(self, partials, want_batch_accum=True, n_partials=None):
        """partials: list of blobs, or (with n_partials) the address of n_partials consecutive blobs in host or device memory"""
        if n_partials is not None:
            bacc = ctypes.create_string_buffer(128) if want_batch_accum else None
            verdict = ctypes.c_int(0)
            self._check(self.lib.h2v_finalize(self._ctx, int(n_partials), ctypes.c_void_p(int(partials)), bacc, ctypes.byref(verdict)))
            return bool(verdict.value), (bacc.raw if bacc is not None else None)
        buf = b"".join(partials)
        bacc = ctypes.create_string_buffer(128) if want_batch_accum else None
        verdict = ctypes.c_int(0)
        self._check(self.lib.h2v_finalize(self._ctx, len(partials), buf, bacc, ctypes.byref(verdict)))
        return bool(verdict.value), (bacc.raw if bacc is not None else None)

    def finalize_groups(self, partials, fold_groups, n_partials=None):
        """partials: one accumulate_shard(..., fold_groups=G) output per rank (or, with n_partials, the address of the
        ranks' outputs concatenated in host or device memory); returns the G batch verdicts"""
        gv = (ctypes.c_uint8 * int(fold_groups))()
        verdict = ctypes.c_int(0)
        if n_partials is not None:
            self._check(self.lib.h2v_finalize_groups(self._ctx, int(n_partials), int(fold_groups), ctypes.c_void_p(int(partials)), gv, ctypes.byref(verdict)))
        else:
            self._check(self.lib.h2v_finalize_groups(self._ctx, len(partials), int(fold_groups), b"".join(partials), gv, ctypes.byref(verdict)))
        return [bool(v) for v in gv]

    def attribute_shard(self, status, group_verdicts=None):
        """per-proof re-check of the shard last processed; with `group_verdicts` only inside the rejected fold groups"""
        arr = (ctypes.c_uint8 * len(status))(*status)
        if group_verdicts is not None:
            gv = (ctypes.c_uint8 * len(group_verdicts))(*[1 if v else 0 for v in group_verdicts])
            self._check(self.lib.h2v_attribute_shard_groups(self._ctx, gv, len(group_verdicts), arr))
        else:
            self._check(self.lib.h2v_attribute_shard(self._ctx, arr))
        return list(arr)

    def timings(self):
        out = (ctypes.c_float * 8)()
        self._check(self.lib.h2v_last_timings(self._ctx, out))
        names = ("total", "decompress", "transcript", "scalar", "rlc_msm", "pairing", "attribution")
        return dict(zip(names, list(out)))

    def msm_geometry(self):
        out = (ctypes.c_uint32 * 4)()
        self.lib.h2v_last_msm_geometry(self._ctx, out)
        return dict(zip(("window_bits", "windows", "terms", "buckets"), list(out)))

    def msm_glv(self):
        """True when the last run's MSM split every scalar into two lifted GLV halves."""
        return self.lib.h2v_last_msm_glv(self._ctx) == 1

    def launch_count(self):
        return int(self.lib.h2v_launch_count(self._ctx))

    def set_graphs(self, on):
        """CUDA-graph replay of the batch kernels (default on); off = direct launches with per-stage event timings."""
        self._check(self.lib.h2v_ctx_set_graphs(self._ctx, 1 if on else 0))

    def stream_handle(self):
        """cudaStream_t of this context as an integer (wrap with torch.cuda.ExternalStream to record events on it)."""
        return int(self.lib.h2v_ctx_stream(self._ctx))


@dataclass
class MixedBatchResult:
    status: List[List[int]]  # one list per member, in member order
    verdict: bool  # every proof of every member accepted
    # folded (L, R) of the whole mix, 2 x 64 B; a multi_params mix: one (L_p, R_p) per params class in class order,
    # classes x 128 B, all-zero for a class without proofs in the call
    batch_accum: Optional[bytes] = None

    def errors(self):
        return [[None if s == 0 else STATUS_ERRORS[s]() for s in st] for st in self.status]


@dataclass
class MixedGroupsResult:
    status: List[List[List[int]]]  # status[q][m]: member m's proofs of group q
    group_verdicts: List[bool]  # group q: its check accepted and every proof of it is valid
    verdict: bool  # every group accepted
    # per group: its classes x 128 B folded (L_p, R_p), as MixedBatchResult.batch_accum for that group alone
    batch_accum: Optional[List[bytes]] = None


class MixedBatchVerifier:
    """Proofs of several BatchVerifiers (verifying keys, SHPLONK or GWC, Blake2b or Keccak) folded into ONE MSM and ONE
    pairing check: the reference's AccumulatorStrategy fed proofs of different VKs under one set of KZG params
    (include/h2v.h "mixed batches").  The members' params must agree on (g, g2, s_g2); k may differ.  The members are not
    owned: they must stay open while the mix is used and must not run their own batches during a mixed one.
    multi_params=True: members may hold up to 8 different params (a different trapdoor or g2); each params class gets its
    own bucket set and lines, and all classes still share one pairing check (`params_classes`, include/h2v.h
    "multi-params mixes")."""

    def __init__(self, members: Sequence[BatchVerifier], multi_params=False):
        self.lib = load_library()
        self.members = list(members)
        self._mx = ctypes.c_void_p()
        ptrs = (ctypes.c_void_p * max(1, len(self.members)))(*[m._ctx for m in self.members])
        create = self.lib.h2v_mix_create_multi_params if multi_params else self.lib.h2v_mix_create
        if create(ctypes.byref(self._mx), ptrs if self.members else None, len(self.members)) != 0:
            self._mx = None
            raise BackendError(self.lib.h2v_mix_last_error(None).decode())
        cls = (ctypes.c_uint32 * len(self.members))()
        self.n_classes = self.lib.h2v_mix_params_classes(self._mx, cls, len(self.members))
        self.params_classes = list(cls)  # params class of each member, numbered by first appearance

    def close(self):
        if getattr(self, "_mx", None):
            self.lib.h2v_mix_destroy(self._mx)
            self._mx = None

    __del__ = close

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()

    def _check(self, rc):
        if rc != 0:
            raise BackendError(self.lib.h2v_mix_last_error(self._mx).decode())

    def verify_batch(self, proofs_per_member, instances_per_member, rlc_scalars: Optional[Sequence[int]] = None, seed=None, key=None,
                     want_batch_accum=False, agg_scalar=None) -> MixedBatchResult:
        """proofs_per_member[m] / instances_per_member[m]: member m's proofs and instances as for its own verify_batch
        (empty lists allowed).  The fold runs over the member-major concatenation: rlc_scalars has one entry per proof of
        it.  Fold randomness as BatchVerifier.verify_batch: OS entropy unless `rlc_scalars` / `key` / `seed` say otherwise."""
        counts, packed = self._pack(proofs_per_member, instances_per_member)
        n = sum(counts)
        if n == 0:
            raise ValueError("a mixed batch needs at least one proof")
        if rlc_scalars is not None and len(rlc_scalars) != n:
            raise ValueError("one fold scalar per proof of the concatenation")
        rlc, seed = self._randomness(proofs_per_member, rlc_scalars, seed, key, agg_scalar)
        status = (ctypes.c_uint8 * n)()
        bacc = ctypes.create_string_buffer(128 * self.n_classes) if want_batch_accum else None
        verdict = ctypes.c_int(0)
        self._check(self.lib.h2v_mix_verify(self._mx, self._u32(counts), *packed[:4], rlc, int(seed), status, bacc, ctypes.byref(verdict)))
        return MixedBatchResult(self._split(list(status), counts), bool(verdict.value), bacc.raw if bacc is not None else None)

    def verify_groups(self, groups, rlc_scalars: Optional[Sequence[int]] = None, seed=None, key=None, want_batch_accum=False,
                      agg_scalar=None) -> MixedGroupsResult:
        """Independent mixed batches in one launch set (include/h2v.h "grouped mixed batches"): groups[q] = (proofs_per_member,
        instances_per_member) as for verify_batch.  Each group is folded, checked and judged on its own; rlc_scalars has one
        entry per proof in call order (group 0's member-major concatenation, then group 1's, ...), so group q's slice is what
        verify_batch takes for group q alone."""
        M = len(self.members)
        groups = list(groups)
        for q, (ppm, ipm) in enumerate(groups):
            if len(ppm) != M or len(ipm) != M:
                raise ValueError(f"group {q}: one proof list and one instance list per member")
            for m in range(M):
                if len(ppm[m]) != len(ipm[m]):
                    raise ValueError(f"group {q}, member {m}: {len(ppm[m])} proofs, {len(ipm[m])} instance lists")
        counts = [len(g[0][m]) for g in groups for m in range(M)]
        n = sum(counts)
        if not groups or n == 0:
            raise ValueError("a grouped mixed batch needs at least one group with proofs")
        if rlc_scalars is not None and len(rlc_scalars) != n:
            raise ValueError("one fold scalar per proof of the call")
        # one _pack per member over its proofs of every group (its ragged-column layout describes its whole upload)
        per_member = []
        for m, bv in enumerate(self.members):
            proofs = [p for g in groups for p in g[0][m]]
            insts = [i for g in groups for i in g[1][m]]
            per_member.append(bv._pack(proofs, insts) if proofs else None)
        pparts, iparts, poffs, ioffs, keep = [], [], [0], [0], []
        first = [0] * M  # next proof of member m in its packed upload
        for q in range(len(groups)):
            for m in range(M):
                c = counts[q * M + m]
                if not c:
                    continue
                pbytes, poff, ibytes, ioff, k = per_member[m]
                keep += k
                a = first[m]
                pparts.append(pbytes[poff[a]:poff[a + c]])
                iparts.append(ibytes[32 * ioff[a]:32 * ioff[a + c]])
                poffs += [poffs[-1] + poff[a + j + 1] - poff[a] for j in range(c)]
                ioffs += [ioffs[-1] + ioff[a + j + 1] - ioff[a] for j in range(c)]
                first[m] += c
        ppm_all = [[p for g in groups for p in g[0][m]] for m in range(M)]
        rlc, seed = self._randomness(ppm_all, rlc_scalars, seed, key, agg_scalar)
        G = len(groups)
        status = (ctypes.c_uint8 * n)()
        gverd = (ctypes.c_uint8 * G)()
        bacc = ctypes.create_string_buffer(128 * self.n_classes * G) if want_batch_accum else None
        verdict = ctypes.c_int(0)
        self._check(self.lib.h2v_mix_verify_groups(self._mx, G, self._u32(counts), b"".join(pparts), (ctypes.c_uint64 * (n + 1))(*poffs),
                                                   b"".join(iparts), (ctypes.c_uint64 * (n + 1))(*ioffs), rlc, int(seed), status, gverd, bacc,
                                                   ctypes.byref(verdict)))
        st, out = list(status), []
        for q in range(G):
            out.append(self._split(st[:sum(counts[q * M:(q + 1) * M])], counts[q * M:(q + 1) * M]))
            st = st[sum(counts[q * M:(q + 1) * M]):]
        per = 128 * self.n_classes
        return MixedGroupsResult(out, [bool(v) for v in gverd], bool(verdict.value),
                                 [bacc.raw[q * per:(q + 1) * per] for q in range(G)] if bacc is not None else None)

    @staticmethod
    def _u32(values):
        return (ctypes.c_uint32 * max(1, len(values)))(*values)

    @staticmethod
    def _split(statuses, counts):
        out = []
        for c in counts:
            out.append(statuses[:c])
            statuses = statuses[c:]
        return out

    def _pack(self, proofs_per_member, instances_per_member):
        """member-major concatenation: (per-member counts, (proofs, proof offsets, instances, instance offsets, keep-alive))"""
        if len(proofs_per_member) != len(self.members) or len(instances_per_member) != len(self.members):
            raise ValueError("one proof list and one instance list per member")
        counts = []
        pparts, iparts, poffs, ioffs, keep = [], [], [0], [0], []
        for m, (bv, proofs, insts) in enumerate(zip(self.members, proofs_per_member, instances_per_member)):
            if len(proofs) != len(insts):
                raise ValueError(f"member {m}: {len(proofs)} proofs, {len(insts)} instance lists")
            counts.append(len(proofs))
            if not proofs:
                continue
            pbytes, poff, ibytes, ioff, k = bv._pack(proofs, insts)  # (sets the member's ragged layout if needed)
            keep += k
            pparts.append(pbytes)
            iparts.append(ibytes)
            poffs += [poffs[-1] + poff[j + 1] for j in range(len(proofs))]
            ioffs += [ioffs[-1] + ioff[j + 1] for j in range(len(proofs))]
        n = len(poffs) - 1
        return counts, (b"".join(pparts), (ctypes.c_uint64 * (n + 1))(*poffs), b"".join(iparts), (ctypes.c_uint64 * (n + 1))(*ioffs), keep)

    def _randomness(self, proofs_per_member, rlc_scalars, seed, key, agg_scalar):
        rlc, seed = _fold_args(rlc_scalars, seed, key, lambda k: self._check(self.lib.h2v_mix_set_rlc_key(self._mx, k)))
        for bv, proofs in zip(self.members, proofs_per_member):  # one rho for every aggregation member with proofs
            if proofs and bv.accumulator is not None:
                bv._set_agg_scalar(agg_scalar)
        return rlc, seed

    # ---- sharded mixed batches (include/h2v.h "sharded mixed batches")
    def _shard_args(self, proofs_per_member, instances_per_member, global_counts, global_base, rlc_scalars, shard_hint):
        """this rank's portions, checked against the split the library derives (sharding.mixed_shard)"""
        from .sharding import mixed_shard_counts
        counts, packed = self._pack(proofs_per_member, instances_per_member)
        if len(global_counts) != len(self.members):
            raise ValueError("one global count per member")
        want = mixed_shard_counts(global_counts, global_base, sum(counts))
        if counts != want:
            raise ValueError(f"proofs per member {counts} are not the share of proofs [{global_base}, {global_base + sum(counts)}) of the global batch: {want}")
        if rlc_scalars is not None and len(rlc_scalars) != sum(global_counts):
            raise ValueError("one fold scalar per proof of the global batch")
        if shard_hint:
            self._check(self.lib.h2v_mix_set_shard_hint(self._mx, int(shard_hint)))
        return sum(counts), counts, packed

    def partial_bytes(self, global_counts) -> int:
        """bytes of one rank's partials for this global batch: one H2V_PARTIAL_BYTES blob per params class with proofs"""
        return int(self.lib.h2v_mix_partial_bytes(self._mx, self._u32(global_counts)))

    def accumulate_shard(self, proofs_per_member, instances_per_member, global_counts, global_base, rlc_scalars=None, seed=None, key=None,
                         shard_hint=0, partial_out=None, agg_scalar=None):
        """This rank's share [global_base, global_base + n) of the member-major global batch of global_counts proofs: returns
        (statuses per member, partials), partials = bytes of partial_bytes(global_counts), or None when `partial_out` (a device
        or host address) receives them.  shard_hint: the largest shard when the shards differ in size."""
        n, counts, packed = self._shard_args(proofs_per_member, instances_per_member, global_counts, global_base, rlc_scalars, shard_hint)
        rlc, seed = self._randomness(proofs_per_member, rlc_scalars, seed, key, agg_scalar)
        status = (ctypes.c_uint8 * max(1, n))()
        buf = ctypes.create_string_buffer(max(1, self.partial_bytes(global_counts))) if partial_out is None else None
        self._check(self.lib.h2v_mix_accumulate_shard(self._mx, self._u32(global_counts), int(global_base), n, *packed[:4], rlc, int(seed), status,
                                                      ctypes.cast(buf, ctypes.c_void_p) if buf is not None else ctypes.c_void_p(int(partial_out))))
        return self._split(list(status)[:n], counts), (buf.raw if buf is not None else None)

    def finalize(self, partials, global_counts, want_batch_accum=True, n_partials=None):
        """partials: one accumulate_shard output per rank, or (with n_partials) the address of n_partials ranks' outputs in host or
        device memory.  Returns (verdict of the one pairing check, classes x 128 B folded (L_p, R_p) or None)."""
        bacc = ctypes.create_string_buffer(128 * self.n_classes) if want_batch_accum else None
        verdict = ctypes.c_int(0)
        if n_partials is None:
            buf = ctypes.create_string_buffer(b"".join(partials), max(1, sum(len(p) for p in partials)))
            n_partials, addr = len(partials), ctypes.cast(buf, ctypes.c_void_p)
        else:
            addr = ctypes.c_void_p(int(partials))
        self._check(self.lib.h2v_mix_finalize(self._mx, self._u32(global_counts), int(n_partials), addr, bacc, ctypes.byref(verdict)))
        return bool(verdict.value), (bacc.raw if bacc is not None else None)

    def attribute_shard(self, status):
        """per-proof re-check of the shard last processed; `status`: its statuses per member (accumulate_shard's)"""
        counts = [len(s) for s in status]
        arr = (ctypes.c_uint8 * max(1, sum(counts)))(*[v for s in status for v in s])
        self._check(self.lib.h2v_mix_attribute_shard(self._mx, arr))
        return self._split(list(arr)[:sum(counts)], counts)

    # device-side exchange over the lead member's channel
    def comm_init(self, rank, world, max_groups=1) -> bytes:
        """the lead's exchange window, for at least as many partials per rank as the mix has params classes (the most bucket
        sets a batch can have; the same on every rank)"""
        h = self.members[0].comm_init(rank, world, max(int(max_groups), self.n_classes))
        self.comm_ready = False
        return h

    def comm_connect(self, handles):
        self.members[0].comm_connect(handles)
        self.comm_ready = True

    comm_ready = False

    def verify_shard(self, proofs_per_member, instances_per_member, global_counts, global_base, root, rlc_scalars=None, seed=None, key=None,
                     shard_hint=0, agg_scalar=None):
        """This rank's share through the device-side exchange: returns (verdict of the global check, statuses per member);
        a rejection is attributed per proof inside this rank's share."""
        n, counts, packed = self._shard_args(proofs_per_member, instances_per_member, global_counts, global_base, rlc_scalars, shard_hint)
        rlc, seed = self._randomness(proofs_per_member, rlc_scalars, seed, key, agg_scalar)
        status = (ctypes.c_uint8 * max(1, n))()
        verdict = ctypes.c_int(0)
        self._check(self.lib.h2v_mix_verify_shard(self._mx, self._u32(global_counts), int(global_base), n, *packed[:4], rlc, int(seed), int(root),
                                                  status, ctypes.byref(verdict)))
        return bool(verdict.value), self._split(list(status)[:n], counts)

    def comm_last_batch_accum(self) -> bytes:
        """root only: classes x 128 B folded (L_p, R_p) of the last exchange launch set"""
        out = ctypes.create_string_buffer(128 * self.n_classes)
        self._check(self.lib.h2v_mix_comm_last_batch_accum(self._mx, out))
        return out.raw

    def cache_stats(self):
        """the lead member's caches: the mix's graph captures and prepared lines are counted there"""
        return self.members[0].cache_stats()


@dataclass
class AbsorbResult:
    statuses: List[int]  # final, except that 0 means "accumulated" (a pairing failure shows at finalize)
    index: int  # record slot of this absorb (FinalizeResult.absorb_verdicts[index])


@dataclass
class FinalizeResult:
    verdict: bool  # the one pairing check on the accumulator accepts
    absorb_verdicts: List[bool]  # one per absorb / merge since the last finalize or reset; False = fails on its own


class Accumulator:
    """The reference's AccumulatorStrategy (poly/kzg/strategy.rs:125-140) as a value that lives across calls (include/h2v.h
    "persistent accumulators"): batches of any BatchVerifier whose params agree with the anchor's are absorbed into one
    device-resident DualMSM, and `finalize` runs one pairing check.  Absorbing proofs in chunks gives the same folded
    (L, R) as one verify_batch over their concatenation with the concatenated fold scalars.  The anchor supplies the params,
    the device and the prepared G2 lines; it is not owned and must stay open while the accumulator is used."""

    def __init__(self, anchor: BatchVerifier, max_absorbs=1024):
        self.lib = load_library()
        self.anchor, self.max_absorbs = anchor, int(max_absorbs)
        self._records = 0
        self._acc = ctypes.c_void_p()
        if self.lib.h2v_acc_create(ctypes.byref(self._acc), anchor._ctx if anchor is not None else None, self.max_absorbs) != 0:
            self._acc = None
            raise BackendError(self.lib.h2v_acc_last_error(None).decode())

    def close(self):
        if getattr(self, "_acc", None):
            self.lib.h2v_acc_destroy(self._acc)
            self._acc = None

    __del__ = close

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()

    def _check(self, rc):
        if rc != 0:
            raise BackendError(self.lib.h2v_acc_last_error(self._acc).decode())

    def absorb(self, verifier: BatchVerifier, proofs: Sequence[bytes], instances, rlc_scalars: Optional[Sequence[int]] = None, seed=None,
               key=None, agg_scalar=None) -> AbsorbResult:
        """AccumulatorStrategy::process for every proof, in order: proof j gets c_j = prod_{i>j} r_i and the accumulator is
        scaled by prod_i r_i before the batch is added.  Fold randomness as BatchVerifier.verify_batch: OS entropy unless
        `rlc_scalars` / `key` / `seed` say otherwise."""
        if len(proofs) != len(instances):
            raise ValueError(f"{len(proofs)} proofs, {len(instances)} instance lists")
        n = len(proofs)
        verifier._set_agg_scalar(agg_scalar)
        pbytes, poff, ibytes, ioff, keep = verifier._pack(proofs, instances)
        rlc, seed = _fold_args(rlc_scalars, seed, key, lambda k: self._check(self.lib.h2v_acc_set_rlc_key(self._acc, k)))
        status = (ctypes.c_uint8 * max(1, n))()
        index = ctypes.c_uint32(0)
        self._check(self.lib.h2v_acc_absorb(self._acc, verifier._ctx, n, pbytes, poff, ibytes, ioff, rlc, seed, status, ctypes.byref(index)))
        self._records = index.value + 1
        return AbsorbResult(list(status)[:n], index.value)

    def finalize(self) -> FinalizeResult:
        """DualMSM::check on the accumulator, then reset (finalize consumes the strategy).  On a rejection every absorb is
        checked on its own: re-verify the batches whose absorb_verdicts entry is False with verify_batch."""
        verdict = ctypes.c_int(0)
        av = (ctypes.c_uint8 * max(1, self._records))()
        self._check(self.lib.h2v_acc_finalize(self._acc, ctypes.byref(verdict), av, len(av)))
        n, self._records = self._records, 0
        return FinalizeResult(bool(verdict.value), [bool(v) for v in av[:n]])

    def to_bytes(self) -> bytes:
        """the affine L | R, 2 x 64 B (the batch_accum layout; all-zero = identity)"""
        out = ctypes.create_string_buffer(128)
        self._check(self.lib.h2v_acc_get(self._acc, out))
        return out.raw

    def merge(self, data: bytes, r: Optional[int] = None):
        """acc <- r acc + P, P = another accumulator's to_bytes() (into an empty accumulator: restore a checkpoint).  r = None
        draws r from the OS.  Non-canonical or off-curve bytes raise BackendError and leave the accumulator unchanged."""
        if len(data) != 128:
            raise ValueError("an accumulator is 128 bytes")
        rb = None if r is None else int(r).to_bytes(32, "little")
        self._check(self.lib.h2v_acc_merge(self._acc, bytes(data), rb))
        self._records += 1

    def reset(self):
        self._check(self.lib.h2v_acc_reset(self._acc))
        self._records = 0


def _fold_args(rlc_scalars, seed, key, set_key):
    """(scalar bytes, seed) of the C call for the fold randomness precedence rlc_scalars > key > seed > OS entropy;
    `set_key(key32)` hands a key to the library object"""
    if rlc_scalars is not None:
        return b"".join(int(r).to_bytes(32, "little") for r in rlc_scalars), 0
    if key is not None:
        if len(key) != 32:
            raise ValueError("the fold key is 32 bytes")
        set_key(bytes(key))
        return None, 0
    if seed is None:
        return None, 0
    if int(seed) == 0:
        raise ValueError("seed 0 is reserved (the C ABI reads it as 'draw from the OS'): pass seed=None for OS entropy")
    return None, int(seed)


def verify_proof(params: ParamsKZG, vk: VerifyingKey, proof: bytes, instances, multiopen="shplonk", transcript="blake2b",
                 device=0, accumulator: Optional[InstanceAccumulator] = None) -> None:
    """verify_proof with SingleStrategy (reference lib.rs:33-46): returns None or raises a plonk Error.
    `instances[column][row]`: public inputs of the single circuit instance.  accumulator: an aggregation proof's carried
    KZG accumulator, checked too (InstanceAccumulator)."""
    with BatchVerifier(params, vk, multiopen, transcript, device, accumulator=accumulator) as bv:
        res = bv.verify_batch([proof], [instances])
    if res.status[0] != 0:
        raise STATUS_ERRORS[res.status[0]]()


def verify_proofs_batch(params: ParamsKZG, vk: VerifyingKey, proofs: Sequence[bytes], instances, multiopen="shplonk",
                        transcript="blake2b", device=0, rlc_scalars=None, seed=None, accumulator: Optional[InstanceAccumulator] = None,
                        agg_scalar=None) -> List[Optional[Error]]:
    """Batch entry point: one folded pairing check for the whole batch (AccumulatorStrategy,
    strategy.rs:125-140), per-proof attribution when the fold is rejected.  Returns one entry per
    proof: None (accepted) or the plonk Error the reference's verify_proof would have returned.
    The fold coefficients come from OS entropy, as in the reference (strategy.rs:129), unless `rlc_scalars` or a
    non-zero test `seed` is given (parity hooks: public coefficients are not sound against an adversarial prover).
    accumulator: aggregation proofs; their carried KZG accumulators are checked inside the fold (InstanceAccumulator)."""
    with BatchVerifier(params, vk, multiopen, transcript, device, accumulator=accumulator) as bv:
        return bv.verify_batch(proofs, instances, rlc_scalars, seed, agg_scalar=agg_scalar).errors()


def verify_proofs_mixed(circuits, device=0, multi_params=False) -> List[List[Optional[Error]]]:
    """Mixed batch entry point: circuits = [(params, vk, proofs, instances, multiopen, transcript), ...] whose params agree
    on (g, g2, s_g2) (k may differ), or, with multi_params=True, under up to 8 different params.  All proofs are folded into
    one MSM and one pairing check (the reference's AccumulatorStrategy over proofs of several VKs), with per-proof
    attribution when the fold is rejected.  Returns one error list per circuit, as verify_proofs_batch does; the fold
    coefficients come from OS entropy."""
    bvs = []
    try:
        for params, vk, _proofs, _insts, multiopen, transcript in circuits:
            bvs.append(BatchVerifier(params, vk, multiopen, transcript, device))
        with MixedBatchVerifier(bvs, multi_params) as mx:
            return mx.verify_batch([c[2] for c in circuits], [c[3] for c in circuits]).errors()
    finally:
        for bv in bvs:
            bv.close()
