"""Host-side mirror of blsful's verification API over the blsgpu C ABI (include/blsgpu.h).

The reference is a Rust crate; this image has no Rust toolchain, so the slice-taking batch entry points the Rust
crate would gain (INTEGRATION.md) are mirrored here in Python over the same C ABI, with the reference's names,
argument meaning and error behaviour:

  Signature::verify            -> verify_batch            (reference src/signature.rs:130-138)
                               -> verify_batch_keyed      (keys decoded once into a KeySet, named by index)
  ProofOfPossession::verify    -> pop_verify_batch        (src/proof_of_possession.rs:77-81)
  AggregateSignature::verify   -> aggregate_verify        (src/aggregate_signature.rs:230-239)
                               -> aggregate_verify_batch_status (q aggregates in one call)
  MultiSignature / AggregateSignature::from_signatures, MultiPublicKey::from_public_keys
                               -> sum_signatures / sum_public_keys (src/multi_signature.rs:80-107, multi_public_key.rs:79-83)
  Signature::verify_secure[_with_mode] -> verify_secure_batch   (src/signature.rs:177-197,256-276)
  aggregate_secure[_with_mode] -> aggregate_secure_batch  (src/secure_aggregation.rs:159-169,338-352)
                               -> verify_secure_batch_keyed / aggregate_secure_batch_keyed (members named by index
                                  into a KeySet)
  MultiSignature::verify(&MultiPublicKey::from_public_keys(..), msg)
                               -> verify_multisig_batch / verify_multisig_batch_keyed (src/multi_signature.rs:127-135)
                               -> sum_points_batch (many from_signatures / from_public_keys sums in one call)

There is no CPU fallback: importing works anywhere, but creating an Engine without the CUDA library or a GPU raises.
"""
from __future__ import annotations

import ctypes
import os
from typing import List, Optional, Sequence, Tuple

import numpy as np

# impls.rs:102-109 / sig_types.rs:8-12 / serialization.rs:10-17
Bls12381G1Impl, Bls12381G2Impl = 1, 2
class SignatureSchemes:
    Basic, MessageAugmentation, ProofOfPossession = 0, 1, 2
class SerializationFormat:
    Legacy, Modern = 0, 1

ST_OK, ST_INVALID_SIGNATURE, ST_SIG_IDENTITY, ST_PK_IDENTITY, ST_DESERIALIZE, ST_LEGACY_FORMAT = 0, 1, 2, 3, 4, 5
ST_INVALID_LENGTH, ST_INVALID_COEFFICIENT, ST_DUPLICATE_MESSAGES, ST_SCHEME, ST_MISMATCHED_LENGTHS = 6, 7, 8, 9, 10
ST_VSSS = 11
ST_INVALID_PROOF, ST_COMMITMENT_IDENTITY, ST_PROOF_IDENTITY, ST_ZERO_CHALLENGE = 12, 13, 14, 15

_STATUS_TEXT = {
    ST_INVALID_SIGNATURE: "invalid signature",
    ST_SIG_IDENTITY: "invalid inputs: signature is the identity point",
    ST_PK_IDENTITY: "invalid inputs: public key is the identity point",
    ST_DESERIALIZE: "deserialization error: invalid point",
    ST_LEGACY_FORMAT: "legacy format error: unexpected bits in byte[0]",
    ST_INVALID_LENGTH: "invalid length",
    ST_INVALID_COEFFICIENT: "invalid coefficient: zero coefficient generated",
    ST_DUPLICATE_MESSAGES: "invalid inputs: duplicate messages detected",
    ST_SCHEME: "Invalid signature scheme",
    ST_MISMATCHED_LENGTHS: "invalid inputs: Mismatched array lengths",
    ST_VSSS: "an error occurred during secret sharing",
    ST_INVALID_PROOF: "invalid proof",
    ST_COMMITMENT_IDENTITY: "invalid inputs: commitment is the identity point",
    ST_PROOF_IDENTITY: "invalid inputs: proof is the identity point",
    ST_ZERO_CHALLENGE: "invalid inputs: y is the zero",
}

STAGES = ["decode_pk", "decode_sig", "hash_to_curve", "scale_sig", "miller", "reduce", "final", "bisect"]
# BLSGPU_KERNEL_* of include/blsgpu.h, in index order
KERNELS = ["k_decode_pk", "k_subgroup_check_pk", "k_decode_sig", "k_subgroup_check_sig", "k_hash", "k_clear_cofactor",
           "k_to_affine_batch", "k_m6_prep", "k_m6_lines", "k_m6_accum"]


class BlsError(Exception):
    """Mirror of blsful::BlsError (reference src/error.rs:5-55); `.status` is the C-ABI status code."""

    def __init__(self, status: int, detail: str = ""):
        self.status = status
        super().__init__(_STATUS_TEXT.get(status, f"status {status}") + (f" ({detail})" if detail else ""))


class EngineError(RuntimeError):
    """Engine-level failure (CUDA, allocation, argument). There is no CPU path to fall back to."""


def pk_len(impl_id: int) -> int:
    return 48 if impl_id == Bls12381G2Impl else 96


def sig_len(impl_id: int) -> int:
    return 96 if impl_id == Bls12381G2Impl else 48


_LIB_NAME = "libblsgpu.so"


def lib_path() -> str:
    if os.environ.get("BLSGPU_LIB"):  # build experiments only
        return os.environ["BLSGPU_LIB"]
    return os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), _LIB_NAME)


_lib = None


def load_library() -> ctypes.CDLL:
    global _lib
    if _lib is not None:
        return _lib
    path = lib_path()
    if not os.path.exists(path):
        raise EngineError(f"{path} is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
                          "(no CPU fallback exists)")
    lib = ctypes.CDLL(path)
    c = ctypes
    u8p, u64p, i64p, vp = c.c_void_p, c.c_void_p, c.c_void_p, c.c_void_p
    sigs = {
        "blsgpu_ctx_create": (c.c_int, [c.POINTER(c.c_int), c.c_int, c.POINTER(vp)]),
        "blsgpu_ctx_destroy": (None, [vp]),
        "blsgpu_last_error": (c.c_char_p, [vp]),
        "blsgpu_ctx_set_rlc_salt": (c.c_int, [vp, u8p]),
        "blsgpu_ctx_set_rlc_bits": (c.c_int, [vp, c.c_int]),
        "blsgpu_ctx_set_stream": (c.c_int, [vp, vp]),
        "blsgpu_verify_batch": (c.c_int, [vp, c.c_int, c.c_int, c.c_int, c.c_size_t, u8p, u8p, u8p, u64p, u8p]),
        "blsgpu_verify_batch_dev": (c.c_int, [vp, c.c_int, c.c_int, c.c_int, c.c_size_t, u8p, u8p, u8p, u64p, u8p]),
        "blsgpu_verify_batch_grouped": (c.c_int, [vp, c.c_int, c.c_int, c.c_int, c.c_size_t, u8p, u8p, vp, c.c_size_t, u8p, u64p, u8p]),
        "blsgpu_keyset_create": (c.c_int, [vp, c.c_int, c.c_int, c.c_size_t, u8p, u8p, c.POINTER(c.c_uint64)]),
        "blsgpu_keyset_destroy": (c.c_int, [vp, c.c_uint64]),
        "blsgpu_keyset_update": (c.c_int, [vp, c.c_uint64, c.c_int, c.c_size_t, vp, u8p, u8p]),
        "blsgpu_keyset_append": (c.c_int, [vp, c.c_uint64, c.c_int, c.c_size_t, u8p, u8p]),
        "blsgpu_verify_batch_keyed": (c.c_int, [vp, c.c_uint64, c.c_int, c.c_int, c.c_size_t, vp, u8p, u8p, u64p, u8p]),
        "blsgpu_verify_batch_grouped_keyed": (c.c_int, [vp, c.c_uint64, c.c_int, c.c_int, c.c_size_t, vp, u8p, vp, c.c_size_t, u8p, u64p, u8p]),
        "blsgpu_miller_partial": (c.c_int, [vp, c.c_int, c.c_int, c.c_int, c.c_size_t, u8p, u8p, u8p, u64p, u8p, u8p]),
        "blsgpu_final_exp_is_one": (c.c_int, [vp, c.c_int, c.c_size_t, u8p, u8p, c.POINTER(c.c_int)]),
        "blsgpu_partial_finish": (c.c_int, [vp, c.c_int, u8p]),
        "blsgpu_pop_verify_batch": (c.c_int, [vp, c.c_int, c.c_int, c.c_size_t, u8p, u8p, u8p]),
        "blsgpu_aggregate_verify": (c.c_int, [vp, c.c_int, c.c_int, c.c_int, c.c_size_t, u8p, u8p, u64p, u8p, u8p, i64p]),
        "blsgpu_aggregate_verify_batch": (c.c_int, [vp, c.c_int, c.c_int, c.c_int, c.c_size_t, u64p, u8p, u8p, u64p, u8p, u8p, i64p]),
        "blsgpu_sum_points": (c.c_int, [vp, c.c_int, c.c_int, c.c_size_t, u8p, u8p, u8p, i64p]),
        "blsgpu_verify_secure_batch": (c.c_int, [vp, c.c_int, c.c_int, c.c_int, c.c_size_t, u64p, u8p, u8p, u8p, u64p, u8p]),
        "blsgpu_aggregate_secure_batch": (c.c_int, [vp, c.c_int, c.c_int, c.c_size_t, u64p, u8p, u8p, u8p, u8p]),
        "blsgpu_verify_secure_batch_keyed": (c.c_int, [vp, c.c_uint64, c.c_int, c.c_int, c.c_size_t, u64p, vp, u8p, u8p, u64p, u8p]),
        "blsgpu_aggregate_secure_batch_keyed": (c.c_int, [vp, c.c_uint64, c.c_int, c.c_size_t, u64p, vp, u8p, u8p, u8p]),
        "blsgpu_verify_multisig_batch": (c.c_int, [vp, c.c_int, c.c_int, c.c_int, c.c_size_t, u64p, u8p, u8p, u8p, u64p, u8p]),
        "blsgpu_verify_multisig_batch_keyed": (c.c_int, [vp, c.c_uint64, c.c_int, c.c_int, c.c_size_t, u64p, vp, u8p, u8p, u64p, u8p]),
        "blsgpu_sum_points_batch": (c.c_int, [vp, c.c_int, c.c_int, c.c_size_t, u64p, u8p, u8p, u8p, i64p]),
        "blsgpu_hash_to_curve_batch": (c.c_int, [vp, c.c_int, c.c_size_t, u8p, u64p, u8p, c.c_size_t, u8p]),
        "blsgpu_recode_points": (c.c_int, [vp, c.c_int, c.c_int, c.c_int, c.c_size_t, u8p, u8p, u8p]),
        "blsgpu_fp_mul_batch": (c.c_int, [vp, c.c_int, c.c_size_t, u8p, u8p, u8p]),
        "blsgpu_pairing_product_is_one": (c.c_int, [vp, c.c_size_t, u8p, u8p, c.POINTER(c.c_int)]),
        "blsgpu_testdata_sign": (c.c_int, [vp, c.c_int, c.c_int, c.c_size_t, u8p, u8p, u64p, u8p, u8p]),
        "blsgpu_combine_shares_batch": (c.c_int, [vp, c.c_int, c.c_size_t, u64p, u8p, u8p, u8p]),
        "blsgpu_verify_batch_wire": (c.c_int, [vp, c.c_int, c.c_size_t, u8p, u8p, u8p, u64p, u8p]),
        "blsgpu_pairing_check_batch": (c.c_int, [vp, c.c_size_t, u64p, u8p, u8p, u8p, u8p]),
        "blsgpu_signcrypt_valid_batch": (c.c_int, [vp, c.c_int, c.c_int, c.c_size_t, u8p, u8p, u8p, u64p, u8p, u8p]),
        "blsgpu_signcrypt_verify_share_batch": (c.c_int, [vp, c.c_int, c.c_int, c.c_size_t, u8p, u8p, u8p, u8p, u8p, u64p, u8p, u8p]),
        "blsgpu_pok_verify_batch": (c.c_int, [vp, c.c_int, c.c_int, c.c_size_t, u8p, u8p, u8p, u8p, u8p, u64p, u8p]),
        "blsgpu_verify_batch_records": (c.c_int, [vp, c.c_int, c.c_int, c.c_int, c.c_size_t, u8p, u64p, u8p, u64p, u8p, u64p, u8p]),
        "blsgpu_selftest": (c.c_int, [vp]),
        "blsgpu_plan_msm": (c.c_int, [c.c_size_t, c.c_int, c.POINTER(c.c_int), c.POINTER(c.c_int), c.POINTER(c.c_int)]),
        "blsgpu_plan_shards": (c.c_int, [c.c_size_t, c.c_void_p, c.c_int, c.c_void_p]),
        "blsgpu_imad_peak": (c.c_int, [vp, c.POINTER(c.c_double)]),
        "blsgpu_verify_share_batch": (c.c_int, [vp, c.c_int, c.c_int, c.c_size_t, vp, vp, vp, vp, vp]),
        "blsgpu_last_stage_ms": (c.c_int, [vp, c.POINTER(c.c_float)]),
        "blsgpu_last_kernel_ms": (c.c_int, [vp, c.POINTER(c.c_float), c.POINTER(c.c_int)]),
        "blsgpu_launch_count": (c.c_uint64, [vp]),
    }
    for name, (res, args) in sigs.items():
        fn = getattr(lib, name)  # AttributeError here means the library does not export what include/blsgpu.h declares
        fn.restype, fn.argtypes = res, args
    _lib = lib
    return lib


EXPORTED_SYMBOLS = [
    "blsgpu_ctx_create", "blsgpu_ctx_destroy", "blsgpu_last_error", "blsgpu_ctx_set_rlc_salt", "blsgpu_ctx_set_rlc_bits",
    "blsgpu_ctx_set_stream",
    "blsgpu_verify_batch", "blsgpu_verify_batch_grouped",
    "blsgpu_keyset_create", "blsgpu_keyset_destroy", "blsgpu_keyset_update", "blsgpu_keyset_append", "blsgpu_verify_batch_keyed", "blsgpu_verify_batch_grouped_keyed",
    "blsgpu_miller_partial", "blsgpu_final_exp_is_one", "blsgpu_partial_finish",
    "blsgpu_verify_batch_dev", "blsgpu_pop_verify_batch", "blsgpu_aggregate_verify", "blsgpu_aggregate_verify_batch", "blsgpu_sum_points",
    "blsgpu_verify_secure_batch", "blsgpu_aggregate_secure_batch",
    "blsgpu_verify_secure_batch_keyed", "blsgpu_aggregate_secure_batch_keyed",
    "blsgpu_verify_multisig_batch", "blsgpu_verify_multisig_batch_keyed", "blsgpu_sum_points_batch", "blsgpu_hash_to_curve_batch", "blsgpu_recode_points",
    "blsgpu_fp_mul_batch", "blsgpu_pairing_product_is_one", "blsgpu_testdata_sign", "blsgpu_imad_peak",
    "blsgpu_combine_shares_batch", "blsgpu_verify_batch_wire", "blsgpu_pairing_check_batch",
    "blsgpu_signcrypt_valid_batch", "blsgpu_signcrypt_verify_share_batch", "blsgpu_pok_verify_batch", "blsgpu_verify_batch_records", "blsgpu_selftest", "blsgpu_plan_msm", "blsgpu_plan_shards", "blsgpu_verify_share_batch", "blsgpu_last_stage_ms", "blsgpu_last_kernel_ms", "blsgpu_launch_count",
]


def _u8(buf) -> np.ndarray:
    if isinstance(buf, np.ndarray):
        a = buf
        if a.dtype != np.uint8:
            a = a.view(np.uint8)
        return np.ascontiguousarray(a).reshape(-1)
    return np.frombuffer(bytes(buf), dtype=np.uint8)


def _ptr(a: Optional[np.ndarray]):
    return None if a is None or a.size == 0 else a.ctypes.data


def shard_range(n: int, rank: int, world: int) -> Tuple[int, int]:
    """Contiguous slice [lo, hi) of an n-item batch owned by `rank` of `world` (one process per GPU; the slices are
    independent units - there is no data-path collective, SURVEY.md 8e)."""
    if world < 1 or not 0 <= rank < world:
        raise ValueError("bad rank/world")
    base, rem = divmod(n, world)
    lo = rank * base + min(rank, rem)
    return lo, lo + base + (1 if rank < rem else 0)


def verify_batch_sharded(verify_slice, n: int, rank: int, world: int, gather=None) -> np.ndarray:
    """Runs `verify_slice(lo, hi) -> uint8[hi-lo]` on this rank's slice and, if `gather` (a torch.distributed-style
    all_gather_object callable) is given, assembles the full status vector on every rank in batch order."""
    lo, hi = shard_range(n, rank, world)
    mine = np.asarray(verify_slice(lo, hi), dtype=np.uint8)
    if mine.shape != (hi - lo,):
        raise ValueError("verify_slice returned the wrong number of statuses")
    if gather is None or world == 1:
        return mine
    parts = gather((lo, mine))
    out = np.empty(n, dtype=np.uint8)
    for plo, part in parts:
        out[plo:plo + part.size] = part
    return out


def verify_batch_folded(eng, impl_id: int, scheme: int, pk: np.ndarray, sg: np.ndarray, data: np.ndarray, off: np.ndarray, rank: int,
                        world: int, all_gather, fmt: int = 1) -> Tuple[int, np.ndarray]:
    """ONE batch over `world` processes (one GPU each), strong scaling (SURVEY.md 8e): this rank folds its contiguous slice
    into one partial product of Miller values and one partial sum (blsgpu_miller_partial), the partial results (672 bytes per
    rank) are exchanged with `all_gather` (a callable: object -> list of every rank's object, e.g. built on
    torch.distributed.all_gather_object), every rank runs the single Miller loop + final exponentiation of the whole batch
    (blsgpu_final_exp_is_one, redundantly: no broadcast needed) and finishes its slice.  Returns (lo, statuses of [lo, hi))."""
    n = off.size - 1
    lo, hi = shard_range(n, rank, world)
    pl, sl = pk_len(impl_id), sig_len(impl_id)
    part = eng.miller_partial(impl_id, scheme, pk[pl * lo:pl * hi], sg[sl * lo:sl * hi], data, off[lo:hi + 1], fmt)
    parts = all_gather(part) if world > 1 else [part]
    ok = eng.final_exp_is_one(impl_id, [p[0] for p in parts], [p[1] for p in parts])
    return lo, eng.partial_finish(hi - lo, ok)


def pack_messages(msgs: Sequence[bytes]) -> Tuple[np.ndarray, np.ndarray]:
    off = np.zeros(len(msgs) + 1, dtype=np.uint64)
    if len(msgs):
        off[1:] = np.cumsum([len(m) for m in msgs], dtype=np.uint64)
    data = np.frombuffer(b"".join(bytes(m) for m in msgs), dtype=np.uint8)
    return data, off


def _pack_points(points, length: int, what: str) -> np.ndarray:
    """Accepts a list of byte strings or one flat uint8 array; enforces the reference's length rule."""
    if isinstance(points, np.ndarray):
        a = _u8(points)
        if a.size % length:
            raise BlsError(ST_INVALID_LENGTH, f"{what}: expected multiples of {length} bytes")
        return a
    for p in points:
        if len(p) != length:
            raise BlsError(ST_INVALID_LENGTH, f"{what}: expected {length} bytes, got {len(p)}")
    return np.frombuffer(b"".join(bytes(p) for p in points), dtype=np.uint8)


class KeySet:
    """Public keys of one impl decoded once on the engine's first device (blsgpu_keyset_create), named by index in
    Engine.verify_batch_keyed / verify_batch_grouped_keyed.  status[i]: ST_OK, ST_DESERIALIZE or ST_LEGACY_FORMAT for key i
    (a key that failed to decode stays in the set and gives its items that status).  The engine owns the device memory:
    close() frees it, and so does Engine.close()."""

    def __init__(self, engine: "Engine", impl_id: int, ident: int, status: np.ndarray):
        self._engine = engine
        self.impl_id = impl_id
        self.id = ident
        self.status = status

    def __len__(self) -> int:
        return self.status.size

    def close(self) -> None:
        if self.id and getattr(self._engine, "_ctx", None):
            self._engine._check(self._engine._lib.blsgpu_keyset_destroy(self._engine._ctx, self.id), "blsgpu_keyset_destroy")
        self.id = 0


class Engine:
    """One blsgpu context (one host thread at a time)."""

    def __init__(self, devices: Sequence[int] = (0,)):
        self._lib = load_library()
        self._ctx = ctypes.c_void_p()
        devs = (ctypes.c_int * len(devices))(*devices)
        rc = self._lib.blsgpu_ctx_create(devs, len(devices), ctypes.byref(self._ctx))
        if rc != 0:
            msg = self._lib.blsgpu_last_error(None)
            raise EngineError(f"blsgpu_ctx_create failed ({rc}): {msg.decode() if msg else ''}")

    def close(self):
        if getattr(self, "_ctx", None):
            self._lib.blsgpu_ctx_destroy(self._ctx)
            self._ctx = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def set_stream(self, cuda_stream: int) -> None:
        """Run on a caller-owned CUDA stream (e.g. torch.cuda.Stream().cuda_stream); 0 restores the engine's own."""
        self._check(self._lib.blsgpu_ctx_set_stream(self._ctx, cuda_stream or None), "blsgpu_ctx_set_stream")

    def set_rlc_salt(self, salt: bytes) -> None:
        """Pins the salt of the batch-check scalars (tests / reproducible runs only; the default is fresh OS randomness per call)."""
        if len(salt) != 32:
            raise ValueError("salt must be 32 bytes")
        buf = np.frombuffer(bytes(salt), dtype=np.uint8)
        self._check(self._lib.blsgpu_ctx_set_rlc_salt(self._ctx, _ptr(buf)), "blsgpu_ctx_set_rlc_salt")

    def set_rlc_bits(self, bits: int) -> None:
        """64- (default) or 128-bit random-linear-combination scalars."""
        self._check(self._lib.blsgpu_ctx_set_rlc_bits(self._ctx, bits), "blsgpu_ctx_set_rlc_bits")

    def _check(self, rc: int, what: str):
        if rc != 0:
            msg = self._lib.blsgpu_last_error(self._ctx)
            raise EngineError(f"{what} failed ({rc}): {msg.decode() if msg else ''}")

    # ---- Signature::verify over slices --------------------------------------------------------------------------
    def verify_batch(self, impl_id: int, scheme: int, pks, sigs, msgs: Sequence[bytes],
                     fmt: int = SerializationFormat.Modern) -> np.ndarray:
        """status[i] == 0  <=>  Signature::verify(&pk_i, msg_i).is_ok(); other values name the reference's error."""
        pk = _pack_points(pks, pk_len(impl_id), "public key")
        sg = _pack_points(sigs, sig_len(impl_id), "signature")
        n = pk.size // pk_len(impl_id)
        if sg.size // sig_len(impl_id) != n or len(msgs) != n:
            raise BlsError(ST_MISMATCHED_LENGTHS)
        data, off = pack_messages(msgs)
        return self.verify_batch_packed(impl_id, scheme, pk, sg, data, off, fmt)

    def verify_batch_packed(self, impl_id, scheme, pk: np.ndarray, sg: np.ndarray, data: np.ndarray, off: np.ndarray,
                            fmt: int = SerializationFormat.Modern) -> np.ndarray:
        n = off.size - 1
        status = np.empty(n, dtype=np.uint8)
        rc = self._lib.blsgpu_verify_batch(self._ctx, impl_id, scheme, fmt, n, _ptr(pk), _ptr(sg), _ptr(data), _ptr(off),
                                           _ptr(status))
        self._check(rc, "blsgpu_verify_batch")
        return status

    def verify_batch_grouped(self, impl_id: int, scheme: int, pks, sigs, msg_idx, msgs: Sequence[bytes],
                             fmt: int = SerializationFormat.Modern) -> np.ndarray:
        """verify_batch where item i signs msgs[msg_idx[i]]: each message is hashed once and items of one message share
        their Miller loops.  The statuses equal verify_batch's on the same items with their messages written out."""
        pk = _pack_points(pks, pk_len(impl_id), "public key")
        sg = _pack_points(sigs, sig_len(impl_id), "signature")
        idx = np.ascontiguousarray(msg_idx, dtype=np.uint32).reshape(-1)
        n = pk.size // pk_len(impl_id)
        if sg.size // sig_len(impl_id) != n or idx.size != n:
            raise BlsError(ST_MISMATCHED_LENGTHS)
        data, off = pack_messages(msgs)
        return self.verify_batch_grouped_packed(impl_id, scheme, pk, sg, idx, data, off, fmt)

    def verify_batch_grouped_packed(self, impl_id, scheme, pk: np.ndarray, sg: np.ndarray, msg_idx: np.ndarray, data: np.ndarray,
                                    off: np.ndarray, fmt: int = SerializationFormat.Modern) -> np.ndarray:
        """Flat-buffer form: msg_idx uint32[n], the q messages as data / off (q + 1 offsets)."""
        msg_idx = np.ascontiguousarray(msg_idx, dtype=np.uint32).reshape(-1)
        n = msg_idx.size
        status = np.empty(n, dtype=np.uint8)
        rc = self._lib.blsgpu_verify_batch_grouped(self._ctx, impl_id, scheme, fmt, n, _ptr(pk), _ptr(sg), _ptr(msg_idx), off.size - 1,
                                                   _ptr(data), _ptr(off), _ptr(status))
        self._check(rc, "blsgpu_verify_batch_grouped")
        return status

    # ---- key sets: public keys decoded once, verify calls that name them by index -----------------------------------
    def key_set(self, impl_id: int, pks, fmt: int = SerializationFormat.Modern) -> KeySet:
        """Decodes and subgroup-checks the keys once; they stay in device memory until KeySet.close() or Engine.close()."""
        pk = _pack_points(pks, pk_len(impl_id), "public key")
        n = pk.size // pk_len(impl_id)
        status = np.zeros(n, dtype=np.uint8)
        ident = ctypes.c_uint64(0)
        self._check(self._lib.blsgpu_keyset_create(self._ctx, impl_id, fmt, n, _ptr(pk), _ptr(status), ctypes.byref(ident)),
                    "blsgpu_keyset_create")
        return KeySet(self, impl_id, ident.value, status)

    def update_key_set(self, keys: KeySet, key_idx, pks, fmt: int = SerializationFormat.Modern) -> np.ndarray:
        """Key key_idx[i] of `keys` becomes pks[i], decoded in fmt (blsgpu_keyset_update): the set keeps its id and every
        other key.  Returns the k decode statuses, which keys.status takes over."""
        pk = _pack_points(pks, pk_len(keys.impl_id), "public key")
        idx = np.ascontiguousarray(key_idx, dtype=np.uint32).reshape(-1)
        k = pk.size // pk_len(keys.impl_id)
        if idx.size != k:
            raise BlsError(ST_MISMATCHED_LENGTHS)
        status = np.zeros(k, dtype=np.uint8)
        self._check(self._lib.blsgpu_keyset_update(self._ctx, keys.id, fmt, k, _ptr(idx), _ptr(pk), _ptr(status)), "blsgpu_keyset_update")
        keys.status = keys.status.copy()
        keys.status[idx] = status
        return status

    def append_key_set(self, keys: KeySet, pks, fmt: int = SerializationFormat.Modern) -> np.ndarray:
        """Appends pks, decoded in fmt, to `keys` (blsgpu_keyset_append): they take indices len(keys) onwards.  Returns their
        decode statuses, which keys.status takes over."""
        pk = _pack_points(pks, pk_len(keys.impl_id), "public key")
        k = pk.size // pk_len(keys.impl_id)
        status = np.zeros(k, dtype=np.uint8)
        self._check(self._lib.blsgpu_keyset_append(self._ctx, keys.id, fmt, k, _ptr(pk), _ptr(status)), "blsgpu_keyset_append")
        keys.status = np.concatenate([keys.status, status])
        return status

    def verify_batch_keyed(self, keys: KeySet, scheme: int, key_idx, sigs, msgs: Sequence[bytes],
                           fmt: int = SerializationFormat.Modern) -> np.ndarray:
        """verify_batch with pks[i] = key key_idx[i] of `keys` (fmt is the signatures' format)."""
        sg = _pack_points(sigs, sig_len(keys.impl_id), "signature")
        idx = np.ascontiguousarray(key_idx, dtype=np.uint32).reshape(-1)
        if sg.size // sig_len(keys.impl_id) != idx.size or len(msgs) != idx.size:
            raise BlsError(ST_MISMATCHED_LENGTHS)
        data, off = pack_messages(msgs)
        return self.verify_batch_keyed_packed(keys, scheme, idx, sg, data, off, fmt)

    def verify_batch_keyed_packed(self, keys: KeySet, scheme: int, key_idx: np.ndarray, sg: np.ndarray, data: np.ndarray, off: np.ndarray,
                                  fmt: int = SerializationFormat.Modern) -> np.ndarray:
        """Flat-buffer form: key_idx uint32[n], sg n signatures, the n messages as data / off (n + 1 offsets)."""
        key_idx = np.ascontiguousarray(key_idx, dtype=np.uint32).reshape(-1)
        n = off.size - 1
        if key_idx.size != n:
            raise BlsError(ST_MISMATCHED_LENGTHS)
        status = np.empty(n, dtype=np.uint8)
        rc = self._lib.blsgpu_verify_batch_keyed(self._ctx, keys.id, scheme, fmt, n, _ptr(key_idx), _ptr(sg), _ptr(data), _ptr(off),
                                                 _ptr(status))
        self._check(rc, "blsgpu_verify_batch_keyed")
        return status

    def verify_batch_grouped_keyed(self, keys: KeySet, scheme: int, key_idx, sigs, msg_idx, msgs: Sequence[bytes],
                                   fmt: int = SerializationFormat.Modern) -> np.ndarray:
        """verify_batch_grouped with pks[i] = key key_idx[i] of `keys` (fmt is the signatures' format)."""
        sg = _pack_points(sigs, sig_len(keys.impl_id), "signature")
        kidx = np.ascontiguousarray(key_idx, dtype=np.uint32).reshape(-1)
        midx = np.ascontiguousarray(msg_idx, dtype=np.uint32).reshape(-1)
        n = kidx.size
        if sg.size // sig_len(keys.impl_id) != n or midx.size != n:
            raise BlsError(ST_MISMATCHED_LENGTHS)
        data, off = pack_messages(msgs)
        return self.verify_batch_grouped_keyed_packed(keys, scheme, kidx, sg, midx, data, off, fmt)

    def verify_batch_grouped_keyed_packed(self, keys: KeySet, scheme: int, key_idx: np.ndarray, sg: np.ndarray, msg_idx: np.ndarray,
                                          data: np.ndarray, off: np.ndarray, fmt: int = SerializationFormat.Modern) -> np.ndarray:
        """Flat-buffer form: key_idx and msg_idx uint32[n], sg n signatures, the q messages as data / off (q + 1 offsets)."""
        key_idx = np.ascontiguousarray(key_idx, dtype=np.uint32).reshape(-1)
        msg_idx = np.ascontiguousarray(msg_idx, dtype=np.uint32).reshape(-1)
        n = msg_idx.size
        if key_idx.size != n:
            raise BlsError(ST_MISMATCHED_LENGTHS)
        status = np.empty(n, dtype=np.uint8)
        rc = self._lib.blsgpu_verify_batch_grouped_keyed(self._ctx, keys.id, scheme, fmt, n, _ptr(key_idx), _ptr(sg), _ptr(msg_idx),
                                                         off.size - 1, _ptr(data), _ptr(off), _ptr(status))
        self._check(rc, "blsgpu_verify_batch_grouped_keyed")
        return status

    def verify_batch_dev(self, impl_id, scheme, n, pk_ptr: int, sig_ptr: int, msg_ptr: int, off_ptr: int, status_ptr: int,
                         fmt: int = SerializationFormat.Modern) -> None:
        rc = self._lib.blsgpu_verify_batch_dev(self._ctx, impl_id, scheme, fmt, n, pk_ptr, sig_ptr, msg_ptr, off_ptr, status_ptr)
        self._check(rc, "blsgpu_verify_batch_dev")

    # ---- one batch over several GPUs / processes: slice-local partial results, fold, finish (SURVEY 8e) ------------
    def miller_partial(self, impl_id, scheme, pk: np.ndarray, sg: np.ndarray, data: np.ndarray, off: np.ndarray,
                       fmt: int = SerializationFormat.Modern) -> Tuple[bytes, bytes]:
        """This slice's (product of Miller values as 576 bytes, sum of r_i sig_i as a compressed point)."""
        n = off.size - 1
        gt = np.zeros(576, dtype=np.uint8)
        sm = np.zeros(sig_len(impl_id), dtype=np.uint8)
        rc = self._lib.blsgpu_miller_partial(self._ctx, impl_id, scheme, fmt, n, _ptr(pk), _ptr(sg), _ptr(data), _ptr(off), _ptr(gt), _ptr(sm))
        self._check(rc, "blsgpu_miller_partial")
        return gt.tobytes(), sm.tobytes()

    def final_exp_is_one(self, impl_id, partial_gts: Sequence[bytes], partial_sums: Sequence[bytes]) -> bool:
        k = len(partial_gts)
        gts = np.frombuffer(b"".join(partial_gts), dtype=np.uint8)
        sums = np.frombuffer(b"".join(partial_sums), dtype=np.uint8)
        res = ctypes.c_int(0)
        self._check(self._lib.blsgpu_final_exp_is_one(self._ctx, impl_id, k, _ptr(gts), _ptr(sums), ctypes.byref(res)), "blsgpu_final_exp_is_one")
        return bool(res.value)

    def partial_finish(self, n: int, batch_ok: bool) -> np.ndarray:
        status = np.zeros(n, dtype=np.uint8)
        self._check(self._lib.blsgpu_partial_finish(self._ctx, 1 if batch_ok else 0, _ptr(status)), "blsgpu_partial_finish")
        return status

    def pop_verify_batch(self, impl_id: int, pks, sigs, fmt: int = SerializationFormat.Modern) -> np.ndarray:
        pk = _pack_points(pks, pk_len(impl_id), "public key")
        sg = _pack_points(sigs, sig_len(impl_id), "proof of possession")
        n = pk.size // pk_len(impl_id)
        if sg.size // sig_len(impl_id) != n:
            raise BlsError(ST_MISMATCHED_LENGTHS)
        status = np.empty(n, dtype=np.uint8)
        self._check(self._lib.blsgpu_pop_verify_batch(self._ctx, impl_id, fmt, n, _ptr(pk), _ptr(sg), _ptr(status)),
                    "blsgpu_pop_verify_batch")
        return status

    # ---- AggregateSignature::verify -------------------------------------------------------------------------------
    def aggregate_verify(self, impl_id: int, scheme: int, pks, msgs: Sequence[bytes], sig: bytes,
                         fmt: int = SerializationFormat.Modern) -> None:
        """Returns None on success, raises BlsError like AggregateSignature::verify (aggregate_signature.rs:230-239)."""
        st, idx = self.aggregate_verify_status(impl_id, scheme, pks, msgs, sig, fmt)
        if st != ST_OK:
            detail = ""
            if st == ST_DUPLICATE_MESSAGES:
                detail = f"at {idx[0]} and {idx[1]}"
            elif st == ST_PK_IDENTITY:
                detail = f"public key at {idx[0]}"
            raise BlsError(st, detail)

    def aggregate_verify_status(self, impl_id, scheme, pks, msgs, sig, fmt=SerializationFormat.Modern):
        pk = _pack_points(pks, pk_len(impl_id), "public key")
        n = pk.size // pk_len(impl_id)
        if len(msgs) != n:
            raise BlsError(ST_MISMATCHED_LENGTHS)
        if len(sig) != sig_len(impl_id):
            raise BlsError(ST_INVALID_LENGTH, "signature")
        data, off = pack_messages(msgs)
        sg = _u8(sig)
        status = np.zeros(1, dtype=np.uint8)
        idx = np.full(2, -1, dtype=np.int64)
        rc = self._lib.blsgpu_aggregate_verify(self._ctx, impl_id, scheme, fmt, n, _ptr(pk), _ptr(data), _ptr(off), _ptr(sg),
                                               _ptr(status), _ptr(idx))
        self._check(rc, "blsgpu_aggregate_verify")
        return int(status[0]), (int(idx[0]), int(idx[1]))

    def aggregate_verify_batch_status(self, impl_id: int, scheme: int, sets: Sequence[Tuple[Sequence[bytes], Sequence[bytes]]],
                                      sigs, fmt: int = SerializationFormat.Modern) -> Tuple[np.ndarray, np.ndarray]:
        """q x aggregate_verify_status in one engine call: sets[j] = (pks, msgs) of aggregate j, sigs[j] its signature.
        Returns (status uint8[q], index int64[q, 2]) with the meaning aggregate_verify_status gives each aggregate alone."""
        q = len(sets)
        pl = pk_len(impl_id)
        flat_pks, flat_msgs = [], []
        soff = np.zeros(q + 1, dtype=np.uint64)
        for j, (pks, msgs) in enumerate(sets):
            pk = _pack_points(pks, pl, "public key")
            if len(msgs) != pk.size // pl:
                raise BlsError(ST_MISMATCHED_LENGTHS)
            flat_pks.append(pk)
            flat_msgs.extend(msgs)
            soff[j + 1] = soff[j] + pk.size // pl
        if isinstance(sigs, np.ndarray):
            sg = _pack_points(sigs, sig_len(impl_id), "signature")
        else:
            for s in sigs:
                if len(s) != sig_len(impl_id):
                    raise BlsError(ST_INVALID_LENGTH, "signature")
            sg = np.frombuffer(b"".join(bytes(s) for s in sigs), dtype=np.uint8)
        if sg.size // sig_len(impl_id) != q:
            raise BlsError(ST_MISMATCHED_LENGTHS)
        pk = np.concatenate(flat_pks) if flat_pks else np.zeros(0, dtype=np.uint8)
        data, off = pack_messages(flat_msgs)
        return self.aggregate_verify_batch_packed(impl_id, scheme, soff, pk, data, off, sg, fmt)

    def aggregate_verify_batch_packed(self, impl_id, scheme, set_off: np.ndarray, pk: np.ndarray, data: np.ndarray, off: np.ndarray,
                                      sg: np.ndarray, fmt: int = SerializationFormat.Modern) -> Tuple[np.ndarray, np.ndarray]:
        """Flat-buffer form: set_off[q + 1] pair offsets per aggregate, pk / data / off over all pairs, sg q signatures."""
        q = set_off.size - 1
        status = np.zeros(q, dtype=np.uint8)
        idx = np.full((q, 2), -1, dtype=np.int64)
        rc = self._lib.blsgpu_aggregate_verify_batch(self._ctx, impl_id, scheme, fmt, q, _ptr(set_off), _ptr(pk), _ptr(data), _ptr(off),
                                                     _ptr(sg), _ptr(status), _ptr(idx))
        self._check(rc, "blsgpu_aggregate_verify_batch")
        return status, idx

    # ---- point sums -------------------------------------------------------------------------------------------------
    def sum_points(self, group: int, points, fmt: int = SerializationFormat.Modern) -> bytes:
        length = 48 if group == 1 else 96
        pts = _pack_points(points, length, "point")
        n = pts.size // length
        out = np.zeros(length, dtype=np.uint8)
        status = np.zeros(1, dtype=np.uint8)
        bad = np.full(1, -1, dtype=np.int64)
        rc = self._lib.blsgpu_sum_points(self._ctx, group, fmt, n, _ptr(pts), _ptr(out), _ptr(status), _ptr(bad))
        self._check(rc, "blsgpu_sum_points")
        if status[0] != ST_OK:
            raise BlsError(int(status[0]), f"element {int(bad[0])}")
        return out.tobytes()

    def sum_signatures(self, impl_id: int, sigs, fmt: int = SerializationFormat.Modern, multi: bool = False,
                       schemes: Optional[Sequence[int]] = None) -> bytes:
        """AggregateSignature/MultiSignature::from_signatures (aggregate_signature.rs:123-148, multi_signature.rs:80-107):
        fewer than 2 signatures -> InvalidSignature; mixed schemes -> InvalidSignatureScheme; MultiSignature rejects
        MessageAugmentation elements at positions >= 1."""
        n = len(sigs) if not isinstance(sigs, np.ndarray) else sigs.size // sig_len(impl_id)
        if n < 2:
            raise BlsError(ST_INVALID_SIGNATURE)
        if schemes is not None:
            for s in schemes[1:]:
                if s != schemes[0] or (multi and s == SignatureSchemes.MessageAugmentation):
                    raise BlsError(ST_SCHEME)
        return self.sum_points(1 if impl_id == Bls12381G1Impl else 2, sigs, fmt)

    def sum_public_keys(self, impl_id: int, pks, fmt: int = SerializationFormat.Modern) -> bytes:
        """MultiPublicKey::from_public_keys (multi_public_key.rs:79-83)."""
        return self.sum_points(2 if impl_id == Bls12381G1Impl else 1, pks, fmt)

    # ---- secure aggregation -------------------------------------------------------------------------------------------
    def verify_secure_batch(self, impl_id: int, scheme: int, key_sets: Sequence[Sequence[bytes]], sigs, msgs: Sequence[bytes],
                            fmt: int = SerializationFormat.Modern) -> np.ndarray:
        q = len(key_sets)
        koff = np.zeros(q + 1, dtype=np.uint64)
        if q:
            koff[1:] = np.cumsum([len(k) for k in key_sets], dtype=np.uint64)
        flat = [k for ks in key_sets for k in ks]
        pk = _pack_points(flat, pk_len(impl_id), "public key")
        sg = _pack_points(sigs, sig_len(impl_id), "signature")
        if sg.size // sig_len(impl_id) != q or len(msgs) != q:
            raise BlsError(ST_MISMATCHED_LENGTHS)
        data, off = pack_messages(msgs)
        return self.verify_secure_batch_packed(impl_id, scheme, koff, pk, sg, data, off, fmt)

    def verify_secure_batch_packed(self, impl_id, scheme, koff, pk, sg, data, off, fmt=SerializationFormat.Modern):
        q = koff.size - 1
        status = np.empty(q, dtype=np.uint8)
        rc = self._lib.blsgpu_verify_secure_batch(self._ctx, impl_id, scheme, fmt, q, _ptr(koff), _ptr(pk), _ptr(sg), _ptr(data),
                                                  _ptr(off), _ptr(status))
        self._check(rc, "blsgpu_verify_secure_batch")
        return status

    def aggregate_secure_batch_packed(self, impl_id: int, koff: np.ndarray, pk: np.ndarray, sg: np.ndarray,
                                      fmt: int = SerializationFormat.Modern) -> Tuple[np.ndarray, np.ndarray]:
        """Flat-buffer form: koff[q + 1] key offsets, pk all keys, sg one signature per key; returns (status[q], q signatures flat)."""
        q = koff.size - 1
        out = np.zeros(q * sig_len(impl_id), dtype=np.uint8)
        status = np.empty(q, dtype=np.uint8)
        rc = self._lib.blsgpu_aggregate_secure_batch(self._ctx, impl_id, fmt, q, _ptr(koff), _ptr(pk), _ptr(sg), _ptr(out), _ptr(status))
        self._check(rc, "blsgpu_aggregate_secure_batch")
        return status, out

    def verify_secure_batch_keyed(self, keys: KeySet, scheme: int, key_idx_sets: Sequence[Sequence[int]], sigs, msgs: Sequence[bytes],
                                  fmt: int = SerializationFormat.Modern) -> np.ndarray:
        """verify_secure_batch with quorum j's keys = keys of `keys` at key_idx_sets[j], encoded in fmt."""
        q = len(key_idx_sets)
        koff = np.zeros(q + 1, dtype=np.uint64)
        if q:
            koff[1:] = np.cumsum([len(k) for k in key_idx_sets], dtype=np.uint64)
        idx = np.array([k for ks in key_idx_sets for k in ks], dtype=np.uint32)
        sg = _pack_points(sigs, sig_len(keys.impl_id), "signature")
        if sg.size // sig_len(keys.impl_id) != q or len(msgs) != q:
            raise BlsError(ST_MISMATCHED_LENGTHS)
        data, off = pack_messages(msgs)
        return self.verify_secure_batch_keyed_packed(keys, scheme, koff, idx, sg, data, off, fmt)

    def verify_secure_batch_keyed_packed(self, keys: KeySet, scheme: int, koff: np.ndarray, key_idx: np.ndarray, sg: np.ndarray,
                                         data: np.ndarray, off: np.ndarray, fmt: int = SerializationFormat.Modern) -> np.ndarray:
        """Flat-buffer form: koff[q + 1] member offsets, key_idx uint32[koff[q]], sg q signatures, the q messages as data / off."""
        koff = np.ascontiguousarray(koff, dtype=np.uint64).reshape(-1)
        key_idx = np.ascontiguousarray(key_idx, dtype=np.uint32).reshape(-1)
        q = koff.size - 1
        if key_idx.size != (int(koff[-1]) if q else 0) or off.size - 1 != q:
            raise BlsError(ST_MISMATCHED_LENGTHS)
        status = np.empty(q, dtype=np.uint8)
        rc = self._lib.blsgpu_verify_secure_batch_keyed(self._ctx, keys.id, scheme, fmt, q, _ptr(koff), _ptr(key_idx), _ptr(sg), _ptr(data),
                                                        _ptr(off), _ptr(status))
        self._check(rc, "blsgpu_verify_secure_batch_keyed")
        return status

    def aggregate_secure_batch_keyed(self, keys: KeySet, key_idx_sets: Sequence[Sequence[int]], sig_sets: Sequence[Sequence[bytes]],
                                     fmt: int = SerializationFormat.Modern) -> Tuple[np.ndarray, List[bytes]]:
        """aggregate_secure_batch with quorum j's keys = keys of `keys` at key_idx_sets[j], encoded in fmt."""
        q = len(key_idx_sets)
        if len(sig_sets) != q or any(len(k) != len(s) for k, s in zip(key_idx_sets, sig_sets)):
            raise BlsError(ST_MISMATCHED_LENGTHS)
        koff = np.zeros(q + 1, dtype=np.uint64)
        if q:
            koff[1:] = np.cumsum([len(k) for k in key_idx_sets], dtype=np.uint64)
        idx = np.array([k for ks in key_idx_sets for k in ks], dtype=np.uint32)
        sg = _pack_points([s for ss in sig_sets for s in ss], sig_len(keys.impl_id), "signature")
        status, out = self.aggregate_secure_batch_keyed_packed(keys, koff, idx, sg, fmt)
        L = sig_len(keys.impl_id)
        return status, [out[j * L:(j + 1) * L].tobytes() for j in range(q)]

    def aggregate_secure_batch_keyed_packed(self, keys: KeySet, koff: np.ndarray, key_idx: np.ndarray, sg: np.ndarray,
                                            fmt: int = SerializationFormat.Modern) -> Tuple[np.ndarray, np.ndarray]:
        """Flat-buffer form: koff[q + 1] member offsets, key_idx uint32[koff[q]], sg one signature per member; returns
        (status[q], q signatures flat)."""
        koff = np.ascontiguousarray(koff, dtype=np.uint64).reshape(-1)
        key_idx = np.ascontiguousarray(key_idx, dtype=np.uint32).reshape(-1)
        sg = _pack_points(sg, sig_len(keys.impl_id), "signature")
        q = koff.size - 1
        m = int(koff[-1]) if q else 0
        if key_idx.size != m or sg.size // sig_len(keys.impl_id) != m:
            raise BlsError(ST_MISMATCHED_LENGTHS)
        out = np.zeros(q * sig_len(keys.impl_id), dtype=np.uint8)
        status = np.empty(q, dtype=np.uint8)
        rc = self._lib.blsgpu_aggregate_secure_batch_keyed(self._ctx, keys.id, fmt, q, _ptr(koff), _ptr(key_idx), _ptr(sg), _ptr(out),
                                                           _ptr(status))
        self._check(rc, "blsgpu_aggregate_secure_batch_keyed")
        return status, out

    # ---- multi-signatures over signer subsets ----------------------------------------------------------------------------
    def verify_multisig_batch(self, impl_id: int, scheme: int, key_sets: Sequence[Sequence[bytes]], sigs, msgs: Sequence[bytes],
                              fmt: int = SerializationFormat.Modern) -> np.ndarray:
        """status[j] == 0  <=>  MultiSignature::verify(&MultiPublicKey::from_public_keys(key_sets[j]), msgs[j]).is_ok()
        (multi_signature.rs:127-135); otherwise the reference's error for sum_points then verify."""
        q = len(key_sets)
        koff = np.zeros(q + 1, dtype=np.uint64)
        if q:
            koff[1:] = np.cumsum([len(k) for k in key_sets], dtype=np.uint64)
        pk = _pack_points([k for ks in key_sets for k in ks], pk_len(impl_id), "public key")
        sg = _pack_points(sigs, sig_len(impl_id), "signature")
        if sg.size // sig_len(impl_id) != q or len(msgs) != q:
            raise BlsError(ST_MISMATCHED_LENGTHS)
        data, off = pack_messages(msgs)
        return self.verify_multisig_batch_packed(impl_id, scheme, koff, pk, sg, data, off, fmt)

    def verify_multisig_batch_packed(self, impl_id: int, scheme: int, koff: np.ndarray, pk: np.ndarray, sg: np.ndarray, data: np.ndarray,
                                     off: np.ndarray, fmt: int = SerializationFormat.Modern) -> np.ndarray:
        """Flat-buffer form: koff[q + 1] key offsets, pk koff[q] keys, sg q signatures, the q messages as data / off."""
        koff = np.ascontiguousarray(koff, dtype=np.uint64).reshape(-1)
        q = koff.size - 1
        pk, sg = _pack_points(pk, pk_len(impl_id), "public key"), _pack_points(sg, sig_len(impl_id), "signature")
        if pk.size != (int(koff[-1]) if q else 0) * pk_len(impl_id) or sg.size != q * sig_len(impl_id) or off.size - 1 != q:
            raise BlsError(ST_MISMATCHED_LENGTHS)
        status = np.empty(q, dtype=np.uint8)
        rc = self._lib.blsgpu_verify_multisig_batch(self._ctx, impl_id, scheme, fmt, q, _ptr(koff), _ptr(pk), _ptr(sg), _ptr(data), _ptr(off),
                                                    _ptr(status))
        self._check(rc, "blsgpu_verify_multisig_batch")
        return status

    def verify_multisig_batch_keyed(self, keys: KeySet, scheme: int, key_idx_sets: Sequence[Sequence[int]], sigs, msgs: Sequence[bytes],
                                    fmt: int = SerializationFormat.Modern) -> np.ndarray:
        """verify_multisig_batch with set j's keys = keys of `keys` at key_idx_sets[j] (fmt is the signatures' format)."""
        q = len(key_idx_sets)
        koff = np.zeros(q + 1, dtype=np.uint64)
        if q:
            koff[1:] = np.cumsum([len(k) for k in key_idx_sets], dtype=np.uint64)
        idx = np.array([k for ks in key_idx_sets for k in ks], dtype=np.uint32)
        sg = _pack_points(sigs, sig_len(keys.impl_id), "signature")
        if sg.size // sig_len(keys.impl_id) != q or len(msgs) != q:
            raise BlsError(ST_MISMATCHED_LENGTHS)
        data, off = pack_messages(msgs)
        return self.verify_multisig_batch_keyed_packed(keys, scheme, koff, idx, sg, data, off, fmt)

    def verify_multisig_batch_keyed_packed(self, keys: KeySet, scheme: int, koff: np.ndarray, key_idx: np.ndarray, sg: np.ndarray,
                                           data: np.ndarray, off: np.ndarray, fmt: int = SerializationFormat.Modern) -> np.ndarray:
        """Flat-buffer form: koff[q + 1] member offsets, key_idx uint32[koff[q]], sg q signatures, the q messages as data / off."""
        koff = np.ascontiguousarray(koff, dtype=np.uint64).reshape(-1)
        key_idx = np.ascontiguousarray(key_idx, dtype=np.uint32).reshape(-1)
        q = koff.size - 1
        sg = _pack_points(sg, sig_len(keys.impl_id), "signature")
        if key_idx.size != (int(koff[-1]) if q else 0) or sg.size != q * sig_len(keys.impl_id) or off.size - 1 != q:
            raise BlsError(ST_MISMATCHED_LENGTHS)
        status = np.empty(q, dtype=np.uint8)
        rc = self._lib.blsgpu_verify_multisig_batch_keyed(self._ctx, keys.id, scheme, fmt, q, _ptr(koff), _ptr(key_idx), _ptr(sg), _ptr(data),
                                                          _ptr(off), _ptr(status))
        self._check(rc, "blsgpu_verify_multisig_batch_keyed")
        return status

    def sum_points_batch(self, group: int, point_sets: Sequence[Sequence[bytes]],
                         fmt: int = SerializationFormat.Modern) -> Tuple[np.ndarray, np.ndarray, List[bytes]]:
        """q x sum_points in one call: (status[q], bad_index[q] counted inside each set, q compressed sums; zeroed where a
        set fails)."""
        q = len(point_sets)
        length = 48 if group == 1 else 96
        soff = np.zeros(q + 1, dtype=np.uint64)
        if q:
            soff[1:] = np.cumsum([len(s) for s in point_sets], dtype=np.uint64)
        pts = _pack_points([p for ps in point_sets for p in ps], length, "point")
        status, bad, out = self.sum_points_batch_packed(group, soff, pts, fmt)
        return status, bad, [out[j * length:(j + 1) * length].tobytes() for j in range(q)]

    def sum_points_batch_packed(self, group: int, set_off: np.ndarray, pts: np.ndarray,
                                fmt: int = SerializationFormat.Modern) -> Tuple[np.ndarray, np.ndarray, np.ndarray]:
        """Flat-buffer form: set_off[q + 1] point offsets, pts set_off[q] points; returns (status, bad_index, q sums flat)."""
        length = 48 if group == 1 else 96
        set_off = np.ascontiguousarray(set_off, dtype=np.uint64).reshape(-1)
        q = set_off.size - 1
        pts = _pack_points(pts, length, "point")
        if pts.size != (int(set_off[-1]) if q else 0) * length:
            raise BlsError(ST_MISMATCHED_LENGTHS)
        out = np.zeros(q * length, dtype=np.uint8)
        status = np.empty(q, dtype=np.uint8)
        bad = np.full(q, -1, dtype=np.int64)
        rc = self._lib.blsgpu_sum_points_batch(self._ctx, group, fmt, q, _ptr(set_off), _ptr(pts), _ptr(out), _ptr(status), _ptr(bad))
        self._check(rc, "blsgpu_sum_points_batch")
        return status, bad, out

    def recode_points_packed(self, group: int, pts: np.ndarray, fmt_in: int, fmt_out: int) -> np.ndarray:
        L = 48 if group == 1 else 96
        n = pts.size // L
        out = np.zeros(n * L, dtype=np.uint8)
        status = np.empty(n, dtype=np.uint8)
        self._check(self._lib.blsgpu_recode_points(self._ctx, group, fmt_in, fmt_out, n, _ptr(pts), _ptr(out), _ptr(status)), "blsgpu_recode_points")
        if n and int(status.max()) != 0:
            raise BlsError(int(status.max()), "recode_points_packed")
        return out

    def aggregate_secure_batch(self, impl_id: int, key_sets: Sequence[Sequence[bytes]], sig_sets: Sequence[Sequence[bytes]],
                               fmt: int = SerializationFormat.Modern) -> Tuple[np.ndarray, List[bytes]]:
        q = len(key_sets)
        status_pre = np.zeros(q, dtype=np.uint8)
        for j in range(q):
            if len(key_sets[j]) != len(sig_sets[j]):
                status_pre[j] = ST_MISMATCHED_LENGTHS
        if status_pre.any():
            raise BlsError(ST_MISMATCHED_LENGTHS)
        koff = np.zeros(q + 1, dtype=np.uint64)
        if q:
            koff[1:] = np.cumsum([len(k) for k in key_sets], dtype=np.uint64)
        pk = _pack_points([k for ks in key_sets for k in ks], pk_len(impl_id), "public key")
        sg = _pack_points([s for ss in sig_sets for s in ss], sig_len(impl_id), "signature")
        out = np.zeros(q * sig_len(impl_id), dtype=np.uint8)
        status = np.empty(q, dtype=np.uint8)
        rc = self._lib.blsgpu_aggregate_secure_batch(self._ctx, impl_id, fmt, q, _ptr(koff), _ptr(pk), _ptr(sg), _ptr(out),
                                                     _ptr(status))
        self._check(rc, "blsgpu_aggregate_secure_batch")
        L = sig_len(impl_id)
        return status, [out[j * L:(j + 1) * L].tobytes() for j in range(q)]

    # ---- building blocks ------------------------------------------------------------------------------------------------
    def hash_to_curve_batch(self, group: int, msgs: Sequence[bytes], dst: bytes) -> List[bytes]:
        data, off = pack_messages(msgs)
        n = len(msgs)
        L = 48 if group == 1 else 96
        out = np.zeros(n * L, dtype=np.uint8)
        d = _u8(dst)
        rc = self._lib.blsgpu_hash_to_curve_batch(self._ctx, group, n, _ptr(data), _ptr(off), _ptr(d), len(dst), _ptr(out))
        self._check(rc, "blsgpu_hash_to_curve_batch")
        return [out[i * L:(i + 1) * L].tobytes() for i in range(n)]

    def recode_points(self, group: int, points, fmt_in: int, fmt_out: int) -> Tuple[np.ndarray, List[bytes]]:
        L = 48 if group == 1 else 96
        pts = _pack_points(points, L, "point")
        n = pts.size // L
        out = np.zeros(n * L, dtype=np.uint8)
        status = np.empty(n, dtype=np.uint8)
        rc = self._lib.blsgpu_recode_points(self._ctx, group, fmt_in, fmt_out, n, _ptr(pts), _ptr(out), _ptr(status))
        self._check(rc, "blsgpu_recode_points")
        return status, [out[i * L:(i + 1) * L].tobytes() for i in range(n)]

    def fp_mul_batch(self, a: np.ndarray, b: np.ndarray, variant: int = 0) -> np.ndarray:
        a, b = _u8(a), _u8(b)
        n = a.size // 48
        out = np.zeros(n * 48, dtype=np.uint8)
        self._check(self._lib.blsgpu_fp_mul_batch(self._ctx, variant, n, _ptr(a), _ptr(b), _ptr(out)), "blsgpu_fp_mul_batch")
        return out

    def pairing_product_is_one(self, g1_points, g2_points) -> bool:
        a = _pack_points(g1_points, 48, "G1 point")
        b = _pack_points(g2_points, 96, "G2 point")
        n = a.size // 48
        res = ctypes.c_int(0)
        self._check(self._lib.blsgpu_pairing_product_is_one(self._ctx, n, _ptr(a), _ptr(b), ctypes.byref(res)),
                    "blsgpu_pairing_product_is_one")
        return bool(res.value)

    def verify_batch_wire(self, impl_id: int, pks, tagged_sigs: Sequence[bytes], msgs: Sequence[bytes]) -> np.ndarray:
        """Signature::try_from(&[u8]) + verify for serde_bare signatures (tag byte + point, signature.rs:112-126,285-286)."""
        pk = _pack_points(pks, pk_len(impl_id), "public key")
        n = pk.size // pk_len(impl_id)
        rec = sig_len(impl_id) + 1
        for t in tagged_sigs:
            if len(t) != rec:
                raise BlsError(ST_DESERIALIZE, "invalid byte sequence")
        if len(tagged_sigs) != n or len(msgs) != n:
            raise BlsError(ST_MISMATCHED_LENGTHS)
        sg = np.frombuffer(b"".join(tagged_sigs), dtype=np.uint8) if n else np.zeros(0, dtype=np.uint8)
        data, off = pack_messages(msgs)
        status = np.zeros(n, dtype=np.uint8)
        rc = self._lib.blsgpu_verify_batch_wire(self._ctx, impl_id, n, _ptr(pk), _ptr(sg), _ptr(data), _ptr(off), _ptr(status))
        self._check(rc, "blsgpu_verify_batch_wire")
        return status

    def pairing_check_batch(self, pair_sets: Sequence[Sequence[Tuple[bytes, bytes]]]) -> Tuple[np.ndarray, np.ndarray]:
        """For every set of (G1 bytes, G2 bytes) pairs: prod e(.,.) == 1 ?  (pairings.rs:50; sign_crypt.rs:69-77,192-207)."""
        q = len(pair_sets)
        off = np.zeros(q + 1, dtype=np.uint64)
        if q:
            off[1:] = np.cumsum([len(s) for s in pair_sets], dtype=np.uint64)
        g1 = _pack_points([p[0] for s in pair_sets for p in s], 48, "G1 point")
        g2 = _pack_points([p[1] for s in pair_sets for p in s], 96, "G2 point")
        ok = np.zeros(q, dtype=np.uint8)
        status = np.zeros(q, dtype=np.uint8)
        rc = self._lib.blsgpu_pairing_check_batch(self._ctx, q, _ptr(off), _ptr(g1), _ptr(g2), _ptr(ok), _ptr(status))
        self._check(rc, "blsgpu_pairing_check_batch")
        return ok, status

    # ---- the other public 2-pairing checks (SURVEY 8f-4) ------------------------------------------------------------
    def signcrypt_valid_batch(self, impl_id: int, scheme: int, us, ws, vs: Sequence[bytes]) -> Tuple[np.ndarray, np.ndarray]:
        """n x SignCryptCiphertext::is_valid (sign_crypt_ciphertext.rs:86-101): returns (valid[n], parse status[n])."""
        u = _pack_points(us, pk_len(impl_id), "U")
        w = _pack_points(ws, sig_len(impl_id), "W")
        n = u.size // pk_len(impl_id)
        if w.size // sig_len(impl_id) != n or len(vs) != n:
            raise BlsError(ST_MISMATCHED_LENGTHS)
        data, off = pack_messages(vs)
        ok, st = np.zeros(n, dtype=np.uint8), np.zeros(n, dtype=np.uint8)
        rc = self._lib.blsgpu_signcrypt_valid_batch(self._ctx, impl_id, scheme, n, _ptr(u), _ptr(w), _ptr(data), _ptr(off), _ptr(ok), _ptr(st))
        self._check(rc, "blsgpu_signcrypt_valid_batch")
        return ok, st

    def signcrypt_verify_share_batch(self, impl_id: int, scheme: int, shares, pk_shares, us, ws, vs: Sequence[bytes]):
        """n x SignDecryptionShare::verify (sign_decryption_share.rs:45-61; the reference passes scheme = Basic)."""
        L = pk_len(impl_id)
        sh, pk, u = (_pack_points(x, L, "share") for x in (shares, pk_shares, us))
        w = _pack_points(ws, sig_len(impl_id), "W")
        n = sh.size // L
        if pk.size // L != n or u.size // L != n or w.size // sig_len(impl_id) != n or len(vs) != n:
            raise BlsError(ST_MISMATCHED_LENGTHS)
        data, off = pack_messages(vs)
        ok, st = np.zeros(n, dtype=np.uint8), np.zeros(n, dtype=np.uint8)
        rc = self._lib.blsgpu_signcrypt_verify_share_batch(self._ctx, impl_id, scheme, n, _ptr(sh), _ptr(pk), _ptr(u), _ptr(w), _ptr(data),
                                                           _ptr(off), _ptr(ok), _ptr(st))
        self._check(rc, "blsgpu_signcrypt_verify_share_batch")
        return ok, st

    def pok_verify_batch(self, impl_id: int, scheme: int, commitments, proofs, pks, ys: Sequence[bytes], msgs: Sequence[bytes]) -> np.ndarray:
        """n x ProofOfKnowledge::verify (proof_of_knowledge.rs:132-165); ys: 32-byte big-endian challenge scalars."""
        cm = _pack_points(commitments, sig_len(impl_id), "commitment")
        pr = _pack_points(proofs, sig_len(impl_id), "proof")
        pk = _pack_points(pks, pk_len(impl_id), "public key")
        n = pk.size // pk_len(impl_id)
        if cm.size // sig_len(impl_id) != n or pr.size // sig_len(impl_id) != n or len(ys) != n or len(msgs) != n:
            raise BlsError(ST_MISMATCHED_LENGTHS)
        for y in ys:
            if len(y) != 32:
                raise BlsError(ST_INVALID_LENGTH, "challenge scalar")
        yb = np.frombuffer(b"".join(ys), dtype=np.uint8) if n else np.zeros(0, dtype=np.uint8)
        data, off = pack_messages(msgs)
        st = np.zeros(n, dtype=np.uint8)
        rc = self._lib.blsgpu_pok_verify_batch(self._ctx, impl_id, scheme, n, _ptr(cm), _ptr(pr), _ptr(pk), _ptr(yb), _ptr(data), _ptr(off), _ptr(st))
        self._check(rc, "blsgpu_pok_verify_batch")
        return st

    def verify_batch_records(self, impl_id: int, fmt: int, scheme_or_tagged: int, pk_records: Sequence[bytes],
                             sig_records: Sequence[bytes], msgs: Sequence[bytes]) -> np.ndarray:
        """Ragged network records (any lengths): PublicKey::from_bytes_with_mode + Signature::from_bytes_with_mode (scheme >= 0)
        or Signature::try_from on the serde_bare form (scheme_or_tagged < 0), then verify.  Length / tag / header errors
        come back as per-item statuses."""
        n = len(pk_records)
        if len(sig_records) != n or len(msgs) != n:
            raise BlsError(ST_MISMATCHED_LENGTHS)
        pk, pko = pack_messages(pk_records)
        sg, sgo = pack_messages(sig_records)
        data, off = pack_messages(msgs)
        st = np.zeros(n, dtype=np.uint8)
        rc = self._lib.blsgpu_verify_batch_records(self._ctx, impl_id, fmt, scheme_or_tagged, n, _ptr(pk), _ptr(pko), _ptr(sg), _ptr(sgo),
                                                   _ptr(data), _ptr(off), _ptr(st))
        self._check(rc, "blsgpu_verify_batch_records")
        return st

    # ---- threshold shares ------------------------------------------------------------------------------------------
    def combine_shares_batch(self, group: int, share_sets: Sequence[Sequence[bytes]]) -> Tuple[np.ndarray, List[bytes]]:
        """Signature::from_shares / PublicKey::from_shares for many share sets (signature.rs:151-165, sig_core.rs:92-105).
        A share is the reference's raw form: 32-byte big-endian identifier || compressed point (lib.rs:117-157)."""
        length = 48 if group == 1 else 96
        q = len(share_sets)
        off = np.zeros(q + 1, dtype=np.uint64)
        if q:
            off[1:] = np.cumsum([len(s) for s in share_sets], dtype=np.uint64)
        flat = [sh for ss in share_sets for sh in ss]
        for sh in flat:
            if len(sh) != 32 + length:
                raise BlsError(ST_DESERIALIZE, "Invalid length for share")  # lib.rs:121-125
        data = np.frombuffer(b"".join(flat), dtype=np.uint8) if flat else np.zeros(0, dtype=np.uint8)
        out = np.zeros(q * length, dtype=np.uint8)
        status = np.zeros(q, dtype=np.uint8)
        rc = self._lib.blsgpu_combine_shares_batch(self._ctx, group, q, _ptr(off), _ptr(data), _ptr(out), _ptr(status))
        self._check(rc, "blsgpu_combine_shares_batch")
        return status, [out[j * length:(j + 1) * length].tobytes() for j in range(q)]

    def verify_share_batch(self, impl_id: int, scheme: int, pk_shares: Sequence[bytes], sig_shares: Sequence[bytes],
                           msgs: Sequence[bytes]) -> np.ndarray:
        """n x PublicKeyShare::verify / SignatureShare::verify (public_key_share.rs:55-71, signature_share.rs:98-101) on raw
        share records: 32-byte big-endian identifier || compressed point (lib.rs:117-157).  Returns BLSGPU_ST_* per item."""
        n = len(pk_shares)
        if len(sig_shares) != n or len(msgs) != n:
            raise BlsError(ST_MISMATCHED_LENGTHS)
        for sh, ln in [(s, 32 + pk_len(impl_id)) for s in pk_shares] + [(s, 32 + sig_len(impl_id)) for s in sig_shares]:
            if len(sh) != ln:
                raise BlsError(ST_DESERIALIZE, "Invalid length for share")  # lib.rs:121-125
        pk = np.frombuffer(b"".join(pk_shares), dtype=np.uint8) if n else np.zeros(0, dtype=np.uint8)
        sg = np.frombuffer(b"".join(sig_shares), dtype=np.uint8) if n else np.zeros(0, dtype=np.uint8)
        data, off = pack_messages(msgs)
        status = np.zeros(n, dtype=np.uint8)
        rc = self._lib.blsgpu_verify_share_batch(self._ctx, impl_id, scheme, n, _ptr(pk), _ptr(sg), _ptr(data), _ptr(off),
                                                 _ptr(status))
        self._check(rc, "blsgpu_verify_share_batch")
        return status

    def testdata_sign(self, impl_id: int, scheme: int, scalars: np.ndarray, msgs_data: np.ndarray, msg_off: np.ndarray):
        """Synthetic data only (see include/blsgpu.h): returns (pks, sigs) flat uint8 arrays."""
        n = msg_off.size - 1
        k = _u8(scalars)
        pks = np.zeros(n * pk_len(impl_id), dtype=np.uint8)
        sigs = np.zeros(n * sig_len(impl_id), dtype=np.uint8)
        rc = self._lib.blsgpu_testdata_sign(self._ctx, impl_id, scheme, n, _ptr(k), _ptr(msgs_data), _ptr(msg_off), _ptr(pks),
                                            _ptr(sigs))
        self._check(rc, "blsgpu_testdata_sign")
        return pks, sigs

    def selftest(self) -> None:
        """Known-answer self-test of the device code (also run automatically at the first context creation)."""
        self._check(self._lib.blsgpu_selftest(self._ctx), "blsgpu_selftest")

    def imad_peak(self) -> float:
        v = ctypes.c_double(0)
        self._check(self._lib.blsgpu_imad_peak(self._ctx, ctypes.byref(v)), "blsgpu_imad_peak")
        return v.value

    def last_stage_ms(self) -> dict:
        arr = (ctypes.c_float * len(STAGES))()
        self._check(self._lib.blsgpu_last_stage_ms(self._ctx, arr), "blsgpu_last_stage_ms")
        return {name: float(arr[i]) for i, name in enumerate(STAGES)}

    def last_kernel_ms(self) -> dict:
        """{kernel: (total ms, launches)} of the hot kernels of the last verify call (CUDA events on their own streams)."""
        ms = (ctypes.c_float * len(KERNELS))()
        cnt = (ctypes.c_int * len(KERNELS))()
        self._check(self._lib.blsgpu_last_kernel_ms(self._ctx, ms, cnt), "blsgpu_last_kernel_ms")
        return {name: (float(ms[i]), int(cnt[i])) for i, name in enumerate(KERNELS)}

    def launch_count(self) -> int:
        return int(self._lib.blsgpu_launch_count(self._ctx))
