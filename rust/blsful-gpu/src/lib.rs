//! Slice-taking verification and public-data aggregation for blsful types, executed by the B200 engine
//! (`libblsgpu.so`, C ABI in `include/blsgpu.h`).
//!
//! Every function here has the result of the blsful call it stands for, item by item:
//!
//! | here | n × (or q ×) the blsful call |
//! |---|---|
//! | [`Engine::verify_batch`] | `Signature::verify` (src/signature.rs:130-138) |
//! | [`Engine::verify_batch_keyed`] / [`Engine::verify_batch_grouped_keyed`] | `Signature::verify` against keys decoded once into a [`KeySet`] |
//! | [`Engine::verify_secure_batch_keyed_with_mode`] / [`Engine::aggregate_secure_batch_keyed_with_mode`] | `verify_secure_with_mode` / `aggregate_secure_with_mode` over quorum members named by index into a [`KeySet`] |
//! | [`Engine::pop_verify_batch`] | `ProofOfPossession::verify` (src/proof_of_possession.rs:77-81) |
//! | [`Engine::aggregate_verify`] | `AggregateSignature::verify` (src/aggregate_signature.rs:230-239) |
//! | [`Engine::aggregate_verify_batch`] | q × `AggregateSignature::verify`, one pipeline per signature scheme present |
//! | [`Engine::aggregate_signature_from`] / [`Engine::multi_signature_from`] / [`Engine::multi_public_key_from`] | `from_signatures` / `from_public_keys` (aggregate_signature.rs:171-188, multi_signature.rs:147-150, multi_public_key.rs:79-82) |
//! | [`Engine::multi_public_keys_from`] / [`Engine::multi_signatures_from`] | q × `from_public_keys` / `MultiSignature::from_signatures` in one call |
//! | [`Engine::multi_signature_verify_batch_with_mode`] / [`Engine::multi_signature_verify_batch_keyed_with_mode`] | q × `MultiSignature::verify` (multi_signature.rs:127-135) against the sum of each set's keys, given as keys or as indices into a [`KeySet`] |
//! | [`Engine::verify_secure_batch`] / [`Engine::verify_secure_batch_with_mode`] | `Signature::verify_secure[_with_mode]` (signature.rs:177-197, 256-276) |
//! | [`Engine::aggregate_secure_batch`] / [`Engine::aggregate_secure_batch_with_mode`] | `aggregate_secure[_with_mode]` (secure_aggregation.rs:159-169, 338-352) |
//! | [`Engine::signatures_from_shares`] / [`Engine::public_keys_from_shares`] | `Signature::from_shares` / `PublicKey::from_shares` (signature.rs:151-165, public_key.rs:128-143) |
//! | [`Engine::verify_share_batch`] | `PublicKeyShare::verify` / `SignatureShare::verify` (public_key_share.rs:55-71) |
//! | [`Engine::signcrypt_valid_batch`] | `SignCryptCiphertext::is_valid` (sign_crypt_ciphertext.rs:86-102) |
//! | [`Engine::signcrypt_verify_share_batch`] | `SignDecryptionShare::verify` (sign_decryption_share.rs:44-62) |
//! | [`Engine::pok_verify_batch`] | `ProofOfKnowledge::verify` (proof_of_knowledge.rs:132-165) |
//! | [`Engine::verify_batch_records`] | `PublicKey::try_from(&[u8])` + `Signature::try_from(&[u8])` + `verify` on wire records |
//! | [`Engine::miller_partial`] + [`Engine::final_exp_is_one`] + [`Engine::partial_finish`] | one batch of `Signature::verify` split over processes / GPUs |
//!
//! No function takes a secret key: signing and key generation stay on blsful's constant-time CPU path.
//! There is no CPU fallback either - an engine failure is an `Err(EngineError)`, never a silently different code path.
//!
//! blsful is `#![deny(unsafe_code)]`; the `unsafe` needed to cross the C ABI is confined to this crate's private
//! `call` helpers, each of which passes pointers and lengths of slices that outlive the call.

use std::ffi::CStr;
use std::fmt;
use std::marker::PhantomData;
use std::os::raw::c_int;
use std::ptr;

use blsful::inner_types::{Group, GroupEncoding};
use blsful::{
    AggregateSignature, Bls12381G1Impl, Bls12381G2Impl, BlsError, BlsResult, BlsSignatureImpl, MultiPublicKey,
    MultiSignature, Pairing, ProofCommitmentChallenge, ProofOfKnowledge, ProofOfPossession, PublicKey, PublicKeyShare,
    SerializationFormat, SignCryptCiphertext, SignDecryptionShare, Signature, SignatureSchemes, SignatureShare,
};
use blsful_gpu_sys as sys;

/// Failure of the engine itself (bad argument, CUDA error, allocation); per-item outcomes are `BlsResult`s.
#[derive(Debug, Clone)]
pub struct EngineError {
    pub code: i32,
    pub message: String,
}

impl fmt::Display for EngineError {
    fn fmt(&self, f: &mut fmt::Formatter<'_>) -> fmt::Result {
        write!(f, "blsgpu error {}: {}", self.code, self.message)
    }
}

impl std::error::Error for EngineError {}

pub type EngineResult<T> = Result<T, EngineError>;

/// The two implementations of the reference (`src/impls/g1.rs`, `src/impls/g2.rs`) as seen by the engine.
pub trait GpuImpl: BlsSignatureImpl {
    /// `impl_id` of the C ABI: 1 = `Bls12381G1Impl`, 2 = `Bls12381G2Impl` (`src/impls.rs:102-109`).
    const IMPL_ID: c_int;
    /// `group` argument for public-key-group points (1 = G1, 2 = G2).
    const PK_GROUP: c_int;
    /// `group` argument for signature-group points.
    const SIG_GROUP: c_int;
    const PK_BYTES: usize;
    const SIG_BYTES: usize;
}

impl GpuImpl for Bls12381G2Impl {
    const IMPL_ID: c_int = 2;
    const PK_GROUP: c_int = 1;
    const SIG_GROUP: c_int = 2;
    const PK_BYTES: usize = 48;
    const SIG_BYTES: usize = 96;
}

impl GpuImpl for Bls12381G1Impl {
    const IMPL_ID: c_int = 1;
    const PK_GROUP: c_int = 2;
    const SIG_GROUP: c_int = 1;
    const PK_BYTES: usize = 96;
    const SIG_BYTES: usize = 48;
}

fn scheme_id(s: SignatureSchemes) -> c_int {
    match s {
        SignatureSchemes::Basic => 0,
        SignatureSchemes::MessageAugmentation => 1,
        SignatureSchemes::ProofOfPossession => 2,
    }
}

fn format_id(f: SerializationFormat) -> c_int {
    match f {
        SerializationFormat::Legacy => 0,
        SerializationFormat::Modern => 1,
    }
}

fn signature_scheme<C: BlsSignatureImpl>(s: &Signature<C>) -> SignatureSchemes {
    match s {
        Signature::Basic(_) => SignatureSchemes::Basic,
        Signature::MessageAugmentation(_) => SignatureSchemes::MessageAugmentation,
        Signature::ProofOfPossession(_) => SignatureSchemes::ProofOfPossession,
    }
}

fn wrap_signature<C: BlsSignatureImpl>(scheme: SignatureSchemes, p: <C as Pairing>::Signature) -> Signature<C> {
    match scheme {
        SignatureSchemes::Basic => Signature::Basic(p),
        SignatureSchemes::MessageAugmentation => Signature::MessageAugmentation(p),
        SignatureSchemes::ProofOfPossession => Signature::ProofOfPossession(p),
    }
}

/// `BLSGPU_ST_*` -> the `BlsError` the reference returns for the same item (include/blsgpu.h:40-55).
/// `index` is the position the reference names in its message where it names one.
pub fn status_to_result(status: u8, index: Option<(i64, i64)>) -> BlsResult<()> {
    let inputs = |s: &str| Err(BlsError::InvalidInputs(s.to_string()));
    match status {
        sys::BLSGPU_ST_OK => Ok(()),
        sys::BLSGPU_ST_INVALID_SIGNATURE => Err(BlsError::InvalidSignature),
        sys::BLSGPU_ST_SIG_IDENTITY => inputs("signature is the identity point"),
        sys::BLSGPU_ST_PK_IDENTITY => match index {
            Some((i, _)) if i >= 0 => Err(BlsError::InvalidInputs(format!("public key at {} is the identity point", i))),
            _ => inputs("public key is the identity point"),
        },
        sys::BLSGPU_ST_DESERIALIZE => Err(BlsError::DeserializationError("Invalid byte sequence".to_string())),
        sys::BLSGPU_ST_LEGACY_FORMAT => Err(BlsError::LegacyFormatError("invalid legacy point encoding".to_string())),
        sys::BLSGPU_ST_INVALID_LENGTH => Err(BlsError::InvalidLength { expected: 0, actual: 0 }),
        sys::BLSGPU_ST_INVALID_COEFFICIENT => Err(BlsError::InvalidCoefficient),
        sys::BLSGPU_ST_DUPLICATE_MESSAGES => match index {
            Some((a, b)) => Err(BlsError::InvalidInputs(format!("duplicate messages detected at {} and {}", a, b))),
            None => inputs("duplicate messages detected"),
        },
        sys::BLSGPU_ST_SCHEME => Err(BlsError::InvalidSignatureScheme),
        sys::BLSGPU_ST_MISMATCHED_LENGTHS => inputs("Mismatched array lengths"),
        sys::BLSGPU_ST_VSSS => Err(BlsError::VsssError),
        sys::BLSGPU_ST_INVALID_PROOF => Err(BlsError::InvalidProof),
        sys::BLSGPU_ST_COMMITMENT_IDENTITY => inputs("commitment is the identity point"),
        sys::BLSGPU_ST_PROOF_IDENTITY => inputs("proof is the identity point"),
        sys::BLSGPU_ST_ZERO_CHALLENGE => inputs("y is the zero"),
        other => Err(BlsError::InvalidInputs(format!("unknown engine status {}", other))),
    }
}

/// Messages packed the way the C ABI takes them: one byte string + n+1 offsets.
pub struct PackedMessages {
    pub bytes: Vec<u8>,
    pub offsets: Vec<u64>,
}

impl PackedMessages {
    pub fn from_iter<B: AsRef<[u8]>, I: IntoIterator<Item = B>>(msgs: I) -> Self {
        let mut bytes = Vec::new();
        let mut offsets = vec![0u64];
        for m in msgs {
            bytes.extend_from_slice(m.as_ref());
            offsets.push(bytes.len() as u64);
        }
        Self { bytes, offsets }
    }

    pub fn len(&self) -> usize {
        self.offsets.len() - 1
    }

    pub fn is_empty(&self) -> bool {
        self.len() == 0
    }
}

fn pack_points<P: GroupEncoding, I: IntoIterator<Item = P>>(points: I, each: usize) -> Vec<u8> {
    let mut out = Vec::new();
    for p in points {
        let b = p.to_bytes();
        debug_assert_eq!(b.as_ref().len(), each);
        out.extend_from_slice(b.as_ref());
    }
    out
}

fn unpack_point<P: GroupEncoding>(bytes: &[u8]) -> Option<P> {
    let mut repr = P::Repr::default();
    if repr.as_ref().len() != bytes.len() {
        return None;
    }
    repr.as_mut().copy_from_slice(bytes);
    Option::from(P::from_bytes(&repr))
}

/// One slice of a batch processed by [`Engine::miller_partial`]: what travels between processes (672 B for G2Impl).
#[derive(Clone)]
pub struct Partial {
    /// Product of the slice's Miller loops before the final exponentiation: 12 × 48-byte big-endian Fp coefficients.
    pub gt: [u8; 576],
    /// Random-linear-combination sum of the slice's signatures, compressed (signature group).
    pub sig_sum: Vec<u8>,
}

/// Public keys decoded once into device memory of the [`Engine`] that made them ([`Engine::key_set`]), named by index
/// in [`Engine::verify_batch_keyed`], [`Engine::verify_batch_grouped_keyed`] and the keyed secure calls
/// ([`Engine::verify_secure_batch_keyed_with_mode`], [`Engine::aggregate_secure_batch_keyed_with_mode`]).  Only the engine's id of the set is held
/// here: [`Engine::drop_key_set`] frees the memory, and so does dropping the engine.  Used with another engine, or after
/// it was freed, the id is an `EngineError` (`BLSGPU_E_ARG`), never undefined behaviour.
pub struct KeySet<C: GpuImpl> {
    id: u64,
    len: usize,
    _impl: PhantomData<C>,
}

impl<C: GpuImpl> KeySet<C> {
    pub fn len(&self) -> usize {
        self.len
    }

    pub fn is_empty(&self) -> bool {
        self.len == 0
    }
}

/// Member offsets and flat key indices of quorums named by index into a key set.
fn pack_index_sets(sets: &[&[u32]]) -> (Vec<u64>, Vec<u32>) {
    let mut off = vec![0u64];
    let mut idx = Vec::new();
    for set in sets {
        idx.extend_from_slice(set);
        off.push(idx.len() as u64);
    }
    (off, idx)
}

// cumulative offsets of sets of the given sizes (q + 1 entries)
fn set_offsets<I: IntoIterator<Item = usize>>(sizes: I) -> Vec<u64> {
    let mut off = vec![0u64];
    for s in sizes {
        off.push(off[off.len() - 1] + s as u64);
    }
    off
}

/// RAII owner of a `blsgpu_ctx` (one per thread; a context is not thread-safe, different contexts are independent).
pub struct Engine {
    ctx: *mut sys::blsgpu_ctx,
}

// A context may move between threads; it must not be shared (`&mut self` on every call enforces that).
unsafe impl Send for Engine {}

impl Drop for Engine {
    fn drop(&mut self) {
        unsafe { sys::blsgpu_ctx_destroy(self.ctx) }
    }
}

impl Engine {
    /// Context on the given CUDA devices.  With more than one device a batch is split across them and the partial
    /// results are folded on the first (include/blsgpu.h, "contexts").  Runs the known-answer self-test once per
    /// process and device; an engine that fails it refuses to start.
    pub fn new(devices: &[i32]) -> EngineResult<Self> {
        let mut ctx: *mut sys::blsgpu_ctx = ptr::null_mut();
        let rc = unsafe { sys::blsgpu_ctx_create(devices.as_ptr(), devices.len() as c_int, &mut ctx) };
        if rc != sys::BLSGPU_OK || ctx.is_null() {
            return Err(EngineError { code: rc, message: "blsgpu_ctx_create failed (no CUDA device, or self-test failure)".into() });
        }
        Ok(Self { ctx })
    }

    fn check(&self, rc: c_int) -> EngineResult<()> {
        if rc == sys::BLSGPU_OK {
            return Ok(());
        }
        let message = unsafe {
            let p = sys::blsgpu_last_error(self.ctx);
            if p.is_null() { String::new() } else { CStr::from_ptr(p).to_string_lossy().into_owned() }
        };
        Err(EngineError { code: rc, message })
    }

    /// 64 (default) or 128 bits for the scalars of the random linear combination: a batch with a bad signature passes
    /// the combined check with probability 2^-bits, after which the exact per-item checks are skipped.
    pub fn set_rlc_bits(&mut self, bits: u32) -> EngineResult<()> {
        let rc = unsafe { sys::blsgpu_ctx_set_rlc_bits(self.ctx, bits as c_int) };
        self.check(rc)
    }

    /// Pins the 32-byte salt of the random linear combination.  TEST HOOK: the default (fresh OS randomness for every
    /// call) is what makes the combination unpredictable to whoever chose the signatures.
    pub fn set_rlc_salt_for_tests(&mut self, salt: &[u8; 32]) -> EngineResult<()> {
        let rc = unsafe { sys::blsgpu_ctx_set_rlc_salt(self.ctx, salt.as_ptr()) };
        self.check(rc)
    }

    pub fn selftest(&mut self) -> EngineResult<()> {
        let rc = unsafe { sys::blsgpu_selftest(self.ctx) };
        self.check(rc)
    }

    // ---------------------------------------------------------------------------------------------------------
    // Signature::verify over slices
    // ---------------------------------------------------------------------------------------------------------

    /// `sigs[i].verify(&pks[i], msgs[i])` for every i.  All signatures of one call share a scheme (mixed batches go
    /// through [`Engine::verify_batch_records`] or are grouped by the caller); a signature of another scheme gets
    /// `InvalidSignatureScheme`.
    pub fn verify_batch<C: GpuImpl, B: AsRef<[u8]>>(
        &mut self,
        pks: &[PublicKey<C>],
        sigs: &[Signature<C>],
        msgs: &[B],
    ) -> EngineResult<Vec<BlsResult<()>>> {
        self.verify_batch_with_mode(pks, sigs, msgs, SerializationFormat::Modern)
    }

    /// As [`Engine::verify_batch`]; `format` only selects the byte form the points cross the boundary in
    /// (`to_bytes_with_mode`), the outcome is the same.
    pub fn verify_batch_with_mode<C: GpuImpl, B: AsRef<[u8]>>(
        &mut self,
        pks: &[PublicKey<C>],
        sigs: &[Signature<C>],
        msgs: &[B],
        _format: SerializationFormat,
    ) -> EngineResult<Vec<BlsResult<()>>> {
        let n = sigs.len();
        if pks.len() != n || msgs.len() != n {
            return Err(EngineError { code: sys::BLSGPU_E_ARG, message: "verify_batch: slice lengths differ".into() });
        }
        if n == 0 {
            return Ok(Vec::new());
        }
        let scheme = signature_scheme(&sigs[0]);
        let pk_bytes = pack_points(pks.iter().map(|p| p.0), C::PK_BYTES);
        let sig_bytes = pack_points(sigs.iter().map(|s| *s.as_raw_value()), C::SIG_BYTES);
        let packed = PackedMessages::from_iter(msgs.iter());
        let status = self.verify_batch_bytes::<C>(scheme, SerializationFormat::Modern, &pk_bytes, &sig_bytes, &packed)?;
        Ok(status
            .iter()
            .zip(sigs)
            .map(|(&st, s)| if signature_scheme(s) != scheme { Err(BlsError::InvalidSignatureScheme) } else { status_to_result(st, None) })
            .collect())
    }

    /// The zero-copy form: points already serialised (`format` says how), one status byte per item.
    pub fn verify_batch_bytes<C: GpuImpl>(
        &mut self,
        scheme: SignatureSchemes,
        format: SerializationFormat,
        pks: &[u8],
        sigs: &[u8],
        msgs: &PackedMessages,
    ) -> EngineResult<Vec<u8>> {
        let n = msgs.len();
        if pks.len() != n * C::PK_BYTES || sigs.len() != n * C::SIG_BYTES {
            return Err(EngineError { code: sys::BLSGPU_E_ARG, message: "verify_batch_bytes: buffer sizes do not match n".into() });
        }
        let mut status = vec![0u8; n];
        let rc = unsafe {
            sys::blsgpu_verify_batch(self.ctx, C::IMPL_ID, scheme_id(scheme), format_id(format), n, pks.as_ptr(),
                sigs.as_ptr(), msgs.bytes.as_ptr(), msgs.offsets.as_ptr(), status.as_mut_ptr())
        };
        self.check(rc)?;
        Ok(status)
    }

    /// `sigs[i].verify(&pks[i], msgs[msg_idx[i]])` for every i, where many items share a message: each message is
    /// hashed once and the items of one message share their Miller loops.  The results equal [`Engine::verify_batch`]'s
    /// on the same items with their messages written out; the scheme rule is the same (a signature of another scheme
    /// than the first gets `InvalidSignatureScheme`).
    pub fn verify_batch_grouped<C: GpuImpl, B: AsRef<[u8]>>(
        &mut self,
        pks: &[PublicKey<C>],
        sigs: &[Signature<C>],
        msg_idx: &[u32],
        msgs: &[B],
    ) -> EngineResult<Vec<BlsResult<()>>> {
        let n = sigs.len();
        if pks.len() != n || msg_idx.len() != n {
            return Err(EngineError { code: sys::BLSGPU_E_ARG, message: "verify_batch_grouped: slice lengths differ".into() });
        }
        if n == 0 {
            return Ok(Vec::new());
        }
        let scheme = signature_scheme(&sigs[0]);
        let pk_bytes = pack_points(pks.iter().map(|p| p.0), C::PK_BYTES);
        let sig_bytes = pack_points(sigs.iter().map(|s| *s.as_raw_value()), C::SIG_BYTES);
        let packed = PackedMessages::from_iter(msgs.iter());
        let status = self.verify_batch_grouped_bytes::<C>(scheme, SerializationFormat::Modern, &pk_bytes, &sig_bytes, msg_idx, &packed)?;
        Ok(status
            .iter()
            .zip(sigs)
            .map(|(&st, s)| if signature_scheme(s) != scheme { Err(BlsError::InvalidSignatureScheme) } else { status_to_result(st, None) })
            .collect())
    }

    /// The zero-copy form of [`Engine::verify_batch_grouped`]: points already serialised (`format` says how), one status
    /// byte per item.
    pub fn verify_batch_grouped_bytes<C: GpuImpl>(
        &mut self,
        scheme: SignatureSchemes,
        format: SerializationFormat,
        pks: &[u8],
        sigs: &[u8],
        msg_idx: &[u32],
        msgs: &PackedMessages,
    ) -> EngineResult<Vec<u8>> {
        let n = msg_idx.len();
        if pks.len() != n * C::PK_BYTES || sigs.len() != n * C::SIG_BYTES {
            return Err(EngineError { code: sys::BLSGPU_E_ARG, message: "verify_batch_grouped_bytes: buffer sizes do not match n".into() });
        }
        let mut status = vec![0u8; n];
        let rc = unsafe {
            sys::blsgpu_verify_batch_grouped(self.ctx, C::IMPL_ID, scheme_id(scheme), format_id(format), n, pks.as_ptr(), sigs.as_ptr(),
                msg_idx.as_ptr(), msgs.len(), msgs.bytes.as_ptr(), msgs.offsets.as_ptr(), status.as_mut_ptr())
        };
        self.check(rc)?;
        Ok(status)
    }

    // ---------------------------------------------------------------------------------------------------------
    // Key sets: public keys decoded once on the device, verify calls that name them by index
    // ---------------------------------------------------------------------------------------------------------

    /// Decodes and subgroup-checks `pks` once into device memory this engine owns (first device).  For key sets that
    /// barely change between calls (a validator set, a masternode list, the signers of a quorum): the keyed calls then
    /// send a 4-byte index per item instead of the key and skip its decode.
    pub fn key_set<C: GpuImpl>(&mut self, pks: &[PublicKey<C>]) -> EngineResult<KeySet<C>> {
        let bytes = pack_points(pks.iter().map(|p| p.0), C::PK_BYTES);
        Ok(self.key_set_bytes::<C>(SerializationFormat::Modern, &bytes)?.0)
    }

    /// The byte form of [`Engine::key_set`]: keys serialised in `format`, with one status per key (`BLSGPU_ST_OK`,
    /// `DESERIALIZE` or `LEGACY_FORMAT`).  A key that fails to decode stays in the set; items that name it get that status.
    pub fn key_set_bytes<C: GpuImpl>(&mut self, format: SerializationFormat, pks: &[u8]) -> EngineResult<(KeySet<C>, Vec<u8>)> {
        if pks.len() % C::PK_BYTES != 0 {
            return Err(EngineError { code: sys::BLSGPU_E_ARG, message: "key_set_bytes: not a whole number of keys".into() });
        }
        let n = pks.len() / C::PK_BYTES;
        let mut status = vec![0u8; n];
        let mut id = 0u64;
        let rc = unsafe { sys::blsgpu_keyset_create(self.ctx, C::IMPL_ID, format_id(format), n, pks.as_ptr(), status.as_mut_ptr(), &mut id) };
        self.check(rc)?;
        Ok((KeySet { id, len: n, _impl: PhantomData }, status))
    }

    /// Frees the device memory of a key set now (dropping the engine frees every set it still holds).
    pub fn drop_key_set<C: GpuImpl>(&mut self, keys: KeySet<C>) -> EngineResult<()> {
        let rc = unsafe { sys::blsgpu_keyset_destroy(self.ctx, keys.id) };
        self.check(rc)
    }

    /// [`Engine::verify_batch`] with `pks[i]` = key `key_idx[i]` of `keys`.  An index at or past the end of the set is an
    /// `EngineError` (`BLSGPU_E_ARG`), as is a set of another engine.
    pub fn verify_batch_keyed<C: GpuImpl, B: AsRef<[u8]>>(
        &mut self,
        keys: &KeySet<C>,
        key_idx: &[u32],
        sigs: &[Signature<C>],
        msgs: &[B],
    ) -> EngineResult<Vec<BlsResult<()>>> {
        let n = sigs.len();
        if key_idx.len() != n || msgs.len() != n {
            return Err(EngineError { code: sys::BLSGPU_E_ARG, message: "verify_batch_keyed: slice lengths differ".into() });
        }
        if n == 0 {
            return Ok(Vec::new());
        }
        let scheme = signature_scheme(&sigs[0]);
        let sig_bytes = pack_points(sigs.iter().map(|s| *s.as_raw_value()), C::SIG_BYTES);
        let packed = PackedMessages::from_iter(msgs.iter());
        let status = self.verify_batch_keyed_bytes(keys, scheme, SerializationFormat::Modern, key_idx, &sig_bytes, &packed)?;
        Ok(status
            .iter()
            .zip(sigs)
            .map(|(&st, s)| if signature_scheme(s) != scheme { Err(BlsError::InvalidSignatureScheme) } else { status_to_result(st, None) })
            .collect())
    }

    /// The zero-copy form of [`Engine::verify_batch_keyed`]: signatures already serialised in `format`.
    pub fn verify_batch_keyed_bytes<C: GpuImpl>(
        &mut self,
        keys: &KeySet<C>,
        scheme: SignatureSchemes,
        format: SerializationFormat,
        key_idx: &[u32],
        sigs: &[u8],
        msgs: &PackedMessages,
    ) -> EngineResult<Vec<u8>> {
        let n = msgs.len();
        if key_idx.len() != n || sigs.len() != n * C::SIG_BYTES {
            return Err(EngineError { code: sys::BLSGPU_E_ARG, message: "verify_batch_keyed_bytes: buffer sizes do not match n".into() });
        }
        let mut status = vec![0u8; n];
        let rc = unsafe {
            sys::blsgpu_verify_batch_keyed(self.ctx, keys.id, scheme_id(scheme), format_id(format), n, key_idx.as_ptr(), sigs.as_ptr(),
                msgs.bytes.as_ptr(), msgs.offsets.as_ptr(), status.as_mut_ptr())
        };
        self.check(rc)?;
        Ok(status)
    }

    /// [`Engine::verify_batch_grouped`] with `pks[i]` = key `key_idx[i]` of `keys`.
    pub fn verify_batch_grouped_keyed<C: GpuImpl, B: AsRef<[u8]>>(
        &mut self,
        keys: &KeySet<C>,
        key_idx: &[u32],
        sigs: &[Signature<C>],
        msg_idx: &[u32],
        msgs: &[B],
    ) -> EngineResult<Vec<BlsResult<()>>> {
        let n = sigs.len();
        if key_idx.len() != n || msg_idx.len() != n {
            return Err(EngineError { code: sys::BLSGPU_E_ARG, message: "verify_batch_grouped_keyed: slice lengths differ".into() });
        }
        if n == 0 {
            return Ok(Vec::new());
        }
        let scheme = signature_scheme(&sigs[0]);
        let sig_bytes = pack_points(sigs.iter().map(|s| *s.as_raw_value()), C::SIG_BYTES);
        let packed = PackedMessages::from_iter(msgs.iter());
        let status = self.verify_batch_grouped_keyed_bytes(keys, scheme, SerializationFormat::Modern, key_idx, &sig_bytes, msg_idx, &packed)?;
        Ok(status
            .iter()
            .zip(sigs)
            .map(|(&st, s)| if signature_scheme(s) != scheme { Err(BlsError::InvalidSignatureScheme) } else { status_to_result(st, None) })
            .collect())
    }

    /// The zero-copy form of [`Engine::verify_batch_grouped_keyed`]: signatures already serialised in `format`.
    pub fn verify_batch_grouped_keyed_bytes<C: GpuImpl>(
        &mut self,
        keys: &KeySet<C>,
        scheme: SignatureSchemes,
        format: SerializationFormat,
        key_idx: &[u32],
        sigs: &[u8],
        msg_idx: &[u32],
        msgs: &PackedMessages,
    ) -> EngineResult<Vec<u8>> {
        let n = msg_idx.len();
        if key_idx.len() != n || sigs.len() != n * C::SIG_BYTES {
            return Err(EngineError { code: sys::BLSGPU_E_ARG, message: "verify_batch_grouped_keyed_bytes: buffer sizes do not match n".into() });
        }
        let mut status = vec![0u8; n];
        let rc = unsafe {
            sys::blsgpu_verify_batch_grouped_keyed(self.ctx, keys.id, scheme_id(scheme), format_id(format), n, key_idx.as_ptr(), sigs.as_ptr(),
                msg_idx.as_ptr(), msgs.len(), msgs.bytes.as_ptr(), msgs.offsets.as_ptr(), status.as_mut_ptr())
        };
        self.check(rc)?;
        Ok(status)
    }

    /// `pops[i].verify(pks[i])` for every i.
    pub fn pop_verify_batch<C: GpuImpl>(
        &mut self,
        pks: &[PublicKey<C>],
        pops: &[ProofOfPossession<C>],
    ) -> EngineResult<Vec<BlsResult<()>>> {
        let n = pops.len();
        if pks.len() != n {
            return Err(EngineError { code: sys::BLSGPU_E_ARG, message: "pop_verify_batch: slice lengths differ".into() });
        }
        let pk_bytes = pack_points(pks.iter().map(|p| p.0), C::PK_BYTES);
        let pop_bytes = pack_points(pops.iter().map(|p| p.0), C::SIG_BYTES);
        let mut status = vec![0u8; n];
        let rc = unsafe {
            sys::blsgpu_pop_verify_batch(self.ctx, C::IMPL_ID, 1, n, pk_bytes.as_ptr(), pop_bytes.as_ptr(), status.as_mut_ptr())
        };
        self.check(rc)?;
        Ok(status.iter().map(|&s| status_to_result(s, None)).collect())
    }

    // ---------------------------------------------------------------------------------------------------------
    // AggregateSignature / MultiSignature / MultiPublicKey
    // ---------------------------------------------------------------------------------------------------------

    /// `sig.verify(data)`: n distinct-message pairings against one aggregate, with the reference's duplicate-message
    /// rule for the Basic scheme (`src/traits/sig_basic.rs:46-58`).
    pub fn aggregate_verify<C: GpuImpl, B: AsRef<[u8]>>(
        &mut self,
        sig: &AggregateSignature<C>,
        data: &[(PublicKey<C>, B)],
    ) -> EngineResult<BlsResult<()>> {
        let (scheme, point) = match sig {
            AggregateSignature::Basic(p) => (SignatureSchemes::Basic, *p),
            AggregateSignature::MessageAugmentation(p) => (SignatureSchemes::MessageAugmentation, *p),
            AggregateSignature::ProofOfPossession(p) => (SignatureSchemes::ProofOfPossession, *p),
        };
        let pk_bytes = pack_points(data.iter().map(|(p, _)| p.0), C::PK_BYTES);
        let packed = PackedMessages::from_iter(data.iter().map(|(_, m)| m.as_ref()));
        let sig_bytes = point.to_bytes();
        let mut status = 0u8;
        let mut index = [-1i64; 2];
        let rc = unsafe {
            sys::blsgpu_aggregate_verify(self.ctx, C::IMPL_ID, scheme_id(scheme), 1, data.len(), pk_bytes.as_ptr(),
                packed.bytes.as_ptr(), packed.offsets.as_ptr(), sig_bytes.as_ref().as_ptr(), &mut status, index.as_mut_ptr())
        };
        self.check(rc)?;
        Ok(status_to_result(status, Some((index[0], index[1]))))
    }

    /// `items[j].0.verify(items[j].1)` for every j, in input order.  One engine call per signature scheme present (the
    /// C entry point takes one scheme); within a call every aggregate is checked by one pipeline with a single final
    /// exponentiation, and a rejected aggregate is rejected by its own exact equation.
    pub fn aggregate_verify_batch<C: GpuImpl, B: AsRef<[u8]>>(
        &mut self,
        items: &[(AggregateSignature<C>, &[(PublicKey<C>, B)])],
    ) -> EngineResult<Vec<BlsResult<()>>> {
        let parts = |s: &AggregateSignature<C>| match s {
            AggregateSignature::Basic(p) => (SignatureSchemes::Basic, *p),
            AggregateSignature::MessageAugmentation(p) => (SignatureSchemes::MessageAugmentation, *p),
            AggregateSignature::ProofOfPossession(p) => (SignatureSchemes::ProofOfPossession, *p),
        };
        let mut out: Vec<Option<BlsResult<()>>> = (0..items.len()).map(|_| None).collect();
        for scheme in [SignatureSchemes::Basic, SignatureSchemes::MessageAugmentation, SignatureSchemes::ProofOfPossession] {
            let idx: Vec<usize> = (0..items.len()).filter(|&j| parts(&items[j].0).0 == scheme).collect();
            if idx.is_empty() {
                continue;
            }
            let q = idx.len();
            let mut set_off = Vec::with_capacity(q + 1);
            set_off.push(0u64);
            for &j in &idx {
                set_off.push(set_off[set_off.len() - 1] + items[j].1.len() as u64);
            }
            let pk_bytes = pack_points(idx.iter().flat_map(|&j| items[j].1.iter().map(|(p, _)| p.0)), C::PK_BYTES);
            let packed = PackedMessages::from_iter(idx.iter().flat_map(|&j| items[j].1.iter().map(|(_, m)| m.as_ref())));
            let sig_bytes = pack_points(idx.iter().map(|&j| parts(&items[j].0).1), C::SIG_BYTES);
            let mut status = vec![0u8; q];
            let mut index = vec![-1i64; 2 * q];
            let rc = unsafe {
                sys::blsgpu_aggregate_verify_batch(self.ctx, C::IMPL_ID, scheme_id(scheme), 1, q, set_off.as_ptr(), pk_bytes.as_ptr(),
                    packed.bytes.as_ptr(), packed.offsets.as_ptr(), sig_bytes.as_ptr(), status.as_mut_ptr(), index.as_mut_ptr())
            };
            self.check(rc)?;
            for (k, &j) in idx.iter().enumerate() {
                out[j] = Some(status_to_result(status[k], Some((index[2 * k], index[2 * k + 1]))));
            }
        }
        Ok(out.into_iter().map(|r| r.expect("every scheme variant is covered")).collect())
    }

    fn sum_points<P: GroupEncoding>(&mut self, group: c_int, bytes: &[u8], each: usize) -> EngineResult<BlsResult<P>> {
        let mut out = vec![0u8; each];
        let (mut status, mut bad) = (0u8, -1i64);
        let rc = unsafe {
            sys::blsgpu_sum_points(self.ctx, group, 1, bytes.len() / each, bytes.as_ptr(), out.as_mut_ptr(), &mut status, &mut bad)
        };
        self.check(rc)?;
        if status != sys::BLSGPU_ST_OK {
            return Ok(status_to_result(status, Some((bad, -1))).map(|_| unreachable!()));
        }
        Ok(unpack_point::<P>(&out).ok_or_else(|| BlsError::DeserializationError("engine returned an invalid point".into())))
    }

    fn same_scheme_sum<C: GpuImpl>(&mut self, sigs: &[Signature<C>]) -> EngineResult<BlsResult<(SignatureSchemes, <C as Pairing>::Signature)>> {
        // the reference's checks (aggregate_signature.rs:127-139): at least two signatures, all of one scheme
        if sigs.len() < 2 {
            return Ok(Err(BlsError::InvalidSignature));
        }
        let scheme = signature_scheme(&sigs[0]);
        if sigs.iter().any(|s| signature_scheme(s) != scheme) {
            return Ok(Err(BlsError::InvalidSignatureScheme));
        }
        let bytes = pack_points(sigs.iter().map(|s| *s.as_raw_value()), C::SIG_BYTES);
        Ok(self.sum_points::<<C as Pairing>::Signature>(C::SIG_GROUP, &bytes, C::SIG_BYTES)?.map(|p| (scheme, p)))
    }

    /// `AggregateSignature::from_signatures(sigs)`.
    pub fn aggregate_signature_from<C: GpuImpl>(&mut self, sigs: &[Signature<C>]) -> EngineResult<BlsResult<AggregateSignature<C>>> {
        Ok(self.same_scheme_sum(sigs)?.map(|(scheme, p)| match scheme {
            SignatureSchemes::Basic => AggregateSignature::Basic(p),
            SignatureSchemes::MessageAugmentation => AggregateSignature::MessageAugmentation(p),
            SignatureSchemes::ProofOfPossession => AggregateSignature::ProofOfPossession(p),
        }))
    }

    /// `MultiSignature::from_signatures(sigs)`.  The reference refuses MessageAugmentation signatures here
    /// (`src/multi_signature.rs:93-95`: each signer's message is prefixed with its own key, so they cannot share a message).
    pub fn multi_signature_from<C: GpuImpl>(&mut self, sigs: &[Signature<C>]) -> EngineResult<BlsResult<MultiSignature<C>>> {
        if sigs.len() >= 2 && sigs[1..].iter().any(|s| matches!(s, Signature::MessageAugmentation(_))) {
            return Ok(Err(BlsError::InvalidSignatureScheme));
        }
        Ok(self.same_scheme_sum(sigs)?.map(|(scheme, p)| match scheme {
            SignatureSchemes::Basic => MultiSignature::Basic(p),
            SignatureSchemes::MessageAugmentation => MultiSignature::MessageAugmentation(p),
            SignatureSchemes::ProofOfPossession => MultiSignature::ProofOfPossession(p),
        }))
    }

    /// `MultiPublicKey::from_public_keys(keys)`.
    pub fn multi_public_key_from<C: GpuImpl>(&mut self, keys: &[PublicKey<C>]) -> EngineResult<BlsResult<MultiPublicKey<C>>> {
        let bytes = pack_points(keys.iter().map(|p| p.0), C::PK_BYTES);
        Ok(self.sum_points::<<C as Pairing>::PublicKey>(C::PK_GROUP, &bytes, C::PK_BYTES)?.map(MultiPublicKey))
    }

    /// q point sums in one engine call (`blsgpu_sum_points_batch`): set j's result is what `sum_points` gives for it alone.
    fn sum_points_batch<P: GroupEncoding>(&mut self, group: c_int, set_off: &[u64], bytes: &[u8], each: usize) -> EngineResult<Vec<BlsResult<P>>> {
        let q = set_off.len() - 1;
        let mut out = vec![0u8; q * each];
        let mut status = vec![0u8; q];
        let mut bad = vec![-1i64; q];
        let rc = unsafe {
            sys::blsgpu_sum_points_batch(self.ctx, group, 1, q, set_off.as_ptr(), bytes.as_ptr(), out.as_mut_ptr(), status.as_mut_ptr(),
                bad.as_mut_ptr())
        };
        self.check(rc)?;
        Ok((0..q)
            .map(|j| {
                status_to_result(status[j], Some((bad[j], -1)))?;
                unpack_point::<P>(&out[j * each..(j + 1) * each])
                    .ok_or_else(|| BlsError::DeserializationError("engine returned an invalid point".into()))
            })
            .collect())
    }

    /// `MultiPublicKey::from_public_keys(key_sets[j])` for every j, in one engine call.
    pub fn multi_public_keys_from<C: GpuImpl>(&mut self, key_sets: &[&[PublicKey<C>]]) -> EngineResult<Vec<BlsResult<MultiPublicKey<C>>>> {
        let set_off = set_offsets(key_sets.iter().map(|s| s.len()));
        let bytes = pack_points(key_sets.iter().flat_map(|s| s.iter().map(|p| p.0)), C::PK_BYTES);
        Ok(self.sum_points_batch::<<C as Pairing>::PublicKey>(C::PK_GROUP, &set_off, &bytes, C::PK_BYTES)?
            .into_iter()
            .map(|r| r.map(MultiPublicKey))
            .collect())
    }

    /// `MultiSignature::from_signatures(sig_sets[j])` for every j, in one engine call; each set keeps
    /// [`Engine::multi_signature_from`]'s rules (at least two signatures, one scheme, no MessageAugmentation after the first).
    pub fn multi_signatures_from<C: GpuImpl>(&mut self, sig_sets: &[&[Signature<C>]]) -> EngineResult<Vec<BlsResult<MultiSignature<C>>>> {
        let rule = |sigs: &[Signature<C>]| -> BlsResult<SignatureSchemes> {
            if sigs.len() < 2 {
                return Err(BlsError::InvalidSignature);
            }
            let scheme = signature_scheme(&sigs[0]);
            if sigs[1..].iter().any(|s| signature_scheme(s) != scheme || matches!(s, Signature::MessageAugmentation(_))) {
                return Err(BlsError::InvalidSignatureScheme);
            }
            Ok(scheme)
        };
        let decided: Vec<BlsResult<SignatureSchemes>> = sig_sets.iter().map(|s| rule(*s)).collect();
        // a set the rules refuse is sent empty and reported here
        let set_off = set_offsets(sig_sets.iter().zip(&decided).map(|(s, d)| if d.is_ok() { s.len() } else { 0 }));
        let bytes = pack_points(sig_sets.iter().zip(&decided).filter(|(_, d)| d.is_ok()).flat_map(|(s, _)| s.iter().map(|x| *x.as_raw_value())),
            C::SIG_BYTES);
        let sums = self.sum_points_batch::<<C as Pairing>::Signature>(C::SIG_GROUP, &set_off, &bytes, C::SIG_BYTES)?;
        Ok(decided
            .into_iter()
            .zip(sums)
            .map(|(d, s)| {
                let (scheme, p) = (d?, s?);
                Ok(match scheme {
                    SignatureSchemes::Basic => MultiSignature::Basic(p),
                    SignatureSchemes::MessageAugmentation => MultiSignature::MessageAugmentation(p),
                    SignatureSchemes::ProofOfPossession => MultiSignature::ProofOfPossession(p),
                })
            })
            .collect())
    }

    // ---------------------------------------------------------------------------------------------------------
    // multi-signatures over signer subsets: q (MultiSignature, signer set, message) per call
    // ---------------------------------------------------------------------------------------------------------

    /// `sigs[j].verify(&MultiPublicKey::from_public_keys(key_sets[j]), msgs[j])` for every j, in input order
    /// (`src/multi_signature.rs:127-135`).  One engine call per signature scheme present; the key sums are formed on the
    /// device.  `format` is the encoding the points cross the bus in.
    pub fn multi_signature_verify_batch_with_mode<C: GpuImpl, B: AsRef<[u8]>>(
        &mut self,
        sigs: &[MultiSignature<C>],
        key_sets: &[&[PublicKey<C>]],
        msgs: &[B],
        format: SerializationFormat,
    ) -> EngineResult<Vec<BlsResult<()>>> {
        if key_sets.len() != sigs.len() || msgs.len() != sigs.len() {
            return Err(EngineError { code: sys::BLSGPU_E_ARG, message: "multi_signature_verify_batch: slice lengths differ".into() });
        }
        self.multisig_by_scheme(sigs, format, |eng, idx, scheme, sig_bytes, packed, status| {
            let sets: Vec<&[PublicKey<C>]> = idx.iter().map(|&j| key_sets[j]).collect();
            let (key_off, pk_bytes) = eng.pack_key_sets::<C>(&sets, format)?;
            let rc = unsafe {
                sys::blsgpu_verify_multisig_batch(eng.ctx, C::IMPL_ID, scheme_id(scheme), format_id(format), idx.len(), key_off.as_ptr(),
                    pk_bytes.as_ptr(), sig_bytes.as_ptr(), packed.bytes.as_ptr(), packed.offsets.as_ptr(), status.as_mut_ptr())
            };
            eng.check(rc)
        }, msgs)
    }

    /// [`Engine::multi_signature_verify_batch_with_mode`] with set j's keys = the keys of `keys` at `key_idx_sets[j]`.  An
    /// index at or past the end of the set is an `EngineError` (`BLSGPU_E_ARG`), as is a set of another engine.
    pub fn multi_signature_verify_batch_keyed_with_mode<C: GpuImpl, B: AsRef<[u8]>>(
        &mut self,
        keys: &KeySet<C>,
        key_idx_sets: &[&[u32]],
        sigs: &[MultiSignature<C>],
        msgs: &[B],
        format: SerializationFormat,
    ) -> EngineResult<Vec<BlsResult<()>>> {
        if key_idx_sets.len() != sigs.len() || msgs.len() != sigs.len() {
            return Err(EngineError { code: sys::BLSGPU_E_ARG, message: "multi_signature_verify_batch_keyed: slice lengths differ".into() });
        }
        self.multisig_by_scheme(sigs, format, |eng, idx, scheme, sig_bytes, packed, status| {
            let sets: Vec<&[u32]> = idx.iter().map(|&j| key_idx_sets[j]).collect();
            let (key_off, key_idx) = pack_index_sets(&sets);
            let rc = unsafe {
                sys::blsgpu_verify_multisig_batch_keyed(eng.ctx, keys.id, scheme_id(scheme), format_id(format), idx.len(), key_off.as_ptr(),
                    key_idx.as_ptr(), sig_bytes.as_ptr(), packed.bytes.as_ptr(), packed.offsets.as_ptr(), status.as_mut_ptr())
            };
            eng.check(rc)
        }, msgs)
    }

    // the multi-signatures of each scheme present (input positions idx), their signatures in `format` and messages, through
    // call(engine, idx, scheme, signature bytes, messages, statuses); the results in input order
    fn multisig_by_scheme<C: GpuImpl, B: AsRef<[u8]>>(
        &mut self,
        sigs: &[MultiSignature<C>],
        format: SerializationFormat,
        call: impl Fn(&mut Self, &[usize], SignatureSchemes, &[u8], &PackedMessages, &mut [u8]) -> EngineResult<()>,
        msgs: &[B],
    ) -> EngineResult<Vec<BlsResult<()>>> {
        let parts = |s: &MultiSignature<C>| match s {
            MultiSignature::Basic(p) => (SignatureSchemes::Basic, *p),
            MultiSignature::MessageAugmentation(p) => (SignatureSchemes::MessageAugmentation, *p),
            MultiSignature::ProofOfPossession(p) => (SignatureSchemes::ProofOfPossession, *p),
        };
        let mut out: Vec<Option<BlsResult<()>>> = (0..sigs.len()).map(|_| None).collect();
        for scheme in [SignatureSchemes::Basic, SignatureSchemes::MessageAugmentation, SignatureSchemes::ProofOfPossession] {
            let idx: Vec<usize> = (0..sigs.len()).filter(|&j| parts(&sigs[j]).0 == scheme).collect();
            if idx.is_empty() {
                continue;
            }
            let sig_bytes = self.recode::<C>(C::SIG_GROUP, pack_points(idx.iter().map(|&j| parts(&sigs[j]).1), C::SIG_BYTES), C::SIG_BYTES, format)?;
            let packed = PackedMessages::from_iter(idx.iter().map(|&j| msgs[j].as_ref()));
            let mut status = vec![0u8; idx.len()];
            call(self, &idx, scheme, &sig_bytes, &packed, &mut status)?;
            for (k, &j) in idx.iter().enumerate() {
                out[j] = Some(status_to_result(status[k], None));
            }
        }
        Ok(out.into_iter().map(|r| r.expect("every scheme variant is covered")).collect())
    }

    // ---------------------------------------------------------------------------------------------------------
    // secure aggregation (rogue-key resistant): q quorums per call
    // ---------------------------------------------------------------------------------------------------------

    /// `sigs[j].verify_secure(&key_sets[j], msgs[j])` for every quorum j.
    pub fn verify_secure_batch<C: GpuImpl, B: AsRef<[u8]>>(
        &mut self,
        key_sets: &[&[PublicKey<C>]],
        sigs: &[Signature<C>],
        msgs: &[B],
    ) -> EngineResult<Vec<BlsResult<()>>> {
        self.verify_secure_batch_with_mode(key_sets, sigs, msgs, SerializationFormat::Modern)
    }

    /// `sigs[j].verify_secure_with_mode(&key_sets[j], msgs[j], format)`: the coefficients hash the keys in `format`'s
    /// byte form (`src/secure_aggregation.rs:269-335`), so Legacy and Modern accept different aggregates.
    pub fn verify_secure_batch_with_mode<C: GpuImpl, B: AsRef<[u8]>>(
        &mut self,
        key_sets: &[&[PublicKey<C>]],
        sigs: &[Signature<C>],
        msgs: &[B],
        format: SerializationFormat,
    ) -> EngineResult<Vec<BlsResult<()>>> {
        let q = key_sets.len();
        if sigs.len() != q || msgs.len() != q {
            return Err(EngineError { code: sys::BLSGPU_E_ARG, message: "verify_secure_batch: slice lengths differ".into() });
        }
        if q == 0 {
            return Ok(Vec::new());
        }
        let scheme = signature_scheme(&sigs[0]);
        let (key_off, pk_bytes) = self.pack_key_sets::<C>(key_sets, format)?;
        let sig_bytes = self.recode::<C>(C::SIG_GROUP, pack_points(sigs.iter().map(|s| *s.as_raw_value()), C::SIG_BYTES), C::SIG_BYTES, format)?;
        let packed = PackedMessages::from_iter(msgs.iter());
        let mut status = vec![0u8; q];
        let rc = unsafe {
            sys::blsgpu_verify_secure_batch(self.ctx, C::IMPL_ID, scheme_id(scheme), format_id(format), q, key_off.as_ptr(),
                pk_bytes.as_ptr(), sig_bytes.as_ptr(), packed.bytes.as_ptr(), packed.offsets.as_ptr(), status.as_mut_ptr())
        };
        self.check(rc)?;
        Ok(status
            .iter()
            .zip(sigs)
            .map(|(&st, s)| if signature_scheme(s) != scheme { Err(BlsError::InvalidSignatureScheme) } else { status_to_result(st, None) })
            .collect())
    }

    /// `aggregate_secure(&key_sets[j], &sig_sets[j])` for every quorum j.
    pub fn aggregate_secure_batch<C: GpuImpl>(
        &mut self,
        key_sets: &[&[PublicKey<C>]],
        sig_sets: &[&[<C as Pairing>::Signature]],
    ) -> EngineResult<Vec<BlsResult<<C as Pairing>::Signature>>> {
        self.aggregate_secure_batch_with_mode(key_sets, sig_sets, SerializationFormat::Modern)
    }

    /// `aggregate_secure_with_mode(&key_sets[j], &sig_sets[j], format)` for every quorum j.
    pub fn aggregate_secure_batch_with_mode<C: GpuImpl>(
        &mut self,
        key_sets: &[&[PublicKey<C>]],
        sig_sets: &[&[<C as Pairing>::Signature]],
        format: SerializationFormat,
    ) -> EngineResult<Vec<BlsResult<<C as Pairing>::Signature>>> {
        let q = key_sets.len();
        if sig_sets.len() != q {
            return Err(EngineError { code: sys::BLSGPU_E_ARG, message: "aggregate_secure_batch: slice lengths differ".into() });
        }
        // a quorum whose two lists differ in length is the reference's "Mismatched array lengths" (secure_aggregation.rs:125-129);
        // the flat layout of the C ABI cannot express it, so it is decided here and the quorum is sent empty
        let mismatched: Vec<bool> = key_sets.iter().zip(sig_sets).map(|(k, s)| k.len() != s.len()).collect();
        let keys: Vec<&[PublicKey<C>]> = key_sets.iter().zip(&mismatched).map(|(k, &m)| if m { &k[..0] } else { *k }).collect();
        let (key_off, pk_bytes) = self.pack_key_sets::<C>(&keys, format)?;
        let mut member = Vec::new();
        for (s, &m) in sig_sets.iter().zip(&mismatched) {
            if !m {
                member.extend_from_slice(&pack_points(s.iter().copied(), C::SIG_BYTES));
            }
        }
        let member = self.recode::<C>(C::SIG_GROUP, member, C::SIG_BYTES, format)?;
        let mut out = vec![0u8; q * C::SIG_BYTES];
        let mut status = vec![0u8; q];
        let rc = unsafe {
            sys::blsgpu_aggregate_secure_batch(self.ctx, C::IMPL_ID, format_id(format), q, key_off.as_ptr(), pk_bytes.as_ptr(),
                member.as_ptr(), out.as_mut_ptr(), status.as_mut_ptr())
        };
        self.check(rc)?;
        let out = self.recode_back::<C>(C::SIG_GROUP, out, C::SIG_BYTES, format)?;
        Ok((0..q)
            .map(|j| {
                if mismatched[j] {
                    return Err(BlsError::InvalidInputs("Mismatched array lengths".to_string()));
                }
                status_to_result(status[j], None)?;
                unpack_point(&out[j * C::SIG_BYTES..(j + 1) * C::SIG_BYTES])
                    .ok_or_else(|| BlsError::DeserializationError("engine returned an invalid point".into()))
            })
            .collect())
    }

    /// [`Engine::verify_secure_batch_with_mode`] with quorum j's keys = the keys of `keys` at `key_idx_sets[j]`.  The set
    /// may have been made in either format; its keys are hashed in `format`'s byte form.  An index at or past the end of the
    /// set is an `EngineError` (`BLSGPU_E_ARG`), as is a set of another engine.
    pub fn verify_secure_batch_keyed_with_mode<C: GpuImpl, B: AsRef<[u8]>>(
        &mut self,
        keys: &KeySet<C>,
        key_idx_sets: &[&[u32]],
        sigs: &[Signature<C>],
        msgs: &[B],
        format: SerializationFormat,
    ) -> EngineResult<Vec<BlsResult<()>>> {
        let q = key_idx_sets.len();
        if sigs.len() != q || msgs.len() != q {
            return Err(EngineError { code: sys::BLSGPU_E_ARG, message: "verify_secure_batch_keyed: slice lengths differ".into() });
        }
        if q == 0 {
            return Ok(Vec::new());
        }
        let scheme = signature_scheme(&sigs[0]);
        let (key_off, key_idx) = pack_index_sets(key_idx_sets);
        let sig_bytes = self.recode::<C>(C::SIG_GROUP, pack_points(sigs.iter().map(|s| *s.as_raw_value()), C::SIG_BYTES), C::SIG_BYTES, format)?;
        let packed = PackedMessages::from_iter(msgs.iter());
        let mut status = vec![0u8; q];
        let rc = unsafe {
            sys::blsgpu_verify_secure_batch_keyed(self.ctx, keys.id, scheme_id(scheme), format_id(format), q, key_off.as_ptr(),
                key_idx.as_ptr(), sig_bytes.as_ptr(), packed.bytes.as_ptr(), packed.offsets.as_ptr(), status.as_mut_ptr())
        };
        self.check(rc)?;
        Ok(status
            .iter()
            .zip(sigs)
            .map(|(&st, s)| if signature_scheme(s) != scheme { Err(BlsError::InvalidSignatureScheme) } else { status_to_result(st, None) })
            .collect())
    }

    /// [`Engine::aggregate_secure_batch_with_mode`] with quorum j's keys = the keys of `keys` at `key_idx_sets[j]`.
    pub fn aggregate_secure_batch_keyed_with_mode<C: GpuImpl>(
        &mut self,
        keys: &KeySet<C>,
        key_idx_sets: &[&[u32]],
        sig_sets: &[&[<C as Pairing>::Signature]],
        format: SerializationFormat,
    ) -> EngineResult<Vec<BlsResult<<C as Pairing>::Signature>>> {
        let q = key_idx_sets.len();
        if sig_sets.len() != q {
            return Err(EngineError { code: sys::BLSGPU_E_ARG, message: "aggregate_secure_batch_keyed: slice lengths differ".into() });
        }
        // as in aggregate_secure_batch_with_mode: a quorum whose two lists differ in length is sent empty and reported here
        let mismatched: Vec<bool> = key_idx_sets.iter().zip(sig_sets).map(|(k, s)| k.len() != s.len()).collect();
        let sets: Vec<&[u32]> = key_idx_sets.iter().zip(&mismatched).map(|(k, &m)| if m { &k[..0] } else { *k }).collect();
        let (key_off, key_idx) = pack_index_sets(&sets);
        let mut member = Vec::new();
        for (s, &m) in sig_sets.iter().zip(&mismatched) {
            if !m {
                member.extend_from_slice(&pack_points(s.iter().copied(), C::SIG_BYTES));
            }
        }
        let member = self.recode::<C>(C::SIG_GROUP, member, C::SIG_BYTES, format)?;
        let mut out = vec![0u8; q * C::SIG_BYTES];
        let mut status = vec![0u8; q];
        let rc = unsafe {
            sys::blsgpu_aggregate_secure_batch_keyed(self.ctx, keys.id, format_id(format), q, key_off.as_ptr(), key_idx.as_ptr(),
                member.as_ptr(), out.as_mut_ptr(), status.as_mut_ptr())
        };
        self.check(rc)?;
        let out = self.recode_back::<C>(C::SIG_GROUP, out, C::SIG_BYTES, format)?;
        Ok((0..q)
            .map(|j| {
                if mismatched[j] {
                    return Err(BlsError::InvalidInputs("Mismatched array lengths".to_string()));
                }
                status_to_result(status[j], None)?;
                unpack_point(&out[j * C::SIG_BYTES..(j + 1) * C::SIG_BYTES])
                    .ok_or_else(|| BlsError::DeserializationError("engine returned an invalid point".into()))
            })
            .collect())
    }

    fn pack_key_sets<C: GpuImpl>(&mut self, key_sets: &[&[PublicKey<C>]], format: SerializationFormat) -> EngineResult<(Vec<u64>, Vec<u8>)> {
        let mut off = vec![0u64];
        let mut bytes = Vec::new();
        for set in key_sets {
            bytes.extend_from_slice(&pack_points(set.iter().map(|p| p.0), C::PK_BYTES));
            off.push((bytes.len() / C::PK_BYTES) as u64);
        }
        Ok((off, self.recode::<C>(C::PK_GROUP, bytes, C::PK_BYTES, format)?))
    }

    /// Modern bytes (what `GroupEncoding::to_bytes` yields) -> `format`'s bytes, on the device (`to_bytes_with_mode`).
    fn recode<C: GpuImpl>(&mut self, group: c_int, bytes: Vec<u8>, each: usize, format: SerializationFormat) -> EngineResult<Vec<u8>> {
        self.recode_dir(group, bytes, each, 1, format_id(format))
    }

    fn recode_back<C: GpuImpl>(&mut self, group: c_int, bytes: Vec<u8>, each: usize, format: SerializationFormat) -> EngineResult<Vec<u8>> {
        self.recode_dir(group, bytes, each, format_id(format), 1)
    }

    fn recode_dir(&mut self, group: c_int, bytes: Vec<u8>, each: usize, from: c_int, to: c_int) -> EngineResult<Vec<u8>> {
        if from == to || bytes.is_empty() {
            return Ok(bytes);
        }
        let n = bytes.len() / each;
        let mut out = vec![0u8; bytes.len()];
        let mut status = vec![0u8; n];
        let rc = unsafe { sys::blsgpu_recode_points(self.ctx, group, from, to, n, bytes.as_ptr(), out.as_mut_ptr(), status.as_mut_ptr()) };
        self.check(rc)?;
        Ok(out)
    }

    // ---------------------------------------------------------------------------------------------------------
    // threshold shares
    // ---------------------------------------------------------------------------------------------------------

    fn combine<P: GroupEncoding>(&mut self, group: c_int, each: usize, sets: &[Vec<Vec<u8>>]) -> EngineResult<Vec<BlsResult<P>>> {
        let rec = 32 + each;
        let mut off = vec![0u64];
        let mut bytes = Vec::new();
        for set in sets {
            for r in set {
                if r.len() != rec {
                    return Err(EngineError { code: sys::BLSGPU_E_ARG, message: "share record of unexpected length".into() });
                }
                bytes.extend_from_slice(r);
            }
            off.push((bytes.len() / rec) as u64);
        }
        let q = sets.len();
        let mut out = vec![0u8; q * each];
        let mut status = vec![0u8; q];
        let rc = unsafe { sys::blsgpu_combine_shares_batch(self.ctx, group, q, off.as_ptr(), bytes.as_ptr(), out.as_mut_ptr(), status.as_mut_ptr()) };
        self.check(rc)?;
        Ok((0..q)
            .map(|j| {
                status_to_result(status[j], None)?;
                unpack_point(&out[j * each..(j + 1) * each]).ok_or_else(|| BlsError::DeserializationError("engine returned an invalid point".into()))
            })
            .collect())
    }

    /// `Signature::from_shares(&share_sets[j])` for every j: Lagrange interpolation at zero in the signature group.
    pub fn signatures_from_shares<C: GpuImpl>(&mut self, share_sets: &[&[SignatureShare<C>]]) -> EngineResult<Vec<BlsResult<Signature<C>>>>
    where
        for<'a> Vec<u8>: From<&'a <C as Pairing>::SignatureShare>,
    {
        let mut schemes = Vec::with_capacity(share_sets.len());
        let mut sets = Vec::with_capacity(share_sets.len());
        for set in share_sets {
            // the reference rejects mixed schemes before interpolating (signature.rs:152-154); fewer than two shares,
            // a zero or a repeated identifier are vsss-rs errors found by the engine (status VSSS -> BlsError::VsssError)
            let scheme = set.first().map(share_scheme);
            let uniform = set.iter().all(|s| Some(share_scheme(s)) == scheme);
            schemes.push((uniform, scheme));
            sets.push(if uniform { set.iter().map(|s| Vec::<u8>::from(s.as_raw_value())).collect() } else { Vec::new() });
        }
        let combined = self.combine::<<C as Pairing>::Signature>(C::SIG_GROUP, C::SIG_BYTES, &sets)?;
        Ok(combined
            .into_iter()
            .zip(schemes)
            .map(|(r, (uniform, scheme))| match (uniform, scheme) {
                (false, _) => Err(BlsError::InvalidSignatureScheme),
                (true, Some(s)) => r.map(|p| wrap_signature::<C>(s, p)),
                (true, None) => Err(BlsError::VsssError),
            })
            .collect())
    }

    /// `PublicKey::from_shares(&share_sets[j])` for every j.
    pub fn public_keys_from_shares<C: GpuImpl>(&mut self, share_sets: &[&[PublicKeyShare<C>]]) -> EngineResult<Vec<BlsResult<PublicKey<C>>>>
    where
        for<'a> Vec<u8>: From<&'a <C as Pairing>::PublicKeyShare>,
    {
        let sets: Vec<Vec<Vec<u8>>> = share_sets.iter().map(|set| set.iter().map(|s| Vec::<u8>::from(&s.0)).collect()).collect();
        let combined = self.combine::<<C as Pairing>::PublicKey>(C::PK_GROUP, C::PK_BYTES, &sets)?;
        Ok(combined.into_iter().map(|r| r.map(PublicKey)).collect())
    }

    /// `pk_shares[i].verify(&sig_shares[i], msgs[i])` for every i (the share values are checked like a key and a
    /// signature, `src/public_key_share.rs:55-71`).
    pub fn verify_share_batch<C: GpuImpl, B: AsRef<[u8]>>(
        &mut self,
        pk_shares: &[PublicKeyShare<C>],
        sig_shares: &[SignatureShare<C>],
        msgs: &[B],
    ) -> EngineResult<Vec<BlsResult<()>>>
    where
        for<'a> Vec<u8>: From<&'a <C as Pairing>::PublicKeyShare> + From<&'a <C as Pairing>::SignatureShare>,
    {
        let n = sig_shares.len();
        if pk_shares.len() != n || msgs.len() != n {
            return Err(EngineError { code: sys::BLSGPU_E_ARG, message: "verify_share_batch: slice lengths differ".into() });
        }
        if n == 0 {
            return Ok(Vec::new());
        }
        let scheme = share_scheme(&sig_shares[0]);
        let mut pk_bytes = Vec::with_capacity(n * (32 + C::PK_BYTES));
        let mut sig_bytes = Vec::with_capacity(n * (32 + C::SIG_BYTES));
        for (p, s) in pk_shares.iter().zip(sig_shares) {
            pk_bytes.extend_from_slice(&Vec::<u8>::from(&p.0));
            sig_bytes.extend_from_slice(&Vec::<u8>::from(s.as_raw_value()));
        }
        let packed = PackedMessages::from_iter(msgs.iter());
        let mut status = vec![0u8; n];
        let rc = unsafe {
            sys::blsgpu_verify_share_batch(self.ctx, C::IMPL_ID, scheme_id(scheme), n, pk_bytes.as_ptr(), sig_bytes.as_ptr(),
                packed.bytes.as_ptr(), packed.offsets.as_ptr(), status.as_mut_ptr())
        };
        self.check(rc)?;
        Ok(status
            .iter()
            .zip(sig_shares)
            .map(|(&st, s)| if share_scheme(s) != scheme { Err(BlsError::InvalidSignatureScheme) } else { status_to_result(st, None) })
            .collect())
    }

    // ---------------------------------------------------------------------------------------------------------
    // the other public two-pairing checks: sign-crypt validity, decryption shares, proofs of knowledge
    // ---------------------------------------------------------------------------------------------------------

    /// `ciphertexts[i].is_valid()` for every i.  All ciphertexts of one call share a scheme.
    pub fn signcrypt_valid_batch<C: GpuImpl>(&mut self, ciphertexts: &[SignCryptCiphertext<C>]) -> EngineResult<Vec<bool>> {
        let n = ciphertexts.len();
        if n == 0 {
            return Ok(Vec::new());
        }
        let scheme = ciphertexts[0].scheme;
        let u = pack_points(ciphertexts.iter().map(|c| c.u), C::PK_BYTES);
        let w = pack_points(ciphertexts.iter().map(|c| c.w), C::SIG_BYTES);
        let v = PackedMessages::from_iter(ciphertexts.iter().map(|c| &c.v));
        let mut ok = vec![0u8; n];
        let mut status = vec![0u8; n];
        let rc = unsafe {
            sys::blsgpu_signcrypt_valid_batch(self.ctx, C::IMPL_ID, scheme_id(scheme), n, u.as_ptr(), w.as_ptr(), v.bytes.as_ptr(),
                v.offsets.as_ptr(), ok.as_mut_ptr(), status.as_mut_ptr())
        };
        self.check(rc)?;
        Ok(ok.iter().zip(ciphertexts).map(|(&o, c)| o == 1 && c.scheme == scheme).collect())
    }

    /// `shares[i].verify(&pk_shares[i], &ciphertexts[i])` for every i.
    pub fn signcrypt_verify_share_batch<C: GpuImpl>(
        &mut self,
        shares: &[SignDecryptionShare<C>],
        pk_shares: &[PublicKeyShare<C>],
        ciphertexts: &[SignCryptCiphertext<C>],
    ) -> EngineResult<Vec<BlsResult<()>>>
    where
        <C as Pairing>::PublicKeyShare: ShareValue<<C as Pairing>::PublicKey>,
    {
        let n = shares.len();
        if pk_shares.len() != n || ciphertexts.len() != n {
            return Err(EngineError { code: sys::BLSGPU_E_ARG, message: "signcrypt_verify_share_batch: slice lengths differ".into() });
        }
        if n == 0 {
            return Ok(Vec::new());
        }
        let scheme = ciphertexts[0].scheme;
        let sh = pack_points(shares.iter().map(|s| s.0.point()), C::PK_BYTES);
        let pk = pack_points(pk_shares.iter().map(|s| s.0.point()), C::PK_BYTES);
        let u = pack_points(ciphertexts.iter().map(|c| c.u), C::PK_BYTES);
        let w = pack_points(ciphertexts.iter().map(|c| c.w), C::SIG_BYTES);
        let v = PackedMessages::from_iter(ciphertexts.iter().map(|c| &c.v));
        let mut ok = vec![0u8; n];
        let mut status = vec![0u8; n];
        let rc = unsafe {
            sys::blsgpu_signcrypt_verify_share_batch(self.ctx, C::IMPL_ID, scheme_id(scheme), n, sh.as_ptr(), pk.as_ptr(), u.as_ptr(),
                w.as_ptr(), v.bytes.as_ptr(), v.offsets.as_ptr(), ok.as_mut_ptr(), status.as_mut_ptr())
        };
        self.check(rc)?;
        Ok(ok
            .iter()
            .zip(ciphertexts)
            .map(|(&o, c)| if o == 1 && c.scheme == scheme { Ok(()) } else { Err(BlsError::InvalidDecryptionShare) })
            .collect())
    }

    /// `proofs[i].verify(pks[i], msgs[i], challenges[i])` for every i.  All proofs of one call share a scheme.
    pub fn pok_verify_batch<C: GpuImpl, B: AsRef<[u8]>>(
        &mut self,
        proofs: &[ProofOfKnowledge<C>],
        pks: &[PublicKey<C>],
        msgs: &[B],
        challenges: &[ProofCommitmentChallenge<C>],
    ) -> EngineResult<Vec<BlsResult<()>>> {
        let n = proofs.len();
        if pks.len() != n || msgs.len() != n || challenges.len() != n {
            return Err(EngineError { code: sys::BLSGPU_E_ARG, message: "pok_verify_batch: slice lengths differ".into() });
        }
        if n == 0 {
            return Ok(Vec::new());
        }
        let parts = |p: &ProofOfKnowledge<C>| match p {
            ProofOfKnowledge::Basic { u, v } => (SignatureSchemes::Basic, *u, *v),
            ProofOfKnowledge::MessageAugmentation { u, v } => (SignatureSchemes::MessageAugmentation, *u, *v),
            ProofOfKnowledge::ProofOfPossession { u, v } => (SignatureSchemes::ProofOfPossession, *u, *v),
        };
        let scheme = parts(&proofs[0]).0;
        let commitments = pack_points(proofs.iter().map(|p| parts(p).1), C::SIG_BYTES);
        let responses = pack_points(proofs.iter().map(|p| parts(p).2), C::SIG_BYTES);
        let pk_bytes = pack_points(pks.iter().map(|p| p.0), C::PK_BYTES);
        let mut y = Vec::with_capacity(32 * n);
        for c in challenges {
            y.extend_from_slice(&c.to_be_bytes());
        }
        let packed = PackedMessages::from_iter(msgs.iter());
        let mut status = vec![0u8; n];
        let rc = unsafe {
            sys::blsgpu_pok_verify_batch(self.ctx, C::IMPL_ID, scheme_id(scheme), n, commitments.as_ptr(), responses.as_ptr(),
                pk_bytes.as_ptr(), y.as_ptr(), packed.bytes.as_ptr(), packed.offsets.as_ptr(), status.as_mut_ptr())
        };
        self.check(rc)?;
        Ok(status
            .iter()
            .zip(proofs)
            .map(|(&st, p)| if parts(p).0 != scheme { Err(BlsError::InvalidSignatureScheme) } else { status_to_result(st, None) })
            .collect())
    }

    // ---------------------------------------------------------------------------------------------------------
    // wire front end: ragged records straight from the network
    // ---------------------------------------------------------------------------------------------------------

    /// Records as they arrive: `pk_records[i]` is what `PublicKey::try_from(&[u8])` / `from_bytes_with_mode` takes,
    /// `sig_records[i]` what `Signature::try_from(&[u8])` takes (`scheme = None`: serde_bare, tag byte + point, schemes
    /// may be mixed) or the raw point bytes of `scheme` in `format`.  A record of the wrong length gets `InvalidLength`
    /// with the lengths filled in here (`src/public_key.rs:159-164`); no length can make the call read out of bounds.
    pub fn verify_batch_records<C: GpuImpl, B: AsRef<[u8]>>(
        &mut self,
        format: SerializationFormat,
        scheme: Option<SignatureSchemes>,
        pk_records: &[&[u8]],
        sig_records: &[&[u8]],
        msgs: &[B],
    ) -> EngineResult<Vec<BlsResult<()>>> {
        let n = sig_records.len();
        if pk_records.len() != n || msgs.len() != n {
            return Err(EngineError { code: sys::BLSGPU_E_ARG, message: "verify_batch_records: slice lengths differ".into() });
        }
        let pk = PackedMessages::from_iter(pk_records.iter());
        let sg = PackedMessages::from_iter(sig_records.iter());
        let packed = PackedMessages::from_iter(msgs.iter());
        let mut status = vec![0u8; n];
        let rc = unsafe {
            sys::blsgpu_verify_batch_records(self.ctx, C::IMPL_ID, format_id(format), scheme.map_or(-1, scheme_id), n, pk.bytes.as_ptr(),
                pk.offsets.as_ptr(), sg.bytes.as_ptr(), sg.offsets.as_ptr(), packed.bytes.as_ptr(), packed.offsets.as_ptr(), status.as_mut_ptr())
        };
        self.check(rc)?;
        let sig_len = C::SIG_BYTES + usize::from(scheme.is_none());
        Ok((0..n)
            .map(|i| match status[i] {
                sys::BLSGPU_ST_INVALID_LENGTH if pk_records[i].len() != C::PK_BYTES => {
                    Err(BlsError::InvalidLength { expected: C::PK_BYTES, actual: pk_records[i].len() })
                }
                sys::BLSGPU_ST_INVALID_LENGTH => Err(BlsError::InvalidLength { expected: sig_len, actual: sig_records[i].len() }),
                st => status_to_result(st, None),
            })
            .collect())
    }

    // ---------------------------------------------------------------------------------------------------------
    // one batch over several processes: slice-local partial result -> fold of K partials -> per-item finish
    // ---------------------------------------------------------------------------------------------------------

    /// Step 1, on every process, over its slice of the batch: decode, hash, random linear combination and Miller
    /// loops; NO final exponentiation.  The 576 + SIG_BYTES bytes returned are all that has to be exchanged.
    pub fn miller_partial<C: GpuImpl>(
        &mut self,
        scheme: SignatureSchemes,
        format: SerializationFormat,
        pks: &[u8],
        sigs: &[u8],
        msgs: &PackedMessages,
    ) -> EngineResult<Partial> {
        let n = msgs.len();
        if pks.len() != n * C::PK_BYTES || sigs.len() != n * C::SIG_BYTES {
            return Err(EngineError { code: sys::BLSGPU_E_ARG, message: "miller_partial: buffer sizes do not match n".into() });
        }
        let mut part = Partial { gt: [0u8; 576], sig_sum: vec![0u8; C::SIG_BYTES] };
        let rc = unsafe {
            sys::blsgpu_miller_partial(self.ctx, C::IMPL_ID, scheme_id(scheme), format_id(format), n, pks.as_ptr(), sigs.as_ptr(),
                msgs.bytes.as_ptr(), msgs.offsets.as_ptr(), part.gt.as_mut_ptr(), part.sig_sum.as_mut_ptr())
        };
        self.check(rc)?;
        Ok(part)
    }

    /// Step 2, anywhere (every process after an all-gather, or one coordinator): ONE final exponentiation over the
    /// product of all K partial results (K ≤ 16 per call; fold folds for more).
    pub fn final_exp_is_one<C: GpuImpl>(&mut self, partials: &[Partial]) -> EngineResult<bool> {
        let mut gts = Vec::with_capacity(576 * partials.len());
        let mut sums = Vec::with_capacity(C::SIG_BYTES * partials.len());
        for p in partials {
            gts.extend_from_slice(&p.gt);
            sums.extend_from_slice(&p.sig_sum);
        }
        let mut one: c_int = 0;
        let rc = unsafe { sys::blsgpu_final_exp_is_one(self.ctx, C::IMPL_ID, partials.len(), gts.as_ptr(), sums.as_ptr(), &mut one) };
        self.check(rc)?;
        Ok(one == 1)
    }

    /// Step 3, on every process: the statuses of its own slice.  `batch_ok` = step 2's answer; if false the slice is
    /// searched locally (its own tree of partial products) and only items of THIS slice can come back invalid.
    pub fn partial_finish(&mut self, n: usize, batch_ok: bool) -> EngineResult<Vec<u8>> {
        let mut status = vec![0u8; n];
        let rc = unsafe { sys::blsgpu_partial_finish(self.ctx, c_int::from(batch_ok), status.as_mut_ptr()) };
        self.check(rc)?;
        Ok(status)
    }

    /// Kernel launches issued by this context so far (observability; `blsgpu_launch_count`).
    pub fn launch_count(&self) -> u64 {
        unsafe { sys::blsgpu_launch_count(self.ctx) }
    }

    /// Per-stage device times of the last `verify_batch*` call, milliseconds (`BLSGPU_STAGE_*` order).
    pub fn last_stage_ms(&self) -> [f32; sys::BLSGPU_STAGE_COUNT] {
        let mut ms = [0f32; sys::BLSGPU_STAGE_COUNT];
        unsafe { sys::blsgpu_last_stage_ms(self.ctx, ms.as_mut_ptr()) };
        ms
    }
}

fn share_scheme<C: BlsSignatureImpl>(s: &SignatureShare<C>) -> SignatureSchemes {
    match s {
        SignatureShare::Basic(_) => SignatureSchemes::Basic,
        SignatureShare::MessageAugmentation(_) => SignatureSchemes::MessageAugmentation,
        SignatureShare::ProofOfPossession(_) => SignatureSchemes::ProofOfPossession,
    }
}

/// The group element inside a point share (`InnerPointShareG1/G2`, reference src/lib.rs:75-100: `.0.value.0`).
pub trait ShareValue<P> {
    fn point(&self) -> P;
}

impl ShareValue<blsful::inner_types::G1Projective> for blsful::InnerPointShareG1 {
    fn point(&self) -> blsful::inner_types::G1Projective {
        self.0.value.0
    }
}

impl ShareValue<blsful::inner_types::G2Projective> for blsful::InnerPointShareG2 {
    fn point(&self) -> blsful::inner_types::G2Projective {
        self.0.value.0
    }
}

/// Keeps `Group` in scope for the `is_identity` checks a caller may want next to these functions.
#[allow(dead_code)]
fn _assert_group<G: Group>() {}
