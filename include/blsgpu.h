/* blsgpu.h - C ABI of the B200-native batch BLS12-381 verification engine.
 *
 * Drop-in boundary for the verification hot path of dashpay/agora-blsful (blsful 3.0.0-pre8): these are the entry
 * points a `blsful-gpu-sys` FFI crate binds (see INTEGRATION.md).  Each function cites the reference interface it
 * replaces (file:line under the reference tree).  Only PUBLIC data (public keys, signatures, messages) crosses this
 * boundary; there is no secret-key API.  There is NO CPU fallback: every function fails with BLSGPU_E_CUDA when no
 * usable CUDA device/kernel is available.
 *
 * Conventions
 *   impl_id : 1 = Bls12381G1Impl (sig in G1 48 B, pk in G2 96 B), 2 = Bls12381G2Impl (sig in G2 96 B, pk in G1 48 B)
 *             (same numbering as reference src/impls.rs:102-109)
 *   scheme  : 0 Basic, 1 MessageAugmentation, 2 ProofOfPossession   (reference src/sig_types.rs:8-12)
 *   format  : 0 Legacy (Dash/relic header), 1 Modern (IETF/ZCash)   (reference src/serialization.rs:10-17)
 *             Legacy exists only for impl_id 2 in the reference (src/signature.rs:201-204, src/impls/legacy.rs:85,129);
 *             the engine accepts it for both.
 *   points  : compressed encodings, G1 48 bytes, G2 96 bytes (x.c1 || x.c0), reference src/impls/legacy.rs:19-170
 *   msgs    : all messages concatenated; msg_off[i]..msg_off[i+1] delimits message i (msg_off has n+1 entries)
 *   buffers : caller-allocated, caller-owned, HOST memory unless the name ends in _dev; inputs are read-only
 *   return  : 0 on success or a negative BLSGPU_E_* engine error; per-item outcomes go to status_out (BLSGPU_ST_*),
 *             which reproduce the reference's BlsResult for that item
 *   threads : one call at a time per context; contexts are independent
 *
 * Arguments (every entry point).  A call that breaks these rules returns BLSGPU_E_ARG before any device work (only the
 * decoded contents of blsgpu_pairing_product_is_one and blsgpu_final_exp_is_one are refused later); blsgpu_last_error names
 * the entry point, and the context stays usable.
 *   empty batches : a call over no items (n = 0 or q = 0) returns 0, and the buffers of the items it has not may be NULL.
 *                   The calls with a result even for no items (blsgpu_aggregate_verify, blsgpu_sum_points,
 *                   blsgpu_miller_partial, blsgpu_pairing_product_is_one) still need the buffers of that result, and the
 *                   msg_off of blsgpu_aggregate_verify, blsgpu_hash_to_curve_batch and blsgpu_verify_batch_wire its one entry
 *   offsets       : an offset array has one entry more than it delimits; its entries are non-decreasing and every record
 *                   (a message, a set of members) is below 2^32 bytes or members.  Records are located from off[0] on, so a
 *                   slice of a larger buffer may be passed as is.  Calls that count members in 32 bits (grouped, multi-
 *                   signature, aggregate-batch and key-set calls, secure aggregation) take at most 2^32 - 16 members:
 *                   off[q] - off[0]
 *   null buffers  : a buffer may be NULL only when it holds no bytes: a NULL msgs with messages that span bytes is refused
 *   key sets      : keyed calls name keys by uint32 index into a set of this context (blsgpu_keyset_create); an id this
 *                   context does not hold and an index at or above the set's size are refused
 */
#ifndef BLSGPU_H
#define BLSGPU_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

/* engine errors (function return values) */
#define BLSGPU_OK 0
#define BLSGPU_E_ARG (-1)    /* bad argument (null pointer, unknown impl/scheme/format) */
#define BLSGPU_E_CUDA (-2)   /* CUDA runtime / launch failure, or no device: see blsgpu_last_error */
#define BLSGPU_E_ALLOC (-3)  /* device or host allocation failed */

/* per-item status = the reference's outcome for that item */
#define BLSGPU_ST_OK 0                  /* Ok(()) */
#define BLSGPU_ST_INVALID_SIGNATURE 1   /* BlsError::InvalidSignature            src/traits/sig_core.rs:144,176 */
#define BLSGPU_ST_SIG_IDENTITY 2        /* InvalidInputs("signature is the identity point")   sig_core.rs:126-130,155-159 */
#define BLSGPU_ST_PK_IDENTITY 3         /* InvalidInputs("public key [at i] is the identity point") sig_core.rs:131-135,162-167 */
#define BLSGPU_ST_DESERIALIZE 4         /* DeserializationError / "Invalid byte sequence"  src/impls/legacy.rs:110,121,154,165; src/public_key.rs:73 */
#define BLSGPU_ST_LEGACY_FORMAT 5       /* LegacyFormatError                     src/impls/legacy.rs:53-58 */
#define BLSGPU_ST_INVALID_LENGTH 6      /* InvalidLength (decided by the caller-side binding)  src/public_key.rs:159-164 */
#define BLSGPU_ST_INVALID_COEFFICIENT 7 /* InvalidCoefficient                    src/secure_aggregation.rs:98-100 */
#define BLSGPU_ST_DUPLICATE_MESSAGES 8  /* InvalidInputs("duplicate messages detected at {a} and {b}")  src/traits/sig_basic.rs:51-56 */
#define BLSGPU_ST_SCHEME 9              /* InvalidSignatureScheme / fewer than 2 signatures (binding side) src/aggregate_signature.rs:127-133 */
#define BLSGPU_ST_MISMATCHED_LENGTHS 10 /* InvalidInputs("Mismatched array lengths")  src/secure_aggregation.rs:125-129 */
#define BLSGPU_ST_VSSS 11               /* BlsError::VsssError (fewer than 2 shares, zero or duplicate identifier)  src/error.rs:24-26,60-64 */
#define BLSGPU_ST_INVALID_PROOF 12      /* BlsError::InvalidProof                src/traits/sig_proof.rs:140 */
#define BLSGPU_ST_COMMITMENT_IDENTITY 13 /* InvalidInputs("commitment is the identity point")  sig_proof.rs:110-114 */
#define BLSGPU_ST_PROOF_IDENTITY 14     /* InvalidInputs("proof is the identity point")  sig_proof.rs:115-119 */
#define BLSGPU_ST_ZERO_CHALLENGE 15     /* InvalidInputs("y is the zero")        sig_proof.rs:125-127 */

typedef struct blsgpu_ctx blsgpu_ctx;

/* Create a context on the given CUDA devices (ndev >= 1).  With several devices, blsgpu_verify_batch and
 * blsgpu_pop_verify_batch cut a batch of at least 4096 items per device into contiguous slices, one per device, each
 * driven by its own host thread; the slices' partial results (one Fp12 and one point each) are folded on the first device
 * into a single Miller loop + final exponentiation for the whole batch, and only a device whose slice fails bisects (no
 * collective: 2 x ndev copies of < 1 KB).  Entry points whose units are independent are cut the same way without a fold:
 * blsgpu_sum_points (per-device partial sums of contiguous slices, from 65,536 points per device, then the sum of the partial
 * results) and blsgpu_verify_secure_batch / blsgpu_aggregate_secure_batch (contiguous runs of key sets, balanced by member
 * count); blsgpu_aggregate_verify cuts its pairs over the devices (from 4096 per device) and folds the partial products of
 * Miller values on the first device; blsgpu_aggregate_verify_batch cuts its aggregates into contiguous runs balanced by pair
 * count (from 4096 pairs per device), each verified on its own device without a fold.  Every other entry point (among them
 * blsgpu_verify_batch_grouped, the key sets, the keyed verify calls, the keyed secure calls, blsgpu_verify_multisig_batch[_keyed]
 * and blsgpu_sum_points_batch), the *_dev variants and blsgpu_ctx_set_stream use the first device.  One process per
 * device with blsgpu_miller_partial / blsgpu_final_exp_is_one does the same across processes. */
int blsgpu_ctx_create(const int* devices, int ndev, blsgpu_ctx** out);
void blsgpu_ctx_destroy(blsgpu_ctx* ctx);
/* Text of the last engine error on this context (or of the last failed blsgpu_ctx_create when ctx is NULL). */
const char* blsgpu_last_error(const blsgpu_ctx* ctx);
/* Run the engine on a caller-owned CUDA stream (a cudaStream_t passed as void*; NULL restores the context's own stream).
 * Lets the caller bracket calls with its own CUDA events (bench.py does). */
int blsgpu_ctx_set_stream(blsgpu_ctx* ctx, void* cuda_stream);
/* Random-linear-combination scalars of the batch checks.  r_i = first `bits` bits of SHA-256(digest of the decoded batch ||
 * salt || i).  By DEFAULT the salt is 32 bytes drawn from the OS CSPRNG (getrandom) for EVERY call, so the scalars cannot be
 * predicted or ground offline by whoever chose the batch: a batch holding an invalid signature is accepted with
 * probability <= 2^-bits per call (the statuses themselves do not depend on the salt otherwise).
 * blsgpu_ctx_set_rlc_salt PINS the salt for this context - a determinism hook for tests and reproducible benchmarks only:
 * with a salt known to the adversary the check degrades to a Fiat-Shamir argument with a 2^bits offline work factor.
 * blsgpu_ctx_set_rlc_bits selects 64-bit (default) or 128-bit scalars (r_i * pk_i and the bucket sum cost twice as much). */
int blsgpu_ctx_set_rlc_salt(blsgpu_ctx* ctx, const uint8_t salt[32]);
int blsgpu_ctx_set_rlc_bits(blsgpu_ctx* ctx, int bits);

/* ---- Signature::verify over a slice --------------------------------------------------------------------------
 * Replaces n calls of Signature::<C>::verify(&pk, msg)   (reference src/signature.rs:130-138 ->
 * src/traits/sig_basic.rs:36-38 | sig_aug.rs:20-24 | sig_pop.rs:37-39 -> core_verify src/traits/sig_core.rs:120-146)
 * including the point decoding the reference does at parse time (src/public_key.rs:55-75,158-171,
 * src/signature.rs:231-253, src/impls/legacy.rs:100-169).
 * status_out[i]: decode error of pk i, else decode error of sig i, else SIG_IDENTITY, PK_IDENTITY, then OK or
 * INVALID_SIGNATURE.  Accepts are decided by one random-linear-combination check over the whole batch, rejections by
 * exact per-item checks reached through bisection, so the vector equals the per-signature reference results. */
int blsgpu_verify_batch(blsgpu_ctx* ctx, int impl_id, int scheme, int format, size_t n, const uint8_t* pks,
                        const uint8_t* sigs, const uint8_t* msgs, const uint64_t* msg_off, uint8_t* status_out);
/* Same with every input already resident in device memory of the context's first device (benchmark "value" leg);
 * status_out_dev receives n bytes on the device.  msg_off_dev holds n + 1 non-decreasing offsets with messages shorter
 * than 2^32 bytes (the host entry points check this, here it is the caller's contract); pks_dev / sigs_dev need no
 * particular alignment (16-byte aligned buffers take the vectorised staging path). */
int blsgpu_verify_batch_dev(blsgpu_ctx* ctx, int impl_id, int scheme, int format, size_t n, const uint8_t* pks_dev,
                            const uint8_t* sigs_dev, const uint8_t* msgs_dev, const uint64_t* msg_off_dev,
                            uint8_t* status_out_dev);
/* n x Signature::verify(&pk_i, msg_{msg_idx[i]}) where many items share a message (reference: the same chain as
 * blsgpu_verify_batch).  q messages: message j = msgs[msg_off[j] .. msg_off[j+1]); item i signs message msg_idx[i] < q
 * (items need not be sorted, a message may have any number of items, including none).  status_out[i] is exactly what
 * blsgpu_verify_batch returns for item i with its own copy of the message.  Basic and ProofOfPossession hash each message
 * once and run one Miller loop per run of up to 96 items of one message; MessageAugmentation hashes pk || msg, so it runs
 * blsgpu_verify_batch's pipeline on per-item messages.  msg_idx[i] >= q is BLSGPU_E_ARG.  First device only. */
int blsgpu_verify_batch_grouped(blsgpu_ctx* ctx, int impl_id, int scheme, int format, size_t n, const uint8_t* pks,
                                const uint8_t* sigs, const uint32_t* msg_idx, size_t q, const uint8_t* msgs,
                                const uint64_t* msg_off, uint8_t* status_out);

/* ---- key sets: public keys decoded once, named by index ---------------------------------------------------------------
 * The reference parses and checks a PublicKey<C> once (src/public_key.rs:55-75); the calls above decode every key again
 * on every call.  A key set holds keys that barely change between calls (a validator set, a masternode list, the signers of
 * a quorum) decoded and subgroup-checked once, in device memory the context owns apart from its per-call scratch: 145 bytes
 * per key of impl_id 2 (G1 keys), 273 bytes per key of impl_id 1 (G2 keys).  First device only.
 *
 * Decode n public keys of impl_id (compressed, in `format`) once and keep them on the context's first device.
 * status_out[i] (may be NULL): BLSGPU_ST_OK, DESERIALIZE or LEGACY_FORMAT for key i.  Keys that fail to decode stay in
 * the set, so that items naming them get exactly the status blsgpu_verify_batch gives for those bytes.
 * *keyset_out: a non-zero id, unique in the process (never reused).  n = 0 makes an empty set; at most 2^32 - 16 keys.
 * Synchronises before returning; on BLSGPU_E_ALLOC or BLSGPU_E_CUDA no set is created.  A destroyed set's id is refused like
 * any id this context does not hold.  blsgpu_ctx_destroy frees the sets still alive. */
int blsgpu_keyset_create(blsgpu_ctx* ctx, int impl_id, int format, size_t n, const uint8_t* pks, uint8_t* status_out,
                         uint64_t* keyset_out);
int blsgpu_keyset_destroy(blsgpu_ctx* ctx, uint64_t keyset);
/* Changing a set in place: the set keeps its id and the indices of the keys that did not change, and the work is that of
 * the k changed keys (their decode, and for each live secure view their encoding and a binary search among the set's keys)
 * plus an O(n) pass over 4-byte ranks on the host and their upload.
 *   equivalence : after any sequence of creates, updates and appends, every keyed call returns byte for byte what it returns
 *                 on a set created from the final key bytes (statuses, aggregates and indices, in both formats).  "The bytes
 *                 a key of the set was created from" in the keyed calls below means the bytes it was last given.
 *   format      : each call has its own `format`, as blsgpu_keyset_create; a key's status is the one the format that last
 *                 decoded it gave.  A key that fails to decode stays in the set with that status, as at creation.
 *   refused     : with BLSGPU_E_ARG before any device work, the set unchanged: an id this context does not hold, a NULL pks
 *                 or key_idx with k > 0, a key_idx[i] at or above the set's size, an index named twice in one update (both
 *                 positions are named in blsgpu_last_error), an append past 2^32 - 16 keys.  k = 0 returns 0.
 *   failures    : on BLSGPU_E_ALLOC the set is unchanged (the keys are decoded into scratch, and an append allocates the
 *                 grown set, before anything is written into the set).  A set that meets BLSGPU_E_CUDA can only be destroyed.
 *   secure views: live views are kept current, so that the next keyed secure call does not rebuild them.  The view's memory
 *                 per key is unchanged.
 * Both calls end a pending blsgpu_miller_partial slice, synchronise before returning and run on the first device only.
 *
 * Key key_idx[i] of the set becomes the key decoded from pks[i] (k compressed keys of the set's impl in `format`).
 * status_out[i] (may be NULL): BLSGPU_ST_OK, DESERIALIZE or LEGACY_FORMAT, exactly what blsgpu_keyset_create gives for
 * those bytes. */
int blsgpu_keyset_update(blsgpu_ctx* ctx, uint64_t keyset, int format, size_t k, const uint32_t* key_idx,
                         const uint8_t* pks, uint8_t* status_out);
/* k keys appended: a set of n keys gives them indices n .. n + k - 1 (statuses as blsgpu_keyset_update).  The set's
 * device arrays are reallocated at the exact new size: the old ones are copied device to device, then freed. */
int blsgpu_keyset_append(blsgpu_ctx* ctx, uint64_t keyset, int format, size_t k, const uint8_t* pks, uint8_t* status_out);
/* blsgpu_verify_batch with pks[i] = the bytes key key_idx[i] of the set was created from; `format` is that of sigs only.
 * No key is decoded: the keys are gathered from the set. */
int blsgpu_verify_batch_keyed(blsgpu_ctx* ctx, uint64_t keyset, int scheme, int format, size_t n, const uint32_t* key_idx,
                              const uint8_t* sigs, const uint8_t* msgs, const uint64_t* msg_off, uint8_t* status_out);
/* blsgpu_verify_batch_grouped with pks[i] = the bytes of key key_idx[i] */
int blsgpu_verify_batch_grouped_keyed(blsgpu_ctx* ctx, uint64_t keyset, int scheme, int format, size_t n,
                                      const uint32_t* key_idx, const uint8_t* sigs, const uint32_t* msg_idx, size_t q,
                                      const uint8_t* msgs, const uint64_t* msg_off, uint8_t* status_out);

/* ---- one batch cut over several GPUs / processes (SURVEY.md section 8e) ---------------------------------------------------
 * The random-linear-combination check of a batch factors over slices: every slice folds into ONE partial product of
 * Miller values F_j = prod_i ML(r_i pk_i, H(m_i)) and ONE partial sum S_j = sum_i r_i sig_i; the batch is valid iff
 * prod_j F_j * e(-g, sum_j S_j) == 1 - a single Miller loop and a single final exponentiation for the whole batch
 * (replaces `multi_miller_loop(..).final_exponentiation()`, reference src/helpers.rs:50,62, across devices).
 *   1. every process:  blsgpu_miller_partial on its slice -> gt_out (576 B: the coefficients of w^0..w^5 of F_j, each c0 || c1
 *      as 48-byte big-endian canonical values) and sum_out (S_j as an IETF compressed point of the signature group, 96 | 48 B).
 *      The slice's decode / identity statuses and its product and sum trees stay in the context.
 *   2. any process (or all, redundantly): blsgpu_final_exp_is_one over the k <= 16 gathered partial results.
 *   3. every process:  blsgpu_partial_finish(batch_ok, status_out[n]): if the batch check passed, the statuses are final;
 *      otherwise the slice checks its own partial results and bisects only if they fail too.
 * A context created on several devices does the same inside blsgpu_verify_batch with one host thread per device.
 * Any other call on the context between steps 1 and 3 discards the pending slice. */
int blsgpu_miller_partial(blsgpu_ctx* ctx, int impl_id, int scheme, int format, size_t n, const uint8_t* pks, const uint8_t* sigs,
                          const uint8_t* msgs, const uint64_t* msg_off, uint8_t gt_out[576], uint8_t* sum_out);
int blsgpu_final_exp_is_one(blsgpu_ctx* ctx, int impl_id, size_t k, const uint8_t* partial_gts, const uint8_t* partial_sums,
                            int* is_one_out);
int blsgpu_partial_finish(blsgpu_ctx* ctx, int batch_ok, uint8_t* status_out);

/* ---- ProofOfPossession::verify over a slice:  core_verify(pk, sig, msg = pk.to_bytes(), POP_DST)
 * (reference src/proof_of_possession.rs:77-81, src/traits/sig_pop.rs:61-70) */
int blsgpu_pop_verify_batch(blsgpu_ctx* ctx, int impl_id, int format, size_t n, const uint8_t* pks, const uint8_t* sigs,
                            uint8_t* status_out);

/* ---- AggregateSignature::verify ------------------------------------------------------------------------------
 * Replaces AggregateSignature::<C>::verify(&[(pk, msg)])  (reference src/aggregate_signature.rs:230-239 ->
 * aggregate_verify sig_basic.rs:41-64 | sig_aug.rs:27-38 | sig_pop.rs:52-58 -> core_aggregate_verify
 * sig_core.rs:149-178).  One result in *status_out.  index_out[0..1]: (old, new) positions for DUPLICATE_MESSAGES,
 * (i+1, -1) for PK_IDENTITY exactly as the reference message reports it, (i, -1) for a pk decode error, else -1. */
int blsgpu_aggregate_verify(blsgpu_ctx* ctx, int impl_id, int scheme, int format, size_t n, const uint8_t* pks,
                            const uint8_t* msgs, const uint64_t* msg_off, const uint8_t* sig, uint8_t* status_out,
                            int64_t index_out[2]);
/* q x AggregateSignature::verify (reference src/aggregate_signature.rs:230-239 -> sig_core.rs:149-178, sig_basic.rs:41-64 |
 * sig_aug.rs:27-38 | sig_pop.rs:52-58).  Aggregate j owns pairs set_off[j]..set_off[j+1]-1 of pks / msgs; msg_off holds
 * one message per pair (entries set_off[0] .. set_off[q]);
 * sigs holds q aggregate signatures.  status_out[j] and index_out[2j..2j+1] (index_out may be NULL) mean exactly what
 * blsgpu_aggregate_verify returns for aggregate j alone; indices are positions INSIDE aggregate j.  Duplicate messages
 * (Basic) are looked for within an aggregate only.  One pipeline and one final exponentiation serve the whole call: every
 * pair of aggregate j is weighted by one random scalar r_j, and a failing check is descended to the failing aggregates, each
 * rejected by an exact equation (DESIGN.md section 2). */
int blsgpu_aggregate_verify_batch(blsgpu_ctx* ctx, int impl_id, int scheme, int format, size_t q, const uint64_t* set_off,
                                  const uint8_t* pks, const uint8_t* msgs, const uint64_t* msg_off, const uint8_t* sigs,
                                  uint8_t* status_out, int64_t* index_out);

/* ---- point sums ----------------------------------------------------------------------------------------------
 * Replaces aggregate_signatures / aggregate_public_keys (reference src/traits/sig_core.rs:38-59),
 * BlsMultiSignature::from_signatures (src/traits/sig_multi.rs:7-13), BlsMultiKey::from_public_keys
 * (src/traits/pk_multi.rs:7-13) and the TryFrom<&[Signature]> sums (src/aggregate_signature.rs:123-148,
 * src/multi_signature.rs:80-107).  group: 1 = G1 points (48 B), 2 = G2 points (96 B).  out receives the compressed
 * sum in `format`.  *status_out = OK or the decode error of the first bad element (*bad_index_out). */
int blsgpu_sum_points(blsgpu_ctx* ctx, int group, int format, size_t n, const uint8_t* points, uint8_t* out,
                      uint8_t* status_out, int64_t* bad_index_out);

/* ---- secure aggregation --------------------------------------------------------------------------------------
 * q independent key sets ("quorums"); set j owns public keys key_off[j]..key_off[j+1] of `pks`.
 * verify: replaces Signature::verify_secure[_with_mode] (reference src/signature.rs:177-197,256-276 ->
 * src/secure_aggregation.rs:173-208 with coefficients from :37-106 / :269-335): sort keys by serialized bytes,
 * t_i = BE(SHA256(be32(i) || SHA256(sorted keys))) mod r, check core_verify(sum t_i pk_i, sig_j, msg_j, DST(scheme)).
 * Empty key set: OK iff sig_j is the identity.  status_out[j] per set. */
int blsgpu_verify_secure_batch(blsgpu_ctx* ctx, int impl_id, int scheme, int format, size_t q, const uint64_t* key_off,
                               const uint8_t* pks, const uint8_t* sigs, const uint8_t* msgs, const uint64_t* msg_off,
                               uint8_t* status_out);
/* aggregate: replaces aggregate_secure[_with_mode] (reference src/secure_aggregation.rs:110-169,338-352) and
 * AggregateSignature::from_signatures_secure (src/aggregate_signature.rs:191-227): member_sigs holds one signature per
 * public key (same order as pks); out_sigs receives q aggregated signatures in `format`.  Duplicate keys reuse the
 * signature of the FIRST equal key, as the reference's `position` lookup does (:140-147). */
int blsgpu_aggregate_secure_batch(blsgpu_ctx* ctx, int impl_id, int format, size_t q, const uint64_t* key_off,
                                  const uint8_t* pks, const uint8_t* member_sigs, uint8_t* out_sigs, uint8_t* status_out);

/* Keyed secure aggregation: quorum j's members are key_idx[key_off[j] .. key_off[j+1]), each an index into a key set
 * (blsgpu_keyset_create); impl_id is the set's.  Each call is the unkeyed call above with pks[i] = key key_idx[i] of the
 * set encoded in the call's `format`, as the reference's *_with_mode on already-parsed keys: when `format` is the set's,
 * those are the bytes the set was created from, and every status and output byte equals the unkeyed call's on them.  A set
 * may be used in either format.  A key that failed to decode at creation gives its quorum the status it was created with
 * (the first bad key in member order decides).  No key is decoded, and no member's key bytes cross the bus: the call uploads key_off and key_idx (4 bytes per member) and sorts the quorums on the device.
 * Secure view: the first keyed secure call in a format builds, once per set and format, every key's encoding in that format
 * and its rank in byte order: 52 bytes per key of impl_id 2 and 100 of impl_id 1 on the device, 4 per key on the host.  The
 * build encodes on the device and sorts on the host (once, O(n log n) for n keys); the view lives until the set is
 * destroyed, and blsgpu_keyset_update / blsgpu_keyset_append keep it current.  First device only. */
int blsgpu_verify_secure_batch_keyed(blsgpu_ctx* ctx, uint64_t keyset, int scheme, int format, size_t q,
                                     const uint64_t* key_off, const uint32_t* key_idx, const uint8_t* sigs,
                                     const uint8_t* msgs, const uint64_t* msg_off, uint8_t* status_out);
int blsgpu_aggregate_secure_batch_keyed(blsgpu_ctx* ctx, uint64_t keyset, int format, size_t q, const uint64_t* key_off,
                                        const uint32_t* key_idx, const uint8_t* member_sigs, uint8_t* out_sigs,
                                        uint8_t* status_out);

/* ---- multi-signatures over signer subsets ------------------------------------------------------------------------
 * q x MultiSignature::verify(MultiPublicKey::from_public_keys(keys of set j), msg_j)  (reference src/multi_signature.rs:127-135,
 * src/multi_public_key.rs:79-83, src/traits/pk_multi.rs:7-13 -> core_verify sig_core.rs:120-146).  Set j owns keys
 * key_off[j] .. key_off[j+1]-1 of pks; one signature and one message per set.
 * status_out[j] is exactly blsgpu_sum_points(pk group, format, keys of set j) followed by blsgpu_verify_batch(impl, scheme,
 * format, [that sum], [sig_j], [msg_j]): the first key of the set (in member order) that fails to decode, else the
 * signature's decode error, else SIG_IDENTITY, else PK_IDENTITY when the sum is the identity (an empty set, P and -P, only
 * identity keys), else OK or INVALID_SIGNATURE.  Identity keys add nothing; a key named twice counts twice.
 * MessageAugmentation hashes the compressed multi key || msg.  Both formats for both impls, as blsgpu_verify_batch.
 * The key sums are one segmented sum on the device, balanced by member count (chunks of 16 members of one set, then levels
 * of ranges of 16 partial sums), recorded as BLSGPU_STAGE_DECODE_PK together with the keys' decode; the q (sum, signature,
 * message) triples then take blsgpu_verify_batch's pipeline (one random-linear-combination check, bisection on failure).
 * First device only. */
int blsgpu_verify_multisig_batch(blsgpu_ctx* ctx, int impl_id, int scheme, int format, size_t q, const uint64_t* key_off,
                                 const uint8_t* pks, const uint8_t* sigs, const uint8_t* msgs, const uint64_t* msg_off,
                                 uint8_t* status_out);
/* the same with set j's keys = keys key_idx[key_off[j] .. key_off[j+1]) of a key set; `format` is that of sigs only.  A key
 * that failed to decode at creation gives its set the status it was created with.  No key is decoded: 4 bytes per member cross the bus. */
int blsgpu_verify_multisig_batch_keyed(blsgpu_ctx* ctx, uint64_t keyset, int scheme, int format, size_t q,
                                       const uint64_t* key_off, const uint32_t* key_idx, const uint8_t* sigs,
                                       const uint8_t* msgs, const uint64_t* msg_off, uint8_t* status_out);
/* q x blsgpu_sum_points: set j = points set_off[j] .. set_off[j+1]-1; out: q compressed sums in `format` (zeroed for a
 * failing set); status_out[j] / bad_index_out[j] (may be NULL): what blsgpu_sum_points returns for set j alone, the index
 * counted inside set j.  MultiSignature::from_signatures / MultiPublicKey::from_public_keys / aggregate_signatures for many
 * sets (the binding applies from_signatures' scheme rules).  The same segmented sum as above.  First device only. */
int blsgpu_sum_points_batch(blsgpu_ctx* ctx, int group, int format, size_t q, const uint64_t* set_off, const uint8_t* points,
                            uint8_t* out, uint8_t* status_out, int64_t* bad_index_out);

/* ---- building blocks (parity tests, metrics) ------------------------------------------------------------------ */
/* hash_to_point (reference src/traits/hash_to_point.rs:6-12, src/impls/g2.rs:15-17, src/impls/g1.rs:17-19):
 * out = compressed Modern points, group 2 -> 96 B each (G2Impl signatures), group 1 -> 48 B each. */
int blsgpu_hash_to_curve_batch(blsgpu_ctx* ctx, int group, size_t n, const uint8_t* msgs, const uint64_t* msg_off,
                               const uint8_t* dst, size_t dst_len, uint8_t* out);
/* LegacyG1Point/LegacyG2Point::deserialize + serialize round trip (reference src/traits/legacy_serdes.rs:25-40,
 * src/impls/legacy.rs:85-170): decodes n points given in `format_in` (curve + subgroup check) and re-encodes the
 * accepted ones in `format_out`; status_out[i] = OK / DESERIALIZE / LEGACY_FORMAT. */
int blsgpu_recode_points(blsgpu_ctx* ctx, int group, int format_in, int format_out, size_t n, const uint8_t* in,
                         uint8_t* out, uint8_t* status_out);
/* n Montgomery products of canonical big-endian 48-byte field elements: out = a*b mod p.  variant 0 = the engine's
 * IMAD.WIDE carry-chain multiplier, 1 = plain CIOS cross-check. */
int blsgpu_fp_mul_batch(blsgpu_ctx* ctx, int variant, size_t n, const uint8_t* a, const uint8_t* b, uint8_t* out);
/* Miller loops of n (G1, G2) pairs given as compressed Modern points; *is_one_out = 1 iff the product of the n
 * pairings is the Gt identity (reference src/helpers.rs:41-63 followed by Gt::is_identity). */
int blsgpu_pairing_product_is_one(blsgpu_ctx* ctx, size_t n, const uint8_t* g1_points, const uint8_t* g2_points,
                                  int* is_one_out);
/* Synthetic-data helper for benchmarks and tests (NOT part of the verification path, not a signing API: it takes no
 * secret-key type and is variable-time): out_pk[i] = [k_i] G, out_sig[i] = [k_i] H(msg_i) for 32-byte big-endian
 * scalars k_i, framed for (impl_id, scheme); scheme 3 produces proofs of possession (message = the key's bytes, POP_DST). */
int blsgpu_testdata_sign(blsgpu_ctx* ctx, int impl_id, int scheme, size_t n, const uint8_t* scalars32,
                         const uint8_t* msgs, const uint64_t* msg_off, uint8_t* out_pks, uint8_t* out_sigs);
/* INT32 multiply-issue roofline probe: runs independent mad.wide.u32 chains on every SM and returns the measured
 * 32x32->64 multiply-accumulate rate (MAC/s) of the context's first device. */
int blsgpu_imad_peak(blsgpu_ctx* ctx, double* mac_per_s_out);

/* Wire-format front end (SURVEY.md section 8f-3): the same check as blsgpu_verify_batch for signatures in the reference's
 * serde_bare form, `Vec::<u8>::from(&Signature<C>)` / `Signature::try_from(&[u8])` (src/signature.rs:112-126): one tag
 * byte {0 Basic, 1 MessageAugmentation, 2 ProofOfPossession} followed by the IETF compressed point (49 | 97 bytes,
 * src/signature.rs:285-286).  The scheme of every item comes from its tag (items of different schemes may be mixed);
 * an unknown tag gives BLSGPU_ST_DESERIALIZE (`InvalidInputs(serde error)`).  Public keys are their plain 48 | 96 bytes
 * (the serde_bare form of PublicKey has no tag). */
int blsgpu_verify_batch_wire(blsgpu_ctx* ctx, int impl_id, size_t n, const uint8_t* pks, const uint8_t* tagged_sigs,
                             const uint8_t* msgs, const uint64_t* msg_off, uint8_t* status_out);

/* Batched pairing-product checks (SURVEY.md section 8f-4): for every set j, is  prod_i e(g1[i], g2[i]) == 1  over its
 * pairs?  The building block of the reference's other public 2-pairing checks - `BlsSignCrypt::valid` / `verify_share`
 * (src/traits/sign_crypt.rs:69-77,192-207: pairing(&[(w, -g), (w', u)]).is_identity()) and `ProofOfKnowledge::verify`
 * (src/traits/sig_proof.rs:102-142) - whose hashed points come from blsgpu_hash_to_curve_batch.  Same pairing as
 * `Pairing::pairing` (src/traits/pairings.rs:50, src/helpers.rs:41-63): identity points contribute 1.
 *   pair_off[q+1] : offsets (in pairs) of the sets;  g1_points 48 B, g2_points 96 B each, IETF compressed
 *   ok_out[q]     : 1 / 0;  status_out[q]: BLSGPU_ST_OK or BLSGPU_ST_DESERIALIZE (some point of the set undecodable) */
int blsgpu_pairing_check_batch(blsgpu_ctx* ctx, size_t q, const uint64_t* pair_off, const uint8_t* g1_points,
                               const uint8_t* g2_points, uint8_t* ok_out, uint8_t* status_out);

/* ---- the reference's other public 2-pairing checks (SURVEY.md section 8f-4), pairs assembled on the device ---------------
 * SignCryptCiphertext::is_valid (reference src/sign_crypt_ciphertext.rs:86-101 -> BlsSignCrypt::valid, src/traits/sign_crypt.rs:69-77):
 * W' = hash_to_point(U.to_bytes() || V, DST(scheme)); valid iff pairing([(W, -g), (W', U)]) is the identity and U, W are not.
 * U: public-key group (48 | 96 B), W: signature group (96 | 48 B), IETF compressed; v_bytes/v_off: the ciphertext bodies.
 *   ok_out[i] 1 | 0;  status_out[i]: BLSGPU_ST_OK or BLSGPU_ST_DESERIALIZE (an undecodable point: the reference fails at parse time) */
int blsgpu_signcrypt_valid_batch(blsgpu_ctx* ctx, int impl_id, int scheme, size_t n, const uint8_t* u_points, const uint8_t* w_points,
                                 const uint8_t* v_bytes, const uint64_t* v_off, uint8_t* ok_out, uint8_t* status_out);
/* SignDecryptionShare::verify (reference src/sign_decryption_share.rs:45-61 -> BlsSignCrypt::verify_share,
 * src/traits/sign_crypt.rs:192-207): ok iff share, pk_share and W are not the identity and
 * pairing([(-W', share), (W, pk_share)]) is the identity.  The reference always passes the Basic DST here (scheme = 0).
 *   shares, pk_shares, u_points: public-key group; w_points: signature group */
int blsgpu_signcrypt_verify_share_batch(blsgpu_ctx* ctx, int impl_id, int scheme, size_t n, const uint8_t* shares, const uint8_t* pk_shares,
                                        const uint8_t* u_points, const uint8_t* w_points, const uint8_t* v_bytes, const uint64_t* v_off,
                                        uint8_t* ok_out, uint8_t* status_out);
/* ProofOfKnowledge::verify (reference src/proof_of_knowledge.rs:132-165 -> BlsSignatureProof::verify,
 * src/traits/sig_proof.rs:102-142): a = hash_to_point(msg, DST(scheme)); OK iff pairing([(proof, g), (commitment + a*y, pk)])
 * is the identity.  commitments, proofs: signature group; pks: public-key group; challenges32: n x 32-byte big-endian
 * scalars y (ProofCommitmentChallenge; the timestamp variant's y = compute_y(u, t) is computed by the caller,
 * sig_proof.rs:37-46).  status_out[i]: OK, DESERIALIZE (a point, or y >= r), COMMITMENT_IDENTITY, PROOF_IDENTITY, PK_IDENTITY,
 * ZERO_CHALLENGE (checked in that order), INVALID_PROOF. */
int blsgpu_pok_verify_batch(blsgpu_ctx* ctx, int impl_id, int scheme, size_t n, const uint8_t* commitments, const uint8_t* proofs,
                            const uint8_t* pks, const uint8_t* challenges32, const uint8_t* msgs, const uint64_t* msg_off, uint8_t* status_out);

/* Wire front end on RAGGED records (SURVEY.md section 8f-3): network buffers as they arrived, each record delimited by
 * offsets; the length rules, the serde tag and the Legacy / Modern header validation are applied per record:
 *   public keys   : PublicKey::from_bytes_with_mode (reference src/public_key.rs:146-179): 48 | 96 bytes in `format`, else
 *                   BLSGPU_ST_INVALID_LENGTH
 *   signatures    : scheme_or_tagged >= 0: raw bytes in `format` under that scheme = Signature::from_bytes_with_mode
 *                   (src/signature.rs:209-253), wrong length -> INVALID_LENGTH;
 *                   scheme_or_tagged < 0: the serde_bare form, tag byte + IETF point (src/signature.rs:112-126,285-286), wrong
 *                   length or unknown tag -> BLSGPU_ST_DESERIALIZE
 * Everything else is blsgpu_verify_batch's status (header rules of src/impls/legacy.rs:39-82 included). */
int blsgpu_verify_batch_records(blsgpu_ctx* ctx, int impl_id, int format, int scheme_or_tagged, size_t n, const uint8_t* pk_bytes,
                                const uint64_t* pk_off, const uint8_t* sig_bytes, const uint64_t* sig_off, const uint8_t* msgs,
                                const uint64_t* msg_off, uint8_t* status_out);

/* Threshold-share combination (SURVEY.md section 8f-2): Signature::from_shares / PublicKey::from_shares
 * (reference src/signature.rs:151-165, src/public_key.rs, src/traits/sig_core.rs:92-105 -> vsss-rs `combine`):
 * Lagrange interpolation at zero over the share identifiers, out_j = sum_i lambda_i * value_i for every share set j.
 *   group      : 1 = G1 values (48-byte points), 2 = G2 values (96-byte points)
 *   shares     : share_off[q] records of 32 + 48|96 bytes, the reference's raw share form (src/lib.rs:117-157):
 *                32-byte big-endian identifier (a scalar < r) followed by the IETF compressed point
 *   share_off  : q + 1 offsets in shares (records, not bytes) delimiting the sets
 *   out        : q compressed points (zeroed for sets that fail);  status_out[q]: BLSGPU_ST_OK, BLSGPU_ST_DESERIALIZE
 *                (identifier >= r or undecodable point) or BLSGPU_ST_VSSS (fewer than 2 shares, zero or duplicate identifier)
 * The scheme-consistency rule (InvalidSignatureScheme, signature.rs:152-154) is decided by the caller-side binding. */
int blsgpu_combine_shares_batch(blsgpu_ctx* ctx, int group, size_t q, const uint64_t* share_off, const uint8_t* shares,
                                uint8_t* out, uint8_t* status_out);

/* Share verification on the raw share records (SURVEY.md section 8f-2/8f-3): n x PublicKeyShare::verify /
 * SignatureShare::verify (reference src/public_key_share.rs:55-71, src/signature_share.rs:98-101), which run the scheme's
 * verify on the share VALUES and ignore the identifiers.  Records are the reference's raw share form (src/lib.rs:117-157,
 * 219-259): 32-byte big-endian identifier || IETF compressed point, i.e. pk_shares: n x (32 + 48|96) bytes,
 * sig_shares: n x (32 + 96|48) bytes for impl 2 | 1.  An identifier that is not a canonical scalar (>= r) fails the
 * record's TryFrom (lib.rs:126-133) -> BLSGPU_ST_DESERIALIZE; everything else is blsgpu_verify_batch's status. */
int blsgpu_verify_share_batch(blsgpu_ctx* ctx, int impl_id, int scheme, size_t n, const uint8_t* pk_shares,
                              const uint8_t* sig_shares, const uint8_t* msgs, const uint64_t* msg_off, uint8_t* status_out);

/* Known-answer self-test of the device code: field multiplication, hash_to_curve, one accepted and one rejected golden
 * signature (reference tests/cpp_integration_test.rs:19-82), the fold of partial results.  Runs automatically at the first
 * blsgpu_ctx_create of a process on a device (a failing build refuses to create contexts); may be called again at any time. */
int blsgpu_selftest(blsgpu_ctx* ctx);

/* Host-only planning query (no device needed): the window layout the bucket multi-scalar multiplication of
 * blsgpu_verify_batch uses for a batch of n signatures with scalar_bits-bit (64 | 128) scalars. */
int blsgpu_plan_msm(size_t n, int scalar_bits, int* window_bits_out, int* windows_out, int* top_window_bits_out);

/* Host-only planning query: how a context on ndev devices cuts `sets` independent sets (key sets of
 * blsgpu_verify_secure_batch / blsgpu_aggregate_secure_batch; set_off = their sets + 1 cumulative member offsets) into
 * contiguous runs of about equal member count: device d takes sets cut_out[d] .. cut_out[d + 1] - 1 (cut_out has ndev + 1
 * entries, cut_out[0] = 0, cut_out[ndev] = sets; runs may be empty). */
int blsgpu_plan_shards(size_t sets, const uint64_t* set_off, int ndev, uint64_t* cut_out);

/* ---- metrics ---------------------------------------------------------------------------------------------------
 * Per-stage device times (CUDA events on the engine's stream) of the LAST verify call on the first device. */
#define BLSGPU_STAGE_DECODE_PK 0 /* blsgpu_verify_multisig_batch[_keyed]: the keys' decode and their segmented sums */
#define BLSGPU_STAGE_DECODE_SIG 1
#define BLSGPU_STAGE_HASH 2
#define BLSGPU_STAGE_SCALE_SIG 3 /* sum r_i sig_i (bucket multi-scalar multiplication) */
#define BLSGPU_STAGE_MILLER 4    /* prep + lines + accumulator kernels */
#define BLSGPU_STAGE_REDUCE 5
#define BLSGPU_STAGE_FINAL 6
#define BLSGPU_STAGE_BISECT 7
#define BLSGPU_STAGE_COUNT 8
int blsgpu_last_stage_ms(const blsgpu_ctx* ctx, float ms_out[BLSGPU_STAGE_COUNT]);

/* Device time of the hot kernels of the last blsgpu_verify_batch[_dev] call on this context (first device): one CUDA-event
 * pair around every launch, recorded on the stream the kernel is launched on; ms_out = total per kernel, launches_out
 * (may be NULL) = how many launches that total covers (more than one only when the Miller stage runs in several passes). */
#define BLSGPU_KERNEL_DECODE_PK 0      /* k_decode<pk group>: decompression (square root) */
#define BLSGPU_KERNEL_SUBGROUP_PK 1    /* k_subgroup_check<pk group> */
#define BLSGPU_KERNEL_DECODE_SIG 2     /* k_decode<sig group> */
#define BLSGPU_KERNEL_SUBGROUP_SIG 3   /* k_subgroup_check<sig group> */
#define BLSGPU_KERNEL_HASH_MAP 4       /* k_hash: expand_message, hash_to_field, 2 x (SSWU + isogeny), point addition */
#define BLSGPU_KERNEL_CLEAR_COFACTOR 5 /* k_clear_cofactor */
#define BLSGPU_KERNEL_TO_AFFINE 6      /* k_to_affine_batch (16 points per inversion) */
#define BLSGPU_KERNEL_M6_PREP 7        /* k_m6_prep: r_i * pk_i and the line scalars */
#define BLSGPU_KERNEL_M6_LINES 8       /* k_m6_lines: 68 line evaluations per pairing */
#define BLSGPU_KERNEL_M6_ACCUM 9       /* k_m6_accum: the shared Fp12 accumulators */
#define BLSGPU_KERNEL_COUNT 10
int blsgpu_last_kernel_ms(const blsgpu_ctx* ctx, float ms_out[BLSGPU_KERNEL_COUNT], int launches_out[BLSGPU_KERNEL_COUNT]);
/* number of kernel launches issued by this context since creation */
uint64_t blsgpu_launch_count(const blsgpu_ctx* ctx);

#ifdef __cplusplus
}
#endif
#endif /* BLSGPU_H */
