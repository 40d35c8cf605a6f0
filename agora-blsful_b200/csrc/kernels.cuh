// Device kernels of the batch verification engine.  Decode, hash, bucket-sum and tree kernels: one thread per item
// (signature, public key, bucket, tree node ...); the Miller stage: two lanes per pair for the lines, six lanes per group
// of six pairs for the shared accumulator.  ~10^4 field multiplications per item, integer-multiply bound; the largest HBM
// stream (39 KB of line records per item) is 1% of the run time (DESIGN.md sections 3-6).
#pragma once
#include <cuda_runtime.h>

#include "h2c.cuh"
#include "pairing.cuh"
#include "miller6.cuh"
#include "finalexp6.cuh"
#include "fr.cuh"

namespace bls {

// ---- group-generic glue ------------------------------------------------------------------------------------------
template <class A>
struct PtInfo;
template <>
struct PtInfo<G1Aff> {
  static const int LEN = 48;
  typedef G1Jac Jac;
  typedef Fp F;
};
template <>
struct PtInfo<G2Aff> {
  static const int LEN = 96;
  typedef G2Jac Jac;
  typedef Fp2 F;
};
__device__ __forceinline__ uint8_t pt_decompress(G1Aff& r, const uint8_t* b, bool chk) { return g1_decompress(r, b, chk); }
__device__ __forceinline__ uint8_t pt_decompress(G2Aff& r, const uint8_t* b, bool chk) { return g2_decompress(r, b, chk); }
__device__ __forceinline__ void pt_compress(uint8_t* o, const G1Aff& p) { g1_compress(o, p); }
__device__ __forceinline__ void pt_compress(uint8_t* o, const G2Aff& p) { g2_compress(o, p); }
__device__ __forceinline__ void pt_generator(G1Aff& g) {
  fp_set(g.x, K_G1X);
  fp_set(g.y, K_G1Y);
  g.inf = 0;
}
__device__ __forceinline__ void pt_generator(G2Aff& g) {
  fp2_set(g.x, K_G2X);
  fp2_set(g.y, K_G2Y);
  g.inf = 0;
}
template <class A>
__device__ __forceinline__ void pt_set_inf(A& p) {
  fzero(p.x);
  fzero(p.y);
  p.inf = 1;
}

// impl_id 2 (Bls12381G2Impl): pk in G1, sig/hash in G2.  impl_id 1 (Bls12381G1Impl): pk in G2, sig/hash in G1.
template <int IMPL>
struct ImplT;
template <>
struct ImplT<2> {
  typedef G1Aff PkAff;
  typedef G2Aff SigAff;
  typedef G1Jac PkJac;
  typedef G2Jac SigJac;
};
template <>
struct ImplT<1> {
  typedef G2Aff PkAff;
  typedef G1Aff SigAff;
  typedef G2Jac PkJac;
  typedef G1Jac SigJac;
};
__device__ __forceinline__ void hash_to_group(G2Jac& r, const uint8_t* pre, uint32_t pl, const uint8_t* m, uint32_t ml,
                                              const uint8_t* dst, uint32_t dl) {
  hash_to_g2(r, pre, pl, m, ml, dst, dl);
}
__device__ __forceinline__ void hash_to_group(G1Jac& r, const uint8_t* pre, uint32_t pl, const uint8_t* m, uint32_t ml,
                                              const uint8_t* dst, uint32_t dl) {
  hash_to_g1(r, pre, pl, m, ml, dst, dl);
}

__device__ __forceinline__ void hash_map_to_curve(G2Jac& r, const uint8_t* pre, uint32_t pl, const uint8_t* m, uint32_t ml,
                                                  const uint8_t* dst, uint32_t dl) {
  hash_map_g2(r, pre, pl, m, ml, dst, dl);
}
__device__ __forceinline__ void hash_map_to_curve(G1Jac& r, const uint8_t* pre, uint32_t pl, const uint8_t* m, uint32_t ml,
                                                  const uint8_t* dst, uint32_t dl) {
  hash_map_g1(r, pre, pl, m, ml, dst, dl);
}
__device__ __forceinline__ void clear_cofactor(G2Jac& r, const G2Jac& q) { g2_clear_cofactor(r, q); }
__device__ __forceinline__ void clear_cofactor(G1Jac& r, const G1Jac& q) { g1_clear_cofactor(r, q); }

struct DstParam {
  uint8_t b[64];
  uint32_t len;
};
struct Digest {
  uint8_t b[32];
};

#define BLS_TID() ((size_t)blockIdx.x * blockDim.x + threadIdx.x)
// resident 128-thread blocks per SM the heavy kernels are compiled for (register cap = 65536 / (128 * BLS_MIN_BLOCKS))
#ifndef BLS_MIN_BLOCKS
#define BLS_MIN_BLOCKS 1
#endif

// k_subgroup_check and k_clear_cofactor are pure curve arithmetic and take a 128-register cap (four blocks per SM) with a
// handful of spilled words; measured at 1M: decode 174 -> 171 ms, hash_to_curve 268 -> 257 ms.  The same cap on every
// kernel gains nothing more and slows the bucket kernels.
#if !defined(BLS_SPLIT_MIN_BLOCKS)
#define BLS_SPLIT_MIN_BLOCKS 4
#endif
// k_hash: three blocks per SM (170 registers).  Left to itself the G2 instance compiles to 164-176 registers depending on
// unrelated inlining decisions, and at 176 it drops to two blocks per SM: 93 -> 100 ms at 1M (seen when the point
// additions were rewritten in round 2).
#if !defined(BLS_HASH_MIN_BLOCKS)
#define BLS_HASH_MIN_BLOCKS 3
#endif
#if !defined(BLS_SPLIT2_MIN_BLOCKS)  // the same two kernels over Fp2 points
#define BLS_SPLIT2_MIN_BLOCKS 4
#endif
template <class A>
struct SplitBlocks {
  static constexpr int value = sizeof(A) > 2 * sizeof(Fp) + 16 ? BLS_SPLIT2_MIN_BLOCKS : BLS_SPLIT_MIN_BLOCKS;
};
// the per-key-set bucket kernel k_secure_msm: pure curve arithmetic as well (cfg 5 verify_secure 809 -> 784 ms at 10,000 x 400)
#if !defined(BLS_MSM_MIN_BLOCKS)
#define BLS_MSM_MIN_BLOCKS 4
#endif
// ---- decode: compressed bytes -> affine Montgomery points, curve + subgroup check --------------------------------
// Input staging: the block's 128 records (48 | 96 bytes each, contiguous) are fetched with coalesced 16-byte loads into
// shared memory and every thread then picks up its own record; a base pointer that is not 16-byte aligned (possible only
// through blsgpu_verify_batch_dev with caller-owned device buffers) takes the byte-wise path.
template <class A>
__global__ void __launch_bounds__(128, BLS_MIN_BLOCKS) k_decode(size_t n, const uint8_t* __restrict__ in, int format, A* __restrict__ out,
                                                uint8_t* __restrict__ st) {
  constexpr int L = PtInfo<A>::LEN;
  __shared__ __align__(16) uint8_t stage[128 * L];
  const size_t first = (size_t)blockIdx.x * blockDim.x;
  const size_t cnt = first < n ? (n - first < blockDim.x ? n - first : blockDim.x) : 0;
  const uint8_t* src = in + first * L;
  if ((reinterpret_cast<uintptr_t>(src) & 15u) == 0) {
    const uint4* v = reinterpret_cast<const uint4*>(src);
    uint4* d = reinterpret_cast<uint4*>(stage);
    const size_t quads = cnt * L / 16, tail = cnt * L - quads * 16;
    for (size_t q = threadIdx.x; q < quads; q += blockDim.x) d[q] = v[q];
    if (threadIdx.x < tail) stage[quads * 16 + threadIdx.x] = src[quads * 16 + threadIdx.x];
  } else {
    for (size_t b = threadIdx.x; b < cnt * L; b += blockDim.x) stage[b] = src[b];
  }
  __syncthreads();
  size_t i = BLS_TID();
  if (i >= n) return;
  uint8_t b[L];
  const uint32_t* rec = reinterpret_cast<const uint32_t*>(stage + threadIdx.x * L);
#pragma unroll
  for (int k = 0; k < L / 4; k++) {
    uint32_t w = rec[k];
    b[4 * k] = (uint8_t)w;
    b[4 * k + 1] = (uint8_t)(w >> 8);
    b[4 * k + 2] = (uint8_t)(w >> 16);
    b[4 * k + 3] = (uint8_t)(w >> 24);
  }
  uint8_t s = header_to_modern(b[0], format);
  A p;
  if (s == ST_OK) s = pt_decompress(p, b, false);  // on the curve; k_subgroup_check decides membership
  if (s != ST_OK) pt_set_inf(p);
  out[i] = p;
  st[i] = s;
}

// second half of the decode: the endomorphism subgroup check (G1: phi(P) + [x^2]P = O, G2: psi(P) = [x]P) on the decoded
// points, a launch of its own for the same reason as k_clear_cofactor (neither half carries the other's stack frame)
__device__ __forceinline__ bool pt_in_subgroup(const G1Aff& p) { return g1_in_subgroup(p); }
__device__ __forceinline__ bool pt_in_subgroup(const G2Aff& p) { return g2_in_subgroup(p); }
template <class A>
__global__ void __launch_bounds__(128, SplitBlocks<A>::value) k_subgroup_check(size_t n, A* __restrict__ pts, uint8_t* __restrict__ st) {
  size_t i = BLS_TID();
  if (i >= n || st[i] != ST_OK) return;
  A p = pts[i];
  if (p.inf || pt_in_subgroup(p)) return;
  pt_set_inf(p);
  pts[i] = p;
  st[i] = ST_DESERIALIZE;
}

// keyed verification: item i takes the decoded point and the decode status of key key_idx[i] of a key set that k_decode and
// k_subgroup_check filled once (a key that failed to decode is the identity there, as k_decode leaves it for the item)
template <class A>
__global__ void __launch_bounds__(128, BLS_MIN_BLOCKS) k_gather_keys(size_t n, const uint32_t* __restrict__ key_idx, const A* __restrict__ set_pts,
                                                     const uint8_t* __restrict__ set_st, A* __restrict__ out, uint8_t* __restrict__ st) {
  size_t i = BLS_TID();
  if (i >= n) return;
  const uint32_t k = key_idx[i];
  out[i] = set_pts[k];
  st[i] = set_st[k];
}

// affine points -> compressed bytes in `format`
template <class A>
__global__ void __launch_bounds__(128, BLS_MIN_BLOCKS) k_encode(size_t n, const A* __restrict__ in, int format, uint8_t* __restrict__ out) {
  size_t i = BLS_TID();
  if (i >= n) return;
  constexpr int L = PtInfo<A>::LEN;
  uint8_t b[L];
  A p = in[i];
  pt_compress(b, p);
  header_from_modern(b[0], format);
  for (int k = 0; k < L; k++) out[i * L + k] = b[k];
}

// Jacobian -> affine (one inversion per thread)
template <class A>
__global__ void __launch_bounds__(128, BLS_MIN_BLOCKS) k_to_affine(size_t n, const typename PtInfo<A>::Jac* __restrict__ in, A* __restrict__ out) {
  size_t i = BLS_TID();
  if (i >= n) return;
  typename PtInfo<A>::Jac p = in[i];
  A a;
  jac_to_aff(a, p);
  out[i] = a;
}

// Jacobian -> affine, TO_AFFINE_BATCH consecutive points per thread sharing one field inversion (the inversion is a
// 380-squaring exponentiation: ~490 of the ~5,300 Fp multiplications of a hash_to_curve; shared 16 ways it is ~30)
#define TO_AFFINE_BATCH 16
template <class A>
__global__ void __launch_bounds__(128) k_to_affine_batch(size_t n, const typename PtInfo<A>::Jac* __restrict__ in, A* __restrict__ out) {
  size_t base = BLS_TID() * TO_AFFINE_BATCH;
  if (base >= n) return;
  size_t left = n - base;
  jac_to_aff_batch<typename PtInfo<A>::F, TO_AFFINE_BATCH>(out + base, in + base, left < TO_AFFINE_BATCH ? (int)left : TO_AFFINE_BATCH);
}

// per-item status before any pairing work, in the reference's order (sig_core.rs:126-135 after the parse errors)
template <class PkA, class SigA>
__global__ void k_prestatus(size_t n, const uint8_t* st_pk, const uint8_t* st_sig, const PkA* pk, const SigA* sig,
                            uint8_t* out) {
  size_t i = BLS_TID();
  if (i >= n) return;
  uint8_t s = st_pk[i];
  if (s == ST_OK) s = st_sig[i];
  if (s == ST_OK && sig[i].inf) s = ST_SIG_IDENTITY;
  if (s == ST_OK && pk[i].inf) s = ST_PK_IDENTITY;
  out[i] = s;
}

// ---- hash_to_curve of the framed message ---------------------------------------------------------------------------
// msg_mode 0: msg ; 1: pk.to_bytes() || msg (MessageAugmentation, sig_aug.rs:20-24) ; 2: pk.to_bytes() (PoP, sig_pop.rs:66-69)
template <class HA, class PkA>
__global__ void __launch_bounds__(128, BLS_HASH_MIN_BLOCKS) k_hash(size_t n, const uint8_t* __restrict__ msgs, const uint64_t* __restrict__ msg_off,
                                              int msg_mode, const PkA* __restrict__ pk, const uint8_t* __restrict__ pre,
                                              DstParam dst, typename PtInfo<HA>::Jac* __restrict__ out) {
  size_t i = BLS_TID();
  if (i >= n) return;
  typename PtInfo<HA>::Jac hj;
  if (pre != nullptr && pre[i] != ST_OK) {
    jac_set_inf(hj);
    out[i] = hj;
    return;
  }
  uint8_t prefix[PtInfo<PkA>::LEN];
  uint32_t plen = 0;
  if (msg_mode != 0) {
    PkA p = pk[i];
    pt_compress(prefix, p);
    plen = PtInfo<PkA>::LEN;
  }
  const uint8_t* m = msgs;
  uint32_t mlen = 0;
  if (msg_mode != 2) {
    uint64_t o0 = msg_off[i], o1 = msg_off[i + 1];
    m = msgs + o0;
    mlen = (uint32_t)(o1 - o0);
  }
  hash_map_to_curve(hj, prefix, plen, m, mlen, dst.b, dst.len);
  out[i] = hj;  // on the curve, not yet in the subgroup: k_clear_cofactor, then k_to_affine_batch, finish the hash
}

// second half of hash_to_curve, in place: the h_eff multiplication (G2: psi method, two 64-bit multiplications; G1: 1 + |x|).
// A launch of its own so that neither half carries the other's stack frame (as one kernel: 9.2 KB of frame per thread and
// 276 ms at 1M; as two: 267 ms.  A third launch for hash_to_field, with map_to_curve per field element, gained nothing.)
// The result stays Jacobian: k_to_affine_batch normalises TO_AFFINE_BATCH points per field inversion.
template <class HA>
__global__ void __launch_bounds__(128, SplitBlocks<HA>::value) k_clear_cofactor(size_t n, typename PtInfo<HA>::Jac* __restrict__ pts) {
  size_t i = BLS_TID();
  if (i >= n) return;
  typename PtInfo<HA>::Jac q = pts[i], r;
  if (jac_is_inf(q)) return;  // items skipped by k_hash
  clear_cofactor(r, q);
  pts[i] = r;
}

// ---- random-linear-combination scalars --------------------------------------------------------------------------------
// leaf_i = SHA256(coordinates and identity flags of pk_i, sig_i, H_i); root = 16-ary SHA-256 tree over the leaves;
// r_i = the first rbits (64 | 128) bits of SHA256(root || salt || i), little-endian, forced non-zero.  The salt is 32
// bytes of OS randomness drawn per call (blsgpu.cu: fresh_salt) unless the caller pinned it for a reproducible run, so
// the scalars are unpredictable to whoever chose the batch; binding them to the inputs as well keeps them from being
// reused across different batches under a pinned salt.  Only explicit fields are hashed (never struct padding).
template <class P>
__device__ __forceinline__ void digest_point(Sha256& s, const P& p) {
  sha256_update(s, reinterpret_cast<const uint8_t*>(&p.x), sizeof(p.x));
  sha256_update(s, reinterpret_cast<const uint8_t*>(&p.y), sizeof(p.y));
  const uint8_t f = p.inf ? 1 : 0;
  sha256_update(s, &f, 1);
}
template <class PkA, class SigA>
__global__ void __launch_bounds__(128, BLS_MIN_BLOCKS) k_leaf_digest(size_t n, const PkA* pk, const SigA* sig, const SigA* h, Digest* out) {
  size_t i = BLS_TID();
  if (i >= n) return;
  Sha256 s;
  sha256_init(s);
  digest_point(s, pk[i]);
  digest_point(s, sig[i]);
  digest_point(s, h[i]);
  Digest d;
  sha256_final(s, d.b);
  out[i] = d;
}
__global__ void __launch_bounds__(128, BLS_MIN_BLOCKS) k_digest_reduce(size_t n_in, const Digest* in, size_t n_out, Digest* out) {
  size_t j = BLS_TID();
  if (j >= n_out) return;
  Sha256 s;
  sha256_init(s);
  for (int m = 0; m < 16; m++) {
    size_t idx = j + (size_t)m * n_out;
    if (idx < n_in) sha256_update(s, in[idx].b, 32);
  }
  Digest d;
  sha256_final(s, d.b);
  out[j] = d;
}
constexpr int RLC_MAX_WORDS = 4;  // 128-bit scalars at most
// k[0 .. rbits/32) = the scalar, remaining words zero
__device__ __forceinline__ void rlc_scalar(uint32_t k[RLC_MAX_WORDS], const Digest* root, size_t i, int rbits) {
  Sha256 s;
  sha256_init(s);
  sha256_update(s, root[0].b, 32);  // root[0] = tree root
  sha256_update(s, root[1].b, 32);  // root[1] = salt of this call
  uint8_t ib[8];
  for (int b = 0; b < 8; b++) ib[b] = (uint8_t)((uint64_t)i >> (8 * b));
  sha256_update(s, ib, 8);
  uint8_t d[32];
  sha256_final(s, d);
  uint32_t any = 0;
#pragma unroll
  for (int w = 0; w < RLC_MAX_WORDS; w++) {
    const uint32_t v = (uint32_t)d[4 * w] | ((uint32_t)d[4 * w + 1] << 8) | ((uint32_t)d[4 * w + 2] << 16) | ((uint32_t)d[4 * w + 3] << 24);
    k[w] = 32 * w < rbits ? v : 0u;
    any |= k[w];
  }
  if (any == 0) k[0] = 1;
}

// ---- per-item Miller loop (exact per-item checks of failing groups): ML(pk_i, H_i) (G2Impl) | ML(H_i, pk_i) (G1Impl) ------
__device__ __forceinline__ void miller_item(Fp12& f, const G1Aff& pk, const G2Aff& h, const uint32_t* k, bool scale) {
  MillerG1 mp;
  if (scale) {
    G1Jac pj;
    jac_mul_aff(pj, pk, k, 2);
    miller_prepare(mp, pj);
  } else {
    miller_prepare(mp, pk);
  }
  miller_loop(f, mp, h);
}
__device__ __forceinline__ void miller_item(Fp12& f, const G2Aff& pk, const G1Aff& h, const uint32_t* k, bool scale) {
  miller_item(f, h, pk, k, scale);
}
// ---- cooperative Miller loop (miller6.cuh): groups of 6 consecutive items, F_g = prod_{i in g} ML(r_i * pk_i, H_i) -------
// Three kernels, so that each keeps its working set on chip (DESIGN.md section 5):
//   k_m6_prep   one thread per item: the RLC scalar and r_i * pk_i, stored as the three Fp scalars the lines need, plus
//               the G2 point as (-x2, y2) for the addition steps (M6Arg, 560 B)
//   k_m6_lines  two lanes per item: the 68 line evaluations of the pair, record file in SHARED memory (10 records per
//               pair, record-major: conflict-free 128-bit accesses), lines streamed to HBM (39 KB per item)
//   k_m6_accum  six lanes per group: the shared Fp12 accumulator, one coefficient per lane, in shared memory (expanded
//               records, updated in place behind a group barrier); the next line is prefetched into L1 from HBM
constexpr int M6_LINES_TPB = 128;
constexpr int M6_LINES_PAIRS = M6_LINES_TPB / 2;
constexpr int M6_LINES_SMEM = M6_NREG * M6_LINES_PAIRS * (int)sizeof(SFp2);  // 71,680 B: three blocks per SM
constexpr int M6_ITEMS_PER_BLOCK = 120;                                   // k_m6_accum: 4 warps x 5 groups x 6 lanes
constexpr int M6_ACCUM_SMEM = 4 * 30 * (int)sizeof(SAccRec);
constexpr size_t M6_LINE_RECS = (size_t)M6_STEPS * 3;                     // records per item in the line stream

__device__ __forceinline__ const G1Aff& m6_g1(const G1Aff* pk, const G2Aff* h, size_t i) { return pk[i]; }
__device__ __forceinline__ const G1Aff& m6_g1(const G2Aff* pk, const G1Aff* h, size_t i) { return h[i]; }
__device__ __forceinline__ const G2Aff& m6_g2(const G1Aff* pk, const G2Aff* h, size_t i) { return h[i]; }
__device__ __forceinline__ const G2Aff& m6_g2(const G2Aff* pk, const G1Aff* h, size_t i) { return pk[i]; }

// items [base, base + n) of the batch -> args[0..n)
template <class PkA, class HA>
__global__ void __launch_bounds__(128, BLS_MIN_BLOCKS) k_m6_prep(size_t n, size_t base, const PkA* __restrict__ pk, const HA* __restrict__ h,
                                                 const uint8_t* __restrict__ pre, const Digest* __restrict__ root, int rbits,
                                                 M6Arg* __restrict__ args) {
  size_t c = BLS_TID();
  if (c >= n) return;
  const size_t i = base + c;
  if (pre[i] != ST_OK) return;
  G1Aff p = m6_g1(pk, h, i);
  MillerG1 mp;
  if (rbits) {  // 0: no random linear combination (aggregate verify), else the scalar width
    uint32_t sc[RLC_MAX_WORDS];
    rlc_scalar(sc, root, i, rbits);
    G1Jac pj;
    jac_mul_aff_w4(pj, p, sc, rbits / 4);
    miller_prepare(mp, pj);
  } else {
    miller_prepare(mp, p);
  }
  M6Arg a;
  const G2Aff q = m6_g2(pk, h, i);
  m6_make_arg(a, mp, q);
  args[c] = a;
}

// Two lanes per pair: lane h computes coefficient h of every program step (sop1), both read the pair's 10 records in
// shared memory (record-major, 112-byte stride between pairs: conflict-free; the two lanes of a pair read the same words).
// 64 pairs per 128-thread block, 71,680 B of shared memory (10 records per pair): three blocks per SM.
template <class PkA, class HA>
__global__ void __launch_bounds__(M6_LINES_TPB, 3) k_m6_lines(size_t n, size_t base, const M6Arg* __restrict__ args, const PkA* __restrict__ pk,
                                                             const HA* __restrict__ h, const uint8_t* __restrict__ pre, SLineRec* __restrict__ lines) {
  extern __shared__ __align__(16) uint8_t m6_smem[];
  const int hh = threadIdx.x & 1, pib = threadIdx.x >> 1;
  const size_t c = (size_t)blockIdx.x * M6_LINES_PAIRS + pib;
  const bool active = c < n && pre[base + (c < n ? c : 0)] == ST_OK;
  const size_t cc = active ? c : 0;
  const G2Aff& q = m6_g2(pk, h, base + cc);
  SopSpaces cx = m6_spaces_line(reinterpret_cast<SFp2*>(m6_smem) + pib, M6_LINES_PAIRS, args + cc, lines + cc * M6_LINE_RECS);
  if (active && hh == 0) {
    const G2Aff qv = q;
    m6_init_point(cx, qv);
  }
  __syncwarp();
  const uint64_t e = K_X_ABS;
#pragma unroll 1
  for (int i = 62; i >= 0; i--) {
#pragma unroll 1
    for (int pass = 0; pass < 1 + (int)((e >> i) & 1); pass++) {
      const M6Op* prog = pass == 0 ? K_M6_DBL : K_M6_ADD;
      const int nops = pass == 0 ? K_M6_DBL_N : K_M6_ADD_N;
#pragma unroll 1
      for (int o = 0; o < nops; o++) {
        const M6Op* op = prog + o;
        int32_t res[NL], other[NL];
        double vb = 0;
        if (active) vb = m6_op_compute(res, op, cx, hh);
        if (op->dst >= SOPX_LINE) {  // the sum run of a line record needs the partner's coefficient (uniform branch)
#pragma unroll
          for (int j = 0; j < NL; j++) other[j] = __shfl_xor_sync(0xffffffffu, res[j], 1);
        }
        __syncwarp();  // every lane has read its operands: results may now overwrite them
        if (active) m6_op_store(op, cx, hh, res, other, vb);
        __syncwarp();
      }
      cx.line += 3;
    }
  }
}

#ifndef M6_ACC_BLOCKS
#define M6_ACC_BLOCKS 3
#endif
__global__ void __launch_bounds__(128, M6_ACC_BLOCKS) k_m6_accum(size_t n, size_t base, const uint8_t* __restrict__ pre, const SLineRec* __restrict__ lines,
                                                     Fp12* __restrict__ out) {
  extern __shared__ __align__(16) uint8_t m6_smem[];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int g = lane / 6, k = lane - 6 * g;
  const bool lane_on = g < 5;  // lanes 30, 31 only keep the warp's barriers company
  SAccRec* F = reinterpret_cast<SAccRec*>(m6_smem) + warp * 30 + 6 * (lane_on ? g : 0);  // updated in place (sopw's barrier)
  const unsigned gsync = lane_on ? 63u << (6 * g) : 0xc0000000u;  // the lanes that share this F
  const size_t group = ((size_t)blockIdx.x * 4 + warp) * 5 + g;  // within the chunk (base is a multiple of 6)
  const size_t item = group * 6 + k;
  const bool active = lane_on && item < n && pre[base + item] == ST_OK;
  const unsigned ball = __ballot_sync(0xffffffffu, active);
  const unsigned gmask = lane_on ? (ball >> (6 * g)) & 63u : 0u;
  if (lane_on) {
    SFp2 init;
    if (k == 0) sfp2_one(init); else sfp2_zero(init);
    sacc_from_sfp2(F[k], init);
  }
  __syncwarp();
  const SLineRec* gl = lines + group * 6 * M6_LINE_RECS;  // the group's six line streams
  const uint64_t e = K_X_ABS;
  int step = 0;
  if (gmask != 0) {  // uniform within the group; every barrier below names the group's lanes only
#pragma unroll 1
    for (int i = 62; i >= 0; i--) {
      if (i != 62) m6_sqr_lane(F + k, F, k, gsync);
      const int nst = 1 + (int)((e >> i) & 1);
#pragma unroll 1
      for (int st = 0; st < nst; st++, step++) {
#pragma unroll 1
        for (int j = 0; j < 6; j++) {
          {
            // the NEXT line of this group (576 B in HBM, used once by all six lanes) starts its way into L1 now
            const int jn = j == 5 ? 0 : j + 1;
            const int sn = j == 5 ? step + 1 : step;
            if (k < 3 && sn < M6_STEPS) {
              const SLineRec* nx = gl + (size_t)jn * M6_LINE_RECS + 3 * sn + k;
              asm volatile("prefetch.global.L1 [%0];" ::"l"(nx));
              asm volatile("prefetch.global.L1 [%0];" ::"l"(reinterpret_cast<const uint8_t*>(nx) + 128));
            }
          }
          if ((gmask >> j) & 1u) m6_mul_line_lane(F + k, F, gl + (size_t)j * M6_LINE_RECS + 3 * step, k, gsync);
        }
      }
    }
  }
  __syncwarp();
  if (lane_on && group * 6 < n) m6_finish_lane(*fp12_coeff(out[base / 6 + group], k), F[k], k);
}

// S_i = r_i * sig_i
template <class SigA>
__global__ void __launch_bounds__(128, BLS_MIN_BLOCKS) k_scale_sig(size_t n, const SigA* __restrict__ sig, const uint8_t* __restrict__ pre,
                                                   const Digest* __restrict__ root, int rbits,
                                                   typename PtInfo<SigA>::Jac* __restrict__ out) {
  size_t i = BLS_TID();
  if (i >= n) return;
  typename PtInfo<SigA>::Jac s;
  if (pre[i] != ST_OK) {
    jac_set_inf(s);
  } else {
    uint32_t k[RLC_MAX_WORDS];
    rlc_scalar(k, root, i, rbits);
    SigA a = sig[i];
    jac_mul_aff(s, a, k, rbits / 32);
  }
  out[i] = s;
}

// ---- S = sum_i r_i * sig_i as a bucket (Pippenger) multi-scalar multiplication ------------------------------------------
// The per-item double-and-add (k_scale_sig: 64 doublings + ~32 additions per signature) is only needed when a batch FAILS
// and the bisection wants per-group sums; the accept path needs the total only: with c-bit windows every signature costs
// one mixed addition per window (4 at c = 16 instead of ~96 point operations).
//   k_msm_count   r_i -> digits, histogram of every window (global atomics)
//   k_msm_scan    exclusive prefix sums of the histograms (one block per window)
//   k_msm_scatter item indices sorted by digit (counting sort; order inside a bucket is irrelevant to the sum)
//   k_msm_bucket  one thread per (window, digit): B = sum of its signatures
//   k_msm_chunk   one thread per 16 buckets: 2^(c w) * sum_j j B_j over the chunk (running sums), then a flat tree sum
constexpr int MSM_CHUNK = 16;
struct RlcScalar {  // little-endian 64-bit halves (hi = 0 for 64-bit scalars)
  uint64_t lo, hi;
};
__device__ __forceinline__ uint32_t msm_digit(const RlcScalar& r, int c, int w) {  // c <= 16
  const int bit = c * w;
  const uint64_t v = bit >= 64 ? r.hi >> (bit - 64) : bit == 0 ? r.lo : (r.lo >> bit) | (r.hi << (64 - bit));
  return (uint32_t)v & ((1u << c) - 1u);
}
__global__ void __launch_bounds__(128) k_msm_count(size_t n, const uint8_t* __restrict__ pre, const Digest* __restrict__ root, int rbits, int c,
                                                   int nwin, RlcScalar* __restrict__ r_out, uint32_t* __restrict__ counts) {
  size_t i = BLS_TID();
  if (i >= n) return;
  RlcScalar r = {0, 0};
  if (pre[i] == ST_OK) {
    uint32_t k[RLC_MAX_WORDS];
    rlc_scalar(k, root, i, rbits);
    r.lo = (uint64_t)k[0] | ((uint64_t)k[1] << 32);
    r.hi = (uint64_t)k[2] | ((uint64_t)k[3] << 32);
  }
  r_out[i] = r;
  for (int w = 0; w < nwin; w++) {
    const uint32_t d = msm_digit(r, c, w);
    if (d) atomicAdd(&counts[((size_t)w << c) + d], 1u);
  }
}
// counts -> exclusive offsets (per window); cursors zeroed.  One block of 1024 threads per window, nb = 2^c entries.
__global__ void __launch_bounds__(1024) k_msm_scan(int c, const uint32_t* __restrict__ counts, uint32_t* __restrict__ offsets,
                                                   uint32_t* __restrict__ cursor) {
  __shared__ uint32_t part[1024];
  const size_t nb = (size_t)1 << c;
  const uint32_t* cnt = counts + (size_t)blockIdx.x * nb;
  uint32_t* off = offsets + (size_t)blockIdx.x * nb;
  uint32_t* cur = cursor + (size_t)blockIdx.x * nb;
  const size_t per = (nb + 1023) / 1024;
  const size_t lo = (size_t)threadIdx.x * per, hi = lo + per < nb ? lo + per : nb;
  uint32_t sum = 0;
  for (size_t j = lo; j < hi; j++) sum += cnt[j];
  part[threadIdx.x] = sum;
  __syncthreads();
  for (int d = 1; d < 1024; d <<= 1) {
    uint32_t v = threadIdx.x >= d ? part[threadIdx.x - d] : 0;
    __syncthreads();
    part[threadIdx.x] += v;
    __syncthreads();
  }
  uint32_t run = part[threadIdx.x] - sum;
  for (size_t j = lo; j < hi; j++) {
    off[j] = run;
    cur[j] = 0;
    run += cnt[j];
  }
}
__global__ void __launch_bounds__(128) k_msm_scatter(size_t n, const RlcScalar* __restrict__ r_in, int c, int nwin, const uint32_t* __restrict__ offsets,
                                                     uint32_t* __restrict__ cursor, uint32_t* __restrict__ sorted) {
  size_t i = BLS_TID();
  if (i >= n) return;
  const RlcScalar r = r_in[i];
  for (int w = 0; w < nwin; w++) {
    const uint32_t d = msm_digit(r, c, w);
    if (d) {
      const size_t b = ((size_t)w << c) + d;
      const uint32_t pos = offsets[b] + atomicAdd(&cursor[b], 1u);
      sorted[(size_t)w * n + pos] = (uint32_t)i;
    }
  }
}
template <class SigA>
__global__ void __launch_bounds__(128, BLS_MIN_BLOCKS) k_msm_bucket(size_t n, size_t nbuckets, const SigA* __restrict__ sig, int c,
                                                    const uint32_t* __restrict__ counts, const uint32_t* __restrict__ offsets,
                                                    const uint32_t* __restrict__ sorted, typename PtInfo<SigA>::Jac* __restrict__ B) {
  size_t b = BLS_TID();
  if (b >= nbuckets) return;
  typename PtInfo<SigA>::Jac acc;
  jac_set_inf(acc);
  const size_t w = b >> c;
  const uint32_t cnt = counts[b], off = offsets[b];
  const uint32_t* idx = sorted + w * n + off;
  for (uint32_t t = 0; t < cnt; t++) {
    SigA a = sig[idx[t]];
    jac_add_mixed(acc, acc, a);
  }
  B[b] = acc;
}
template <class J>
__device__ __forceinline__ void jac_mul_small(J& r, const J& p, uint32_t k) {
  J acc;
  jac_set_inf(acc);
  bool started = false;  // doubling the identity costs as much as doubling a point
  for (int b = 31; b >= 0; b--) {
    if (started) jac_dbl(acc, acc);
    if ((k >> b) & 1u) {
      jac_add(acc, acc, p);
      started = true;
    }
  }
  r = acc;
}
template <class J>
__global__ void __launch_bounds__(128, BLS_MIN_BLOCKS) k_msm_chunk(size_t nchunks, int c, const J* __restrict__ B, J* __restrict__ V) {
  size_t t = BLS_TID();
  if (t >= nchunks) return;
  const size_t per_win = ((size_t)1 << c) / MSM_CHUNK;  // chunks per window
  const size_t w = t / per_win, tc = t % per_win;
  const size_t j0 = (w << c) + tc * MSM_CHUNK;             // first bucket of the chunk; its digit is tc * MSM_CHUNK
  J run, ws;
  jac_set_inf(run);
  jac_set_inf(ws);
  for (int j = MSM_CHUNK - 1; j >= 0; j--) {
    J bj = B[j0 + j];
    jac_add(run, run, bj);
    jac_add(ws, ws, run);  // ws = sum_j (j + 1) B_{j0 + j}
  }
  // sum_j (digit_j) B = ws + (tc * MSM_CHUNK - 1) * run
  const uint32_t base = (uint32_t)(tc * MSM_CHUNK);
  J res;
  if (base == 0) {
    J nr;
    jac_neg(nr, run);
    jac_add(res, ws, nr);
  } else {
    J m;
    jac_mul_small(m, run, base - 1u);
    jac_add(res, ws, m);
  }
  if (!jac_is_inf(res))
    for (size_t s = 0; s < w * (size_t)c; s++) jac_dbl(res, res);
  V[t] = res;
}

// ---- failure path: S of every LEVEL-1 node of the product tree, without per-item scalar multiplications -----------------
// A failed batch needs sum r_i sig_i per tree node.  Round 1 multiplied every signature by its 64-bit scalar (64 doublings +
// ~32 additions per item: +370 ms at 1M).  A level-1 node covers 16 groups of 6 items (groups j + m * n1, m < 16): one warp
// per node runs a small bucket method over its 96 signatures - lane = (4-bit window w = lane & 15, half = lane >> 4 of the
// node's groups): 48 mixed additions into 15 buckets + 30 additions of the running-sum reduction per lane, then the halves
// are added and the 16 window sums folded by k_node_combine.  ~21 point operations per item instead of ~96; the levels above
// come from the usual tree sums, and per-item work is left for the (few) level-1 nodes that fail.
constexpr int NODE_BUCKETS = 15;
// (no register cap here: measured at 1M with one bad signature, the G2 instance under a 128-register cap made the failure
// path 60 ms slower - 204 registers and 2 blocks per SM is its better point, unlike k_secure_msm below)
template <class SigA>
__global__ void __launch_bounds__(128, BLS_MIN_BLOCKS) k_node_msm(size_t n, size_t n1, size_t ng, const SigA* __restrict__ sig, const uint8_t* __restrict__ pre,
                                                  const RlcScalar* __restrict__ r, typename PtInfo<SigA>::Jac* __restrict__ buckets,
                                                  typename PtInfo<SigA>::Jac* __restrict__ W) {
  typedef typename PtInfo<SigA>::Jac J;
  const int lane = threadIdx.x & 31, w = lane & 15, half = lane >> 4;
  const size_t warp = (size_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5), nwarps = (size_t)gridDim.x * (blockDim.x >> 5);
  J* mine = buckets + (warp * 32 + lane) * NODE_BUCKETS;
  for (size_t node = warp; node < n1; node += nwarps) {
    uint32_t full = 0;
    for (int m = 8 * half; m < 8 * half + 8; m++) {
      const size_t g = node + (size_t)m * n1;
      if (g >= ng) break;
      for (int t = 0; t < M6_GROUP; t++) {
        const size_t i = g * M6_GROUP + t;
        if (i >= n || pre[i] != ST_OK) continue;
        const RlcScalar k = r[i];
        const uint32_t d = (uint32_t)(k.lo >> (4 * w)) & 15u;  // 64-bit scalars: 16 windows of 4 bits
        if (d == 0) continue;
        SigA p = sig[i];
        J acc;
        if ((full >> (d - 1)) & 1u) {
          acc = mine[d - 1];
          jac_add_mixed(acc, acc, p);
        } else {
          jac_from_aff(acc, p);
          full |= 1u << (d - 1);
        }
        mine[d - 1] = acc;
      }
    }
    J run, tot;
    jac_set_inf(run);
    jac_set_inf(tot);
    bool any = false;
    for (int b = NODE_BUCKETS - 1; b >= 0; b--) {
      if ((full >> b) & 1u) {
        J t = mine[b];
        jac_add(run, run, t);
        any = true;
      }
      if (any) jac_add(tot, tot, run);
    }
    W[node * 32 + lane] = tot;
  }
}
// S[node] = sum_w 16^w (W[node][w] + W[node][16 + w])
template <class J>
__global__ void __launch_bounds__(128, BLS_MIN_BLOCKS) k_node_combine(size_t n1, const J* __restrict__ W, J* __restrict__ S) {
  size_t node = BLS_TID();
  if (node >= n1) return;
  J acc;
  jac_set_inf(acc);
  for (int w = 15; w >= 0; w--) {
    if (!jac_is_inf(acc))
      for (int k = 0; k < 4; k++) jac_dbl(acc, acc);
    J a = W[node * 32 + w], b = W[node * 32 + 16 + w];
    jac_add(acc, acc, a);
    jac_add(acc, acc, b);
  }
  S[node] = acc;
}
// S_i = r_i * sig_i for the listed items only
template <class SigA>
__global__ void __launch_bounds__(128, BLS_MIN_BLOCKS) k_scale_sig_list(size_t cnt, const uint32_t* __restrict__ idx, const SigA* __restrict__ sig,
                                                        const uint8_t* __restrict__ pre, const Digest* __restrict__ root, int rbits,
                                                        typename PtInfo<SigA>::Jac* __restrict__ out) {
  size_t c = BLS_TID();
  if (c >= cnt) return;
  const size_t i = idx[c];
  typename PtInfo<SigA>::Jac s;
  if (pre[i] != ST_OK) {
    jac_set_inf(s);
  } else {
    uint32_t k[RLC_MAX_WORDS];
    rlc_scalar(k, root, i, rbits);
    SigA a = sig[i];
    jac_mul_aff(s, a, k, rbits / 32);
  }
  out[i] = s;
}
// S_g for the listed groups
template <class J>
__global__ void __launch_bounds__(128, BLS_MIN_BLOCKS) k_group_sum_list(size_t cnt, const uint32_t* __restrict__ groups, size_t n, const J* __restrict__ in,
                                                        J* __restrict__ out) {
  size_t c = BLS_TID();
  if (c >= cnt) return;
  const size_t g = groups[c];
  J acc = in[g * M6_GROUP];
  for (int m = 1; m < M6_GROUP; m++) {
    size_t i = g * M6_GROUP + m;
    if (i < n) {
      J t = in[i];
      jac_add(acc, acc, t);
    }
  }
  out[g] = acc;
}

// ---- 16-ary strided reduction trees: out[j] = op over in[j + m*n_out], m = 0..15 -------------------------------------
__global__ void __launch_bounds__(128, BLS_MIN_BLOCKS) k_reduce_fp12(size_t n_in, const Fp12* __restrict__ in, size_t n_out, Fp12* __restrict__ out) {
  size_t j = BLS_TID();
  if (j >= n_out) return;
  Fp12 acc = in[j];
  for (int m = 1; m < 16; m++) {
    size_t idx = j + (size_t)m * n_out;
    if (idx < n_in) {
      Fp12 t = in[idx];
      fp12_mul(acc, acc, t);
    }
  }
  out[j] = acc;
}
template <class J>
__global__ void __launch_bounds__(128, BLS_MIN_BLOCKS) k_reduce_jac(size_t n_in, const J* __restrict__ in, size_t n_out, J* __restrict__ out) {
  size_t j = BLS_TID();
  if (j >= n_out) return;
  J acc = in[j];
  for (int m = 1; m < 16; m++) {
    size_t idx = j + (size_t)m * n_out;
    if (idx < n_in) {
      J t = in[idx];
      jac_add(acc, acc, t);
    }
  }
  out[j] = acc;
}
// The same levels with SIXTEEN lanes per output node (lane m loads child m, four shuffle-and-multiply steps): a level with
// few nodes is pure latency - 15 dependent Fp12 products (~100 us each) or point additions (~70 us) per thread - and this
// form has 4 on its critical path.  It spends 4 x 16 lane-operations per node instead of 15, so it is only used where the
// narrow form cannot fill the GPU anyway (REDUCE_WIDE_MAX output nodes; blsgpu.cu REDUCE_FP12 / REDUCE_JAC).
template <class T>
__device__ __forceinline__ void words_shfl_xor(T& r, const T& p, int mask) {
  static_assert(sizeof(T) % 4 == 0, "records are whole words");
  const uint32_t* src = reinterpret_cast<const uint32_t*>(&p);
  uint32_t* dst = reinterpret_cast<uint32_t*>(&r);
#pragma unroll 8
  for (size_t i = 0; i < sizeof(T) / 4; i++) dst[i] = __shfl_xor_sync(0xffffffffu, src[i], mask);
}
__global__ void __launch_bounds__(128, BLS_MIN_BLOCKS) k_reduce_fp12_w(size_t n_in, const Fp12* __restrict__ in, size_t n_out, Fp12* __restrict__ out) {
  const size_t t = BLS_TID(), j = t >> 4;
  const int m = (int)(t & 15);
  const size_t idx = j + (size_t)m * n_out;
  Fp12 acc;
  if (j < n_out && idx < n_in) acc = in[idx]; else fp12_one(acc);
#pragma unroll 1
  for (int s = 1; s < 16; s <<= 1) {
    Fp12 other;
    words_shfl_xor(other, acc, s);
    if ((m & (2 * s - 1)) == 0) fp12_mul(acc, acc, other);
  }
  if (j < n_out && m == 0) out[j] = acc;
}
template <class J>
__global__ void __launch_bounds__(128, BLS_MIN_BLOCKS) k_reduce_jac_w(size_t n_in, const J* __restrict__ in, size_t n_out, J* __restrict__ out) {
  const size_t t = BLS_TID(), j = t >> 4;
  const int m = (int)(t & 15);
  const size_t idx = j + (size_t)m * n_out;
  J acc;
  if (j < n_out && idx < n_in) acc = in[idx]; else jac_set_inf(acc);
#pragma unroll 1
  for (int s = 1; s < 16; s <<= 1) {
    J other;
    words_shfl_xor(other, acc, s);
    if ((m & (2 * s - 1)) == 0) jac_add(acc, acc, other);
  }
  if (j < n_out && m == 0) out[j] = acc;
}
// same for affine inputs (first level of a plain point sum)
template <class A>
__global__ void __launch_bounds__(128, BLS_MIN_BLOCKS) k_reduce_aff(size_t n_in, const A* __restrict__ in, size_t n_out,
                                                    typename PtInfo<A>::Jac* __restrict__ out) {
  size_t j = BLS_TID();
  if (j >= n_out) return;
  typename PtInfo<A>::Jac acc;
  jac_set_inf(acc);
  for (int m = 0; m < 16; m++) {
    size_t idx = j + (size_t)m * n_out;
    if (idx < n_in) {
      A t = in[idx];
      jac_add_mixed(acc, acc, t);
    }
  }
  out[j] = acc;
}

// ---- probes: is  F * prod_j e(P_j, Q_j)  == 1 after the final exponentiation? --------------------------------------------
// A probe is one GROUP of the cooperative Miller kernels (up to six pairs at items 6c .. 6c + 5 of a scratch batch) followed
// by the six-lane final exponentiation (finalexp6.cuh).  Round 1 ran every probe on ONE thread (Miller loop 9 ms + final
// exponentiation 14 ms of latency per bisection level); the cooperative kernels bring a level to ~3 ms.
//   node probe : F = the node's product of Miller values, one pair (-g, S_node):   e(pk-side generator negated, sum r_i sig_i)
//   leaf probe : F = 1, two pairs (pk_i, H_i), (-g, sig_i): the exact per-item equation of core_verify (sig_core.rs:138-145)
// k_probe_fill_* write the scratch batch (points + per-item status; everything not written stays "skip").
constexpr uint8_t PROBE_SKIP = 0xfe;  // any status != ST_OK makes the Miller kernels skip the item
template <class PkA, class SigA>
__global__ void __launch_bounds__(128, BLS_MIN_BLOCKS) k_probe_fill_nodes(size_t cnt, const uint32_t* __restrict__ idx,
                                                          const typename PtInfo<SigA>::Jac* __restrict__ S, PkA* __restrict__ xpk,
                                                          SigA* __restrict__ xh, uint8_t* __restrict__ xpre) {
  size_t c = BLS_TID();
  if (c >= cnt) return;
  const size_t j = idx ? idx[c] : c;
  typename PtInfo<SigA>::Jac s = S[j];
  SigA sa;
  jac_to_aff(sa, s);
  PkA ng;
  pt_generator(ng);
  aff_neg(ng, ng);
  xpk[6 * c] = ng;
  xh[6 * c] = sa;
  xpre[6 * c] = sa.inf ? PROBE_SKIP : ST_OK;  // S = O contributes e(., O) = 1
  for (int m = 1; m < 6; m++) xpre[6 * c + m] = PROBE_SKIP;
}
template <class PkA, class SigA>
__global__ void __launch_bounds__(128, BLS_MIN_BLOCKS) k_probe_fill_leaves(size_t cnt, const uint32_t* __restrict__ idx, const PkA* __restrict__ pk,
                                                           const SigA* __restrict__ h, const SigA* __restrict__ sig,
                                                           const uint8_t* __restrict__ status, PkA* __restrict__ xpk,
                                                           SigA* __restrict__ xh, uint8_t* __restrict__ xpre) {
  size_t c = BLS_TID();
  if (c >= cnt) return;
  const size_t i = idx[c];
  const bool on = status[i] == ST_OK;  // anything else was decided before the pairing: its probe is the empty product
  if (on) {
    PkA ng;
    pt_generator(ng);
    aff_neg(ng, ng);
    xpk[6 * c] = pk[i];
    xh[6 * c] = h[i];
    xpk[6 * c + 1] = ng;
    xh[6 * c + 1] = sig[i];
  }
  xpre[6 * c] = xpre[6 * c + 1] = on ? ST_OK : PROBE_SKIP;
  for (int m = 2; m < 6; m++) xpre[6 * c + m] = PROBE_SKIP;
}
// ok[c] = ( F[idx ? idx[c] : c] * T[c] )^(3 (p^12-1)/r) == 1 ; F == nullptr: F = 1.  Five probes per warp, six lanes each.
constexpr int FE6_PER_WARP = 5;
constexpr int FE6_SMEM = FE6_PER_WARP * (FE6_NREG * 6 * (int)sizeof(SAccRec) + (int)sizeof(Fp12));
__global__ void __launch_bounds__(32) k_final6(size_t cnt, const uint32_t* __restrict__ idx, const Fp12* __restrict__ F,
                                               const Fp12* __restrict__ T, uint8_t* __restrict__ ok) {
  extern __shared__ __align__(16) uint8_t fe6_smem[];
  const int lane = threadIdx.x, g = lane / 6, k = lane - 6 * g;
  const size_t c = (size_t)blockIdx.x * FE6_PER_WARP + g;
  if (g >= FE6_PER_WARP || c >= cnt) return;  // whole groups leave together: every barrier below names one group's lanes
  Fe6 cx;
  cx.R = reinterpret_cast<SAccRec*>(fe6_smem) + g * FE6_NREG * 6;
  cx.scratch = reinterpret_cast<Fp12*>(fe6_smem + FE6_PER_WARP * FE6_NREG * 6 * sizeof(SAccRec)) + g;
  cx.k = k;
  cx.mask = 63u << (6 * g);
  {
    Fp12 t = T[c];
    fe6_load_coeff(fe6_reg(cx, F ? 1 : 0)[k], *fp12_coeff(t, k));
  }
  if (F) {
    Fp12 f = F[idx ? idx[c] : c];
    fe6_load_coeff(fe6_reg(cx, 2)[k], *fp12_coeff(f, k));
    __syncwarp(cx.mask);
    fe6_mul(cx, 0, 1, 2);
  } else {
    __syncwarp(cx.mask);
  }
  fe6_final_exponentiation(cx);
  const unsigned votes = __ballot_sync(cx.mask, fe6_lane_is_one(cx, k));
  if (k == 0) ok[c] = ((votes >> (6 * g)) & 63u) == 63u ? 1 : 0;
}

// S_g = sum of the (up to) 6 consecutive per-item points of group g
template <class J>
__global__ void __launch_bounds__(128, BLS_MIN_BLOCKS) k_group_sum(size_t n, const J* __restrict__ in, size_t ng, J* __restrict__ out) {
  size_t g = BLS_TID();
  if (g >= ng) return;
  J acc = in[g * M6_GROUP];
  for (int m = 1; m < M6_GROUP; m++) {
    size_t idx = g * M6_GROUP + m;
    if (idx < n) {
      J t = in[idx];
      jac_add(acc, acc, t);
    }
  }
  out[g] = acc;
}

// leaves that failed their exact check
__global__ void k_mark_invalid(size_t cnt, const uint32_t* idx, const uint8_t* ok, uint8_t* status) {
  size_t c = BLS_TID();
  if (c >= cnt) return;
  if (!ok[c]) status[idx[c]] = ST_INVALID_SIGNATURE;
}

// ---- secure aggregation (reference src/secure_aggregation.rs) ------------------------------------------------------------
// base_j = SHA256(sorted key bytes of key set j)            (:45-59, :284-298)
__global__ void __launch_bounds__(128) k_secure_base(size_t q, const uint64_t* __restrict__ key_off, const uint32_t* __restrict__ ord,
                                                     const uint8_t* __restrict__ key_bytes, int key_len, Digest* __restrict__ base) {
  size_t j = BLS_TID();
  if (j >= q) return;
  Sha256 s;
  sha256_init(s);
  for (uint64_t i = key_off[j]; i < key_off[j + 1]; i++) sha256_update(s, key_bytes + (size_t)ord[i] * key_len, (uint32_t)key_len);
  Digest d;
  sha256_final(s, d.b);
  base[j] = d;
}
// t = BE(SHA256(be32(pos) || base)) mod r as 8 little-endian words; returns false if t == 0   (:61-103, :300-331)
__device__ __forceinline__ bool secure_coefficient(uint32_t t[8], uint32_t pos, const Digest& base) {
  Sha256 s;
  sha256_init(s);
  uint8_t ib[4] = {(uint8_t)(pos >> 24), (uint8_t)(pos >> 16), (uint8_t)(pos >> 8), (uint8_t)pos};
  sha256_update(s, ib, 4);
  sha256_update(s, base.b, 32);
  uint8_t d[32];
  sha256_final(s, d);
  for (int w = 0; w < 8; w++) {
    const uint8_t* p = d + 28 - 4 * w;
    t[w] = ((uint32_t)p[0] << 24) | ((uint32_t)p[1] << 16) | ((uint32_t)p[2] << 8) | p[3];
  }
  // 2^256 < 3r: at most two subtractions of r
  for (int rep = 0; rep < 2; rep++) {
    uint32_t u[8];
    int64_t br = 0;
    for (int w = 0; w < 8; w++) {
      int64_t v = (int64_t)t[w] - (int64_t)K_R_ORDER[w] + br;
      u[w] = (uint32_t)v;
      br = v >> 32;
    }
    if (br == 0)
      for (int w = 0; w < 8; w++) t[w] = u[w];
  }
  uint32_t any = 0;
  for (int w = 0; w < 8; w++) any |= t[w];
  return any != 0;
}
// ---- the coefficient multi-scalar multiplication of a key set: sum_i t_i * P_i (secure_aggregation.rs:150-153, 201-204) ------
// Round 1 multiplied every member by its 255-bit coefficient on its own thread (255 doublings + ~128 additions each) and
// added a quorum's 400 products on ONE thread.  Now: Pippenger's bucket method per key set with signed 8-bit windows -
// 32 windows = the 32 lanes of ONE WARP per key set.  Lane w drops every member into one of its 128 buckets (one mixed
// addition per member and window, the sign folded into the point), then sums its buckets with the running-sum trick;
// k_secure_combine folds the 32 window sums (8 doublings + 1 addition each).  Per member of a 400-key set:
// 32 x (11 + 2 x 127 x 16 / 400) Fp multiplications in G1 ~ 680 instead of ~2,800.
//   k_secure_digits  t_m -> 32 signed base-256 digits in [-128, 127] (one byte per window), zero[m] = (t_m == 0)
constexpr int SECURE_WINDOWS = 32, SECURE_BUCKETS = 128;
// a scalar < r (8 little-endian words) as 32 signed base-256 digits in [-128, 127]; `out` is 4-byte aligned
__device__ __forceinline__ void signed_digits_256(int8_t* out, const uint32_t t[8]) {
  int carry = 0;
  uint32_t* o = reinterpret_cast<uint32_t*>(out);
#pragma unroll
  for (int w8 = 0; w8 < 8; w8++) {
    uint32_t pk = 0;
#pragma unroll
    for (int k = 0; k < 4; k++) {
      int v = (int)((t[w8] >> (8 * k)) & 255u) + carry;
      carry = v >= 128;
      v -= carry << 8;                       // [-128, 127]; the top digit stays below 128 because t < r < 2^255
      pk |= ((uint32_t)v & 255u) << (8 * k);
    }
    o[w8] = pk;
  }
}
__global__ void __launch_bounds__(128) k_secure_digits(size_t M, const uint32_t* __restrict__ set_of, const uint32_t* __restrict__ pos,
                                                       const Digest* __restrict__ base, int8_t* __restrict__ digits, uint8_t* __restrict__ zero) {
  size_t m = BLS_TID();
  if (m >= M) return;
  uint32_t t[8];
  Digest b = base[set_of[m]];
  zero[m] = secure_coefficient(t, pos[m], b) ? 0 : 1;
  signed_digits_256(digits + m * SECURE_WINDOWS, t);
}
// one warp per key set (warp-stride loop), lane = window.  src[m] = index of member m's point (sorted position -> point);
// buckets: scratch of SECURE_BUCKETS Jacobian points per resident lane; W[set * 32 + lane] = the window's sum.
template <class A>
__global__ void __launch_bounds__(128, BLS_MSM_MIN_BLOCKS) k_secure_msm(size_t q, const uint64_t* __restrict__ key_off, const uint32_t* __restrict__ src,
                                                    const int8_t* __restrict__ digits, const A* __restrict__ points,
                                                    typename PtInfo<A>::Jac* __restrict__ buckets, typename PtInfo<A>::Jac* __restrict__ W) {
  typedef typename PtInfo<A>::Jac J;
  const int lane = threadIdx.x & 31;
  const size_t warp = (size_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5), nwarps = (size_t)gridDim.x * (blockDim.x >> 5);
  J* mine = buckets + (warp * 32 + lane) * SECURE_BUCKETS;
  for (size_t set = warp; set < q; set += nwarps) {
    uint32_t full[SECURE_BUCKETS / 32] = {0, 0, 0, 0};  // which buckets hold a point (no initialisation pass over memory)
    const size_t lo = (size_t)key_off[set], hi = (size_t)key_off[set + 1];
    for (size_t m = lo; m < hi; m++) {
      const int d = digits[m * SECURE_WINDOWS + lane];
      if (d == 0) continue;
      A p = points[src[m]];
      if (p.inf) continue;
      if (d < 0) aff_neg(p, p);
      const int b = (d < 0 ? -d : d) - 1;
      J acc;
      if ((full[b >> 5] >> (b & 31)) & 1u) {
        acc = mine[b];
        jac_add_mixed(acc, acc, p);
      } else {
        jac_from_aff(acc, p);
        full[b >> 5] |= 1u << (b & 31);
      }
      mine[b] = acc;
    }
    // sum_b (b + 1) * bucket[b] by running sums from the top
    J run, tot;
    jac_set_inf(run);
    jac_set_inf(tot);
    bool any = false;
    for (int b = SECURE_BUCKETS - 1; b >= 0; b--) {
      if ((full[b >> 5] >> (b & 31)) & 1u) {
        J t = mine[b];
        jac_add(run, run, t);
        any = true;
      }
      if (any) jac_add(tot, tot, run);
    }
    W[set * SECURE_WINDOWS + lane] = tot;
  }
}
// sum_w 2^(8w) W[w] per key set (Horner from the top window)
template <class J>
__global__ void __launch_bounds__(128, BLS_MIN_BLOCKS) k_secure_combine(size_t q, const J* __restrict__ W, J* __restrict__ out) {
  size_t set = BLS_TID();
  if (set >= q) return;
  J acc = W[set * SECURE_WINDOWS + SECURE_WINDOWS - 1];
  for (int w = SECURE_WINDOWS - 2; w >= 0; w--) {
    if (!jac_is_inf(acc))
      for (int k = 0; k < 8; k++) jac_dbl(acc, acc);
    J t = W[set * SECURE_WINDOWS + w];
    jac_add(acc, acc, t);
  }
  out[set] = acc;
}
// keyed secure aggregation: the plan make_secure_plan (blsgpu.cu) builds on the host, built per quorum on the device from
// the dense byte-order ranks of a key set's secure view.  One block per quorum j with members key_idx[lo..hi):
//   keyst[j]  the set status of its first bad key in member order (ST_OK if none), for every quorum;
//   and for quorums of at most `slots` members (the host plans the others): (rank, member position) sorted in shared
//   memory, ties by position = the reference's stable sort on the byte strings.  Sorted member i (lo <= i < hi) gets
//   ord[i] = its key's SET index, set_of[i] = j, pos[i] = i - lo, first[i] = the member index of the first member of its
//   equal-rank run (the first match of duplicate keys, secure_aggregation.rs:140-147).
// slots: a power of two, the dynamic shared memory is slots 64-bit words.
__global__ void __launch_bounds__(256) k_secure_plan_keyed(size_t q, const uint64_t* __restrict__ key_off, const uint32_t* __restrict__ key_idx,
                                                           const uint32_t* __restrict__ rank, const uint8_t* __restrict__ set_st, uint32_t slots,
                                                           uint32_t* __restrict__ ord, uint32_t* __restrict__ set_of, uint32_t* __restrict__ pos,
                                                           uint32_t* __restrict__ first, uint8_t* __restrict__ keyst) {
  extern __shared__ unsigned long long srt[];
  __shared__ uint32_t bad;
  const size_t j = blockIdx.x;
  if (j >= q) return;
  const uint64_t lo = key_off[j];
  const uint32_t cnt = (uint32_t)(key_off[j + 1] - lo);
  if (threadIdx.x == 0) bad = 0xffffffffu;
  __syncthreads();
  for (uint32_t p = threadIdx.x; p < cnt; p += blockDim.x)
    if (set_st[key_idx[lo + p]] != ST_OK) atomicMin(&bad, p);
  __syncthreads();
  if (threadIdx.x == 0) keyst[j] = bad == 0xffffffffu ? (uint8_t)ST_OK : set_st[key_idx[lo + bad]];
  if (cnt > slots) return;
  uint32_t N = 1;
  while (N < cnt) N <<= 1;
  for (uint32_t t = threadIdx.x; t < N; t += blockDim.x)  // ranks are below 2^32 - 16: the padding sorts last
    srt[t] = t < cnt ? ((unsigned long long)rank[key_idx[lo + t]] << 32) | t : ~0ull;
  __syncthreads();
  for (uint32_t k = 2; k <= N; k <<= 1)  // bitonic sort, ascending
    for (uint32_t h = k >> 1; h > 0; h >>= 1) {
      for (uint32_t t = threadIdx.x; t < N; t += blockDim.x) {
        const uint32_t u = t ^ h;
        if (u > t) {
          const unsigned long long a = srt[t], b = srt[u];
          if ((a > b) == ((t & k) == 0)) {
            srt[t] = b;
            srt[u] = a;
          }
        }
      }
      __syncthreads();
    }
  for (uint32_t t = threadIdx.x; t < cnt; t += blockDim.x) {
    const unsigned long long v = srt[t];
    const uint32_t r = (uint32_t)(v >> 32);
    uint32_t a = 0, b = t;  // the start of t's equal-rank run: the lowest member position of that rank
    while (a < b) {
      const uint32_t m = (a + b) >> 1;
      if ((uint32_t)(srt[m] >> 32) < r)
        a = m + 1;
      else
        b = m;
    }
    ord[lo + t] = key_idx[lo + (uint32_t)v];
    set_of[lo + t] = (uint32_t)j;
    pos[lo + t] = t;
    first[lo + t] = (uint32_t)lo + (uint32_t)srt[a];
  }
}

// ---- threshold-share combination (vsss-rs `combine` behind Signature::from_shares / PublicKey::from_shares) ------------
// identifiers: 32 big-endian bytes -> raw words; flag 1: >= r (DeserializationError), 2: zero (VsssError)
__global__ void __launch_bounds__(128) k_share_ids(size_t M, const uint8_t* __restrict__ ids_be, uint32_t* __restrict__ ids_raw, uint8_t* __restrict__ flag) {
  size_t i = BLS_TID();
  if (i >= M) return;
  uint8_t b[32];
  for (int k = 0; k < 32; k++) b[k] = ids_be[i * 32 + k];
  uint32_t w[8];
  fr_raw_from_be32(w, b);
  uint32_t any = 0;
  for (int k = 0; k < 8; k++) any |= w[k];
  uint8_t f = fr_raw_ge_r(w) ? 1 : any == 0 ? 2 : 0;
  if (f == 1)
    for (int k = 0; k < 8; k++) w[k] = 0;
  for (int k = 0; k < 8; k++) ids_raw[i * 8 + k] = w[k];
  flag[i] = f;
}
// one thread per share: its Lagrange coefficient at zero within its set as signed window digits for k_secure_msm (all zero
// for sets the host flagged bad and for duplicate identifiers, which set dup[i] = 1)
__global__ void __launch_bounds__(128, BLS_MIN_BLOCKS) k_share_digits(size_t M, const uint32_t* __restrict__ set_of, const uint64_t* __restrict__ share_off,
                                                      const uint8_t* __restrict__ bad, const uint32_t* __restrict__ ids_raw,
                                                      int8_t* __restrict__ digits, uint8_t* __restrict__ dup) {
  size_t i = BLS_TID();
  if (i >= M) return;
  uint32_t lam[8] = {0, 0, 0, 0, 0, 0, 0, 0};
  uint8_t d = 0;
  const uint32_t s = set_of[i];
  if (!bad[s]) {
    const uint64_t lo = share_off[s], hi = share_off[s + 1];
    if (!fr_lagrange_at_zero(lam, ids_raw + 8 * lo, (uint32_t)(hi - lo), (uint32_t)(i - lo))) {
      d = 1;
      for (int k = 0; k < 8; k++) lam[k] = 0;
    }
  }
  dup[i] = d;
  signed_digits_256(digits + i * SECURE_WINDOWS, lam);
}

// ---- building blocks ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(128, BLS_MIN_BLOCKS) k_fp_mul(size_t n, int variant, const uint8_t* a, const uint8_t* b, uint8_t* out) {
  size_t i = BLS_TID();
  if (i >= n) return;
  uint8_t ba[48], bb[48];
  for (int k = 0; k < 48; k++) {
    ba[k] = a[i * 48 + k];
    bb[k] = b[i * 48 + k];
  }
  Fp ra, rb, x, y, z;
  fp_from_be48_raw(ra, ba);
  fp_from_be48_raw(rb, bb);
  fp_to_mont(x, ra);
  fp_to_mont(y, rb);
  if (variant == 0)
    fp_mul_inl(z, x, y);
  else if (variant == 1)
    fp_mul(z, x, y);
  else
    fp_sqr_inl(z, x);
  fp_from_mont(ra, z);
  fp_to_be48_raw(ba, ra);
  for (int k = 0; k < 48; k++) out[i * 48 + k] = ba[k];
}

// Miller loop of decoded (G1, G2) pairs (no scaling)
__global__ void __launch_bounds__(128, BLS_MIN_BLOCKS) k_miller_pairs(size_t n, const G1Aff* p, const G2Aff* q, Fp12* out) {
  size_t i = BLS_TID();
  if (i >= n) return;
  Fp12 f;
  G1Aff a = p[i];
  G2Aff b = q[i];
  if (a.inf || b.inf) {
    fp12_one(f);
  } else {
    MillerG1 mp;
    miller_prepare(mp, a);
    miller_loop(f, mp, b);
  }
  out[i] = f;
}
// per set: product of its Miller values, final exponentiation, == 1 ?   (one thread per set)
__global__ void __launch_bounds__(64) k_set_final_is_one(size_t q, const uint64_t* __restrict__ off, const Fp12* __restrict__ F,
                                                         uint8_t* __restrict__ ok) {
  size_t j = BLS_TID();
  if (j >= q) return;
  Fp12 acc;
  fp12_one(acc);
  for (uint64_t i = off[j]; i < off[j + 1]; i++) {
    Fp12 t = F[i];
    fp12_mul(acc, acc, t);
  }
  Fp12 e;
  final_exponentiation(e, acc);
  ok[j] = fp12_is_one(e) ? 1 : 0;
}
__global__ void k_final_is_one(const Fp12* f, uint8_t* ok) {
  if (BLS_TID() != 0) return;
  Fp12 g = f[0], e;
  final_exponentiation(e, g);
  ok[0] = fp12_is_one(e) ? 1 : 0;
}

// ---- partial results of a batch cut over several devices / processes (SURVEY.md section 8e) --------------------------------
// 576-byte form of an Fp12: the coefficients of w^0 .. w^5, each as c0 || c1 in 48-byte big-endian canonical form
__global__ void k_fp12_to_bytes(size_t n, const Fp12* __restrict__ in, uint8_t* __restrict__ out) {
  size_t t = BLS_TID();
  if (t >= 6 * n) return;
  Fp12 f = in[t / 6];
  const Fp2 c = *fp12_coeff(f, (int)(t % 6));
  Fp raw;
  uint8_t b[48];
  fp_from_mont(raw, c.c0);
  fp_to_be48_raw(b, raw);
  for (int k = 0; k < 48; k++) out[96 * t + k] = b[k];
  fp_from_mont(raw, c.c1);
  fp_to_be48_raw(b, raw);
  for (int k = 0; k < 48; k++) out[96 * t + 48 + k] = b[k];
}
// One thread per field element (12 per value); bad[i] = 1 if some coefficient of value i is not canonical.
// (The first version built the value in a local Fp12 and assigned each Fp2 through `*fp12_coeff(f, k) = c`; cicc 12.9
// compiled the final `out[i] = f` to THREE 32-bit stores - tools/repro/cicc_struct_copy_repro.cu, DESIGN.md section 9.
// Rule for this code base: never assign a multi-member aggregate through a pointer chosen at run time.)
__global__ void k_fp12_from_bytes(size_t n, const uint8_t* __restrict__ in, Fp12* __restrict__ out, uint8_t* __restrict__ bad) {
  size_t t = BLS_TID();
  if (t >= 12 * n) return;
  const size_t i = t / 12;
  const int k = (int)((t % 12) >> 1), h = (int)(t & 1);
  uint8_t b[48];
  for (int j = 0; j < 48; j++) b[j] = in[576 * i + 96 * k + 48 * h + j];
  uint8_t flag = (b[0] & 0xe0) ? 1 : 0;
  b[0] &= 0x1f;
  Fp raw, m;
  if (!fp_from_be48_raw(raw, b)) flag = 1;
  fp_to_mont(m, raw);
  Fp2* c = fp12_coeff(out[i], k);
  if (h) c->c1 = m; else c->c0 = m;
  if (flag) bad[i] = 1;  // bad[] is zeroed by the caller
}
// affine -> Jacobian (the partial sums of the slices arrive as compressed points)
template <class A>
__global__ void k_aff_to_jac(size_t n, const A* __restrict__ in, typename PtInfo<A>::Jac* __restrict__ out) {
  size_t i = BLS_TID();
  if (i >= n) return;
  A a = in[i];
  typename PtInfo<A>::Jac j;
  jac_from_aff(j, a);
  out[i] = j;
}

// ---- the reference's other public 2-pairing checks (SURVEY.md section 8f-4) ---------------------------------------------
// Every item becomes two (G1, G2) pairs at 2i, 2i + 1; k_miller_pairs + k_set_final_is_one decide prod e(.,.) == 1 per item.
__device__ __forceinline__ void put_pair(G1Aff* g1, G2Aff* g2, size_t idx, const G1Aff& a, const G2Aff& b) {
  g1[idx] = a;
  g2[idx] = b;
}
__device__ __forceinline__ void put_pair(G1Aff* g1, G2Aff* g2, size_t idx, const G2Aff& b, const G1Aff& a) { put_pair(g1, g2, idx, a, b); }
// 32 big-endian bytes -> 8 little-endian words
__device__ __forceinline__ void scalar_words_be32(uint32_t k[8], const uint8_t* b) {
  for (int w = 0; w < 8; w++) {
    const uint8_t* q = b + 28 - 4 * w;
    k[w] = ((uint32_t)q[0] << 24) | ((uint32_t)q[1] << 16) | ((uint32_t)q[2] << 8) | q[3];
  }
}
// ProofOfKnowledge::verify (reference src/traits/sig_proof.rs:102-142): status before the pairing, in the reference's order.
// yflag: 0 fine, 1 not a canonical scalar (parse error), 2 zero
template <class PkA, class SigA>
__global__ void k_pok_prestatus(size_t n, const uint8_t* st_cm, const uint8_t* st_pr, const uint8_t* st_pk, const uint8_t* yflag,
                                const SigA* cm, const SigA* pr, const PkA* pk, uint8_t* out) {
  size_t i = BLS_TID();
  if (i >= n) return;
  uint8_t s = st_cm[i];
  if (s == ST_OK) s = st_pr[i];
  if (s == ST_OK) s = st_pk[i];
  if (s == ST_OK && yflag[i] == 1) s = ST_DESERIALIZE;
  if (s == ST_OK && cm[i].inf) s = ST_COMMITMENT_IDENTITY;
  if (s == ST_OK && pr[i].inf) s = ST_PROOF_IDENTITY;
  if (s == ST_OK && pk[i].inf) s = ST_PK_IDENTITY;
  if (s == ST_OK && yflag[i] == 2) s = ST_ZERO_CHALLENGE;
  out[i] = s;
}
// pairs of item i: (proof, g), (commitment + [y] a, pk)   with a = hash_to_point(msg)   (sig_proof.rs:130-136)
template <class PkA, class SigA>
__global__ void __launch_bounds__(128, BLS_MIN_BLOCKS) k_pok_pairs(size_t n, const uint8_t* __restrict__ pre, const SigA* __restrict__ a,
                                                   const SigA* __restrict__ cm, const SigA* __restrict__ pr, const PkA* __restrict__ pk,
                                                   const uint8_t* __restrict__ y_be32, G1Aff* __restrict__ g1, G2Aff* __restrict__ g2) {
  size_t i = BLS_TID();
  if (i >= n) return;
  PkA gen, key;
  SigA proof, target;
  if (pre[i] != ST_OK) {  // identity pairs: the product is 1, the status already says why the item failed
    pt_set_inf(gen);
    pt_set_inf(key);
    pt_set_inf(proof);
    pt_set_inf(target);
  } else {
    uint32_t k[8];
    scalar_words_be32(k, y_be32 + 32 * i);
    SigA h = a[i], c = cm[i];
    typename PtInfo<SigA>::Jac t;
    jac_mul_aff(t, h, k, 8);
    jac_add_mixed(t, t, c);
    jac_to_aff(target, t);
    pt_generator(gen);
    key = pk[i];
    proof = pr[i];
  }
  put_pair(g1, g2, 2 * i, gen, proof);
  put_pair(g1, g2, 2 * i + 1, key, target);
}
// BlsSignCrypt::verify_share (reference src/traits/sign_crypt.rs:192-207): pairs (-W', share), (w, pk); flag = 0 if share, pk
// or w is the identity (the check is then false without a pairing)
template <class PkA, class SigA>
__global__ void __launch_bounds__(128, BLS_MIN_BLOCKS) k_signcrypt_share_pairs(size_t n, const uint8_t* __restrict__ pre, const SigA* __restrict__ wt,
                                                               const PkA* __restrict__ share, const PkA* __restrict__ pk,
                                                               const SigA* __restrict__ w, G1Aff* __restrict__ g1, G2Aff* __restrict__ g2,
                                                               uint8_t* __restrict__ flag) {
  size_t i = BLS_TID();
  if (i >= n) return;
  PkA s, k;
  SigA h, ww;
  uint8_t f = 0;
  if (pre[i] == ST_OK) {
    s = share[i];
    k = pk[i];
    ww = w[i];
    h = wt[i];
    f = !(s.inf || k.inf || ww.inf);
  }
  if (!f) {
    pt_set_inf(s);
    pt_set_inf(k);
    pt_set_inf(h);
    pt_set_inf(ww);
  } else {
    aff_neg(h, h);
  }
  put_pair(g1, g2, 2 * i, s, h);
  put_pair(g1, g2, 2 * i + 1, k, ww);
  flag[i] = f;
}
__global__ void k_pair_offsets(size_t q, uint64_t* off) {  // off[j] = 2 j, j = 0..q
  size_t j = BLS_TID();
  if (j <= q) off[j] = 2 * j;
}
// status / ok from the pairing results: PoK: ok ? OK : INVALID_PROOF (keeping earlier statuses)
__global__ void k_pok_finish(size_t n, const uint8_t* ok, uint8_t* status) {
  size_t i = BLS_TID();
  if (i >= n) return;
  if (status[i] == ST_OK && !ok[i]) status[i] = ST_INVALID_PROOF;
}
__global__ void k_and_flags(size_t n, const uint8_t* flag, uint8_t* ok) {
  size_t i = BLS_TID();
  if (i >= n) return;
  ok[i] = ok[i] && flag[i];
}

// ---- many aggregate signatures in one call (blsgpu_aggregate_verify_batch) ------------------------------------------------
// Aggregate j owns pairs set_off[j] .. set_off[j+1]-1 and whole Miller groups of slots: its pairs are copied to slots, the
// rest of its last group is padding (status "skip"), so no group straddles two aggregates.  One scalar r_j per aggregate.
//
// leaves of the digest that binds the scalars: one per pair (pk_i, H_i), then one per aggregate (sig_j, its pair range)
template <class PkA, class SigA>
__global__ void __launch_bounds__(128, BLS_MIN_BLOCKS) k_agg_leaf_digest(size_t np, size_t q, const PkA* __restrict__ pk, const SigA* __restrict__ h,
                                                         const SigA* __restrict__ sig, const uint64_t* __restrict__ set_off,
                                                         Digest* __restrict__ out) {
  const size_t t = BLS_TID();
  if (t >= np + q) return;
  Sha256 s;
  sha256_init(s);
  if (t < np) {
    digest_point(s, pk[t]);
    digest_point(s, h[t]);
  } else {
    const size_t j = t - np;
    digest_point(s, sig[j]);
    uint8_t b[16];
    for (int k = 0; k < 8; k++) {
      b[k] = (uint8_t)(set_off[j] >> (8 * k));
      b[8 + k] = (uint8_t)(set_off[j + 1] >> (8 * k));
    }
    sha256_update(s, b, 16);
  }
  Digest d;
  sha256_final(s, d.b);
  out[t] = d;
}
// slot s <- pair src[s]; src[s] == 0xffffffff: padding or an aggregate decided before the pairing (skipped)
template <class PkA, class SigA>
__global__ void __launch_bounds__(128, BLS_MIN_BLOCKS) k_agg_slots(size_t nslots, const uint32_t* __restrict__ src, const PkA* __restrict__ pk,
                                                   const SigA* __restrict__ h, PkA* __restrict__ pk_s, SigA* __restrict__ h_s,
                                                   uint8_t* __restrict__ pre_s) {
  const size_t s = BLS_TID();
  if (s >= nslots) return;
  const uint32_t i = src[s];
  if (i == 0xffffffffu) {
    pre_s[s] = PROBE_SKIP;
    return;
  }
  pk_s[s] = pk[i];
  h_s[s] = h[i];
  pre_s[s] = ST_OK;
}
// k_m6_prep with the scalar of the slot's AGGREGATE: r_{set(i)} = rlc_scalar(root, g_set[i / 6])
template <class PkA, class HA>
__global__ void __launch_bounds__(128, BLS_MIN_BLOCKS) k_m6_prep_sets(size_t n, size_t base, const PkA* __restrict__ pk, const HA* __restrict__ h,
                                                      const uint8_t* __restrict__ pre, const uint32_t* __restrict__ g_set,
                                                      const Digest* __restrict__ root, int rbits, M6Arg* __restrict__ args) {
  size_t c = BLS_TID();
  if (c >= n) return;
  const size_t i = base + c;
  if (pre[i] != ST_OK) return;
  G1Aff p = m6_g1(pk, h, i);
  uint32_t sc[RLC_MAX_WORDS];
  rlc_scalar(sc, root, g_set[i / M6_GROUP], rbits);
  G1Jac pj;
  jac_mul_aff_w4(pj, p, sc, rbits / 4);
  MillerG1 mp;
  miller_prepare(mp, pj);
  M6Arg a;
  const G2Aff q = m6_g2(pk, h, i);
  m6_make_arg(a, mp, q);
  args[c] = a;
}
// One level of the segmented product: out[j] = prod in[off[j] .. off[j+1]), ranges of at most 16 consecutive nodes of one
// aggregate.  A thread per output node, or (_w, for levels with few nodes) sixteen lanes per node as in k_reduce_fp12_w.
__global__ void __launch_bounds__(128, BLS_MIN_BLOCKS) k_seg_reduce_fp12(size_t n_out, const uint32_t* __restrict__ off, const Fp12* __restrict__ in,
                                                         Fp12* __restrict__ out) {
  const size_t j = BLS_TID();
  if (j >= n_out) return;
  const uint32_t lo = off[j], hi = off[j + 1];
  Fp12 acc = in[lo];
  for (uint32_t m = lo + 1; m < hi; m++) {
    Fp12 t = in[m];
    fp12_mul(acc, acc, t);
  }
  out[j] = acc;
}
__global__ void __launch_bounds__(128, BLS_MIN_BLOCKS) k_seg_reduce_fp12_w(size_t n_out, const uint32_t* __restrict__ off, const Fp12* __restrict__ in,
                                                           Fp12* __restrict__ out) {
  const size_t t = BLS_TID(), j = t >> 4;
  const int m = (int)(t & 15);
  Fp12 acc;
  if (j < n_out && off[j] + m < off[j + 1]) acc = in[off[j] + m]; else fp12_one(acc);
#pragma unroll 1
  for (int s = 1; s < 16; s <<= 1) {
    Fp12 other;
    words_shfl_xor(other, acc, s);
    if ((m & (2 * s - 1)) == 0) fp12_mul(acc, acc, other);
  }
  if (j < n_out && m == 0) out[j] = acc;
}

// ---- segmented point sums (blsgpu_verify_multisig_batch[_keyed], blsgpu_sum_points_batch) --------------------------------------
// The first level: a thread per CHUNK of at most 16 consecutive members of one set (members coff[c] .. coff[c+1]-1 of set
// cset[c]; a chunk of an empty set has none and gives the identity).  Member m's point is pts[idx[m]] (members named by index
// into a key set) or pts[m] (idx null: points decoded in member order); a point that failed to decode is the identity there
// (k_decode / k_subgroup_check), so it adds nothing.  The same pass finds each set's first member whose status is not OK:
// first_bad[set] = min over such members of (m << 8 | status), ~0 where there is none.
template <class A>
__global__ void __launch_bounds__(128, BLS_MIN_BLOCKS) k_seg_sum_gather(size_t nchunks, const uint32_t* __restrict__ coff,
                                                        const uint32_t* __restrict__ cset, const uint32_t* __restrict__ idx,
                                                        const A* __restrict__ pts, const uint8_t* __restrict__ st,
                                                        typename PtInfo<A>::Jac* __restrict__ out, unsigned long long* __restrict__ first_bad) {
  const size_t c = BLS_TID();
  if (c >= nchunks) return;
  const uint32_t lo = coff[c], hi = coff[c + 1];
  typename PtInfo<A>::Jac acc;
  jac_set_inf(acc);
  unsigned long long bad = ~0ull;
  for (uint32_t m = lo; m < hi; m++) {
    const uint32_t k = idx ? idx[m] : m;
    const uint8_t s = st[k];
    if (s != ST_OK && bad == ~0ull) bad = ((unsigned long long)m << 8) | s;
    A p = pts[k];
    jac_add_mixed(acc, acc, p);
  }
  out[c] = acc;
  if (bad != ~0ull) atomicMin(first_bad + cset[c], bad);
}
// per set: the status of its first member that failed to decode (k_seg_sum_gather), or OK
__global__ void k_seg_first_bad_status(size_t q, const unsigned long long* __restrict__ first_bad, uint8_t* __restrict__ st) {
  const size_t j = BLS_TID();
  if (j >= q) return;
  const unsigned long long b = first_bad[j];
  st[j] = b == ~0ull ? (uint8_t)ST_OK : (uint8_t)(b & 0xff);
}
// One level of the segmented sum: out[j] = sum in[off[j] .. off[j+1]), the Jacobian twins of k_seg_reduce_fp12 / _w.
template <class J>
__global__ void __launch_bounds__(128, BLS_MIN_BLOCKS) k_seg_reduce_jac(size_t n_out, const uint32_t* __restrict__ off, const J* __restrict__ in,
                                                        J* __restrict__ out) {
  const size_t j = BLS_TID();
  if (j >= n_out) return;
  const uint32_t lo = off[j], hi = off[j + 1];
  J acc = in[lo];
  for (uint32_t m = lo + 1; m < hi; m++) {
    J t = in[m];
    jac_add(acc, acc, t);
  }
  out[j] = acc;
}
template <class J>
__global__ void __launch_bounds__(128, BLS_MIN_BLOCKS) k_seg_reduce_jac_w(size_t n_out, const uint32_t* __restrict__ off, const J* __restrict__ in,
                                                          J* __restrict__ out) {
  const size_t t = BLS_TID(), j = t >> 4;
  const int m = (int)(t & 15);
  J acc;
  if (j < n_out && off[j] + m < off[j + 1]) acc = in[off[j] + m]; else jac_set_inf(acc);
#pragma unroll 1
  for (int s = 1; s < 16; s <<= 1) {
    J other;
    words_shfl_xor(other, acc, s);
    if ((m & (2 * s - 1)) == 0) jac_add(acc, acc, other);
  }
  if (j < n_out && m == 0) out[j] = acc;
}

// ---- signatures over shared messages (blsgpu_verify_batch_grouped) --------------------------------------------------------
// The host counting-sorts the items by message (order[]) and cuts every message's run into LEAVES of at most
// GROUPED_LEAF consecutive entries of order[].  The Miller stage runs over the leaves: ML(P_l, H_l) with
// P_l = sum_{i in l} r_i pk_i, since prod_{i in l} e(r_i pk_i, H) = e(P_l, H) when every item of l signs H.
struct GLeaf {
  uint32_t first, count, msg;  // order[first .. first + count) sign message `msg`
};
// leaf digest of item i: pk_i, sig_i, the hash of its message and the message's index (binds the grouping into the scalars)
template <class PkA, class SigA>
__global__ void __launch_bounds__(128, BLS_MIN_BLOCKS) k_grouped_leaf_digest(size_t n, const PkA* __restrict__ pk, const SigA* __restrict__ sig,
                                                             const SigA* __restrict__ hq, const uint32_t* __restrict__ msg_idx,
                                                             Digest* __restrict__ out) {
  size_t i = BLS_TID();
  if (i >= n) return;
  const uint32_t m = msg_idx[i];
  Sha256 s;
  sha256_init(s);
  digest_point(s, pk[i]);
  digest_point(s, sig[i]);
  digest_point(s, hq[m]);
  const uint8_t b[4] = {(uint8_t)m, (uint8_t)(m >> 8), (uint8_t)(m >> 16), (uint8_t)(m >> 24)};
  sha256_update(s, b, 4);
  Digest d;
  sha256_final(s, d.b);
  out[i] = d;
}
// window w (4 bits) of a 64- or 128-bit scalar
__device__ __forceinline__ uint32_t rlc_nibble(const RlcScalar& k, int w) {
  return (uint32_t)(w < 16 ? k.lo >> (4 * w) : k.hi >> (4 * (w - 16))) & 15u;
}
// Sum_{i in leaf} r_i * pts[i] for the listed leaves, ONE WARP per leaf (warp-stride loop): lane = (4-bit window w, part of
// the leaf).  64-bit scalars: 16 windows x 2 halves of the leaf's items; 128-bit: 32 windows, each lane over every item.
// Every lane drops its items into 15 buckets by its digit (one mixed addition each), then sums the buckets by running sums;
// W[c * 32 + lane] = that window sum, folded by k_leaf_combine.  Items with r_i = 0 (status not OK) add nothing.
// Per item of a full 96-item leaf ~ 26 point operations in lane-time against ~90 for r_i * P on its own (k_leaf_scale).
constexpr int LEAF_BUCKETS = 15;
template <class A>
__global__ void __launch_bounds__(128, BLS_MIN_BLOCKS) k_leaf_msm(size_t cnt, const uint32_t* __restrict__ list, const GLeaf* __restrict__ leaves,
                                                  const uint32_t* __restrict__ order, const A* __restrict__ pts,
                                                  const RlcScalar* __restrict__ r, int rbits, typename PtInfo<A>::Jac* __restrict__ buckets,
                                                  typename PtInfo<A>::Jac* __restrict__ W) {
  typedef typename PtInfo<A>::Jac J;
  const int nwin = rbits / 4, parts = 32 / nwin;
  const int lane = threadIdx.x & 31, w = lane % nwin, part = lane / nwin;
  const size_t warp = (size_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5), nwarps = (size_t)gridDim.x * (blockDim.x >> 5);
  J* mine = buckets + (warp * 32 + lane) * LEAF_BUCKETS;
  for (size_t c = warp; c < cnt; c += nwarps) {
    const GLeaf lf = leaves[list[c]];
    uint32_t full = 0;
    for (uint32_t t = part; t < lf.count; t += parts) {
      const uint32_t i = order[lf.first + t];
      const uint32_t d = rlc_nibble(r[i], w);
      if (d == 0) continue;
      A p = pts[i];
      J acc;
      if ((full >> (d - 1)) & 1u) {
        acc = mine[d - 1];
        jac_add_mixed(acc, acc, p);
      } else {
        jac_from_aff(acc, p);
        full |= 1u << (d - 1);
      }
      mine[d - 1] = acc;
    }
    J run, tot;
    jac_set_inf(run);
    jac_set_inf(tot);
    bool any = false;
    for (int b = LEAF_BUCKETS - 1; b >= 0; b--) {
      if ((full >> b) & 1u) {
        J t = mine[b];
        jac_add(run, run, t);
        any = true;
      }
      if (any) jac_add(tot, tot, run);
    }
    W[c * 32 + lane] = tot;
  }
}
// out[list[c]] = sum_w 16^w (sum over the parts of W[c * 32 + part * nwin + w])
template <class J>
__global__ void __launch_bounds__(128, BLS_MIN_BLOCKS) k_leaf_combine(size_t cnt, const uint32_t* __restrict__ list, int rbits, const J* __restrict__ W,
                                                      J* __restrict__ out) {
  size_t c = BLS_TID();
  if (c >= cnt) return;
  const int nwin = rbits / 4, parts = 32 / nwin;
  J acc;
  jac_set_inf(acc);
  for (int w = nwin - 1; w >= 0; w--) {
    if (!jac_is_inf(acc))
      for (int k = 0; k < 4; k++) jac_dbl(acc, acc);
    for (int p = 0; p < parts; p++) {
      J t = W[c * 32 + p * nwin + w];
      jac_add(acc, acc, t);
    }
  }
  out[list[c]] = acc;
}
// the same sum for leaves too small for a warp's buckets to pay: one thread per leaf, r_i * pts[i] per item, then the sum
template <class A>
__global__ void __launch_bounds__(128, BLS_MIN_BLOCKS) k_leaf_scale(size_t cnt, const uint32_t* __restrict__ list, const GLeaf* __restrict__ leaves,
                                                    const uint32_t* __restrict__ order, const A* __restrict__ pts,
                                                    const RlcScalar* __restrict__ r, int rbits, typename PtInfo<A>::Jac* __restrict__ out) {
  typedef typename PtInfo<A>::Jac J;
  size_t c = BLS_TID();
  if (c >= cnt) return;
  const GLeaf lf = leaves[list[c]];
  J acc;
  jac_set_inf(acc);
  for (uint32_t t = 0; t < lf.count; t++) {
    const uint32_t i = order[lf.first + t];
    const RlcScalar k = r[i];
    if ((k.lo | k.hi) == 0) continue;
    const uint32_t kw[RLC_MAX_WORDS] = {(uint32_t)k.lo, (uint32_t)(k.lo >> 32), (uint32_t)k.hi, (uint32_t)(k.hi >> 32)};
    A p = pts[i];
    J pj;
    jac_mul_aff_w4(pj, p, kw, rbits / 4);
    jac_add(acc, acc, pj);
  }
  out[list[c]] = acc;
}
// per leaf: H_l = H of its message, and the Miller stage's status (P_l = O adds e(O, H) = 1: skipped)
template <class PkA, class HA>
__global__ void __launch_bounds__(128, BLS_MIN_BLOCKS) k_leaf_gather(size_t nl, const GLeaf* __restrict__ leaves, const PkA* __restrict__ p,
                                                     const HA* __restrict__ hq, HA* __restrict__ h_leaf, uint8_t* __restrict__ pre) {
  size_t l = BLS_TID();
  if (l >= nl) return;
  h_leaf[l] = hq[leaves[l].msg];
  pre[l] = p[l].inf ? PROBE_SKIP : ST_OK;
}
// k_probe_fill_leaves for items whose hash is that of their message: H_i = hq[msg_idx[i]]
template <class PkA, class SigA>
__global__ void __launch_bounds__(128, BLS_MIN_BLOCKS) k_probe_fill_grouped(size_t cnt, const uint32_t* __restrict__ idx, const PkA* __restrict__ pk,
                                                            const uint32_t* __restrict__ msg_idx, const SigA* __restrict__ hq,
                                                            const SigA* __restrict__ sig, const uint8_t* __restrict__ status,
                                                            PkA* __restrict__ xpk, SigA* __restrict__ xh, uint8_t* __restrict__ xpre) {
  size_t c = BLS_TID();
  if (c >= cnt) return;
  const size_t i = idx[c];
  const bool on = status[i] == ST_OK;
  if (on) {
    PkA ng;
    pt_generator(ng);
    aff_neg(ng, ng);
    xpk[6 * c] = pk[i];
    xh[6 * c] = hq[msg_idx[i]];
    xpk[6 * c + 1] = ng;
    xh[6 * c + 1] = sig[i];
  }
  xpre[6 * c] = xpre[6 * c + 1] = on ? ST_OK : PROBE_SKIP;
  for (int m = 2; m < 6; m++) xpre[6 * c + m] = PROBE_SKIP;
}

// synthetic data: pk = [k]G, sig = [k]H(frame(msg))
template <class PkA, class SigA>
__global__ void __launch_bounds__(128, BLS_MIN_BLOCKS) k_testdata_sign(size_t n, const uint8_t* scalars, const uint8_t* msgs, const uint64_t* msg_off,
                                                       int msg_mode, DstParam dst, uint8_t* out_pk, uint8_t* out_sig) {
  size_t i = BLS_TID();
  if (i >= n) return;
  uint32_t k[8];
  for (int w = 0; w < 8; w++) {
    const uint8_t* q = scalars + i * 32 + 28 - 4 * w;
    k[w] = ((uint32_t)q[0] << 24) | ((uint32_t)q[1] << 16) | ((uint32_t)q[2] << 8) | q[3];
  }
  PkA g, pk;
  pt_generator(g);
  typename PtInfo<PkA>::Jac pj;
  jac_mul_aff(pj, g, k, 8);
  jac_to_aff(pk, pj);
  uint8_t pkb[PtInfo<PkA>::LEN];
  pt_compress(pkb, pk);
  for (int b = 0; b < PtInfo<PkA>::LEN; b++) out_pk[i * PtInfo<PkA>::LEN + b] = pkb[b];
  uint64_t o0 = msg_off[i], o1 = msg_off[i + 1];
  typename PtInfo<SigA>::Jac hj, sj;
  SigA h, s;
  hash_to_group(hj, pkb, msg_mode ? PtInfo<PkA>::LEN : 0, msgs + o0, msg_mode == 2 ? 0 : (uint32_t)(o1 - o0), dst.b, dst.len);
  jac_to_aff(h, hj);
  jac_mul_aff(sj, h, k, 8);
  jac_to_aff(s, sj);
  uint8_t sb[PtInfo<SigA>::LEN];
  pt_compress(sb, s);
  for (int b = 0; b < PtInfo<SigA>::LEN; b++) out_sig[i * PtInfo<SigA>::LEN + b] = sb[b];
}

// INT32 multiply roofline probe: 8 independent 64-bit accumulators per thread, iters*64 IMAD.WIDE.U32 each.  The operands
// change every group of 8 (a += low word of an accumulator, b += odd constant) so that neither nvcc nor ptxas can hoist
// the product out of the loop - an earlier probe with loop-invariant operands compiled to 64-bit ADDs and overstated the
// peak by 2x.  SASS check: the loop body must show 64 IMAD.WIDE.U32 per iteration (DESIGN.md section 6).
__global__ void __launch_bounds__(256) k_imad_peak(uint32_t iters, uint32_t seed, uint64_t* sink) {
  uint32_t a[8], b = seed * 3 + blockIdx.x;
  uint64_t c[8];
#pragma unroll
  for (int k = 0; k < 8; k++) {
    a[k] = seed + threadIdx.x * 8 + k;
    c[k] = a[k];
  }
  for (uint32_t it = 0; it < iters; it++) {
#pragma unroll
    for (int u = 0; u < 8; u++) {
#pragma unroll
      for (int k = 0; k < 8; k++) asm volatile("mad.wide.u32 %0, %1, %2, %0;" : "+l"(c[k]) : "r"(a[k]), "r"(b));
      b += 0x9e3779b9u;
    }
#pragma unroll
    for (int k = 0; k < 8; k++) a[k] ^= (uint32_t)c[(k + 1) & 7];
  }
  uint64_t r = 0;
#pragma unroll
  for (int k = 0; k < 8; k++) r ^= c[k];
  if (r == 0x123456789abcdefull) sink[0] = r;  // keeps the chains alive
}

}  // namespace bls
