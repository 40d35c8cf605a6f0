// C ABI of the engine (include/blsgpu.h): host orchestration of the kernels in kernels.cuh.
// No CPU arithmetic lives here: every field/curve/pairing operation runs on the device; the host only stages buffers,
// launches kernels, walks the bisection tree and applies the reference's host-side rules (duplicate messages, sorting).
#include <cuda_runtime.h>
#include <nvtx3/nvToolsExt.h>  // header-only: ranges cost nothing unless a profiler is attached (SURVEY.md section 5: tracing)
#include <sys/random.h>

#include <algorithm>
#include <atomic>
#include <functional>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <memory>
#include <mutex>
#include <string>
#include <unordered_map>
#include <thread>
#include <vector>

#include "../../include/blsgpu.h"
#include "kernels.cuh"

using namespace bls;

namespace {

thread_local std::string g_create_error;

// NVTX range over a C-ABI call or a pipeline stage (visible in Nsight Systems / ncu --nvtx)
struct NvtxRange {
  explicit NvtxRange(const char* name) { nvtxRangePushA(name); }
  ~NvtxRange() { nvtxRangePop(); }
  NvtxRange(const NvtxRange&) = delete;
  NvtxRange& operator=(const NvtxRange&) = delete;
};
#define NVTX_RANGE(name) NvtxRange nvtx_range_(name)

#define CK(expr)                                                                                   \
  do {                                                                                             \
    cudaError_t e_ = (expr);                                                                       \
    if (e_ != cudaSuccess) {                                                                       \
      ctx->err = std::string(#expr) + ": " + cudaGetErrorString(e_);                               \
      return (e_ == cudaErrorMemoryAllocation) ? BLSGPU_E_ALLOC : BLSGPU_E_CUDA;                   \
    }                                                                                              \
  } while (0)
#define CKR(expr)                         \
  do {                                    \
    int r_ = (expr);                      \
    if (r_ != BLSGPU_OK) return r_;       \
  } while (0)

constexpr int TPB = 128;
constexpr size_t MSM_MIN_ITEMS = 4096;  // below this the per-item scaling is as fast as the bucket method's fixed costs
// Items per pass of the Miller kernels (a multiple of 120).  Measured on B200 at n = 1M: every extra pass costs ~8 ms of
// kernel ramp-up and tail (444 ms in one pass, 452 in three, 468 in six), and HBM is there to be used: 39 KB per item.
// The pass size of a call is planned from the memory that is actually free (plan_m6_chunk below): a context next to
// other tenants, or on a smaller device, takes more passes instead of failing with BLSGPU_E_ALLOC.
constexpr size_t M6_CHUNK_MAX = (size_t)8736 * 120;  // 1,048,320 items = 41 GB of line records: a 1M batch in one pass
constexpr size_t M6_CHUNK_MIN = 120;
inline unsigned blocks_for(size_t n, int tpb = TPB) { return (unsigned)((n + tpb - 1) / tpb); }
// one level of a 16-ary product / sum tree: levels with few output nodes take the 16-lanes-per-node kernels (kernels.cuh)
constexpr size_t REDUCE_WIDE_MAX = 4096;
#define REDUCE_FP12(n_in, in, n_out, out)                                                                       \
  do {                                                                                                          \
    if ((size_t)(n_out) <= REDUCE_WIDE_MAX)                                                                     \
      LAUNCH(k_reduce_fp12_w, blocks_for((size_t)(n_out) * 16), TPB, (size_t)(n_in), in, (size_t)(n_out), out); \
    else                                                                                                        \
      LAUNCH(k_reduce_fp12, blocks_for(n_out), TPB, (size_t)(n_in), in, (size_t)(n_out), out);                  \
  } while (0)
#define REDUCE_JAC(J, n_in, in, n_out, out)                                                                          \
  do {                                                                                                               \
    if ((size_t)(n_out) <= REDUCE_WIDE_MAX)                                                                          \
      LAUNCH((k_reduce_jac_w<J>), blocks_for((size_t)(n_out) * 16), TPB, (size_t)(n_in), in, (size_t)(n_out), out);  \
    else                                                                                                             \
      LAUNCH((k_reduce_jac<J>), blocks_for(n_out), TPB, (size_t)(n_in), in, (size_t)(n_out), out);                   \
  } while (0)

// bump allocator over one device buffer, regrown between calls
struct Arena {
  uint8_t* base = nullptr;
  size_t cap = 0, budget = 0, off = 0;  // budget: the bytes the call counted its takes to need (cap may hold more)
  bool over = false;  // a take ran past the call's budget: every later launch is refused (ARENA_OK)
  template <class T>
  static size_t bytes(size_t count) {
    return (count * sizeof(T) + 255) & ~size_t(255);
  }
  template <class T>
  T* take(size_t count) {
    T* p = reinterpret_cast<T*>(base + off);
    off += bytes<T>(count);
    if (off > budget) over = true;
    return p;
  }
};
// counts what a sequence of Arena takes occupies at its peak, without memory: every budget is its takes counted
struct ArenaSize {
  size_t off = 0, peak = 0;
  template <class T>
  T* take(size_t count) {
    off += Arena::bytes<T>(count);
    peak = std::max(peak, off);
    return nullptr;
  }
};
// `count` T of scratch handed back to the arena at once: later takes reuse it, which is safe for work ordered after its
// last reader on one stream
template <class T, class A>
T* take_back(A& a, size_t count) {
  const size_t mark = a.off;
  T* p = a.template take<T>(count);
  a.off = mark;
  return p;
}
// the peak of the takes that takes(a) makes
template <class Takes>
size_t counted(const Takes& takes) {
  ArenaSize a;
  takes(a);
  return a.peak;
}

struct Level {
  size_t off, cnt;
};

}  // namespace

// the slice-local state blsgpu_miller_partial leaves behind for blsgpu_partial_finish (lives in the arena)
struct PendingSlice {
  virtual ~PendingSlice() {}
  virtual int finish(blsgpu_ctx* ctx, bool batch_ok, uint8_t* status_out) = 0;
};

// public keys decoded once (blsgpu_keyset_create): n affine points of the impl's key group and their decode statuses, in a
// device allocation of their own on the first device (apart from the arena, so that regrowing the arena keeps them)
// The secure view of a key set in one format (ensure_secure_view, built by the first keyed secure call in that format, and
// kept current by the set's updates and appends, keyset_change_impl):
// every key re-encoded in the format, and its dense rank in memcmp order of those encodings (equal bytes, equal rank).
struct SecureView {
  uint8_t* enc = nullptr;            // device, n encodings
  uint32_t* rank = nullptr;          // device, n ranks
  std::vector<uint32_t> host_rank;  // the same ranks, for quorums the host plans
  size_t ranks = 0;                 // distinct encodings (the largest rank + 1)
};
struct KeySet {
  int impl_id = 0;
  size_t n = 0;
  void* pts = nullptr;
  uint8_t* st = nullptr;
  SecureView view[2];  // by format
};
// every device allocation of a key set (cudaFree waits for the work that may still read it); the first error
static cudaError_t free_keyset(const KeySet& s) {
  cudaError_t e = cudaSuccess;
  for (void* p : {s.pts, (void*)s.st, (void*)s.view[0].enc, (void*)s.view[0].rank, (void*)s.view[1].enc, (void*)s.view[1].rank}) {
    const cudaError_t r = cudaFree(p);
    if (e == cudaSuccess) e = r;
  }
  return e;
}

struct blsgpu_ctx {
  std::vector<int> devices;
  std::unique_ptr<PendingSlice> pending;  // invalidated by every call that re-plans the arena
  std::unordered_map<uint64_t, KeySet> keysets;  // by id: ids come from a process-wide counter and are never reused
  Arena fold;  // small device buffer of the fold (blsgpu_final_exp_is_one, fold_roots), apart from the arena
  std::vector<blsgpu_ctx*> peers;  // one single-device context per further device (devices[1..]); see verify_host_common
  cudaStream_t stream = nullptr;
  cudaStream_t own_stream = nullptr;
  int sm_count = 148;
  // the Miller stage runs its two big kernels on two side streams so that one block of each shares every SM (kernels.cuh)
  cudaStream_t side[2] = {nullptr, nullptr};
  cudaStream_t aux = nullptr;  // the signature side of the batch equation (bucket sum, its Miller loop), concurrent with the Miller stage
  cudaEvent_t ev_aux = nullptr;
  cudaEvent_t ev_fork = nullptr, ev_lines[2] = {nullptr, nullptr}, ev_accum[2] = {nullptr, nullptr};
  Arena arena;
  std::string err;
  uint8_t salt[32];        // salt of the current call's random-linear-combination scalars
  bool salt_pinned = false;  // blsgpu_ctx_set_rlc_salt: reproducible scalars (tests); otherwise fresh OS randomness per call
  int rlc_bits = 64;       // width of the scalars: 64 | 128
  size_t m6_chunk = M6_CHUNK_MAX;  // items per pass of the Miller kernels for the current call (plan_m6_chunk)
  cudaEvent_t ev[BLSGPU_STAGE_COUNT + 1];
  bool ev_valid[BLSGPU_STAGE_COUNT + 1];
  float stage_ms[BLSGPU_STAGE_COUNT];
  // per-kernel CUDA-event pairs of the hot kernels, recorded on the stream each kernel is launched on (blsgpu_last_kernel_ms)
  struct KernelMark {
    int id;
    cudaEvent_t begin, end;
  };
  std::vector<KernelMark> kmarks;
  size_t kmarks_used = 0;
  float kernel_ms[BLSGPU_KERNEL_COUNT];
  int kernel_launches[BLSGPU_KERNEL_COUNT];
  uint64_t launches = 0;
};

namespace {

// an arena of at least `bytes`, the call's budget (an ArenaSize count of its takes)
int ensure_arena(blsgpu_ctx* ctx, size_t bytes) {
  ctx->pending.reset();  // the arena is about to be handed out again
  ctx->arena.off = 0;
  ctx->arena.over = false;
  ctx->arena.budget = bytes;
  if (ctx->arena.cap >= bytes) return BLSGPU_OK;
  if (ctx->arena.base) CK(cudaFree(ctx->arena.base));  // the device may not hold the old and the new arena at once
  ctx->arena.base = nullptr;
  ctx->arena.cap = 0;
  size_t want = bytes + (bytes >> 3) + (1 << 20);
  if (cudaMalloc(&ctx->arena.base, want) != cudaSuccess) {
    (void)cudaGetLastError();
    want = bytes;  // no head-room available: the exact size
    ctx->arena.base = nullptr;
    CK(cudaMalloc(&ctx->arena.base, want));
  }
  ctx->arena.cap = want;
  return BLSGPU_OK;
}

// Pass size of the Miller kernels for a call over n items whose other scratch is `other_bytes`: as many items per pass as
// fit into ~85% of the memory this context may use (what is free now plus its own arena), at most M6_CHUNK_MAX, at least
// M6_CHUNK_MIN, a multiple of 120.  BLSGPU_M6_CHUNK overrides it (experiments and the multi-pass test), same clamps.
constexpr size_t M6_ITEM_BYTES = sizeof(M6Arg) + (size_t)M6_LINE_RECS * sizeof(SLineRec) + 512;
void plan_m6_chunk(blsgpu_ctx* ctx, size_t n, size_t other_bytes) {
  size_t chunk = M6_CHUNK_MAX;
  const char* e = getenv("BLSGPU_M6_CHUNK");
  if (e != nullptr && atoll(e) > 0) {
    chunk = (size_t)atoll(e);
  } else {
    size_t free_b = 0, total_b = 0;
    if (cudaMemGetInfo(&free_b, &total_b) == cudaSuccess) {
      const size_t usable = (free_b + ctx->arena.cap) / 20 * 17;
      const size_t room = usable > other_bytes ? usable - other_bytes : 0;
      const size_t one_pass = std::max<size_t>(n, 1) * M6_ITEM_BYTES;
      if (one_pass > room) chunk = room / (2 * M6_ITEM_BYTES);  // several passes run on two line buffers
    } else {
      (void)cudaGetLastError();
    }
  }
  chunk = std::min(chunk, M6_CHUNK_MAX) / 120 * 120;
  ctx->m6_chunk = std::max(chunk, M6_CHUNK_MIN);
}

// The salt of this call's random-linear-combination scalars: 32 bytes from the OS CSPRNG unless the caller pinned one.
int fresh_salt(blsgpu_ctx* ctx) {
  if (ctx->salt_pinned) return BLSGPU_OK;
  size_t got = 0;
  while (got < 32) {
    ssize_t r = getrandom(ctx->salt + got, 32 - got, 0);
    if (r <= 0) {
      ctx->err = "getrandom failed: no randomness for the batch-check scalars";
      return BLSGPU_E_CUDA;
    }
    got += (size_t)r;
  }
  return BLSGPU_OK;
}

int check_launch(blsgpu_ctx* ctx, const char* what) {
  ctx->launches++;
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) {
    ctx->err = std::string(what) + " launch: " + cudaGetErrorString(e);
    return BLSGPU_E_CUDA;
  }
  return BLSGPU_OK;
}
#define ARENA_OK()                                                          \
  do {                                                                      \
    if (ctx->arena.over || ctx->fold.over) {                                \
      ctx->err = "internal: device scratch arena sized too small";          \
      return BLSGPU_E_ALLOC;                                                \
    }                                                                       \
  } while (0)
#define LAUNCH(name, grid, block, ...)                          \
  do {                                                          \
    ARENA_OK();                                                 \
    name<<<(grid), (block), 0, ctx->stream>>>(__VA_ARGS__);     \
    CKR(check_launch(ctx, #name));                              \
  } while (0)

#define LAUNCH_TIMED(kid, name, grid, block, ...)               \
  do {                                                          \
    ARENA_OK();                                                 \
    const size_t km_ = kernel_begin(ctx, (kid), ctx->stream);   \
    name<<<(grid), (block), 0, ctx->stream>>>(__VA_ARGS__);     \
    kernel_end(ctx, km_, ctx->stream);                          \
    CKR(check_launch(ctx, #name));                              \
  } while (0)

// sizes the arena for the takes that takes(a) makes, then makes them on it
template <class Takes>
int arena_takes(blsgpu_ctx* ctx, const Takes& takes) {
  CKR(ensure_arena(ctx, counted(takes)));
  takes(ctx->arena);
  ARENA_OK();
  return BLSGPU_OK;
}

size_t kernel_begin(blsgpu_ctx* ctx, int id, cudaStream_t stream);
void kernel_end(blsgpu_ctx* ctx, size_t k, cudaStream_t stream);

void stage_mark(blsgpu_ctx* ctx, int idx) {
  static const char* const names[BLSGPU_STAGE_COUNT + 1] = {"stage:decode_pk", "stage:decode_sig", "stage:hash_to_curve", "stage:scale_sig",
                                                            "stage:miller", "stage:reduce", "stage:final", "stage:bisect", "stage:done"};
  nvtxMarkA(names[idx]);  // host-side marker of the stage's launches (the device times are the CUDA events below)
  cudaEventRecord(ctx->ev[idx], ctx->stream);
  ctx->ev_valid[idx] = true;
}
void stage_reset(blsgpu_ctx* ctx) {
  for (int i = 0; i <= BLSGPU_STAGE_COUNT; i++) ctx->ev_valid[i] = false;
  for (int i = 0; i < BLSGPU_STAGE_COUNT; i++) ctx->stage_ms[i] = 0.f;
  ctx->kmarks_used = 0;
  for (int i = 0; i < BLSGPU_KERNEL_COUNT; i++) {
    ctx->kernel_ms[i] = 0.f;
    ctx->kernel_launches[i] = 0;
  }
}
// event pair around ONE launch of a hot kernel, on the stream it is launched on; id < 0: not timed
size_t kernel_begin(blsgpu_ctx* ctx, int id, cudaStream_t stream) {
  if (id < 0) return (size_t)-1;
  if (ctx->kmarks_used == ctx->kmarks.size()) {
    blsgpu_ctx::KernelMark m{id, nullptr, nullptr};
    if (cudaEventCreate(&m.begin) != cudaSuccess || cudaEventCreate(&m.end) != cudaSuccess) return (size_t)-1;
    ctx->kmarks.push_back(m);
  }
  const size_t k = ctx->kmarks_used++;
  ctx->kmarks[k].id = id;
  cudaEventRecord(ctx->kmarks[k].begin, stream);
  return k;
}
void kernel_end(blsgpu_ctx* ctx, size_t k, cudaStream_t stream) {
  if (k != (size_t)-1) cudaEventRecord(ctx->kmarks[k].end, stream);
}
void stage_collect(blsgpu_ctx* ctx) {
  if (ctx->ev_valid[BLSGPU_STAGE_COUNT]) cudaEventSynchronize(ctx->ev[BLSGPU_STAGE_COUNT]);
  for (size_t k = 0; k < ctx->kmarks_used; k++) {
    float ms = 0.f;
    const blsgpu_ctx::KernelMark& m = ctx->kmarks[k];
    if (cudaEventSynchronize(m.end) == cudaSuccess && cudaEventElapsedTime(&ms, m.begin, m.end) == cudaSuccess) {
      ctx->kernel_ms[m.id] += ms;
      ctx->kernel_launches[m.id]++;
    }
  }
  for (int i = 0; i < BLSGPU_STAGE_COUNT; i++) {
    if (ctx->ev_valid[i] && ctx->ev_valid[i + 1]) {
      float ms = 0.f;
      if (cudaEventElapsedTime(&ms, ctx->ev[i], ctx->ev[i + 1]) == cudaSuccess) ctx->stage_ms[i] = ms;
    }
  }
}

bool make_dst(DstParam& d, int impl_id, int scheme, bool pop_proof) {
  // reference src/impls/g2.rs:107-118, src/impls/g1.rs:109-120
  const char* g = impl_id == 2 ? "G2" : "G1";
  const char* tag = scheme == 0 ? "NUL_" : scheme == 1 ? "AUG_" : "POP_";
  char buf[64];
  int n = snprintf(buf, sizeof buf, "BLS_%s_BLS12381%s_XMD:SHA-256_SSWU_RO_%s", pop_proof ? "POP" : "SIG", g, tag);
  if (n <= 0 || n > 63) return false;
  memset(d.b, 0, sizeof d.b);
  memcpy(d.b, buf, n);
  d.len = (uint32_t)n;
  return true;
}

// Window width of the bucket multi-scalar multiplication over rbits-bit scalars: >= 4 signatures per bucket, and only
// widths whose TOP window (rbits - (nwin - 1) c bits) is not much narrower than the others - a 4-bit top window would put
// n/16 signatures into each of 16 buckets, one thread each (measured: 1.5 s at n = 500,000 with c = 15).
// A bucket is summed by ONE thread, ~70 us per addition: what a slice of a batch cut over several GPUs pays is the LENGTH of
// the buckets, not the number of additions (round 2, measured with >= 16 per bucket: 21 ms at n = 125,000 with c = 11 and 61
// signatures per bucket, against 13 ms at n = 250,000 with c = 13 and 30 per bucket) - hence the wider windows.
int msm_window_bits(size_t n, int rbits = 64) {
  static const int widths64[] = {16, 13, 11, 8, 5, 4};    // top windows of 16, 12, 9, 8, 4, 4 bits
  static const int widths128[] = {16, 13, 10, 8, 5, 4};   // top windows of 16, 11, 8, 8, 3, 4 bits
  for (int w : (rbits == 128 ? widths128 : widths64))
    if (((size_t)1 << (w + 2)) <= n) return w;
  return 4;
}

std::vector<Level> make_levels(size_t n) {
  std::vector<Level> lv;
  size_t off = 0, cnt = n;
  lv.push_back({off, cnt});
  while (cnt > 1) {
    off += cnt;
    cnt = (cnt + 15) / 16;
    lv.push_back({off, cnt});
  }
  return lv;
}
size_t levels_total(const std::vector<Level>& lv) { return lv.back().off + lv.back().cnt; }

// A segmented 16-ary reduction over segments of cnt[j] >= 1 nodes: levels of ranges of at most 16 consecutive nodes of one
// segment, until one node per segment.  n[k]: the nodes of level k (n[0]: every segment's nodes, in segment order); off: the
// n[k] + 1 range offsets of every level k >= 1, concatenated.
struct SegLevels {
  std::vector<uint32_t> off;
  std::vector<size_t> n;
  size_t below_top() const {  // the nodes of every level but the last (the last is one node per segment)
    size_t t = 0;
    for (size_t k = 0; k + 1 < n.size(); k++) t += n[k];
    return t;
  }
};
SegLevels seg_levels(std::vector<size_t> cnt) {
  SegLevels s;
  const size_t q = cnt.size();
  size_t total = 0;
  for (size_t c : cnt) total += c;
  s.n.push_back(total);
  while (s.n.back() > q) {
    uint32_t in = 0;
    size_t outs = 0;
    s.off.push_back(0);
    for (size_t j = 0; j < q; j++) {
      const size_t o = (cnt[j] + 15) / 16;
      for (size_t k = 0; k < o; k++) {
        in += (uint32_t)std::min<size_t>(16, cnt[j] - 16 * k);
        s.off.push_back(in);
      }
      cnt[j] = o;
      outs += o;
    }
    s.n.push_back(outs);
  }
  return s;
}

// -----------------------------------------------------------------------------------------------------------------
// The batch pipeline on decoded points.  PkA/SigA are the affine types of the impl.
//   pre[i]   : status before pairing work (non-OK items are excluded from the batch equation)
//   use_rlc  : true  -> per-item check  e(pk_i,H_i) e(-g,sig_i) == 1 for all i, decided by one random linear combination
//                       and bisection on failure (writes INVALID_SIGNATURE into status[i] for the exact failures);
//              false -> aggregate check prod e(pk_i,H_i) * e(-g, sig_0) == 1 (sig has ONE element)
// Three phases, so that a batch cut over several devices can be folded (SURVEY 8e): pipeline_partials leaves the slice's
// product of Miller values (root of the product tree) and its sum of r_i sig_i in device memory; pipeline_check decides
// F * e(-g, S) == 1 for this slice alone; pipeline_bisect finds the exact failures of a slice whose check failed.
// -----------------------------------------------------------------------------------------------------------------
// The bucket multi-scalar multiplication S = sum r_i sig_i over n items, r_i = rlc_scalar(root, i) (0 for an item whose
// status is not OK): its window plan, and its takes
struct MsmPlan {
  int c, nwin;
  size_t nbuckets, nchunks;
  std::vector<Level> lm;  // the tree over the chunk sums
  MsmPlan(size_t n, int rbits) : c(msm_window_bits(n, rbits)), nwin((rbits + c - 1) / c) {
    nbuckets = ((size_t)1 << c) * nwin;
    nchunks = nbuckets / MSM_CHUNK;
    lm = make_levels(nchunks);
  }
};
template <class SigJ>
struct MsmScratch {
  RlcScalar* r = nullptr;
  uint32_t *cnt = nullptr, *sorted = nullptr;  // cnt: histograms, offsets, cursors
  SigJ *B = nullptr, *V = nullptr;
};
template <class SigJ, class A>
void take_msm(A& a, size_t n, const MsmPlan& m, MsmScratch<SigJ>& s) {
  s.r = a.template take<RlcScalar>(n);
  s.cnt = a.template take<uint32_t>(3 * m.nbuckets);
  s.sorted = a.template take<uint32_t>((size_t)m.nwin * n);
  s.B = a.template take<SigJ>(m.nbuckets);
  s.V = a.template take<SigJ>(levels_total(m.lm));
}

// blocks of the node-level bucket method of the failure path (a warp per level-1 node, four per block)
size_t node_msm_blocks(const blsgpu_ctx* ctx, size_t n1) { return std::max<size_t>(1, std::min<size_t>((n1 + 3) / 4, (size_t)ctx->sm_count * 4)); }
constexpr size_t PROBE_SMALL = 16;  // probes the dedicated scratch holds (the root check; small batches' bisection levels)
template <class PkA, class SigA>
struct Pipe {
  typedef typename PtInfo<SigA>::Jac SigJ;
  size_t n = 0, ng = 0;
  bool use_rlc = true, use_msm = false;
  int rbits = 0;
  std::vector<Level> lv;
  const PkA* d_pk = nullptr;
  const SigA *d_sig = nullptr, *d_h = nullptr;
  uint8_t* d_status = nullptr;
  Fp12* d_F = nullptr;
  SigJ *d_S = nullptr, *d_Sitem = nullptr, *d_msm_root = nullptr;
  MsmScratch<SigJ> msm;  // the bucket path (use_msm); its scalars msm.r are kept for the failure path
  Digest *d_dig = nullptr, *d_root = nullptr;
  // the failure path's node bucket method (by_nodes): bucket scratch, window sums of the level-1 nodes, item / group lists
  bool by_nodes = false;
  SigJ *node_buckets = nullptr, *node_W = nullptr;
  uint32_t* d_list = nullptr;
  uint8_t* d_ok = nullptr;
  uint32_t* d_idx = nullptr;
  // probe scratch: a small dedicated one, and (after the Miller stage) the first line buffer for levels with many probes
  PkA* x_pk = nullptr;
  SigA* x_h = nullptr;
  uint8_t* x_pre = nullptr;
  M6Arg* x_args = nullptr;
  SLineRec* x_lines = nullptr;
  Fp12* x_T = nullptr;
  size_t x_cap = 0;            // probes per launch the point / status / T scratch holds
  // the line buffers of the Miller stage (take_lines); buffer 0 is free for the probes once the stage is done
  M6Arg* m6_args[2] = {nullptr, nullptr};
  SLineRec* m6_lines[2] = {nullptr, nullptr};
  size_t big_items = 0;
  bool root_T_ready = false;   // T = ML(-g, S_root) already computed beside the Miller stage (x_T[0])
  const Fp12* rootF() const { return d_F + lv.back().off; }
  const SigJ* rootS() const { return use_msm ? d_msm_root : use_rlc ? d_S + lv.back().off : d_S; }
  // `count` probes go in rounds of PROBE_SMALL through the dedicated scratch, or (big) in rounds of as many as line buffer 0
  // and the point scratch hold
  bool big_rounds(size_t count) const { return count > PROBE_SMALL && big_items >= 6 * PROBE_SMALL; }
  size_t round_size(size_t count) const { return big_rounds(count) ? std::min(x_cap, big_items / 6) : PROBE_SMALL; }
};

// probes per launch of a tree with `leaves` leaves: as many as one bisection level can ask for at once (16 per failing node, at
// most one node per leaf)
size_t probe_cap(size_t leaves) { return std::max<size_t>(PROBE_SMALL, std::min<size_t>(leaves, 4096) + 16); }
// The probe scratch of P for `cap` probes per launch: indices and verdicts, the points and statuses of six pairs per probe,
// the T values, and the Miller buffers of one small round.  A takes from an Arena, or counts bytes (ArenaSize).
template <class PkA, class SigA, class A>
void take_probe_scratch(A& a, Pipe<PkA, SigA>& P, size_t cap) {
  const size_t small = std::min(cap, PROBE_SMALL);
  P.x_cap = cap;
  P.d_ok = a.template take<uint8_t>(cap);
  P.d_idx = a.template take<uint32_t>(cap);
  P.x_pk = a.template take<PkA>(6 * cap);
  P.x_h = a.template take<SigA>(6 * cap);
  P.x_pre = a.template take<uint8_t>(6 * cap);
  P.x_T = a.template take<Fp12>(cap);
  P.x_args = a.template take<M6Arg>(6 * small);
  P.x_lines = a.template take<SLineRec>(6 * small * M6_LINE_RECS);
}
// The line buffers of a Miller stage over n items in passes of `chunk` (miller_stage): one, or two when the stage takes
// several passes.  chunk 0 takes none: a call's takes counted with chunk 0 are what plan_m6_chunk plans the passes around.
template <class PkA, class SigA, class A>
void take_lines(A& a, Pipe<PkA, SigA>& P, size_t n, size_t chunk) {
  if (chunk == 0) return;
  P.big_items = std::max<size_t>(std::min(n, chunk), 6 * PROBE_SMALL);
  for (int b = 0; b < (n > chunk ? 2 : 1); b++) {
    P.m6_args[b] = a.template take<M6Arg>(P.big_items);
    P.m6_lines[b] = a.template take<SLineRec>(P.big_items * M6_LINE_RECS);
  }
}
// dynamic shared memory of the probe kernels, per device and per call (microseconds): a context per device may run this
// from several host threads
template <class PkA, class SigA>
int set_probe_smem(blsgpu_ctx* ctx) {
  CK(cudaFuncSetAttribute(k_m6_lines<PkA, SigA>, cudaFuncAttributeMaxDynamicSharedMemorySize, M6_LINES_SMEM));
  CK(cudaFuncSetAttribute(k_m6_accum, cudaFuncAttributeMaxDynamicSharedMemorySize, M6_ACCUM_SMEM));
  CK(cudaFuncSetAttribute(k_final6, cudaFuncAttributeMaxDynamicSharedMemorySize, FE6_SMEM));
  return BLSGPU_OK;
}

// the levels above `first` of a 16-ary product tree over F and / or sum tree over S (a null tree is skipped); per level the
// F launch goes first
template <class J>
int reduce_levels(blsgpu_ctx* ctx, const std::vector<Level>& lv, size_t first, Fp12* F, J* S) {
  for (size_t k = first; k + 1 < lv.size(); k++) {
    if (F) REDUCE_FP12(lv[k].cnt, (const Fp12*)(F + lv[k].off), lv[k + 1].cnt, F + lv[k + 1].off);
    if (S) REDUCE_JAC(J, lv[k].cnt, (const J*)(S + lv[k].off), lv[k + 1].cnt, S + lv[k + 1].off);
  }
  return BLSGPU_OK;
}

// the levels of a segmented reduction (seg_levels; d_off = its offsets on the device): level 0 in nodes[0 .. n[0]), the
// levels between in nodes after it, the last level (one node per segment) in top.  A level of few nodes takes the
// sixteen-lanes-per-node kernel, as REDUCE_FP12 / REDUCE_JAC do.
int seg_reduce(blsgpu_ctx* ctx, size_t n_out, const uint32_t* off, const Fp12* in, Fp12* out) {
  if (n_out <= REDUCE_WIDE_MAX)
    LAUNCH(k_seg_reduce_fp12_w, blocks_for(n_out * 16), TPB, n_out, off, in, out);
  else
    LAUNCH(k_seg_reduce_fp12, blocks_for(n_out), TPB, n_out, off, in, out);
  return BLSGPU_OK;
}
template <class J>
int seg_reduce(blsgpu_ctx* ctx, size_t n_out, const uint32_t* off, const J* in, J* out) {
  if (n_out <= REDUCE_WIDE_MAX)
    LAUNCH((k_seg_reduce_jac_w<J>), blocks_for(n_out * 16), TPB, n_out, off, in, out);
  else
    LAUNCH((k_seg_reduce_jac<J>), blocks_for(n_out), TPB, n_out, off, in, out);
  return BLSGPU_OK;
}
template <class T>
int seg_reduce_levels(blsgpu_ctx* ctx, const SegLevels& s, const uint32_t* d_off, T* nodes, T* top) {
  size_t in_off = 0, out_off = s.n[0], o = 0;
  for (size_t k = 1; k < s.n.size(); k++) {
    const size_t n_out = s.n[k];
    CKR(seg_reduce(ctx, n_out, d_off + o, (const T*)(nodes + in_off), k + 1 == s.n.size() ? top : nodes + out_off));
    o += n_out + 1;
    in_off = out_off;
    out_off += n_out;
  }
  return BLSGPU_OK;
}

// d_dig[0 .. leaves) holds the leaf digests: the 16-ary SHA-256 tree over them, then d_root = [root, salt of this call]
int digest_root(blsgpu_ctx* ctx, size_t leaves, Digest* d_dig, Digest* d_root) {
  const std::vector<Level> ld = make_levels(leaves);
  for (size_t k = 0; k + 1 < ld.size(); k++)
    LAUNCH(k_digest_reduce, blocks_for(ld[k + 1].cnt), TPB, ld[k].cnt, d_dig + ld[k].off, ld[k + 1].cnt, d_dig + ld[k + 1].off);
  CK(cudaMemcpyAsync(d_root, d_dig + ld.back().off, sizeof(Digest), cudaMemcpyDeviceToDevice, ctx->stream));
  CK(cudaMemcpyAsync(d_root + 1, ctx->salt, 32, cudaMemcpyHostToDevice, ctx->stream));
  return BLSGPU_OK;
}

// T[c] = product of the Miller values of probe c's pairs, c < cnt, on `stream`; the scratch batch was filled by k_probe_fill_*
template <class PkA, class SigA>
int probe_miller(blsgpu_ctx* ctx, Pipe<PkA, SigA>& P, cudaStream_t stream, size_t cnt, M6Arg* args, SLineRec* lines) {
  const size_t items = 6 * cnt;
  ARENA_OK();
  k_m6_prep<PkA, SigA><<<blocks_for(items), TPB, 0, stream>>>(items, 0, (const PkA*)P.x_pk, (const SigA*)P.x_h, (const uint8_t*)P.x_pre,
                                                               (const Digest*)nullptr, 0, args);
  CKR(check_launch(ctx, "k_m6_prep(probe)"));
  k_m6_lines<PkA, SigA><<<blocks_for(items, M6_LINES_PAIRS), M6_LINES_TPB, M6_LINES_SMEM, stream>>>(items, 0, args, (const PkA*)P.x_pk, (const SigA*)P.x_h,
                                                                                                       (const uint8_t*)P.x_pre, lines);
  CKR(check_launch(ctx, "k_m6_lines(probe)"));
  k_m6_accum<<<blocks_for(items, M6_ITEMS_PER_BLOCK), 128, M6_ACCUM_SMEM, stream>>>(items, 0, (const uint8_t*)P.x_pre, lines, P.x_T);
  CKR(check_launch(ctx, "k_m6_accum(probe)"));
  return BLSGPU_OK;
}
// ok[c] = final_exp(F[idx[c]] * T[c]) == 1 for the cnt probes whose T sits in x_T
template <class PkA, class SigA>
int probe_final(blsgpu_ctx* ctx, Pipe<PkA, SigA>& P, size_t cnt, const uint32_t* d_idx, const Fp12* F, uint8_t* d_ok) {
  ARENA_OK();
  k_final6<<<blocks_for(cnt, FE6_PER_WARP), 32, FE6_SMEM, ctx->stream>>>(cnt, d_idx, F, (const Fp12*)P.x_T, d_ok);
  CKR(check_launch(ctx, "k_final6"));
  return BLSGPU_OK;
}
// The probes of idx in rounds (P.round_size): a round copies its indices to P.d_idx, fill(cnt) fills the probe batch, then
// the Miller loops and the final exponentiation against F[idx] (F null: the probes' own pairs only), then after(lo, cnt)
// consumes the verdicts in P.d_ok; the round ends with a stream synchronisation.
template <class PkA, class SigA, class Fill, class After>
int probe_rounds(blsgpu_ctx* ctx, Pipe<PkA, SigA>& P, const std::vector<uint32_t>& idx, const Fp12* F, const Fill& fill, const After& after) {
  const bool big = P.big_rounds(idx.size());
  const size_t per = P.round_size(idx.size());
  for (size_t lo = 0; lo < idx.size(); lo += per) {
    const size_t cnt = std::min(per, idx.size() - lo);
    CK(cudaMemcpyAsync(P.d_idx, idx.data() + lo, cnt * 4, cudaMemcpyHostToDevice, ctx->stream));
    CKR(fill(cnt));
    CKR((probe_miller<PkA, SigA>(ctx, P, ctx->stream, cnt, big ? P.m6_args[0] : P.x_args, big ? P.m6_lines[0] : P.x_lines)));
    CKR((probe_final<PkA, SigA>(ctx, P, cnt, F ? P.d_idx : nullptr, F, P.d_ok)));
    CKR(after(lo, cnt));
    CK(cudaStreamSynchronize(ctx->stream));
  }
  return BLSGPU_OK;
}
// node probes over one tree level: res[c] = ( F[cand[c]] * e(-g, S[cand[c]]) == 1 )
template <class PkA, class SigA>
int probe_level(blsgpu_ctx* ctx, Pipe<PkA, SigA>& P, const std::vector<uint32_t>& cand, const Fp12* F, const typename Pipe<PkA, SigA>::SigJ* S,
                std::vector<uint8_t>& res) {
  res.resize(cand.size());
  return probe_rounds(
      ctx, P, cand, F,
      [&](size_t cnt) -> int {
        LAUNCH((k_probe_fill_nodes<PkA, SigA>), blocks_for(cnt), TPB, cnt, (const uint32_t*)P.d_idx, S, P.x_pk, P.x_h, P.x_pre);
        return BLSGPU_OK;
      },
      [&](size_t lo, size_t cnt) -> int {
        CK(cudaMemcpyAsync(res.data() + lo, P.d_ok, cnt, cudaMemcpyDeviceToHost, ctx->stream));
        return BLSGPU_OK;
      });
}

// The Miller stage over n items: F[g] = prod over the items of group g of ML(r pk, H), after ctx->ev_fork.  prep(stream, cn,
// base, args) launches the kernel that fills the M6Arg records of items [base, base + cn).  The line stream is 39 KB per item:
// batches beyond one pass (ctx->m6_chunk) go through in chunks with two line buffers (P.m6_*, taken by take_lines with the
// same chunk), chunk c's lines produced on side stream 0 while chunk c-1's accumulator consumes the other buffer on side
// stream 1.
template <class PkA, class SigA, class Prep>
int miller_stage(blsgpu_ctx* ctx, Pipe<PkA, SigA>& P, size_t n, const PkA* d_pk, const SigA* d_h, const uint8_t* d_status, Fp12* d_F,
                 const Prep& prep) {
  const size_t M6_CHUNK = ctx->m6_chunk;  // planned by the entry point together with the arena size (plan_m6_chunk)
  const int nbuf = n > M6_CHUNK ? 2 : 1;
  M6Arg* const* d_args = P.m6_args;
  SLineRec* const* d_lines = P.m6_lines;
  ARENA_OK();
  CK(cudaStreamWaitEvent(ctx->side[0], ctx->ev_fork, 0));
  CK(cudaStreamWaitEvent(ctx->side[1], ctx->ev_fork, 0));
  size_t ci = 0;
  for (size_t base = 0; base < n; base += M6_CHUNK, ci++) {
    const size_t cn = std::min(M6_CHUNK, n - base);
    const int b = (int)(ci % nbuf);
    if (ci >= (size_t)nbuf) CK(cudaStreamWaitEvent(ctx->side[0], ctx->ev_accum[b], 0));  // the buffer's previous reader is done
    size_t km = kernel_begin(ctx, BLSGPU_KERNEL_M6_PREP, ctx->side[0]);
    prep(ctx->side[0], cn, base, d_args[b]);
    kernel_end(ctx, km, ctx->side[0]);
    CKR(check_launch(ctx, "k_m6_prep"));
    km = kernel_begin(ctx, BLSGPU_KERNEL_M6_LINES, ctx->side[0]);
    k_m6_lines<PkA, SigA><<<blocks_for(cn, M6_LINES_PAIRS), M6_LINES_TPB, M6_LINES_SMEM, ctx->side[0]>>>(
        cn, base, d_args[b], d_pk, d_h, d_status, d_lines[b]);
    kernel_end(ctx, km, ctx->side[0]);
    CKR(check_launch(ctx, "k_m6_lines"));
    CK(cudaEventRecord(ctx->ev_lines[b], ctx->side[0]));
    CK(cudaStreamWaitEvent(ctx->side[1], ctx->ev_lines[b], 0));
    km = kernel_begin(ctx, BLSGPU_KERNEL_M6_ACCUM, ctx->side[1]);
    k_m6_accum<<<blocks_for(cn, M6_ITEMS_PER_BLOCK), 128, M6_ACCUM_SMEM, ctx->side[1]>>>(cn, base, d_status, d_lines[b], d_F);
    kernel_end(ctx, km, ctx->side[1]);
    CKR(check_launch(ctx, "k_m6_accum"));
    CK(cudaEventRecord(ctx->ev_accum[b], ctx->side[1]));
  }
  // join: everything later on the caller's stream waits for the last accumulator (which waited for every line kernel)
  CK(cudaStreamWaitEvent(ctx->stream, ctx->ev_accum[(ci - 1) % nbuf], 0));
  if (ci >= 2) CK(cudaStreamWaitEvent(ctx->stream, ctx->ev_accum[(ci - 2) % nbuf], 0));
  return BLSGPU_OK;
}

// S = sum r_i sig_i in the scratch s (take_msm with MsmPlan(n, rbits)): s.r = the scalars (kept for the failure path and the
// key side of blsgpu_verify_batch_grouped), *sum_out = S
template <class SigA>
int msm_sum(blsgpu_ctx* ctx, size_t n, const SigA* d_sig, const uint8_t* d_status, const Digest* d_root, int rbits,
            const MsmScratch<typename PtInfo<SigA>::Jac>& s, typename PtInfo<SigA>::Jac** sum_out) {
  typedef typename PtInfo<SigA>::Jac SigJ;
  const MsmPlan m(n, rbits);
  const int c = m.c, nwin = m.nwin;
  const size_t nbuckets = m.nbuckets, nchunks = m.nchunks;
  RlcScalar* d_r = s.r;
  uint32_t *d_cnt = s.cnt, *d_sorted = s.sorted;
  SigJ *d_B = s.B, *d_V = s.V;
  uint32_t *d_off = d_cnt + nbuckets, *d_cur = d_off + nbuckets;
  CK(cudaMemsetAsync(d_cnt, 0, nbuckets * sizeof(uint32_t), ctx->stream));
  LAUNCH(k_msm_count, blocks_for(n), TPB, n, (const uint8_t*)d_status, (const Digest*)d_root, rbits, c, nwin, d_r, d_cnt);
  LAUNCH(k_msm_scan, (unsigned)nwin, 1024, c, (const uint32_t*)d_cnt, d_off, d_cur);
  LAUNCH(k_msm_scatter, blocks_for(n), TPB, n, (const RlcScalar*)d_r, c, nwin, (const uint32_t*)d_off, d_cur, d_sorted);
  LAUNCH((k_msm_bucket<SigA>), blocks_for(nbuckets), TPB, n, nbuckets, d_sig, c, (const uint32_t*)d_cnt, (const uint32_t*)d_off,
         (const uint32_t*)d_sorted, d_B);
  LAUNCH((k_msm_chunk<SigJ>), blocks_for(nchunks), TPB, nchunks, c, (const SigJ*)d_B, d_V);
  CKR(reduce_levels(ctx, m.lm, 0, nullptr, d_V));
  *sum_out = d_V + m.lm.back().off;
  return BLSGPU_OK;
}

// Every take of the pipeline over n items (pipeline_partials): the product / sum trees, the leaf digests, the probe scratch
// (the line records of big levels go through the Miller stage's buffer 0), the bucket MSM, the Miller line buffers for passes
// of `chunk` items, and pipeline_bisect's scratch for the worst case it allows (every level-1 node and group failing).
template <class PkA, class SigA, class A>
void take_pipe(A& a, Pipe<PkA, SigA>& P, const blsgpu_ctx* ctx, size_t n, bool use_rlc, size_t chunk) {
  typedef typename PtInfo<SigA>::Jac SigJ;
  P.n = n;
  P.use_rlc = use_rlc;
  P.rbits = use_rlc ? ctx->rlc_bits : 0;
  P.use_msm = use_rlc && n >= MSM_MIN_ITEMS;
  // leaves of the product/sum trees are GROUPS of 6 consecutive items (the cooperative Miller kernel's unit)
  const size_t ng = P.ng = (n + M6_GROUP - 1) / M6_GROUP;
  P.lv = make_levels(ng);
  const size_t total = levels_total(P.lv);
  P.d_F = a.template take<Fp12>(total);
  P.d_S = a.template take<SigJ>(use_rlc ? total : 1);
  P.d_Sitem = a.template take<SigJ>(use_rlc ? n : 1);
  P.d_dig = a.template take<Digest>(levels_total(make_levels(n)) + 2);  // the digest tree, then [root, salt]
  take_probe_scratch(a, P, probe_cap(ng));
  if (P.use_msm) take_msm(a, n, MsmPlan(n, P.rbits), P.msm);
  take_lines(a, P, n, chunk);
  P.by_nodes = P.use_msm && P.rbits == 64 && P.lv.size() >= 3;
  if (P.by_nodes) {
    const size_t n1 = P.lv[1].cnt;
    P.node_buckets = a.template take<SigJ>(node_msm_blocks(ctx, n1) * 128 * NODE_BUCKETS);
    P.node_W = a.template take<SigJ>(n1 * 32);
    P.d_list = a.template take<uint32_t>(n + ng);
  }
}

// the pipeline over the n items of P (taken by take_pipe with ctx->m6_chunk)
template <class PkA, class SigA>
int pipeline_partials(blsgpu_ctx* ctx, Pipe<PkA, SigA>& P, const PkA* d_pk, const SigA* d_sig, const SigA* d_h, uint8_t* d_status) {
  typedef typename PtInfo<SigA>::Jac SigJ;
  const size_t n = P.n;
  const bool use_rlc = P.use_rlc;
  P.d_pk = d_pk;
  P.d_sig = d_sig;
  P.d_h = d_h;
  P.d_status = d_status;
  const size_t ng = P.ng;
  const std::vector<Level>& lv = P.lv;
  Fp12* d_F = P.d_F;
  SigJ* d_S = P.d_S;
  Digest* d_dig = P.d_dig;
  Digest* d_root = P.d_root = d_dig + levels_total(make_levels(n));
  CKR((set_probe_smem<PkA, SigA>(ctx)));

  const int rbits = P.rbits;
  if (use_rlc) {
    CKR(fresh_salt(ctx));
    LAUNCH((k_leaf_digest<PkA, SigA>), blocks_for(n), TPB, n, d_pk, d_sig, d_h, d_dig);
    CKR(digest_root(ctx, n, d_dig, d_root));
  }
  // S = sum r_i sig_i.  Large batches: bucket multi-scalar multiplication for the total only (the per-group sums the
  // bisection needs are computed if the batch fails) BEFORE the Miller stage, so that its Miller loop T = ML(-g, S) can
  // run on the aux stream beside the Miller kernels.  Small batches: per-item scaling.
  // (Running the bucket kernels themselves beside the Miller stage was measured: they evict Miller blocks, +70 ms at 1M.)
  stage_mark(ctx, BLSGPU_STAGE_SCALE_SIG);
  const bool use_msm = P.use_msm;
  if (use_msm) CKR((msm_sum<SigA>(ctx, n, d_sig, d_status, d_root, rbits, P.msm, &P.d_msm_root)));
  CK(cudaEventRecord(ctx->ev_fork, ctx->stream));
  P.root_T_ready = false;
  if (use_msm) {
    // the signature side of the batch equation, T = ML(-g, S): one cooperative probe on the aux stream, beside the Miller stage
    CK(cudaStreamWaitEvent(ctx->aux, ctx->ev_fork, 0));
    ARENA_OK();
    k_probe_fill_nodes<PkA, SigA><<<1, TPB, 0, ctx->aux>>>((size_t)1, (const uint32_t*)nullptr, (const SigJ*)P.d_msm_root, P.x_pk, P.x_h, P.x_pre);
    CKR(check_launch(ctx, "k_probe_fill_nodes"));
    CKR((probe_miller<PkA, SigA>(ctx, P, ctx->aux, 1, P.x_args, P.x_lines)));
    CK(cudaEventRecord(ctx->ev_aux, ctx->aux));
    P.root_T_ready = true;
  }
  stage_mark(ctx, BLSGPU_STAGE_MILLER);
  CKR((miller_stage<PkA, SigA>(ctx, P, n, d_pk, d_h, d_status, d_F, [&](cudaStream_t s, size_t cn, size_t base, M6Arg* args) {
    k_m6_prep<PkA, SigA><<<blocks_for(cn), TPB, 0, s>>>(cn, base, d_pk, d_h, (const uint8_t*)d_status, (const Digest*)d_root, rbits, args);
  })));
  if (use_msm) CK(cudaStreamWaitEvent(ctx->stream, ctx->ev_aux, 0));  // T = ML(-g, S) ran beside the Miller stage
  if (use_rlc && !use_msm) {
    LAUNCH((k_scale_sig<SigA>), blocks_for(n), TPB, n, d_sig, d_status, d_root, rbits, P.d_Sitem);
    LAUNCH((k_group_sum<SigJ>), blocks_for(ng), TPB, n, (const SigJ*)P.d_Sitem, ng, d_S);
  }
  stage_mark(ctx, BLSGPU_STAGE_REDUCE);
  CKR(reduce_levels(ctx, lv, 0, d_F, use_rlc && !use_msm ? d_S : nullptr));
  if (!use_rlc) LAUNCH((k_reduce_aff<SigA>), 1, 32, (size_t)1, d_sig, (size_t)1, d_S);  // S = the single aggregate signature
  return BLSGPU_OK;
}

// F_root * e(-g, S_root) == 1 for this slice?  (synchronises the stream)
template <class PkA, class SigA>
int pipeline_check(blsgpu_ctx* ctx, Pipe<PkA, SigA>& P, bool* ok_out) {
  typedef typename PtInfo<SigA>::Jac SigJ;
  stage_mark(ctx, BLSGPU_STAGE_FINAL);
  if (!P.root_T_ready) {
    LAUNCH((k_probe_fill_nodes<PkA, SigA>), 1, TPB, (size_t)1, (const uint32_t*)nullptr, (const SigJ*)P.rootS(), P.x_pk, P.x_h, P.x_pre);
    CKR((probe_miller<PkA, SigA>(ctx, P, ctx->stream, 1, P.x_args, P.x_lines)));
    P.root_T_ready = true;
  }
  CKR((probe_final<PkA, SigA>(ctx, P, 1, nullptr, P.rootF(), P.d_ok)));
  uint8_t ok = 0;
  CK(cudaMemcpyAsync(&ok, P.d_ok, 1, cudaMemcpyDeviceToHost, ctx->stream));
  stage_mark(ctx, BLSGPU_STAGE_BISECT);
  CK(cudaStreamSynchronize(ctx->stream));
  *ok_out = ok != 0;
  return BLSGPU_OK;
}

// Walks a failing tree (P.lv over P.d_F / P.d_S, root failed) down to its failing leaves: bad = the leaf indices whose node
// probe fails.  Children of node j at level k+1 are {j + m * cnt(k+1)} at level k.  A round of probes costs ~9 ms whatever
// its size (one cooperative Miller pass + one final-exponentiation launch, both latency), so a round goes down as many levels
// as it can while the candidates stay below BISECT_FANOUT: one bad signature in 1M is found in 3 rounds instead of 6.
// before_leaves(cand) runs once, before the probes of the leaf level (it may fill in leaf sums of P.d_S).
template <class PkA, class SigA, class BeforeLeaves>
int descend_tree(blsgpu_ctx* ctx, Pipe<PkA, SigA>& P, std::vector<uint32_t>& bad, const BeforeLeaves& before_leaves) {
  const std::vector<Level>& lv = P.lv;
  const size_t BISECT_FANOUT = std::min<size_t>(1024, P.round_size(SIZE_MAX));  // at most one round of probe_level
  auto children = [&](const std::vector<uint32_t>& nodes, size_t level) {  // nodes at `level` -> their children at level - 1
    std::vector<uint32_t> out;
    const size_t cn = lv[level].cnt;
    for (uint32_t j : nodes)
      for (int m = 0; m < 16; m++) {
        size_t idx = (size_t)j + (size_t)m * cn;
        if (idx < lv[level - 1].cnt) out.push_back((uint32_t)idx);
      }
    return out;
  };
  bad.assign(1, 0);
  std::vector<uint8_t> res;
  for (size_t k = lv.size() - 1; k > 0;) {
    std::vector<uint32_t> cand = children(bad, k);
    k--;
    while (k > 0 && cand.size() * 16 <= BISECT_FANOUT) {
      cand = children(cand, k);
      k--;
    }
    if (cand.empty()) break;
    if (k == 0) CKR(before_leaves(cand));
    CKR((probe_level<PkA, SigA>(ctx, P, cand, P.d_F + lv[k].off, P.d_S + lv[k].off, res)));
    bad.clear();
    for (size_t c = 0; c < cand.size(); c++)
      if (!res[c]) bad.push_back(cand[c]);
    if (bad.empty()) break;  // cannot happen for a failing parent; defensive
  }
  return BLSGPU_OK;
}

// the slice's check failed: per-group sums, descent of the 16-ary tree, exact per-item checks of the failing groups
template <class PkA, class SigA>
int pipeline_bisect(blsgpu_ctx* ctx, Pipe<PkA, SigA>& P) {
  typedef typename PtInfo<SigA>::Jac SigJ;
  const size_t n = P.n, ng = P.ng;
  const std::vector<Level>& lv = P.lv;
  // The bucket method gave the total only.  64-bit scalars: the sums of the LEVEL-1 nodes come from a small bucket method per
  // node (k_node_msm: ~21 point operations per item), the levels above from the tree, and only the groups of level-1 nodes
  // that FAIL get per-item scalar multiplications.  Otherwise (128-bit scalars): per-item scaling of the whole batch.
  const bool by_nodes = P.by_nodes;
  if (P.use_msm && !by_nodes) {
    LAUNCH((k_scale_sig<SigA>), blocks_for(n), TPB, n, P.d_sig, P.d_status, P.d_root, P.rbits, P.d_Sitem);
    LAUNCH((k_group_sum<SigJ>), blocks_for(ng), TPB, n, (const SigJ*)P.d_Sitem, ng, P.d_S);
    CKR(reduce_levels(ctx, lv, 0, nullptr, P.d_S));
  }
  if (by_nodes) {
    const size_t n1 = lv[1].cnt, nblocks = node_msm_blocks(ctx, n1);
    LAUNCH((k_node_msm<SigA>), (unsigned)nblocks, 128, n, n1, ng, P.d_sig, (const uint8_t*)P.d_status, (const RlcScalar*)P.msm.r, P.node_buckets,
           P.node_W);
    LAUNCH((k_node_combine<SigJ>), blocks_for(n1), TPB, n1, (const SigJ*)P.node_W, P.d_S + lv[1].off);
    CKR(reduce_levels(ctx, lv, 1, nullptr, P.d_S));
  }
  std::vector<uint32_t> bad;
  CKR((descend_tree<PkA, SigA>(ctx, P, bad, [&](const std::vector<uint32_t>& cand) -> int {
    if (!by_nodes) return BLSGPU_OK;
    // the candidate groups (children of failing level-1 nodes) get their sums now: r_i sig_i for their items only
    std::vector<uint32_t> its;
    for (uint32_t g : cand)
      for (int m = 0; m < M6_GROUP; m++)
        if ((size_t)g * M6_GROUP + m < n) its.push_back(g * M6_GROUP + m);
    uint32_t* d_list = P.d_list;  // its.size() <= n, cand.size() <= ng
    CK(cudaMemcpyAsync(d_list, its.data(), its.size() * 4, cudaMemcpyHostToDevice, ctx->stream));
    CK(cudaMemcpyAsync(d_list + its.size(), cand.data(), cand.size() * 4, cudaMemcpyHostToDevice, ctx->stream));
    LAUNCH((k_scale_sig_list<SigA>), blocks_for(its.size()), TPB, its.size(), (const uint32_t*)d_list, P.d_sig, (const uint8_t*)P.d_status,
           (const Digest*)P.d_root, P.rbits, P.d_Sitem);
    LAUNCH((k_group_sum_list<SigJ>), blocks_for(cand.size()), TPB, cand.size(), (const uint32_t*)(d_list + its.size()), n, (const SigJ*)P.d_Sitem,
           P.d_S + lv[0].off);
    CK(cudaStreamSynchronize(ctx->stream));  // the host vectors go out of scope
    return BLSGPU_OK;
  })));
  // every item of a failing group is decided by its own exact equation e(pk_i, H_i) e(-g, sig_i) == 1
  std::vector<uint32_t> items;
  for (uint32_t gidx : bad)
    for (int m = 0; m < M6_GROUP; m++) {
      size_t i = (size_t)gidx * M6_GROUP + m;
      if (i < n) items.push_back((uint32_t)i);
    }
  return probe_rounds(
      ctx, P, items, nullptr,
      [&](size_t cnt) -> int {
        LAUNCH((k_probe_fill_leaves<PkA, SigA>), blocks_for(cnt), TPB, cnt, (const uint32_t*)P.d_idx, P.d_pk, P.d_h, P.d_sig,
               (const uint8_t*)P.d_status, P.x_pk, P.x_h, P.x_pre);
        return BLSGPU_OK;
      },
      [&](size_t, size_t cnt) -> int {
        LAUNCH(k_mark_invalid, blocks_for(cnt), TPB, cnt, (const uint32_t*)P.d_idx, (const uint8_t*)P.d_ok, P.d_status);
        return BLSGPU_OK;
      });
}

// the slice's verdict on its own: root check, bisection if it fails; the call's last stage ends here
template <class PkA, class SigA>
int check_and_bisect(blsgpu_ctx* ctx, Pipe<PkA, SigA>& P) {
  bool ok = false;
  CKR((pipeline_check<PkA, SigA>(ctx, P, &ok)));
  if (!ok) CKR((pipeline_bisect<PkA, SigA>(ctx, P)));
  stage_mark(ctx, BLSGPU_STAGE_COUNT);
  return BLSGPU_OK;
}

// Plans the pass size of the Miller kernels for a call over n Miller items and sizes the arena for takes(a, chunk), the
// call's takes with line buffers for passes of `chunk` items (take_lines).  If the allocation fails the pass size is halved
// (more passes) until it fits or reaches the minimum.
template <class Takes>
int ensure_miller_arena(blsgpu_ctx* ctx, size_t n, const Takes& takes) {
  auto bytes = [&](size_t chunk) { return counted([&](auto& a) { takes(a, chunk); }); };
  plan_m6_chunk(ctx, n, bytes(0));
  for (;;) {
    const int r = ensure_arena(ctx, bytes(ctx->m6_chunk));
    if (r != BLSGPU_E_ALLOC || ctx->m6_chunk <= M6_CHUNK_MIN || n <= M6_CHUNK_MIN) return r;
    (void)cudaGetLastError();
    ctx->m6_chunk = std::max(M6_CHUNK_MIN, std::min(ctx->m6_chunk, n) / 2 / 120 * 120);
  }
}

// compressed bytes -> affine points + per-item status: decompression (square root), then the subgroup check
template <class A>
int decode_points(blsgpu_ctx* ctx, size_t n, const uint8_t* d_in, int format, A* d_out, uint8_t* d_st, int kid = -1) {
  LAUNCH_TIMED(kid, (k_decode<A>), blocks_for(n), TPB, n, d_in, format, d_out, d_st);
  LAUNCH_TIMED(kid < 0 ? -1 : kid + 1, (k_subgroup_check<A>), blocks_for(n), TPB, n, d_out, d_st);
  return BLSGPU_OK;
}

// The public keys of a verify call: n compressed keys in the call's format (`bytes`), or, for the keyed entry points, the
// index of every item's key (`idx`) in a key set decoded once (`set`).  Host pointers until the call uploads them.
struct Keys {
  const uint8_t* bytes = nullptr;
  KeySet* set = nullptr;
  const uint32_t* idx = nullptr;
  Keys(const uint8_t* b = nullptr) : bytes(b) {}
  Keys(KeySet* s, const uint32_t* i) : set(s), idx(i) {}
};
// the key step of a verify call, the one step where keyed and unkeyed calls differ: d_pk / d_st of the n items, by decoding
// their bytes or by gathering them from the key set (no decode or subgroup check)
template <class PkA>
int load_keys(blsgpu_ctx* ctx, size_t n, const Keys& d_keys, int format, PkA* d_pk, uint8_t* d_st) {
  if (!d_keys.set) return decode_points<PkA>(ctx, n, d_keys.bytes, format, d_pk, d_st, BLSGPU_KERNEL_DECODE_PK);
  LAUNCH((k_gather_keys<PkA>), blocks_for(n), TPB, n, d_keys.idx, (const PkA*)d_keys.set->pts, (const uint8_t*)d_keys.set->st, d_pk, d_st);
  return BLSGPU_OK;
}

// the Jacobian scratch of hash_points over n messages: handed back to the arena at once, later takes reuse it
template <class HA, class A>
typename PtInfo<HA>::Jac* take_hash_scratch(A& a, size_t n) {
  return take_back<typename PtInfo<HA>::Jac>(a, n);
}
// hash_to_curve of n framed messages into affine points: k_hash leaves Jacobian points in d_hj (take_hash_scratch),
// k_to_affine_batch normalises them 16 per inversion
template <class HA, class PkA>
int hash_points(blsgpu_ctx* ctx, size_t n, const uint8_t* d_msgs, const uint64_t* d_moff, int msg_mode, const PkA* d_pk,
                const uint8_t* d_pre, const DstParam& dst, typename PtInfo<HA>::Jac* d_hj, HA* d_h) {
  typedef typename PtInfo<HA>::Jac HJ;
  LAUNCH_TIMED(BLSGPU_KERNEL_HASH_MAP, (k_hash<HA, PkA>), blocks_for(n), TPB, n, d_msgs, d_moff, msg_mode, d_pk, d_pre, dst, d_hj);
  LAUNCH_TIMED(BLSGPU_KERNEL_CLEAR_COFACTOR, (k_clear_cofactor<HA>), blocks_for(n), TPB, n, d_hj);
  LAUNCH_TIMED(BLSGPU_KERNEL_TO_AFFINE, (k_to_affine_batch<HA>), blocks_for((n + TO_AFFINE_BATCH - 1) / TO_AFFINE_BATCH), TPB, n,
               (const HJ*)d_hj, d_h);
  return BLSGPU_OK;
}

// the takes of verify_points_partials over n items: the message points, the hash scratch, the pipeline (take_pipe)
template <int IMPL, class A>
void take_verify_points(A& a, const blsgpu_ctx* ctx, size_t n, size_t chunk, typename ImplT<IMPL>::SigAff*& d_h,
                        typename PtInfo<typename ImplT<IMPL>::SigAff>::Jac*& d_hj, Pipe<typename ImplT<IMPL>::PkAff, typename ImplT<IMPL>::SigAff>& P) {
  d_h = a.template take<typename ImplT<IMPL>::SigAff>(n);
  d_hj = take_hash_scratch<typename ImplT<IMPL>::SigAff>(a, n);
  take_pipe(a, P, ctx, n, true, chunk);
}
// the same counted, for the budget of a call that ends in verify_points_partials
template <int IMPL, class A>
void take_verify_points(A& a, const blsgpu_ctx* ctx, size_t n, size_t chunk) {
  typename ImplT<IMPL>::SigAff* d_h;
  typename PtInfo<typename ImplT<IMPL>::SigAff>::Jac* d_hj;
  Pipe<typename ImplT<IMPL>::PkAff, typename ImplT<IMPL>::SigAff> P;
  take_verify_points<IMPL>(a, ctx, n, chunk, d_h, d_hj, P);
}

// verify over decoded points: per-item pre-status, hash_to_curve of the framed message, pairing pipeline
template <int IMPL>
int verify_points_partials(blsgpu_ctx* ctx, Pipe<typename ImplT<IMPL>::PkAff, typename ImplT<IMPL>::SigAff>& P, int msg_mode, const DstParam& dst,
                           size_t n, const typename ImplT<IMPL>::PkAff* d_pk, const typename ImplT<IMPL>::SigAff* d_sig, const uint8_t* d_stpk,
                           const uint8_t* d_stsig, const uint8_t* d_msgs, const uint64_t* d_moff, uint8_t* d_status_out) {
  typedef typename ImplT<IMPL>::PkAff PkA;
  typedef typename ImplT<IMPL>::SigAff SigA;
  SigA* d_h;
  typename PtInfo<SigA>::Jac* d_hj;
  take_verify_points<IMPL>(ctx->arena, ctx, n, ctx->m6_chunk, d_h, d_hj, P);
  LAUNCH((k_prestatus<PkA, SigA>), blocks_for(n), TPB, n, d_stpk, d_stsig, d_pk, d_sig, d_status_out);
  stage_mark(ctx, BLSGPU_STAGE_HASH);
  CKR((hash_points<SigA, PkA>(ctx, n, d_msgs, d_moff, msg_mode, d_pk, (const uint8_t*)d_status_out, dst, d_hj, d_h)));
  return pipeline_partials<PkA, SigA>(ctx, P, d_pk, d_sig, d_h, d_status_out);
}
template <int IMPL>
int verify_points(blsgpu_ctx* ctx, int msg_mode, const DstParam& dst, size_t n, const typename ImplT<IMPL>::PkAff* d_pk,
                  const typename ImplT<IMPL>::SigAff* d_sig, const uint8_t* d_stpk, const uint8_t* d_stsig, const uint8_t* d_msgs,
                  const uint64_t* d_moff, uint8_t* d_status_out) {
  typedef typename ImplT<IMPL>::PkAff PkA;
  typedef typename ImplT<IMPL>::SigAff SigA;
  Pipe<PkA, SigA> P;
  CKR((verify_points_partials<IMPL>(ctx, P, msg_mode, dst, n, d_pk, d_sig, d_stpk, d_stsig, d_msgs, d_moff, d_status_out)));
  return check_and_bisect(ctx, P);
}

// verify over device-resident inputs: compressed signatures, keys as bytes or key-set indices.  msg_mode: 0 msg, 1 pk||msg,
// 2 pk bytes (PoP).  verify_dev_partials stops after the slice's partial results (its product of Miller values and sum of r_i sig_i).
// n decoded keys and signatures and their statuses
template <int IMPL>
struct Decoded {
  typename ImplT<IMPL>::PkAff* pk = nullptr;
  typename ImplT<IMPL>::SigAff* sig = nullptr;
  uint8_t *stpk = nullptr, *stsig = nullptr;
};
template <int IMPL, class A>
void take_decoded(A& a, size_t n, Decoded<IMPL>& D) {
  D.pk = a.template take<typename ImplT<IMPL>::PkAff>(n);
  D.sig = a.template take<typename ImplT<IMPL>::SigAff>(n);
  D.stpk = a.template take<uint8_t>(n);
  D.stsig = a.template take<uint8_t>(n);
}
// the takes of verify_dev_partials over n items counted, for the budget of a call that ends in it
template <int IMPL, class A>
void take_verify_dev(A& a, const blsgpu_ctx* ctx, size_t n, size_t chunk) {
  Decoded<IMPL> D;
  take_decoded(a, n, D);
  take_verify_points<IMPL>(a, ctx, n, chunk);
}
template <int IMPL>
int verify_dev_partials(blsgpu_ctx* ctx, Pipe<typename ImplT<IMPL>::PkAff, typename ImplT<IMPL>::SigAff>& P, int msg_mode, const DstParam& dst,
                        int format, size_t n, const Keys& d_keys, const uint8_t* d_sigs, const uint8_t* d_msgs, const uint64_t* d_moff,
                        uint8_t* d_status_out) {
  typedef typename ImplT<IMPL>::PkAff PkA;
  typedef typename ImplT<IMPL>::SigAff SigA;
  Decoded<IMPL> D;
  take_decoded(ctx->arena, n, D);
  PkA* d_pk = D.pk;
  SigA* d_sig = D.sig;
  uint8_t *d_stpk = D.stpk, *d_stsig = D.stsig;
  stage_reset(ctx);
  stage_mark(ctx, BLSGPU_STAGE_DECODE_PK);
  CKR((load_keys<PkA>(ctx, n, d_keys, format, d_pk, d_stpk)));
  stage_mark(ctx, BLSGPU_STAGE_DECODE_SIG);
  CKR((decode_points<SigA>(ctx, n, d_sigs, format, d_sig, d_stsig, BLSGPU_KERNEL_DECODE_SIG)));
  return verify_points_partials<IMPL>(ctx, P, msg_mode, dst, n, d_pk, d_sig, d_stpk, d_stsig, d_msgs, d_moff, d_status_out);
}
template <int IMPL>
int verify_dev(blsgpu_ctx* ctx, int msg_mode, const DstParam& dst, int format, size_t n, const uint8_t* d_pks, const uint8_t* d_sigs,
               const uint8_t* d_msgs, const uint64_t* d_moff, uint8_t* d_status_out) {
  Pipe<typename ImplT<IMPL>::PkAff, typename ImplT<IMPL>::SigAff> P;
  CKR((verify_dev_partials<IMPL>(ctx, P, msg_mode, dst, format, n, d_pks, d_sigs, d_msgs, d_moff, d_status_out)));
  CKR(check_and_bisect(ctx, P));
  stage_collect(ctx);
  return BLSGPU_OK;
}

// ---- the fold: partial results of several slices -> one verdict ------------------------------------------------------------
// d_F[k], d_S[k] on this context's device: is  prod F_j * e(-g, sum S_j)  == 1 ?   One product/sum launch, one cooperative
// probe, one six-lane final exponentiation - the "host multiplies the partials and runs a single final exponentiation" step
// of the north star, executed on a GPU because the engine has no CPU arithmetic.
// fold_check's takes: the product / sum of the partial results, and the probe scratch (only that of P is used)
template <class PkA, class SigA, class A>
void take_fold_check(A& a, Pipe<PkA, SigA>& P, Fp12*& d_Froot, typename PtInfo<SigA>::Jac*& d_Sroot) {
  d_Froot = a.template take<Fp12>(1);
  d_Sroot = a.template take<typename PtInfo<SigA>::Jac>(1);
  take_probe_scratch(a, P, 1);
}
// Sizes the fold scratch (a small device buffer apart from the arena, regrown between calls) for head(a) followed by
// fold_check's takes, and makes head's takes from it.
template <class PkA, class SigA, class Head>
int fold_takes(blsgpu_ctx* ctx, const Head& head) {
  const size_t bytes = counted([&](auto& a) {
    head(a);
    Pipe<PkA, SigA> P;
    Fp12* F;
    typename PtInfo<SigA>::Jac* S;
    take_fold_check(a, P, F, S);
  });
  Arena& A = ctx->fold;
  if (A.cap < bytes) {
    if (A.base) CK(cudaFree(A.base));
    A.base = nullptr;
    A.cap = 0;
    CK(cudaMalloc(&A.base, bytes));
    A.cap = bytes;
  }
  A.off = 0;
  A.budget = bytes;
  A.over = false;
  head(A);
  ARENA_OK();
  return BLSGPU_OK;
}
template <class PkA, class SigA>
int fold_check(blsgpu_ctx* ctx, size_t k, const Fp12* d_F, const typename PtInfo<SigA>::Jac* d_S, bool* ok_out) {
  typedef typename PtInfo<SigA>::Jac SigJ;
  Pipe<PkA, SigA> P;
  Fp12* d_Froot;
  SigJ* d_Sroot;
  take_fold_check(ctx->fold, P, d_Froot, d_Sroot);
  CKR((set_probe_smem<PkA, SigA>(ctx)));
  if (k > 16) {
    ctx->err = "fold: at most 16 partial results";
    return BLSGPU_E_ARG;
  }
  REDUCE_FP12(k, d_F, 1, d_Froot);  // 16-ary: one level covers up to 16 slices
  REDUCE_JAC(SigJ, k, d_S, 1, d_Sroot);
  LAUNCH((k_probe_fill_nodes<PkA, SigA>), 1, TPB, (size_t)1, (const uint32_t*)nullptr, (const SigJ*)d_Sroot, P.x_pk, P.x_h, P.x_pre);
  CKR((probe_miller<PkA, SigA>(ctx, P, ctx->stream, 1, P.x_args, P.x_lines)));
  CKR((probe_final<PkA, SigA>(ctx, P, 1, nullptr, (const Fp12*)d_Froot, P.d_ok)));
  uint8_t ok = 0;
  CK(cudaMemcpyAsync(&ok, P.d_ok, 1, cudaMemcpyDeviceToHost, ctx->stream));
  CK(cudaStreamSynchronize(ctx->stream));
  *ok_out = ok != 0;
  return BLSGPU_OK;
}
// the partial results of the slices in P (the roots of their trees, on device d for P[d]) meet on the first device
template <class PkA, class SigA>
int fold_roots(blsgpu_ctx* ctx, const std::vector<const Pipe<PkA, SigA>*>& P, bool* ok_out) {
  typedef typename PtInfo<SigA>::Jac SigJ;
  const size_t ndev = P.size();
  Fp12* d_Fk;
  SigJ* d_Sk;
  CKR((fold_takes<PkA, SigA>(ctx, [&](auto& a) {
    d_Fk = a.template take<Fp12>(ndev);
    d_Sk = a.template take<SigJ>(ndev);
  })));
  for (size_t d = 0; d < ndev; d++) {
    CK(cudaMemcpyPeerAsync(d_Fk + d, ctx->devices[0], P[d]->rootF(), ctx->devices[d], sizeof(Fp12), ctx->stream));
    CK(cudaMemcpyPeerAsync(d_Sk + d, ctx->devices[0], P[d]->rootS(), ctx->devices[d], sizeof(SigJ), ctx->stream));
  }
  return fold_check<PkA, SigA>(ctx, ndev, d_Fk, d_Sk, ok_out);
}

bool args_ok(int impl_id, int scheme, int format) {
  return (impl_id == 1 || impl_id == 2) && scheme >= 0 && scheme <= 2 && (format == 0 || format == 1);
}
// f(std::integral_constant<int, IMPL>) for impl_id 2 (Bls12381G2Impl) or 1 (Bls12381G1Impl): the template instance of the impl
template <class F>
int with_impl(int impl_id, const F& f) {
  return impl_id == 2 ? f(std::integral_constant<int, 2>()) : f(std::integral_constant<int, 1>());
}
// f(PointType<A>) for group 1 (G1 points) or 2 (G2 points): the affine point type of the group
template <class A>
struct PointType {
  typedef A type;
};
template <class F>
int with_group(int group, const F& f) {
  return group == 1 ? f(PointType<G1Aff>()) : f(PointType<G2Aff>());
}

// off[lo .. hi] rebased to off[lo]: the offsets of a run of records as the run's own
std::vector<uint64_t> rebased(const uint64_t* off, size_t lo, size_t hi) {
  std::vector<uint64_t> r(hi - lo + 1);
  for (size_t i = lo; i <= hi; i++) r[i - lo] = off[i] - off[lo];
  return r;
}

// ---- the argument rules of the entry points (include/blsgpu.h, "Arguments").  Each check returns a BLSGPU_* code and
// names the entry point (`what`) in ctx->err.
constexpr uint64_t MEMBERS_CAP = 0xfffffff0ull;  // items / members of a call that counts them in 32 bits (2^32 - 16)
constexpr uint64_t NO_CAP = ~0ull;

int arg_error(blsgpu_ctx* ctx, const char* what, const std::string& why) {
  ctx->err = std::string(what) + ": " + why;
  return BLSGPU_E_ARG;
}
// a buffer of `count` elements may be null only when it holds none
int check_buffer(blsgpu_ctx* ctx, const char* what, const char* name, const void* buf, uint64_t count) {
  return buf || count == 0 ? (int)BLSGPU_OK : arg_error(ctx, what, std::string(name) + " is null");
}
// n + 1 offsets: non-decreasing, every record below 2^32 (the kernels keep lengths and counts in 32 bits)
int check_offsets(blsgpu_ctx* ctx, const char* what, const char* name, const uint64_t* off, size_t n) {
  CKR(check_buffer(ctx, what, name, off, 1));
  for (size_t i = 0; i < n; i++)
    if (off[i + 1] < off[i] || off[i + 1] - off[i] > 0xffffffffull)
      return arg_error(ctx, what, std::string(name) + ": offsets must be non-decreasing with records below 2^32");
  return BLSGPU_OK;
}
// ragged records buf / off[0..n]: the offsets' rule, and buf non-null when the records span bytes
int check_records(blsgpu_ctx* ctx, const char* what, const char* buf_name, const uint8_t* buf, const char* off_name, const uint64_t* off,
                  size_t n) {
  CKR(check_offsets(ctx, what, off_name, off, n));
  return check_buffer(ctx, what, buf_name, buf, off[n] - off[0]);
}
// q sets of members (key_off, set_off, share_off, pair_off): the offsets' rule and at most `cap` members in all.
// off0 = the offsets rebased to 0; the caller shifts its member buffers by off[0] members once.
int check_sets(blsgpu_ctx* ctx, const char* what, const char* name, const uint64_t* off, size_t q, uint64_t cap, std::vector<uint64_t>& off0) {
  CKR(check_buffer(ctx, what, name, off, 1));
  off0.resize(q + 1);
  off0[0] = 0;
  for (size_t j = 0; j < q; j++) {
    if (off[j + 1] < off[j] || off[j + 1] - off[j] > 0xffffffffull)
      return arg_error(ctx, what, std::string(name) + ": offsets must be non-decreasing with sets below 2^32 members");
    off0[j + 1] = off[j + 1] - off[0];
  }
  return off0[q] > cap ? arg_error(ctx, what, "at most 2^32 - 16 members per call") : (int)BLSGPU_OK;
}
// the key set `id` of this context (an id that was destroyed, never issued, or is another context's is refused)
int find_keyset(blsgpu_ctx* ctx, const char* what, uint64_t id, KeySet*& set) {
  const auto it = ctx->keysets.find(id);
  if (it == ctx->keysets.end()) return arg_error(ctx, what, "key set " + std::to_string(id) + " is not held by this context");
  set = &it->second;
  return BLSGPU_OK;
}
// the keys of `count` members from member `first` on: the call's key bytes, or indices into a key set (at most 2^32 - 16,
// each below the set's size).  keys comes back shifted to `first`.
int check_keys(blsgpu_ctx* ctx, const char* what, int impl_id, Keys& keys, uint64_t first, uint64_t count) {
  if (!keys.set) {
    if (keys.bytes) keys.bytes += first * (impl_id == 2 ? 48 : 96);
    return check_buffer(ctx, what, "pks", keys.bytes, count);
  }
  if (keys.idx) keys.idx += first;
  CKR(check_buffer(ctx, what, "key_idx", keys.idx, count));
  if (count > MEMBERS_CAP) return arg_error(ctx, what, "at most 2^32 - 16 members per call");
  for (uint64_t i = 0; i < count; i++)
    if (keys.idx[i] >= keys.set->n)
      return arg_error(ctx, what, "key_idx[" + std::to_string(i) + "] is not below the key set's size " + std::to_string(keys.set->n));
  return BLSGPU_OK;
}

// the device copy of `count` host T (take_up, then upload)
template <class T, class A>
T* take_up(A& a, size_t count) {
  return a.template take<T>(std::max<size_t>(count, 1));
}
template <class T>
int upload(blsgpu_ctx* ctx, const T* d, const T* h, size_t count) {
  ARENA_OK();
  if (count) CK(cudaMemcpyAsync((void*)d, h, count * sizeof(T), cudaMemcpyHostToDevice, ctx->stream));
  return BLSGPU_OK;
}
// checked ragged records on the device as records from byte 0: the bytes off[0] .. off[n] and the offsets rebased to 0 (the
// caller's offsets go up as they are when they start at 0: no host copy)
template <class A>
void take_records(A& a, const uint64_t* off, size_t n, uint8_t*& d_buf, uint64_t*& d_off) {
  d_buf = take_up<uint8_t>(a, (size_t)(off[n] - off[0]));
  d_off = take_up<uint64_t>(a, n + 1);
}
int upload_records(blsgpu_ctx* ctx, const uint8_t* buf, const uint64_t* off, size_t n, uint8_t* d_buf, uint64_t* d_off) {
  CKR(upload(ctx, d_buf, off[n] > off[0] ? buf + off[0] : buf, (size_t)(off[n] - off[0])));
  if (off[0] == 0) return upload(ctx, d_off, off, n + 1);
  const std::vector<uint64_t> r = rebased(off, 0, n);
  return upload(ctx, d_off, r.data(), n + 1);
}
// the keys of a call on the device: its compressed key bytes, or its key indices, in the arena
template <class PkA, class A>
void take_keys(A& a, size_t n, const Keys& keys, Keys& d_keys) {
  d_keys = keys;
  if (keys.set)
    d_keys.idx = take_up<uint32_t>(a, n);
  else
    d_keys.bytes = take_up<uint8_t>(a, n * PtInfo<PkA>::LEN);
}
template <class PkA>
int upload_keys(blsgpu_ctx* ctx, size_t n, const Keys& keys, const Keys& d_keys) {
  return keys.set ? upload(ctx, d_keys.idx, keys.idx, n) : upload(ctx, d_keys.bytes, keys.bytes, n * PtInfo<PkA>::LEN);
}

int set_device(blsgpu_ctx* ctx) {
  CK(cudaSetDevice(ctx->devices[0]));
  return BLSGPU_OK;
}

}  // namespace

// =====================================================================================================================
// (C linkage comes from the declarations in include/blsgpu.h)

int blsgpu_ctx_create(const int* devices, int ndev, blsgpu_ctx** out) {
  NVTX_RANGE("blsgpu_ctx_create");
  if (!out || ndev < 1 || !devices) {
    g_create_error = "blsgpu_ctx_create: bad arguments";
    return BLSGPU_E_ARG;
  }
  int count = 0;
  cudaError_t e = cudaGetDeviceCount(&count);
  if (e != cudaSuccess || count == 0) {
    g_create_error = std::string("no CUDA device: ") + cudaGetErrorString(e) + " (this engine has no CPU fallback)";
    return BLSGPU_E_CUDA;
  }
  for (int i = 0; i < ndev; i++)
    if (devices[i] < 0 || devices[i] >= count) {
      g_create_error = "device index out of range";
      return BLSGPU_E_ARG;
    }
  blsgpu_ctx* ctx = new blsgpu_ctx();
  ctx->devices.assign(devices, devices + ndev);
  memset(ctx->salt, 0, 32);  // every batch check draws its own salt (fresh_salt) unless blsgpu_ctx_set_rlc_salt pinned one
  e = cudaSetDevice(devices[0]);
  if (e == cudaSuccess) e = cudaStreamCreateWithFlags(&ctx->own_stream, cudaStreamNonBlocking);
  ctx->stream = ctx->own_stream;
  if (e == cudaSuccess) e = cudaDeviceGetAttribute(&ctx->sm_count, cudaDevAttrMultiProcessorCount, devices[0]);
  int prio_lo = 0, prio_hi = 0;
  if (e == cudaSuccess) e = cudaDeviceGetStreamPriorityRange(&prio_lo, &prio_hi);
  for (int i = 0; e == cudaSuccess && i < 2; i++) {
    // side[0] (k_m6_lines, one block per SM) outranks side[1] (k_m6_accum): free SM resources go to a line block first,
    // the accumulator kernel takes what is left - that is what makes the two kernels share every SM
    e = cudaStreamCreateWithPriority(&ctx->side[i], cudaStreamNonBlocking, i == 0 ? prio_hi : prio_lo);
    if (e == cudaSuccess) e = cudaEventCreateWithFlags(&ctx->ev_lines[i], cudaEventDisableTiming);
    if (e == cudaSuccess) e = cudaEventCreateWithFlags(&ctx->ev_accum[i], cudaEventDisableTiming);
  }
  if (e == cudaSuccess) e = cudaEventCreateWithFlags(&ctx->ev_fork, cudaEventDisableTiming);
  if (e == cudaSuccess) e = cudaStreamCreateWithPriority(&ctx->aux, cudaStreamNonBlocking, prio_hi);
  if (e == cudaSuccess) e = cudaEventCreateWithFlags(&ctx->ev_aux, cudaEventDisableTiming);
  for (int i = 0; e == cudaSuccess && i <= BLSGPU_STAGE_COUNT; i++) e = cudaEventCreate(&ctx->ev[i]);
  if (e != cudaSuccess) {
    g_create_error = std::string("context setup: ") + cudaGetErrorString(e);
    delete ctx;
    return BLSGPU_E_CUDA;
  }
  stage_reset(ctx);
  for (int i = 1; i < ndev; i++) {
    blsgpu_ctx* peer = nullptr;
    int r = blsgpu_ctx_create(devices + i, 1, &peer);
    if (r != BLSGPU_OK) {
      blsgpu_ctx_destroy(ctx);
      return r;
    }
    ctx->peers.push_back(peer);
  }
  cudaSetDevice(devices[0]);
  // the device code vouches for itself once per process (and per first device): ~50 ms; BLSGPU_SKIP_SELFTEST=1 skips it
  static std::mutex selftest_mutex;
  static std::vector<int> selftested;
  {
    std::lock_guard<std::mutex> lock(selftest_mutex);
    const char* skip = getenv("BLSGPU_SKIP_SELFTEST");
    if (!(skip && skip[0] == '1') && std::find(selftested.begin(), selftested.end(), devices[0]) == selftested.end()) {
      selftested.push_back(devices[0]);  // before the call: the self-test's own entry points do not create contexts, but stay safe
      const int r = blsgpu_selftest(ctx);
      if (r != BLSGPU_OK) {
        g_create_error = ctx->err;
        blsgpu_ctx_destroy(ctx);
        return r;
      }
      ctx->launches = 0;
    }
  }
  *out = ctx;
  return BLSGPU_OK;
}

void blsgpu_ctx_destroy(blsgpu_ctx* ctx) {
  NVTX_RANGE("blsgpu_ctx_destroy");
  if (!ctx) return;
  for (blsgpu_ctx* peer : ctx->peers) blsgpu_ctx_destroy(peer);
  cudaSetDevice(ctx->devices[0]);
  ctx->pending.reset();
  for (const auto& ks : ctx->keysets) free_keyset(ks.second);
  if (ctx->arena.base) cudaFree(ctx->arena.base);
  if (ctx->fold.base) cudaFree(ctx->fold.base);
  for (int i = 0; i <= BLSGPU_STAGE_COUNT; i++) cudaEventDestroy(ctx->ev[i]);
  for (const blsgpu_ctx::KernelMark& m : ctx->kmarks) {
    cudaEventDestroy(m.begin);
    cudaEventDestroy(m.end);
  }
  if (ctx->own_stream) cudaStreamDestroy(ctx->own_stream);
  for (int i = 0; i < 2; i++) {
    if (ctx->side[i]) cudaStreamDestroy(ctx->side[i]);
    if (ctx->ev_lines[i]) cudaEventDestroy(ctx->ev_lines[i]);
    if (ctx->ev_accum[i]) cudaEventDestroy(ctx->ev_accum[i]);
  }
  if (ctx->ev_fork) cudaEventDestroy(ctx->ev_fork);
  if (ctx->aux) cudaStreamDestroy(ctx->aux);
  if (ctx->ev_aux) cudaEventDestroy(ctx->ev_aux);
  delete ctx;
}

const char* blsgpu_last_error(const blsgpu_ctx* ctx) { return ctx ? ctx->err.c_str() : g_create_error.c_str(); }

int blsgpu_ctx_set_stream(blsgpu_ctx* ctx, void* cuda_stream) {
  if (!ctx) return BLSGPU_E_ARG;
  ctx->stream = cuda_stream ? static_cast<cudaStream_t>(cuda_stream) : ctx->own_stream;
  return BLSGPU_OK;
}

int blsgpu_ctx_set_rlc_salt(blsgpu_ctx* ctx, const uint8_t salt[32]) {
  if (!ctx || !salt) return BLSGPU_E_ARG;
  memcpy(ctx->salt, salt, 32);
  ctx->salt_pinned = true;
  for (blsgpu_ctx* peer : ctx->peers) {
    memcpy(peer->salt, salt, 32);
    peer->salt_pinned = true;
  }
  return BLSGPU_OK;
}

int blsgpu_ctx_set_rlc_bits(blsgpu_ctx* ctx, int bits) {
  if (!ctx || (bits != 64 && bits != 128)) return BLSGPU_E_ARG;
  ctx->rlc_bits = bits;
  for (blsgpu_ctx* peer : ctx->peers) peer->rlc_bits = bits;
  return BLSGPU_OK;
}

int blsgpu_last_stage_ms(const blsgpu_ctx* ctx, float ms_out[BLSGPU_STAGE_COUNT]) {
  if (!ctx || !ms_out) return BLSGPU_E_ARG;
  for (int i = 0; i < BLSGPU_STAGE_COUNT; i++) ms_out[i] = ctx->stage_ms[i];
  return BLSGPU_OK;
}
int blsgpu_last_kernel_ms(const blsgpu_ctx* ctx, float ms_out[BLSGPU_KERNEL_COUNT], int launches_out[BLSGPU_KERNEL_COUNT]) {
  if (!ctx || !ms_out) return BLSGPU_E_ARG;
  for (int i = 0; i < BLSGPU_KERNEL_COUNT; i++) {
    ms_out[i] = ctx->kernel_ms[i];
    if (launches_out) launches_out[i] = ctx->kernel_launches[i];
  }
  return BLSGPU_OK;
}
uint64_t blsgpu_launch_count(const blsgpu_ctx* ctx) {
  if (!ctx) return 0;
  uint64_t total = ctx->launches;
  for (const blsgpu_ctx* peer : ctx->peers) total += peer->launches;
  return total;
}

int blsgpu_verify_batch_dev(blsgpu_ctx* ctx, int impl_id, int scheme, int format, size_t n, const uint8_t* pks_dev,
                            const uint8_t* sigs_dev, const uint8_t* msgs_dev, const uint64_t* msg_off_dev, uint8_t* status_out_dev) {
  NVTX_RANGE("blsgpu_verify_batch_dev");
  if (!ctx) return BLSGPU_E_ARG;
  if (!args_ok(impl_id, scheme, format) || (n && (!pks_dev || !sigs_dev || !msg_off_dev || !status_out_dev))) return arg_error(ctx, __func__, "bad arguments");
  if (n == 0) return BLSGPU_OK;
  CKR(set_device(ctx));
  DstParam dst;
  make_dst(dst, impl_id, scheme, false);
  int mode = scheme == 1 ? 1 : 0;
  return with_impl(impl_id, [&](auto I) {
    CKR(ensure_miller_arena(ctx, n, [&](auto& a, size_t chunk) { take_verify_dev<decltype(I)::value>(a, ctx, n, chunk); }));
    return verify_dev<I>(ctx, mode, dst, format, n, pks_dev, sigs_dev, msgs_dev, msg_off_dev, status_out_dev);
  });
}

namespace {
// takes that make none (the tail of a call that takes nothing after its last step)
struct NoTakes {
  template <class A>
  void operator()(A&) const {}
};
// host buffers of one slice -> its partial results (state in P, statuses so far in *d_st_out); the stream is synchronised.
// The arena is sized for tail(a) as well: the takes the caller makes after this.
template <int IMPL, class Tail = NoTakes>
int host_partials(blsgpu_ctx* ctx, Pipe<typename ImplT<IMPL>::PkAff, typename ImplT<IMPL>::SigAff>& P, int msg_mode, const DstParam& dst, int format,
                  size_t n, const Keys& keys, const uint8_t* sigs, const uint8_t* msgs, const uint64_t* msg_off, uint8_t** d_st_out,
                  const Tail& tail = Tail()) {
  CKR(set_device(ctx));
  const size_t sig_len = IMPL == 2 ? 96 : 48;
  const std::vector<uint64_t> no_msgs(msg_off ? 0 : n + 1, 0);  // PoP: every message empty
  if (!msg_off) msg_off = no_msgs.data();
  uint8_t *d_sigs, *d_msgs, *d_st;
  uint64_t* d_off;
  Keys d_keys;
  auto head = [&](auto& a) {
    take_keys<typename ImplT<IMPL>::PkAff>(a, n, keys, d_keys);
    d_sigs = take_up<uint8_t>(a, n * sig_len);
    take_records(a, msg_off, n, d_msgs, d_off);
    d_st = a.template take<uint8_t>(n);
  };
  CKR(ensure_miller_arena(ctx, n, [&](auto& a, size_t chunk) {
    head(a);
    take_verify_dev<IMPL>(a, ctx, n, chunk);
    tail(a);
  }));
  head(ctx->arena);
  CKR(upload_keys<typename ImplT<IMPL>::PkAff>(ctx, n, keys, d_keys));
  CKR(upload(ctx, d_sigs, sigs, n * sig_len));
  CKR(upload_records(ctx, msgs, msg_off, n, d_msgs, d_off));
  *d_st_out = d_st;
  CKR((verify_dev_partials<IMPL>(ctx, P, msg_mode, dst, format, n, d_keys, d_sigs, d_msgs, d_off, d_st)));
  CK(cudaStreamSynchronize(ctx->stream));
  return BLSGPU_OK;
}
// batch_ok: the verdict of the fold over all slices.  A slice of a failed batch checks its own partial results and bisects
// only if they fail too (SURVEY 8e: only the devices holding bad items do extra work).
template <int IMPL>
int host_finish(blsgpu_ctx* ctx, Pipe<typename ImplT<IMPL>::PkAff, typename ImplT<IMPL>::SigAff>& P, bool batch_ok, const uint8_t* d_st, size_t n,
                uint8_t* status_out) {
  CKR(set_device(ctx));
  if (batch_ok)
    stage_mark(ctx, BLSGPU_STAGE_COUNT);
  else
    CKR(check_and_bisect(ctx, P));
  CK(cudaMemcpyAsync(status_out, d_st, n, cudaMemcpyDeviceToHost, ctx->stream));
  CK(cudaStreamSynchronize(ctx->stream));
  stage_collect(ctx);
  return BLSGPU_OK;
}

template <int IMPL>
int verify_host_one(blsgpu_ctx* ctx, int msg_mode, const DstParam& dst, int format, size_t n, const Keys& keys, const uint8_t* sigs,
                    const uint8_t* msgs, const uint64_t* msg_off, uint8_t* status_out) {
  Pipe<typename ImplT<IMPL>::PkAff, typename ImplT<IMPL>::SigAff> P;
  uint8_t* d_st = nullptr;
  CKR((host_partials<IMPL>(ctx, P, msg_mode, dst, format, n, keys, sigs, msgs, msg_off, &d_st)));
  return host_finish<IMPL>(ctx, P, false, d_st, n, status_out);
}

// A context on several devices: independent work (point sums of slices, key sets, quorums) goes to the devices in contiguous
// runs, one host thread per device on the device's own child context - the same sharding blsgpu_verify_batch does, minus the
// fold (nothing is shared between the runs).  cut[d] .. cut[d + 1] is device d's run; f(device context, d) returns a BLSGPU_* code.
int run_on_devices(blsgpu_ctx* ctx, const std::function<int(blsgpu_ctx*, size_t)>& f) {
  const size_t ndev = 1 + ctx->peers.size();
  std::vector<int> rc(ndev, BLSGPU_OK);
  auto body = [&](size_t d) {
    blsgpu_ctx* c = d == 0 ? ctx : ctx->peers[d - 1];
    rc[d] = set_device(c);
    if (rc[d] == BLSGPU_OK) rc[d] = f(c, d);
  };
  std::vector<std::thread> workers;
  for (size_t d = 1; d < ndev; d++) workers.emplace_back(body, d);
  body(0);
  for (std::thread& w : workers) w.join();
  for (size_t d = 0; d < ndev; d++)
    if (rc[d] != BLSGPU_OK) {
      if (d) ctx->err = "device " + std::to_string(ctx->devices[d]) + ": " + ctx->peers[d - 1]->err;
      return rc[d];
    }
  return set_device(ctx);
}
// cut points of `sets` sets with cumulative weights off[0..sets] into ndev runs of about equal weight
std::vector<size_t> balanced_cuts(size_t sets, const uint64_t* off, size_t ndev) {
  std::vector<size_t> cut(ndev + 1, sets);
  cut[0] = 0;
  const uint64_t total = off[sets] - off[0];
  size_t j = 0;
  for (size_t d = 1; d < ndev; d++) {
    const uint64_t want = off[0] + total * d / ndev;
    while (j < sets && off[j] < want) j++;
    cut[d] = j;
  }
  return cut;
}
// sets 0 .. sets-1 cut into contiguous runs over the devices, balanced by the cumulative weights off[0 .. sets]:
// run(device context, lo, hi) handles sets lo .. hi-1; a device whose run is empty does nothing
int run_cut(blsgpu_ctx* ctx, size_t sets, const uint64_t* off, const std::function<int(blsgpu_ctx*, size_t, size_t)>& run) {
  const std::vector<size_t> cut = balanced_cuts(sets, off, 1 + ctx->peers.size());
  return run_on_devices(ctx, [&](blsgpu_ctx* c, size_t d) { return cut[d] == cut[d + 1] ? (int)BLSGPU_OK : run(c, cut[d], cut[d + 1]); });
}

// A context created on several devices cuts a host-buffer batch into contiguous slices, one per device, each driven by its
// own host thread (SURVEY 8e).  Every device folds its slice into ONE partial product of Miller values and ONE partial sum
// of r_i sig_i; the partial results meet on the first device, which multiplies / adds them and runs a single Miller loop
// and a single final exponentiation for the whole batch.  Only if that check fails does a device look at its own partial
// results, and only a device whose slice fails bisects.  No collective: 2 x ndev small copies.
// Below SHARD_MIN_ITEMS per device the first device takes the whole batch.
constexpr size_t SHARD_MIN_ITEMS = 4096;
template <int IMPL>
int verify_host_fold(blsgpu_ctx* ctx, int msg_mode, const DstParam& dst, int format, size_t n, const uint8_t* pks, const uint8_t* sigs,
                     const uint8_t* msgs, const uint64_t* msg_off, uint8_t* status_out) {
  typedef typename ImplT<IMPL>::PkAff PkA;
  typedef typename ImplT<IMPL>::SigAff SigA;
  const size_t ndev = 1 + ctx->peers.size();
  const size_t pk_len = IMPL == 2 ? 48 : 96, sig_len = IMPL == 2 ? 96 : 48;
  std::vector<Pipe<PkA, SigA>> P(ndev);
  std::vector<uint8_t*> d_st(ndev, nullptr);
  auto lo = [&](size_t d) { return n * d / ndev; };
  CKR(run_on_devices(ctx, [&](blsgpu_ctx* c, size_t d) {
    const size_t s = lo(d), e = lo(d + 1);
    return host_partials<IMPL>(c, P[d], msg_mode, dst, format, e - s, pks + s * pk_len, sigs + s * sig_len, msgs, msg_off ? msg_off + s : nullptr,
                               &d_st[d]);
  }));
  std::vector<const Pipe<PkA, SigA>*> roots;
  for (const Pipe<PkA, SigA>& p : P) roots.push_back(&p);
  bool ok = false;
  CKR((fold_roots<PkA, SigA>(ctx, roots, &ok)));
  return run_on_devices(ctx, [&](blsgpu_ctx* c, size_t d) {
    const size_t s = lo(d), e = lo(d + 1);
    return host_finish<IMPL>(c, P[d], ok, d_st[d], e - s, status_out + s);
  });
}

int verify_host_common(blsgpu_ctx* ctx, int impl_id, int msg_mode, const DstParam& dst, int format, size_t n, const uint8_t* pks,
                       const uint8_t* sigs, const uint8_t* msgs, const uint64_t* msg_off, uint8_t* status_out) {
  const size_t ndev = 1 + ctx->peers.size();
  const bool fold = ndev > 1 && n >= ndev * SHARD_MIN_ITEMS;
  return with_impl(impl_id, [&](auto I) {
    return fold ? verify_host_fold<I>(ctx, msg_mode, dst, format, n, pks, sigs, msgs, msg_off, status_out)
                : verify_host_one<I>(ctx, msg_mode, dst, format, n, pks, sigs, msgs, msg_off, status_out);
  });
}

// blsgpu_verify_batch and its keyed form (which stays on the first device)
int verify_batch_common(blsgpu_ctx* ctx, const char* what, int impl_id, int scheme, int format, size_t n, Keys keys, const uint8_t* sigs,
                        const uint8_t* msgs, const uint64_t* msg_off, uint8_t* status_out) {
  if (!args_ok(impl_id, scheme, format) || (n && (!sigs || !status_out))) return arg_error(ctx, what, "bad arguments");
  if (n == 0) return BLSGPU_OK;
  CKR(check_keys(ctx, what, impl_id, keys, 0, n));
  CKR(check_records(ctx, what, "msgs", msgs, "msg_off", msg_off, n));
  DstParam dst;
  make_dst(dst, impl_id, scheme, false);
  const int mode = scheme == 1 ? 1 : 0;
  if (!keys.set) return verify_host_common(ctx, impl_id, mode, dst, format, n, keys.bytes, sigs, msgs, msg_off, status_out);
  return with_impl(impl_id, [&](auto I) { return verify_host_one<I>(ctx, mode, dst, format, n, keys, sigs, msgs, msg_off, status_out); });
}

template <int IMPL>
struct PendingImpl : PendingSlice {
  Pipe<typename ImplT<IMPL>::PkAff, typename ImplT<IMPL>::SigAff> P;
  uint8_t* d_st = nullptr;
  size_t n = 0;
  int finish(blsgpu_ctx* ctx, bool batch_ok, uint8_t* status_out) override { return host_finish<IMPL>(ctx, P, batch_ok, d_st, n, status_out); }
};
template <int IMPL>
int miller_partial_impl(blsgpu_ctx* ctx, int msg_mode, const DstParam& dst, int format, size_t n, const uint8_t* pks, const uint8_t* sigs,
                        const uint8_t* msgs, const uint64_t* msg_off, uint8_t* gt_out, uint8_t* sum_out) {
  typedef typename ImplT<IMPL>::SigAff SigA;
  typedef typename PtInfo<SigA>::Jac SigJ;
  const size_t Ls = PtInfo<SigA>::LEN;
  std::unique_ptr<PendingImpl<IMPL>> pend(new PendingImpl<IMPL>());
  pend->n = n;
  uint8_t *d_gt, *d_enc;
  SigA* d_aff;
  auto tail = [&](auto& a) {
    d_gt = a.template take<uint8_t>(576);
    d_aff = a.template take<SigA>(1);
    d_enc = a.template take<uint8_t>(Ls);
  };
  CKR((host_partials<IMPL>(ctx, pend->P, msg_mode, dst, format, n, pks, sigs, msgs, msg_off, &pend->d_st, tail)));
  tail(ctx->arena);
  LAUNCH(k_fp12_to_bytes, 1, 32, (size_t)1, pend->P.rootF(), d_gt);
  LAUNCH((k_to_affine<SigA>), 1, 32, (size_t)1, (const SigJ*)pend->P.rootS(), d_aff);
  LAUNCH((k_encode<SigA>), 1, 32, (size_t)1, (const SigA*)d_aff, 1, d_enc);
  CK(cudaMemcpyAsync(gt_out, d_gt, 576, cudaMemcpyDeviceToHost, ctx->stream));
  CK(cudaMemcpyAsync(sum_out, d_enc, Ls, cudaMemcpyDeviceToHost, ctx->stream));
  CK(cudaStreamSynchronize(ctx->stream));
  ctx->pending = std::move(pend);
  return BLSGPU_OK;
}
template <int IMPL>
int fold_bytes_impl(blsgpu_ctx* ctx, const char* what, size_t k, const uint8_t* gts, const uint8_t* sums, int* ok_out) {
  typedef typename ImplT<IMPL>::PkAff PkA;
  typedef typename ImplT<IMPL>::SigAff SigA;
  typedef typename PtInfo<SigA>::Jac SigJ;
  const size_t Ls = PtInfo<SigA>::LEN;
  uint8_t *d_gt, *d_sb, *d_flag;
  Fp12* d_Fk;
  SigA* d_aff;
  SigJ* d_Sk;
  CKR((fold_takes<PkA, SigA>(ctx, [&](auto& a) {
    d_gt = a.template take<uint8_t>(576 * k);
    d_sb = a.template take<uint8_t>(Ls * k);
    d_Fk = a.template take<Fp12>(k);
    d_aff = a.template take<SigA>(k);
    d_Sk = a.template take<SigJ>(k);
    d_flag = a.template take<uint8_t>(2 * k);
  })));
  CK(cudaMemcpyAsync(d_gt, gts, 576 * k, cudaMemcpyHostToDevice, ctx->stream));
  CK(cudaMemcpyAsync(d_sb, sums, Ls * k, cudaMemcpyHostToDevice, ctx->stream));
  CK(cudaMemsetAsync(d_flag, 0, 2 * k, ctx->stream));
  LAUNCH(k_fp12_from_bytes, blocks_for(12 * k), TPB, k, (const uint8_t*)d_gt, d_Fk, d_flag);
  CKR((decode_points<SigA>(ctx, k, (const uint8_t*)d_sb, 1, d_aff, d_flag + k)));
  LAUNCH((k_aff_to_jac<SigA>), blocks_for(k), TPB, k, (const SigA*)d_aff, d_Sk);
  std::vector<uint8_t> flag(2 * k);
  CK(cudaMemcpyAsync(flag.data(), d_flag, 2 * k, cudaMemcpyDeviceToHost, ctx->stream));
  CK(cudaStreamSynchronize(ctx->stream));
  for (uint8_t f : flag)
    if (f) return arg_error(ctx, what, "a partial result is not a canonical field element / group element");
  bool ok = false;
  CKR((fold_check<PkA, SigA>(ctx, k, d_Fk, d_Sk, &ok)));
  *ok_out = ok ? 1 : 0;
  return BLSGPU_OK;
}
}  // namespace

int blsgpu_miller_partial(blsgpu_ctx* ctx, int impl_id, int scheme, int format, size_t n, const uint8_t* pks, const uint8_t* sigs,
                          const uint8_t* msgs, const uint64_t* msg_off, uint8_t gt_out[576], uint8_t* sum_out) {
  NVTX_RANGE("blsgpu_miller_partial");
  if (!ctx) return BLSGPU_E_ARG;
  if (!args_ok(impl_id, scheme, format) || !gt_out || !sum_out || (n && (!pks || !sigs))) return arg_error(ctx, __func__, "bad arguments");
  const size_t Ls = impl_id == 2 ? 96 : 48;
  if (n == 0) {  // the empty slice: (1, O)
    ctx->pending.reset();
    memset(gt_out, 0, 576);
    gt_out[47] = 1;
    memset(sum_out, 0, Ls);
    sum_out[0] = 0xc0;
    return BLSGPU_OK;
  }
  CKR(check_records(ctx, __func__, "msgs", msgs, "msg_off", msg_off, n));
  DstParam dst;
  make_dst(dst, impl_id, scheme, false);
  const int mode = scheme == 1 ? 1 : 0;
  return with_impl(impl_id, [&](auto I) { return miller_partial_impl<I>(ctx, mode, dst, format, n, pks, sigs, msgs, msg_off, gt_out, sum_out); });
}

int blsgpu_final_exp_is_one(blsgpu_ctx* ctx, int impl_id, size_t k, const uint8_t* partial_gts, const uint8_t* partial_sums, int* is_one_out) {
  NVTX_RANGE("blsgpu_final_exp_is_one");
  if (!ctx) return BLSGPU_E_ARG;
  if ((impl_id != 1 && impl_id != 2) || k == 0 || k > 16 || !partial_gts || !partial_sums || !is_one_out)
    return arg_error(ctx, __func__, "bad arguments (1 to 16 partial results)");
  CKR(set_device(ctx));
  return with_impl(impl_id, [&](auto I) { return fold_bytes_impl<I>(ctx, __func__, k, partial_gts, partial_sums, is_one_out); });
}

int blsgpu_partial_finish(blsgpu_ctx* ctx, int batch_ok, uint8_t* status_out) {
  NVTX_RANGE("blsgpu_partial_finish");
  if (!ctx) return BLSGPU_E_ARG;
  if (!ctx->pending) return BLSGPU_OK;  // an empty slice, or nothing pending
  if (!status_out) return arg_error(ctx, __func__, "status_out is null");
  std::unique_ptr<PendingSlice> p = std::move(ctx->pending);
  return p->finish(ctx, batch_ok != 0, status_out);
}

int blsgpu_verify_batch(blsgpu_ctx* ctx, int impl_id, int scheme, int format, size_t n, const uint8_t* pks, const uint8_t* sigs,
                        const uint8_t* msgs, const uint64_t* msg_off, uint8_t* status_out) {
  NVTX_RANGE("blsgpu_verify_batch");
  if (!ctx) return BLSGPU_E_ARG;
  return verify_batch_common(ctx, __func__, impl_id, scheme, format, n, pks, sigs, msgs, msg_off, status_out);
}

int blsgpu_pop_verify_batch(blsgpu_ctx* ctx, int impl_id, int format, size_t n, const uint8_t* pks, const uint8_t* sigs,
                            uint8_t* status_out) {
  NVTX_RANGE("blsgpu_pop_verify_batch");
  if (!ctx) return BLSGPU_E_ARG;
  if (!args_ok(impl_id, 2, format) || (n && (!pks || !sigs || !status_out))) return arg_error(ctx, __func__, "bad arguments");
  if (n == 0) return BLSGPU_OK;
  DstParam dst;
  make_dst(dst, impl_id, 2, true);
  return verify_host_common(ctx, impl_id, 2, dst, format, n, pks, sigs, nullptr, nullptr, status_out);
}

// AggregateSignature::verify in phases, so that a context on several devices can cut the pairs over its devices (SURVEY 8e,
// cfg 4): (1) every device decodes its slice of the keys (the first one also the signature), (2) the host applies the
// reference's checks in the reference's order over the whole input, (3) every device hashes its messages and folds its pairs
// into one product of Miller values, (4) the products meet on the first device: one Miller loop against -g, one final
// exponentiation.
template <int IMPL>
struct AggSlice {
  typedef typename ImplT<IMPL>::PkAff PkA;
  typedef typename ImplT<IMPL>::SigAff SigA;
  size_t n = 0;
  PkA* d_pk = nullptr;
  SigA *d_sig = nullptr, *d_h = nullptr;
  uint8_t *d_msgs = nullptr, *d_status = nullptr;
  uint64_t* d_off = nullptr;
  typename PtInfo<SigA>::Jac* d_hj = nullptr;
  Pipe<PkA, SigA> P;
};
// (1) st_out[n] and inf_out[n] get the slice's decode statuses and identity flags; with `sig` also st_out[n] / inf_out[n]
// (the signature's); without it the slice's signature slot holds the identity (it adds nothing to the fold).
template <int IMPL>
static int agg_decode(blsgpu_ctx* ctx, AggSlice<IMPL>& S, int format, size_t n, const uint8_t* pks, const uint8_t* msgs, const uint64_t* msg_off,
                      const uint8_t* sig, uint8_t* st_out, uint32_t* inf_out) {
  typedef typename ImplT<IMPL>::PkAff PkA;
  typedef typename ImplT<IMPL>::SigAff SigA;
  const size_t pk_len = PtInfo<PkA>::LEN, sig_len = PtInfo<SigA>::LEN;
  S.n = n;
  uint8_t *d_pks, *d_sigb, *d_stpk;
  // every take of the slice: its inputs and decoded points here, the hash scratch and the pipeline for agg_partials
  auto takes = [&](auto& a, size_t chunk) {
    d_pks = take_up<uint8_t>(a, n * pk_len);
    take_records(a, msg_off, n, S.d_msgs, S.d_off);
    d_sigb = a.template take<uint8_t>(sig_len);
    S.d_pk = a.template take<PkA>(std::max<size_t>(n, 1));
    S.d_sig = a.template take<SigA>(1);
    S.d_h = a.template take<SigA>(std::max<size_t>(n, 1));
    d_stpk = a.template take<uint8_t>(n + 1);
    S.d_status = a.template take<uint8_t>(std::max<size_t>(n, 1));
    S.d_hj = take_hash_scratch<SigA>(a, n);
    take_pipe(a, S.P, ctx, n, false, chunk);
  };
  CKR(ensure_miller_arena(ctx, n, takes));
  takes(ctx->arena, ctx->m6_chunk);
  CKR(upload(ctx, d_pks, pks, n * pk_len));
  CKR(upload_records(ctx, msgs, msg_off, n, S.d_msgs, S.d_off));
  stage_reset(ctx);
  if (n) CKR((decode_points<PkA>(ctx, n, (const uint8_t*)d_pks, format, S.d_pk, d_stpk)));
  if (sig) {
    CK(cudaMemcpyAsync(d_sigb, sig, sig_len, cudaMemcpyHostToDevice, ctx->stream));
    CKR((decode_points<SigA>(ctx, (size_t)1, (const uint8_t*)d_sigb, format, S.d_sig, d_stpk + n)));
  } else {
    SigA ident;
    memset(&ident, 0, sizeof(ident));
    ident.inf = 1;
    CK(cudaMemcpyAsync(S.d_sig, &ident, sizeof(ident), cudaMemcpyHostToDevice, ctx->stream));  // pageable source: staged before the call returns
  }
  CK(cudaMemcpyAsync(st_out, d_stpk, n + (sig ? 1 : 0), cudaMemcpyDeviceToHost, ctx->stream));
  // identity flags: read the `inf` words back (strided copy)
  if (n) CK(cudaMemcpy2DAsync(inf_out, 4, reinterpret_cast<const uint8_t*>(S.d_pk) + offsetof(PkA, inf), sizeof(PkA), 4, n, cudaMemcpyDeviceToHost,
                              ctx->stream));
  if (sig) CK(cudaMemcpyAsync(inf_out + n, reinterpret_cast<const uint8_t*>(S.d_sig) + offsetof(SigA, inf), 4, cudaMemcpyDeviceToHost, ctx->stream));
  CK(cudaStreamSynchronize(ctx->stream));
  return BLSGPU_OK;
}
// (2) the reference's checks before any pairing work, in its order (sig_core.rs:149-178, sig_basic.rs:46-58); true = decided
static bool agg_host_checks(int scheme, size_t n, const uint8_t* st, const uint32_t* inf, const uint8_t* msgs, const uint64_t* msg_off,
                            uint8_t* status_out, int64_t index_out[2]) {
  index_out[0] = index_out[1] = -1;
  for (size_t i = 0; i < n; i++)
    if (st[i] != BLSGPU_ST_OK) {
      *status_out = st[i];
      index_out[0] = (int64_t)i;
      return true;
    }
  if (st[n] != BLSGPU_ST_OK) {
    *status_out = st[n];
    return true;
  }
  if (scheme == 0) {
    // Basic: duplicate messages are rejected before any curve work (reference src/traits/sig_basic.rs:46-58)
    std::unordered_map<std::string, size_t> seen;
    seen.reserve(n * 2);
    for (size_t i = 0; i < n; i++) {
      std::string m(reinterpret_cast<const char*>(msgs + msg_off[i]), (size_t)(msg_off[i + 1] - msg_off[i]));
      auto it = seen.find(m);
      if (it != seen.end()) {
        *status_out = BLSGPU_ST_DUPLICATE_MESSAGES;
        index_out[0] = (int64_t)it->second;
        index_out[1] = (int64_t)i;
        return true;
      }
      seen.emplace(std::move(m), i);
    }
  }
  if (inf[n]) {
    *status_out = BLSGPU_ST_SIG_IDENTITY;
    return true;
  }
  for (size_t i = 0; i < n; i++)
    if (inf[i]) {
      *status_out = BLSGPU_ST_PK_IDENTITY;
      index_out[0] = (int64_t)i + 1;  // the reference reports i+1 (sig_core.rs:162-167)
      return true;
    }
  if (n == 0) {
    // only the (sig, -g) pair remains and sig != identity: never the Gt identity (SURVEY appendix A)
    *status_out = BLSGPU_ST_INVALID_SIGNATURE;
    return true;
  }
  return false;
}
// (3) hash the slice's messages, Miller loops of its pairs, product tree: S.P.rootF() / S.P.rootS() (the stream is NOT synchronised)
template <int IMPL>
static int agg_partials(blsgpu_ctx* ctx, AggSlice<IMPL>& S, int scheme) {
  typedef typename ImplT<IMPL>::PkAff PkA;
  typedef typename ImplT<IMPL>::SigAff SigA;
  DstParam dst;
  make_dst(dst, IMPL, scheme, false);
  CK(cudaMemsetAsync(S.d_status, 0, S.n, ctx->stream));
  CKR((hash_points<SigA, PkA>(ctx, S.n, (const uint8_t*)S.d_msgs, (const uint64_t*)S.d_off, scheme == 1 ? 1 : 0, (const PkA*)S.d_pk,
                              (const uint8_t*)nullptr, dst, S.d_hj, S.d_h)));
  return pipeline_partials<PkA, SigA>(ctx, S.P, S.d_pk, S.d_sig, S.d_h, S.d_status);
}
template <int IMPL>
static int aggregate_verify_impl(blsgpu_ctx* ctx, int scheme, int format, size_t n, const uint8_t* pks, const uint8_t* msgs,
                                 const uint64_t* msg_off, const uint8_t* sig, uint8_t* status_out, int64_t index_out[2]) {
  typedef typename ImplT<IMPL>::PkAff PkA;
  typedef typename ImplT<IMPL>::SigAff SigA;
  AggSlice<IMPL> S;
  std::vector<uint8_t> st(n + 1);
  std::vector<uint32_t> inf(n + 1, 0);
  CKR((agg_decode<IMPL>(ctx, S, format, n, pks, msgs, msg_off, sig, st.data(), inf.data())));
  if (agg_host_checks(scheme, n, st.data(), inf.data(), msgs, msg_off, status_out, index_out)) return BLSGPU_OK;
  CKR((agg_partials<IMPL>(ctx, S, scheme)));
  bool ok = false;
  CKR((pipeline_check<PkA, SigA>(ctx, S.P, &ok)));
  stage_mark(ctx, BLSGPU_STAGE_COUNT);
  *status_out = ok ? BLSGPU_ST_OK : BLSGPU_ST_INVALID_SIGNATURE;
  return BLSGPU_OK;
}
// the same over the devices of a context: contiguous slices of the pairs, the signature travels with the first slice
template <int IMPL>
static int aggregate_verify_multi(blsgpu_ctx* ctx, int scheme, int format, size_t n, const uint8_t* pks, const uint8_t* msgs,
                                  const uint64_t* msg_off, const uint8_t* sig, uint8_t* status_out, int64_t index_out[2]) {
  typedef typename ImplT<IMPL>::PkAff PkA;
  typedef typename ImplT<IMPL>::SigAff SigA;
  const size_t ndev = 1 + ctx->peers.size(), pk_len = PtInfo<PkA>::LEN;
  std::vector<AggSlice<IMPL>> S(ndev);
  std::vector<uint8_t> st(n + 1);
  std::vector<uint32_t> inf(n + 1, 0);
  auto lo = [&](size_t d) { return n * d / ndev; };
  // the signature's status and identity flag come back at the END of slice 0's arrays: stage them, then move them to [n]
  std::vector<uint8_t> st0(lo(1) + 1);
  std::vector<uint32_t> inf0(lo(1) + 1, 0);
  CKR(run_on_devices(ctx, [&](blsgpu_ctx* c, size_t d) {
    const size_t s0 = lo(d), cnt = lo(d + 1) - s0;
    return agg_decode<IMPL>(c, S[d], format, cnt, pks + s0 * pk_len, msgs, msg_off + s0, d == 0 ? sig : nullptr,
                            d == 0 ? st0.data() : st.data() + s0, d == 0 ? inf0.data() : inf.data() + s0);
  }));
  std::copy(st0.begin(), st0.end() - 1, st.begin());
  std::copy(inf0.begin(), inf0.end() - 1, inf.begin());
  st[n] = st0.back();
  inf[n] = inf0.back();
  if (agg_host_checks(scheme, n, st.data(), inf.data(), msgs, msg_off, status_out, index_out)) return BLSGPU_OK;
  CKR(run_on_devices(ctx, [&](blsgpu_ctx* c, size_t d) {
    int rc = agg_partials<IMPL>(c, S[d], scheme);
    if (rc != BLSGPU_OK) return rc;
    if (cudaStreamSynchronize(c->stream) != cudaSuccess) {
      c->err = "aggregate_verify: device synchronisation failed";
      return (int)BLSGPU_E_CUDA;
    }
    return (int)BLSGPU_OK;
  }));
  std::vector<const Pipe<PkA, SigA>*> roots;
  for (const AggSlice<IMPL>& slice : S) roots.push_back(&slice.P);
  bool ok = false;
  CKR((fold_roots<PkA, SigA>(ctx, roots, &ok)));
  *status_out = ok ? BLSGPU_ST_OK : BLSGPU_ST_INVALID_SIGNATURE;
  return BLSGPU_OK;
}

int blsgpu_aggregate_verify(blsgpu_ctx* ctx, int impl_id, int scheme, int format, size_t n, const uint8_t* pks, const uint8_t* msgs,
                            const uint64_t* msg_off, const uint8_t* sig, uint8_t* status_out, int64_t index_out[2]) {
  NVTX_RANGE("blsgpu_aggregate_verify");
  if (!ctx) return BLSGPU_E_ARG;
  int64_t dummy[2];
  if (!index_out) index_out = dummy;
  if (!args_ok(impl_id, scheme, format) || !sig || !status_out || (n && !pks)) return arg_error(ctx, __func__, "bad arguments");
  CKR(check_records(ctx, __func__, "msgs", msgs, "msg_off", msg_off, n));
  CKR(set_device(ctx));
  const bool multi = !ctx->peers.empty() && n >= (1 + ctx->peers.size()) * SHARD_MIN_ITEMS;
  return with_impl(impl_id, [&](auto I) {
    return multi ? aggregate_verify_multi<I>(ctx, scheme, format, n, pks, msgs, msg_off, sig, status_out, index_out)
                 : aggregate_verify_impl<I>(ctx, scheme, format, n, pks, msgs, msg_off, sig, status_out, index_out);
  });
}

// ---------------------------------------------------------------------------------------------------------------------
// q x AggregateSignature::verify in one pipeline.  The host applies agg_host_checks per aggregate; the live aggregates share
// one Miller stage in which aggregate j fills whole groups of slots and every pair of it is scaled by ONE scalar r_j, so
//   F_j = prod_{i in j} ML(r_j pk_i, H_i)          (segmented product of its groups' values)
//   S_j = r_j sig_j                                   (k_scale_sig with the aggregate as the item)
// and a 16-ary tree over the q leaves (F_j, S_j) is checked at its root and descended with node probes on failure.
// set_off / msg_off start at 0 here (the entry point rebases them).
template <int IMPL>
static int aggregate_batch_impl(blsgpu_ctx* ctx, int scheme, int format, size_t q, const uint64_t* set_off, const uint8_t* pks,
                                const uint8_t* msgs, const uint64_t* msg_off, const uint8_t* sigs, uint8_t* status_out, int64_t* index_out) {
  typedef typename ImplT<IMPL>::PkAff PkA;
  typedef typename ImplT<IMPL>::SigAff SigA;
  typedef typename PtInfo<SigA>::Jac SigJ;
  const size_t Lp = PtInfo<PkA>::LEN, Ls = PtInfo<SigA>::LEN;
  const size_t np = (size_t)set_off[q], msg_bytes = (size_t)msg_off[np];
  // layout: aggregate j owns groups g_first[j] .. g_first[j+1]-1, at least one (an empty or decided aggregate's group is all
  // padding, so its F_j is 1)
  std::vector<size_t> g_first(q + 1, 0);
  for (size_t j = 0; j < q; j++) g_first[j + 1] = g_first[j] + std::max<size_t>(1, (size_t)(set_off[j + 1] - set_off[j] + M6_GROUP - 1) / M6_GROUP);
  const size_t ng = g_first[q], nslots = ng * M6_GROUP;
  // the segmented product: levels of ranges of <= 16 consecutive nodes of one aggregate, until one node per aggregate
  std::vector<size_t> cnt(q);
  for (size_t j = 0; j < q; j++) cnt[j] = g_first[j + 1] - g_first[j];
  const SegLevels seg = seg_levels(std::move(cnt));
  const std::vector<uint32_t>& seg_off = seg.off;
  const size_t seg_total = seg.below_top();  // the last level is the set tree's leaves
  Pipe<PkA, SigA> P;
  P.lv = make_levels(q);
  const size_t qtotal = levels_total(P.lv), ndig = levels_total(make_levels(np + q));
  uint8_t *d_pkb, *d_sigb, *d_msgs, *d_st, *d_pair_pre, *d_agg_pre, *d_pres;
  uint64_t *d_moff, *d_soff;
  uint32_t *d_src, *d_gset, *d_segoff;
  PkA *d_pk, *d_pks;
  SigA *d_sig, *d_h, *d_hs;
  SigJ* d_hj;
  Digest* d_dig;
  Fp12* d_Fseg;
  auto takes = [&](auto& a, size_t chunk) {
    d_pkb = take_up<uint8_t>(a, np * Lp);
    d_sigb = take_up<uint8_t>(a, q * Ls);
    d_msgs = take_up<uint8_t>(a, msg_bytes);
    d_moff = take_up<uint64_t>(a, np + 1);
    d_soff = take_up<uint64_t>(a, q + 1);
    d_pk = a.template take<PkA>(std::max<size_t>(np, 1));
    d_sig = a.template take<SigA>(q);
    d_st = a.template take<uint8_t>(np + q);  // decode statuses: the pks, then the signatures
    d_pair_pre = take_up<uint8_t>(a, np);
    d_agg_pre = take_up<uint8_t>(a, q);
    d_src = take_up<uint32_t>(a, nslots);
    d_gset = take_up<uint32_t>(a, ng);
    d_segoff = take_up<uint32_t>(a, seg_off.size());
    d_h = a.template take<SigA>(std::max<size_t>(np, 1));
    d_hj = take_hash_scratch<SigA>(a, np);
    d_dig = a.template take<Digest>(ndig + 2);
    d_pks = a.template take<PkA>(nslots);
    d_hs = a.template take<SigA>(nslots);
    d_pres = a.template take<uint8_t>(nslots);
    // the pipe of the set tree: leaves (F_j, S_j), probe scratch, the Miller stage's line buffers
    P.d_F = a.template take<Fp12>(qtotal);
    P.d_S = a.template take<SigJ>(qtotal);
    take_probe_scratch(a, P, probe_cap(q));
    d_Fseg = a.template take<Fp12>(std::max<size_t>(seg_total, 1));
    take_lines(a, P, nslots, chunk);
  };
  CKR(ensure_miller_arena(ctx, nslots, takes));
  takes(ctx->arena, ctx->m6_chunk);
  stage_reset(ctx);
  CKR(upload(ctx, d_pkb, pks, np * Lp));
  CKR(upload(ctx, d_sigb, sigs, q * Ls));
  CKR(upload(ctx, d_msgs, msgs, msg_bytes));
  CKR(upload(ctx, d_moff, msg_off, np + 1));
  CKR(upload(ctx, d_soff, set_off, q + 1));
  stage_mark(ctx, BLSGPU_STAGE_DECODE_PK);
  if (np) CKR((decode_points<PkA>(ctx, np, (const uint8_t*)d_pkb, format, d_pk, d_st, BLSGPU_KERNEL_DECODE_PK)));
  stage_mark(ctx, BLSGPU_STAGE_DECODE_SIG);
  CKR((decode_points<SigA>(ctx, q, (const uint8_t*)d_sigb, format, d_sig, d_st + np, BLSGPU_KERNEL_DECODE_SIG)));
  std::vector<uint8_t> st(np + q);
  std::vector<uint32_t> inf(np + q);
  CK(cudaMemcpyAsync(st.data(), d_st, np + q, cudaMemcpyDeviceToHost, ctx->stream));
  if (np) CK(cudaMemcpy2DAsync(inf.data(), 4, reinterpret_cast<const uint8_t*>(d_pk) + offsetof(PkA, inf), sizeof(PkA), 4, np, cudaMemcpyDeviceToHost,
                               ctx->stream));
  CK(cudaMemcpy2DAsync(inf.data() + np, 4, reinterpret_cast<const uint8_t*>(d_sig) + offsetof(SigA, inf), sizeof(SigA), 4, q, cudaMemcpyDeviceToHost,
                       ctx->stream));
  CK(cudaStreamSynchronize(ctx->stream));
  // the reference's checks per aggregate, in its order; a decided aggregate takes no part in the pairing work
  std::vector<uint8_t> agg_pre(q, BLSGPU_ST_OK), pair_pre(np, PROBE_SKIP);
  std::vector<uint32_t> slot_src(nslots, 0xffffffffu), g_set(ng);
  size_t live = 0;
  {
    std::vector<uint8_t> st_j;
    std::vector<uint32_t> inf_j;
    for (size_t j = 0; j < q; j++) {
      const size_t lo = (size_t)set_off[j], n = (size_t)set_off[j + 1] - lo;
      st_j.assign(st.begin() + lo, st.begin() + lo + n);
      st_j.push_back(st[np + j]);
      inf_j.assign(inf.begin() + lo, inf.begin() + lo + n);
      inf_j.push_back(inf[np + j]);
      for (size_t g = g_first[j]; g < g_first[j + 1]; g++) g_set[g] = (uint32_t)j;
      if (agg_host_checks(scheme, n, st_j.data(), inf_j.data(), msgs, msg_off + lo, status_out + j, index_out + 2 * j)) {
        agg_pre[j] = PROBE_SKIP;
        continue;
      }
      live++;
      for (size_t i = 0; i < n; i++) {
        pair_pre[lo + i] = BLSGPU_ST_OK;
        slot_src[g_first[j] * M6_GROUP + i] = (uint32_t)(lo + i);
      }
    }
  }
  if (live == 0) {
    stage_collect(ctx);
    return BLSGPU_OK;
  }
  CKR(upload(ctx, d_pair_pre, pair_pre.data(), np));
  CKR(upload(ctx, d_agg_pre, agg_pre.data(), q));
  CKR(upload(ctx, d_src, slot_src.data(), nslots));
  CKR(upload(ctx, d_gset, g_set.data(), ng));
  CKR(upload(ctx, d_segoff, seg_off.data(), seg_off.size()));
  DstParam dst;
  make_dst(dst, IMPL, scheme, false);
  stage_mark(ctx, BLSGPU_STAGE_HASH);
  CKR((hash_points<SigA, PkA>(ctx, np, (const uint8_t*)d_msgs, (const uint64_t*)d_moff, scheme == 1 ? 1 : 0, (const PkA*)d_pk,
                              (const uint8_t*)d_pair_pre, dst, d_hj, d_h)));
  // the scalars: r_j = rlc_scalar(root, j), root = 16-ary SHA-256 tree over every pk, hashed message, signature and range
  Digest* d_root = d_dig + ndig;  // [root, salt]
  CKR(fresh_salt(ctx));
  LAUNCH((k_agg_leaf_digest<PkA, SigA>), blocks_for(np + q), TPB, np, q, (const PkA*)d_pk, (const SigA*)d_h, (const SigA*)d_sig,
         (const uint64_t*)d_soff, d_dig);
  CKR(digest_root(ctx, np + q, d_dig, d_root));
  LAUNCH((k_agg_slots<PkA, SigA>), blocks_for(nslots), TPB, nslots, (const uint32_t*)d_src, (const PkA*)d_pk, (const SigA*)d_h, d_pks, d_hs, d_pres);
  P.n = nslots;
  P.ng = q;
  P.use_rlc = true;
  P.use_msm = false;
  const int rbits = P.rbits = ctx->rlc_bits;
  P.d_pk = d_pks;
  P.d_h = d_hs;
  P.d_status = d_pres;
  P.d_root = d_root;
  CKR((set_probe_smem<PkA, SigA>(ctx)));
  stage_mark(ctx, BLSGPU_STAGE_SCALE_SIG);
  LAUNCH((k_scale_sig<SigA>), blocks_for(q), TPB, q, (const SigA*)d_sig, (const uint8_t*)d_agg_pre, (const Digest*)d_root, rbits, P.d_S);
  CK(cudaEventRecord(ctx->ev_fork, ctx->stream));
  P.root_T_ready = false;
  stage_mark(ctx, BLSGPU_STAGE_MILLER);
  const bool segmented = seg.n.size() > 1;  // some aggregate spans more than one group
  CKR((miller_stage<PkA, SigA>(ctx, P, nslots, d_pks, d_hs, d_pres, segmented ? d_Fseg : P.d_F,
                               [&](cudaStream_t s, size_t cn, size_t base, M6Arg* args) {
                                 k_m6_prep_sets<PkA, SigA><<<blocks_for(cn), TPB, 0, s>>>(cn, base, d_pks, d_hs, (const uint8_t*)d_pres,
                                                                                          (const uint32_t*)d_gset, (const Digest*)d_root, rbits, args);
                               })));
  stage_mark(ctx, BLSGPU_STAGE_REDUCE);
  CKR(seg_reduce_levels<Fp12>(ctx, seg, d_segoff, d_Fseg, P.d_F));
  CKR(reduce_levels(ctx, P.lv, 0, P.d_F, P.d_S));
  bool ok = false;
  CKR((pipeline_check<PkA, SigA>(ctx, P, &ok)));
  for (size_t j = 0; j < q; j++)
    if (agg_pre[j] == BLSGPU_ST_OK) status_out[j] = BLSGPU_ST_OK;
  if (!ok) {
    std::vector<uint32_t> bad;
    CKR((descend_tree<PkA, SigA>(ctx, P, bad, [](const std::vector<uint32_t>&) { return (int)BLSGPU_OK; })));
    // Leaf j is exact, not a probabilistic verdict: its probe is final_exp(F_j * ML(-g, r_j sig_j)) =
    // (prod_i e(pk_i, H_i) * e(-g, sig_j))^(3 r_j).  rlc_scalar never returns 0 and r_j < 2^128 < r, so gcd(3 r_j, r) = 1,
    // and Gt has prime order r: the leaf is 1 exactly when aggregate j is valid.  Only an ACCEPT rests on the combination
    // (probability >= 1 - 2^-bits per call, as for blsgpu_verify_batch).
    for (uint32_t j : bad) status_out[j] = BLSGPU_ST_INVALID_SIGNATURE;
  }
  stage_mark(ctx, BLSGPU_STAGE_COUNT);
  stage_collect(ctx);
  return BLSGPU_OK;
}

int blsgpu_aggregate_verify_batch(blsgpu_ctx* ctx, int impl_id, int scheme, int format, size_t q, const uint64_t* set_off, const uint8_t* pks,
                                  const uint8_t* msgs, const uint64_t* msg_off, const uint8_t* sigs, uint8_t* status_out, int64_t* index_out) {
  NVTX_RANGE("blsgpu_aggregate_verify_batch");
  if (!ctx) return BLSGPU_E_ARG;
  if (!args_ok(impl_id, scheme, format) || (q && (!sigs || !status_out))) return arg_error(ctx, __func__, "bad arguments");
  if (q == 0) return BLSGPU_OK;
  std::vector<uint64_t> so;
  CKR(check_sets(ctx, __func__, "set_off", set_off, q, MEMBERS_CAP, so));
  const size_t np = (size_t)so[q];
  Keys keys(pks);
  CKR(check_keys(ctx, __func__, impl_id, keys, set_off[0], np));
  CKR(check_buffer(ctx, __func__, "msg_off", msg_off, 1));
  msg_off += set_off[0];  // one message per pair
  CKR(check_records(ctx, __func__, "msgs", msgs, "msg_off", msg_off, np));
  CKR(set_device(ctx));
  std::vector<int64_t> idx_scratch;
  if (!index_out) {
    idx_scratch.resize(2 * q);
    index_out = idx_scratch.data();
  }
  const size_t pk_len = impl_id == 2 ? 48 : 96, sig_len = impl_id == 2 ? 96 : 48;
  // aggregates lo .. hi-1 on context c, with their pair and message offsets rebased to 0
  auto run = [&](blsgpu_ctx* c, size_t lo, size_t hi) -> int {
    const size_t a = (size_t)so[lo], b = (size_t)so[hi];
    const std::vector<uint64_t> s = rebased(so.data(), lo, hi), mo = rebased(msg_off, a, b);
    const uint8_t* pk = keys.bytes ? keys.bytes + a * pk_len : nullptr;
    const uint8_t* ms = msgs ? msgs + msg_off[a] : nullptr;
    return with_impl(impl_id, [&](auto I) {
      return aggregate_batch_impl<I>(c, scheme, format, hi - lo, s.data(), pk, ms, mo.data(), sigs + lo * sig_len, status_out + lo, index_out + 2 * lo);
    });
  };
  const size_t ndev = 1 + ctx->peers.size();
  if (ndev == 1 || np < ndev * SHARD_MIN_ITEMS) return run(ctx, 0, q);
  // aggregates are independent: contiguous runs per device, balanced by pair count, nothing to fold
  return run_cut(ctx, q, so.data(), run);
}

// ---------------------------------------------------------------------------------------------------------------------
// n x Signature::verify where many items share a message.  The batch equation of blsgpu_verify_batch regroups by bilinearity:
//   prod_i e(r_i pk_i, H(m_i)) = prod_l e(P_l, H_l),   P_l = sum_{i in leaf l} r_i pk_i
// so the q messages are hashed once each and the Miller stage runs once per LEAF (at most GROUPED_LEAF items of one message)
// instead of once per item.  The scalars are blsgpu_verify_batch's (rlc_scalar(root, i), item order), the root binds every
// pk, signature, message hash and message index.  A failing check descends the tree of Miller groups of leaves, probes the
// leaves of the failing groups, and decides every item of a failing leaf by its own exact equation (DESIGN.md section 2).
#ifndef BLSGPU_GROUPED_LEAF
#define BLSGPU_GROUPED_LEAF 96
#endif
namespace {
constexpr uint32_t GROUPED_LEAF = BLSGPU_GROUPED_LEAF;  // items per leaf at most (DESIGN.md section 6: the measured trade)
constexpr uint32_t LEAF_MSM_MIN = 16;  // leaves with fewer items take k_leaf_scale: 32 lanes of buckets do not pay below this
template <class PkA, class SigA>
struct Grouped {
  typedef typename PtInfo<PkA>::Jac PkJ;
  typedef typename PtInfo<SigA>::Jac SigJ;
  size_t n = 0, q = 0, nl = 0, nbig = 0, nsmall = 0, msg_bytes = 0, blocks = 1;
  bool keyed = false;  // the keys come from a key set: key indices instead of key bytes
  uint8_t *pkb, *sigb, *msgs, *mpre, *stpk, *stsig, *status, *lpre;
  uint32_t* kidx;
  uint64_t* moff;
  uint32_t *midx, *order, *big, *small;  // big / small: the leaves of k_leaf_msm / k_leaf_scale
  GLeaf* leaves;
  PkA* pk;
  SigA *sig, *hq, *hl;  // hq: per message, hl: per leaf
  SigJ* hj;             // hash_points' scratch
  Digest* dig;          // leaf digests, their tree, [root, salt]
  RlcScalar* r;         // the scalars of the per-item route (the bucket route's come from msm_sum)
  SigJ* s_item;         // per-item route: r_i sig_i and the tree over them
  PkJ *p_jac, *p_buckets, *p_W;
  PkA* p_aff;
  SigJ *s_jac, *s_buckets, *s_W;  // failure path: S_l per leaf
  SigA* s_aff;
  Pipe<PkA, SigA> P;  // the tree over the Miller groups of leaves
};
// every take of the grouped pipeline, with Miller line buffers for passes of `chunk` leaves
template <class PkA, class SigA, class A>
void take_grouped(A& a, Grouped<PkA, SigA>& G, int rbits, size_t chunk) {
  typedef typename Grouped<PkA, SigA>::PkJ PkJ;
  typedef typename Grouped<PkA, SigA>::SigJ SigJ;
  const size_t n = G.n, nl = G.nl, ng = (nl + M6_GROUP - 1) / M6_GROUP, ndig = levels_total(make_levels(n));
  if (G.keyed)
    G.kidx = a.template take<uint32_t>(n);
  else
    G.pkb = a.template take<uint8_t>(n * PtInfo<PkA>::LEN);
  G.sigb = a.template take<uint8_t>(n * PtInfo<SigA>::LEN);
  G.msgs = a.template take<uint8_t>(std::max<size_t>(G.msg_bytes, 1));
  G.moff = a.template take<uint64_t>(G.q + 1);
  G.mpre = a.template take<uint8_t>(G.q);
  G.midx = a.template take<uint32_t>(n);
  G.order = a.template take<uint32_t>(n);
  G.leaves = a.template take<GLeaf>(nl);
  G.big = a.template take<uint32_t>(std::max<size_t>(G.nbig, 1));
  G.small = a.template take<uint32_t>(std::max<size_t>(G.nsmall, 1));
  G.pk = a.template take<PkA>(n);
  G.sig = a.template take<SigA>(n);
  G.stpk = a.template take<uint8_t>(n);
  G.stsig = a.template take<uint8_t>(n);
  G.status = a.template take<uint8_t>(n);
  G.hq = a.template take<SigA>(G.q);
  G.hj = take_hash_scratch<SigA>(a, G.q);
  G.dig = a.template take<Digest>(ndig + 2);
  if (n < MSM_MIN_ITEMS) {
    G.r = a.template take<RlcScalar>(n);
    G.s_item = a.template take<SigJ>(ndig);
  }
  G.p_jac = a.template take<PkJ>(nl);
  G.p_aff = a.template take<PkA>(nl);
  G.hl = a.template take<SigA>(nl);
  G.lpre = a.template take<uint8_t>(nl);
  G.p_buckets = a.template take<PkJ>(G.nbig ? G.blocks * 128 * LEAF_BUCKETS : 1);
  G.p_W = a.template take<PkJ>(G.nbig * 32 + 1);
  G.s_jac = a.template take<SigJ>(nl);
  G.s_aff = a.template take<SigA>(nl);
  G.s_buckets = a.template take<SigJ>(G.nbig ? G.blocks * 128 * LEAF_BUCKETS : 1);
  G.s_W = a.template take<SigJ>(G.nbig * 32 + 1);
  const size_t gtotal = levels_total(make_levels(ng));
  G.P.d_F = a.template take<Fp12>(gtotal);
  G.P.d_S = a.template take<SigJ>(gtotal);
  take_probe_scratch(a, G.P, probe_cap(ng));
  if (n >= MSM_MIN_ITEMS) take_msm(a, n, MsmPlan(n, rbits), G.P.msm);
  take_lines(a, G.P, nl, chunk);
}
// sum_{i in l} r_i * pts[i] into out[l] for every leaf: the bucket kernel for the big leaves, per-item scaling for the small
template <class A, class G>
int leaf_sums(blsgpu_ctx* ctx, const G& g, const A* pts, const RlcScalar* d_r, int rbits, typename PtInfo<A>::Jac* buckets,
              typename PtInfo<A>::Jac* W, typename PtInfo<A>::Jac* out) {
  typedef typename PtInfo<A>::Jac J;
  if (g.nbig) {
    LAUNCH((k_leaf_msm<A>), (unsigned)g.blocks, 128, g.nbig, (const uint32_t*)g.big, (const GLeaf*)g.leaves, (const uint32_t*)g.order, pts, d_r,
           rbits, buckets, W);
    LAUNCH((k_leaf_combine<J>), blocks_for(g.nbig), TPB, g.nbig, (const uint32_t*)g.big, rbits, (const J*)W, out);
  }
  if (g.nsmall)
    LAUNCH((k_leaf_scale<A>), blocks_for(g.nsmall), TPB, g.nsmall, (const uint32_t*)g.small, (const GLeaf*)g.leaves, (const uint32_t*)g.order, pts,
           d_r, rbits, out);
  return BLSGPU_OK;
}

template <int IMPL>
int verify_grouped_impl(blsgpu_ctx* ctx, int scheme, int format, size_t n, const Keys& keys, const uint8_t* sigs, const uint32_t* msg_idx,
                        size_t q, const uint8_t* msgs, const uint64_t* msg_off, uint8_t* status_out) {
  typedef typename ImplT<IMPL>::PkAff PkA;
  typedef typename ImplT<IMPL>::SigAff SigA;
  typedef typename PtInfo<PkA>::Jac PkJ;
  typedef typename PtInfo<SigA>::Jac SigJ;
  // group: counting sort of the items by message, then every message's run cut into leaves
  std::vector<uint32_t> order(n), start(q + 1, 0);
  for (size_t i = 0; i < n; i++) start[msg_idx[i] + 1]++;
  for (size_t j = 0; j < q; j++) start[j + 1] += start[j];
  {
    std::vector<uint32_t> cur(start.begin(), start.end() - 1);
    for (size_t i = 0; i < n; i++) order[cur[msg_idx[i]]++] = (uint32_t)i;
  }
  std::vector<GLeaf> leaves;
  std::vector<uint32_t> big, small;
  std::vector<uint8_t> mpre(q, PROBE_SKIP);  // a message no item signs is not hashed
  for (size_t j = 0; j < q; j++)
    for (uint32_t f = start[j]; f < start[j + 1]; f += GROUPED_LEAF) {
      const uint32_t cnt = std::min(GROUPED_LEAF, start[j + 1] - f);
      (cnt >= LEAF_MSM_MIN ? big : small).push_back((uint32_t)leaves.size());
      leaves.push_back({f, cnt, (uint32_t)j});
      mpre[j] = BLSGPU_ST_OK;
    }
  Grouped<PkA, SigA> G;
  G.n = n;
  G.q = q;
  G.keyed = keys.set != nullptr;
  G.nl = leaves.size();
  G.nbig = big.size();
  G.nsmall = small.size();
  G.msg_bytes = (size_t)(msg_off[q] - msg_off[0]);
  G.blocks = node_msm_blocks(ctx, G.nbig);
  const int rbits = ctx->rlc_bits;
  CKR(ensure_miller_arena(ctx, G.nl, [&](auto& a, size_t chunk) { take_grouped(a, G, rbits, chunk); }));
  take_grouped(ctx->arena, G, rbits, ctx->m6_chunk);
  ARENA_OK();
  Pipe<PkA, SigA>& P = G.P;
  stage_reset(ctx);
  const std::vector<uint64_t> moff = rebased(msg_off, 0, q);
  Keys d_keys = keys;
  if (G.keyed) {
    CK(cudaMemcpyAsync(G.kidx, keys.idx, n * 4, cudaMemcpyHostToDevice, ctx->stream));
    d_keys.idx = G.kidx;
  } else {
    CK(cudaMemcpyAsync(G.pkb, keys.bytes, n * PtInfo<PkA>::LEN, cudaMemcpyHostToDevice, ctx->stream));
    d_keys.bytes = G.pkb;
  }
  CK(cudaMemcpyAsync(G.sigb, sigs, n * PtInfo<SigA>::LEN, cudaMemcpyHostToDevice, ctx->stream));
  if (G.msg_bytes) CK(cudaMemcpyAsync(G.msgs, msgs + msg_off[0], G.msg_bytes, cudaMemcpyHostToDevice, ctx->stream));
  CK(cudaMemcpyAsync(G.moff, moff.data(), (q + 1) * 8, cudaMemcpyHostToDevice, ctx->stream));
  CK(cudaMemcpyAsync(G.mpre, mpre.data(), q, cudaMemcpyHostToDevice, ctx->stream));
  CK(cudaMemcpyAsync(G.midx, msg_idx, n * 4, cudaMemcpyHostToDevice, ctx->stream));
  CK(cudaMemcpyAsync(G.order, order.data(), n * 4, cudaMemcpyHostToDevice, ctx->stream));
  CK(cudaMemcpyAsync(G.leaves, leaves.data(), G.nl * sizeof(GLeaf), cudaMemcpyHostToDevice, ctx->stream));
  if (G.nbig) CK(cudaMemcpyAsync(G.big, big.data(), G.nbig * 4, cudaMemcpyHostToDevice, ctx->stream));
  if (G.nsmall) CK(cudaMemcpyAsync(G.small, small.data(), G.nsmall * 4, cudaMemcpyHostToDevice, ctx->stream));
  // decode, per-item statuses (item order throughout)
  stage_mark(ctx, BLSGPU_STAGE_DECODE_PK);
  CKR((load_keys<PkA>(ctx, n, d_keys, format, G.pk, G.stpk)));
  stage_mark(ctx, BLSGPU_STAGE_DECODE_SIG);
  CKR((decode_points<SigA>(ctx, n, (const uint8_t*)G.sigb, format, G.sig, G.stsig, BLSGPU_KERNEL_DECODE_SIG)));
  LAUNCH((k_prestatus<PkA, SigA>), blocks_for(n), TPB, n, (const uint8_t*)G.stpk, (const uint8_t*)G.stsig, (const PkA*)G.pk, (const SigA*)G.sig,
         G.status);
  // one hash per message, then the scalars of blsgpu_verify_batch
  stage_mark(ctx, BLSGPU_STAGE_HASH);
  DstParam dst;
  make_dst(dst, IMPL, scheme, false);
  CKR((hash_points<SigA, PkA>(ctx, q, (const uint8_t*)G.msgs, (const uint64_t*)G.moff, 0, (const PkA*)nullptr, (const uint8_t*)G.mpre, dst, G.hj, G.hq)));
  CKR(fresh_salt(ctx));
  const size_t ndig = levels_total(make_levels(n));
  Digest* d_root = G.dig + ndig;
  LAUNCH((k_grouped_leaf_digest<PkA, SigA>), blocks_for(n), TPB, n, (const PkA*)G.pk, (const SigA*)G.sig, (const SigA*)G.hq, (const uint32_t*)G.midx,
         G.dig);
  CKR(digest_root(ctx, n, G.dig, d_root));
  // the signature side: S = sum r_i sig_i (the bucket method, or per-item scaling and a tree for small batches)
  stage_mark(ctx, BLSGPU_STAGE_SCALE_SIG);
  RlcScalar* d_r = nullptr;
  SigJ* d_S = nullptr;
  if (n >= MSM_MIN_ITEMS) {
    CKR((msm_sum<SigA>(ctx, n, G.sig, G.status, d_root, rbits, P.msm, &d_S)));
    d_r = P.msm.r;
  } else {
    d_r = G.r;
    const std::vector<Level> lvn = make_levels(n);
    LAUNCH(k_msm_count, blocks_for(n), TPB, n, (const uint8_t*)G.status, (const Digest*)d_root, rbits, 0, 0, d_r, (uint32_t*)nullptr);
    LAUNCH((k_scale_sig<SigA>), blocks_for(n), TPB, n, (const SigA*)G.sig, (const uint8_t*)G.status, (const Digest*)d_root, rbits, G.s_item);
    CKR(reduce_levels(ctx, lvn, 0, nullptr, G.s_item));
    d_S = G.s_item + lvn.back().off;
  }
  // the key side: P_l = sum_{i in l} r_i pk_i, affine, with H of the leaf's message
  stage_mark(ctx, BLSGPU_STAGE_MILLER);
  CKR((leaf_sums<PkA>(ctx, G, (const PkA*)G.pk, (const RlcScalar*)d_r, rbits, G.p_buckets, G.p_W, G.p_jac)));
  LAUNCH((k_to_affine_batch<PkA>), blocks_for((G.nl + TO_AFFINE_BATCH - 1) / TO_AFFINE_BATCH), TPB, G.nl, (const PkJ*)G.p_jac, G.p_aff);
  LAUNCH((k_leaf_gather<PkA, SigA>), blocks_for(G.nl), TPB, G.nl, (const GLeaf*)G.leaves, (const PkA*)G.p_aff, (const SigA*)G.hq, G.hl, G.lpre);
  // the tree over Miller groups of six leaves; its root is checked against S
  const size_t ng = (G.nl + M6_GROUP - 1) / M6_GROUP;
  P.n = G.nl;
  P.ng = ng;
  P.lv = make_levels(ng);
  P.use_rlc = true;
  P.use_msm = true;  // rootS() = the total S
  P.rbits = rbits;
  P.d_pk = G.p_aff;
  P.d_sig = G.s_aff;
  P.d_h = G.hl;
  P.d_status = G.lpre;
  P.d_root = d_root;
  P.d_msm_root = d_S;
  CKR((set_probe_smem<PkA, SigA>(ctx)));
  CK(cudaEventRecord(ctx->ev_fork, ctx->stream));
  // T = ML(-g, S) on the aux stream, beside the Miller stage
  CK(cudaStreamWaitEvent(ctx->aux, ctx->ev_fork, 0));
  ARENA_OK();
  k_probe_fill_nodes<PkA, SigA><<<1, TPB, 0, ctx->aux>>>((size_t)1, (const uint32_t*)nullptr, (const SigJ*)d_S, P.x_pk, P.x_h, P.x_pre);
  CKR(check_launch(ctx, "k_probe_fill_nodes"));
  CKR((probe_miller<PkA, SigA>(ctx, P, ctx->aux, 1, P.x_args, P.x_lines)));
  CK(cudaEventRecord(ctx->ev_aux, ctx->aux));
  P.root_T_ready = true;
  // the leaves are weighted already: the stock prep with rbits = 0
  CKR((miller_stage<PkA, SigA>(ctx, P, G.nl, G.p_aff, G.hl, G.lpre, P.d_F, [&](cudaStream_t s, size_t cn, size_t base, M6Arg* args) {
    k_m6_prep<PkA, SigA><<<blocks_for(cn), TPB, 0, s>>>(cn, base, (const PkA*)G.p_aff, (const SigA*)G.hl, (const uint8_t*)G.lpre, (const Digest*)nullptr,
                                                        0, args);
  })));
  CK(cudaStreamWaitEvent(ctx->stream, ctx->ev_aux, 0));
  stage_mark(ctx, BLSGPU_STAGE_REDUCE);
  CKR(reduce_levels(ctx, P.lv, 0, P.d_F, (SigJ*)nullptr));
  bool ok = false;
  CKR((pipeline_check<PkA, SigA>(ctx, P, &ok)));
  if (!ok) {
    // S_l per leaf (the same kernels over the signatures), summed per Miller group and up the tree
    CKR((leaf_sums<SigA>(ctx, G, (const SigA*)G.sig, (const RlcScalar*)d_r, rbits, G.s_buckets, G.s_W, G.s_jac)));
    LAUNCH((k_group_sum<SigJ>), blocks_for(ng), TPB, G.nl, (const SigJ*)G.s_jac, ng, P.d_S);
    CKR(reduce_levels(ctx, P.lv, 0, (Fp12*)nullptr, P.d_S));
    LAUNCH((k_to_affine_batch<SigA>), blocks_for((G.nl + TO_AFFINE_BATCH - 1) / TO_AFFINE_BATCH), TPB, G.nl, (const SigJ*)G.s_jac, G.s_aff);
    std::vector<uint32_t> bad;
    CKR((descend_tree<PkA, SigA>(ctx, P, bad, [](const std::vector<uint32_t>&) { return (int)BLSGPU_OK; })));
    // the leaves of the failing groups: e(P_l, H_l) e(-g, S_l) == 1 ?
    std::vector<uint32_t> cand;
    for (uint32_t g : bad)
      for (int m = 0; m < M6_GROUP; m++)
        if ((size_t)g * M6_GROUP + m < G.nl) cand.push_back(g * M6_GROUP + m);
    std::vector<uint8_t> res(cand.size());
    CKR(probe_rounds(
        ctx, P, cand, nullptr,
        [&](size_t cnt) -> int {
          LAUNCH((k_probe_fill_leaves<PkA, SigA>), blocks_for(cnt), TPB, cnt, (const uint32_t*)P.d_idx, (const PkA*)G.p_aff, (const SigA*)G.hl,
                 (const SigA*)G.s_aff, (const uint8_t*)G.lpre, P.x_pk, P.x_h, P.x_pre);
          return BLSGPU_OK;
        },
        [&](size_t lo, size_t cnt) -> int {
          CK(cudaMemcpyAsync(res.data() + lo, P.d_ok, cnt, cudaMemcpyDeviceToHost, ctx->stream));
          return BLSGPU_OK;
        }));
    // every item of a failing leaf is decided by its own exact equation e(pk_i, H(m_i)) e(-g, sig_i) == 1
    std::vector<uint32_t> items;
    for (size_t c = 0; c < cand.size(); c++)
      if (!res[c])
        for (uint32_t t = 0; t < leaves[cand[c]].count; t++) items.push_back(order[leaves[cand[c]].first + t]);
    CKR(probe_rounds(
        ctx, P, items, nullptr,
        [&](size_t cnt) -> int {
          LAUNCH((k_probe_fill_grouped<PkA, SigA>), blocks_for(cnt), TPB, cnt, (const uint32_t*)P.d_idx, (const PkA*)G.pk, (const uint32_t*)G.midx,
                 (const SigA*)G.hq, (const SigA*)G.sig, (const uint8_t*)G.status, P.x_pk, P.x_h, P.x_pre);
          return BLSGPU_OK;
        },
        [&](size_t, size_t cnt) -> int {
          LAUNCH(k_mark_invalid, blocks_for(cnt), TPB, cnt, (const uint32_t*)P.d_idx, (const uint8_t*)P.d_ok, G.status);
          return BLSGPU_OK;
        }));
  }
  stage_mark(ctx, BLSGPU_STAGE_COUNT);
  CK(cudaMemcpyAsync(status_out, G.status, n, cudaMemcpyDeviceToHost, ctx->stream));
  CK(cudaStreamSynchronize(ctx->stream));
  stage_collect(ctx);
  return BLSGPU_OK;
}

// blsgpu_verify_batch_grouped and its keyed form: the argument checks, then the grouped pipeline, or for MessageAugmentation
// blsgpu_verify_batch's pipeline on per-item messages
int verify_grouped_common(blsgpu_ctx* ctx, const char* what, int impl_id, int scheme, int format, size_t n, Keys keys, const uint8_t* sigs,
                          const uint32_t* msg_idx, size_t q, const uint8_t* msgs, const uint64_t* msg_off, uint8_t* status_out) {
  if (!args_ok(impl_id, scheme, format) || (n && (!sigs || !msg_idx || !status_out))) return arg_error(ctx, what, "bad arguments");
  if (n == 0) return BLSGPU_OK;
  if (n > MEMBERS_CAP) return arg_error(ctx, what, "at most 2^32 - 16 items per call");
  CKR(check_keys(ctx, what, impl_id, keys, 0, n));
  CKR(check_records(ctx, what, "msgs", msgs, "msg_off", msg_off, q));
  for (size_t i = 0; i < n; i++)
    if (msg_idx[i] >= q) return arg_error(ctx, what, "msg_idx[" + std::to_string(i) + "] is not below q");
  CKR(set_device(ctx));
  if (scheme == 1) {
    // MessageAugmentation hashes pk || msg: no two items share a hash.  Per-item messages through blsgpu_verify_batch's pipeline.
    std::vector<uint64_t> off(n + 1, 0);
    for (size_t i = 0; i < n; i++) off[i + 1] = off[i] + (msg_off[msg_idx[i] + 1] - msg_off[msg_idx[i]]);
    std::vector<uint8_t> data(std::max<uint64_t>(off[n], 1));
    for (size_t i = 0; i < n; i++)
      if (off[i + 1] > off[i]) memcpy(data.data() + off[i], msgs + msg_off[msg_idx[i]], (size_t)(off[i + 1] - off[i]));
    DstParam dst;
    make_dst(dst, impl_id, scheme, false);
    return with_impl(impl_id, [&](auto I) { return verify_host_one<I>(ctx, 1, dst, format, n, keys, sigs, data.data(), off.data(), status_out); });
  }
  return with_impl(impl_id, [&](auto I) { return verify_grouped_impl<I>(ctx, scheme, format, n, keys, sigs, msg_idx, q, msgs, msg_off, status_out); });
}

// n compressed keys -> a key set of this context: decoded and subgroup-checked once into a device allocation of its own
template <class PkA>
int keyset_create_impl(blsgpu_ctx* ctx, int impl_id, int format, size_t n, const uint8_t* pks, uint8_t* status_out, uint64_t* keyset_out) {
  static std::atomic<uint64_t> next_id{1};
  KeySet s;
  s.impl_id = impl_id;
  s.n = n;
  uint8_t* d_bytes = nullptr;
  const int r = [&]() -> int {
    CK(cudaMalloc(&s.pts, std::max<size_t>(n, 1) * sizeof(PkA)));
    CK(cudaMalloc(&s.st, std::max<size_t>(n, 1)));
    if (n) {
      CK(cudaMalloc(&d_bytes, n * PtInfo<PkA>::LEN));
      CK(cudaMemcpyAsync(d_bytes, pks, n * PtInfo<PkA>::LEN, cudaMemcpyHostToDevice, ctx->stream));
      CKR((decode_points<PkA>(ctx, n, (const uint8_t*)d_bytes, format, (PkA*)s.pts, s.st)));
      if (status_out) CK(cudaMemcpyAsync(status_out, s.st, n, cudaMemcpyDeviceToHost, ctx->stream));
    }
    CK(cudaStreamSynchronize(ctx->stream));
    return BLSGPU_OK;
  }();
  cudaFree(d_bytes);
  if (r != BLSGPU_OK) {  // no set is created
    cudaFree(s.pts);
    cudaFree(s.st);
    (void)cudaGetLastError();
    return r;
  }
  const uint64_t id = next_id.fetch_add(1);
  ctx->keysets[id] = s;
  *keyset_out = id;
  return BLSGPU_OK;
}

// The dense ranks of a secure view after some of its keys change, equal to those a fresh ensure_secure_view gives over the
// final encodings.  h: the old ranks of the n keys, over `ranks` distinct encodings.  Key idx[j] (j < k; at or above n for
// an appended key) takes encoding enc[j] (L bytes), which k_rank_search placed at pos[j] = 2 * lb + eq among the old ranks.
// Two kept keys are equal iff their old ranks are; a new key equals the keys of old rank lb when eq is set, and otherwise
// lies between old ranks lb - 1 and lb; new keys are ordered among themselves by memcmp.  An old rank that neither a kept
// key nor an equal new key holds disappears.  out: the n1 new ranks; returns the new count of distinct encodings.
// O(n + ranks) integer work, and a sort of the k new keys.
size_t merge_ranks(const std::vector<uint32_t>& h, size_t ranks, size_t n1, size_t k, const uint32_t* idx, const uint8_t* enc,
                   const uint64_t* pos, size_t L, std::vector<uint32_t>& out) {
  const size_t n = h.size();
  std::vector<uint8_t> kept(n, 1), alive(ranks, 0);
  for (size_t j = 0; j < k; j++)
    if (idx[j] < n) kept[idx[j]] = 0;
  for (size_t i = 0; i < n; i++)
    if (kept[i]) alive[h[i]] = 1;
  std::vector<uint32_t> ord(k);
  for (size_t j = 0; j < k; j++) ord[j] = (uint32_t)j;
  // by lb, then by bytes: the new keys equal to rank lb come after those below it
  std::sort(ord.begin(), ord.end(), [&](uint32_t a, uint32_t b) {
    if (pos[a] >> 1 != pos[b] >> 1) return pos[a] >> 1 < pos[b] >> 1;
    return memcmp(enc + (size_t)a * L, enc + (size_t)b * L, L) < 0;
  });
  std::vector<uint32_t> remap(ranks), fresh(k);
  size_t c = 0, p = 0;
  for (size_t r = 0; r <= ranks; r++) {
    const uint8_t* last = nullptr;  // the previous new encoding below old rank r
    for (; p < k && pos[ord[p]] >> 1 == r && !(pos[ord[p]] & 1); p++) {
      const uint8_t* e = enc + (size_t)ord[p] * L;
      if (!last || memcmp(last, e, L) != 0) c++;
      fresh[ord[p]] = (uint32_t)(c - 1);
      last = e;
    }
    if (r == ranks) break;
    bool held = alive[r];
    for (; p < k && pos[ord[p]] >> 1 == r; p++) {  // equal to old rank r
      fresh[ord[p]] = (uint32_t)c;
      held = true;
    }
    if (held) remap[r] = (uint32_t)c++;
  }
  out.resize(n1);
  for (size_t i = 0; i < n; i++)
    if (kept[i]) out[i] = remap[h[i]];
  for (size_t j = 0; j < k; j++) out[idx[j]] = fresh[j];
  return c;
}

// k keys of set s change (blsgpu_keyset_update: key_idx are distinct indices below n) or are appended (append: key_idx =
// n .. n + k - 1).  The keys are decoded into arena scratch, and for every live secure view encoded in its format and placed
// among its ranks by a binary search; the new ranks are merged on the host (merge_ranks).  Only then is the set written: an
// append first allocates every array at the size n + k and copies the old contents device to device, then the points,
// statuses and encodings are scattered to key_idx and the ranks uploaded.  The old arrays of an append are freed last.
template <class PkA>
int keyset_change_impl(blsgpu_ctx* ctx, KeySet& s, int format, size_t k, const uint32_t* key_idx, const uint8_t* pks, uint8_t* status_out,
                       bool append) {
  constexpr int L = PtInfo<PkA>::LEN;
  const size_t n = s.n, n1 = append ? n + k : n;
  bool live[2];
  for (int f = 0; f < 2; f++) live[f] = s.view[f].enc != nullptr;
  uint8_t *d_bytes, *d_st;
  uint32_t* d_idx;
  PkA* d_pts;
  uint8_t* d_enc[2] = {nullptr, nullptr};
  uint64_t* d_pos[2] = {nullptr, nullptr};
  uint32_t* d_rep[2] = {nullptr, nullptr};
  CKR(arena_takes(ctx, [&](auto& a) {
    d_bytes = take_up<uint8_t>(a, k * L);
    d_idx = take_up<uint32_t>(a, k);
    d_pts = a.template take<PkA>(k);
    d_st = a.template take<uint8_t>(k);
    for (int f = 0; f < 2; f++) {
      if (!live[f]) continue;
      d_enc[f] = a.template take<uint8_t>(k * L);
      d_pos[f] = a.template take<uint64_t>(k);
      d_rep[f] = a.template take<uint32_t>(std::max<size_t>(s.view[f].ranks, 1));
    }
  }));
  CKR(upload(ctx, d_bytes, pks, k * L));
  CKR(upload(ctx, d_idx, key_idx, k));
  CKR((decode_points<PkA>(ctx, k, (const uint8_t*)d_bytes, format, d_pts, d_st)));
  if (status_out) CK(cudaMemcpyAsync(status_out, d_st, k, cudaMemcpyDeviceToHost, ctx->stream));
  std::vector<uint8_t> enc[2];
  std::vector<uint64_t> pos[2];
  for (int f = 0; f < 2; f++) {
    if (!live[f]) continue;
    const SecureView& v = s.view[f];
    LAUNCH((k_encode<PkA>), blocks_for(k), TPB, k, (const PkA*)d_pts, f, d_enc[f]);
    if (n) LAUNCH(k_rank_reps, blocks_for(n), TPB, n, (const uint32_t*)v.rank, d_rep[f]);
    LAUNCH((k_rank_search<L>), blocks_for(k), TPB, k, (const uint8_t*)d_enc[f], (const uint8_t*)v.enc, (const uint32_t*)d_rep[f], v.ranks, d_pos[f]);
    enc[f].resize(k * L);
    pos[f].resize(k);
    CK(cudaMemcpyAsync(enc[f].data(), d_enc[f], k * L, cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaMemcpyAsync(pos[f].data(), d_pos[f], k * 8, cudaMemcpyDeviceToHost, ctx->stream));
  }
  CK(cudaStreamSynchronize(ctx->stream));
  std::vector<uint32_t> rank[2];
  size_t ranks[2] = {0, 0};
  for (int f = 0; f < 2; f++)
    if (live[f]) ranks[f] = merge_ranks(s.view[f].host_rank, s.view[f].ranks, n1, k, key_idx, enc[f].data(), pos[f].data(), L, rank[f]);

  KeySet g;  // the device arrays written: the set's own, or for an append the grown ones
  if (!append) {
    g.pts = s.pts;
    g.st = s.st;
    for (int f = 0; f < 2; f++) {
      g.view[f].enc = s.view[f].enc;
      g.view[f].rank = s.view[f].rank;
    }
  }
  const int r = [&]() -> int {
    if (append) {
      CK(cudaMalloc(&g.pts, n1 * sizeof(PkA)));
      CK(cudaMalloc(&g.st, n1));
      for (int f = 0; f < 2; f++) {
        if (!live[f]) continue;
        CK(cudaMalloc(&g.view[f].enc, n1 * L));
        CK(cudaMalloc(&g.view[f].rank, n1 * 4));
      }
      if (n) {
        CK(cudaMemcpyAsync(g.pts, s.pts, n * sizeof(PkA), cudaMemcpyDeviceToDevice, ctx->stream));
        CK(cudaMemcpyAsync(g.st, s.st, n, cudaMemcpyDeviceToDevice, ctx->stream));
        for (int f = 0; f < 2; f++)
          if (live[f]) CK(cudaMemcpyAsync(g.view[f].enc, s.view[f].enc, n * L, cudaMemcpyDeviceToDevice, ctx->stream));
      }
    }
    LAUNCH((k_scatter_keys<PkA>), blocks_for(k), TPB, k, (const uint32_t*)d_idx, (const PkA*)d_pts, (const uint8_t*)d_st, (PkA*)g.pts, g.st);
    for (int f = 0; f < 2; f++) {
      if (!live[f]) continue;
      LAUNCH((k_scatter_enc<L>), blocks_for(k), TPB, k, (const uint32_t*)d_idx, (const uint8_t*)d_enc[f], g.view[f].enc);
      CK(cudaMemcpyAsync(g.view[f].rank, rank[f].data(), n1 * 4, cudaMemcpyHostToDevice, ctx->stream));
    }
    CK(cudaStreamSynchronize(ctx->stream));
    return BLSGPU_OK;
  }();
  if (r != BLSGPU_OK) {
    if (append) {  // the set keeps its old arrays
      free_keyset(g);
      (void)cudaGetLastError();
    }
    return r;
  }
  if (append) {
    free_keyset(s);
    s.pts = g.pts;
    s.st = g.st;
    s.n = n1;
  }
  for (int f = 0; f < 2; f++) {
    if (!live[f]) continue;
    s.view[f].enc = g.view[f].enc;
    s.view[f].rank = g.view[f].rank;
    s.view[f].host_rank = std::move(rank[f]);
    s.view[f].ranks = ranks[f];
  }
  return BLSGPU_OK;
}

// the k target keys of an update: each below the set's size, none named twice
int check_update_keys(blsgpu_ctx* ctx, const char* what, KeySet* set, size_t k, const uint32_t* key_idx) {
  Keys keys(set, key_idx);
  CKR(check_keys(ctx, what, set->impl_id, keys, 0, k));
  std::vector<std::pair<uint32_t, uint32_t>> o(k);  // (key, position)
  for (size_t i = 0; i < k; i++) o[i] = {key_idx[i], (uint32_t)i};
  std::sort(o.begin(), o.end());
  for (size_t i = 1; i < k; i++)
    if (o[i].first == o[i - 1].first)
      return arg_error(ctx, what, "key_idx[" + std::to_string(o[i - 1].second) + "] and key_idx[" + std::to_string(o[i].second) +
                                      "] both name key " + std::to_string(o[i].first));
  return BLSGPU_OK;
}
}  // namespace

int blsgpu_verify_batch_grouped(blsgpu_ctx* ctx, int impl_id, int scheme, int format, size_t n, const uint8_t* pks, const uint8_t* sigs,
                                const uint32_t* msg_idx, size_t q, const uint8_t* msgs, const uint64_t* msg_off, uint8_t* status_out) {
  NVTX_RANGE("blsgpu_verify_batch_grouped");
  if (!ctx) return BLSGPU_E_ARG;
  return verify_grouped_common(ctx, __func__, impl_id, scheme, format, n, pks, sigs, msg_idx, q, msgs, msg_off, status_out);
}

// ---- key sets -----------------------------------------------------------------------------------------------------------
int blsgpu_keyset_create(blsgpu_ctx* ctx, int impl_id, int format, size_t n, const uint8_t* pks, uint8_t* status_out, uint64_t* keyset_out) {
  NVTX_RANGE("blsgpu_keyset_create");
  if (!ctx) return BLSGPU_E_ARG;
  if ((impl_id != 1 && impl_id != 2) || (format != 0 && format != 1) || !keyset_out) return arg_error(ctx, __func__, "bad arguments");
  CKR(check_buffer(ctx, __func__, "pks", pks, n));
  if (n > MEMBERS_CAP) return arg_error(ctx, __func__, "at most 2^32 - 16 keys per set");
  CKR(set_device(ctx));
  CKR(ensure_arena(ctx, 0));  // takes nothing from the arena: ends a pending slice like any other call
  return with_impl(impl_id, [&](auto I) { return keyset_create_impl<typename ImplT<I>::PkAff>(ctx, impl_id, format, n, pks, status_out, keyset_out); });
}

int blsgpu_keyset_destroy(blsgpu_ctx* ctx, uint64_t keyset) {
  NVTX_RANGE("blsgpu_keyset_destroy");
  if (!ctx) return BLSGPU_E_ARG;
  KeySet* s = nullptr;
  CKR(find_keyset(ctx, __func__, keyset, s));
  ctx->pending.reset();
  CKR(set_device(ctx));
  const cudaError_t e = free_keyset(*s);
  ctx->keysets.erase(keyset);
  CK(e);
  return BLSGPU_OK;
}

int blsgpu_keyset_update(blsgpu_ctx* ctx, uint64_t keyset, int format, size_t k, const uint32_t* key_idx, const uint8_t* pks,
                         uint8_t* status_out) {
  NVTX_RANGE("blsgpu_keyset_update");
  if (!ctx) return BLSGPU_E_ARG;
  KeySet* set = nullptr;
  CKR(find_keyset(ctx, __func__, keyset, set));
  if (format != 0 && format != 1) return arg_error(ctx, __func__, "bad arguments");
  CKR(check_buffer(ctx, __func__, "pks", pks, k));
  CKR(check_update_keys(ctx, __func__, set, k, key_idx));
  if (k == 0) return BLSGPU_OK;
  CKR(set_device(ctx));
  return with_impl(set->impl_id, [&](auto I) {
    return keyset_change_impl<typename ImplT<I>::PkAff>(ctx, *set, format, k, key_idx, pks, status_out, false);
  });
}

int blsgpu_keyset_append(blsgpu_ctx* ctx, uint64_t keyset, int format, size_t k, const uint8_t* pks, uint8_t* status_out) {
  NVTX_RANGE("blsgpu_keyset_append");
  if (!ctx) return BLSGPU_E_ARG;
  KeySet* set = nullptr;
  CKR(find_keyset(ctx, __func__, keyset, set));
  if (format != 0 && format != 1) return arg_error(ctx, __func__, "bad arguments");
  CKR(check_buffer(ctx, __func__, "pks", pks, k));
  if (k > MEMBERS_CAP - set->n) return arg_error(ctx, __func__, "at most 2^32 - 16 keys per set");
  if (k == 0) return BLSGPU_OK;
  std::vector<uint32_t> idx(k);
  for (size_t i = 0; i < k; i++) idx[i] = (uint32_t)(set->n + i);
  CKR(set_device(ctx));
  return with_impl(set->impl_id, [&](auto I) {
    return keyset_change_impl<typename ImplT<I>::PkAff>(ctx, *set, format, k, idx.data(), pks, status_out, true);
  });
}

int blsgpu_verify_batch_keyed(blsgpu_ctx* ctx, uint64_t keyset, int scheme, int format, size_t n, const uint32_t* key_idx, const uint8_t* sigs,
                              const uint8_t* msgs, const uint64_t* msg_off, uint8_t* status_out) {
  NVTX_RANGE("blsgpu_verify_batch_keyed");
  if (!ctx) return BLSGPU_E_ARG;
  KeySet* set = nullptr;
  CKR(find_keyset(ctx, __func__, keyset, set));
  return verify_batch_common(ctx, __func__, set->impl_id, scheme, format, n, Keys(set, key_idx), sigs, msgs, msg_off, status_out);
}

int blsgpu_verify_batch_grouped_keyed(blsgpu_ctx* ctx, uint64_t keyset, int scheme, int format, size_t n, const uint32_t* key_idx, const uint8_t* sigs,
                                      const uint32_t* msg_idx, size_t q, const uint8_t* msgs, const uint64_t* msg_off, uint8_t* status_out) {
  NVTX_RANGE("blsgpu_verify_batch_grouped_keyed");
  if (!ctx) return BLSGPU_E_ARG;
  KeySet* set = nullptr;
  CKR(find_keyset(ctx, __func__, keyset, set));
  return verify_grouped_common(ctx, __func__, set->impl_id, scheme, format, n, Keys(set, key_idx), sigs, msg_idx, q, msgs, msg_off, status_out);
}

// ---------------------------------------------------------------------------------------------------------------------
template <class A>
static int sum_points_impl(blsgpu_ctx* ctx, int format, size_t n, const uint8_t* points, uint8_t* out, uint8_t* status_out,
                           int64_t* bad_index_out) {
  typedef typename PtInfo<A>::Jac J;
  const size_t L = PtInfo<A>::LEN;
  std::vector<Level> lv = make_levels(std::max<size_t>(n, 1));
  uint8_t *d_in, *d_st, *d_out;
  A *d_pts, *d_res;
  J* d_tree;
  CKR(arena_takes(ctx, [&](auto& a) {
    d_in = take_up<uint8_t>(a, n * L);
    d_pts = a.template take<A>(std::max<size_t>(n, 1));
    d_st = a.template take<uint8_t>(std::max<size_t>(n, 1));
    d_tree = a.template take<J>(levels_total(lv) + 1);
    d_res = a.template take<A>(1);
    d_out = a.template take<uint8_t>(L);
  }));
  CKR(upload(ctx, d_in, points, n * L));
  *bad_index_out = -1;
  std::vector<uint8_t> st(n);
  if (n) {
    CKR((decode_points<A>(ctx, n, (const uint8_t*)d_in, format, d_pts, d_st)));
    CK(cudaMemcpyAsync(st.data(), d_st, n, cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    for (size_t i = 0; i < n; i++)
      if (st[i] != BLSGPU_ST_OK) {
        *status_out = st[i];
        *bad_index_out = (int64_t)i;
        return BLSGPU_OK;
      }
  }
  // level 1 from the affine leaves, then Jacobian levels
  const size_t n1 = n ? (n + 15) / 16 : 1;
  LAUNCH((k_reduce_aff<A>), blocks_for(n1), TPB, n, (const A*)d_pts, n1, d_tree);
  const std::vector<Level> lj = make_levels(n1);
  CKR(reduce_levels(ctx, lj, 0, nullptr, d_tree));
  LAUNCH((k_to_affine<A>), 1, 32, (size_t)1, (const J*)(d_tree + lj.back().off), d_res);
  LAUNCH((k_encode<A>), 1, 32, (size_t)1, (const A*)d_res, format, d_out);
  CK(cudaMemcpyAsync(out, d_out, L, cudaMemcpyDeviceToHost, ctx->stream));
  CK(cudaStreamSynchronize(ctx->stream));
  *status_out = BLSGPU_ST_OK;
  return BLSGPU_OK;
}

constexpr size_t SHARD_MIN_POINTS = 65536;  // per device, for the entry points without pairing work

int blsgpu_sum_points(blsgpu_ctx* ctx, int group, int format, size_t n, const uint8_t* points, uint8_t* out, uint8_t* status_out,
                      int64_t* bad_index_out) {
  NVTX_RANGE("blsgpu_sum_points");
  if (!ctx) return BLSGPU_E_ARG;
  int64_t dummy;
  if (!bad_index_out) bad_index_out = &dummy;
  if ((group != 1 && group != 2) || (format != 0 && format != 1) || !out || !status_out || (n && !points)) return arg_error(ctx, __func__, "bad arguments");
  CKR(set_device(ctx));
  auto one = [&](blsgpu_ctx* c, size_t cnt, const uint8_t* pts, uint8_t* o, uint8_t* st, int64_t* bad) {
    return with_group(group, [&](auto G) { return sum_points_impl<typename decltype(G)::type>(c, format, cnt, pts, o, st, bad); });
  };
  const size_t ndev = 1 + ctx->peers.size(), L = group == 1 ? 48 : 96;
  if (ndev == 1 || n < SHARD_MIN_POINTS * ndev) return one(ctx, n, points, out, status_out, bad_index_out);
  // per-device partial sums of contiguous slices (SURVEY 8e, cfg 3), then the sum of the ndev partial results on the first device
  std::vector<uint8_t> part(ndev * L), st(ndev, BLSGPU_ST_OK);
  std::vector<int64_t> bad(ndev, -1);
  CKR(run_on_devices(ctx, [&](blsgpu_ctx* c, size_t d) {
    const size_t lo = n * d / ndev, hi = n * (d + 1) / ndev;
    return one(c, hi - lo, points + lo * L, &part[d * L], &st[d], &bad[d]);
  }));
  for (size_t d = 0; d < ndev; d++)
    if (st[d] != BLSGPU_ST_OK) {  // the first bad element of the whole input is in the first slice that has one
      *status_out = st[d];
      *bad_index_out = (int64_t)(n * d / ndev) + bad[d];
      return BLSGPU_OK;
    }
  return one(ctx, ndev, part.data(), out, status_out, bad_index_out);
}

// ---------------------------------------------------------------------------------------------------------------------
template <class A>
static int hash_batch_impl(blsgpu_ctx* ctx, size_t n, const uint8_t* msgs, const uint64_t* msg_off, const DstParam& dst, uint8_t* out) {
  const size_t L = PtInfo<A>::LEN;
  uint8_t *d_msgs, *d_out;
  uint64_t* d_off;
  A* d_h;
  typename PtInfo<A>::Jac* d_hj;
  CKR(arena_takes(ctx, [&](auto& a) {
    take_records(a, msg_off, n, d_msgs, d_off);
    d_h = a.template take<A>(n);
    d_out = a.template take<uint8_t>(n * L);
    d_hj = take_hash_scratch<A>(a, n);
  }));
  CKR(upload_records(ctx, msgs, msg_off, n, d_msgs, d_off));
  CKR((hash_points<A, G1Aff>(ctx, n, (const uint8_t*)d_msgs, (const uint64_t*)d_off, 0, (const G1Aff*)nullptr, (const uint8_t*)nullptr,
                             dst, d_hj, d_h)));
  LAUNCH((k_encode<A>), blocks_for(n), TPB, n, (const A*)d_h, 1, d_out);
  CK(cudaMemcpyAsync(out, d_out, n * L, cudaMemcpyDeviceToHost, ctx->stream));
  CK(cudaStreamSynchronize(ctx->stream));
  return BLSGPU_OK;
}

int blsgpu_hash_to_curve_batch(blsgpu_ctx* ctx, int group, size_t n, const uint8_t* msgs, const uint64_t* msg_off, const uint8_t* dst,
                               size_t dst_len, uint8_t* out) {
  NVTX_RANGE("blsgpu_hash_to_curve_batch");
  if (!ctx) return BLSGPU_E_ARG;
  if ((group != 1 && group != 2) || !dst || dst_len == 0 || dst_len > 63 || (n && !out))
    return arg_error(ctx, __func__, "bad arguments (dst_len must be 1..63)");
  CKR(check_records(ctx, __func__, "msgs", msgs, "msg_off", msg_off, n));
  if (n == 0) return BLSGPU_OK;
  CKR(set_device(ctx));
  DstParam d;
  memset(d.b, 0, sizeof d.b);
  memcpy(d.b, dst, dst_len);
  d.len = (uint32_t)dst_len;
  return with_group(group, [&](auto G) { return hash_batch_impl<typename decltype(G)::type>(ctx, n, msgs, msg_off, d, out); });
}

template <class A>
static int recode_impl(blsgpu_ctx* ctx, int fin, int fout, size_t n, const uint8_t* in, uint8_t* out, uint8_t* status_out) {
  const size_t L = PtInfo<A>::LEN;
  uint8_t *d_in, *d_st, *d_out;
  A* d_pts;
  CKR(arena_takes(ctx, [&](auto& a) {
    d_in = take_up<uint8_t>(a, n * L);
    d_pts = a.template take<A>(n);
    d_st = a.template take<uint8_t>(n);
    d_out = a.template take<uint8_t>(n * L);
  }));
  CKR(upload(ctx, d_in, in, n * L));
  CKR((decode_points<A>(ctx, n, (const uint8_t*)d_in, fin, d_pts, d_st)));
  LAUNCH((k_encode<A>), blocks_for(n), TPB, n, (const A*)d_pts, fout, d_out);
  CK(cudaMemcpyAsync(out, d_out, n * L, cudaMemcpyDeviceToHost, ctx->stream));
  CK(cudaMemcpyAsync(status_out, d_st, n, cudaMemcpyDeviceToHost, ctx->stream));
  CK(cudaStreamSynchronize(ctx->stream));
  return BLSGPU_OK;
}

int blsgpu_recode_points(blsgpu_ctx* ctx, int group, int format_in, int format_out, size_t n, const uint8_t* in, uint8_t* out,
                         uint8_t* status_out) {
  NVTX_RANGE("blsgpu_recode_points");
  if (!ctx) return BLSGPU_E_ARG;
  if ((group != 1 && group != 2) || (format_in | format_out) & ~1 || (n && (!in || !out || !status_out))) return arg_error(ctx, __func__, "bad arguments");
  if (n == 0) return BLSGPU_OK;
  CKR(set_device(ctx));
  return with_group(group, [&](auto G) { return recode_impl<typename decltype(G)::type>(ctx, format_in, format_out, n, in, out, status_out); });
}

int blsgpu_fp_mul_batch(blsgpu_ctx* ctx, int variant, size_t n, const uint8_t* a, const uint8_t* b, uint8_t* out) {
  NVTX_RANGE("blsgpu_fp_mul_batch");
  if (!ctx) return BLSGPU_E_ARG;
  if ((variant != 0 && variant != 1) || (n && (!a || !b || !out))) return arg_error(ctx, __func__, "bad arguments");
  if (n == 0) return BLSGPU_OK;
  CKR(set_device(ctx));
  uint8_t *d_a, *d_b, *d_o;
  CKR(arena_takes(ctx, [&](auto& ar) {
    d_a = take_up<uint8_t>(ar, n * 48);
    d_b = take_up<uint8_t>(ar, n * 48);
    d_o = ar.template take<uint8_t>(n * 48);
  }));
  CKR(upload(ctx, d_a, a, n * 48));
  CKR(upload(ctx, d_b, b, n * 48));
  LAUNCH(k_fp_mul, blocks_for(n), TPB, n, variant, (const uint8_t*)d_a, (const uint8_t*)d_b, d_o);
  CK(cudaMemcpyAsync(out, d_o, n * 48, cudaMemcpyDeviceToHost, ctx->stream));
  CK(cudaStreamSynchronize(ctx->stream));
  return BLSGPU_OK;
}

int blsgpu_pairing_product_is_one(blsgpu_ctx* ctx, size_t n, const uint8_t* g1_points, const uint8_t* g2_points, int* is_one_out) {
  NVTX_RANGE("blsgpu_pairing_product_is_one");
  if (!ctx) return BLSGPU_E_ARG;
  if (!is_one_out || (n && (!g1_points || !g2_points))) return arg_error(ctx, __func__, "bad arguments");
  if (n == 0) {
    *is_one_out = 1;
    return BLSGPU_OK;
  }
  CKR(set_device(ctx));
  std::vector<Level> lv = make_levels(n);
  uint8_t *d_a, *d_b, *d_st, *d_ok;
  G1Aff* d_p;
  G2Aff* d_q;
  Fp12* d_F;
  CKR(arena_takes(ctx, [&](auto& a) {
    d_a = take_up<uint8_t>(a, n * 48);
    d_b = take_up<uint8_t>(a, n * 96);
    d_p = a.template take<G1Aff>(n);
    d_q = a.template take<G2Aff>(n);
    d_st = a.template take<uint8_t>(2 * n);
    d_F = a.template take<Fp12>(levels_total(lv));
    d_ok = a.template take<uint8_t>(1);
  }));
  CKR(upload(ctx, d_a, g1_points, n * 48));
  CKR(upload(ctx, d_b, g2_points, n * 96));
  CKR((decode_points<G1Aff>(ctx, n, (const uint8_t*)d_a, 1, d_p, d_st)));
  CKR((decode_points<G2Aff>(ctx, n, (const uint8_t*)d_b, 1, d_q, d_st + n)));
  std::vector<uint8_t> st(2 * n);
  CK(cudaMemcpyAsync(st.data(), d_st, 2 * n, cudaMemcpyDeviceToHost, ctx->stream));
  CK(cudaStreamSynchronize(ctx->stream));
  for (uint8_t s : st)
    if (s != BLSGPU_ST_OK) return arg_error(ctx, __func__, "undecodable point");
  LAUNCH(k_miller_pairs, blocks_for(n), TPB, n, (const G1Aff*)d_p, (const G2Aff*)d_q, d_F);
  CKR(reduce_levels(ctx, lv, 0, d_F, (PtInfo<G1Aff>::Jac*)nullptr));
  LAUNCH(k_final_is_one, 1, 32, (const Fp12*)(d_F + lv.back().off), d_ok);
  uint8_t ok = 0;
  CK(cudaMemcpyAsync(&ok, d_ok, 1, cudaMemcpyDeviceToHost, ctx->stream));
  CK(cudaStreamSynchronize(ctx->stream));
  *is_one_out = ok;
  return BLSGPU_OK;
}

int blsgpu_testdata_sign(blsgpu_ctx* ctx, int impl_id, int scheme, size_t n, const uint8_t* scalars32, const uint8_t* msgs,
                         const uint64_t* msg_off, uint8_t* out_pks, uint8_t* out_sigs) {
  NVTX_RANGE("blsgpu_testdata_sign");
  if (!ctx) return BLSGPU_E_ARG;
  const bool pop_proof = scheme == 3;  // proof of possession: message = the key's own bytes, BLS_POP_ DST
  if (!args_ok(impl_id, pop_proof ? 2 : scheme, 1) || (n && (!scalars32 || !out_pks || !out_sigs))) return arg_error(ctx, __func__, "bad arguments");
  if (n == 0) return BLSGPU_OK;
  CKR(check_records(ctx, __func__, "msgs", msgs, "msg_off", msg_off, n));
  CKR(set_device(ctx));
  size_t pk_len = impl_id == 2 ? 48 : 96, sig_len = impl_id == 2 ? 96 : 48;
  uint8_t *d_k, *d_m, *d_pk, *d_sig;
  uint64_t* d_off;
  CKR(arena_takes(ctx, [&](auto& a) {
    d_k = take_up<uint8_t>(a, n * 32);
    take_records(a, msg_off, n, d_m, d_off);
    d_pk = a.template take<uint8_t>(n * pk_len);
    d_sig = a.template take<uint8_t>(n * sig_len);
  }));
  CKR(upload(ctx, d_k, scalars32, n * 32));
  CKR(upload_records(ctx, msgs, msg_off, n, d_m, d_off));
  DstParam dst;
  make_dst(dst, impl_id, pop_proof ? 2 : scheme, pop_proof);
  int mode = pop_proof ? 2 : scheme == 1 ? 1 : 0;
  CKR(with_impl(impl_id, [&](auto I) {
    LAUNCH((k_testdata_sign<typename ImplT<I>::PkAff, typename ImplT<I>::SigAff>), blocks_for(n), TPB, n, (const uint8_t*)d_k, (const uint8_t*)d_m,
           (const uint64_t*)d_off, mode, dst, d_pk, d_sig);
    return BLSGPU_OK;
  }));
  CK(cudaMemcpyAsync(out_pks, d_pk, n * pk_len, cudaMemcpyDeviceToHost, ctx->stream));
  CK(cudaMemcpyAsync(out_sigs, d_sig, n * sig_len, cudaMemcpyDeviceToHost, ctx->stream));
  CK(cudaStreamSynchronize(ctx->stream));
  return BLSGPU_OK;
}

int blsgpu_imad_peak(blsgpu_ctx* ctx, double* mac_per_s_out) {
  NVTX_RANGE("blsgpu_imad_peak");
  if (!ctx || !mac_per_s_out) return BLSGPU_E_ARG;
  CKR(set_device(ctx));
  uint64_t* d_sink;
  CKR(arena_takes(ctx, [&](auto& a) { d_sink = a.template take<uint64_t>(1); }));
  cudaDeviceProp prop;
  CK(cudaGetDeviceProperties(&prop, ctx->devices[0]));
  const int blocks = prop.multiProcessorCount * 8, threads = 256;
  const uint32_t iters = 4096;
  cudaEvent_t a, b;
  CK(cudaEventCreate(&a));
  CK(cudaEventCreate(&b));
  LAUNCH(k_imad_peak, blocks, threads, 256u, 12345u, d_sink);  // warm-up
  float best = 1e30f;
  for (int rep = 0; rep < 3; rep++) {
    CK(cudaEventRecord(a, ctx->stream));
    LAUNCH(k_imad_peak, blocks, threads, iters, 12345u + rep, d_sink);
    CK(cudaEventRecord(b, ctx->stream));
    CK(cudaEventSynchronize(b));
    float ms = 0.f;
    CK(cudaEventElapsedTime(&ms, a, b));
    best = std::min(best, ms);
  }
  cudaEventDestroy(a);
  cudaEventDestroy(b);
  double macs = (double)blocks * threads * (double)iters * 64.0;
  *mac_per_s_out = macs / (best * 1e-3);
  return BLSGPU_OK;
}

// ---------------------------------------------------------------------------------------------------------------------
// Secure aggregation.  Host side: the reference's ordering rules (stable sort of the serialized keys, first-match lookup
// for duplicate keys); device side: SHA-256 coefficient derivation, the t_i * P_i scalar multiplications, segmented sums.
namespace {

struct SecurePlan {
  size_t q = 0, M = 0;
  std::vector<uint32_t> ord, set_of, pos, first;  // per sorted member: original key index, key set, position; first equal key
  std::vector<uint32_t> c_start, c_cnt, s_start, s_cnt;  // level-1 chunks of 16 members, level-2 chunk ranges per key set
};

// sorts every key set by serialized bytes (reference src/secure_aggregation.rs:42,281: sort_by on the byte strings; the
// sort is stable, and a valid compressed encoding is canonical, so the caller's bytes are the reference's sort keys)
// blocks of the key-set multi-scalar multiplication: four warps (= four key sets in flight) per block, a few blocks per SM
size_t secure_msm_blocks(const blsgpu_ctx* ctx, size_t q) { return std::max<size_t>(1, std::min<size_t>((q + 3) / 4, (size_t)ctx->sm_count * 4)); }

SecurePlan make_secure_plan(size_t q, const uint64_t* key_off, const uint8_t* pks, size_t L) {
  SecurePlan pl;
  pl.q = q;
  pl.M = (size_t)key_off[q];
  pl.ord.resize(pl.M);
  pl.set_of.resize(pl.M);
  pl.pos.resize(pl.M);
  pl.first.resize(pl.M);
  for (size_t j = 0; j < q; j++) {
    size_t lo = (size_t)key_off[j], hi = (size_t)key_off[j + 1];
    for (size_t i = lo; i < hi; i++) pl.ord[i] = (uint32_t)i;
    std::stable_sort(pl.ord.begin() + lo, pl.ord.begin() + hi,
                     [&](uint32_t a, uint32_t b) { return memcmp(pks + (size_t)a * L, pks + (size_t)b * L, L) < 0; });
    for (size_t i = lo; i < hi; i++) {
      pl.set_of[i] = (uint32_t)j;
      pl.pos[i] = (uint32_t)(i - lo);
      // equal keys are adjacent after sorting and keep their original order: the run's first element is the first match
      if (i > lo && memcmp(pks + (size_t)pl.ord[i] * L, pks + (size_t)pl.ord[i - 1] * L, L) == 0)
        pl.first[i] = pl.first[i - 1];
      else
        pl.first[i] = pl.ord[i];
    }
    pl.s_start.push_back((uint32_t)pl.c_start.size());
    for (size_t i = lo; i < hi; i += 16) {
      pl.c_start.push_back((uint32_t)i);
      pl.c_cnt.push_back((uint32_t)std::min<size_t>(16, hi - i));
    }
    pl.s_cnt.push_back((uint32_t)pl.c_start.size() - pl.s_start.back());
  }
  return pl;
}

// device part shared by verify and aggregate: out_sum[j] = sum_i t_i * points[src(i)] ; zero_out[m] flags t_m == 0.
// One bucket multi-scalar multiplication per key set: a warp per set, a lane per 8-bit window (kernels.cuh k_secure_msm).
// The plan is on the device: d_ord indexes d_key_bytes, d_src indexes d_points.  Its scratch (take_weighted_sums): the
// per-set digest bases, the members' window digits, the bucket scratch and the window sums.
template <class J>
struct WeightedSums {
  Digest* base = nullptr;
  int8_t* digits = nullptr;
  J *buckets = nullptr, *W = nullptr;
};
template <class J, class A>
void take_weighted_sums(A& a, const blsgpu_ctx* ctx, size_t q, size_t M, WeightedSums<J>& w) {
  w.base = a.template take<Digest>(q);
  w.digits = a.template take<int8_t>(std::max<size_t>(M, 1) * SECURE_WINDOWS);
  w.buckets = a.template take<J>(secure_msm_blocks(ctx, q) * 128 * SECURE_BUCKETS);
  w.W = a.template take<J>(q * SECURE_WINDOWS);
}
template <class A>
int secure_weighted_sums(blsgpu_ctx* ctx, size_t q, size_t M, const uint64_t* d_koff, const uint32_t* d_ord, const uint32_t* d_set,
                         const uint32_t* d_pos, const uint8_t* d_key_bytes, int key_len, const uint32_t* d_src, const A* d_points,
                         const WeightedSums<typename PtInfo<A>::Jac>& w, typename PtInfo<A>::Jac* d_sum, uint8_t* d_zero) {
  typedef typename PtInfo<A>::Jac J;
  Digest* d_base = w.base;
  int8_t* d_digits = w.digits;
  const size_t nblocks = secure_msm_blocks(ctx, q);
  J* d_buckets = w.buckets;
  J* d_W = w.W;
  LAUNCH(k_secure_base, blocks_for(q), TPB, q, d_koff, d_ord, d_key_bytes, key_len, d_base);
  if (M) LAUNCH(k_secure_digits, blocks_for(M), TPB, M, d_set, d_pos, (const Digest*)d_base, d_digits, d_zero);
  LAUNCH((k_secure_msm<A>), (unsigned)nblocks, 128, q, d_koff, d_src, (const int8_t*)d_digits, d_points, d_buckets, d_W);
  LAUNCH((k_secure_combine<J>), blocks_for(q), TPB, q, (const J*)d_W, d_sum);
  return BLSGPU_OK;
}

// Quorums of at most this many members are planned by k_secure_plan_keyed in shared memory (8 bytes per member, so 32 KB:
// within the default limit of dynamic shared memory, 10x Dash's largest quorum of 400); larger ones by make_secure_plan on
// the host, over 4-byte big-endian ranks.
constexpr uint32_t SECURE_PLAN_CAP = 4096;

// A secure call's keys on the device, as the key step (secure_keys) leaves them: the plan (koff, and per sorted member
// ord = the index of its key in key_bytes and pts, set, pos, and first = the member index of the first equal key), the
// keys' encodings in the call's format and their decoded points, and the key statuses: per member (st_per_member) or
// already reduced to each quorum's first bad key.
template <class PkA>
struct SecureKeys {
  const uint64_t* koff = nullptr;
  const uint32_t *ord = nullptr, *set = nullptr, *pos = nullptr, *first = nullptr;
  const uint8_t* key_bytes = nullptr;
  const PkA* pts = nullptr;
  const uint8_t* st = nullptr;
  bool st_per_member = false;
  std::vector<SecurePlan> host_plans;  // host-side plans whose uploads may still be in flight
};

// The key step of a secure call, the one step where keyed and unkeyed calls differ.  Unkeyed: upload the members' key
// bytes, decode them, plan on the host by those bytes (make_secure_plan) and upload the plan.  Keyed: upload key_idx, plan
// on the device by the set's secure view in `format` (k_secure_plan_keyed; make_secure_plan over the ranks for quorums
// above SECURE_PLAN_CAP), and take the keys' encodings and points from the view and the set.  with_first: the plan's
// `first` is needed (aggregate).
// The arena scratch of secure_keys: unkeyed, the key bytes, their points and statuses; keyed, the key indices and the
// quorums' key statuses; both, the key offsets and the plan.
template <class PkA>
struct SecureKeyBufs {
  uint8_t *pkb = nullptr, *st = nullptr;
  PkA* pk = nullptr;
  uint64_t* koff = nullptr;
  uint32_t *kidx = nullptr, *ord = nullptr, *set = nullptr, *pos = nullptr, *first = nullptr;
};
template <class PkA, class A>
void take_secure_keys(A& a, size_t q, size_t M, const Keys& keys, bool with_first, SecureKeyBufs<PkA>& b) {
  if (!keys.set) {
    b.pkb = take_up<uint8_t>(a, M * PtInfo<PkA>::LEN);
    b.pk = a.template take<PkA>(std::max<size_t>(M, 1));
    b.st = a.template take<uint8_t>(std::max<size_t>(M, 1));
  }
  b.koff = take_up<uint64_t>(a, q + 1);
  if (keys.set) b.kidx = take_up<uint32_t>(a, M);
  b.ord = take_up<uint32_t>(a, M);
  b.set = take_up<uint32_t>(a, M);
  b.pos = take_up<uint32_t>(a, M);
  if (with_first || keys.set) b.first = take_up<uint32_t>(a, M);
  if (keys.set) b.st = a.template take<uint8_t>(q);
}
template <class PkA>
int secure_keys(blsgpu_ctx* ctx, int format, size_t q, const uint64_t* key_off, const Keys& keys, bool with_first, const SecureKeyBufs<PkA>& b,
                SecureKeys<PkA>& K) {
  const size_t M = (size_t)key_off[q], Lp = PtInfo<PkA>::LEN;
  uint64_t* d_koff = b.koff;
  if (!keys.set) {
    K.host_plans.push_back(make_secure_plan(q, key_off, keys.bytes, Lp));
    const SecurePlan& pl = K.host_plans.back();
    uint8_t* d_pkb = b.pkb;
    CKR(upload(ctx, d_pkb, keys.bytes, M * Lp));
    PkA* d_pk = b.pk;
    uint8_t* d_stpk = b.st;
    if (M) CKR((decode_points<PkA>(ctx, M, (const uint8_t*)d_pkb, format, d_pk, d_stpk)));
    uint32_t *d_ord = b.ord, *d_set = b.set, *d_pos = b.pos, *d_first = with_first ? b.first : nullptr;
    CKR(upload(ctx, d_koff, key_off, q + 1));
    CKR(upload(ctx, d_ord, pl.ord.data(), M));
    CKR(upload(ctx, d_set, pl.set_of.data(), M));
    CKR(upload(ctx, d_pos, pl.pos.data(), M));
    if (with_first) CKR(upload(ctx, d_first, pl.first.data(), M));
    K.koff = d_koff;
    K.ord = d_ord;
    K.set = d_set;
    K.pos = d_pos;
    K.first = d_first;
    K.key_bytes = d_pkb;
    K.pts = d_pk;
    K.st = d_stpk;
    K.st_per_member = true;
    return BLSGPU_OK;
  }
  const SecureView& v = keys.set->view[format];
  uint32_t* d_kidx = b.kidx;
  CKR(upload(ctx, d_koff, key_off, q + 1));
  CKR(upload(ctx, d_kidx, keys.idx, M));
  uint32_t *d_ord = b.ord, *d_set = b.set, *d_pos = b.pos, *d_first = b.first;
  uint8_t* d_keyst = b.st;
  uint32_t slots = 1;
  for (size_t j = 0; j < q; j++) {
    const uint64_t cnt = key_off[j + 1] - key_off[j];
    while (cnt <= SECURE_PLAN_CAP && slots < cnt) slots <<= 1;
  }
  ARENA_OK();
  k_secure_plan_keyed<<<(unsigned)q, 256, slots * sizeof(unsigned long long), ctx->stream>>>(q, d_koff, d_kidx, v.rank, keys.set->st, slots, d_ord,
                                                                                             d_set, d_pos, d_first, d_keyst);
  CKR(check_launch(ctx, "k_secure_plan_keyed"));
  for (size_t j = 0; j < q; j++) {
    const size_t lo = (size_t)key_off[j], cnt = (size_t)(key_off[j + 1] - lo);
    if (cnt <= SECURE_PLAN_CAP) continue;
    std::vector<uint8_t> be(cnt * 4);
    for (size_t p = 0; p < cnt; p++) {
      const uint32_t r = v.host_rank[keys.idx[lo + p]];
      for (int b = 0; b < 4; b++) be[p * 4 + b] = (uint8_t)(r >> (24 - 8 * b));
    }
    const uint64_t one[2] = {0, cnt};
    K.host_plans.push_back(make_secure_plan(1, one, be.data(), 4));
    SecurePlan& pl = K.host_plans.back();
    for (size_t i = 0; i < cnt; i++) {  // to the call's indices: set indices in ord, member indices in first
      pl.ord[i] = keys.idx[lo + pl.ord[i]];
      pl.set_of[i] = (uint32_t)j;
      pl.first[i] += (uint32_t)lo;
    }
    CK(cudaMemcpyAsync(d_ord + lo, pl.ord.data(), cnt * 4, cudaMemcpyHostToDevice, ctx->stream));
    CK(cudaMemcpyAsync(d_set + lo, pl.set_of.data(), cnt * 4, cudaMemcpyHostToDevice, ctx->stream));
    CK(cudaMemcpyAsync(d_pos + lo, pl.pos.data(), cnt * 4, cudaMemcpyHostToDevice, ctx->stream));
    CK(cudaMemcpyAsync(d_first + lo, pl.first.data(), cnt * 4, cudaMemcpyHostToDevice, ctx->stream));
  }
  K.koff = d_koff;
  K.ord = d_ord;
  K.set = d_set;
  K.pos = d_pos;
  K.first = d_first;
  K.key_bytes = v.enc;
  K.pts = (const PkA*)keys.set->pts;
  K.st = d_keyst;
  K.st_per_member = false;
  return BLSGPU_OK;
}
// quorum j's key status (its first bad key in member order) from the statuses secure_keys left, downloaded to `st`
template <class PkA>
uint8_t secure_key_status(const SecureKeys<PkA>& K, const std::vector<uint8_t>& st, const uint64_t* key_off, size_t j) {
  if (!K.st_per_member) return st[j];
  uint8_t s = BLSGPU_ST_OK;
  for (size_t i = (size_t)key_off[j]; i < (size_t)key_off[j + 1] && s == BLSGPU_ST_OK; i++) s = st[i];
  return s;
}

template <int IMPL>
int verify_secure_impl(blsgpu_ctx* ctx, int scheme, int format, size_t q, const uint64_t* key_off, const Keys& keys, const uint8_t* sigs,
                       const uint8_t* msgs, const uint64_t* msg_off, uint8_t* status_out) {
  typedef typename ImplT<IMPL>::PkAff PkA;
  typedef typename ImplT<IMPL>::SigAff SigA;
  typedef typename ImplT<IMPL>::PkJac PkJ;
  const size_t Lp = PtInfo<PkA>::LEN, Ls = PtInfo<SigA>::LEN;
  const size_t M = (size_t)key_off[q];
  SecureKeyBufs<PkA> kb;
  WeightedSums<PkJ> ws;
  uint8_t *d_sigb, *d_msgs, *d_stsig, *d_zero, *d_setst, *d_status;
  uint64_t* d_moff;
  SigA* d_sig;
  PkJ* d_sum;
  PkA* d_agg;
  auto head = [&](auto& a) {
    take_secure_keys(a, q, M, keys, false, kb);
    d_sigb = take_up<uint8_t>(a, q * Ls);
    take_records(a, msg_off, q, d_msgs, d_moff);
    d_sig = a.template take<SigA>(q);
    d_stsig = a.template take<uint8_t>(q);
    d_zero = a.template take<uint8_t>(std::max<size_t>(M, 1));
    d_sum = a.template take<PkJ>(q);
    d_agg = a.template take<PkA>(q);
    d_setst = a.template take<uint8_t>(q);
    d_status = a.template take<uint8_t>(q);
    take_weighted_sums(a, ctx, q, M, ws);
  };
  CKR(ensure_miller_arena(ctx, q, [&](auto& a, size_t chunk) {
    head(a);
    take_verify_points<IMPL>(a, ctx, q, chunk);
  }));
  head(ctx->arena);
  stage_reset(ctx);
  SecureKeys<PkA> K;
  CKR((secure_keys<PkA>(ctx, format, q, key_off, keys, false, kb, K)));
  CKR(upload(ctx, d_sigb, sigs, q * Ls));
  CKR(upload_records(ctx, msgs, msg_off, q, d_msgs, d_moff));
  CKR((decode_points<SigA>(ctx, q, (const uint8_t*)d_sigb, format, d_sig, d_stsig)));
  CKR((secure_weighted_sums<PkA>(ctx, q, M, K.koff, K.ord, K.set, K.pos, K.key_bytes, (int)Lp, K.ord, K.pts, ws, d_sum, d_zero)));
  LAUNCH((k_to_affine<PkA>), blocks_for(q), TPB, q, (const PkJ*)d_sum, d_agg);
  const size_t nst = K.st_per_member ? M : q;
  std::vector<uint8_t> stpk(nst), stsig(q), zero(M);
  std::vector<uint32_t> siginf(q);
  if (nst) CK(cudaMemcpyAsync(stpk.data(), K.st, nst, cudaMemcpyDeviceToHost, ctx->stream));
  if (M) CK(cudaMemcpyAsync(zero.data(), d_zero, M, cudaMemcpyDeviceToHost, ctx->stream));
  CK(cudaMemcpyAsync(stsig.data(), d_stsig, q, cudaMemcpyDeviceToHost, ctx->stream));
  CK(cudaMemcpy2DAsync(siginf.data(), 4, reinterpret_cast<const uint8_t*>(d_sig) + offsetof(SigA, inf), sizeof(SigA), 4, q,
                       cudaMemcpyDeviceToHost, ctx->stream));
  CK(cudaStreamSynchronize(ctx->stream));
  // set-level status in the reference's order: key decode errors (first bad key), signature decode error, empty key set
  // (secure_aggregation.rs:189-195), zero coefficient (:98-100); everything else is core_verify on the device
  std::vector<uint8_t> pre(q, BLSGPU_ST_OK);
  for (size_t j = 0; j < q; j++) {
    size_t lo = (size_t)key_off[j], hi = (size_t)key_off[j + 1];
    uint8_t s = secure_key_status(K, stpk, key_off, j);
    if (s == BLSGPU_ST_OK) s = stsig[j];
    if (s == BLSGPU_ST_OK && lo == hi) s = siginf[j] ? 0xff : BLSGPU_ST_INVALID_SIGNATURE;  // 0xff: "OK, nothing to check"
    if (s == BLSGPU_ST_OK)
      for (size_t i = lo; i < hi; i++)
        if (zero[i]) s = BLSGPU_ST_INVALID_COEFFICIENT;
    pre[j] = s;
  }
  CK(cudaMemcpyAsync(d_setst, pre.data(), q, cudaMemcpyHostToDevice, ctx->stream));
  CK(cudaMemsetAsync(d_stsig, 0, q, ctx->stream));
  DstParam dst;
  make_dst(dst, IMPL, scheme, false);
  // MessageAugmentation uses its DST but does NOT prepend the aggregated key here (secure_aggregation.rs:236-247)
  CKR((verify_points<IMPL>(ctx, 0, dst, q, d_agg, d_sig, d_setst, d_stsig, d_msgs, d_moff, d_status)));
  CK(cudaMemcpyAsync(status_out, d_status, q, cudaMemcpyDeviceToHost, ctx->stream));
  CK(cudaStreamSynchronize(ctx->stream));
  for (size_t j = 0; j < q; j++)
    if (status_out[j] == 0xff) status_out[j] = BLSGPU_ST_OK;
  stage_collect(ctx);
  return BLSGPU_OK;
}

template <int IMPL>
int aggregate_secure_impl(blsgpu_ctx* ctx, int format, size_t q, const uint64_t* key_off, const Keys& keys, const uint8_t* member_sigs,
                          uint8_t* out_sigs, uint8_t* status_out) {
  typedef typename ImplT<IMPL>::PkAff PkA;
  typedef typename ImplT<IMPL>::SigAff SigA;
  typedef typename ImplT<IMPL>::SigJac SigJ;
  const size_t Lp = PtInfo<PkA>::LEN, Ls = PtInfo<SigA>::LEN;
  const size_t M = (size_t)key_off[q];
  SecureKeyBufs<PkA> kb;
  WeightedSums<SigJ> ws;
  uint8_t *d_sigb, *d_stsig, *d_zero, *d_out;
  SigA *d_sig, *d_agg;
  SigJ* d_sum;
  CKR(arena_takes(ctx, [&](auto& a) {
    take_secure_keys(a, q, M, keys, true, kb);
    d_sigb = take_up<uint8_t>(a, M * Ls);
    d_sig = a.template take<SigA>(std::max<size_t>(M, 1));
    d_stsig = a.template take<uint8_t>(std::max<size_t>(M, 1));
    d_zero = a.template take<uint8_t>(std::max<size_t>(M, 1));
    d_sum = a.template take<SigJ>(q);
    d_agg = a.template take<SigA>(q);
    d_out = a.template take<uint8_t>(q * Ls);
    take_weighted_sums(a, ctx, q, M, ws);
  }));
  SecureKeys<PkA> K;
  CKR((secure_keys<PkA>(ctx, format, q, key_off, keys, true, kb, K)));
  CKR(upload(ctx, d_sigb, member_sigs, M * Ls));
  if (M) CKR((decode_points<SigA>(ctx, M, (const uint8_t*)d_sigb, format, d_sig, d_stsig)));
  // sum_i t_i * sig[first original index whose key bytes equal sorted key i]   (secure_aggregation.rs:138-153)
  CKR((secure_weighted_sums<SigA>(ctx, q, M, K.koff, K.ord, K.set, K.pos, K.key_bytes, (int)Lp, K.first, d_sig, ws, d_sum, d_zero)));
  LAUNCH((k_to_affine<SigA>), blocks_for(q), TPB, q, (const SigJ*)d_sum, d_agg);
  LAUNCH((k_encode<SigA>), blocks_for(q), TPB, q, (const SigA*)d_agg, format, d_out);
  const size_t nst = K.st_per_member ? M : q;
  std::vector<uint8_t> stpk(nst), stsig(M), zero(M);
  if (nst) CK(cudaMemcpyAsync(stpk.data(), K.st, nst, cudaMemcpyDeviceToHost, ctx->stream));
  if (M) {
    CK(cudaMemcpyAsync(stsig.data(), d_stsig, M, cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaMemcpyAsync(zero.data(), d_zero, M, cudaMemcpyDeviceToHost, ctx->stream));
  }
  CK(cudaMemcpyAsync(out_sigs, d_out, q * Ls, cudaMemcpyDeviceToHost, ctx->stream));
  CK(cudaStreamSynchronize(ctx->stream));
  for (size_t j = 0; j < q; j++) {
    size_t lo = (size_t)key_off[j], hi = (size_t)key_off[j + 1];
    uint8_t s = secure_key_status(K, stpk, key_off, j);
    for (size_t i = lo; i < hi && s == BLSGPU_ST_OK; i++) s = stsig[i];
    if (s == BLSGPU_ST_OK)
      for (size_t i = lo; i < hi; i++)
        if (zero[i]) s = BLSGPU_ST_INVALID_COEFFICIENT;
    status_out[j] = s;
    if (s != BLSGPU_ST_OK) memset(out_sigs + j * Ls, 0, Ls);
  }
  return BLSGPU_OK;
}

// The secure view of key set s in `format` (SecureView), built once: k_encode of every key, the encodings downloaded and
// ranked on the host, the ranks uploaded.  Device allocations of its own, like the set; freed with the set.
template <class PkA>
int ensure_secure_view(blsgpu_ctx* ctx, KeySet& s, int format) {
  SecureView& v = s.view[format];
  if (v.enc) return BLSGPU_OK;
  const size_t n = s.n, L = PtInfo<PkA>::LEN;
  SecureView nv;
  nv.host_rank.resize(n);
  const int r = [&]() -> int {
    CK(cudaMalloc(&nv.enc, std::max<size_t>(n, 1) * L));
    CK(cudaMalloc(&nv.rank, std::max<size_t>(n, 1) * 4));
    if (n) {
      std::vector<uint8_t> enc(n * L);
      LAUNCH((k_encode<PkA>), blocks_for(n), TPB, n, (const PkA*)s.pts, format, nv.enc);
      CK(cudaMemcpyAsync(enc.data(), nv.enc, n * L, cudaMemcpyDeviceToHost, ctx->stream));
      CK(cudaStreamSynchronize(ctx->stream));
      // sort by the first 8 bytes, then by all of them: memcmp order
      std::vector<std::pair<uint64_t, uint32_t>> o(n);
      for (size_t i = 0; i < n; i++) {
        uint64_t pre = 0;
        for (int b = 0; b < 8; b++) pre = (pre << 8) | enc[i * L + b];
        o[i] = {pre, (uint32_t)i};
      }
      std::sort(o.begin(), o.end(), [&](const std::pair<uint64_t, uint32_t>& a, const std::pair<uint64_t, uint32_t>& b) {
        if (a.first != b.first) return a.first < b.first;
        return memcmp(&enc[(size_t)a.second * L], &enc[(size_t)b.second * L], L) < 0;
      });
      uint32_t rk = 0;
      for (size_t i = 0; i < n; i++) {
        if (i && (o[i].first != o[i - 1].first || memcmp(&enc[(size_t)o[i].second * L], &enc[(size_t)o[i - 1].second * L], L) != 0)) rk++;
        nv.host_rank[o[i].second] = rk;
      }
      nv.ranks = (size_t)rk + 1;
      CK(cudaMemcpyAsync(nv.rank, nv.host_rank.data(), n * 4, cudaMemcpyHostToDevice, ctx->stream));
      CK(cudaStreamSynchronize(ctx->stream));
    }
    return BLSGPU_OK;
  }();
  if (r != BLSGPU_OK) {  // no view is kept
    cudaFree(nv.enc);
    cudaFree(nv.rank);
    (void)cudaGetLastError();
    return r;
  }
  v = std::move(nv);
  return BLSGPU_OK;
}

// The secure calls and their keyed forms.  A keyed call runs on the first device over the set's secure view in `format`;
// the unkeyed calls cut their quorums over the devices of the context (SURVEY 8e, cfg 5): contiguous runs, balanced by
// member count.  f(device context, quorums, key_off from 0, keys of the first member, quorum offset) runs a set of quorums.
template <int IMPL, class F>
int secure_route(blsgpu_ctx* ctx, int format, size_t q, const std::vector<uint64_t>& ko, const Keys& keys, const F& f) {
  if (keys.set) {
    CKR((ensure_secure_view<typename ImplT<IMPL>::PkAff>(ctx, *keys.set, format)));
    return f(ctx, q, ko.data(), keys, (size_t)0);
  }
  const size_t ndev = 1 + ctx->peers.size();
  if (ndev == 1 || q < 2 * ndev || ko[q] < SHARD_MIN_ITEMS * ndev) return f(ctx, q, ko.data(), keys, (size_t)0);
  return run_cut(ctx, q, ko.data(), [&](blsgpu_ctx* c, size_t lo, size_t hi) {
    const std::vector<uint64_t> run = rebased(ko.data(), lo, hi);
    return f(c, hi - lo, run.data(), Keys(keys.bytes + ko[lo] * PtInfo<typename ImplT<IMPL>::PkAff>::LEN), lo);
  });
}

// the argument rules the secure calls share: Legacy only for Bls12381G2Impl, key_off (at most 2^32 - 16 members), the keys.
// ko: key_off from 0; keys: from the first member on.
int check_secure(blsgpu_ctx* ctx, const char* what, int impl_id, int scheme, int format, size_t q, const uint64_t* key_off, Keys& keys,
                 bool outputs, std::vector<uint64_t>& ko) {
  if (!args_ok(impl_id, scheme, format) || (q && !outputs) || (impl_id == 1 && format == 0))
    return arg_error(ctx, what, "bad arguments (Legacy mode exists only for Bls12381G2Impl)");
  if (q == 0) return BLSGPU_OK;
  CKR(check_sets(ctx, what, "key_off", key_off, q, MEMBERS_CAP, ko));
  return check_keys(ctx, what, impl_id, keys, key_off[0], ko[q]);
}

int verify_secure_common(blsgpu_ctx* ctx, const char* what, int impl_id, int scheme, int format, size_t q, const uint64_t* key_off, Keys keys,
                         const uint8_t* sigs, const uint8_t* msgs, const uint64_t* msg_off, uint8_t* status_out) {
  std::vector<uint64_t> ko;
  CKR(check_secure(ctx, what, impl_id, scheme, format, q, key_off, keys, sigs && status_out, ko));
  if (q == 0) return BLSGPU_OK;
  CKR(check_records(ctx, what, "msgs", msgs, "msg_off", msg_off, q));
  CKR(set_device(ctx));
  const size_t sig_len = impl_id == 2 ? 96 : 48;
  return with_impl(impl_id, [&](auto I) {
    return secure_route<I>(ctx, format, q, ko, keys, [&](blsgpu_ctx* c, size_t cnt, const uint64_t* k, const Keys& ks, size_t lo) {
      return verify_secure_impl<I>(c, scheme, format, cnt, k, ks, sigs + lo * sig_len, msgs, msg_off + lo, status_out + lo);
    });
  });
}

int aggregate_secure_common(blsgpu_ctx* ctx, const char* what, int impl_id, int format, size_t q, const uint64_t* key_off, Keys keys,
                            const uint8_t* member_sigs, uint8_t* out_sigs, uint8_t* status_out) {
  std::vector<uint64_t> ko;
  CKR(check_secure(ctx, what, impl_id, 0, format, q, key_off, keys, out_sigs && status_out, ko));
  if (q == 0) return BLSGPU_OK;
  const size_t sig_len = impl_id == 2 ? 96 : 48;
  if (member_sigs) member_sigs += key_off[0] * sig_len;
  CKR(check_buffer(ctx, what, "member_sigs", member_sigs, ko[q]));
  CKR(set_device(ctx));
  return with_impl(impl_id, [&](auto I) {
    return secure_route<I>(ctx, format, q, ko, keys, [&](blsgpu_ctx* c, size_t cnt, const uint64_t* k, const Keys& ks, size_t lo) {
      return aggregate_secure_impl<I>(c, format, cnt, k, ks, member_sigs + ko[lo] * sig_len, out_sigs + lo * sig_len, status_out + lo);
    });
  });
}

}  // namespace

int blsgpu_verify_secure_batch(blsgpu_ctx* ctx, int impl_id, int scheme, int format, size_t q, const uint64_t* key_off, const uint8_t* pks,
                               const uint8_t* sigs, const uint8_t* msgs, const uint64_t* msg_off, uint8_t* status_out) {
  NVTX_RANGE("blsgpu_verify_secure_batch");
  if (!ctx) return BLSGPU_E_ARG;
  return verify_secure_common(ctx, __func__, impl_id, scheme, format, q, key_off, pks, sigs, msgs, msg_off, status_out);
}

int blsgpu_aggregate_secure_batch(blsgpu_ctx* ctx, int impl_id, int format, size_t q, const uint64_t* key_off, const uint8_t* pks,
                                  const uint8_t* member_sigs, uint8_t* out_sigs, uint8_t* status_out) {
  NVTX_RANGE("blsgpu_aggregate_secure_batch");
  if (!ctx) return BLSGPU_E_ARG;
  return aggregate_secure_common(ctx, __func__, impl_id, format, q, key_off, pks, member_sigs, out_sigs, status_out);
}

int blsgpu_verify_secure_batch_keyed(blsgpu_ctx* ctx, uint64_t keyset, int scheme, int format, size_t q, const uint64_t* key_off,
                                     const uint32_t* key_idx, const uint8_t* sigs, const uint8_t* msgs, const uint64_t* msg_off,
                                     uint8_t* status_out) {
  NVTX_RANGE("blsgpu_verify_secure_batch_keyed");
  if (!ctx) return BLSGPU_E_ARG;
  KeySet* set = nullptr;
  CKR(find_keyset(ctx, __func__, keyset, set));
  return verify_secure_common(ctx, __func__, set->impl_id, scheme, format, q, key_off, Keys(set, key_idx), sigs, msgs, msg_off, status_out);
}

int blsgpu_aggregate_secure_batch_keyed(blsgpu_ctx* ctx, uint64_t keyset, int format, size_t q, const uint64_t* key_off,
                                        const uint32_t* key_idx, const uint8_t* member_sigs, uint8_t* out_sigs, uint8_t* status_out) {
  NVTX_RANGE("blsgpu_aggregate_secure_batch_keyed");
  if (!ctx) return BLSGPU_E_ARG;
  KeySet* set = nullptr;
  CKR(find_keyset(ctx, __func__, keyset, set));
  return aggregate_secure_common(ctx, __func__, set->impl_id, format, q, key_off, Keys(set, key_idx), member_sigs, out_sigs, status_out);
}

// ---------------------------------------------------------------------------------------------------------------------
// Multi-signatures over signer subsets, and point sums of many sets: MultiSignature::verify(MultiPublicKey of set j, msg_j)
// is core_verify against the SUM of set j's keys, so the q key sums are formed on the device (a segmented sum balanced by
// member count) and the q (sum, signature, message) triples go through verify_points like any batch of q signatures.
namespace {

// The segmented sum of q point sets, set j = members off[j] .. off[j+1]-1 (off rebased to 0): chunks of at most 16 members of
// one set for k_seg_sum_gather (an empty set has one chunk without members, so that every set has a node), then the levels of
// seg_levels over each set's chunks.  A set of 2^20 members is 65,536 chunks next to one chunk per set of 3: the threads
// of every launch do about equal work however skewed the set sizes are.
struct SegSumPlan {
  size_t q;
  std::vector<uint32_t> coff, cset;  // chunk c: members coff[c] .. coff[c+1]-1 of set cset[c]
  SegLevels lv;
  SegSumPlan(size_t q_, const uint64_t* off) : q(q_) {
    std::vector<size_t> cnt(q);
    coff.push_back(0);
    for (size_t j = 0; j < q; j++) {
      const uint64_t lo = off[j], hi = off[j + 1];
      cnt[j] = 0;
      for (uint64_t m = lo; m < hi || cnt[j] == 0; m += 16, cnt[j]++) {
        coff.push_back((uint32_t)std::min<uint64_t>(m + 16, hi));
        cset.push_back((uint32_t)j);
      }
    }
    lv = seg_levels(std::move(cnt));
  }
  size_t nchunks() const { return cset.size(); }
};
// the arena scratch of seg_point_sums over a plan: the plan's chunks and level offsets, the levels' nodes, and per set its
// first bad member and its sum
template <class J>
struct SegSums {
  uint32_t *coff = nullptr, *cset = nullptr, *segoff = nullptr;
  J *nodes = nullptr, *sum = nullptr;
  unsigned long long* bad = nullptr;
};
template <class J, class A>
void take_seg_sums(A& a, const SegSumPlan& pl, SegSums<J>& s) {
  s.coff = take_up<uint32_t>(a, pl.coff.size());
  s.cset = take_up<uint32_t>(a, pl.cset.size());
  s.segoff = take_up<uint32_t>(a, pl.lv.off.size());
  s.nodes = a.template take<J>(std::max<size_t>(pl.lv.below_top(), 1));
  s.bad = a.template take<unsigned long long>(pl.q);
  s.sum = a.template take<J>(pl.q);
}

// s.sum[j] = the sum of set j's points (the identity for an empty set), s.bad[j] = (member << 8 | status) of its first
// member that failed to decode or ~0 (kernels.cuh k_seg_sum_gather).  Member m's point is d_pts[d_idx[m]], or d_pts[m] when
// d_idx is null; likewise its status in d_st.
template <class A>
int seg_point_sums(blsgpu_ctx* ctx, const SegSumPlan& pl, const SegSums<typename PtInfo<A>::Jac>& s, const uint32_t* d_idx, const A* d_pts,
                   const uint8_t* d_st) {
  typedef typename PtInfo<A>::Jac J;
  uint32_t *d_coff = s.coff, *d_cset = s.cset, *d_segoff = s.segoff;
  CKR(upload(ctx, d_coff, pl.coff.data(), pl.coff.size()));
  CKR(upload(ctx, d_cset, pl.cset.data(), pl.cset.size()));
  CKR(upload(ctx, d_segoff, pl.lv.off.data(), pl.lv.off.size()));
  J* d_nodes = s.nodes;
  unsigned long long* d_bad = s.bad;
  J* d_sum = s.sum;
  CK(cudaMemsetAsync(d_bad, 0xff, pl.q * sizeof(unsigned long long), ctx->stream));
  const bool levels = pl.lv.n.size() > 1;  // some set has more than one chunk
  LAUNCH((k_seg_sum_gather<A>), blocks_for(pl.nchunks()), TPB, pl.nchunks(), (const uint32_t*)d_coff, (const uint32_t*)d_cset, d_idx, d_pts, d_st,
         levels ? d_nodes : d_sum, d_bad);
  if (levels) CKR(seg_reduce_levels<J>(ctx, pl.lv, d_segoff, d_nodes, d_sum));
  return BLSGPU_OK;
}

// q x MultiSignature::verify: the key step (upload and decode the members' keys, or their indices into a key set), the
// segmented key sums, then verify_points on (sum_j, sig_j, msg_j).  Key offsets start at 0 (the entry points rebase them).
// The per-set status before any pairing work is k_prestatus's over (first bad key of the set, signature decode status,
// signature identity, sum identity): the reference's order for sum_points followed by verify.
template <int IMPL>
int verify_multisig_impl(blsgpu_ctx* ctx, int scheme, int format, size_t q, const uint64_t* key_off, const Keys& keys, const uint8_t* sigs,
                         const uint8_t* msgs, const uint64_t* msg_off, uint8_t* status_out) {
  typedef typename ImplT<IMPL>::PkAff PkA;
  typedef typename ImplT<IMPL>::SigAff SigA;
  typedef typename ImplT<IMPL>::PkJac PkJ;
  const size_t Ls = PtInfo<SigA>::LEN;
  const size_t M = (size_t)key_off[q];
  const SegSumPlan pl(q, key_off);
  Keys d_keys;
  PkA *d_pk = nullptr, *d_agg;
  uint8_t *d_stpk = nullptr, *d_setst, *d_sigb, *d_msgs, *d_stsig, *d_status;
  uint64_t* d_moff;
  SigA* d_sig;
  SegSums<PkJ> ss;
  auto head = [&](auto& a) {
    take_keys<PkA>(a, M, keys, d_keys);
    if (!keys.set) {
      d_pk = a.template take<PkA>(std::max<size_t>(M, 1));
      d_stpk = a.template take<uint8_t>(std::max<size_t>(M, 1));
    }
    take_seg_sums(a, pl, ss);
    d_agg = a.template take<PkA>(q);
    d_setst = a.template take<uint8_t>(q);
    d_sigb = take_up<uint8_t>(a, q * Ls);
    take_records(a, msg_off, q, d_msgs, d_moff);
    d_sig = a.template take<SigA>(q);
    d_stsig = a.template take<uint8_t>(q);
    d_status = a.template take<uint8_t>(q);
  };
  CKR(ensure_miller_arena(ctx, q, [&](auto& a, size_t chunk) {
    head(a);
    take_verify_points<IMPL>(a, ctx, q, chunk);
  }));
  head(ctx->arena);
  stage_reset(ctx);
  stage_mark(ctx, BLSGPU_STAGE_DECODE_PK);  // the key side: decode (unkeyed calls) and the segmented sums
  CKR(upload_keys<PkA>(ctx, M, keys, d_keys));
  const PkA* d_pts = keys.set ? (const PkA*)keys.set->pts : d_pk;
  const uint8_t* d_st = keys.set ? (const uint8_t*)keys.set->st : d_stpk;
  if (!keys.set && M) CKR((decode_points<PkA>(ctx, M, d_keys.bytes, format, d_pk, d_stpk, BLSGPU_KERNEL_DECODE_PK)));
  CKR((seg_point_sums<PkA>(ctx, pl, ss, keys.set ? d_keys.idx : nullptr, d_pts, d_st)));
  LAUNCH((k_to_affine_batch<PkA>), blocks_for((q + TO_AFFINE_BATCH - 1) / TO_AFFINE_BATCH), TPB, q, (const PkJ*)ss.sum, d_agg);
  LAUNCH(k_seg_first_bad_status, blocks_for(q), TPB, q, (const unsigned long long*)ss.bad, d_setst);
  stage_mark(ctx, BLSGPU_STAGE_DECODE_SIG);
  CKR(upload(ctx, d_sigb, sigs, q * Ls));
  CKR(upload_records(ctx, msgs, msg_off, q, d_msgs, d_moff));
  CKR((decode_points<SigA>(ctx, q, (const uint8_t*)d_sigb, format, d_sig, d_stsig, BLSGPU_KERNEL_DECODE_SIG)));
  DstParam dst;
  make_dst(dst, IMPL, scheme, false);
  // MessageAugmentation hashes the multi key || msg (sig_aug.rs:20-24 on the MultiPublicKey's bytes)
  CKR((verify_points<IMPL>(ctx, scheme == 1 ? 1 : 0, dst, q, d_agg, d_sig, d_setst, d_stsig, d_msgs, d_moff, d_status)));
  CK(cudaMemcpyAsync(status_out, d_status, q, cudaMemcpyDeviceToHost, ctx->stream));
  CK(cudaStreamSynchronize(ctx->stream));
  stage_collect(ctx);
  return BLSGPU_OK;
}

// q x blsgpu_sum_points in one pass: decode, segmented sums, encode; per set the first bad element, counted inside the set
template <class A>
int sum_points_batch_impl(blsgpu_ctx* ctx, int format, size_t q, const uint64_t* set_off, const uint8_t* points, uint8_t* out,
                          uint8_t* status_out, int64_t* bad_index_out) {
  typedef typename PtInfo<A>::Jac J;
  const size_t L = PtInfo<A>::LEN, M = (size_t)set_off[q];
  const SegSumPlan pl(q, set_off);
  uint8_t *d_in, *d_st, *d_out;
  A *d_pts, *d_res;
  SegSums<J> ss;
  CKR(arena_takes(ctx, [&](auto& a) {
    d_in = take_up<uint8_t>(a, M * L);
    d_pts = a.template take<A>(std::max<size_t>(M, 1));
    d_st = a.template take<uint8_t>(std::max<size_t>(M, 1));
    take_seg_sums(a, pl, ss);
    d_res = a.template take<A>(q);
    d_out = a.template take<uint8_t>(q * L);
  }));
  CKR(upload(ctx, d_in, points, M * L));
  if (M) CKR((decode_points<A>(ctx, M, (const uint8_t*)d_in, format, d_pts, d_st)));
  CKR((seg_point_sums<A>(ctx, pl, ss, nullptr, d_pts, d_st)));
  unsigned long long* d_bad = ss.bad;
  LAUNCH((k_to_affine_batch<A>), blocks_for((q + TO_AFFINE_BATCH - 1) / TO_AFFINE_BATCH), TPB, q, (const J*)ss.sum, d_res);
  LAUNCH((k_encode<A>), blocks_for(q), TPB, q, (const A*)d_res, format, d_out);
  std::vector<unsigned long long> bad(q);
  CK(cudaMemcpyAsync(out, d_out, q * L, cudaMemcpyDeviceToHost, ctx->stream));
  CK(cudaMemcpyAsync(bad.data(), d_bad, q * sizeof(unsigned long long), cudaMemcpyDeviceToHost, ctx->stream));
  CK(cudaStreamSynchronize(ctx->stream));
  for (size_t j = 0; j < q; j++) {
    if (bad[j] == ~0ull) {
      status_out[j] = BLSGPU_ST_OK;
      if (bad_index_out) bad_index_out[j] = -1;
      continue;
    }
    status_out[j] = (uint8_t)(bad[j] & 0xff);
    if (bad_index_out) bad_index_out[j] = (int64_t)((bad[j] >> 8) - set_off[j]);
    memset(out + j * L, 0, L);
  }
  return BLSGPU_OK;
}

// both multi-signature calls (both formats for both impls, as blsgpu_verify_batch): the pipeline sees key_off from 0 and the
// keys from the first member on
int verify_multisig_common(blsgpu_ctx* ctx, const char* what, int impl_id, int scheme, int format, size_t q, const uint64_t* key_off, Keys keys,
                           const uint8_t* sigs, const uint8_t* msgs, const uint64_t* msg_off, uint8_t* status_out) {
  if (!args_ok(impl_id, scheme, format) || (q && (!sigs || !status_out))) return arg_error(ctx, what, "bad arguments");
  if (q == 0) return BLSGPU_OK;
  std::vector<uint64_t> ko;
  CKR(check_sets(ctx, what, "key_off", key_off, q, MEMBERS_CAP, ko));
  CKR(check_keys(ctx, what, impl_id, keys, key_off[0], ko[q]));
  CKR(check_records(ctx, what, "msgs", msgs, "msg_off", msg_off, q));
  CKR(set_device(ctx));
  return with_impl(impl_id, [&](auto I) { return verify_multisig_impl<I>(ctx, scheme, format, q, ko.data(), keys, sigs, msgs, msg_off, status_out); });
}

}  // namespace

int blsgpu_verify_multisig_batch(blsgpu_ctx* ctx, int impl_id, int scheme, int format, size_t q, const uint64_t* key_off, const uint8_t* pks,
                                 const uint8_t* sigs, const uint8_t* msgs, const uint64_t* msg_off, uint8_t* status_out) {
  NVTX_RANGE("blsgpu_verify_multisig_batch");
  if (!ctx) return BLSGPU_E_ARG;
  return verify_multisig_common(ctx, __func__, impl_id, scheme, format, q, key_off, pks, sigs, msgs, msg_off, status_out);
}

int blsgpu_verify_multisig_batch_keyed(blsgpu_ctx* ctx, uint64_t keyset, int scheme, int format, size_t q, const uint64_t* key_off,
                                       const uint32_t* key_idx, const uint8_t* sigs, const uint8_t* msgs, const uint64_t* msg_off,
                                       uint8_t* status_out) {
  NVTX_RANGE("blsgpu_verify_multisig_batch_keyed");
  if (!ctx) return BLSGPU_E_ARG;
  KeySet* set = nullptr;
  CKR(find_keyset(ctx, __func__, keyset, set));
  return verify_multisig_common(ctx, __func__, set->impl_id, scheme, format, q, key_off, Keys(set, key_idx), sigs, msgs, msg_off, status_out);
}

int blsgpu_sum_points_batch(blsgpu_ctx* ctx, int group, int format, size_t q, const uint64_t* set_off, const uint8_t* points, uint8_t* out,
                            uint8_t* status_out, int64_t* bad_index_out) {
  NVTX_RANGE("blsgpu_sum_points_batch");
  if (!ctx) return BLSGPU_E_ARG;
  if ((group != 1 && group != 2) || (format != 0 && format != 1) || (q && (!out || !status_out))) return arg_error(ctx, __func__, "bad arguments");
  if (q == 0) return BLSGPU_OK;
  std::vector<uint64_t> so;
  CKR(check_sets(ctx, __func__, "set_off", set_off, q, MEMBERS_CAP, so));
  if (points) points += set_off[0] * (group == 1 ? 48 : 96);
  CKR(check_buffer(ctx, __func__, "points", points, so[q]));
  CKR(set_device(ctx));
  return with_group(group, [&](auto G) {
    return sum_points_batch_impl<typename decltype(G)::type>(ctx, format, q, so.data(), points, out, status_out, bad_index_out);
  });
}

// ---------------------------------------------------------------------------------------------------------------------
// Threshold-share combination.  Host side: splitting the records, the set-level rules of vsss-rs `combine` (at least two
// shares, non-zero and distinct identifiers); device side: identifier parsing, Lagrange coefficients in Fr, the
// lambda_i * value_i multiplications, segmented sums, encoding.
template <class A>
static int combine_shares_impl(blsgpu_ctx* ctx, size_t q, const uint64_t* share_off, const uint8_t* shares, uint8_t* out, uint8_t* status_out) {
  typedef typename PtInfo<A>::Jac J;
  const size_t L = PtInfo<A>::LEN, REC = 32 + L, M = (size_t)share_off[q];
  std::vector<uint8_t> ids(M * 32), pts(M * L);
  std::vector<uint32_t> set_of(M), iota(M);
  for (size_t j = 0; j < q; j++)
    for (size_t i = (size_t)share_off[j]; i < (size_t)share_off[j + 1]; i++) {
      memcpy(&ids[i * 32], shares + i * REC, 32);
      memcpy(&pts[i * L], shares + i * REC + 32, L);
      set_of[i] = (uint32_t)j;
      iota[i] = (uint32_t)i;
    }
  const size_t nblocks = secure_msm_blocks(ctx, q);
  uint8_t *d_ids, *d_pts, *d_idflag, *d_stpt, *d_dup, *d_bad, *d_out;
  uint32_t *d_set, *d_iota, *d_raw;
  uint64_t* d_off;
  A *d_p, *d_res;
  int8_t* d_digits;
  J *d_buckets, *d_W, *d_sum;
  CKR(arena_takes(ctx, [&](auto& a) {
    d_ids = take_up<uint8_t>(a, M * 32);
    d_pts = take_up<uint8_t>(a, M * L);
    d_set = take_up<uint32_t>(a, M);
    d_iota = take_up<uint32_t>(a, M);
    d_off = take_up<uint64_t>(a, q + 1);
    d_raw = a.template take<uint32_t>(std::max<size_t>(M, 1) * 8);
    d_idflag = a.template take<uint8_t>(std::max<size_t>(M, 1));
    d_stpt = a.template take<uint8_t>(std::max<size_t>(M, 1));
    d_dup = a.template take<uint8_t>(std::max<size_t>(M, 1));
    d_bad = a.template take<uint8_t>(q);
    d_p = a.template take<A>(std::max<size_t>(M, 1));
    d_digits = a.template take<int8_t>(std::max<size_t>(M, 1) * SECURE_WINDOWS);
    d_buckets = a.template take<J>(nblocks * 128 * SECURE_BUCKETS);
    d_W = a.template take<J>(q * SECURE_WINDOWS);
    d_sum = a.template take<J>(q);
    d_res = a.template take<A>(q);
    d_out = a.template take<uint8_t>(q * L);
  }));
  CKR(upload(ctx, d_ids, ids.data(), M * 32));
  CKR(upload(ctx, d_pts, pts.data(), M * L));
  CKR(upload(ctx, d_set, set_of.data(), M));
  CKR(upload(ctx, d_iota, iota.data(), M));
  CKR(upload(ctx, d_off, share_off, q + 1));
  std::vector<uint8_t> idflag(M), stpt(M), dup(M), bad(q, 0);
  if (M) {
    LAUNCH(k_share_ids, blocks_for(M), TPB, M, (const uint8_t*)d_ids, d_raw, d_idflag);
    CKR((decode_points<A>(ctx, M, (const uint8_t*)d_pts, 1, d_p, d_stpt)));
    CK(cudaMemcpyAsync(idflag.data(), d_idflag, M, cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaMemcpyAsync(stpt.data(), d_stpt, M, cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
  }
  // parse errors first (every share is parsed before `combine` runs), then the set rules
  for (size_t j = 0; j < q; j++) {
    const size_t lo = (size_t)share_off[j], hi = (size_t)share_off[j + 1];
    uint8_t s = BLSGPU_ST_OK;
    for (size_t i = lo; i < hi && s == BLSGPU_ST_OK; i++)
      if (idflag[i] == 1 || stpt[i] != BLSGPU_ST_OK) s = BLSGPU_ST_DESERIALIZE;
    if (s == BLSGPU_ST_OK && hi - lo < 2) s = BLSGPU_ST_VSSS;
    for (size_t i = lo; i < hi && s == BLSGPU_ST_OK; i++)
      if (idflag[i] == 2) s = BLSGPU_ST_VSSS;
    status_out[j] = s;
    bad[j] = s != BLSGPU_ST_OK;
  }
  CK(cudaMemcpyAsync(d_bad, bad.data(), q, cudaMemcpyHostToDevice, ctx->stream));
  if (M) {
    // lambda_i as window digits, then one bucket multi-scalar multiplication per share set (a warp per set)
    LAUNCH(k_share_digits, blocks_for(M), TPB, M, (const uint32_t*)d_set, (const uint64_t*)d_off, (const uint8_t*)d_bad, (const uint32_t*)d_raw,
           d_digits, d_dup);
    CK(cudaMemcpyAsync(dup.data(), d_dup, M, cudaMemcpyDeviceToHost, ctx->stream));
  }
  LAUNCH((k_secure_msm<A>), (unsigned)nblocks, 128, q, (const uint64_t*)d_off, (const uint32_t*)d_iota, (const int8_t*)d_digits, (const A*)d_p,
         d_buckets, d_W);
  LAUNCH((k_secure_combine<J>), blocks_for(q), TPB, q, (const J*)d_W, d_sum);
  LAUNCH((k_to_affine<A>), blocks_for(q), TPB, q, (const J*)d_sum, d_res);
  LAUNCH((k_encode<A>), blocks_for(q), TPB, q, (const A*)d_res, 1, d_out);
  CK(cudaMemcpyAsync(out, d_out, q * L, cudaMemcpyDeviceToHost, ctx->stream));
  CK(cudaStreamSynchronize(ctx->stream));
  for (size_t j = 0; j < q; j++) {
    if (status_out[j] == BLSGPU_ST_OK)
      for (size_t i = (size_t)share_off[j]; i < (size_t)share_off[j + 1]; i++)
        if (dup[i]) status_out[j] = BLSGPU_ST_VSSS;
    if (status_out[j] != BLSGPU_ST_OK) memset(out + j * L, 0, L);
  }
  return BLSGPU_OK;
}

int blsgpu_combine_shares_batch(blsgpu_ctx* ctx, int group, size_t q, const uint64_t* share_off, const uint8_t* shares, uint8_t* out,
                                uint8_t* status_out) {
  NVTX_RANGE("blsgpu_combine_shares_batch");
  if (!ctx) return BLSGPU_E_ARG;
  if ((group != 1 && group != 2) || (q && (!out || !status_out))) return arg_error(ctx, __func__, "bad arguments");
  if (q == 0) return BLSGPU_OK;
  std::vector<uint64_t> so;
  CKR(check_sets(ctx, __func__, "share_off", share_off, q, NO_CAP, so));
  if (shares) shares += share_off[0] * (32 + (group == 1 ? 48 : 96));
  CKR(check_buffer(ctx, __func__, "shares", shares, so[q]));
  CKR(set_device(ctx));
  return with_group(group, [&](auto G) { return combine_shares_impl<typename decltype(G)::type>(ctx, q, so.data(), shares, out, status_out); });
}

// ---------------------------------------------------------------------------------------------------------------------
// Wire-format front end: tagged signatures, schemes mixed in one call.  Fixed-size records: blsgpu_verify_batch_records in
// tagged mode does the rest.
int blsgpu_verify_batch_wire(blsgpu_ctx* ctx, int impl_id, size_t n, const uint8_t* pks, const uint8_t* tagged_sigs, const uint8_t* msgs,
                             const uint64_t* msg_off, uint8_t* status_out) {
  NVTX_RANGE("blsgpu_verify_batch_wire");
  if (!ctx) return BLSGPU_E_ARG;
  if ((impl_id != 1 && impl_id != 2) || (n && (!pks || !tagged_sigs || !status_out))) return arg_error(ctx, __func__, "bad arguments");
  CKR(check_records(ctx, __func__, "msgs", msgs, "msg_off", msg_off, n));
  const size_t pk_len = impl_id == 2 ? 48 : 96, rec = (impl_id == 2 ? 96 : 48) + 1;
  std::vector<uint64_t> pk_off(n + 1), sig_off(n + 1);
  for (size_t i = 0; i <= n; i++) {
    pk_off[i] = i * pk_len;
    sig_off[i] = i * rec;
  }
  return blsgpu_verify_batch_records(ctx, impl_id, 1, -1, n, pks, pk_off.data(), tagged_sigs, sig_off.data(), msgs, msg_off, status_out);
}

// ---------------------------------------------------------------------------------------------------------------------
// Share verification on raw share records: strip (and validate) the identifiers on the host, verify the values.
int blsgpu_verify_share_batch(blsgpu_ctx* ctx, int impl_id, int scheme, size_t n, const uint8_t* pk_shares, const uint8_t* sig_shares,
                              const uint8_t* msgs, const uint64_t* msg_off, uint8_t* status_out) {
  NVTX_RANGE("blsgpu_verify_share_batch");
  if (!ctx) return BLSGPU_E_ARG;
  if (!args_ok(impl_id, scheme, 1) || (n && (!pk_shares || !sig_shares || !msg_off || !status_out))) return arg_error(ctx, __func__, "bad arguments");
  if (n == 0) return BLSGPU_OK;
  static const uint8_t R_BE[32] = {0x73, 0xed, 0xa7, 0x53, 0x29, 0x9d, 0x7d, 0x48, 0x33, 0x39, 0xd8, 0x08, 0x09, 0xa1, 0xd8, 0x05,
                                   0x53, 0xbd, 0xa4, 0x02, 0xff, 0xfe, 0x5b, 0xfe, 0xff, 0xff, 0xff, 0xff, 0x00, 0x00, 0x00, 0x01};
  const size_t pk_len = impl_id == 2 ? 48 : 96, sig_len = impl_id == 2 ? 96 : 48;
  std::vector<uint8_t> p(n * pk_len), g(n * sig_len), bad_id(n, 0);
  for (size_t i = 0; i < n; i++) {
    const uint8_t* pr = pk_shares + i * (32 + pk_len);
    const uint8_t* sr = sig_shares + i * (32 + sig_len);
    bad_id[i] = memcmp(pr, R_BE, 32) >= 0 || memcmp(sr, R_BE, 32) >= 0;  // Scalar::from_be_bytes rejects values >= r
    memcpy(&p[i * pk_len], pr + 32, pk_len);
    memcpy(&g[i * sig_len], sr + 32, sig_len);
  }
  CKR(verify_batch_common(ctx, __func__, impl_id, scheme, 1, n, p.data(), g.data(), msgs, msg_off, status_out));
  for (size_t i = 0; i < n; i++)
    if (bad_id[i]) status_out[i] = BLSGPU_ST_DESERIALIZE;
  return BLSGPU_OK;
}

// ---------------------------------------------------------------------------------------------------------------------
int blsgpu_pairing_check_batch(blsgpu_ctx* ctx, size_t q, const uint64_t* pair_off, const uint8_t* g1_points, const uint8_t* g2_points,
                               uint8_t* ok_out, uint8_t* status_out) {
  NVTX_RANGE("blsgpu_pairing_check_batch");
  if (!ctx) return BLSGPU_E_ARG;
  if (q && (!ok_out || !status_out)) return arg_error(ctx, __func__, "bad arguments");
  if (q == 0) return BLSGPU_OK;
  std::vector<uint64_t> po;
  CKR(check_sets(ctx, __func__, "pair_off", pair_off, q, NO_CAP, po));
  const size_t M = (size_t)po[q];
  if (g1_points) g1_points += pair_off[0] * 48;
  if (g2_points) g2_points += pair_off[0] * 96;
  CKR(check_buffer(ctx, __func__, "g1_points", g1_points, M));
  CKR(check_buffer(ctx, __func__, "g2_points", g2_points, M));
  pair_off = po.data();
  CKR(set_device(ctx));
  uint8_t *d_a, *d_b, *d_st, *d_ok;
  uint64_t* d_off;
  G1Aff* d_p;
  G2Aff* d_q;
  Fp12* d_F;
  CKR(arena_takes(ctx, [&](auto& a) {
    d_a = take_up<uint8_t>(a, M * 48);
    d_b = take_up<uint8_t>(a, M * 96);
    d_off = take_up<uint64_t>(a, q + 1);
    d_p = a.template take<G1Aff>(std::max<size_t>(M, 1));
    d_q = a.template take<G2Aff>(std::max<size_t>(M, 1));
    d_st = a.template take<uint8_t>(2 * std::max<size_t>(M, 1));
    d_F = a.template take<Fp12>(std::max<size_t>(M, 1));
    d_ok = a.template take<uint8_t>(q);
  }));
  CKR(upload(ctx, d_a, g1_points, M * 48));
  CKR(upload(ctx, d_b, g2_points, M * 96));
  CKR(upload(ctx, d_off, pair_off, q + 1));
  std::vector<uint8_t> st(2 * M);
  if (M) {
    CKR((decode_points<G1Aff>(ctx, M, (const uint8_t*)d_a, 1, d_p, d_st)));
    CKR((decode_points<G2Aff>(ctx, M, (const uint8_t*)d_b, 1, d_q, d_st + M)));
    LAUNCH(k_miller_pairs, blocks_for(M), TPB, M, (const G1Aff*)d_p, (const G2Aff*)d_q, d_F);  // undecodable -> identity -> 1
    CK(cudaMemcpyAsync(st.data(), d_st, 2 * M, cudaMemcpyDeviceToHost, ctx->stream));
  }
  LAUNCH(k_set_final_is_one, blocks_for(q, 64), 64, q, (const uint64_t*)d_off, (const Fp12*)d_F, d_ok);
  CK(cudaMemcpyAsync(ok_out, d_ok, q, cudaMemcpyDeviceToHost, ctx->stream));
  CK(cudaStreamSynchronize(ctx->stream));
  for (size_t j = 0; j < q; j++) {
    status_out[j] = BLSGPU_ST_OK;
    for (size_t i = (size_t)pair_off[j]; i < (size_t)pair_off[j + 1]; i++)
      if (st[i] != BLSGPU_ST_OK || st[M + i] != BLSGPU_ST_OK) status_out[j] = BLSGPU_ST_DESERIALIZE;
    if (status_out[j] != BLSGPU_ST_OK) ok_out[j] = 0;
  }
  return BLSGPU_OK;
}

// ---------------------------------------------------------------------------------------------------------------------
// The reference's other public 2-pairing checks (SURVEY.md section 8f-4), pairs assembled on the device.

// SignCryptCiphertext::is_valid -> BlsSignCrypt::valid(u, v, w, dst)  ==  core_verify(pk = u, sig = w, msg = u.to_bytes() || v, dst)
// as a boolean: both check  pairing([(w, -g), (hash_to_point(u_bytes || v), u)]) == 1  and reject identity u / w.
int blsgpu_signcrypt_valid_batch(blsgpu_ctx* ctx, int impl_id, int scheme, size_t n, const uint8_t* u_points, const uint8_t* w_points,
                                 const uint8_t* v_bytes, const uint64_t* v_off, uint8_t* ok_out, uint8_t* status_out) {
  NVTX_RANGE("blsgpu_signcrypt_valid_batch");
  if (!ctx) return BLSGPU_E_ARG;
  if (!args_ok(impl_id, scheme, 1) || (n && (!u_points || !w_points || !ok_out || !status_out))) return arg_error(ctx, __func__, "bad arguments");
  if (n == 0) return BLSGPU_OK;
  CKR(check_records(ctx, __func__, "v_bytes", v_bytes, "v_off", v_off, n));
  DstParam dst;
  make_dst(dst, impl_id, scheme, false);
  CKR(verify_host_common(ctx, impl_id, 1, dst, 1, n, u_points, w_points, v_bytes, v_off, status_out));
  for (size_t i = 0; i < n; i++) {
    ok_out[i] = status_out[i] == BLSGPU_ST_OK;
    if (status_out[i] != BLSGPU_ST_DESERIALIZE) status_out[i] = BLSGPU_ST_OK;  // only parse errors are errors; the rest is `false`
  }
  return BLSGPU_OK;
}

namespace {
static const uint8_t R_ORDER_BE[32] = {0x73, 0xed, 0xa7, 0x53, 0x29, 0x9d, 0x7d, 0x48, 0x33, 0x39, 0xd8, 0x08, 0x09, 0xa1, 0xd8, 0x05,
                                       0x53, 0xbd, 0xa4, 0x02, 0xff, 0xfe, 0x5b, 0xfe, 0xff, 0xff, 0xff, 0xff, 0x00, 0x00, 0x00, 0x01};

// the scratch of pair2_check over n items: the pairs' Miller values and the item offsets
struct Pair2 {
  Fp12* F = nullptr;
  uint64_t* off = nullptr;
};
template <class A>
void take_pair2(A& a, size_t n, Pair2& s) {
  s.F = a.template take<Fp12>(2 * n);
  s.off = a.template take<uint64_t>(n + 1);
}
// prod over the two pairs of every item == 1 ?  (one thread per pair / per item: these checks are low-volume)
int pair2_check(blsgpu_ctx* ctx, size_t n, const Pair2& s, const G1Aff* d_g1, const G2Aff* d_g2, uint8_t* d_ok) {
  Fp12* d_F = s.F;
  uint64_t* d_off = s.off;
  LAUNCH(k_pair_offsets, blocks_for(n + 1), TPB, n, d_off);
  LAUNCH(k_miller_pairs, blocks_for(2 * n), TPB, 2 * n, d_g1, d_g2, d_F);
  LAUNCH(k_set_final_is_one, blocks_for(n, 64), 64, n, (const uint64_t*)d_off, (const Fp12*)d_F, d_ok);
  return BLSGPU_OK;
}

template <int IMPL>
int pok_verify_impl(blsgpu_ctx* ctx, int scheme, size_t n, const uint8_t* commitments, const uint8_t* proofs, const uint8_t* pks,
                    const uint8_t* ys, const uint8_t* msgs, const uint64_t* msg_off, uint8_t* status_out) {
  typedef typename ImplT<IMPL>::PkAff PkA;
  typedef typename ImplT<IMPL>::SigAff SigA;
  typedef typename PtInfo<SigA>::Jac SigJ;
  const size_t Lp = PtInfo<PkA>::LEN, Ls = PtInfo<SigA>::LEN;
  std::vector<uint8_t> yflag(n);
  for (size_t i = 0; i < n; i++) {
    const uint8_t* y = ys + 32 * i;
    bool zero = true;
    for (int b = 0; b < 32; b++) zero = zero && y[b] == 0;
    yflag[i] = memcmp(y, R_ORDER_BE, 32) >= 0 ? 1 : zero ? 2 : 0;  // Scalar parsing rejects values >= r
  }
  uint8_t *d_cmb, *d_prb, *d_pkb, *d_y, *d_yf, *d_msgs, *d_st, *d_ok;
  uint64_t* d_moff;
  SigA *d_cm, *d_pr, *d_a;
  PkA* d_pk;
  SigJ* d_hj;
  G1Aff* d_g1;
  G2Aff* d_g2;
  Pair2 p2;
  CKR(arena_takes(ctx, [&](auto& a) {
    d_cmb = take_up<uint8_t>(a, n * Ls);
    d_prb = take_up<uint8_t>(a, n * Ls);
    d_pkb = take_up<uint8_t>(a, n * Lp);
    d_y = take_up<uint8_t>(a, n * 32);
    d_yf = take_up<uint8_t>(a, n);
    take_records(a, msg_off, n, d_msgs, d_moff);
    d_cm = a.template take<SigA>(n);
    d_pr = a.template take<SigA>(n);
    d_a = a.template take<SigA>(n);
    d_pk = a.template take<PkA>(n);
    d_st = a.template take<uint8_t>(4 * n);
    d_ok = a.template take<uint8_t>(n);
    d_g1 = a.template take<G1Aff>(2 * n);
    d_g2 = a.template take<G2Aff>(2 * n);
    d_hj = take_hash_scratch<SigA>(a, n);
    take_pair2(a, n, p2);
  }));
  CKR(upload(ctx, d_cmb, commitments, n * Ls));
  CKR(upload(ctx, d_prb, proofs, n * Ls));
  CKR(upload(ctx, d_pkb, pks, n * Lp));
  CKR(upload(ctx, d_y, ys, n * 32));
  CKR(upload(ctx, d_yf, yflag.data(), n));
  CKR(upload_records(ctx, msgs, msg_off, n, d_msgs, d_moff));
  uint8_t *d_stcm = d_st, *d_stpr = d_st + n, *d_stpk = d_st + 2 * n, *d_status = d_st + 3 * n;
  CKR((decode_points<SigA>(ctx, n, (const uint8_t*)d_cmb, 1, d_cm, d_stcm)));
  CKR((decode_points<SigA>(ctx, n, (const uint8_t*)d_prb, 1, d_pr, d_stpr)));
  CKR((decode_points<PkA>(ctx, n, (const uint8_t*)d_pkb, 1, d_pk, d_stpk)));
  LAUNCH((k_pok_prestatus<PkA, SigA>), blocks_for(n), TPB, n, (const uint8_t*)d_stcm, (const uint8_t*)d_stpr, (const uint8_t*)d_stpk,
         (const uint8_t*)d_yf, (const SigA*)d_cm, (const SigA*)d_pr, (const PkA*)d_pk, d_status);
  DstParam dst;
  make_dst(dst, IMPL, scheme, false);
  CKR((hash_points<SigA, PkA>(ctx, n, (const uint8_t*)d_msgs, (const uint64_t*)d_moff, 0, (const PkA*)d_pk, (const uint8_t*)d_status, dst, d_hj, d_a)));
  LAUNCH((k_pok_pairs<PkA, SigA>), blocks_for(n), TPB, n, (const uint8_t*)d_status, (const SigA*)d_a, (const SigA*)d_cm, (const SigA*)d_pr,
         (const PkA*)d_pk, (const uint8_t*)d_y, d_g1, d_g2);
  CKR(pair2_check(ctx, n, p2, d_g1, d_g2, d_ok));
  LAUNCH(k_pok_finish, blocks_for(n), TPB, n, (const uint8_t*)d_ok, d_status);
  CK(cudaMemcpyAsync(status_out, d_status, n, cudaMemcpyDeviceToHost, ctx->stream));
  CK(cudaStreamSynchronize(ctx->stream));
  return BLSGPU_OK;
}

template <int IMPL>
int signcrypt_share_impl(blsgpu_ctx* ctx, int scheme, size_t n, const uint8_t* shares, const uint8_t* pks, const uint8_t* us, const uint8_t* ws,
                         const uint8_t* v_bytes, const uint64_t* v_off, uint8_t* ok_out, uint8_t* status_out) {
  typedef typename ImplT<IMPL>::PkAff PkA;
  typedef typename ImplT<IMPL>::SigAff SigA;
  typedef typename PtInfo<SigA>::Jac SigJ;
  const size_t Lp = PtInfo<PkA>::LEN, Ls = PtInfo<SigA>::LEN;
  uint8_t *d_shb, *d_pkb, *d_ub, *d_wb, *d_v, *d_st;
  uint64_t* d_voff;
  PkA *d_sh, *d_pk, *d_u;
  SigA *d_w, *d_wt;
  SigJ* d_hj;
  G1Aff* d_g1;
  G2Aff* d_g2;
  Pair2 p2;
  CKR(arena_takes(ctx, [&](auto& a) {
    d_shb = take_up<uint8_t>(a, n * Lp);
    d_pkb = take_up<uint8_t>(a, n * Lp);
    d_ub = take_up<uint8_t>(a, n * Lp);
    d_wb = take_up<uint8_t>(a, n * Ls);
    take_records(a, v_off, n, d_v, d_voff);
    d_sh = a.template take<PkA>(n);
    d_pk = a.template take<PkA>(n);
    d_u = a.template take<PkA>(n);
    d_w = a.template take<SigA>(n);
    d_wt = a.template take<SigA>(n);
    d_st = a.template take<uint8_t>(6 * n);
    d_g1 = a.template take<G1Aff>(2 * n);
    d_g2 = a.template take<G2Aff>(2 * n);
    d_hj = take_hash_scratch<SigA>(a, n);
    take_pair2(a, n, p2);
  }));
  CKR(upload(ctx, d_shb, shares, n * Lp));
  CKR(upload(ctx, d_pkb, pks, n * Lp));
  CKR(upload(ctx, d_ub, us, n * Lp));
  CKR(upload(ctx, d_wb, ws, n * Ls));
  CKR(upload_records(ctx, v_bytes, v_off, n, d_v, d_voff));
  uint8_t *d_s0 = d_st, *d_s1 = d_st + n, *d_s2 = d_st + 2 * n, *d_s3 = d_st + 3 * n, *d_flag = d_st + 4 * n, *d_ok = d_st + 5 * n;
  CKR((decode_points<PkA>(ctx, n, (const uint8_t*)d_shb, 1, d_sh, d_s0)));
  CKR((decode_points<PkA>(ctx, n, (const uint8_t*)d_pkb, 1, d_pk, d_s1)));
  CKR((decode_points<PkA>(ctx, n, (const uint8_t*)d_ub, 1, d_u, d_s2)));
  CKR((decode_points<SigA>(ctx, n, (const uint8_t*)d_wb, 1, d_w, d_s3)));
  std::vector<uint8_t> st(4 * n);
  CK(cudaMemcpyAsync(st.data(), d_st, 4 * n, cudaMemcpyDeviceToHost, ctx->stream));
  CK(cudaStreamSynchronize(ctx->stream));
  for (size_t i = 0; i < n; i++) {
    uint8_t s = st[i];
    for (int k = 1; k < 4 && s == BLSGPU_ST_OK; k++) s = st[k * n + i];
    status_out[i] = s;
  }
  CK(cudaMemcpyAsync(d_s0, status_out, n, cudaMemcpyHostToDevice, ctx->stream));  // d_s0 now holds the combined parse status
  DstParam dst;
  make_dst(dst, IMPL, scheme, false);
  // W' = hash_to_point(u.to_bytes() || v): the pk-prefix framing with u in the key's place (compute_w, sign_crypt.rs:151-158)
  CKR((hash_points<SigA, PkA>(ctx, n, (const uint8_t*)d_v, (const uint64_t*)d_voff, 1, (const PkA*)d_u, (const uint8_t*)d_s0, dst, d_hj, d_wt)));
  LAUNCH((k_signcrypt_share_pairs<PkA, SigA>), blocks_for(n), TPB, n, (const uint8_t*)d_s0, (const SigA*)d_wt, (const PkA*)d_sh, (const PkA*)d_pk,
         (const SigA*)d_w, d_g1, d_g2, d_flag);
  CKR(pair2_check(ctx, n, p2, d_g1, d_g2, d_ok));
  LAUNCH(k_and_flags, blocks_for(n), TPB, n, (const uint8_t*)d_flag, d_ok);
  CK(cudaMemcpyAsync(ok_out, d_ok, n, cudaMemcpyDeviceToHost, ctx->stream));
  CK(cudaStreamSynchronize(ctx->stream));
  return BLSGPU_OK;
}
}  // namespace

int blsgpu_pok_verify_batch(blsgpu_ctx* ctx, int impl_id, int scheme, size_t n, const uint8_t* commitments, const uint8_t* proofs,
                            const uint8_t* pks, const uint8_t* challenges32, const uint8_t* msgs, const uint64_t* msg_off, uint8_t* status_out) {
  NVTX_RANGE("blsgpu_pok_verify_batch");
  if (!ctx) return BLSGPU_E_ARG;
  if (!args_ok(impl_id, scheme, 1) || (n && (!commitments || !proofs || !pks || !challenges32 || !status_out))) return arg_error(ctx, __func__, "bad arguments");
  if (n == 0) return BLSGPU_OK;
  CKR(check_records(ctx, __func__, "msgs", msgs, "msg_off", msg_off, n));
  CKR(set_device(ctx));
  return with_impl(impl_id, [&](auto I) { return pok_verify_impl<I>(ctx, scheme, n, commitments, proofs, pks, challenges32, msgs, msg_off, status_out); });
}

int blsgpu_signcrypt_verify_share_batch(blsgpu_ctx* ctx, int impl_id, int scheme, size_t n, const uint8_t* shares, const uint8_t* pk_shares,
                                        const uint8_t* u_points, const uint8_t* w_points, const uint8_t* v_bytes, const uint64_t* v_off,
                                        uint8_t* ok_out, uint8_t* status_out) {
  NVTX_RANGE("blsgpu_signcrypt_verify_share_batch");
  if (!ctx) return BLSGPU_E_ARG;
  if (!args_ok(impl_id, scheme, 1) || (n && (!shares || !pk_shares || !u_points || !w_points || !ok_out || !status_out)))
    return arg_error(ctx, __func__, "bad arguments");
  if (n == 0) return BLSGPU_OK;
  CKR(check_records(ctx, __func__, "v_bytes", v_bytes, "v_off", v_off, n));
  CKR(set_device(ctx));
  return with_impl(impl_id, [&](auto I) {
    return signcrypt_share_impl<I>(ctx, scheme, n, shares, pk_shares, u_points, w_points, v_bytes, v_off, ok_out, status_out);
  });
}

// ---------------------------------------------------------------------------------------------------------------------
// Wire front end on ragged records (SURVEY.md section 8f-3): length rules, tags and the Legacy / Modern header validation
// happen here, so callers hand over network buffers as they arrived.
int blsgpu_verify_batch_records(blsgpu_ctx* ctx, int impl_id, int format, int scheme_or_tagged, size_t n, const uint8_t* pk_bytes,
                                const uint64_t* pk_off, const uint8_t* sig_bytes, const uint64_t* sig_off, const uint8_t* msgs,
                                const uint64_t* msg_off, uint8_t* status_out) {
  NVTX_RANGE("blsgpu_verify_batch_records");
  if (!ctx) return BLSGPU_E_ARG;
  const bool tagged = scheme_or_tagged < 0;
  if ((impl_id != 1 && impl_id != 2) || (format != 0 && format != 1) || scheme_or_tagged > 2 || (n && !status_out))
    return arg_error(ctx, __func__, "bad arguments");
  if (n == 0) return BLSGPU_OK;
  CKR(check_records(ctx, __func__, "pk_bytes", pk_bytes, "pk_off", pk_off, n));
  CKR(check_records(ctx, __func__, "sig_bytes", sig_bytes, "sig_off", sig_off, n));
  CKR(check_records(ctx, __func__, "msgs", msgs, "msg_off", msg_off, n));
  const size_t pk_len = impl_id == 2 ? 48 : 96, sig_len = impl_id == 2 ? 96 : 48;
  // InvalidLength (public_key.rs:159-164, signature.rs:236-241) and the serde_bare tag (signature.rs:120-126) per record;
  // well-formed records are regrouped by scheme and go through blsgpu_verify_batch in `format`
  std::vector<int8_t> scheme_of(n, -1);
  for (size_t i = 0; i < n; i++) {
    const size_t pl = (size_t)(pk_off[i + 1] - pk_off[i]), sl = (size_t)(sig_off[i + 1] - sig_off[i]);
    status_out[i] = BLSGPU_ST_OK;
    if (pl != pk_len) {
      status_out[i] = BLSGPU_ST_INVALID_LENGTH;
    } else if (tagged) {
      // serde_bare: a short or long buffer and an unknown tag are both `InvalidInputs(serde error)`
      if (sl != sig_len + 1 || sig_bytes[sig_off[i]] > 2) status_out[i] = BLSGPU_ST_DESERIALIZE;
      else scheme_of[i] = (int8_t)sig_bytes[sig_off[i]];
    } else if (sl != sig_len) {
      status_out[i] = BLSGPU_ST_INVALID_LENGTH;
    } else {
      scheme_of[i] = (int8_t)scheme_or_tagged;
    }
  }
  for (int scheme = 0; scheme < 3; scheme++) {
    std::vector<size_t> idx;
    for (size_t i = 0; i < n; i++)
      if (scheme_of[i] == scheme) idx.push_back(i);
    if (idx.empty()) continue;
    std::vector<uint8_t> p(idx.size() * pk_len), g(idx.size() * sig_len), m, st(idx.size());
    std::vector<uint64_t> off(idx.size() + 1, 0);
    for (size_t k = 0; k < idx.size(); k++) {
      const size_t i = idx[k];
      memcpy(&p[k * pk_len], pk_bytes + pk_off[i], pk_len);
      memcpy(&g[k * sig_len], sig_bytes + sig_off[i] + (tagged ? 1 : 0), sig_len);
      if (msg_off[i + 1] > msg_off[i]) m.insert(m.end(), msgs + msg_off[i], msgs + msg_off[i + 1]);
      off[k + 1] = m.size();
    }
    // the tagged (serde) form always carries the IETF encoding; raw records are in the caller's format
    CKR(blsgpu_verify_batch(ctx, impl_id, scheme, tagged ? 1 : format, idx.size(), p.data(), g.data(), m.empty() ? p.data() : m.data(), off.data(),
                            st.data()));
    for (size_t k = 0; k < idx.size(); k++) status_out[idx[k]] = st[k];
  }
  return BLSGPU_OK;
}

// ---------------------------------------------------------------------------------------------------------------------
// Known-answer self-test of the device code.  This code base has met device-only wrong results that were compiler
// artefacts (DESIGN.md section 9: a dropped struct copy in cicc, stack colouring): a build that miscompiles the arithmetic
// must fail HERE, loudly, not return wrong verdicts.  Vectors: the first C++ bls-signatures triple of the reference's
// tests/cpp_integration_test.rs:19-82 (message "hello") and H("hello") derived from it (sig = sk * H).
int blsgpu_selftest(blsgpu_ctx* ctx) {
  NVTX_RANGE("blsgpu_selftest");
  if (!ctx) return BLSGPU_E_ARG;
  static const uint8_t PK1[48] = {0xb1, 0x45, 0xdf, 0xcb, 0x3c, 0xbd, 0xef, 0x21, 0x50, 0x2f, 0x30, 0x5d, 0x1b, 0xa1, 0xcb, 0xa5, 0x84, 0x79, 0x69, 0x18, 0x57, 0x1e, 0x8b, 0x5d, 0x85, 0xbe, 0x17, 0x6f, 0x34, 0x45, 0xac, 0x7a, 0xd9, 0x9a, 0xec, 0x19, 0xe1, 0x93, 0x1b, 0x69, 0x34, 0xd7, 0x29, 0x0b, 0x97, 0xec, 0x2d, 0x75};
  static const uint8_t SIG1[96] = {0x82, 0xc8, 0x08, 0x03, 0xa3, 0x24, 0x6f, 0x5d, 0x10, 0xb5, 0x19, 0x23, 0xd4, 0x96, 0x7b, 0xef, 0x55, 0x7c, 0xf0, 0x41, 0x6f, 0xa3, 0x06, 0x05, 0x94, 0x9c, 0xaa, 0xc6, 0x27, 0x3b, 0x59, 0x93, 0xd2, 0x6f, 0xef, 0x27, 0x8e, 0xb4, 0x86, 0x75, 0xc6, 0x2b, 0x42, 0x26, 0x6f, 0x9b, 0x01, 0x48, 0x0a, 0x8d, 0xc0, 0x7e, 0xf1, 0x68, 0xed, 0xd3, 0xf1, 0xa9, 0xca, 0xd3, 0x63, 0x30, 0x83, 0xdc, 0xb3, 0xc2, 0xdf, 0x37, 0x27, 0x89, 0xb8, 0x78, 0x71, 0x24, 0x9d, 0xab, 0x38, 0x0b, 0x07, 0x1d, 0xd4, 0x80, 0xd7, 0x42, 0xd0, 0x27, 0xf3, 0x7c, 0x36, 0xf8, 0x9e, 0x63, 0xb5, 0xf1, 0xe0, 0x93};
  static const uint8_t SIG2[96] = {0xb2, 0xca, 0x57, 0x80, 0x16, 0xe8, 0x96, 0x20, 0xb4, 0x94, 0x03, 0xa0, 0x29, 0xad, 0x96, 0x40, 0x27, 0x2c, 0x18, 0x45, 0x5a, 0x5f, 0xdd, 0xc4, 0x0f, 0x99, 0x9b, 0xd7, 0x5c, 0xb9, 0xda, 0xc0, 0x71, 0x61, 0x3c, 0xb5, 0xa6, 0x64, 0xe0, 0xa7, 0x19, 0xa2, 0x29, 0xff, 0x65, 0x51, 0xfd, 0x52, 0x0b, 0x6d, 0x92, 0x96, 0x75, 0x08, 0xd5, 0xf1, 0xf5, 0x8c, 0xd4, 0x14, 0xcb, 0xde, 0x44, 0xc9, 0xe3, 0x91, 0x18, 0x73, 0xb4, 0xa2, 0xe9, 0x54, 0x44, 0x29, 0xb8, 0x67, 0x6f, 0xca, 0x69, 0xcb, 0x97, 0xab, 0xc6, 0xf4, 0x99, 0x16, 0xd0, 0x8c, 0xee, 0xda, 0x42, 0xb0, 0x6b, 0xe3, 0x6f, 0xf4};
  static const uint8_t FA[48] = {0x00, 0x00, 0x00, 0x00, 0x00, 0x00, 0x00, 0x00, 0x00, 0x00, 0x00, 0x00, 0x00, 0x00, 0x00, 0x00, 0x00, 0x00, 0x00, 0x00, 0x00, 0x00, 0x01, 0x00, 0x00, 0x00, 0x00, 0x00, 0x00, 0x00, 0x00, 0x00, 0x00, 0x00, 0x00, 0x00, 0x00, 0x00, 0x00, 0x00, 0x00, 0x00, 0x00, 0x00, 0x00, 0x00, 0x30, 0x39};
  static const uint8_t FB[48] = {0x1a, 0x01, 0x11, 0xea, 0x39, 0x7f, 0xe6, 0x9a, 0x4b, 0x1b, 0xa7, 0xb6, 0x43, 0x4b, 0xac, 0xd7, 0x64, 0x77, 0x4b, 0x84, 0xf3, 0x85, 0x12, 0xbf, 0x67, 0x30, 0xd2, 0xa0, 0xf6, 0xb0, 0xf6, 0x24, 0x1e, 0xab, 0xff, 0xfe, 0xb1, 0x53, 0xff, 0xff, 0xb9, 0xfe, 0xff, 0xff, 0xff, 0xff, 0xaa, 0xa9};
  static const uint8_t FAB[48] = {0x1a, 0x01, 0x11, 0xea, 0x39, 0x7f, 0xe6, 0x9a, 0x4b, 0x1b, 0xa7, 0xb6, 0x43, 0x4b, 0xac, 0xd7, 0x64, 0x77, 0x4b, 0x84, 0xf3, 0x85, 0x10, 0xbf, 0x67, 0x30, 0xd2, 0xa0, 0xf6, 0xb0, 0xf6, 0x24, 0x1e, 0xab, 0xff, 0xfe, 0xb1, 0x53, 0xff, 0xff, 0xb9, 0xfe, 0xff, 0xff, 0xff, 0xff, 0x4a, 0x39};
  static const uint8_t HHELLO[96] = {0x8d, 0xbf, 0x4d, 0x3c, 0x42, 0x6b, 0xad, 0xac, 0x1e, 0x66, 0x42, 0x1c, 0x7d, 0x65, 0xdc, 0x01, 0x7c, 0x05, 0xfb, 0x76, 0x31, 0x83, 0x3f, 0x3c, 0x9a, 0x72, 0xf5, 0x31, 0xbe, 0xdf, 0x79, 0x95, 0xf2, 0x30, 0x9d, 0x2f, 0xd6, 0x83, 0x10, 0x18, 0xc8, 0x3d, 0xe0, 0xc2, 0x7b, 0x6a, 0x10, 0xc8, 0x10, 0x94, 0x69, 0x37, 0xad, 0x15, 0x67, 0x4b, 0x2f, 0x39, 0x76, 0xd1, 0x0f, 0x50, 0xae, 0x5a, 0x66, 0xa0, 0x7f, 0x5d, 0xa2, 0x3a, 0x4f, 0x17, 0x78, 0x70, 0x70, 0x2d, 0x0d, 0xbf, 0x84, 0x63, 0x22, 0x5a, 0x49, 0x3a, 0x8c, 0x22, 0x10, 0x32, 0xe1, 0x5d, 0x44, 0x5a, 0xfe, 0xac, 0x74, 0x8a};
  static const uint8_t MSG[5] = {'h', 'e', 'l', 'l', 'o'};
  static const char DST[] = "BLS_SIG_BLS12381G2_XMD:SHA-256_SSWU_RO_NUL_";
  auto fail = [&](const char* what) {
    ctx->err = std::string("self-test failed: ") + what + " (this build of libblsgpu.so computes wrong results; do not use it)";
    return BLSGPU_E_CUDA;
  };
  uint8_t out[96];
  for (int variant = 0; variant < 2; variant++) {
    CKR(blsgpu_fp_mul_batch(ctx, variant, 1, FA, FB, out));
    if (memcmp(out, FAB, 48) != 0) return fail("field multiplication");
  }
  const uint64_t off1[2] = {0, 5};
  CKR(blsgpu_hash_to_curve_batch(ctx, 2, 1, MSG, off1, reinterpret_cast<const uint8_t*>(DST), sizeof(DST) - 1, out));
  if (memcmp(out, HHELLO, 96) != 0) return fail("hash_to_curve");
  uint8_t pks[96], sigs[192], msgs[10], st[2] = {9, 9};
  memcpy(pks, PK1, 48); memcpy(pks + 48, PK1, 48);
  memcpy(sigs, SIG1, 96); memcpy(sigs + 96, SIG2, 96);
  memcpy(msgs, MSG, 5); memcpy(msgs + 5, MSG, 5);
  const uint64_t off2[3] = {0, 5, 10};
  CKR(blsgpu_verify_batch(ctx, 2, 0, 1, 2, pks, sigs, msgs, off2, st));
  if (st[0] != BLSGPU_ST_OK || st[1] != BLSGPU_ST_INVALID_SIGNATURE) return fail("signature verification (pairing, final exponentiation, bisection)");
  uint8_t gt[576], sum[96];
  int one = 0;
  CKR(blsgpu_miller_partial(ctx, 2, 0, 1, 1, PK1, SIG1, MSG, off1, gt, sum));
  CKR(blsgpu_final_exp_is_one(ctx, 2, 1, gt, sum, &one));
  CKR(blsgpu_partial_finish(ctx, one, st));
  if (!one || st[0] != BLSGPU_ST_OK) return fail("fold of partial results (byte conversions)");
  gt[100] ^= 1;
  CKR(blsgpu_final_exp_is_one(ctx, 2, 1, gt, sum, &one));
  if (one) return fail("fold of a tampered partial result");
  return BLSGPU_OK;
}

int blsgpu_plan_msm(size_t n, int scalar_bits, int* window_bits_out, int* windows_out, int* top_window_bits_out) {
  if (!window_bits_out || !windows_out || !top_window_bits_out || (scalar_bits != 64 && scalar_bits != 128)) return BLSGPU_E_ARG;
  const int c = msm_window_bits(n, scalar_bits), nwin = (scalar_bits + c - 1) / c;
  *window_bits_out = c;
  *windows_out = nwin;
  *top_window_bits_out = scalar_bits - (nwin - 1) * c;
  return BLSGPU_OK;
}

int blsgpu_plan_shards(size_t sets, const uint64_t* set_off, int ndev, uint64_t* cut_out) {
  if (!set_off || !cut_out || ndev < 1) return BLSGPU_E_ARG;
  for (size_t j = 0; j < sets; j++)
    if (set_off[j + 1] < set_off[j]) return BLSGPU_E_ARG;
  const std::vector<size_t> cut = balanced_cuts(sets, set_off, (size_t)ndev);
  for (int d = 0; d <= ndev; d++) cut_out[d] = cut[d];
  return BLSGPU_OK;
}
