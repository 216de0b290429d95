// Internal declarations shared by the translation units of libfrg.so (not part of the ABI).
#pragma once

#include <cuda_runtime.h>
#include <cuda_bf16.h>
#include <stdint.h>

#include <cmath>

#include <map>
#include <mutex>
#include <string>
#include <unordered_map>
#include <vector>

#include "frg.h"

namespace frg {

constexpr int kWarp = 32;
constexpr float kNoScore = -1.0f;   // the scan's initial best_score (infrenceServer.py:536)
constexpr int32_t kNoRow = -1;

// ---- error plumbing -----------------------------------------------------------------------
void set_error(const char* fmt, ...);
int cuda_fail(cudaError_t e, const char* what, const char* file, int line);

#define FRG_CUDA(call)                                                        \
  do {                                                                        \
    cudaError_t e__ = (call);                                                 \
    if (e__ != cudaSuccess) return ::frg::cuda_fail(e__, #call, __FILE__, __LINE__); \
  } while (0)

#define FRG_CHECK(expr)                     \
  do {                                      \
    int rc__ = (expr);                      \
    if (rc__ != FRG_OK) return rc__;        \
  } while (0)

void note_launch(const char* variant_or_null);   // launch accounting for frg_last_launch_count()
void reset_launches();
// bench-only timing of the dominant kernel(s): bracket them with profile_begin/profile_end
enum ProfileStage { kStagePrep = 0, kStagePrepass = 1, kStageFloor = 2, kStageDominant = 3, kStageSelect = 4,
                    kStageFallback = 5 };
void profile_begin(cudaStream_t st, int stage = kStageDominant);
void profile_end(cudaStream_t st, int launches);

// ---- programmatic dependent launch (PDL) ------------------------------------------------------
// The kernels of one match run back to back on one stream.  A kernel launched with the programmatic-
// serialization attribute may be SCHEDULED while its predecessor is still running (once every CTA of the
// predecessor has called pdl_trigger() or exited): its launch latency and prologue (barrier init, TMEM
// allocation, descriptor prefetch) overlap the predecessor's tail.  pdl_wait() then blocks until the
// predecessor has completed and its writes are visible - it precedes every read of earlier results.
// Without the attribute both calls are no-ops.
#ifdef __CUDACC__
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
__device__ __forceinline__ void pdl_trigger() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }
#endif
#ifdef __CUDACC__
// order-preserving float <-> uint32 key (a < b  <=>  key(a) < key(b) for non-NaN floats): lets atomicMax fold float
// maxima and redux.sync find a warp's best score in one instruction
__device__ __forceinline__ uint32_t float_key(float x) {
  const uint32_t b = __float_as_uint(x);
  return (b & 0x80000000u) ? ~b : (b | 0x80000000u);
}
__device__ __forceinline__ float key_float(uint32_t k) {
  return __uint_as_float((k & 0x80000000u) ? (k & 0x7fffffffu) : ~k);
}
// (float_key(-1.0f) == 0x407FFFFF: the value normalise_queries_kernel resets the group keys to)

// Lane of the warp's best (score desc, row asc, lane asc) entry.  One REDUX over the ordered keys and a ballot; only
// when several lanes hold exactly the best score (exact ties; exhausted lists, where every lane holds the sentinel)
// does the (row, lane) butterfly run.  -0.0 and +0.0 compare equal, as in the float comparison.  No NaNs in `s`.
template <typename RowT>
__device__ __forceinline__ int warp_argbest(float s, RowT r, RowT none, int lane) {
  const uint32_t key = float_key(s + 0.0f);
  const uint32_t mx = __reduce_max_sync(0xffffffffu, key);
  const unsigned tied = __ballot_sync(0xffffffffu, key == mx);
  if ((tied & (tied - 1u)) == 0u) return __ffs(tied) - 1;
  RowT br = key == mx ? r : none;
  int bl = key == mx ? lane : 64;
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    const RowT orow = __shfl_xor_sync(0xffffffffu, br, o);
    const int ol = __shfl_xor_sync(0xffffffffu, bl, o);
    if (orow < br || (orow == br && ol < bl)) { br = orow; bl = ol; }
  }
  return bl;
}
#endif

template <typename... KArgs, typename... Args>
inline cudaError_t launch_kernel(void (*kern)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t st,
                                 Args&&... args) {
  cudaLaunchConfig_t cfg{};
  cfg.gridDim = grid; cfg.blockDim = block; cfg.dynamicSmemBytes = smem; cfg.stream = st;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  return cudaLaunchKernelEx(&cfg, kern, static_cast<KArgs>(args)...);
}

// Function attributes are sticky per (function, device): set them once per thread and device instead of in front
// of every launch (a handful of driver calls per match otherwise).
template <typename F>
inline cudaError_t func_attr_once(F* kern, cudaFuncAttribute attr, int value) {
  struct Key { const void* f; int dev, attr, value; };
  static thread_local std::vector<Key> done;
  int dev = 0;
  cudaError_t e = cudaGetDevice(&dev);
  if (e != cudaSuccess) return e;
  const void* f = reinterpret_cast<const void*>(kern);
  for (const Key& k : done)
    if (k.f == f && k.dev == dev && k.attr == int(attr) && k.value == value) return cudaSuccess;
  e = cudaFuncSetAttribute(kern, attr, value);
  if (e == cudaSuccess) done.push_back(Key{f, dev, int(attr), value});
  return e;
}

// Pieces of one workspace allocation: take(bytes) returns the 256-byte aligned offset of the next piece; `off` is the
// end of the last piece, the bytes to allocate.
struct Carve {
  size_t off = 0;
  size_t take(size_t bytes) { const size_t o = (off + 255) & ~size_t(255); off = o + bytes; return o; }
};

struct DeviceInfo {
  int sm_count = 0;
  int cc_major = 0, cc_minor = 0;
  size_t smem_optin = 0;
};
int device_info(int device, DeviceInfo* out);

// RAII device switch
struct DeviceGuard {
  int prev = -1;
  bool ok = true;
  explicit DeviceGuard(int dev) {
    if (cudaGetDevice(&prev) != cudaSuccess) { ok = false; return; }
    if (prev != dev && cudaSetDevice(dev) != cudaSuccess) ok = false;
  }
  ~DeviceGuard() { if (prev >= 0) cudaSetDevice(prev); }
};

}  // namespace frg

// ---- the store ------------------------------------------------------------------------------
struct frg_store {
  int device = 0;
  int dim = 0;
  uint32_t flags = 0;
  int64_t capacity = 0;
  int64_t rows = 0;       // next append position
  int64_t live = 0;       // maintained on the host from upsert/remove arguments when possible (-1 = unknown)
  int64_t version = 0;
  bool maybe_dead = false;            // a row was tombstoned since the last compaction (or tag -1 was upserted)
  float* master = nullptr;            // [capacity][dim] fp32, unit rows
  __nv_bfloat16* plane = nullptr;     // [capacity][plane_dim] bf16 image (scan plane of raw and bf16-only stores) or null
  // Unit-row store with FRG_STORE_BF16_PLANE: the scan plane is int8 instead, [capacity][dim], element =
  // clamp(rint(g / i8_gallery_step(dim)), -127, 127) (plane stays null).  gmax_bits[1] holds its largest residual.
  int8_t* plane8 = nullptr;
  // plane_dim == dim for unit-row stores.  A FRG_STORE_RAW store's plane is the EUCLIDEAN scan plane:
  // plane_dim = dim + kEuclidPad (16): columns dim..dim+2 hold -0.5*||g||^2 split exactly into three bf16 terms,
  // columns dim+3..dim+5 the row's error-bound terms ||g - bf16(g)||, ||g||, ||g||^2 rounded up (the rest 0), so that
  // Qaug . Gaug = q.g - 0.5*||g||^2 +- bound with Qaug = [q, 1, 1, 1, +-A, +-B, +-C, 0...] (queries.cu, tc_match.cu)
  int plane_dim = 0;
  uint32_t* gmax_bits = nullptr;      // device uint32[2], float bits: [0] max ||g||^2 ever ingested (raw stores with a
                                      // Euclidean plane), [1] max ||g - g^||^2 (any store with a plane; g^ = the
                                      // row's bf16 image, or its int8 image times the store's step)
  int32_t* tags = nullptr;            // [capacity]
  // Fault word in pinned, device-mapped host memory: a kernel whose TMA / MMA pipeline barrier timed out sets it
  // instead of trapping (a trap would kill the CUDA context of the whole service).  Sticky; reported by
  // frg_store_stats (faults) and by every *_host call as FRG_ERR_CUDA.
  uint32_t* fault_host = nullptr;
  uint32_t* fault_dev = nullptr;
  std::mutex mu;                      // guards the fields above and the stream bookkeeping
  cudaEvent_t last_write = nullptr;   // recorded after every mutation
  bool has_write = false;
  std::vector<cudaStream_t> readers;  // streams that matched since the last mutation
  // Row extent [lo, hi) every tenant tag can sit in (a superset: never shrunk by removals, rebuilt exactly by
  // compact()).  A tenant-filtered match scans only that window: infrenceServer.py:343-380 filters EVERY frame
  // by company, and a company's people are typically enrolled as one contiguous block.  Known only while every
  // mutation carried its tags / rows in host memory (the *_host entry points, fill_synthetic).
  struct Extent { int64_t lo, hi; };
  std::unordered_map<int32_t, Extent> extents;
  bool extents_known = true;
  // ... and, finer, the disjoint row intervals [lo, hi) of every tag (same provenance, same superset rule).  When
  // a tenant's window is mostly other tenants' rows - one person re-enrolled at the end of the gallery stretches it
  // over everything - the tensor-core kernels walk only the TILES these intervals touch (tile list, cached per
  // store version and tile size).  A tag with more than kMaxSpans intervals (interleaved companies) is "scattered":
  // no list, the masked scan of the window as before.
  static constexpr size_t kMaxSpans = 4096;
  struct Spans { std::map<int64_t, int64_t> iv; int64_t covered = 0; bool scattered = false; };
  std::unordered_map<int32_t, Spans> spans;
  struct TileList { int64_t version = -1; int32_t* dev = nullptr; int64_t cap = 0; int n = 0; bool use = false;
                    cudaEvent_t ready = nullptr; };
  std::map<std::pair<int32_t, int>, TileList> tile_lists;       // (tenant, rows per tile)
  std::vector<void*> retired;                                   // outgrown list buffers, freed with the store
};

namespace frg {
// Dequantisation step of a unit store's int8 scan plane, fixed per dim: alpha / 127 with alpha = 0.165 * sqrt(512 /
// dim), i.e. 3.73 standard deviations of an element of a random unit vector.  At dim 512 alpha = 0.165 sits just above
// the largest element of the synthetic gallery (0.161; its row maxima: median 0.125, 99.9th percentile 0.149), so
// ordinary rows never saturate; a row that does is clamped to +-127 and its larger residual is measured like any
// other (gmax_bits[1]), so the filter's bound stays rigorous.
inline float i8_gallery_step(int dim) { return float(0.165 * std::sqrt(512.0 / double(dim)) / 127.0); }
// What the match kernels see of a store: the whole gallery, or the row window of one tenant.
struct GalleryWindow {
  const float* master = nullptr;
  const __nv_bfloat16* plane = nullptr;
  const int8_t* plane8 = nullptr;
  const int32_t* tags = nullptr;
  uint32_t* gmax_bits = nullptr;
  uint32_t* fault = nullptr;          // frg_store::fault_dev
  int64_t rows = 0;       // rows in the window
  int64_t row0 = 0;       // store row of the window's first row (added to every returned row)
  int dim = 0, plane_dim = 0;
  uint32_t flags = 0;
  bool maybe_dead = false;
  // tenant-filtered call over a window that is mostly other tenants' rows: the tensor-core kernels may ask the
  // store for the tenant's tile list (store_tile_list; the caller holds owner->mu)
  frg_store* owner = nullptr;
  bool want_tile_list = false;
  int32_t list_tenant = -1;
};
}  // namespace frg

namespace frg {

// order a mutation on `stream` after every match enqueued so far; call with s->mu held
int store_begin_write(frg_store* s, cudaStream_t stream);
int store_end_write(frg_store* s, cudaStream_t stream);
// order a match on `stream` after the last mutation; call with s->mu held
int store_begin_read(frg_store* s, cudaStream_t stream);

// api.cu: device-resident list of the tiles (`gran` rows each, absolute tile indices, ascending) that hold rows of
// `tenant`, rebuilt when the store's version changed; *list == nullptr: not worth it.  s->mu held; the list is
// valid for work enqueued on `st` after the call.
int store_tile_list(frg_store* s, int32_t tenant, int gran, cudaStream_t st, const int32_t** list, int* n);
// tc_match.cu
int64_t tc_effective_rows(const GalleryWindow* s, int nq, cudaStream_t st, const int32_t** list, int* n_list);

// ---- kernels' host launchers (defined in the .cu named in the comment) ----------------------
// queries.cu: qn[f] = q[f] / ||q[f]|| (fp32), optional bf16 image
// eps / bounds (tensor-core variants): eps[f] = rigorous bound of |bf16 filter score - fp32 score| for query f
// against ANY row of the store, from the measured rounding residual of the query and bounds[1], the largest
// residual of a stored row (store_kernels.cu)
int launch_normalise_queries(const float* q, int nq, int dim, bool normalise, float* qn,
                             __nv_bfloat16* qn_bf16, uint32_t* group_keys, int* cand_total, int* n_flagged,
                             cudaStream_t st, float* eps = nullptr, const uint32_t* bounds = nullptr);
// queries.cu: the int8 filter's prep (unit store with an int8 plane): qn = unit fp32 queries, qi8 = int8 image
// rint(qn / c_q) with c_q = max|qn| / 127, qstep[f] = c_q * i8_gallery_step(dim) (S = integer product * qstep),
// eps[f] = rigorous bound of |S - fp32 score| against any row of the store (bounds[1]: the rows' largest residual).
// Resets the 64-bit group keys of the pre-pass (group_keys: [nq][32] uint64) and the counters.
int launch_prepare_queries_i8(const float* q, int nq, int dim, float* qn, int8_t* qi8, float* qstep, float* eps,
                              const uint32_t* bounds, unsigned long long* group_keys, int* cand_total, int* n_flagged,
                              cudaStream_t st);
// queries.cu: Euclidean tensor-core prep: qn = q as given, bf16 image [nq][dim + kEuclidQPad] = [q, 1, 1, 1, 0...],
// eps[f] = filter error bound of query f from ||q|| and the store's max row norm
// q_aug: the filter's image [q, 1, 1, 1, +A, +B, +C, 0...], q_aug_lo: the pre-pass image (-A, -B, -C); coef[f][4] = the
// bf16 coefficient values A, B, C of query f (select recomputes a candidate's bound from them); eps[f] = 0
int launch_prepare_queries_euclid(const float* q, int nq, int dim, const uint32_t* gmax_bits, float* qn,
                                  __nv_bfloat16* q_aug, __nv_bfloat16* q_aug_lo, float* coef, float* eps,
                                  uint32_t* group_keys, int* cand_total, int* n_flagged, cudaStream_t st);

struct XPush;      // exchange.cu, below
// scan_f32.cu: exact scan; writes nq x k best (score desc, row asc) into rows32/scores
struct ScanArgs {
  const float* master; const __nv_bfloat16* plane = nullptr;   // master == nullptr: bf16-only store, scan the plane
  const int32_t* tags; int64_t rows; int dim;
  const float* qn; int nq; int k; int metric; int32_t tenant;
  int sm_count;
};
int scan_f32_workspace_bytes(const ScanArgs& a, size_t* bytes);
int launch_scan_f32(const ScanArgs& a, void* workspace, int64_t row_offset, float threshold,
                    int64_t* out_rows, float* out_scores, uint8_t* out_accept, cudaStream_t st);

// scan_f32.cu: exact re-do of the queries listed on the device (tensor-core candidate overflow)
// push: row-sharded gallery - the last CTA sends every redone query's final top-k to all ranks
int launch_scan_f32_flagged(const ScanArgs& a, const int* flagged, int* n_flagged_and_ticket, int64_t row_offset,
                            float threshold, const XPush& push, int64_t* out_rows, float* out_scores,
                            uint8_t* out_accept, cudaStream_t st);

// merge.cu: generic k-way merge of sorted partial lists
int launch_merge_i64(const float* scores, const int64_t* rows, int parts, int nq, int k_in, int k_out,
                     int metric, float threshold, int64_t row_offset, bool finalize_euclid,
                     int64_t* out_rows, float* out_scores, uint8_t* out_accept, cudaStream_t st);
int launch_merge_i64_strided(const float* scores, int64_t score_stride, const int64_t* rows, int64_t row_stride,
                             int parts, int nq, int k, int metric, float threshold, int64_t* out_rows,
                             float* out_scores, uint8_t* out_accept, cudaStream_t st);
int launch_merge_i32(const float* scores, const int32_t* rows, int parts, int nq, int k_in, int k_out,
                     int metric, float threshold, int64_t row_offset, bool finalize_euclid,
                     int64_t* out_rows, float* out_scores, uint8_t* out_accept, cudaStream_t st);

// exchange.cu: multi-GPU tail over NVLink peer memory.  XPush describes where this rank's results go:
// into slot `rank` of every rank's exchange buffer, as 8-byte {payload, epoch} packets.
// Buffer layout: [header kExchangeHeader][parity 0: world blocks][parity 1: world blocks]; the header holds
//   [0, 512)    hello packets [parity][source rank]: {(nq << 5) | k, epoch} - what the source believes this
//               call is; a rank that polls first checks them, so a call-count or shape mismatch between ranks
//               is REPORTED (status record) instead of waited on
//   [512, 576)  status record of this rank's own poll kernel (XStatus), read by frg_exchange_status
constexpr int kExchangeHeader = 1024;
constexpr int kExchangeMaxWorld = 32;
constexpr int kExchangeStatusOff = 512;
enum XCode : uint32_t { kXOk = 0, kXHelloTimeout = 1, kXHelloMismatch = 2, kXDataTimeout = 3 };
struct XStatus { uint32_t code, peer, epoch, seen_epoch, want_hello, seen_hello, query, pad; };
struct XPush {
  unsigned char* const* peer_bufs = nullptr;   // DEVICE array of `world` peer-mapped buffer pointers; null = no exchange
  int rank = 0, world = 1;
  uint32_t epoch = 0;                          // 1, 2, 3, ... one more per collective call; never 0
  uint32_t hello = 0;                          // (nq << 5) | k
  int64_t block_cap = 0;                       // bytes per (parity, source rank) block >= nslots * 24
  int64_t nslots = 0;                          // nq * k
  unsigned long long timeout_ns = 0;           // bound of the poll kernel's wait for a peer
};
#ifdef __CUDACC__
__device__ __forceinline__ void xpush_slot(const XPush& x, int peer, int64_t slot, int64_t row, float score) {
  uint2* b = reinterpret_cast<uint2*>(x.peer_bufs[peer] + kExchangeHeader +
                                      (size_t(x.epoch & 1u) * x.world + x.rank) * size_t(x.block_cap));
  const uint64_t r = uint64_t(row);
  asm volatile("st.relaxed.sys.global.v2.u32 [%0], {%1, %2};" ::"l"(b + slot), "r"(uint32_t(r)), "r"(x.epoch) : "memory");
  asm volatile("st.relaxed.sys.global.v2.u32 [%0], {%1, %2};" ::"l"(b + x.nslots + slot), "r"(uint32_t(r >> 32)), "r"(x.epoch) : "memory");
  asm volatile("st.relaxed.sys.global.v2.u32 [%0], {%1, %2};" ::"l"(b + 2 * x.nslots + slot), "r"(__float_as_uint(score)), "r"(x.epoch) : "memory");
}
// "rank x.rank is in call x.epoch with this (nq, k)" -> header of `peer`
__device__ __forceinline__ void xpush_hello(const XPush& x, int peer) {
  uint2* h = reinterpret_cast<uint2*>(x.peer_bufs[peer]) + (x.epoch & 1u) * kExchangeMaxWorld + x.rank;
  asm volatile("st.relaxed.sys.global.v2.u32 [%0], {%1, %2};" ::"l"(h), "r"(x.hello), "r"(x.epoch) : "memory");
}
#endif
// hello word, slot count and the poll bound (FRG_EXCHANGE_TIMEOUT_MS, default 2000) of a call
void exchange_fill_defaults(XPush* x, int nq, int k);
// push kernel: hello + the listed queries' (or all queries') local top-k to every rank.  Only needed where no
// earlier kernel of the match pushed (variants without a select stage; results computed elsewhere).
int launch_exchange_push(const XPush& x, const int64_t* local_rows, const float* local_scores, int nq, int k,
                         int sm_count, cudaStream_t st);
// poll kernel: waits (bounded) for every rank's packets of this call and merges them.  It never pushes: every
// local push was issued by an EARLIER kernel of the stream, so no CTA of it waits for a push that sits in a
// CTA which is not resident yet.
int launch_exchange_merge(const XPush& x, int nq, int k, int metric, float threshold, int sm_count,
                          int64_t* out_rows, float* out_scores, uint8_t* out_accept, cudaStream_t st);

// tc_match.cu: tcgen05 filter + exact rescoring.  Cosine: dim multiple of 64 and <= 512 (unit rows);
// Euclidean: dim 128 / 256 over a raw store's augmented plane (plane_dim = dim + kEuclidPad).
constexpr int kEuclidPad = 16;      // plane: one more 32-byte group of k (one UMMA K step) for the three bias columns
constexpr int kEuclidQPad = 64;     // query image: padded to a whole 128-byte swizzle row (the tile's k-block)
constexpr float kEuclidNone = -3.0e38f;   // "no score yet" of the Euclidean filter (scores are unbounded below)
int tc_supported(int dim, int metric, const char** why);

// Candidate entries per query of a range-mode filter (range search and self-join; DESIGN.md section 7.3)
constexpr int kRangeBudget = 4096;

// The plan of one ungrouped tensor-core call over `rows` rows (the window's, or listed tiles x rows per tile): grid,
// pre-pass sample and the sizes of its workspace.  dim < 0: Euclidean plane of |dim| columns.  range: no pre-pass and
// kRangeBudget dense entries per query (range search); i8: the int8 filter of a unit store.
struct TcPlan {
  bool pair;              // CTA-pair kernels (F > 128)
  bool fused;             // pre-pass folded into the filter kernel (probe tile + published group maxima)
  int qtiles, stride, chunks_pre, chunks_main, kreg, seg;
  int stage_entries;      // the dense width: dense list entries per query
  int64_t cand_entries;   // candidate segment entries (int2): nq x chunks_main x (kEpiWarps / 4) x seg
};
void tc_plan(int64_t rows, int dim, int nq, int k, int sm_count, TcPlan* pl, bool range, bool i8);

// The workspace of the filter behind every tensor-core call of nq queries (top-k, range search, one self-join slab, a
// per-query-tenant batch).  The query prep resets keys, cand_total and n_flagged[0..2].
struct TcWs {
  unsigned long long* keys;   // [nq][32] group keys: uint64 (int8 filter), uint32 (bf16 and Euclidean filters)
  int* cand_total;            // [nq] candidates per query
  int* flagged;               // [nq] queries whose candidates overflowed, then their count, the fallback's ticket and
                              // the fused kernel's probe-arrival counter
  int* n_flagged;             // flagged + nq
  float* floor;               // [nq] per-query float floor of the int8 filter (null otherwise)
  int2* dense;                // [nq][dense_cap] packed candidates
  int2* cand;                 // the filter's candidate segments
  int dense_cap;
};
// Bytes of that workspace when the filter writes cand_entries segment entries (int2); with ws, its pieces in *out.
// i8: 64-bit group keys and the floor.
size_t tc_workspace(int nq, int64_t cand_entries, int dense_cap, bool i8, unsigned char* ws, TcWs* out);

// metric cosine, int8 plane (s->plane8): qi8 / qstep / eps from launch_prepare_queries_i8, qb unused.
// metric cosine, bf16 plane (bf16-only store): qb = [nq][dim] bf16 unit queries, eps[nq] per-query bounds.
// metric euclidean: qb = [nq][dim + kEuclidQPad] augmented image, eps[nq] per-query bounds.
// pl: tc_plan over the rows the call scans (tile_list: the listed tiles of a tenant-filtered call whose window is
// mostly other tenants' rows, tc_effective_rows); w: tc_workspace of pl, its keys and counters reset by the query prep.
// Queries whose candidates overflowed are left in (w.flagged, w.n_flagged) for launch_scan_f32_flagged.
// push: the select stage sends every query's final top-k straight to all ranks (XPush::peer_bufs != null)
int launch_tc_match(const GalleryWindow* s, int metric, const float* qn, const __nv_bfloat16* qb, const float* eps,
                    int nq, int k, int32_t tenant, bool rescore, float threshold, int64_t row_offset,
                    const TcPlan& pl, const TcWs& w, int sm_count, const XPush& push, int64_t* out_rows,
                    float* out_scores, uint8_t* out_accept, cudaStream_t st, const int32_t* tile_list, int n_list,
                    const __nv_bfloat16* qb_prepass = nullptr, const float* coef = nullptr,
                    const int8_t* qi8 = nullptr, const float* qstep = nullptr);

// ---- the GROUPED int8 filter grid (per-query tenants, self-join).  A query tile holds queries q0 .. q0 + nq - 1
// (nq <= kTcTileRows) of one tenant (the filter masks with it; -1 = none), which scan the absolute kTcTileRows-row
// tiles list[0 .. n_tiles) or tile0 .. tile0 + n_tiles - 1 (a masked range).
constexpr int kTcTileRows = 128;
struct TcTenantGroup { int32_t tenant; int q0, nq; int tile0, n_tiles; const int32_t* list; };
// tc_match.cu, host: the grid's CTA descriptors over the query tiles.  k >= 1 (top-k): each tile takes the pre-pass
// stride and candidate budget of a single-tenant tc_plan over its tiles, and the grid has a pre-pass; k = 0 (range
// search, self-join): kRangeBudget candidates per query, no pre-pass.
struct TcGroupPlan {
  std::vector<unsigned char> ctas;    // [n_pre pre-pass descriptors][n_main filter descriptors]
  int n_pre = 0, n_main = 0;
  int64_t cand_entries = 0;           // candidate segment entries (int2) the filter grid writes
  int dense_cap = 0;                  // dense list entries per query
};
void tc_group_plan(const std::vector<TcTenantGroup>& tiles, int k, int dim, int sm_count, TcGroupPlan* out);
// tc_match.cu: out[i] = q[perm[i]] (rows of dim floats)
int launch_gather_queries(const float* q, const int32_t* perm, int nq, int dim, float* out, cudaStream_t st);
// tc_match.cu: out[perm[i]] = sorted result i: rows / scores [nq][width] and field[nq] (F = uint8_t: top-k's accept,
// out_field may be null; F = int64_t: range search's counts)
template <typename F>
int launch_scatter_sorted(const int64_t* rows, const float* scores, const F* field, const int32_t* perm, int nq,
                          int width, int64_t* out_rows, float* out_scores, F* out_field, cudaStream_t st);
// scan_f32.cu: the exact re-do of launch_scan_f32_flagged, each flagged query q with its own tenant q_tenant[q]
// (device array; cosine, fp32 master, a.tenant ignored)
int launch_scan_f32_flagged_tenants(const ScanArgs& a, const int32_t* q_tenant, const int* flagged,
                                    int* n_flagged_and_ticket, int64_t row_offset, float threshold, int64_t* out_rows,
                                    float* out_scores, uint8_t* out_accept, cudaStream_t st);
// api.cu: host -> device copy through the per-thread pinned staging ring (pageable copy when larger than a slot)
int stage_upload(void* dev, const void* host, size_t bytes, cudaStream_t st);

// tc_match.cu: top-k with a tenant per query (frg_match_tenants) on the int8 filter of a unit cosine store, over the
// tenant-sorted batch: qn / qi8 / qstep / eps from launch_prepare_queries_i8 (which reset w's keys and counters),
// d_ctas the uploaded descriptors of tc_group_plan (k >= 1; n_pre pre-pass, then n_main filter).  Pre-pass, floor,
// filter and select-rescore into out_* (sorted order); queries whose candidates overflowed are left in (w.flagged,
// w.n_flagged) for launch_scan_f32_flagged_tenants.  s: the whole store.
int launch_tc_match_grouped(const GalleryWindow* s, const float* qn, const int8_t* qi8, const float* qstep,
                            const float* eps, int nq, const void* d_ctas, int n_pre, int n_main, int k, float threshold,
                            int64_t row_offset, const TcWs& w, int64_t* out_rows, float* out_scores,
                            uint8_t* out_accept, cudaStream_t st);

// tc_match.cu: range search over a unit cosine store (frg_match_range).  The filter keeps every row with
// S >= threshold - eps[q] (no pre-pass); range_select_kernel rescores each candidate exactly, keeps those that pass
// (score >= threshold, '>' when strict), writes the first max_hits in gallery order and the count.  pl: tc_plan in
// range mode over the rows scanned (tile_list as in launch_tc_match); w: tc_workspace of pl.  Queries whose
// candidates overflowed the plan are left in (w.flagged, w.n_flagged) for launch_range_scan's flagged mode.
int launch_tc_range(const GalleryWindow* s, const float* qn, const int8_t* qi8, const float* qstep, const float* eps,
                    int nq, int max_hits, int32_t tenant, float threshold, bool strict, int64_t row_offset,
                    const TcPlan& pl, const TcWs& w, int64_t* out_counts, int64_t* out_rows, float* out_scores,
                    cudaStream_t st, const int32_t* tile_list, int n_list);

// scan_f32.cu: exact, counting range scan.  Pass 1: every warp owns a contiguous row range and counts its hits per
// query; a per-query exclusive scan over the warp counts gives the total and each warp's output offset; pass 2: the
// warps whose offset is below max_hits recompute and write their hits in row order.  flagged == nullptr: all nq
// queries; else only the n_flagged[0] listed ones (device-side count, the tensor-core path's overflow fallback).
int range_scan_supported(int dim, const char** why);
int launch_range_scan(const ScanArgs& a, const int* flagged, const int* n_flagged, int max_hits, float threshold,
                      bool strict, int64_t row_offset, int64_t* out_counts, int64_t* out_rows, float* out_scores,
                      cudaStream_t st);

// ---- range search with a tenant per query (frg_match_range_tenants): the batch is sorted by tenant; sorted query q
// has its tenant q_tenant[q] (-1 = all) and its row window [q_lo[q], q_hi[q]) (device arrays; rows < 2^31).
// scan_f32.cu: launch_range_scan's passes with that tenant and window per query.  a: the whole store, a.qn / a.nq the
// sorted queries (unit for cosine), a.tenant ignored.  flagged == nullptr: every query; else the n_flagged[0] listed ones.
int launch_range_tenants_scan(const ScanArgs& a, const int32_t* q_tenant, const int32_t* q_lo, const int32_t* q_hi,
                              const int* flagged, const int* n_flagged, int max_hits, float threshold, bool strict,
                              int64_t row_offset, int64_t* out_counts, int64_t* out_rows, float* out_scores,
                              cudaStream_t st);
// tc_match.cu: launch_tc_range's path with the GROUPED filter over the uploaded descriptors (d_table, n_ctas from
// tc_group_plan in range mode; none when 0).  Queries whose candidates overflowed are left in (w.flagged, w.n_flagged)
// for launch_range_tenants_scan.  s: the whole store.
int launch_tc_range_grouped(const GalleryWindow* s, const float* qn, const int8_t* qi8, const float* qstep,
                            const float* eps, int nq, const void* d_table, int n_ctas, int max_hits, float threshold,
                            bool strict, int64_t row_offset, const TcWs& w, int64_t* out_counts,
                            int64_t* out_rows, float* out_scores, cudaStream_t st);

// ---- gallery self-join (frg_self_join): the queries are the store's own rows qrow0 .. qrow0 + nq - 1 of one slab,
// and a pair (a, b) counts only for b > a (plus the tag rule: tenant >= 0 -> both rows carry it; same_tag -> tag[b] ==
// tag[a]).  Query tile u of the slab holds queries 128u .. 128u + 127.
// tc_match.cu: the int8 filter path of one slab, launch_tc_range's with the GROUPED filter over the uploaded
// descriptors (d_table, n_ctas from tc_group_plan in range mode; none when 0) and join_select_kernel (exact rescoring, b > a, tag rule, counts and the first
// max_hits hits in gallery order).  Queries whose candidates overflowed are left in (w.flagged, w.n_flagged) for
// launch_join_scan.  s: the whole store.
int launch_tc_join(const GalleryWindow* s, const float* qn, const int8_t* qi8, const float* qstep, const float* eps,
                   int nq, const void* d_table, int n_ctas, int64_t qrow0, int32_t tenant, bool same_tag,
                   float threshold, bool strict, int max_hits, int64_t row_offset, const TcWs& w,
                   int64_t* out_counts, int64_t* out_rows, float* out_scores, cudaStream_t st);
// scan_f32.cu: exact, counting join scan (launch_range_scan's passes with the join rules).  a: the whole store, a.qn /
// a.nq the slab's unit queries, a.tenant the tenant rule, cosine.  tile_end[u]: exclusive end row of query tile u's
// plan (device).  A pass of queries reads only the rows from its lowest live query row + 1 to its largest end.
// flagged == nullptr: every query of the slab; else only the n_flagged[0] listed ones.  ws: join_scan_workspace_bytes.
size_t join_scan_workspace_bytes(const ScanArgs& a);
int launch_join_scan(const ScanArgs& a, int64_t qrow0, const int32_t* tile_end, bool same_tag, const int* flagged,
                     const int* n_flagged, int max_hits, float threshold, bool strict, int64_t row_offset, void* ws,
                     int64_t* out_counts, int64_t* out_rows, float* out_scores, cudaStream_t st);

// scan_f32.cu: frg_cluster_observe_host's device work.  a: the store's first a.rows rows (the clusters before the call),
// a.qn / a.nq the faces as given, a.tenant the call's filter.  Pre-pass: launch_range_scan of every face against those
// rows (hit budget kClusterHits); then ONE CTA resolves the faces in order, writing the means to master, the tags of the
// new rows (new_tag) and the ring, and out_cluster / out_created (device).  master / tags: the store's, with room for
// a.rows + a.nq rows.
constexpr int kClusterHits = 16;
int launch_cluster_observe(const ScanArgs& a, float* master, int32_t* tags, float threshold, bool strict,
                           int32_t new_tag, const frg_cluster_ring_t& ring, int64_t* out_cluster, uint8_t* out_created,
                           cudaStream_t st);

// first_match.cu
int launch_first_match(const float* master, const int32_t* tags, int64_t rows, int dim, const float* qn, int nq,
                       int32_t tenant, float threshold, bool strict, int64_t row_offset, unsigned long long* scratch,
                       int sm_count, int64_t* out_rows, float* out_scores, cudaStream_t st);

// store_kernels.cu
// plane_dim > dim: Euclidean scan plane (bias columns written, gmax_bits folded); else plane_dim == dim
// plane8: the int8 scan plane of a unit store (written instead of plane, residual folded into gmax_bits[1])
int launch_ingest(const float* vecs, const int64_t* rows, const int32_t* tags, int64_t n, int64_t append_at,
                  int dim, bool normalise, float* master, __nv_bfloat16* plane, int8_t* plane8, int plane_dim,
                  uint32_t* gmax_bits, int32_t* tag_out, cudaStream_t st);
int launch_tombstone(const int64_t* rows, int64_t n, int64_t limit, int32_t* tags, cudaStream_t st);
int launch_synth(int64_t n, int64_t append_at, int64_t global_row0, uint64_t seed, int32_t tag, int dim,
                 float* master, __nv_bfloat16* plane, int8_t* plane8, int plane_dim, uint32_t* gmax_bits,
                 int32_t* tag_out, cudaStream_t st);
// plane_row_bytes: bytes of a scan-plane row (multiple of 8), 0 = no plane
int launch_gather_rows(const int64_t* src_rows, int64_t n, int dim, int plane_row_bytes, const float* master_in,
                       const void* plane_in, const int32_t* tags_in, float* master_out, void* plane_out,
                       int32_t* tags_out, cudaStream_t st);

}  // namespace frg
