// Tensor-core variants (FRG_VARIANT_TC_EXACT / FRG_VARIANT_TC_BF16): the query x gallery contraction
// on tcgen05 with the threshold / top-k in the epilogue, so no score matrix reaches HBM.  Which store runs which filter:
//   - a unit cosine store with an fp32 master: the int8 filter (I8; pre-pass, i8_floor_kernel, filter, select);
//   - the Euclidean plane of a raw store and a bf16-only store: the bf16 filter described below;
//   - a bf16-only store matched with nq <= 8 queries: the bf16 filter with the pre-pass folded in (MODE = FUSED);
//   - per-query tenants on a unit cosine store (frg_match_tenants): the int8 pre-pass and filter in their GROUPED
//     single-CTA form, every CTA one (query tile of one tenant, chunk of that tenant's tiles) of a host-built table.
//
//   S[q, r] = sum_k Qb[q, k] * Gb[r, k]        Qb, Gb = bf16 images of the unit fp32 vectors
//
// The bf16 product is only a FILTER.  |S - s| <= eps[q], a rigorous, data-dependent bound from measured
// rounding residuals: |q^.g^ - q.g| <= ||q^|| ||g^ - g|| + ||q^ - q|| ||g||, the row side folded at ingest
// (largest residual of any stored row), the query side measured by the prep kernel (queries.cu); ~3.6e-3 for
// ordinary data, never above the a-priori 2u + u^2 = 7.8e-3 (u = 2^-8, bf16 round-to-nearest).  So every row
// of the true top-k has S >= tau - 2*eps, tau = k-th best coarse score.  Pipeline per batch:
//
//   1. pre-pass  (tc_scan_kernel<GROUPMAX>) over every stride-th 128-row tile of the scan plane:
//      per query, the running maximum of each of 32 disjoint row groups (row mod 32), folded across
//      CTAs with atomicMax on order-preserving keys.  The k-th largest of those 32 maxima (derived by
//      every FILTER thread in its prologue) is attained by k distinct rows, hence L[q] <= tau.
//   2. filter    (tc_scan_kernel<FILTER>) over the whole plane: append every (row, S) with
//      S >= L[q] - 2*eps to the query's candidate list (a few hundred rows out of 10^6).
//   3. select + rescore (select_rescore_kernel): tau from the candidates, keep S >= tau - 2*eps,
//      recompute those few scores EXACTLY in fp32 from the master rows (same arithmetic as the
//      streaming scan), order by (score desc, row asc), apply the threshold.
//   4. queries whose lists overflowed (adversarial duplicates, sparse tenants) are re-done by the
//      exact streaming scan inside the same enqueue (scan_f32_flagged_kernel) - never by the host.
//   For a handful of queries on a bf16-only store (nq <= 8) steps 1 and 2 run as ONE kernel (MODE = FUSED: every
//   CTA probes its first tile, publishes the group maxima, derives the floor, filters, re-visits the probe tile).
//
// Kernel anatomy (one CTA per SM, 320 threads):
//   warp 0   TMA producer: gallery tiles [128 rows x 64 k] bf16, 128B-swizzled, 6-stage mbarrier ring
//   warp 1   MMA issuer: one elected lane, tcgen05.mma cta_group::1 kind::f16, M=128 (queries) x N=128
//            (gallery rows) x K=16, A = the query tile resident in smem (128 x 512 bf16 = 128 KB),
//            B = the staged gallery tile; accumulators in TMEM, double buffered (2 x 128 columns)
//   warps 2-9 epilogue (two per TMEM lane quarter, splitting the columns): tcgen05.ld 32 lanes x 32
//            columns, software-pipelined; thread = one query, columns = gallery rows:
//            a running max against the query's threshold (1 FMNMX per score), rare slow path.
// The gallery is read once per 128-query tile: algorithmic bytes = rows * dim * 2 per launch and
// query tile; flops = 2 * 128 * rows * dim.
#include <cuda.h>

#include <cmath>
#include <cstring>

#include "frg_internal.cuh"

namespace frg {

// ------------------------------------------------------------------------------------------ PTX
__device__ __forceinline__ uint32_t smem_u32(const void* p) {
  return static_cast<uint32_t>(__cvta_generic_to_shared(p));
}

__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint32_t bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint32_t bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint32_t bar, uint32_t parity) {
  uint32_t ok;
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t}"
      : "=r"(ok) : "r"(bar), "r"(parity) : "memory");
  return ok != 0;
}
// A broken pipeline must neither hang the GPU nor kill the CUDA context of a long-running service (a trap
// would): bounded spin, then the CTA's abort flag is raised.  Every role loop leaves at its next iteration, the
// CTA tears down normally, the store's fault word is set (frg_store_stats / the *_host calls report it as a
// status code) and the results of that call are void.
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity, volatile int* abort_flag) {
  uint32_t spins = 0;
  while (!mbar_try_wait(bar, parity)) {
    if ((++spins & 1023u) == 0u) {
      if (*abort_flag) return;
      if (spins > (1u << 24)) { *abort_flag = 1; return; }
    }
  }
}
// one lane of a converged warp (PTX elect.sync): lets the rest of the warp stay on the uniform datapath
__device__ __forceinline__ bool elect_one() {
  uint32_t pred;
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "elect.sync _|p, 0xffffffff;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t}"
      : "=r"(pred));
  return pred != 0;
}
__device__ __forceinline__ void fence_barrier_init() {
  asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void fence_proxy_async() {
  asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
}

constexpr uint64_t kEvictFirst = 0x12F0000000000000ull;
constexpr uint64_t kEvictLast = 0x14F0000000000000ull;

__device__ __forceinline__ void tma_load_2d(uint32_t dst, const CUtensorMap* map, uint32_t bar, int c0, int c1,
                                            uint64_t hint) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint"
      " [%0], [%1, {%3, %4}], [%2], %5;"
      ::"r"(dst), "l"(reinterpret_cast<uint64_t>(map)), "r"(bar), "r"(c0), "r"(c1), "l"(hint)
      : "memory");
}
// CTA-pair (cta_group::2) flavours: both CTAs of the pair issue their half of the load, the
// transaction bytes land on the LEADER's mbarrier (peer bit of the shared::cluster address cleared)
__device__ __forceinline__ void tma_load_2d_pair(uint32_t dst, const CUtensorMap* map, uint32_t bar, int c0, int c1,
                                                 uint64_t hint) {
  asm volatile(
      "cp.async.bulk.tensor.2d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint"
      " [%0], [%1, {%3, %4}], [%2], %5;"
      ::"r"(dst), "l"(reinterpret_cast<uint64_t>(map)), "r"(bar & 0xFEFFFFFFu), "r"(c0), "r"(c1), "l"(hint)
      : "memory");
}
__device__ __forceinline__ uint32_t cluster_ctarank() {
  uint32_t r;
  asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
  return r;
}
__device__ __forceinline__ void cluster_sync_all() {
  asm volatile("barrier.cluster.arrive.release.aligned;\n\tbarrier.cluster.wait.acquire.aligned;" ::: "memory");
}
// arrive on the same-offset mbarrier of CTA `cta` of the cluster
__device__ __forceinline__ void mbar_arrive_remote(uint32_t bar, uint32_t cta) {
  asm volatile(
      "{\n\t.reg .b32 r;\n\t"
      "mapa.shared::cluster.u32 r, %0, %1;\n\t"
      "mbarrier.arrive.shared::cluster.b64 _, [r];\n\t}"
      ::"r"(bar), "r"(cta) : "memory");
}
__device__ __forceinline__ void tmem_alloc_pair(uint32_t dst_smem, uint32_t ncols) {
  asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(dst_smem), "r"(ncols) : "memory");
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc_pair(uint32_t taddr, uint32_t ncols) {
  asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}
__device__ __forceinline__ void umma_bf16_pair(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc,
                                               uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, p;\n\t}"
      ::"r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
      : "memory");
}
__device__ __forceinline__ void umma_i8_pair(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc,
                                             uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::2.kind::i8 [%0], %1, %2, %3, p;\n\t}"
      ::"r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
      : "memory");
}
// arrives on the same-offset mbarrier of BOTH CTAs of the pair once the issued MMAs have retired
__device__ __forceinline__ void umma_commit_pair(uint32_t bar) {
  asm volatile(
      "tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;"
      ::"r"(bar), "h"(uint16_t(3)) : "memory");
}

__device__ __forceinline__ void tma_prefetch_desc(const CUtensorMap* map) {
  asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(map)) : "memory");
}

__device__ __forceinline__ void tmem_alloc(uint32_t dst_smem, uint32_t ncols) {
  asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(dst_smem), "r"(ncols) : "memory");
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr, uint32_t ncols) {
  asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }

__device__ __forceinline__ void umma_bf16(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc,
                                          uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}"
      ::"r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
      : "memory");
}
__device__ __forceinline__ void umma_i8(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc,
                                        uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::i8 [%0], %1, %2, %3, p;\n\t}"
      ::"r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
      : "memory");
}
// arrives on the mbarrier once every previously issued tcgen05.mma of this thread has completed
__device__ __forceinline__ void umma_commit(uint32_t bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar) : "memory");
}

template <typename T>     // float (kind::f16 accumulators) or int (kind::i8)
__device__ __forceinline__ void tmem_ld32(uint32_t taddr, T (&v)[32]) {
  static_assert(sizeof(T) == 4, "32-bit accumulators");
  uint32_t* r = reinterpret_cast<uint32_t*>(v);
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32"
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15,"
      " %16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),
        "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]),
        "=r"(r[16]), "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]),
        "=r"(r[24]), "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
      : "r"(taddr)
      : "memory");
}
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }

// K-major, 128B-swizzled operand tile: rows of 64 bf16 or 128 int8 (128 B), 8-row groups 1024 B apart.
// Field layout: start>>4 [0,14) | LBO>>4 [16,30) | SBO>>4 [32,46) | version=1 [46,48) | swizzle [61,64).
__device__ __forceinline__ uint64_t umma_desc_sw128(uint32_t smem_addr) {
  return uint64_t((smem_addr & 0x3FFFFu) >> 4) | (uint64_t(1) << 16) | (uint64_t(1024 >> 4) << 32) |
         (uint64_t(1) << 46) | (uint64_t(2) << 61);
}

// K-major, 32B-swizzled operand tile of ONE UMMA K step: rows of 16 bf16 (32 B), 8-row groups 256 B apart
// (layout type 6).  The Euclidean plane's pad block: only 16 columns per gallery row are staged and multiplied.
__device__ __forceinline__ uint64_t umma_desc_sw32(uint32_t smem_addr) {
  return uint64_t((smem_addr & 0x3FFFFu) >> 4) | (uint64_t(1) << 16) | (uint64_t(256 >> 4) << 32) |
         (uint64_t(1) << 46) | (uint64_t(6) << 61);
}

// ------------------------------------------------------------------------------------------ shapes
constexpr int kTileQ = 128;          // queries per CTA tile (TMEM lanes); UMMA M = 128, or 256 across a CTA pair
constexpr int kTileR = 128;          // gallery rows staged per CTA and k-block (TMA box rows)
constexpr int kBlockK = 64;          // one 128-byte swizzle row of bf16
constexpr int kBlockKI8 = 128;       // ... of int8
constexpr int kMaxStages = 8;        // barrier slots of the ring; kStages (6) of them are used
constexpr int kMaxKBlocks = 8;       // 512 columns / 64
constexpr int kStageBytes = kTileR * kBlockK * 2;          // 16 KB
constexpr int kPadStageBytes = kTileR * kEuclidPad * 2;    // 4 KB of a stage: the Euclidean plane's pad block
constexpr int kEpiWarps = 8;          // two per TMEM lane quarter: they split a tile's columns
constexpr int kTcThreads = 64 + 32 * kEpiWarps;
// accumulator: double-buffered, N columns each (N = 128 single CTA, 256 for a CTA pair)
constexpr float kCoarseEps = 7.9e-3f;                      // a-priori |bf16 filter score - fp32 score| bound (no eps[] given)
// instruction descriptor, kind::f16: D=f32 [4,6)=1, A=bf16 [7,10)=1, B=bf16 [10,13)=1, K-major both,
// N>>3 at [17,23), M>>4 at [24,29)
constexpr uint32_t make_idesc(int m, int n) {
  return (1u << 4) | (1u << 7) | (1u << 10) | (uint32_t(n >> 3) << 17) | (uint32_t(m >> 4) << 24);
}
// kind::i8: D=s32 [4,6)=2, A=signed int8 [7,10)=1, B=signed int8 [10,13)=1, K-major both, same N / M fields
constexpr uint32_t make_idesc_i8(int m, int n) {
  return (2u << 4) | (1u << 7) | (1u << 10) | (uint32_t(n >> 3) << 17) | (uint32_t(m >> 4) << 24);
}

// The epilogue's element: fp32 scores of the bf16 filter, raw s32 products of the int8 filter (compared with an
// integer floor: one IMNMX per score, no conversion)
template <bool I8> struct Acc;
template <> struct Acc<false> {
  using T = float;
  static __device__ __forceinline__ T none() { return -INFINITY; }
  static __device__ __forceinline__ T mx(T a, T b) { return fmaxf(a, b); }
  static __device__ __forceinline__ int bits(T a) { return __float_as_int(a); }
};
template <> struct Acc<true> {
  using T = int;
  static __device__ __forceinline__ T none() { return INT_MIN; }
  static __device__ __forceinline__ T mx(T a, T b) { return max(a, b); }
  static __device__ __forceinline__ int bits(T a) { return a; }
};

enum TcMode { kModeGroupMax = 0, kModeFilter = 1, kModeFused = 2 };
constexpr int kGroups = 32;

// (float_key / key_float, frg_internal.cuh: the group maxima of all pre-pass CTAs are folded with one atomicMax per
// (query, group) on order-preserving keys)

// GROUPED launch (frg_match_tenants): what one CTA of a grid over many (query tile, tenant) pairs works on.  Queries
// q0 .. q0 + nq - 1 of the tenant-sorted batch (one tenant), chunk `chunk` of `chunks` over its gallery tiles: the
// absolute 128-row tiles list[0 .. n_tiles) or, without a list, tile0 .. tile0 + n_tiles - 1; every scale-th of them
// (pre-pass sample).  Its candidate segments start at cand[cand0], seg entries each.
struct TcGroupCta {
  int q0, nq, tenant, chunk, chunks, tile0, n_tiles, scale, seg;
  long long cand0;
  const int32_t* list;
};

struct TcScanParams {
  int dim;                 // 512 etc. (multiple of 64; of 128 for the int8 filter)
  int n_rows;              // gallery rows
  int tile_scale;          // pre-pass: only every tile_scale-th 128-row tile is visited (1 = all)
  int nq;                  // real queries
  int32_t tenant;
  const int32_t* tags;     // per REAL row
  // GROUPMAX output: [nq][32] maxima of the row groups (row mod 32) as ordered keys, atomicMax-folded
  uint32_t* group_key;
  // int8 filter: GROUPMAX folds [nq][32] 64-bit keys (s32 product biased by 2^31 << 32 | row): each group's winning
  // row is known, i8_floor_kernel rescores the k best of them exactly.  FILTER reads floor[q] (a floor of the exact
  // score, float) and qstep[q] (S = s32 product * qstep) and compares with the integer floor derived from them.
  unsigned long long* group_key64;
  const float* floor;
  const float* qstep;
  // FILTER inputs / outputs
  int k;                   // L[q] = k-th largest of the 32 group maxima (computed in the prologue)
  int* arrive;             // FUSED: CTAs that have published their probe-tile maxima
  int arrive_target;       // FUSED: wait (bounded) for this many before deriving the floor; 0 = do not wait
  int probe_div;           // FUSED: the probe is 1/probe_div of every CTA's chunk (at least one tile)
  int seg;                 // candidate slots per (query, chunk) private segment
  int2* cand;              // [nq][chunks][seg] (row, score bits): written while scanning
  int* cand_total;         // [nq] candidates of the query over all chunks (atomicAdd at the CTA's end)
  int2* dense;             // [nq][dense_cap]: the segments, packed per query for the select kernel
  int dense_cap;
  // error bound of the filter: eps == nullptr -> kCoarseEps for every query (unit vectors, cosine);
  // else eps[q] (Euclidean plane: scales with ||q|| and the store's largest row norm)
  const float* eps;
  float none_score;        // "nothing seen": kNoScore (cosine, scores > -1) or kEuclidNone
  // Euclidean plane: the LAST k-block of the query tile meets a 16-column pad block of the plane (pad_map:
  // box 16 x 128 rows, 32B swizzle, 4 KB per stage) with ONE K = 16 MMA instead of four
  int pad;
  int stages;              // depth of the TMA ring (kStages)
  uint32_t* fault;         // the store's fault word (host-mapped): set when a pipeline barrier timed out
  // Tile list (tenant-filtered calls over a window that is mostly other tenants' rows): the kernel walks
  // n_list listed tiles instead of every tile of the window; entry = absolute tile index (tile = kAccN rows)
  const int32_t* tile_list;
  int n_list;
  // GROUPED: one descriptor per CTA (blockIdx.x), frg_match_tenants
  const TcGroupCta* groups;
};

// MASKED: rows can be invalid for this call (tombstones, or a tenant filter): their tags are read
// once per 32-row block, one row per lane, and turned into a warp-uniform bit mask with a ballot -
// no per-candidate global load sits on the epilogue's dependent path.
// PAIR: the CTA pair variant (cluster of 2 along x = two query tiles against the same gallery rows).
// tcgen05.mma.cta_group::2 multiplies M = 256 queries (128 per CTA) by N = 256 gallery rows, each CTA
// staging only ITS 128-row half of every B tile: half the shared-memory operand traffic per flop of
// the single-CTA form, which is what lifts the tensor pipe at large batches.  The leader CTA (rank 0)
// owns the full/tmem_empty barriers and issues the MMAs; commits are multicast to both CTAs.
// I8: int8 operands (unit cosine store's int8 plane): tcgen05.mma kind::i8, K = 32 per MMA, 128 int8 per k-block,
// exact s32 accumulators; half the MMA time and half the plane bytes of bf16 per score.  Not FUSED.
// GROUPED: blockIdx.x selects a TcGroupCta (single-CTA int8 form only); the query tile, tenant, tile source and chunk
// come from it instead of the grid and the scalar parameters.
template <int MODE, bool MASKED, bool PAIR, bool I8 = false, bool GROUPED = false>
__global__ void __launch_bounds__(kTcThreads, 1)
tc_scan_kernel(const __grid_constant__ CUtensorMap q_map, const __grid_constant__ CUtensorMap g_map,
               const __grid_constant__ CUtensorMap pad_map, const TcScanParams p) {
  static_assert(!(I8 && MODE == kModeFused), "the int8 filter takes its floor from i8_floor_kernel");
  static_assert(!GROUPED || (I8 && MASKED && !PAIR), "the grouped form is the single-CTA int8 masked filter");
  using A = Acc<I8>;
  using AccT = typename A::T;
  constexpr int kAccN = PAIR ? 2 * kTileR : kTileR;        // accumulator columns = gallery rows per tile
  constexpr int kTmemCols = 2 * kAccN;
  constexpr int kBlk = I8 ? kBlockKI8 : kBlockK;             // elements per 128-byte k-block
  constexpr uint32_t kIdesc = I8 ? make_idesc_i8(PAIR ? 2 * kTileQ : kTileQ, kAccN)
                                 : make_idesc(PAIR ? 2 * kTileQ : kTileQ, kAccN);
  const uint32_t cta_rank = PAIR ? cluster_ctarank() : 0u;
  const bool leader = cta_rank == 0;
  extern __shared__ unsigned char smem_raw[];
  // 128B swizzle wants 1024-byte aligned tiles
  const uint32_t raw = smem_u32(smem_raw);
  const uint32_t base = (raw + 1023u) & ~1023u;
  unsigned char* sm = smem_raw + (base - raw);
  const int kblocks = p.dim / kBlk;
  const uint32_t q_bytes = uint32_t(kTileQ) * p.dim * (I8 ? 1 : 2);   // resident query tile
  const uint32_t q_smem = base;
  const uint32_t stage_smem = base + q_bytes;
  const int nstages = p.stages;
  uint64_t* bars = reinterpret_cast<uint64_t*>(sm + q_bytes + nstages * kStageBytes);
  const uint32_t bar0 = smem_u32(bars);
  auto bar_full = [&](int s) { return bar0 + 8u * s; };
  auto bar_empty = [&](int s) { return bar0 + 8u * (kMaxStages + s); };
  auto bar_tfull = [&](int b) { return bar0 + 8u * (2 * kMaxStages + b); };
  auto bar_tempty = [&](int b) { return bar0 + 8u * (2 * kMaxStages + 2 + b); };
  // one barrier per k-block of the resident query tile: the first MMAs start when 16 KB of it have
  // landed, not all 128 KB
  auto bar_q = [&](int kb) { return bar0 + 8u * (2 * kMaxStages + 4 + kb); };
  uint32_t* tmem_holder = reinterpret_cast<uint32_t*>(bars + 2 * kMaxStages + 4 + kMaxKBlocks);
  volatile int* abort_flag = reinterpret_cast<volatile int*>(tmem_holder + 1);

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  const int qtile = blockIdx.x;
  TcGroupCta gd{};
  if constexpr (GROUPED) gd = p.groups[blockIdx.x];     // written by the host copy that precedes the whole match
  const int chunk = GROUPED ? gd.chunk : int(blockIdx.y), chunks = GROUPED ? gd.chunks : int(gridDim.y);
  const int tile_scale = GROUPED ? gd.scale : p.tile_scale;
  // view tile v stands for gallery tile v * tile_scale (the pre-pass samples whole 128-row tiles:
  // contiguous 128 KB reads, spread evenly over the gallery)
  const int tiles_all = GROUPED ? gd.n_tiles : (p.tile_list ? p.n_list : (p.n_rows + kAccN - 1) / kAccN);
  const int tiles_total = (tiles_all + tile_scale - 1) / tile_scale;
  // gallery tile behind view tile v
  auto gtile = [&](int v) {
    const int i = v * tile_scale;
    if constexpr (GROUPED) return gd.list ? __ldg(gd.list + i) : gd.tile0 + i;
    else return p.tile_list ? __ldg(p.tile_list + i) : i;
  };
  const int tile_begin = int((int64_t(tiles_total) * chunk) / chunks);
  const int tile_end = int((int64_t(tiles_total) * (chunk + 1)) / chunks);
  // FUSED: the CTA's first n_probe tiles (1/64 of its chunk, at least one) are visited twice - first as
  // a probe (group maxima only, published to all CTAs so that everyone can derive the floor L[q]),
  // and once more at the very end to emit from them
  const int n_tiles = tile_end - tile_begin;
  const int n_probe = MODE == kModeFused ? (n_tiles + p.probe_div - 1) / p.probe_div : 0;
  const int n_iter = n_tiles + n_probe;
  auto tile_of = [&](int it) { return it < n_tiles ? tile_begin + it : tile_begin + (it - n_tiles); };

  if (threadIdx.x == 0) {
    *abort_flag = 0;
    for (int s = 0; s < nstages; ++s) { mbar_init(bar_full(s), 1); mbar_init(bar_empty(s), 1); }
    for (int b = 0; b < 2; ++b) { mbar_init(bar_tfull(b), 1); mbar_init(bar_tempty(b), PAIR ? 2 * kEpiWarps : kEpiWarps); }
    for (int kb = 0; kb < kblocks; ++kb) mbar_init(bar_q(kb), 1);
    fence_barrier_init();
  }
  if (warp == 1) {
    if (PAIR) tmem_alloc_pair(smem_u32(tmem_holder), kTmemCols);
    else tmem_alloc(smem_u32(tmem_holder), kTmemCols);
  }
  tc_fence_before();
  if (PAIR) cluster_sync_all();        // the peer's barriers must exist before anything signals them
  else __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_holder;
  // everything above ran while the previous kernel of the match was still finishing (PDL); from here on
  // its results are read (query image, group maxima, counters)
  pdl_wait();
  pdl_trigger();

  if (warp == 0) {
    // ===== TMA producer =====
    if (lane == 0) {
      tma_prefetch_desc(&q_map);
      tma_prefetch_desc(&g_map);
      if (p.pad) tma_prefetch_desc(&pad_map);
      const uint64_t g_hint = gridDim.x > (PAIR ? 2 : 1) ? kEvictLast : kEvictFirst;
      constexpr uint32_t kQBlockBytes = kTileQ * 128;
      int stage = 0; uint32_t phase = 0;
      for (int it = 0; it < n_iter && !*abort_flag; ++it) {
        const int t = tile_of(it);
        const int row0 = gtile(t) * kAccN + int(cta_rank) * kTileR;   // this CTA's half of the tile
        for (int kb = 0; kb < kblocks; ++kb) {
          if (it == 0) {
            // the query tile's k-block kb, issued just ahead of the first gallery block that meets it
            if (PAIR) {
              if (leader) mbar_expect_tx(bar_q(kb), 2 * kQBlockBytes);
              tma_load_2d_pair(q_smem + kb * kQBlockBytes, &q_map, bar_q(kb), kb * kBlk, GROUPED ? gd.q0 : qtile * kTileQ, kEvictLast);
            } else {
              mbar_expect_tx(bar_q(kb), kQBlockBytes);
              tma_load_2d(q_smem + kb * kQBlockBytes, &q_map, bar_q(kb), kb * kBlk, GROUPED ? gd.q0 : qtile * kTileQ, kEvictLast);
            }
          }
          mbar_wait(bar_empty(stage), phase ^ 1, abort_flag);
          const bool padkb = p.pad && kb == kblocks - 1;
          const CUtensorMap* map = padkb ? &pad_map : &g_map;
          const uint32_t bytes = padkb ? kPadStageBytes : kStageBytes;
          const int c0 = padkb ? 0 : kb * kBlk;
          if (PAIR) {
            if (leader) mbar_expect_tx(bar_full(stage), 2 * bytes);
            tma_load_2d_pair(stage_smem + stage * kStageBytes, map, bar_full(stage), c0, row0, g_hint);
          } else {
            mbar_expect_tx(bar_full(stage), bytes);
            tma_load_2d(stage_smem + stage * kStageBytes, map, bar_full(stage), c0, row0, g_hint);
          }
          if (++stage == nstages) { stage = 0; phase ^= 1; }
        }
      }
    }
  } else if (warp == 1) {
    // ===== MMA issuer (leader CTA only in pair mode) =====
    // The whole warp runs the loop (waits, descriptor arithmetic) so that every operand of
    // tcgen05.mma is warp-uniform and lives in uniform registers; only the tcgen05 instructions
    // themselves are issued by one elected lane.  (Running the loop under `lane == 0` costs an
    // ELECT + R2UR chain per MMA operand and makes the issue path, not the tensor pipe, the limit.)
    if (leader) {
      int stage = 0; uint32_t phase = 0;
      int buf = 0; uint32_t tphase = 0;
      const uint64_t a_base = umma_desc_sw128(q_smem);
      const uint64_t b_base = umma_desc_sw128(stage_smem);
      const uint64_t pad_base = umma_desc_sw32(stage_smem);
      for (int it = 0; it < n_iter && !*abort_flag; ++it) {
        mbar_wait(bar_tempty(buf), tphase ^ 1, abort_flag);
        tc_fence_after();
        const uint32_t d_tmem = tmem_base + uint32_t(buf * kAccN);
        for (int kb = 0; kb < kblocks; ++kb) {
          if (it == 0) mbar_wait(bar_q(kb), 0, abort_flag);          // first tile: the query k-block must have landed
          mbar_wait(bar_full(stage), phase, abort_flag);
          tc_fence_after();
          // descriptor start-address field is (addr >> 4): a k-block of A is 16 KB, a stage of B 16 KB
          const uint64_t a0 = a_base + uint64_t(kb * ((kTileQ * 128) >> 4));
          const uint64_t b0 = b_base + uint64_t(stage * (kStageBytes >> 4));
          const bool padkb = p.pad && kb == kblocks - 1;
          if (elect_one()) {
            if (padkb) {
              // the query tile's last k-block (128B swizzle, columns 0..15) x the staged 16-column pad block
              const uint64_t bp = pad_base + uint64_t(stage * (kStageBytes >> 4));
              if (PAIR) umma_bf16_pair(d_tmem, a0, bp, kIdesc, 1u);
              else umma_bf16(d_tmem, a0, bp, kIdesc, 1u);
            } else {
#pragma unroll
              for (int kk = 0; kk < 4; ++kk) {
                // advance one MMA's K (16 bf16 / 32 int8) = 32 bytes inside the swizzle row: +2 in the (addr >> 4) field
                const uint32_t acc = (kb | kk) != 0 ? 1u : 0u;
                if (I8) {
                  if (PAIR) umma_i8_pair(d_tmem, a0 + uint64_t(kk * 2), b0 + uint64_t(kk * 2), kIdesc, acc);
                  else umma_i8(d_tmem, a0 + uint64_t(kk * 2), b0 + uint64_t(kk * 2), kIdesc, acc);
                } else {
                  if (PAIR) umma_bf16_pair(d_tmem, a0 + uint64_t(kk * 2), b0 + uint64_t(kk * 2), kIdesc, acc);
                  else umma_bf16(d_tmem, a0 + uint64_t(kk * 2), b0 + uint64_t(kk * 2), kIdesc, acc);
                }
              }
            }
            // smem slot reusable / accumulator readable once these MMAs retire (both CTAs in pair mode)
            if (PAIR) {
              umma_commit_pair(bar_empty(stage));
              if (kb == kblocks - 1) umma_commit_pair(bar_tfull(buf));
            } else {
              umma_commit(bar_empty(stage));
              if (kb == kblocks - 1) umma_commit(bar_tfull(buf));
            }
          }
          __syncwarp();
          if (++stage == nstages) { stage = 0; phase ^= 1; }
        }
        if (++buf == 2) { buf = 0; tphase ^= 1; }
      }
    }
  } else {
    // ===== epilogue: thread = query (TMEM lane), columns = gallery rows =====
    const int quarter = warp & 3;                        // tcgen05.ld: warp w may touch lanes 32*(w%4)..+31
    // FILTER: the two warps of a quarter split every tile's columns (the epilogue is issue-latency
    // bound, two warps per scheduler hide it).  bf16 GROUPMAX: one warp per quarter does all columns (the
    // other only keeps the barrier protocol), so each (query, group) maximum costs ONE atomic per CTA.
    // I8 GROUPMAX splits the columns like the filter and folds the two warps' maxima in shared memory at the end.
    constexpr bool kSplitCols = MODE != kModeGroupMax || I8;
    constexpr int kSplit = kSplitCols ? kEpiWarps / 4 : 1;
    const int half = kSplitCols ? (warp - 2) >> 2 : 0;
    const bool idle = !kSplitCols && warp >= 6;
    constexpr int kBlocksPerWarp = (kAccN / 32) / kSplit;
    const int q_local = quarter * 32 + lane;
    const int q = (GROUPED ? gd.q0 : qtile * kTileQ) + q_local;
    const bool q_real = GROUPED ? q_local < gd.nq : q < p.nq;
    const int32_t tenant = GROUPED ? gd.tenant : p.tenant;

    // GROUPMAX / FUSED probe: running maximum per row group.  I8 GROUPMAX keeps ONE packed key per group instead,
    // acc * 256 + lb (|acc| <= 127^2 * 512 < 2^23, so the key is exact and orders by (acc, lb)), lb = the CTA-local
    // 32-row block of the maximum within a window of kWinTiles tiles: one IMAD + IMNMX per score carries the winner.
    // The larger block wins an exact tie; any winner is a valid distinct row of its group.
    AccT gmax[kGroups];
    constexpr int kTileBlocks = kAccN / 32;
    constexpr int kWinTiles = 256 / kTileBlocks;
    AccT thr;
    if constexpr (I8) thr = INT_MAX;
    else thr = INFINITY;
    int emitted = 0;
    int2* my_seg = nullptr;
    // L[q] = k-th largest of the 32 group maxima published so far.  The groups are disjoint row sets,
    // so that value is reached by k distinct valid rows: L[q] <= tau, whatever subset has been seen.
    auto derive_thr = [&]() {
      const uint4* src = reinterpret_cast<const uint4*>(p.group_key + size_t(q) * kGroups);
      float g[kGroups];
#pragma unroll
      for (int j = 0; j < kGroups; j += 4) {
        uint4 x;
        if (MODE == kModeFused) {           // other CTAs are still publishing: bypass the non-coherent path
          asm volatile("ld.global.cg.v4.u32 {%0,%1,%2,%3}, [%4];"
                       : "=r"(x.x), "=r"(x.y), "=r"(x.z), "=r"(x.w) : "l"(src + j / 4) : "memory");
        } else {
          x = __ldg(src + j / 4);
        }
        g[j] = key_float(x.x); g[j + 1] = key_float(x.y); g[j + 2] = key_float(x.z); g[j + 3] = key_float(x.w);
      }
      float floor_v = p.none_score;
      for (int r = 0; r < p.k; ++r) {
        float m = g[0];
#pragma unroll
        for (int j = 1; j < kGroups; ++j) m = fmaxf(m, g[j]);
        floor_v = m;
        bool popped = false;                 // remove ONE instance of the maximum
#pragma unroll
        for (int j = 0; j < kGroups; ++j) {
          const bool hit = !popped && g[j] == m;
          g[j] = hit ? -INFINITY : g[j];
          popped |= hit;
        }
      }
      // fewer than k usable groups so far: no bound, every valid row is a candidate
      // (finite, so that masked columns, which are set to -inf, still fail the comparison)
      const float eps_q = p.eps ? __ldg(p.eps + q) : kCoarseEps;
      return (floor_v <= p.none_score) ? -3.0e38f : floor_v - 2.0f * eps_q;
    };
    // int8 filter: the integer floor of the s32 products, from the float floor (i8_floor_kernel, or threshold - eps
    // for a range search) and the query's step, rounded down with a margin of 3 (|floor / qstep| < 2^23: the fp32
    // quotient is within 1 of the real one).  NaN floor (a NaN query, which no row can match): no candidates.
    auto derive_thr_i8 = [&]() {
      const float f = __ldg(p.floor + q);
      if (!(f == f)) return INT_MAX;
      const float t = fminf(fmaxf(__fdiv_rn(f, __ldg(p.qstep + q)), -1.0e9f), 1.0e9f);
      return __float2int_rd(t) - 3;
    };
    if (MODE != kModeFilter) {
#pragma unroll
      for (int j = 0; j < kGroups; ++j) {
        if constexpr (I8) gmax[j] = A::none();
        else gmax[j] = p.none_score;
      }
    }
    // I8 GROUPMAX: fold the packed keys of the window that began at iteration it0 into the (query, group) 64-bit keys,
    // (s32 product biased by 2^31) << 32 | row
    auto publish_i8 = [&](int it0) {
      if constexpr (I8) {
        unsigned long long* o = p.group_key64 + size_t(q) * kGroups;
#pragma unroll
        for (int j = 0; j < kGroups; ++j) {
          if (gmax[j] != A::none()) {
            const int lb = gmax[j] & 255;
            const int row = gtile(tile_of(it0 + lb / kTileBlocks)) * kAccN + (lb % kTileBlocks) * 32 + j;
            atomicMax(o + j, (uint64_t(uint32_t(gmax[j] >> 8) ^ 0x80000000u) << 32) | uint32_t(row));
          }
        }
      }
    };
    if (MODE != kModeGroupMax && q_real) {
      if constexpr (I8) thr = derive_thr_i8();
      else if (MODE == kModeFilter) thr = derive_thr();
      if constexpr (GROUPED) my_seg = p.cand + gd.cand0 + ((size_t(q_local) * chunks + chunk) * (kEpiWarps / 4) + half) * gd.seg;
      else my_seg = p.cand + ((size_t(q) * chunks + chunk) * (kEpiWarps / 4) + half) * p.seg;
    }

    int buf = 0; uint32_t tphase = 0;
    int win0 = 0;                                          // I8 GROUPMAX: first iteration of the current lb window
    for (int it = 0; it < n_iter && !*abort_flag; ++it) {
      const int t = tile_of(it);
      const int tile_row0 = gtile(t) * kAccN;              // first gallery row of this tile
      const bool probe = MODE == kModeGroupMax || (MODE == kModeFused && it < n_probe);
      if (idle) {
        mbar_wait(bar_tfull(buf), tphase, abort_flag);
        if (lane == 0) {
          if (PAIR) mbar_arrive_remote(bar_tempty(buf), 0);
          else mbar_arrive(bar_tempty(buf));
        }
        if (++buf == 2) { buf = 0; tphase ^= 1; }
        continue;
      }
      // validity of this tile's rows (32 per ballot), fetched while the tile's MMAs are still running
      uint32_t vmask[kBlocksPerWarp];
#pragma unroll
      for (int b = 0; b < kBlocksPerWarp; ++b) {
        const int row = tile_row0 + (half * kBlocksPerWarp + b) * 32 + lane;
        bool ok = row < p.n_rows;
        if (MASKED && ok) {
          const int32_t tag = __ldg(p.tags + row);
          ok = tag >= 0 && (tenant < 0 || tag == tenant);
        }
        vmask[b] = __ballot_sync(0xffffffffu, ok);
      }
      mbar_wait(bar_tfull(buf), tphase, abort_flag);
      tc_fence_after();
      const uint32_t taddr = tmem_base + (uint32_t(quarter * 32) << 16) +
                             uint32_t(buf * kAccN + half * kBlocksPerWarp * 32);
      // software-pipelined TMEM reads: the load of block b+1 is in flight while block b is processed
      AccT va[32], vb[32];
      auto process = [&](AccT (&v)[32], int b) {
        const uint32_t vm = vmask[b];
        if (!(I8 && MODE == kModeGroupMax) && vm != 0xffffffffu) {   // warp-uniform: tombstones / other tenants / rows past the end
#pragma unroll
          for (int j = 0; j < 32; ++j) v[j] = (vm >> j) & 1u ? v[j] : A::none();
        }
        if (MODE == kModeGroupMax) {
          // column j of every 32-row block belongs to group j (tiles start at multiples of 32)
          if constexpr (I8) {
            const int lb = (it % kWinTiles) * kTileBlocks + half * kBlocksPerWarp + b;
            if (vm == 0xffffffffu) {
#pragma unroll
              for (int j = 0; j < 32; ++j) gmax[j] = max(gmax[j], v[j] * 256 + lb);
            } else {
#pragma unroll
              for (int j = 0; j < 32; ++j) gmax[j] = max(gmax[j], (vm >> j) & 1u ? v[j] * 256 + lb : A::none());
            }
          } else {
#pragma unroll
            for (int j = 0; j < 32; ++j) gmax[j] = fmaxf(gmax[j], v[j]);
          }
        } else if (MODE == kModeFused && probe) {
          // this warp sees half of the tile's rows: it owns 16 of the 32 groups, (column mod 16)
#pragma unroll
          for (int j = 0; j < 32; ++j) gmax[j & 15] = A::mx(gmax[j & 15], v[j]);
        } else {
          // The block maximum is built from four 8-column group maxima, and a thread that holds a candidate walks
          // only the group(s) that contain one: ~35 instructions instead of ~110 for all 32 columns.  A warp takes
          // this path whenever one of its 32 queries has a candidate among the 32 rows (about a quarter of all
          // blocks), and (bf16) the slowest epilogue warp decides when the accumulator buffer goes back to the MMA warp.
          // Measured against the 32-column walk (profiles/r02_ab_grouped.txt, same box, sustained clocks): -3.6 /
          // -4.8 / -7 % of the step at F = 256 / 512 / 1024, neutral at F <= 128 (HBM-bound, the epilogue has slack).
          AccT g0 = v[0], g1 = v[8], g2 = v[16], g3 = v[24];
#pragma unroll
          for (int j = 1; j < 8; ++j) {
            g0 = A::mx(g0, v[j]); g1 = A::mx(g1, v[8 + j]); g2 = A::mx(g2, v[16 + j]); g3 = A::mx(g3, v[24 + j]);
          }
          if (A::mx(A::mx(g0, g1), A::mx(g2, g3)) >= thr) {
            const int row0 = tile_row0 + (half * kBlocksPerWarp + b) * 32;
            const AccT gm[4] = {g0, g1, g2, g3};
#pragma unroll
            for (int g = 0; g < 4; ++g) {
              if (gm[g] >= thr) {
#pragma unroll
                for (int j = 8 * g; j < 8 * g + 8; ++j) {
                  if (v[j] >= thr) {
                    if (emitted < (GROUPED ? gd.seg : p.seg)) my_seg[emitted] = make_int2(row0 + j, A::bits(v[j]));
                    ++emitted;
                  }
                }
              }
            }
          }
        }
      };
      __syncwarp();
      if constexpr (I8 && MODE == kModeFilter) {
        // Early release: the int8 MMA takes as long as the TMEM reads of its tile (~2048 clk per pair tile at dim
        // 512), so a buffer held through the rare paths stalls the tensor pipe.  All of the warp's blocks go to
        // registers first; the buffer goes back to the MMA warp before any of them is processed.
        AccT vs[kBlocksPerWarp][32];
#pragma unroll
        for (int b = 0; b < kBlocksPerWarp; ++b) tmem_ld32(taddr + b * 32, vs[b]);
        tmem_ld_wait();
        tc_fence_before();
        __syncwarp();
        if (lane == 0) {
          if (PAIR) mbar_arrive_remote(bar_tempty(buf), 0);
          else mbar_arrive(bar_tempty(buf));
        }
#pragma unroll
        for (int b = 0; b < kBlocksPerWarp; ++b) process(vs[b], b);
      } else {
        tmem_ld32(taddr, va);
#pragma unroll
        for (int b = 0; b < kBlocksPerWarp; b += 2) {
          tmem_ld_wait();                    // va (block b) has landed
          __syncwarp();                      // tcgen05.ld is .sync.aligned: reconverge after a slow path
          tmem_ld32(taddr + (b + 1) * 32, vb);
          process(va, b);
          tmem_ld_wait();                    // vb (block b + 1)
          __syncwarp();
          if (b + 2 < kBlocksPerWarp) tmem_ld32(taddr + (b + 2) * 32, va);
          process(vb, b + 1);
        }
        tc_fence_before();
        __syncwarp();
        if (lane == 0) {
          if (PAIR) mbar_arrive_remote(bar_tempty(buf), 0);      // the leader's MMA thread waits on it
          else mbar_arrive(bar_tempty(buf));
        }
      }
      if (++buf == 2) { buf = 0; tphase ^= 1; }
      if constexpr (MODE == kModeGroupMax && I8) {
        // a window's blocks fill the 8 bits of lb: publish this warp's keys and start the next window
        if ((it + 1) % kWinTiles == 0 && it + 1 < n_iter) {
          if (q_real) publish_i8(win0);
#pragma unroll
          for (int j = 0; j < kGroups; ++j) gmax[j] = A::none();
          win0 = it + 1;
        }
      }

      if constexpr (MODE == kModeFused && !I8) {
        const int since = it - (n_probe - 1);           // 0 at the last probe tile
        if (since == 0) {
          // publish the probe tile's maxima (groups half*16 .. +15), tell the grid, derive the floor
          if (q_real) {
            uint32_t* o = p.group_key + size_t(q) * kGroups + half * 16;
#pragma unroll
            for (int j = 0; j < 16; ++j)
              if (gmax[j] > p.none_score) atomicMax(o + j, float_key(gmax[j]));
          }
          __threadfence();
          asm volatile("bar.sync 1, %0;" ::"n"(32 * kEpiWarps) : "memory");     // the epilogue warps only
          if (warp == 2 && lane == 0) atomicAdd(p.arrive, 1);
          if (p.arrive_target > 0) {
            // single-wave grid: give the other CTAs a few microseconds to publish too.  Bounded: a late
            // CTA only makes this one's floor a little looser, never wrong.
            for (int spin = 0; spin < 48; ++spin) {
              if (*reinterpret_cast<volatile int*>(p.arrive) >= p.arrive_target) break;
              __nanosleep(128);
            }
          }
          if (q_real) thr = derive_thr();
        } else if (since > 0 && (since & (since - 1)) == 0 && q_real && it < n_iter - 1) {
          thr = derive_thr();              // late publishers: refresh 1, 2, 4, 8, ... tiles later
        }
      }
    }
    if constexpr (MODE == kModeGroupMax && I8) {
      // fold the two warps of the quarter through shared memory (the ring: the last tile's MMAs have retired),
      // then ONE 64-bit atomicMax per (query, group) and CTA
      int* fold = reinterpret_cast<int*>(sm + q_bytes);
      if (half == 1) {
#pragma unroll
        for (int j = 0; j < kGroups; ++j) fold[j * kTileQ + q_local] = gmax[j];
      }
      asm volatile("bar.sync %0, 64;" ::"r"(2 + quarter) : "memory");
      if (half == 0) {
#pragma unroll
        for (int j = 0; j < kGroups; ++j) gmax[j] = max(gmax[j], fold[j * kTileQ + q_local]);
        if (q_real) publish_i8(win0);
      }
    } else if (q_real && !idle) {
      if (MODE == kModeGroupMax) {
        uint32_t* o = p.group_key + size_t(q) * kGroups;
#pragma unroll
        for (int j = 0; j < kGroups; ++j)
          if (gmax[j] > p.none_score) atomicMax(o + j, float_key(gmax[j]));
      } else {
        // pack this thread's few candidates into the query's dense list: one atomicAdd per (query, CTA),
        // outside the scan loop.  A private-segment overflow poisons the total so that select flags it
        // (2^20 > any dense_cap; a query has at most 2 * 148 segments, so the sum of poisons cannot wrap).
        const int seg = GROUPED ? gd.seg : p.seg;
        const int base = atomicAdd(p.cand_total + q, emitted > seg ? (1 << 20) : emitted);
        const int mine_n = emitted < seg ? emitted : seg;
        for (int i = 0; i < mine_n; ++i)
          if (unsigned(base + i) < unsigned(p.dense_cap)) p.dense[size_t(q) * p.dense_cap + base + i] = my_seg[i];
      }
    }
  }

  tc_fence_before();
  if (PAIR) cluster_sync_all();        // the leader's MMAs read the peer's shared memory until the very end
  else __syncthreads();
  if (threadIdx.x == 0 && *abort_flag && p.fault)      // zero-copy word in pinned host memory: only ever written here
    asm volatile("st.relaxed.sys.global.u32 [%0], %1;" ::"l"(p.fault), "r"(uint32_t(1 + MODE)) : "memory");
  if (warp == 1) {
    __syncwarp();
    if (PAIR) tmem_dealloc_pair(tmem_base, kTmemCols);
    else tmem_dealloc(tmem_base, kTmemCols);
  }
}

// ------------------------------------------------------------------------------------------ int8 floor
// One warp per query, between the int8 pre-pass and the filter: the pre-pass left, per row group, the (s32 product,
// row) of the group's best sampled row.  The k best of those are k DISTINCT valid rows (the groups are disjoint);
// they are rescored exactly, with the streaming scan's arithmetic, so e_k = the smallest of those k exact scores is
// <= tau, the k-th best exact score.  Every row of the true top-k has S >= s - eps >= tau - eps >= e_k - eps:
// floor[q] = e_k - eps[q] is rigorous, without the coarse error of a sampled floor or a second eps.  Fewer than k
// groups seen: no floor.  NaN eps (a NaN query, which no row matches): NaN floor, no candidates.
__global__ void __launch_bounds__(128)
i8_floor_kernel(const unsigned long long* __restrict__ keys, int nq, int k, int dim, const float* __restrict__ qn,
                const float* __restrict__ master, const float* __restrict__ eps, float* __restrict__ floor_out) {
  pdl_wait();             // the pre-pass's group keys
  pdl_trigger();
  const int lane = threadIdx.x & 31;
  const int w = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  if (w >= nq) return;
  unsigned long long key = keys[size_t(w) * kGroups + lane];
  const float4* qq = reinterpret_cast<const float4*>(qn + size_t(w) * dim);
  const int nvec = dim >> 2;
  float e_k = INFINITY;
  int got = 0;
  for (int r = 0; r < k; ++r) {
    const uint32_t hi = uint32_t(key >> 32), lo = uint32_t(key);
    const uint32_t mh = __reduce_max_sync(0xffffffffu, hi);
    if (mh == 0u) break;                               // warp-uniform: no group left
    const uint32_t ml = __reduce_max_sync(0xffffffffu, hi == mh ? lo : 0u);
    if (hi == mh && lo == ml) key = 0ull;              // rows are distinct across groups: exactly one lane
    const float4* g = reinterpret_cast<const float4*>(master + size_t(ml) * dim);
    float a = 0.f;
#pragma unroll 4
    for (int v = lane; v < nvec; v += 32) {
      const float4 x = __ldg(g + v), y = __ldg(qq + v);
      a = fmaf(x.x, y.x, a); a = fmaf(x.y, y.y, a); a = fmaf(x.z, y.z, a); a = fmaf(x.w, y.w, a);
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) a += __shfl_xor_sync(0xffffffffu, a, o);
    e_k = fminf(e_k, a == a ? a : -INFINITY);
    ++got;
  }
  if (lane == 0) {
    const float e = __ldg(eps + w);
    floor_out[w] = !(e == e) ? NAN : (got < k ? -3.0e38f : e_k - e);
  }
}

// ------------------------------------------------------------------------------------------ stage 3
// One CTA per query: tau from the candidate list, keep the rows that can still be in the top-k, rescore in fp32, top-k.
constexpr int kMaxKeep = 256;      // rescored rows per query before the query is handed to the fallback

template <int K>
__device__ __forceinline__ void lane_insert(float (&sc)[K], int32_t (&ix)[K], float s, int32_t r) {
  if (s > sc[K - 1] || (s == sc[K - 1] && r < ix[K - 1])) {
    sc[K - 1] = s; ix[K - 1] = r;
#pragma unroll
    for (int t = K - 1; t > 0; --t) {
      if (sc[t] > sc[t - 1] || (sc[t] == sc[t - 1] && ix[t] < ix[t - 1])) {
        float ts = sc[t]; sc[t] = sc[t - 1]; sc[t - 1] = ts;
        int32_t tr = ix[t]; ix[t] = ix[t - 1]; ix[t - 1] = tr;
      }
    }
  }
}

// pops the warp-wide best (score desc, row asc) of the lane-local sorted lists
template <int K>
__device__ __forceinline__ void warp_pop_best(float (&sc)[K], int32_t (&ix)[K], int lane, float sentinel,
                                              float* best_s, int32_t* best_r) {
  const int bl = warp_argbest<int32_t>(sc[0], ix[0], 0x7fffffff, lane);
  const float bs = __shfl_sync(0xffffffffu, sc[0], bl);
  const int32_t br = __shfl_sync(0xffffffffu, ix[0], bl);
  if (lane == bl) {
#pragma unroll
    for (int t = 0; t < K - 1; ++t) { sc[t] = sc[t + 1]; ix[t] = ix[t + 1]; }
    sc[K - 1] = sentinel; ix[K - 1] = 0x7fffffff;
  }
  *best_s = bs; *best_r = br;
}

constexpr int kSelectWarps = 4;

// ONE CTA (4 warps) per query.  The dense candidate list of a query (a few hundred entries, L2-resident:
// the filter kernel has just written it) is read twice straight from global memory, each warp taking every
// fourth 32-entry slice; the warps meet in shared memory three times (their k best coarse scores -> tau,
// the compacted survivors, the exact scores).  With one WARP per query the kernel ran ~3900 dependent
// instructions per query at 5 warps per SM (40 us at 1024 queries, ncu: 83 % of cycles no eligible warp);
// four warps per query cut the chain and quadruple the warps in flight.
// EUCLID: the coarse scores are S = q.g - 0.5*||g||^2 (larger = nearer); the kept rows are rescored as the
// exact direct-difference d^2 = sum (g - q)^2 (the streaming scan's arithmetic and order), ranked by
// (-d^2 desc, row asc) and reported as distances; accept iff d <= threshold.
// Cosine with rescoring: two steps.  The k best coarse rows are rescored first; the smallest of their exact scores,
// tau_e, is <= the true k-th best tau (k distinct rows reach it), so every row of the true top-k has
// S >= tau - eps >= tau_e - eps: only those are rescored next (about 30 rows at dim 512 with the int8 filter's eps,
// instead of ~140 above tau_c - 2 eps).
// qstep != nullptr: the candidates carry the int8 filter's s32 products, S = product * qstep[q].
template <int K, bool EUCLID>
__global__ void __launch_bounds__(kSelectWarps * 32)
select_rescore_kernel(const int2* __restrict__ dense, const int* __restrict__ cand_total,
                      int dense_cap, int nq, int k, int dim, const float* __restrict__ qn,
                      const float* __restrict__ eps, const __nv_bfloat16* __restrict__ plane, int plane_dim,
                      const float* __restrict__ coef, const float* __restrict__ qstep,
                      const float* __restrict__ master, int rescore, float threshold, int64_t row_offset,
                      int64_t* __restrict__ out_rows, float* __restrict__ out_scores,
                      uint8_t* __restrict__ out_accept, int* __restrict__ flagged, int* __restrict__ n_flagged,
                      const XPush x) {
  __shared__ int keep_row[kMaxKeep];
  __shared__ float keep_sc[kMaxKeep];
  __shared__ float top_s[kSelectWarps][FRG_MAX_K];
  __shared__ int32_t top_r[kSelectWarps][FRG_MAX_K];
  __shared__ int s_m;
  const int lane = threadIdx.x & 31;
  const int w = threadIdx.x >> 5;
  const int q = blockIdx.x;
  pdl_wait();             // the filter kernel's candidate lists
  pdl_trigger();
  // row-sharded gallery: tell every rank which call this is before the first result goes out (exchange.cu)
  if (x.peer_bufs && blockIdx.x == 0 && int(threadIdx.x) < x.world) xpush_hello(x, threadIdx.x);

  const int total = cand_total[q];
  if (total > dense_cap) {                           // also set by a poisoned total (segment overflow)
    // the dense list is incomplete (and partly unwritten): leave the query to the exact fallback
    if (threadIdx.x == 0) flagged[atomicAdd(n_flagged, 1)] = q;
    return;
  }
  const int n = total;
  const int2* mine = dense + size_t(q) * dense_cap;
  if (threadIdx.x == 0) s_m = 0;

  // EUCLID: an entry's coarse score is an UPPER bound U of the row's exact score (the filter's query image adds the
  // row's own error bound, queries.cu); tau must be a floor of the true k-th best, so entries are ranked by their
  // LOWER bounds L = U - 2 err, err recomputed from the row's bound columns (the same bf16 numbers the tensor core
  // multiplied) - and every entry with U >= tau survives.  Cosine: ranked by the score itself (below: tau_e - eps).
  const float ca = EUCLID ? coef[size_t(q) * 4] : 0.f, cb = EUCLID ? coef[size_t(q) * 4 + 1] : 0.f,
              cc = EUCLID ? coef[size_t(q) * 4 + 2] : 0.f;
  const float step = qstep ? __ldg(qstep + q) : 0.f;
  auto coarse = [&](int y) { return qstep ? float(y) * step : __int_as_float(y); };
  auto rank_key = [&](const int2& e) {
    const float u_ = coarse(e.y);
    if (!EUCLID) return u_;
    const __nv_bfloat16* pr = plane + size_t(e.x) * plane_dim + dim + 3;
    const float err = fmaf(ca, __bfloat162float(pr[0]), fmaf(cb, __bfloat162float(pr[1]), cc * __bfloat162float(pr[2])));
    return u_ - 2.0001f * err;
  };
  // (a) this warp's k best coarse scores: lane-local top-K over its slices, then k rounds of warp arg-max
  float sc[K];
  int32_t ix[K];
#pragma unroll
  for (int j = 0; j < K; ++j) { sc[j] = -INFINITY; ix[j] = 0x7fffffff; }
  for (int c0 = w * 32 + lane; c0 < n; c0 += 4 * kSelectWarps * 32) {
    int2 e[4];
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      const int c = c0 + u * kSelectWarps * 32;
      e[u] = c < n ? mine[c] : make_int2(0x7fffffff, __float_as_int(-INFINITY));
    }
#pragma unroll
    for (int u = 0; u < 4; ++u)
      if (c0 + u * kSelectWarps * 32 < n) lane_insert<K>(sc, ix, rank_key(e[u]), e[u].x);
  }
  for (int j = 0; j < k; ++j) {
    float bs; int32_t br;
    warp_pop_best<K>(sc, ix, lane, -INFINITY, &bs, &br);
    if (lane == 0) { top_s[w][j] = bs; top_r[w][j] = br; }
  }
  __syncthreads();

  // tau = k-th best of the 4 x k warp winners (every warp folds them: no second barrier for a broadcast)
#pragma unroll
  for (int j = 0; j < K; ++j) { sc[j] = -INFINITY; ix[j] = 0x7fffffff; }
  for (int c = lane; c < kSelectWarps * k; c += 32) {
    const int ww = c / k, j = c - ww * k;
    lane_insert<K>(sc, ix, top_s[ww][j], top_r[ww][j]);
  }
  float tau = -INFINITY;
  float top_sc = 0.f; int32_t top_ix = -1;     // lane j keeps the j-th coarse winner (TC_BF16 output)
  for (int j = 0; j < k; ++j) {
    float bs; int32_t br;
    warp_pop_best<K>(sc, ix, lane, -INFINITY, &bs, &br);
    if (lane == j) { top_sc = bs; top_ix = br == 0x7fffffff ? -1 : br; }
    tau = bs;                                   // -inf when fewer than k candidates exist: keep all
  }

  if (!rescore) {
    // bf16 gallery mode: report the coarse scores themselves (own tolerance, DESIGN.md)
    if (w == 0 && lane < k) {
      const bool filled = top_ix >= 0 && top_sc > kNoScore;
      const int64_t r_out = filled ? int64_t(top_ix) + row_offset : int64_t(kNoRow);
      const float s_out = filled ? top_sc : kNoScore;
      out_rows[size_t(q) * k + lane] = r_out;
      out_scores[size_t(q) * k + lane] = s_out;
      if (lane == 0 && out_accept) out_accept[q] = (filled && top_sc >= threshold) ? 1 : 0;
      if (x.peer_bufs)
        for (int i = 0; i < x.world; ++i) xpush_slot(x, (x.rank + 1 + i) % x.world, int64_t(q) * k + lane, r_out, s_out);
    }
    return;
  }

  const int nvec = dim >> 2;
  const float4* qq = reinterpret_cast<const float4*>(qn + size_t(q) * dim);
  // exact fp32 rescoring of keep_row[i0 .. m) into keep_sc, 2 rows per warp and round - the typical k + 3 survivors
  // occupy all four warps - with the row's 16-byte loads unrolled four deep (a 512-d row = 4 loads per lane: one DRAM
  // round trip, not four); same element -> lane mapping and summation order as the streaming scan
  auto rescore_rows = [&](int i_begin, int m_end) {
    constexpr int kRescoreRows = 2;
    for (int i0 = i_begin + w * kRescoreRows; i0 < m_end; i0 += kSelectWarps * kRescoreRows) {
      float a[kRescoreRows];
      const float4* g[kRescoreRows];
#pragma unroll
      for (int u = 0; u < kRescoreRows; ++u) {
        a[u] = 0.f;
        const int i = i0 + u < m_end ? i0 + u : i0;
        g[u] = reinterpret_cast<const float4*>(master + size_t(keep_row[i]) * dim);
      }
#pragma unroll 4
      for (int v = lane; v < nvec; v += 32) {
        const float4 y = __ldg(qq + v);
        float4 x[kRescoreRows];
#pragma unroll
        for (int u = 0; u < kRescoreRows; ++u) x[u] = __ldg(g[u] + v);
#pragma unroll
        for (int u = 0; u < kRescoreRows; ++u) {
          if (EUCLID) {
            float d;
            d = x[u].x - y.x; a[u] = fmaf(d, d, a[u]); d = x[u].y - y.y; a[u] = fmaf(d, d, a[u]);
            d = x[u].z - y.z; a[u] = fmaf(d, d, a[u]); d = x[u].w - y.w; a[u] = fmaf(d, d, a[u]);
          } else {
            a[u] = fmaf(x[u].x, y.x, a[u]); a[u] = fmaf(x[u].y, y.y, a[u]);
            a[u] = fmaf(x[u].z, y.z, a[u]); a[u] = fmaf(x[u].w, y.w, a[u]);
          }
        }
      }
#pragma unroll
      for (int u = 0; u < kRescoreRows; ++u) {
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) a[u] += __shfl_xor_sync(0xffffffffu, a[u], o);
        if (lane == 0 && i0 + u < m_end) keep_sc[i0 + u] = EUCLID ? -a[u] : a[u];
      }
    }
  };

  // (b) cosine: rescore the m0 <= k coarse winners first (every warp holds them in lanes 0..k-1); keep threshold
  //     tau_e - eps.  Euclidean: keep U >= tau (the lower-bound ranking above).
  int m0 = 0;
  float keep_thr = tau;
  if (!EUCLID) {
    m0 = __popc(__ballot_sync(0xffffffffu, lane < k && top_ix >= 0));
    if (w == 0 && lane < m0) keep_row[lane] = top_ix;
    __syncthreads();
    rescore_rows(0, m0);
    __syncthreads();
    float te = m0 < k ? -INFINITY : INFINITY;
    for (int i = 0; i < m0; ++i) { const float x = keep_sc[i]; te = fminf(te, x == x ? x : -INFINITY); }
    keep_thr = te - (eps ? __ldg(eps + q) : kCoarseEps);
  }
  // compact the other rows that can still be in the true top-k (their order is irrelevant: the final order below
  // is total) behind the m0 rescored ones
  for (int c0 = w * 32; c0 < n; c0 += 4 * kSelectWarps * 32) {     // 4 independent loads per lane per round
    int2 e[4];
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      const int c = c0 + u * kSelectWarps * 32 + lane;
      e[u] = c < n ? mine[c] : make_int2(-1, 0);
    }
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      const float sv = EUCLID ? __int_as_float(e[u].y) : coarse(e[u].y);
      bool kp = (c0 + u * kSelectWarps * 32 + lane < n) && sv >= keep_thr;
      if (kp)
        for (int i = 0; i < m0; ++i) kp &= keep_row[i] != e[u].x;     // already rescored
      const unsigned bal = __ballot_sync(0xffffffffu, kp);
      if (bal) {
        int base = 0;
        if (lane == 0) base = atomicAdd(&s_m, __popc(bal));
        base = __shfl_sync(0xffffffffu, base, 0);
        const int pos = m0 + base + __popc(bal & ((1u << lane) - 1));
        if (kp && pos < kMaxKeep) keep_row[pos] = e[u].x;
      }
    }
  }
  __syncthreads();
  int m = m0 + s_m;
  const bool overflow = m > kMaxKeep;            // too many survivors: rescored in part, then redone by the fallback
  if (overflow) m = kMaxKeep;

  // (c) exact fp32 rescoring of the rest
  rescore_rows(m0, m);
  __syncthreads();
  if (w != 0) return;

  // (d) final order (score desc, row asc) over the m exact scores; lane-local lists + warp merge
  const float sentinel = EUCLID ? -INFINITY : kNoScore;     // the exact scan's initial best
#pragma unroll
  for (int j = 0; j < K; ++j) { sc[j] = sentinel; ix[j] = 0x7fffffff; }
  for (int c = lane; c < m; c += 32) {
    const float s = keep_sc[c];
    if (s > sentinel) lane_insert<K>(sc, ix, s, keep_row[c]);   // scores <= -1 (d = inf) and NaN never match
  }
  for (int j = 0; j < k; ++j) {
    float bs; int32_t br;
    warp_pop_best<K>(sc, ix, lane, sentinel, &bs, &br);
    const bool filled = br != 0x7fffffff;
    const int64_t r_out = filled ? int64_t(br) + row_offset : int64_t(kNoRow);
    const float s_out = EUCLID ? (filled ? __fsqrt_rn(fmaxf(-bs, 0.f)) : INFINITY) : (filled ? bs : kNoScore);
    if (lane == 0) {
      out_rows[size_t(q) * k + j] = r_out;
      out_scores[size_t(q) * k + j] = s_out;
      if (j == 0 && out_accept) out_accept[q] = (filled && (EUCLID ? s_out <= threshold : bs >= threshold)) ? 1 : 0;
    }
    // row-sharded gallery: this slot is final - send it to every rank now (lane p -> rank p), unless the
    // query goes to the exact fallback, whose result the exchange kernel pushes
    if (x.peer_bufs && !overflow)
      for (int pr = lane; pr < x.world; pr += 32) xpush_slot(x, pr, int64_t(q) * k + j, r_out, s_out);
  }
  if (overflow && lane == 0) flagged[atomicAdd(n_flagged, 1)] = q;
}

// ------------------------------------------------------------------------------------------ host side
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static int get_encode(EncodeTiledFn* out) {
  static EncodeTiledFn fn = nullptr;
  if (!fn) {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult qres;
    FRG_CUDA(cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &qres));
    if (!p || qres != cudaDriverEntryPointSuccess) { set_error("cuTensorMapEncodeTiled not available"); return FRG_ERR_CUDA; }
    fn = reinterpret_cast<EncodeTiledFn>(p);
  }
  *out = fn;
  return FRG_OK;
}

// 2-D bf16 row-major [rows][dim] view with a row pitch (bytes), box = box_k x box_rows; box_k = 64 with the
// 128B swizzle (a k-block) or 16 with the 32B swizzle (the Euclidean pad block).  i8: an int8 view, box = one
// 128-byte k-block of 128 elements, 128B swizzle.
static int make_map(CUtensorMap* map, const void* ptr, int dim, int64_t rows, size_t pitch_bytes, int box_rows,
                    int box_k = kBlockK, bool i8 = false) {
  EncodeTiledFn enc = nullptr;
  FRG_CHECK(get_encode(&enc));
  if (i8) box_k = kBlockKI8;
  cuuint64_t gdim[2] = {cuuint64_t(dim), cuuint64_t(rows)};
  cuuint64_t gstride[1] = {cuuint64_t(pitch_bytes)};
  cuuint32_t box[2] = {cuuint32_t(box_k), cuuint32_t(box_rows)};
  cuuint32_t estr[2] = {1, 1};
  CUresult r = enc(map, i8 ? CU_TENSOR_MAP_DATA_TYPE_UINT8 : CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, const_cast<void*>(ptr),
                   gdim, gstride, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                   (i8 || box_k == kBlockK) ? CU_TENSOR_MAP_SWIZZLE_128B : CU_TENSOR_MAP_SWIZZLE_32B,
                   CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) { set_error("cuTensorMapEncodeTiled failed (%d): rows=%lld pitch=%zu", int(r), (long long)rows, pitch_bytes); return FRG_ERR_CUDA; }
  return FRG_OK;
}

static int gcd_int(int a, int b) { while (b) { int t = a % b; a = b; b = t; } return a; }

// dynamic shared memory: [alignment slack 1 KB][query tile][ring][barriers 256 B].  Six 16 KB stages
// (96 KB in flight per SM) already reach the HBM peak; a deeper ring beside shorter query tiles
// (up to 12 stages) measured no faster at dim 128 / 256 - those shapes are bound by the TMEM read
// rate of the epilogue (DESIGN.md section 4.2), not by bytes in flight.
constexpr size_t kSmemLimit = 227 * 1024;
constexpr int kStages = 6;
// q_row_bytes: bytes of one query row of the resident tile (dim x 2 bf16, dim x 1 int8)
static size_t tc_smem_bytes(int q_row_bytes) {
  return size_t(kTileQ) * q_row_bytes + size_t(kStages) * kStageBytes + 256 + 1024;
}
static_assert(kStages <= kMaxStages && size_t(kTileQ) * 512 * 2 + size_t(kStages) * kStageBytes + 256 + 1024 <= kSmemLimit,
              "the ring must fit beside the largest query tile (512 bf16 columns)");

int tc_supported(int dim, int metric, const char** why) {
  // the tiles take any multiple of 64 up to 512 columns; the exact pass behind the filter (rescoring
  // order, overflow fallback) is the streaming scan's, which is built for 128 / 256 / 512
  if (dim != 128 && dim != 256 && dim != 512) { *why = "tensor-core variants are built for dim 128, 256 and 512"; return 0; }
  if (metric == FRG_METRIC_EUCLIDEAN && dim + kEuclidQPad > 512) {
    *why = "the Euclidean tensor-core filter needs dim <= 448 (one more k-block carries the norm terms)";
    return 0;
  }
  return 1;
}

struct TcPlan {
  bool pair;              // CTA-pair kernels (F > 128)
  bool fused;             // pre-pass folded into the filter kernel (probe tile + published group maxima)
  int qtiles, stride, chunks_pre, chunks_main, kreg, seg, stage_entries;
  size_t off_keys, off_cnt, off_cand, off_dense, off_flag, off_floor, total;
};

// FUSED: share of every CTA's chunk probed before the floor is derived (1/64; larger probes, up to 1/8, measured no
// faster, DESIGN.md section 4.2)
constexpr int kProbeDiv = 64;

bool tc_uses_pairs(int nq);

static int reg_k(int k) { return k == 1 ? 1 : (k <= 4 ? 4 : (k <= 8 ? 8 : 16)); }

// dim < 0: Euclidean plane (|dim| columns).  Its probe and filter phases need DIFFERENT query images (lower / upper
// bounds of the exact score), so the pre-pass is never folded into the filter kernel there.
// Range search (range = true): no pre-pass, and a fixed dense list of kRangeBudget entries per query instead of one
// sized from k (DESIGN.md section 7.3).
// i8: the int8 filter - pre-pass at most every 16th tile, floor from i8_floor_kernel, never fused.
static void tc_plan(int64_t rows, int dim, int nq, int k, int sm_count, TcPlan* pl, bool range = false, bool i8 = false) {
  const bool euclid_plane = dim < 0;
  pl->qtiles = (nq + kTileQ - 1) / kTileQ;
  pl->pair = tc_uses_pairs(nq);
  if (pl->pair) pl->qtiles = (pl->qtiles + 1) & ~1;      // clusters of 2 along x; a padding tile holds no query
  // Fusing the pre-pass into the filter kernel saves a launch and a query-tile reload but probes a
  // smaller sample (one tile per CTA), i.e. a looser floor and more candidates: measured on B200 it
  // wins for a handful of queries (F = 1: 198 vs 208 us) and loses from F = 64 on (F = 1024: 814 vs
  // 735 us).
  pl->fused = !euclid_plane && !range && !i8 && nq <= 8;
  const int tile_rows = pl->pair ? 2 * kTileR : kTileR;
  // pre-pass sample: every stride-th 128-row tile, stride the largest power of two <= 64 (int8: <= 16) that still
  // leaves >= 16 K sampled rows
  const int max_stride = i8 ? 16 : 64;
  int stride = 1;
  while (stride < max_stride && rows / (stride * 2) >= 16384) stride *= 2;
  pl->stride = stride;
  const int tiles_all = int((rows + tile_rows - 1) / tile_rows);
  auto chunks_for = [&](int tiles) {
    // (query tiles x chunks) a whole number of waves over the SMs (SM pairs in pair mode)
    const int units = pl->pair ? sm_count / 2 : sm_count;
    const int cols = pl->pair ? pl->qtiles / 2 : pl->qtiles;
    int c = units / gcd_int(units, cols);
    if (c > tiles) c = tiles;
    return c < 1 ? 1 : c;
  };
  // pre-pass: a few tiles per CTA, so the fixed cost of a CTA (query-tile load, TMEM allocation, the
  // group-max atomics at its end) matters - never more than ONE wave (1024 queries: 72 CTA pairs with
  // 7 tiles each instead of 148 pairs in two waves of 3-4)
  {
    const int units = pl->pair ? sm_count / 2 : sm_count;
    const int cols = pl->pair ? pl->qtiles / 2 : pl->qtiles;
    const int tiles_pre = (tiles_all + stride - 1) / stride;
    int c = cols <= units ? units / cols : 1;
    if (c > tiles_pre) c = tiles_pre;
    pl->chunks_pre = c < 1 ? 1 : c;
  }
  pl->chunks_main = chunks_for(tiles_all);
  pl->kreg = reg_k(k);
  // Expected candidates per query ~ 2 * stride * Gamma(k): the k-th best of a 1/stride sample sits
  // at tail mass Gamma(k)/n_view, and the 2*eps widening about doubles the count at dim 512.  Room for
  // mean + ~10 sigma keeps the overflow probability negligible; the exact fallback covers the rest.
  // (x1.5: the group-max floor is a little looser than an exact k-th best of the sample)
  // int8 filter: its eps is ~4x bf16's, but its floor e_k - eps drops the second eps and the group-max error; the
  // CPU rehearsal of the synthetic gallery (tools/int8_band_sim.py, 1 M x 512, k = 5, 128 queries) gives 399 / 791 /
  // 815 (median / p99 / max) candidates per query at stride 16 and 218 / 468 / 534 at stride 8, against 1793 and 896
  // entries from the same formula (profiles/r04_int8_band_sim.json).
  // fused: the probe is 1/64 of every chunk, or one tile per CTA if that is more
  int eff_stride = stride;
  if (pl->fused) {
    const int64_t probe_rows = int64_t((tiles_all / pl->chunks_main + kProbeDiv - 1) / kProbeDiv) * pl->chunks_main * tile_rows;
    eff_stride = int(rows / (probe_rows > 0 ? probe_rows : 1)) + 1;
    if (eff_stride > 64) eff_stride = 64;
  }
  int stage_entries = int(3.0 * eff_stride * (k + 10.0 * sqrt(double(k)) + 10.0));
  if (stage_entries < 256) stage_entries = 256;
  if (stage_entries > 8192) stage_entries = 8192;
  if (range) stage_entries = kRangeBudget;
  pl->stage_entries = stage_entries;
  // private segments: one per (query, chunk, column half); x2 headroom for imbalance across them
  const int nseg = pl->chunks_main * (kEpiWarps / 4);
  int seg = (2 * stage_entries + nseg - 1) / nseg;
  if (seg < 12) seg = 12;
  pl->seg = seg;
  size_t off = 0;
  auto take = [&](size_t bytes) { size_t o = off; off = (off + bytes + 255) & ~size_t(255); return o; };
  pl->off_keys = take(size_t(nq) * kGroups * (i8 ? 8 : 4));
  pl->off_cnt = take(size_t(nq) * 4);
  pl->off_cand = take(size_t(nq) * nseg * seg * 8);
  pl->off_dense = take(size_t(nq) * stage_entries * 8);
  pl->off_flag = take(size_t(nq) * 4 + 12);    // flagged[nq], count, ticket, probe-arrival counter
  pl->off_floor = take(i8 ? size_t(nq) * 4 : 0);
  pl->total = off;
}

template <int MODE, bool MASKED, bool PAIR, bool I8, bool GROUPED = false>
static int launch_tc_scan(const CUtensorMap& qm, const CUtensorMap& gm, const CUtensorMap& pm, const TcScanParams& p,
                          int qtiles, int chunks, cudaStream_t st) {
  const size_t smem = tc_smem_bytes(I8 ? p.dim : 2 * p.dim);
  auto kern = tc_scan_kernel<MODE, MASKED, PAIR, I8, GROUPED>;
  FRG_CUDA(func_attr_once(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, int(kSmemLimit)));
  cudaLaunchConfig_t cfg{};
  cfg.gridDim = dim3(qtiles, chunks);
  cfg.blockDim = dim3(kTcThreads);
  cfg.dynamicSmemBytes = smem;
  cfg.stream = st;
  cudaLaunchAttribute attr[2];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = PAIR ? 2 : 1;
  attr[0].val.clusterDim.y = 1;
  attr[0].val.clusterDim.z = 1;
  attr[1].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[1].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 2;
  FRG_CUDA(cudaLaunchKernelEx(&cfg, kern, qm, gm, pm, p));
  note_launch(nullptr);
  return FRG_OK;
}

template <int MODE, bool I8 = false>
static int launch_tc_scan_m(bool masked, bool pair, const CUtensorMap& qm, const CUtensorMap& gm,
                            const CUtensorMap& pm, const TcScanParams& p, int qtiles, int chunks, cudaStream_t st) {
  if (pair)
    return masked ? launch_tc_scan<MODE, true, true, I8>(qm, gm, pm, p, qtiles, chunks, st)
                  : launch_tc_scan<MODE, false, true, I8>(qm, gm, pm, p, qtiles, chunks, st);
  return masked ? launch_tc_scan<MODE, true, false, I8>(qm, gm, pm, p, qtiles, chunks, st)
                : launch_tc_scan<MODE, false, false, I8>(qm, gm, pm, p, qtiles, chunks, st);
}

bool tc_uses_pairs(int nq) { return (nq + kTileQ - 1) / kTileQ >= 2; }

// rows the plan is made for: the window's, or (tile list in use) listed tiles x rows per tile
int64_t tc_effective_rows(const GalleryWindow* s, int nq, cudaStream_t st, const int32_t** list, int* n_list) {
  *list = nullptr; *n_list = 0;
  if (!s->owner || !s->want_tile_list) return s->rows;
  const int gran = tc_uses_pairs(nq) ? 2 * kTileR : kTileR;
  const int32_t* l = nullptr; int n = 0;
  if (store_tile_list(s->owner, s->list_tenant, gran, st, &l, &n) != FRG_OK) return -1;
  if (!l) return s->rows;                 // not worth it / not known: the masked scan of the window
  *list = l; *n_list = n;
  return int64_t(n) * gran;
}

size_t tc_workspace_bytes(int64_t rows, int dim, int nq, int k, int sm_count, bool range, bool i8) {
  TcPlan pl;
  tc_plan(rows, dim, nq, k, sm_count, &pl, range, i8);
  return pl.total;
}

// the pieces of the workspace the query-prep kernel initialises (group keys := "nothing seen", counters := 0)
void tc_workspace_init_targets(int64_t rows, int dim, int nq, int k, int sm_count, unsigned char* ws,
                               void** keys, int** cand_total, int** n_flagged, bool range, bool i8) {
  TcPlan pl;
  tc_plan(rows, dim, nq, k, sm_count, &pl, range, i8);
  *keys = ws + pl.off_keys;
  *cand_total = reinterpret_cast<int*>(ws + pl.off_cnt);
  *n_flagged = reinterpret_cast<int*>(ws + pl.off_flag) + nq;
}

// qn / qb: normalised fp32 queries and their bf16 image [nq][dim]; ws: tc_workspace_bytes() of scratch.
// Leaves the overflowed queries in (flagged, n_flagged) for the caller's exact fallback pass.
int launch_tc_match(const GalleryWindow* s, int metric, const float* qn, const __nv_bfloat16* qb, const float* eps,
                    int nq, int k, int32_t tenant, bool rescore, float threshold, int64_t row_offset,
                    unsigned char* ws, int sm_count, const XPush& push, int64_t* out_rows, float* out_scores,
                    uint8_t* out_accept, int** flagged_out, int** n_flagged_out, cudaStream_t st,
                    int64_t plan_rows, const int32_t* tile_list, int n_list, const __nv_bfloat16* qb_prepass,
                    const float* coef, const int8_t* qi8, const float* qstep) {
  const bool euclid = metric == FRG_METRIC_EUCLIDEAN;
  const bool i8 = s->plane8 != nullptr;
  if (euclid && (!qb_prepass || !coef)) { set_error("tc_match: the Euclidean filter needs both query images"); return FRG_ERR_INVALID; }
  if (euclid ? (!s->plane || s->plane_dim == s->dim) : (i8 ? !qi8 || !qstep || !eps || !rescore : !s->plane)) {
    set_error("tc_match: metric / query image does not fit the store's scan plane");
    return FRG_ERR_UNSUPPORTED;
  }
  // columns of the query tile: dim, or dim + kEuclidQPad (its last k-block meets the plane's 16-column pad block)
  const int kdim = euclid ? s->dim + kEuclidQPad : s->dim;
  const size_t pitch = i8 ? size_t(s->dim) : size_t(s->plane_dim) * 2;
  // (tile_list: a tenant-filtered call whose window is mostly other tenants' rows walks only the tiles that hold
  // rows of the tenant; everything is planned for plan_rows = listed tiles x rows per tile)
  TcPlan pl;
  tc_plan(plan_rows, euclid ? -s->dim : s->dim, nq, k, sm_count, &pl, false, i8);
  uint32_t* keys = reinterpret_cast<uint32_t*>(ws + pl.off_keys);
  int* cnt = reinterpret_cast<int*>(ws + pl.off_cnt);
  int2* cand = reinterpret_cast<int2*>(ws + pl.off_cand);
  int2* dense = reinterpret_cast<int2*>(ws + pl.off_dense);
  int* flagged = reinterpret_cast<int*>(ws + pl.off_flag);
  int* n_flagged = flagged + nq;
  *flagged_out = flagged;
  *n_flagged_out = n_flagged;
  const bool masked = tenant >= 0 || s->maybe_dead;

  CUtensorMap qm, qm_pre, gm_full, pm;
  if (i8) FRG_CHECK(make_map(&qm, qi8, kdim, nq, size_t(kdim), kTileQ, kBlockK, true));
  else FRG_CHECK(make_map(&qm, qb, kdim, nq, size_t(kdim) * 2, kTileQ));
  if (euclid) FRG_CHECK(make_map(&qm_pre, qb_prepass, kdim, nq, size_t(kdim) * 2, kTileQ));   // lower-bound image
  else qm_pre = qm;
  if (i8) FRG_CHECK(make_map(&gm_full, s->plane8, s->dim, s->rows, pitch, kTileR, kBlockK, true));
  else FRG_CHECK(make_map(&gm_full, s->plane, s->dim, s->rows, pitch, kTileR));   // box = one CTA's half
  if (euclid) FRG_CHECK(make_map(&pm, s->plane + s->dim, kEuclidPad, s->rows, pitch, kTileR, kEuclidPad));
  else pm = gm_full;                                                          // never dereferenced (p.pad == 0)

  TcScanParams p{};
  p.fault = s->fault;
  p.tile_list = tile_list; p.n_list = n_list;
  p.eps = eps; p.none_score = euclid ? kEuclidNone : kNoScore; p.pad = euclid ? 1 : 0;
  p.stages = kStages;
  p.dim = kdim; p.nq = nq; p.tenant = tenant; p.tags = s->tags;
  p.n_rows = int(s->rows); p.group_key = keys; p.k = k;
  p.seg = pl.seg; p.cand = cand; p.cand_total = cnt; p.dense = dense; p.dense_cap = pl.stage_entries;
  int rc;
  if (i8) {
    // 1. int8 pre-pass over the sampled tiles: (s32 product, row) of every row group's best sampled row
    p.group_key64 = reinterpret_cast<unsigned long long*>(ws + pl.off_keys);
    p.floor = reinterpret_cast<float*>(ws + pl.off_floor);
    p.qstep = qstep;
    p.tile_scale = pl.stride;
    profile_begin(st, kStagePrepass);
    FRG_CHECK((launch_tc_scan_m<kModeGroupMax, true>(masked, pl.pair, qm, gm_full, gm_full, p, pl.qtiles, pl.chunks_pre, st)));
    profile_end(st, 1);
    // 2. exact floor e_k - eps from the k best group winners
    profile_begin(st, kStageFloor);
    FRG_CUDA(launch_kernel(i8_floor_kernel, dim3((nq + 3) / 4), dim3(128), 0, st, p.group_key64, nq, k, s->dim,
                           qn, s->master, eps, const_cast<float*>(p.floor)));
    note_launch(nullptr);
    profile_end(st, 1);
    // 3. filter over the whole plane against the integer floor
    p.tile_scale = 1;
    profile_begin(st, kStageDominant);
    rc = launch_tc_scan_m<kModeFilter, true>(masked, pl.pair, qm, gm_full, gm_full, p, pl.qtiles, pl.chunks_main, st);
    FRG_CHECK(rc);
    profile_end(st, 1);
  } else if (pl.fused) {
    // 1+2. ONE kernel: every CTA probes its first tile, publishes the group maxima, derives L[q] from
    // what all CTAs published, filters the rest of its chunk and finally the probe tile itself
    p.tile_scale = 1;
    p.probe_div = kProbeDiv;
    p.arrive = n_flagged + 2;
    {
      // the first wave holds min(all CTAs, one per SM): later waves find the counter already there
      const int ctas = pl.qtiles * pl.chunks_main;
      p.arrive_target = ctas < sm_count ? ctas : sm_count;
    }
    profile_begin(st, kStageDominant);
    rc = launch_tc_scan_m<kModeFused>(masked, pl.pair, qm, gm_full, pm, p, pl.qtiles, pl.chunks_main, st);
    FRG_CHECK(rc);
    profile_end(st, 1);
  } else {
    // 1. pre-pass over the sampled tiles
    p.tile_scale = pl.stride;
    profile_begin(st, kStagePrepass);
    FRG_CHECK(launch_tc_scan_m<kModeGroupMax>(masked, pl.pair, qm_pre, gm_full, pm, p, pl.qtiles, pl.chunks_pre, st));
    profile_end(st, 1);
    // 2. filter over the whole plane
    p.tile_scale = 1;
    profile_begin(st, kStageDominant);
    rc = launch_tc_scan_m<kModeFilter>(masked, pl.pair, qm, gm_full, pm, p, pl.qtiles, pl.chunks_main, st);
    FRG_CHECK(rc);
    profile_end(st, 1);
  }
  // 3. select + exact rescoring
  profile_begin(st, kStageSelect);
  const int grid = nq;                                   // one CTA per query
  const int rs = rescore ? 1 : 0;
#define FRG_SELECT_M(KK, EU)                                                                                    \
  FRG_CUDA(func_attr_once(select_rescore_kernel<KK, EU>, cudaFuncAttributePreferredSharedMemoryCarveout, 100)); \
  FRG_CUDA(launch_kernel(select_rescore_kernel<KK, EU>, dim3(grid), dim3(kSelectWarps * 32), 0, st, dense, \
      cnt, pl.stage_entries, nq, k, s->dim, qn, eps, s->plane, s->plane_dim, coef, i8 ? qstep : nullptr,         \
      s->master, rs, threshold,                                                                                    \
      row_offset, out_rows, out_scores,                                                                             \
      out_accept, flagged, n_flagged, push))
#define FRG_SELECT(KK)                                                                                          \
  if (euclid) { FRG_SELECT_M(KK, true); } else { FRG_SELECT_M(KK, false); }
  switch (pl.kreg) {
    case 1: FRG_SELECT(1); break;
    case 4: FRG_SELECT(4); break;
    case 8: FRG_SELECT(8); break;
    default: FRG_SELECT(16); break;
  }
#undef FRG_SELECT
#undef FRG_SELECT_M
  note_launch(nullptr);
  FRG_CUDA(cudaGetLastError());
  profile_end(st, 1);
  return FRG_OK;
}


// ------------------------------------------------------------------------------------------ range search
// The filter's floor for a range search is the fixed threshold - eps[q] (rigorous: |S - s| <= eps[q], so every row
// with exact s >= threshold has S >= the floor), not a sampled floor: no pre-pass runs.  It goes into the per-query
// floor array the int8 filter's prologue reads (eps[q] already covers the fp32 rounding of the subtraction).
__global__ void __launch_bounds__(256)
range_floor_kernel(const float* __restrict__ eps, float threshold, float* __restrict__ floor_out, int nq) {
  pdl_wait();             // the query prep's eps[]
  pdl_trigger();
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < nq) floor_out[i] = threshold - __ldg(eps + i);
}

// ONE CTA (4 warps) per query over the dense candidate list of a range-mode filter: every candidate is rescored
// exactly in fp32 from the master (same element -> lane mapping and xor 16..1 reduction as the streaming scan, so
// the scores are bit-identical to launch_range_scan's), the survivors of the threshold rule are packed as
// (row << 32 | score bits) in shared memory, sorted by row (bitonic) and the first max_hits written in gallery order.
__global__ void __launch_bounds__(kSelectWarps * 32)
range_select_kernel(const int2* __restrict__ dense, const int* __restrict__ cand_total, int dense_cap, int dim,
                    const float* __restrict__ qn, const float* __restrict__ master, float threshold, int strict,
                    int max_hits, int64_t row_offset, int64_t* __restrict__ out_counts,
                    int64_t* __restrict__ out_rows, float* __restrict__ out_scores, int* __restrict__ flagged,
                    int* __restrict__ n_flagged) {
  extern __shared__ unsigned long long hits[];        // [pow2 >= dense_cap]
  __shared__ int s_m;
  const int lane = threadIdx.x & 31;
  const int w = threadIdx.x >> 5;
  const int q = blockIdx.x;
  pdl_wait();             // the filter kernel's candidate lists
  pdl_trigger();
  const int total = cand_total[q];
  if (total > dense_cap) {                           // also set by a poisoned total (segment overflow)
    if (threadIdx.x == 0) flagged[atomicAdd(n_flagged, 1)] = q;
    return;
  }
  if (threadIdx.x == 0) s_m = 0;
  __syncthreads();
  const int2* mine = dense + size_t(q) * dense_cap;
  const int nvec = dim >> 2;
  const float4* qq = reinterpret_cast<const float4*>(qn + size_t(q) * dim);
  for (int c = w; c < total; c += kSelectWarps) {
    const int row = mine[c].x;
    const float4* g = reinterpret_cast<const float4*>(master + size_t(row) * dim);
    float a = 0.f;
#pragma unroll 4
    for (int v = lane; v < nvec; v += 32) {
      const float4 x = __ldg(g + v), y = __ldg(qq + v);
      a = fmaf(x.x, y.x, a); a = fmaf(x.y, y.y, a); a = fmaf(x.z, y.z, a); a = fmaf(x.w, y.w, a);
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) a += __shfl_xor_sync(0xffffffffu, a, o);
    const bool pass = strict ? (a > threshold) : (a >= threshold);      // false for NaN
    if (lane == 0 && pass) hits[atomicAdd(&s_m, 1)] = (uint64_t(uint32_t(row)) << 32) | __float_as_uint(a);
  }
  __syncthreads();
  const int m = s_m;
  int n2 = 1;
  while (n2 < m) n2 <<= 1;
  for (int i = m + threadIdx.x; i < n2; i += blockDim.x) hits[i] = ~0ull;
  __syncthreads();
  // rows are distinct: ascending keys = gallery order
  for (int kk = 2; kk <= n2; kk <<= 1) {
    for (int j = kk >> 1; j > 0; j >>= 1) {
      for (int i = threadIdx.x; i < n2; i += blockDim.x) {
        const int ij = i ^ j;
        if (ij > i) {
          const unsigned long long x = hits[i], y = hits[ij];
          if ((x > y) == ((i & kk) == 0)) { hits[i] = y; hits[ij] = x; }
        }
      }
      __syncthreads();
    }
  }
  for (int i = threadIdx.x; i < max_hits; i += blockDim.x) {
    const bool filled = i < m;
    out_rows[size_t(q) * max_hits + i] = filled ? int64_t(hits[i] >> 32) + row_offset : int64_t(kNoRow);
    out_scores[size_t(q) * max_hits + i] = filled ? __uint_as_float(uint32_t(hits[i])) : kNoScore;
  }
  if (threadIdx.x == 0) out_counts[q] = m;
}

int launch_tc_range(const GalleryWindow* s, const float* qn, const int8_t* qi8, const float* qstep, const float* eps,
                    int nq, int max_hits, int32_t tenant, float threshold, bool strict, int64_t row_offset,
                    unsigned char* ws, int sm_count, int64_t* out_counts, int64_t* out_rows, float* out_scores,
                    int** flagged_out, int** n_flagged_out, cudaStream_t st, int64_t plan_rows,
                    const int32_t* tile_list, int n_list) {
  if (!s->plane8) { set_error("tc_range: the store has no int8 scan plane"); return FRG_ERR_UNSUPPORTED; }
  TcPlan pl;
  tc_plan(plan_rows, s->dim, nq, 1, sm_count, &pl, true, true);
  int* cnt = reinterpret_cast<int*>(ws + pl.off_cnt);
  int2* cand = reinterpret_cast<int2*>(ws + pl.off_cand);
  int2* dense = reinterpret_cast<int2*>(ws + pl.off_dense);
  int* flagged = reinterpret_cast<int*>(ws + pl.off_flag);
  int* n_flagged = flagged + nq;
  *flagged_out = flagged;
  *n_flagged_out = n_flagged;
  const bool masked = tenant >= 0 || s->maybe_dead;

  CUtensorMap qm, gm;
  FRG_CHECK(make_map(&qm, qi8, s->dim, nq, size_t(s->dim), kTileQ, kBlockK, true));
  FRG_CHECK(make_map(&gm, s->plane8, s->dim, s->rows, size_t(s->dim), kTileR, kBlockK, true));

  TcScanParams p{};
  p.fault = s->fault;
  p.tile_list = tile_list; p.n_list = n_list;
  p.eps = eps; p.none_score = kNoScore; p.pad = 0; p.stages = kStages;
  p.dim = s->dim; p.nq = nq; p.tenant = tenant; p.tags = s->tags;
  p.n_rows = int(s->rows); p.k = 1;
  p.floor = reinterpret_cast<float*>(ws + pl.off_floor); p.qstep = qstep;
  p.seg = pl.seg; p.cand = cand; p.cand_total = cnt; p.dense = dense; p.dense_cap = pl.stage_entries;
  p.tile_scale = 1;
  profile_begin(st, kStageFloor);
  FRG_CUDA(launch_kernel(range_floor_kernel, dim3((nq + 255) / 256), dim3(256), 0, st, eps, threshold,
                         const_cast<float*>(p.floor), nq));
  note_launch(nullptr);
  profile_end(st, 1);
  profile_begin(st, kStageDominant);
  FRG_CHECK((launch_tc_scan_m<kModeFilter, true>(masked, pl.pair, qm, gm, gm, p, pl.qtiles, pl.chunks_main, st)));
  profile_end(st, 1);

  profile_begin(st, kStageSelect);
  int n2 = 1;
  while (n2 < pl.stage_entries) n2 <<= 1;
  const size_t smem = size_t(n2) * sizeof(unsigned long long);
  FRG_CUDA(func_attr_once(range_select_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, int(smem)));
  FRG_CUDA(launch_kernel(range_select_kernel, dim3(nq), dim3(kSelectWarps * 32), smem, st, dense, cnt,
                         pl.stage_entries, s->dim, qn, s->master, threshold, strict ? 1 : 0, max_hits, row_offset,
                         out_counts, out_rows, out_scores, flagged, n_flagged));
  note_launch(nullptr);
  FRG_CUDA(cudaGetLastError());
  profile_end(st, 1);
  return FRG_OK;
}

// ------------------------------------------------------------------------------------------ per-query tenants
static_assert(kTileR == kTcTileRows, "the host plans tile sources in kTcTileRows-row tiles");

// rows -> original query position: sorted[i] = q[perm[i]]
__global__ void __launch_bounds__(128)
gather_queries_kernel(const float* __restrict__ q, const int32_t* __restrict__ perm, int nq, int dim,
                      float* __restrict__ out) {
  pdl_wait();
  pdl_trigger();
  const int lane = threadIdx.x & 31;
  const int w = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  if (w >= nq) return;
  const float4* src = reinterpret_cast<const float4*>(q + size_t(__ldg(perm + w)) * dim);
  float4* dst = reinterpret_cast<float4*>(out + size_t(w) * dim);
  for (int v = lane; v < (dim >> 2); v += 32) dst[v] = __ldg(src + v);
}

// results of sorted query i -> the caller's slot perm[i]
__global__ void __launch_bounds__(256)
scatter_results_kernel(const int64_t* __restrict__ rows, const float* __restrict__ scores,
                       const uint8_t* __restrict__ accept, const int32_t* __restrict__ perm, int nq, int k,
                       int64_t* __restrict__ out_rows, float* __restrict__ out_scores, uint8_t* __restrict__ out_accept) {
  pdl_wait();
  pdl_trigger();
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= nq * k) return;
  const int q = i / k, j = i - q * k;
  const size_t o = size_t(__ldg(perm + q)) * k + j;
  out_rows[o] = rows[i];
  out_scores[o] = scores[i];
  if (out_accept && j == 0) out_accept[o / k] = accept[q];
}

int launch_gather_queries(const float* q, const int32_t* perm, int nq, int dim, float* out, cudaStream_t st) {
  if (nq <= 0) return FRG_OK;
  FRG_CUDA(launch_kernel(gather_queries_kernel, dim3((nq + 3) / 4), dim3(128), 0, st, q, perm, nq, dim, out));
  note_launch(nullptr);
  return FRG_OK;
}

int launch_scatter_results(const int64_t* rows, const float* scores, const uint8_t* accept, const int32_t* perm, int nq,
                           int k, int64_t* out_rows, float* out_scores, uint8_t* out_accept, cudaStream_t st) {
  if (nq <= 0) return FRG_OK;
  FRG_CUDA(launch_kernel(scatter_results_kernel, dim3((nq * k + 255) / 256), dim3(256), 0, st, rows, scores, accept,
                         perm, nq, k, out_rows, out_scores, out_accept));
  note_launch(nullptr);
  return FRG_OK;
}

// Chunks of each unit in proportion to its tiles, so that the whole grid stays near one wave of sm_count CTAs
// (at least one chunk per unit, at most one per tile).
static std::vector<int> proportional_chunks(const std::vector<int>& tiles, int sm_count) {
  int64_t total = 0;
  for (int t : tiles) total += t;
  std::vector<int> c(tiles.size(), 0);
  for (size_t i = 0; i < tiles.size(); ++i) {
    if (tiles[i] <= 0) continue;
    int64_t x = total > 0 ? int64_t(sm_count) * tiles[i] / total : 1;
    if (x < 1) x = 1;
    if (x > tiles[i]) x = tiles[i];
    c[i] = int(x);
  }
  return c;
}

// One query tile of a GROUPED grid: queries q0 .. q0 + nq - 1 (nq <= kTileQ) of src's tenant, which scan src's tiles
// with `entries` candidates per query and (pre-pass) every stride-th tile.
struct GroupUnit { const TcTenantGroup* src; int q0, nq, entries, stride; };

// The descriptors of a GROUPED filter grid (main) and, when pre != nullptr, of its pre-pass grid: each unit's tiles cut
// into chunks in proportion to its share of all tiles, its candidate segments one per (query, chunk, column half) with
// x2 headroom (as tc_plan).  Returns the candidate entries (int2) the filter grid writes.
static int64_t plan_group_ctas(const std::vector<GroupUnit>& units, int sm_count, std::vector<TcGroupCta>* pre,
                               std::vector<TcGroupCta>* main) {
  std::vector<int> tiles_main(units.size()), tiles_pre(units.size());
  for (size_t u = 0; u < units.size(); ++u) {
    tiles_main[u] = units[u].src->n_tiles;
    tiles_pre[u] = (tiles_main[u] + units[u].stride - 1) / units[u].stride;
  }
  const std::vector<int> ch_main = proportional_chunks(tiles_main, sm_count);
  const std::vector<int> ch_pre = proportional_chunks(tiles_pre, sm_count);
  int64_t cand_entries = 0;
  for (size_t u = 0; u < units.size(); ++u) {
    const TcTenantGroup& G = *units[u].src;
    if (tiles_main[u] == 0) continue;                  // an unknown tag: no rows, nothing to scan
    const int nseg = ch_main[u] * (kEpiWarps / 4);
    int seg = (2 * units[u].entries + nseg - 1) / nseg;
    if (seg < 12) seg = 12;
    TcGroupCta d{};
    d.q0 = units[u].q0; d.nq = units[u].nq; d.tenant = G.tenant; d.tile0 = G.tile0; d.n_tiles = G.n_tiles;
    d.list = G.list; d.seg = seg; d.cand0 = cand_entries;
    for (int c = 0; c < ch_main[u]; ++c) { d.chunk = c; d.chunks = ch_main[u]; d.scale = 1; main->push_back(d); }
    if (pre)
      for (int c = 0; c < ch_pre[u]; ++c) { d.chunk = c; d.chunks = ch_pre[u]; d.scale = units[u].stride; pre->push_back(d); }
    cand_entries += int64_t(kTileQ) * nseg * seg;
  }
  return cand_entries;
}

int launch_tc_match_grouped(const GalleryWindow* s, const float* q, const std::vector<int32_t>& perm,
                            const std::vector<TcTenantGroup>& groups, int k, float threshold, int64_t row_offset,
                            int sm_count, int64_t* out_rows, float* out_scores, uint8_t* out_accept, cudaStream_t st) {
  const int nq = int(perm.size());
  const int dim = s->dim;
  if (!s->plane8 || !s->master || s->rows <= 0 || s->rows > 0x7fffffff) {
    set_error("tc_match_grouped: needs a non-empty unit store with an int8 plane and an fp32 master");
    return FRG_ERR_UNSUPPORTED;
  }
  // ---- plan: query tiles of at most kTileQ queries, never across tenants
  std::vector<GroupUnit> units;
  for (int g = 0; g < int(groups.size()); ++g)
    for (int a = 0; a < groups[g].nq; a += kTileQ)
      units.push_back(GroupUnit{&groups[g], groups[g].q0 + a, groups[g].nq - a < kTileQ ? groups[g].nq - a : kTileQ, 0, 0});
  int dense_cap = 0;
  for (GroupUnit& U : units) {
    // the plan of a single-tenant match over the same tiles (tc_plan): pre-pass stride and candidate budget
    TcPlan pl;
    tc_plan(int64_t(U.src->n_tiles) * kTileR, dim, 1, k, sm_count, &pl, false, true);
    U.stride = pl.stride;
    U.entries = pl.stage_entries;
    if (pl.stage_entries > dense_cap) dense_cap = pl.stage_entries;
  }
  std::vector<TcGroupCta> pre, main;
  const int64_t cand_entries = plan_group_ctas(units, sm_count, &pre, &main);
  if (dense_cap < 256) dense_cap = 256;
  // ---- workspace (one stream-ordered allocation)
  size_t off = 0;
  auto take = [&](size_t bytes) { size_t o = off; off = (off + bytes + 255) & ~size_t(255); return o; };
  const size_t o_qs = take(size_t(nq) * dim * 4), o_qn = take(size_t(nq) * dim * 4), o_qi8 = take(size_t(nq) * dim);
  const size_t o_eps = take(size_t(nq) * 4), o_step = take(size_t(nq) * 4), o_keys = take(size_t(nq) * kGroups * 8);
  const size_t o_cnt = take(size_t(nq) * 4), o_flag = take(size_t(nq) * 4 + 12), o_floor = take(size_t(nq) * 4);
  const size_t o_cand = take(size_t(cand_entries > 0 ? cand_entries : 1) * 8);
  const size_t o_dense = take(size_t(nq) * dense_cap * 8);
  const size_t o_rows = take(size_t(nq) * k * 8), o_sc = take(size_t(nq) * k * 4), o_acc = take(size_t(nq));
  // the only host -> device copy of the call: [perm][tenant of each sorted query][pre-pass CTAs][filter CTAs]
  std::vector<unsigned char> table;
  const size_t t_perm = 0, t_ten = size_t(nq) * 4, t_pre = (t_ten + size_t(nq) * 4 + 15) & ~size_t(15);
  const size_t t_main = t_pre + pre.size() * sizeof(TcGroupCta);
  table.resize(t_main + main.size() * sizeof(TcGroupCta));
  memcpy(table.data() + t_perm, perm.data(), size_t(nq) * 4);
  for (const TcTenantGroup& G : groups)
    for (int i = 0; i < G.nq; ++i) memcpy(table.data() + t_ten + size_t(G.q0 + i) * 4, &G.tenant, 4);
  if (!pre.empty()) memcpy(table.data() + t_pre, pre.data(), pre.size() * sizeof(TcGroupCta));
  if (!main.empty()) memcpy(table.data() + t_main, main.data(), main.size() * sizeof(TcGroupCta));
  const size_t o_table = take(table.size());
  unsigned char* ws = nullptr;
  FRG_CUDA(cudaMallocAsync(reinterpret_cast<void**>(&ws), off, st));
  float* qs = reinterpret_cast<float*>(ws + o_qs);
  float* qn = reinterpret_cast<float*>(ws + o_qn);
  int8_t* qi8 = reinterpret_cast<int8_t*>(ws + o_qi8);
  float* eps = reinterpret_cast<float*>(ws + o_eps);
  float* qstep = reinterpret_cast<float*>(ws + o_step);
  unsigned long long* keys = reinterpret_cast<unsigned long long*>(ws + o_keys);
  int* cnt = reinterpret_cast<int*>(ws + o_cnt);
  int* flagged = reinterpret_cast<int*>(ws + o_flag);
  int* n_flagged = flagged + nq;
  float* floor_v = reinterpret_cast<float*>(ws + o_floor);
  int64_t* srows = reinterpret_cast<int64_t*>(ws + o_rows);
  float* sscores = reinterpret_cast<float*>(ws + o_sc);
  uint8_t* sacc = ws + o_acc;
  const int32_t* dperm = reinterpret_cast<const int32_t*>(ws + o_table + t_perm);
  const int32_t* dten = reinterpret_cast<const int32_t*>(ws + o_table + t_ten);
  int rc = stage_upload(ws + o_table, table.data(), table.size(), st);
  if (rc == FRG_OK) rc = launch_gather_queries(q, dperm, nq, dim, qs, st);
  profile_begin(st, kStagePrep);
  if (rc == FRG_OK)
    rc = launch_prepare_queries_i8(qs, nq, dim, qn, qi8, qstep, eps, s->gmax_bits, keys, cnt, n_flagged, st);
  profile_end(st, 1);
  CUtensorMap qm, gm;
  if (rc == FRG_OK) rc = make_map(&qm, qi8, dim, nq, size_t(dim), kTileQ, kBlockK, true);
  if (rc == FRG_OK) rc = make_map(&gm, s->plane8, dim, s->rows, size_t(dim), kTileR, kBlockK, true);
  TcScanParams p{};
  p.fault = s->fault; p.eps = eps; p.none_score = kNoScore; p.pad = 0; p.stages = kStages;
  p.dim = dim; p.nq = nq; p.tenant = -1; p.tags = s->tags; p.n_rows = int(s->rows); p.k = k; p.tile_scale = 1;
  p.group_key64 = keys; p.floor = floor_v; p.qstep = qstep;
  p.cand = reinterpret_cast<int2*>(ws + o_cand); p.cand_total = cnt;
  p.dense = reinterpret_cast<int2*>(ws + o_dense); p.dense_cap = dense_cap;
  // 1. int8 pre-pass, 2. exact floor, 3. filter: every (query tile, chunk) of every tenant in one grid each
  profile_begin(st, kStagePrepass);
  if (rc == FRG_OK && !pre.empty()) {
    p.groups = reinterpret_cast<const TcGroupCta*>(ws + o_table + t_pre);
    rc = launch_tc_scan<kModeGroupMax, true, false, true, true>(qm, gm, gm, p, int(pre.size()), 1, st);
  }
  profile_end(st, 1);
  profile_begin(st, kStageFloor);
  if (rc == FRG_OK) {
    cudaError_t e = launch_kernel(i8_floor_kernel, dim3((nq + 3) / 4), dim3(128), 0, st, keys, nq, k, dim, qn,
                                  s->master, eps, floor_v);
    if (e != cudaSuccess) rc = cuda_fail(e, "i8_floor_kernel", __FILE__, __LINE__);
    else note_launch(nullptr);
  }
  profile_end(st, 1);
  profile_begin(st, kStageDominant);
  if (rc == FRG_OK && !main.empty()) {
    p.groups = reinterpret_cast<const TcGroupCta*>(ws + o_table + t_main);
    rc = launch_tc_scan<kModeFilter, true, false, true, true>(qm, gm, gm, p, int(main.size()), 1, st);
  }
  profile_end(st, 1);
  // 4. select + exact rescoring into the sorted scratch (the tenant filter was applied by the filter's tag check)
  profile_begin(st, kStageSelect);
  if (rc == FRG_OK) {
    cudaError_t e = cudaSuccess;
#define FRG_SELECT_G(KK)                                                                                          \
  e = func_attr_once(select_rescore_kernel<KK, false>, cudaFuncAttributePreferredSharedMemoryCarveout, 100);       \
  if (e == cudaSuccess)                                                                                          \
    e = launch_kernel(select_rescore_kernel<KK, false>, dim3(nq), dim3(kSelectWarps * 32), 0, st,               \
                      const_cast<const int2*>(p.dense), const_cast<const int*>(cnt), dense_cap, nq, k, dim,       \
                      const_cast<const float*>(qn), const_cast<const float*>(eps),                              \
                      static_cast<const __nv_bfloat16*>(nullptr), dim, static_cast<const float*>(nullptr),        \
                      const_cast<const float*>(qstep), s->master, 1, threshold, row_offset, srows, sscores, sacc,  \
                      flagged, n_flagged, XPush())
    switch (reg_k(k)) {
      case 1: FRG_SELECT_G(1); break;
      case 4: FRG_SELECT_G(4); break;
      case 8: FRG_SELECT_G(8); break;
      default: FRG_SELECT_G(16); break;
    }
#undef FRG_SELECT_G
    if (e != cudaSuccess) rc = cuda_fail(e, "select_rescore_kernel", __FILE__, __LINE__);
    else note_launch(nullptr);
  }
  profile_end(st, 1);
  // 5. the queries whose candidates overflowed: exact scan of the whole store, each with its own tenant
  profile_begin(st, kStageFallback);
  if (rc == FRG_OK) {
    ScanArgs a;
    a.master = s->master; a.plane = nullptr; a.tags = s->tags; a.rows = s->rows; a.dim = dim;
    a.qn = qn; a.nq = nq; a.k = k; a.metric = FRG_METRIC_COSINE; a.tenant = -1; a.sm_count = sm_count;
    rc = launch_scan_f32_flagged_tenants(a, dten, flagged, n_flagged, row_offset, threshold, srows, sscores, sacc, st);
  }
  profile_end(st, 1);
  if (rc == FRG_OK) rc = launch_scatter_results(srows, sscores, sacc, dperm, nq, k, out_rows, out_scores, out_accept, st);
  if (rc == FRG_OK) { cudaError_t e = cudaGetLastError(); if (e != cudaSuccess) rc = cuda_fail(e, "grouped match", __FILE__, __LINE__); }
  cudaError_t e = cudaFreeAsync(ws, st);
  if (rc == FRG_OK && e != cudaSuccess) rc = cuda_fail(e, "cudaFreeAsync", __FILE__, __LINE__);
  return rc;
}

// ------------------------------------------------------------------------------------------ gallery self-join
// range_select_kernel for a slab of the self-join: query q is the stored row a = qrow0 + q.  A dead query, or one
// outside the tenant, has no pairs.  A candidate counts when b > a and, with same_tag, tag[b] == tag[a] (the filter
// has masked dead rows, and other tenants' rows when its descriptor carried a tenant); it is rescored with the same
// arithmetic as range_select_kernel, so the scores are bit-identical to a range search with row a as the query.
__global__ void __launch_bounds__(kSelectWarps * 32)
join_select_kernel(const int2* __restrict__ dense, const int* __restrict__ cand_total, int dense_cap, int dim,
                   const float* __restrict__ qn, const float* __restrict__ master, const int32_t* __restrict__ tags,
                   int64_t qrow0, int32_t tenant, int same_tag, float threshold, int strict, int max_hits,
                   int64_t row_offset, int64_t* __restrict__ out_counts, int64_t* __restrict__ out_rows,
                   float* __restrict__ out_scores, int* __restrict__ flagged, int* __restrict__ n_flagged) {
  extern __shared__ unsigned long long hits[];        // [pow2 >= dense_cap]
  __shared__ int s_m;
  const int lane = threadIdx.x & 31;
  const int w = threadIdx.x >> 5;
  const int q = blockIdx.x;
  const int64_t a = qrow0 + q;
  pdl_wait();             // the filter kernel's candidate lists
  pdl_trigger();
  const int32_t ta = __ldg(tags + a);
  const bool live = ta >= 0 && (tenant < 0 || ta == tenant);
  const int total = live ? cand_total[q] : 0;
  if (total > dense_cap) {                           // also set by a poisoned total (segment overflow)
    if (threadIdx.x == 0) flagged[atomicAdd(n_flagged, 1)] = q;
    return;
  }
  if (threadIdx.x == 0) s_m = 0;
  __syncthreads();
  const int2* mine = dense + size_t(q) * dense_cap;
  const int nvec = dim >> 2;
  const float4* qq = reinterpret_cast<const float4*>(qn + size_t(q) * dim);
  for (int c = w; c < total; c += kSelectWarps) {
    const int row = mine[c].x;
    if (row <= a || (same_tag && __ldg(tags + row) != ta)) continue;     // warp-uniform
    const float4* g = reinterpret_cast<const float4*>(master + size_t(row) * dim);
    float acc = 0.f;
#pragma unroll 4
    for (int v = lane; v < nvec; v += 32) {
      const float4 x = __ldg(g + v), y = __ldg(qq + v);
      acc = fmaf(x.x, y.x, acc); acc = fmaf(x.y, y.y, acc); acc = fmaf(x.z, y.z, acc); acc = fmaf(x.w, y.w, acc);
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
    const bool pass = strict ? (acc > threshold) : (acc >= threshold);      // false for NaN
    if (lane == 0 && pass) hits[atomicAdd(&s_m, 1)] = (uint64_t(uint32_t(row)) << 32) | __float_as_uint(acc);
  }
  __syncthreads();
  const int m = s_m;
  int n2 = 1;
  while (n2 < m) n2 <<= 1;
  for (int i = m + threadIdx.x; i < n2; i += blockDim.x) hits[i] = ~0ull;
  __syncthreads();
  // rows are distinct: ascending keys = gallery order
  for (int kk = 2; kk <= n2; kk <<= 1) {
    for (int j = kk >> 1; j > 0; j >>= 1) {
      for (int i = threadIdx.x; i < n2; i += blockDim.x) {
        const int ij = i ^ j;
        if (ij > i) {
          const unsigned long long x = hits[i], y = hits[ij];
          if ((x > y) == ((i & kk) == 0)) { hits[i] = y; hits[ij] = x; }
        }
      }
      __syncthreads();
    }
  }
  for (int i = threadIdx.x; i < max_hits; i += blockDim.x) {
    const bool filled = i < m;
    out_rows[size_t(q) * max_hits + i] = filled ? int64_t(hits[i] >> 32) + row_offset : int64_t(kNoRow);
    out_scores[size_t(q) * max_hits + i] = filled ? __uint_as_float(uint32_t(hits[i])) : kNoScore;
  }
  if (threadIdx.x == 0) out_counts[q] = m;
}

void tc_join_plan(const std::vector<TcTenantGroup>& tiles, int sm_count, std::vector<unsigned char>* table,
                  int* n_ctas, int64_t* cand_entries) {
  std::vector<GroupUnit> units;
  for (const TcTenantGroup& t : tiles) units.push_back(GroupUnit{&t, t.q0, t.nq, kRangeBudget, 1});
  std::vector<TcGroupCta> main;
  *cand_entries = plan_group_ctas(units, sm_count, nullptr, &main);
  *n_ctas = int(main.size());
  table->resize(main.size() * sizeof(TcGroupCta));
  if (!main.empty()) memcpy(table->data(), main.data(), table->size());
}

int launch_tc_join(const GalleryWindow* s, const float* qn, const int8_t* qi8, const float* qstep, const float* eps,
                   int nq, const void* d_table, int n_ctas, int64_t qrow0, int32_t tenant, bool same_tag,
                   float threshold, bool strict, int max_hits, int64_t row_offset, int2* cand, int* cand_total,
                   int2* dense, float* floor_v, int* flagged, int* n_flagged, int64_t* out_counts, int64_t* out_rows,
                   float* out_scores, cudaStream_t st) {
  if (!s->plane8 || !s->master || s->row0 != 0 || s->rows > 0x7fffffff) {
    set_error("tc_join: needs the whole unit store with an int8 plane and an fp32 master");
    return FRG_ERR_UNSUPPORTED;
  }
  CUtensorMap qm, gm;
  FRG_CHECK(make_map(&qm, qi8, s->dim, nq, size_t(s->dim), kTileQ, kBlockK, true));
  FRG_CHECK(make_map(&gm, s->plane8, s->dim, s->rows, size_t(s->dim), kTileR, kBlockK, true));
  TcScanParams p{};
  p.fault = s->fault; p.eps = eps; p.none_score = kNoScore; p.pad = 0; p.stages = kStages;
  p.dim = s->dim; p.nq = nq; p.tenant = -1; p.tags = s->tags; p.n_rows = int(s->rows); p.k = 1; p.tile_scale = 1;
  p.floor = floor_v; p.qstep = qstep;
  p.cand = cand; p.cand_total = cand_total; p.dense = dense; p.dense_cap = kRangeBudget;
  p.groups = static_cast<const TcGroupCta*>(d_table);
  profile_begin(st, kStageFloor);
  FRG_CUDA(launch_kernel(range_floor_kernel, dim3((nq + 255) / 256), dim3(256), 0, st, eps, threshold, floor_v, nq));
  note_launch(nullptr);
  profile_end(st, 1);
  profile_begin(st, kStageDominant);
  if (n_ctas > 0) FRG_CHECK((launch_tc_scan<kModeFilter, true, false, true, true>(qm, gm, gm, p, n_ctas, 1, st)));
  profile_end(st, n_ctas > 0 ? 1 : 0);
  profile_begin(st, kStageSelect);
  int n2 = 1;
  while (n2 < kRangeBudget) n2 <<= 1;
  const size_t smem = size_t(n2) * sizeof(unsigned long long);
  FRG_CUDA(func_attr_once(join_select_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, int(smem)));
  FRG_CUDA(launch_kernel(join_select_kernel, dim3(nq), dim3(kSelectWarps * 32), smem, st,
                         const_cast<const int2*>(dense), const_cast<const int*>(cand_total), kRangeBudget, s->dim, qn,
                         s->master, s->tags, qrow0, tenant, same_tag ? 1 : 0, threshold, strict ? 1 : 0, max_hits,
                         row_offset, out_counts, out_rows, out_scores, flagged, n_flagged));
  note_launch(nullptr);
  FRG_CUDA(cudaGetLastError());
  profile_end(st, 1);
  return FRG_OK;
}

}  // namespace frg
