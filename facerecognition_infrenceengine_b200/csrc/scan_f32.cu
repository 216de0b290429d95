// Exact fp32 streaming scan (FRG_VARIANT_SCAN_F32): the reference's inner loop
//   for person_id, g in embeddings.items(): s = np.dot(q, g); if s > best: ...
// (infrenceServer.py:538-542, peopleCount.py:869-873) for up to QB queries per pass, on CUDA cores.
//
// HBM-bound by construction: every gallery row (dim * 4 B) is read exactly once per pass with
// 16-byte streaming loads, a warp owning whole rows (512 B per load instruction, fully coalesced);
// the QB unit queries live in registers (lane L holds elements j*128 + 4L .. +3 of each), the QB
// row-dots are reduced with a halving butterfly (QB + log2(32/QB) shuffles instead of 5*QB) and the
// running top-k of each (warp, query) sits in shared memory, touched only when a score beats the
// current k-th best.  Per-CTA lists go to a small partial buffer folded by merge.cu, so no score
// matrix ever reaches HBM.
//
// Algorithmic bytes per launch = rows * dim * 4 (DESIGN.md); grid = 2 CTAs x SM count.
#include "merge_device.cuh"

namespace frg {

constexpr int kScanWarps = 8;

__device__ __forceinline__ float4 ldg_stream(const float4* p) {
  float4 v;
  asm volatile("ld.global.nc.L1::no_allocate.v4.f32 {%0,%1,%2,%3}, [%4];"
               : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "l"(p));
  return v;
}

// the same 4 elements per lane and 128-element chunk, from the bf16 scan plane (bf16-only stores)
__device__ __forceinline__ float4 ldg_stream_bf16(const uint2* p) {
  uint2 v;
  asm volatile("ld.global.nc.L1::no_allocate.v2.u32 {%0,%1}, [%2];" : "=r"(v.x), "=r"(v.y) : "l"(p));
  return make_float4(__uint_as_float(v.x << 16), __uint_as_float(v.x & 0xffff0000u),
                     __uint_as_float(v.y << 16), __uint_as_float(v.y & 0xffff0000u));
}

// Reduce QB per-lane partial dots across the warp.  After the call, the returned value on lane L is
// the full dot for query `lane_query<QB>(L)`, replicated on the 32/QB lanes that share it.
template <int QB>
__device__ __forceinline__ float butterfly(float (&acc)[QB], int lane) {
  int width = 16;
#pragma unroll
  for (int n = QB; n > 1; n >>= 1) {
    const bool upper = (lane & width) != 0;
#pragma unroll
    for (int i = 0; i < n / 2; ++i) {
      const float keep = upper ? acc[i + n / 2] : acc[i];
      const float send = upper ? acc[i] : acc[i + n / 2];
      acc[i] = keep + __shfl_xor_sync(0xffffffffu, send, width);
    }
    width >>= 1;
  }
#pragma unroll
  for (int w = 16; w > 0; w >>= 1)
    if (w <= width) acc[0] += __shfl_xor_sync(0xffffffffu, acc[0], w);
  return acc[0];
}

template <int QB>
__device__ __forceinline__ int lane_query(int lane) {
  int q = 0, width = 16;
#pragma unroll
  for (int n = QB; n > 1; n >>= 1) {
    if (lane & width) q += n / 2;
    width >>= 1;
  }
  return q;
}

template <int QB>
__device__ __forceinline__ bool lane_is_rep(int lane) {
  // lowest lane of the group sharing a query: all non-query bits clear
  int mask = 0, width = 16;
#pragma unroll
  for (int n = QB; n > 1; n >>= 1) { mask |= width; width >>= 1; }
  return (lane & ~mask) == 0;
}

template <int NJ, int QB, int METRIC>
__device__ __forceinline__ void row_dots(const float4 (&g)[NJ], const float4 (&q)[QB][NJ], float (&acc)[QB]) {
#pragma unroll
  for (int b = 0; b < QB; ++b) {
    float a = 0.f;
#pragma unroll
    for (int j = 0; j < NJ; ++j) {
      if (METRIC == FRG_METRIC_COSINE) {
        a = fmaf(g[j].x, q[b][j].x, a); a = fmaf(g[j].y, q[b][j].y, a);
        a = fmaf(g[j].z, q[b][j].z, a); a = fmaf(g[j].w, q[b][j].w, a);
      } else {
        float d;
        d = g[j].x - q[b][j].x; a = fmaf(d, d, a);
        d = g[j].y - q[b][j].y; a = fmaf(d, d, a);
        d = g[j].z - q[b][j].z; a = fmaf(d, d, a);
        d = g[j].w - q[b][j].w; a = fmaf(d, d, a);
      }
    }
    acc[b] = a;
  }
}

// Insert (s, row) into the descending list [sc, ix] of length K held in shared memory.  Rows reach a
// warp in increasing order, so strict '>' keeps the earliest row on exact ties.
__device__ __forceinline__ void list_insert(float* sc, int32_t* ix, int K, float s, int32_t row) {
  int t = K - 1;
  while (t > 0 && s > sc[t - 1]) { sc[t] = sc[t - 1]; ix[t] = ix[t - 1]; --t; }
  sc[t] = s; ix[t] = row;
}

// One pass over the gallery for the queries q_of[0..nq_pass): fills part_[sc|ix][(block*part_stride + part_q0 + b)*K ..].
// ROW = float: fp32 master rows.  ROW = __nv_bfloat16: rows of the bf16 scan plane, widened exactly.
// SPARSE: few rows of the window can take part (a tenant whose row window was stretched by one late
// re-enrolment; a gallery full of tombstones).  Tags are read FIRST - 32 per warp and step, one coalesced load,
// the next step's prefetched - and only the rows that can match are fetched at all: a 10 000-row company inside
// a 1 M-row window costs 4 MB of tags + 20 MB of rows per pass instead of 2 GB.
template <int NJ, int QB, int METRIC, typename ROW = float, bool SPARSE = false>
__device__ __forceinline__ void scan_pass(const ROW* __restrict__ master, const int32_t* __restrict__ tags,
                                          int64_t rows, const float* __restrict__ qn, const int (&q_of)[QB],
                                          int nq_pass, int part_stride, int part_q0, int K, int32_t tenant,
                                          float* __restrict__ part_sc, int32_t* __restrict__ part_ix,
                                          float* l_sc, int32_t* l_ix, const int32_t* w_list = nullptr, int w_n = -1) {
  constexpr int DIM = NJ * 128;
  const int lane = threadIdx.x & 31;
  const int warp = threadIdx.x >> 5;
  const float sentinel = METRIC == FRG_METRIC_COSINE ? kNoScore : -INFINITY;

  for (int i = threadIdx.x; i < kScanWarps * QB * K; i += blockDim.x) { l_sc[i] = sentinel; l_ix[i] = 0x7fffffff; }

  float4 q[QB][NJ];
#pragma unroll
  for (int b = 0; b < QB; ++b) {
#pragma unroll
    for (int j = 0; j < NJ; ++j) {
      q[b][j] = (b < nq_pass)
                    ? __ldg(reinterpret_cast<const float4*>(qn + size_t(q_of[b]) * DIM) + j * 32 + lane)
                    : make_float4(0.f, 0.f, 0.f, 0.f);
    }
  }
  __syncthreads();

  const int my_q = lane_query<QB>(lane);
  const bool rep = lane_is_rep<QB>(lane);
  float* my_sc = l_sc + (warp * QB + my_q) * K;
  int32_t* my_ix = l_ix + (warp * QB + my_q) * K;
  float kth = sentinel;

  const int64_t gw = int64_t(blockIdx.x) * kScanWarps + warp;
  const int64_t tw = int64_t(gridDim.x) * kScanWarps;

  auto load_row = [&](int64_t r, float4 (&g)[NJ]) {
    if constexpr (sizeof(ROW) == 4) {
      const float4* pr = reinterpret_cast<const float4*>(master + r * DIM) + lane;
#pragma unroll
      for (int j = 0; j < NJ; ++j) g[j] = ldg_stream(pr + j * 32);
    } else {
      const uint2* pr = reinterpret_cast<const uint2*>(master + r * DIM) + lane;
#pragma unroll
      for (int j = 0; j < NJ; ++j) g[j] = ldg_stream_bf16(pr + j * 32);
    }
  };
  auto consume = [&](const float4 (&g)[NJ], int64_t r) {
    float a[QB];
    row_dots<NJ, QB, METRIC>(g, q, a);
    float sdot = butterfly<QB>(a, lane);
    if (METRIC == FRG_METRIC_EUCLIDEAN) sdot = -sdot;
    const bool ins = sdot > kth;                     // false for NaN
    if (__any_sync(0xffffffffu, ins)) {
      if (ins && rep) list_insert(my_sc, my_ix, K, sdot, int32_t(r));
      __syncwarp();
      kth = my_sc[K - 1];
    }
  };
  if (SPARSE && w_n >= 0) {
    // this warp's valid rows were listed once for the whole kernel (sparse_row_list): two in flight
    for (int i = 0; i < w_n; i += 2) {
      const bool two = i + 1 < w_n;
      const int64_t r0 = w_list[i], r1 = two ? w_list[i + 1] : r0;
      float4 g0[NJ], g1[NJ];
      load_row(r0, g0);
      if (two) load_row(r1, g1);
      consume(g0, r0);
      if (two) consume(g1, r1);
    }
  } else if constexpr (SPARSE) {
    const int64_t nblk = (rows + 31) >> 5;
    auto tag_of = [&](int64_t b) {
      const int64_t r = b * 32 + lane;
      return (b < nblk && r < rows) ? __ldg(tags + r) : int32_t(-1);
    };
    int32_t tg_next = tag_of(gw);
    for (int64_t b = gw; b < nblk; b += tw) {
      const int32_t tg = tg_next;
      tg_next = tag_of(b + tw);
      unsigned vm = __ballot_sync(0xffffffffu, tg >= 0 && (tenant < 0 || tg == tenant));
      while (vm) {                                   // valid rows of the block, in row order, two in flight
        const int j0 = __ffs(vm) - 1;
        vm &= vm - 1;
        const int j1 = vm ? __ffs(vm) - 1 : -1;
        if (j1 >= 0) vm &= vm - 1;
        float4 g0[NJ], g1[NJ];
        load_row(b * 32 + j0, g0);
        if (j1 >= 0) load_row(b * 32 + j1, g1);
        consume(g0, b * 32 + j0);
        if (j1 >= 0) consume(g1, b * 32 + j1);
      }
    }
  }
  // R rows in flight per warp (R * NJ 16-byte loads per lane): enough bytes in flight per SM to
  // cover the HBM latency even for short rows
  constexpr int R = NJ >= 4 ? 2 : (NJ == 2 ? 4 : 8);
  for (int64_t rb = SPARSE ? rows : gw; rb < rows; rb += int64_t(R) * tw) {
    float4 g[R][NJ];
    int32_t tg[R];
#pragma unroll
    for (int u = 0; u < R; ++u) {
      const int64_t r = rb + int64_t(u) * tw;
      const bool has = r < rows;
      if constexpr (sizeof(ROW) == 4) {
        const float4* pr = reinterpret_cast<const float4*>(master + (has ? r : rb) * DIM) + lane;
#pragma unroll
        for (int j = 0; j < NJ; ++j) g[u][j] = ldg_stream(pr + j * 32);
      } else {
        const uint2* pr = reinterpret_cast<const uint2*>(master + (has ? r : rb) * DIM) + lane;
#pragma unroll
        for (int j = 0; j < NJ; ++j) g[u][j] = ldg_stream_bf16(pr + j * 32);
      }
      tg[u] = has ? __ldg(tags + r) : -1;
    }
#pragma unroll
    for (int u = 0; u < R; ++u) {
      float a[QB];
      row_dots<NJ, QB, METRIC>(g[u], q, a);
      float sdot = butterfly<QB>(a, lane);
      if (METRIC == FRG_METRIC_EUCLIDEAN) sdot = -sdot;
      // removed rows (tag -1) and other tenants never take part (infrenceServer.py:343-380)
      const bool valid = tg[u] >= 0 && (tenant < 0 || tg[u] == tenant);
      const bool ins = valid && sdot > kth;          // false for NaN
      if (__any_sync(0xffffffffu, ins)) {
        if (ins && rep) list_insert(my_sc, my_ix, K, sdot, int32_t(rb + int64_t(u) * tw));
        __syncwarp();
        kth = my_sc[K - 1];
      }
    }
  }
  __syncthreads();

  // fold the kScanWarps lists of each query: thread b < nq_pass walks the heads
  if (threadIdx.x < nq_pass) {
    const int b = threadIdx.x;
    int head[kScanWarps];
#pragma unroll
    for (int w = 0; w < kScanWarps; ++w) head[w] = 0;
    float* o_sc = part_sc + (size_t(blockIdx.x) * part_stride + part_q0 + b) * K;
    int32_t* o_ix = part_ix + (size_t(blockIdx.x) * part_stride + part_q0 + b) * K;
    for (int j = 0; j < K; ++j) {
      float bs = sentinel; int32_t br = 0x7fffffff; int bw = -1;
#pragma unroll
      for (int w = 0; w < kScanWarps; ++w) {
        if (head[w] < K) {
          const float s = l_sc[(w * QB + b) * K + head[w]];
          const int32_t r = l_ix[(w * QB + b) * K + head[w]];
          if (s > bs || (s == bs && r < br)) { bs = s; br = r; bw = w; }
        }
      }
#pragma unroll
      for (int w = 0; w < kScanWarps; ++w) if (w == bw) head[w]++;
      o_sc[j] = bs;
      o_ix[j] = (br == 0x7fffffff) ? -1 : br;
    }
  }
}

template <int NJ, int QB, int METRIC>
__global__ void __launch_bounds__(kScanWarps * 32, 2)
scan_f32_kernel(const float* __restrict__ master, const int32_t* __restrict__ tags, int64_t rows,
                const float* __restrict__ qn, int nq_total, int q0, int nq_pass, int K, int32_t tenant,
                float* __restrict__ part_sc, int32_t* __restrict__ part_ix) {
  extern __shared__ unsigned char smem_raw[];
  float* l_sc = reinterpret_cast<float*>(smem_raw);                          // [warp][query][K]
  int32_t* l_ix = reinterpret_cast<int32_t*>(l_sc + kScanWarps * QB * K);
  int q_of[QB];
#pragma unroll
  for (int b = 0; b < QB; ++b) q_of[b] = q0 + b;
  scan_pass<NJ, QB, METRIC>(master, tags, rows, qn, q_of, nq_pass, nq_total, q0, K, tenant, part_sc, part_ix,
                            l_sc, l_ix);
}

// SPARSE fallback: the rows that can take part are the same for every pass of the kernel - each warp lists ITS
// valid rows once (tags read 32 at a time, ascending), up to kSparseCap; a warp with more keeps sweeping the tags
// in every pass (returns -1).
constexpr int kSparseCap = 96;
__device__ __forceinline__ int sparse_row_list(const int32_t* __restrict__ tags, int64_t rows, int32_t tenant,
                                               int32_t* list) {
  const int lane = threadIdx.x & 31;
  const int64_t gw = int64_t(blockIdx.x) * kScanWarps + (threadIdx.x >> 5);
  const int64_t tw = int64_t(gridDim.x) * kScanWarps;
  const int64_t nblk = (rows + 31) >> 5;
  int n = 0;
  for (int64_t b0 = gw; b0 < nblk; b0 += 4 * tw) {           // four independent tag loads per round
    int32_t tg[4];
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      const int64_t r = (b0 + u * tw) * 32 + lane;
      tg[u] = (b0 + u * tw < nblk && r < rows) ? __ldg(tags + r) : int32_t(-1);
    }
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      const bool ok = tg[u] >= 0 && (tenant < 0 || tg[u] == tenant);
      const unsigned vm = __ballot_sync(0xffffffffu, ok);
      const int pos = n + __popc(vm & ((1u << lane) - 1u));
      if (ok && pos < kSparseCap) list[pos] = int32_t((b0 + u * tw) * 32 + lane);
      n += __popc(vm);
    }
  }
  __syncwarp();
  return n <= kSparseCap ? n : -1;
}

// Exact re-do of the queries a tensor-core pass could not settle (candidate overflow).  The list
// and its length live on the device; the kernel loops over it, so nothing waits for the host, and
// the CTA that finishes last folds the per-CTA lists into the final results (ticket counter), so an
// empty list costs ONE idle launch.  ctl[0] = number of flagged queries, ctl[1] = ticket (starts 0).
template <int NJ, int QB, int METRIC, int KMAX, typename ROW, bool SPARSE>
__global__ void __launch_bounds__(kScanWarps * 32, 2)
scan_f32_flagged_kernel(const ROW* __restrict__ master, const int32_t* __restrict__ tags, int64_t rows,
                        const float* __restrict__ qn, int nq_total, const int* __restrict__ flagged,
                        int* __restrict__ ctl, int K, int32_t tenant, float threshold, int64_t row_offset,
                        float* __restrict__ part_sc, int32_t* __restrict__ part_ix,
                        int64_t* __restrict__ out_rows, float* __restrict__ out_scores,
                        uint8_t* __restrict__ out_accept, const XPush x) {
  extern __shared__ unsigned char smem_raw[];
  float* l_sc = reinterpret_cast<float*>(smem_raw);
  int32_t* l_ix = reinterpret_cast<int32_t*>(l_sc + kScanWarps * QB * K);
  __shared__ int is_last;
  __shared__ int32_t s_list[SPARSE ? kScanWarps : 1][SPARSE ? kSparseCap : 1];
  pdl_wait();             // the select kernel's list of flagged queries
  pdl_trigger();
  const int nf = ctl[0];
  int w_n = -1;
  const int32_t* w_list = s_list[SPARSE ? (threadIdx.x >> 5) : 0];
  if (SPARSE && nf > 0) w_n = sparse_row_list(tags, rows, tenant, s_list[SPARSE ? (threadIdx.x >> 5) : 0]);
  for (int q0 = 0; q0 < nf; q0 += QB) {
    const int nq_pass = nf - q0 < QB ? nf - q0 : QB;
    int q_of[QB];
#pragma unroll
    for (int b = 0; b < QB; ++b) q_of[b] = b < nq_pass ? flagged[q0 + b] : 0;
    scan_pass<NJ, QB, METRIC, ROW, SPARSE>(master, tags, rows, qn, q_of, nq_pass, nq_total, q0, K, tenant, part_sc,
                                           part_ix, l_sc, l_ix, w_list, w_n);
    __syncthreads();
  }
  if (nf == 0) return;
  __threadfence();
  __syncthreads();
  if (threadIdx.x == 0) is_last = atomicAdd(ctl + 1, 1) == int(gridDim.x) - 1;
  __syncthreads();
  if (!is_last) return;
  __threadfence();
  for (int slot = threadIdx.x >> 5; slot < nf; slot += kScanWarps) {
    const int q = flagged[slot];
    merge_one<int32_t, KMAX>(part_sc, part_ix, int(gridDim.x), nq_total, K, K, METRIC, threshold, row_offset,
                             /*internal_euclid=*/METRIC == FRG_METRIC_EUCLIDEAN ? 1 : 0, slot, q, int64_t(nq_total) * K, int64_t(nq_total) * K, out_rows, out_scores,
                             out_accept);
    if (x.peer_bufs) {
      // row-sharded gallery: the redone query's top-k is final now - send it to every rank (select skipped it)
      __syncwarp();                // lane 0's result stores are visible to the warp
      const int lane = threadIdx.x & 31;
      for (int c = lane; c < x.world * K; c += 32) {
        const int peer = c / K, j = c - peer * K;
        const int64_t s_ = int64_t(q) * K + j;
        xpush_slot(x, (x.rank + 1 + peer) % x.world, s_, out_rows[s_], out_scores[s_]);
      }
    }
  }
}

// The exact re-do of scan_f32_flagged_kernel for a batch whose queries carry their own tenants (frg_match_tenants):
// flagged query q is scanned alone with tenant q_tenant[q] - a tenant-filtered one reads the tags first and fetches
// only its tenant's rows (SPARSE sweep), an unfiltered one streams every row.  Same partial lists, ticket and merge.
template <int NJ, int KMAX>
__global__ void __launch_bounds__(kScanWarps * 32, 2)
scan_f32_flagged_tenants_kernel(const float* __restrict__ master, const int32_t* __restrict__ tags, int64_t rows,
                                const float* __restrict__ qn, int nq_total, const int32_t* __restrict__ q_tenant,
                                const int* __restrict__ flagged, int* __restrict__ ctl, int K, float threshold,
                                int64_t row_offset, float* __restrict__ part_sc, int32_t* __restrict__ part_ix,
                                int64_t* __restrict__ out_rows, float* __restrict__ out_scores,
                                uint8_t* __restrict__ out_accept) {
  extern __shared__ unsigned char smem_raw[];
  float* l_sc = reinterpret_cast<float*>(smem_raw);
  int32_t* l_ix = reinterpret_cast<int32_t*>(l_sc + kScanWarps * K);
  __shared__ int is_last;
  pdl_wait();             // the select kernel's list of flagged queries
  pdl_trigger();
  const int nf = ctl[0];
  for (int slot = 0; slot < nf; ++slot) {
    const int q_of[1] = {flagged[slot]};
    const int32_t tenant = q_tenant[q_of[0]];
    if (tenant >= 0)
      scan_pass<NJ, 1, FRG_METRIC_COSINE, float, true>(master, tags, rows, qn, q_of, 1, nq_total, slot, K, tenant,
                                                       part_sc, part_ix, l_sc, l_ix);
    else
      scan_pass<NJ, 1, FRG_METRIC_COSINE>(master, tags, rows, qn, q_of, 1, nq_total, slot, K, -1, part_sc, part_ix,
                                          l_sc, l_ix);
    __syncthreads();
  }
  if (nf == 0) return;
  __threadfence();
  __syncthreads();
  if (threadIdx.x == 0) is_last = atomicAdd(ctl + 1, 1) == int(gridDim.x) - 1;
  __syncthreads();
  if (!is_last) return;
  __threadfence();
  for (int slot = threadIdx.x >> 5; slot < nf; slot += kScanWarps)
    merge_one<int32_t, KMAX>(part_sc, part_ix, int(gridDim.x), nq_total, K, K, FRG_METRIC_COSINE, threshold, row_offset,
                             0, slot, flagged[slot], int64_t(nq_total) * K, int64_t(nq_total) * K, out_rows, out_scores,
                             out_accept);
}

template <int NJ, int KMAX>
static int launch_flagged_tenants_k(const ScanArgs& a, int grid, const int32_t* q_tenant, const int* flagged, int* ctl,
                                    float threshold, int64_t row_offset, float* ps, int32_t* pi, int64_t* out_rows,
                                    float* out_scores, uint8_t* out_accept, cudaStream_t st) {
  const size_t smem = size_t(kScanWarps) * a.k * (sizeof(float) + sizeof(int32_t));
  auto kern = scan_f32_flagged_tenants_kernel<NJ, KMAX>;
  FRG_CUDA(func_attr_once(kern, cudaFuncAttributePreferredSharedMemoryCarveout, 100));
  FRG_CUDA(launch_kernel(kern, dim3(grid), dim3(kScanWarps * 32), smem, st, a.master, a.tags, a.rows, a.qn, a.nq,
                         q_tenant, flagged, ctl, a.k, threshold, row_offset, ps, pi, out_rows, out_scores, out_accept));
  note_launch(nullptr);
  return FRG_OK;
}

template <int NJ>
static int launch_flagged_tenants_t(const ScanArgs& a, int grid, const int32_t* q_tenant, const int* flagged, int* ctl,
                                    float threshold, int64_t row_offset, float* ps, int32_t* pi, int64_t* out_rows,
                                    float* out_scores, uint8_t* out_accept, cudaStream_t st) {
#define FRG_FT(KM) return launch_flagged_tenants_k<NJ, KM>(a, grid, q_tenant, flagged, ctl, threshold, row_offset, ps, \
                                                            pi, out_rows, out_scores, out_accept, st)
  if (a.k == 1) FRG_FT(1);
  if (a.k <= 4) FRG_FT(4);
  if (a.k <= 8) FRG_FT(8);
  FRG_FT(16);
#undef FRG_FT
}

int launch_scan_f32_flagged_tenants(const ScanArgs& a, const int32_t* q_tenant, const int* flagged, int* ctl,
                                    int64_t row_offset, float threshold, int64_t* out_rows, float* out_scores,
                                    uint8_t* out_accept, cudaStream_t st) {
  if (a.rows <= 0 || a.nq <= 0) return FRG_OK;
  if (!a.master || a.metric != FRG_METRIC_COSINE) { set_error("flagged scan: per-query tenants need a cosine master"); return FRG_ERR_UNSUPPORTED; }
  const int grid = a.sm_count;
  const size_t n_part = size_t(grid) * a.nq * a.k;
  unsigned char* ws = nullptr;
  FRG_CUDA(cudaMallocAsync(reinterpret_cast<void**>(&ws), n_part * 8, st));
  float* ps = reinterpret_cast<float*>(ws);
  int32_t* pi = reinterpret_cast<int32_t*>(ps + n_part);
  int rc;
  switch (a.dim) {
    case 128: rc = launch_flagged_tenants_t<1>(a, grid, q_tenant, flagged, ctl, threshold, row_offset, ps, pi, out_rows, out_scores, out_accept, st); break;
    case 256: rc = launch_flagged_tenants_t<2>(a, grid, q_tenant, flagged, ctl, threshold, row_offset, ps, pi, out_rows, out_scores, out_accept, st); break;
    case 512: rc = launch_flagged_tenants_t<4>(a, grid, q_tenant, flagged, ctl, threshold, row_offset, ps, pi, out_rows, out_scores, out_accept, st); break;
    default: set_error("flagged scan: dim %d not built", a.dim); rc = FRG_ERR_UNSUPPORTED; break;
  }
  cudaError_t e = cudaFreeAsync(ws, st);
  if (rc == FRG_OK && e != cudaSuccess) rc = cuda_fail(e, "cudaFreeAsync", __FILE__, __LINE__);
  return rc;
}

static int scan_grid(const ScanArgs& a) {
  const int r = a.dim >= 512 ? 2 : (a.dim == 256 ? 4 : 8);     // rows in flight per warp (scan_pass)
  int64_t want = (a.rows + kScanWarps * r - 1) / (kScanWarps * r);
  int64_t cap = int64_t(a.sm_count) * 2;
  if (want > cap) want = cap;
  if (want < 1) want = 1;
  return int(want);
}

static int scan_qb(int dim, int nq) {
  const int nj = dim / 128;
  int qb = 16 / nj;                 // register budget: QB * NJ float4 <= 16 (64 registers of queries)
  if (qb > 8) qb = 8;               // 16 would spill under the 128-register cap of 2 CTAs / SM
  if (qb < 1) qb = 1;
  while (qb > 1 && qb / 2 >= nq) qb /= 2;
  return qb;
}

int scan_f32_workspace_bytes(const ScanArgs& a, size_t* bytes) {
  const int grid = scan_grid(a);
  *bytes = size_t(grid) * size_t(a.nq > 0 ? a.nq : 1) * a.k * (sizeof(float) + sizeof(int32_t));
  return FRG_OK;
}

template <int NJ, int QB, int METRIC>
static int launch_one(const ScanArgs& a, int grid, int q0, int nq_pass, float* part_sc, int32_t* part_ix,
                      cudaStream_t st) {
  const size_t smem = size_t(kScanWarps) * QB * a.k * (sizeof(float) + sizeof(int32_t));
  scan_f32_kernel<NJ, QB, METRIC><<<grid, kScanWarps * 32, smem, st>>>(
      a.master, a.tags, a.rows, a.qn, a.nq, q0, nq_pass, a.k, a.tenant, part_sc, part_ix);
  note_launch(nullptr);
  FRG_CUDA(cudaGetLastError());
  return FRG_OK;
}

template <int NJ, int QB>
static int launch_metric(const ScanArgs& a, int grid, int q0, int nq_pass, float* ps, int32_t* pi, cudaStream_t st) {
  if (a.metric == FRG_METRIC_COSINE) return launch_one<NJ, QB, FRG_METRIC_COSINE>(a, grid, q0, nq_pass, ps, pi, st);
  return launch_one<NJ, QB, FRG_METRIC_EUCLIDEAN>(a, grid, q0, nq_pass, ps, pi, st);
}

template <int NJ>
static int launch_qb(const ScanArgs& a, int qb, int grid, int q0, int nq_pass, float* ps, int32_t* pi, cudaStream_t st) {
  if (qb == 1) return launch_metric<NJ, 1>(a, grid, q0, nq_pass, ps, pi, st);
  if (qb == 2) return launch_metric<NJ, 2>(a, grid, q0, nq_pass, ps, pi, st);
  if constexpr (NJ <= 4) { if (qb == 4) return launch_metric<NJ, 4>(a, grid, q0, nq_pass, ps, pi, st); }
  if constexpr (NJ <= 2) { if (qb == 8) return launch_metric<NJ, 8>(a, grid, q0, nq_pass, ps, pi, st); }
  set_error("scan_f32: unsupported queries-per-pass %d for dim %d", qb, NJ * 128);
  return FRG_ERR_UNSUPPORTED;
}

int launch_scan_f32(const ScanArgs& a, void* workspace, int64_t row_offset, float threshold,
                    int64_t* out_rows, float* out_scores, uint8_t* out_accept, cudaStream_t st) {
  if (a.dim != 128 && a.dim != 256 && a.dim != 512 && a.dim != 1024) {
    set_error("scan_f32: dim %d not built (128, 256, 512, 1024)", a.dim);
    return FRG_ERR_UNSUPPORTED;
  }
  if (a.k < 1 || a.k > FRG_MAX_K) { set_error("k=%d out of range 1..%d", a.k, FRG_MAX_K); return FRG_ERR_INVALID; }
  if (a.rows > 0x7fffffff) { set_error("scan_f32: more than 2^31-1 rows in one shard"); return FRG_ERR_UNSUPPORTED; }
  const int grid = a.rows > 0 ? scan_grid(a) : 0;
  float* part_sc = static_cast<float*>(workspace);
  int32_t* part_ix = reinterpret_cast<int32_t*>(part_sc + size_t(grid > 0 ? grid : 1) * a.nq * a.k);
  if (a.rows > 0) {
    const int qb = scan_qb(a.dim, a.nq);
    profile_begin(st);
    int passes = 0;
    for (int q0 = 0; q0 < a.nq; q0 += qb) {
      ++passes;
      const int nq_pass = a.nq - q0 < qb ? a.nq - q0 : qb;
      int rc;
      switch (a.dim) {
        case 128: rc = launch_qb<1>(a, qb, grid, q0, nq_pass, part_sc, part_ix, st); break;
        case 256: rc = launch_qb<2>(a, qb, grid, q0, nq_pass, part_sc, part_ix, st); break;
        case 512: rc = launch_qb<4>(a, qb, grid, q0, nq_pass, part_sc, part_ix, st); break;
        default:  rc = launch_qb<8>(a, qb, grid, q0, nq_pass, part_sc, part_ix, st); break;
      }
      FRG_CHECK(rc);
    }
    profile_end(st, passes);
  }
  return launch_merge_i32(part_sc, part_ix, grid, a.nq, a.k, a.k, a.metric, threshold, row_offset,
                          /*finalize_euclid=*/a.metric == FRG_METRIC_EUCLIDEAN, out_rows, out_scores,
                          out_accept, st);
}

template <int NJ, int QB, int KMAX>
static int launch_flagged_k(const ScanArgs& a, int grid, const int* flagged, int* ctl, float threshold,
                            int64_t row_offset, float* ps, int32_t* pi, const XPush& push, int64_t* out_rows,
                            float* out_scores, uint8_t* out_accept, cudaStream_t st) {
  const size_t smem = size_t(kScanWarps) * QB * a.k * (sizeof(float) + sizeof(int32_t));
  // a tenant-filtered call whose queries overflowed: the tenant's rows are concentrated inside a wide window
  // (DESIGN.md section 4.4) - read the tags first and fetch only that tenant's rows
  if (a.master && a.metric == FRG_METRIC_COSINE && a.tenant >= 0) {
    auto kern = scan_f32_flagged_kernel<NJ, QB, FRG_METRIC_COSINE, KMAX, float, true>;
    FRG_CUDA(func_attr_once(kern, cudaFuncAttributePreferredSharedMemoryCarveout, 100));
    FRG_CUDA(launch_kernel(kern, dim3(grid), dim3(kScanWarps * 32), smem, st, a.master, a.tags, a.rows, a.qn,
                           a.nq, flagged, ctl, a.k, a.tenant, threshold, row_offset, ps, pi, out_rows, out_scores,
                           out_accept, push));
  } else if (a.master && a.metric == FRG_METRIC_EUCLIDEAN) {
    auto kern = scan_f32_flagged_kernel<NJ, QB, FRG_METRIC_EUCLIDEAN, KMAX, float, false>;
    FRG_CUDA(func_attr_once(kern, cudaFuncAttributePreferredSharedMemoryCarveout, 100));
    FRG_CUDA(launch_kernel(kern, dim3(grid), dim3(kScanWarps * 32), smem, st, a.master, a.tags, a.rows, a.qn,
                           a.nq, flagged, ctl, a.k, a.tenant, threshold, row_offset, ps, pi, out_rows, out_scores,
                           out_accept, push));
  } else if (a.master) {
    auto kern = scan_f32_flagged_kernel<NJ, QB, FRG_METRIC_COSINE, KMAX, float, false>;
    FRG_CUDA(func_attr_once(kern, cudaFuncAttributePreferredSharedMemoryCarveout, 100));
    FRG_CUDA(launch_kernel(kern, dim3(grid), dim3(kScanWarps * 32), smem, st, a.master, a.tags, a.rows, a.qn,
                           a.nq, flagged, ctl, a.k, a.tenant, threshold, row_offset, ps, pi, out_rows, out_scores,
                           out_accept, push));
  } else {
    // bf16-only store: the exact re-do reads the scan plane (fp32 query x bf16 row, fp32 accumulation)
    auto kern = scan_f32_flagged_kernel<NJ, QB, FRG_METRIC_COSINE, KMAX, __nv_bfloat16, false>;
    FRG_CUDA(func_attr_once(kern, cudaFuncAttributePreferredSharedMemoryCarveout, 100));
    FRG_CUDA(launch_kernel(kern, dim3(grid), dim3(kScanWarps * 32), smem, st, a.plane, a.tags, a.rows, a.qn,
                           a.nq, flagged, ctl, a.k, a.tenant, threshold, row_offset, ps, pi, out_rows, out_scores,
                           out_accept, push));
  }
  note_launch(nullptr);
  FRG_CUDA(cudaGetLastError());
  return FRG_OK;
}

template <int NJ, int QB>
static int launch_flagged_t(const ScanArgs& a, int grid, const int* flagged, int* ctl, float threshold,
                            int64_t row_offset, float* ps, int32_t* pi, const XPush& push, int64_t* out_rows,
                            float* out_scores, uint8_t* out_accept, cudaStream_t st) {
  if (a.k == 1) return launch_flagged_k<NJ, QB, 1>(a, grid, flagged, ctl, threshold, row_offset, ps, pi, push, out_rows, out_scores, out_accept, st);
  if (a.k <= 4) return launch_flagged_k<NJ, QB, 4>(a, grid, flagged, ctl, threshold, row_offset, ps, pi, push, out_rows, out_scores, out_accept, st);
  if (a.k <= 8) return launch_flagged_k<NJ, QB, 8>(a, grid, flagged, ctl, threshold, row_offset, ps, pi, push, out_rows, out_scores, out_accept, st);
  return launch_flagged_k<NJ, QB, 16>(a, grid, flagged, ctl, threshold, row_offset, ps, pi, push, out_rows, out_scores, out_accept, st);
}

// ctl: device int[2] = {number of flagged queries, ticket counter (0)}
int launch_scan_f32_flagged(const ScanArgs& a, const int* flagged, int* ctl, int64_t row_offset,
                            float threshold, const XPush& push, int64_t* out_rows, float* out_scores,
                            uint8_t* out_accept, cudaStream_t st) {
  if (a.rows <= 0 || a.nq <= 0) return FRG_OK;
  const int grid = a.sm_count;       // partial lists are sized for the worst case (every query flagged)
  const size_t n_part = size_t(grid) * a.nq * a.k;
  unsigned char* ws = nullptr;
  FRG_CUDA(cudaMallocAsync(reinterpret_cast<void**>(&ws), n_part * 8, st));
  float* ps = reinterpret_cast<float*>(ws);
  int32_t* pi = reinterpret_cast<int32_t*>(ps + n_part);
  int rc;
  switch (a.dim) {
    case 128: rc = launch_flagged_t<1, 4>(a, grid, flagged, ctl, threshold, row_offset, ps, pi, push, out_rows, out_scores, out_accept, st); break;
    case 256: rc = launch_flagged_t<2, 4>(a, grid, flagged, ctl, threshold, row_offset, ps, pi, push, out_rows, out_scores, out_accept, st); break;
    case 512: rc = launch_flagged_t<4, 4>(a, grid, flagged, ctl, threshold, row_offset, ps, pi, push, out_rows, out_scores, out_accept, st); break;
    default: set_error("flagged scan: dim %d not built", a.dim); rc = FRG_ERR_UNSUPPORTED; break;
  }
  cudaError_t e = cudaFreeAsync(ws, st);
  if (rc == FRG_OK && e != cudaSuccess) rc = cuda_fail(e, "cudaFreeAsync", __FILE__, __LINE__);
  return rc;
}


// ------------------------------------------------------------------------------------------ range search
// Exact, counting range scan (frg_match_range: the SCAN_F32 variant over all queries, and the tensor-core path's
// fallback over the flagged ones).  Deterministic and sort-free: warp gw of W owns the contiguous rows
// [gw * rows / W, (gw + 1) * rows / W), so the concatenation of the warps' hits in warp order IS gallery order.
//   pass 1 (range_count_kernel):  per (query, warp) hit count -> cnt[slot][W]
//   range_offsets_kernel:         per query, exclusive scan over the W counts -> off[slot][W], total -> out_counts;
//                                 the slots past min(total, max_hits) get the "none" marker
//   pass 2 (range_write_kernel):  a warp with hits whose offset is below max_hits recomputes its rows and writes
//                                 its hits at off, off + 1, ... (row order) while they are below max_hits
// Scores come from row_dots + butterfly, the arithmetic of scan_pass: bit-identical to the other exact paths.
// Queries are taken QB at a time (slot = position in `flagged`, or the query itself); the number of slots is read
// on the device, so with nothing flagged every launch exits at once.
__device__ __forceinline__ int64_t range_warp_row(int64_t rows, int64_t w, int64_t nw) { return rows * w / nw; }

template <int METRIC>
__device__ __forceinline__ bool range_pass(float sdot, float threshold, int strict) {
  if (METRIC == FRG_METRIC_COSINE) return strict ? (sdot > threshold) : (sdot >= threshold);   // false for NaN
  const float d = __fsqrt_rn(sdot);                                                            // sdot = d^2 >= 0
  return strict ? (d < threshold) : (d <= threshold);
}

template <int NJ, int QB, int METRIC, bool WRITE>
__global__ void __launch_bounds__(kScanWarps * 32, 2)
range_scan_kernel(const float* __restrict__ master, const int32_t* __restrict__ tags, int64_t rows,
                  const float* __restrict__ qn, int nq, const int* __restrict__ flagged,
                  const int* __restrict__ n_flagged, int32_t tenant, float threshold, int strict, int max_hits,
                  int64_t row_offset, int* __restrict__ cnt, const int* __restrict__ off,
                  int64_t* __restrict__ out_rows, float* __restrict__ out_scores) {
  constexpr int DIM = NJ * 128;
  pdl_wait();
  pdl_trigger();
  const int n_slots = flagged ? *n_flagged : nq;
  const int lane = threadIdx.x & 31;
  const int64_t nw = int64_t(gridDim.x) * kScanWarps;
  const int64_t gw = int64_t(blockIdx.x) * kScanWarps + (threadIdx.x >> 5);
  const int64_t r0 = range_warp_row(rows, gw, nw), r1 = range_warp_row(rows, gw + 1, nw);
  const int my_b = lane_query<QB>(lane);
  const bool rep = lane_is_rep<QB>(lane);
  for (int s0 = 0; s0 < n_slots; s0 += QB) {
    const int nb = n_slots - s0 < QB ? n_slots - s0 : QB;
    const int slot = s0 + (my_b < nb ? my_b : 0);
    const int q = flagged ? flagged[slot] : slot;
    // pass 2: this lane's query needs this warp iff the warp has hits that land below max_hits
    int pos = 0, room = 0;
    if (WRITE) {
      if (my_b < nb && cnt[size_t(slot) * nw + gw] > 0) {
        pos = off[size_t(slot) * nw + gw];
        room = max_hits;
      }
      if (!__any_sync(0xffffffffu, pos < room)) continue;
    }
    float4 qv[QB][NJ];
#pragma unroll
    for (int b = 0; b < QB; ++b) {
      const int qb_ = flagged ? flagged[s0 + (b < nb ? b : 0)] : s0 + (b < nb ? b : 0);
#pragma unroll
      for (int j = 0; j < NJ; ++j) qv[b][j] = __ldg(reinterpret_cast<const float4*>(qn + size_t(qb_) * DIM) + j * 32 + lane);
    }
    int count = 0;
    for (int64_t r = r0; r < r1; ++r) {
      const int32_t tg = __ldg(tags + r);
      float4 g[NJ];                                                     // issued together with the tag load
      const float4* pr = reinterpret_cast<const float4*>(master + r * DIM) + lane;
#pragma unroll
      for (int j = 0; j < NJ; ++j) g[j] = ldg_stream(pr + j * 32);
      if (tg < 0 || (tenant >= 0 && tg != tenant)) continue;           // warp-uniform
      float a[QB];
      row_dots<NJ, QB, METRIC>(g, qv, a);
      const float sdot = butterfly<QB>(a, lane);
      const bool hit = my_b < nb && range_pass<METRIC>(sdot, threshold, strict);
      if (WRITE) {
        if (hit && pos < room) {
          if (rep) {
            out_rows[size_t(q) * max_hits + pos] = r + row_offset;
            out_scores[size_t(q) * max_hits + pos] = METRIC == FRG_METRIC_COSINE ? sdot : __fsqrt_rn(sdot);
          }
          ++pos;
        }
        if (!__any_sync(0xffffffffu, pos < room)) break;
      } else {
        count += hit ? 1 : 0;
      }
    }
    if (!WRITE && rep && my_b < nb) cnt[size_t(slot) * nw + gw] = count;
  }
}

// one CTA per slot: exclusive scan of the slot's nw warp counts (each thread a contiguous strip, then a block scan
// of the strip sums), the total, and the "none" marker in the unused output slots
__global__ void __launch_bounds__(256)
range_offsets_kernel(int nq, const int* __restrict__ flagged, const int* __restrict__ n_flagged, int nw,
                     const int* __restrict__ cnt, int* __restrict__ off, int max_hits, float none_score,
                     int64_t* __restrict__ out_counts, int64_t* __restrict__ out_rows, float* __restrict__ out_scores) {
  __shared__ long long part[256];
  pdl_wait();
  pdl_trigger();
  const int slot = blockIdx.x;
  if (slot >= (flagged ? *n_flagged : nq)) return;
  const int q = flagged ? flagged[slot] : slot;
  const int t = threadIdx.x;
  const int per = (nw + blockDim.x - 1) / blockDim.x;
  const int a = t * per < nw ? t * per : nw, b = a + per < nw ? a + per : nw;
  const int* c = cnt + size_t(slot) * nw;
  long long sum = 0;
  for (int i = a; i < b; ++i) sum += c[i];
  part[t] = sum;
  __syncthreads();
  for (int o = 1; o < int(blockDim.x); o <<= 1) {          // Hillis-Steele inclusive scan
    const long long v = t >= o ? part[t - o] : 0;
    __syncthreads();
    part[t] += v;
    __syncthreads();
  }
  long long run = part[t] - sum;
  int* o_ = off + size_t(slot) * nw;
  for (int i = a; i < b; ++i) {
    o_[i] = run < max_hits ? int(run) : max_hits;
    run += c[i];
  }
  const long long total = part[blockDim.x - 1];
  if (t == 0) out_counts[q] = total;
  for (long long i = (total < max_hits ? total : max_hits) + t; i < max_hits; i += blockDim.x) {
    out_rows[size_t(q) * max_hits + i] = kNoRow;
    out_scores[size_t(q) * max_hits + i] = none_score;
  }
}

int range_scan_supported(int dim, const char** why) {
  if (dim != 128 && dim != 256 && dim != 512 && dim != 1024) { *why = "the range scan is built for dim 128, 256, 512 and 1024"; return 0; }
  return 1;
}

template <int NJ, int QB, int METRIC>
static int launch_range_passes(const ScanArgs& a, int grid, const int* flagged, const int* n_flagged, int max_hits,
                               float threshold, bool strict, int64_t row_offset, int* cnt, int* off,
                               int64_t* out_counts, int64_t* out_rows, float* out_scores, cudaStream_t st) {
  const int nw = grid * kScanWarps;
  const int s = strict ? 1 : 0;
  FRG_CUDA(launch_kernel(range_scan_kernel<NJ, QB, METRIC, false>, dim3(grid), dim3(kScanWarps * 32), 0, st,
                         a.master, a.tags, a.rows, a.qn, a.nq, flagged, n_flagged, a.tenant, threshold, s, max_hits,
                         row_offset, cnt, off, out_rows, out_scores));
  note_launch(nullptr);
  FRG_CUDA(launch_kernel(range_offsets_kernel, dim3(a.nq), dim3(256), 0, st, a.nq, flagged, n_flagged, nw, cnt,
                         off, max_hits, METRIC == FRG_METRIC_COSINE ? kNoScore : INFINITY, out_counts, out_rows,
                         out_scores));
  note_launch(nullptr);
  FRG_CUDA(launch_kernel(range_scan_kernel<NJ, QB, METRIC, true>, dim3(grid), dim3(kScanWarps * 32), 0, st,
                         a.master, a.tags, a.rows, a.qn, a.nq, flagged, n_flagged, a.tenant, threshold, s, max_hits,
                         row_offset, cnt, off, out_rows, out_scores));
  note_launch(nullptr);
  FRG_CUDA(cudaGetLastError());
  return FRG_OK;
}

template <int NJ, int QB>
static int launch_range_m(const ScanArgs& a, int grid, const int* flagged, const int* n_flagged, int max_hits,
                          float threshold, bool strict, int64_t row_offset, int* cnt, int* off, int64_t* out_counts,
                          int64_t* out_rows, float* out_scores, cudaStream_t st) {
  if (a.metric == FRG_METRIC_COSINE)
    return launch_range_passes<NJ, QB, FRG_METRIC_COSINE>(a, grid, flagged, n_flagged, max_hits, threshold, strict,
                                                          row_offset, cnt, off, out_counts, out_rows, out_scores, st);
  return launch_range_passes<NJ, QB, FRG_METRIC_EUCLIDEAN>(a, grid, flagged, n_flagged, max_hits, threshold, strict,
                                                           row_offset, cnt, off, out_counts, out_rows, out_scores, st);
}

template <int NJ>
static int launch_range_qb(const ScanArgs& a, int qb, int grid, const int* flagged, const int* n_flagged,
                           int max_hits, float threshold, bool strict, int64_t row_offset, int* cnt, int* off,
                           int64_t* out_counts, int64_t* out_rows, float* out_scores, cudaStream_t st) {
#define FRG_RANGE_QB(QB) return launch_range_m<NJ, QB>(a, grid, flagged, n_flagged, max_hits, threshold, strict, \
                                                      row_offset, cnt, off, out_counts, out_rows, out_scores, st)
  if (qb == 1) { FRG_RANGE_QB(1); }
  if (qb == 2) { FRG_RANGE_QB(2); }
  if constexpr (NJ <= 4) { if (qb == 4) { FRG_RANGE_QB(4); } }
  if constexpr (NJ <= 2) { if (qb == 8) { FRG_RANGE_QB(8); } }
#undef FRG_RANGE_QB
  set_error("range scan: unsupported queries-per-pass %d for dim %d", qb, NJ * 128);
  return FRG_ERR_UNSUPPORTED;
}

int launch_range_scan(const ScanArgs& a, const int* flagged, const int* n_flagged, int max_hits, float threshold,
                      bool strict, int64_t row_offset, int64_t* out_counts, int64_t* out_rows, float* out_scores,
                      cudaStream_t st) {
  const char* why = "";
  if (!range_scan_supported(a.dim, &why)) { set_error("range scan: %s", why); return FRG_ERR_UNSUPPORTED; }
  if (a.nq <= 0) return FRG_OK;
  if (flagged && a.rows <= 0) return FRG_OK;
  // the same rows-in-flight sizing as the top-k scan; at least one warp, so an empty gallery still gets its counts
  const int grid = scan_grid(a);
  const size_t n_cnt = size_t(grid) * kScanWarps * a.nq;
  unsigned char* ws = nullptr;
  FRG_CUDA(cudaMallocAsync(reinterpret_cast<void**>(&ws), n_cnt * 2 * sizeof(int), st));
  int* cnt = reinterpret_cast<int*>(ws);
  int* off = cnt + n_cnt;
  const int qb = scan_qb(a.dim, a.nq);
  int rc;
  switch (a.dim) {
    case 128: rc = launch_range_qb<1>(a, qb, grid, flagged, n_flagged, max_hits, threshold, strict, row_offset, cnt, off, out_counts, out_rows, out_scores, st); break;
    case 256: rc = launch_range_qb<2>(a, qb, grid, flagged, n_flagged, max_hits, threshold, strict, row_offset, cnt, off, out_counts, out_rows, out_scores, st); break;
    case 512: rc = launch_range_qb<4>(a, qb, grid, flagged, n_flagged, max_hits, threshold, strict, row_offset, cnt, off, out_counts, out_rows, out_scores, st); break;
    default:  rc = launch_range_qb<8>(a, qb, grid, flagged, n_flagged, max_hits, threshold, strict, row_offset, cnt, off, out_counts, out_rows, out_scores, st); break;
  }
  cudaError_t e = cudaFreeAsync(ws, st);
  if (rc == FRG_OK && e != cudaSuccess) rc = cuda_fail(e, "cudaFreeAsync", __FILE__, __LINE__);
  return rc;
}

// ------------------------------------------------------------------------------------------ gallery self-join
// range_scan_kernel with the join rules (cosine): query q of the slab is the stored row a = qrow0 + q, and row b counts
// for it only when b > a and (same_tag) tag[b] == tag[a]; a dead query, or one outside the tenant, counts nothing.  A
// pass of QB queries reads only the rows [lowest live a + 1, largest plan end of its queries), split into contiguous
// strips in warp order as range_scan_kernel splits the whole gallery, so pass 2 finds the same strips and the
// concatenation of the warps' hits is gallery order.  The scores come from row_dots + butterfly: bit-identical.
template <int NJ, int QB, bool WRITE>
__global__ void __launch_bounds__(kScanWarps * 32, 2)
join_scan_kernel(const float* __restrict__ master, const int32_t* __restrict__ tags, const float* __restrict__ qn,
                 int nq, int64_t qrow0, const int32_t* __restrict__ tile_end, const int* __restrict__ flagged,
                 const int* __restrict__ n_flagged, int32_t tenant, int same_tag, float threshold, int strict,
                 int max_hits, int64_t row_offset, int* __restrict__ cnt, const int* __restrict__ off,
                 int64_t* __restrict__ out_rows, float* __restrict__ out_scores) {
  constexpr int DIM = NJ * 128;
  pdl_wait();
  pdl_trigger();
  const int n_slots = flagged ? *n_flagged : nq;
  const int lane = threadIdx.x & 31;
  const int64_t nw = int64_t(gridDim.x) * kScanWarps;
  const int64_t gw = int64_t(blockIdx.x) * kScanWarps + (threadIdx.x >> 5);
  const int my_b = lane_query<QB>(lane);
  const bool rep = lane_is_rep<QB>(lane);
  for (int s0 = 0; s0 < n_slots; s0 += QB) {
    const int nb = n_slots - s0 < QB ? n_slots - s0 : QB;
    const int slot = s0 + (my_b < nb ? my_b : 0);
    const int q = flagged ? flagged[slot] : slot;
    const int a = int(qrow0 + q);                                     // rows < 2^31 (frg_self_join)
    const int32_t ta = __ldg(tags + a);
    const bool live = my_b < nb && ta >= 0 && (tenant < 0 || ta == tenant);
    // rows of this pass: [lowest live a + 1, largest plan end); none when no query of the pass is live
    const int lo = __reduce_min_sync(0xffffffffu, live ? a + 1 : 0x7fffffff);
    const int hi = __reduce_max_sync(0xffffffffu, live ? __ldg(tile_end + q / 128) : 0);
    const int64_t span = hi > lo ? int64_t(hi - lo) : 0;
    const int64_t r0 = lo + span * gw / nw, r1 = lo + span * (gw + 1) / nw;
    int pos = 0, room = 0;
    if (WRITE) {
      if (my_b < nb && cnt[size_t(slot) * nw + gw] > 0) {
        pos = off[size_t(slot) * nw + gw];
        room = max_hits;
      }
      if (!__any_sync(0xffffffffu, pos < room)) continue;
    }
    float4 qv[QB][NJ];
#pragma unroll
    for (int b = 0; b < QB; ++b) {
      const int qb_ = flagged ? flagged[s0 + (b < nb ? b : 0)] : s0 + (b < nb ? b : 0);
#pragma unroll
      for (int j = 0; j < NJ; ++j) qv[b][j] = __ldg(reinterpret_cast<const float4*>(qn + size_t(qb_) * DIM) + j * 32 + lane);
    }
    int count = 0;
    for (int64_t r = r0; r < r1; ++r) {
      const int32_t tg = __ldg(tags + r);
      float4 g[NJ];                                                     // issued together with the tag load
      const float4* pr = reinterpret_cast<const float4*>(master + r * DIM) + lane;
#pragma unroll
      for (int j = 0; j < NJ; ++j) g[j] = ldg_stream(pr + j * 32);
      if (tg < 0 || (tenant >= 0 && tg != tenant)) continue;           // warp-uniform
      const bool mine = live && r > a && (!same_tag || tg == ta);
      if (!__any_sync(0xffffffffu, mine)) continue;
      float acc[QB];
      row_dots<NJ, QB, FRG_METRIC_COSINE>(g, qv, acc);
      const float sdot = butterfly<QB>(acc, lane);
      const bool hit = mine && range_pass<FRG_METRIC_COSINE>(sdot, threshold, strict);
      if (WRITE) {
        if (hit && pos < room) {
          if (rep) {
            out_rows[size_t(q) * max_hits + pos] = r + row_offset;
            out_scores[size_t(q) * max_hits + pos] = sdot;
          }
          ++pos;
        }
        if (!__any_sync(0xffffffffu, pos < room)) break;
      } else {
        count += hit ? 1 : 0;
      }
    }
    if (!WRITE && rep && my_b < nb) cnt[size_t(slot) * nw + gw] = count;
  }
}

size_t join_scan_workspace_bytes(const ScanArgs& a) {
  return size_t(scan_grid(a)) * kScanWarps * size_t(a.nq > 0 ? a.nq : 1) * 2 * sizeof(int);
}

template <int NJ, int QB>
static int launch_join_passes(const ScanArgs& a, int grid, int64_t qrow0, const int32_t* tile_end, bool same_tag,
                              const int* flagged, const int* n_flagged, int max_hits, float threshold, bool strict,
                              int64_t row_offset, int* cnt, int* off, int64_t* out_counts, int64_t* out_rows,
                              float* out_scores, cudaStream_t st) {
  const int nw = grid * kScanWarps;
  const int s = strict ? 1 : 0, t = same_tag ? 1 : 0;
  FRG_CUDA(launch_kernel(join_scan_kernel<NJ, QB, false>, dim3(grid), dim3(kScanWarps * 32), 0, st, a.master, a.tags,
                         a.qn, a.nq, qrow0, tile_end, flagged, n_flagged, a.tenant, t, threshold, s, max_hits,
                         row_offset, cnt, const_cast<const int*>(off), out_rows, out_scores));
  note_launch(nullptr);
  FRG_CUDA(launch_kernel(range_offsets_kernel, dim3(a.nq), dim3(256), 0, st, a.nq, flagged, n_flagged, nw,
                         const_cast<const int*>(cnt), off, max_hits, kNoScore, out_counts, out_rows, out_scores));
  note_launch(nullptr);
  FRG_CUDA(launch_kernel(join_scan_kernel<NJ, QB, true>, dim3(grid), dim3(kScanWarps * 32), 0, st, a.master, a.tags,
                         a.qn, a.nq, qrow0, tile_end, flagged, n_flagged, a.tenant, t, threshold, s, max_hits,
                         row_offset, cnt, const_cast<const int*>(off), out_rows, out_scores));
  note_launch(nullptr);
  FRG_CUDA(cudaGetLastError());
  return FRG_OK;
}

template <int NJ>
static int launch_join_qb(const ScanArgs& a, int qb, int grid, int64_t qrow0, const int32_t* tile_end, bool same_tag,
                          const int* flagged, const int* n_flagged, int max_hits, float threshold, bool strict,
                          int64_t row_offset, int* cnt, int* off, int64_t* out_counts, int64_t* out_rows,
                          float* out_scores, cudaStream_t st) {
#define FRG_JOIN_QB(QB) return launch_join_passes<NJ, QB>(a, grid, qrow0, tile_end, same_tag, flagged, n_flagged,     \
                                                         max_hits, threshold, strict, row_offset, cnt, off, out_counts, \
                                                         out_rows, out_scores, st)
  if (qb == 1) { FRG_JOIN_QB(1); }
  if (qb == 2) { FRG_JOIN_QB(2); }
  if constexpr (NJ <= 4) { if (qb == 4) { FRG_JOIN_QB(4); } }
  if constexpr (NJ <= 2) { if (qb == 8) { FRG_JOIN_QB(8); } }
#undef FRG_JOIN_QB
  set_error("join scan: unsupported queries-per-pass %d for dim %d", qb, NJ * 128);
  return FRG_ERR_UNSUPPORTED;
}

int launch_join_scan(const ScanArgs& a, int64_t qrow0, const int32_t* tile_end, bool same_tag, const int* flagged,
                     const int* n_flagged, int max_hits, float threshold, bool strict, int64_t row_offset, void* ws,
                     int64_t* out_counts, int64_t* out_rows, float* out_scores, cudaStream_t st) {
  const char* why = "";
  if (!range_scan_supported(a.dim, &why)) { set_error("join scan: %s", why); return FRG_ERR_UNSUPPORTED; }
  if (a.nq <= 0) return FRG_OK;
  const int grid = scan_grid(a);
  int* cnt = static_cast<int*>(ws);
  int* off = cnt + size_t(grid) * kScanWarps * a.nq;
  const int qb = scan_qb(a.dim, a.nq);
  switch (a.dim) {
    case 128: return launch_join_qb<1>(a, qb, grid, qrow0, tile_end, same_tag, flagged, n_flagged, max_hits, threshold, strict, row_offset, cnt, off, out_counts, out_rows, out_scores, st);
    case 256: return launch_join_qb<2>(a, qb, grid, qrow0, tile_end, same_tag, flagged, n_flagged, max_hits, threshold, strict, row_offset, cnt, off, out_counts, out_rows, out_scores, st);
    case 512: return launch_join_qb<4>(a, qb, grid, qrow0, tile_end, same_tag, flagged, n_flagged, max_hits, threshold, strict, row_offset, cnt, off, out_counts, out_rows, out_scores, st);
    default:  return launch_join_qb<8>(a, qb, grid, qrow0, tile_end, same_tag, flagged, n_flagged, max_hits, threshold, strict, row_offset, cnt, off, out_counts, out_rows, out_scores, st);
  }
}

}  // namespace frg
