// Gallery-store kernels: ingest (normalise + write master / scan plane (bf16 or int8) / tag), tombstone, stable
// gather (compaction) and the synthetic generator.  All are HBM-bound row movers: one warp per
// row, 16-byte accesses, no shared memory.
#include "frg_internal.cuh"

namespace frg {

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

// writes the bf16 image of v and returns ||v - bf16(v)||^2 of the four elements (each difference is exact in fp32)
__device__ __forceinline__ float store_bf16x4(__nv_bfloat16* dst, float4 v) {
  __nv_bfloat162 lo = __floats2bfloat162_rn(v.x, v.y);
  __nv_bfloat162 hi = __floats2bfloat162_rn(v.z, v.w);
  uint2 packed;
  packed.x = *reinterpret_cast<uint32_t*>(&lo);
  packed.y = *reinterpret_cast<uint32_t*>(&hi);
  *reinterpret_cast<uint2*>(dst) = packed;
  const float2 l = __bfloat1622float2(lo), h = __bfloat1622float2(hi);
  const float a = v.x - l.x, b = v.y - l.y, c = v.z - h.x, d = v.w - h.y;
  return fmaf(a, a, fmaf(b, b, fmaf(c, c, d * d)));
}

// writes the int8 image of v (step c: element = clamp(rint(x / c), -127, 127), NaN -> 0) and returns ||v - c * i8(v)||^2
// of the four elements.  Saturated elements are clamped, not wrapped: their larger residual is part of the sum.
__device__ __forceinline__ float store_i8x4(int8_t* dst, float4 v, float c) {
  const float x[4] = {v.x, v.y, v.z, v.w};
  uint32_t packed = 0;
  float rr = 0.f;
#pragma unroll
  for (int e = 0; e < 4; ++e) {
    float t = rintf(__fdiv_rn(x[e], c));
    t = t == t ? fminf(fmaxf(t, -127.f), 127.f) : 0.f;
    const float d = fmaf(-t, c, x[e]);
    rr = fmaf(d, d, rr);
    packed |= (uint32_t(int(t)) & 0xFFu) << (8 * e);
  }
  *reinterpret_cast<uint32_t*>(dst) = packed;
  return rr;
}

// The tensor-core filter's error bound is DATA-DEPENDENT and rigorous: |q^.g^ - q.g| <= ||q^|| ||g^ - g|| +
// ||q^ - q|| ||g|| (q^, g^ the bf16 images, or the int8 images times their steps).  bounds[1] keeps the largest ||g^ - g||^2 of any row ever stored
// (non-negative floats order like their bit patterns); the query side is measured per query (queries.cu).
// A NaN row (zero vector) is left out: it can never match either way.
__device__ __forceinline__ float fold_residual(uint32_t* bounds, float rr, int lane) {
  rr = warp_sum(rr);
  if (bounds && lane == 0 && rr < INFINITY) atomicMax(bounds + 1, __float_as_uint(rr));
  return rr;                // the row's ||g - bf16(g)||^2, on every lane
}

// Euclidean scan plane (raw stores): columns dim .. dim+15 of the row = [hi, mid, lo, 0 ...], the exact
// three-term bf16 split of c = -0.5 * ||g||^2 (24 significand bits = 3 x 8), so that the tensor-core
// product with a query image [q, 1, 1, 1, 0 ...] accumulates q.g - 0.5*||g||^2.  The largest ||g||^2
// ever stored is folded into gmax_bits[0] (non-negative floats order like their bit patterns); it scales
// the filter's error bound.  Non-finite norms are left out: such rows can never match either way.
// Columns 3..5 carry THIS ROW's share of the filter's error bound, each rounded UP to bf16: R = ||g - bf16(g)||,
// N = ||g||, SS = ||g||^2.  The query image holds the matching coefficients (queries.cu), so the tensor core
// itself adds (filter) or subtracts (pre-pass) the bound: scores come out as upper / lower bounds of the exact
// score, per row - one row of huge norm no longer loosens the bound of every other row.
__device__ __forceinline__ uint32_t bf16_up(float x) {          // smallest bf16 >= x, for x >= 0 (bits)
  __nv_bfloat16 b = __float2bfloat16_rn(x);
  uint32_t u = __bfloat16_as_ushort(b);
  if (__bfloat162float(b) < x) ++u;                              // next bf16 up (x >= 0: bit patterns are ordered)
  return u;
}
__device__ __forceinline__ void store_bias_columns(__nv_bfloat16* row_aug, float ss, float rr, uint32_t* gmax_bits,
                                                   int lane) {
  if (lane < kEuclidPad / 4) {
    uint2 packed = make_uint2(0u, 0u);
    if (lane == 0) {
      const float c = -0.5f * ss;
      const __nv_bfloat16 hi = __float2bfloat16_rn(c);
      const float r1 = c - __bfloat162float(hi);
      const __nv_bfloat16 mid = __float2bfloat16_rn(r1);
      const float r2 = r1 - __bfloat162float(mid);
      const __nv_bfloat16 lo = __float2bfloat16_rn(r2);
      packed.x = uint32_t(__bfloat16_as_ushort(hi)) | (uint32_t(__bfloat16_as_ushort(mid)) << 16);
      packed.y = uint32_t(__bfloat16_as_ushort(lo)) | (bf16_up(__fsqrt_ru(rr)) << 16);
      if (gmax_bits && ss < INFINITY) atomicMax(gmax_bits, __float_as_uint(ss));
    } else if (lane == 1) {
      packed.x = bf16_up(__fsqrt_ru(ss)) | (bf16_up(ss) << 16);
    }
    reinterpret_cast<uint2*>(row_aug)[lane] = packed;
  }
}

// `embedding / np.linalg.norm(embedding)` at load time: infrenceServer.py:271,324; peopleCount.py:788,806.
// norm = sqrt(sum x^2) in fp32 (numpy's sdot-based norm; summation order differs by a few ulp).
__global__ void __launch_bounds__(256)
ingest_kernel(const float* __restrict__ vecs, const int64_t* __restrict__ rows,
              const int32_t* __restrict__ tags, int64_t n, int64_t append_at, int64_t limit, int dim,
              int normalise, float* __restrict__ master, __nv_bfloat16* __restrict__ plane,
              int8_t* __restrict__ plane8, float step8, int plane_dim, uint32_t* __restrict__ gmax_bits,
              int32_t* __restrict__ tag_out) {
  const int lane = threadIdx.x & 31;
  const int64_t warp = (int64_t(blockIdx.x) * blockDim.x + threadIdx.x) >> 5;
  const int64_t nwarps = (int64_t(gridDim.x) * blockDim.x) >> 5;
  const int nvec = dim >> 2;
  for (int64_t i = warp; i < n; i += nwarps) {
    const int64_t dst = rows ? rows[i] : append_at + i;
    if (dst < 0 || dst >= limit) continue;   // host-side entry points validate; device callers are skipped
    const float4* src = reinterpret_cast<const float4*>(vecs + i * dim);
    float inv_or_norm = 1.0f;
    if (normalise) {
      float ss = 0.f;
      for (int v = lane; v < nvec; v += 32) {
        float4 x = __ldg(src + v);
        ss = fmaf(x.x, x.x, ss); ss = fmaf(x.y, x.y, ss); ss = fmaf(x.z, x.z, ss); ss = fmaf(x.w, x.w, ss);
      }
      inv_or_norm = __fsqrt_rn(warp_sum(ss));
    }
    float4* m = master ? reinterpret_cast<float4*>(master + dst * dim) : nullptr;   // null: bf16-only store
    float ss_stored = 0.f;                    // ||stored row||^2, for the Euclidean plane's bias columns
    float rr = 0.f;                           // ||row - bf16(row)||^2
    for (int v = lane; v < nvec; v += 32) {
      float4 x = __ldg(src + v);
      if (normalise) {
        x.x = __fdiv_rn(x.x, inv_or_norm); x.y = __fdiv_rn(x.y, inv_or_norm);
        x.z = __fdiv_rn(x.z, inv_or_norm); x.w = __fdiv_rn(x.w, inv_or_norm);
      }
      ss_stored = fmaf(x.x, x.x, ss_stored); ss_stored = fmaf(x.y, x.y, ss_stored);
      ss_stored = fmaf(x.z, x.z, ss_stored); ss_stored = fmaf(x.w, x.w, ss_stored);
      if (m) m[v] = x;
      if (plane) rr += store_bf16x4(plane + dst * plane_dim + v * 4, x);
      if (plane8) rr += store_i8x4(plane8 + dst * dim + v * 4, x, step8);
    }
    if (plane || plane8) rr = fold_residual(gmax_bits, rr, lane);
    if (plane && plane_dim > dim) store_bias_columns(plane + dst * plane_dim + dim, warp_sum(ss_stored), rr, gmax_bits, lane);
    if (lane == 0) tag_out[dst] = tags ? tags[i] : 0;
  }
}

__global__ void tombstone_kernel(const int64_t* __restrict__ rows, int64_t n, int64_t limit,
                                 int32_t* __restrict__ tags) {
  int64_t i = int64_t(blockIdx.x) * blockDim.x + threadIdx.x;
  if (i < n) {
    int64_t r = rows[i];
    if (r >= 0 && r < limit) tags[r] = -1;
  }
}

__global__ void __launch_bounds__(256)
gather_rows_kernel(const int64_t* __restrict__ src_rows, int64_t n, int dim, int plane_row_bytes,
                   const float* __restrict__ master_in, const unsigned char* __restrict__ plane_in,
                   const int32_t* __restrict__ tags_in, float* __restrict__ master_out,
                   unsigned char* __restrict__ plane_out, int32_t* __restrict__ tags_out) {
  const int lane = threadIdx.x & 31;
  const int64_t warp = (int64_t(blockIdx.x) * blockDim.x + threadIdx.x) >> 5;
  const int64_t nwarps = (int64_t(gridDim.x) * blockDim.x) >> 5;
  const int nvec = dim >> 2;
  for (int64_t i = warp; i < n; i += nwarps) {
    const int64_t s = src_rows[i];
    if (master_in) {
      const float4* mi = reinterpret_cast<const float4*>(master_in + s * dim);
      float4* mo = reinterpret_cast<float4*>(master_out + i * dim);
      for (int v = lane; v < nvec; v += 32) mo[v] = mi[v];
    }
    if (plane_in) {
      const uint2* pi = reinterpret_cast<const uint2*>(plane_in + s * plane_row_bytes);
      uint2* po = reinterpret_cast<uint2*>(plane_out + i * plane_row_bytes);
      for (int v = lane; v < (plane_row_bytes >> 3); v += 32) po[v] = pi[v];
    }
    if (lane == 0) tags_out[i] = tags_in[s];
  }
}

// ---- synthetic gallery "frg-synth-v1" (CPU twin: oracle/synth.py) ----------------------------
__device__ __forceinline__ void philox4x32_10(uint32_t c0, uint32_t c1, uint32_t c2, uint32_t c3,
                                              uint32_t k0, uint32_t k1, uint32_t out[4]) {
#pragma unroll
  for (int r = 0; r < 10; ++r) {
    const uint32_t hi0 = __umulhi(0xD2511F53u, c0), lo0 = 0xD2511F53u * c0;
    const uint32_t hi1 = __umulhi(0xCD9E8D57u, c2), lo1 = 0xCD9E8D57u * c2;
    const uint32_t n0 = hi1 ^ c1 ^ k0, n2 = hi0 ^ c3 ^ k1;
    c0 = n0; c1 = lo1; c2 = n2; c3 = lo0;
    k0 += 0x9E3779B9u; k1 += 0xBB67AE85u;
  }
  out[0] = c0; out[1] = c1; out[2] = c2; out[3] = c3;
}

__device__ __forceinline__ int nibble_sum(uint32_t h) {
  return int(h & 0xF) + int((h >> 4) & 0xF) + int((h >> 8) & 0xF) + int((h >> 12) & 0xF) - 30;
}

// one warp per row; lane handles 8-element blocks lane, lane+32, ... (dim/8 blocks, <= 4 per lane
// for dim <= 1024).  sum(x^2) is an exact integer, so norm and quotients are bit-identical to numpy.
__global__ void __launch_bounds__(256)
synth_kernel(int64_t n, int64_t append_at, int64_t global_row0, uint32_t k0, uint32_t k1, int32_t tag,
             int dim, float* __restrict__ master, __nv_bfloat16* __restrict__ plane, int8_t* __restrict__ plane8,
             float step8, int plane_dim, uint32_t* __restrict__ gmax_bits, int32_t* __restrict__ tag_out) {
  const int lane = threadIdx.x & 31;
  const int64_t warp = (int64_t(blockIdx.x) * blockDim.x + threadIdx.x) >> 5;
  const int64_t nwarps = (int64_t(gridDim.x) * blockDim.x) >> 5;
  const int nblk = dim >> 3;
  for (int64_t i = warp; i < n; i += nwarps) {
    const uint64_t g = uint64_t(global_row0 + i);
    const int64_t dst = append_at + i;
    int x[4][8];
    int ss = 0;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const int b = lane + 32 * j;
      if (b < nblk) {
        uint32_t w[4];
        philox4x32_10(uint32_t(g), uint32_t(g >> 32), uint32_t(b), 0u /* stream: gallery */, k0, k1, w);
#pragma unroll
        for (int e = 0; e < 8; ++e) {
          const int v = nibble_sum((w[e >> 1] >> (16 * (e & 1))) & 0xFFFFu);
          x[j][e] = v;
          ss += v * v;
        }
      }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) ss += __shfl_xor_sync(0xffffffffu, ss, o);
    const float norm = __fsqrt_rn(float(ss));
    float ss_stored = 0.f;
    float rr = 0.f;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const int b = lane + 32 * j;
      if (b < nblk) {
        float4 lo, hi;
        lo.x = __fdiv_rn(float(x[j][0]), norm); lo.y = __fdiv_rn(float(x[j][1]), norm);
        lo.z = __fdiv_rn(float(x[j][2]), norm); lo.w = __fdiv_rn(float(x[j][3]), norm);
        hi.x = __fdiv_rn(float(x[j][4]), norm); hi.y = __fdiv_rn(float(x[j][5]), norm);
        hi.z = __fdiv_rn(float(x[j][6]), norm); hi.w = __fdiv_rn(float(x[j][7]), norm);
        if (master) {
          float4* m = reinterpret_cast<float4*>(master + dst * dim + b * 8);
          m[0] = lo; m[1] = hi;
        }
        if (plane) {
          rr += store_bf16x4(plane + dst * plane_dim + b * 8, lo);
          rr += store_bf16x4(plane + dst * plane_dim + b * 8 + 4, hi);
        }
        if (plane8) {
          rr += store_i8x4(plane8 + dst * dim + b * 8, lo, step8);
          rr += store_i8x4(plane8 + dst * dim + b * 8 + 4, hi, step8);
        }
        ss_stored = fmaf(lo.x, lo.x, ss_stored); ss_stored = fmaf(lo.y, lo.y, ss_stored);
        ss_stored = fmaf(lo.z, lo.z, ss_stored); ss_stored = fmaf(lo.w, lo.w, ss_stored);
        ss_stored = fmaf(hi.x, hi.x, ss_stored); ss_stored = fmaf(hi.y, hi.y, ss_stored);
        ss_stored = fmaf(hi.z, hi.z, ss_stored); ss_stored = fmaf(hi.w, hi.w, ss_stored);
      }
    }
    if (plane || plane8) rr = fold_residual(gmax_bits, rr, lane);
    if (plane && plane_dim > dim) store_bias_columns(plane + dst * plane_dim + dim, warp_sum(ss_stored), rr, gmax_bits, lane);
    if (lane == 0) tag_out[dst] = tag;
  }
}

static int grid_for_rows(int64_t n, int warps_per_block) {
  int64_t blocks = (n + warps_per_block - 1) / warps_per_block;
  if (blocks > 148 * 16) blocks = 148 * 16;
  if (blocks < 1) blocks = 1;
  return int(blocks);
}

int launch_ingest(const float* vecs, const int64_t* rows, const int32_t* tags, int64_t n, int64_t append_at,
                  int dim, bool normalise, float* master, __nv_bfloat16* plane, int8_t* plane8, int plane_dim,
                  uint32_t* gmax_bits, int32_t* tag_out, cudaStream_t st) {
  if (n <= 0) return FRG_OK;
  // limit: appended rows land below append_at + n, in-place rows below append_at
  const int64_t limit = rows ? append_at : append_at + n;
  ingest_kernel<<<grid_for_rows(n, 8), 256, 0, st>>>(vecs, rows, tags, n, append_at, limit, dim,
                                                     normalise ? 1 : 0, master, plane, plane8, i8_gallery_step(dim),
                                                     plane_dim, gmax_bits, tag_out);
  note_launch(nullptr);
  FRG_CUDA(cudaGetLastError());
  return FRG_OK;
}

int launch_tombstone(const int64_t* rows, int64_t n, int64_t limit, int32_t* tags, cudaStream_t st) {
  if (n <= 0) return FRG_OK;
  tombstone_kernel<<<int((n + 255) / 256), 256, 0, st>>>(rows, n, limit, tags);
  note_launch(nullptr);
  FRG_CUDA(cudaGetLastError());
  return FRG_OK;
}

int launch_synth(int64_t n, int64_t append_at, int64_t global_row0, uint64_t seed, int32_t tag, int dim,
                 float* master, __nv_bfloat16* plane, int8_t* plane8, int plane_dim, uint32_t* gmax_bits,
                 int32_t* tag_out, cudaStream_t st) {
  if (n <= 0) return FRG_OK;
  synth_kernel<<<grid_for_rows(n, 8), 256, 0, st>>>(n, append_at, global_row0, uint32_t(seed),
                                                    uint32_t(seed >> 32), tag, dim, master, plane, plane8,
                                                    i8_gallery_step(dim), plane_dim, gmax_bits, tag_out);
  note_launch(nullptr);
  FRG_CUDA(cudaGetLastError());
  return FRG_OK;
}

int launch_gather_rows(const int64_t* src_rows, int64_t n, int dim, int plane_row_bytes, const float* master_in,
                       const void* plane_in, const int32_t* tags_in, float* master_out, void* plane_out,
                       int32_t* tags_out, cudaStream_t st) {
  if (n <= 0) return FRG_OK;
  gather_rows_kernel<<<grid_for_rows(n, 8), 256, 0, st>>>(src_rows, n, dim, plane_in ? plane_row_bytes : 0, master_in,
                                                          static_cast<const unsigned char*>(plane_in), tags_in,
                                                          master_out, static_cast<unsigned char*>(plane_out), tags_out);
  note_launch(nullptr);
  FRG_CUDA(cudaGetLastError());
  return FRG_OK;
}

}  // namespace frg
