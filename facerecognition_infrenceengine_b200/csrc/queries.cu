// Query preparation: the reference re-normalises every face embedding before the scan
// (`face.normed_embedding / np.linalg.norm(face.normed_embedding)`, infrenceServer.py:532,
// peopleCount.py:863).  One warp per query; writes the fp32 unit query and, for the tensor-core
// variants, its bf16 or int8 image.
#include <cstring>

#include "frg_internal.cuh"

namespace frg {

__global__ void __launch_bounds__(128)
normalise_queries_kernel(const float* __restrict__ q, int nq, int dim, int normalise,
                         float* __restrict__ qn, __nv_bfloat16* __restrict__ qb,
                         uint32_t* __restrict__ group_keys, int* __restrict__ cand_total,
                         int* __restrict__ n_flagged, float* __restrict__ eps, const uint32_t* __restrict__ bounds) {
  // launched with the programmatic-serialization attribute: the launch overlaps the tail of whatever kernel
  // precedes it in the stream (the previous match of a back-to-back caller); nothing is read or written before
  // that kernel has completed
  pdl_wait();
  pdl_trigger();          // the next kernel of the match may be scheduled now (it waits before reading)
  const int lane = threadIdx.x & 31;
  const int w = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  if (w >= nq) return;
  // per-query scratch of the tensor-core pipeline starts from "nothing seen": 32 group maxima at the
  // ordered key of -1.0f, flagged-query counter at 0 (saves a memset node per match)
  if (group_keys) group_keys[size_t(w) * 32 + lane] = 0x407FFFFFu;
  if (cand_total && lane == 0) cand_total[w] = 0;
  if (n_flagged && w == 0 && lane < 3) n_flagged[lane] = 0;      // count, ticket, probe arrivals
  const float4* src = reinterpret_cast<const float4*>(q + size_t(w) * dim);
  const int nvec = dim >> 2;
  float norm = 1.0f;
  if (normalise) {
    float ss = 0.f;
    for (int v = lane; v < nvec; v += 32) {
      float4 x = __ldg(src + v);
      ss = fmaf(x.x, x.x, ss); ss = fmaf(x.y, x.y, ss); ss = fmaf(x.z, x.z, ss); ss = fmaf(x.w, x.w, ss);
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) ss += __shfl_xor_sync(0xffffffffu, ss, o);
    norm = __fsqrt_rn(ss);
  }
  float rq = 0.f;          // ||q - bf16(q)||^2 (each difference is exact in fp32)
  for (int v = lane; v < nvec; v += 32) {
    float4 x = __ldg(src + v);
    if (normalise) {
      x.x = __fdiv_rn(x.x, norm); x.y = __fdiv_rn(x.y, norm);
      x.z = __fdiv_rn(x.z, norm); x.w = __fdiv_rn(x.w, norm);
    }
    reinterpret_cast<float4*>(qn + size_t(w) * dim)[v] = x;
    if (qb) {
      __nv_bfloat162 lo = __floats2bfloat162_rn(x.x, x.y);
      __nv_bfloat162 hi = __floats2bfloat162_rn(x.z, x.w);
      uint2 p;
      p.x = *reinterpret_cast<uint32_t*>(&lo);
      p.y = *reinterpret_cast<uint32_t*>(&hi);
      reinterpret_cast<uint2*>(qb + size_t(w) * dim)[v] = p;
      const float2 l = __bfloat1622float2(lo), h = __bfloat1622float2(hi);
      const float a = x.x - l.x, b = x.y - l.y, c = x.z - h.x, d = x.w - h.y;
      rq = fmaf(a, a, fmaf(b, b, fmaf(c, c, fmaf(d, d, rq))));
    }
  }
  if (eps) {
    // |q^.g^ - q.g| <= ||q^|| ||g^ - g|| + ||q^ - q|| ||g||  with unit q, g (to fp32 rounding) and ||q^|| <= 1 + 2^-8;
    // + 1 % for the fp32 evaluation of the residual norms, + 1e-4 for the tensor core's fp32 accumulation of 512
    // exact products.  ~3.6e-3 for ordinary data, at most 2^-7 + 2^-16 (every element rounded the same way).
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) rq += __shfl_xor_sync(0xffffffffu, rq, o);
    if (lane == 0) {
      const float rg = bounds ? __uint_as_float(bounds[1]) : 6.2e-5f;      // (2^-7)^2: the a-priori worst case
      eps[w] = 1.01f * (1.00390625f * __fsqrt_rn(rg) + __fsqrt_rn(rq)) + 1e-4f;
    }
  }
}

// Int8 filter prep (unit store with an int8 plane, tc_match.cu).  Per query: the unit fp32 query, its int8 image
// qi = rint(q / c_q) with c_q = max|q| / 127 (no element saturates), the integer product's step
// qstep = c_q * c_g (S = sum qi * gi * qstep, exact up to that one fp32 product: the tensor core accumulates in s32),
// and eps = a rigorous bound of |S - s| for every row of the store:
//   |q^.g^ - q.g| <= ||q^|| ||g^ - g|| + ||q^ - q|| ||g||,   ||q^|| <= 1 + ||q^ - q||,  ||g|| = 1
// with q^ = c_q qi, g^ = c_g gi, ||g^ - g|| <= sqrt(bounds[1]) (the largest residual of any stored row) and ||q^ - q||
// measured here.  + 1 % for the fp32 evaluation of the residual norms; + 4e-5 for the fp32 accumulation of the exact
// scan whose scores are the results (<= dim 2^-24 ||q|| ||g|| = 3.1e-5 at dim 512) and the fp32 conversions of the
// floor.  ~1.9e-2 for ordinary 512-d data.
__global__ void __launch_bounds__(128)
prepare_queries_i8_kernel(const float* __restrict__ q, int nq, int dim, float step_g, float* __restrict__ qn,
                          int8_t* __restrict__ qi8, float* __restrict__ qstep, float* __restrict__ eps,
                          const uint32_t* __restrict__ bounds, unsigned long long* __restrict__ group_keys,
                          int* __restrict__ cand_total, int* __restrict__ n_flagged) {
  pdl_wait();
  pdl_trigger();
  const int lane = threadIdx.x & 31;
  const int w = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  if (w >= nq) return;
  // the pre-pass folds (score, row) keys with a 64-bit atomicMax: 0 = nothing seen
  group_keys[size_t(w) * 32 + lane] = 0ull;
  if (lane == 0) cand_total[w] = 0;
  if (w == 0 && lane < 3) n_flagged[lane] = 0;      // count, ticket, probe arrivals
  const float4* src = reinterpret_cast<const float4*>(q + size_t(w) * dim);
  float4* dst = reinterpret_cast<float4*>(qn + size_t(w) * dim);
  const int nvec = dim >> 2;
  float ss = 0.f;
  for (int v = lane; v < nvec; v += 32) {
    const float4 x = __ldg(src + v);
    ss = fmaf(x.x, x.x, ss); ss = fmaf(x.y, x.y, ss); ss = fmaf(x.z, x.z, ss); ss = fmaf(x.w, x.w, ss);
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) ss += __shfl_xor_sync(0xffffffffu, ss, o);
  const float norm = __fsqrt_rn(ss);
  float amax = 0.f;
  for (int v = lane; v < nvec; v += 32) {
    float4 x = __ldg(src + v);
    x.x = __fdiv_rn(x.x, norm); x.y = __fdiv_rn(x.y, norm);
    x.z = __fdiv_rn(x.z, norm); x.w = __fdiv_rn(x.w, norm);
    dst[v] = x;
    amax = fmaxf(amax, fmaxf(fmaxf(fabsf(x.x), fabsf(x.y)), fmaxf(fabsf(x.z), fabsf(x.w))));
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) amax = fmaxf(amax, __shfl_xor_sync(0xffffffffu, amax, o));
  // a zero / non-finite query (NaN elements: no row can match it) keeps step 1 and an all-zero image; its eps is NaN
  const float c_q = amax > 0.f && amax < INFINITY ? amax / 127.f : 1.f;
  float rq = ss == ss && norm > 0.f ? 0.f : NAN;
  for (int v = lane; v < nvec; v += 32) {
    const float4 x4 = dst[v];                  // this lane's own writes
    const float x[4] = {x4.x, x4.y, x4.z, x4.w};
    uint32_t packed = 0;
#pragma unroll
    for (int e = 0; e < 4; ++e) {
      float t = rintf(__fdiv_rn(x[e], c_q));
      t = t == t ? fminf(fmaxf(t, -127.f), 127.f) : 0.f;
      const float d = fmaf(-t, c_q, x[e]);
      rq = fmaf(d, d, rq);
      packed |= (uint32_t(int(t)) & 0xFFu) << (8 * e);
    }
    reinterpret_cast<uint32_t*>(qi8 + size_t(w) * dim)[v] = packed;
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) rq += __shfl_xor_sync(0xffffffffu, rq, o);
  if (lane == 0) {
    const float rq_n = __fsqrt_rn(rq);
    const float rg_n = __fsqrt_rn(__uint_as_float(bounds[1]));
    qstep[w] = c_q * step_g;
    eps[w] = 1.01f * ((1.0f + rq_n) * rg_n + rq_n) + 4e-5f;
  }
}

int launch_prepare_queries_i8(const float* q, int nq, int dim, float* qn, int8_t* qi8, float* qstep, float* eps,
                              const uint32_t* bounds, unsigned long long* group_keys, int* cand_total, int* n_flagged,
                              cudaStream_t st) {
  if (nq <= 0) return FRG_OK;
  FRG_CUDA(func_attr_once(prepare_queries_i8_kernel, cudaFuncAttributePreferredSharedMemoryCarveout, 100));
  FRG_CUDA(launch_kernel(prepare_queries_i8_kernel, dim3((nq + 3) / 4), dim3(128), 0, st, q, nq, dim,
                         i8_gallery_step(dim), qn, qi8, qstep, eps, bounds, group_keys, cand_total, n_flagged));
  note_launch(nullptr);
  FRG_CUDA(cudaGetLastError());
  return FRG_OK;
}

__device__ __forceinline__ uint32_t bf16_up_bits(float x) {      // smallest bf16 >= x, x >= 0
  __nv_bfloat16 b = __float2bfloat16_rn(x);
  uint32_t u = __bfloat16_as_ushort(b);
  if (__bfloat162float(b) < x) ++u;
  return u;
}

// Euclidean tensor-core prep (BASELINE config 3; ours, not in the reference).  The query is used as
// given; its bf16 image gets kEuclidQPad more columns [1, 1, 1, 0 ...] that pick up the three bias terms of
// the Euclidean scan plane, so that the tensor-core score is S = q.g - 0.5*||g||^2 = (||q||^2 - d^2) / 2:
// largest S <=> smallest distance.  eps[w] bounds |S - exact| for every row of the store:
//   bf16 rounding of both operands  (2u + u^2) ||q|| ||g||,  u = 2^-9   ->  < 3.92e-3 ||q|| Gmax
//   fp32 bias / accumulation          O(dim * 2^-24) (||q|| ||g|| + ||g||^2 / 2)
__global__ void __launch_bounds__(128)
prepare_queries_euclid_kernel(const float* __restrict__ q, int nq, int dim, const uint32_t* __restrict__ gmax_bits,
                              float* __restrict__ qn, __nv_bfloat16* __restrict__ q_aug,
                              __nv_bfloat16* __restrict__ q_aug_lo, float* __restrict__ coef, float* __restrict__ eps,
                              uint32_t* __restrict__ group_keys, uint32_t none_key, int* __restrict__ cand_total,
                              int* __restrict__ n_flagged) {
  pdl_wait();
  pdl_trigger();
  const int lane = threadIdx.x & 31;
  const int w = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  if (w >= nq) return;
  if (group_keys) group_keys[size_t(w) * 32 + lane] = none_key;
  if (cand_total && lane == 0) cand_total[w] = 0;
  if (n_flagged && w == 0 && lane < 3) n_flagged[lane] = 0;
  const float4* src = reinterpret_cast<const float4*>(q + size_t(w) * dim);
  const int nvec = dim >> 2;
  const int aug = dim + kEuclidQPad;
  float ss = 0.f, rq = 0.f;
  for (int v = lane; v < nvec; v += 32) {
    const float4 x = __ldg(src + v);
    ss = fmaf(x.x, x.x, ss); ss = fmaf(x.y, x.y, ss); ss = fmaf(x.z, x.z, ss); ss = fmaf(x.w, x.w, ss);
    reinterpret_cast<float4*>(qn + size_t(w) * dim)[v] = x;
    __nv_bfloat162 lo = __floats2bfloat162_rn(x.x, x.y);
    __nv_bfloat162 hi = __floats2bfloat162_rn(x.z, x.w);
    uint2 p;
    p.x = *reinterpret_cast<uint32_t*>(&lo);
    p.y = *reinterpret_cast<uint32_t*>(&hi);
    reinterpret_cast<uint2*>(q_aug + size_t(w) * aug)[v] = p;
    reinterpret_cast<uint2*>(q_aug_lo + size_t(w) * aug)[v] = p;
    const float2 l = __bfloat1622float2(lo), h = __bfloat1622float2(hi);
    const float a = x.x - l.x, b = x.y - l.y, c = x.z - h.x, d = x.w - h.y;
    rq = fmaf(a, a, fmaf(b, b, fmaf(c, c, fmaf(d, d, rq))));
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    ss += __shfl_xor_sync(0xffffffffu, ss, o);
    rq += __shfl_xor_sync(0xffffffffu, rq, o);
  }
  // |S - s| <= ||q^|| ||g^ - g|| + ||q^ - q|| ||g|| + fp32 accumulation  =  A R_g + B N_g + C SS_g   per ROW, with
  //   A = 1.01 (1 + 2^-8) ||q||,  B = 1.01 ||q - bf16(q)|| + 1e-4 ||q||,  C = 1e-4
  // (R_g, N_g, SS_g: the row's bound columns, store_kernels.cu; the bias columns carry -0.5*||g||^2 exactly).  The
  // coefficients, rounded UP to bf16, sit behind the three ones of the image: +A, +B, +C in the filter's image (the
  // tensor core returns an UPPER bound of the exact score), -A, -B, -C in the pre-pass image (a LOWER bound: its
  // k-th best is a floor of the true k-th best).  No eps arithmetic is left for the epilogue: eps[w] = 0.
  (void)gmax_bits;
  const float nq_ = __fsqrt_ru(ss);
  const uint32_t a = bf16_up_bits(1.01f * 1.00390625f * nq_);
  const uint32_t b = bf16_up_bits(1.01f * __fsqrt_ru(rq) + 1e-4f * nq_);
  const uint32_t c = bf16_up_bits(1e-4f);
  if (lane < kEuclidQPad / 4) {
    // bf16(1.0) = 0x3F80; sign bit 0x8000
    uint2 hi_img = make_uint2(0u, 0u), lo_img = make_uint2(0u, 0u);
    if (lane == 0) {
      hi_img = make_uint2(0x3F803F80u, 0x00003F80u | (a << 16));
      lo_img = make_uint2(0x3F803F80u, 0x00003F80u | ((a | 0x8000u) << 16));
    } else if (lane == 1) {
      hi_img = make_uint2(b | (c << 16), 0u);
      lo_img = make_uint2((b | 0x8000u) | ((c | 0x8000u) << 16), 0u);
    }
    reinterpret_cast<uint2*>(q_aug + size_t(w) * aug + dim)[lane] = hi_img;
    reinterpret_cast<uint2*>(q_aug_lo + size_t(w) * aug + dim)[lane] = lo_img;
  }
  if (lane == 0) {
    eps[w] = 0.f;
    coef[size_t(w) * 4 + 0] = __uint_as_float(a << 16);        // the bf16 values the tensor core multiplies with
    coef[size_t(w) * 4 + 1] = __uint_as_float(b << 16);
    coef[size_t(w) * 4 + 2] = __uint_as_float(c << 16);
    coef[size_t(w) * 4 + 3] = 0.f;
  }
}

int launch_prepare_queries_euclid(const float* q, int nq, int dim, const uint32_t* gmax_bits, float* qn,
                                  __nv_bfloat16* q_aug, __nv_bfloat16* q_aug_lo, float* coef, float* eps,
                                  uint32_t* group_keys, int* cand_total, int* n_flagged, cudaStream_t st) {
  if (nq <= 0) return FRG_OK;
  FRG_CUDA(func_attr_once(prepare_queries_euclid_kernel, cudaFuncAttributePreferredSharedMemoryCarveout, 100));
  // group maxima start from "nothing seen" = the ordered key of -3e38 (Euclidean scores are unbounded below)
  uint32_t none_bits;
  const float none = kEuclidNone;
  memcpy(&none_bits, &none, sizeof(none_bits));
  const uint32_t none_key = ~none_bits;        // float_key() of a negative value: all bits complemented
  FRG_CUDA(launch_kernel(prepare_queries_euclid_kernel, dim3((nq + 3) / 4), dim3(128), 0, st, q, nq, dim, gmax_bits,
                         qn, q_aug, q_aug_lo, coef, eps, group_keys, none_key, cand_total, n_flagged));
  note_launch(nullptr);
  FRG_CUDA(cudaGetLastError());
  return FRG_OK;
}

int launch_normalise_queries(const float* q, int nq, int dim, bool normalise, float* qn,
                             __nv_bfloat16* qn_bf16, uint32_t* group_keys, int* cand_total, int* n_flagged,
                             cudaStream_t st, float* eps, const uint32_t* bounds) {
  if (nq <= 0) return FRG_OK;
  const int warps_per_block = 4;
  // same smem/L1 split as the tensor-core kernels that follow: no carve-out switch between launches
  FRG_CUDA(func_attr_once(normalise_queries_kernel, cudaFuncAttributePreferredSharedMemoryCarveout, 100));
  FRG_CUDA(launch_kernel(normalise_queries_kernel, dim3((nq + warps_per_block - 1) / warps_per_block), dim3(128), 0, st,
                         q, nq, dim, normalise ? 1 : 0, qn, qn_bf16, group_keys, cand_total, n_flagged, eps, bounds));
  note_launch(nullptr);
  FRG_CUDA(cudaGetLastError());
  return FRG_OK;
}

}  // namespace frg
