// Warp-per-pair exact fp64 scorer shared by the finish kernel (K4 family) and the MMR selection (K8): the exact key of
// (an fp64 "query" row, one stored row) on the stored values, one warp per pair, every lane returns it.
//   COSINE dot / (|q| |g|),  DOT dot,  EUCLID -sum (q - g)^2,  MANHATTAN -sum |q - g|
#pragma once

#include "rbod_common.cuh"
#include "rbod_internal.h"

namespace rbod {

// 8 consecutive elements of one lane: a += the products (EUCLID: squared differences, MANHATTAN: absolute differences),
// b += x^2 (COSINE only).
template <int METRIC>
__device__ __forceinline__ void score_step8(const double* __restrict__ q8, const float (&x)[8], double& a, double& b) {
#pragma unroll
  for (int i = 0; i < 8; ++i) {
    const double xd = (double)x[i];
    if (METRIC == RBOD_EUCLID) {
      const double d = q8[i] - xd;
      a = fma(d, d, a);
    } else if (METRIC == RBOD_MANHATTAN) {
      a += fabs(q8[i] - xd);
    } else {
      a = fma(q8[i], xd, a);
      if (METRIC == RBOD_COSINE) b = fma(xd, xd, b);
    }
  }
}

__device__ __forceinline__ void unpack8(const uint4& h, int kind16, float (&x)[8]) {
  const uint32_t w[4] = {h.x, h.y, h.z, h.w};
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    x[2 * i] = h16_to_f32(static_cast<uint16_t>(w[i] & 0xffffu), kind16);
    x[2 * i + 1] = h16_to_f32(static_cast<uint16_t>(w[i] >> 16), kind16);
  }
}

template <int METRIC>
__device__ __forceinline__ double finish_score(double a, double b, double qq) {
  a = warp_sum_f64(a);
  if (METRIC == RBOD_EUCLID || METRIC == RBOD_MANHATTAN) return -a;
  if (METRIC == RBOD_DOT) return a;
  b = warp_sum_f64(b);
  const double den = sqrt(qq) * sqrt(b);
  return den > 0.0 ? a / den : 0.0;
}

// Exact score of (query, stored row) with the query already widened to fp64 (qq = |q|^2, read by COSINE only).
// Vector path (dim % 8 == 0, row 16-byte aligned): 8 elements per lane and step, lane l takes columns 8 l + 256 i.
template <int METRIC>
__device__ __forceinline__ double exact_score_q64(const double* __restrict__ q64, double qq,
                                                  const float* __restrict__ g32, const uint16_t* __restrict__ g16,
                                                  int kind16, int dim, int lane) {
  double a = 0.0, b = 0.0;
  const bool vec = (dim & 7) == 0 &&
                   (g32 ? (reinterpret_cast<uintptr_t>(g32) & 15) == 0 : (reinterpret_cast<uintptr_t>(g16) & 15) == 0);
  if (vec) {
    for (int c0 = lane * 8; c0 < dim; c0 += 256) {
      float x[8];
      if (g32) {
        const float4 g0 = __ldg(reinterpret_cast<const float4*>(g32 + c0));
        const float4 g1 = __ldg(reinterpret_cast<const float4*>(g32 + c0 + 4));
        x[0] = g0.x; x[1] = g0.y; x[2] = g0.z; x[3] = g0.w;
        x[4] = g1.x; x[5] = g1.y; x[6] = g1.z; x[7] = g1.w;
      } else {
        unpack8(__ldg(reinterpret_cast<const uint4*>(g16 + c0)), kind16, x);
      }
      score_step8<METRIC>(q64 + c0, x, a, b);
    }
  } else {
    for (int c = lane; c < dim; c += 32) {
      const double xd = g32 ? (double)g32[c] : (double)h16_to_f32(g16[c], kind16);
      if (METRIC == RBOD_EUCLID) {
        const double d = q64[c] - xd;
        a = fma(d, d, a);
      } else if (METRIC == RBOD_MANHATTAN) {
        a += fabs(q64[c] - xd);
      } else {
        a = fma(q64[c], xd, a);
        if (METRIC == RBOD_COSINE) b = fma(xd, xd, b);
      }
    }
  }
  return finish_score<METRIC>(a, b, qq);
}

}  // namespace rbod
