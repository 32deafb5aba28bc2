// K8 mmr_select: maximal marginal relevance over a query's exact candidate list (rbod_search_mmr, include/rbod.h).
//
// Input per query: the candidates c_0 .. c_{L-1} of an rbod_search with k = L (row slot, fp32 score, fp64 key), ordered
// by (key desc, row slot asc), -1 padded.  With sim(y) = y (-sqrt(-y) for EUCLID), rel(c) = sim(key(q, c)) and
// lambda = 1 - diversity, the first pick is c_0 and every later pick is the unpicked candidate with the largest
//   mmr(c) = lambda * rel(c) - diversity * max over picked s of sim(key(s, c))
// (fp64, in exactly that order: no contraction into an fma), exact ties to the smaller candidate rank.  key(s, c) is the
// exact fp64 search key with the picked STORED row s as the query side, from the stored values.
//
// One CTA per query (a grid-stride loop when the picks are widened into global scratch).  Shared memory holds the
// candidates' slots, rel, a running maxsim and a picked flag.  Each step widens the last pick to fp64 once (shared
// memory up to MMR_SMEM_DIM columns, the CTA's row of global scratch beyond), every warp scores the unpicked candidates
// w, w + 8, ... against it with the finish kernel's warp-per-pair scorer (rbod_exact_score.cuh) and updates maxsim, and a
// block arg-max over (mmr desc, rank asc) makes the next pick.  So a query costs (limit - 1) * L pair keys, not L^2.
#include "rbod_exact_score.cuh"

#include <algorithm>

namespace rbod {

namespace {

constexpr int MMR_THREADS = 256;
constexpr int MMR_WARPS = MMR_THREADS / 32;

template <int METRIC>
__device__ __forceinline__ double mmr_sim(double key) {
  return METRIC == RBOD_EUCLID ? -sqrt(-key) : key;
}

// |q|^2 of a widened row in the lane order exact_score_q64 sums a stored row's b in, so key(s, c) == key(c, s) bit for
// bit for COSINE (the products are the same, and so are both norms).
__device__ __forceinline__ double row_sq_q64(const double* q64, int dim, int lane) {
  double b = 0.0;
  if ((dim & 7) == 0) {
    for (int c0 = lane * 8; c0 < dim; c0 += 256)
#pragma unroll
      for (int i = 0; i < 8; ++i) b = fma(q64[c0 + i], q64[c0 + i], b);
  } else {
    for (int c = lane; c < dim; c += 32) b = fma(q64[c], q64[c], b);
  }
  return warp_sum_f64(b);
}

template <int METRIC>
__global__ void __launch_bounds__(MMR_THREADS) mmr_select_kernel(const MmrArgs A) {
  extern __shared__ __align__(16) unsigned char mmr_smem[];
  const int L = A.L, dim = A.dim;
  const bool wide = dim > MMR_SMEM_DIM;
  double* s_rel = reinterpret_cast<double*>(mmr_smem);
  double* s_maxsim = s_rel + L;
  double* q64 = wide ? A.q64_scratch + (size_t)blockIdx.x * dim : s_maxsim + L;
  uint32_t* s_row = reinterpret_cast<uint32_t*>(s_maxsim + L + (wide ? 0 : dim));
  unsigned char* s_picked = reinterpret_cast<unsigned char*>(s_row + L);
  __shared__ double s_bval[MMR_WARPS];
  __shared__ int s_bidx[MMR_WARPS];
  __shared__ int s_n, s_pick;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const bool dist = METRIC == RBOD_EUCLID || METRIC == RBOD_MANHATTAN;
  const float no_score = dist ? INFINITY : -INFINITY;

  for (int64_t q = blockIdx.x; q < A.Q; q += gridDim.x) {
    const double div = A.diversity[q];
    const double lam = __dsub_rn(1.0, div);
    const float thr = A.score_threshold ? A.score_threshold[q] : NAN;
    const int64_t* crow = A.cand_rows + q * L;
    const float* csc = A.cand_scores + q * L;
    const double* ckey = A.cand_keys + q * L;
    if (tid == 0) s_n = L;
    __syncthreads();
    // candidates that take part: a row, with a score passing the threshold.  The list is ordered by key and the fp32
    // score is monotone in the key, so they are a prefix of it; its length is the first rank that fails.
    for (int j = tid; j < L; j += MMR_THREADS) {
      const int64_t r = crow[j];
      const float sc = csc[j];
      const bool ok = r >= 0 && (thr != thr || (dist ? sc <= thr : sc >= thr));
      if (!ok) atomicMin(&s_n, j);
      s_row[j] = static_cast<uint32_t>(r);
      s_rel[j] = mmr_sim<METRIC>(ckey[j]);
      s_maxsim[j] = -INFINITY;
      s_picked[j] = 0;
    }
    __syncthreads();
    const int n = s_n;
    const int picks = min(A.limit, n);
    float* o_s = A.out_scores + q * A.limit;
    int64_t* o_r = A.out_rows + q * A.limit;
    double* o_k = A.out_keys + q * A.limit;
    for (int j = picks + tid; j < A.limit; j += MMR_THREADS) {
      o_s[j] = no_score;
      o_r[j] = -1;
      o_k[j] = -INFINITY;
    }
    int pick = 0;   // c_0
    for (int t = 0; t < picks; ++t) {
      if (tid == 0) {
        s_picked[pick] = 1;
        o_s[t] = csc[pick];
        o_r[t] = crow[pick];
        o_k[t] = ckey[pick];
      }
      if (t + 1 == picks) break;
      // widen the pick once
      const int64_t srow = s_row[pick];
      if (A.master32) {
        const float* src = A.master32 + srow * A.ld32;
        for (int c = tid; c < dim; c += MMR_THREADS) q64[c] = (double)src[c];
      } else {
        const uint16_t* src = A.rows16 + srow * A.ld16;
        for (int c = tid; c < dim; c += MMR_THREADS) q64[c] = (double)h16_to_f32(src[c], A.kind16);
      }
      __syncthreads();
      const double qq = METRIC == RBOD_COSINE ? row_sq_q64(q64, dim, lane) : 0.0;
      // a warp per unpicked candidate: sim(key(pick, c)) into maxsim
      for (int j = warp; j < n; j += MMR_WARPS) {
        if (s_picked[j]) continue;
        const int64_t r = s_row[j];
        const double key = exact_score_q64<METRIC>(q64, qq, A.master32 ? A.master32 + r * A.ld32 : nullptr,
                                                   A.master32 ? nullptr : A.rows16 + r * A.ld16, A.kind16, dim, lane);
        const double s = mmr_sim<METRIC>(key);
        if (lane == 0 && s > s_maxsim[j]) s_maxsim[j] = s;
      }
      __syncthreads();
      // block arg-max over (mmr desc, rank asc)
      double bv = -INFINITY;
      int bi = 0x7fffffff;
      for (int j = tid; j < n; j += MMR_THREADS) {
        if (s_picked[j]) continue;
        const double m = __dsub_rn(__dmul_rn(lam, s_rel[j]), __dmul_rn(div, s_maxsim[j]));
        if (bi == 0x7fffffff || m > bv) {   // j ascends: an equal value keeps the smaller rank
          bv = m;
          bi = j;
        }
      }
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) {
        const double ov = __shfl_xor_sync(FULL_MASK, bv, o);
        const int oi = __shfl_xor_sync(FULL_MASK, bi, o);
        if (oi != 0x7fffffff && (bi == 0x7fffffff || ov > bv || (ov == bv && oi < bi))) {
          bv = ov;
          bi = oi;
        }
      }
      if (lane == 0) {
        s_bval[warp] = bv;
        s_bidx[warp] = bi;
      }
      __syncthreads();
      if (tid == 0) {
        double v = s_bval[0];
        int i = s_bidx[0];
        for (int w = 1; w < MMR_WARPS; ++w) {
          const double ov = s_bval[w];
          const int oi = s_bidx[w];
          if (oi != 0x7fffffff && (i == 0x7fffffff || ov > v || (ov == v && oi < i))) {
            v = ov;
            i = oi;
          }
        }
        s_pick = i;
      }
      __syncthreads();
      pick = s_pick;
    }
    __syncthreads();   // the next query rewrites the shared arrays
  }
}

}  // namespace

int launch_mmr_select(int metric, const MmrArgs& A, int num_sms, cudaStream_t st) {
  if (A.Q <= 0) return RBOD_OK;
  if (A.L < 1 || A.L > MMR_MAX_CANDIDATES || A.limit < 1 || A.limit > A.L)
    return set_error(RBOD_E_INVAL, "mmr_select: limit %d / candidates %d", A.limit, A.L);
  const bool wide = A.dim > MMR_SMEM_DIM;
  if (wide && A.q64_scratch == nullptr) return set_error(RBOD_E_INVAL, "mmr_select: no scratch for %d columns", A.dim);
  const size_t smem = (size_t)A.L * (8 + 8 + 4 + 1) + (wide ? 0 : (size_t)A.dim * 8);
  const int64_t grid = mmr_grid(A.Q, A.dim, num_sms);
  auto go = [&](auto kern) -> int {
    RBOD_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    kern<<<(unsigned)grid, MMR_THREADS, smem, st>>>(A);
    RBOD_CUDA(cudaGetLastError());
    return RBOD_OK;
  };
  switch (metric) {
    case RBOD_COSINE: return go(mmr_select_kernel<RBOD_COSINE>);
    case RBOD_DOT: return go(mmr_select_kernel<RBOD_DOT>);
    case RBOD_EUCLID: return go(mmr_select_kernel<RBOD_EUCLID>);
    case RBOD_MANHATTAN: return go(mmr_select_kernel<RBOD_MANHATTAN>);
  }
  return set_error(RBOD_E_INVAL, "mmr_select: metric %d", metric);
}

}  // namespace rbod
