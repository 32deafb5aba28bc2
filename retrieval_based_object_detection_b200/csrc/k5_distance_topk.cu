// K5  distance_topk -- exact top-k by a sweep of the whole gallery on the CUDA cores in fp64 (B200 issues 64 DFMA
// per clock per SM), for every metric.  It answers what the tcgen05 pass does not cover: Distance.MANHATTAN
// (util/qdrant_manager.py:61-66, chosen at :68-79 and passed to recreate_collection at :82-85; L1 distance is not a
// contraction at all, and the reference only ever creates such collections at script scale), k beyond the K3
// candidate lists, rows wider than K3 takes -- and the finish path's queries the certification left open.  Keys:
//
//   key(q, g) = dot / (|q| |g|)  (COSINE)     = dot  (DOT)
//             = -sum_i (q_i - g_i)^2   (EUCLID)      = -sum_i |q_i - g_i|   (MANHATTAN)
//
// computed in fp64 from the fp32 query and the stored row, so larger key = closer and the ordering
// (key desc, row asc) needs no certification.  Selection without a Q x N matrix:
//   1. sample pass: keys of a strided sample of <= cap rows; the k-th best sample key is a threshold no
//      member of the true top-k can fall below (a caller that already holds such a bound passes it instead);
//   2. sweep: one pass over the gallery records every row whose key >= threshold (expected k * stride
//      rows); a list that overflows `cap` tightens its threshold to the k-th best key it did record --
//      still a lower bound of the true k-th key -- and only those queries are swept again;
//   3. select: sort each list in shared memory, emit (distance, row) ascending by distance.
// Every lane owns one gallery row and scores it against a batch of up to 32 queries staged in shared memory (32
// independent DFMA chains per lane, no cross-lane reduction), so the gallery is read once per batch of 32 queries.
#include "rbod_common.cuh"
#include "rbod_internal.h"

#include <algorithm>

namespace rbod {

namespace {

// fp32 queries of one batch -> fp64 (done once, so the sweep's inner loop has no conversions)
// One warp per query; also |q| (fp64), which the COSINE key divides by.
__global__ void __launch_bounds__(256)
dist_widen_queries_kernel(const float* __restrict__ q, const int* __restrict__ qsel, int nf, int dim,
                          double* __restrict__ q64, double* __restrict__ qnorm) {
  const int lane = threadIdx.x & 31;
  for (int f = blockIdx.x * 8 + (threadIdx.x >> 5); f < nf; f += gridDim.x * 8) {
    const float* src = q + (int64_t)qsel[f] * dim;
    double ss = 0.0;
    for (int c = lane; c < dim; c += 32) {
      const double x = (double)src[c];
      q64[(int64_t)f * dim + c] = x;
      ss = fma(x, x, ss);
    }
    ss = warp_sum_f64(ss);
    if (lane == 0) qnorm[f] = sqrt(ss);
  }
}

__device__ __forceinline__ void cp_async_4(void* smem_dst, const void* gsrc) {
  asm volatile("cp.async.ca.shared.global [%0], [%1], 4;" ::"r"(smem_u32(smem_dst)), "l"(gsrc) : "memory");
}
__device__ __forceinline__ void cp_async_8(void* smem_dst, const void* gsrc) {
  asm volatile("cp.async.ca.shared.global [%0], [%1], 8;" ::"r"(smem_u32(smem_dst)), "l"(gsrc) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
__device__ __forceinline__ void cp_async_wait_1() { asm volatile("cp.async.wait_group 1;" ::: "memory"); }

constexpr int K5_CH = 64;        // columns per staged chunk
constexpr int K5_ROWS = 256;     // gallery rows per CTA step: 8 warps x 32 lanes, one row per lane

// Rows r = row0, row0 + stride, ... < n_rows.  A CTA takes 256 of them at a time and every LANE owns one row, so a
// row's distance to a query is a private fp64 accumulator: no reduction across lanes, NQ independent DFMA chains
// per lane.  The work is staged through shared memory in chunks of 64 columns, double-buffered with cp.async: each
// warp copies its 32 rows' chunk (coalesced, a row at a time, pitch odd so lane-strided reads are conflict-free),
// the CTA copies the chunk of the NQ fp64 queries once for all 8 warps, and the inner loop is one broadcast
// LDS.128 (two query elements) per four fp64 operations.  q64 is [32, dim], zero rows beyond the batch; `wpr` =
// 4-byte words per chunk row (64 for fp32 rows, 32 for 16-bit rows), `pitch` = wpr + 1.
template <int METRIC, int NQ>
__global__ void __launch_bounds__(256, 1)
dist_collect_kernel(const double* __restrict__ q64, const float* __restrict__ master32,
                    const uint16_t* __restrict__ rows16, int kind16, int dim, int64_t ld32, int64_t ld16,
                    int64_t n_rows, int64_t row0, int64_t stride, const uint32_t* __restrict__ row_mask,
                    int64_t mask_words, const int* __restrict__ slot_mask, const double* __restrict__ thr, const uint32_t* __restrict__ thr_row, const int* __restrict__ active,
                    const double* __restrict__ qnorm, int nf, int cap, double* __restrict__ coll_key,
                    uint32_t* __restrict__ coll_idx, int* __restrict__ coll_cnt) {
  extern __shared__ __align__(16) uint8_t k5_smem[];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const bool f32rows = master32 != nullptr;
  const int wpr = f32rows ? K5_CH : K5_CH / 2, pitch = wpr + 1;
  double* qs = reinterpret_cast<double*>(k5_smem);                                   // [2][NQ][K5_CH]
  uint32_t* xs = reinterpret_cast<uint32_t*>(k5_smem + (size_t)2 * NQ * K5_CH * 8);  // [2][8][32][pitch]
  __shared__ double thr_s[32], qn_s[32];
  __shared__ uint32_t thr_row_s[32];   // with thr_s a (key, row) pair bound: rows tying with the key count up to this row
  __shared__ int mask_s[32];            // per-query masks: the mask slot f reads, -1 = none
  if (threadIdx.x < 32) {
    thr_s[threadIdx.x] = (threadIdx.x < nf && active[threadIdx.x]) ? thr[threadIdx.x] : INFINITY;
    thr_row_s[threadIdx.x] = (threadIdx.x < nf && thr_row != nullptr) ? thr_row[threadIdx.x] : 0xffffffffu;
    qn_s[threadIdx.x] = threadIdx.x < nf ? qnorm[threadIdx.x] : 0.0;
    mask_s[threadIdx.x] = (threadIdx.x < nf && slot_mask != nullptr) ? slot_mask[threadIdx.x] : -1;
  }
  __syncthreads();
  constexpr bool kInner = METRIC == RBOD_COSINE || METRIC == RBOD_DOT;   // keys built from q . g
  double gg = 0.0;                                                        // |row|^2 of this lane's row (COSINE)

  const int64_t n_visit = n_rows > row0 ? (n_rows - row0 + stride - 1) / stride : 0;   // rows of this pass
  const int n_chunks = (dim + K5_CH - 1) / K5_CH;
  const int64_t n_groups = (n_visit + K5_ROWS - 1) / K5_ROWS;
  const int64_t my_groups = n_groups > blockIdx.x ? (n_groups - blockIdx.x + gridDim.x - 1) / gridDim.x : 0;
  const int64_t n_steps = my_groups * n_chunks;     // (group, chunk) pairs this CTA walks, in order

  auto row_of = [&](int64_t g, int l) -> int64_t {  // gallery row of lane l of this warp in group g, or -1
    const int64_t v = (blockIdx.x + g * gridDim.x) * K5_ROWS + warp * 32 + l;
    if (v >= n_visit) return -1;
    const int64_t r = row0 + v * stride;
    // one mask for the whole batch: masked rows are not even loaded
    if (row_mask != nullptr && slot_mask == nullptr && !((row_mask[r >> 5] >> (r & 31)) & 1u)) return -1;
    return r;
  };
  auto issue = [&](int64_t step, int b) {
    const int64_t g = step / n_chunks;
    const int c0 = (int)(step - g * n_chunks) * K5_CH;
    const int cw = min(K5_CH, dim - c0);
    // this warp's 32 rows, one row per iteration, lanes across the chunk's words
    uint32_t* xb = xs + ((size_t)b * 8 + warp) * 32 * pitch;
    for (int j = 0; j < 32; ++j) {
      const int64_t r = row_of(g, j);
      if (r < 0) continue;
      if (f32rows) {
        const uint32_t* src = reinterpret_cast<const uint32_t*>(master32 + r * ld32 + c0);
        for (int w = lane; w < cw; w += 32) cp_async_4(xb + j * pitch + w, src + w);
      } else {
        const uint32_t* src = reinterpret_cast<const uint32_t*>(rows16 + r * ld16 + c0);   // padded to 64 elements
        cp_async_4(xb + j * pitch + lane, src + lane);
      }
    }
    // the CTA's query chunk
    double* qb = qs + (size_t)b * NQ * K5_CH;
    for (int i = threadIdx.x; i < NQ * K5_CH; i += 256) {
      const int f = i / K5_CH, c = i - f * K5_CH;
      if (c < cw) cp_async_8(qb + i, q64 + (int64_t)f * dim + c0 + c);
    }
    cp_async_commit();
  };

  double acc[NQ];
  if (n_steps > 0) issue(0, 0);
  for (int64_t step = 0; step < n_steps; ++step) {
    const int b = (int)(step & 1);
    const int64_t g = step / n_chunks;
    const int ci = (int)(step - g * n_chunks);
    if (step + 1 < n_steps) issue(step + 1, b ^ 1); else cp_async_commit();
    cp_async_wait_1();
    __syncthreads();
    if (ci == 0) {
#pragma unroll
      for (int f = 0; f < NQ; ++f) acc[f] = 0.0;
      gg = 0.0;
    }
    const int cw = min(K5_CH, dim - ci * K5_CH);
    const uint32_t* xr = xs + (((size_t)b * 8 + warp) * 32 + lane) * pitch;
    const double* qb = qs + (size_t)b * NQ * K5_CH;
    auto elem = [&](int c) -> double {
      if (f32rows) return (double)__uint_as_float(xr[c]);
      const uint32_t w = xr[c >> 1];
      return (double)h16_to_f32((uint16_t)((c & 1) ? (w >> 16) : (w & 0xffffu)), kind16);
    };
    int c = 0;
    for (; c + 1 < cw; c += 2) {
      const double x0 = elem(c), x1 = elem(c + 1);
      if (METRIC == RBOD_COSINE) gg = fma(x1, x1, fma(x0, x0, gg));
#pragma unroll
      for (int f = 0; f < NQ; ++f) {
        const double2 qq = *reinterpret_cast<const double2*>(qb + f * K5_CH + c);
        if (kInner) {
          acc[f] = fma(qq.y, x1, fma(qq.x, x0, acc[f]));
        } else {
          const double d0 = qq.x - x0, d1 = qq.y - x1;
          if (METRIC == RBOD_EUCLID) acc[f] = fma(d1, d1, fma(d0, d0, acc[f]));
          else acc[f] += fabs(d0) + fabs(d1);
        }
      }
    }
    if (c < cw) {
      const double x0 = elem(c);
      if (METRIC == RBOD_COSINE) gg = fma(x0, x0, gg);
#pragma unroll
      for (int f = 0; f < NQ; ++f) {
        if (kInner) {
          acc[f] = fma(qb[f * K5_CH + c], x0, acc[f]);
        } else {
          const double d0 = qb[f * K5_CH + c] - x0;
          if (METRIC == RBOD_EUCLID) acc[f] = fma(d0, d0, acc[f]);
          else acc[f] += fabs(d0);
        }
      }
    }
    if (ci == n_chunks - 1) {
      const int64_t r = row_of(g, lane);
      if (r >= 0) {
#pragma unroll
        for (int f = 0; f < NQ; ++f) {
          double key;
          if (METRIC == RBOD_COSINE) {
            const double den = qn_s[f] * sqrt(gg);
            key = den > 0.0 ? acc[f] / den : 0.0;        // the formula of cosine_similarity, 33_…py:76-77
          } else if (METRIC == RBOD_DOT) {
            key = acc[f];
          } else {
            key = -acc[f];
          }
          // thr_s is +inf for slots beyond the batch and for finished queries; a list that overflowed was tightened to
          // the k-th best (key, row) pair it had recorded, so a cluster of duplicates wider than the list resolves to
          // its smallest row slots instead of overflowing for ever
          // per-query masks (slot_mask != nullptr): a row slot f's mask excludes is never recorded for it
          if ((key > thr_s[f] || (key == thr_s[f] && (uint32_t)r <= thr_row_s[f])) &&
              (mask_s[f] < 0 || ((row_mask[(int64_t)mask_s[f] * mask_words + (r >> 5)] >> (r & 31)) & 1u))) {
            const int slot = atomicAdd(coll_cnt + f, 1);
            if (slot < cap) {
              coll_key[(size_t)f * cap + slot] = key;
              coll_idx[(size_t)f * cap + slot] = (uint32_t)r;
            }
          }
        }
      }
    }
    __syncthreads();   // everyone is done with buffer b before the copy of step + 2 lands in it
  }
}

// Monotone map double -> uint64 (larger double <=> larger key).
__device__ __forceinline__ unsigned long long f64_to_ordered(double d) {
  const unsigned long long b = (unsigned long long)__double_as_longlong(d);
  return (b >> 63) ? ~b : (b | 0x8000000000000000ull);
}

// One CTA per query of the batch: the recorded (key, row) pairs are sorted in shared memory (bitonic, key
// descending then row ascending), then
//   sample != 0         : thr[f] = k-th best recorded key (-inf if fewer than k were recorded); no output.
//   list fits (<= cap)  : the first k entries are the answer, active[f] = 0.
//   list overflowed     : thr[f] = k-th best key among the `cap` rows that were recorded, active[f] stays 1.
// Shared memory: p2 * 12 bytes, p2 = capacity rounded up to a power of two.
__global__ void __launch_bounds__(256)
dist_select_kernel(const double* __restrict__ coll_key, const uint32_t* __restrict__ coll_idx,
                   int* __restrict__ coll_cnt, const int* __restrict__ qsel, int cap, int p2_max, int k, int sample,
                   int metric, double* __restrict__ thr, uint32_t* __restrict__ thr_row, int* __restrict__ active,
                   int* __restrict__ n_active, float* __restrict__ out_scores, int64_t* __restrict__ out_rows, double* __restrict__ out_keys) {
  extern __shared__ __align__(16) uint8_t k5_sel_smem[];
  unsigned long long* sk = reinterpret_cast<unsigned long long*>(k5_sel_smem);       // [p2_max] ordered keys
  uint32_t* si = reinterpret_cast<uint32_t*>(k5_sel_smem + (size_t)p2_max * 8);      // [p2_max] rows
  const int f = blockIdx.x;
  if (!active[f]) return;
  const int total = coll_cnt[f];
  const int cnt = total < cap ? total : cap;
  const bool overflow = total > cap;
  const int64_t q = qsel[f];
  const bool emit = !sample && !overflow;
  int p2 = 1;
  while (p2 < cnt) p2 <<= 1;
  for (int i = threadIdx.x; i < p2; i += blockDim.x) {
    const bool have = i < cnt;
    sk[i] = have ? f64_to_ordered(coll_key[(size_t)f * cap + i]) : 0ull;   // 0 sorts below every real key
    si[i] = have ? coll_idx[(size_t)f * cap + i] : 0xffffffffu;
  }
  __syncthreads();
  for (int size = 2; size <= p2; size <<= 1) {
    for (int strd = size >> 1; strd > 0; strd >>= 1) {
      for (int i = threadIdx.x; i < (p2 >> 1); i += blockDim.x) {
        const int lo = 2 * i - (i & (strd - 1));
        const int hi = lo + strd;
        const bool desc = (lo & size) == 0;
        const unsigned long long ka = sk[lo], kb = sk[hi];
        const uint32_t ia = si[lo], ib = si[hi];
        const bool a_first = ka > kb || (ka == kb && ia < ib);   // a belongs before b in the final order
        if (desc ? !a_first : a_first) {
          sk[lo] = kb; sk[hi] = ka;
          si[lo] = ib; si[hi] = ia;
        }
      }
      __syncthreads();
    }
  }
  if (emit) {
    for (int j = threadIdx.x; j < k; j += blockDim.x) {
      const bool have = j < cnt;
      // recover the key from the row's recorded value order: re-read by position is not possible after the sort,
      // so invert the ordered map
      const unsigned long long o = have ? sk[j] : 0ull;
      const unsigned long long bits = (o >> 63) ? (o & 0x7fffffffffffffffull) : ~o;
      const double key = have ? __longlong_as_double((long long)bits) : -INFINITY;
      const bool dist = metric == RBOD_EUCLID || metric == RBOD_MANHATTAN;
      out_scores[q * k + j] = !have ? (dist ? INFINITY : -INFINITY)
                                    : (float)(metric == RBOD_EUCLID ? sqrt(-key) : (metric == RBOD_MANHATTAN ? -key : key));
      out_rows[q * k + j] = have ? (int64_t)si[j] : -1;
      if (out_keys) out_keys[q * k + j] = key;
    }
  } else if (threadIdx.x == 0 && cnt >= k) {
    const unsigned long long o = sk[k - 1];
    const unsigned long long bits = (o >> 63) ? (o & 0x7fffffffffffffffull) : ~o;
    thr[f] = __longlong_as_double((long long)bits);
    // a sampled threshold must admit every tie (the sample saw only some rows); an overflowed list's bound is the pair
    if (thr_row != nullptr) thr_row[f] = sample ? 0xffffffffu : si[k - 1];
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    if (emit) active[f] = 0;
    else atomicAdd(n_active, 1);
    coll_cnt[f] = 0;
  }
}

}  // namespace

int launch_dist_widen_queries(const float* q, const int* qsel, int nf, int dim, double* q64, double* qnorm,
                              cudaStream_t st) {
  if (nf <= 0) return RBOD_OK;
  dist_widen_queries_kernel<<<(unsigned)((nf + 7) / 8), 256, 0, st>>>(q, qsel, nf, dim, q64, qnorm);
  RBOD_CUDA(cudaGetLastError());
  return RBOD_OK;
}

int launch_dist_collect(int metric, const double* q64, const float* master32, const uint16_t* rows16, int kind16,
                        int dim, int64_t ld32, int64_t ld16, int64_t n_rows, int64_t row0, int64_t stride,
                        const uint32_t* row_mask, int64_t mask_words, const int* slot_mask, const double* thr,
                        const uint32_t* thr_row, const int* active, const double* qnorm, int nf, int cap,
                        double* coll_key, uint32_t* coll_idx, int* coll_cnt, int num_sms, cudaStream_t st) {
  if (nf <= 0 || n_rows <= 0) return RBOD_OK;
  if (nf > 32) return set_error(RBOD_E_INVAL, "dist_collect: at most 32 queries per pass");
  const int64_t rows_visited = (n_rows - row0 + stride - 1) / stride;
  const int64_t groups = (rows_visited + K5_ROWS - 1) / K5_ROWS;
  const int grid = (int)std::max<int64_t>(1, std::min<int64_t>(groups, (int64_t)num_sms));
  const int pitch = (master32 ? K5_CH : K5_CH / 2) + 1;
#define RBOD_K5_GO(METRIC, NQ)                                                                                 \
  do {                                                                                                         \
    const size_t smem = (size_t)2 * NQ * K5_CH * 8 + (size_t)2 * 8 * 32 * pitch * 4;                           \
    RBOD_CUDA(cudaFuncSetAttribute(dist_collect_kernel<METRIC, NQ>, cudaFuncAttributeMaxDynamicSharedMemorySize, \
                                   (int)smem));                                                                \
    dist_collect_kernel<METRIC, NQ><<<grid, 256, smem, st>>>(q64, master32, rows16, kind16, dim, ld32, ld16,    \
                                                             n_rows, row0, stride, row_mask, mask_words,       \
                                                             slot_mask, thr, thr_row, active,                  \
                                                             qnorm, nf, cap, coll_key, coll_idx, coll_cnt);    \
  } while (0)
  // 8 accumulators per lane for batches of up to 8 queries (single-query searches of the scripts), 32 otherwise
  if (metric == RBOD_EUCLID) {
    if (nf <= 8) RBOD_K5_GO(RBOD_EUCLID, 8); else RBOD_K5_GO(RBOD_EUCLID, 32);
  } else if (metric == RBOD_MANHATTAN) {
    if (nf <= 8) RBOD_K5_GO(RBOD_MANHATTAN, 8); else RBOD_K5_GO(RBOD_MANHATTAN, 32);
  } else if (metric == RBOD_DOT) {
    if (nf <= 8) RBOD_K5_GO(RBOD_DOT, 8); else RBOD_K5_GO(RBOD_DOT, 32);
  } else {
    if (nf <= 8) RBOD_K5_GO(RBOD_COSINE, 8); else RBOD_K5_GO(RBOD_COSINE, 32);
  }
#undef RBOD_K5_GO
  RBOD_CUDA(cudaGetLastError());
  return RBOD_OK;
}

int launch_dist_select(const double* coll_key, const uint32_t* coll_idx, int* coll_cnt, const int* qsel, int nf,
                       int cap, int k, int sample, int metric, double* thr, uint32_t* thr_row, int* active,
                       int* n_active, float* out_scores, int64_t* out_rows, double* out_keys, cudaStream_t st) {
  if (nf <= 0) return RBOD_OK;
  int p2 = 1;
  while (p2 < cap) p2 <<= 1;
  const size_t smem = (size_t)p2 * 12;
  if (smem > 200 * 1024) return set_error(RBOD_E_INVAL, "dist_select: list capacity %d too large", cap);
  RBOD_CUDA(cudaFuncSetAttribute(dist_select_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  dist_select_kernel<<<nf, 256, smem, st>>>(coll_key, coll_idx, coll_cnt, qsel, cap, p2, k, sample, metric, thr, thr_row,
                                            active, n_active, out_scores, out_rows, out_keys);
  RBOD_CUDA(cudaGetLastError());
  return RBOD_OK;
}

}  // namespace rbod
