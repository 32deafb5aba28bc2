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
// The row loop is slot_sweep (rbod_slot_sweep.cuh), shared with K6 and K7: every lane owns one gallery row and scores
// it against a pass of up to 32 queries staged in shared memory (32 independent DFMA chains per lane, no cross-lane
// reduction), so the gallery is read once per 32 queries.  A query is a request of one slot and its end of a row,
// KeyRow below, records the key itself; K6 and K7 fold a request's slots into one score instead.  The widening and
// the selection below serve all three, and so does the host loop (rbod_api.cu: sweep).
#include "rbod_slot_sweep.cuh"

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

// End of a row: a query is a request of one slot, whose score is its key.
struct KeyRow {
  static constexpr bool kSlotIsRequest = true;
  double key = 0.0;
  __device__ __forceinline__ void fold(int, double k) { key = k; }
  __device__ __forceinline__ double score(int) const { return key; }
  __device__ __forceinline__ void reset() {}
};

template <int METRIC, int NS>
__global__ void __launch_bounds__(256, 1)
key_collect_kernel(const double* __restrict__ q64, const float* __restrict__ master32,
                   const uint16_t* __restrict__ rows16, int kind16, int dim, int64_t ld32, int64_t ld16,
                   int64_t n_rows, int64_t row0, int64_t stride, const uint32_t* __restrict__ row_mask,
                   int64_t mask_words, const int* __restrict__ slot_tab, const int* __restrict__ req_mask,
                   const double* __restrict__ thr, const uint32_t* __restrict__ thr_row,
                   const int* __restrict__ active, const double* __restrict__ qnorm, int n_slots, int n_req, int cap,
                   double* __restrict__ coll_key, uint32_t* __restrict__ coll_idx, int* __restrict__ coll_cnt) {
  slot_sweep<METRIC, NS, KeyRow>(q64, master32, rows16, kind16, dim, ld32, ld16, n_rows, row0, stride, row_mask,
                                 mask_words, slot_tab, req_mask, thr, thr_row, active, qnorm, n_slots, n_req, cap,
                                 coll_key, coll_idx, coll_cnt);
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

int launch_key_collect(int metric, const double* q64, const float* master32, const uint16_t* rows16, int kind16,
                       int dim, int64_t ld32, int64_t ld16, int64_t n_rows, int64_t row0, int64_t stride,
                       const uint32_t* row_mask, int64_t mask_words, const int* slot_tab, const int* req_mask,
                       const double* thr, const uint32_t* thr_row, const int* active, const double* qnorm,
                       int n_slots, int n_req, int cap, double* coll_key, uint32_t* coll_idx, int* coll_cnt,
                       int num_sms, cudaStream_t st) {
  static const SlotKernel kernels[4][2] = {
      {key_collect_kernel<RBOD_COSINE, 8>, key_collect_kernel<RBOD_COSINE, 32>},
      {key_collect_kernel<RBOD_DOT, 8>, key_collect_kernel<RBOD_DOT, 32>},
      {key_collect_kernel<RBOD_EUCLID, 8>, key_collect_kernel<RBOD_EUCLID, 32>},
      {key_collect_kernel<RBOD_MANHATTAN, 8>, key_collect_kernel<RBOD_MANHATTAN, 32>}};
  return launch_slot_kernel(kernels, "key_collect", metric, q64, master32, rows16, kind16, dim, ld32, ld16, n_rows,
                            row0, stride, row_mask, mask_words, slot_tab, req_mask, thr, thr_row, active, qnorm,
                            n_slots, n_req, cap, coll_key, coll_idx, coll_cnt, num_sms, st);
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
