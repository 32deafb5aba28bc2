// K6  recommend -- exact recommendation top-k ("like these examples, unlike those") by the best_score rule, swept over
// the whole gallery on the CUDA cores in fp64.  A pass holds up to 32 example vectors ("slots") of up to 32 requests;
// request r owns a contiguous run of slots, each a positive or a negative example.  For a row g:
//
//   key(e, g) = K5's key (COSINE dot/(|e||g|), DOT dot, EUCLID -sum (e-g)^2, MANHATTAN -sum |e-g|), fp64
//   bp = max over r's positives, bn = max over r's negatives (-inf when there are none)
//   sim(x) = x, or -sqrt(-x) for EUCLID;  s(y) = 0.5 (y / (1 + |y|) + 1)
//   K(r, g) = s(sim(bp)) if bp > bn, else -s(sim(bn))
//
// K is larger-is-better for every metric, so the selection is K5's (key desc, row asc) with K as the key: the sample
// pass, the threshold sweep, the tightening of an overflowing list and the final sort are K5's, through its launchers
// (launch_dist_widen_queries widens the examples, launch_dist_select sorts the per-request lists).  Only the collecting
// kernel differs: K5 records one key per slot, K6 folds a request's slots into one K before it records.
#include "rbod_common.cuh"
#include "rbod_internal.h"

#include <algorithm>

namespace rbod {

namespace {

__device__ __forceinline__ void cp_async_4(void* smem_dst, const void* gsrc) {
  asm volatile("cp.async.ca.shared.global [%0], [%1], 4;" ::"r"(smem_u32(smem_dst)), "l"(gsrc) : "memory");
}
__device__ __forceinline__ void cp_async_8(void* smem_dst, const void* gsrc) {
  asm volatile("cp.async.ca.shared.global [%0], [%1], 8;" ::"r"(smem_u32(smem_dst)), "l"(gsrc) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
__device__ __forceinline__ void cp_async_wait_1() { asm volatile("cp.async.wait_group 1;" ::: "memory"); }

constexpr int K6_CH = 64;        // columns per staged chunk
constexpr int K6_ROWS = 256;     // gallery rows per CTA step: 8 warps x 32 lanes, one row per lane

template <int METRIC>
__device__ __forceinline__ double reco_sim(double key) {
  return METRIC == RBOD_EUCLID ? -sqrt(-key) : key;
}
__device__ __forceinline__ double reco_sigmoid(double y) { return 0.5 * (y / (1.0 + fabs(y)) + 1.0); }

// The row loop is dist_collect_kernel's (k5_distance_topk.cu): every lane owns one gallery row, NS private fp64
// accumulators (one per example slot, no cross-lane reduction), 64-column chunks double-buffered with cp.async, the
// fp64 examples of the pass staged once per CTA.  At the end of a row the slots are scanned in (unrolled) order with a
// running bp / bn; a request's last slot forms its K and records (K, row) in the request's list when it beats the
// request's (threshold, row) bound and the request's mask allows the row.
// slot_tab[s] = request index | RECO_LAST (s is its request's last slot) | RECO_NEG (negative example); req_mask[r] =
// the mask request r reads (-1 = none); thr / thr_row / active are per request, as K5's are per query.
constexpr int RECO_REQ = 31, RECO_LAST = 32, RECO_NEG = 64;

template <int METRIC, int NS>
__global__ void __launch_bounds__(256, 1)
reco_collect_kernel(const double* __restrict__ q64, const float* __restrict__ master32,
                    const uint16_t* __restrict__ rows16, int kind16, int dim, int64_t ld32, int64_t ld16,
                    int64_t n_rows, int64_t row0, int64_t stride, const uint32_t* __restrict__ row_mask,
                    int64_t mask_words, const int* __restrict__ slot_tab, const int* __restrict__ req_mask,
                    const double* __restrict__ thr, const uint32_t* __restrict__ thr_row,
                    const int* __restrict__ active, const double* __restrict__ qnorm, int n_slots, int n_req, int cap,
                    double* __restrict__ coll_key, uint32_t* __restrict__ coll_idx, int* __restrict__ coll_cnt) {
  extern __shared__ __align__(16) uint8_t k6_smem[];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const bool f32rows = master32 != nullptr;
  const int wpr = f32rows ? K6_CH : K6_CH / 2, pitch = wpr + 1;
  double* qs = reinterpret_cast<double*>(k6_smem);                                   // [2][NS][K6_CH]
  uint32_t* xs = reinterpret_cast<uint32_t*>(k6_smem + (size_t)2 * NS * K6_CH * 8);  // [2][8][32][pitch]
  __shared__ double thr_s[32], qn_s[32];
  __shared__ uint32_t thr_row_s[32];
  __shared__ int slot_s[32], rmask_s[32];
  if (threadIdx.x < 32) {
    const int t = threadIdx.x;
    thr_s[t] = (t < n_req && active[t]) ? thr[t] : INFINITY;   // +inf: beyond the pass, or the request is finished
    thr_row_s[t] = t < n_req ? thr_row[t] : 0xffffffffu;
    rmask_s[t] = t < n_req ? req_mask[t] : -1;
    qn_s[t] = t < n_slots ? qnorm[t] : 0.0;
    slot_s[t] = t < n_slots ? slot_tab[t] : 0;                  // slots beyond the pass end no request
  }
  __syncthreads();
  constexpr bool kInner = METRIC == RBOD_COSINE || METRIC == RBOD_DOT;
  double gg = 0.0;

  const int64_t n_visit = n_rows > row0 ? (n_rows - row0 + stride - 1) / stride : 0;
  const int n_chunks = (dim + K6_CH - 1) / K6_CH;
  const int64_t n_groups = (n_visit + K6_ROWS - 1) / K6_ROWS;
  const int64_t my_groups = n_groups > blockIdx.x ? (n_groups - blockIdx.x + gridDim.x - 1) / gridDim.x : 0;
  const int64_t n_steps = my_groups * n_chunks;

  auto row_of = [&](int64_t g, int l) -> int64_t {
    const int64_t v = (blockIdx.x + g * gridDim.x) * K6_ROWS + warp * 32 + l;
    return v < n_visit ? row0 + v * stride : -1;
  };
  auto issue = [&](int64_t step, int b) {
    const int64_t g = step / n_chunks;
    const int c0 = (int)(step - g * n_chunks) * K6_CH;
    const int cw = min(K6_CH, dim - c0);
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
    double* qb = qs + (size_t)b * NS * K6_CH;
    for (int i = threadIdx.x; i < NS * K6_CH; i += 256) {
      const int f = i / K6_CH, c = i - f * K6_CH;
      if (c < cw) cp_async_8(qb + i, q64 + (int64_t)f * dim + c0 + c);
    }
    cp_async_commit();
  };

  double acc[NS];
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
      for (int f = 0; f < NS; ++f) acc[f] = 0.0;
      gg = 0.0;
    }
    const int cw = min(K6_CH, dim - ci * K6_CH);
    const uint32_t* xr = xs + (((size_t)b * 8 + warp) * 32 + lane) * pitch;
    const double* qb = qs + (size_t)b * NS * K6_CH;
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
      for (int f = 0; f < NS; ++f) {
        const double2 qq = *reinterpret_cast<const double2*>(qb + f * K6_CH + c);
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
      for (int f = 0; f < NS; ++f) {
        if (kInner) {
          acc[f] = fma(qb[f * K6_CH + c], x0, acc[f]);
        } else {
          const double d0 = qb[f * K6_CH + c] - x0;
          if (METRIC == RBOD_EUCLID) acc[f] = fma(d0, d0, acc[f]);
          else acc[f] += fabs(d0);
        }
      }
    }
    if (ci == n_chunks - 1) {
      const int64_t r = row_of(g, lane);
      if (r >= 0) {
        const double gn = sqrt(gg);
        double bp = -INFINITY, bn = -INFINITY;
#pragma unroll
        for (int f = 0; f < NS; ++f) {
          double key;
          if (METRIC == RBOD_COSINE) {
            const double den = qn_s[f] * gn;
            key = den > 0.0 ? acc[f] / den : 0.0;
          } else if (METRIC == RBOD_DOT) {
            key = acc[f];
          } else {
            key = -acc[f];
          }
          const int tab = slot_s[f];
          if (tab & RECO_NEG) bn = fmax(bn, key); else bp = fmax(bp, key);
          if (tab & RECO_LAST) {
            const int q = tab & RECO_REQ;
            const double K = bp > bn ? reco_sigmoid(reco_sim<METRIC>(bp)) : -reco_sigmoid(reco_sim<METRIC>(bn));
            if ((K > thr_s[q] || (K == thr_s[q] && (uint32_t)r <= thr_row_s[q])) &&
                (rmask_s[q] < 0 || ((row_mask[(int64_t)rmask_s[q] * mask_words + (r >> 5)] >> (r & 31)) & 1u))) {
              const int slot = atomicAdd(coll_cnt + q, 1);
              if (slot < cap) {
                coll_key[(size_t)q * cap + slot] = K;
                coll_idx[(size_t)q * cap + slot] = (uint32_t)r;
              }
            }
            bp = -INFINITY;
            bn = -INFINITY;
          }
        }
      }
    }
    __syncthreads();   // everyone is done with buffer b before the copy of step + 2 lands in it
  }
}

}  // namespace

int launch_reco_collect(int metric, const double* q64, const float* master32, const uint16_t* rows16, int kind16,
                        int dim, int64_t ld32, int64_t ld16, int64_t n_rows, int64_t row0, int64_t stride,
                        const uint32_t* row_mask, int64_t mask_words, const int* slot_tab, const int* req_mask,
                        const double* thr, const uint32_t* thr_row, const int* active, const double* qnorm,
                        int n_slots, int n_req, int cap, double* coll_key, uint32_t* coll_idx, int* coll_cnt,
                        int num_sms, cudaStream_t st) {
  if (n_slots <= 0 || n_req <= 0 || n_rows <= 0) return RBOD_OK;
  if (n_slots > 32 || n_req > 32) return set_error(RBOD_E_INVAL, "reco_collect: at most 32 examples per pass");
  const int64_t rows_visited = (n_rows - row0 + stride - 1) / stride;
  const int64_t groups = (rows_visited + K6_ROWS - 1) / K6_ROWS;
  const int grid = (int)std::max<int64_t>(1, std::min<int64_t>(groups, (int64_t)num_sms));
  const int pitch = (master32 ? K6_CH : K6_CH / 2) + 1;
#define RBOD_K6_GO(METRIC, NS)                                                                                 \
  do {                                                                                                         \
    const size_t smem = (size_t)2 * NS * K6_CH * 8 + (size_t)2 * 8 * 32 * pitch * 4;                           \
    RBOD_CUDA(cudaFuncSetAttribute(reco_collect_kernel<METRIC, NS>, cudaFuncAttributeMaxDynamicSharedMemorySize, \
                                   (int)smem));                                                                \
    reco_collect_kernel<METRIC, NS><<<grid, 256, smem, st>>>(q64, master32, rows16, kind16, dim, ld32, ld16,    \
                                                             n_rows, row0, stride, row_mask, mask_words,       \
                                                             slot_tab, req_mask, thr, thr_row, active, qnorm,  \
                                                             n_slots, n_req, cap, coll_key, coll_idx,          \
                                                             coll_cnt);                                        \
  } while (0)
  // 8 accumulators per lane for passes of up to 8 example slots (a request or two), 32 otherwise
  if (metric == RBOD_EUCLID) {
    if (n_slots <= 8) RBOD_K6_GO(RBOD_EUCLID, 8); else RBOD_K6_GO(RBOD_EUCLID, 32);
  } else if (metric == RBOD_MANHATTAN) {
    if (n_slots <= 8) RBOD_K6_GO(RBOD_MANHATTAN, 8); else RBOD_K6_GO(RBOD_MANHATTAN, 32);
  } else if (metric == RBOD_DOT) {
    if (n_slots <= 8) RBOD_K6_GO(RBOD_DOT, 8); else RBOD_K6_GO(RBOD_DOT, 32);
  } else {
    if (n_slots <= 8) RBOD_K6_GO(RBOD_COSINE, 8); else RBOD_K6_GO(RBOD_COSINE, 32);
  }
#undef RBOD_K6_GO
  RBOD_CUDA(cudaGetLastError());
  return RBOD_OK;
}

}  // namespace rbod
