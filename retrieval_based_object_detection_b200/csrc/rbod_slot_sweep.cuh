// The row loop of the exact fp64 sweep, shared by K5 (search), K6 (recommend) and K7 (discover), which differ only in
// the end of a row, a policy: a pass of up to 32 vectors ("slots": queries or examples) of up to 32 whole requests.
// Every lane owns one gallery row and NS private fp64 accumulators (one per slot, no cross-lane reduction); 64-column
// chunks of the rows and of the fp64 slots are double-buffered in shared memory with cp.async.  At the end of a row
// the lane scans the slots in (unrolled) order: the policy folds each slot's key into its running values, and at a
// request's last slot forms the request's score, which is recorded as (score, row) in the request's list when it beats
// the request's (threshold, row) bound and the request's mask allows the row.  A K5 query is a request of one slot.
//
// slot_tab[s] = request of the pass | SLOT_LAST (s is its request's last slot) | the policy's flags (rbod_internal.h);
// req_mask[r] = the mask request r reads (-1 = none), or nullptr: every request reads mask 0 of row_mask (if any), and
// the rows it excludes are not even loaded; thr / thr_row / active are per request.
//
// A policy End is default-constructed at the start of each row with its running values reset, and provides
//   static constexpr bool kSlotIsRequest   true: slot f is request f of the pass (and its last slot), no table is read
//   void fold(int tab, double key)    the key of the slot whose table entry is tab
//   double score(int tab)             at the request's last slot (tab is that slot's entry)
//   void reset()                      after the score is recorded, before the next request's first slot
#pragma once

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

constexpr int SLOT_CH = 64;        // columns per staged chunk
constexpr int SLOT_ROWS = 256;     // gallery rows per CTA step: 8 warps x 32 lanes, one row per lane

// sim(x) of the example-based queries: x, or -sqrt(-x) for EUCLID (minus the L2 distance);  s(y) = 0.5 (y/(1+|y|) + 1)
template <int METRIC>
__device__ __forceinline__ double reco_sim(double key) {
  return METRIC == RBOD_EUCLID ? -sqrt(-key) : key;
}
__device__ __forceinline__ double reco_sigmoid(double y) { return 0.5 * (y / (1.0 + fabs(y)) + 1.0); }

// The body of a collecting kernel launched with 256 threads and
// 2 * NS * SLOT_CH * 8 + 2 * 8 * 32 * (row words per chunk + 1) * 4 bytes of dynamic shared memory.
template <int METRIC, int NS, class End>
__device__ __forceinline__ void slot_sweep(const double* __restrict__ q64, const float* __restrict__ master32,
                                           const uint16_t* __restrict__ rows16, int kind16, int dim, int64_t ld32,
                                           int64_t ld16, int64_t n_rows, int64_t row0, int64_t stride,
                                           const uint32_t* __restrict__ row_mask, int64_t mask_words,
                                           const int* __restrict__ slot_tab, const int* __restrict__ req_mask,
                                           const double* __restrict__ thr, const uint32_t* __restrict__ thr_row,
                                           const int* __restrict__ active, const double* __restrict__ qnorm,
                                           int n_slots, int n_req, int cap, double* __restrict__ coll_key,
                                           uint32_t* __restrict__ coll_idx, int* __restrict__ coll_cnt) {
  extern __shared__ __align__(16) uint8_t slot_smem[];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const bool f32rows = master32 != nullptr;
  const int wpr = f32rows ? SLOT_CH : SLOT_CH / 2, pitch = wpr + 1;
  double* qs = reinterpret_cast<double*>(slot_smem);                                     // [2][NS][SLOT_CH]
  uint32_t* xs = reinterpret_cast<uint32_t*>(slot_smem + (size_t)2 * NS * SLOT_CH * 8);  // [2][8][32][pitch]
  __shared__ double thr_s[32], qn_s[32];
  __shared__ uint32_t thr_row_s[32];
  __shared__ int slot_s[32], rmask_s[32];
  if (threadIdx.x < 32) {
    const int t = threadIdx.x;
    thr_s[t] = (t < n_req && active[t]) ? thr[t] : INFINITY;   // +inf: beyond the pass, or the request is finished
    thr_row_s[t] = t < n_req ? thr_row[t] : 0xffffffffu;
    rmask_s[t] = (t < n_req && req_mask != nullptr) ? req_mask[t] : -1;
    qn_s[t] = t < n_slots ? qnorm[t] : 0.0;
    slot_s[t] = t < n_slots ? slot_tab[t] : 0;                  // slots beyond the pass end no request
  }
  __syncthreads();
  constexpr bool kInner = METRIC == RBOD_COSINE || METRIC == RBOD_DOT;
  double gg = 0.0;

  const int64_t n_visit = n_rows > row0 ? (n_rows - row0 + stride - 1) / stride : 0;
  const int n_chunks = (dim + SLOT_CH - 1) / SLOT_CH;
  const int64_t n_groups = (n_visit + SLOT_ROWS - 1) / SLOT_ROWS;
  const int64_t my_groups = n_groups > blockIdx.x ? (n_groups - blockIdx.x + gridDim.x - 1) / gridDim.x : 0;
  const int64_t n_steps = my_groups * n_chunks;

  auto visit = [&](int64_t g, int l) -> int64_t { return (blockIdx.x + g * gridDim.x) * SLOT_ROWS + warp * 32 + l; };
  // the gallery row lane l of this warp reads in group g, or -1: beyond the pass, or excluded by the one mask of the
  // whole pass (req_mask == nullptr) -- such rows are not even loaded
  auto row_of = [&](int64_t g, int l) -> int64_t {
    const int64_t v = visit(g, l);
    if (v >= n_visit) return -1;
    const int64_t r = row0 + v * stride;
    if (row_mask != nullptr && req_mask == nullptr && !((row_mask[r >> 5] >> (r & 31)) & 1u)) return -1;
    return r;
  };
  auto issue = [&](int64_t step, int b) {
    const int64_t g = step / n_chunks;
    const int c0 = (int)(step - g * n_chunks) * SLOT_CH;
    const int cw = min(SLOT_CH, dim - c0);
    uint32_t* xb = xs + ((size_t)b * 8 + warp) * 32 * pitch;
    const unsigned live = __ballot_sync(0xffffffffu, row_of(g, lane) >= 0);   // one test per lane, not one per row
    for (int j = 0; j < 32; ++j) {
      if (!((live >> j) & 1u)) continue;
      const int64_t r = row0 + visit(g, j) * stride;
      if (f32rows) {
        const uint32_t* src = reinterpret_cast<const uint32_t*>(master32 + r * ld32 + c0);
        for (int w = lane; w < cw; w += 32) cp_async_4(xb + j * pitch + w, src + w);
      } else {
        const uint32_t* src = reinterpret_cast<const uint32_t*>(rows16 + r * ld16 + c0);   // padded to 64 elements
        cp_async_4(xb + j * pitch + lane, src + lane);
      }
    }
    double* qb = qs + (size_t)b * NS * SLOT_CH;
    for (int i = threadIdx.x; i < NS * SLOT_CH; i += 256) {
      const int f = i / SLOT_CH, c = i - f * SLOT_CH;
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
    const int cw = min(SLOT_CH, dim - ci * SLOT_CH);
    const uint32_t* xr = xs + (((size_t)b * 8 + warp) * 32 + lane) * pitch;
    const double* qb = qs + (size_t)b * NS * SLOT_CH;
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
        const double2 qq = *reinterpret_cast<const double2*>(qb + f * SLOT_CH + c);
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
          acc[f] = fma(qb[f * SLOT_CH + c], x0, acc[f]);
        } else {
          const double d0 = qb[f * SLOT_CH + c] - x0;
          if (METRIC == RBOD_EUCLID) acc[f] = fma(d0, d0, acc[f]);
          else acc[f] += fabs(d0);
        }
      }
    }
    if (ci == n_chunks - 1) {
      const int64_t r = row_of(g, lane);
      if (r >= 0) {
        const double gn = sqrt(gg);
        End end;
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
          // a policy whose every slot is its own request (slot f = request f) reads no slot table: q = f at compile time
          const int tab = End::kSlotIsRequest ? (f | SLOT_LAST) : slot_s[f];
          end.fold(tab, key);
          if (tab & SLOT_LAST) {
            const int q = tab & SLOT_REQ;
            const double K = end.score(tab);
            if ((K > thr_s[q] || (K == thr_s[q] && (uint32_t)r <= thr_row_s[q])) &&
                (rmask_s[q] < 0 || ((row_mask[(int64_t)rmask_s[q] * mask_words + (r >> 5)] >> (r & 31)) & 1u))) {
              const int slot = atomicAdd(coll_cnt + q, 1);
              if (slot < cap) {
                coll_key[(size_t)q * cap + slot] = K;
                coll_idx[(size_t)q * cap + slot] = (uint32_t)r;
              }
            }
            end.reset();
          }
        }
      }
    }
    __syncthreads();   // everyone is done with buffer b before the copy of step + 2 lands in it
  }
}

using SlotKernel = void (*)(const double*, const float*, const uint16_t*, int, int, int64_t, int64_t, int64_t, int64_t,
                            int64_t, const uint32_t*, int64_t, const int*, const int*, const double*, const uint32_t*,
                            const int*, const double*, int, int, int, double*, uint32_t*, int*);

// Launches kernels[metric][NS == 32] (a kernel whose body is slot_sweep<metric, NS>) over the gallery rows row0,
// row0 + stride, ...: 8 accumulators per lane for passes of up to 8 slots, 32 otherwise.
inline int launch_slot_kernel(const SlotKernel (&kernels)[4][2], const char* who, int metric, const double* q64,
                              const float* master32, const uint16_t* rows16, int kind16, int dim, int64_t ld32,
                              int64_t ld16, int64_t n_rows, int64_t row0, int64_t stride, const uint32_t* row_mask,
                              int64_t mask_words, const int* slot_tab, const int* req_mask, const double* thr,
                              const uint32_t* thr_row, const int* active, const double* qnorm, int n_slots, int n_req,
                              int cap, double* coll_key, uint32_t* coll_idx, int* coll_cnt, int num_sms,
                              cudaStream_t st) {
  if (n_slots <= 0 || n_req <= 0 || n_rows <= 0) return RBOD_OK;
  if (n_slots > 32 || n_req > 32) return set_error(RBOD_E_INVAL, "%s: at most 32 examples per pass", who);
  if (metric < 0 || metric > 3) return set_error(RBOD_E_INVAL, "%s: unknown metric %d", who, metric);
  const int64_t rows_visited = (n_rows - row0 + stride - 1) / stride;
  const int64_t groups = (rows_visited + SLOT_ROWS - 1) / SLOT_ROWS;
  const int grid = (int)std::max<int64_t>(1, std::min<int64_t>(groups, (int64_t)num_sms));
  const int pitch = (master32 ? SLOT_CH : SLOT_CH / 2) + 1;
  const int ns = n_slots <= 8 ? 8 : 32;
  const SlotKernel kern = kernels[metric][ns == 32];
  const size_t smem = (size_t)2 * ns * SLOT_CH * 8 + (size_t)2 * 8 * 32 * pitch * 4;
  RBOD_CUDA(cudaFuncSetAttribute(reinterpret_cast<const void*>(kern), cudaFuncAttributeMaxDynamicSharedMemorySize,
                                 (int)smem));
  kern<<<grid, 256, smem, st>>>(q64, master32, rows16, kind16, dim, ld32, ld16, n_rows, row0, stride, row_mask,
                                mask_words, slot_tab, req_mask, thr, thr_row, active, qnorm, n_slots, n_req, cap,
                                coll_key, coll_idx, coll_cnt);
  RBOD_CUDA(cudaGetLastError());
  return RBOD_OK;
}

}  // namespace

}  // namespace rbod
