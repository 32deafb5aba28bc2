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
// (launch_dist_widen_queries widens the examples, launch_dist_select sorts the per-request lists) and its host loop.
// Only the end of a row differs: K5 records one key per slot, K6 folds a request's slots into one K before it records.
// The row loop is slot_sweep (rbod_slot_sweep.cuh, shared with K5 and K7); the end of a row is RecoRow below.
#include "rbod_slot_sweep.cuh"

namespace rbod {

namespace {

// End of a row: a running bp / bn over the request's slots; SLOT_NEG marks a negative example.
template <int METRIC>
struct RecoRow {
  static constexpr bool kSlotIsRequest = false;
  double bp = -INFINITY, bn = -INFINITY;
  __device__ __forceinline__ void fold(int tab, double key) {
    if (tab & SLOT_NEG) bn = fmax(bn, key); else bp = fmax(bp, key);
  }
  __device__ __forceinline__ double score(int) const {
    return bp > bn ? reco_sigmoid(reco_sim<METRIC>(bp)) : -reco_sigmoid(reco_sim<METRIC>(bn));
  }
  __device__ __forceinline__ void reset() {
    bp = -INFINITY;
    bn = -INFINITY;
  }
};

template <int METRIC, int NS>
__global__ void __launch_bounds__(256, 1)
reco_collect_kernel(const double* __restrict__ q64, const float* __restrict__ master32,
                    const uint16_t* __restrict__ rows16, int kind16, int dim, int64_t ld32, int64_t ld16,
                    int64_t n_rows, int64_t row0, int64_t stride, const uint32_t* __restrict__ row_mask,
                    int64_t mask_words, const int* __restrict__ slot_tab, const int* __restrict__ req_mask,
                    const double* __restrict__ thr, const uint32_t* __restrict__ thr_row,
                    const int* __restrict__ active, const double* __restrict__ qnorm, int n_slots, int n_req, int cap,
                    double* __restrict__ coll_key, uint32_t* __restrict__ coll_idx, int* __restrict__ coll_cnt) {
  slot_sweep<METRIC, NS, RecoRow<METRIC>>(q64, master32, rows16, kind16, dim, ld32, ld16, n_rows, row0, stride,
                                          row_mask, mask_words, slot_tab, req_mask, thr, thr_row, active, qnorm,
                                          n_slots, n_req, cap, coll_key, coll_idx, coll_cnt);
}

}  // namespace

int launch_reco_collect(int metric, const double* q64, const float* master32, const uint16_t* rows16, int kind16,
                        int dim, int64_t ld32, int64_t ld16, int64_t n_rows, int64_t row0, int64_t stride,
                        const uint32_t* row_mask, int64_t mask_words, const int* slot_tab, const int* req_mask,
                        const double* thr, const uint32_t* thr_row, const int* active, const double* qnorm,
                        int n_slots, int n_req, int cap, double* coll_key, uint32_t* coll_idx, int* coll_cnt,
                        int num_sms, cudaStream_t st) {
  static const SlotKernel kernels[4][2] = {
      {reco_collect_kernel<RBOD_COSINE, 8>, reco_collect_kernel<RBOD_COSINE, 32>},
      {reco_collect_kernel<RBOD_DOT, 8>, reco_collect_kernel<RBOD_DOT, 32>},
      {reco_collect_kernel<RBOD_EUCLID, 8>, reco_collect_kernel<RBOD_EUCLID, 32>},
      {reco_collect_kernel<RBOD_MANHATTAN, 8>, reco_collect_kernel<RBOD_MANHATTAN, 32>}};
  return launch_slot_kernel(kernels, "reco_collect", metric, q64, master32, rows16, kind16, dim, ld32, ld16, n_rows,
                            row0, stride, row_mask, mask_words, slot_tab, req_mask, thr, thr_row, active, qnorm,
                            n_slots, n_req, cap, coll_key, coll_idx, coll_cnt, num_sms, st);
}

}  // namespace rbod
