// K7  discover -- exact discovery and context search ("like this target, on the positive side of these pairs"), swept
// over the whole gallery on the CUDA cores in fp64.  A request is an optional target t followed by pairs (p, n) of
// examples; a pass holds the examples ("slots") of up to 32 whole requests.  For a row g, with K6's key and sim:
//
//   P = key(p, g), N = key(n, g), f(y) = y / (1 + |y|), s(y) = 0.5 (f(y) + 1), MARGIN = 2^-23
//   rank_pair = +1 if P > N else -1;   loss_pair = f(min(sim(P) - sim(N) - MARGIN, 0))
//   discovery (a target):  K = sum rank_pair + s(sim(key(t, g)))
//   context (no target):   K = sum loss_pair, summed in pair order
//
// K is larger-is-better for every metric, so the selection, the sample pass, the sweep and the tightening are K5's and
// K6's (rbod_api.cu: sweep); the row loop is slot_sweep (rbod_slot_sweep.cuh).  Only the end of a row differs: DiscRow
// below.
#include "rbod_slot_sweep.cuh"

namespace rbod {

namespace {

__device__ __forceinline__ double disc_f(double y) { return y / (1.0 + fabs(y)); }

// End of a row: the target slot stores t, a pair's positive stores P, its negative closes the pair into the running
// rank and loss; the request's last slot picks its score by SLOT_DISC.
template <int METRIC>
struct DiscRow {
  static constexpr bool kSlotIsRequest = false;
  double t = 0.0, p = 0.0, loss = 0.0;
  int rank = 0;
  __device__ __forceinline__ void fold(int tab, double key) {
    if (tab & SLOT_TARGET) {
      t = key;
    } else if (!(tab & SLOT_NEG)) {
      p = key;
    } else {
      rank += p > key ? 1 : -1;
      loss += disc_f(fmin(reco_sim<METRIC>(p) - reco_sim<METRIC>(key) - 0x1p-23, 0.0));
    }
  }
  __device__ __forceinline__ double score(int tab) const {
    return (tab & SLOT_DISC) ? (double)rank + reco_sigmoid(reco_sim<METRIC>(t)) : loss;
  }
  __device__ __forceinline__ void reset() {
    loss = 0.0;
    rank = 0;
  }
};

template <int METRIC, int NS>
__global__ void __launch_bounds__(256, 1)
disc_collect_kernel(const double* __restrict__ q64, const float* __restrict__ master32,
                    const uint16_t* __restrict__ rows16, int kind16, int dim, int64_t ld32, int64_t ld16,
                    int64_t n_rows, int64_t row0, int64_t stride, const uint32_t* __restrict__ row_mask,
                    int64_t mask_words, const int* __restrict__ slot_tab, const int* __restrict__ req_mask,
                    const double* __restrict__ thr, const uint32_t* __restrict__ thr_row,
                    const int* __restrict__ active, const double* __restrict__ qnorm, int n_slots, int n_req, int cap,
                    double* __restrict__ coll_key, uint32_t* __restrict__ coll_idx, int* __restrict__ coll_cnt) {
  slot_sweep<METRIC, NS, DiscRow<METRIC>>(q64, master32, rows16, kind16, dim, ld32, ld16, n_rows, row0, stride,
                                          row_mask, mask_words, slot_tab, req_mask, thr, thr_row, active, qnorm,
                                          n_slots, n_req, cap, coll_key, coll_idx, coll_cnt);
}

}  // namespace

int launch_disc_collect(int metric, const double* q64, const float* master32, const uint16_t* rows16, int kind16,
                        int dim, int64_t ld32, int64_t ld16, int64_t n_rows, int64_t row0, int64_t stride,
                        const uint32_t* row_mask, int64_t mask_words, const int* slot_tab, const int* req_mask,
                        const double* thr, const uint32_t* thr_row, const int* active, const double* qnorm,
                        int n_slots, int n_req, int cap, double* coll_key, uint32_t* coll_idx, int* coll_cnt,
                        int num_sms, cudaStream_t st) {
  static const SlotKernel kernels[4][2] = {
      {disc_collect_kernel<RBOD_COSINE, 8>, disc_collect_kernel<RBOD_COSINE, 32>},
      {disc_collect_kernel<RBOD_DOT, 8>, disc_collect_kernel<RBOD_DOT, 32>},
      {disc_collect_kernel<RBOD_EUCLID, 8>, disc_collect_kernel<RBOD_EUCLID, 32>},
      {disc_collect_kernel<RBOD_MANHATTAN, 8>, disc_collect_kernel<RBOD_MANHATTAN, 32>}};
  return launch_slot_kernel(kernels, "disc_collect", metric, q64, master32, rows16, kind16, dim, ld32, ld16, n_rows,
                            row0, stride, row_mask, mask_words, slot_tab, req_mask, thr, thr_row, active, qnorm,
                            n_slots, n_req, cap, coll_key, coll_idx, coll_cnt, num_sms, st);
}

}  // namespace rbod
