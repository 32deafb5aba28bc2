// Internal declarations shared by the rbod translation units (host side).
#pragma once

#include <cuda.h>
#include <cuda_runtime.h>
#include <cstdint>
#include <cstdarg>
#include <cstddef>

#include <algorithm>

#include "../../include/rbod.h"

namespace rbod {

// ---- error plumbing (rbod_api.cu) -------------------------------------------------------
int set_error(int code, const char* fmt, ...);
#define RBOD_CUDA(expr)                                                                            \
  do {                                                                                             \
    cudaError_t _e = (expr);                                                                       \
    if (_e != cudaSuccess)                                                                         \
      return ::rbod::set_error(RBOD_E_IO, "%s failed: %s (%s:%d)", #expr, cudaGetErrorString(_e),  \
                               __FILE__, __LINE__);                                                \
  } while (0)
#define RBOD_TRY(expr)            \
  do {                            \
    int _rc = (expr);             \
    if (_rc != RBOD_OK) return _rc; \
  } while (0)

// ---- growable device buffers ------------------------------------------------------------
struct DevBuf {
  void* p = nullptr;
  size_t cap = 0;
  int ensure(size_t bytes);  // contents are NOT preserved on growth
  void release();
  template <class T>
  T* as() const { return static_cast<T*>(p); }
};

constexpr int K2_SEG_CHUNK = 256;    // rows per K2 work item (one warp)

// ---- K3 geometry ------------------------------------------------------------------------
constexpr int K3_TILE_M = 128;       // queries per CTA (TMEM lanes)
constexpr int K3_TILE_N = 128;       // gallery rows per accumulator buffer (one tcgen05.mma N)
constexpr int K3_KBLOCK = 64;        // 16-bit elements per 128-byte swizzle row
constexpr int K3_MAX_DP = 768;       // query tile resident in TMEM (+ smem tail): A operand must fit 384 TMEM columns
constexpr int K3_MAX_DP_WIDE = 2048; // wider rows (up to this) stream the query tile through shared memory (variant 1)
constexpr int K3_THREADS = 192;      // warp0 TMA, warp1 MMA, warps 2-5 epilogue
constexpr int K3_MAX_KC = 128;
constexpr int K3_COLLECT_CAP = 1024; // rows a collecting pass records per query before it reports overflow
constexpr int K3_SAMPLE_GROUPS = 8;  // threshold pre-pass: groups whose row maxima are compared
constexpr int K3_SAMPLE_RATIO = 16;  // rows per group = N / (ratio * kc)
constexpr int K3_TAU_REFRESH = 32;   // tiles between two looks at the threshold shared by a query's slices

struct K3Launch {
  CUtensorMap tmap_b;     // gallery [rows, dp] 16-bit, box {64, 128}, SWIZZLE_128B
  CUtensorMap tmap_a;     // queries [Qpad, dp] 16-bit, box {64, 128} (variant 1 only)
  const uint16_t* q16;    // [Qpad, dp]
  int dp;
  int64_t n_rows;         // valid gallery rows
  int tiles_total;        // ceil(n_rows / K3_TILE_N)
  int num_qt;             // Qpad / 128
  int slices;
  int64_t q_valid;
  int64_t q_pad;
  int kc;                 // candidates a prune keeps per (query, slice) list, <= K3_MAX_KC
  int num_stages;
  int a_tmem_kb;          // k-blocks of the query tile kept in TMEM (rest resident in smem)
  int variant;            // 0 = A in TMEM, 1 = A streamed through smem, 2 = A in TMEM + CTA pairs (cta_group::2)
  int kbs;                // k-blocks per pipeline stage of the variant-0 kernel (2 or 4)
  int a_fmt, b_fmt;       // 0 = f16, 1 = bf16
  uint2* lists;           // [slices][q_pad][list_stride] candidate lists {score bits, row index} (select mode)
  int* list_cnt;          // [slices][q_pad] entries per list when its unit is done
  int list_cap;           // prune trigger: 64 (kc <= 32), 128 (kc <= 64) or 256
  int list_stride;        // list_cap + K3_TILE_N
  int final_cap;          // lists longer than this get a last exact prune to kc entries
  const uint32_t* row_mask;       // [n_masks][mask_words] row bitmasks, or nullptr
  const int* mask_of_query;       // [q_pad] mask id per query row (-1 = no mask), or nullptr = all rows read mask 0
  int64_t mask_words;
  const float* row_bias;  // EUCLID collections: [capacity rounded up to whole tiles] -|g|^2 / 2 per stored row
  uint32_t* tau_shared;   // [q_pad] ordered-key thresholds shared across slices, preset to key(-inf); or nullptr
  const float* collect_thr;   // collect mode (second pass for uncertified queries), see k3_cosine_topk.cu
  uint32_t* coll_idx;
  int* coll_cnt;
  int coll_cap;
  float* groupmax_out;        // sample mode: [slices][q_pad] row maxima (threshold pre-pass)
  int group_stride, group_tiles, group_splits;
  float* dump;            // optional raw scores [q_pad][dump_ld]
  int64_t dump_ld;
  int* sync_counters;     // zeroed [slices * sync_span * sync_windows] ints, or nullptr
  int sync_window, sync_lead, sync_span, sync_windows;
  int debug_epi;          // bring-up: 1 = epilogue selects nothing, 2 = epilogue does not read the tile
  unsigned long long* prof;   // optional [16] wait-cycle counters (option k3_prof), see k3_cosine_topk.cu
  int grid;
  size_t smem_bytes;
  int no_coop;            // profiling only: keep the throttle but skip the cooperative-launch attribute
  int* coop_refused;      // optional host counter: ++ when the cooperative launch was refused and the throttle dropped
};

// kernels (each returns RBOD_OK or sets the error) -----------------------------------------
// K1
int launch_l2norm_pack(const float* in, int64_t n, int dim, const int64_t* slots_dev, int64_t slot0,
                       int normalize, int cosine, float* master32, int64_t ld32, uint16_t* out16, int64_t ld16,
                       int kind16, uint16_t* shadow16, float* out_norms, float* stats, int num_sms, cudaStream_t st);
int launch_row_bias(const float* master32, const uint16_t* rows16, int kind16, int dim, int64_t ld32, int64_t ld16,
                    const int64_t* slots_dev, int64_t slot0, int64_t n, float* row_bias, cudaStream_t st);
int launch_gather_rows(const float* master32, const uint16_t* rows16, int kind16, int dim, int64_t ld32,
                       int64_t ld16, const int64_t* rows, int64_t n, int64_t n_valid, float* out, int* err_flag,
                       cudaStream_t st);
// K2
int launch_segment_mean(const float* master32, const uint16_t* rows16, int kind16, int dim, int64_t ld32,
                        int64_t ld16, int64_t n_valid, const int64_t* row_idx, const int64_t* offsets,
                        int64_t n_classes, int64_t n_items_upper, double* partials, int* chunk_prefix,
                        unsigned int* arrive_cnt, float* out, double* sums_out, int normalize, int* err_flag,
                        cudaStream_t st);
int launch_segment_finish(const double* sums, const int64_t* counts, int64_t n_classes, int dim, int normalize,
                          float* out, cudaStream_t st);
int launch_segment_delegates(const float* master32, const uint16_t* rows16, int kind16, int dim, int64_t ld32,
                             int64_t ld16, int64_t n_valid, const int64_t* row_idx, const int64_t* offsets,
                             int64_t n_classes, int kind, double alpha, int cosine, double* scratch, float* out,
                             int64_t* out_member, int* err_flag, int64_t max_class_rows, cudaStream_t st);
// K3
int k3_configure(int device);
int k3_plan(int variant, int want_kbs, int dp, int smem_optin, int allow_hybrid, int* num_stages,
            int* a_tmem_kb, int* kbs_out, size_t* smem_bytes);
int k3_box_rows(int variant);   // gallery rows per TMA box (64 for the CTA-pair kernel)
int launch_k3(const K3Launch& L, cudaStream_t st);
// query preparation: normalise, round to 16 bit, per-query error radius and |q|^2
int launch_prep_queries(const float* q, int64_t Q, int64_t q_pad, int dim, int dp, int kind16, int normalize,
                        uint16_t* q16, float* q_dq, double* q_qq, uint32_t* tau_shared, cudaStream_t st);
// K4 family
int launch_tau_init(const float* groupmax, int groups, int splits, int64_t q_pad, uint32_t* tau_shared,
                    float* tau_init, cudaStream_t st);
// finish: merge of a query's per-slice lists, exact rescoring, top-k, certification (one CTA per query)
struct FinishArgs {
  const uint2* lists;      // [slices][q_pad][list_stride] {score bits, row index}
  const int* list_cnt;     // [slices][q_pad]
  int slices, list_stride, n_cap, kc, k;
  int64_t q_pad;
  const float* tau_init;   // [q_pad] pre-sampled starting thresholds, or nullptr
  const float* q;          // [Q, dim] queries as given
  const double* q_qq;      // [q_pad] |q|^2
  const float* q_dq;       // [q_pad] rounding radius of the 16-bit query
  const float* stats;      // gallery maxima (K1)
  const float* master32;
  const uint16_t* rows16;
  int kind16, dim, metric, master16, shadow, dp;
  int64_t ld32, ld16;
  float* out_scores;
  int64_t* out_rows;
  double* out_scores64;
  int* n_flag;
  int* flag_q;
  double* flag_thr;
  float* flag_lo;
  float* max_eps;
  // split search (rbod_search_begin / rbod_search_end): FIN_SELECT stops after the selection and publishes it,
  // FIN_RESUME picks it up, rescoring only what can still reach the global answer
  int mode, approx_m;
  unsigned long long* sel_keys;   // [Q][kc] selected candidates
  int* sel_n;                     // [Q]
  float* sel_tau;                 // [Q] threshold below which rows were dropped
  float* out_approx;              // [Q][approx_m + 1]: best approximate scores (descending), then the error bound
  const float2* ext_cut;          // [Q] {global k-th best approximate score, largest error bound of any shard}
  double* ubound;                 // [Q] upper bound (exact-key domain) on the rows this shard never listed
};
enum { FIN_FULL = 0, FIN_SELECT = 1, FIN_RESUME = 2 };
int launch_finish(const FinishArgs& A, int64_t Q, cudaStream_t st);
int launch_global_cut(const float* gathered, int G, int64_t Q, int m, int k, float* out_cut2, cudaStream_t st);
int launch_gather_flagged(const uint16_t* q16, int dp, const int* flag_q, int f0, int nf, int64_t nf_pad,
                          uint16_t* fq16, int* coll_cnt, const int* mask_of_query, int* fmask, cudaStream_t st);
int launch_rescore_collected(const float* q, const double* q_qq, const float* master32, const uint16_t* rows16,
                             int kind16, int dim, int64_t ld32, int64_t ld16, int metric, const int* flag_q, int f0,
                             int nf, int cap, const uint32_t* coll_idx, const int* coll_cnt, double* coll_score,
                             cudaStream_t st);
int launch_select_collected(const double* coll_score, const uint32_t* coll_idx, const int* coll_cnt,
                            const int* flag_q, int f0, int nf, int cap, int k, int metric, float* out_scores,
                            int64_t* out_rows, double* out_scores64, cudaStream_t st);
// K5 / K6 / K7: the exact fp64 sweep (rbod_slot_sweep.cuh), one collecting kernel per end of a row, with K5's widening
// and selection.  Slot table of a pass: request of the pass | SLOT_LAST (the request's last slot) | the slot's flags:
// SLOT_NEG (a negative example, K6; a pair's negative, K7), SLOT_TARGET (K7's target) and SLOT_DISC (K7, on every slot
// of a request with a target: the request is scored as a discovery, not a context search).  A K5 query has no flags.
int launch_dist_widen_queries(const float* q, const int* qsel, int nf, int dim, double* q64, double* qnorm,
                              cudaStream_t st);
int launch_dist_select(const double* coll_key, const uint32_t* coll_idx, int* coll_cnt, const int* qsel, int nf,
                       int cap, int k, int sample, int metric, double* thr, uint32_t* thr_row, int* active,
                       int* n_active, float* out_scores, int64_t* out_rows, double* out_keys, cudaStream_t st);
constexpr int SLOT_REQ = 31, SLOT_LAST = 32, SLOT_NEG = 64, SLOT_TARGET = 128, SLOT_DISC = 256;
using CollectLauncher = int (*)(int metric, const double* q64, const float* master32, const uint16_t* rows16,
                                int kind16, int dim, int64_t ld32, int64_t ld16, int64_t n_rows, int64_t row0,
                                int64_t stride, const uint32_t* row_mask, int64_t mask_words, const int* slot_tab,
                                const int* req_mask, const double* thr, const uint32_t* thr_row, const int* active,
                                const double* qnorm, int n_slots, int n_req, int cap, double* coll_key,
                                uint32_t* coll_idx, int* coll_cnt, int num_sms, cudaStream_t st);
int launch_key_collect(int metric, const double* q64, const float* master32, const uint16_t* rows16, int kind16,
                       int dim, int64_t ld32, int64_t ld16, int64_t n_rows, int64_t row0, int64_t stride,
                       const uint32_t* row_mask, int64_t mask_words, const int* slot_tab, const int* req_mask,
                       const double* thr, const uint32_t* thr_row, const int* active, const double* qnorm,
                       int n_slots, int n_req, int cap, double* coll_key, uint32_t* coll_idx, int* coll_cnt,
                       int num_sms, cudaStream_t st);
int launch_reco_collect(int metric, const double* q64, const float* master32, const uint16_t* rows16, int kind16,
                        int dim, int64_t ld32, int64_t ld16, int64_t n_rows, int64_t row0, int64_t stride,
                        const uint32_t* row_mask, int64_t mask_words, const int* slot_tab, const int* req_mask,
                        const double* thr, const uint32_t* thr_row, const int* active, const double* qnorm,
                        int n_slots, int n_req, int cap, double* coll_key, uint32_t* coll_idx, int* coll_cnt,
                        int num_sms, cudaStream_t st);
int launch_disc_collect(int metric, const double* q64, const float* master32, const uint16_t* rows16, int kind16,
                        int dim, int64_t ld32, int64_t ld16, int64_t n_rows, int64_t row0, int64_t stride,
                        const uint32_t* row_mask, int64_t mask_words, const int* slot_tab, const int* req_mask,
                        const double* thr, const uint32_t* thr_row, const int* active, const double* qnorm,
                        int n_slots, int n_req, int cap, double* coll_key, uint32_t* coll_idx, int* coll_cnt,
                        int num_sms, cudaStream_t st);
// K8: maximal marginal relevance over each query's exact candidate list (k8_mmr.cu).  Device pointers throughout.
constexpr int MMR_MAX_CANDIDATES = 1024;
constexpr int MMR_SMEM_DIM = 4096;   // picks up to this many columns are widened into shared memory, wider ones into
                                     // q64_scratch: one row per CTA of mmr_grid
struct MmrArgs {
  int64_t Q;
  int L, limit;
  const int64_t* cand_rows;   // [Q][L] the candidate search's answer: row slots (-1 padded), fp32 scores, fp64 keys
  const float* cand_scores;
  const double* cand_keys;
  const double* diversity;    // [Q] in [0, 1]
  const float* score_threshold;   // [Q] (NaN = none) or nullptr
  const float* master32;
  const uint16_t* rows16;
  int kind16, dim;
  int64_t ld32, ld16;
  double* q64_scratch;        // [mmr_grid][dim] when dim > MMR_SMEM_DIM, else unused
  float* out_scores;          // [Q][limit] in selection order
  int64_t* out_rows;
  double* out_keys;
};
inline int64_t mmr_grid(int64_t Q, int dim, int num_sms) {
  return dim > MMR_SMEM_DIM ? std::min<int64_t>(Q, 2 * (int64_t)num_sms) : Q;
}
int launch_mmr_select(int metric, const MmrArgs& A, int num_sms, cudaStream_t st);
int launch_merge_topk(const double* scores64, const int64_t* ids, int64_t shard_stride, const int64_t* row0_host,
                      int G, int64_t Q, int k, float* out_scores, int64_t* out_ids, double* out_scores64,
                      cudaStream_t st, const double* ubound = nullptr, int* flag_q = nullptr, int* n_flag = nullptr);
// bf16 collection -> fp16 search operand built after the fact (rbod_api.cu: auto_shadow)
int launch_build_shadow(const uint16_t* rows16, int64_t n, int dp, uint16_t* shadow16, float* stats, cudaStream_t st);

}  // namespace rbod

struct rbod_gallery {
  int dim = 0, dp = 0, dtype = 0, metric = 0, device = 0;
  int kind16 = 1;  // 16-bit search operand: 1 = bf16, 2 = fp16
  int64_t rows = 0, capacity = 0;
  float* master32 = nullptr;    // [capacity, dim]  (dtype == RBOD_F32 only)
  uint16_t* rows16 = nullptr;   // [capacity, dp]
  uint16_t* shadow16 = nullptr; // [capacity, dp] fp16 copy of a bf16 gallery used as the search operand (option)
  float* row_bias = nullptr;    // [capacity + 128] EUCLID collections: -|stored row|^2 / 2 (the K3 epilogue adds it)
  int use_shadow = 0;
  int auto_shadow = 1;          // bf16 COSINE collections: build the fp16 shadow when a search with k > 40 arrives
  float* stats = nullptr;       // device [4]: max ||row16||, max ||row16 - unit(master)||, max ||shadow||,
                                // max ||shadow - row16||
  int num_sms = 148;
  // options
  int k3_variant = -1;    // -1 = by batch size (CTA pairs above 128 queries), 0 / 1 / 2 force a kernel flavour
  int k3_kbs = 0;         // k-blocks per stage of the single-CTA kernel: 0 = by batch size, 2, 4
  int slack = -1;  // -1 = automatic
  int time_k3 = 0;
  int debug_epi = 0;
  int coop_launch = 1;       // 0 (profiling only): throttled launches do not ask for a cooperative launch
  int debug_grid_scale = 1;  // test hook: launch this many times the planned CTAs (forces a cooperative-launch refusal)
  int coop_refusals = 0;     // K3 launches that fell back to an ordinary grid (rbod_info reports it)
  int k3_prof = 0;        // accumulate where the K3 warp roles wait (rbod_debug_profile reads and clears)
  int presample = 1;      // threshold pre-pass over a strided sample of the gallery (needs tau_share)
  int collect_pass = 1;   // uncertified queries get a collecting tensor-core pass before the fp64 sweep
  int tau_share = 1;      // slices of one query share their candidate threshold through global memory
  int hybrid = 1;         // allow the query tile to be split between TMEM and resident smem
  int l2_sync = 1;        // producer throttle that keeps slice-mates within an L2 window
  int sync_window = 16, sync_lead = 4;
  // workspaces
  rbod::DevBuf stage_rows, stage_slots, stage_norms;          // upsert staging
  rbod::DevBuf q32, q16, q_dq, q_qq, tau_shared;              // query prep
  rbod::DevBuf lists, list_cnt;                                // K3 candidate lists
  rbod::DevBuf out_scores, out_rows, out_scores64;
  rbod::DevBuf flags;      // ints: [0]=n_flag [2]=err; float max_eps at [3]; [4]=queries the pre-pass cut short
  rbod::DevBuf flag_q, flag_thr, flag_lo, fq16, groupmax, tau_init;
  rbod::DevBuf coll_score, coll_idx, coll_cnt;
  rbod::DevBuf mask_dev, dump, sync_counters, prof;
  rbod::DevBuf mask_ids, fmask_ids;   // per-query mask ids: [q_pad] of the main pass, [q_pad] of the collecting pass
  rbod::DevBuf sel_keys, sel_n, sel_tau;       // split search: the selection rbod_search_begin leaves for rbod_search_end
  struct {                                     // what rbod_search_end needs to know about the pending rbod_search_begin
    int64_t Q = 0;
    int k = 0, kc = 0, approx_m = 0, valid = 0;
    int64_t q_pad = 0;
    const float* q_dev = nullptr;
    int64_t launches = 0;
  } pending;
  rbod::DevBuf seg_idx, seg_off, seg_out, seg_partials, seg_prefix, seg_arrive, seg_scratch, seg_member;
  rbod::DevBuf gather_idx, gather_out;
  rbod::DevBuf dist_q64, dist_thr, dist_ctl;   // K5-K7 sweep: widened slots of a pass, thresholds, the pass's control
  rbod::DevBuf mmr_scores, mmr_rows, mmr_keys;  // K8: the candidate search's answer [Q][L] (search_impl writes it directly)
  rbod::DevBuf mmr_ctl, mmr_q64;                // K8: {diversity, threshold} per query; widened picks of wide rows
  cudaEvent_t ev0 = nullptr, ev1 = nullptr;
};
