// C ABI of librbod.so (see include/rbod.h for the contract and the reference call sites each
// entry point replaces).  Host-side orchestration only: handle lifetime, host<->device staging,
// work decomposition for the tcgen05 pass, and the certify / fallback loop.
#include "rbod_internal.h"

#include <algorithm>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <ctime>
#include <new>
#include <vector>

namespace rbod {

int make_tmap_2d_sw128(CUtensorMap* out, const void* base, int64_t rows, int dp, int box_rows);

static thread_local char g_err[512] = "";

int set_error(int code, const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
  return code;
}

int DevBuf::ensure(size_t bytes) {
  if (bytes <= cap) return RBOD_OK;
  if (p) cudaFree(p);
  p = nullptr;
  cap = 0;
  size_t want = bytes + bytes / 8 + 256;
  cudaError_t e = cudaMalloc(&p, want);
  if (e != cudaSuccess) {
    cudaGetLastError();
    want = bytes;
    e = cudaMalloc(&p, want);
  }
  if (e != cudaSuccess) {
    cudaGetLastError();
    p = nullptr;
    return set_error(RBOD_E_NOMEM, "cudaMalloc of %zu bytes failed: %s", bytes, cudaGetErrorString(e));
  }
  cap = want;
  return RBOD_OK;
}
void DevBuf::release() {
  if (p) cudaFree(p);
  p = nullptr;
  cap = 0;
}

static bool is_device_ptr(const void* p) {
  if (!p) return false;
  cudaPointerAttributes a;
  if (cudaPointerGetAttributes(&a, p) != cudaSuccess) {
    cudaGetLastError();
    return false;
  }
  return a.type == cudaMemoryTypeDevice || a.type == cudaMemoryTypeManaged;
}

// Returns a device view of `src` (bytes): the pointer itself when it already is device memory,
// otherwise an async copy into `buf`.
static int to_device(const void* src, size_t bytes, DevBuf& buf, cudaStream_t st, const void** out) {
  if (bytes == 0 || is_device_ptr(src)) {
    *out = src;
    return RBOD_OK;
  }
  RBOD_TRY(buf.ensure(bytes));
  RBOD_CUDA(cudaMemcpyAsync(buf.p, src, bytes, cudaMemcpyHostToDevice, st));
  *out = buf.p;
  return RBOD_OK;
}

static int copy_out(void* dst, const void* src_dev, size_t bytes, cudaStream_t st) {
  if (bytes == 0 || dst == nullptr || dst == src_dev) return RBOD_OK;
  RBOD_CUDA(cudaMemcpyAsync(dst, src_dev, bytes, cudaMemcpyDefault, st));
  return RBOD_OK;
}

static size_t elem16_bytes() { return 2; }

static size_t gallery_bytes(const rbod_gallery* g) {
  size_t b = (size_t)g->capacity * g->dp * elem16_bytes();
  if (g->master32) b += (size_t)g->capacity * g->dim * 4;
  if (g->shadow16) b += (size_t)g->capacity * g->dp * 2;
  return b;
}

static int grow(rbod_gallery* g, int64_t need, cudaStream_t st) {
  if (need <= g->capacity) return RBOD_OK;
  int64_t cap = std::max<int64_t>(need, g->capacity + g->capacity / 2);
  cap = std::max<int64_t>(cap, 1024);
  cap = (cap + 63) / 64 * 64;
  uint16_t *n16 = nullptr, *nsh = nullptr;
  float* n32 = nullptr;
  cudaError_t e = cudaMalloc(&n16, (size_t)cap * g->dp * 2);
  if (e != cudaSuccess) {
    cudaGetLastError();
    return set_error(RBOD_E_NOMEM, "gallery: cudaMalloc of %zu bytes failed", (size_t)cap * g->dp * 2);
  }
  if (g->use_shadow) {
    e = cudaMalloc(&nsh, (size_t)cap * g->dp * 2);
    if (e != cudaSuccess) {
      cudaGetLastError();
      cudaFree(n16);
      return set_error(RBOD_E_NOMEM, "gallery: cudaMalloc of %zu bytes (fp16 shadow) failed", (size_t)cap * g->dp * 2);
    }
  }
  if (g->dtype == RBOD_F32) {
    e = cudaMalloc(&n32, (size_t)cap * g->dim * 4);
    if (e != cudaSuccess) {
      cudaGetLastError();
      cudaFree(n16);
      if (nsh) cudaFree(nsh);
      return set_error(RBOD_E_NOMEM, "gallery: cudaMalloc of %zu bytes failed", (size_t)cap * g->dim * 4);
    }
  }
  float* nbias = nullptr;
  if (g->metric == RBOD_EUCLID) {
    e = cudaMalloc(&nbias, (size_t)(cap + K3_TILE_N) * 4);   // whole tiles: the K3 epilogue reads 128 entries at a time
    if (e != cudaSuccess) {
      cudaGetLastError();
      cudaFree(n16);
      if (nsh) cudaFree(nsh);
      if (n32) cudaFree(n32);
      return set_error(RBOD_E_NOMEM, "gallery: cudaMalloc of %zu bytes (row bias) failed", (size_t)(cap + K3_TILE_N) * 4);
    }
    RBOD_CUDA(cudaMemsetAsync(nbias, 0, (size_t)(cap + K3_TILE_N) * 4, st));
    if (g->rows > 0 && g->row_bias)
      RBOD_CUDA(cudaMemcpyAsync(nbias, g->row_bias, (size_t)g->rows * 4, cudaMemcpyDeviceToDevice, st));
  }
  // zero the new tail (keeps the dim..dp padding columns zero), then carry the old rows over
  const size_t old16 = (size_t)g->rows * g->dp * 2;
  RBOD_CUDA(cudaMemsetAsync(reinterpret_cast<uint8_t*>(n16) + old16, 0, (size_t)cap * g->dp * 2 - old16, st));
  if (nsh) RBOD_CUDA(cudaMemsetAsync(reinterpret_cast<uint8_t*>(nsh) + old16, 0, (size_t)cap * g->dp * 2 - old16, st));
  if (g->rows > 0) {
    RBOD_CUDA(cudaMemcpyAsync(n16, g->rows16, old16, cudaMemcpyDeviceToDevice, st));
    if (nsh && g->shadow16) RBOD_CUDA(cudaMemcpyAsync(nsh, g->shadow16, old16, cudaMemcpyDeviceToDevice, st));
    if (n32)
      RBOD_CUDA(cudaMemcpyAsync(n32, g->master32, (size_t)g->rows * g->dim * 4, cudaMemcpyDeviceToDevice, st));
  }
  RBOD_CUDA(cudaStreamSynchronize(st));
  if (g->rows16) cudaFree(g->rows16);
  if (g->master32) cudaFree(g->master32);
  if (g->shadow16) cudaFree(g->shadow16);
  if (g->row_bias) cudaFree(g->row_bias);
  g->rows16 = n16;
  g->master32 = n32;
  g->shadow16 = nsh;
  g->row_bias = nbias;
  g->capacity = cap;
  return RBOD_OK;
}

static int round_up(int x, int m) { return (x + m - 1) / m * m; }

struct SearchPlan {
  int variant;   // kernel flavour this plan is for (0 single CTA, 1 streamed query tile, 2 CTA pairs)
  int kc, slices, grid, num_qt, tiles_total, num_stages, a_tmem_kb, kbs;
  int list_cap, list_stride, final_cap, n_cap;   // candidate-list geometry (see K3Launch / FinishArgs)
  int64_t q_pad;
  size_t smem;
};

static int plan_search(const rbod_gallery* g, int64_t Q, int k, int variant, int smem_optin, SearchPlan* P) {
  // Candidates kept per (query, slice).  Galleries too small for the threshold pre-pass (< 320 tiles = 40 960 rows)
  // never warm their heaps, so the selection, not the contraction, is their cost and it grows with the list length:
  // 10^4 queries x 10^4 rows, k = 5: 1.77 ms with 32 candidates, 1.10 ms with 16, 0.82 ms with 8 -- including the
  // collecting pass for the 55 queries that 3 spare candidates did not certify, which is cheap at this size.
  const int tiles = (int)((g->rows + K3_TILE_N - 1) / K3_TILE_N);
  int kc;
  if (g->slack >= 0) kc = round_up(k + g->slack, 8);
  else if (tiles < 320) kc = std::min(K3_MAX_KC, std::max(8, round_up(k + 3, 8)));
  else kc = k <= 10 ? 32 : (k <= 40 ? 64 : 128);
  if (kc > K3_MAX_KC || kc < k)
    return set_error(RBOD_E_UNSUPPORTED, "search: k=%d (+slack) needs %d candidates per query, max is %d", k, kc,
                     K3_MAX_KC);
  P->kc = kc;
  P->variant = variant;
  const int q_per_unit = variant == 2 ? 2 * K3_TILE_M : K3_TILE_M;   // a CTA pair owns 256 queries
  const int workers = variant == 2 ? std::max(1, g->num_sms / 2) : g->num_sms;
  P->q_pad = (Q + q_per_unit - 1) / q_per_unit * q_per_unit;
  P->num_qt = (int)(P->q_pad / q_per_unit);
  P->tiles_total = (int)((g->rows + K3_TILE_N - 1) / K3_TILE_N);
  // slices: balance (units per CTA) x (tiles per unit); fewer slices on ties (less merge work)
  const int max_slices = std::max(1, std::min({P->tiles_total, 8192 / kc, 2 * workers, 512}));
  double best = 1e300;
  int best_s = 1;
  for (int s = 1; s <= max_slices; ++s) {
    const int64_t units = (int64_t)s * P->num_qt;
    const int64_t per_cta = (units + workers - 1) / workers;
    const double tiles_per_unit = std::ceil((double)P->tiles_total / s);
    const double cost = (double)per_cta * (tiles_per_unit + 24.0);  // +24 ~ per-unit setup in tile units
    if (cost < best * 0.97) { best = cost; best_s = s; }
  }
  P->slices = best_s;
  const int64_t units = (int64_t)P->slices * P->num_qt;
  P->grid = (int)std::min<int64_t>(units, workers) * (variant == 2 ? 2 : 1);
  // Coarse 4-k-block stages (fewer barrier round trips per tile) whenever a CTA pair of query tiles or more is in
  // flight; fine 2-k-block stages for a single query tile, where the launch is HBM-bound and a later first MMA costs
  // more than the round trips.  With the candidate lists out of shared memory both layouts keep the hybrid query tile
  // and two accumulators at any k.  Same-box A/B (tools/k3_where.py, kbs 2 -> 4): 10M x 768 bf16 Q=10^4 1107 -> 1166
  // TF/s; its 8-GPU shard (1.25M rows) 1099 -> 1274 (k = 100: 1074 -> 1211); 1M x 512 fp32 Q=10^4 1105 -> 1178;
  // 12.5M x 768 fp16 Q=1024 1042 -> 1127, Q=256 1039 -> 1062, Q=128 854 -> 762 (worse), Q <= 16 equal.
  const int want_kbs = g->k3_kbs ? g->k3_kbs : ((variant == 2 || P->num_qt >= 2) ? 4 : 2);
  RBOD_TRY(k3_plan(variant, want_kbs, g->dp, smem_optin, g->hybrid, &P->num_stages, &P->a_tmem_kb, &P->kbs,
                   &P->smem));
  // Candidate lists: a list is pruned back to ~kc entries whenever it reaches list_cap (>= 2 kc, so at least kc
  // appends pay for one prune); a tile may append 128 entries before the check, hence the stride.  Lists are left
  // unpruned at the end of a unit unless the query's slices together could exceed what the finish kernel sorts.
  P->list_cap = kc <= 32 ? 64 : (kc <= 64 ? 128 : 256);
  P->list_stride = P->list_cap + K3_TILE_N;
  P->final_cap = std::max(kc, std::min(P->list_stride - 1, 8192 / P->slices));
  P->n_cap = std::min(8192, P->slices * P->final_cap);
  return RBOD_OK;
}

}  // namespace rbod

using namespace rbod;

// =============================================================================================
extern "C" {

const char* rbod_last_error(void) { return g_err; }
int rbod_abi_version(void) { return RBOD_ABI_VERSION; }

int rbod_create(int32_t dim, int32_t dtype, int32_t metric, int64_t capacity_hint, int32_t device,
                rbod_gallery** out) {
  if (!out) return set_error(RBOD_E_INVAL, "rbod_create: out is NULL");
  *out = nullptr;
  if (dim < 1 || dim > 65536) return set_error(RBOD_E_INVAL, "rbod_create: dim %d out of range", dim);
  if (dtype != RBOD_F32 && dtype != RBOD_BF16 && dtype != RBOD_F16)
    return set_error(RBOD_E_INVAL, "rbod_create: unknown dtype %d", dtype);
  if (metric != RBOD_COSINE && metric != RBOD_DOT && metric != RBOD_EUCLID && metric != RBOD_MANHATTAN)
    return set_error(RBOD_E_INVAL, "rbod_create: unknown metric %d", metric);
  int ndev = 0;
  if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) {
    cudaGetLastError();
    return set_error(RBOD_E_IO, "rbod_create: no CUDA device available (this library has no CPU path)");
  }
  if (device < 0 || device >= ndev) return set_error(RBOD_E_INVAL, "rbod_create: device %d of %d", device, ndev);
  RBOD_CUDA(cudaSetDevice(device));
  cudaDeviceProp prop;
  RBOD_CUDA(cudaGetDeviceProperties(&prop, device));
  if (prop.major != 10)
    return set_error(RBOD_E_UNSUPPORTED, "rbod_create: device %d is sm_%d%d; this build is sm_100a only", device,
                     prop.major, prop.minor);
  rbod_gallery* g = new (std::nothrow) rbod_gallery();
  if (!g) return set_error(RBOD_E_NOMEM, "rbod_create: out of host memory");
  g->dim = dim;
  g->dp = round_up(dim, K3_KBLOCK);
  g->dtype = dtype;
  g->metric = metric;
  g->device = device;
  // 16-bit search operand: the master itself for bf16/fp16 galleries; for fp32 galleries an fp16
  // shadow (unit vectors are well inside fp16 range and it halves the rounding radius of bf16),
  // bf16 when the rows are not normalised.
  g->kind16 = dtype == RBOD_BF16 ? 1 : (dtype == RBOD_F16 ? 2 : (metric == RBOD_COSINE ? 2 : 1));
  g->num_sms = prop.multiProcessorCount;
  cudaError_t e = cudaMalloc(&g->stats, 4 * sizeof(float));
  if (e != cudaSuccess) {
    cudaGetLastError();
    delete g;
    return set_error(RBOD_E_NOMEM, "rbod_create: cudaMalloc failed");
  }
  cudaMemset(g->stats, 0, 4 * sizeof(float));
  cudaEventCreate(&g->ev0);
  cudaEventCreate(&g->ev1);
  int rc = grow(g, std::max<int64_t>(capacity_hint, 1), nullptr);
  if (rc != RBOD_OK) {
    rbod_destroy(g);
    return rc;
  }
  *out = g;
  return RBOD_OK;
}

int rbod_destroy(rbod_gallery* g) {
  if (!g) return RBOD_OK;
  cudaSetDevice(g->device);
  cudaDeviceSynchronize();
  if (g->rows16) cudaFree(g->rows16);
  if (g->master32) cudaFree(g->master32);
  if (g->shadow16) cudaFree(g->shadow16);
  if (g->row_bias) cudaFree(g->row_bias);
  if (g->stats) cudaFree(g->stats);
  DevBuf* bufs[] = {&g->stage_rows, &g->stage_slots, &g->stage_norms, &g->q32, &g->q16, &g->q_dq, &g->q_qq, &g->tau_shared,
                    &g->lists, &g->list_cnt, &g->out_scores,
                    &g->out_rows, &g->out_scores64, &g->flags, &g->flag_q, &g->flag_thr, &g->flag_lo, &g->fq16, &g->groupmax, &g->tau_init, &g->coll_score,
                    &g->coll_idx, &g->coll_cnt, &g->mask_dev, &g->mask_ids, &g->fmask_ids, &g->dump, &g->sync_counters, &g->prof, &g->seg_idx, &g->seg_off, &g->seg_out,
                    &g->seg_partials, &g->seg_prefix, &g->seg_arrive, &g->seg_scratch, &g->seg_member, &g->gather_idx,
                    &g->gather_out, &g->dist_q64, &g->dist_thr, &g->dist_ctl, &g->mmr_scores, &g->mmr_rows,
                    &g->mmr_keys, &g->mmr_ctl, &g->mmr_q64};
  for (DevBuf* b : bufs) b->release();
  if (g->ev0) cudaEventDestroy(g->ev0);
  if (g->ev1) cudaEventDestroy(g->ev1);
  cudaGetLastError();
  delete g;
  return RBOD_OK;
}

int64_t rbod_count(const rbod_gallery* g) { return g ? g->rows : (int64_t)set_error(RBOD_E_INVAL, "NULL handle"); }

int rbod_info(const rbod_gallery* g, rbod_gallery_info* out) {
  if (!g || !out) return set_error(RBOD_E_INVAL, "rbod_info: NULL argument");
  RBOD_CUDA(cudaSetDevice(g->device));
  memset(out, 0, sizeof(*out));
  out->dim = g->dim;
  out->dim_padded = g->dp;
  out->dtype = g->dtype;
  out->metric = g->metric;
  out->device = g->device;
  out->rows = g->rows;
  out->capacity = g->capacity;
  out->coop_refusals = g->coop_refusals;
  size_t ws = 0;
  const DevBuf* bufs[] = {&g->stage_rows, &g->q32, &g->q16, &g->lists, &g->list_cnt, &g->out_scores, &g->out_rows, &g->out_scores64, &g->coll_score,
                          &g->coll_idx, &g->mask_dev, &g->mask_ids, &g->fmask_ids, &g->dump, &g->seg_idx, &g->seg_out, &g->seg_partials,
                          &g->gather_out};
  for (const DevBuf* b : bufs) ws += b->cap;
  out->bytes_device = (int64_t)(gallery_bytes(g) + ws);
  float st[2] = {0, 0};
  RBOD_CUDA(cudaMemcpy(st, g->stats, sizeof(st), cudaMemcpyDeviceToHost));
  out->max_row_norm = st[0];
  out->max_row_dev = st[1];
  return RBOD_OK;
}

int rbod_truncate(rbod_gallery* g, int64_t rows) {
  if (!g) return set_error(RBOD_E_INVAL, "rbod_truncate: NULL handle");
  if (rows < 0 || rows > g->rows) return set_error(RBOD_E_RANGE, "rbod_truncate: %lld not in [0, %lld]",
                                                   (long long)rows, (long long)g->rows);
  g->rows = rows;
  if (rows == 0) {
    RBOD_CUDA(cudaSetDevice(g->device));
    RBOD_CUDA(cudaMemset(g->stats, 0, 4 * sizeof(float)));
  }
  return RBOD_OK;
}

int rbod_set_option(rbod_gallery* g, const char* key, int64_t value) {
  if (!g || !key) return set_error(RBOD_E_INVAL, "rbod_set_option: NULL argument");
  if (!strcmp(key, "k3_variant")) {
    if (value < -1 || value > 2) return set_error(RBOD_E_INVAL, "k3_variant must be -1 (by batch size), 0, 1 or 2");
    g->k3_variant = (int)value;
  } else if (!strcmp(key, "k3_kbs")) {
    if (value != 0 && value != 2 && value != 4) return set_error(RBOD_E_INVAL, "k3_kbs must be 0 (auto), 2 or 4");
    g->k3_kbs = (int)value;
  } else if (!strcmp(key, "slack")) {
    if (value < -1 || value > 118) return set_error(RBOD_E_INVAL, "slack must be in [-1, 118]");
    g->slack = (int)value;
  } else if (!strcmp(key, "time_k3")) {
    g->time_k3 = value != 0;
  } else if (!strcmp(key, "shadow16")) {
    // fp16 search operand for a bf16 collection (doubles its device memory); must be chosen while it is empty
    if (g->dtype != RBOD_BF16) return set_error(RBOD_E_INVAL, "shadow16 applies to bf16 collections only");
    if (g->rows != 0) return set_error(RBOD_E_INVAL, "shadow16 must be set before the first upsert");
    if ((value != 0) != (g->use_shadow != 0)) {
      g->use_shadow = value != 0;
      if (g->shadow16) { cudaFree(g->shadow16); g->shadow16 = nullptr; }
      if (g->use_shadow) {
        RBOD_CUDA(cudaSetDevice(g->device));
        RBOD_CUDA(cudaMalloc(&g->shadow16, (size_t)g->capacity * g->dp * 2));
        RBOD_CUDA(cudaMemset(g->shadow16, 0, (size_t)g->capacity * g->dp * 2));
      }
    }
  } else if (!strcmp(key, "auto_shadow")) {
    g->auto_shadow = value != 0;
  } else if (!strcmp(key, "presample")) {
    if (value < 0 || value > 2) return set_error(RBOD_E_INVAL, "presample must be 0 (off), 1 (when it pays) or 2 (always)");
    g->presample = (int)value;
  } else if (!strcmp(key, "collect_pass")) {
    g->collect_pass = value != 0;
  } else if (!strcmp(key, "tau_share")) {
    g->tau_share = value != 0;
  } else if (!strcmp(key, "debug_epi")) {
    g->debug_epi = (int)value;   // bring-up only: results are wrong when non-zero
  } else if (!strcmp(key, "coop_launch")) {
    g->coop_launch = value != 0;   // 0 is for profilers that cannot replay cooperative cluster launches (ncu): nothing
                                   // then guarantees that the CTAs the throttle makes wait for each other are co-resident
  } else if (!strcmp(key, "debug_grid_scale")) {
    if (value < 1 || value > 8) return set_error(RBOD_E_INVAL, "debug_grid_scale must be in [1, 8]");
    g->debug_grid_scale = (int)value;
  } else if (!strcmp(key, "k3_prof")) {
    g->k3_prof = value != 0;
  } else if (!strcmp(key, "hybrid")) {
    g->hybrid = value != 0;
  } else if (!strcmp(key, "l2_sync")) {
    g->l2_sync = value != 0;
  } else if (!strcmp(key, "sync_window")) {
    if (value < 1 || value > 4096) return set_error(RBOD_E_INVAL, "sync_window must be in [1, 4096]");
    g->sync_window = (int)value;
  } else if (!strcmp(key, "sync_lead")) {
    if (value < 1 || value > 64) return set_error(RBOD_E_INVAL, "sync_lead must be in [1, 64]");
    g->sync_lead = (int)value;
  } else {
    return set_error(RBOD_E_INVAL, "rbod_set_option: unknown key '%s'", key);
  }
  return RBOD_OK;
}

// ---------------------------------------------------------------------------------------------
int rbod_upsert(rbod_gallery* g, const float* rows, int64_t n, const int64_t* row_slots, float* out_norms,
                int32_t flags, void* stream) {
  if (!g) return set_error(RBOD_E_INVAL, "rbod_upsert: NULL handle");
  if (n < 0 || (n > 0 && !rows)) return set_error(RBOD_E_INVAL, "rbod_upsert: bad rows/n");
  if (n == 0) return RBOD_OK;
  RBOD_CUDA(cudaSetDevice(g->device));
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  std::vector<int64_t> slots_host;
  if (row_slots && is_device_ptr(row_slots)) {
    // slots living on the device are read back: they are validated (range, no holes) on the host
    slots_host.resize((size_t)n);
    RBOD_CUDA(cudaMemcpyAsync(slots_host.data(), row_slots, (size_t)n * 8, cudaMemcpyDeviceToHost, st));
    RBOD_CUDA(cudaStreamSynchronize(st));
    row_slots = slots_host.data();
  }

  int64_t new_rows = g->rows + n;
  if (row_slots) {
    int64_t mn = INT64_MAX, mx = -1, fresh = 0;
    for (int64_t i = 0; i < n; ++i) {
      if (row_slots[i] < 0) return set_error(RBOD_E_RANGE, "rbod_upsert: negative slot at %lld", (long long)i);
      mn = std::min(mn, row_slots[i]);
      mx = std::max(mx, row_slots[i]);
    }
    if (mx - g->rows >= n)   // a hole whatever the slots are; also bounds the bitmap below
      return set_error(RBOD_E_RANGE, "rbod_upsert: slots would leave holes (max slot %lld, rows %lld)",
                       (long long)mx, (long long)g->rows);
    // Slots must be distinct: two K1 warps would write a repeated slot in no defined order (master, 16-bit row and
    // bias each from either input, stats from both), and counted twice below it would hide a hole.  One bit per slot
    // of [mn, mx], no sort: a bulk overwrite may carry millions of slots, a delete's move carries one.
    std::vector<uint64_t> seen((size_t)((mx - mn) / 64 + 1), 0);
    for (int64_t i = 0; i < n; ++i) {
      const uint64_t off = (uint64_t)(row_slots[i] - mn), bit = 1ull << (off % 64);
      if (seen[off / 64] & bit)
        return set_error(RBOD_E_INVAL, "rbod_upsert: slot %lld appears more than once", (long long)row_slots[i]);
      seen[off / 64] |= bit;
      if (row_slots[i] >= g->rows) ++fresh;
    }
    new_rows = std::max(g->rows, mx + 1);
    if (mx + 1 > g->rows + fresh)
      return set_error(RBOD_E_RANGE, "rbod_upsert: slots would leave holes (max slot %lld, rows %lld)",
                       (long long)mx, (long long)g->rows);
  }
  RBOD_TRY(grow(g, new_rows, st));

  const int normalize = (g->metric == RBOD_COSINE) && !(flags & RBOD_UPSERT_RAW);
  const int cosine = g->metric == RBOD_COSINE;
  const bool rows_dev = is_device_ptr(rows);
  const bool norms_dev = out_norms && is_device_ptr(out_norms);
  // chunking bounds the staging buffers for host input
  const int64_t chunk_rows = rows_dev ? n : std::max<int64_t>(1, std::min<int64_t>(n, (256ll << 20) / ((int64_t)g->dim * 4)));
  for (int64_t r0 = 0; r0 < n; r0 += chunk_rows) {
    const int64_t m = std::min(chunk_rows, n - r0);
    const float* src = rows + r0 * g->dim;
    if (!rows_dev) {
      RBOD_TRY(g->stage_rows.ensure((size_t)m * g->dim * 4));
      RBOD_CUDA(cudaMemcpyAsync(g->stage_rows.p, src, (size_t)m * g->dim * 4, cudaMemcpyHostToDevice, st));
      src = g->stage_rows.as<float>();
    }
    const int64_t* slots_dev = nullptr;
    if (row_slots) {
      RBOD_TRY(g->stage_slots.ensure((size_t)m * 8));
      RBOD_CUDA(cudaMemcpyAsync(g->stage_slots.p, row_slots + r0, (size_t)m * 8, cudaMemcpyHostToDevice, st));
      slots_dev = g->stage_slots.as<int64_t>();
    }
    float* norms_dst = nullptr;
    if (out_norms) {
      if (norms_dev) norms_dst = out_norms + r0;
      else {
        RBOD_TRY(g->stage_norms.ensure((size_t)m * 4));
        norms_dst = g->stage_norms.as<float>();
      }
    }
    RBOD_TRY(launch_l2norm_pack(src, m, g->dim, slots_dev, g->rows + r0, normalize, cosine, g->master32, g->dim,
                                g->rows16, g->dp, g->kind16, g->shadow16, norms_dst, g->stats, g->num_sms, st));
    if (g->row_bias)
      RBOD_TRY(launch_row_bias(g->master32, g->rows16, g->kind16, g->dim, g->dim, g->dp, slots_dev, g->rows + r0, m,
                               g->row_bias, st));
    if (out_norms && !norms_dev)
      RBOD_CUDA(cudaMemcpyAsync(out_norms + r0, norms_dst, (size_t)m * 4, cudaMemcpyDeviceToHost, st));
    if (!rows_dev || row_slots) RBOD_CUDA(cudaStreamSynchronize(st));  // staging buffers are reused
  }
  g->rows = new_rows;
  if (out_norms && !norms_dev) RBOD_CUDA(cudaStreamSynchronize(st));
  return RBOD_OK;
}

int rbod_get_rows(rbod_gallery* g, const int64_t* rows, int64_t n, float* out, void* stream) {
  if (!g) return set_error(RBOD_E_INVAL, "rbod_get_rows: NULL handle");
  if (n < 0 || (n > 0 && (!rows || !out))) return set_error(RBOD_E_INVAL, "rbod_get_rows: bad arguments");
  if (n == 0) return RBOD_OK;
  RBOD_CUDA(cudaSetDevice(g->device));
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const void* rows_dev = nullptr;
  RBOD_TRY(to_device(rows, (size_t)n * 8, g->gather_idx, st, &rows_dev));
  const bool out_dev = is_device_ptr(out);
  float* dst = out;
  if (!out_dev) {
    RBOD_TRY(g->gather_out.ensure((size_t)n * g->dim * 4));
    dst = g->gather_out.as<float>();
  }
  RBOD_TRY(g->flags.ensure(64));
  RBOD_CUDA(cudaMemsetAsync(g->flags.p, 0, 64, st));
  RBOD_TRY(launch_gather_rows(g->master32, g->rows16, g->kind16, g->dim, g->dim, g->dp,
                              static_cast<const int64_t*>(rows_dev), n, g->rows, dst, g->flags.as<int>() + 2, st));
  if (!out_dev) RBOD_CUDA(cudaMemcpyAsync(out, dst, (size_t)n * g->dim * 4, cudaMemcpyDeviceToHost, st));
  int err = 0;
  RBOD_CUDA(cudaMemcpyAsync(&err, g->flags.as<int>() + 2, 4, cudaMemcpyDeviceToHost, st));
  RBOD_CUDA(cudaStreamSynchronize(st));
  if (err) return set_error(RBOD_E_RANGE, "rbod_get_rows: row index outside [0, %lld)", (long long)g->rows);
  return RBOD_OK;
}

int rbod_l2norm_pack(const float* in, int64_t n, int32_t dim, int32_t out_dtype, void* out, int64_t out_ld,
                     float* out_norms, void* stream) {
  if (n < 0 || dim < 1 || (n > 0 && (!in || !out))) return set_error(RBOD_E_INVAL, "rbod_l2norm_pack: bad arguments");
  if (out_ld < dim) return set_error(RBOD_E_INVAL, "rbod_l2norm_pack: out_ld < dim");
  if (n == 0) return RBOD_OK;
  if (!is_device_ptr(in) || !is_device_ptr(out) || (out_norms && !is_device_ptr(out_norms)))
    return set_error(RBOD_E_INVAL, "rbod_l2norm_pack: device pointers only");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  int dev = 0, sms = 148;
  RBOD_CUDA(cudaGetDevice(&dev));
  RBOD_CUDA(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
  if (out_dtype == RBOD_F32)
    return launch_l2norm_pack(in, n, dim, nullptr, 0, 1, 1, static_cast<float*>(out), out_ld, nullptr, 0, 1,
                              nullptr, out_norms, nullptr, sms, st);
  if (out_dtype == RBOD_BF16 || out_dtype == RBOD_F16)
    return launch_l2norm_pack(in, n, dim, nullptr, 0, 1, 1, nullptr, 0, static_cast<uint16_t*>(out), out_ld,
                              out_dtype == RBOD_BF16 ? 1 : 2, nullptr, out_norms, nullptr, sms, st);
  return set_error(RBOD_E_INVAL, "rbod_l2norm_pack: unknown out_dtype %d", out_dtype);
}

// ---------------------------------------------------------------------------------------------
// K2 front end.  out_centroids != NULL: finished delegate vectors [C, dim] fp32 (host or device);
// out_sums != NULL: raw fp64 column sums [C, dim] (device only) for the sharded build.
static int segment_mean_impl(rbod_gallery* g, const int64_t* row_idx, const int64_t* offsets, int64_t n_classes,
                             float* out_centroids, double* out_sums, void* stream) {
  if (!g) return set_error(RBOD_E_INVAL, "rbod_segment_mean: NULL handle");
  if (n_classes < 0 || (n_classes > 0 && (!offsets || (!out_centroids && !out_sums))))
    return set_error(RBOD_E_INVAL, "rbod_segment_mean: bad arguments");
  if (out_sums && !is_device_ptr(out_sums))
    return set_error(RBOD_E_INVAL, "rbod_segment_sums: out_sums must be a device pointer");
  if (n_classes == 0) return RBOD_OK;
  if (n_classes > (1ll << 30)) return set_error(RBOD_E_INVAL, "rbod_segment_mean: too many classes");
  RBOD_CUDA(cudaSetDevice(g->device));
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  int64_t first = 0, total = 0;
  if (is_device_ptr(offsets)) {
    RBOD_CUDA(cudaMemcpyAsync(&first, offsets, 8, cudaMemcpyDeviceToHost, st));
    RBOD_CUDA(cudaMemcpyAsync(&total, offsets + n_classes, 8, cudaMemcpyDeviceToHost, st));
    RBOD_CUDA(cudaStreamSynchronize(st));
  } else {
    first = offsets[0];
    total = offsets[n_classes];
    for (int64_t c = 0; c < n_classes; ++c)
      if (offsets[c + 1] < offsets[c]) return set_error(RBOD_E_INVAL, "rbod_segment_mean: offsets not monotone");
  }
  if (first < 0 || total < first) return set_error(RBOD_E_INVAL, "rbod_segment_mean: bad offsets");
  if (!row_idx && total > g->rows) return set_error(RBOD_E_RANGE, "rbod_segment_mean: offsets exceed row count");
  const void *idx_dev = nullptr, *off_dev = nullptr;
  if (row_idx) RBOD_TRY(to_device(row_idx, (size_t)total * 8, g->seg_idx, st, &idx_dev));
  RBOD_TRY(to_device(offsets, (size_t)(n_classes + 1) * 8, g->seg_off, st, &off_dev));
  const bool out_dev = out_sums != nullptr || is_device_ptr(out_centroids);
  float* dst = out_centroids;
  if (!out_dev) {
    RBOD_TRY(g->seg_out.ensure((size_t)n_classes * g->dim * 4));
    dst = g->seg_out.as<float>();
  }
  const int64_t items_upper = (total - first) / K2_SEG_CHUNK + n_classes + 1;
  const int64_t parts_upper = 2 * ((total - first) / K2_SEG_CHUNK) + 2;
  if (items_upper > 0x7fffffff) return set_error(RBOD_E_INVAL, "rbod_segment_mean: problem too large");
  RBOD_TRY(g->seg_partials.ensure((size_t)parts_upper * g->dim * 8));
  RBOD_TRY(g->seg_prefix.ensure((size_t)(2 * n_classes + 2) * 4));
  RBOD_TRY(g->seg_arrive.ensure((size_t)parts_upper * 4));   // one flag word per partial slot (tree reduction)
  RBOD_CUDA(cudaMemsetAsync(g->seg_arrive.p, 0, (size_t)parts_upper * 4, st));
  RBOD_TRY(g->flags.ensure(64));
  RBOD_CUDA(cudaMemsetAsync(g->flags.p, 0, 64, st));
  RBOD_TRY(launch_segment_mean(g->master32, g->rows16, g->kind16, g->dim, g->dim, g->dp, g->rows,
                               static_cast<const int64_t*>(idx_dev), static_cast<const int64_t*>(off_dev), n_classes,
                               items_upper, g->seg_partials.as<double>(), g->seg_prefix.as<int>(),
                               g->seg_arrive.as<unsigned int>(), dst, out_sums, g->metric == RBOD_COSINE,
                               g->flags.as<int>() + 2, st));
  if (!out_dev)
    RBOD_CUDA(cudaMemcpyAsync(out_centroids, dst, (size_t)n_classes * g->dim * 4, cudaMemcpyDeviceToHost, st));
  int err = 0;
  RBOD_CUDA(cudaMemcpyAsync(&err, g->flags.as<int>() + 2, 4, cudaMemcpyDeviceToHost, st));
  RBOD_CUDA(cudaStreamSynchronize(st));
  if (err) return set_error(RBOD_E_RANGE, "rbod_segment_mean: row index outside [0, %lld)", (long long)g->rows);
  return RBOD_OK;
}

int rbod_segment_mean(rbod_gallery* g, const int64_t* row_idx, const int64_t* offsets, int64_t n_classes,
                      float* out_centroids, void* stream) {
  if (n_classes > 0 && !out_centroids) return set_error(RBOD_E_INVAL, "rbod_segment_mean: out_centroids is NULL");
  return segment_mean_impl(g, row_idx, offsets, n_classes, out_centroids, nullptr, stream);
}

int rbod_segment_sums(rbod_gallery* g, const int64_t* row_idx, const int64_t* offsets, int64_t n_classes,
                      double* out_sums, void* stream) {
  if (n_classes > 0 && !out_sums) return set_error(RBOD_E_INVAL, "rbod_segment_sums: out_sums is NULL");
  return segment_mean_impl(g, row_idx, offsets, n_classes, nullptr, out_sums, stream);
}

int rbod_segment_finish(const double* sums, const int64_t* counts, int64_t n_classes, int32_t dim, int32_t normalize,
                        float* out_vectors, void* stream) {
  if (n_classes < 0 || dim < 1 || (n_classes > 0 && (!sums || !counts || !out_vectors)))
    return set_error(RBOD_E_INVAL, "rbod_segment_finish: bad arguments");
  if (n_classes == 0) return RBOD_OK;
  if (!is_device_ptr(sums) || !is_device_ptr(counts) || !is_device_ptr(out_vectors))
    return set_error(RBOD_E_INVAL, "rbod_segment_finish: device pointers only");
  return launch_segment_finish(sums, counts, n_classes, dim, normalize, out_vectors, static_cast<cudaStream_t>(stream));
}

int rbod_segment_delegates(rbod_gallery* g, int32_t kind, const int64_t* row_idx, const int64_t* offsets,
                           int64_t n_classes, double alpha, float* out_vectors, int64_t* out_member_rows,
                           void* stream) {
  if (!g) return set_error(RBOD_E_INVAL, "rbod_segment_delegates: NULL handle");
  if (kind == RBOD_DELEGATE_AVERAGE) {
    RBOD_TRY(rbod_segment_mean(g, row_idx, offsets, n_classes, out_vectors, stream));
    if (out_member_rows && n_classes > 0) {
      if (is_device_ptr(out_member_rows))
        RBOD_CUDA(cudaMemsetAsync(out_member_rows, 0xff, (size_t)n_classes * 8, static_cast<cudaStream_t>(stream)));
      else
        for (int64_t c = 0; c < n_classes; ++c) out_member_rows[c] = -1;
    }
    return RBOD_OK;
  }
  if (kind != RBOD_DELEGATE_CENTROID && kind != RBOD_DELEGATE_WEIGHTED && kind != RBOD_DELEGATE_MEDOID)
    return set_error(RBOD_E_INVAL, "rbod_segment_delegates: unknown kind %d", kind);
  if (n_classes < 0 || (n_classes > 0 && (!offsets || !out_vectors)))
    return set_error(RBOD_E_INVAL, "rbod_segment_delegates: bad arguments");
  if (n_classes == 0) return RBOD_OK;
  if (n_classes > 0x7fffffffll) return set_error(RBOD_E_INVAL, "rbod_segment_delegates: too many classes");
  RBOD_CUDA(cudaSetDevice(g->device));
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  int64_t first = 0, total = 0, max_class = 0;
  {
    // the class sizes decide which medoid kernel a class takes: a device-resident offsets array is read back once
    std::vector<int64_t> off_host;
    const int64_t* oh = offsets;
    if (is_device_ptr(offsets)) {
      off_host.resize((size_t)n_classes + 1);
      RBOD_CUDA(cudaMemcpyAsync(off_host.data(), offsets, (size_t)(n_classes + 1) * 8, cudaMemcpyDeviceToHost, st));
      RBOD_CUDA(cudaStreamSynchronize(st));
      oh = off_host.data();
    }
    first = oh[0];
    total = oh[n_classes];
    for (int64_t c = 0; c < n_classes; ++c) {
      if (oh[c + 1] < oh[c]) return set_error(RBOD_E_INVAL, "rbod_segment_delegates: offsets not monotone");
      max_class = std::max(max_class, oh[c + 1] - oh[c]);
    }
  }
  if (first < 0 || total < first) return set_error(RBOD_E_INVAL, "rbod_segment_delegates: bad offsets");
  if (!row_idx && total > g->rows) return set_error(RBOD_E_RANGE, "rbod_segment_delegates: offsets exceed row count");
  const void *idx_dev = nullptr, *off_dev = nullptr;
  if (row_idx) RBOD_TRY(to_device(row_idx, (size_t)total * 8, g->seg_idx, st, &idx_dev));
  RBOD_TRY(to_device(offsets, (size_t)(n_classes + 1) * 8, g->seg_off, st, &off_dev));
  const bool out_dev = is_device_ptr(out_vectors);
  float* dst = out_vectors;
  if (!out_dev) {
    RBOD_TRY(g->seg_out.ensure((size_t)n_classes * g->dim * 4));
    dst = g->seg_out.as<float>();
  }
  int64_t* mem_dst = nullptr;
  const bool mem_dev = out_member_rows && is_device_ptr(out_member_rows);
  if (out_member_rows) {
    if (mem_dev) mem_dst = out_member_rows;
    else {
      RBOD_TRY(g->seg_member.ensure((size_t)n_classes * 8));
      mem_dst = g->seg_member.as<int64_t>();
    }
  }
  RBOD_TRY(g->seg_scratch.ensure((size_t)std::max<int64_t>(total, 1) * 8));
  RBOD_TRY(g->flags.ensure(64));
  RBOD_CUDA(cudaMemsetAsync(g->flags.p, 0, 64, st));
  RBOD_TRY(launch_segment_delegates(g->master32, g->rows16, g->kind16, g->dim, g->dim, g->dp, g->rows,
                                    static_cast<const int64_t*>(idx_dev), static_cast<const int64_t*>(off_dev),
                                    n_classes, kind, alpha, g->metric == RBOD_COSINE, g->seg_scratch.as<double>(), dst,
                                    mem_dst, g->flags.as<int>() + 2, max_class, st));
  if (!out_dev)
    RBOD_CUDA(cudaMemcpyAsync(out_vectors, dst, (size_t)n_classes * g->dim * 4, cudaMemcpyDeviceToHost, st));
  if (out_member_rows && !mem_dev)
    RBOD_CUDA(cudaMemcpyAsync(out_member_rows, mem_dst, (size_t)n_classes * 8, cudaMemcpyDeviceToHost, st));
  int err = 0;
  RBOD_CUDA(cudaMemcpyAsync(&err, g->flags.as<int>() + 2, 4, cudaMemcpyDeviceToHost, st));
  RBOD_CUDA(cudaStreamSynchronize(st));
  if (err) return set_error(RBOD_E_RANGE, "rbod_segment_delegates: row index outside [0, %lld)", (long long)g->rows);
  return RBOD_OK;
}

// ---------------------------------------------------------------------------------------------
// 16-bit type the (unit-norm) queries are rounded to for the tensor-core pass: the gallery's own.
// (Measured on B200: a kind::f16 MMA whose instruction descriptor mixes an fp16 A with a bf16 B
// raises "illegal instruction", so both operands must share one format.)
// The kernel flavour a collection's searches run on: rows wider than the TMEM-resident query tile allows (768 columns)
// stream the query tile through shared memory next to the gallery tile (variant 1: twice the L2 -> SM traffic per
// flop, still two orders of magnitude faster than the fp64 sweep such collections took before).
// Otherwise (option k3_variant = -1, the default): CTA pairs (cta_group::2, M = 256 per pair, each CTA streaming half
// of every gallery tile) as soon as a second query tile exists -- 1555 vs 1166 TFLOP/s on the headline shape, same box
// -- and the single-CTA kernel for batches of at most 128 queries, where a pair would idle one of its two SMs.
static int search_variant(const rbod_gallery* g, int64_t Q) {
  if (g->dp > K3_MAX_DP) return 1;
  if (g->k3_variant >= 0) return g->k3_variant;
  return Q > K3_TILE_M ? 2 : 0;
}

static int query_kind(const rbod_gallery* g) { return g->use_shadow ? 2 : g->kind16; }
static const uint16_t* search_operand(const rbod_gallery* g) { return g->use_shadow ? g->shadow16 : g->rows16; }

struct K3Collect {
  const float* thr;
  uint32_t* idx;
  int* cnt;
  int cap;
};

struct K3Sample {
  float* groupmax;   // [groups * splits][q_pad]
  int stride, tiles, splits;
};

// Row masks of one search.  `dev`: [n_masks][words] bitmasks on the device, nullptr = no filter.  `of_query`: the mask
// each query row of the K3 launch reads ([q_pad] on the device, -1 = none) and `of_query_host` the same ids by query (or
// request) index ([Q] on the host, read by the sweep's batch control); both nullptr = every query reads mask 0.
struct SearchMasks {
  const uint32_t* dev;
  int64_t words;
  const int* of_query;
  const int* of_query_host;
};

static int run_k3(rbod_gallery* g, const SearchPlan& P, int64_t Q, const uint16_t* q16, const SearchMasks& M,
                  const K3Collect* collect, float* dump, int64_t dump_ld, cudaStream_t st,
                  const K3Sample* sample = nullptr) {
  K3Launch L;
  memset(&L, 0, sizeof(L));
  RBOD_TRY(make_tmap_2d_sw128(&L.tmap_b, search_operand(g), g->rows, g->dp, k3_box_rows(P.variant)));
  RBOD_TRY(make_tmap_2d_sw128(&L.tmap_a, q16, P.q_pad, g->dp, K3_TILE_M));
  L.q16 = q16;
  if (collect) {
    L.collect_thr = collect->thr;
    L.coll_idx = collect->idx;
    L.coll_cnt = collect->cnt;
    L.coll_cap = collect->cap;
  }
  L.dp = g->dp;
  L.n_rows = g->rows;
  L.tiles_total = P.tiles_total;
  L.num_qt = P.num_qt;
  L.slices = P.slices;
  L.q_valid = Q;
  L.q_pad = P.q_pad;
  L.kc = P.kc;
  L.num_stages = P.num_stages;
  L.a_tmem_kb = P.a_tmem_kb;
  L.variant = P.variant;
  L.kbs = P.kbs;
  L.debug_epi = g->debug_epi;
  if (g->k3_prof && collect == nullptr && sample == nullptr && dump == nullptr) {
    if (g->prof.p == nullptr) {
      RBOD_TRY(g->prof.ensure(16 * sizeof(unsigned long long)));
      RBOD_CUDA(cudaMemsetAsync(g->prof.p, 0, 16 * sizeof(unsigned long long), st));
    }
    L.prof = g->prof.as<unsigned long long>();
  }
  L.a_fmt = query_kind(g) == 1 ? 1 : 0;
  L.b_fmt = query_kind(g) == 1 ? 1 : 0;
  L.lists = g->lists.as<uint2>();
  L.list_cnt = g->list_cnt.as<int>();
  L.list_cap = P.list_cap;
  L.list_stride = P.list_stride;
  L.final_cap = P.final_cap;
  L.row_mask = M.dev;
  L.mask_of_query = M.dev != nullptr ? M.of_query : nullptr;
  L.mask_words = M.words;
  L.row_bias = g->metric == RBOD_EUCLID ? g->row_bias : nullptr;
  L.tau_shared = (g->tau_share && dump == nullptr && collect == nullptr && sample == nullptr)
                     ? g->tau_shared.as<uint32_t>() : nullptr;
  if (sample) {
    L.groupmax_out = sample->groupmax;
    L.group_stride = sample->stride;
    L.group_tiles = sample->tiles;
    L.group_splits = sample->splits;
  }
  L.dump = dump;
  L.dump_ld = dump_ld;
  L.grid = P.grid * std::max(1, g->debug_grid_scale);   // > 1 only under the test hook: the extra CTAs find no unit
  L.smem_bytes = P.smem;
  L.coop_refused = &g->coop_refusals;
  L.no_coop = !g->coop_launch;
  if (g->l2_sync && dump == nullptr && sample == nullptr) {
    const int workers = P.variant == 2 ? P.grid / 2 : P.grid;
    const int max_tiles = (P.tiles_total + P.slices - 1) / P.slices + 1;
    L.sync_window = std::max(1, g->sync_window);
    L.sync_lead = std::max(1, g->sync_lead);
    L.sync_span = P.num_qt / std::max(1, workers) + 2;
    L.sync_windows = max_tiles / L.sync_window + 2;
    const size_t n = (size_t)P.slices * L.sync_span * L.sync_windows;
    RBOD_TRY(g->sync_counters.ensure(n * sizeof(int)));
    RBOD_CUDA(cudaMemsetAsync(g->sync_counters.p, 0, n * sizeof(int), st));
    L.sync_counters = g->sync_counters.as<int>();
  }
  return launch_k3(L, st);
}

// RBOD_TRACE=1: rbod_search prints the host wall-clock time between its phases (microseconds) to stderr -- where the
// part of a call that is not kernel time goes.
struct Trace {
  bool on;
  double t0, last;
  char buf[512];
  int len;
  static double now() {
    timespec ts;
    clock_gettime(CLOCK_MONOTONIC, &ts);
    return ts.tv_sec * 1e6 + ts.tv_nsec * 1e-3;
  }
  Trace() : len(0) {
    static const bool enabled = getenv("RBOD_TRACE") != nullptr && getenv("RBOD_TRACE")[0] == '1';
    on = enabled;
    t0 = last = on ? now() : 0.0;
    buf[0] = 0;
  }
  void mark(const char* what) {
    if (!on) return;
    const double t = now();
    len += snprintf(buf + len, sizeof(buf) - len, " %s=%.0f", what, t - last);
    last = t;
  }
  ~Trace() {
    if (on) fprintf(stderr, "rbod_search trace (us): total=%.0f%s\n", now() - t0, buf);
  }
};

static int ensure_lists(rbod_gallery* g, const SearchPlan& P) {
  RBOD_TRY(g->lists.ensure((size_t)P.slices * P.q_pad * P.list_stride * sizeof(uint2)));
  RBOD_TRY(g->list_cnt.ensure((size_t)P.slices * P.q_pad * sizeof(int)));
  return RBOD_OK;
}

static int prepare_queries(rbod_gallery* g, const float* queries, int64_t Q, const SearchPlan& P, cudaStream_t st,
                           const float** q_dev) {
  const void* qd = nullptr;
  RBOD_TRY(to_device(queries, (size_t)Q * g->dim * 4, g->q32, st, &qd));
  *q_dev = static_cast<const float*>(qd);
  RBOD_TRY(g->q16.ensure((size_t)P.q_pad * g->dp * 2));
  RBOD_TRY(g->q_dq.ensure((size_t)P.q_pad * 4));
  RBOD_TRY(g->q_qq.ensure((size_t)P.q_pad * 8));
  RBOD_TRY(g->tau_shared.ensure((size_t)P.q_pad * 4));
  return launch_prep_queries(*q_dev, Q, P.q_pad, g->dim, g->dp, query_kind(g), g->metric == RBOD_COSINE,
                             g->q16.as<uint16_t>(),
                             g->q_dq.as<float>(), g->q_qq.as<double>(), g->tau_shared.as<uint32_t>(), st);
}

// A call's answer, n entries each of fp32 scores, rows and fp64 keys (keys optional): the caller's arrays, and where
// the kernels write them -- the caller's array when it is device memory, else the handle's out_* workspace.
struct Answer {
  float* scores;
  int64_t* rows;
  double* keys;
  float* d_scores;
  int64_t* d_rows;
  double* d_keys;
  size_t n;
};

static int stage_answer(rbod_gallery* g, float* scores, int64_t* rows, double* keys, size_t n, Answer* a) {
  RBOD_TRY(g->out_scores.ensure(n * 4));
  RBOD_TRY(g->out_rows.ensure(n * 8));
  RBOD_TRY(g->out_scores64.ensure(n * 8));
  *a = {scores, rows, keys, is_device_ptr(scores) ? scores : g->out_scores.as<float>(),
        is_device_ptr(rows) ? rows : g->out_rows.as<int64_t>(),
        (keys && is_device_ptr(keys)) ? keys : g->out_scores64.as<double>(), n};
  return RBOD_OK;
}

// Queues the copy of a staged answer into the caller's arrays (where they are not the same).
static int copy_out(const Answer& a, cudaStream_t st) {
  RBOD_TRY(copy_out(a.scores, a.d_scores, a.n * 4, st));
  RBOD_TRY(copy_out(a.rows, a.d_rows, a.n * 8, st));
  return copy_out(a.keys, a.d_keys, a.n * 8, st);
}

// The answer of an empty gallery, written straight to the caller's arrays: every entry is "no result" -- row -1, key
// -inf, score -inf, or +inf where `metric` ranks by distance (as dist_select_kernel pads a short list).
static int answer_none(float* scores, int64_t* rows, double* keys, size_t n, int metric, cudaStream_t st) {
  std::vector<float> hs(n, (metric == RBOD_EUCLID || metric == RBOD_MANHATTAN) ? INFINITY : -INFINITY);
  std::vector<int64_t> hr(n, -1);
  std::vector<double> hd(n, -INFINITY);
  RBOD_CUDA(cudaMemcpyAsync(scores, hs.data(), n * 4, cudaMemcpyDefault, st));
  RBOD_CUDA(cudaMemcpyAsync(rows, hr.data(), n * 8, cudaMemcpyDefault, st));
  if (keys) RBOD_CUDA(cudaMemcpyAsync(keys, hd.data(), n * 8, cudaMemcpyDefault, st));
  RBOD_CUDA(cudaStreamSynchronize(st));
  return RBOD_OK;
}

// The per-item mask ids of a filtered call (n of them, in host or device memory), read to the host and checked before
// anything is launched: each must be -1 (no mask) or one of the n_masks masks; `fmt` reports the first that is not,
// from (who, its index, its value, n_masks).  `ids` stays empty without ids, and without masks (all ids are -1 then).
static int read_mask_ids(const char* who, const char* fmt, rbod_gallery* g, const int32_t* src, int64_t n,
                         int32_t n_masks, cudaStream_t st, std::vector<int>* ids) {
  if (src == nullptr || n <= 0) return RBOD_OK;
  ids->resize((size_t)n);
  if (is_device_ptr(src)) {
    if (!g) return set_error(RBOD_E_INVAL, "%s: NULL handle", who);
    RBOD_CUDA(cudaSetDevice(g->device));
    RBOD_CUDA(cudaMemcpyAsync(ids->data(), src, (size_t)n * 4, cudaMemcpyDeviceToHost, st));
    RBOD_CUDA(cudaStreamSynchronize(st));
  } else {
    memcpy(ids->data(), src, (size_t)n * 4);
  }
  for (int64_t i = 0; i < n; ++i)
    if ((*ids)[i] < -1 || (*ids)[i] >= n_masks) return set_error(RBOD_E_INVAL, fmt, who, (long long)i, (*ids)[i], n_masks);
  if (n_masks == 0) ids->clear();
  return RBOD_OK;
}

// Exact fp64 sweep (kernels K5 search, K6 recommend, K7 discover): requests are packed whole, in order, into passes of
// at most 32 slots and 32 requests.  Request r is the examples off[r] .. off[r + 1] - 1 of ex_dev ([*, dim] fp32, on
// the device) or, without offsets, the one example sel[r] (host; r when sel is null).  It answers into rows o * k of
// a's device arrays, o = sel[r] (or r), its slots carry the flags of its examples (rbod_internal.h; none when flags is
// null), and it reads the mask M.of_query_host[o] -- or mask 0 when M has masks but no ids, and then the rows mask 0
// excludes are not even loaded.  Per pass a strided sample pass gives every request its starting threshold, unless kth
// does (host, one per request, or null: a provisional k-th key, -inf if there were fewer than k candidates, a lower
// bound of the true k-th key); then the gallery is swept, and the requests whose list overflowed are tightened and
// swept again.  Nothing a request's answer depends on (its slots' accumulators, its threshold, its list, its mask) is
// shared with another request of the pass, so the packing does not change any answer.  collect: the kernel's
// launcher; metric: what the selection is given -- the gallery's for a search, which turns keys into distances, COSINE
// for K6 / K7, which emits the score as it is and pads with -inf; who: the entry point named in errors, kth_of: what a
// list overflows around in them ("key of a query", "score of a request").
static int sweep(rbod_gallery* g, const char* who, const char* kth_of, CollectLauncher collect, int metric,
                 const float* ex_dev, const int* flags, const int64_t* off, const int* sel, int64_t R, const double* kth,
                 int k, const SearchMasks& M, const Answer& a, int64_t* launches, int64_t* resweeps, cudaStream_t st) {
  // lists hold 8192 rows and so does the sample: ~k * stride rows pass the threshold it yields (1M rows, k = 10:
  // ~1200), so one sweep is enough unless k * rows / 8192 exceeds a list (then a second sweep with the tightened
  // threshold finishes it)
  const int cap = 8192, sample_cap = 8192, batch = 32, max_iter = 12;
  if (k > 1024) return set_error(RBOD_E_UNSUPPORTED, "%s: k=%d > 1024", who, k);
  RBOD_TRY(g->dist_q64.ensure((size_t)batch * g->dim * 8));
  RBOD_TRY(g->dist_thr.ensure((size_t)2 * batch * 8 + (size_t)batch * 4));   // thresholds, slot norms, row bounds
  RBOD_TRY(g->dist_ctl.ensure((size_t)(5 * batch + 1) * 4));
  RBOD_TRY(g->coll_score.ensure((size_t)batch * cap * 8));
  RBOD_TRY(g->coll_idx.ensure((size_t)batch * cap * 4));
  RBOD_TRY(g->coll_cnt.ensure((size_t)batch * 4));
  int* d_wsel = g->dist_ctl.as<int>();   // slot -> example (what the widening reads)
  int* d_slot = d_wsel + batch;           // slot table of the pass (rbod_internal.h)
  int* d_out = d_wsel + 2 * batch;        // request of the pass -> its output row
  int* d_active = d_wsel + 3 * batch;
  int* d_rmask = d_wsel + 4 * batch;      // the mask each request of the pass reads, -1 = none
  int* d_nactive = d_wsel + 5 * batch;
  const bool per_request = M.dev != nullptr && M.of_query_host != nullptr;
  double* d_thr = g->dist_thr.as<double>();
  double* d_qnorm = d_thr + batch;
  uint32_t* d_thr_row = reinterpret_cast<uint32_t*>(d_qnorm + batch);
  std::vector<double> h_thr(batch, -INFINITY);
  std::vector<int> h_ctl(5 * batch + 1);
  const int64_t sample_stride = (g->rows + sample_cap - 1) / sample_cap;   // > 1 iff more than `sample_cap` rows
  auto n_slots = [&](int64_t r) { return off ? (int)(off[r + 1] - off[r]) : 1; };
  for (int64_t r0 = 0; r0 < R;) {
    int nreq = 0, ns = 0;
    for (; r0 + nreq < R && nreq < batch && ns + n_slots(r0 + nreq) <= batch; ++nreq) ns += n_slots(r0 + nreq);
    std::fill(h_ctl.begin(), h_ctl.end(), 0);
    for (int q = 0, s = 0; q < nreq; ++q) {
      const int64_t r = r0 + q, o = sel ? sel[r] : r;
      const int64_t e0 = off ? off[r] : o, e1 = off ? off[r + 1] : o + 1;
      for (int64_t e = e0; e < e1; ++e, ++s) {
        h_ctl[s] = (int)e;
        h_ctl[batch + s] = q | (e == e1 - 1 ? SLOT_LAST : 0) | (flags ? flags[e] : 0);
      }
      h_ctl[2 * batch + q] = (int)o;
      h_ctl[3 * batch + q] = 1;
      h_ctl[4 * batch + q] = per_request ? M.of_query_host[o] : -1;
      // kth was summed in another order than this sweep sums, so the very row that set it may come out an ulp lower
      // here: seed a margin far above fp64 summation noise below it (-inf stays -inf)
      if (kth) h_thr[q] = kth[r] - 1e-12 * std::max(1.0, std::fabs(kth[r]));
    }
    RBOD_CUDA(cudaMemcpyAsync(d_wsel, h_ctl.data(), h_ctl.size() * 4, cudaMemcpyHostToDevice, st));
    RBOD_CUDA(cudaMemcpyAsync(d_thr, h_thr.data(), (size_t)batch * 8, cudaMemcpyHostToDevice, st));
    RBOD_CUDA(cudaMemsetAsync(d_thr_row, 0xff, (size_t)batch * 4, st));   // no row bound: every tie with the threshold counts
    RBOD_CUDA(cudaMemsetAsync(g->coll_cnt.p, 0, (size_t)batch * 4, st));
    if (ns < batch) RBOD_CUDA(cudaMemsetAsync(g->dist_q64.p, 0, (size_t)batch * g->dim * 8, st));   // zero rows pad the pass
    RBOD_TRY(launch_dist_widen_queries(ex_dev, d_wsel, ns, g->dim, g->dist_q64.as<double>(), d_qnorm, st));
    ++*launches;
    // one collecting pass over the rows 0, stride, 2 stride, ... and the selection of its lists
    auto collect_select = [&](int64_t stride, int sample) {
      RBOD_TRY(collect(g->metric, g->dist_q64.as<double>(), g->master32, g->rows16, g->kind16, g->dim, g->dim, g->dp,
                       g->rows, 0, stride, M.dev, M.words, d_slot, per_request ? d_rmask : nullptr, d_thr, d_thr_row,
                       d_active, d_qnorm, ns, nreq, cap, g->coll_score.as<double>(), g->coll_idx.as<uint32_t>(),
                       g->coll_cnt.as<int>(), g->num_sms, st));
      RBOD_TRY(launch_dist_select(g->coll_score.as<double>(), g->coll_idx.as<uint32_t>(), g->coll_cnt.as<int>(), d_out,
                                  nreq, cap, k, sample, metric, d_thr, d_thr_row, d_active, d_nactive, a.d_scores,
                                  a.d_rows, a.d_keys, st));
      *launches += 2;
      return RBOD_OK;
    };
    if (!kth && sample_stride > 1) RBOD_TRY(collect_select(sample_stride, 1));
    int iter = 0, left = nreq;
    for (; iter < max_iter && left > 0; ++iter) {
      RBOD_CUDA(cudaMemsetAsync(d_nactive, 0, 4, st));
      RBOD_TRY(collect_select(1, 0));
      RBOD_CUDA(cudaMemcpyAsync(&left, d_nactive, 4, cudaMemcpyDeviceToHost, st));
      RBOD_CUDA(cudaStreamSynchronize(st));
      if (iter > 0) ++*resweeps;
    }
    if (left > 0)
      return set_error(RBOD_E_OVERFLOW, "%s: more than %d rows tie around the k-th %s", who, cap, kth_of);
    r0 += nreq;
  }
  return RBOD_OK;
}

// The exact sweep's front end, past the entry point's argument checks: rbod_search / rbod_search_masks (what the
// tensor-core pass does not cover), rbod_recommend and rbod_discover.  The answer of an empty gallery, or: the outputs
// staged, the masks and the examples uploaded, the sweep, the copy-out and the stats.  ids: the checked host mask ids,
// one per request, or null (every request reads mask 0, if there are masks).
static int sweep_search(rbod_gallery* g, const char* who, const char* kth_of, CollectLauncher collect, int metric,
                        const float* examples,
                        int64_t n_examples, const int* flags, const int64_t* off, int64_t R, int k,
                        const uint32_t* row_masks, int32_t n_masks, const int* ids, float* out_scores,
                        int64_t* out_rows, double* out_keys, rbod_search_stats* stats, cudaStream_t st) {
  Answer a;
  RBOD_TRY(stage_answer(g, out_scores, out_rows, out_keys, (size_t)R * k, &a));
  if (g->rows == 0) return answer_none(out_scores, out_rows, out_keys, a.n, metric, st);
  SearchMasks M = {nullptr, (g->rows + 31) / 32, nullptr, ids};
  const void* md = nullptr;
  if (n_masks > 0) RBOD_TRY(to_device(row_masks, (size_t)n_masks * M.words * 4, g->mask_dev, st, &md));
  M.dev = static_cast<const uint32_t*>(md);
  const void* xd = nullptr;
  RBOD_TRY(to_device(examples, (size_t)n_examples * g->dim * 4, g->q32, st, &xd));
  int64_t launches = 0, resweeps = 0;
  RBOD_TRY(sweep(g, who, kth_of, collect, metric, static_cast<const float*>(xd), flags, off, nullptr, R, nullptr, k, M,
                 a, &launches, &resweeps, st));
  RBOD_TRY(copy_out(a, st));
  RBOD_CUDA(cudaStreamSynchronize(st));
  if (stats) {
    stats->queries = R;
    stats->total_launches = launches;
    stats->sweep_queries = R;        // every query or request is answered by the fp64 sweep
    stats->fallback_queries = resweeps;
  }
  return RBOD_OK;
}

// bf16 COSINE collections: a bf16 query sits up to 2e-3 from the exact unit query, more than the gap between the
// k-th and the (k + slack)-th score once k reaches the high tens (10M rows, k = 100: 17-37 % of the queries were
// not certified and took the collecting second pass).  An fp16 copy of the stored rows as the search operand brings
// the margin to 4e-4 -- bf16 -> fp16 is exact for values of magnitude >= 2^-14 -- at the price of 2 more bytes per
// element, so it is built the first time such a search arrives (one HBM-bound pass) and kept up to date by K1.
static int maybe_build_shadow(rbod_gallery* g, int k, cudaStream_t st) {
  if (g->dtype == RBOD_BF16 && g->metric == RBOD_COSINE && !g->use_shadow && g->auto_shadow && k > 40 && g->rows > 0) {
    uint16_t* nsh = nullptr;
    if (cudaMalloc(&nsh, (size_t)g->capacity * g->dp * 2) == cudaSuccess) {
      RBOD_CUDA(cudaMemsetAsync(nsh, 0, (size_t)g->capacity * g->dp * 2, st));
      RBOD_CUDA(cudaMemsetAsync(g->stats + 2, 0, 2 * sizeof(float), st));
      RBOD_TRY(launch_build_shadow(g->rows16, g->rows, g->dp, nsh, g->stats, st));
      g->shadow16 = nsh;
      g->use_shadow = 1;
    } else {
      cudaGetLastError();
      g->auto_shadow = 0;   // no room for it: searches stay on the bf16 operand (still exact, more second passes)
    }
  }
  return RBOD_OK;
}

// Threshold pre-pass: row maxima over K3_SAMPLE_GROUPS strided samples of the gallery give every query a
// starting threshold, so the candidate lists of the main pass skip their cold start (see tau_init_kernel).
// Each group's comb is split over enough units to fill the chip, so a small batch does not stream the sample on
// eight SMs (Q <= 128 on 12.5M x 768: 0.48 ms before the split, next to a 2.9 ms main pass).  Batches of at most
// 8 queries skip it: their epilogue has almost nothing to insert (measured: Q = 1 is 0.47 ms faster without,
// Q = 16 already 0.17 ms slower).  presample = 2 forces it.
static bool presample_pays(const rbod_gallery* g, const SearchPlan& P, int64_t Q, int* sample_tiles) {
  *sample_tiles = std::max(1, P.tiles_total / (K3_SAMPLE_RATIO * P.kc));
  const bool sample_pays = g->presample >= 2 || Q > 8;
  return g->tau_share && g->presample && sample_pays && P.tiles_total >= 10 * P.kc &&
         P.tiles_total / *sample_tiles >= K3_SAMPLE_GROUPS;
}

// Everything of a search up to and including the main K3 launch: flags cleared, queries prepared, the optional
// threshold pre-pass, the candidate lists filled.
static int launch_front(rbod_gallery* g, const float* queries, int64_t Q, const SearchPlan& P, const SearchMasks& M,
                        bool use_sample, int sample_tiles, cudaStream_t st, const float** q_dev_out,
                        const float** tau_init_out, int64_t* launches_io, Trace& tr) {
  int64_t launches = *launches_io;
  const float* q_dev = nullptr;
  RBOD_CUDA(cudaMemsetAsync(g->flags.p, 0, 64, st));
  tr.mark("setup");
  RBOD_TRY(prepare_queries(g, queries, Q, P, st, &q_dev));
  ++launches;
  tr.mark("prep");
  if (g->time_k3) RBOD_CUDA(cudaEventRecord(g->ev0, st));
  const float* tau_init = nullptr;
  if (use_sample) {
    SearchPlan PA = P;
    const int workers = P.variant == 2 ? std::max(1, g->num_sms / 2) : g->num_sms;
    const int splits = std::max(1, std::min({16, sample_tiles, workers / (K3_SAMPLE_GROUPS * std::max(1, PA.num_qt))}));
    PA.slices = K3_SAMPLE_GROUPS * splits;
    PA.grid = (int)std::min<int64_t>((int64_t)PA.slices * PA.num_qt, workers) * (P.variant == 2 ? 2 : 1);
    RBOD_TRY(g->groupmax.ensure((size_t)PA.slices * P.q_pad * 4));
    RBOD_TRY(g->tau_init.ensure((size_t)P.q_pad * 4));
    K3Sample S;
    S.groupmax = g->groupmax.as<float>();
    S.tiles = sample_tiles;
    S.stride = P.tiles_total / sample_tiles;
    S.splits = splits;
    RBOD_TRY(run_k3(g, PA, Q, g->q16.as<uint16_t>(), M, nullptr, nullptr, 0, st, &S));
    RBOD_TRY(launch_tau_init(g->groupmax.as<float>(), K3_SAMPLE_GROUPS, splits, P.q_pad,
                             g->tau_shared.as<uint32_t>(), g->tau_init.as<float>(), st));
    tau_init = g->tau_init.as<float>();
    launches += 2;
  }
  RBOD_TRY(run_k3(g, P, Q, g->q16.as<uint16_t>(), M, nullptr, nullptr, 0, st));
  if (g->time_k3) RBOD_CUDA(cudaEventRecord(g->ev1, st));
  ++launches;
  tr.mark("k3_launches");
  *q_dev_out = q_dev;
  *tau_init_out = tau_init;
  *launches_io = launches;
  return RBOD_OK;
}

static void fill_finish(rbod_gallery* g, const SearchPlan& P, int k, const float* tau_init, const float* q_dev,
                        float* d_scores, int64_t* d_rows, double* d_scores64, FinishArgs* Fp) {
  FinishArgs& F = *Fp;
  int* d_flags = g->flags.as<int>();
  memset(&F, 0, sizeof(F));
  F.lists = g->lists.as<uint2>();
  F.list_cnt = g->list_cnt.as<int>();
  F.slices = P.slices;
  F.list_stride = P.list_stride;
  F.n_cap = P.n_cap;
  F.kc = P.kc;
  F.k = k;
  F.q_pad = P.q_pad;
  F.tau_init = tau_init;
  F.q = q_dev;
  F.q_qq = g->q_qq.as<double>();
  F.q_dq = g->q_dq.as<float>();
  F.stats = g->stats;
  F.master32 = g->master32;
  F.rows16 = g->rows16;
  F.kind16 = g->kind16;
  F.dim = g->dim;
  F.metric = g->metric;
  F.master16 = g->dtype != RBOD_F32;
  F.shadow = g->use_shadow;
  F.dp = g->dp;
  F.ld32 = g->dim;
  F.ld16 = g->dp;
  F.out_scores = d_scores;
  F.out_rows = d_rows;
  F.out_scores64 = d_scores64;
  F.n_flag = d_flags;
  F.flag_q = g->flag_q.as<int>();
  F.flag_thr = g->flag_thr.as<double>();
  F.flag_lo = g->flag_lo.as<float>();
  F.max_eps = reinterpret_cast<float*>(d_flags + 3);
}

// rbod_search and rbod_search_masks: a search with one shared mask is the case "every query reads mask 0".
static int search_impl(rbod_gallery* g, const float* queries, int64_t Q, int32_t k, const uint32_t* row_masks,
                       int32_t n_masks, const int32_t* mask_of_query, float* out_scores, int64_t* out_rows,
                       double* out_scores64, rbod_search_stats* stats, void* stream) {
  if (!g) return set_error(RBOD_E_INVAL, "rbod_search: NULL handle");
  if (Q < 0 || k < 1 || (Q > 0 && (!queries || !out_scores || !out_rows)))
    return set_error(RBOD_E_INVAL, "rbod_search: bad arguments");
  if (n_masks < 0 || (n_masks > 0 && !row_masks))
    return set_error(RBOD_E_INVAL, "rbod_search_masks: %d masks, row_masks %s", n_masks, row_masks ? "set" : "NULL");
  if (stats) memset(stats, 0, sizeof(*stats));
  g->pending.valid = 0;   // a full search reuses the query buffers a pending rbod_search_begin left behind
  if (Q == 0) return RBOD_OK;
  // What the tensor-core pass does not cover takes the exact fp64 sweep (K5): MANHATTAN (not a contraction), vectors
  // wider than K3_MAX_DP_WIDE columns, and k beyond the K3 candidate lists.  Everything else -- COSINE, DOT and EUCLID
  // (row-bias epilogue) up to 2048 columns, k <= 128 -- runs on the tensor cores.
  const bool distance_metric = g->metric == RBOD_MANHATTAN || g->dp > K3_MAX_DP_WIDE || k > K3_MAX_KC;
  if (Q > (1ll << 24)) return set_error(RBOD_E_INVAL, "rbod_search: Q too large");
  if (g->rows >= 0xffffffffll) return set_error(RBOD_E_UNSUPPORTED, "rbod_search: more than 2^32-2 rows per shard");
  RBOD_CUDA(cudaSetDevice(g->device));
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  std::vector<int> ids_h;
  RBOD_TRY(read_mask_ids("rbod_search_masks", "%s: mask_of_query[%lld] = %d is outside [-1, %d)", g, mask_of_query, Q,
                         n_masks, st, &ids_h));
  const int* ids = ids_h.empty() ? nullptr : ids_h.data();

  if (distance_metric)
    return sweep_search(g, "rbod_search", "key of a query", launch_key_collect, g->metric, queries, Q, nullptr, nullptr,
                        Q, k, row_masks, n_masks, ids, out_scores, out_rows, out_scores64, stats, st);

  const int smem_optin = k3_configure(g->device);
  if (smem_optin < 0) return smem_optin;

  RBOD_TRY(maybe_build_shadow(g, k, st));

  Answer a;
  RBOD_TRY(stage_answer(g, out_scores, out_rows, out_scores64, (size_t)Q * k, &a));

  Trace tr;
  SearchPlan P;
  RBOD_TRY(plan_search(g, Q, k, search_variant(g, Q), smem_optin, &P));
  tr.mark("plan");
  if (stats) {
    stats->queries = Q;
    stats->candidates = P.kc;
    stats->slices = P.slices;
  }

  RBOD_TRY(g->flags.ensure(64));
  int* d_flags = g->flags.as<int>();
  int64_t launches = 0;

  if (g->rows == 0) return answer_none(out_scores, out_rows, out_scores64, a.n, g->metric, st);

  SearchMasks M = {nullptr, (g->rows + 31) / 32, nullptr, ids};
  const void* mask_dev = nullptr;
  if (n_masks > 0) RBOD_TRY(to_device(row_masks, (size_t)n_masks * M.words * 4, g->mask_dev, st, &mask_dev));
  M.dev = static_cast<const uint32_t*>(mask_dev);
  std::vector<int> ids_pad;
  if (ids != nullptr) {
    // the K3 launches read one id per query row of the padded tile: pad rows read no mask
    ids_pad.assign(ids, ids + Q);
    ids_pad.resize((size_t)P.q_pad, -1);
    RBOD_TRY(g->mask_ids.ensure((size_t)P.q_pad * 4));
    RBOD_CUDA(cudaMemcpyAsync(g->mask_ids.p, ids_pad.data(), (size_t)P.q_pad * 4, cudaMemcpyHostToDevice, st));
    M.of_query = g->mask_ids.as<int>();
  }

  RBOD_TRY(ensure_lists(g, P));
  RBOD_TRY(g->flag_q.ensure((size_t)Q * 4));
  RBOD_TRY(g->flag_thr.ensure((size_t)Q * 8));
  RBOD_TRY(g->flag_lo.ensure((size_t)P.q_pad * 4 + 1024));   // read as [q_pad of the second pass]

  int sample_tiles = 1;
  bool use_sample = presample_pays(g, P, Q, &sample_tiles);
  int hflags[8] = {0, 0, 0, 0, 0, 0, 0, 0};
  const float* q_dev = nullptr;
  int64_t retries = 0;
  for (int attempt = 0;; ++attempt) {
    const float* tau_init = nullptr;
    RBOD_TRY(launch_front(g, queries, Q, P, M, use_sample, sample_tiles, st, &q_dev, &tau_init, &launches, tr));
    FinishArgs F;
    fill_finish(g, P, k, tau_init, q_dev, a.d_scores, a.d_rows, a.d_keys, &F);
    RBOD_TRY(launch_finish(F, Q, st));
    ++launches;
    tr.mark("finish_launch");

    // The answer and the certification flags travel together: in the common case (every query certified) this is
    // the only synchronisation of the call.
    RBOD_TRY(copy_out(a, st));
    RBOD_CUDA(cudaMemcpyAsync(hflags, d_flags, sizeof(hflags), cudaMemcpyDeviceToHost, st));
    tr.mark("copies");
    RBOD_CUDA(cudaStreamSynchronize(st));
    tr.mark("sync");
    if (hflags[4] > 0 && tau_init != nullptr && attempt == 0) {
      // a starting threshold cut below k candidates for some query: once more without the pre-pass
      retries = hflags[4];
      use_sample = false;
      continue;
    }
    break;
  }
  const int n_flag = hflags[0];
  float max_eps;
  memcpy(&max_eps, &hflags[3], 4);

  int n_sweep = n_flag;   // queries that still need the exact fp64 sweep
  int64_t k3_launches = 1;
  const int cap = K3_COLLECT_CAP;
  std::vector<int> cnt_h(n_flag), fq_h(n_flag);
  std::vector<double> thr_h(n_flag);
  if (n_flag > 0 && g->collect_pass) {
    // Second tensor-core pass over the uncertified queries only: record every row whose approximate
    // score can still reach the query's provisional k-th exact score, rescore those exactly, select.
    SearchPlan P2;
    RBOD_TRY(plan_search(g, n_flag, k, search_variant(g, n_flag), smem_optin, &P2));
    RBOD_TRY(g->fq16.ensure((size_t)P2.q_pad * g->dp * 2));
    RBOD_TRY(g->coll_cnt.ensure((size_t)P2.q_pad * 4));
    RBOD_TRY(g->coll_idx.ensure((size_t)P2.q_pad * cap * 4));
    RBOD_TRY(g->coll_score.ensure((size_t)n_flag * cap * 8));
    SearchMasks M2 = M;   // the gathered query rows keep their queries' masks
    if (M.of_query != nullptr) {
      RBOD_TRY(g->fmask_ids.ensure((size_t)P2.q_pad * 4));
      M2.of_query = g->fmask_ids.as<int>();
    }
    RBOD_TRY(launch_gather_flagged(g->q16.as<uint16_t>(), g->dp, g->flag_q.as<int>(), 0, n_flag, P2.q_pad,
                                   g->fq16.as<uint16_t>(), g->coll_cnt.as<int>(), M.of_query, g->fmask_ids.as<int>(),
                                   st));
    K3Collect C;
    C.thr = g->flag_lo.as<float>();
    C.idx = g->coll_idx.as<uint32_t>();
    C.cnt = g->coll_cnt.as<int>();
    C.cap = cap;
    RBOD_TRY(run_k3(g, P2, n_flag, g->fq16.as<uint16_t>(), M2, &C, nullptr, 0, st));
    RBOD_TRY(launch_rescore_collected(q_dev, g->q_qq.as<double>(), g->master32, g->rows16, g->kind16, g->dim, g->dim,
                                      g->dp, g->metric, g->flag_q.as<int>(), 0, n_flag, cap, g->coll_idx.as<uint32_t>(),
                                      g->coll_cnt.as<int>(), g->coll_score.as<double>(), st));
    RBOD_TRY(launch_select_collected(g->coll_score.as<double>(), g->coll_idx.as<uint32_t>(), g->coll_cnt.as<int>(),
                                     g->flag_q.as<int>(), 0, n_flag, cap, k, g->metric, a.d_scores, a.d_rows,
                                     a.d_keys, st));
    launches += 4;
    ++k3_launches;
    RBOD_CUDA(cudaMemcpyAsync(cnt_h.data(), g->coll_cnt.p, (size_t)n_flag * 4, cudaMemcpyDeviceToHost, st));
  }
  if (n_flag > 0) {
    RBOD_CUDA(cudaMemcpyAsync(fq_h.data(), g->flag_q.p, (size_t)n_flag * 4, cudaMemcpyDeviceToHost, st));
    RBOD_CUDA(cudaMemcpyAsync(thr_h.data(), g->flag_thr.p, (size_t)n_flag * 8, cudaMemcpyDeviceToHost, st));
    RBOD_CUDA(cudaStreamSynchronize(st));
    if (g->collect_pass) {
      // queries whose list overflowed (a tie cluster wider than `cap`) keep going to the exact sweep
      n_sweep = 0;
      for (int f = 0; f < n_flag; ++f)
        if (cnt_h[f] > cap) {
          fq_h[n_sweep] = fq_h[f];
          thr_h[n_sweep] = thr_h[f];
          ++n_sweep;
        }
    }
    if (n_sweep > 0) {
      int64_t resweeps = 0;   // not reported: fallback_queries counts the uncertified queries here
      RBOD_TRY(sweep(g, "rbod_search", "key of a query", launch_key_collect, g->metric, q_dev, nullptr, nullptr,
                     fq_h.data(), n_sweep, thr_h.data(), k, M, a, &launches, &resweeps, st));
    }
    // the second pass rewrote the flagged queries' rows of the answer
    RBOD_TRY(copy_out(a, st));
    RBOD_CUDA(cudaStreamSynchronize(st));
  }

  if (stats) {
    stats->fallback_queries = n_flag;
    stats->k3_launches = k3_launches;
    stats->sweep_queries = n_sweep;
    stats->total_launches = launches;
    stats->max_eps = max_eps;
    stats->presample_retries = retries;
    if (g->time_k3) {
      float ms = 0.f;
      RBOD_CUDA(cudaEventElapsedTime(&ms, g->ev0, g->ev1));
      stats->k3_ms = ms;
    }
  }
  return RBOD_OK;
}

int rbod_search(rbod_gallery* g, const float* queries, int64_t Q, int32_t k, const uint32_t* row_mask,
                float* out_scores, int64_t* out_rows, double* out_scores64, rbod_search_stats* stats,
                void* stream) {
  return search_impl(g, queries, Q, k, row_mask, row_mask ? 1 : 0, nullptr, out_scores, out_rows, out_scores64, stats,
                     stream);
}

int rbod_search_masks(rbod_gallery* g, const float* queries, int64_t Q, int32_t k, const uint32_t* row_masks,
                      int32_t n_masks, const int32_t* mask_of_query, float* out_scores, int64_t* out_rows,
                      double* out_scores64, rbod_search_stats* stats, void* stream) {
  return search_impl(g, queries, Q, k, row_masks, n_masks, mask_of_query, out_scores, out_rows, out_scores64, stats,
                     stream);
}

// Maximal marginal relevance: the exact top-`candidates` of every query (search_impl, unchanged, into the handle's K8
// workspaces), then K8's greedy selection of `limit` of them, then the copy-out.
int rbod_search_mmr(rbod_gallery* g, const float* queries, int64_t Q, int32_t limit, int32_t candidates,
                    const double* diversity, const float* score_threshold, const uint32_t* row_masks, int32_t n_masks,
                    const int32_t* mask_of_query, float* out_scores, int64_t* out_rows, double* out_keys,
                    rbod_search_stats* stats, void* stream) {
  const char* who = "rbod_search_mmr";
  if (Q < 0 || Q > (1ll << 24)) return set_error(RBOD_E_INVAL, "%s: Q = %lld out of range", who, (long long)Q);
  if (limit < 1) return set_error(RBOD_E_INVAL, "%s: limit = %d < 1", who, limit);
  if (candidates < limit)
    return set_error(RBOD_E_INVAL, "%s: candidates = %d < limit = %d", who, candidates, limit);
  if (n_masks < 0 || (n_masks > 0 && !row_masks))
    return set_error(RBOD_E_INVAL, "%s: %d masks, row_masks %s", who, n_masks, row_masks ? "set" : "NULL");
  if (Q > 0 && !diversity) return set_error(RBOD_E_INVAL, "%s: diversity is NULL", who);
  if (Q > 0 && (!queries || !out_scores || !out_rows)) return set_error(RBOD_E_INVAL, "%s: NULL queries or outputs", who);
  for (int64_t q = 0; q < Q; ++q)
    if (!(diversity[q] >= 0.0 && diversity[q] <= 1.0))
      return set_error(RBOD_E_INVAL, "%s: query %lld: diversity %g is not in [0, 1]", who, (long long)q, diversity[q]);
  // mask ids are checked here, on the host, and handed to the search as a host array
  std::vector<int> ids;
  RBOD_TRY(read_mask_ids(who, "%s: query %lld: mask_of_query = %d is outside [-1, %d)", g, mask_of_query, Q, n_masks,
                         static_cast<cudaStream_t>(stream), &ids));
  if (candidates > MMR_MAX_CANDIDATES)
    return set_error(RBOD_E_UNSUPPORTED, "%s: candidates = %d > %d", who, candidates, MMR_MAX_CANDIDATES);
  if (!g) return set_error(RBOD_E_INVAL, "%s: NULL handle", who);
  if (stats) memset(stats, 0, sizeof(*stats));
  if (Q == 0) return RBOD_OK;
  RBOD_CUDA(cudaSetDevice(g->device));
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  if (g->rows == 0) {
    if (stats) stats->queries = Q;
    return answer_none(out_scores, out_rows, out_keys, (size_t)Q * limit, g->metric, st);
  }

  // 1. the candidates: an ordinary search with k = candidates, written straight into the K8 workspaces
  const size_t n_cand = (size_t)Q * candidates;
  RBOD_TRY(g->mmr_scores.ensure(n_cand * 4));
  RBOD_TRY(g->mmr_rows.ensure(n_cand * 8));
  RBOD_TRY(g->mmr_keys.ensure(n_cand * 8));
  RBOD_TRY(search_impl(g, queries, Q, candidates, row_masks, n_masks, ids.empty() ? nullptr : ids.data(),
                       g->mmr_scores.as<float>(), g->mmr_rows.as<int64_t>(), g->mmr_keys.as<double>(), stats, stream));

  // 2. K8
  std::vector<double> ctl_d(diversity, diversity + Q);
  std::vector<float> ctl_t;
  if (score_threshold) ctl_t.assign(score_threshold, score_threshold + Q);
  RBOD_TRY(g->mmr_ctl.ensure((size_t)Q * 12));
  RBOD_CUDA(cudaMemcpyAsync(g->mmr_ctl.p, ctl_d.data(), (size_t)Q * 8, cudaMemcpyHostToDevice, st));
  if (score_threshold)
    RBOD_CUDA(cudaMemcpyAsync(g->mmr_ctl.as<double>() + Q, ctl_t.data(), (size_t)Q * 4, cudaMemcpyHostToDevice, st));
  Answer a;
  RBOD_TRY(stage_answer(g, out_scores, out_rows, out_keys, (size_t)Q * limit, &a));
  MmrArgs A;
  A.Q = Q;
  A.L = candidates;
  A.limit = limit;
  A.cand_rows = g->mmr_rows.as<int64_t>();
  A.cand_scores = g->mmr_scores.as<float>();
  A.cand_keys = g->mmr_keys.as<double>();
  A.diversity = g->mmr_ctl.as<double>();
  A.score_threshold = score_threshold ? reinterpret_cast<const float*>(g->mmr_ctl.as<double>() + Q) : nullptr;
  A.master32 = g->master32;
  A.rows16 = g->rows16;
  A.kind16 = g->kind16;
  A.dim = g->dim;
  A.ld32 = g->dim;
  A.ld16 = g->dp;
  A.q64_scratch = nullptr;
  if (g->dim > MMR_SMEM_DIM) {
    RBOD_TRY(g->mmr_q64.ensure((size_t)mmr_grid(Q, g->dim, g->num_sms) * g->dim * 8));
    A.q64_scratch = g->mmr_q64.as<double>();
  }
  A.out_scores = a.d_scores;
  A.out_rows = a.d_rows;
  A.out_keys = a.d_keys;
  RBOD_TRY(launch_mmr_select(g->metric, A, g->num_sms, st));

  // 3. copy-out
  RBOD_TRY(copy_out(a, st));
  RBOD_CUDA(cudaStreamSynchronize(st));
  if (stats) stats->total_launches += 1;
  return RBOD_OK;
}

// Checks common to rbod_recommend and rbod_discover, made on the host before anything touches a device, in the order
// they are reported: counts, masks, NULL pointers, offsets (request sizes 1 to 32).  `what` names the per-example array.
static int check_example_args(const char* who, const char* what, const float* examples, int64_t n_examples,
                              const void* per_example, const int64_t* off, int64_t R, int k,
                              const uint32_t* row_masks, int32_t n_masks, const float* out_scores,
                              const int64_t* out_rows) {
  if (R < 0 || R > (1ll << 24)) return set_error(RBOD_E_INVAL, "%s: R = %lld out of range", who, (long long)R);
  if (k < 1) return set_error(RBOD_E_INVAL, "%s: k = %d < 1", who, k);
  if (n_examples < 0) return set_error(RBOD_E_INVAL, "%s: n_examples = %lld", who, (long long)n_examples);
  if (n_masks < 0 || (n_masks > 0 && !row_masks))
    return set_error(RBOD_E_INVAL, "%s: %d masks, row_masks %s", who, n_masks, row_masks ? "set" : "NULL");
  if (R > 0 && (!examples || !per_example || !off || !out_scores || !out_rows))
    return set_error(RBOD_E_INVAL, "%s: NULL examples, %s, offsets or outputs", who, what);
  if (off) {
    if (off[0] != 0 || off[R] != n_examples)
      return set_error(RBOD_E_INVAL, "%s: request_offsets must run from 0 to n_examples = %lld", who,
                       (long long)n_examples);
    for (int64_t r = 0; r < R; ++r) {
      const int64_t n = off[r + 1] - off[r];
      if (n < 1 || n > 32)
        return set_error(RBOD_E_INVAL, "%s: request %lld has %lld examples, not 1 to 32 (offsets monotone)", who,
                         (long long)r, (long long)n);
    }
  }
  return RBOD_OK;
}

// The rest of rbod_recommend / rbod_discover once the requests themselves are checked: the host mask ids, k, the
// handle, then the sweep's front end with `collect` over the examples whose slot-table flags are `flags` [n_examples].
static int example_search(const char* who, CollectLauncher collect, rbod_gallery* g, const float* examples,
                          int64_t n_examples, const int* flags, const int64_t* request_offsets, int64_t R, int32_t k,
                          const uint32_t* row_masks, int32_t n_masks, const int32_t* mask_of_request,
                          float* out_scores, int64_t* out_rows, double* out_keys, rbod_search_stats* stats,
                          void* stream) {
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const char* bad_id = "%s: mask_of_request[%lld] = %d is outside [-1, %d)";
  // ids in host memory are checked before the handle is; ids in device memory are read once the device is set, and
  // only when there are masks to read
  const bool ids_dev = is_device_ptr(mask_of_request);
  std::vector<int> ids;
  if (!ids_dev) RBOD_TRY(read_mask_ids(who, bad_id, g, mask_of_request, R, n_masks, st, &ids));
  if (k > 1024) return set_error(RBOD_E_UNSUPPORTED, "%s: k=%d > 1024", who, k);
  if (!g) return set_error(RBOD_E_INVAL, "%s: NULL handle", who);
  if (stats) {
    memset(stats, 0, sizeof(*stats));
    stats->queries = R;   // what an empty gallery reports too
  }
  if (R == 0) return RBOD_OK;
  if (g->rows >= 0xffffffffll) return set_error(RBOD_E_UNSUPPORTED, "%s: more than 2^32-2 rows per shard", who);
  RBOD_CUDA(cudaSetDevice(g->device));
  if (ids_dev && n_masks > 0) RBOD_TRY(read_mask_ids(who, bad_id, g, mask_of_request, R, n_masks, st, &ids));
  // K is larger-is-better: the selection takes it as a COSINE key, emitted as it is and padded with -inf
  return sweep_search(g, who, "score of a request", collect, RBOD_COSINE, examples, n_examples, flags, request_offsets,
                      R, k, row_masks, n_masks, ids.empty() ? nullptr : ids.data(), out_scores, out_rows, out_keys, stats,
                      st);
}

int rbod_recommend(rbod_gallery* g, const float* examples, int64_t n_examples, const int8_t* example_sign,
                   const int64_t* request_offsets, int64_t R, int32_t k, const uint32_t* row_masks, int32_t n_masks,
                   const int32_t* mask_of_request, float* out_scores, int64_t* out_rows, double* out_keys,
                   rbod_search_stats* stats, void* stream) {
  RBOD_TRY(check_example_args("rbod_recommend", "signs", examples, n_examples, example_sign, request_offsets, R, k,
                              row_masks, n_masks, out_scores, out_rows));
  const int64_t E = R > 0 ? n_examples : 0;
  std::vector<int> flags(E);
  for (int64_t e = 0; e < E; ++e) {
    if (example_sign[e] != 1 && example_sign[e] != -1)
      return set_error(RBOD_E_INVAL, "rbod_recommend: example_sign[%lld] = %d is not +1 or -1", (long long)e,
                       (int)example_sign[e]);
    flags[e] = example_sign[e] < 0 ? SLOT_NEG : 0;
  }
  return example_search("rbod_recommend", launch_reco_collect, g, examples, n_examples, flags.data(), request_offsets,
                        R, k, row_masks, n_masks, mask_of_request, out_scores, out_rows, out_keys, stats, stream);
}

int rbod_discover(rbod_gallery* g, const float* examples, int64_t n_examples, const int8_t* example_role,
                  const int64_t* request_offsets, int64_t R, int32_t k, const uint32_t* row_masks, int32_t n_masks,
                  const int32_t* mask_of_request, float* out_scores, int64_t* out_rows, double* out_keys,
                  rbod_search_stats* stats, void* stream) {
  RBOD_TRY(check_example_args("rbod_discover", "roles", examples, n_examples, example_role, request_offsets, R, k,
                              row_masks, n_masks, out_scores, out_rows));
  const int64_t E = R > 0 ? n_examples : 0;
  for (int64_t e = 0; e < E; ++e)
    if (example_role[e] < -1 || example_role[e] > 1)
      return set_error(RBOD_E_INVAL, "rbod_discover: example_role[%lld] = %d is not 0, +1 or -1", (long long)e,
                       (int)example_role[e]);
  // an optional target first, then (+1, -1) pairs; a request with a target is a discovery, without one a context search
  std::vector<int> flags(E);
  for (int64_t r = 0; r < R; ++r) {
    const int64_t e0 = request_offsets[r], e1 = request_offsets[r + 1];
    const int disc = example_role[e0] == 0 ? SLOT_DISC : 0;
    for (int64_t e = e0; e < e1; ++e) {
      const int role = example_role[e];
      if (role == 0 && e != e0)
        return set_error(RBOD_E_INVAL, "rbod_discover: request %lld: %s target at example %lld (a target comes first)",
                         (long long)r, disc ? "a second" : "a", (long long)e);
      if (role == 1 && (e + 1 == e1 || example_role[e + 1] != -1))
        return set_error(RBOD_E_INVAL, "rbod_discover: request %lld: positive example %lld is not followed by a negative",
                         (long long)r, (long long)e);
      if (role == -1 && (e == e0 || example_role[e - 1] != 1))
        return set_error(RBOD_E_INVAL, "rbod_discover: request %lld: negative example %lld is not preceded by a positive",
                         (long long)r, (long long)e);
      flags[e] = disc | (role == 0 ? SLOT_TARGET : role < 0 ? SLOT_NEG : 0);
    }
  }
  return example_search("rbod_discover", launch_disc_collect, g, examples, n_examples, flags.data(), request_offsets,
                        R, k, row_masks, n_masks, mask_of_request, out_scores, out_rows, out_keys, stats, stream);
}

// ---- split search: the two halves of rbod_search around an exchange between shards ---------------------------
// begin: query prep, threshold pre-pass, K3, selection of the kc best approximate candidates per query; publishes
// the approx_m best approximate scores and the error bound.  end: exact scores for the candidates that can still
// reach the GLOBAL top k (cut = the k-th best approximate score over all shards), local ranking, and an upper bound
// on everything the shard never listed, which rbod_merge_topk_certified checks against the merged k-th score.
int rbod_search_begin(rbod_gallery* g, const float* queries, int64_t Q, int32_t k, int32_t approx_m,
                      const uint32_t* row_mask, float* out_approx, rbod_search_stats* stats, void* stream) {
  if (!g) return set_error(RBOD_E_INVAL, "rbod_search_begin: NULL handle");
  g->pending.valid = 0;
  if (Q < 1 || k < 1 || !queries || !out_approx || approx_m < 1 || approx_m > k)
    return set_error(RBOD_E_INVAL, "rbod_search_begin: bad arguments");
  if (!is_device_ptr(out_approx)) return set_error(RBOD_E_INVAL, "rbod_search_begin: out_approx must be device memory");
  if (stats) memset(stats, 0, sizeof(*stats));
  if (g->metric == RBOD_MANHATTAN || g->dp > K3_MAX_DP_WIDE || k > K3_MAX_KC)
    return set_error(RBOD_E_UNSUPPORTED, "rbod_search_begin: this collection / k is answered by the exact sweep; use rbod_search");
  if (Q > (1ll << 24)) return set_error(RBOD_E_INVAL, "rbod_search_begin: Q too large");
  if (g->rows >= 0xffffffffll) return set_error(RBOD_E_UNSUPPORTED, "rbod_search_begin: more than 2^32-2 rows per shard");
  RBOD_CUDA(cudaSetDevice(g->device));
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  if (g->rows < 1) {
    // an empty shard takes part in the exchange with nothing to offer: no scores, no error bound, nothing dropped
    std::vector<float> ha((size_t)Q * (approx_m + 1), -INFINITY);
    for (int64_t q = 0; q < Q; ++q) ha[(size_t)q * (approx_m + 1) + approx_m] = 0.0f;
    RBOD_CUDA(cudaMemcpyAsync(out_approx, ha.data(), ha.size() * 4, cudaMemcpyHostToDevice, st));
    RBOD_CUDA(cudaStreamSynchronize(st));   // the host vector goes out of scope
    g->pending.Q = Q;
    g->pending.k = k;
    g->pending.kc = 0;
    g->pending.approx_m = approx_m;
    g->pending.q_dev = nullptr;
    g->pending.launches = 0;
    g->pending.valid = 2;   // pending, empty shard
    if (stats) stats->queries = Q;
    return RBOD_OK;
  }
  const int smem_optin = k3_configure(g->device);
  if (smem_optin < 0) return smem_optin;
  RBOD_TRY(maybe_build_shadow(g, k, st));
  Trace tr;
  SearchPlan P;
  RBOD_TRY(plan_search(g, Q, k, search_variant(g, Q), smem_optin, &P));
  RBOD_TRY(g->flags.ensure(64));
  const void* mask_dev = nullptr;
  if (row_mask) RBOD_TRY(to_device(row_mask, (size_t)((g->rows + 31) / 32) * 4, g->mask_dev, st, &mask_dev));
  RBOD_TRY(ensure_lists(g, P));
  RBOD_TRY(g->sel_keys.ensure((size_t)Q * P.kc * 8));
  RBOD_TRY(g->sel_n.ensure((size_t)Q * 4));
  RBOD_TRY(g->sel_tau.ensure((size_t)Q * 4));
  int sample_tiles = 1;
  const bool use_sample = presample_pays(g, P, Q, &sample_tiles);
  const float* q_dev = nullptr;
  const float* tau_init = nullptr;
  int64_t launches = 0;
  const SearchMasks M = {static_cast<const uint32_t*>(mask_dev), (g->rows + 31) / 32, nullptr, nullptr};
  RBOD_TRY(launch_front(g, queries, Q, P, M, use_sample, sample_tiles, st, &q_dev, &tau_init, &launches, tr));
  FinishArgs F;
  fill_finish(g, P, k, tau_init, q_dev, nullptr, nullptr, nullptr, &F);
  F.mode = FIN_SELECT;
  F.approx_m = approx_m;
  F.sel_keys = g->sel_keys.as<unsigned long long>();
  F.sel_n = g->sel_n.as<int>();
  F.sel_tau = g->sel_tau.as<float>();
  F.out_approx = out_approx;
  RBOD_TRY(launch_finish(F, Q, st));
  ++launches;
  g->pending.Q = Q;
  g->pending.k = k;
  g->pending.kc = P.kc;
  g->pending.approx_m = approx_m;
  g->pending.q_pad = P.q_pad;
  g->pending.q_dev = q_dev;
  g->pending.launches = launches;
  g->pending.valid = 1;
  if (stats) {
    stats->queries = Q;
    stats->candidates = P.kc;
    stats->slices = P.slices;
    stats->k3_launches = 1;
    stats->total_launches = launches;
  }
  return RBOD_OK;
}

int rbod_global_cut(const float* gathered_approx, int32_t G, int64_t Q, int32_t approx_m, int32_t k, float* out_cut,
                    void* stream) {
  if (!gathered_approx || !out_cut || Q < 0) return set_error(RBOD_E_INVAL, "rbod_global_cut: bad arguments");
  if (!is_device_ptr(gathered_approx) || !is_device_ptr(out_cut))
    return set_error(RBOD_E_INVAL, "rbod_global_cut: device pointers only");
  return launch_global_cut(gathered_approx, G, Q, approx_m, k, out_cut, static_cast<cudaStream_t>(stream));
}

int rbod_search_end(rbod_gallery* g, const float* cut, int64_t Q, int32_t k, double* out_scores64, int64_t* out_rows,
                    double* out_ubound, rbod_search_stats* stats, void* stream) {
  if (!g) return set_error(RBOD_E_INVAL, "rbod_search_end: NULL handle");
  if (!g->pending.valid || g->pending.Q != Q || g->pending.k != k)
    return set_error(RBOD_E_INVAL, "rbod_search_end: no matching rbod_search_begin is pending on this handle");
  g->pending.valid = 0;
  if (!cut || !out_scores64 || !out_rows || !out_ubound)
    return set_error(RBOD_E_INVAL, "rbod_search_end: bad arguments");
  if (!is_device_ptr(cut) || !is_device_ptr(out_scores64) || !is_device_ptr(out_rows) || !is_device_ptr(out_ubound))
    return set_error(RBOD_E_INVAL, "rbod_search_end: device pointers only");
  RBOD_CUDA(cudaSetDevice(g->device));
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  if (g->pending.kc == 0) {
    // the empty shard of rbod_search_begin: an empty list per query, and no row it could have left unlisted
    const size_t n = (size_t)Q * k;
    std::vector<double> hs(n, -INFINITY), hu((size_t)Q, -INFINITY);
    std::vector<int64_t> hr(n, -1);
    RBOD_CUDA(cudaMemcpyAsync(out_scores64, hs.data(), n * 8, cudaMemcpyHostToDevice, st));
    RBOD_CUDA(cudaMemcpyAsync(out_rows, hr.data(), n * 8, cudaMemcpyHostToDevice, st));
    RBOD_CUDA(cudaMemcpyAsync(out_ubound, hu.data(), (size_t)Q * 8, cudaMemcpyHostToDevice, st));
    RBOD_CUDA(cudaStreamSynchronize(st));
    if (stats) {
      memset(stats, 0, sizeof(*stats));
      stats->queries = Q;
    }
    return RBOD_OK;
  }
  RBOD_TRY(g->out_scores.ensure((size_t)Q * k * 4));
  SearchPlan P;
  memset(&P, 0, sizeof(P));
  P.kc = g->pending.kc;
  P.q_pad = g->pending.q_pad;
  P.slices = 1;
  P.n_cap = 1;
  FinishArgs F;
  fill_finish(g, P, k, nullptr, g->pending.q_dev, g->out_scores.as<float>(), out_rows, out_scores64, &F);
  F.mode = FIN_RESUME;
  F.sel_keys = g->sel_keys.as<unsigned long long>();
  F.sel_n = g->sel_n.as<int>();
  F.sel_tau = g->sel_tau.as<float>();
  F.ext_cut = reinterpret_cast<const float2*>(cut);
  F.ubound = out_ubound;
  RBOD_TRY(launch_finish(F, Q, st));
  if (stats) {
    memset(stats, 0, sizeof(*stats));
    stats->queries = Q;
    stats->candidates = P.kc;
    stats->k3_launches = 1;
    stats->total_launches = g->pending.launches + 1;   // k3_ms: rbod_last_k3_ms, after the caller's own synchronisation
  }
  return RBOD_OK;
}

int rbod_last_k3_ms(rbod_gallery* g, float* out_ms) {
  if (!g || !out_ms) return set_error(RBOD_E_INVAL, "rbod_last_k3_ms: bad arguments");
  if (!g->time_k3) return set_error(RBOD_E_INVAL, "rbod_last_k3_ms: option time_k3 is off");
  RBOD_CUDA(cudaSetDevice(g->device));
  RBOD_CUDA(cudaEventSynchronize(g->ev1));
  RBOD_CUDA(cudaEventElapsedTime(out_ms, g->ev0, g->ev1));
  return RBOD_OK;
}

int rbod_merge_topk_certified(const void* gathered, const int64_t* shard_row0, int32_t G, int64_t Q, int32_t k,
                              float* out_scores, int64_t* out_ids, double* out_scores64, int32_t* out_flag_q,
                              int32_t* out_n_flag, void* stream) {
  if (!gathered || !out_scores || !out_ids || !out_flag_q || !out_n_flag || Q < 0 || k < 1)
    return set_error(RBOD_E_INVAL, "rbod_merge_topk_certified: bad arguments");
  if (!is_device_ptr(gathered) || !is_device_ptr(out_scores) || !is_device_ptr(out_ids) || !is_device_ptr(out_flag_q) ||
      !is_device_ptr(out_n_flag) || (out_scores64 && !is_device_ptr(out_scores64)))
    return set_error(RBOD_E_INVAL, "rbod_merge_topk_certified: device pointers only (shard_row0 is a host array)");
  if (shard_row0 && is_device_ptr(shard_row0))
    return set_error(RBOD_E_INVAL, "rbod_merge_topk_certified: shard_row0 must be a host pointer (or NULL)");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  RBOD_CUDA(cudaMemsetAsync(out_n_flag, 0, 4, st));
  const double* sc = static_cast<const double*>(gathered);
  const int64_t* id = static_cast<const int64_t*>(gathered) + Q * k;
  return launch_merge_topk(sc, id, 2 * Q * k + Q, shard_row0, G, Q, k, out_scores, out_ids, out_scores64, st,
                           sc + 2 * Q * k, out_flag_q, out_n_flag);
}

int rbod_debug_scores(rbod_gallery* g, const float* queries, int64_t Q, float* out, void* stream) {
  if (!g || !queries || !out || Q < 1) return set_error(RBOD_E_INVAL, "rbod_debug_scores: bad arguments");
  if (g->rows < 1) return set_error(RBOD_E_INVAL, "rbod_debug_scores: empty gallery");
  if (g->dp > K3_MAX_DP_WIDE) return set_error(RBOD_E_UNSUPPORTED, "rbod_debug_scores: dim too large");
  if ((double)Q * (double)g->rows > (double)(1ll << 28))
    return set_error(RBOD_E_INVAL, "rbod_debug_scores: Q * rows > 2^28");
  RBOD_CUDA(cudaSetDevice(g->device));
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const int smem_optin = k3_configure(g->device);
  if (smem_optin < 0) return smem_optin;
  SearchPlan P;
  RBOD_TRY(plan_search(g, Q, 1, search_variant(g, Q), smem_optin, &P));
  const float* q_dev = nullptr;
  RBOD_TRY(prepare_queries(g, queries, Q, P, st, &q_dev));
  RBOD_TRY(ensure_lists(g, P));
  const int64_t ld = g->rows;
  const bool out_dev = is_device_ptr(out);
  float* dst = out;
  if (!out_dev) {
    RBOD_TRY(g->dump.ensure((size_t)Q * ld * 4));
    dst = g->dump.as<float>();
  }
  RBOD_CUDA(cudaMemsetAsync(dst, 0xff, (size_t)Q * ld * 4, st));  // NaN pattern: unwritten cells show up
  const SearchMasks none = {nullptr, 0, nullptr, nullptr};
  RBOD_TRY(run_k3(g, P, Q, g->q16.as<uint16_t>(), none, nullptr, dst, ld, st));
  if (!out_dev) RBOD_CUDA(cudaMemcpyAsync(out, dst, (size_t)Q * ld * 4, cudaMemcpyDeviceToHost, st));
  RBOD_CUDA(cudaStreamSynchronize(st));
  return RBOD_OK;
}

int rbod_debug_profile(rbod_gallery* g, int64_t* out16) {
  if (!g || !out16) return set_error(RBOD_E_INVAL, "rbod_debug_profile: NULL argument");
  memset(out16, 0, 16 * sizeof(int64_t));
  if (g->prof.p == nullptr) return RBOD_OK;
  RBOD_CUDA(cudaSetDevice(g->device));
  RBOD_CUDA(cudaDeviceSynchronize());
  RBOD_CUDA(cudaMemcpy(out16, g->prof.p, 16 * sizeof(int64_t), cudaMemcpyDeviceToHost));
  RBOD_CUDA(cudaMemset(g->prof.p, 0, 16 * sizeof(int64_t)));
  return RBOD_OK;
}

int rbod_debug_plan(int32_t dim, int64_t rows, int64_t Q, int32_t k, int32_t variant, int32_t num_sms,
                    int32_t smem_optin, int64_t* out) {
  if (!out || dim < 1 || rows < 1 || Q < 1 || k < 1 || variant < -1 || variant > 2 || num_sms < 2)
    return set_error(RBOD_E_INVAL, "rbod_debug_plan: bad arguments");
  rbod_gallery g;                 // host fields only: nothing is allocated, nothing touches a device
  g.dim = dim;
  g.dp = round_up(dim, K3_KBLOCK);
  g.rows = rows;
  g.num_sms = num_sms;
  if (g.dp > K3_MAX_DP_WIDE || k > K3_MAX_KC)
    return set_error(RBOD_E_UNSUPPORTED, "rbod_debug_plan: dim %d / k %d take the fp64 sweep, not the tensor-core pass",
                     dim, k);
  g.k3_variant = variant;
  SearchPlan P;
  RBOD_TRY(plan_search(&g, Q, k, search_variant(&g, Q), smem_optin, &P));
  out[0] = P.kc;
  out[1] = P.slices;
  out[2] = P.grid;
  out[3] = P.num_qt;
  out[4] = P.tiles_total;
  out[5] = P.num_stages;
  out[6] = P.kbs;
  out[7] = P.a_tmem_kb;
  out[8] = (int64_t)P.smem;
  out[9] = P.list_cap;
  out[10] = P.list_stride;
  out[11] = P.final_cap;
  out[12] = P.n_cap;
  return RBOD_OK;
}

int rbod_merge_topk(const double* scores64, const int64_t* ids, int32_t G, int64_t Q, int32_t k,
                    float* out_scores, int64_t* out_ids, double* out_scores64, void* stream) {
  if (!scores64 || !ids || !out_scores || !out_ids || Q < 0 || k < 1)
    return set_error(RBOD_E_INVAL, "rbod_merge_topk: bad arguments");
  if (!is_device_ptr(scores64) || !is_device_ptr(ids) || !is_device_ptr(out_scores) || !is_device_ptr(out_ids) ||
      (out_scores64 && !is_device_ptr(out_scores64)))
    return set_error(RBOD_E_INVAL, "rbod_merge_topk: device pointers only");
  return launch_merge_topk(scores64, ids, Q * k, nullptr, G, Q, k, out_scores, out_ids, out_scores64,
                           static_cast<cudaStream_t>(stream));
}

int rbod_merge_topk_packed(const void* gathered, const int64_t* shard_row0, int32_t G, int64_t Q, int32_t k,
                           float* out_scores, int64_t* out_ids, double* out_scores64, void* stream) {
  if (!gathered || !out_scores || !out_ids || Q < 0 || k < 1)
    return set_error(RBOD_E_INVAL, "rbod_merge_topk_packed: bad arguments");
  if (!is_device_ptr(gathered) || !is_device_ptr(out_scores) || !is_device_ptr(out_ids) ||
      (out_scores64 && !is_device_ptr(out_scores64)))
    return set_error(RBOD_E_INVAL, "rbod_merge_topk_packed: device pointers only (shard_row0 is a host array)");
  if (shard_row0 && is_device_ptr(shard_row0))
    return set_error(RBOD_E_INVAL, "rbod_merge_topk_packed: shard_row0 must be a host pointer (or NULL)");
  const double* sc = static_cast<const double*>(gathered);
  const int64_t* id = static_cast<const int64_t*>(gathered) + Q * k;
  return launch_merge_topk(sc, id, 2 * Q * k, shard_row0, G, Q, k, out_scores, out_ids, out_scores64,
                           static_cast<cudaStream_t>(stream));
}

}  // extern "C"
