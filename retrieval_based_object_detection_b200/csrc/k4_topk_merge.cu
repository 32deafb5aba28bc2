// K4 family -- everything between the tensor-core pass and the answer:
//
//   finish           one CTA per query, everything between the tensor-core pass and the answer:
//                    (1) gather the query's per-slice candidate lists (K3's append lists) as packed
//                        64-bit keys, (2) radix-select the kc best approximate candidates (tau = the
//                        kc-th best approximate score: every row K3 or this step dropped scores <= tau),
//                        (3) rescore them exactly in fp64 on the stored values -- dot / (|q| * |g|),
//                        the formula of cosine_similarity (33_run_all_experiments.py:76-77) --
//                        (4) order by (score desc, row asc), emit the top k, and (5) certify them: if
//                        tau + eps < (k-th exact score) no dropped row can belong to the top k.
//                        Uncertified queries are appended to a flag list.  (Round 1 ran this as three
//                        kernels -- bitonic merge, rescore, select -- with the candidates round-tripping
//                        through global memory; the bitonic sort of up to 8192 keys per query was the
//                        largest fixed cost of a sharded search.)
//   select_collected answer of the collecting second pass for flagged queries: the rows the collecting K3
//                    launch recorded, rescored exactly.  A query whose list overflows goes on to the exact
//                    fp64 sweep (K5), seeded with its provisional k-th score.  This is the guarantee behind
//                    "identical ids".
//   merge_topk       (K4 proper) G sorted per-GPU lists -> global top k, after the NCCL
//                    all-gather in the row-sharded multi-GPU search.
//
// All of it is small, latency/HBM-bound integer and fp64 work on CUDA cores.
#include "rbod_common.cuh"
#include "rbod_exact_score.cuh"
#include "rbod_internal.h"

#include <algorithm>

namespace rbod {

namespace {

__device__ __forceinline__ bool beats(double sa, uint32_t ia, double sb, uint32_t ib) {
  return sa > sb || (sa == sb && ia < ib);
}

// Exact score of one (query, stored row) pair, one warp per pair, fp64 on the stored values; every lane returns it.
//   COSINE : dot / (|q| |g|)  -- cosine_similarity, 33_run_all_experiments.py:76-77
//   DOT    : dot
//   EUCLID : the ordering key -sum (q_i - g_i)^2, accumulated directly (no |q|^2 - 2 q.g + |g|^2 cancellation)
__device__ __forceinline__ double exact_pair_score(const float* __restrict__ qv, double qq,
                                                   const float* __restrict__ g32, const uint16_t* __restrict__ g16,
                                                   int kind16, int dim, int metric, int lane) {
  double a = 0.0, b = 0.0;
  auto acc = [&](double qc, double x) {
    if (metric == RBOD_EUCLID) {
      const double d = qc - x;
      a = fma(d, d, a);
    } else {
      a = fma(qc, x, a);
      b = fma(x, x, b);
    }
  };
  const bool vec = (dim & 7) == 0 && (reinterpret_cast<uintptr_t>(qv) & 15) == 0 &&
                   (g32 ? (reinterpret_cast<uintptr_t>(g32) & 15) == 0 : (reinterpret_cast<uintptr_t>(g16) & 15) == 0);
  if (vec) {
    // 8 elements per lane and step: 16-byte loads of the stored row, two float4 of the query
    for (int c0 = lane * 8; c0 < dim; c0 += 256) {
      const float4 q0 = *reinterpret_cast<const float4*>(qv + c0);
      const float4 q1 = *reinterpret_cast<const float4*>(qv + c0 + 4);
      float x[8];
      if (g32) {
        const float4 g0 = *reinterpret_cast<const float4*>(g32 + c0);
        const float4 g1 = *reinterpret_cast<const float4*>(g32 + c0 + 4);
        x[0] = g0.x; x[1] = g0.y; x[2] = g0.z; x[3] = g0.w;
        x[4] = g1.x; x[5] = g1.y; x[6] = g1.z; x[7] = g1.w;
      } else {
        const uint4 h = *reinterpret_cast<const uint4*>(g16 + c0);
        const uint32_t w[4] = {h.x, h.y, h.z, h.w};
#pragma unroll
        for (int i = 0; i < 4; ++i) {
          x[2 * i] = h16_to_f32(static_cast<uint16_t>(w[i] & 0xffffu), kind16);
          x[2 * i + 1] = h16_to_f32(static_cast<uint16_t>(w[i] >> 16), kind16);
        }
      }
      acc((double)q0.x, (double)x[0]);
      acc((double)q0.y, (double)x[1]);
      acc((double)q0.z, (double)x[2]);
      acc((double)q0.w, (double)x[3]);
      acc((double)q1.x, (double)x[4]);
      acc((double)q1.y, (double)x[5]);
      acc((double)q1.z, (double)x[6]);
      acc((double)q1.w, (double)x[7]);
    }
  } else {
    for (int c = lane; c < dim; c += 32)
      acc((double)qv[c], g32 ? (double)g32[c] : (double)h16_to_f32(g16[c], kind16));
  }
  a = warp_sum_f64(a);
  if (metric == RBOD_EUCLID) return -a;
  if (metric == RBOD_DOT) return a;
  b = warp_sum_f64(b);
  const double den = sqrt(qq) * sqrt(b);
  return den > 0.0 ? a / den : 0.0;
}

// What the caller sees for an internal score: EUCLID keys (-d^2) come out as the distance d (fp32) and keep the
// key in the fp64 output (the order the multi-GPU merge uses); "no result" is an infinite distance.
__device__ __forceinline__ float user_score(double s, int metric) {
  return metric == RBOD_EUCLID ? (float)sqrt(-s) : (float)s;
}
__device__ __forceinline__ float user_no_result(int metric) { return metric == RBOD_EUCLID ? INFINITY : -INFINITY; }

// ---------------------------------------------------------------------------------------------
// tau_init: starting threshold of a query = the smallest of its `groups` sample-group maxima.  Every
// group holds one row scoring at least that much, and with N / (rows per group) = 16 * kc the expected
// number of gallery rows above it is ~ 16 * kc * H(groups): far fewer than N, so the candidate heaps
// skip their cold start, yet fewer than k rows beat it only with probability ~ (k / (16 kc))^groups
// per query (8 groups: < 1e-9 even at k = 100, kc = 128); the host then redoes the call without it.
// ---------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256)
tau_init_kernel(const float* __restrict__ groupmax, int groups, int splits, int64_t q_pad,
                uint32_t* __restrict__ tau_shared, float* __restrict__ tau_init) {
  const int64_t q = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (q >= q_pad) return;
  // a group's maximum = the largest of its splits' maxima (each split visited part of the group's comb)
  float t = INFINITY;
  for (int g = 0; g < groups; ++g) {
    float m = -INFINITY;
    for (int s = 0; s < splits; ++s) m = fmaxf(m, groupmax[((size_t)g * splits + s) * q_pad + q]);
    t = fminf(t, m);
  }
  if (!(t > -INFINITY)) t = -INFINITY;   // an empty (or fully masked) group: no starting threshold
  tau_init[q] = t;
  tau_shared[q] = f32_to_ordered(t);
}

// ---------------------------------------------------------------------------------------------
// finish: one CTA per query (see the file header)
// ---------------------------------------------------------------------------------------------
constexpr int FIN_THREADS = 256;
constexpr int FIN_WARPS = FIN_THREADS / 32;
constexpr int FIN_MAX_SLICES = 2 * FIN_THREADS;
constexpr int FIN_MAX_KEYS = 8192;

// The error model of the tensor-core pass for one query (one thread): eps bounds |approximate score - exact score in
// the approximate domain| for EVERY row of the collection, given that tau bounds the approximate scores in play.
//   |approx - exact cosine| <= ||q16 - unit(q)|| * max||g16||      (query rounding, Cauchy-Schwarz)
//                            + dp * 2^-23 * max||g16||              (fp32 accumulation in the tensor core)
//                            + row term
// The row term is ||g16 - unit(G)|| for fp32 masters (their 16-bit shadow is rounded independently);
// for 16-bit masters g16 IS the stored row and only its norm deviates from 1 by d = stats[1], which
// scales the score instead of adding to it: (|tau| + e) * d / (1 - d).
// With an fp16 shadow as the search operand, the operand norm is stats[2] and its distance to the stored
// row, stats[3], adds to the query term.
// DOT collections: nothing is normalised, so every term scales with the query norm |q| and the row term is
// |q| * ||g16 - g|| (zero for 16-bit masters, whose operand is the stored row).
// EUCLID collections: the tensor-core pass scores a = q16 . g16 + bias32 with bias32 = fp32(-|g|^2 / 2), an
// approximation of (key + |q|^2) / 2 for the exact key = -|q - g|^2.  Nothing is normalised, so the dot-product
// terms are those of DOT, plus the rounding of the bias and of its addition: 2^-23 (|q| G + G^2), G = max |g|.
struct QueryMargin { float e, row_term, bias_term, eps, gdev; bool unnorm, master16; double qq_half; };

__device__ QueryMargin query_margin(const FinishArgs& P, int64_t q, float tau) {
  QueryMargin M;
  const float* stats = P.stats;
  const int metric = P.metric;
  M.master16 = P.master16 != 0;
  const bool shadow = P.shadow != 0;
  const float gmax = (shadow ? stats[2] : stats[0]) * 1.000001f;
  M.gdev = stats[1] * 1.000001f;
  M.unnorm = metric != RBOD_COSINE;
  const float qn = M.unnorm ? (float)sqrt(P.q_qq[q]) * 1.000001f + P.q_dq[q] : 1.0f;
  M.e = P.q_dq[q] * gmax + (float)P.dp * 1.2e-7f * gmax * qn + (shadow ? stats[3] * 1.000001f * qn : 0.0f);
  M.row_term = M.unnorm ? (M.master16 ? 0.0f : qn * M.gdev)
                        : (M.master16 ? (fabsf(tau) + M.e) * M.gdev / (1.0f - M.gdev) : M.gdev);
  const float gbig = gmax + (M.master16 ? 0.0f : M.gdev);
  M.bias_term = metric == RBOD_EUCLID ? 1.2e-7f * (qn * gbig + gbig * gbig) : 0.0f;
  M.eps = M.e + M.row_term + M.bias_term + fabsf(tau) * 1e-6f + 1e-7f;
  M.qq_half = metric == RBOD_EUCLID ? 0.5 * P.q_qq[q] : 0.0;
  return M;
}

// Certification of one query's answer (one thread).  tau bounds the approximate score of every row that was dropped
// anywhere; kth is the k-th exact score (if k candidates exist): if tau + eps < kth no dropped row can belong to the
// top k.  Otherwise the query joins the flag list of the collecting second pass.
__device__ void certify_query(const FinishArgs& P, int64_t q, float tau, const QueryMargin& M, bool have_kth, double kth) {
  const int metric = P.metric;
  bool flagged = true;
  if (have_kth) {
    // the k-th exact score in the domain the tensor-core pass works in
    const double kth_a = metric == RBOD_EUCLID ? 0.5 * kth + M.qq_half : kth;
    flagged = !((double)tau + (double)M.eps < kth_a);
  } else {
    // Fewer than k candidates although rows were dropped: the pre-sampled starting threshold sat above this
    // query's k-th best score (possible only when the sample misrepresents the gallery).  The host reruns the
    // search without the pre-pass.
    kth = -INFINITY;
    atomicAdd(P.n_flag + 4, 1);
  }
  atomic_max_nonneg(P.max_eps, M.eps);
  if (flagged) {
    const int slot = atomicAdd(P.n_flag, 1);
    P.flag_q[slot] = (int)q;
    P.flag_thr[slot] = kth;
    // Threshold for the collecting second pass: every row whose exact score reaches kth has an
    // approximate score above lo (same error model, applied from the exact side).
    const float kf = (float)(metric == RBOD_EUCLID ? 0.5 * kth + M.qq_half : kth);
    const float lo = M.unnorm ? kf - M.e - M.row_term - M.bias_term
                              : (M.master16 ? kf - fabsf(kf) * M.gdev - M.e : kf - M.e - M.gdev);
    P.flag_lo[slot] = kth == -INFINITY ? -INFINITY : lo - fabsf(kf) * 2e-6f - 2e-7f;
  }
}

// A stored 16-bit row of up to 1024 columns as this lane's share of it: 8 consecutive elements per 256-column step.
struct RowRegs { uint4 h[4]; };
__device__ __forceinline__ void load_row16(RowRegs& R, const uint16_t* __restrict__ g16, int dim, int lane) {
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const int c0 = lane * 8 + 256 * i;
    R.h[i] = c0 < dim ? __ldg(reinterpret_cast<const uint4*>(g16 + c0)) : make_uint4(0u, 0u, 0u, 0u);
  }
}

template <int METRIC>
__device__ __forceinline__ double exact_score_regs(const double* __restrict__ q64, double qq, const RowRegs& R, int kind16,
                                                   int dim, int lane) {
  double a = 0.0, b = 0.0;
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const int c0 = lane * 8 + 256 * i;
    if (c0 < dim) {
      float x[8];
      unpack8(R.h[i], kind16, x);
      score_step8<METRIC>(q64 + c0, x, a, b);
    }
  }
  return finish_score<METRIC>(a, b, qq);
}

// Exact scores of the candidates s_sel2[0..nres): warp w takes candidates w, w + 8, ...  For 16-bit masters up to 1024
// columns the NEXT candidate's row is already in flight while the current one is scored (software pipelining: the
// rescoring is a gather of 1.5 KB rows from all over HBM, and its latency, not its arithmetic, is what costs).
template <int METRIC>
__device__ __forceinline__ void rescore_candidates(const FinishArgs& P, const double* __restrict__ q64, double qq,
                                                   const unsigned long long* __restrict__ sel, int nres,
                                                   double* __restrict__ out_sc, int warp, int lane) {
  const bool pipelined = P.master32 == nullptr && (P.dim & 7) == 0 && P.dim <= 1024 &&
                         (reinterpret_cast<uintptr_t>(P.rows16) & 15) == 0 && (P.ld16 & 7) == 0;
  if (pipelined) {
    RowRegs cur, nxt;
    int cnd = warp;
    if (cnd < nres) load_row16(cur, P.rows16 + (int64_t)(~static_cast<uint32_t>(sel[cnd])) * P.ld16, P.dim, lane);
    for (; cnd < nres; cnd += FIN_WARPS) {
      const int nx = cnd + FIN_WARPS;
      if (nx < nres) load_row16(nxt, P.rows16 + (int64_t)(~static_cast<uint32_t>(sel[nx])) * P.ld16, P.dim, lane);
      const double sc = exact_score_regs<METRIC>(q64, qq, cur, P.kind16, P.dim, lane);
      if (lane == 0) out_sc[cnd] = sc;
      cur = nxt;
    }
    return;
  }
  for (int cnd = warp; cnd < nres; cnd += FIN_WARPS) {
    const uint32_t idx = ~static_cast<uint32_t>(sel[cnd]);
    const float* g32 = P.master32 ? P.master32 + (int64_t)idx * P.ld32 : nullptr;
    const uint16_t* g16 = P.master32 ? nullptr : P.rows16 + (int64_t)idx * P.ld16;
    const double sc = exact_score_q64<METRIC>(q64, qq, g32, g16, P.kind16, P.dim, lane);
    if (lane == 0) out_sc[cnd] = sc;
  }
}

__global__ void __launch_bounds__(FIN_THREADS) finish_kernel(const FinishArgs P) {
  extern __shared__ unsigned long long keys[];   // [n_cap]: ordered(score) << 32 | ~row; distinct, larger = better
  __shared__ int s_off[FIN_MAX_SLICES + 1];
  __shared__ int s_wsum[FIN_WARPS];
  __shared__ unsigned int s_cnt[3];
  __shared__ uint32_t s_hmax[FIN_WARPS], s_hmin[FIN_WARPS];
  __shared__ unsigned long long s_sel[K3_MAX_KC], s_sel2[K3_MAX_KC];
  __shared__ double s_sc[K3_MAX_KC];
  __shared__ float s_cut;
  __shared__ int s_nsel, s_nres, s_have_kth;
  __shared__ double s_kth;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int64_t q = blockIdx.x;
  const int kc = P.kc, k = P.k;
  int total = 0, nsel = 0;

  if (P.mode == FIN_RESUME) {
    // second half of a split search (rbod_search_end): the selection of the first half comes back from global memory
    if (tid == 0) {
      s_nres = 0;
      s_have_kth = 0;
      s_kth = -INFINITY;
    }
    nsel = min(max(P.sel_n[q], 0), min(kc, K3_MAX_KC));
    if (tid < nsel) s_sel[tid] = P.sel_keys[q * kc + tid];
  } else {
    // (1) list lengths -> exclusive offsets (two slices per thread)
    int c0 = 0, c1 = 0;
    if (2 * tid < P.slices) c0 = min(max(P.list_cnt[(size_t)(2 * tid) * P.q_pad + q], 0), P.list_stride);
    if (2 * tid + 1 < P.slices) c1 = min(max(P.list_cnt[(size_t)(2 * tid + 1) * P.q_pad + q], 0), P.list_stride);
    int incl = c0 + c1;
  #pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const int t = __shfl_up_sync(FULL_MASK, incl, o);
      if (lane >= o) incl += t;
    }
    if (lane == 31) s_wsum[warp] = incl;
    if (tid == 0) {
      s_cnt[0] = s_cnt[1] = s_cnt[2] = 0u;
      s_nsel = 0;
      s_nres = 0;
      s_have_kth = 0;
      s_kth = -INFINITY;
    }
    __syncthreads();
    int wbase = 0;
    total = 0;
  #pragma unroll
    for (int w = 0; w < FIN_WARPS; ++w) {
      if (w < warp) wbase += s_wsum[w];
      total += s_wsum[w];
    }
    const int excl = wbase + incl - c0 - c1;
    if (2 * tid < P.slices) s_off[2 * tid] = excl;
    if (2 * tid + 1 < P.slices) s_off[2 * tid + 1] = excl + c0;
    if (tid == 0) s_off[P.slices] = total;
    const int n_tot = min(total, P.n_cap);
    __syncthreads();

    // gather the lists as packed keys
    for (int s = warp; s < P.slices; s += FIN_WARPS) {
      const int off = s_off[s], cs = s_off[s + 1] - off;
      const uint2* lst = P.lists + ((size_t)s * P.q_pad + q) * P.list_stride;
      for (int j = lane; j < cs; j += 32)
        if (off + j < n_tot) {
          const uint2 e = lst[j];
          keys[off + j] = (static_cast<unsigned long long>(f32_to_ordered(__uint_as_float(e.x))) << 32) |
                          static_cast<unsigned long long>(~e.y);
        }
    }
    __syncthreads();

    // (2) the kc-th largest key by a most-significant-bit-first radix descent, one block-wide count per bit, starting
    // at the first bit in which the scores differ at all.  Keys are distinct (a row appears once), so the descent ends
    // with exactly kc keys at or above the decided prefix -- usually long before the last bit.
    unsigned long long T = 0ull;
    if (n_tot > kc) {
      uint32_t hmax = 0u, hmin = 0xffffffffu;
      for (int j = tid; j < n_tot; j += FIN_THREADS) {
        const uint32_t h = static_cast<uint32_t>(keys[j] >> 32);
        hmax = max(hmax, h);
        hmin = min(hmin, h);
      }
      hmax = __reduce_max_sync(FULL_MASK, hmax);
      hmin = __reduce_min_sync(FULL_MASK, hmin);
      if (lane == 0) {
        s_hmax[warp] = hmax;
        s_hmin[warp] = hmin;
      }
      __syncthreads();
  #pragma unroll
      for (int w = 0; w < FIN_WARPS; ++w) {
        hmax = max(hmax, s_hmax[w]);
        hmin = min(hmin, s_hmin[w]);
      }
      const uint32_t diff = hmax ^ hmin;
      int b = diff ? 32 + (31 - __clz(diff)) : 31;
      unsigned long long prefix = static_cast<unsigned long long>(diff ? (hmax & ~((2u << (b - 32)) - 1u)) : hmax) << 32;
      int remaining = kc, share = n_tot, it = 0;
      while (b >= 0 && share != remaining) {
        const unsigned long long want = (prefix >> b) | 1ull;
        int cc = 0;
        for (int j = tid; j < n_tot; j += FIN_THREADS) cc += ((keys[j] >> b) == want) ? 1 : 0;
        cc = __reduce_add_sync(FULL_MASK, cc);
        if (lane == 0 && cc) atomicAdd(&s_cnt[it % 3], (unsigned int)cc);
        if (tid == 0) s_cnt[(it + 1) % 3] = 0u;   // last read two iterations ago, next used after this barrier
        __syncthreads();
        const int ctot = (int)s_cnt[it % 3];
        if (ctot >= remaining) {
          prefix |= 1ull << b;
          share = ctot;
        } else {
          remaining -= ctot;
          share -= ctot;
        }
        --b;
        ++it;
      }
      T = prefix;
    }
    for (int j = tid; j < n_tot; j += FIN_THREADS) {
      const unsigned long long key = keys[j];
      if (key >= T) {
        const int pos = atomicAdd(&s_nsel, 1);
        if (pos < K3_MAX_KC) s_sel[pos] = key;
      }
    }
  }
  if (P.mode != FIN_SELECT)
    for (int j = tid; j < k; j += FIN_THREADS) {
      P.out_scores[q * k + j] = user_no_result(P.metric);
      P.out_rows[q * k + j] = -1;
      if (P.out_scores64) P.out_scores64[q * k + j] = -INFINITY;
    }
  __syncthreads();
  if (P.mode != FIN_RESUME) nsel = min(min(s_nsel, kc), K3_MAX_KC);

  // kc or more candidates: everything dropped (by a prune of K3 or by the selection above) scores at most the
  // kc-th best approximate score.  Fewer: no list was ever pruned, only the pre-sampled threshold dropped rows.
  uint32_t hmin = 0xffffffffu, hbest = 0u;
  for (int i = lane; i < nsel; i += 32) {
    hmin = min(hmin, static_cast<uint32_t>(s_sel[i] >> 32));
    hbest = max(hbest, static_cast<uint32_t>(s_sel[i] >> 32));
  }
  hmin = __reduce_min_sync(FULL_MASK, hmin);
  hbest = __reduce_max_sync(FULL_MASK, hbest);
  float tau;
  if (P.mode == FIN_RESUME) {
    tau = P.sel_tau[q];
  } else {
    tau = total >= kc ? ordered_to_f32(hmin) : -INFINITY;
    if (P.tau_init != nullptr) tau = fmaxf(tau, P.tau_init[q]);
  }
  const QueryMargin M = query_margin(P, q, tau);
  // the same bound for the CANDIDATES, whose scores reach up to the best approximate score: for unit-norm 16-bit
  // masters the row term scales with the score it perturbs
  const float s_best = nsel > 0 ? fabsf(ordered_to_f32(hbest)) : 0.0f;
  const float eps_cand = (!M.unnorm && M.master16)
                             ? M.e + (fmaxf(s_best, fabsf(tau) == INFINITY ? 0.0f : fabsf(tau)) + M.e) * M.gdev / (1.0f - M.gdev) +
                                   s_best * 1e-6f + 1e-7f
                             : M.eps + s_best * 1e-6f;

  if (P.mode == FIN_SELECT) {
    // first half of a split search (rbod_search_begin): keep the selection and the threshold, and publish the
    // approx_m best approximate scores plus this shard's error bound for them -- what the other shards need to
    // place the GLOBAL k-th best approximate score
    if (tid < nsel) {
      const unsigned long long mykey = s_sel[tid];
      P.sel_keys[q * kc + tid] = mykey;
      int above = 0;
      for (int i = 0; i < nsel; ++i) above += s_sel[i] > mykey ? 1 : 0;
      if (above < P.approx_m) P.out_approx[q * (P.approx_m + 1) + above] = ordered_to_f32(static_cast<uint32_t>(mykey >> 32));
    }
    for (int j = nsel + tid; j < P.approx_m; j += FIN_THREADS) P.out_approx[q * (P.approx_m + 1) + j] = -INFINITY;
    if (tid == 0) {
      P.sel_n[q] = nsel;
      P.sel_tau[q] = tau;
      P.out_approx[q * (P.approx_m + 1) + P.approx_m] = eps_cand;
    }
    return;
  }

  // (3) exact scores.  Not every candidate needs one: the error model puts every row's approximate score within eps
  // of its exact score (in the approximate domain), so a candidate more than 2 eps below the k-th best APPROXIMATE
  // score is beaten by k others exactly as well and cannot be in the answer.  The keys of the candidates that stay
  // are compacted to the front; the query is widened to fp64 once, into the (now free) key buffer.
  double* q64 = reinterpret_cast<double*>(keys);
  const float* qv = P.q + q * P.dim;
  for (int c = tid; c < P.dim; c += FIN_THREADS) q64[c] = (double)qv[c];
  unsigned long long mykey = 0ull;
  bool keep = false;
  if (tid < nsel) {
    mykey = s_sel[tid];
    keep = true;
    if (nsel > k) {
      int above = 0;
      for (int i = 0; i < nsel; ++i) above += s_sel[i] > mykey ? 1 : 0;
      if (above == k - 1) s_cut = ordered_to_f32(static_cast<uint32_t>(mykey >> 32));   // the k-th best approximate score
    }
  }
  __syncthreads();
  if (P.mode == FIN_RESUME) {
    // the cut is the k-th best approximate score over ALL shards and the bound the largest any shard reported: a
    // candidate more than 2 eps below it is beaten exactly by k rows somewhere and cannot be in the global answer
    const float2 ext = P.ext_cut[q];
    if (tid < nsel) keep = ordered_to_f32(static_cast<uint32_t>(mykey >> 32)) >= ext.x - 2.0f * fmaxf(eps_cand, ext.y);
  } else if (tid < nsel && nsel > k) {
    keep = ordered_to_f32(static_cast<uint32_t>(mykey >> 32)) >= s_cut - 2.0f * eps_cand;
  }
  if (keep) {
    const int pos = atomicAdd(&s_nres, 1);
    s_sel2[pos] = mykey;
  }
  __syncthreads();
  const int nres = s_nres;
  const double qq = P.q_qq[q];
  if (P.metric == RBOD_COSINE) rescore_candidates<RBOD_COSINE>(P, q64, qq, s_sel2, nres, s_sc, warp, lane);
  else if (P.metric == RBOD_DOT) rescore_candidates<RBOD_DOT>(P, q64, qq, s_sel2, nres, s_sc, warp, lane);
  else rescore_candidates<RBOD_EUCLID>(P, q64, qq, s_sel2, nres, s_sc, warp, lane);
  __syncthreads();

  // (4) rank by counting over the rescored candidates
  if (tid < nres) {
    const double sv = s_sc[tid];
    const uint32_t ix = ~static_cast<uint32_t>(s_sel2[tid]);
    int rank = 0;
    for (int i = 0; i < nres; ++i)
      if (beats(s_sc[i], ~static_cast<uint32_t>(s_sel2[i]), sv, ix)) ++rank;
    if (rank < k) {
      P.out_scores[q * k + rank] = user_score(sv, P.metric);
      P.out_rows[q * k + rank] = (int64_t)ix;
      if (P.out_scores64) P.out_scores64[q * k + rank] = sv;
      if (rank == k - 1) {
        s_kth = sv;
        s_have_kth = 1;
      }
    }
  }
  __syncthreads();

  // (5) certification
  if (P.mode == FIN_RESUME) {
    // The local list is complete only down to the global cut, so the k-th local score certifies nothing; what the
    // merge needs is an upper bound, in the domain of the exact keys, on every row this shard never listed
    if (tid == 0) {
      double ub = -INFINITY;
      if (tau != -INFINITY) {
        ub = (double)tau + (double)M.eps;
        if (P.metric == RBOD_EUCLID) ub = 2.0 * (ub - M.qq_half);
        atomic_max_nonneg(P.max_eps, M.eps);
      }
      P.ubound[q] = ub;
    }
    return;
  }
  if (tid == 0 && tau != -INFINITY) certify_query(P, q, tau, M, s_have_kth != 0, s_kth);   // else exact by construction
}

// k-th largest approximate score of a query over the lists the shards published (rbod_search_begin), and the largest
// error bound among them: one warp per query, MSB-first descent over the order-preserving integer image.
__global__ void __launch_bounds__(128) global_cut_kernel(const float* __restrict__ gathered, int G, int64_t Q, int m, int k,
                                                         float2* __restrict__ out) {
  extern __shared__ uint32_t gc_vals[];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int64_t q = (int64_t)blockIdx.x * (blockDim.x >> 5) + warp;
  if (q >= Q) return;
  uint32_t* v = gc_vals + (size_t)warp * G * m;
  const int n = G * m;
  float eps = 0.0f;
  for (int g = 0; g < G; ++g) {
    const float* src = gathered + ((size_t)g * Q + q) * (m + 1);
    for (int j = lane; j < m; j += 32) v[g * m + j] = f32_to_ordered(src[j]);
    eps = fmaxf(eps, src[m]);
  }
  __syncwarp();
  uint32_t prefix = 0u;
  int remaining = k;   // the answer is the remaining-th largest among the values that share the decided prefix
  for (int b = 31; b >= 0; --b) {
    const uint32_t want = (prefix >> b) | 1u;
    int c = 0;
    for (int j = lane; j < n; j += 32) c += ((v[j] >> b) == want) ? 1 : 0;
    c = __reduce_add_sync(FULL_MASK, c);
    if (c >= remaining) prefix |= 1u << b;
    else remaining -= c;
  }
  if (lane == 0) out[q] = make_float2(n >= k ? ordered_to_f32(prefix) : -INFINITY, eps);
}

// The answer of a collecting second pass from its rescored list (one CTA per flagged query).  A list that overflowed
// is left alone: the host sends that query on to the exact sweep (K5).
__global__ void __launch_bounds__(256)
select_collected_kernel(const double* __restrict__ coll_score, const uint32_t* __restrict__ coll_idx,
                        const int* __restrict__ coll_cnt, const int* __restrict__ flag_q, int f0, int cap, int k,
                        int metric, float* __restrict__ out_scores, int64_t* __restrict__ out_rows,
                        double* __restrict__ out_scores64) {
  const int f = blockIdx.x;
  const int q = flag_q[f0 + f];
  const int cnt = coll_cnt[f];
  if (cnt > cap) return;
  const double* sc = coll_score + (size_t)f * cap;
  const uint32_t* ix = coll_idx + (size_t)f * cap;
  for (int j = threadIdx.x; j < k; j += blockDim.x) {
    out_scores[(int64_t)q * k + j] = user_no_result(metric);
    out_rows[(int64_t)q * k + j] = -1;
    if (out_scores64) out_scores64[(int64_t)q * k + j] = -INFINITY;
  }
  __syncthreads();
  for (int j = threadIdx.x; j < cnt; j += blockDim.x) {
    const double s = sc[j];
    const uint32_t id = ix[j];
    int rank = 0;
    for (int i = 0; i < cnt; ++i)
      if (beats(sc[i], ix[i], s, id)) ++rank;
    if (rank < k) {
      out_scores[(int64_t)q * k + rank] = user_score(s, metric);
      out_rows[(int64_t)q * k + rank] = (int64_t)id;
      if (out_scores64) out_scores64[(int64_t)q * k + rank] = s;
    }
  }
}

// ---------------------------------------------------------------------------------------------
// second pass for uncertified queries (tensor-core collect): pack their 16-bit rows into a dense
// query matrix, then rescore whatever the collecting K3 launch recorded.
// ---------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256)
gather_flagged_kernel(const uint16_t* __restrict__ q16, int dp, const int* __restrict__ flag_q, int f0, int nf,
                      int64_t nf_pad, uint16_t* __restrict__ fq16, int* __restrict__ coll_cnt,
                      const int* __restrict__ mask_of_query, int* __restrict__ fmask) {
  const int lane = threadIdx.x & 31;
  const int64_t w0 = (int64_t)blockIdx.x * 8 + (threadIdx.x >> 5);
  const int64_t nw = (int64_t)gridDim.x * 8;
  for (int64_t f = w0; f < nf_pad; f += nw) {
    uint4* dst = reinterpret_cast<uint4*>(fq16 + f * dp);
    if (f < nf) {
      const uint4* src = reinterpret_cast<const uint4*>(q16 + (int64_t)flag_q[f0 + f] * dp);
      for (int c = lane; c < dp / 8; c += 32) dst[c] = src[c];
    } else {
      for (int c = lane; c < dp / 8; c += 32) dst[c] = make_uint4(0u, 0u, 0u, 0u);
    }
    if (lane == 0) {
      coll_cnt[f] = 0;
      // per-query masks: the gathered row keeps its query's mask (pad rows read none)
      if (mask_of_query != nullptr) fmask[f] = f < nf ? mask_of_query[flag_q[f0 + f]] : -1;
    }
  }
}

// one warp per (flagged query, recorded row); grid.y = flagged query
__global__ void __launch_bounds__(256)
rescore_collected_kernel(const float* __restrict__ q, const double* __restrict__ q_qq,
                         const float* __restrict__ master32, const uint16_t* __restrict__ rows16, int kind16,
                         int dim, int64_t ld32, int64_t ld16, int metric, const int* __restrict__ flag_q, int f0, int cap,
                         const uint32_t* __restrict__ coll_idx, const int* __restrict__ coll_cnt,
                         double* __restrict__ coll_score) {
  const int lane = threadIdx.x & 31;
  const int f = blockIdx.y;
  const int cnt = min(coll_cnt[f], cap);
  const int qi = flag_q[f0 + f];
  const float* qv = q + (int64_t)qi * dim;
  for (int j = blockIdx.x * 8 + (threadIdx.x >> 5); j < cnt; j += gridDim.x * 8) {
    const uint32_t idx = coll_idx[(size_t)f * cap + j];
    const double sc = exact_pair_score(qv, q_qq[qi], master32 ? master32 + (int64_t)idx * ld32 : nullptr,
                                       master32 ? nullptr : rows16 + (int64_t)idx * ld16, kind16, dim, metric, lane);
    if (lane == 0) coll_score[(size_t)f * cap + j] = sc;
  }
}

// ---------------------------------------------------------------------------------------------
// merge_topk: one warp per query, lane g walks the (sorted) list of shard g.  G <= 32.
// Shard g's scores start at scores64 + g * shard_stride, its ids at ids + g * shard_stride (8-byte words), so the
// same kernel reads two separately gathered arrays (stride Q * k) or ONE gathered buffer in which every rank sent
// its scores and its local row slots back to back (stride 2 * Q * k); row0[g] >= 0 turns local slots into global ids.
// ---------------------------------------------------------------------------------------------
struct MergeRow0 { long long v[32]; };

__global__ void __launch_bounds__(256)
merge_topk_kernel(const double* __restrict__ scores64, const int64_t* __restrict__ ids, int64_t shard_stride, int G,
                  int64_t Q, int k, const MergeRow0 row0, float* __restrict__ out_scores,
                  int64_t* __restrict__ out_ids, double* __restrict__ out_scores64,
                  const double* __restrict__ ubound, int* __restrict__ flag_q, int* __restrict__ n_flag) {
  const int lane = threadIdx.x & 31;
  const int64_t q = (int64_t)blockIdx.x * 8 + (threadIdx.x >> 5);
  if (q >= Q) return;
  double kth = -INFINITY;   // the k-th merged score, if there are k
  int pos = 0;
  const int src = lane < G ? lane : 0;
  const double* sc = scores64 + (size_t)src * shard_stride + q * k;
  const int64_t* id = ids + (size_t)src * shard_stride + q * k;
  const long long off = row0.v[src];
  const long long kEmpty = 0x7fffffffffffffffll;
  double hs = -INFINITY;
  long long hi = kEmpty;
  if (lane < G && k > 0 && id[0] >= 0) { hs = sc[0]; hi = id[0] + off; }
  for (int j = 0; j < k; ++j) {
    // warp arg-best over (score desc, id asc); empty heads lose
    double bs = hs;
    long long bi = hi;
    int bl = lane;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      const double os = __shfl_xor_sync(FULL_MASK, bs, o);
      const long long oi = __shfl_xor_sync(FULL_MASK, bi, o);
      const int ol = __shfl_xor_sync(FULL_MASK, bl, o);
      const bool take = (oi != kEmpty) && (bi == kEmpty || os > bs || (os == bs && (oi < bi || (oi == bi && ol < bl))));
      if (take) { bs = os; bi = oi; bl = ol; }
    }
    if (lane == 0) {
      const bool valid = bi != kEmpty;
      out_scores[q * k + j] = valid ? (float)bs : -INFINITY;
      out_ids[q * k + j] = valid ? (int64_t)bi : -1;
      if (out_scores64) out_scores64[q * k + j] = valid ? bs : -INFINITY;
    }
    if (j == k - 1 && bi != kEmpty) kth = bs;
    if (bi == kEmpty) continue;  // uniform: all lanes agree on the winner
    if (lane == bl) {
      ++pos;
      if (pos < k && id[pos] >= 0) { hs = sc[pos]; hi = id[pos] + off; }
      else { hs = -INFINITY; hi = kEmpty; }
    }
  }
  if (ubound != nullptr) {
    // split searches (rbod_search_end): shard g vouches that no row it left unlisted scores above ubound[g][q]; the
    // merged answer is exact when its k-th score beats every shard's bound
    double ub = lane < G ? ubound[(size_t)lane * shard_stride + q] : -INFINITY;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) ub = fmax(ub, __shfl_xor_sync(FULL_MASK, ub, o));
    if (lane == 0 && ub != -INFINITY && !(ub < kth)) flag_q[atomicAdd(n_flag, 1)] = (int)q;
  }
}

}  // namespace

int launch_tau_init(const float* groupmax, int groups, int splits, int64_t q_pad, uint32_t* tau_shared,
                    float* tau_init, cudaStream_t st) {
  if (q_pad <= 0) return RBOD_OK;
  tau_init_kernel<<<(unsigned)((q_pad + 255) / 256), 256, 0, st>>>(groupmax, groups, splits, q_pad, tau_shared,
                                                                   tau_init);
  RBOD_CUDA(cudaGetLastError());
  return RBOD_OK;
}

int launch_finish(const FinishArgs& A, int64_t Q, cudaStream_t st) {
  if (Q <= 0) return RBOD_OK;
  if (A.kc < 1 || A.kc > K3_MAX_KC || A.k < 1 || A.k > A.kc)
    return set_error(RBOD_E_INVAL, "finish: k %d / kc %d outside [1, %d]", A.k, A.kc, K3_MAX_KC);
  if (A.slices < 1 || A.slices > FIN_MAX_SLICES)
    return set_error(RBOD_E_INVAL, "finish: %d slices outside [1, %d]", A.slices, FIN_MAX_SLICES);
  if (A.dim > FIN_MAX_KEYS) return set_error(RBOD_E_UNSUPPORTED, "finish: dim %d > %d", A.dim, FIN_MAX_KEYS);
  if (A.n_cap < 1 || A.n_cap > FIN_MAX_KEYS)
    return set_error(RBOD_E_INVAL, "finish: %d candidates per query exceed %d", A.n_cap, FIN_MAX_KEYS);
  static bool configured[64] = {false};   // raising the dynamic shared-memory limit: once per device and process
  int dev = 0;
  RBOD_CUDA(cudaGetDevice(&dev));
  if (dev < 0 || dev >= 64 || !configured[dev]) {
    RBOD_CUDA(cudaFuncSetAttribute(finish_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, FIN_MAX_KEYS * 8));
    if (dev >= 0 && dev < 64) configured[dev] = true;
  }
  finish_kernel<<<(unsigned)Q, FIN_THREADS, (size_t)std::max(A.n_cap, A.dim) * 8, st>>>(A);
  RBOD_CUDA(cudaGetLastError());
  return RBOD_OK;
}

int launch_select_collected(const double* coll_score, const uint32_t* coll_idx, const int* coll_cnt,
                            const int* flag_q, int f0, int nf, int cap, int k, int metric, float* out_scores,
                            int64_t* out_rows, double* out_scores64, cudaStream_t st) {
  if (nf <= 0) return RBOD_OK;
  select_collected_kernel<<<nf, 256, 0, st>>>(coll_score, coll_idx, coll_cnt, flag_q, f0, cap, k, metric, out_scores,
                                              out_rows, out_scores64);
  RBOD_CUDA(cudaGetLastError());
  return RBOD_OK;
}

int launch_gather_flagged(const uint16_t* q16, int dp, const int* flag_q, int f0, int nf, int64_t nf_pad,
                          uint16_t* fq16, int* coll_cnt, const int* mask_of_query, int* fmask, cudaStream_t st) {
  if (nf_pad <= 0) return RBOD_OK;
  const int64_t want = (nf_pad + 7) / 8;
  gather_flagged_kernel<<<(unsigned)(want < 148 * 8 ? want : 148 * 8), 256, 0, st>>>(q16, dp, flag_q, f0, nf, nf_pad,
                                                                                    fq16, coll_cnt, mask_of_query,
                                                                                    fmask);
  RBOD_CUDA(cudaGetLastError());
  return RBOD_OK;
}

int launch_rescore_collected(const float* q, const double* q_qq, const float* master32, const uint16_t* rows16,
                             int kind16, int dim, int64_t ld32, int64_t ld16, int metric, const int* flag_q, int f0,
                             int nf, int cap, const uint32_t* coll_idx, const int* coll_cnt, double* coll_score,
                             cudaStream_t st) {
  if (nf <= 0) return RBOD_OK;
  for (int y0 = 0; y0 < nf; y0 += 32768) {   // grid.y limit
    const int ny = nf - y0 < 32768 ? nf - y0 : 32768;
    rescore_collected_kernel<<<dim3(4, (unsigned)ny), 256, 0, st>>>(
        q, q_qq, master32, rows16, kind16, dim, ld32, ld16, metric, flag_q, f0 + y0, cap, coll_idx + (size_t)y0 * cap,
        coll_cnt + y0, coll_score + (size_t)y0 * cap);
  }
  RBOD_CUDA(cudaGetLastError());
  return RBOD_OK;
}

int launch_global_cut(const float* gathered, int G, int64_t Q, int m, int k, float* out_cut2, cudaStream_t st) {
  if (Q <= 0) return RBOD_OK;
  if (G < 1 || G > 32 || m < 1 || m > K3_MAX_KC || k < 1 || (int64_t)G * m < k)
    return set_error(RBOD_E_INVAL, "global_cut: G=%d lists of %d scores for k=%d", G, m, k);
  const size_t per_warp = (size_t)G * m * 4;
  const int warps = (int)std::max<size_t>(1, std::min<size_t>(4, (48 * 1024) / per_warp));
  global_cut_kernel<<<(unsigned)((Q + warps - 1) / warps), warps * 32, per_warp * warps, st>>>(
      gathered, G, Q, m, k, reinterpret_cast<float2*>(out_cut2));
  RBOD_CUDA(cudaGetLastError());
  return RBOD_OK;
}

int launch_merge_topk(const double* scores64, const int64_t* ids, int64_t shard_stride, const int64_t* row0_host,
                      int G, int64_t Q, int k, float* out_scores, int64_t* out_ids, double* out_scores64,
                      cudaStream_t st, const double* ubound, int* flag_q, int* n_flag) {
  if (Q <= 0 || k <= 0) return RBOD_OK;
  if (G < 1 || G > 32) return set_error(RBOD_E_UNSUPPORTED, "merge_topk: G=%d outside [1, 32]", G);
  MergeRow0 r0;
  for (int g = 0; g < 32; ++g) r0.v[g] = (row0_host != nullptr && g < G) ? (long long)row0_host[g] : 0ll;
  merge_topk_kernel<<<(unsigned)((Q + 7) / 8), 256, 0, st>>>(scores64, ids, shard_stride, G, Q, k, r0, out_scores,
                                                            out_ids, out_scores64, ubound, flag_q, n_flag);
  RBOD_CUDA(cudaGetLastError());
  return RBOD_OK;
}

}  // namespace rbod
