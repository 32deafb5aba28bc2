// K3  cosine_topk -- query x gallery cosine scores on the tcgen05 tensor cores with the top-k
// selection fused into the epilogue, so the Q x N score matrix never leaves the SM.
//
// Replaces: cosine_similarity (33_run_all_experiments.py:76-77, used at :151), generalised from
// one (test vector, delegate) pair to Q queries against N stored rows, plus the top-k a Qdrant
// `search` would return.
//
// Shape of the computation (D[M=queries, N=gallery rows] = A[M,K] * B[N,K]^T, K = dim):
//   * One CTA owns 128 queries = the 128 TMEM lanes.  In variant 0 the whole 16-bit query tile
//     (128 x dp) is parked in TMEM columns [0, dp/2) for the life of a work unit and used as the
//     A operand straight from tensor memory (tcgen05.mma with A in TMEM), so the only operand
//     that streams is the gallery: HBM -> L2 -> shared memory by TMA (128-byte swizzle, boxes of
//     64 rows x 64 elements), 2 or 4 k-blocks per pipeline stage (chosen by the planner).
//   * Accumulators: 128x128 fp32 tiles (one N=128 MMA shape: measured 90% of peak per clock and
//     ~23% less energy per flop than N=64) at the top of TMEM, two buffers, so the MMA of tile j+1
//     overlaps the epilogue of tile j.  For dim > 512 the last k-blocks of the query tile live in
//     shared memory instead of TMEM to leave room for both buffers (hybrid layout); the epilogue
//     copies a tile to registers and releases its TMEM buffer before it starts selecting.
//   * Epilogue (4 warps, one thread per query row): tcgen05.ld the 128 scores of the row, compare
//     against the row's running threshold (one FMNMX per score on the fast path); survivors are
//     APPENDED to the row's candidate list in global memory (one 8-byte store, L2-resident).  When a
//     list reaches its capacity the warp prunes it cooperatively: a radix descent over the 32 lanes'
//     registers finds the kc-th best score, the list is compacted to the rows at or above it and that
//     score becomes the row's new threshold.  No shared memory is spent on candidates, so the gallery
//     pipeline keeps all of it whatever k is (round 1 kept a kc-deep heap per row in shared memory:
//     128 KB at k = 100, which cost the second accumulator buffer and ~500 cycles per insert).
//   * Work unit = (gallery slice, query tile).  Units are ordered slice-major so that CTAs
//     running at the same time stream the same gallery slice and share it through L2.
// Output: per (slice, query) a list of at least the `kc` best approximate scores of the slice with
// their row indices (unsorted, plus whatever else passed the threshold since the last prune).  The
// finish kernel (k4_topk_merge.cu) merges the slices, rescores exactly in fp64 and certifies.
// The same kernel serves DOT collections (nothing normalised) and, in its BIAS instantiation,
// EUCLID collections (a per-row -|g|^2/2 added to the scores; util/qdrant_manager.py:61-66).
//
// Warp roles (192 threads): warp 0 = TMA producer, warp 1 = TMEM allocator + MMA issuer,
// warps 2..5 = epilogue (TMEM lane quadrant = warp % 4).
// Variant 1 streams the A tile through shared memory as well (plain SS MMA); it exists to
// cross-check the TMEM-resident path.
#include "rbod_common.cuh"
#include "rbod_internal.h"

#include <cstring>

namespace rbod {

namespace {

constexpr int TMEM_COLS = 512;
constexpr int MAX_STAGES = 8;
constexpr int A_TILE_KB_BYTES = K3_TILE_M * 128;   // one k-block of a 128-row query tile in smem: 16 KB

struct alignas(64) K3Params {
  CUtensorMap tmap_b;
  CUtensorMap tmap_a;
  const uint16_t* q16;
  uint2* lists;           // [slices][q_pad][list_stride] candidate lists: {score bits, row index}
  int* list_cnt;          // [slices][q_pad] entries in each list when its unit is done
  int list_cap;           // a list is pruned back to ~kc entries once it holds this many (64, 128 or 256)
  int list_stride;        // list_cap + 128: a tile can append 128 entries before the capacity check
  int final_cap;          // lists longer than this get a last exact prune to kc entries (keeps the merge within 8192)
  const uint32_t* row_mask;   // [n_masks][mask_words] row bitmasks, or nullptr = every row allowed
  const int* mask_of_query;   // [q_pad] mask each query row reads (-1 = none), or nullptr = every row reads mask 0
  int64_t mask_words;
  const float* row_bias;  // BIAS kernels (EUCLID collections): score = q . g + row_bias[row], row_bias = -|g|^2 / 2
  uint32_t* tau_shared;   // [q_pad] per-query lower bound on the kc-th best score, as ordered keys (nullptr = off)
  const float* collect_thr;   // collect mode: [q_pad] fixed per-query thresholds; every row scoring above is recorded
  uint32_t* coll_idx;         //   [q_pad][coll_cap] recorded row indices
  int* coll_cnt;              //   [q_pad] rows recorded (may exceed coll_cap: overflow, caller falls back)
  int coll_cap;
  float* groupmax_out;        // sample mode: [slices][q_pad] row maxima over the unit's tiles (no candidate lists)
  int group_stride;           // > 0: unit `slice` visits tiles slice, slice + stride, ... (at most group_tiles of them)
  int group_tiles;
  int group_splits;           // sample mode: each group's comb is dealt round-robin to this many units (>= 1)
  float* dump;
  int64_t dump_ld;
  int64_t n_rows;
  int64_t q_valid;
  int64_t q_pad;
  int dp;
  int num_kb;
  int tiles_total;
  int num_qt;
  int slices;
  int kc;
  int num_stages;
  int variant;
  int* sync_counters;   // [groups][sync_windows] issue-progress counters (nullptr = no throttle)
  int sync_window;      // tiles per progress window
  int sync_lead;        // windows a CTA may run ahead of the slowest CTA of its group
  int sync_span;        // groups per slice (a slice's units may fall into several rounds)
  int sync_windows;     // counters per group
  int a_tmem_kb;   // k-blocks of the query tile held in TMEM; the rest sits in shared memory (resident)
  int num_acc;     // accumulator buffers (1 or 2)
  int acc_col0;    // first accumulator column in TMEM
  int debug_epi;   // bring-up only: 1 = epilogue loads the tile but selects nothing, 2 = does not even load it
  unsigned long long* prof;   // optional [16] cycle counters (option "k3_prof"): where each warp role waits
  uint32_t idesc;
};

struct K3Barriers {
  uint64_t full[MAX_STAGES];
  uint64_t empty[MAX_STAGES];
  uint64_t tfull[2];
  uint64_t tempty[2];
  uint64_t a_ready;
  uint32_t tmem_base;
  uint32_t pad;
};

// Blocking wait that, when profiling is on, adds the cycles it took to `acc` (a register of the calling role).
__device__ __forceinline__ void k3_wait(uint64_t* bar, uint32_t parity, int tag, bool prof, unsigned long long& acc) {
  if (prof) {
    const long long t0 = clock64();
    mbar_wait(bar, parity, tag);
    acc += (unsigned long long)(clock64() - t0);
  } else {
    mbar_wait(bar, parity, tag);
  }
}
enum { K3P_PROD_EMPTY = 0, K3P_PROD_THROTTLE, K3P_MMA_AREADY, K3P_MMA_TEMPTY, K3P_MMA_FULL, K3P_EPI_TFULL, K3P_EPI_PRUNE,
       K3P_CTA_CYCLES, K3P_CTAS, K3P_EPI_WARPS, K3P_PRUNES, K3P_PROD_EMPTY_FOLLOWER, K3P_PROD_ISSUE, K3P_MMA_ISSUE };

// Per-row candidate list = an append-only array of {score bits, row index} in global memory, owned by the row's
// epilogue thread for the life of a work unit.  Appending costs one 8-byte store; nothing is ordered.  When a list
// holds `list_cap` entries the whole warp prunes it: each lane takes the entries j = lane, lane + 32, ... into
// registers as order-preserving integer keys, a most-significant-bit-first radix descent (one warp-wide count per
// bit, starting at the first bit in which the keys differ at all) finds the keep-th largest key, and the entries
// at or above it are compacted to the front of the list with a ballot scan.  The descent stops as soon as at most
// keep + 16 entries survive (the threshold is then the decided prefix with zeros below, a slightly lower but still
// valid bound); `exact` runs it to the last bit and resolves score ties by the smaller row index, leaving exactly
// `keep` entries.  Returns (entries kept << 32) | threshold key: `keep` rows of this unit score at least that much.
template <int MAXCH>
__device__ __noinline__ unsigned long long k3_prune_list(uint2* lst, int n, int keep, int exact) {
  const int lane = threadIdx.x & 31;
  __syncwarp();   // the entries were written by other lanes of this warp
  uint32_t key[MAXCH], idx[MAXCH];
  uint32_t kmax = 0u, kmin = 0xffffffffu;
#pragma unroll
  for (int i = 0; i < MAXCH; ++i) {
    const int j = 32 * i + lane;
    key[i] = 0u;             // 0 is below every real key (even -inf maps to 0x007fffff)
    idx[i] = 0xffffffffu;
    if (j < n) {
      const uint2 e = __ldcg(lst + j);
      key[i] = f32_to_ordered(__uint_as_float(e.x));
      idx[i] = e.y;
      kmax = max(kmax, key[i]);
      kmin = min(kmin, key[i]);
    }
  }
  if (n <= keep) return (static_cast<unsigned long long>(static_cast<uint32_t>(n)) << 32) | f32_to_ordered(-INFINITY);
  kmax = __reduce_max_sync(FULL_MASK, kmax);
  kmin = __reduce_min_sync(FULL_MASK, kmin);
  const uint32_t diff = kmax ^ kmin;
  int b = diff ? 31 - __clz(diff) : -1;
  uint32_t prefix = diff ? (kmax & ~((2u << b) - 1u)) : kmax;   // the bits all keys share
  // invariant: the keep-th largest key is the `remaining`-th largest of the `share` keys that carry `prefix`
  int remaining = keep, share = n;
  const int slack = exact ? 0 : 16;
  while (b >= 0 && share - remaining > slack) {
    const uint32_t want = (prefix >> b) | 1u;
    int c = 0;
#pragma unroll
    for (int i = 0; i < MAXCH; ++i) c += ((key[i] >> b) == want) ? 1 : 0;
    c = __reduce_add_sync(FULL_MASK, c);
    if (c >= remaining) {
      prefix |= 1u << b;
      share = c;
    } else {
      remaining -= c;
      share -= c;
    }
    --b;
  }
  uint32_t istar = 0u;   // entries equal to `prefix` survive when ~idx >= istar
  if (share - remaining > slack) {
    // every bit is decided and more rows tie with the keep-th score than may stay: keep the `remaining` of them
    // with the smallest row index (the order the exact selection uses), found by the same descent over ~idx
    int rem2 = remaining, sh2 = share;
    for (int bb = 31; bb >= 0 && sh2 > rem2; --bb) {
      const uint32_t want = (istar >> bb) | 1u;
      int c = 0;
#pragma unroll
      for (int i = 0; i < MAXCH; ++i) c += (key[i] == prefix && ((~idx[i]) >> bb) == want) ? 1 : 0;
      c = __reduce_add_sync(FULL_MASK, c);
      if (c >= rem2) {
        istar |= 1u << bb;
        sh2 = c;
      } else {
        rem2 -= c;
        sh2 -= c;
      }
    }
  }
  int base = 0;
#pragma unroll
  for (int i = 0; i < MAXCH; ++i) {
    const bool kp = key[i] > prefix || (key[i] == prefix && (~idx[i]) >= istar);   // prefix > 0, so padding never passes
    const unsigned bal = __ballot_sync(FULL_MASK, kp);
    if (kp)
      __stcg(lst + base + __popc(bal & ((1u << lane) - 1u)),
             make_uint2(__float_as_uint(ordered_to_f32(key[i])), idx[i]));
    base += __popc(bal);
  }
  __syncwarp();
  return (static_cast<unsigned long long>(static_cast<uint32_t>(base)) << 32) | prefix;
}

__device__ __forceinline__ unsigned long long k3_prune(uint2* lst, int n, int keep, int exact, int list_cap) {
  if (list_cap <= 64) return k3_prune_list<6>(lst, n, keep, exact);
  if (list_cap <= 128) return k3_prune_list<8>(lst, n, keep, exact);
  return k3_prune_list<12>(lst, n, keep, exact);
}

// Tiles a work unit visits: t0, t0 + step, ... (n of them).  Normal launches cut the gallery into `slices`
// contiguous ranges; sample launches (group_stride > 0) give unit `slice` a strided comb of tiles, which stays
// representative when the gallery is stored in class order.
struct K3TileRange { int t0, n, step; };
__device__ __forceinline__ K3TileRange k3_unit_tiles(const K3Params& P, int slice) {
  K3TileRange r;
  if (P.group_stride > 0) {
    // unit = (group g, split s).  Group g starts g/groups of a stride in, so even one-tile groups are spread over
    // the whole gallery; its comb of group_tiles tiles is dealt round-robin to the group's splits, so a small
    // batch still spreads the sample over the whole chip.
    const int S = P.group_splits, groups = P.slices / S;
    const int g = slice / S, s = slice - g * S;
    const int t0g = (int)(((int64_t)g * P.group_stride) / groups);
    const int avail = t0g < P.tiles_total ? (P.tiles_total - t0g + P.group_stride - 1) / P.group_stride : 0;
    const int ng = min(P.group_tiles, avail);
    r.t0 = t0g + s * P.group_stride;
    r.step = P.group_stride * S;
    r.n = ng > s ? (ng - s + S - 1) / S : 0;
  } else {
    r.t0 = (int)(((int64_t)slice * P.tiles_total) / P.slices);
    r.n = (int)(((int64_t)(slice + 1) * P.tiles_total) / P.slices) - r.t0;
    r.step = 1;
  }
  return r;
}

// Geometry of one kernel flavour.
//   PAIR = 0: one CTA per 128 queries, the CTA streams whole 128-row gallery tiles.
//   PAIR = 1: a 2-CTA cluster (tcgen05 cta_group::2) owns 256 queries; each CTA holds its own 128 query
//             rows in TMEM and streams only HALF of every gallery tile (64 rows); the leader CTA issues
//             M=256 MMAs that read both halves.  L2 -> SM operand traffic per flop is halved.
//   KBS     : k-blocks (64 elements of K) per pipeline stage.  Coarser stages mean fewer barrier round trips per
//             tile -- measured on the headline shape, same box: 1 -> 1019 TF/s, 2 -> 1209-1218, 4 -> 1264 -- but a
//             later first MMA and half as many stages in flight, which costs small, HBM-bound batches 5-10 %.
template <int VARIANT, int PAIR, int KBS_>
struct K3Geom {
  static constexpr int BOX_N = PAIR ? K3_TILE_N / 2 : K3_TILE_N;   // gallery rows this CTA loads per tile
  static constexpr int B_KB_BYTES = BOX_N * 128;
  static constexpr int A_KB_BYTES = VARIANT == 1 ? A_TILE_KB_BYTES : 0;   // streamed A (variant 1 only)
  static constexpr int KBS = KBS_;                                 // k-blocks per pipeline stage
  static constexpr int STAGE_BYTES = KBS * (B_KB_BYTES + A_KB_BYTES);
  static constexpr int Q_PER_UNIT = PAIR ? 2 * K3_TILE_M : K3_TILE_M;
  static constexpr uint32_t EPI_ARRIVALS = PAIR ? 8 : 4;   // one arrival per epilogue warp
};

// Issues the MMAs of one full pipeline stage as straight-line code: per MMA one uniform add for the
// A address / descriptor and one for the B descriptor.  A_SMEM: the A operand of this stage comes from
// shared memory (streamed tile in variant 1, resident tail of the query tile otherwise).
template <int VARIANT, int PAIR, int KBS, int A_SMEM>
__device__ __forceinline__ void issue_full_stage(uint32_t d_tmem, uint32_t a_tmem0, uint64_t adesc, uint64_t bdesc,
                                                 uint32_t idesc, uint32_t first_accumulate) {
  using G = K3Geom<VARIANT, PAIR, KBS>;
#pragma unroll
  for (int j = 0; j < G::KBS; ++j) {
#pragma unroll
    for (int kk = 0; kk < 4; ++kk) {
      const uint32_t accumulate = (j == 0 && kk == 0) ? first_accumulate : 1u;
      const uint64_t bd = bdesc + (uint64_t)(j * (G::B_KB_BYTES >> 4) + kk * 2);
      const uint32_t at = a_tmem0 + (uint32_t)((j * 4 + kk) * 8);
      const uint64_t ad = adesc + (uint64_t)(j * (A_TILE_KB_BYTES >> 4) + kk * 2);
      if (A_SMEM) {
        if (PAIR) mma_f16_ss_pair(d_tmem, ad, bd, idesc, accumulate);
        else mma_f16_ss(d_tmem, ad, bd, idesc, accumulate);
      } else {
        if (PAIR) mma_f16_ts_pair(d_tmem, at, bd, idesc, accumulate);
        else mma_f16_ts(d_tmem, at, bd, idesc, accumulate);
      }
    }
  }
}

// BIAS = 1 (EUCLID collections): the epilogue adds a per-gallery-row term to every score before anything looks at
// it, so thresholds, candidate lists, the collecting pass and the sampled pre-pass all work on
// q . g - |g|^2 / 2 = (|q|^2 - |q - g|^2) / 2, which orders rows by Euclidean distance.
template <int VARIANT, int PAIR, int KBS, int BIAS>
__global__ void __launch_bounds__(K3_THREADS, 1) k3_cosine_topk_kernel(const __grid_constant__ K3Params P) {
  using G = K3Geom<VARIANT, PAIR, KBS>;
  extern __shared__ uint8_t smem_raw[];
  // 1024-byte alignment for the 128B-swizzled operand tiles
  const uint32_t raw_addr = smem_u32(smem_raw);
  uint8_t* smem = smem_raw + ((1024u - (raw_addr & 1023u)) & 1023u);

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  const uint32_t rank = PAIR ? cluster_ctarank() : 0u;          // 0 = leader of the pair
  const int worker = PAIR ? (int)(blockIdx.x >> 1) : (int)blockIdx.x;
  const int num_workers = PAIR ? (int)(gridDim.x >> 1) : (int)gridDim.x;

  uint8_t* stage_base = smem;
  uint8_t* a_tail = smem + (size_t)P.num_stages * G::STAGE_BYTES;       // resident query-tile tail (k-blocks >= a_tmem_kb)
  const int tail_kb = VARIANT == 1 ? 0 : (P.num_kb - P.a_tmem_kb);
  K3Barriers* bars = reinterpret_cast<K3Barriers*>(a_tail + (size_t)tail_kb * A_TILE_KB_BYTES);

  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&P.tmap_b);
    if (VARIANT == 1) tma_prefetch_desc(&P.tmap_a);
    for (int s = 0; s < P.num_stages; ++s) {
      mbar_init(&bars->full[s], 1);   // CTA pair: the leader's expect_tx covers both halves, the follower only sends bytes
      mbar_init(&bars->empty[s], 1);
    }
    for (int b = 0; b < 2; ++b) {
      mbar_init(&bars->tfull[b], 1);
      mbar_init(&bars->tempty[b], G::EPI_ARRIVALS);
    }
    mbar_init(&bars->a_ready, G::EPI_ARRIVALS);
    fence_mbar_init();
  }
  if (warp == 1) {
    if (PAIR) tmem_alloc_pair(&bars->tmem_base, TMEM_COLS);
    else tmem_alloc(&bars->tmem_base, TMEM_COLS);
  }
  tc_fence_before();
  if (PAIR) cluster_sync_all(); else __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = bars->tmem_base;

  const int num_units = P.slices * P.num_qt;
  const int num_chunks = (P.num_kb + G::KBS - 1) / G::KBS;

  if (warp == 0) {
    // ================================ TMA producer ================================
    // The whole warp walks the schedule (warp-uniform control flow); one elected lane issues.
    int stage = 0;
    uint32_t phase = 0;
    const bool prof = P.prof != nullptr;
    unsigned long long w_empty = 0ull, w_throttle = 0ull, w_issue = 0ull;
    const long long t_start = prof ? clock64() : 0ll;
    for (int u = worker; u < num_units; u += num_workers) {
      const int slice = u / P.num_qt, qt = u - slice * P.num_qt;
      const K3TileRange tr = k3_unit_tiles(P, slice);
      // L2 sharing throttle: the CTAs that stream this slice in this round form a group; nobody
      // issues window w before every member has issued window w - lead.  That keeps the group's
      // working set (lead + 1 windows) hot in L2, so each gallery tile is fetched from HBM once per
      // group instead of once per CTA.  Dependencies only point to the same or earlier rounds.
      int* cnt = nullptr;
      int gsize = 0;
      if (P.sync_counters != nullptr && rank == 0) {
        const int round = u / num_workers;
        const int first_round = (slice * P.num_qt) / num_workers;
        const int lo = max(slice * P.num_qt, round * num_workers);
        const int hi = min((slice + 1) * P.num_qt, (round + 1) * num_workers);
        gsize = hi - lo;
        cnt = P.sync_counters + ((size_t)slice * P.sync_span + (round - first_round)) * P.sync_windows;
      }
      for (int ti = 0; ti < tr.n; ++ti) {
        const int t = tr.t0 + ti * tr.step;
        if (cnt != nullptr && gsize > 1 && ti % P.sync_window == 0) {
          const int w = ti / P.sync_window;
          if (elect_one()) {
            if (w > 0) {
              __threadfence();
              atomicAdd(cnt + (w - 1), 1);
            }
            if (w >= P.sync_lead) {
              const volatile int* flag = cnt + (w - P.sync_lead);
              if (*flag < gsize) {
                const long long c0 = prof ? clock64() : 0ll;
                const uint64_t w0 = global_timer_ns();
                while (*flag < gsize) {
                  __nanosleep(128);
                  if (global_timer_ns() - w0 > 4000000000ull) {
                    printf("rbod: L2 throttle watchdog: block %d unit %d window %d count %d/%d\n", (int)blockIdx.x, u,
                           w, *flag, gsize);
                    __trap();
                  }
                }
                if (prof) w_throttle += (unsigned long long)(clock64() - c0);
              }
            }
          }
          __syncwarp();
        }
        for (int ch = 0; ch < num_chunks; ++ch) {
          const int kb0 = ch * G::KBS;
          const int nkb = min(G::KBS, P.num_kb - kb0);
          k3_wait(&bars->empty[stage], phase ^ 1u, 1, prof, w_empty);
          const long long i0 = prof ? clock64() : 0ll;
          if (elect_one()) {
            uint8_t* sb = stage_base + (size_t)stage * G::STAGE_BYTES;
            if (PAIR) {
              // Both halves report their bytes to the leader's barrier, which expects the whole tile; the leader's
              // arrive.expect_tx is the barrier's only arrival.  (Bytes of the follower may land before the leader has
              // armed the phase: the transaction count goes negative for a moment, the phase cannot complete before
              // the leader's arrival.  A second, remote arrival from the follower -- release semantics at cluster
              // scope -- kept the follower's producer busy 95 % of the time and starved the MMA issuer for half of it.)
              const uint32_t full_leader = mapa_u32(smem_u32(&bars->full[stage]), 0);
              if (rank == 0) mbar_arrive_expect_tx(&bars->full[stage], 2u * nkb * G::B_KB_BYTES);
              for (int j = 0; j < nkb; ++j)
                tma_load_2d_pair(sb + j * G::B_KB_BYTES, &P.tmap_b, full_leader, (kb0 + j) * K3_KBLOCK,
                                 t * K3_TILE_N + (int)rank * G::BOX_N);
            } else {
              mbar_arrive_expect_tx(&bars->full[stage], nkb * (G::B_KB_BYTES + G::A_KB_BYTES));
              for (int j = 0; j < nkb; ++j)
                tma_load_2d(sb + j * G::B_KB_BYTES, &P.tmap_b, &bars->full[stage], (kb0 + j) * K3_KBLOCK,
                            t * K3_TILE_N);
              if (VARIANT == 1) {
                uint8_t* sa = sb + G::KBS * G::B_KB_BYTES;
                for (int j = 0; j < nkb; ++j)
                  tma_load_2d(sa + j * G::A_KB_BYTES, &P.tmap_a, &bars->full[stage], (kb0 + j) * K3_KBLOCK,
                              qt * K3_TILE_M);
              }
            }
          }
          __syncwarp();
          if (prof) w_issue += (unsigned long long)(clock64() - i0);
          if (++stage == P.num_stages) { stage = 0; phase ^= 1u; }
        }
      }
    }
    if (prof && lane == 0) {
      atomicAdd(P.prof + (rank == 0 ? K3P_PROD_EMPTY : K3P_PROD_EMPTY_FOLLOWER), w_empty);
      atomicAdd(P.prof + K3P_PROD_ISSUE, w_issue);
      atomicAdd(P.prof + K3P_PROD_THROTTLE, w_throttle);
      atomicAdd(P.prof + K3P_CTA_CYCLES, (unsigned long long)(clock64() - t_start));
      atomicAdd(P.prof + K3P_CTAS, 1ull);
    }
  } else if (warp == 1) {
    // ================================ MMA issuer ==================================
    // Warp-converged loop; elect.sync picks the issuing lane so descriptors stay in uniform registers.
    // In a CTA pair only the leader issues (its MMAs drive both SMs).
    if (rank == 0) {
      int stage = 0;
      uint32_t phase = 0;
      int acc = 0;
      uint32_t acc_phase = 0, unit_par = 0;
      const bool prof = P.prof != nullptr;
      unsigned long long w_aready = 0ull, w_tempty = 0ull, w_full = 0ull, w_mma = 0ull;
      const uint32_t tmem_b = __shfl_sync(FULL_MASK, tmem_base, 0);
      const uint32_t smem_stage0 = __shfl_sync(FULL_MASK, smem_u32(stage_base), 0);
      const uint32_t smem_tail0 = __shfl_sync(FULL_MASK, smem_u32(a_tail), 0);
      const uint64_t desc_hi = make_smem_desc_sw128(0);  // everything except the start address
      for (int u = worker; u < num_units; u += num_workers) {
        const int slice = u / P.num_qt;
        const K3TileRange tr = k3_unit_tiles(P, slice);
        if (VARIANT == 0) {
          k3_wait(&bars->a_ready, unit_par, 2, prof, w_aready);
          unit_par ^= 1u;
          tc_fence_after();
        }
        for (int ti = 0; ti < tr.n; ++ti) {
          k3_wait(&bars->tempty[acc], acc_phase ^ 1u, 3, prof, w_tempty);
          tc_fence_after();
          const uint32_t d_tmem = tmem_b + (uint32_t)(P.acc_col0 + acc * K3_TILE_N);
          for (int ch = 0; ch < num_chunks; ++ch) {
            const int kb0 = ch * G::KBS;
            const int nkb = min(G::KBS, P.num_kb - kb0);
            k3_wait(&bars->full[stage], phase, 4, prof, w_full);
            const long long m0 = prof ? clock64() : 0ll;
            tc_fence_after();
            if (elect_one()) {
              const uint32_t sb = smem_stage0 + (uint32_t)stage * (uint32_t)G::STAGE_BYTES;
              const uint64_t bdesc = desc_hi | (uint64_t)((sb >> 4) & 0x3fffu);
              const uint32_t first = ch > 0 ? 1u : 0u;
              // A operand of this stage: streamed tile (variant 1), TMEM columns, or the smem-resident tail
              const bool a_smem = VARIANT == 1 || kb0 >= P.a_tmem_kb;
              const uint32_t sa = VARIANT == 1 ? sb + G::KBS * G::B_KB_BYTES
                                               : smem_tail0 + (uint32_t)(kb0 - P.a_tmem_kb) * (uint32_t)A_TILE_KB_BYTES;
              const uint64_t adesc = desc_hi | (uint64_t)((sa >> 4) & 0x3fffu);
              const uint32_t a_tmem0 = tmem_b + (uint32_t)kb0 * 32u;   // 4 K=16 steps x 8 columns per k-block
              if (nkb == G::KBS) {
                if (a_smem) issue_full_stage<VARIANT, PAIR, KBS, 1>(d_tmem, a_tmem0, adesc, bdesc, P.idesc, first);
                else issue_full_stage<VARIANT, PAIR, KBS, 0>(d_tmem, a_tmem0, adesc, bdesc, P.idesc, first);
              } else {
                for (int j = 0; j < nkb; ++j) {
                  const bool js = VARIANT == 1 || (kb0 + j) >= P.a_tmem_kb;
                  for (int kk = 0; kk < 4; ++kk) {
                    const uint32_t accumulate = (ch > 0 || j > 0 || kk > 0) ? 1u : 0u;
                    const uint64_t bd = bdesc + (uint64_t)(j * (G::B_KB_BYTES >> 4) + kk * 2);
                    const uint32_t at = a_tmem0 + (uint32_t)((j * 4 + kk) * 8);
                    const uint64_t ad = adesc + (uint64_t)(j * (A_TILE_KB_BYTES >> 4) + kk * 2);
                    if (js) {
                      if (PAIR) mma_f16_ss_pair(d_tmem, ad, bd, P.idesc, accumulate);
                      else mma_f16_ss(d_tmem, ad, bd, P.idesc, accumulate);
                    } else {
                      if (PAIR) mma_f16_ts_pair(d_tmem, at, bd, P.idesc, accumulate);
                      else mma_f16_ts(d_tmem, at, bd, P.idesc, accumulate);
                    }
                  }
                }
              }
              if (PAIR) {
                mma_commit_pair(&bars->empty[stage], 3);
                if (ch == num_chunks - 1) mma_commit_pair(&bars->tfull[acc], 3);
              } else {
                mma_commit(&bars->empty[stage]);
                if (ch == num_chunks - 1) mma_commit(&bars->tfull[acc]);
              }
            }
            __syncwarp();
            if (prof) w_mma += (unsigned long long)(clock64() - m0);
            if (++stage == P.num_stages) { stage = 0; phase ^= 1u; }
          }
          if (++acc == P.num_acc) { acc = 0; acc_phase ^= 1u; }
        }
      }
      if (prof && lane == 0) {
        atomicAdd(P.prof + K3P_MMA_AREADY, w_aready);
        atomicAdd(P.prof + K3P_MMA_TEMPTY, w_tempty);
        atomicAdd(P.prof + K3P_MMA_FULL, w_full);
        atomicAdd(P.prof + K3P_MMA_ISSUE, w_mma);
      }
    }
  } else {
    // ================================ epilogue ====================================
    const int quad = warp & 3;
    const int wrow0 = quad * 32;
    const int row = wrow0 + lane;
    const uint32_t lane_addr = static_cast<uint32_t>(wrow0) << 16;
    const int kc = P.kc;
    int acc = 0;
    uint32_t acc_phase = 0;
    const bool prof = P.prof != nullptr;
    unsigned long long w_tfull = 0ull, w_prune = 0ull, n_prune = 0ull;
    // barriers the MMA issuer waits on live in the leader CTA
    const uint32_t a_ready_leader = PAIR ? mapa_u32(smem_u32(&bars->a_ready), 0) : 0u;
    const uint32_t tempty_leader0 = PAIR ? mapa_u32(smem_u32(&bars->tempty[0]), 0) : 0u;
    const uint32_t tempty_leader1 = PAIR ? mapa_u32(smem_u32(&bars->tempty[1]), 0) : 0u;

    for (int u = worker; u < num_units; u += num_workers) {
      const int slice = u / P.num_qt, qt = u - slice * P.num_qt;
      const K3TileRange tr = k3_unit_tiles(P, slice);
      const int64_t q_unit0 = (int64_t)qt * G::Q_PER_UNIT + (int64_t)rank * K3_TILE_M;   // first query row of this CTA
      const int64_t qg = q_unit0 + row;

      if (VARIANT == 0) {
        // Park this thread's query row.  K-blocks < a_tmem_kb go to TMEM (lane = row, column c holds
        // elements 2c, 2c+1); the rest goes to shared memory in the K-major 128B-swizzled layout the MMA
        // descriptor expects: row r at r*128 B inside its k-block, 16-byte chunk c at position c ^ (r & 7).
        const uint4* src = reinterpret_cast<const uint4*>(P.q16 + qg * P.dp);
        const int n16_tmem = P.a_tmem_kb * 4;
        for (int c = 0; c < n16_tmem; ++c) {
          const uint4 x0 = __ldg(src + 2 * c), x1 = __ldg(src + 2 * c + 1);
          const uint32_t r[8] = {x0.x, x0.y, x0.z, x0.w, x1.x, x1.y, x1.z, x1.w};
          tmem_st_32x32b_x8(tmem_base + lane_addr + (uint32_t)c * 8u, r);
        }
        if (tail_kb > 0) {
          for (int kb = 0; kb < tail_kb; ++kb) {
            uint8_t* dst = a_tail + (size_t)kb * A_TILE_KB_BYTES + row * 128;
            const uint4* s8 = src + (size_t)(P.a_tmem_kb + kb) * 8;
#pragma unroll
            for (int c = 0; c < 8; ++c)
              *reinterpret_cast<uint4*>(dst + ((c ^ (row & 7)) << 4)) = __ldg(s8 + c);
          }
          fence_proxy_async_smem();   // generic-proxy writes -> visible to the tensor core's async proxy
        }
        tmem_st_wait();
        tc_fence_before();
        __syncwarp();
        if (lane == 0) {
          if (PAIR) mbar_arrive_cluster(a_ready_leader); else mbar_arrive(&bars->a_ready);
        }
      }
      // Threshold shared between the units (gallery slices) of one query.  A unit publishes the threshold a prune
      // of its list leaves behind: kc rows of the unit score at least that much, so no row below it can be among
      // the kc best of the whole gallery, whichever slice it sits in.  Other units start from, and periodically
      // re-read, the best published bound, which removes almost all list traffic after the first slice of a query
      // has warmed up.  Rows that only pad the query tile never append anything.
      uint32_t* tau_cell = P.tau_shared != nullptr ? P.tau_shared + qg : nullptr;
      float tau = tau_cell != nullptr ? ordered_to_f32(ld_relaxed_u32(tau_cell)) : -INFINITY;
      float tau_published = tau;
      const bool collect = P.collect_thr != nullptr;
      if (collect) tau = qg < P.q_valid ? P.collect_thr[qg] : INFINITY;
      else if (qg >= P.q_valid) tau = INFINITY;
      // this row's candidate list (select mode only): `wp` is where the next survivor goes
      uint2* const my_list = P.lists + ((size_t)slice * P.q_pad + qg) * P.list_stride;
      uint2* wp = my_list;

      const bool groupmax = P.groupmax_out != nullptr;
      float gmax_run = -INFINITY;
      for (int ti = 0; ti < tr.n; ++ti) {
        const int t = tr.t0 + ti * tr.step;
        if (tau_cell != nullptr && (ti & (K3_TAU_REFRESH - 1)) == K3_TAU_REFRESH - 1)
          tau = fmaxf(tau, ordered_to_f32(ld_relaxed_u32(tau_cell)));
        k3_wait(&bars->tfull[acc], acc_phase, 5, prof, w_tfull);
        tc_fence_after();
        if (P.debug_epi == 2) {
          tc_fence_before();
          __syncwarp();
          if (lane == 0) {
            if (PAIR) mbar_arrive_cluster_relaxed(acc == 0 ? tempty_leader0 : tempty_leader1);
            else mbar_arrive(&bars->tempty[acc]);
          }
          if (++acc == P.num_acc) { acc = 0; acc_phase ^= 1u; }
          continue;
        }
        float v[K3_TILE_N];
        {
          const uint32_t taddr = tmem_base + lane_addr + (uint32_t)(P.acc_col0 + acc * K3_TILE_N);
          uint32_t raw[4][32];
#pragma unroll
          for (int h = 0; h < 4; ++h) tmem_ld_32x32b_x32(taddr + 32u * h, raw[h]);
          tmem_ld_wait();
          tc_fence_before();
          __syncwarp();
          // TMEM tile is in registers: hand it back to the MMA issuer (one arrival per warp)
          if (lane == 0) {
            if (PAIR) mbar_arrive_cluster_relaxed(acc == 0 ? tempty_leader0 : tempty_leader1);
            else mbar_arrive(&bars->tempty[acc]);
          }
#pragma unroll
          for (int h = 0; h < 4; ++h)
#pragma unroll
            for (int c = 0; c < 32; ++c) v[h * 32 + c] = __uint_as_float(raw[h][c]);
        }
        if (++acc == P.num_acc) { acc = 0; acc_phase ^= 1u; }
        const int64_t col0 = (int64_t)t * K3_TILE_N;
        if (BIAS) {
          // the same 512 bytes for all four epilogue warps: L1-resident after the first touch (the array is
          // allocated in whole tiles, rows beyond n_rows are masked below)
          const float4* bp = reinterpret_cast<const float4*>(P.row_bias + col0);
#pragma unroll
          for (int c4 = 0; c4 < K3_TILE_N / 4; ++c4) {
            const float4 b4 = __ldg(bp + c4);
            v[4 * c4 + 0] += b4.x;
            v[4 * c4 + 1] += b4.y;
            v[4 * c4 + 2] += b4.z;
            v[4 * c4 + 3] += b4.w;
          }
        }

        if (P.dump != nullptr && qg < P.q_valid) {
#pragma unroll
          for (int c = 0; c < K3_TILE_N; ++c)
            if (col0 + c < P.n_rows) P.dump[qg * P.dump_ld + col0 + c] = v[c];
        }

        if (col0 + K3_TILE_N > P.n_rows || P.row_mask != nullptr) {
          // the mask this row's query reads (index into P.row_mask), -1 = none; pad rows of the tile read none.  Looked
          // up per tile (an L1 hit) rather than held in a register across the tile loop, which is at its register limit.
          const int mask_id = P.mask_of_query == nullptr ? 0 : (qg < P.q_valid ? __ldg(P.mask_of_query + qg) : -1);
#pragma unroll
          for (int half = 0; half < 2; ++half) {
            const int64_t c0 = col0 + 64 * half;
            uint64_t allow = ~0ull;
            if (c0 + 64 > P.n_rows) {
              const int64_t valid = P.n_rows - c0;
              allow = valid <= 0 ? 0ull : (valid >= 64 ? ~0ull : ((1ull << valid) - 1ull));
            }
            if (P.row_mask != nullptr && mask_id >= 0) {
              // one broadcast address per warp with a shared mask; per-query masks read the row's own words (L1 / L2)
              const uint32_t* mask = P.row_mask + (int64_t)mask_id * P.mask_words;
              const int64_t w0 = c0 >> 5;
              const int64_t nwords = (P.n_rows + 31) >> 5;
              const uint64_t lo = w0 < nwords ? mask[w0] : 0u;
              const uint64_t hi = (w0 + 1) < nwords ? mask[w0 + 1] : 0u;
              allow &= (lo | (hi << 32));
            }
#pragma unroll
            for (int c = 0; c < 64; ++c)
              if (!((allow >> c) & 1ull)) v[64 * half + c] = -INFINITY;
          }
        }

        // group maxima (16 columns each) -> row maximum; almost always everything is below the threshold
        float gm[K3_TILE_N / 16];
#pragma unroll
        for (int gi = 0; gi < K3_TILE_N / 16; ++gi) {
          float a = fmaxf(v[16 * gi], v[16 * gi + 1]);
#pragma unroll
          for (int c = 2; c < 16; ++c) a = fmaxf(a, v[16 * gi + c]);
          gm[gi] = a;
        }
        float m = gm[0];
#pragma unroll
        for (int gi = 1; gi < K3_TILE_N / 16; ++gi) m = fmaxf(m, gm[gi]);
        if (P.debug_epi == 1) {
          if (m == 12345.678f) tau = m;   // keep the loads and maxima alive
          continue;
        }
        if (groupmax) {
          gmax_run = fmaxf(gmax_run, m);
          continue;
        }
        if (collect) {
          // second pass over uncertified queries: record every row above the query's fixed threshold
          if (m > tau) {
#pragma unroll
            for (int gi = 0; gi < K3_TILE_N / 16; ++gi) {
              if (gm[gi] > tau) {
#pragma unroll
                for (int c = 0; c < 16; ++c)
                  if (v[16 * gi + c] > tau) {
                    const int slot = atomicAdd(P.coll_cnt + qg, 1);
                    if (slot < P.coll_cap) P.coll_idx[(size_t)qg * P.coll_cap + slot] = (uint32_t)(col0 + 16 * gi + c);
                  }
              }
            }
          }
          continue;
        }
        // Select mode.  The branches are warp-uniform (votes), the appends inside are predicated stores: what a
        // tile costs depends on how many 16-column groups hold a survivor in ANY of the warp's 32 rows, not on the
        // number of survivors.
        if (__any_sync(FULL_MASK, m > tau)) {
#pragma unroll
          for (int gi = 0; gi < K3_TILE_N / 16; ++gi) {
            if (__any_sync(FULL_MASK, gm[gi] > tau)) {
#pragma unroll
              for (int c = 0; c < 16; ++c) {
                const float s = v[16 * gi + c];
                if (s > tau) {
                  __stcg(wp, make_uint2(__float_as_uint(s), (uint32_t)(col0 + 16 * gi + c)));
                  ++wp;
                }
              }
            }
          }
          const int cnt = (int)(wp - my_list);
          unsigned need = __ballot_sync(FULL_MASK, cnt >= P.list_cap);
          const long long p0 = (prof && need) ? clock64() : 0ll;
          if (prof) n_prune += __popc(need);
          while (need) {
            const int L = __ffs(need) - 1;
            need &= need - 1;
            const int n = __shfl_sync(FULL_MASK, cnt, L);
            uint2* lst = P.lists + ((size_t)slice * P.q_pad + (q_unit0 + wrow0 + L)) * P.list_stride;
            const unsigned long long r = k3_prune(lst, n, kc, 0, P.list_cap);
            if (lane == L) {
              wp = my_list + (int)(r >> 32);
              tau = fmaxf(tau, ordered_to_f32((uint32_t)r));
              if (tau_cell != nullptr && tau > tau_published) {
                atomicMax(tau_cell, f32_to_ordered(tau));
                tau_published = tau;
              }
            }
          }
          if (prof && p0) w_prune += (unsigned long long)(clock64() - p0);
        }
      }

      // unit done
      if (groupmax) P.groupmax_out[(size_t)slice * P.q_pad + qg] = gmax_run;
      if (!collect && !groupmax) {
        // lists the merge could not hold get a last, exact prune to kc entries; the others stay as they are
        int cnt = (int)(wp - my_list);
        unsigned need = __ballot_sync(FULL_MASK, cnt > P.final_cap);
        while (need) {
          const int L = __ffs(need) - 1;
          need &= need - 1;
          const int n = __shfl_sync(FULL_MASK, cnt, L);
          uint2* lst = P.lists + ((size_t)slice * P.q_pad + (q_unit0 + wrow0 + L)) * P.list_stride;
          const unsigned long long r = k3_prune(lst, n, kc, 1, P.list_cap);
          if (lane == L) cnt = (int)(r >> 32);
        }
        if (qg < P.q_valid) P.list_cnt[(size_t)slice * P.q_pad + qg] = cnt;
      }
    }
    if (prof && lane == 0) {
      atomicAdd(P.prof + K3P_EPI_TFULL, w_tfull);
      atomicAdd(P.prof + K3P_EPI_PRUNE, w_prune);
      atomicAdd(P.prof + K3P_EPI_WARPS, 1ull);
      atomicAdd(P.prof + K3P_PRUNES, n_prune);
    }
  }

  tc_fence_before();
  if (PAIR) cluster_sync_all(); else __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    if (PAIR) tmem_dealloc_pair(tmem_base, TMEM_COLS);
    else tmem_dealloc(tmem_base, TMEM_COLS);
  }
}

// One warp per query: |q|^2 in fp64, (unit) query rounded to the 16-bit operand type, and
// dq = || fp(q16) - target ||_2 (the query's share of the certification margin), target = q/|q| (COSINE) or q (DOT).
__global__ void __launch_bounds__(256)
prep_queries_kernel(const float* __restrict__ q, int64_t Q, int64_t q_pad, int dim, int dp, int kind16, int normalize,
                    uint16_t* __restrict__ q16, float* __restrict__ q_dq, double* __restrict__ q_qq,
                    uint32_t* __restrict__ tau_shared) {
  const int lane = threadIdx.x & 31;
  const int64_t w0 = (int64_t)blockIdx.x * 8 + (threadIdx.x >> 5);
  const int64_t nw = (int64_t)gridDim.x * 8;
  for (int64_t i = w0; i < q_pad; i += nw) {
    uint16_t* dst = q16 + i * dp;
    if (lane == 0 && tau_shared != nullptr) tau_shared[i] = f32_to_ordered(-INFINITY);
    if (i >= Q) {
      for (int c = lane; c < dp; c += 32) dst[c] = 0;
      continue;
    }
    const float* src = q + i * dim;
    double ss = 0.0;
    for (int c = lane; c < dim; c += 32) {
      const double x = (double)src[c];
      ss = fma(x, x, ss);
    }
    ss = warp_sum_f64(ss);
    // COSINE: the operand is the unit query; DOT: the query itself (fp16 operands saturate instead of overflowing,
    // the clamp error lands in dq like any other rounding error)
    const double r = normalize ? (ss > 0.0 ? 1.0 / sqrt(ss) : 0.0) : 1.0;
    double dd = 0.0;
    for (int c = lane; c < dp; c += 32) {
      uint16_t h = 0;
      if (c < dim) {
        const double u = (double)src[c] * r;
        float uf = (float)u;
        if (kind16 == 2) uf = fminf(fmaxf(uf, -65504.0f), 65504.0f);
        h = f32_to_h16(uf, kind16);
        const double e = (double)h16_to_f32(h, kind16) - u;
        dd = fma(e, e, dd);
      }
      dst[c] = h;
    }
    dd = warp_sum_f64(dd);
    if (lane == 0) {
      q_dq[i] = (float)(sqrt(dd) * 1.000001 + 1e-12);
      q_qq[i] = ss;
    }
  }
}

typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

EncodeTiledFn get_encode_fn() {
  static EncodeTiledFn fn = nullptr;
  if (fn) return fn;
  void* p = nullptr;
  cudaDriverEntryPointQueryResult qres;
  if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &qres) != cudaSuccess ||
      qres != cudaDriverEntryPointSuccess)
    return nullptr;
  fn = reinterpret_cast<EncodeTiledFn>(p);
  return fn;
}

}  // namespace

// [rows, dp] 16-bit row-major -> 2D map with box {64 elements, box_rows}, 128-byte swizzle.
int make_tmap_2d_sw128(CUtensorMap* out, const void* base, int64_t rows, int dp, int box_rows) {
  EncodeTiledFn fn = get_encode_fn();
  if (!fn) return set_error(RBOD_E_IO, "cuTensorMapEncodeTiled entry point not available");
  cuuint64_t gdim[2] = {(cuuint64_t)dp, (cuuint64_t)rows};
  cuuint64_t gstride[1] = {(cuuint64_t)dp * 2};
  cuuint32_t box[2] = {(cuuint32_t)K3_KBLOCK, (cuuint32_t)box_rows};
  cuuint32_t estr[2] = {1, 1};
  CUresult rc = fn(out, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, const_cast<void*>(base), gdim, gstride, box, estr,
                   CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                   CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (rc != CUDA_SUCCESS) return set_error(RBOD_E_IO, "cuTensorMapEncodeTiled failed with CUresult %d", (int)rc);
  return RBOD_OK;
}

static size_t k3_stage_bytes(int variant, int kbs) {
  if (variant == 1) return (size_t)K3Geom<1, 0, 2>::STAGE_BYTES;
  if (variant == 2) return kbs == 4 ? (size_t)K3Geom<0, 1, 4>::STAGE_BYTES : (size_t)K3Geom<0, 1, 2>::STAGE_BYTES;
  return kbs == 4 ? (size_t)K3Geom<0, 0, 4>::STAGE_BYTES : (size_t)K3Geom<0, 0, 2>::STAGE_BYTES;
}

size_t k3_smem_bytes(int variant, int kbs, int num_stages, int tail_kb) {
  return 1024 + (size_t)num_stages * k3_stage_bytes(variant, kbs) + (size_t)tail_kb * A_TILE_KB_BYTES +
         sizeof(K3Barriers);
}

// Chooses where the query tile lives and how deep the gallery pipeline is.
//   dp <= 512            : whole tile in TMEM (<= 256 columns), two accumulator buffers.
//   dp  > 512, room left : first 8 k-blocks in TMEM, the tail resident in shared memory, two buffers.
//   dp  > 512, smem short: whole tile in TMEM (384 columns), one accumulator buffer.
// `want_kbs` = 4 asks for the coarse 4-k-block stages of the single-CTA kernel.  Candidate lists live in global
// memory, so the plan does not depend on k.
int k3_plan(int variant, int want_kbs, int dp, int smem_optin, int allow_hybrid, int* num_stages,
            int* a_tmem_kb, int* kbs_out, size_t* smem_bytes) {
  const int num_kb = dp / K3_KBLOCK;
  auto attempt = [&](int kbs, int min_stages_hybrid, int* st_out, int* tmem_out, int* tail_out) -> bool {
    auto fit = [&](int tail_kb) {
      int st = MAX_STAGES;
      while (st > 0 && k3_smem_bytes(variant, kbs, st, tail_kb) > (size_t)smem_optin) --st;
      return st;
    };
    int tmem_kb = num_kb, tail = 0;
    if (variant == 1) {
      tmem_kb = 0;
    } else if (num_kb > 8 && allow_hybrid) {
      if (fit(num_kb - 8) >= min_stages_hybrid) { tmem_kb = 8; tail = num_kb - 8; }
    }
    const int st = fit(tail);
    *st_out = st;
    *tmem_out = tmem_kb;
    *tail_out = tail;
    return !(st < 1 || (variant != 1 && st < 2));
  };
  int st = 0, tmem_kb = 0, tail = 0, kbs = variant == 2 ? 4 : 2;
  bool ok = false;
  if (variant == 2 && want_kbs == 2) {
    ok = attempt(2, 2, &st, &tmem_kb, &tail);
    if (ok) kbs = 2;
  }
  if (!ok && variant == 0 && want_kbs == 4) {
    ok = attempt(4, 2, &st, &tmem_kb, &tail);
    // two accumulator buffers matter more than coarse stages: never trade the hybrid layout for them
    if (ok && num_kb > 8 && allow_hybrid && tail == 0) ok = false;
    if (ok) kbs = 4;
  }
  if (!ok) {
    kbs = variant == 2 ? 4 : 2;
    ok = attempt(kbs, variant == 2 ? 2 : 3, &st, &tmem_kb, &tail);
  }
  if (!ok)
    return set_error(RBOD_E_UNSUPPORTED, "search: variant %d with %d columns does not fit shared memory", variant, dp);
  *num_stages = st;
  *a_tmem_kb = tmem_kb;
  *kbs_out = kbs;
  *smem_bytes = k3_smem_bytes(variant, kbs, st, tail);
  return RBOD_OK;
}

int k3_box_rows(int variant) { return variant == 2 ? K3Geom<0, 1, 4>::BOX_N : K3_TILE_N; }

int k3_configure(int device) {
  // once per device and process: the four attribute calls cost ~40 us, which a sharded search pays on every call
  static int cached_optin[64] = {0};
  if (device >= 0 && device < 64 && cached_optin[device] > 0) return cached_optin[device];
  int optin = 0;
  RBOD_CUDA(cudaDeviceGetAttribute(&optin, cudaDevAttrMaxSharedMemoryPerBlockOptin, device));
  RBOD_CUDA(cudaFuncSetAttribute(k3_cosine_topk_kernel<0, 0, 2, 0>, cudaFuncAttributeMaxDynamicSharedMemorySize, optin));
  RBOD_CUDA(cudaFuncSetAttribute(k3_cosine_topk_kernel<0, 0, 4, 0>, cudaFuncAttributeMaxDynamicSharedMemorySize, optin));
  RBOD_CUDA(cudaFuncSetAttribute(k3_cosine_topk_kernel<0, 0, 2, 1>, cudaFuncAttributeMaxDynamicSharedMemorySize, optin));
  RBOD_CUDA(cudaFuncSetAttribute(k3_cosine_topk_kernel<0, 0, 4, 1>, cudaFuncAttributeMaxDynamicSharedMemorySize, optin));
  RBOD_CUDA(cudaFuncSetAttribute(k3_cosine_topk_kernel<1, 0, 2, 0>, cudaFuncAttributeMaxDynamicSharedMemorySize, optin));
  RBOD_CUDA(cudaFuncSetAttribute(k3_cosine_topk_kernel<1, 0, 2, 1>, cudaFuncAttributeMaxDynamicSharedMemorySize, optin));
  RBOD_CUDA(cudaFuncSetAttribute(k3_cosine_topk_kernel<0, 1, 4, 0>, cudaFuncAttributeMaxDynamicSharedMemorySize, optin));
  RBOD_CUDA(cudaFuncSetAttribute(k3_cosine_topk_kernel<0, 1, 2, 0>, cudaFuncAttributeMaxDynamicSharedMemorySize, optin));
  RBOD_CUDA(cudaFuncSetAttribute(k3_cosine_topk_kernel<0, 1, 4, 1>, cudaFuncAttributeMaxDynamicSharedMemorySize, optin));
  if (device >= 0 && device < 64) cached_optin[device] = optin;
  return optin;
}

int launch_k3(const K3Launch& L, cudaStream_t st) {
  K3Params P;
  memset(&P, 0, sizeof(P));
  P.tmap_b = L.tmap_b;
  P.tmap_a = L.tmap_a;
  P.q16 = L.q16;
  P.lists = L.lists;
  P.list_cnt = L.list_cnt;
  P.list_cap = L.list_cap;
  P.list_stride = L.list_stride;
  P.final_cap = L.final_cap;
  P.row_mask = L.row_mask;
  P.mask_of_query = L.mask_of_query;
  P.mask_words = L.mask_words;
  P.row_bias = L.row_bias;
  P.tau_shared = L.tau_shared;
  P.collect_thr = L.collect_thr;
  P.coll_idx = L.coll_idx;
  P.coll_cnt = L.coll_cnt;
  P.coll_cap = L.coll_cap;
  P.groupmax_out = L.groupmax_out;
  P.group_stride = L.group_stride;
  P.group_tiles = L.group_tiles;
  P.group_splits = L.group_splits > 0 ? L.group_splits : 1;
  P.dump = L.dump;
  P.dump_ld = L.dump_ld;
  P.n_rows = L.n_rows;
  P.q_valid = L.q_valid;
  P.q_pad = L.q_pad;
  P.dp = L.dp;
  P.num_kb = L.dp / K3_KBLOCK;
  P.tiles_total = L.tiles_total;
  P.num_qt = L.num_qt;
  P.slices = L.slices;
  P.kc = L.kc;
  P.num_stages = L.num_stages;
  P.variant = L.variant;
  P.sync_counters = L.sync_counters;
  P.sync_window = L.sync_window;
  P.sync_lead = L.sync_lead;
  P.sync_span = L.sync_span;
  P.sync_windows = L.sync_windows;
  P.a_tmem_kb = L.a_tmem_kb;
  P.debug_epi = L.debug_epi;
  P.prof = L.prof;
  P.num_acc = (L.variant == 1 || L.a_tmem_kb * 32 + 2 * K3_TILE_N <= TMEM_COLS) ? 2 : 1;
  P.acc_col0 = TMEM_COLS - P.num_acc * K3_TILE_N;
  P.idesc = make_idesc_f16(L.a_fmt, L.b_fmt, L.variant == 2 ? 2 * K3_TILE_M : K3_TILE_M, K3_TILE_N);
  if (L.num_stages < 1 || L.num_stages > MAX_STAGES)
    return set_error(RBOD_E_INVAL, "k3: bad stage count %d", L.num_stages);
  const bool select_mode = L.collect_thr == nullptr && L.groupmax_out == nullptr;
  if (select_mode && (L.lists == nullptr || L.list_cnt == nullptr || L.kc < 1 || L.kc > K3_MAX_KC ||
                      (L.list_cap != 64 && L.list_cap != 128 && L.list_cap != 256) || L.list_cap < 2 * L.kc ||
                      L.list_stride != L.list_cap + K3_TILE_N || L.final_cap < L.kc))
    return set_error(RBOD_E_INVAL, "k3: bad candidate-list geometry (kc %d, cap %d, stride %d, final %d)", L.kc,
                     L.list_cap, L.list_stride, L.final_cap);
  if (L.variant == 2 && L.grid % 2) return set_error(RBOD_E_INVAL, "k3: pair kernel needs an even grid");
  cudaLaunchConfig_t cfg;
  memset(&cfg, 0, sizeof(cfg));
  cfg.gridDim = dim3((unsigned)L.grid);
  cfg.blockDim = dim3(K3_THREADS);
  cfg.dynamicSmemBytes = L.smem_bytes;
  cfg.stream = st;
  cudaLaunchAttribute attr[2];
  int na = 0;
  if (L.variant == 2) {
    attr[na].id = cudaLaunchAttributeClusterDimension;
    attr[na].val.clusterDim.x = 2;
    attr[na].val.clusterDim.y = 1;
    attr[na].val.clusterDim.z = 1;
    ++na;
  }
  if (L.sync_counters != nullptr && !L.no_coop) {
    // The L2-sharing throttle makes CTAs of one launch wait for each other: ask for a cooperative launch so
    // the runtime guarantees (or refuses) co-residency of the whole grid (grid <= number of SMs, 1 CTA per SM).
    attr[na].id = cudaLaunchAttributeCooperative;
    attr[na].val.cooperative = 1;
    ++na;
  }
  cfg.attrs = attr;
  cfg.numAttrs = na;
  if (L.variant == 2 && L.row_bias != nullptr && L.kbs != 4)
    return set_error(RBOD_E_UNSUPPORTED, "k3: the row-bias (EUCLID) CTA-pair kernel is built with 4-k-block stages only");
  auto launch = [&]() -> cudaError_t {
    if (L.variant == 2 && L.row_bias != nullptr) return cudaLaunchKernelEx(&cfg, k3_cosine_topk_kernel<0, 1, 4, 1>, P);
    if (L.variant == 2 && L.kbs == 2) return cudaLaunchKernelEx(&cfg, k3_cosine_topk_kernel<0, 1, 2, 0>, P);
    if (L.variant == 2) return cudaLaunchKernelEx(&cfg, k3_cosine_topk_kernel<0, 1, 4, 0>, P);
    if (L.variant == 0 && L.row_bias != nullptr && L.kbs == 4) return cudaLaunchKernelEx(&cfg, k3_cosine_topk_kernel<0, 0, 4, 1>, P);
    if (L.variant == 0 && L.row_bias != nullptr) return cudaLaunchKernelEx(&cfg, k3_cosine_topk_kernel<0, 0, 2, 1>, P);
    if (L.variant == 0 && L.kbs == 4) return cudaLaunchKernelEx(&cfg, k3_cosine_topk_kernel<0, 0, 4, 0>, P);
    if (L.variant == 0) return cudaLaunchKernelEx(&cfg, k3_cosine_topk_kernel<0, 0, 2, 0>, P);
    if (L.row_bias != nullptr) return cudaLaunchKernelEx(&cfg, k3_cosine_topk_kernel<1, 0, 2, 1>, P);
    return cudaLaunchKernelEx(&cfg, k3_cosine_topk_kernel<1, 0, 2, 0>, P);
  };
  cudaError_t e = launch();
  if (e == cudaErrorCooperativeLaunchTooLarge && L.sync_counters != nullptr && !L.no_coop) {
    // The runtime cannot keep the whole grid resident (fewer SMs than the planner assumed: another tenant, MPS, a green
    // context).  CTAs that wait for each other are then not allowed: drop the L2-sharing throttle -- the only thing
    // that needs co-residency -- and launch again as an ordinary grid.  Same result, more DRAM traffic.
    cudaGetLastError();
    P.sync_counters = nullptr;
    cfg.numAttrs = na - 1;          // the cooperative attribute was added last
    if (L.coop_refused) ++*L.coop_refused;
    e = launch();
  }
  if (e != cudaSuccess) return set_error(RBOD_E_IO, "k3 launch failed: %s", cudaGetErrorString(e));
  RBOD_CUDA(cudaGetLastError());
  return RBOD_OK;
}

int launch_prep_queries(const float* q, int64_t Q, int64_t q_pad, int dim, int dp, int kind16, int normalize,
                        uint16_t* q16, float* q_dq, double* q_qq, uint32_t* tau_shared, cudaStream_t st) {
  const int64_t want = (q_pad + 7) / 8;
  const int grid = (int)(want < 148 * 8 ? want : 148 * 8);
  prep_queries_kernel<<<grid, 256, 0, st>>>(q, Q, q_pad, dim, dp, kind16, normalize, q16, q_dq, q_qq, tau_shared);
  RBOD_CUDA(cudaGetLastError());
  return RBOD_OK;
}

}  // namespace rbod
