/*
 * rbod.h -- C ABI of the B200-native retrieval hot path ("rbod" = retrieval based object
 * detection).  One shared library, librbod.so, exports exactly these symbols; the Python
 * package `qdrant_client` in this repo (the drop-in for the third-party client the reference
 * scripts import) binds them with ctypes.  No torch / C++ types cross this boundary: plain
 * pointers, sizes and an opaque handle.
 *
 * What each entry point replaces in the reference (paths relative to the reference repo):
 *
 *   rbod_create / rbod_destroy / rbod_count / rbod_truncate
 *       client.recreate_collection(name, VectorParams(size, distance))
 *           util/qdrant_manager.py:82-85 (defaults :56, :74), 02_qdrant_environment_setting.txt:12-14
 *       client.get_collection(n).points_count      util/qdrant_manager.py:46-47, 112-113
 *       client.count(n, exact=True).count          32_create_delegate_vector.py:67
 *       client.delete_collection(n)                util/qdrant_manager.py:121, 138
 *   rbod_upsert                                    (kernel K1 l2norm_pack)
 *       client.upsert(collection, points=[PointStruct(id, vector, payload)])
 *           31_clip_embedding_and_save_vector.py:178-179, 32_create_delegate_vector.py:41-42
 *       plus the L2 normalisation a COSINE collection applies to every stored vector
 *       (third-party Qdrant behaviour, see oracle/oracle_np.py header).
 *   rbod_get_rows
 *       client.scroll(..., with_vectors=True) -> Record.vector
 *           32_create_delegate_vector.py:123-131,137; 33_run_all_experiments.py:96-110,139-149
 *   rbod_segment_mean                              (kernel K2 segmented_mean_renorm)
 *       compute_average  32_create_delegate_vector.py:9-10  (+ renormalise on upsert :41-42)
 *   rbod_search                                    (kernel K3 cosine_topk + exact rescoring)
 *       cosine_similarity(a, b)  33_run_all_experiments.py:76-77, used at :151, generalised
 *       from one pair to Q x N with top-k selection (client.search / query_points semantics).
 *       Distance.MANHATTAN collections (util/qdrant_manager.py:61-66), vectors wider than 768 columns and
 *       k > 128 are answered by kernel K5 distance_topk (exact fp64 sweep) behind the same entry point.
 *   rbod_search_masks                              (the same kernels, one row mask per query)
 *       client.search_batch(requests=[SearchRequest(vector, filter, limit, ...)]), one payload filter per
 *       request (filters as at 32_create_delegate_vector.py:125-129, 33_run_all_experiments.py:98-103,117-137).
 *   rbod_recommend                                 (kernel K6 recommend, exact fp64 sweep)
 *       client.recommend(positive=[...], negative=[...], strategy=RecommendStrategy.BEST_SCORE), recommend_batch and
 *       query_points(query=RecommendQuery(...)): "stored objects like these examples and unlike those" (refining a
 *       class from a few labelled crops, mining hard negatives).  The average_vector strategy needs no entry point of
 *       its own: it is one rbod_search of the composed vector.
 *   rbod_discover                                  (kernel K7 discover, exact fp64 sweep)
 *       client.discover(target=..., context=[ContextExamplePair(positive, negative), ...]), discover_batch and
 *       query_points(query=DiscoverQuery(...) | ContextQuery(...)): "like this target, on the right side of these
 *       corrections" (pairs such as "this crop is the class, that near-identical one is not").
 *   rbod_search_mmr                                (the search's kernels, then kernel K8 mmr_select)
 *       client.query_points(query=NearestQuery(nearest=v, mmr=Mmr(diversity, candidates_limit))) and
 *       query_batch_points: a top-k that is not ten near-copies of one object (the gallery holds ~18 augmented variants
 *       of every crop, 23_augmentation.py / 31_...py).
 *   rbod_merge_topk                                (kernel K4 topk_merge)
 *       no reference call site; merges per-GPU top-k lists after the NCCL all-gather.
 *
 * Conventions
 *   - Every function returns 0 (RBOD_OK) or a negative errno-style code; rbod_last_error()
 *     returns a thread-local, human-readable message for the last failure.  Nothing aborts.
 *   - Pointers marked "host or device" are classified with cudaPointerGetAttributes; host
 *     buffers are copied to / from device workspaces inside the call (pass pinned memory to
 *     keep those copies at full PCIe speed).
 *   - `stream` is a cudaStream_t passed as void* (NULL = legacy default stream).  Calls that
 *     write host outputs synchronise the stream before returning; rbod_search always does
 *     (it reports certification statistics).
 *   - A handle is used from one thread at a time.  One handle lives on one GPU; multi-GPU
 *     search runs one process per GPU and merges with rbod_merge_topk.
 */
#ifndef RBOD_H_
#define RBOD_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define RBOD_ABI_VERSION 1

/* return codes */
#define RBOD_OK 0
#define RBOD_E_IO (-5)           /* CUDA runtime / driver failure */
#define RBOD_E_NOMEM (-12)       /* allocation failed */
#define RBOD_E_INVAL (-22)       /* bad argument */
#define RBOD_E_RANGE (-34)       /* row index / slot out of range */
#define RBOD_E_OVERFLOW (-75)    /* tie cluster larger than the exact-fallback buffer */
#define RBOD_E_UNSUPPORTED (-95) /* valid request this build does not implement */

/* storage dtype of the gallery (the arithmetic is always fp32-accumulate + fp64 rescoring) */
#define RBOD_F32 0
#define RBOD_BF16 1
#define RBOD_F16 2

/* distance of the collection (Distance enum, util/qdrant_manager.py:61-66) */
#define RBOD_COSINE 0
#define RBOD_DOT 1
#define RBOD_EUCLID 2    /* score = L2 distance, smaller is closer; tensor-core pass with a row-bias epilogue (K3) up to
                            768 columns, exact fp64 sweep on CUDA cores (K5) beyond */
#define RBOD_MANHATTAN 3 /* score = L1 distance, smaller is closer; exact fp64 sweep on CUDA cores (kernel K5) */

/* rbod_upsert flags */
#define RBOD_UPSERT_RAW 1 /* rows are already in stored form: do not normalise (used on reload) */

typedef struct rbod_gallery rbod_gallery;

typedef struct rbod_gallery_info {
  int32_t dim;            /* logical vector size                                   */
  int32_t dim_padded;     /* row stride (elements) of the 16-bit search operand    */
  int32_t dtype;          /* RBOD_F32 / RBOD_BF16 / RBOD_F16                       */
  int32_t metric;         /* RBOD_COSINE / RBOD_DOT / RBOD_EUCLID / RBOD_MANHATTAN */
  int32_t device;         /* CUDA device ordinal                                   */
  int32_t coop_refusals;    /* tensor-core launches that ran without the L2-sharing throttle because the runtime */
                            /* refused a cooperative launch (grid not co-resident); 0 on a whole B200           */
  int64_t rows;           /* number of row slots in use (max slot + 1)             */
  int64_t capacity;       /* allocated row slots                                   */
  int64_t bytes_device;   /* device bytes held by the handle (gallery + workspace) */
  float max_row_norm;     /* max ||stored 16-bit row||                             */
  float max_row_dev;      /* max ||stored 16-bit row - unit(master row)||          */
} rbod_gallery_info;

typedef struct rbod_search_stats {
  int64_t queries;          /* Q                                                         */
  int64_t fallback_queries; /* queries whose top-k was not certified by the first        */
                            /* tensor-core pass (they get a collecting second pass)      */
  int64_t k3_launches;      /* kernel launches of the tcgen05 pass (1, or 2 with the     */
                            /* collecting pass)                                          */
  int64_t total_launches;   /* all kernel launches issued by this call                   */
  int32_t candidates;       /* candidates kept per query before rescoring (k + slack)    */
  int32_t slices;           /* gallery slices the tcgen05 pass was split into            */
  float max_eps;            /* largest certification margin used                         */
  float k3_ms;              /* device time of the first tcgen05 pass (CUDA events), 0 if */
                            /* off                                                       */
  int64_t sweep_queries;    /* queries that needed the exact fp64 sweep over the gallery */
                            /* (tie cluster wider than the collecting pass records)      */
  int64_t presample_retries;/* > 0: the sampled starting thresholds were too high for    */
                            /* this many queries and the call was redone without them    */
} rbod_search_stats;

const char* rbod_last_error(void);
int rbod_abi_version(void);

/* --- collection lifetime -------------------------------------------------------------- */
int rbod_create(int32_t dim, int32_t dtype, int32_t metric, int64_t capacity_hint, int32_t device,
                rbod_gallery** out);
int rbod_destroy(rbod_gallery* g);
int64_t rbod_count(const rbod_gallery* g);
int rbod_info(const rbod_gallery* g, rbod_gallery_info* out);
/* Shrinks the number of used row slots (rows beyond `rows` are forgotten). */
int rbod_truncate(rbod_gallery* g, int64_t rows);
/* Tunables: "k3_variant" (-1 = chosen per search: CTA pairs above 128 queries, single CTA below; 0 = query tile
 * resident in TMEM, 1 = query tile streamed through smem, 2 = TMEM-resident + CTA pairs / cta_group::2; rows wider
 * than 768 columns always use 1), "k3_kbs" (64-element k-blocks per pipeline stage of variant 0:
 * 0 = chosen by batch size, 2, 4), "slack" (extra candidates kept per query),
 * "time_k3" (1 = fill stats.k3_ms), "tau_share" (slices of a query share their threshold),
 * "collect_pass" (tensor-core second pass for uncertified queries), "presample" (sampled
 * starting thresholds: 0 = never, 1 = for batches of more than 8 queries, 2 = always), "l2_sync" / "sync_window" /
 * "sync_lead" (L2-sharing producer throttle), "hybrid" (query tile split TMEM / smem), "auto_shadow" (bf16 COSINE
 * collections build an fp16 search operand on the first search with k > 40; default 1), "k3_prof" (wait-cycle
 * counters, see rbod_debug_profile), "debug_grid_scale" (test hook: over-sized grid, exercises the fallback taken
 * when a cooperative launch is refused). */
int rbod_set_option(rbod_gallery* g, const char* key, int64_t value);

/* --- K1: normalise + pack on upsert ----------------------------------------------------
 * rows:      [n, dim] fp32, host or device.
 * row_slots: [n] int64 destination slots (host or device; a device array is read back for validation), or NULL to
 *            append.
 *            A slot equal to the current count appends; smaller overwrites (upsert-by-id
 *            is resolved to a slot by the caller).  Slots must be distinct (a repeated slot is
 *            RBOD_E_INVAL) and the new slots must fill [count, max slot] without holes
 *            (RBOD_E_RANGE); a call refused for its slots changes nothing.
 * out_norms: optional [n] fp32 L2 norms of the incoming rows (host or device), or NULL.   */
int rbod_upsert(rbod_gallery* g, const float* rows, int64_t n, const int64_t* row_slots, float* out_norms,
                int32_t flags, void* stream);

/* Stored rows widened to fp32: out[i, :] = gallery[rows[i], :].  rows/out host or device. */
int rbod_get_rows(rbod_gallery* g, const int64_t* rows, int64_t n, float* out, void* stream);

/* Same kernel on caller-owned buffers (no handle): in [n, dim] fp32 device -> out [n, out_ld]
 * of out_dtype, plus optional norms.  Device pointers only.                               */
int rbod_l2norm_pack(const float* in, int64_t n, int32_t dim, int32_t out_dtype, void* out, int64_t out_ld,
                     float* out_norms, void* stream);

/* --- K2: delegate ("average") vectors ---------------------------------------------------
 * Class c owns gallery rows row_idx[offsets[c] .. offsets[c+1]) (row_idx == NULL: the rows
 * themselves are label-sorted, i.e. row_idx[i] = i).  out_centroids[c, :] is the fp32 mean of those
 * stored rows, L2-normalised for COSINE collections (the stored form an upsert of the mean would
 * leave); an empty class or a zero mean gives zeros.
 * row_idx / offsets / out_centroids: host or device.                                      */
int rbod_segment_mean(rbod_gallery* g, const int64_t* row_idx, const int64_t* offsets, int64_t n_classes,
                      float* out_centroids, void* stream);

/* Sharded build of the same delegates (SURVEY.md 8(e), K2 row "per-rank partial sums + all-reduce"): every rank
 * calls rbod_segment_sums on its own rows with the same class list, the [n_classes, dim] fp64 sums and the
 * per-class row counts are summed over the ranks (ncclAllReduce, issued by the caller), and rbod_segment_finish
 * turns them into the stored form: fp32(sum / count), L2-normalised when `normalize` is non-zero.  A class with
 * count 0 gives zeros.  out_sums / sums / counts / out_vectors: device pointers.                              */
int rbod_segment_sums(rbod_gallery* g, const int64_t* row_idx, const int64_t* offsets, int64_t n_classes,
                      double* out_sums, void* stream);
int rbod_segment_finish(const double* sums, const int64_t* counts, int64_t n_classes, int32_t dim, int32_t normalize,
                        float* out_vectors, void* stream);

/* Other delegate types of 32_create_delegate_vector.py, one vector per class, float64 arithmetic on the
 * stored rows like the reference, output in stored form (fp32, L2-normalised for COSINE collections):
 *   RBOD_DELEGATE_AVERAGE  compute_average           :9-10   (same result as rbod_segment_mean)
 *   RBOD_DELEGATE_CENTROID compute_centroid          :12-15  member nearest to the mean
 *   RBOD_DELEGATE_WEIGHTED compute_weighted_average  :17-21  softmax(-alpha * distance to mean) weights
 *   RBOD_DELEGATE_MEDOID   compute_medoid            :23-26  member with the smallest distance sum
 * out_member_rows: optional [n_classes] int64, the row slot of the chosen member (centroid / medoid),
 * -1 for the other kinds and for empty classes.  Pointers host or device.                            */
#define RBOD_DELEGATE_AVERAGE 0
#define RBOD_DELEGATE_CENTROID 1
#define RBOD_DELEGATE_WEIGHTED 2
#define RBOD_DELEGATE_MEDOID 3
int rbod_segment_delegates(rbod_gallery* g, int32_t kind, const int64_t* row_idx, const int64_t* offsets,
                           int64_t n_classes, double alpha, float* out_vectors, int64_t* out_member_rows,
                           void* stream);

/* --- K3: cosine top-k (K5 for EUCLID / MANHATTAN collections) ---------------------------
 * queries:      [Q, dim] fp32 (any norm), host or device.
 * row_mask:     optional bitmask over row slots (bit r%32 of word r/32 set = row allowed),
 *               ceil(rows/32) words, host or device; NULL = all rows.
 * out_scores:   [Q, k] fp32 cosine, descending; ties broken by smaller row slot.
 * out_rows:     [Q, k] int64 row slots; -1 (score -inf) where fewer than k rows qualify.
 * out_scores64: optional [Q, k] fp64 scores (what the multi-GPU merge consumes), or NULL.
 * stats:        optional.
 * COSINE, DOT and EUCLID collections up to 2048 columns with k <= 128 run on the tensor-core pass; MANHATTAN, wider
 * vectors and larger k (up to 1024) take the exact fp64 sweep on the CUDA cores (kernel K5) -- same results.
 * EUCLID / MANHATTAN collections: out_scores holds the DISTANCE (sqrt of the squared sum / sum of absolute
 * differences), ascending, +inf where fewer than k rows qualify; ties broken by smaller row slot;
 * out_scores64 holds the ordering key (-squared distance / -L1 distance, larger = closer), which is what
 * rbod_merge_topk orders by.  MANHATTAN (and EUCLID wider than 2048 columns): k <= 1024.   */
int rbod_search(rbod_gallery* g, const float* queries, int64_t Q, int32_t k, const uint32_t* row_mask,
                float* out_scores, int64_t* out_rows, double* out_scores64, rbod_search_stats* stats,
                void* stream);

/* Like rbod_search, but each query has its own row mask (one filtered request per query, in one pass).
 * row_masks:     [n_masks][ceil(rows/32)] uint32, the same bit layout as rbod_search's row_mask. Host or device.
 *                NULL only when n_masks == 0.
 * mask_of_query: [Q] int32, the mask each query uses. -1 means no filter. Host or device (a device array is read
 *                back, Q * 4 bytes, to be checked before anything is launched).
 *                NULL means every query uses mask 0 (or no mask when n_masks == 0).
 * Every other argument and output is as for rbod_search.  An id outside [-1, n_masks), n_masks < 0, or n_masks > 0
 * with row_masks == NULL is RBOD_E_INVAL.
 * Result: row q is identical, bit for bit in out_scores / out_rows / out_scores64, to
 * rbod_search(queries + q*dim, 1, k, row_masks + mask_of_query[q]*words, ...).
 * rbod_search(..., row_mask, ...) is rbod_search_masks(..., row_mask, row_mask ? 1 : 0, NULL, ...).           */
int rbod_search_masks(rbod_gallery* g, const float* queries, int64_t Q, int32_t k,
                      const uint32_t* row_masks, int32_t n_masks, const int32_t* mask_of_query,
                      float* out_scores, int64_t* out_rows, double* out_scores64,
                      rbod_search_stats* stats, void* stream);

/* --- K8: maximal marginal relevance (MMR) ------------------------------------------------
 * For a query q with the exact candidates c_0 .. c_{L-1} of rbod_search_masks(..., k = candidates, ...), ordered as that
 * search orders them (key desc, row slot asc), and with
 *   key(x, g)  the search key in fp64 from the stored values (the fp32 master of an f32 collection, the 16-bit rows
 *              otherwise, never the fp16 shadow): COSINE dot / (|x| |g|), DOT dot, EUCLID -sum (x - g)^2,
 *              MANHATTAN -sum |x - g|,
 *   sim(y)     y, or -sqrt(-y) for EUCLID (rbod_recommend's sim: larger is better for every metric),
 *   rel(c)     sim(key(q, c)), the candidate search's own fp64 key,
 *   lambda     1 - diversity[q],
 * the first pick is c_0 and every later pick maximises, over the candidates not yet picked,
 *   mmr(c) = lambda * rel(c) - diversity * max over picked s of sim(key(s, c))
 * computed in fp64 in exactly that order (the picked stored row s is the query side of the pairwise key); exact ties go
 * to the smaller candidate rank.  Results come in SELECTION order, each with its ordinary search score (cosine / dot, or
 * the distance for EUCLID / MANHATTAN), so they are not sorted by score; diversity 0 returns the search's first `limit`
 * rows.  (Qdrant >= 1.15 documents the same kind of rule; this one was not checked against a live Qdrant or its source.
 * The EUCLID sim and the tie rule are choices of this library.)
 * queries:         [Q, dim] fp32, host or device.
 * limit:           results per query; candidates: L, limit <= L <= 1024.
 * diversity:       [Q] fp64 in [0, 1], host.
 * score_threshold: [Q] fp32, host, or NULL; NaN = none.  A candidate takes part only if its fp32 search score is >= the
 *                  threshold (<= for EUCLID / MANHATTAN, whose scores are distances), so a request still fills `limit`
 *                  when enough candidates pass.
 * row_masks / n_masks / mask_of_query: as rbod_search_masks.
 * out_scores:      [Q, limit] fp32 search scores in selection order; -inf (COSINE, DOT) or +inf (EUCLID, MANHATTAN) where
 *                  fewer candidates exist.
 * out_rows:        [Q, limit] int64 row slots in selection order, -1 padded.
 * out_keys:        optional [Q, limit] fp64 search keys (-inf padded), or NULL.  Outputs host or device.
 * stats:           optional: the candidate search's, total_launches counting K8.
 * RBOD_E_INVAL (checked on the host before anything is launched, a device mask_of_query after reading it back): limit < 1,
 * candidates < limit, a diversity that is NaN or outside [0, 1], diversity == NULL with Q > 0, a mask id outside
 * [-1, n_masks), n_masks < 0, n_masks > 0 with row_masks == NULL, NULL queries or outputs with Q > 0.  candidates > 1024
 * is RBOD_E_UNSUPPORTED.  Q = 0 and an empty collection return RBOD_OK (the latter with padding).
 * Result: row q is identical, bit for bit, whether query q is sent alone or with others.                    */
int rbod_search_mmr(rbod_gallery* g, const float* queries, int64_t Q, int32_t limit, int32_t candidates,
                    const double* diversity, const float* score_threshold, const uint32_t* row_masks, int32_t n_masks,
                    const int32_t* mask_of_query, float* out_scores, int64_t* out_rows, double* out_keys,
                    rbod_search_stats* stats, void* stream);

/* --- K6: recommendation, best_score strategy ---------------------------------------------
 * A request is a set of 1 to 32 examples, each positive ("like this") or negative ("unlike this").  For an example e and
 * a stored row g the key is rbod_search's exact fp64 ordering key, computed from the fp32 example and the stored row:
 *   COSINE dot / (|e| |g|),  DOT dot,  EUCLID -sum (e - g)^2,  MANHATTAN -sum |e - g|.
 * bp = the largest key over the request's positives, bn = over its negatives (-inf where there are none), and
 *   sim(x) = x (COSINE, DOT, MANHATTAN) or -sqrt(-x) (EUCLID),   s(y) = 0.5 * (y / (1 + |y|) + 1),
 *   score  = s(sim(bp)) if bp > bn, else -s(sim(bn))
 * (the best_score rule of Qdrant >= 1.7, merge_similarities / scaled_fast_sigmoid; not checked against a live Qdrant).
 * The score is larger-is-better for every metric: rows come ordered by (score desc, row slot asc).
 * examples:        [n_examples, dim] fp32, host or device.  Example points given by id are passed as their stored rows
 *                  (rbod_get_rows); leaving those rows out of a request's answer is the caller's business.
 * example_sign:    [n_examples] int8, +1 (positive) or -1 (negative), host.
 * request_offsets: [R + 1] int64, host: request r owns examples [request_offsets[r], request_offsets[r + 1]); they run
 *                  from 0 to n_examples and every request has 1 to 32 examples.
 * row_masks / n_masks / mask_of_request: as rbod_search_masks's row_masks / n_masks / mask_of_query, one id per request
 *                  (-1 = no filter; NULL = every request reads mask 0, or no mask when n_masks == 0).
 * out_scores:      [R, k] fp32 (float)score; -inf where fewer than k rows are allowed.
 * out_rows:        [R, k] int64 row slots; -1 where fewer than k rows are allowed.
 * out_keys:        optional [R, k] fp64 score (-inf padded), or NULL.  Outputs host or device.
 * stats:           optional: queries = sweep_queries = R, total_launches, fallback_queries = re-sweeps of requests
 *                  whose list of rows at or above the threshold overflowed.
 * RBOD_E_INVAL (checked on the host before anything is launched, a device mask_of_request after reading it back): a
 * request without examples or with more than 32, a sign other than +1 / -1, offsets that are not monotone or do not
 * run from 0 to n_examples, a mask id outside [-1, n_masks), n_masks < 0, n_masks > 0 with row_masks == NULL, k < 1.
 * k > 1024 is RBOD_E_UNSUPPORTED.  R = 0 and an empty collection return RBOD_OK (the latter with padding).  More than
 * 8192 rows tied with a request's k-th score is RBOD_E_OVERFLOW, as for rbod_search.
 * Result: row r is identical, bit for bit, whether request r is sent alone or with others.                  */
int rbod_recommend(rbod_gallery* g, const float* examples, int64_t n_examples, const int8_t* example_sign,
                   const int64_t* request_offsets, int64_t R, int32_t k, const uint32_t* row_masks, int32_t n_masks,
                   const int32_t* mask_of_request, float* out_scores, int64_t* out_rows, double* out_keys,
                   rbod_search_stats* stats, void* stream);

/* --- K7: discovery and context search ---------------------------------------------------
 * A request is an optional target t followed by pairs (p, n) of examples ("like p, not n"): 1 to 32 examples, 0 to 15
 * pairs with a target, 1 to 16 without.  Keys and sim are rbod_recommend's: for an example e and a stored row g the
 * fp64 key of the fp32 example and the stored row (COSINE dot / (|e| |g|), DOT dot, EUCLID -sum (e - g)^2, MANHATTAN
 * -sum |e - g|), sim(x) = x (-sqrt(-x) for EUCLID).  With
 *   f(y) = y / (1 + |y|),  s(y) = 0.5 * (f(y) + 1),  MARGIN = 2^-23 (f32 epsilon),  P = key(p, g),  N = key(n, g):
 *   rank_pair = +1 if P > N else -1 (a tie counts -1),  loss_pair = f(min(sim(P) - sim(N) - MARGIN, 0))
 *   discovery (with a target):  score = sum of rank_pair + s(sim(key(t, g)))
 *   context (no target):        score = sum of loss_pair, summed in pair order; 0 for every row on the positive
 *                               side of every pair, so the top k is often a plateau of rows tied at 0
 * (the rule of Qdrant >= 1.7, DiscoveryQuery::score_by / ContextPair::loss_by, as read from its source; not checked
 * against a live Qdrant.  The EUCLID sim is best_score's, a choice of this library.)  The score is larger-is-better for
 * every metric: rows come ordered by (score desc, row slot asc).  A request of a target alone scores s(sim(key(t, g))),
 * the order of rbod_search.
 * examples:        [n_examples, dim] fp32, host or device; example points given by id are passed as their stored rows.
 * example_role:    [n_examples] int8, host: 0 = target (only as a request's first example), +1 = a pair's positive
 *                  (always followed by its negative), -1 = a pair's negative (always preceded by its positive).
 * request_offsets, row_masks, n_masks, mask_of_request, out_scores, out_rows, out_keys, stats: as rbod_recommend.
 * RBOD_E_INVAL (checked on the host before anything is launched, a device mask_of_request after reading it back): a
 * request without examples or with more than 32, offsets that are not monotone or do not run from 0 to n_examples, a
 * role outside {0, +1, -1}, a target that is not its request's first example (or a second target), a +1 not followed
 * by a -1 or a -1 not preceded by a +1, a mask id outside [-1, n_masks), n_masks < 0, n_masks > 0 with row_masks ==
 * NULL, k < 1.  k > 1024 is RBOD_E_UNSUPPORTED.  R = 0 and an empty collection return RBOD_OK (the latter with
 * padding).  More than 8192 rows tied with a request's k-th score after the re-sweeps is RBOD_E_OVERFLOW.
 * Result: row r is identical, bit for bit, whether request r is sent alone or with others.                  */
int rbod_discover(rbod_gallery* g, const float* examples, int64_t n_examples, const int8_t* example_role,
                  const int64_t* request_offsets, int64_t R, int32_t k, const uint32_t* row_masks, int32_t n_masks,
                  const int32_t* mask_of_request, float* out_scores, int64_t* out_rows, double* out_keys,
                  rbod_search_stats* stats, void* stream);

/* --- K4: merge of per-shard top-k lists -------------------------------------------------
 * scores64 / ids: [G, Q, k] as produced by an all-gather of each rank's rbod_search output
 * (ids already global; id < 0 = empty).  Output: the global top-k per query, ordered by
 * (score desc, id asc).  Device pointers only.                                            */
int rbod_merge_topk(const double* scores64, const int64_t* ids, int32_t G, int64_t Q, int32_t k,
                    float* out_scores, int64_t* out_ids, double* out_scores64, void* stream);

/* The same merge over ONE gathered buffer: every rank contributes [2][Q][k] 8-byte words -- its fp64 scores
 * (rbod_search's out_scores64) followed by its LOCAL row slots (out_rows) -- so a sharded search needs a single
 * all-gather; gathered = [G][2][Q][k] (device).  shard_row0: host array of G global row offsets added to the
 * non-negative slots of shard g (NULL = slots are already global ids).                                     */
int rbod_merge_topk_packed(const void* gathered, const int64_t* shard_row0, int32_t G, int64_t Q, int32_t k,
                           float* out_scores, int64_t* out_ids, double* out_scores64, void* stream);

/* --- Split search for row-sharded collections (multi-GPU, SURVEY.md 8(e)) --------------------------------------
 * rbod_search makes every shard compute exact scores for its own k best candidates although the merge keeps k of the
 * G*k.  The split form puts one small exchange in the middle so that a shard rescoring only what can still be in the
 * GLOBAL answer:
 *   1. rbod_search_begin   query prep, threshold pre-pass, K3, selection.  Writes out_approx [Q][approx_m + 1] (device,
 *                          fp32): the shard's approx_m best APPROXIMATE scores, descending, -inf padded, then the
 *                          bound on |approximate - exact| for this query on this shard.  1 <= approx_m <= k; the
 *                          global cut below is exact when no shard holds more than approx_m of the global top k and
 *                          a valid (lower) bound otherwise, G * approx_m >= k is required.  No synchronisation.
 *   2. (caller)            all-gather of out_approx -> [G][Q][approx_m + 1]
 *   3. rbod_global_cut     out_cut [Q][2] (device, fp32): {k-th largest gathered score, largest gathered bound}
 *   4. rbod_search_end     exact fp64 scores for the candidates within 2 bounds of the cut, ranked; writes the
 *                          shard's list in the packed layout rbod_merge_topk_packed takes -- out_scores64 [Q][k],
 *                          out_rows [Q][k] (local slots, -1 padded) -- and out_ubound [Q] (fp64): an upper bound, in
 *                          the domain of out_scores64, on every row of the shard that was never a candidate (-inf if
 *                          none was dropped).  Device pointers only; the three are normally slices of ONE buffer of
 *                          2*Q*k + Q 8-byte words.  Must follow rbod_search_begin on the same handle with the same
 *                          Q and k, nothing else searched in between; device `queries` must stay valid until then.
 *   5. (caller)            all-gather of that buffer -> [G][2*Q*k + Q]
 *   6. rbod_merge_topk_certified   K4 over the gathered buffer, plus the certification: query q is exact when the
 *                          merged k-th score beats every shard's bound; the others are listed in out_flag_q
 *                          [up to Q] (device int32, unordered), their number in out_n_flag (device int32).  The caller
 *                          answers those with rbod_search (+ rbod_merge_topk_packed) and overwrites their rows.
 * Collections / k that rbod_search answers with the exact sweep (MANHATTAN, > 2048 columns, k > 128) are refused by
 * rbod_search_begin with RBOD_E_UNSUPPORTED: use rbod_search there.  A shard without rows takes part with empty lists. */
int rbod_search_begin(rbod_gallery* g, const float* queries, int64_t Q, int32_t k, int32_t approx_m,
                      const uint32_t* row_mask, float* out_approx, rbod_search_stats* stats, void* stream);
int rbod_global_cut(const float* gathered_approx, int32_t G, int64_t Q, int32_t approx_m, int32_t k, float* out_cut,
                    void* stream);
int rbod_search_end(rbod_gallery* g, const float* cut, int64_t Q, int32_t k, double* out_scores64, int64_t* out_rows,
                    double* out_ubound, rbod_search_stats* stats, void* stream);
int rbod_merge_topk_certified(const void* gathered, const int64_t* shard_row0, int32_t G, int64_t Q, int32_t k,
                              float* out_scores, int64_t* out_ids, double* out_scores64, int32_t* out_flag_q,
                              int32_t* out_n_flag, void* stream);
/* K3 time (threshold pre-pass + main pass) of the handle's last search, option time_k3 = 1; waits for that search. */
int rbod_last_k3_ms(rbod_gallery* g, float* out_ms);

/* --- test hook --------------------------------------------------------------------------
 * Raw scores of the tcgen05 pass (before top-k and rescoring): out[q, r] for r < rows,
 * fp32, device or host.  Small problems only (Q * rows <= 2^28).                          */
int rbod_debug_scores(rbod_gallery* g, const float* queries, int64_t Q, float* out, void* stream);

/* With option "k3_prof" = 1 the main tensor-core launches of this collection's searches accumulate SM cycles spent
 * waiting, summed over CTAs (warp role: what it waited for): out16[0] producer: a free pipeline stage, [1] producer:
 * the L2-sharing throttle, [2] MMA issuer: the query tile, [3] MMA issuer: a free accumulator (epilogue behind),
 * [4] MMA issuer: gallery data (TMA behind), [5] epilogue warps: a finished accumulator, [6] epilogue warps: list
 * prunes, [7] total cycles of the CTAs, [8] CTAs, [9] epilogue warps, [10] prunes, [11] as [0] for the second CTA of a pair,
 * [12] producer: issuing TMA loads, [13] MMA issuer: issuing MMAs and commits.  Reads and clears the counters. */
int rbod_debug_profile(rbod_gallery* g, int64_t* out16);

/* Host-only: the work decomposition rbod_search would choose for a tensor-core search of Q queries, top k, over a
 * gallery of `rows` vectors of `dim` columns (`variant` as the "k3_variant" option, -1 = automatic) on a device with `num_sms` SMs and `smem_optin` bytes of opt-in shared
 * memory per CTA (B200: 148, 232448).  Needs no GPU.  out[0..12] = candidates per query, slices, grid, query tiles,
 * gallery tiles, pipeline stages, k-blocks per stage, query-tile k-blocks kept in TMEM, dynamic shared memory bytes,
 * candidate-list prune trigger, list stride, longest list handed to the merge, keys the merge holds per query.
 * Returns RBOD_E_UNSUPPORTED when the shape must take the fp64 sweep instead (k > 128 or more than 768 columns). */
int rbod_debug_plan(int32_t dim, int64_t rows, int64_t Q, int32_t k, int32_t variant, int32_t num_sms,
                    int32_t smem_optin, int64_t* out);

#ifdef __cplusplus
}
#endif
#endif /* RBOD_H_ */
