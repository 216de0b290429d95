/*
 * frg.h - C ABI of the B200-native face-gallery matcher (libfrg.so).
 *
 * This is the drop-in boundary for ONE path of bharatlytics/faceRecognition_InfrenceEngine:
 * matching query face embeddings against the enrolled gallery.  The reference has no native
 * code and no FFI; its path is an inline Python loop plus an in-process dict cache.  Each
 * entry point below names the reference lines it replaces (paths relative to the reference
 * root).  A ctypes binding for the reference's two call sites is shown in INTEGRATION.md.
 *
 * Conventions
 *   - every function returns an int status (FRG_OK = 0); frg_last_error() returns a
 *     thread-local description of the last failure.  Nothing throws or aborts across the ABI.
 *   - "_host" entry points take HOST pointers, copy in/out themselves and return when the
 *     result is in the caller's buffers.  The others take DEVICE pointers plus a CUDA stream
 *     (cudaStream_t passed as void*; NULL = legacy default stream) and only enqueue work.
 *   - the caller owns every buffer it passes; the library owns only the store handle.
 *   - a "row" is a position in gallery order = insertion order of the reference's dict
 *     (infrenceServer.py:49, peopleCount.py:707).  Exact score ties resolve to the LOWER row,
 *     which is the reference's strict '>' scan (infrenceServer.py:540, peopleCount.py:871).
 *   - no match: row = -1, score = -1.0f (the scan's initial best_score; infrenceServer.py:536).
 *   - there is no CPU fallback: without a CUDA device every compute entry point fails.
 */
#ifndef FRG_H_
#define FRG_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define FRG_ABI_VERSION 1

#if defined(__GNUC__)
#define FRG_API __attribute__((visibility("default")))
#else
#define FRG_API
#endif

/* status codes */
#define FRG_OK               0
#define FRG_ERR_INVALID      1   /* bad argument */
#define FRG_ERR_CUDA         2   /* a CUDA call failed; see frg_last_error() */
#define FRG_ERR_NOMEM        3
#define FRG_ERR_UNSUPPORTED  4   /* shape / mode not built (e.g. dim not in {128,256,512,1024}) */
#define FRG_ERR_STATE        5   /* e.g. row out of range, store full and not growable */

/* metric */
#define FRG_METRIC_COSINE    0   /* dot of unit vectors: infrenceServer.py:539, peopleCount.py:870 */
#define FRG_METRIC_EUCLIDEAN 1   /* ||g - q||_2, smallest wins.  NOT in the reference (BASELINE config 3) */

/* kernel variant */
#define FRG_VARIANT_AUTO      0  /* dispatch table by batch size (DESIGN.md) */
#define FRG_VARIANT_SCAN_F32  1  /* exact fp32 streaming scan on CUDA cores, reads the fp32 master */
#define FRG_VARIANT_TC_EXACT  2  /* tcgen05 bf16 filter over the scan plane + exact fp32 rescoring (cosine: unit-row
                                    stores; euclidean: FRG_STORE_RAW stores with a scan plane, dim 128 / 256) */
#define FRG_VARIANT_TC_BF16   3  /* tcgen05 bf16 scores returned as-is ("bf16 gallery mode", own tolerance) */

/* frg_store_create flags */
#define FRG_STORE_BF16_PLANE  1u /* keep a scan plane next to the fp32 master (needed by TC variants).  For a unit
                                   (non-raw) store it is an INT8 plane, dim bytes per row, one store-wide scale fixed
                                   by dim (0.165 / 127 per step at dim 512; saturating): a 512-d row takes 2.5 KB.
                                   FRG_VARIANT_TC_BF16 on such a store returns exact scores. */
#define FRG_STORE_RAW         2u /* never normalise on ingest (Euclidean galleries, cluster means).  Together with
                                   FRG_STORE_BF16_PLANE the plane is the EUCLIDEAN scan plane: each row carries
                                   -0.5*||g||^2 (and its own error-bound terms) in 16 more bf16 columns, so that the
                                   tensor-core product with [q, 1, 1, 1, +-A, +-B, +-C, 0..] is an upper / lower bound
                                   of q.g - 0.5*||g||^2 = (||q||^2 - d^2) / 2 */
#define FRG_STORE_BF16_ONLY   4u /* keep ONLY the bf16 scan plane (1 KB / 512-d row instead of 3 KB): "bf16 gallery
                                   mode".  Matches run as FRG_VARIANT_TC_BF16 (scores within the measured bound, ~3.6e-3 of fp32 for ordinary data, DESIGN.md);
                                   the exact variants, first_match and the Euclidean metric are not available. */

/* upsert flags */
#define FRG_ROWS_PRENORMALISED 1u /* store vectors as given (snapshot reload; exact-score fixtures) */

#define FRG_MAX_K 16

typedef struct frg_store frg_store;

typedef struct frg_store_stats_t {
  int64_t rows;        /* rows in use, including tombstones (= next append position) */
  int64_t live;        /* rows that can match (tag >= 0) */
  int64_t capacity;    /* rows allocated */
  int64_t version;     /* bumped by every mutation: the snapshot epoch a match observes */
  int64_t bytes;       /* device bytes held */
  int32_t dim;
  int32_t device;
  uint32_t flags;
  uint32_t faults;     /* != 0: a match kernel's internal pipeline barrier timed out (never a trap: the context
                          stays usable); sticky - results since are void, recreate the store.  The *_host entry
                          points return FRG_ERR_CUDA once it is set. */
} frg_store_stats_t;

typedef struct frg_match_params_t {
  int32_t metric;      /* FRG_METRIC_* */
  int32_t variant;     /* FRG_VARIANT_* */
  float   threshold;   /* cosine: accept iff score >= threshold, compared in fp32 (NumPy>=2 semantics of
                          infrenceServer.py:545 / peopleCount.py:876); euclidean: accept iff dist <= threshold */
  int32_t tenant;      /* < 0: all tenants (peopleCount.py:848); else only rows with this tag
                          (company subset, infrenceServer.py:343-380).  The store remembers the row extent each
                          tag can sit in (as long as tags / rows reach it through the *_host mutators or
                          fill_synthetic; frg_store_compact re-tightens it): a tenant-filtered call scans only
                          that window, so enrol a company's people together */
  int64_t row_offset;  /* added to every returned row (global row of a shard's first row) */
  uint32_t flags;      /* FRG_QUERY_PRENORMALISED (match and first_match), FRG_FIRST_STRICT (first_match) */
  uint32_t reserved;
} frg_match_params_t;

FRG_API int         frg_abi_version(void);
FRG_API const char* frg_last_error(void);
/* number of CUDA devices visible; FRG_ERR_CUDA when the driver / device is missing */
FRG_API int         frg_device_count(int32_t* count);

/* ---- gallery store: replaces EmbeddingManager.embeddings, the Dict[str, np.ndarray] cache
 *      (infrenceServer.py:36-60, peopleCount.py:695-714).  Holds, per row: the unit fp32 vector
 *      (master), optionally its bf16 image (scan plane), and an int32 tag (tenant >= 0, -1 = removed). */
FRG_API int frg_store_create(int32_t device, int32_t dim, int64_t capacity, uint32_t flags, frg_store** out);
FRG_API int frg_store_destroy(frg_store* s);
FRG_API int frg_store_reserve(frg_store* s, int64_t capacity);           /* grow; contents and order kept */
FRG_API int frg_store_stats(frg_store* s, frg_store_stats_t* out);       /* get_stats(): infrenceServer.py:386-398 */

/* Upsert n rows.  rows == NULL: append at [stats.rows, stats.rows + n) (a NEW id in the dict);
 * else rows[i] < stats.rows is overwritten in place (an EXISTING id keeps its position).
 * Vectors are divided by their L2 norm on ingest unless FRG_ROWS_PRENORMALISED / FRG_STORE_RAW:
 * `embedding / np.linalg.norm(embedding)`, infrenceServer.py:271,324; peopleCount.py:788,806
 * (a zero vector becomes a NaN row that never matches).  tags == NULL: tag 0. */
FRG_API int frg_store_upsert(frg_store* s, const int64_t* rows, const float* vecs, const int32_t* tags,
                     int64_t n, uint32_t flags, void* stream);
/* Host arrays.  Returns once the caller's arrays have been consumed (they may be reused at once); batches up to
 * 4 MB are staged through pinned memory and the call does NOT wait for the device - every match enqueued
 * afterwards, on any stream, is ordered after the mutation on the device.  Larger (bulk) batches are copied
 * straight from the caller's arrays and waited for. */
FRG_API int frg_store_upsert_host(frg_store* s, const int64_t* rows, const float* vecs, const int32_t* tags,
                          int64_t n, uint32_t flags);
/* Tombstone rows (tag := -1): `del self.embeddings[id]`, infrenceServer.py:234-258. */
FRG_API int frg_store_remove(frg_store* s, const int64_t* rows, int64_t n, void* stream);
FRG_API int frg_store_remove_host(frg_store* s, const int64_t* rows, int64_t n);
/* Stable compaction: drops tombstones, keeps order.  old_to_new (host, stats.rows entries, may be
 * NULL) receives the new row of every old row or -1. */
FRG_API int frg_store_compact(frg_store* s, int64_t* old_to_new);
/* Copy rows [row0, row0+n) back to the host (snapshot / verification): get_all(), peopleCount.py:816. */
FRG_API int frg_store_read_host(frg_store* s, int64_t row0, int64_t n, float* vecs, int32_t* tags);
/* Append n rows of the counter-based synthetic gallery "frg-synth-v1" (oracle/synth.py is the
 * bit-identical CPU twin): row i is generated from (seed, global_row0 + i) only. */
FRG_API int frg_store_fill_synthetic(frg_store* s, int64_t n, int64_t global_row0, uint64_t seed,
                             int32_t tag, void* stream);

/* ---- match: replaces the per-face loop of FaceRecognitionProcessor.recognize_faces
 *      (infrenceServer.py:530-552) and CameraProcessor.process_frame (peopleCount.py:860-887).
 * q: nq x dim RAW query embeddings (face.normed_embedding); they are re-normalised inside,
 *    as the reference does (infrenceServer.py:532, peopleCount.py:863).
 * out_rows [nq*k] int64, out_scores [nq*k] fp32: the k best rows per query, best first
 *    (k = 1 is the reference's scan; k > 1 is its stable-sort extension, SURVEY.md section 8a row a6).
 * out_accept [nq] uint8: the decision on slot 0 (infrenceServer.py:545; peopleCount.py:876).
 * An empty gallery is not an error: every query gets row -1 / reject (infrenceServer.py:523-525). */
FRG_API int frg_match(frg_store* s, const float* q, int32_t nq, int32_t k, const frg_match_params_t* p,
              int64_t* out_rows, float* out_scores, uint8_t* out_accept, void* stream);
FRG_API int frg_match_host(frg_store* s, const float* q, int32_t nq, int32_t k, const frg_match_params_t* p,
                   int64_t* out_rows, float* out_scores, uint8_t* out_accept);

/* ---- one match call in which every query carries its own tenant filter (a server for many companies' cameras).
 * tenants: HOST array [nq]; tenants[i] < 0 = all tenants, else only rows tagged tenants[i] (a tag no row carries:
 *   every slot of that query row -1 / reject).  p->tenant is not read; everything else of *p applies to all queries.
 * Result of query i == frg_match(s, q_i, 1, k, p') with p' = *p, p'.tenant = tenants[i], bit for bit (rows,
 *   scores, accept), in the caller's query order.
 * A unit cosine store with an fp32 master and a scan plane (AUTO / TC_EXACT / TC_BF16 with dim 128 / 256 / 512)
 *   runs every tenant in ONE pass of the int8 tensor-core filter (frg_last_variant() "tc_exact_grouped"; the launch
 *   count does not grow with the number of tenants).  All queries on one tenant: exactly frg_match.  Every other
 *   store or variant (SCAN_F32, raw / Euclidean, bf16-only, no plane) runs frg_match's path once per tenant inside
 *   the same call - correct, but no faster than separate calls. */
FRG_API int frg_match_tenants(frg_store* s, const float* q, int32_t nq, int32_t k, const frg_match_params_t* p,
                              const int32_t* tenants, int64_t* out_rows, float* out_scores, uint8_t* out_accept,
                              void* stream);
FRG_API int frg_match_tenants_host(frg_store* s, const float* q, int32_t nq, int32_t k, const frg_match_params_t* p,
                                   const int32_t* tenants, int64_t* out_rows, float* out_scores, uint8_t* out_accept);

/* ---- first row, in gallery order, whose score reaches the threshold (exact fp32).  Replaces the two
 *      "first hit" scans next to the matching path:
 *        trainingServer.py:170-200  duplicate face at enrolment: first stored template with cos > 0.4
 *                                   (FRG_FIRST_STRICT)
 *        peopleCount.py:446-452     unknown-person clustering: first cluster, in creation order, with
 *                                   dot(avg_embedding, q) >= 0.65 (a FRG_STORE_RAW store of cluster means,
 *                                   FRG_QUERY_PRENORMALISED)
 *      p->flags: FRG_FIRST_STRICT ('>' instead of '>='), FRG_QUERY_PRENORMALISED (use q as given).
 *      out_rows [nq] (-1 = none), out_scores [nq] (score of that row, -1.0f = none). */
#define FRG_FIRST_STRICT        1u
#define FRG_QUERY_PRENORMALISED 2u
FRG_API int frg_first_match(frg_store* s, const float* q, int32_t nq, const frg_match_params_t* p,
                    int64_t* out_rows, float* out_scores, void* stream);
FRG_API int frg_first_match_host(frg_store* s, const float* q, int32_t nq, const frg_match_params_t* p,
                         int64_t* out_rows, float* out_scores);

/* ---- every row whose score reaches the threshold ("range search"; NOT in the reference: parity unpinned, the
 *      generalisation of trainingServer.py:170-200 from "first hit" to "all hits": watchlists, template clean-up,
 *      duplicate audits of a whole gallery).
 * out_counts [nq] int64: the exact number of live rows (tenant-filtered) with score >= p->threshold (cosine; '>'
 *   with FRG_FIRST_STRICT) or dist <= p->threshold (euclidean; '<' with FRG_FIRST_STRICT).
 * out_rows [nq*max_hits] int64, out_scores [nq*max_hits] fp32: the FIRST min(count, max_hits) of those rows IN
 *   GALLERY ORDER (row ascending, + p->row_offset) with their exact fp32 scores (euclidean: distances); unused slots
 *   row -1 / score -1.0f (euclidean +inf).  count > max_hits tells the caller the list is truncated.
 * p->flags: FRG_FIRST_STRICT, FRG_QUERY_PRENORMALISED.  p->variant: AUTO (the tensor-core filter for unit cosine
 *   stores with a scan plane and dim 128 / 256 / 512, else the exact scan), TC_EXACT (cosine only) or SCAN_F32;
 *   TC_BF16 and bf16-only stores: FRG_ERR_UNSUPPORTED.  max_hits >= 1.  An empty gallery gives counts 0.
 * The scores are bit-identical on both paths; frg_last_variant() names the one that ran (range_tc / range_scan). */
FRG_API int frg_match_range(frg_store* s, const float* q, int32_t nq, int32_t max_hits, const frg_match_params_t* p,
                            int64_t* out_counts, int64_t* out_rows, float* out_scores, void* stream);
FRG_API int frg_match_range_host(frg_store* s, const float* q, int32_t nq, int32_t max_hits,
                                 const frg_match_params_t* p, int64_t* out_counts, int64_t* out_rows,
                                 float* out_scores);

/* ---- range search in which every query carries its own tenant filter (watchlists per company on a server that mixes
 *      companies in one batch; a batch of enrolment duplicate checks: max_hits = 1 with FRG_FIRST_STRICT).
 * tenants: HOST array [nq]; tenants[i] < 0 = all tenants, else only rows tagged tenants[i] (a tag no row carries:
 *   count 0 and "none" slots).  p->tenant is not read; everything else of *p applies to all queries.
 * Result of query i (out_counts[i], out_rows[i*max_hits ..], out_scores[i*max_hits ..]) == frg_match_range(s, q_i, 1,
 *   max_hits, p') with p' = *p, p'.tenant = tenants[i], bit for bit, in the caller's query order, for every metric,
 *   variant, flag and store frg_match_range accepts.  Its refusals apply unchanged; tenants == NULL with nq > 0:
 *   FRG_ERR_INVALID.  A store of more than 2^31 - 1 rows: FRG_ERR_UNSUPPORTED (unless all queries share one tenant).
 * All queries on one tenant: exactly frg_match_range.  Otherwise every tenant runs in ONE set of launches (the launch
 *   count does not grow with the number of tenants): the int8 tensor-core filter where frg_match_range takes it
 *   (frg_last_variant() "range_tc_grouped"), else one exact counting scan in which each query reads only its
 *   tenant's row window ("range_scan_tenants"). */
FRG_API int frg_match_range_tenants(frg_store* s, const float* q, int32_t nq, int32_t max_hits,
                                    const frg_match_params_t* p, const int32_t* tenants, int64_t* out_counts,
                                    int64_t* out_rows, float* out_scores, void* stream);
FRG_API int frg_match_range_tenants_host(frg_store* s, const float* q, int32_t nq, int32_t max_hits,
                                         const frg_match_params_t* p, const int32_t* tenants, int64_t* out_counts,
                                         int64_t* out_rows, float* out_scores);

/* ---- gallery self-join: every pair of stored rows a < b whose score reaches the threshold, in one pass over the
 *      upper triangle on the device (NOT in the reference: the duplicate rule of trainingServer.py:170-200 applied to
 *      what is already enrolled - after a bulk import or a snapshot load).  The queries are the store's own rows; no
 *      row travels to the host.  For each row a in [row0, row0 + n):
 * out_counts[a - row0] int64: the exact number of rows b with a < b < stats.rows such that
 *   score rule:  score(a, b) >= p->threshold ('>' with FRG_FIRST_STRICT);
 *   tag rule:    row b is live; with p->tenant >= 0 both a and b carry that tag; with FRG_JOIN_SAME_TAG
 *                tag[b] == tag[a] (every tenant at once, each within itself).
 *   A dead row a, or one outside p->tenant, has count 0.
 * score(a, b) equals, bit for bit, what frg_match_range returns for row b given the stored fp32 row a as a query.
 * out_rows [n*max_hits] int64, out_scores [n*max_hits] fp32: the FIRST min(count, max_hits) such rows IN GALLERY ORDER
 *   (+ p->row_offset) with their scores; unused slots row -1 / score -1.0f (the range-search layout).
 * Supported: unit cosine stores with an fp32 master.  p->variant: AUTO (the int8 tensor-core filter when the store
 *   keeps a scan plane and dim is 128 / 256 / 512, else the exact scan), TC_EXACT (needs that plane and dim) or
 *   SCAN_F32.  Raw (FRG_STORE_RAW), Euclidean and bf16-only stores, TC_BF16 and FRG_QUERY_PRENORMALISED:
 *   FRG_ERR_UNSUPPORTED (scores on a raw store are not symmetric).  row0 < 0, row0 + n > stats.rows or max_hits < 1:
 *   FRG_ERR_INVALID.  frg_last_variant(): "join_tc" or "join_scan".
 * The call works through [row0, row0 + n) in slabs of FRG_JOIN_SLAB_ROWS query rows with ONE device workspace, whatever
 *   n is: below 2^27 bytes (128 MB) for dim 512 on a 148-SM device, about FRG_JOIN_SLAB_ROWS * (5 * dim + 120 KB).
 *   The launch count is fixed per slab (it does not grow with the number of tenants). */
#define FRG_JOIN_SAME_TAG   4u   /* p->flags: only pairs whose two rows carry the same tag */
#define FRG_JOIN_SLAB_ROWS  1024
FRG_API int frg_self_join(frg_store* s, int64_t row0, int64_t n, int32_t max_hits, const frg_match_params_t* p,
                          int64_t* out_counts, int64_t* out_rows, float* out_scores, void* stream);
FRG_API int frg_self_join_host(frg_store* s, int64_t row0, int64_t n, int32_t max_hits,
                               const frg_match_params_t* p, int64_t* out_counts, int64_t* out_rows, float* out_scores);

/* ---- online clustering of unknown faces, a whole batch in one call (peopleCount.py:432-500, the rule of
 *      frg_first_match's clustering use applied face after face).  The store holds the cluster means: row r is the
 *      mean of cluster r's last `window` faces, which the caller-owned ring keeps on the device.
 * Result == observing q_0, q_1, ... one at a time: face i (used as given) joins the FIRST live row, in row order, with
 *   dot(mean, q_i) >= p->threshold ('>' with FRG_FIRST_STRICT; p->tenant filters as in frg_first_match) - every mean
 *   as the earlier faces of the batch left it - else founds a new row (mean = q_i, tag p->tenant, or 0 when
 *   p->tenant < 0).  On a join q_i is appended to the row's window (the oldest member evicted when it is full) and the
 *   mean becomes the fp32 sum of the members from +0.0f, oldest first, divided by their number (NumPy's
 *   np.mean(window, axis=0), bit for bit).  The dot is frg_first_match's arithmetic, bit for bit.
 * out_cluster [nq] int64: the row face i joined or founded; out_created [nq] uint8: 1 when it founded it.  New rows are
 *   appended at stats.rows, stats.rows + 1, ... in face order.
 * Only FRG_STORE_RAW stores without a scan plane (FRG_ERR_UNSUPPORTED otherwise); the store grows itself.  Refused
 *   with FRG_ERR_INVALID and the store unchanged: ring->capacity < stats.rows + nq, a window outside 1..16, NULL
 *   pointers with nq > 0.  The call synchronises (the number of new rows is known only on the device).
 *   frg_last_variant(): "cluster_observe". */
#define FRG_CLUSTER_MAX_WINDOW 16
typedef struct frg_cluster_ring_t {
  float*   members;   /* DEVICE [capacity][window][dim] fp32: the last `window` faces of cluster row r */
  int32_t* len;       /* DEVICE [capacity] members held, 1..window */
  int32_t* head;      /* DEVICE [capacity] slot of the oldest member */
  int64_t  capacity;  /* cluster rows the ring has room for */
  int32_t  window;    /* 1..FRG_CLUSTER_MAX_WINDOW */
} frg_cluster_ring_t;
FRG_API int frg_cluster_observe_host(frg_store* s, const float* q, int32_t nq, const frg_match_params_t* p,
                                     const frg_cluster_ring_t* ring, int64_t* out_cluster, uint8_t* out_created);

/* ---- k-way merge of per-shard results (multi-GPU tail, SURVEY.md section 8e).
 * scores/rows: [parts][nq][k] (each list best-first, unfilled slots row -1), e.g. the output of an
 * all-gather of every rank's frg_match result.  Order: score desc (euclidean: asc), then row asc. */
FRG_API int frg_merge_topk(int32_t device, const float* scores, const int64_t* rows, int32_t parts,
                   int32_t nq, int32_t k, int32_t metric, float threshold,
                   int64_t* out_rows, float* out_scores, uint8_t* out_accept, void* stream);
/* Same, for lists that sit `score_part_stride` floats / `row_part_stride` int64s apart (0 = nq*k,
 * i.e. contiguous): lets ONE all-gather of a packed [rows | scores] block per rank feed the merge. */
FRG_API int frg_merge_topk_strided(int32_t device, const float* scores, int64_t score_part_stride,
                           const int64_t* rows, int64_t row_part_stride, int32_t parts, int32_t nq, int32_t k,
                           int32_t metric, float threshold, int64_t* out_rows, float* out_scores,
                           uint8_t* out_accept, void* stream);

/* ---- the same tail over NVLink peer memory, no collective-library call on the data path.
 * Every rank owns an exchange buffer of frg_exchange_bytes() bytes, zero-initialised once and peer-mapped
 * into all ranks (e.g. torch symmetric memory: rendezvous(...).buffer_ptrs_dev is `peer_bufs`).  A rank's
 * local top-k travels as 8-byte {payload, epoch} packets written straight into slot `rank` of every rank's
 * buffer; a packet is valid when its epoch word matches, so there is no fence, flag or rendezvous.
 * Collective: every rank makes the same call with the same nq, k and epoch = 1, 2, 3, ... */
#define FRG_XCHG_PUSH_ONLY  1u   /* run the local match and push its result; merge later (same epoch) */
#define FRG_XCHG_MERGE_ONLY 2u   /* the result of this epoch went out earlier: only wait for all ranks and merge */
#define FRG_XCHG_TIMEOUT_MS(ms) ((uint32_t)(ms) << 8)   /* per-call bound of the merge kernel's waits, 1 .. 2^24-1 ms
                                                          (0 = FRG_EXCHANGE_TIMEOUT_MS from the environment, else 2000) */
typedef struct frg_exchange_t {
  int32_t rank, world;     /* world <= 32 */
  void* const* peer_bufs;  /* DEVICE array of `world` device pointers */
  int64_t block_cap;       /* from frg_exchange_bytes() */
  uint32_t epoch;          /* one more per call, never 0 */
  uint32_t flags;          /* 0, or FRG_XCHG_PUSH_ONLY / FRG_XCHG_MERGE_ONLY: the two halves of a call, issued
                              separately (e.g. ranks emulated one after the other on a single device);
                              | FRG_XCHG_TIMEOUT_MS(ms) */
} frg_exchange_t;
FRG_API int frg_exchange_bytes(int32_t world, int32_t nq, int32_t k, int64_t* block_cap, int64_t* total);   /* world <= 32 */
/* frg_match on this rank's shard + exchange + merge in one enqueue: the select stage pushes every query's
 * top-k to all ranks the moment it is final (the exact fallback pushes the queries it redoes); a last kernel,
 * which only waits, merges each query's `world` lists as their packets arrive.  local_rows / local_scores:
 * [nq][k] device scratch for this shard's own result (global rows: params->row_offset).  out_*: the merged
 * result, identical on every rank. */
FRG_API int frg_match_exchange(frg_store* s, const float* q, int32_t nq, int32_t k, const frg_match_params_t* p,
                       const frg_exchange_t* x, int64_t* local_rows, float* local_scores,
                       int64_t* out_rows, float* out_scores, uint8_t* out_accept, void* stream);
/* Exchange + merge of results computed elsewhere ([nq][k] local lists, global rows). */
FRG_API int frg_exchange_merge_topk(int32_t device, const frg_exchange_t* x, const int64_t* local_rows,
                            const float* local_scores, int32_t nq, int32_t k, int32_t metric, float threshold,
                            int64_t* out_rows, float* out_scores, uint8_t* out_accept, void* stream);

/* Waits are bounded (FRG_EXCHANGE_TIMEOUT_MS, default 2000): when a rank never announces the call (the ranks made
 * different numbers of collective calls; a rank died), announces a different (nq, k), or a packet never arrives,
 * the merge kernel gives up, writes "no match" results and a status record into the header of this rank's
 * buffer - it never traps, never hangs.  frg_exchange_status copies that record out (own_buf = this rank's
 * buffer, device pointer; synchronises `stream`): FRG_OK, or FRG_ERR_STATE with frg_last_error() naming call,
 * rank and shapes.  The record is sticky until cleared (clear != 0) or the buffer is zeroed again. */
typedef struct frg_exchange_status_t {
  int32_t code;            /* 0 ok, 1 a rank never announced the call, 2 (nq, k) mismatch, 3 a packet never arrived */
  int32_t peer;            /* the rank concerned */
  uint32_t epoch;          /* the failing call on this rank */
  uint32_t peer_epoch;     /* what that rank's header slot / packet carried instead */
  int32_t nq, k;           /* this rank's shape */
  int32_t peer_nq, peer_k; /* code 2: the peer's */
  int32_t slot;            /* code 3: nq*k slot that never arrived */
  int32_t reserved;
} frg_exchange_status_t;
FRG_API int frg_exchange_status(int32_t device, const void* own_buf, int32_t clear, void* stream,
                                frg_exchange_status_t* out);

/* ---- introspection for tests / bench: name and launch count of the kernels the LAST frg_match /
 * frg_match_host on this thread enqueued (bench.py reports it as gpu_launches). */
FRG_API int frg_last_launch_count(void);
FRG_API const char* frg_last_variant(void);

/* ---- kernel timing for bench.py's roofline: while enabled, every frg_match brackets its DOMINANT
 * kernel launches (the gallery scan / tensor-core pass, not the query prep or the merge) with CUDA
 * events on the caller's stream.  frg_profile_collect waits for those events, returns the summed
 * device time and launch count since the last collect, and clears them.  Thread-local. */
/* on: 0 = off, 1 = every stage of the pipeline (frg_profile_stage_ms), 2 = the dominant kernel only
 * (two event records per match), 3 = as 2 but only every 4th match of this thread, starting with the
 * next one (what bench.py keeps inside its timed region: an event pair costs ~6 us of stream time) */
FRG_API int frg_profile_enable(int32_t on);
FRG_API int frg_profile_collect(float* dominant_ms, int32_t* dominant_launches);
/* Per-stage device time of the matches since the last frg_profile_collect (filled by that call):
 * stage 0 query prep, 1 pre-pass, 2 floor merge, 3 dominant scan/filter, 4 select+rescore, 5 fallback. */
#define FRG_PROFILE_STAGES 6
FRG_API int frg_profile_stage_ms(int32_t stage, float* ms);

#ifdef __cplusplus
}
#endif
#endif  /* FRG_H_ */
