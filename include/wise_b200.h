/* wise_b200.h - C-ABI of libwiseb200.so, the B200 (sm_100a) search-index backend for WISE.
 *
 * The reference (ox-vgg/wise) has no FFI: its hot path is the Python object protocol of the
 * faiss CPU classes held in FeatureSearchIndex.index.  Every entry point below names the
 * reference call it replaces (paths under /root/reference).  A maintainer binds these with
 * ctypes (see INTEGRATION.md); wise_b200/faiss_compat.py is that binding.
 *
 * Conventions
 *   - every function returns 0 on success, non-zero on error; wb_last_error() gives the
 *     message of the last error on the calling thread.  Nothing throws across the boundary.
 *   - the caller owns every buffer; "host" pointers are ordinary (pageable or pinned) host
 *     memory, "_dev" variants take device pointers on the index's GPU and a cudaStream_t
 *     (passed as void*) and do not synchronise.
 *   - a buffer (host or device) needs only the natural alignment of its element type: 4 bytes for float and int32,
 *     8 bytes for int64.  Any view into a larger allocation at such an offset is a valid argument.
 *   - one handle must not be used from two threads at the same time; different handles (also of one GPU) may be.
 *   - one index lives on one GPU.  Several GPUs serve one set of rows either from one process per GPU (rows are
 *     sharded across processes by the host layer, wise_b200/sharded.py; the per-GPU top-k lists are exchanged and
 *     merged through NVLink peer memory by wb_exch_search*, below - NCCL is not on the search path) or from one
 *     process through a shard group (wb_group_*, below).
 *   - results: D float32[nq*k] sorted by score descending, ties broken by lowest insertion
 *     position; I int64[nq*k]; unfilled slots are (-FLT_MAX, -1) exactly like faiss.
 *   - there is no CPU fallback: without a CUDA device every compute call fails.
 *   - streams: host-pointer entry points run on the handle's own stream and return synchronised.  "_dev" entry
 *     points enqueue on the caller's stream; calls on ONE stream are ordered, but the caller must synchronise that
 *     stream before it uses another stream or a host-pointer entry point on the same handle (an add that has to grow
 *     the store synchronises the caller's stream itself; wb_reserve up front avoids the growth).
 */
#ifndef WISE_B200_H
#define WISE_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct wb_index wb_index;

#define WB_MAX_K 2048 /* top-k / nprobe limit of the fused selection (faiss-gpu has the same cap) */

/* ---- library ---------------------------------------------------------------------------- */
const char* wb_last_error(void);
const char* wb_version(void);
int wb_device_count(int* count);

/* ---- construction ----------------------------------------------------------------------- */
/* faiss.IndexFlatIP(d) [+ faiss.IndexIDMap(index)]   src/index/feature_search_index.py:47-52.
 * One object serves both: rows added without ids get id = insertion position. */
int wb_flat_create(int d, int device, wb_index** out);
/* faiss.IndexIVFFlat(quantizer, d, nlist, METRIC_INNER_PRODUCT)   feature_search_index.py:60 */
int wb_ivf_create(int d, int64_t nlist, int device, wb_index** out);
int wb_free(wb_index* h);

/* ---- properties: index.d / .ntotal / .is_trained / .nlist   feature_search_index.py:73,76 --- */
int64_t wb_dim(const wb_index* h);
int64_t wb_ntotal(const wb_index* h);
int wb_is_trained(const wb_index* h);
int64_t wb_nlist(const wb_index* h); /* 0 for a flat index */
int wb_is_ivf(const wb_index* h);

/* ---- build ------------------------------------------------------------------------------ */
/* Pre-size HBM for n rows (FeatureStore.feature_count is known before the add loop,
 * feature_search_index.py:44) so adds never re-allocate. Optional. */
int wb_reserve(wb_index* h, int64_t n);
/* Rows the store holds without growing, and the free memory of the index's GPU (a growth allocates the new store,
 * at least 1.5x the old, before it frees the old one): lets a multi-GPU index decide when a shard is full. */
int wb_capacity(wb_index* h, int64_t* cap_rows, int64_t* free_bytes);
/* index.add_with_ids(X, ids)   feature_search_index.py:81.  ids may be NULL (index.add).
 * IVF: also assigns each row to its max-inner-product centroid (ties -> lowest list). */
int wb_add_with_ids(wb_index* h, int64_t n, const float* x_host, const int64_t* ids_host);
int wb_add_with_ids_dev(wb_index* h, int64_t n, const float* x_dev, const int64_t* ids_dev, void* stream);

/* Pinned, overlapped ingest: the add loop of feature_search_index.py:79-82 with the host->HBM copy and the IVF
 * assignment of batch i running while the loader decodes batch i+1.  x / ids live in pinned host memory
 * (wb_pinned_alloc); the call enqueues and returns; `slot` (0..7) names the buffer and wb_add_slot_wait(slot) blocks
 * until the GPU has finished reading it; wb_sync waits for everything enqueued on the handle. */
int wb_pinned_alloc(int64_t bytes, void** out);
int wb_pinned_free(void* p);
int wb_add_with_ids_pinned(wb_index* h, int64_t n, const float* x_pinned, const int64_t* ids_pinned, int slot);
int wb_ivf_add_preassigned_pinned(wb_index* h, int64_t n, const float* x_pinned, const int64_t* ids_pinned,
                                  const int32_t* assign_pinned, int slot); /* read_index of an IwFl file: lists known */
int wb_add_slot_wait(wb_index* h, int slot);
int wb_sync(wb_index* h);

/* index.train(train_features)   feature_search_index.py:75  (k-means with max-inner-product assignment, niter
 * iterations, faiss Clustering defaults: niter=10, seed=1234, spherical=false).  Sets is_trained. */
int wb_ivf_train(wb_index* h, int64_t n, const float* x_host, int niter, int64_t seed);
/* index.cp.spherical (faiss ClusteringParameters): renormalise the centroids after every update.  Default off, like
 * the IndexIVFFlat the reference constructs (feature_search_index.py:60). */
int wb_ivf_set_spherical(wb_index* h, int on);
/* The quantizer's centroids (what faiss keeps in index.quantizer): used to load a trained
 * index (read_index) and to compare search on the reference's own centroids. */
int wb_ivf_set_centroids(wb_index* h, const float* centroids_host /* [nlist*d] */);
int wb_ivf_get_centroids(const wb_index* h, float* centroids_host /* [nlist*d] */);
/* A trainer that drives the k-means pieces below itself (sharded training) declares the result final. */
int wb_ivf_mark_trained(wb_index* h);
/* One k-means iteration from the current centroids over device-resident points; exposed so a
 * sharded trainer can all-reduce sums/counts between the two halves.
 *   assign: x -> int32 list per row, objective = sum of max inner products
 *   accumulate: per-list fp32 sums [nlist*d] and int64 counts [nlist] of the local rows
 *   update: centroids <- sums/counts (L2-normalised when spherical), empty lists split (eps = 1/1024) */
int wb_kmeans_assign_dev(wb_index* h, int64_t n, const float* x_dev, int32_t* assign_dev,
                         double* objective_host, void* stream);
/* Same, with plain-TF32 scores (one tensor-core term): for TRAINING iterations only - two centroids whose scores differ
 * by less than ~2e-3 |x||c| may swap (SURVEY.md 8d).  wb_ivf_train uses it; add-time assignment never does. */
int wb_kmeans_assign_fast_dev(wb_index* h, int64_t n, const float* x_dev, int32_t* assign_dev,
                              double* objective_host, void* stream);
int wb_kmeans_accumulate_dev(wb_index* h, int64_t n, const float* x_dev, const int32_t* assign_dev,
                             float* sums_dev, int64_t* counts_dev, void* stream);
int wb_kmeans_update_dev(wb_index* h, const float* sums_dev, const int64_t* counts_dev, int64_t n_total,
                         int64_t seed, int64_t* nsplit_host, void* stream);

/* ---- search ----------------------------------------------------------------------------- */
/* dist, ids = index.search(x, k)   feature_search_index.py:113, api/routes.py:1407.
 * nprobe is ignored by flat indices (index.nprobe, api/routes.py:899-902). 1 <= k <= WB_MAX_K.
 * Batches of 5+ queries take the tensor-core path, which synchronises `stream` once at the end (it has to
 * read the candidate-overflow flag); smaller batches and IVF list scans stay fully asynchronous in _dev and are
 * ONE kernel launch (the scan kernel's last CTA merges the per-CTA lists and writes D / I). */
int wb_search(wb_index* h, int64_t nq, const float* q_host, int64_t k, int64_t nprobe,
              float* D_host, int64_t* I_host);
int wb_search_dev(wb_index* h, int64_t nq, const float* q_dev, int64_t k, int64_t nprobe,
                  float* D_dev, int64_t* I_dev, void* stream);
/* ---- filtered search ---------------------------------------------------------------------------
 * index.search(x, k, params=faiss.SearchParameters(sel=...)) / SearchParametersIVF(sel=..., nprobe=...) [faiss-upstream]:
 * the exact top-k over the rows a selector keeps.  A selector tests the EXTERNAL id of a row (the id given to
 * add_with_ids; the insertion position for rows added without ids).  Order, tie rule and padding are those of
 * wb_search; the IVF coarse quantizer is not filtered (candidates = the selected rows of the nprobe probed lists).
 *
 * A wb_filter is bound to the index it was created for (using it with another index is an error) and must be freed
 * before that index.  It keeps its definition, a device bitmap with one bit per insertion position, and the number of
 * rows it selects.  Creation evaluates it on the device and synchronises once to read that number; a search with it
 * needs no further synchronisation, except after the index has grown: the next search re-evaluates the bitmap, and a
 * _dev search then synchronises the caller's stream first (as an add that grows the store does).  The first flat
 * search with a very selective filter (below 1/kSparseCutoffDen of the rows, DESIGN.md "Filtered search") also
 * gathers the selected rows into a compact copy that the filter keeps and later searches reuse.
 * f == NULL in the search calls means unfiltered. */
typedef struct wb_filter wb_filter;
/* IDSelectorBatch(ids) (invert = 0) or IDSelectorNot(IDSelectorBatch(ids)) (invert = 1): ids in any order,
 * duplicates allowed, n may be 0. */
int wb_filter_create_ids(wb_index* h, int64_t n, const int64_t* ids_host, int invert, wb_filter** out);
/* IDSelectorRange(imin, imax): imin <= id < imax (empty when imin >= imax); invert = 1 for IDSelectorNot of it. */
int wb_filter_create_range(wb_index* h, int64_t imin, int64_t imax, int invert, wb_filter** out);
int64_t wb_filter_count(const wb_filter* f); /* rows selected when the filter was last evaluated */
int wb_filter_free(wb_filter* f);            /* before the index it belongs to */
int wb_search_filtered(wb_index* h, wb_filter* f, int64_t nq, const float* q_host, int64_t k, int64_t nprobe,
                       float* D_host, int64_t* I_host);
int wb_search_filtered_dev(wb_index* h, wb_filter* f, int64_t nq, const float* q_dev, int64_t k, int64_t nprobe,
                           float* D_dev, int64_t* I_dev, void* stream);

/* ---- range search (DESIGN.md "Range search") ----------------------------------------------------
 * Every row whose fp32 inner product with the query is strictly greater than `thresh` (the score returned in D is the
 * one compared), per query in score-descending order, equal scores by insertion position.  Flat: every row is a
 * candidate; IVF: the rows of the nprobe lists the coarse quantizer of wb_search picks; with a filter, only the rows it
 * selects.  There is no cap on the result size (WB_MAX_K does not apply): query i's results are entries
 * [lims[i], lims[i+1]) of D and I.  A query whose hits alone exceed the device budget of one call (2^28 hits) is an
 * error; the index stays usable.
 * Results come back in a wb_range_result that owns its memory (host memory, or device memory for wb_range_search_dev):
 * it does not depend on the index's scratch or lifetime, so a later search cannot clobber it, and it may outlive the
 * index. */
typedef struct wb_range_result wb_range_result;
/* index.range_search(x, thresh, params=...) [faiss-upstream].  f may be NULL (unfiltered); nprobe is ignored by flat
 * indices.  Synchronises once the hit counts are known; fills lims_host[0..nq] before returning. */
int wb_range_search(wb_index* h, wb_filter* f, int64_t nq, const float* q_host, float thresh, int64_t nprobe,
                    int64_t* lims_host, wb_range_result** out);
/* The same search with queries [nq, d] on the index's GPU, run on `stream`, which is synchronised once per query chunk
 * to read the hit counts; lims_host is filled before returning.  The result holds D and I in device memory of the
 * index's GPU, written on `stream`: no host copy is made. */
int wb_range_search_dev(wb_index* h, wb_filter* f, int64_t nq, const float* q_dev, float thresh, int64_t nprobe,
                        int64_t* lims_host, wb_range_result** out, void* stream);
/* Copy a result (host or device) out, lims_host[nq] entries each.  wb_range_result_copy synchronises the device of a
 * device result first; wb_range_result_copy_dev enqueues the copies on `stream` (for a device result: the stream it
 * was written on, or one ordered after it). */
int wb_range_result_copy(const wb_range_result* r, float* D_host, int64_t* I_host);
int wb_range_result_copy_dev(const wb_range_result* r, float* D_dev, int64_t* I_dev, void* stream);
int wb_range_result_free(wb_range_result* r); /* a device result's memory is freed on its GPU */

/* Sharded range search: merge the range results of the same nq queries from `nparts` parts (one per rank, rank p
 * holding the p-th contiguous slice of the rows).  Part p's hits for query q are entries
 * p * part_stride + [lims_p[q], lims_p[q+1]) of D_parts / I_parts (the padded all-gather layout), lims_p =
 * lims_parts_dev + p * (nq + 1).  lims_dev[nq + 1] is the sum of the parts' lims.  The result is the single-index
 * order: score descending, equal scores by part, then by order inside the part.  No synchronisation, no allocation. */
int wb_range_merge_dev(int device, int64_t nq, int64_t nparts, const int64_t* lims_parts_dev, int64_t part_stride,
                       const float* D_parts_dev, const int64_t* I_parts_dev, const int64_t* lims_dev, float* D_dev,
                       int64_t* I_dev, void* stream);

/* Merge `nparts` sorted partial results (layout [part][nq][k], e.g. the all-gathered per-GPU
 * top-k) into the global top-k.  Order: score desc, then part asc, then rank-in-part asc - with
 * contiguous row sharding that is exactly "lowest insertion position". */
int wb_merge_topk_dev(int device, int64_t nq, int64_t k, int64_t nparts, const float* D_parts_dev,
                      const int64_t* I_parts_dev, float* D_dev, int64_t* I_dev, void* stream);

/* ---- multi-GPU exchange over NVLink peer memory (one process per GPU) ---------------------------
 * The all-gather of the k candidates and the final merge as ONE kernel: every rank stores its rows
 * straight into the mailboxes of its peers (cudaIpc-mapped), raises per-query flags, waits for the
 * others' flags and merges.  Setup: wb_exch_create on every rank, exchange the 64-byte handles
 * (any host-side all-gather), wb_exch_open_peers.  Every rank must then call
 * wb_exch_merge_dev the same number of times with the same nq and k. */
typedef struct wb_exchange wb_exchange;
int wb_exch_create(int device, int rank, int world, int64_t max_queries, int64_t max_entries, wb_exchange** out);
int wb_exch_local_handle(wb_exchange* ex, void* handle64 /* 64 bytes out */);
int wb_exch_open_peers(wb_exchange* ex, const void* handles /* [world][64] */);
int wb_exch_merge_dev(wb_exchange* ex, int64_t nq, int64_t k, const float* D_local_dev, const int64_t* I_local_dev,
                      float* D_dev, int64_t* I_dev, void* stream);
/* index.search(x, k) on a row-sharded index (every rank passes the same queries): local search + exchange + merge.
 * Searches served by the scan kernel (flat batches <= 4, every IVF list scan) are ONE launch per GPU: the last CTA of
 * the scan merges the per-CTA lists, pushes the winners to the peers' mailboxes and emits the global top-k. */
int wb_exch_search(wb_index* h, wb_exchange* ex, int64_t nq, const float* q_host, int64_t k, int64_t nprobe,
                   float* D_host, int64_t* I_host);
int wb_exch_search_dev(wb_index* h, wb_exchange* ex, int64_t nq, const float* q_dev, int64_t k, int64_t nprobe,
                       float* D_dev, int64_t* I_dev, void* stream);
/* Filtered sharded search: every rank passes a filter built from the same selector over its own rows.  A rank whose
 * filter selects nothing still takes part in the exchange. */
int wb_exch_search_filtered(wb_index* h, wb_exchange* ex, wb_filter* f, int64_t nq, const float* q_host, int64_t k,
                            int64_t nprobe, float* D_host, int64_t* I_host);
int wb_exch_search_filtered_dev(wb_index* h, wb_exchange* ex, wb_filter* f, int64_t nq, const float* q_dev, int64_t k,
                                int64_t nprobe, float* D_dev, int64_t* I_dev, void* stream);
/* *timed_out = 1 when a kernel of this exchange gave up waiting for a peer (20 s): that search's results are invalid.
 * wb_exch_search checks it itself; callers of the _dev entry points check it after synchronising their stream. */
int wb_exch_status(wb_exchange* ex, int* timed_out);
/* exchange_merge_kernel launches so far (0 for searches whose exchange ran inside the scan kernel). */
int64_t wb_exch_launch_count(const wb_exchange* ex);
int wb_exch_free(wb_exchange* ex);

/* ---- in-process shard group: one index over several GPUs of one process (DESIGN.md "Shard group") -----------------
 * faiss index_cpu_to_all_gpus(index, co) with co.shard = True.  shards[0..n) are indices of the same kind (flat / IVF),
 * the same d (and nlist) and, for IVF, bit-identical centroids, each on its own GPU; shard s holds the s-th contiguous
 * slice of insertion order.  A search of the group returns exactly what one index holding all the rows in that order
 * returns (equal scores by shard, then by local order == global insertion position).
 *   - shards[0]'s GPU is the root: the _dev queries, the results and the caller's stream live there.
 *   - creation enables peer access between every ordered pair of the GPUs and builds one exchange (rank s of n) whose
 *     mailboxes are the other shards' device memory.  Searches of at most max_queries queries and max_entries = nq * k
 *     results run the exchange in the search kernels' tail; larger ones, and every search of a group with a pair of
 *     GPUs without peer access, search each shard locally, copy the results to the root (cudaMemcpyPeerAsync) and
 *     merge them there (wb_merge_topk_dev).  With n = 1 every call is the plain single-index call.
 *   - filters: NULL (unfiltered) or filters[s] = a wb_filter of shards[s] (NULL entries allowed), each built from the
 *     same selector over its shard's rows.
 *   - threads: searches of 1-4 queries (flat or IVF) are enqueued on every GPU from the calling thread.  Larger
 *     batches may take the tensor-core path (the flat scan, or the coarse step of IVF), which synchronises once: the
 *     group keeps one host thread per non-root shard (created here, joined by wb_group_free) that runs those shards'
 *     searches.  One group must not be
 *     used from two threads at the same time, and its shards must not be used elsewhere during a group call.
 *   - streams: wb_group_search runs on the shards' own streams and returns synchronised on every GPU; a time-out of
 *     the exchange (wb_exch_status) is its error.  wb_group_search_dev does not synchronise for searches of 1-4 queries:
 *     the non-root shards' streams wait for `stream`, copy q_dev to their GPUs, and `stream` waits for those copies,
 *     so the caller may overwrite q_dev with later work on `stream`; D_dev / I_dev are complete when `stream` is.
 *   - wb_group_free comes before the free of its shards; shards grow (add) only between group calls. */
typedef struct wb_group wb_group;
int wb_group_create(int n, wb_index* const* shards, int64_t max_queries, int64_t max_entries, wb_group** out);
int wb_group_search(wb_group* g, wb_filter* const* filters /* [n] or NULL */, int64_t nq, const float* q_host,
                    int64_t k, int64_t nprobe, float* D_host, int64_t* I_host);
int wb_group_search_dev(wb_group* g, wb_filter* const* filters, int64_t nq, const float* q_dev, int64_t k,
                        int64_t nprobe, float* D_dev, int64_t* I_dev, void* stream);
int wb_group_free(wb_group* g);

/* ---- row access ------------------------------------------------------------------------- */
/* index.reconstruct_batch(ids)   api/routes.py:1078 (after index.make_direct_map, :907).
 * Looks rows up by external id; an unknown id is an error (faiss raises). */
int wb_reconstruct_batch(wb_index* h, int64_t m, const int64_t* ids_host, float* out_host /* [m*d] */);
/* The insertion position of each id, -1 for an id the index does not hold (the shard lookup of a group's
 * reconstruct_batch: an unknown id is not an error here). */
int wb_lookup_ids(wb_index* h, int64_t m, const int64_t* ids_host, int64_t* pos_host /* [m] */);
/* Bulk export for faiss.write_index (feature_search_index.py:84): storage rows [start,start+n), their ids, and (IVF)
 * their list assignment.  Storage order is insertion order for flat indices and for IVF indices that have not been
 * searched / finalized yet; afterwards it is list by list.  Any output may be NULL. */
int wb_export_rows(wb_index* h, int64_t start, int64_t n, float* x_host, int64_t* ids_host, int32_t* assign_host);
/* Bulk import for faiss.read_index (feature_search_index.py:96) of an IVF index: rows with a
 * known list assignment (no coarse quantisation is run). */
int wb_ivf_add_preassigned(wb_index* h, int64_t n, const float* x_host, const int64_t* ids_host,
                           const int32_t* assign_host);

/* IVF: bring the inverted lists up to date now (K8: device histogram + scan + stable scatter, then the row store is
 * regrouped list by list).  faiss does this inside add_with_ids (invlists->add_entry); here it happens lazily at the
 * first search after an add, or when this is called (faiss.write_index does, feature_search_index.py:84).  After it,
 * wb_export_rows returns rows in STORAGE order = list by list, insertion order inside a list. */
int wb_ivf_finalize(wb_index* h);
int wb_ivf_list_offsets(wb_index* h, int64_t* list_off_host /* [nlist + 1] */, int* grouped_out);

/* ---- FeatureStore fast ingest (host only, no GPU needed) -----------------------------------------------
 * One pass over a WebdatasetStore shard `<media>-%06d.tar` (src/feature/store/webdataset_store.py:33-35):
 * tar headers are walked directly and the float32 payload of every `%010d.features.pyd` member
 * (pickle.dumps(ndarray (m,d) f32), :93-99) is located without creating python objects - replaces the
 * per-vector loop of iter_batch (:116-141) that feeds index.add_with_ids (feature_search_index.py:79-82).
 * A non-zero return means "use the python reader for this shard" (unknown pickle dialect, I/O error). */
int wb_tar_scan(const char* path, int64_t* rows_out, int64_t* members_out, int64_t* d_out);
int wb_tar_read(const char* path, int64_t d, int64_t cap, int64_t* ids_host, float* x_host, int64_t* rows_out);

/* ---- introspection for bench.py / tests --------------------------------------------------- */
/* TF32 tensor-pipe peak (TFLOP/s) of `device`, measured with the library's own instruction shape: back-to-back
 * tcgen05.mma.cta_group::2.kind::tf32 M=256 N=256 K=8 on every SM pair, no loads (the denominator of the
 * batched-search roofline; replaces nothing in the reference).  burst = best single launch of `iters` x 4 MMAs per
 * pair; sustained (optional) = the second half of `reps` back-to-back launches, i.e. under the settled power cap. */
int wb_tf32_peak(int device, int iters, int reps, double* tflops_burst_out, double* tflops_sustained_out);
/* Device pointer and row stride (floats) of the resident row store, for reading.  Writing rows through it is not
 * supported: the int8 image that 1-2 query flat searches stream would no longer match the rows. */
int wb_storage(wb_index* h, void** rows_dev, int64_t* ld);
/* Number of this library's kernels launched on behalf of `h` since creation. */
int64_t wb_launch_count(const wb_index* h);
/* Tensor-core path (batches of 5+ queries on large stores): epochs of the GEMM kernels launched so far, and how many
 * batches had to be repaired by the CUDA-core scan after a candidate-list overflow. */
int wb_gemm_stats(const wb_index* h, int64_t* epochs, int64_t* fallbacks);
/* IVF searches of up to 4 queries run as ONE cooperative launch: the coarse quantizer (faiss quantizer->search at the top
 * of IndexIVF::search, reached from /root/reference/src/index/feature_search_index.py:113) is the prologue of the list
 * scan.  Number of searches served that way so far (the others took the coarse scan + list scan launches). */
int64_t wb_ivf_fused_searches(const wb_index* h);
/* Flat searches of 1-2 queries over a large store stream an int8 image of it and re-score the candidates exactly in
 * fp32: the number of searches served by the image so far, and the (row, query) pairs they re-scored.  Waits for the
 * device.  (The name predates the int8 image, which replaced a bf16 one.) */
int wb_flat_bf16_stats(wb_index* h, int64_t* searches, int64_t* rescored);
/* Device bytes held by that image: 0 until a search builds it, then capacity x (16 + d rounded up to 16). */
int64_t wb_flat_image_bytes(const wb_index* h);
/* The CUDA-core scan plan of a search of nq queries with k results (k = 0: a range search) over the whole store
 * (gather = 0) or over nprobe probed lists (gather = 1): out = {queries per CTA, rows per warp, floats per staged row
 * chunk, chunks per row, ring stages}.  Chunks per row > 1 is the fallback for rows too wide for two whole-row stages.
 * Fails with the planner's message when no plan fits shared memory.  Read-only. */
int wb_scan_plan(wb_index* h, int64_t nq, int64_t k, int gather, int64_t nprobe, int out[5]);
/* Diagnostics (replaces nothing in the reference): with WB_PHASE_TS=1 in the environment the scan kernel's CTAs stamp
 * %globaltimer at their phase boundaries (scan.cuh ScanParams::phase_ts lists the 10 phases); this copies the stamps of
 * the first `ctas` CTAs of the last scan-served search, 16 uint64 per CTA (scripts/phase_times.py prints them). */
int wb_phase_stamps(wb_index* h, uint64_t* out_host, int ctas);
/* Device time (ms, CUDA events on the index's stream) of the scan kernel(s) of the last
 * wb_search / wb_search_dev call that finished; -1 if timing was off. */
int wb_set_timing(wb_index* h, int on);
float wb_last_scan_ms(wb_index* h);
/* Durations (ms) of the most recent timed scan launches, oldest first; returns how many (<= cap, <= 128). */
int wb_scan_ms_history(wb_index* h, float* out_ms, int cap);

#ifdef __cplusplus
}
#endif
#endif /* WISE_B200_H */
