/*
 * pecos_b200 C ABI  --  libpecos_b200_float32.so
 *
 * Drop-in replacement, on one NVIDIA B200 (sm_100a), for the two inference hot paths that the reference exports
 * from pecos/core/libpecos.cpp and binds through ctypes in pecos/core/base.py:
 *
 *   XR-Linear beam-search prediction   (libpecos.cpp:116-176,  base.py:799-976, :990-1095)
 *   HNSW dense search                  (libpecos.cpp:449-564,  base.py:1865-1964)
 *
 * The `c_*` entry points below have byte-identical signatures, argument meaning and ownership rules to the reference
 * symbols of the same name, so `pecos.core.base.corelib` can bind them unchanged (see INTEGRATION.md).
 * The `pb200_*` entry points are additions (device selection, device-resident batches for benchmarking, profiling
 * counters, host-only model inspection for tests).
 *
 * Conventions (same as the reference): no error codes.  The reference lets C++ exceptions escape `extern "C"`
 * (=> std::terminate); this library prints the message to stderr and calls abort().  There is NO CPU fallback:
 * every compute entry point requires a CUDA device and fails loudly without one.
 * `threads` arguments are accepted and ignored (the GPU schedules the work).
 */
#ifndef PECOS_B200_H_
#define PECOS_B200_H_

#include <stdbool.h>
#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

/* ---- plain-C views of scipy/numpy buffers: pecos/core/utils/matrix.hpp:43-73, ctypes mirrors base.py:177-310 ---- */
typedef struct {
    uint32_t rows, cols;
    uint64_t* col_ptr;
    uint32_t* row_idx;
    float* val;
} ScipyCscF32;

typedef struct {
    uint32_t rows, cols;
    uint64_t* row_ptr;
    uint32_t* col_idx;
    float* val;
} ScipyCsrF32;

typedef struct {
    uint32_t rows, cols;
    float* val; /* row-major */
} ScipyDrmF32;

/* Result allocator callback (matrix.hpp:47; Python side base.py:407-478):
 *   pred_alloc(is_col_major=false, rows, cols, nnz, &indices /u32[nnz]/, &indptr /u64[rows+1]/, &data /f32[nnz]/)
 * Called exactly once per predict call, from the calling thread. */
typedef void (*py_sparse_allocator_t)(bool, uint64_t, uint64_t, uint64_t, void*, void*, void*);

/* ======================================= XR-Linear (reference-compatible) ======================================= */

/* libpecos.cpp:116  model_path = the `ranker/` folder of an XLinearModel; default layer type. */
void* c_xlinear_load_model_from_disk(const char* model_path);
/* libpecos.cpp:121  weight_matrix_type in {0 CSC, 1 HASH_CHUNKED, 2 BINARY_SEARCH_CHUNKED} (base.py:49).
 * All three are served by the one HBM chunk layout; the requested type is remembered and reported back by
 * c_xlinear_get_layer_type (pecos/xmc/base.py:1736-1743 gates features on it).  Rejects mmap folders. */
void* c_xlinear_load_model_from_disk_ext(const char* model_path, int weight_matrix_type);
/* libpecos.cpp:128  folder written by c_xlinear_compile_mmap_model (W/C/perm.mmap_store per layer). */
void* c_xlinear_load_mmap_model_from_disk(const char* model_path, const bool lazy_load);
/* libpecos.cpp:140 */
/* libpecos.cpp:133-138  npz model folder (ranker/) -> the reference's mmap format (param.json with is_mmap = true; per layer
 * W.mmap_store = chunked matrix, C.mmap_store, perm.mmap_store when the tree is not contiguously ordered; formats: SURVEY.md
 * Appendix B).  Host-only: needs no GPU.  The output loads in the reference library and here. */
void c_xlinear_compile_mmap_model(const char* model_path, const char* mmap_model_path);
void c_xlinear_destruct_model(void* ptr);
/* libpecos.cpp:147  attr in {"depth","nr_features","nr_labels","nr_codes"} (inference.hpp:2367-2379). */
uint32_t c_xlinear_get_int_attr(void* ptr, const char* attr);
/* libpecos.cpp:152 */
int c_xlinear_get_layer_type(void* ptr, int layer_depth);
/* libpecos.cpp:158-175  0 / NULL overrides mean "use the value stored with each layer". */
void c_xlinear_predict_csr_f32(void* ptr, const ScipyCsrF32* input_x, const uint32_t overridden_beam_size,
                               const char* overridden_post_processor_str, const uint32_t overridden_only_topk,
                               const int threads, py_sparse_allocator_t pred_alloc);
/* libpecos.cpp:176 */
void c_xlinear_predict_drm_f32(void* ptr, const ScipyDrmF32* input_x, const uint32_t overridden_beam_size,
                               const char* overridden_post_processor_str, const uint32_t overridden_only_topk,
                               const int threads, py_sparse_allocator_t pred_alloc);

/* libpecos.cpp:179-198  predict_on_selected_outputs: scores of exactly the (query, label) pairs of the CSR pattern
 * selected_outputs_csr (rows x nr_labels; values ignored), pushed through the hierarchy (transform + combine per layer), no
 * top-k (HierarchicalMLModel::predict_on_selected_outputs, pecos/core/xmc/inference.hpp:2507-2571).  Result: CSR with the
 * selected rows' lengths; a row's entries come in the reference's order (parents in the previous layer's order, children
 * in C's column order); labels without a path to the root leave zero entries at the row's end, like the reference.
 * The reference serves this from CSC layers only (inference.hpp:2143-2147; its Python gates on get_layer_type == CSC):
 * here every handle can, and the arithmetic is the beam-search kernels' (bit-identical raw scores). */
void c_xlinear_predict_on_selected_outputs_csr_f32(void* ptr, const ScipyCsrF32* X, const ScipyCsrF32* selected_outputs_csr,
                                                   const char* overridden_post_processor_str, const int threads,
                                                   py_sparse_allocator_t pred_alloc);
void c_xlinear_predict_on_selected_outputs_drm_f32(void* ptr, const ScipyDrmF32* X, const ScipyCsrF32* selected_outputs_csr,
                                                   const char* overridden_post_processor_str, const int threads,
                                                   py_sparse_allocator_t pred_alloc);

/* libpecos.cpp:32-36  one npz layer folder (param.json + W.npz [+ C.npz]) -> the single-layer mmap format read by
 * c_mlmodel_load_mmap_model (MLModel<csc_t>::save_mmap, inference.hpp:2274-2289).  Host-only, needs no GPU. */
void c_mlmodel_compile_mmap_model(const char* model_path, const char* mmap_model_path);
/* libpecos.cpp:37-113  Single-layer handles over ONE mmap-format MLModel folder (MLModel<csc_t>::save_mmap,
 * pecos/core/xmc/inference.hpp:2274-2289: param.json with is_mmap = true + W.mmap_store + C.mmap_store in csc_t's mmap
 * format, pecos/core/utils/matrix.hpp:386-407).  c_mlmodel_get_int_attr: nr_labels | nr_codes | nr_features.
 * c_mlmodel_predict_*: csr_codes = previous layer's prediction or NULL (= ones(rows x nr_codes), no combine);
 * overridden_post_processor NULL / overridden_only_topk 0 = the values stored with the layer.
 * Folders written by this library's or by the reference's c_mlmodel_compile_mmap_model are interchangeable. */
void* c_mlmodel_load_mmap_model(const char* model_path, const bool lazy_load);
void c_mlmodel_destruct_model(void* ptr);
uint32_t c_mlmodel_get_int_attr(void* ptr, const char* attr);
void c_mlmodel_predict_csr_f32(void* ptr, const ScipyCsrF32* input_x, const ScipyCsrF32* csr_codes,
                               const char* overridden_post_processor, const uint32_t overridden_only_topk, const int num_threads,
                               py_sparse_allocator_t pred_alloc);
void c_mlmodel_predict_drm_f32(void* ptr, const ScipyDrmF32* input_x, const ScipyCsrF32* csr_codes,
                               const char* overridden_post_processor, const uint32_t overridden_only_topk, const int num_threads,
                               py_sparse_allocator_t pred_alloc);
void c_mlmodel_predict_on_selected_outputs_csr_f32(void* ptr, const ScipyCsrF32* input_x, const ScipyCsrF32* selected_outputs_csr,
                                                   const ScipyCsrF32* csr_codes, const char* overridden_post_processor,
                                                   const int num_threads, py_sparse_allocator_t pred_alloc);
void c_mlmodel_predict_on_selected_outputs_drm_f32(void* ptr, const ScipyDrmF32* input_x, const ScipyCsrF32* selected_outputs_csr,
                                                   const ScipyCsrF32* csr_codes, const char* overridden_post_processor,
                                                   const int num_threads, py_sparse_allocator_t pred_alloc);

/* libpecos.cpp:201-235  One layer of the python prediction chain (pecos/xmc/base.py:890-949, is_predict_only=False
 * models): W ((nr_features [+1 bias row]) x nr_labels) and C (nr_labels x nr_codes) are handed over on every call;
 * csr_codes = the previous layer's prediction (rows x nr_codes, entries consumed in stored order) or NULL for the first
 * layer (= ones, no combine).  post_processor_str must be given; only_topk as passed (0 keeps nothing, like the
 * reference).  The chunked HBM layout of (W, C, bias) is built on first use and kept in a small LRU cache keyed by the
 * matrices' shapes, value pointer and a sampled content fingerprint (PB200_LAYER_CACHE entries, default 8): the
 * matrices are assumed immutable while cached (pb200_layer_cache_clear() drops them).
 * Validated on a B200 (tests/test_single_layer_gpu.py); oracle pinned against the reference in tests/test_oracle_cpu.py. */
void c_xlinear_single_layer_predict_csr_f32(const ScipyCsrF32* input_x, const ScipyCsrF32* csr_codes, ScipyCscF32* W,
                                            ScipyCscF32* C, const char* post_processor_str, const uint32_t only_topk,
                                            const int num_threads, const float bias, py_sparse_allocator_t pred_alloc);
void c_xlinear_single_layer_predict_drm_f32(const ScipyDrmF32* input_x, const ScipyCsrF32* csr_codes, ScipyCscF32* W,
                                            ScipyCscF32* C, const char* post_processor_str, const uint32_t only_topk,
                                            const int num_threads, const float bias, py_sparse_allocator_t pred_alloc);
/* libpecos.cpp:238-273  the same single layer, scores of exactly the (query, label) pairs of selected_outputs_csr
 * (MLModel::predict_on_selected_outputs, inference.hpp:2129-2224; pecos/xmc/base.py:1003 = predict_on_selected_outputs of
 * is_predict_only=False models).  Result: the pattern of selected_outputs_csr, values = transformed (+ combined) scores. */
void c_xlinear_single_layer_predict_on_selected_outputs_csr_f32(const ScipyCsrF32* input_x, const ScipyCsrF32* selected_outputs_csr,
                                                                const ScipyCsrF32* csr_codes, ScipyCscF32* W, ScipyCscF32* C,
                                                                const char* post_processor_str, const int num_threads,
                                                                const float bias, py_sparse_allocator_t pred_alloc);
void c_xlinear_single_layer_predict_on_selected_outputs_drm_f32(const ScipyDrmF32* input_x, const ScipyCsrF32* selected_outputs_csr,
                                                                const ScipyCsrF32* csr_codes, ScipyCscF32* W, ScipyCscF32* C,
                                                                const char* post_processor_str, const int num_threads,
                                                                const float bias, py_sparse_allocator_t pred_alloc);
/* drops every cached single-layer engine; returns how many were held */
uint32_t pb200_layer_cache_clear(void);
/* out[0] = entries held, out[1] = hits, out[2] = misses (builds) since load */
void pb200_layer_cache_info(uint64_t* out);

/* ========================================= HNSW (reference-compatible) ========================================== */

/* libpecos.cpp:471-480  model_dir = ".../c_model" holding config.json + index.mmap_store (hnsw.hpp:534-552). */
void* c_ann_hnsw_load_drm_ip_f32(const char* model_dir, const bool lazy_load);
void* c_ann_hnsw_load_drm_l2_f32(const char* model_dir, const bool lazy_load);
/* libpecos.cpp:492-499 */
void c_ann_hnsw_destruct_drm_ip_f32(void* model_ptr);
void c_ann_hnsw_destruct_drm_l2_f32(void* model_ptr);
/* libpecos.cpp:501-524  opaque scratch pool; here: pre-allocated per-query device scratch. */
void* c_ann_hnsw_searchers_create_drm_ip_f32(void* model_ptr, uint32_t num_searcher);
void* c_ann_hnsw_searchers_create_drm_l2_f32(void* model_ptr, uint32_t num_searcher);
void c_ann_hnsw_searchers_destruct_drm_ip_f32(void* searchers_ptr);
void c_ann_hnsw_searchers_destruct_drm_l2_f32(void* searchers_ptr);
/* libpecos.cpp:527-564  caller passes zeroed Q x topk arrays; row q gets its neighbours in ascending distance. */
void c_ann_hnsw_predict_drm_ip_f32(void* model_ptr, const ScipyDrmF32* pX, uint32_t* ret_idx, float* ret_val,
                                   uint32_t efS, uint32_t topk, int32_t threads, void* searchers_ptr);
void c_ann_hnsw_predict_drm_l2_f32(void* model_ptr, const ScipyDrmF32* pX, uint32_t* ret_idx, float* ret_val,
                                   uint32_t efS, uint32_t topk, int32_t threads, void* searchers_ptr);
/* Sparse (csr) indices: HNSW<float, FeatVecSparse{IP,L2}Simd<uint32_t, float>> (libpecos.cpp:449-450, :479-480, :497-498,
 * :508-513, :522-523, :563-564; distances pecos/core/ann/feat_vectors.hpp:186-210 + distance_impl/common.hpp:15-86).  Rows of the
 * index and of the queries carry strictly ascending column indices (what scipy's sort_indices()/sum_duplicates() give and
 * the reference's block intersection assumes).  The reference's sparse "l2" evaluates to -2<x,y> (feat_vectors.hpp:186-192: the
 * squared norms are taken as do_l2_distance_simd(x, x) = 0); this library returns the same values. */
void* c_ann_hnsw_load_csr_ip_f32(const char* model_dir, const bool lazy_load);
void* c_ann_hnsw_load_csr_l2_f32(const char* model_dir, const bool lazy_load);
void c_ann_hnsw_destruct_csr_ip_f32(void* model_ptr);
void c_ann_hnsw_destruct_csr_l2_f32(void* model_ptr);
void* c_ann_hnsw_searchers_create_csr_ip_f32(void* model_ptr, uint32_t num_searcher);
void* c_ann_hnsw_searchers_create_csr_l2_f32(void* model_ptr, uint32_t num_searcher);
void c_ann_hnsw_searchers_destruct_csr_ip_f32(void* searchers_ptr);
void c_ann_hnsw_searchers_destruct_csr_l2_f32(void* searchers_ptr);
void c_ann_hnsw_predict_csr_ip_f32(void* model_ptr, const ScipyCsrF32* pX, uint32_t* ret_idx, float* ret_val,
                                   uint32_t efS, uint32_t topk, int32_t threads, void* searchers_ptr);
void c_ann_hnsw_predict_csr_l2_f32(void* model_ptr, const ScipyCsrF32* pX, uint32_t* ret_idx, float* ret_val,
                                   uint32_t efS, uint32_t topk, int32_t threads, void* searchers_ptr);

/* ============================================ pecos_b200 additions ============================================== */

const char* pb200_version(void);
/* Number of visible CUDA devices (0 when there is none; never aborts). */
int pb200_device_count(void);
/* Device used by subsequently created model handles (default 0). Returns 0 on success. */
int pb200_set_device(int device);
int pb200_get_device(void);
/* Pinned host memory for end-to-end runs (cudaMallocHost / cudaFreeHost). */
void* pb200_host_alloc(size_t bytes);
void pb200_host_free(void* ptr);
/* Overwrite a scratch buffer larger than L2 (126 MB) so the next timed iteration starts cold. */
void pb200_l2_flush(void);

/* Device-resident query batch: upload once, run the layers with inputs already in HBM, fetch when wanted. */
void pb200_xlinear_resident_upload_csr(void* ptr, const ScipyCsrF32* input_x);
/* Returns the device time (ms, CUDA events on the engine's stream) of one pass over the resident batch. */
double pb200_xlinear_resident_predict(void* ptr, uint32_t overridden_beam_size, const char* overridden_post_processor_str,
                                      uint32_t overridden_only_topk, int collect_stats);
void pb200_xlinear_resident_fetch(void* ptr, py_sparse_allocator_t pred_alloc);

/* Index sharding of the leaf layer over `shard_world` GPUs (one process per GPU; SURVEY.md 8e).  Upper layers are
 * replicated, so every rank walks the identical global beam; rank r keeps the weights of a contiguous range of leaf
 * chunks and scores only those.  weight_matrix_type < 0 loads an mmap folder.
 *   local:  runs all layers, writes this rank's top-k {u64 key, u32 id, f32 value}[rows][stride] and u32 count[rows]
 *           into CALLER-OWNED DEVICE buffers (the send buffers of ONE ncclAllGather); returns stride (<= capacity).
 *   merge:  gathered [world][rows][stride] lists -> global top-k, returned through pred_alloc like c_xlinear_predict_*.
 * The result is bit-identical to the unsharded prediction (keys carry the candidate's global position). */
void* pb200_xlinear_load_sharded(const char* model_path, int weight_matrix_type, uint32_t shard_rank, uint32_t shard_world);
void pb200_xlinear_get_shard(void* ptr, uint32_t* out /* rank, world, leaf_chunk_begin, leaf_chunk_end */);
uint32_t pb200_xlinear_sharded_local_csr(void* ptr, const ScipyCsrF32* input_x, uint32_t overridden_beam_size,
                                         const char* overridden_post_processor_str, uint32_t overridden_only_topk,
                                         uint32_t stride_capacity, void* keys_dev, void* ids_dev, void* vals_dev, void* cnt_dev);
void pb200_xlinear_sharded_merge(void* ptr, uint32_t world, uint32_t rows, uint32_t stride, uint32_t overridden_only_topk,
                                 const void* g_keys, const void* g_ids, const void* g_vals, const void* g_cnt,
                                 py_sparse_allocator_t pred_alloc);

/* Packed form of the exchange: rec_dev / g_rec hold 16-byte records {u64 key, u32 id, f32 value} ([rows][stride] locally,
 * [world][rows][stride] gathered); key == 0 marks an empty slot, so no count array travels and the whole exchange is ONE
 * ncclAllGather of one buffer (16 B x rows x stride per rank). */
uint32_t pb200_xlinear_sharded_local_csr_packed(void* ptr, const ScipyCsrF32* input_x, uint32_t overridden_beam_size,
                                                const char* overridden_post_processor_str, uint32_t overridden_only_topk,
                                                uint32_t stride_capacity, void* rec_dev);
void pb200_xlinear_sharded_merge_packed(void* ptr, uint32_t world, uint32_t rows, uint32_t stride, uint32_t overridden_only_topk,
                                        const void* g_rec, py_sparse_allocator_t pred_alloc);

/* Per-layer kernel timing (CUDA events) and algorithmic-byte counters.
 *   profile: out[2*d] = chunk-score kernel ms, out[2*d+1] = top-k kernel ms   (accumulated since reset)
 *   stats:   out[7*d + {0..6}] = chunks, sum R, sum m, sum e, sum c, sum nnz(x), sum beam-out   (last stats pass) */
void pb200_xlinear_set_profile(void* ptr, int on);
/* Kernel generation selector for A/B tests (results are identical): 0 = row-list streaming + block-wide sort,
 * 1 = default (feature-map kernels + warp top-k; query-warp kernel for beams of many narrow chunks), 2 = feature-map
 * lookups with one warp per chunk only, 3 = query-warp kernel wherever it is eligible, 4 = as 1 but the warp top-k
 * evaluates the post-processor for every candidate (no single-precision estimate filter), 5 = as 1 plus the EXPERIMENTAL
 * chunk-major score kernel on eligible layers (written without GPU access at the end of round 1, not validated yet).
 * Returns 1 when every layer has a feature map (PB200_FEATMAP_MB caps their total size at load time, default 32768). */
int pb200_xlinear_set_lookup(void* ptr, int on);
void pb200_xlinear_reset_profile(void* ptr);
void pb200_xlinear_get_profile(void* ptr, double* out);
/* out[2*depth]: per layer {score kernel, top-k kernel} of the last call.  Score: 0 row-list streaming, 1 feature-map
 * lookup (xl_chunk_scores_kernel), 2 dense, 3 xl_query_warp_scores_kernel, 4 xl_cm_scores_kernel (experimental).  Top-k: 0 xl_topk_kernel, 1 xl_topk_warp_kernel,
 * 2 xl_topk_filter_kernel. */
void pb200_xlinear_get_kernel_ids(void* ptr, int* out);
void pb200_xlinear_get_stats(void* ptr, uint64_t* out);
uint64_t pb200_xlinear_launches(void* ptr);
uint64_t pb200_xlinear_model_bytes(void* ptr);
/* Replicas held by a handle: 1, or one per entry of PB200_DEVICES ("0,1,..." | "all", read at load time).  With replicas a
 * c_xlinear_predict_* / c_ann_hnsw_predict_* call splits its rows over the devices (one host thread + stream each) and
 * concatenates the results in row order -- the multi-GPU form of the reference's OpenMP loop over queries
 * (pecos/core/xmc/inference.hpp:969-1005, pecos/core/libpecos.cpp:540-548). */
uint32_t pb200_xlinear_replicas(void* ptr);
uint32_t pb200_hnsw_replicas(void* model_ptr);

/* HNSW: device-resident query batch, search-kernel time (ms, CUDA events), algorithmic counters of the last search
 *   counters out[4] = {distance evaluations, level-0 expansions, upper-level neighbourhood reads, queries}
 *   info     out[8] = {num_node, feat_dim, maxM, maxM0, max_level, init_node, index bytes in HBM, kernel launches} */
void pb200_hnsw_resident_upload(void* model_ptr, const ScipyDrmF32* pX);
double pb200_hnsw_resident_predict(void* model_ptr, uint32_t efS, uint32_t topk);
void pb200_hnsw_resident_fetch(void* model_ptr, uint32_t* ret_idx, float* ret_val);
void pb200_hnsw_get_counters(void* model_ptr, uint64_t* out);
/* sparse (csr) indices: resident csr batch; stored entries (8 bytes each) of the base rows evaluated by the last search */
void pb200_hnsw_resident_upload_csr(void* model_ptr, const ScipyCsrF32* pX);
uint64_t pb200_hnsw_sparse_entries(void* model_ptr);
/* libpecos.cpp:482-490  c_ann_hnsw_save_drm_{ip,l2}_f32(model_ptr, model_dir): for an index loaded by THIS library the saved
 * form is what it was loaded from (config.json + index.mmap_store are copied to model_dir).
 *
 * Handles are library-specific: an index TRAINED by the reference (c_ann_hnsw_train_* is not served here) is a reference
 * handle, but after the overlay the reference's Python passes it to this library's destruct / searchers / predict / save.
 * pb200_hnsw_set_foreign registers the reference's own functions for one index type (0 = drm ip, 1 = drm l2, 2 = csr ip, 3 = csr l2); handles and searcher tokens
 * that were not created here are forwarded to them (pecos_b200.integration.overlay does this).  Without the registration a
 * foreign handle is a fatal error with a clear message. */
void c_ann_hnsw_save_drm_ip_f32(void* model_ptr, const char* model_dir);
void c_ann_hnsw_save_drm_l2_f32(void* model_ptr, const char* model_dir);
void c_ann_hnsw_save_csr_ip_f32(void* model_ptr, const char* model_dir);
void c_ann_hnsw_save_csr_l2_f32(void* model_ptr, const char* model_dir);
void pb200_hnsw_set_foreign(int metric, void* destruct, void* searchers_create, void* searchers_destruct, void* predict, void* save);

/* base-vector rows kept in flight per warp by the bulk-copy (TMA) ring: 0 = direct loads, 4 (default) or 8; returns the
 * value in effect.  Results are identical for every setting. */
int pb200_hnsw_set_stages(void* model_ptr, int stages);
void pb200_hnsw_get_info(void* model_ptr, uint64_t* out);
/* Host-only ingest check of an HNSW index folder (<model>/c_model), no GPU needed: the loader's validation of config.json
 * (hnsw_t string of the requested metric / data type, version) and of index.mmap_store (record sizes; sparse: record offsets,
 * strictly ascending in-range indices).  metric 0 = ip, 1 = l2; sparse 0 = drm, 1 = csr.  Returns 0 and
 * out[8] = {num_node, feat_dim, maxM, maxM0, max_level, init_node, stored vector entries, level-0 degree sum}, or 1 (reason on stderr). */
int pb200_hnsw_host_info(const char* model_dir, int metric, int sparse, uint64_t* out);
/* Distance work of the GPU builder for SPARSE (csr) indices (pecos_b200/hnsw_build.py).  All pointers are CALLER-OWNED DEVICE
 * buffers; the kernels are enqueued on `stream` (a cudaStream_t, e.g. torch.cuda.current_stream().cuda_stream) of `device` and
 * the calls return without synchronising.  Distances have the reference's bits (FeatVecSparse{IP,L2}Simd::distance: ordered
 * sum of the matched products; ip = 1 - dot, l2 = -2 dot); orders are by (distance, id).  metric 0 = ip, 1 = l2.  Rows are a
 * canonical csr (row_ptr i64 [n+1], col_idx i32 ascending per row, val f32).  Both return 0, or 1 (reason on stderr).
 *   knn:    for every row q < n, its k nearest rows among 0..q-1.  post_ptr i64 [cols+1] / post_entries {i32 row, f32 value}
 *           [nnz] are the posting lists (csc, rows ascending), self_pos i64 [nnz] the position of every csr entry in its
 *           posting list, cursor i64 [nnz] scratch.  out_keys i64 [n][k] ascending: (orderable(distance) << 32 | row) with
 *           the sign bit flipped (signed order = key order); INT64_MAX pads rows with fewer than k earlier rows.
 *   select: the neighbour-selection heuristic (hnsw.hpp:556-592) for n nodes: cand i64 [n][C] global row ids (-1 = empty),
 *           ascending by (cand_d f32 [n][C], id); keep u8 [n][C] receives 1 for the kept candidates (at most cap). */
int pb200_hnsw_build_sparse_knn(int device, void* stream, uint32_t n, uint32_t k, int metric, const void* row_ptr,
                                const void* col_idx, const void* val, const void* post_ptr, const void* post_entries,
                                const void* self_pos, void* cursor, void* out_keys);
int pb200_hnsw_build_sparse_select(int device, void* stream, uint32_t n, uint32_t C, uint32_t cap, int metric,
                                   const void* row_ptr, const void* col_idx, const void* val, const void* cand,
                                   const void* cand_d, void* keep);
/* A query whose candidate queue outgrows the per-warp scratch (PB200_HNSW_VCAP entries, default 32768) makes the engine re-run
 * the batch with twice the capacity (up to num_node + 1, which cannot overflow) -- this counts those re-runs. */
uint32_t pb200_hnsw_vcap_retries(void* model_ptr);

/* Host-only model ingest (no GPU needed): loads + builds the chunk layout, for layout tests.
 *   kind: 0 = npz folder, 1 = mmap folder.  dims out[8] = {w_rows, n_cols, out_cols, n_chunks, c_max, meta_len,
 *   n_entries, label_of_col_len}.  export copies the arrays into caller buffers (any may be NULL). */
void* pb200_xlinear_host_load(const char* model_path, int kind);
/* host-only: the one-layer model c_xlinear_single_layer_predict_* builds from in-memory W / C (same handle type) */
void* pb200_xlinear_host_from_csc(const ScipyCscF32* W, const ScipyCscF32* C, float bias);
void pb200_xlinear_host_free(void* hptr);
uint32_t pb200_xlinear_host_depth(void* hptr);
void pb200_xlinear_host_layer_dims(void* hptr, uint32_t layer, uint64_t* out);
void pb200_xlinear_host_layer_export(void* hptr, uint32_t layer, void* chunks32, uint32_t* meta, void* entries8,
                                     uint32_t* label_of_col);

#ifdef __cplusplus
}
#endif
#endif /* PECOS_B200_H_ */
