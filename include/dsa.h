/*
 * libdsa — C ABI of the B200-native engine behind DynamicSparseArrays.jl's hot path.
 *
 * The reference (atoptima/DynamicSparseArrays.jl v0.7.2) is pure Julia and has no FFI /
 * plugin boundary (SURVEY.md §8b); this header is the boundary a maintainer binds with
 * `ccall` from vector.jl / matrix.jl / buffer.jl (INTEGRATION.md shows the stubs).  Every
 * entry point cites the reference seam (file:line under /root/reference/src) it replaces.
 *
 * Conventions
 *   - plain C: opaque handles, `int64_t*` / `double*` buffers, sizes; no C++/torch types.
 *   - keys are Int64, values Float64 (the device path of BASELINE.json's configs).
 *   - every call returns 0 on success or a DSA_ERR_* code; dsa_last_error() gives the
 *     thread-local message.  The glue re-throws the reference's exception type:
 *     DSA_ERR_ARGUMENT -> ArgumentError, DSA_ERR_BOUNDS -> BoundsError,
 *     DSA_ERR_ERROR -> ErrorException.  A failed call leaves the structure unchanged.
 *   - host-pointer entry points copy in/out on the handle's stream and are synchronous on
 *     return; `_d` variants take DEVICE pointers (same layout) and only enqueue + sync
 *     where a host decision is needed.
 *   - positions in exports are 1-based, exactly like the reference's `semaphores` vector.
 *   - a handle is not thread-safe (neither is the reference); distinct handles are
 *     independent.  All work of a handle runs on one CUDA stream (dsa_*_set_stream).
 *   - there is NO CPU fallback: without a CUDA device every compute call fails with
 *     DSA_ERR_CUDA.
 */
#ifndef DSA_H
#define DSA_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define DSA_OK 0
#define DSA_ERR_ARGUMENT 1 /* Julia ArgumentError  (pcsr.jl:208, vector.jl:50, pcsr.jl:440)            */
#define DSA_ERR_BOUNDS 2   /* Julia BoundsError    (pcsr.jl:190, moves.jl:10-11)                        */
#define DSA_ERR_ERROR 3    /* Julia ErrorException (pcsr.jl:299, matrix.jl:73,84,96,105,127, writes.jl:39) */
#define DSA_ERR_CUDA 10
#define DSA_ERR_OOM 11
#define DSA_ERR_INTERNAL 12

/* combine operators of the builders (vector.jl:44, pcsr.jl:354): left fold in input order */
#define DSA_COMBINE_ADD 0
#define DSA_COMBINE_MUL 1
#define DSA_COMBINE_LAST 2
#define DSA_COMBINE_FIRST 3
#define DSA_COMBINE_MIN 4
#define DSA_COMBINE_MAX 5

#define DSA_COLMAJOR 0
#define DSA_ROWMAJOR 1

typedef struct dsa_vec dsa_vec_t;       /* DynamicSparseVector{Int64,Float64}      (vector.jl:1-4)  */
typedef struct dsa_matrix dsa_matrix_t; /* DynamicSparseMatrix{Int64,Int64,Float64} (matrix.jl:1-8) */

/* ---------------------------------------------------------------- library -------------- */
int dsa_version(void);
const char* dsa_last_error(void);
int dsa_device_count(int* count_out);
int dsa_set_device(int device);

/* ---------------------------------------------------------------- host logic (no GPU) -- */
/* _pma geometry (pma.jl:42-55,64,88): out = {capacity, segment_capacity, nb_segments, height}; n == 0 -> empty ctor */
int dsa_pma_geometry(int64_t nb_elements, int64_t* out4);
/* integer count bounds per level from the Float64 thresholds of pma.jl:119-123; mn/mx have height+1 entries */
int dsa_level_bounds(int64_t segment_capacity, int64_t height, int64_t* mn, int64_t* mx);
/* closed form of spread! (moves.jl:120-172): 0-based offset of the element of rank r in a window of c cells holding m elements */
int64_t dsa_spread_dest(int64_t c, int64_t m, int64_t r);
/* inverse: rank of the element stored at 0-based offset p, or -1 if spread! leaves a gap there */
int64_t dsa_spread_rank(int64_t c, int64_t m, int64_t p);
/* column-map planning of a batch (addcolumn! slot logic, pcsr.jl:148-169, replayed in arrival order).
 * in : slot_key/slot_live[nslots] = current col_keys with tombstones; new_keys[nnew] = distinct absent keys in first-arrival order
 * out: out_key/out_live/out_old[<= nslots+nnew] = new col_keys; out_old[s] = old 1-based slot of new slot s (0 = new or tombstone)
 * returns the new slot count (or a negative error) */
int64_t dsa_colmap_plan(const int64_t* slot_key, const uint8_t* slot_live, int64_t nslots, const int64_t* new_keys, int64_t nnew,
                        int64_t* out_key, uint8_t* out_live, int64_t* out_old);

/* ---------------------------------------------------------------- DynamicSparseVector -- */
/* PackedMemoryArray(K,T; expected_nb_elems) (pma.jl:86) wrapped as dynamicsparsevec(Int[],Float64[]) */
int dsa_vec_create(int64_t expected_nb_elems, dsa_vec_t** out);
/* dynamicsparsevec(I, V, combine, n) (vector.jl:38-62): stable sort, left-fold combine, bulk build; zeros are kept */
int dsa_vec_build(const int64_t* keys, const double* vals, int64_t n, int combine, int64_t len, int len_given, dsa_vec_t** out);
int dsa_vec_destroy(dsa_vec_t* v);
int dsa_vec_clone(const dsa_vec_t* v, dsa_vec_t** out); /* deepcopy (sparsevector.jl:163-182) */
int dsa_vec_set_stream(dsa_vec_t* v, void* cuda_stream);
/* batched setindex! (vector.jl:76-81 -> pma.jl:196-213): last writer wins, value 0.0 deletes, n = max(n, key) for non-zeros */
int dsa_vec_set_batch(dsa_vec_t* v, const int64_t* keys, const double* vals, int64_t n);
int dsa_vec_set_batch_d(dsa_vec_t* v, const int64_t* d_keys, const double* d_vals, int64_t n);
/* batched getindex (vector.jl:72 -> pma.jl:189-193): value or 0.0 */
int dsa_vec_get_batch(dsa_vec_t* v, const int64_t* keys, int64_t n, double* out);
/* out = {capacity, segment_capacity, nb_segments, nnz, height, n(length)} (pma.jl:8-24, vector.jl:2) */
int dsa_vec_info(const dsa_vec_t* v, int64_t* out6);
/* nonzeroinds / nonzeros / iterate (vector.jl:93-109, pma.jl:165-180): ascending; two-call size query via count_out */
int dsa_vec_nonzeros(dsa_vec_t* v, int64_t* keys_out, double* vals_out, int64_t cap, int64_t* count_out);
/* shrink_size! (vector.jl:64): n = max stored key */
int dsa_vec_shrink_size(dsa_vec_t* v, int64_t* n_out);
/* raw layout dump for parity: occupied[capacity] (1 = element, 0 = nothing), keys, vals */
int dsa_vec_export(dsa_vec_t* v, uint8_t* occupied, int64_t* keys, double* vals);

/* ---------------------------------------------------------------- DynamicSparseMatrix -- */
/* dynamicsparse(Int, Int, Float64; fill_mode = false) (matrix.jl:31-41): two empty MappedPackedCSC */
int dsa_matrix_create(dsa_matrix_t** out);
/* dynamicsparse(I, J, V, m, n) (matrix.jl:15-19) and closefillmode! (matrix.jl:126-134; the Dict buffer of buffer.jl stays in the
 * glue and is flushed as COO): builds BOTH orientations (pcsr.jl:354-449). Duplicates folded with `combine` in input order. */
int dsa_matrix_build_coo(const int64_t* rows, const int64_t* cols, const double* vals, int64_t n, int64_t m, int64_t ncols,
                         int dims_given, int combine, dsa_matrix_t** out);
int dsa_matrix_destroy(dsa_matrix_t* A);
int dsa_matrix_clone(const dsa_matrix_t* A, dsa_matrix_t** out); /* deepcopy (pcsr.jl:70-71) */
int dsa_matrix_set_stream(dsa_matrix_t* A, void* cuda_stream);
/* batched setindex! (matrix.jl:43-62 -> pcsr.jl:341-347 twice): LWW, 0.0 deletes, absent rows/columns are created
 * (addcolumn!, pcsr.jl:148-169), m/n grow on non-zeros. In-array keys must be >= 1 (key 0 is the semaphore key, pcsr.jl:23). */
int dsa_matrix_set_batch(dsa_matrix_t* A, const int64_t* rows, const int64_t* cols, const double* vals, int64_t n);
int dsa_matrix_set_batch_d(dsa_matrix_t* A, const int64_t* d_rows, const int64_t* d_cols, const double* d_vals, int64_t n);
/* The buffered-write flush, double-buffered: dsa_matrix_stage_batch starts the host->device copy of a batch on the handle's
 * copy stream and returns at once (the host buffers must stay valid, and should be pinned, until the matching
 * dsa_matrix_apply_staged returns); dsa_matrix_apply_staged applies the oldest staged batch exactly like dsa_matrix_set_batch.
 * Staging batch k+1 before applying batch k overlaps its PCIe transfer with the kernels of batch k.  At most 2 batches staged. */
int dsa_matrix_stage_batch(dsa_matrix_t* A, const int64_t* rows, const int64_t* cols, const double* vals, int64_t n);
int dsa_matrix_apply_staged(dsa_matrix_t* A);
/* batched getindex (matrix.jl:64-68 -> pcsr.jl:261-267); which = orientation to read (both hold the same values) */
int dsa_matrix_get_batch(dsa_matrix_t* A, int which, const int64_t* rows, const int64_t* cols, int64_t n, double* out);
/* deletecolumn! / deleterow! for a list (matrix.jl:95-111 -> pcsr.jl:188-212, writes.jl:80-92); DSA_ERR_ARGUMENT if one is absent */
int dsa_matrix_delete_columns(dsa_matrix_t* A, const int64_t* cols, int64_t n);
int dsa_matrix_delete_rows(dsa_matrix_t* A, const int64_t* rows, int64_t n);
/* view(matrix, :, col) / view(matrix, row, :) (matrix.jl:70-88, views.jl:15-35; pcsr.jl:285-291): compacted span, ascending */
int dsa_matrix_column(dsa_matrix_t* A, int64_t col, int64_t* keys_out, double* vals_out, int64_t cap, int64_t* count_out);
int dsa_matrix_row(dsa_matrix_t* A, int64_t row, int64_t* keys_out, double* vals_out, int64_t cap, int64_t* count_out);
/* mat * x (trans = 0) and transpose(mat) * x (trans = 1) with a sparse x given as ascending (key, value) pairs
 * (operations.jl:14-36, 62-135). Output = touched rows only, ascending, stored zeros kept (sparsevec(::Dict, n)). */
int dsa_matrix_spmv(dsa_matrix_t* A, int trans, const int64_t* x_keys, const double* x_vals, int64_t nx, int64_t* y_keys,
                    double* y_vals, int64_t cap, int64_t* count_out);
/* dense-x variant: x_j = x[j-1] for j in 1..nx (every entry stored); y[i-1] for i in 1..ny, 0.0 where no entry */
int dsa_matrix_spmv_dense(dsa_matrix_t* A, int trans, const double* x, int64_t nx, double* y, int64_t ny);
int dsa_matrix_spmv_dense_d(dsa_matrix_t* A, int trans, const double* d_x, int64_t nx, double* d_y, int64_t ny);
/* mat * X (trans = 0) / transpose(mat) * X (trans = 1) for a dense row-major X (nx rows, k columns, row stride ldx >= k):
 * Y[i-1, c] for i in 1..ny, c < k (row stride ldy >= k), 0.0 where no entry; columns k..ldy-1 of Y are not written.
 * Column c equals dsa_matrix_spmv_dense of column c bit for bit.  k == 0: nothing is written.  nx, ny or k < 0, ldx < k or
 * ldy < k: DSA_ERR_ARGUMENT, nothing is launched.  One pass over the matrix carries up to 32 columns; X is read in place when
 * ldx and k are multiples of 4 and X is 32-byte aligned, otherwise re-laid on the device first. */
int dsa_matrix_spmm_dense(dsa_matrix_t* A, int trans, const double* X, int64_t nx, int64_t k, int64_t ldx, double* Y, int64_t ny,
                          int64_t ldy);
int dsa_matrix_spmm_dense_d(dsa_matrix_t* A, int trans, const double* d_X, int64_t nx, int64_t k, int64_t ldx, double* d_Y,
                            int64_t ny, int64_t ldy);
/* the CUDA stream the handle's work is enqueued on (so that a caller can order its own streams against it) */
int dsa_matrix_get_stream(const dsa_matrix_t* A, void** cuda_stream_out);
/* which = DSA_COLMAJOR | DSA_ROWMAJOR; out = {capacity, segment_capacity, nb_segments, nb_elements, height, nb_partitions,
 * len(semaphores), m, n, nnz} (pma.jl:8-24, pcsr.jl:4-21, matrix.jl:1-8,91) */
int dsa_matrix_info(const dsa_matrix_t* A, int which, int64_t* out10);
/* raw layout dump: occupied/keys/vals[capacity], semaphores[len] (1-based position, 0 = nothing), col_keys[len], col_live[len] */
int dsa_matrix_export(dsa_matrix_t* A, int which, uint8_t* occupied, int64_t* keys, double* vals, int64_t* semaphores,
                      int64_t* col_keys, uint8_t* col_live);
/* Compressed snapshot of ONE orientation: the column / row gathers of every partition at once (pcsr.jl:234-291) in iteration
 * order (pma.jl:165-180), gaps and semaphore cells dropped.  which = DSA_COLMAJOR gives CSC (partition = column, index = row),
 * DSA_ROWMAJOR gives CSR (partition = row, index = column).  Partitions in ascending key, entries in ascending in-array key
 * inside each: sorted indices, no duplicates.  Values are copied bit for bit (stored zeros, NaN payloads and -0.0 kept); nnz is
 * that of dsa_matrix_info.
 * Sparse-pointer form, any keys: counts_out2 = {np, nnz}; part_keys[np] = keys of the live partitions (empty ones included),
 * ptr[np + 1] = 0-based offsets of their entries, keys[nnz] = raw in-array keys, vals[nnz].  Two-call size query: when an
 * output is NULL (one whose length is 0 may be) or cap_parts < np (part_keys holds cap_parts, ptr cap_parts + 1) or
 * cap_nnz < nnz, only the counts are returned and nothing is written. */
int dsa_matrix_compress(dsa_matrix_t* A, int which, int64_t* part_keys, int64_t* ptr, int64_t* keys, double* vals, int64_t cap_parts,
                        int64_t cap_nnz, int64_t* counts_out2);
int dsa_matrix_compress_d(dsa_matrix_t* A, int which, int64_t* d_part_keys, int64_t* d_ptr, int64_t* d_keys, double* d_vals,
                          int64_t cap_parts, int64_t cap_nnz, int64_t* counts_out2);
/* Dense-pointer form (scipy / torch / cuSPARSE / SparseMatrixCSC): the entries of partition key k (1 <= k <= dim) are
 * ptr[k-1]-base .. ptr[k]-base-1 of ind / vals; ptr has dim + 1 entries, ind = in-array key - 1 + base; base = 0 or 1, else
 * DSA_ERR_ARGUMENT (as is dim < 0 or idim < 0).  nnz_out = nnz; size query as above (NULL output or cap_nnz < nnz).
 * DSA_ERR_BOUNDS, nothing written, if a partition holding an entry has key > dim or an entry's in-array key is > idim
 * (dynamicsparse(I, J, V, m, n) stores entries outside m x n); an EMPTY live partition above dim is simply not represented.
 * The `_d` variant synchronises only when the host cannot rule such an entry out (a live partition key > dim, or an in-array
 * key > idim may be stored): the count pass reports it, and the host reads that report before anything is written. */
int dsa_matrix_compress_dense(dsa_matrix_t* A, int which, int64_t dim, int64_t idim, int base, int64_t* ptr, int64_t* ind, double* vals,
                              int64_t cap_nnz, int64_t* nnz_out);
int dsa_matrix_compress_dense_d(dsa_matrix_t* A, int which, int64_t dim, int64_t idim, int base, int64_t* d_ptr, int64_t* d_ind,
                                double* d_vals, int64_t cap_nnz, int64_t* nnz_out);

/* ---------------------------------------------------------------- multi-GPU (SURVEY.md §8e) ---- */
/* One process per GPU.  A dsa_dist_t is this rank's seat in a group of `world` ranks on one NVLink box; a dsa_dmatrix_t is a
 * DynamicSparseMatrix sharded by key range over the group: rank r owns the column-major PCSR of the columns in
 * [col_split[r], col_split[r+1]) and the row-major PCSR of the rows in [row_split[r], row_split[r+1]).  The Julia methods these
 * replace are the same as for dsa_matrix_* (matrix.jl:15-19,43-68,95-111; operations.jl:14-36); what is new is that each is a
 * COLLECTIVE: every rank of the group must make the same call in the same order.
 * Communication: routed updates travel as direct NVLink stores into the owner's receive regions (CUDA IPC peer memory), fused
 * into the routing kernel; NCCL carries only the 2 x world send counts of a batch (one small all-gather, which is also the
 * barrier) and the all-gather of the SpMV result.  DSA_DIST_TRANSPORT=nccl selects grouped ncclSend/ncclRecv instead. */
typedef struct dsa_dist dsa_dist_t;
typedef struct dsa_dmatrix dsa_dmatrix_t;
#define DSA_ERR_NCCL 13
#define DSA_UNIQUE_ID_BYTES 128
/* rank 0 creates the id (ncclGetUniqueId) and hands the 128 bytes to the other ranks by any host-side means */
int dsa_dist_unique_id(void* id_out128);
/* joins the group on the CURRENT CUDA device (collective): creates an NCCL communicator owned by the handle */
int dsa_dist_init(const void* id128, int rank, int world, dsa_dist_t** out);
/* same, on a communicator the host already has (an `ncclComm_t` of the same libnccl); it is not destroyed with the handle */
int dsa_dist_init_comm(void* nccl_comm, int rank, int world, dsa_dist_t** out);
int dsa_dist_destroy(dsa_dist_t* d);
/* out = {rank, world, transport (0 = peer-memory stores, 1 = nccl send/recv), nccl version} */
int dsa_dist_info(const dsa_dist_t* d, int64_t* out4);
/* empty m x n matrix sharded over the group (collective).  row_split / col_split: world + 1 ascending first-owned keys
 * (split[0] = 1, split[world] = dimension + 1), or NULL for equal key ranges.  max_share = the largest number of updates ONE
 * rank will pass to a single set_batch / build round: it sizes the receive regions (a full share per (source, owner) pair and
 * orientation, double-buffered: 96 x world x max_share bytes per rank), so no skew can overflow them. */
int dsa_dmatrix_create(dsa_dist_t* d, int64_t m, int64_t n, const int64_t* row_split, const int64_t* col_split, int64_t max_share,
                       dsa_dmatrix_t** out);
int dsa_dmatrix_destroy(dsa_dmatrix_t* D);
int dsa_dmatrix_set_stream(dsa_dmatrix_t* D, void* cuda_stream);
/* this rank's shards as a plain matrix handle (owned by D): for dsa_matrix_info / dsa_matrix_export / dsa_matrix_column ... */
dsa_matrix_t* dsa_dmatrix_local(dsa_dmatrix_t* D);
/* dynamicsparse(I, J, V, m, n) (matrix.jl:15-19) over the group: every rank passes ITS share of the global COO (host
 * pointers, any split); entries are routed to the owners of both orientations in rounds of max_share, then each shard is
 * bulk-built (pcsr.jl:354-449).  Duplicate (i, j) are folded in global order = round-major, then rank-major, then arrival. */
int dsa_dmatrix_build_coo(dsa_dmatrix_t* D, const int64_t* rows, const int64_t* cols, const double* vals, int64_t n, int combine);
/* shard-local bulk build without any exchange: the caller passes exactly the entries of ITS shard of one orientation
 * ((rows, cols) for DSA_COLMAJOR within its column range, (cols, rows) for DSA_ROWMAJOR within its row range) */
int dsa_dmatrix_build_local(dsa_dmatrix_t* D, int which, const int64_t* inkeys, const int64_t* partkeys, const double* vals,
                            int64_t n, int combine);
int dsa_dmatrix_build_local_d(dsa_dmatrix_t* D, int which, const int64_t* d_inkeys, const int64_t* d_partkeys, const double* d_vals,
                              int64_t n, int combine);
/* batched setindex! (matrix.jl:43-62) over the group: every rank passes its share (n <= max_share, may be 0) of ONE global
 * batch whose op order is rank-major, then arrival within a rank: last writer wins in that order, 0.0 deletes. */
int dsa_dmatrix_set_batch(dsa_dmatrix_t* D, const int64_t* rows, const int64_t* cols, const double* vals, int64_t n);
int dsa_dmatrix_set_batch_d(dsa_dmatrix_t* D, const int64_t* d_rows, const int64_t* d_cols, const double* d_vals, int64_t n);
/* The same batch in two halves, so that the exchange of batch k+1 overlaps the kernels of batch k (both collective):
 * dsa_dmatrix_stage_batch[_d] routes the share and pushes it into the owners' receive regions on a side stream and returns at
 * once (host buffers must stay valid, and should be pinned, until the matching apply returns; device buffers until it has been
 * applied); dsa_dmatrix_apply_staged applies the oldest staged batch.  At most 2 batches staged; reads and products between
 * the two calls see the matrix without the staged batch. */
int dsa_dmatrix_stage_batch(dsa_dmatrix_t* D, const int64_t* rows, const int64_t* cols, const double* vals, int64_t n);
int dsa_dmatrix_stage_batch_d(dsa_dmatrix_t* D, const int64_t* d_rows, const int64_t* d_cols, const double* d_vals, int64_t n);
int dsa_dmatrix_apply_staged(dsa_dmatrix_t* D);
/* mat * x (trans = 0) / transpose(mat) * x (trans = 1), x replicated on every rank, y (ny entries) returned on every rank:
 * each rank computes its slice from its row-major (col-major) shard into the gather buffer, one ncclAllGather (operations.jl:14-36) */
int dsa_dmatrix_spmv_dense(dsa_dmatrix_t* D, int trans, const double* x, int64_t nx, double* y, int64_t ny);
int dsa_dmatrix_spmv_dense_d(dsa_dmatrix_t* D, int trans, const double* d_x, int64_t nx, double* d_y, int64_t ny);
/* batched getindex (matrix.jl:64-68): every rank may ask for different (row, col) pairs (n may differ); answered by the owners */
int dsa_dmatrix_get_batch(dsa_dmatrix_t* D, int which, const int64_t* rows, const int64_t* cols, int64_t n, double* out);
/* deletecolumn! / deleterow! (matrix.jl:95-111) over the group: the SAME list on every rank; owner(col) purges its partitions
 * and the (row, col) delete list is routed to the owners of the rows (SURVEY.md §8e (3)).  DSA_ERR_ARGUMENT on every rank, with
 * nothing changed, if a listed column does not exist. */
int dsa_dmatrix_delete_columns(dsa_dmatrix_t* D, const int64_t* cols, int64_t n);
int dsa_dmatrix_delete_rows(dsa_dmatrix_t* D, const int64_t* rows, int64_t n);
/* out = {m, n, nnz over all ranks (matrix.jl:91: of the row-major shards), col-major partitions over all ranks, row-major
 * partitions over all ranks, max_share, nnz of the col-major shards over all ranks, transport} (collective) */
int dsa_dmatrix_info(dsa_dmatrix_t* D, int64_t* out8);

/* ---------------------------------------------------------------- memory --------------- */
/* device buffers are recycled through a size-class cache (growth of a structure would otherwise pay cudaMalloc/cudaFree of
 * 100 MB-class blocks per batch); dsa_trim_memory returns the cached blocks to the driver */
int dsa_trim_memory(void);
int64_t dsa_cached_bytes(void);

/* ---------------------------------------------------------------- tuning --------------- */
/* How a batched setindex! of a matrix orientation (pcsr.jl:341-347 per op) is applied.  0: always the random-access pipeline
 * (per-partition buckets / radix sort, locate in HBM, leaf merge).  1 (default): batches of at least capacity/40 ops are
 * tile-streamed (one pass over the array, every op located and every accepted leaf re-laid in shared memory); a batch that
 * creates columns or overflows a tile's bucket starts over on the random-access pipeline.  2: tile-streamed whenever the
 * structure allows it (tests).  Both pipelines leave the same layout, bit for bit.  Returns the previous mode. */
int dsa_set_tile_mode(int mode);

/* ---------------------------------------------------------------- measurement ---------- */
/* kernel launches issued by this library since load (bench.py's gpu_launches) */
int64_t dsa_launch_count(void);
/* per-kernel CUDA-event timing (adds a sync per launch: use outside timed regions only) */
int dsa_prof_enable(int on);
int dsa_prof_reset(void);
/* writes "name,count,total_ms\n" lines; returns bytes needed */
int64_t dsa_prof_dump(char* buf, int64_t cap);

#ifdef __cplusplus
}
#endif
#endif /* DSA_H */
