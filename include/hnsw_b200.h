/* libhnsw_b200.so — C ABI of the B200-native HNSW search/insert engine.
 *
 * Part 1 re-exports, with identical names, argument order and #[repr(C)] struct layouts, the
 * extern "C" surface the reference crate (jean-pierreBoth/hnswlib-rs) defines in
 * /root/reference/src/libext.rs, for the f32 instantiation (the hot path named by
 * BASELINE.json).  A caller of the reference cdylib (Julia's HnswAnn.jl, C, or the Rust shim in
 * hnswlib-rs_b200/rust_shim/) can link this library instead.
 * Part 2 are `hnsw_b200_*` extensions: explicit frees (the reference leaks its answers to the
 * caller and exports no free, libext.rs:194-200,236-251), flat-array batch calls, options,
 * graph import/export, filter upload, stand-alone distance / brute-force kernels, statistics.
 *
 * No torch types, plain pointers and sizes only.  Every call needing the GPU fails loudly (NULL /
 * negative status + hnsw_b200_last_error()) when no CUDA device is usable; there is no CPU fallback.
 */
#ifndef HNSW_B200_H
#define HNSW_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

/* ------------------------------------------------------------------ Part 1: reference symbols */

/* opaque handle; libext.rs:38-50,100 (declare_myapi_type!(HnswApif32, f32)) */
typedef struct HnswApif32 HnswApif32;

/* libext.rs:64-71   #[repr(C)] pub struct Neighbour_api { id: usize, d: f32 }   (16 bytes) */
typedef struct Neighbour_api {
  size_t id;
  float d;
} Neighbour_api;

/* libext.rs:82-87   #[repr(C)] pub struct Neighbourhood_api { nbgh: i64, neighbours: *const Neighbour_api } */
typedef struct Neighbourhood_api {
  int64_t nbgh;
  const Neighbour_api* neighbours;
} Neighbourhood_api;

/* libext.rs:58-62   #[repr(C)] pub struct Vec_api<T> { len: i64, ptr: *const T }, T = Neighbourhood_api */
typedef struct Vec_api_Neighbourhood_api {
  int64_t len;
  const Neighbourhood_api* ptr;
} Vec_api_Neighbourhood_api;

/* libext.rs:458-525.  Hnsw::<f32,D>::new(max_nb_conn, 10000, 16, ef_const, D).  cdistname is NOT
 * NUL-terminated (namelen bytes).  Accepted: "DistL1" "DistL2" "DistDot" "DistHellinger"
 * "DistJeffreys" "DistJensenShannon" as upstream, plus "DistCosine" (upstream reaches it only
 * through load_hnswdump_f32_DistCosine).  Unknown name or no usable GPU => NULL. */
const HnswApif32* init_hnsw_f32(size_t max_nb_conn, size_t ef_const, size_t namelen, const uint8_t* cdistname);

/* libext.rs:532-620 */
const HnswApif32* new_hnsw_f32(size_t max_nb_conn, size_t ef_const, size_t namelen, const uint8_t* cdistname,
                               size_t max_elements, size_t max_layer);

/* libext.rs:626-630 */
void drop_hnsw_f32(const HnswApif32* p);

/* libext.rs:643-655.  A host function pointer cannot be evaluated inside a kernel; this entry
 * point exists for link compatibility and always returns NULL (see INTEGRATION.md). */
const HnswApif32* init_hnsw_ptrdist_f32(size_t max_nb_conn, size_t ef_const,
                                        float (*c_func)(const float*, const float*, unsigned long long));

/* libext.rs:661-677.  The vector is copied; `len` fixes the index dimension on first use and must
 * match afterwards (the flat point store needs one dimension; mismatches are ignored with an error
 * recorded in hnsw_b200_last_error()). */
void insert_f32(HnswApif32* hnsw_api, size_t len, const float* data, size_t id);

/* libext.rs:683-722 */
void parallel_insert_f32(HnswApif32* hnsw_api, size_t nb_vec, size_t vec_len, const float** datas, const size_t* ids);

/* libext.rs:728-767.  Result is owned by the caller; release with hnsw_b200_free_neighbourhood(). */
const Neighbourhood_api* search_neighbours_f32(const HnswApif32* hnsw_api, size_t len, const float* data, size_t knbn,
                                               size_t ef_search);

/* libext.rs:205-254 (instantiated :770).  Answers in input order.  Release with hnsw_b200_free_vec_api(). */
const Vec_api_Neighbourhood_api* parallel_search_neighbours_f32(const HnswApif32* hnsw_api, size_t nb_vec,
                                                                int64_t vec_len, const float** data, size_t knbn,
                                                                size_t ef_search);

/* libext.rs:257-275 (instantiated :771).  Returns 1 on success, -1 on failure. */
int64_t file_dump_f32(const HnswApif32* hnsw_api, size_t namelen, const uint8_t* filename);


/* ---- integer element types (libext.rs:779-1116).  Same pattern as f32; accepted distance names as upstream:
 * i32: DistL1 DistL2 DistHamming (:779-810) | u32: DistL1 DistL2 DistJaccard DistHamming (:843-881) |
 * u16: DistL1 DistL2 DistHamming DistJaccard (:914-958; DistLevenshtein is a variable-length edit distance and is not
 * offered by this engine) | u8: DistL1 DistL2 DistHamming DistJaccard (:1058-1095).
 * Upstream exports drop_hnsw_f32 and drop_hnsw_u16 only; hnsw_b200_drop() releases a handle of any type. */
typedef struct HnswApii32 HnswApii32; /* libext.rs:779-835 */
const HnswApii32* init_hnsw_i32(size_t max_nb_conn, size_t ef_const, size_t namelen, const uint8_t* cdistname);
const HnswApii32* init_hnsw_ptrdist_i32(size_t max_nb_conn, size_t ef_const,
                                        float (*c_func)(const int32_t*, const int32_t*, unsigned long long)); /* always NULL */
void insert_i32(HnswApii32* hnsw_api, size_t len, const int32_t* data, size_t id);
void parallel_insert_i32(HnswApii32* hnsw_api, size_t nb_vec, size_t vec_len, const int32_t** datas, const size_t* ids);
const Neighbourhood_api* search_neighbours_i32(const HnswApii32* hnsw_api, size_t len, const int32_t* data, size_t knbn,
                                               size_t ef_search);
const Vec_api_Neighbourhood_api* parallel_search_neighbours_i32(const HnswApii32* hnsw_api, size_t nb_vec,
                                                                int64_t vec_len, const int32_t** data, size_t knbn,
                                                                size_t ef_search);
int64_t file_dump_i32(const HnswApii32* hnsw_api, size_t namelen, const uint8_t* filename);
typedef struct HnswApiu32 HnswApiu32; /* libext.rs:843-904 */
const HnswApiu32* init_hnsw_u32(size_t max_nb_conn, size_t ef_const, size_t namelen, const uint8_t* cdistname);
const HnswApiu32* init_hnsw_ptrdist_u32(size_t max_nb_conn, size_t ef_const,
                                        float (*c_func)(const uint32_t*, const uint32_t*, unsigned long long)); /* always NULL */
void insert_u32(HnswApiu32* hnsw_api, size_t len, const uint32_t* data, size_t id);
void parallel_insert_u32(HnswApiu32* hnsw_api, size_t nb_vec, size_t vec_len, const uint32_t** datas, const size_t* ids);
const Neighbourhood_api* search_neighbours_u32(const HnswApiu32* hnsw_api, size_t len, const uint32_t* data, size_t knbn,
                                               size_t ef_search);
const Vec_api_Neighbourhood_api* parallel_search_neighbours_u32(const HnswApiu32* hnsw_api, size_t nb_vec,
                                                                int64_t vec_len, const uint32_t** data, size_t knbn,
                                                                size_t ef_search);
int64_t file_dump_u32(const HnswApiu32* hnsw_api, size_t namelen, const uint8_t* filename);
typedef struct HnswApiu16 HnswApiu16; /* libext.rs:908-1048 */
const HnswApiu16* init_hnsw_u16(size_t max_nb_conn, size_t ef_const, size_t namelen, const uint8_t* cdistname);
const HnswApiu16* init_hnsw_ptrdist_u16(size_t max_nb_conn, size_t ef_const,
                                        float (*c_func)(const uint16_t*, const uint16_t*, unsigned long long)); /* always NULL */
void insert_u16(HnswApiu16* hnsw_api, size_t len, const uint16_t* data, size_t id);
void parallel_insert_u16(HnswApiu16* hnsw_api, size_t nb_vec, size_t vec_len, const uint16_t** datas, const size_t* ids);
const Neighbourhood_api* search_neighbours_u16(const HnswApiu16* hnsw_api, size_t len, const uint16_t* data, size_t knbn,
                                               size_t ef_search);
const Vec_api_Neighbourhood_api* parallel_search_neighbours_u16(const HnswApiu16* hnsw_api, size_t nb_vec,
                                                                int64_t vec_len, const uint16_t** data, size_t knbn,
                                                                size_t ef_search);
int64_t file_dump_u16(const HnswApiu16* hnsw_api, size_t namelen, const uint8_t* filename);
typedef struct HnswApiu8 HnswApiu8; /* libext.rs:1052-1116 */
const HnswApiu8* init_hnsw_u8(size_t max_nb_conn, size_t ef_const, size_t namelen, const uint8_t* cdistname);
const HnswApiu8* init_hnsw_ptrdist_u8(size_t max_nb_conn, size_t ef_const,
                                        float (*c_func)(const uint8_t*, const uint8_t*, unsigned long long)); /* always NULL */
void insert_u8(HnswApiu8* hnsw_api, size_t len, const uint8_t* data, size_t id);
void parallel_insert_u8(HnswApiu8* hnsw_api, size_t nb_vec, size_t vec_len, const uint8_t** datas, const size_t* ids);
const Neighbourhood_api* search_neighbours_u8(const HnswApiu8* hnsw_api, size_t len, const uint8_t* data, size_t knbn,
                                               size_t ef_search);
const Vec_api_Neighbourhood_api* parallel_search_neighbours_u8(const HnswApiu8* hnsw_api, size_t nb_vec,
                                                                int64_t vec_len, const uint8_t** data, size_t knbn,
                                                                size_t ef_search);
int64_t file_dump_u8(const HnswApiu8* hnsw_api, size_t namelen, const uint8_t* filename);
const HnswApiu16* new_hnsw_u16(size_t max_nb_conn, size_t ef_const, size_t namelen, const uint8_t* cdistname,
                               size_t max_elements, size_t max_layer); /* libext.rs:964-1028 */
void drop_hnsw_u16(const HnswApiu16* p);                               /* libext.rs:636-640 */

/* ---- dump reload (libext.rs:27-33, 280-451, 1121-1232).  Files: <basename>.hnsw.graph + <basename>.hnsw.data in the
 * reference's native format (hnswio.rs), so dumps written by hnsw_rs load here and the other way round. */
typedef struct HnswIo HnswIo;
HnswIo* get_hnswio(uint64_t flen, const uint8_t* name); /* libext.rs:27-33: basename, looked up in "." */
const HnswApif32* load_hnswdump_f32_DistL1(HnswIo* io); /* libext.rs:310-345 */
const HnswApif32* load_hnswdump_f32_DistL2(HnswIo* io);
const HnswApif32* load_hnswdump_f32_DistCosine(HnswIo* io);
const HnswApif32* load_hnswdump_f32_DistDot(HnswIo* io);
const HnswApif32* load_hnswdump_f32_DistJensenShannon(HnswIo* io);
const HnswApif32* load_hnswdump_f32_DistJeffreys(HnswIo* io);
const HnswApii32* load_hnswdump_i32_DistL1(HnswIo* io); /* libext.rs:348-365 */
const HnswApii32* load_hnswdump_i32_DistL2(HnswIo* io);
const HnswApii32* load_hnswdump_i32_DistHamming(HnswIo* io);
const HnswApiu32* load_hnswdump_u32_DistL1(HnswIo* io); /* libext.rs:368-391 */
const HnswApiu32* load_hnswdump_u32_DistL2(HnswIo* io);
const HnswApiu32* load_hnswdump_u32_DistHamming(HnswIo* io);
const HnswApiu32* load_hnswdump_u32_DistJaccard(HnswIo* io);
const HnswApiu16* load_hnswdump_u16_DistL1(HnswIo* io); /* libext.rs:394-417 (DistLevenshtein: not offered) */
const HnswApiu16* load_hnswdump_u16_DistL2(HnswIo* io);
const HnswApiu16* load_hnswdump_u16_DistHamming(HnswIo* io);
const HnswApiu8* load_hnswdump_u8_DistL1(HnswIo* io); /* libext.rs:420-443 */
const HnswApiu8* load_hnswdump_u8_DistL2(HnswIo* io);
const HnswApiu8* load_hnswdump_u8_DistHamming(HnswIo* io);
const HnswApiu8* load_hnswdump_u8_DistJaccard(HnswIo* io);

/* libext.rs:1121-1141   #[repr(C)] pub struct DescriptionFFI (64 bytes) */
typedef struct DescriptionFFI {
  uint8_t dumpmode;
  uint8_t max_nb_connection;
  uint8_t nb_layer;
  size_t ef;
  size_t nb_point;
  size_t data_dimension;
  size_t distname_len;
  const uint8_t* distname;
  size_t t_name_len;
  const uint8_t* t_name;
} DescriptionFFI;
/* libext.rs:1170-1232; `name` is the path of the .hnsw.graph file */
const DescriptionFFI* load_hnsw_description(size_t flen, const uint8_t* name);

/* libext.rs:1238-1240.  No-op here (diagnostics go through hnsw_b200_last_error). */
void init_rust_log(void);

/* ------------------------------------------------------------------ Part 2: extensions
 * `h` is a handle of ANY element type (HnswApif32*, HnswApii32*, HnswApiu32*, HnswApiu16*, HnswApiu8*) passed as
 * void*; vector / query arguments are arrays of that handle's element type. */

/* dtype: 0 f32, 1 u8, 2 u16, 3 u32, 4 i32.  new_hnsw_<ty> with max_elements / max_layer for every element type. */
void* hnsw_b200_new(int dtype, size_t max_nb_conn, size_t ef_const, size_t namelen, const uint8_t* cdistname,
                    size_t max_elements, size_t max_layer);
void hnsw_b200_drop(const void* h);


const char* hnsw_b200_last_error(void);
int hnsw_b200_device_count(void);
/* Limits: max_nb_connection <= 256; fewer than 2^31 points; one query (or insert) must fit 220 KB of shared memory:
 * 16 * ceil(dim * sizeof(T) / 128) * 8 bytes for the query (twice that for an insert) plus 8 bytes per ef (ef_construction)
 * slot, i.e. dimensions up to ~13 000 f32 at ef = 64.  Wide rows or big ef make the kernels run fewer warps per block, not fail. */
/* select the CUDA device used by handles created afterwards on this thread's process (default 0) */
int hnsw_b200_set_device(int device);

void hnsw_b200_free_neighbourhood(const Neighbourhood_api* p);
void hnsw_b200_free_vec_api(const Vec_api_Neighbourhood_api* p);

/* Hnsw setters/getters, /root/reference/src/hnsw.rs:810-905 */
int hnsw_b200_set_extend_candidates(void* h, int flag);  /* hnsw.rs:858 */
/* The flag as the engine applies it.  The reference turns it on at every reload (hnswio.rs:510, 599); the engine can honour
 * it only when ef_construction > 2 * max_nb_connection (select_neighbours extends only when it holds <= max neighbours
 * candidates, hnsw.rs:1318-1362, which with such an ef means the search ran out of reachable points and the extension set is
 * empty): after reloading an index built with a smaller ef_construction this returns 0, and inserts into it keep every
 * candidate where the reference would run the extension + heuristic. */
int hnsw_b200_get_extend_candidates(const void* h);
int hnsw_b200_set_keeping_pruned(void* h, int flag);     /* hnsw.rs:845 */
int hnsw_b200_modify_level_scale(void* h, double scale); /* hnsw.rs:876-905, scale in [0.2,1] */
int hnsw_b200_set_searching_mode(void* h, int flag);     /* hnsw.rs:834 */
/* How unfiltered searches order EQUAL distances.  0 (default): by (distance, internal id), a total order; identical to the
 * reference whenever no two compared distances are equal.  1: the reference's own behaviour, its two std BinaryHeaps
 * (Ord = distance only, /root/reference/src/hnsw.rs:273-297, 940-1053, 1544) replayed literally: same neighbour ids as the
 * reference on tie-heavy metrics (Hamming, Jaccard, integer L1), several times slower (one lane drives the heaps). */
int hnsw_b200_set_tie_mode(void* h, int mode);
int hnsw_b200_set_level_seed(void* h, uint64_t seed);
uint64_t hnsw_b200_get_nb_point(const void* h);          /* hnsw.rs:810 */
int hnsw_b200_get_max_level_observed(const void* h);     /* hnsw.rs:474 */
int hnsw_b200_get_dim(const void* h);
/* max in-flight inserts of one GPU batch = clamp(nb_point / ratio, 1, max_batch) (DESIGN.md "batched insert") */
int hnsw_b200_set_insert_batching(void* h, uint32_t ratio, uint32_t max_batch);

/* Flat batched insert: vecs[n][dim] row-major host memory, ids[n] (may be NULL => running index),
 * levels[n] (may be NULL => drawn from the reference's level law, hnsw.rs:363-374). 0 on success. */
int hnsw_b200_insert_flat(void* h, const void* vecs, uint64_t n, uint64_t dim, const uint64_t* ids,
                          const int32_t* levels);

/* Flat batched search.  queries[nq][dim] host memory (pinned memory is used directly).
 * Outputs, each [nq][knbn] except counts[nq]; any of out_internal/out_pid may be NULL:
 *   out_ids  = origin ids (DataId), out_dist = distances (ascending), missing slots = ~0 / +inf
 *   out_internal = internal ids, out_pid = PointId (level, rank) pairs as int32[nq][knbn][2]
 * Filter (FilterT, /root/reference/src/filter.rs:7-24): filter_mode 0 none, 1 sorted origin-id
 * list (filter_ids / nfilter), 2 predicate callback evaluated ONCE per stored origin id on the
 * host and materialised to a device bitmap.  0 on success. */
typedef int (*hnsw_b200_filter_fn)(uint64_t origin_id, void* ctx);
int hnsw_b200_search_flat(const void* h, const void* queries, uint64_t nq, uint64_t dim, uint64_t knbn,
                          uint64_t ef_search, int filter_mode, const uint64_t* filter_ids, uint64_t nfilter,
                          hnsw_b200_filter_fn fn, void* ctx, uint64_t* out_ids, float* out_dist,
                          uint32_t* out_internal, int32_t* out_pid, int32_t* out_counts);

/* One FilterT (sorted Vec<usize> of origin ids, filter.rs:11-15) per query: query i admits
 * filter_ids[filter_offsets[i] .. filter_offsets[i+1]), ascending (repeats allowed).
 * An empty range admits nothing.  Outputs as hnsw_b200_search_flat.  Sharded over replicas like it.
 * filter_offsets has nq + 1 entries.  Every point whose origin id is listed is admitted (several points may share one);
 * ids absent from the index are ignored.  Each query's list is packed for the device as ascending internal ids, or as
 * a bitmap over the points when that is no larger (32 * ids >= points).  Tie mode "std" (hnsw_b200_set_tie_mode) does
 * not apply, as with filter_mode != 0.  Refused (< 0, nothing launched, the handle stays usable): NULL arrays when
 * nq > 0, filter_offsets[0] != 0, decreasing offsets, a list that is not ascending, packed filters of 2^32 words or
 * more. */
int hnsw_b200_search_flat_filters(const void* h, const void* queries, uint64_t nq, uint64_t dim, uint64_t knbn,
                                  uint64_t ef_search, const uint64_t* filter_offsets, const uint64_t* filter_ids,
                                  uint64_t* out_ids, float* out_dist, uint32_t* out_internal, int32_t* out_pid,
                                  int32_t* out_counts);

/* The same search (unfiltered; sharded over the replicas when hnsw_b200_replicate was called) split in two calls, so that ONE host thread keeps several batches in
 * flight: submit enqueues the batch and returns a ticket (>= 0; < 0 on error) at once, wait blocks until its answers
 * are in the arrays given to submit.  Up to 4 batches may be in flight per handle (a fifth submit blocks); the query and
 * output arrays must stay valid and untouched until wait returns; calls that change the index wait for outstanding
 * tickets (so a thread must collect its own tickets before it inserts).  Batches in flight together overlap on the GPU (see hnsw_b200_search_device). */
int64_t hnsw_b200_search_flat_submit(const void* h, const void* queries, uint64_t nq, uint64_t dim, uint64_t knbn,
                                     uint64_t ef_search, uint64_t* out_ids, float* out_dist, uint32_t* out_internal,
                                     int32_t* out_pid, int32_t* out_counts);
int hnsw_b200_search_flat_wait(const void* h, int64_t ticket);

/* Device-resident variant (kernel-only timing, multi-GPU sharding): d_queries [nq][dim] elements and
 * d_out (Neighbour_api[nq][knbn], internal id in the tail padding) / d_counts (int32[nq]) are
 * DEVICE pointers owned by the caller.  sync != 0: returns when the answers are there; kernel_ms (may be
 * NULL) receives the CUDA-event duration of the search kernel.  sync == 0: the launch is ordered AFTER
 * everything enqueued so far on the handle's stream and runs on one of two alternating internal streams,
 * so that consecutive launches overlap (the last, long searches of one launch leave most SMs idle); the
 * handle's stream does not wait for it until hnsw_b200_join(h); hnsw_b200_stream_wait_last(h, s) makes
 * stream s (NULL = the handle's) wait for the most recent launch only.  Use distinct output buffers for
 * launches that may be in flight together. */
int hnsw_b200_search_device(const void* h, const void* d_queries, uint64_t nq, uint64_t knbn,
                            uint64_t ef_search, void* d_out, int32_t* d_counts, int sync, float* kernel_ms);

/* Run this handle's kernels and copies on a caller-owned CUDA stream (cudaStream_t passed as void*; NULL
 * restores the handle's own stream), e.g. so that torch.cuda.Event on torch's current stream brackets them. */
int hnsw_b200_join(void* h);
int hnsw_b200_stream_wait_last(void* h, void* cuda_stream);
int hnsw_b200_set_stream(void* h, void* cuda_stream);
/* After asynchronous hnsw_b200_search_device calls: synchronise and report 1 if a per-warp visited table
 * overflowed (those answers are empty; re-run them with sync != 0, which grows the tables), 0 if not, <0 on error. */
int hnsw_b200_check_status(void* h);

/* Dump helpers: explicit directory, overwrite flag (DumpInit, hnswio.rs:150-236: with overwrite = 0 an existing
 * <basename>.hnsw.data is kept and a unique "<basename>-<n>" is used; it is returned in used_basename), loaders by name. */
HnswIo* hnsw_b200_get_hnswio(const char* dir, const char* basename);
void hnsw_b200_free_hnswio(HnswIo* io);
int hnsw_b200_file_dump(const void* h, const char* dir, const char* basename, int overwrite, char* used_basename,
                        size_t used_cap);
void* hnsw_b200_load_dump(HnswIo* io, int dtype, size_t namelen, const uint8_t* cdistname);
void hnsw_b200_free_description(const DescriptionFFI* d);

/* Traversal statistics of all searches since the last reset (device counters):
 * out[0] distance evaluations, out[1] expansions, out[2] adjacency ids read, out[3] queries.
 * Collection is off by default; enable != 0 turns it on. */
int hnsw_b200_enable_stats(void* h, int enable);
int hnsw_b200_get_stats(const void* h, uint64_t* out4, int reset);

/* Graph export / import as flat arrays (parity tests, NCCL broadcast, dump writer).
 * Layers are CSR: offsets[nb_point+1], ids[], dists[] (distance to the list owner). */
int hnsw_b200_export_points(const void* h, uint8_t* levels, int32_t* ranks, uint64_t* origin, int64_t* entry);
int hnsw_b200_export_vectors(const void* h, void* out /* [nb_point][dim] elements */);
int64_t hnsw_b200_layer_edges(const void* h, int layer);
int hnsw_b200_export_layer(const void* h, int layer, uint64_t* offsets, uint32_t* ids, float* dists);
/* FlatNeighborhood (/root/reference/src/flatten.rs:50-126): the graph-only view, neighbours of all layers merged and
 * sorted by distance.  flat_neighbours = get_neighbours(DataId); flatten = the whole table (call with NULL arrays first
 * to size them: returns the total neighbour count). */
int64_t hnsw_b200_flat_neighbours(const void* h, uint64_t origin_id, Neighbour_api* out, uint64_t cap);
int64_t hnsw_b200_flatten(const void* h, uint64_t* offsets, uint64_t* nb_origin, float* nb_dist);
/* import into an EMPTY handle: nlayers CSR layers (layer l at offsets[l], ids[l], dists[l]; dists[l] may be NULL) */
int hnsw_b200_import_graph(void* h, const void* vecs, uint64_t n, uint64_t dim, const uint64_t* origin,
                           const uint8_t* levels, int64_t entry, int nlayers, const uint64_t* const* offsets,
                           const uint32_t* const* ids, const float* const* dists);

/* Frozen-index blobs in device memory, for replication over NCCL (one rank builds, the others
 * allocate with hnsw_b200_blob_alloc from the broadcast header, then broadcast every blob).
 * header: 16 x uint64 (see DESIGN.md "replication header"). */
int hnsw_b200_blob_header(const void* h, uint64_t* header16);
int hnsw_b200_blob_alloc(void* h, const uint64_t* header16);
int hnsw_b200_blob_count(const void* h);
int hnsw_b200_blob_info(const void* h, int i, void** dev_ptr, uint64_t* nbytes);
int hnsw_b200_blob_commit(void* h); /* after the broadcasts: pull the small host mirrors back */

/* ---- Multi-GPU search (SURVEY 8e).  The reference's parallel_search (/root/reference/src/hnsw.rs:1612-1635) fans one
 * batch out over the host's cores; these entry points fan it out over the GPUs of one box.  NCCL is bound at run time
 * (libnccl.so.2), used only to copy the frozen index between devices and to gather device-resident answers.
 *
 * One process, N devices.  hnsw_b200_replicate copies the index held by `h` (on devices[0], which must be the handle's
 * device) to devices[1..ndev) with ncclBroadcast.  Afterwards hnsw_b200_search_flat and parallel_search_neighbours_<ty> on
 * `h` split a batch of >= 64 * ndev queries into ndev contiguous shards; every device copies its shard in, searches it and
 * writes its slice of the caller's output arrays (input order kept, no gather step).  Inserting into `h` marks the copies
 * stale; they are re-broadcast before the next sharded search.  ndev = 1 drops the copies. */
int hnsw_b200_replicate(void* h, int ndev, const int* devices);
int hnsw_b200_replica_count(const void* h);
/* One process per GPU.  Rank 0 calls hnsw_b200_nccl_unique_id and hands the 128 bytes to the other ranks by the host's own
 * means; every rank calls hnsw_b200_nccl_init on its (possibly empty) handle, then hnsw_b200_nccl_broadcast_index(root):
 * the root's index is copied into every other rank's handle, which must be empty and created with the same
 * max_nb_connection / distance / element type.  hnsw_b200_nccl_allgather gathers bytes_per_rank bytes of device memory from
 * every rank into d_recv (nranks * bytes_per_rank) on cuda_stream (NULL = the handle's stream), asynchronously. */
int hnsw_b200_nccl_unique_id(uint8_t* id128);
int hnsw_b200_nccl_init(void* h, int nranks, int rank, const uint8_t* id128);
int hnsw_b200_nccl_broadcast_index(void* h, int root);
int hnsw_b200_nccl_allgather(void* h, const void* d_send, void* d_recv, uint64_t bytes_per_rank, void* cuda_stream);

/* Stand-alone kernels.  dist_batch: out[nq][m] = dist(queries[i], base[cand[i][j]]) on the index's
 * point store (host pointers).  bruteforce: exact k nearest (ascending) of each query over the
 * index's point store: out_ids are INTERNAL ids. */
int hnsw_b200_dist_batch(const void* h, const void* queries, uint64_t nq, uint64_t dim, const uint32_t* cand,
                         uint64_t m, float* out);
int hnsw_b200_bruteforce(const void* h, const void* queries, uint64_t nq, uint64_t dim, uint64_t k,
                         uint32_t* out_ids, float* out_dist);

#ifdef __cplusplus
}
#endif
#endif /* HNSW_B200_H */
