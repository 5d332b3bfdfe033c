// Host side of the engine: owns the HBM-resident index, schedules insert batches and query
// launches.  Replaces, above the kernels, what PointIndexation / Hnsw::new / parallel_insert /
// parallel_search do on the CPU in the reference (/root/reference/src/hnsw.rs:395-557, 739-905,
// 1224-1238, 1612-1635): point bookkeeping (level draw, PointId ranks, entry point), and the
// rayon fan-out, which here is a persistent-warp kernel launch.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include <atomic>
#include <functional>
#include <map>
#include <memory>
#include <condition_variable>
#include <mutex>
#include <shared_mutex>
#include <tuple>
#include <string>
#include <thread>
#include <vector>

#include "kernels.h"

namespace hb {

struct SplitMix64 {
  uint64_t s;
  uint64_t next() {
    uint64_t z = (s += 0x9E3779B97F4A7C15ull);
    z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ull;
    z = (z ^ (z >> 27)) * 0x94D049BB133111EBull;
    return z ^ (z >> 31);
  }
  double unif() { return (double)(next() >> 11) * (1.0 / 9007199254740992.0); }
};

// restores the calling thread's current device on scope exit (the library switches devices when it works on replicas;
// a host that tracks the current device itself, e.g. torch, must find it unchanged after every call)
struct DeviceRestore {
  int prev = -1;
  DeviceRestore() { cudaGetDevice(&prev); }
  ~DeviceRestore() {
    if (prev >= 0) cudaSetDevice(prev);
  }
};

template <class T>
struct DevArray {  // growable device array, contents preserved on growth
  T* p = nullptr;
  size_t cap = 0;
};

struct DumpDescription {  // Description, /root/reference/src/hnswio.rs:846-870
  int format_version = 0;
  uint8_t dumpmode = 0, max_nb_connection = 0, nb_layer = 0;
  double level_scale = 1.0;
  uint64_t ef = 0, nb_point = 0, dimension = 0;
  std::string distname, t_name;
  long header_bytes = 0;
};
int read_description(const std::string& graph_path, DumpDescription& out, std::string& err);
int metric_from_type_name(const std::string& full);
int dtype_from_type_name(const std::string& s);

class Index {
 public:
  Index(int M, size_t max_elements, int max_layer, int ef_c, int metric, int dtype, int device);
  ~Index();
  bool ok() const { return ok_; }

  // ---- configuration (Hnsw::new and setters, hnsw.rs:771-905)
  int M, max_layer, ef_c, metric, dtype, es, device;  // es = bytes per element
  size_t max_elements;
  bool extend_candidates = false, keep_pruned = false, searching = false;
  bool tie_std_ = false;  // hnsw_b200_set_tie_mode: equal-distance ties resolved like the reference's std BinaryHeaps (search_std.cu)
  double level_scale;  // 1/ln(M) * factor
  SplitMix64 rng{397};
  uint32_t batch_ratio = 16, batch_max = 16384;

  // ---- state
  int dim = 0, row_bytes = 0;  // row_bytes = dim*es rounded up to whole 128-byte lines
  size_t n = 0;          // points stored (all linked: inserts are synchronous per call)
  size_t n_ul = 0;       // upper lists allocated
  size_t layer_count[MAX_LAYERS];
  uint32_t entry = INVALID_ID;
  int entry_level = -1;
  std::vector<uint8_t> h_level, h_plevel;
  std::vector<int32_t> h_rank;
  std::vector<uint64_t> h_origin;
  std::vector<uint32_t> h_upoff;

  // ---- operations (return 0 or a negative status; message in err())
  int set_dim(int d);
  int draw_level();
  int insert_batch(const void* vecs, size_t n_new, size_t stride, const void* const* rows, const uint64_t* ids,
                   const int32_t* levels);
  int import_graph(const void* vecs, size_t n_new, int d, const uint64_t* origin, const uint8_t* levels,
                   int64_t entry_id, int nlayers, const uint64_t* const* offsets, const uint32_t* const* ids,
                   const float* const* dists);
  // host queries (flat or row pointers); results to host NeighbourOut[nq][k] + counts
  int search_host(const void* queries, const void* const* rows, size_t nq, int d, size_t k, size_t ef,
                  const uint32_t* filter_bits_host, NeighbourOut* out, int32_t* counts);
  // same on context c (a CtxLease), answers left in the context's pinned buffer (valid until the lease ends)
  // qdesc / qpay: per-query filters instead of filter_bits_host (QueryFilterSet below; qdesc[i] is query i's, its offset
  // counts from qpay, which only the range those nq descriptors name is read of)
  int search_host_begin(int c, const void* queries, const void* const* rows, size_t nq, int d, size_t k, size_t ef,
                        const uint32_t* filter_bits_host, const QueryFilter* qdesc = nullptr, const uint32_t* qpay = nullptr);
  int search_host_finish(int c, const NeighbourOut** out, const int32_t** counts);
  // submitted-but-not-waited host searches: anything that changes the graph waits for them (drain_pending)
  std::atomic<int> pending_{0};
  void drain_pending() const {
    while (pending_.load() != 0) std::this_thread::yield();
  }
  int search_host_staged(int c, const void* queries, const void* const* rows, size_t nq, int d, size_t k, size_t ef,
                         const uint32_t* filter_bits_host, const NeighbourOut** out, const int32_t** counts,
                         const QueryFilter* qdesc = nullptr, const uint32_t* qpay = nullptr);
  int search_device(const void* d_queries, size_t nq, size_t k, size_t ef, const uint32_t* d_filter_bits,
                    NeighbourOut* d_out, int32_t* d_counts, bool sync, float* kernel_ms);
  // filter materialisation: bit per internal id from a sorted origin-id list or a callback
  int make_filter_bits(int mode, const uint64_t* sorted_ids, size_t nids, int (*fn)(uint64_t, void*), void* ctx,
                       std::vector<uint32_t>& bits) const;
  // One FilterT per query: query i admits the points whose origin id is in ids[offsets[i] .. offsets[i+1]) (ascending,
  // repeats allowed; every point sharing an admitted origin id is admitted, ids not in the index are ignored).  Translated
  // to internal ids and packed per query as a list or a bitmap (QueryFilter, kernels.h).  The caller validates the input.
  // Searches with per-query filters always run the filtered kernel; tie mode "std" does not apply to them, as to batch
  // filters.
  struct QueryFilterSet {
    std::vector<QueryFilter> desc;  // [nq], offsets into payload
    std::vector<uint32_t> payload;
  };
  int make_query_filters(size_t nq, const uint64_t* offsets, const uint64_t* ids, QueryFilterSet& out) const;

  int export_layer(int layer, uint64_t* offsets, uint32_t* ids, float* dists, int64_t* total) const;
  int export_vectors(void* out) const;
  // FlatNeighborhood (/root/reference/src/flatten.rs:50-126): per point, the neighbours of ALL layers merged and
  // sorted by distance; CSR over internal ids, neighbours named by origin id
  int flatten(std::vector<uint64_t>& offsets, std::vector<uint64_t>& nb_origin, std::vector<float>& nb_dist) const;
  // dump / reload in the reference's two-file format (hnswio.cu)
  int file_dump(const std::string& dir, const std::string& basename, bool overwrite, std::string* used_basename);
  int load_dump(const std::string& dir, const std::string& basename);
  int enable_stats(bool on);
  int get_stats(uint64_t* out4, bool reset);

  // replication blobs
  int blob_header(uint64_t* h16) const;
  int blob_alloc(const uint64_t* h16);
  int blob_count() const { return 9; }
  int blob_info(int i, void** p, uint64_t* bytes) const;
  int blob_commit();

  // ---- multi-GPU (multi.cu).  One process, N devices: replicate() builds a copy of the frozen index on every listed
  // device (NCCL broadcast) and for_each_shard() runs a batch split into contiguous shards, one worker thread per
  // device.  One process per GPU: nccl_init() + nccl_broadcast_index() + nccl_allgather().
  int replicate(int ndev, const int* devices);
  size_t replica_count() const { return replicas_.size(); }
  int for_each_shard(size_t nq, const std::function<int(Index*, size_t, size_t)>& run);
  // same shards, visited one after the other on the calling thread (asynchronous enqueues: submit)
  int for_each_shard_inline(size_t nq, const std::function<int(Index*, size_t, size_t)>& run);
  // outstanding submit tickets: (index, context) per device
  struct Ticket {
    std::vector<std::pair<Index*, int>> parts;
  };
  int finish_parts(const std::vector<std::pair<Index*, int>>& parts, const std::function<int(Index*, int)>& fn);
  int64_t park_ticket(Ticket&& t);
  bool take_ticket(int64_t id, Ticket& out);
  void drop_replicas();
  static int nccl_unique_id(unsigned char* out128);
  int nccl_init(int nranks, int rank, const unsigned char* id128);
  int nccl_broadcast_index(int root);
  int nccl_allgather(const void* d_send, void* d_recv, size_t bytes_per_rank, cudaStream_t s);
  void nccl_destroy();

  // ---- search contexts.  Everything a running search owns besides the (read-only) graph: stream, work counter,
  // status flag, visited tables, staging buffers.  Up to NCTX searches are in flight at once: calls from several host
  // threads (the reference serves concurrent searches, hnsw.rs:830-833) and consecutive asynchronous device-resident
  // launches, whose last queries then overlap the next launch's first (a launch ends with a few long searches that
  // leave most SMs idle).
  struct VisitedPool {
    uint32_t* tab = nullptr;
    uint32_t* epoch = nullptr;
    size_t slots = 0, cap = 0;
    int id_bits = 0;
  };
  struct SearchCtx {
    cudaStream_t stream = nullptr;
    cudaEvent_t fork = nullptr, join = nullptr, ev0 = nullptr, ev1 = nullptr;
    unsigned int* d_counter = nullptr;
    int* d_status = nullptr;
    VisitedPool vis, fvis;  // unfiltered / filtered searches
    void *d_q = nullptr, *d_out = nullptr, *d_cnt = nullptr, *d_fbits = nullptr, *d_cbuf = nullptr, *d_qf = nullptr;
    size_t d_q_bytes = 0, d_out_bytes = 0, d_cnt_bytes = 0, d_fbits_bytes = 0, d_cbuf_bytes = 0, d_qf_bytes = 0;
    void *h_pin = nullptr, *h_res = nullptr;  // pinned, mapped: query staging / answers
    size_t h_pin_bytes = 0, h_res_bytes = 0;
    bool busy = false;
    struct Pending {  // a host search enqueued by search_host_begin, completed by search_host_finish
      const void* d_queries = nullptr;
      const uint32_t* dfb = nullptr;
      const QueryFilter* dqf = nullptr;  // per-query filters: descriptors and payload in d_qf
      const uint32_t* dqpay = nullptr;
      NeighbourOut *k_out = nullptr, *hout = nullptr;
      int32_t *k_cnt = nullptr, *hcnt = nullptr, *hstatus = nullptr;
      size_t nq = 0, k = 0, ef = 0, out_bytes = 0, cnt_bytes = 0;
      bool direct = false, enqueued = false;
      // where hnsw_b200_search_flat_wait unpacks to
      uint64_t* u_ids = nullptr;
      float* u_dist = nullptr;
      uint32_t* u_internal = nullptr;
      int32_t *u_pid = nullptr, *u_counts = nullptr;
    } pend;
  };
  static constexpr int NCTX = 4;    // leased by synchronous calls (host threads)
  static constexpr int NASYNC = 2;  // alternated by asynchronous device-resident launches (never leased)
  int acquire_ctx();            // blocks until a context is free
  void release_ctx(int c);
  SearchCtx& ctx(int c) { return ctx_[c]; }
  struct CtxLease {             // RAII: answers returned by search_host_staged live in the context until release
    Index* ix;
    int c;
    explicit CtxLease(Index* i) : ix(i), c(i->acquire_ctx()) {}
    ~CtxLease() { ix->release_ctx(c); }
    CtxLease(const CtxLease&) = delete;
    CtxLease& operator=(const CtxLease&) = delete;
  };

  int dist_batch(const void* queries, size_t nq, int d, const uint32_t* cand, size_t m, float* out);
  int bruteforce(const void* queries, size_t nq, int d, size_t k, uint32_t* out_ids, float* out_dist);

  std::string err() const;
  GraphView view() const;
  cudaStream_t stream() const { return stream_; }
  int join();                           // the handle's stream waits for every asynchronous launch enqueued so far
  int stream_wait_last(cudaStream_t s);  // `s` waits for the most recent asynchronous launch
  int set_stream(cudaStream_t s);   // run on a caller-owned stream (e.g. torch's current stream); nullptr = own stream
  int check_status();               // synchronise; 0 ok, 1 = a visited table overflowed since the last check
  // the C ABI allows calls from many host threads (hnsw.rs:830-833): searches share the graph, anything that changes it
  // (insert, import, load, replicate) holds it exclusively
  mutable std::shared_mutex mu;

 private:
  int fail(const std::string& m) const;
  int cuda_fail(cudaError_t e, const char* what) const;
  int ensure_points(size_t need);
  int ensure_upper(size_t need_lists);
  int ensure_visited(VisitedPool& v, size_t slots, size_t cap_entries, cudaStream_t st);
  int fill_visited_cfg(VisitedPool& v, VisitedCfg& c, cudaStream_t st);
  int ensure_scratch(void** p, size_t* cur, size_t need, cudaStream_t st);
  int grow_plevel(uint32_t id, int new_plevel);
  int run_insert_range(size_t first, size_t count, const std::vector<uint16_t>& masks, size_t mask_off);
  int check_insert_fit();
  void rollback_points(size_t keep);
  template <class T>
  int grow(DevArray<T>& a, size_t need_elems, size_t keep_elems, int fill_byte);

  struct Worker;
  struct WorkerDeleter {
    void operator()(Worker* w) const;
  };
  int broadcast_to_replicas();
  std::vector<std::unique_ptr<Index>> replicas_;  // replicas_[i] lives on replica_devices_[i + 1]
  std::vector<std::unique_ptr<Worker, WorkerDeleter>> workers_;
  std::vector<void*> comms_;                      // ncclComm_t per device, rank 0 = this index
  std::vector<int> replica_devices_;
  bool replicas_stale_ = false;                   // the index changed after the last broadcast
  void* comm_ = nullptr;                          // ncclComm_t of the one-process-per-GPU mode
  int nranks_ = 1, rank_ = 0;

  bool ok_ = false;
  bool poisoned_ = false;  // a CUDA failure interrupted an insert: the graph may hold half-written links
  std::string poison_msg_;
  mutable std::string err_;
  mutable std::mutex err_mu_;
  cudaStream_t stream_ = nullptr, own_stream_ = nullptr;
  int sm_count_ = 0;

  size_t cap_ = 0, cap_ul_ = 0;
  DevArray<unsigned char> d_vec_;
  DevArray<uint32_t> d_adj0_, d_adjU_, d_upoff_;
  DevArray<float> d_adj0d_, d_adjUd_;
  DevArray<uint8_t> d_level_, d_plevel_;
  DevArray<uint64_t> d_origin_;
  DevArray<int> d_locks_;

  VisitedPool vis_;  // visited tables of the insert kernel (searches: SearchCtx)
  SearchCtx ctx_[NCTX + NASYNC];
  int search_on_ctx(SearchCtx& c, const void* d_queries, size_t nq, size_t k, size_t ef_arg, const uint32_t* d_filter_bits,
                    NeighbourOut* d_out, int32_t* d_counts, bool sync, float* kernel_ms, const QueryFilter* d_qf = nullptr,
                    const uint32_t* d_qpay = nullptr);
  std::mutex ctx_mu_;
  std::condition_variable ctx_cv_;
  std::mutex ticket_mu_, shard_mu_;
  std::map<int64_t, Ticket> tickets_;
  int64_t next_ticket_ = 0;
  int last_async_ = -1;
  unsigned ctx_rr_ = 0;        // round robin of the asynchronous device-resident launches
  std::mutex occ_mu_;
  int kernel_pref_ = 0;        // env HNSW_B200_KERNEL=warp (A/B measurements): 1 = always the generic warp kernel
  bool zero_copy_ = true;      // env HNSW_B200_ZERO_COPY=0: explicit H2D / D2H copies instead of kernel access to pinned host memory

  // small device scratch (insert path; searches: SearchCtx)
  unsigned int* d_counter_ = nullptr;
  int* d_status_ = nullptr;
  unsigned long long* d_stats_ = nullptr;
  bool stats_on_ = false;
  std::atomic<uint64_t> stat_queries_{0};

  // staging of the insert path
  void* h_pin_ = nullptr;
  size_t h_pin_bytes_ = 0;
  std::map<std::tuple<int, int, int, size_t>, int> occ_cache_;  // (filtered, queue kind, d4, smem) -> CTAs/SM
  void* d_mask_ = nullptr;
  size_t d_mask_bytes_ = 0;

  // (origin id, internal id) sorted, for make_query_filters: built on first use, dropped wherever h_origin changes
  mutable std::mutex origin_mu_;
  mutable std::vector<std::pair<uint64_t, uint32_t>> origin_table_;
  mutable bool origin_table_ok_ = false;
  void invalidate_origin_table() {
    std::lock_guard<std::mutex> lk(origin_mu_);
    origin_table_ok_ = false;
    origin_table_.clear();
    origin_table_.shrink_to_fit();
  }
};

}  // namespace hb
