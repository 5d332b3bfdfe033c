// Host-visible declarations of the kernel launchers (search.cu, build.cu, aux.cu).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdlib.h>

#include "common.cuh"

namespace hb {

enum DType : int { DT_F32 = 0, DT_U8 = 1, DT_U16 = 2, DT_U32 = 3, DT_I32 = 4 };
inline int dtype_size(int dt) { return dt == DT_U8 ? 1 : dt == DT_U16 ? 2 : 4; }

constexpr int SEARCH_THREADS = 256;  // 8 warps = 8 queries in flight per CTA
constexpr int BUILD_THREADS = 128;   // 4 warps = 4 inserts in flight per CTA
constexpr int LEAN_THREADS = 32;      // lean kernel (search_lean.cuh): one warp per CTA, so that a finished query frees its slot at once
#ifndef HB_LEAN_BLOCKS
#define HB_LEAN_BLOCKS 28
#endif
constexpr int LEAN_MIN_BLOCKS = HB_LEAN_BLOCKS;  // 28 one-warp CTAs per SM, <= 72 registers per thread (measured: 24, 28, 32 warps within 3 %)

// One answer slot.  Same 16-byte layout as the reference's #[repr(C)] Neighbour_api {id: usize, d: f32}
// (/root/reference/src/libext.rs:64-71); the internal id rides in what is tail padding there.
struct NeighbourOut {
  uint64_t origin;
  float dist;
  uint32_t internal;
};

// One query's FilterT on the device.  form QF_LIST: payload[off .. off+len) are ascending internal ids; form QF_BITMAP:
// payload[off .. off+ceil(n/32)) is a bit per internal id (len = ids admitted).  The host picks the bitmap when the list
// would be at least as large (32 * len >= n), so a query never costs more than 4 bytes per admitted id.
enum : uint32_t { QF_LIST = 0, QF_BITMAP = 1 };
struct __align__(16) QueryFilter {
  uint32_t off;  // in 32-bit words
  uint32_t len;
  uint32_t form;
  uint32_t pad;
};
inline bool qf_use_bitmap(uint64_t len, uint64_t n) { return 32 * len >= n; }

struct SearchParams {
  GraphView g;
  const void* queries;  // device, raw element bytes, row i at i * q_stride_bytes
  int q_bytes;          // bytes of one query = dim * sizeof(T)
  int q_stride_bytes;
  uint32_t nq;
  int k;
  int ef;      // already max(ef_arg, k), hnsw.rs:1531
  int layer0;  // lowest layer holding a point of exactly that level (hnsw.rs:1534-1540), normally 0
  VisitedCfg vis;
  unsigned int* work_counter;
  NeighbourOut* out_nb;  // [nq][k]
  int32_t* out_count;    // [nq]
  const uint32_t* filter_bits;  // nullptr = no batch filter; bit per internal id, one filter for every query
  unsigned long long* stats;    // nullptr or [3]: evals, expansions, adjacency ids read
  int* status;                  // set to 1 on visited-table overflow
  int smem_per_warp;
  int threads;  // threads per CTA of this launch (a multiple of 32)
  int q_smem;  // queue slots in shared memory
  int q_kind;  // QueueSel kind
  uint64_t* cbuf;  // filtered search only: candidate queue C, [slots][ccap] keys
  uint32_t ccap;
  // per-query filters (filter_bits == nullptr): query qi admits what qfilters[qi] describes in qpayload
  const QueryFilter* qfilters;  // nullptr = none; [nq]
  const uint32_t* qpayload;
};

// rows of up to 512 bytes are (partly) staged by TMA: STAGE_ROWS rows + an mbarrier per warp
__host__ __device__ inline size_t stage_bytes(int d4) { return d4 <= 32 ? (size_t)STAGE_ROWS * d4 * 16 : 0; }
// register-queue stripes for a given ef (0 = queue in shared memory)
// Queue kind for a given ef (see QueueSel): compile-time chunked shared-memory queue up to ef = 256, generic beyond.
// (A register-resident variant was measured ~5 % slower at 64 registers/thread because it spills, and a speculative
// two-candidates-per-iteration loop was exact but 5-13 % slower; both were removed, see profiles/README.md.)
inline int queue_kind(int ef, int metric, int dtype) {
  const bool common = dtype == DT_F32 && (metric == METRIC_L1 || metric == METRIC_L2 || metric == METRIC_DOT || metric == METRIC_COSINE);
  if (!common || ef > 256) return 0;
  if (ef <= 32) return 101;
  if (ef <= 64) return 102;
  if (ef <= 128) return 104;
  return 108;
}
inline int queue_slots(int kind, int ef) { return kind >= 100 ? 32 * (kind - 100) : ef; }
inline size_t search_smem_per_warp(int d4, int q_smem) {
  size_t b = stage_bytes(d4) + (size_t)d4 * 16 + (size_t)q_smem * 8 + 64 * 8 + 16;
  return (b + 127) & ~(size_t)127;
}

// ---- lean kernel (search_lean.cuh): eligibility and shared-memory footprint
// rows of 128 / 256 / 512 bytes (compile-time chunk count), ef <= 128, no filter
inline int lean_queue_slots(int ef) { return ef <= 64 ? 64 : (ef <= 128 ? 128 : 0); }
inline bool lean_eligible(int d4, int ef) { return (d4 == 8 || d4 == 16 || d4 == 32) && lean_queue_slots(ef) != 0; }
inline size_t lean_smem_per_warp(int qc) { return (size_t)qc * 8 + 256; }

struct InsertParams {
  GraphView g;
  uint32_t first;   // internal id of the first point of the batch
  uint32_t count;   // points in the batch
  const uint16_t* layer_mask;  // [count] bit l set <=> some point of exact level l exists when this point searches
  int ef_c;
  int keep_pruned;
  int extend;  // extend_candidates flag (hnsw.rs:858), only with ef_c > 2M
  VisitedCfg vis;
  unsigned int* work_counter;
  int* locks;  // [capacity] per-point spin locks (phase B)
  unsigned long long* stats;
  int* status;
  int smem_per_warp;
  int threads;  // threads per CTA of the search phase (a multiple of 32)
  int q_smem;
  int q_kind;
};

inline size_t insert_smem_per_warp(int d4, int ef_c, int deg0, int q_smem) {
  size_t b = stage_bytes(d4) + (size_t)d4 * 32 + (size_t)q_smem * 8 + 512 + 16 + (size_t)deg0 * 12 + (size_t)ef_c * 2;
  return (b + 127) & ~(size_t)127;
}

cudaError_t launch_insert_search(const InsertParams& p, int metric, int dtype, int grid, size_t smem, cudaStream_t st,
                                 bool query_only, int* blocks_per_sm);
cudaError_t launch_insert_link(const InsertParams& p, int grid, cudaStream_t st);

cudaError_t launch_search_filtered(const SearchParams& p, int metric, int dtype, int grid, size_t smem, cudaStream_t st,
                                   bool query_only, int* blocks_per_sm);
cudaError_t launch_search(const SearchParams& p, int metric, int dtype, int grid, size_t smem, cudaStream_t st, bool query_only,
                          int* blocks_per_sm);
cudaError_t launch_search_std(const SearchParams& p, int metric, int dtype, int grid, size_t smem, cudaStream_t st, bool query_only,
                              int* blocks_per_sm);
cudaError_t launch_search_lean(const SearchParams& p, int metric, int dtype, int grid, size_t smem, cudaStream_t st,
                               bool query_only, int* blocks_per_sm);
cudaError_t launch_search_lean_u8(const SearchParams& p, int metric, int grid, size_t smem, cudaStream_t st, bool query_only,
                                  int* blocks_per_sm);
cudaError_t launch_search_lean_u16(const SearchParams& p, int metric, int grid, size_t smem, cudaStream_t st, bool query_only,
                                   int* blocks_per_sm);

// ---- (metric, element type) -> distance functor.  f is called as f(OpTag<Op>{}) and returns cudaError_t.
template <class Op>
struct OpTag {
  typedef Op type;
};
// CH-specialised kernels (compile-time row length) are only built for the common f32 metrics
template <class Op>
struct Specialise {
  static constexpr bool value = false;
};
template <> struct Specialise<OpL1> { static constexpr bool value = true; };
template <> struct Specialise<OpL2> { static constexpr bool value = true; };
template <> struct Specialise<OpDot> { static constexpr bool value = true; };
template <> struct Specialise<OpCosine> { static constexpr bool value = true; };

// (metric, element type) pairs the lean kernel (search_lean.cuh) is instantiated for
inline bool lean_op_supported(int metric, int dtype) {
  if (dtype == DT_F32) return metric == METRIC_L1 || metric == METRIC_L2 || metric == METRIC_DOT || metric == METRIC_COSINE;
  if (dtype == DT_U8 || dtype == DT_U16)
    return metric == METRIC_L1 || metric == METRIC_L2 || metric == METRIC_HAMMING || metric == METRIC_JACCARD;
  return false;
}

template <class T, class F>
cudaError_t dispatch_int(int metric, bool with_jaccard, F&& f) {
  switch (metric) {
    case METRIC_L1: return f(OpTag<OpCast<T, OpL1>>{});
    case METRIC_L2: return f(OpTag<OpCast<T, OpL2>>{});
    case METRIC_HAMMING: return f(OpTag<OpHamming<T>>{});
    case METRIC_JACCARD:
      if (with_jaccard) return f(OpTag<OpJaccard<T>>{});
      break;
  }
  return cudaErrorInvalidValue;
}

template <class F>
cudaError_t dispatch_op(int metric, int dtype, F&& f) {
  switch (dtype) {
    case DT_F32:
      switch (metric) {
        case METRIC_L1: return f(OpTag<OpL1>{});
        case METRIC_L2: return f(OpTag<OpL2>{});
        case METRIC_DOT: return f(OpTag<OpDot>{});
        case METRIC_COSINE: return f(OpTag<OpCosine>{});
        case METRIC_HELLINGER: return f(OpTag<OpHellinger>{});
        case METRIC_JEFFREYS: return f(OpTag<OpJeffreys>{});
        case METRIC_JENSENSHANNON: return f(OpTag<OpJS>{});
      }
      break;
    case DT_U8: return dispatch_int<uint8_t>(metric, true, f);
    case DT_U16: return dispatch_int<uint16_t>(metric, true, f);
    case DT_U32: return dispatch_int<uint32_t>(metric, true, f);
    case DT_I32: return dispatch_int<int32_t>(metric, false, f);
  }
  return cudaErrorInvalidValue;
}

// which (metric, dtype) pairs exist (mirrors init_hnsw_{f32,i32,u32,u16,u8} in /root/reference/src/libext.rs)
inline bool metric_supported(int metric, int dtype) {
  if (dtype == DT_F32)
    return metric == METRIC_L1 || metric == METRIC_L2 || metric == METRIC_DOT || metric == METRIC_COSINE ||
           metric == METRIC_HELLINGER || metric == METRIC_JEFFREYS || metric == METRIC_JENSENSHANNON;
  if (metric == METRIC_L1 || metric == METRIC_L2 || metric == METRIC_HAMMING) return true;
  return metric == METRIC_JACCARD && dtype != DT_I32;
}

}  // namespace hb
