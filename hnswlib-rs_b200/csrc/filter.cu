// Filtered query kernel: search_filter with Some(filter) (/root/reference/src/hnsw.rs:1487-1580) and the
// filter branches of search_layer (/root/reference/src/hnsw.rs:981-1001, 1037-1050).
//
// With a filter the reference's loop differs from the unfiltered one in ways that break the
// "C is the unexpanded part of W" argument of search_core.cuh:
//   * W only receives candidates that pass the filter (plus the unfiltered entry point), but C receives
//     every accepted candidate, so C is not a subset of W;
//   * the stop rule does not return: when d(c) > d(f) it only drops non-passing points from W (if |W| >= ef)
//     and keeps expanding, until C is empty.
// So here C is a real queue: an unsorted array of keys per warp in global memory, pop = warp-wide min scan
// (consumed entries are overwritten with ~0).  W is the same sorted shared-memory array as elsewhere.
// The FilterT predicate (filter.rs:7-24) is a policy (Pol below), tested at four sites: the retain pass over W, the
// per-candidate pass mask, the W.n == 1 entry-point check and the post-filter after truncation.
//   * BatchBits: one device bitmap over internal ids for the whole batch, materialised by the host;
//   * PerQuery: query qi's own filter (QueryFilter, kernels.h), loaded when the warp picks the query up: a bitmap, or an
//     ascending list of internal ids that each lane binary-searches for its own id.
#include "kernels.h"
#include "search_core.cuh"

namespace hb {

__device__ __forceinline__ bool filter_pass(const uint32_t* bits, uint32_t id) {
  return (__ldg(bits + (id >> 5)) >> (id & 31)) & 1u;
}

struct BatchBits {
  const SearchParams& p;  // reads p.filter_bits where it is used, as the kernel did before it took a policy
  __device__ __forceinline__ explicit BatchBits(const SearchParams& sp) : p(sp) {}
  __device__ __forceinline__ void load(const SearchParams&, uint32_t) {}
  __device__ __forceinline__ bool pass(uint32_t id) const { return filter_pass(p.filter_bits, id); }
};

struct PerQuery {
  const uint32_t* data;  // this query's payload
  uint32_t len;
  bool bitmap;
  __device__ __forceinline__ explicit PerQuery(const SearchParams&) : data(nullptr), len(0), bitmap(false) {}
  // every lane loads the same descriptor (one 16-byte load)
  __device__ __forceinline__ void load(const SearchParams& p, uint32_t qi) {
    const uint4 d = __ldg(reinterpret_cast<const uint4*>(p.qfilters + qi));
    data = p.qpayload + d.x;
    len = d.y;
    bitmap = d.z == QF_BITMAP;
  }
  __device__ __forceinline__ bool pass(uint32_t id) const {
    if (bitmap) return filter_pass(data, id);
    uint32_t lo = 0, hi = len;  // first position with data[pos] >= id
    while (lo < hi) {
      const uint32_t mid = (lo + hi) >> 1;
      if (__ldg(data + mid) < id) lo = mid + 1;
      else hi = mid;
    }
    return lo < len && __ldg(data + lo) == id;
  }
};

template <class Op, int CH, int U, class Pol>
__device__ __forceinline__ void search_layer_filtered(const GraphView& g, const WarpSmem& s, Visited& vis, SortedQueue& W,
                                                      uint64_t* cbuf, uint32_t ccap, const Pol& filt, uint32_t ep,
                                                      int ef, int layer, Stats& st, bool& overflow) {
  const int lane = lane_id();
  const uint4* vec4 = reinterpret_cast<const uint4*>(g.vec);
  vis.begin();
  __syncwarp();  // the descent's reads of cand_id happen-before the write below
  if (lane == 0) s.cand_id[0] = ep;
  __syncwarp();
  warp_dists<Op, CH, U>(vec4, g.d4, g.dim, s.q4, s.cand_id, 1, s.cand_d);  // hnsw.rs:952
  __syncwarp();
  st.evals += 1;
  const float d0 = Op::post(s.cand_d[0]);
  vis.test_and_set(ep, lane == 0);
  W.reset(s.wbuf, ef);
  if (lane == 0) {
    s.wbuf[0] = make_key(d0, ep);  // ep enters W unfiltered (hnsw.rs:964-967)
    cbuf[0] = make_key(d0, ep);    // and C (960-963)
  }
  W.n = 1;
  uint32_t cn = 1;
  __syncwarp();
  for (;;) {
    // ---- C.pop(): nearest candidate (hnsw.rs:971)
    uint64_t best = ~0ull;
    uint32_t bpos = 0;
    for (uint32_t b = 0; b < cn; b += 32) {
      const uint32_t i = b + lane;
      const uint64_t v = i < cn ? __ldcg(cbuf + i) : ~0ull;
      if (v < best) {
        best = v;
        bpos = i;
      }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      const uint64_t ov = __shfl_xor_sync(FULL, best, o);
      const uint32_t op = __shfl_xor_sync(FULL, bpos, o);
      if (ov < best) {
        best = ov;
        bpos = op;
      }
    }
    if (best == ~0ull) break;  // C is empty (969)
    if (lane == 0) __stcg(cbuf + bpos, ~0ull);
    // trim consumed entries at the tail so the scan stays short
    if (bpos == cn - 1) cn -= 1;
    __syncwarp();
    // The reference unwraps W.peek() here (973) and would panic on an empty W (possible only when the
    // entry point fails the filter, ef == 1 and it was retained away); we return the empty W instead.
    if (W.n == 0) break;
    const uint64_t fkey = W.w[W.n - 1] & ~1ull;
    // 981: the reference compares DISTANCES here (-(c.dist) > f.dist); with equal distances a larger id must not
    // trigger the retain pass (Hamming / Jaccard / integer L1 tie often)
    if ((best >> 32) > (fkey >> 32) && W.n >= ef) {  // 994-1000: retain only the points passing the filter
      int out = 0;
      for (int b = 0; b < W.n; b += 32) {
        const int i = b + lane;
        uint64_t v = 0;
        bool keep = false;
        if (i < W.n) {
          v = W.w[i];
          keep = filt.pass(key_id(v));
        }
        const unsigned m = __ballot_sync(FULL, keep);
        __syncwarp();
        if (keep) W.w[out + __popc(m & ((1u << lane) - 1u))] = v;
        out += __popc(m);
        __syncwarp();
      }
      W.n = out;
    }
    const uint32_t c = key_id(best);
    int cap;
    const uint32_t* ids = list_ids(g, c, layer, cap);  // 1006
    st.expansions += 1;
    bool done = false;
    for (int base = 0; base < cap && !done; base += 32) {
      const uint32_t nid = (base + lane < cap) ? ids[base + lane] : INVALID_ID;
      const unsigned valid = __ballot_sync(FULL, nid != INVALID_ID);
      st.adj += __popc(valid);
      const bool fresh = vis.test_and_set(nid, nid != INVALID_ID);  // 1016-1017
      const unsigned m = __ballot_sync(FULL, fresh);
      const int cnt = __popc(m);
      if (cnt) {
        const int pos = __popc(m & ((1u << lane) - 1u));
        if (fresh) s.cand_id[pos] = nid;
        __syncwarp();
        warp_dists<Op, CH, U>(vec4, g.d4, g.dim, s.q4, s.cand_id, cnt, s.cand_d);  // 1026
        __syncwarp();
        st.evals += cnt;
        const uint32_t my_id = lane < cnt ? s.cand_id[lane] : 0u;
        const uint64_t key = lane < cnt ? make_key(Op::post(s.cand_d[lane]), my_id) : ~0ull;
        const bool my_pass = lane < cnt && filt.pass(my_id);
        const unsigned passmask = __ballot_sync(FULL, my_pass);
        for (int j = 0; j < cnt; ++j) {  // strictly in list order: the accept rule sees the W of that moment
          if (W.n == 0) {                // 1019-1024
            done = true;
            break;
          }
          const uint64_t kj = __shfl_sync(FULL, key, j);
          if (W.n < ef || kj < (W.w[W.n - 1] & ~1ull)) {  // 1028
            if (cn >= ccap) {
              overflow = true;
              done = true;
              break;
            }
            if (lane == 0) __stcg(cbuf + cn, kj);  // 1035-1036: every accepted candidate goes to C
            cn += 1;
            if ((passmask >> j) & 1u) {  // 1040-1049
              if (W.n == 1 && !filt.pass(key_id(W.w[0]))) W.n = 0;
              __syncwarp();
              W.insert(kj);  // push, and pop the farthest when over ef (1051-1053)
            }
          }
        }
        __syncwarp();
      }
      if (valid != FULL) break;
    }
    if (done && W.n == 0) break;
    if (overflow || vis.overflowing()) {
      overflow = true;
      break;
    }
  }
}

template <class Op, int CH, int U, class Pol>
__global__ void __launch_bounds__(SEARCH_THREADS) search_filter_kernel(SearchParams p) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const GraphView& g = p.g;
  unsigned char* base = smem_raw + (size_t)warp * p.smem_per_warp;
  const size_t stb = stage_bytes(g.d4);  // same per-warp layout as search.cu (the stage is unused here)
  WarpSmem s;
  s.q4 = reinterpret_cast<uint4*>(base + stb);
  s.wbuf = reinterpret_cast<uint64_t*>(base + stb + (size_t)g.d4 * 16);
  s.cand_id = reinterpret_cast<uint32_t*>(base + stb + (size_t)g.d4 * 16 + (size_t)p.q_smem * 8);
  s.cand_d = reinterpret_cast<float*>(s.cand_id + 32);
  const uint32_t slot = blockIdx.x * (blockDim.x >> 5) + warp;  // the host launches fewer warps per CTA when shared memory is short
  Visited vis;
  vis.init(p.vis, slot);
  uint64_t* cbuf = p.cbuf + (size_t)slot * p.ccap;
  SortedQueue W;
  Stats st{0, 0, 0};
  const uint4* vec4 = reinterpret_cast<const uint4*>(g.vec);
  Pol filt(p);

  for (;;) {
    uint32_t qi = 0;
    if (lane == 0) qi = atomicAdd(p.work_counter, 1u);
    qi = __shfl_sync(FULL, qi, 0);
    if (qi >= p.nq) break;
    filt.load(p, qi);
    stage_row_bytes(s.q4, reinterpret_cast<const char*>(p.queries) + (size_t)qi * p.q_stride_bytes, p.q_bytes, g.d4 * 16);
    int count = 0;
    bool overflow = false;
    W.reset(s.wbuf, p.ef);
    if (g.entry != INVALID_ID) {
      // descent identical to the unfiltered kernel (hnsw.rs:1511-1529: the filter plays no role here)
      uint32_t pivot = g.entry;
      if (lane == 0) s.cand_id[0] = pivot;
      __syncwarp();
      warp_dists<Op, CH, U>(vec4, g.d4, g.dim, s.q4, s.cand_id, 1, s.cand_d);
      __syncwarp();
      st.evals += 1;
      float best = Op::post(s.cand_d[0]);
      for (int layer = g.entry_level; layer >= 1; --layer) {
        int cap;
        const uint32_t* ids = list_ids(g, pivot, layer, cap);
        uint32_t new_pivot = pivot;
        for (int b = 0; b < cap; b += 32) {
          const uint32_t nid = (b + lane < cap) ? ids[b + lane] : INVALID_ID;
          const unsigned valid = __ballot_sync(FULL, nid != INVALID_ID);
          const int cnt = __popc(valid);
          if (cnt) {
            __syncwarp();
            if (lane < cnt) s.cand_id[lane] = nid;
            __syncwarp();
            warp_dists<Op, CH, U>(vec4, g.d4, g.dim, s.q4, s.cand_id, cnt, s.cand_d);
            __syncwarp();
            st.evals += cnt;
            st.adj += cnt;
            uint64_t key = lane < cnt ? (((uint64_t)__float_as_uint(Op::post(s.cand_d[lane])) << 32) | (uint32_t)lane) : ~0ull;
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) {
              uint64_t other = __shfl_xor_sync(FULL, key, o);
              key = other < key ? other : key;
            }
            const float dmin = __uint_as_float((uint32_t)(key >> 32));
            if (dmin < best) {
              best = dmin;
              new_pivot = s.cand_id[(uint32_t)key & 31u];
            }
          }
          if (valid != FULL) break;
        }
        pivot = new_pivot;
      }
      search_layer_filtered<Op, CH, U, Pol>(g, s, vis, W, cbuf, p.ccap, filt, pivot, p.ef, p.layer0, st, overflow);
      count = min(p.k, min(p.ef, W.n));  // hnsw.rs:1547
    }
    if (overflow) {
      if (lane == 0) atomicExch(p.status, 1);
      count = 0;
    }
    // post-filter AFTER truncation (hnsw.rs:1549-1563): only the entry point can fail here
    const size_t ob = (size_t)qi * p.k;
    int outn = 0;
    for (int b = 0; b < count; b += 32) {
      const int j = b + lane;
      uint64_t key = 0;
      bool keep = false;
      if (j < count) {
        key = W.w[j];
        keep = filt.pass(key_id(key));
      }
      const unsigned m = __ballot_sync(FULL, keep);
      if (keep) {
        const uint32_t id = key_id(key);
        p.out_nb[ob + outn + __popc(m & ((1u << lane) - 1u))] = NeighbourOut{g.origin[id], key_dist(key), id};
      }
      outn += __popc(m);
    }
    for (int j = outn + lane; j < p.k; j += 32) p.out_nb[ob + j] = NeighbourOut{~0ull, __int_as_float(0x7f800000), INVALID_ID};
    if (lane == 0) p.out_count[qi] = outn;
    __syncwarp();
  }
  vis.save(p.vis, slot);
  if (p.stats && lane == 0) {
    atomicAdd(p.stats + 0, (unsigned long long)st.evals);
    atomicAdd(p.stats + 1, (unsigned long long)st.expansions);
    atomicAdd(p.stats + 2, (unsigned long long)st.adj);
  }
}

template <class Op, class Pol>
static cudaError_t launch_filter_for_op(const SearchParams& p, int grid, size_t smem, cudaStream_t st, bool query_only,
                                        int* blocks_per_sm) {
  const int ch = p.g.d4 / 8;
#define HB_LAUNCH(CHV, UV)                                                                              \
  do {                                                                                                  \
    auto kern = search_filter_kernel<Op, CHV, UV, Pol>;                                                 \
    cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem); \
    if (e != cudaSuccess) return e;                                                                     \
    if (blocks_per_sm) {                                                                                \
      e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(blocks_per_sm, kern, p.threads, smem);     \
      if (e != cudaSuccess) return e;                                                                   \
    }                                                                                                   \
    if (!query_only) kern<<<grid, p.threads, smem, st>>>(p);                                       \
    return cudaGetLastError();                                                                          \
  } while (0)
  if constexpr (Specialise<Op>::value) {
    if (ch == 4) HB_LAUNCH(4, 2);
  }
  HB_LAUNCH(0, 2);
#undef HB_LAUNCH
}

cudaError_t launch_search_filtered(const SearchParams& p, int metric, int dtype, int grid, size_t smem, cudaStream_t st,
                                   bool query_only, int* blocks_per_sm) {
  return dispatch_op(metric, dtype, [&](auto tag) -> cudaError_t {
    using Op = typename decltype(tag)::type;
    if (p.qfilters) return launch_filter_for_op<Op, PerQuery>(p, grid, smem, st, query_only, blocks_per_sm);
    return launch_filter_for_op<Op, BatchBits>(p, grid, smem, st, query_only, blocks_per_sm);
  });
}

}  // namespace hb
