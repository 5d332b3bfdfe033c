// Host-side index: HBM allocation, insert-batch scheduling, query launches, import/export.
// See index.h for what it replaces in the reference.
#include "index.h"

#include <algorithm>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>

namespace hb {

#define HB_CUDA(call)                                   \
  do {                                                  \
    cudaError_t e__ = (call);                           \
    if (e__ != cudaSuccess) return cuda_fail(e__, #call); \
  } while (0)

static size_t next_pow2(size_t x) {
  size_t p = 1;
  while (p < x) p <<= 1;
  return p;
}
static int ilog2(size_t p) {
  int r = 0;
  while (((size_t)1 << r) < p) ++r;
  return r;
}

// searches run concurrently: the message of the last failure is guarded (the C ABI copies it into a thread-local string)
int Index::fail(const std::string& m) const {
  std::lock_guard<std::mutex> lk(err_mu_);
  err_ = m;
  return -1;
}
int Index::cuda_fail(cudaError_t e, const char* what) const {
  std::lock_guard<std::mutex> lk(err_mu_);
  err_ = std::string("CUDA error: ") + cudaGetErrorString(e) + " at " + what;
  return -2;
}
std::string Index::err() const {
  std::lock_guard<std::mutex> lk(err_mu_);
  return err_;
}

Index::Index(int M_, size_t max_elements_, int max_layer_, int ef_c_, int metric_, int dtype_, int device_)
    : M(M_), max_layer(std::min(max_layer_, MAX_LAYERS)), ef_c(ef_c_), metric(metric_), dtype(dtype_),
      es(dtype_size(dtype_)), device(device_),
      max_elements(max_elements_) {
  for (int l = 0; l < MAX_LAYERS; ++l) layer_count[l] = 0;
  level_scale = 1.0 / std::log((double)M);  // hnsw.rs:327
  int ndev = 0;
  cudaError_t e = cudaGetDeviceCount(&ndev);
  if (e != cudaSuccess || ndev <= 0) {
    err_ = std::string("no usable CUDA device: ") + cudaGetErrorString(e) + " (this engine has no CPU fallback)";
    return;
  }
  if (device >= ndev) {
    err_ = "device index out of range";
    return;
  }
  if ((e = cudaSetDevice(device)) != cudaSuccess || (e = cudaStreamCreateWithFlags(&stream_, cudaStreamNonBlocking)) != cudaSuccess) {
    err_ = std::string("CUDA init failed: ") + cudaGetErrorString(e);
    return;
  }
  for (SearchCtx& c : ctx_) {
    if ((e = cudaStreamCreateWithFlags(&c.stream, cudaStreamNonBlocking)) != cudaSuccess ||
        (e = cudaEventCreateWithFlags(&c.fork, cudaEventDisableTiming)) != cudaSuccess ||
        (e = cudaEventCreateWithFlags(&c.join, cudaEventDisableTiming)) != cudaSuccess ||
        (e = cudaEventCreate(&c.ev0)) != cudaSuccess || (e = cudaEventCreate(&c.ev1)) != cudaSuccess ||
        (e = cudaMalloc(&c.d_counter, sizeof(unsigned int))) != cudaSuccess || (e = cudaMalloc(&c.d_status, sizeof(int))) != cudaSuccess ||
        (e = cudaMemset(c.d_status, 0, sizeof(int))) != cudaSuccess) {
      err_ = std::string("CUDA init failed: ") + cudaGetErrorString(e);
      return;
    }
  }
  cudaDeviceProp prop;
  if ((e = cudaGetDeviceProperties(&prop, device)) != cudaSuccess) {
    err_ = std::string("cudaGetDeviceProperties: ") + cudaGetErrorString(e);
    return;
  }
  own_stream_ = stream_;
  sm_count_ = prop.multiProcessorCount;
  if (const char* k = getenv("HNSW_B200_KERNEL")) kernel_pref_ = strcmp(k, "warp") == 0 ? 1 : 0;
  if (const char* k = getenv("HNSW_B200_ZERO_COPY")) zero_copy_ = atoi(k) != 0;
  if ((e = cudaMalloc(&d_counter_, sizeof(unsigned int))) != cudaSuccess || (e = cudaMalloc(&d_status_, sizeof(int))) != cudaSuccess ||
      (e = cudaMalloc(&d_stats_, 4 * sizeof(unsigned long long))) != cudaSuccess) {
    err_ = std::string("cudaMalloc: ") + cudaGetErrorString(e);
    return;
  }
  cudaMemset(d_stats_, 0, 4 * sizeof(unsigned long long));
  cudaMemset(d_status_, 0, sizeof(int));
  ok_ = true;
}

Index::~Index() {
  DeviceRestore keep;
  drop_replicas();
  nccl_destroy();
  cudaSetDevice(device);
  if (stream_) cudaStreamSynchronize(stream_);
  cudaFree(d_vec_.p); cudaFree(d_adj0_.p); cudaFree(d_adjU_.p); cudaFree(d_upoff_.p); cudaFree(d_adj0d_.p);
  cudaFree(d_adjUd_.p); cudaFree(d_level_.p); cudaFree(d_plevel_.p); cudaFree(d_origin_.p); cudaFree(d_locks_.p);
  cudaFree(vis_.tab); cudaFree(vis_.epoch); cudaFree(d_counter_); cudaFree(d_status_); cudaFree(d_stats_); cudaFree(d_mask_);
  if (h_pin_) cudaFreeHost(h_pin_);
  for (SearchCtx& c : ctx_) {
    if (c.stream) cudaStreamSynchronize(c.stream);
    cudaFree(c.vis.tab); cudaFree(c.vis.epoch); cudaFree(c.fvis.tab); cudaFree(c.fvis.epoch); cudaFree(c.d_counter); cudaFree(c.d_status);
    cudaFree(c.d_q); cudaFree(c.d_out); cudaFree(c.d_cnt); cudaFree(c.d_fbits); cudaFree(c.d_cbuf);
    cudaFree(c.d_qf);
    if (c.h_pin) cudaFreeHost(c.h_pin);
    if (c.h_res) cudaFreeHost(c.h_res);
    if (c.fork) cudaEventDestroy(c.fork);
    if (c.join) cudaEventDestroy(c.join);
    if (c.ev0) cudaEventDestroy(c.ev0);
    if (c.ev1) cudaEventDestroy(c.ev1);
    if (c.stream) cudaStreamDestroy(c.stream);
  }
  if (own_stream_) cudaStreamDestroy(own_stream_);
}

template <class T>
int Index::grow(DevArray<T>& a, size_t need, size_t keep, int fill) {
  if (need <= a.cap) return 0;
  T* np = nullptr;
  HB_CUDA(cudaMalloc(&np, need * sizeof(T)));
  HB_CUDA(cudaMemsetAsync(np, fill, need * sizeof(T), stream_));
  if (keep && a.p) HB_CUDA(cudaMemcpyAsync(np, a.p, keep * sizeof(T), cudaMemcpyDeviceToDevice, stream_));
  HB_CUDA(cudaStreamSynchronize(stream_));
  cudaFree(a.p);
  a.p = np;
  a.cap = need;
  return 0;
}

int Index::set_dim(int d) {
  if (d <= 0) return fail("dimension must be positive");
  if (dim == 0) {
    dim = d;
    row_bytes = (d * es + 127) / 128 * 128;
    return 0;
  }
  if (dim != d) return fail("vector length differs from the index dimension (the flat point store needs one dimension)");
  return 0;
}

int Index::ensure_points(size_t need) {
  if (need <= cap_) return 0;
  if (need >= (size_t)1 << 31) return fail("more than 2^31 points are not supported");
  size_t nc = std::max(need, cap_ * 2);
  if (cap_ == 0) nc = std::max(nc, std::max<size_t>(max_elements, 1024));
  const size_t deg0 = (size_t)2 * M;
  int r;
  if ((r = grow(d_vec_, nc * (size_t)row_bytes, n * (size_t)row_bytes, 0))) return r;
  if ((r = grow(d_adj0_, nc * deg0, n * deg0, 0xFF))) return r;
  if ((r = grow(d_adj0d_, nc * deg0, n * deg0, 0))) return r;
  if ((r = grow(d_upoff_, nc, n, 0xFF))) return r;
  if ((r = grow(d_level_, nc, n, 0))) return r;
  if ((r = grow(d_plevel_, nc, n, 0))) return r;
  if ((r = grow(d_origin_, nc, n, 0))) return r;
  if ((r = grow(d_locks_, nc, n, 0))) return r;
  cap_ = nc;
  return 0;
}

int Index::ensure_upper(size_t need) {
  if (need <= cap_ul_) return 0;
  size_t nc = std::max(need, std::max<size_t>(cap_ul_ * 2, 1024));
  int r;
  if ((r = grow(d_adjU_, nc * M, n_ul * M, 0xFF))) return r;
  if ((r = grow(d_adjUd_, nc * M, n_ul * M, 0))) return r;
  cap_ul_ = nc;
  return 0;
}

// A pool is laid out as [slots][cap] for the (slots, cap) it was last sized for.  Insert and filtered search share one
// pool (large tables); unfiltered searches own another, so that their small L2-resident tables are not inflated by
// the insert path's (4x larger: ef_construction instead of ef).
int Index::ensure_visited(VisitedPool& v, size_t slots, size_t cap_entries, cudaStream_t st) {
  if (slots <= v.slots && cap_entries <= v.cap) return 0;
  size_t ns = std::max(slots, v.slots), nc = std::max(cap_entries, v.cap);
  if (ns * nc * sizeof(uint32_t) > ((size_t)8 << 30)) {  // do not carry a huge shape over (filtered searches use few, big tables)
    ns = slots;
    nc = cap_entries;
  }
  HB_CUDA(cudaStreamSynchronize(st));
  cudaFree(v.tab);
  cudaFree(v.epoch);
  v.tab = v.epoch = nullptr;
  v.slots = v.cap = 0;
  HB_CUDA(cudaMalloc(&v.tab, ns * nc * sizeof(uint32_t)));
  HB_CUDA(cudaMalloc(&v.epoch, ns * sizeof(uint32_t)));
  HB_CUDA(cudaMemsetAsync(v.tab, 0, ns * nc * sizeof(uint32_t), st));
  // epoch = max forces a table clear on first use whatever id_bits is (Visited::begin)
  HB_CUDA(cudaMemsetAsync(v.epoch, 0xFF, ns * sizeof(uint32_t), st));
  v.slots = ns;
  v.cap = nc;
  return 0;
}

int Index::fill_visited_cfg(VisitedPool& v, VisitedCfg& c, cudaStream_t st) {
  const int id_bits = std::max(1, ilog2(std::max<size_t>(cap_, 2)));
  if (id_bits != v.id_bits) {  // entries are (epoch << id_bits) | id: a new split invalidates every table
    HB_CUDA(cudaMemsetAsync(v.epoch, 0xFF, v.slots * sizeof(uint32_t), st));
    v.id_bits = id_bits;
  }
  c.tables = v.tab;
  c.epochs = v.epoch;
  c.cap = (uint32_t)v.cap;
  c.shift = 32 - ilog2(v.cap);
  c.id_bits = id_bits;
  return 0;
}

int Index::ensure_scratch(void** p, size_t* cur, size_t need, cudaStream_t st) {
  if (need <= *cur) return 0;
  HB_CUDA(cudaStreamSynchronize(st));
  cudaFree(*p);
  *p = nullptr;
  *cur = 0;
  size_t nb = std::max(need, (size_t)4096);
  HB_CUDA(cudaMalloc(p, nb));
  *cur = nb;
  return 0;
}

GraphView Index::view() const {
  GraphView g;
  g.vec = d_vec_.p;
  g.d4 = row_bytes / 16;
  g.dim = dim;
  g.adj0 = d_adj0_.p;
  g.adj0_d = d_adj0d_.p;
  g.deg0 = 2 * M;
  g.adjU = d_adjU_.p;
  g.adjU_d = d_adjUd_.p;
  g.M = M;
  g.up_off = d_upoff_.p;
  g.plevel = d_plevel_.p;
  g.level = d_level_.p;
  g.origin = d_origin_.p;
  g.n = (uint32_t)n;
  g.entry = entry;
  g.entry_level = entry_level;
  return g;
}

// LayerGenerator::generate, hnsw.rs:363-374 (law only; the reference's StdRng stream needs the rand crate)
int Index::draw_level() {
  double xsi = rng.unif();
  if (xsi <= 0.) xsi = 1e-300;
  double level = -std::log(xsi) * level_scale;
  size_t ul = (size_t)std::floor(level);
  if (ul >= (size_t)max_layer) ul = (size_t)(rng.next() % (uint64_t)max_layer);
  return (int)ul;
}

// ------------------------------------------------------------------------------------------------
// insert
int Index::grow_plevel(uint32_t id, int new_pl) {
  const int old = h_plevel[id];
  if (new_pl <= old) return 0;
  int r;
  if ((r = ensure_upper(n_ul + new_pl))) return r;
  if (old > 0) {
    const size_t src = (size_t)h_upoff[id] * M, dst = n_ul * M, cnt = (size_t)old * M;
    HB_CUDA(cudaMemcpyAsync(d_adjU_.p + dst, d_adjU_.p + src, cnt * 4, cudaMemcpyDeviceToDevice, stream_));
    HB_CUDA(cudaMemcpyAsync(d_adjUd_.p + dst, d_adjUd_.p + src, cnt * 4, cudaMemcpyDeviceToDevice, stream_));
  }
  h_upoff[id] = (uint32_t)n_ul;
  h_plevel[id] = (uint8_t)new_pl;
  n_ul += new_pl;
  HB_CUDA(cudaMemcpyAsync(d_upoff_.p + id, &h_upoff[id], 4, cudaMemcpyHostToDevice, stream_));
  HB_CUDA(cudaMemcpyAsync(d_plevel_.p + id, &h_plevel[id], 1, cudaMemcpyHostToDevice, stream_));
  HB_CUDA(cudaStreamSynchronize(stream_));
  return 0;
}

// shared-memory footprint of the insert kernel for this (dimension, ef_construction, M): checked before an insert
// changes any state
int Index::check_insert_fit() {
  int qk = queue_kind(ef_c, metric, dtype);
  if (qk != 0 && qk < 104) qk = 104;
  const size_t spw = insert_smem_per_warp(row_bytes / 16, ef_c, 2 * M, queue_slots(qk, ef_c));
  if (spw > 220 * 1024)
    return fail("ef_construction / dimension too large: one insert needs " + std::to_string(spw) + " bytes of shared memory (limit 220 KB)");
  return 0;
}

// forget the points [keep, n): they were stored but never linked (a failed insert call)
void Index::rollback_points(size_t keep) {
  invalidate_origin_table();
  n = keep;
  h_level.resize(keep);
  h_plevel.resize(keep);
  h_rank.resize(keep);
  h_origin.resize(keep);
  h_upoff.resize(keep);
  for (int l = 0; l < MAX_LAYERS; ++l) layer_count[l] = 0;
  n_ul = 0;
  for (size_t p = 0; p < keep; ++p) {
    layer_count[h_level[p]]++;
    if (h_plevel[p] > 0) n_ul = std::max<size_t>(n_ul, (size_t)h_upoff[p] + h_plevel[p]);
  }
}

int Index::run_insert_range(size_t first, size_t count, const std::vector<uint16_t>& masks, size_t mask_off) {
  (void)masks;
  InsertParams p;
  p.g = view();
  p.first = (uint32_t)first;
  p.count = (uint32_t)count;
  p.layer_mask = reinterpret_cast<const uint16_t*>(d_mask_) + mask_off;
  p.ef_c = ef_c;
  p.keep_pruned = keep_pruned ? 1 : 0;
  p.extend = extend_candidates ? 1 : 0;
  p.work_counter = d_counter_;
  p.locks = d_locks_.p;
  p.stats = stats_on_ ? d_stats_ : nullptr;  // insert-path distance evaluations / expansions / adjacency ids read
  p.status = d_status_;
  p.q_kind = queue_kind(ef_c, metric, dtype);
  if (p.q_kind != 0 && p.q_kind < 104) p.q_kind = 104;  // the insert kernel is built for 128 / 256-slot queues only
  p.q_smem = queue_slots(p.q_kind, ef_c);
  const size_t spw = insert_smem_per_warp(p.g.d4, ef_c, p.g.deg0, p.q_smem);
  p.smem_per_warp = (int)spw;
  int wpb = BUILD_THREADS / 32;
  while (wpb > 1 && spw * wpb > 220 * 1024) wpb >>= 1;  // fewer inserts per CTA when one warp's share is large
  const size_t smem = spw * wpb;
  if (smem > 220 * 1024) return fail("ef_construction / dimension too large for the insert kernel's shared memory");
  p.threads = wpb * 32;
  int bps = 0;
  HB_CUDA(launch_insert_search(p, metric, dtype, 0, smem, stream_, true, &bps));
  if (bps < 1) return fail("insert kernel does not fit on an SM");
  int grid = (int)std::min<size_t>((size_t)sm_count_ * bps, (count + wpb - 1) / wpb);
  size_t vcap = next_pow2(std::max<size_t>(1024, (size_t)2 * (ef_c + 16) * p.g.deg0));
  for (int attempt = 0;; ++attempt) {
    int r;
    if ((r = ensure_visited(vis_, (size_t)grid * wpb, vcap, stream_))) return r;
    if ((r = fill_visited_cfg(vis_, p.vis, stream_))) return r;
    HB_CUDA(cudaMemsetAsync(d_counter_, 0, sizeof(unsigned int), stream_));
    HB_CUDA(launch_insert_search(p, metric, dtype, grid, smem, stream_, false, nullptr));
    int status = 0;
    HB_CUDA(cudaMemcpyAsync(&status, d_status_, sizeof(int), cudaMemcpyDeviceToHost, stream_));
    HB_CUDA(cudaStreamSynchronize(stream_));
    if (status == 0) break;
    if (attempt >= 8) return fail("visited table overflow persists");
    HB_CUDA(cudaMemsetAsync(d_status_, 0, sizeof(int), stream_));
    vcap = vis_.cap * 2;  // rare: a search wandered further than 2*(ef+16)*degree nodes
  }
  int lgrid = (int)std::min<size_t>((size_t)sm_count_ * 8, (count + wpb - 1) / wpb);
  HB_CUDA(launch_insert_link(p, lgrid, stream_));
  return 0;
}

int Index::insert_batch(const void* vecs, size_t n_new, size_t stride, const void* const* rows, const uint64_t* ids,
                        const int32_t* levels) {
  if (n_new == 0) return 0;
  if (dim == 0) return fail("dimension not set");
  if (poisoned_) return fail(poison_msg_);
  HB_CUDA(cudaSetDevice(device));
  int fit = check_insert_fit();
  if (fit) return fit;
  replicas_stale_ = !replicas_.empty();  // the copies on the other devices are re-broadcast before the next sharded search
  // ---- levels, PointId ranks, upper-list allocation (generate_new_point, hnsw.rs:503-531)
  std::vector<int> lv(n_new);
  size_t need_ul = 0;
  for (size_t i = 0; i < n_new; ++i) {
    int l = levels ? levels[i] : draw_level();
    if (l < 0) l = 0;
    if (l >= max_layer) l = max_layer - 1;
    lv[i] = l;
    need_ul += l;
  }
  int r;
  if ((r = ensure_points(n + n_new))) return r;
  if ((r = ensure_upper(n_ul + need_ul + 2 * MAX_LAYERS))) return r;
  const size_t first = n;
  invalidate_origin_table();
  h_level.resize(first + n_new);
  h_plevel.resize(first + n_new);
  h_rank.resize(first + n_new);
  h_origin.resize(first + n_new);
  h_upoff.resize(first + n_new);
  std::vector<uint16_t> masks(n_new);
  for (size_t i = 0; i < n_new; ++i) {
    const size_t id = first + i;
    h_level[id] = (uint8_t)lv[i];
    h_plevel[id] = (uint8_t)lv[i];
    h_rank[id] = (int32_t)layer_count[lv[i]];
    layer_count[lv[i]]++;
    h_origin[id] = ids ? ids[i] : (uint64_t)id;
    if (lv[i] > 0) {
      h_upoff[id] = (uint32_t)n_ul;
      n_ul += lv[i];
    } else {
      h_upoff[id] = INVALID_ID;
    }
    uint16_t m = 0;
    for (int l = 0; l < MAX_LAYERS; ++l)
      if (layer_count[l] > 0) m |= (uint16_t)(1u << l);
    masks[i] = m;
  }
  // ---- upload vectors (rows padded to d_pad on the device; the padding was zero-filled at allocation)
  if (rows) {
    const size_t rb = (size_t)dim * es;  // bytes of one user row
    const size_t chunk = std::max<size_t>(1, (size_t)(8u << 20) / rb);
    if (h_pin_bytes_ < chunk * rb) {
      if (h_pin_) cudaFreeHost(h_pin_);
      h_pin_ = nullptr;
      h_pin_bytes_ = 0;
      HB_CUDA(cudaMallocHost(&h_pin_, chunk * rb));
      h_pin_bytes_ = chunk * rb;
    }
    for (size_t b = 0; b < n_new; b += chunk) {
      const size_t c = std::min(chunk, n_new - b);
      unsigned char* st = (unsigned char*)h_pin_;
      for (size_t i = 0; i < c; ++i) memcpy(st + i * rb, rows[b + i], rb);
      HB_CUDA(cudaMemcpy2DAsync(d_vec_.p + (first + b) * (size_t)row_bytes, (size_t)row_bytes, st, rb, rb, c,
                                cudaMemcpyHostToDevice, stream_));
      HB_CUDA(cudaStreamSynchronize(stream_));
    }
  } else {
    HB_CUDA(cudaMemcpy2DAsync(d_vec_.p + first * (size_t)row_bytes, (size_t)row_bytes, vecs, stride * es, (size_t)dim * es, n_new,
                              cudaMemcpyHostToDevice, stream_));
  }
  HB_CUDA(cudaMemcpyAsync(d_level_.p + first, h_level.data() + first, n_new, cudaMemcpyHostToDevice, stream_));
  HB_CUDA(cudaMemcpyAsync(d_plevel_.p + first, h_plevel.data() + first, n_new, cudaMemcpyHostToDevice, stream_));
  HB_CUDA(cudaMemcpyAsync(d_origin_.p + first, h_origin.data() + first, n_new * 8, cudaMemcpyHostToDevice, stream_));
  HB_CUDA(cudaMemcpyAsync(d_upoff_.p + first, h_upoff.data() + first, n_new * 4, cudaMemcpyHostToDevice, stream_));
  if ((r = ensure_scratch(&d_mask_, &d_mask_bytes_, n_new * 2, stream_))) return r;
  HB_CUDA(cudaMemcpyAsync(d_mask_, masks.data(), n_new * 2, cudaMemcpyHostToDevice, stream_));
  n = first + n_new;  // stored; points become reachable as their batch links them
  // ---- schedule batches
  size_t done = 0;
  while (done < n_new) {
    const size_t id = first + done;
    if (entry == INVALID_ID) {  // very first point: becomes the entry point (hnsw.rs:1106-1109)
      entry = (uint32_t)id;
      entry_level = lv[done];
      done++;
      continue;
    }
    const size_t linked = first + done;
    size_t nb = std::min<size_t>(std::max<size_t>(linked / std::max<uint32_t>(batch_ratio, 1), 1), batch_max);
    nb = std::min(nb, n_new - done);
    bool promo = false;
    for (size_t j = 0; j < nb; ++j) {
      if (lv[done + j] > entry_level) {  // a new top level: alone in its batch (check_entry_point, hnsw.rs:534-557)
        if (j == 0) {
          nb = 1;
          promo = true;
        } else {
          nb = j;
        }
        break;
      }
    }
    r = promo ? grow_plevel(entry, lv[done]) : 0;  // old entry point gains lists up to the new top
    if (!r) r = run_insert_range(id, nb, masks, done);
    if (r) {
      // the batches before this one are fully linked and stay; the rest of the call is forgotten.  A CUDA failure can
      // leave half-written links behind: the handle then refuses further work instead of serving a broken graph.
      const std::string why = err_;
      if (r == -2) {
        poisoned_ = true;
        poison_msg_ = "index unusable after a CUDA failure during insert: " + why;
      }
      rollback_points(id);
      err_ = why + " (insert rolled back to " + std::to_string(id) + " points)";
      return r;
    }
    if (promo) {
      entry = (uint32_t)id;
      entry_level = lv[done];
    }
    done += nb;
  }
  HB_CUDA(cudaStreamSynchronize(stream_));
  return 0;
}

// ------------------------------------------------------------------------------------------------
// import of a graph built elsewhere (oracle, another rank, a dump)
int Index::import_graph(const void* vecs, size_t n_new, int d, const uint64_t* origin, const uint8_t* levels,
                        int64_t entry_id, int nlayers, const uint64_t* const* offsets, const uint32_t* const* ids,
                        const float* const* dists) {
  if (n != 0) return fail("import_graph needs an empty index");
  if (n_new == 0) return 0;
  HB_CUDA(cudaSetDevice(device));
  int r;
  if ((r = set_dim(d))) return r;
  if (nlayers > MAX_LAYERS) nlayers = MAX_LAYERS;
  // present level: plevel[p] = highest layer at which p can be visited = max(level, highest layer l where p
  // appears in the layer-l list of a point present at l).  Fixpoint per layer, top down.
  std::vector<uint8_t> pl(levels, levels + n_new);
  for (int l = nlayers - 1; l >= 1; --l) {
    std::vector<uint32_t> work;
    std::vector<uint8_t> in(n_new, 0);
    for (size_t p = 0; p < n_new; ++p)
      if (pl[p] >= l) {
        in[p] = 1;
        work.push_back((uint32_t)p);
      }
    while (!work.empty()) {
      uint32_t q = work.back();
      work.pop_back();
      for (uint64_t j = offsets[l][q]; j < offsets[l][q + 1]; ++j) {
        uint32_t p = ids[l][j];
        if (p < n_new && !in[p]) {
          in[p] = 1;
          if (pl[p] < l) pl[p] = (uint8_t)l;
          work.push_back(p);
        }
      }
    }
  }
  size_t need_ul = 0;
  for (size_t p = 0; p < n_new; ++p) need_ul += pl[p];
  if ((r = ensure_points(n_new))) return r;
  if ((r = ensure_upper(need_ul + 2 * MAX_LAYERS))) return r;
  const size_t deg0 = (size_t)2 * M;
  h_level.assign(levels, levels + n_new);
  h_plevel = pl;
  h_rank.resize(n_new);
  invalidate_origin_table();  // also the path of a dump load (load_dump)
  h_origin.assign(origin, origin + n_new);
  h_upoff.resize(n_new);
  for (int l = 0; l < MAX_LAYERS; ++l) layer_count[l] = 0;
  n_ul = 0;
  for (size_t p = 0; p < n_new; ++p) {
    h_rank[p] = (int32_t)layer_count[levels[p]]++;
    if (pl[p] > 0) {
      h_upoff[p] = (uint32_t)n_ul;
      n_ul += pl[p];
    } else {
      h_upoff[p] = INVALID_ID;
    }
  }
  std::vector<uint32_t> a0(n_new * deg0, INVALID_ID), aU(std::max<size_t>(n_ul, 1) * M, INVALID_ID);
  std::vector<float> a0d(n_new * deg0, 0.f), aUd(std::max<size_t>(n_ul, 1) * M, 0.f);
  for (size_t p = 0; p < n_new; ++p) {
    if (nlayers > 0) {
      uint64_t b = offsets[0][p], e = offsets[0][p + 1];
      if (e - b > deg0) return fail("layer-0 list longer than 2*max_nb_connection");
      for (uint64_t j = b; j < e; ++j) {
        a0[p * deg0 + (j - b)] = ids[0][j];
        if (dists && dists[0]) a0d[p * deg0 + (j - b)] = dists[0][j];
      }
    }
    for (int l = 1; l <= pl[p] && l < nlayers; ++l) {
      uint64_t b = offsets[l][p], e = offsets[l][p + 1];
      if (e - b > (uint64_t)M) return fail("upper-layer list longer than max_nb_connection");
      const size_t li = (size_t)h_upoff[p] + (l - 1);
      for (uint64_t j = b; j < e; ++j) {
        aU[li * M + (j - b)] = ids[l][j];
        if (dists && dists[l]) aUd[li * M + (j - b)] = dists[l][j];
      }
    }
  }
  HB_CUDA(cudaMemcpy2DAsync(d_vec_.p, (size_t)row_bytes, vecs, (size_t)dim * es, (size_t)dim * es, n_new, cudaMemcpyHostToDevice, stream_));
  HB_CUDA(cudaMemcpyAsync(d_adj0_.p, a0.data(), a0.size() * 4, cudaMemcpyHostToDevice, stream_));
  HB_CUDA(cudaMemcpyAsync(d_adj0d_.p, a0d.data(), a0d.size() * 4, cudaMemcpyHostToDevice, stream_));
  if (n_ul) {
    HB_CUDA(cudaMemcpyAsync(d_adjU_.p, aU.data(), n_ul * M * 4, cudaMemcpyHostToDevice, stream_));
    HB_CUDA(cudaMemcpyAsync(d_adjUd_.p, aUd.data(), n_ul * M * 4, cudaMemcpyHostToDevice, stream_));
  }
  HB_CUDA(cudaMemcpyAsync(d_level_.p, h_level.data(), n_new, cudaMemcpyHostToDevice, stream_));
  HB_CUDA(cudaMemcpyAsync(d_plevel_.p, h_plevel.data(), n_new, cudaMemcpyHostToDevice, stream_));
  HB_CUDA(cudaMemcpyAsync(d_origin_.p, h_origin.data(), n_new * 8, cudaMemcpyHostToDevice, stream_));
  HB_CUDA(cudaMemcpyAsync(d_upoff_.p, h_upoff.data(), n_new * 4, cudaMemcpyHostToDevice, stream_));
  HB_CUDA(cudaStreamSynchronize(stream_));
  n = n_new;
  if (entry_id >= 0 && (size_t)entry_id < n_new) {
    entry = (uint32_t)entry_id;
    entry_level = levels[entry_id];
  }
  return 0;
}

// ------------------------------------------------------------------------------------------------
// search
int Index::acquire_ctx() {
  std::unique_lock<std::mutex> lk(ctx_mu_);
  for (;;) {
    for (int i = 0; i < NCTX; ++i)
      if (!ctx_[i].busy) {
        ctx_[i].busy = true;
        return i;
      }
    ctx_cv_.wait(lk);
  }
}
void Index::release_ctx(int c) {
  {
    std::lock_guard<std::mutex> lk(ctx_mu_);
    ctx_[c].busy = false;
  }
  ctx_cv_.notify_one();
}

// Device-resident search.  sync: runs on a leased context, returns when the answers are there.  Asynchronous: the launch
// is forked from the handle's stream (it waits for everything enqueued there so far) onto the next of two alternating
// context streams, so that two consecutive launches overlap.  The handle's stream does NOT wait for it: join() (or
// check_status, set_stream, any synchronous call's own synchronisation) makes it do so; stream_wait_last() makes any
// stream wait for the most recent launch alone.
int Index::search_device(const void* d_queries, size_t nq, size_t k, size_t ef_arg, const uint32_t* d_filter_bits,
                         NeighbourOut* d_out, int32_t* d_counts, bool sync, float* kernel_ms) {
  if (nq == 0) return 0;
  HB_CUDA(cudaSetDevice(device));
  if (sync) {
    CtxLease lease(this);
    SearchCtx& c = ctx_[lease.c];
    HB_CUDA(cudaEventRecord(c.fork, stream_));
    HB_CUDA(cudaStreamWaitEvent(c.stream, c.fork, 0));
    return search_on_ctx(c, d_queries, nq, k, ef_arg, d_filter_bits, d_out, d_counts, true, kernel_ms);
  }
  int ci;
  {
    std::lock_guard<std::mutex> lk(ctx_mu_);
    ci = NCTX + (int)(ctx_rr_++ % NASYNC);  // two contexts alternate: the tail of one launch overlaps the bulk of the next
  }
  SearchCtx& c = ctx_[ci];
  HB_CUDA(cudaEventRecord(c.fork, stream_));
  HB_CUDA(cudaStreamWaitEvent(c.stream, c.fork, 0));
  int r = search_on_ctx(c, d_queries, nq, k, ef_arg, d_filter_bits, d_out, d_counts, false, nullptr);
  if (r) return r;
  HB_CUDA(cudaEventRecord(c.join, c.stream));
  last_async_ = ci;
  return 0;
}

int Index::join() {
  HB_CUDA(cudaSetDevice(device));
  for (int i = NCTX; i < NCTX + NASYNC; ++i) {
    HB_CUDA(cudaEventRecord(ctx_[i].join, ctx_[i].stream));
    HB_CUDA(cudaStreamWaitEvent(stream_, ctx_[i].join, 0));
  }
  return 0;
}

int Index::stream_wait_last(cudaStream_t s) {
  HB_CUDA(cudaSetDevice(device));
  if (last_async_ >= 0) HB_CUDA(cudaStreamWaitEvent(s ? s : stream_, ctx_[last_async_].join, 0));
  return 0;
}

int Index::search_on_ctx(SearchCtx& c, const void* d_queries, size_t nq, size_t k, size_t ef_arg, const uint32_t* d_filter_bits,
                         NeighbourOut* d_out, int32_t* d_counts, bool sync, float* kernel_ms, const QueryFilter* d_qf,
                         const uint32_t* d_qpay) {
  if (k == 0) return fail("knbn must be positive");
  if (poisoned_) return fail(poison_msg_);
  cudaStream_t st = c.stream;
  if (dim == 0) {  // empty index: every answer is empty (hnsw.rs:1498-1503)
    HB_CUDA(cudaMemsetAsync(d_counts, 0, nq * sizeof(int32_t), st));
    if (sync) HB_CUDA(cudaStreamSynchronize(st));
    return 0;
  }
  SearchParams p;
  p.g = view();
  p.queries = d_queries;
  p.q_bytes = dim * es;
  p.q_stride_bytes = dim * es;
  p.nq = (uint32_t)nq;
  p.k = (int)k;
  p.ef = (int)std::max(ef_arg, k);  // hnsw.rs:1531
  int layer0 = 0;                   // hnsw.rs:1534-1540
  while (layer0 < MAX_LAYERS - 1 && layer_count[layer0] == 0) layer0++;
  if (n == 0) layer0 = 0;
  p.layer0 = layer0;
  p.work_counter = c.d_counter;
  p.out_nb = d_out;
  p.out_count = d_counts;
  p.filter_bits = d_filter_bits;
  p.qfilters = d_qf;
  p.qpayload = d_qpay;
  p.stats = stats_on_ ? d_stats_ : nullptr;
  p.status = c.d_status;
  const bool filtered = d_filter_bits != nullptr || d_qf != nullptr;
  // kernel choice: lean (search_lean.cuh) whenever it applies, else the generic warp kernel (search.cu / filter.cu)
  // tie mode "std" (search_std.cu): the reference's heaps replayed literally, unfiltered searches only
  const bool stdtie = tie_std_ && !filtered;
  const bool lean = !stdtie && !filtered && kernel_pref_ == 0 && entry != INVALID_ID && lean_eligible(p.g.d4, p.ef) && lean_op_supported(metric, dtype);
  p.q_kind = (filtered || lean || stdtie) ? 0 : queue_kind(p.ef, metric, dtype);
  p.q_smem = stdtie ? p.ef + 2 : (lean ? lean_queue_slots(p.ef) : queue_slots(p.q_kind, p.ef));
  size_t spw = stdtie ? (((size_t)p.g.d4 * 16 + (size_t)p.q_smem * 8 + 256 + 127) & ~(size_t)127)
                      : (lean ? lean_smem_per_warp(p.q_smem) : search_smem_per_warp(p.g.d4, p.q_smem));
  p.smem_per_warp = (int)spw;
  // warps per CTA: as many as the kernel is built for, fewer when one warp's share of shared memory is large (wide rows,
  // big ef); a single warp must fit
  int wpb = (lean ? LEAN_THREADS : SEARCH_THREADS) / 32;
  while (wpb > 1 && spw * wpb > 220 * 1024) wpb >>= 1;
  const size_t smem = spw * wpb;
  if (smem > 220 * 1024)
    return fail("ef / dimension too large: one query needs " + std::to_string(spw) + " bytes of shared memory (limit 220 KB)");
  p.threads = wpb * 32;
  p.cbuf = nullptr;
  p.ccap = 0;
  int bps = 0;
  {
    std::lock_guard<std::mutex> lk(occ_mu_);
    const auto key = std::make_tuple(stdtie ? 4 : (lean ? 3 : (d_qf ? 5 : (int)filtered)), (lean ? p.q_smem : p.q_kind) * 64 + wpb, p.g.d4, smem);
    auto it = occ_cache_.find(key);
    if (it != occ_cache_.end()) {
      bps = it->second;
    } else {
      if (stdtie) HB_CUDA(launch_search_std(p, metric, dtype, 0, smem, st, true, &bps));
      else if (lean) HB_CUDA(launch_search_lean(p, metric, dtype, 0, smem, st, true, &bps));
      else if (filtered) HB_CUDA(launch_search_filtered(p, metric, dtype, 0, smem, st, true, &bps));
      else HB_CUDA(launch_search(p, metric, dtype, 0, smem, st, true, &bps));
      occ_cache_[key] = bps;
    }
  }
  if (bps < 1) return fail("search kernel does not fit on an SM");
  const size_t per_cta = (size_t)wpb;
  int grid = (int)std::min<size_t>((size_t)sm_count_ * bps, (nq + per_cta - 1) / per_cta);
  const int deg = layer0 == 0 ? 2 * M : M;
  // visited-table capacity per query slot: a search inserts ~ (ef + a few) * (fresh neighbours per expansion) ids.  An
  // overflow is detected in the kernel and the batch re-run with doubled tables.  (The insert path has its own pool:
  // its tables are 4x larger, ef_construction instead of ef, and would push the search's out of L2.)
  size_t vcap = next_pow2(std::max<size_t>(1024, (size_t)2 * (p.ef + 16) * deg));
  VisitedPool& pool = filtered ? c.fvis : c.vis;
  for (int attempt = 0;; ++attempt) {
    int r;
    if (filtered) {
      // a filtered search keeps expanding until its candidate queue is empty (hnsw.rs:992-1001) and may visit the
      // whole graph: keep (visited table + candidate queue) under ~6 GB by running fewer warps when tables are big
      const size_t per_slot = std::max(vcap, pool.cap) * 12;
      const size_t max_slots = std::max<size_t>(wpb, ((size_t)6 << 30) / per_slot);
      grid = (int)std::max<size_t>(1, std::min<size_t>(grid, max_slots / wpb));
    }
    if ((r = ensure_visited(pool, (size_t)grid * per_cta, vcap, st))) return r;
    if ((r = fill_visited_cfg(pool, p.vis, st))) return r;
    if (filtered || stdtie) {  // candidate queue C: one region per warp slot
      if ((r = ensure_scratch(&c.d_cbuf, &c.d_cbuf_bytes, (size_t)grid * wpb * pool.cap * 8, st))) return r;
      p.cbuf = (uint64_t*)c.d_cbuf;
      p.ccap = (uint32_t)pool.cap;
    }
    HB_CUDA(cudaMemsetAsync(c.d_counter, 0, sizeof(unsigned int), st));
    HB_CUDA(cudaEventRecord(c.ev0, st));
    if (stdtie) HB_CUDA(launch_search_std(p, metric, dtype, grid, smem, st, false, nullptr));
    else if (lean) HB_CUDA(launch_search_lean(p, metric, dtype, grid, smem, st, false, nullptr));
    else if (filtered) HB_CUDA(launch_search_filtered(p, metric, dtype, grid, smem, st, false, nullptr));
    else HB_CUDA(launch_search(p, metric, dtype, grid, smem, st, false, nullptr));
    HB_CUDA(cudaEventRecord(c.ev1, st));
    if (!sync) break;
    int status = 0;
    HB_CUDA(cudaMemcpyAsync(&status, c.d_status, sizeof(int), cudaMemcpyDeviceToHost, st));
    HB_CUDA(cudaStreamSynchronize(st));
    if (status == 0) {
      if (kernel_ms) HB_CUDA(cudaEventElapsedTime(kernel_ms, c.ev0, c.ev1));
      break;
    }
    if (attempt >= 24) return fail("visited table overflow persists");
    HB_CUDA(cudaMemsetAsync(c.d_status, 0, sizeof(int), st));
    vcap = pool.cap * 2;
  }
  if (stats_on_) stat_queries_ += nq;
  return 0;
}

// pointer the device can dereference for a host buffer: pinned (page-locked) memory is mapped into the device's
// address space under unified addressing; pageable memory is not (nullptr)
static const void* device_view_of_host(const void* p) {
  cudaPointerAttributes at;
  if (cudaPointerGetAttributes(&at, p) != cudaSuccess) {
    cudaGetLastError();
    return nullptr;
  }
  if (at.type == cudaMemoryTypeHost || at.type == cudaMemoryTypeManaged) return at.devicePointer;
  return nullptr;
}

// Host queries in, host answers out.  ZERO-COPY when the memory allows it: a pinned query buffer is read by the
// kernel itself (each query crosses the bus once, 512 bytes when its warp picks it up, while thousands of other
// queries are being searched), and the answers are written by the kernel straight into the index's pinned result
// buffer: no cudaMemcpy before or after the launch, one synchronisation.  Pageable queries and row pointers are
// gathered into the index's own pinned staging buffer first (the only host-side copy), which the kernel then reads
// the same way.  zero_copy_ = false (env HNSW_B200_ZERO_COPY=0) restores explicit H2D / D2H copies.
int Index::search_host_begin(int ci, const void* queries, const void* const* rows, size_t nq, int d, size_t k, size_t ef,
                             const uint32_t* filter_bits_host, const QueryFilter* qdesc, const uint32_t* qpay) {
  SearchCtx& c = ctx_[ci];
  cudaStream_t st = c.stream;
  c.pend = SearchCtx::Pending();
  if (nq == 0) return 0;
  HB_CUDA(cudaSetDevice(device));
  if (dim != 0 && d != dim) return fail("query length differs from the index dimension");
  int r;
  const size_t out_bytes = nq * k * sizeof(NeighbourOut), cnt_bytes = nq * sizeof(int32_t);
  if (c.h_res_bytes < out_bytes + cnt_bytes + 16) {
    if (c.h_res) cudaFreeHost(c.h_res);
    c.h_res = nullptr;
    c.h_res_bytes = 0;
    HB_CUDA(cudaHostAlloc(&c.h_res, out_bytes + cnt_bytes + 16, cudaHostAllocMapped | cudaHostAllocPortable));
    c.h_res_bytes = out_bytes + cnt_bytes + 16;
  }
  NeighbourOut* hout = (NeighbourOut*)c.h_res;
  int32_t* hcnt = (int32_t*)((char*)c.h_res + out_bytes);
  int32_t* hstatus = hcnt + nq;
  c.pend.hout = hout;
  c.pend.hcnt = hcnt;
  c.pend.hstatus = hstatus;
  c.pend.nq = nq;
  c.pend.k = k;
  c.pend.ef = ef;
  c.pend.out_bytes = out_bytes;
  c.pend.cnt_bytes = cnt_bytes;
  if (dim == 0) {  // empty index: every answer is empty (hnsw.rs:1498-1500)
    for (size_t i = 0; i < nq; ++i) hcnt[i] = 0;
    for (size_t i = 0; i < nq * k; ++i) hout[i] = NeighbourOut{~0ull, __builtin_inff(), INVALID_ID};
    return 0;
  }
  const size_t qbytes = nq * (size_t)dim * es;
  const void* d_queries = nullptr;  // what the kernel reads
  const void* host_src = queries;
  if (rows || !(zero_copy_ && device_view_of_host(queries))) {
    // gather into pinned staging (rows: one pointer per query, libext.rs parallel_search_neighbours_<ty>)
    if (rows || !device_view_of_host(queries)) {
      if (c.h_pin_bytes < qbytes) {
        if (c.h_pin) cudaFreeHost(c.h_pin);
        c.h_pin = nullptr;
        c.h_pin_bytes = 0;
        HB_CUDA(cudaHostAlloc(&c.h_pin, qbytes, cudaHostAllocMapped | cudaHostAllocPortable));
        c.h_pin_bytes = qbytes;
      }
      unsigned char* st = (unsigned char*)c.h_pin;
      if (rows)
        for (size_t i = 0; i < nq; ++i) memcpy(st + i * (size_t)dim * es, rows[i], (size_t)dim * es);
      else
        memcpy(st, queries, qbytes);
      host_src = st;
    }
  }
  if (zero_copy_) d_queries = device_view_of_host(host_src);
  if (!d_queries) {
    if ((r = ensure_scratch(&c.d_q, &c.d_q_bytes, qbytes, st))) return r;
    HB_CUDA(cudaMemcpyAsync(c.d_q, host_src, qbytes, cudaMemcpyHostToDevice, st));
    d_queries = c.d_q;
  }
  NeighbourOut* k_out = nullptr;  // where the kernel writes
  int32_t* k_cnt = nullptr;
  const void* dv = zero_copy_ ? device_view_of_host(c.h_res) : nullptr;
  if (dv) {
    k_out = (NeighbourOut*)dv;
    k_cnt = (int32_t*)((char*)dv + out_bytes);
  } else {
    if ((r = ensure_scratch(&c.d_out, &c.d_out_bytes, out_bytes, st))) return r;
    if ((r = ensure_scratch(&c.d_cnt, &c.d_cnt_bytes, cnt_bytes, st))) return r;
    k_out = (NeighbourOut*)c.d_out;
    k_cnt = (int32_t*)c.d_cnt;
  }
  const uint32_t* dfb = nullptr;
  if (filter_bits_host) {
    const size_t fb = ((n + 31) / 32) * 4;
    if ((r = ensure_scratch(&c.d_fbits, &c.d_fbits_bytes, fb, st))) return r;
    HB_CUDA(cudaMemcpyAsync(c.d_fbits, filter_bits_host, fb, cudaMemcpyHostToDevice, st));
    dfb = (const uint32_t*)c.d_fbits;
  }
  const QueryFilter* dqf = nullptr;
  const uint32_t* dqpay = nullptr;
  if (qdesc) {  // per-query filters: this batch's descriptors, re-based, then the payload range they name
    const size_t words = (n + 31) / 32;
    size_t lo = SIZE_MAX, hi = 0;
    for (size_t i = 0; i < nq; ++i) {
      lo = std::min<size_t>(lo, qdesc[i].off);
      hi = std::max<size_t>(hi, (size_t)qdesc[i].off + (qdesc[i].form == QF_BITMAP ? words : qdesc[i].len));
    }
    std::vector<QueryFilter> rb(qdesc, qdesc + nq);
    for (QueryFilter& q : rb) q.off -= (uint32_t)lo;
    const size_t db = nq * sizeof(QueryFilter), pb = (hi - lo) * 4;
    if ((r = ensure_scratch(&c.d_qf, &c.d_qf_bytes, db + pb, st))) return r;
    // pageable sources: the calls return once the bytes are staged, so rb may go out of scope
    HB_CUDA(cudaMemcpyAsync(c.d_qf, rb.data(), db, cudaMemcpyHostToDevice, st));
    if (pb) HB_CUDA(cudaMemcpyAsync((char*)c.d_qf + db, qpay + lo, pb, cudaMemcpyHostToDevice, st));
    dqf = (const QueryFilter*)c.d_qf;
    dqpay = (const uint32_t*)((char*)c.d_qf + db);
  }
  // one enqueue (copies if any, kernel, status); search_host_finish synchronises once and takes the slow path (a visited
  // table overflowed: grow and re-run) only when the status says so
  c.pend.d_queries = d_queries;
  c.pend.dfb = dfb;
  c.pend.dqf = dqf;
  c.pend.dqpay = dqpay;
  c.pend.k_out = k_out;
  c.pend.k_cnt = k_cnt;
  c.pend.direct = dv != nullptr;
  c.pend.enqueued = true;
  if ((r = search_on_ctx(c, d_queries, nq, k, ef, dfb, k_out, k_cnt, false, nullptr, dqf, dqpay))) return r;
  if (!c.pend.direct) {
    HB_CUDA(cudaMemcpyAsync(hout, c.d_out, out_bytes, cudaMemcpyDeviceToHost, st));
    HB_CUDA(cudaMemcpyAsync(hcnt, c.d_cnt, cnt_bytes, cudaMemcpyDeviceToHost, st));
  }
  HB_CUDA(cudaMemcpyAsync(hstatus, c.d_status, sizeof(int32_t), cudaMemcpyDeviceToHost, st));
  return 0;
}

int Index::search_host_finish(int ci, const NeighbourOut** out, const int32_t** counts) {
  SearchCtx& c = ctx_[ci];
  cudaStream_t st = c.stream;
  SearchCtx::Pending& p = c.pend;
  *out = p.hout;
  *counts = p.hcnt;
  if (!p.enqueued) return 0;  // empty batch or empty index: the answers (if any) were filled by search_host_begin
  HB_CUDA(cudaSetDevice(device));
  HB_CUDA(cudaStreamSynchronize(st));
  if (*p.hstatus == 0) return 0;
  HB_CUDA(cudaMemsetAsync(c.d_status, 0, sizeof(int), st));
  int r;
  if ((r = search_on_ctx(c, p.d_queries, p.nq, p.k, p.ef, p.dfb, p.k_out, p.k_cnt, true, nullptr, p.dqf, p.dqpay)))
    return r;  // grows the tables
  if (!p.direct) {
    HB_CUDA(cudaMemcpyAsync(p.hout, c.d_out, p.out_bytes, cudaMemcpyDeviceToHost, st));
    HB_CUDA(cudaMemcpyAsync(p.hcnt, c.d_cnt, p.cnt_bytes, cudaMemcpyDeviceToHost, st));
    HB_CUDA(cudaStreamSynchronize(st));
  }
  return 0;
}

int Index::search_host_staged(int ci, const void* queries, const void* const* rows, size_t nq, int d, size_t k, size_t ef,
                              const uint32_t* filter_bits_host, const NeighbourOut** out, const int32_t** counts,
                              const QueryFilter* qdesc, const uint32_t* qpay) {
  *out = nullptr;
  *counts = nullptr;
  int r = search_host_begin(ci, queries, rows, nq, d, k, ef, filter_bits_host, qdesc, qpay);
  if (r) return r;
  return search_host_finish(ci, out, counts);
}

int Index::search_host(const void* queries, const void* const* rows, size_t nq, int d, size_t k, size_t ef,
                       const uint32_t* filter_bits_host, NeighbourOut* out, int32_t* counts) {
  CtxLease lease(this);
  const NeighbourOut* so;
  const int32_t* sc;
  int r = search_host_staged(lease.c, queries, rows, nq, d, k, ef, filter_bits_host, &so, &sc);
  if (r || nq == 0) return r;
  memcpy(counts, sc, nq * sizeof(int32_t));
  memcpy(out, so, nq * k * sizeof(NeighbourOut));
  return 0;
}

int Index::make_filter_bits(int mode, const uint64_t* sorted_ids, size_t nids, int (*fn)(uint64_t, void*), void* ctx,
                            std::vector<uint32_t>& bits) const {
  bits.assign((n + 31) / 32 + 1, 0u);
  for (size_t i = 0; i < n; ++i) {
    bool pass;
    if (mode == 2) {
      if (!fn) return fail("filter callback is NULL");
      pass = fn(h_origin[i], ctx) != 0;  // Fn(&DataId)->bool, filter.rs:17-24
    } else {
      pass = std::binary_search(sorted_ids, sorted_ids + nids, h_origin[i]);  // Vec<usize> filter, filter.rs:11-15
    }
    if (pass) bits[i >> 5] |= 1u << (i & 31);
  }
  return 0;
}

// Per-query filters.  Origin ids are translated through origin_table_, (origin, internal) sorted once per change of
// h_origin: a short list binary-searches it (resuming where the previous id was found), a long one walks it in step.
// Two passes over contiguous chunks of queries on host threads: the first counts each query's internal ids, which fixes
// its form and its place in the payload (so the size limit is checked exactly, before anything is allocated); the
// second translates again and writes the query's list or bitmap in place.
int Index::make_query_filters(size_t nq, const uint64_t* offsets, const uint64_t* ids, QueryFilterSet& out) const {
  {
    std::lock_guard<std::mutex> lk(origin_mu_);
    if (!origin_table_ok_) {
      origin_table_.resize(n);
      for (size_t i = 0; i < n; ++i) origin_table_[i] = {h_origin[i], (uint32_t)i};
      std::sort(origin_table_.begin(), origin_table_.end());
      origin_table_ok_ = true;
    }
  }
  // the table changes only under the index's exclusive lock, which no search holds: read it without origin_mu_
  const std::pair<uint64_t, uint32_t>* T = origin_table_.data();
  const size_t nt = origin_table_.size(), words = (n + 31) / 32;
  unsigned lg = 1;
  while (lg < 63 && ((size_t)1 << lg) < nt) ++lg;
  // calls range(lo, hi) for every run T[lo .. hi) of points whose origin id is in query q's list
  auto translate = [&](size_t q, auto&& range) {
    const uint64_t* a = ids + offsets[q];
    const size_t len = offsets[q + 1] - offsets[q];
    const bool walk = len * lg >= nt;
    size_t pos = 0;
    for (size_t j = 0; j < len; ++j) {
      if (j && a[j] == a[j - 1]) continue;
      size_t end;
      if (walk) {
        while (pos < nt && T[pos].first < a[j]) ++pos;
        for (end = pos; end < nt && T[end].first == a[j];) ++end;
      } else {
        pos = std::lower_bound(T + pos, T + nt, std::make_pair(a[j], (uint32_t)0)) - T;
        end = std::upper_bound(T + pos, T + nt, std::make_pair(a[j], UINT32_MAX)) - T;
      }
      if (end > pos) range(pos, end);
      pos = end;
    }
  };
  const size_t hw = std::max(1u, std::thread::hardware_concurrency());
  const size_t nth = std::max<size_t>(1, std::min<size_t>(std::min<size_t>(hw, 32), nq / 16));
  auto parallel = [&](const std::function<void(size_t, size_t)>& fn) {  // fn(first query, end) per chunk
    if (nth == 1) return fn(0, nq);
    std::vector<std::thread> th;
    for (size_t t = 0; t < nth; ++t) th.emplace_back(fn, nq * t / nth, nq * (t + 1) / nth);
    for (auto& x : th) x.join();
  };
  out.desc.assign(nq, QueryFilter{0, 0, QF_LIST, 0});
  parallel([&](size_t q0, size_t q1) {
    for (size_t q = q0; q < q1; ++q) {
      size_t c = 0;
      translate(q, [&](size_t lo, size_t hi) { c += hi - lo; });
      out.desc[q].len = (uint32_t)c;  // c <= n < 2^32
      out.desc[q].form = qf_use_bitmap(c, n) ? QF_BITMAP : QF_LIST;
    }
  });
  size_t total = 0;
  for (QueryFilter& d : out.desc) {
    if (total > UINT32_MAX) break;
    d.off = (uint32_t)total;
    total += d.form == QF_BITMAP ? words : d.len;
  }
  if (total > UINT32_MAX)
    return fail("per-query filters: the packed filters need more than 2^32 - 1 32-bit words");
  out.payload.assign(total, 0u);
  parallel([&](size_t q0, size_t q1) {
    for (size_t q = q0; q < q1; ++q) {
      uint32_t* dst = out.payload.data() + out.desc[q].off;
      if (out.desc[q].form == QF_BITMAP) {
        translate(q, [&](size_t lo, size_t hi) {
          for (size_t i = lo; i < hi; ++i) dst[T[i].second >> 5] |= 1u << (T[i].second & 31);
        });
      } else {
        size_t c = 0;
        translate(q, [&](size_t lo, size_t hi) {
          for (size_t i = lo; i < hi; ++i) dst[c++] = T[i].second;
        });
        std::sort(dst, dst + c);
      }
    }
  });
  return 0;
}

// ------------------------------------------------------------------------------------------------
// export
int Index::export_layer(int layer, uint64_t* offsets, uint32_t* ids, float* dists, int64_t* total) const {
  if (layer < 0 || layer >= MAX_LAYERS) return fail("bad layer");
  cudaSetDevice(device);
  const size_t deg0 = (size_t)2 * M;
  std::vector<uint32_t> a;
  std::vector<float> ad;
  if (layer == 0) {
    a.resize(n * deg0);
    ad.resize(n * deg0);
    if (n) {
      HB_CUDA(cudaMemcpy(a.data(), d_adj0_.p, a.size() * 4, cudaMemcpyDeviceToHost));
      HB_CUDA(cudaMemcpy(ad.data(), d_adj0d_.p, ad.size() * 4, cudaMemcpyDeviceToHost));
    }
  } else {
    a.resize(n_ul * M);
    ad.resize(n_ul * M);
    if (n_ul) {
      HB_CUDA(cudaMemcpy(a.data(), d_adjU_.p, a.size() * 4, cudaMemcpyDeviceToHost));
      HB_CUDA(cudaMemcpy(ad.data(), d_adjUd_.p, ad.size() * 4, cudaMemcpyDeviceToHost));
    }
  }
  uint64_t o = 0;
  for (size_t p = 0; p < n; ++p) {
    if (offsets) offsets[p] = o;
    const uint32_t* l = nullptr;
    const float* ld = nullptr;
    size_t cap = 0;
    if (layer == 0) {
      l = a.data() + p * deg0;
      ld = ad.data() + p * deg0;
      cap = deg0;
    } else if (layer <= h_plevel[p]) {
      const size_t li = (size_t)h_upoff[p] + (layer - 1);
      l = a.data() + li * M;
      ld = ad.data() + li * M;
      cap = M;
    }
    for (size_t j = 0; j < cap && l[j] != INVALID_ID; ++j) {
      if (ids) ids[o] = l[j];
      if (dists) dists[o] = ld[j];
      ++o;
    }
  }
  if (offsets) offsets[n] = o;
  if (total) *total = (int64_t)o;
  return 0;
}

int Index::flatten(std::vector<uint64_t>& offsets, std::vector<uint64_t>& nb_origin, std::vector<float>& nb_dist) const {
  std::vector<std::vector<std::pair<float, uint32_t>>> per(n);
  int top = 0;
  for (size_t p = 0; p < n; ++p) top = std::max<int>(top, h_plevel[p]);
  for (int l = 0; l <= top && l < MAX_LAYERS; ++l) {
    int64_t total = 0;
    int r;
    if ((r = export_layer(l, nullptr, nullptr, nullptr, &total))) return r;
    std::vector<uint64_t> off(n + 1);
    std::vector<uint32_t> ids((size_t)total);
    std::vector<float> ds((size_t)total);
    if ((r = export_layer(l, off.data(), ids.data(), ds.data(), nullptr))) return r;
    for (size_t p = 0; p < n; ++p)
      for (uint64_t j = off[p]; j < off[p + 1]; ++j) per[p].emplace_back(ds[j], ids[j]);
  }
  offsets.assign(n + 1, 0);
  nb_origin.clear();
  nb_dist.clear();
  for (size_t p = 0; p < n; ++p) {
    std::sort(per[p].begin(), per[p].end());  // flatten.rs:82 sort_unstable by distance (ties: by internal id here)
    offsets[p] = nb_origin.size();
    for (auto& e : per[p]) {
      nb_origin.push_back(h_origin[e.second]);
      nb_dist.push_back(e.first);
    }
  }
  offsets[n] = nb_origin.size();
  return 0;
}

int Index::export_vectors(void* out) const {
  if (n == 0) return 0;
  cudaSetDevice(device);
  HB_CUDA(cudaMemcpy2D(out, (size_t)dim * es, d_vec_.p, (size_t)row_bytes, (size_t)dim * es, n, cudaMemcpyDeviceToHost));
  return 0;
}

int Index::set_stream(cudaStream_t s) {
  HB_CUDA(cudaSetDevice(device));
  for (SearchCtx& c : ctx_) HB_CUDA(cudaStreamSynchronize(c.stream));
  HB_CUDA(cudaStreamSynchronize(stream_));
  stream_ = s ? s : own_stream_;
  return 0;
}

int Index::check_status() {
  HB_CUDA(cudaSetDevice(device));
  HB_CUDA(cudaStreamSynchronize(stream_));
  int any = 0;
  for (SearchCtx& c : ctx_) {
    int status = 0;
    HB_CUDA(cudaMemcpyAsync(&status, c.d_status, sizeof(int), cudaMemcpyDeviceToHost, c.stream));
    HB_CUDA(cudaStreamSynchronize(c.stream));
    if (status) HB_CUDA(cudaMemset(c.d_status, 0, sizeof(int)));
    any |= status;
  }
  return any ? 1 : 0;
}

int Index::enable_stats(bool on) {
  stats_on_ = on;
  return 0;
}

int Index::get_stats(uint64_t* out4, bool reset) {
  cudaSetDevice(device);
  unsigned long long h[4];
  HB_CUDA(cudaStreamSynchronize(stream_));
  HB_CUDA(cudaMemcpy(h, d_stats_, sizeof(h), cudaMemcpyDeviceToHost));
  out4[0] = h[0];
  out4[1] = h[1];
  out4[2] = h[2];
  out4[3] = stat_queries_;
  if (reset) {
    HB_CUDA(cudaMemset(d_stats_, 0, sizeof(h)));
    stat_queries_ = 0;
  }
  return 0;
}

// ------------------------------------------------------------------------------------------------
// replication blobs: 0 vec, 1 adj0, 2 adjU, 3 up_off, 4 plevel, 5 level, 6 origin, 7 adj0_d, 8 adjU_d
static const uint64_t BLOB_MAGIC = 0x68623230306e7377ull;

int Index::blob_header(uint64_t* h) const {
  for (int i = 0; i < 16; ++i) h[i] = 0;
  h[0] = BLOB_MAGIC;
  h[1] = n;
  h[2] = (uint64_t)dim;
  h[3] = (uint64_t)M;
  h[4] = (uint64_t)max_layer;
  h[5] = (uint64_t)ef_c;
  h[6] = (uint64_t)metric;
  h[7] = n_ul;
  h[8] = entry;
  h[9] = (uint64_t)(int64_t)entry_level;
  h[10] = 1;  // distances included
  h[11] = (uint64_t)dtype;
  return 0;
}

int Index::blob_alloc(const uint64_t* h) {
  if (h[0] != BLOB_MAGIC) return fail("bad replication header");
  if (n != 0) return fail("blob_alloc needs an empty index");
  if ((int)h[3] != M || (int)h[6] != metric || (int)h[11] != dtype)
    return fail("replication header does not match this handle's M / metric / element type");
  HB_CUDA(cudaSetDevice(device));
  int r;
  if ((r = set_dim((int)h[2]))) return r;
  if ((r = ensure_points((size_t)h[1]))) return r;
  if ((r = ensure_upper((size_t)h[7] + 2 * MAX_LAYERS))) return r;
  n = (size_t)h[1];
  n_ul = (size_t)h[7];
  entry = (uint32_t)h[8];
  entry_level = (int)(int64_t)h[9];
  max_layer = (int)h[4];
  ef_c = (int)h[5];
  return 0;
}

int Index::blob_info(int i, void** p, uint64_t* bytes) const {
  const size_t deg0 = (size_t)2 * M;
  switch (i) {
    case 0: *p = d_vec_.p; *bytes = n * (size_t)row_bytes; return 0;
    case 1: *p = d_adj0_.p; *bytes = n * deg0 * 4; return 0;
    case 2: *p = d_adjU_.p; *bytes = n_ul * M * 4; return 0;
    case 3: *p = d_upoff_.p; *bytes = n * 4; return 0;
    case 4: *p = d_plevel_.p; *bytes = n; return 0;
    case 5: *p = d_level_.p; *bytes = n; return 0;
    case 6: *p = d_origin_.p; *bytes = n * 8; return 0;
    case 7: *p = d_adj0d_.p; *bytes = n * deg0 * 4; return 0;
    case 8: *p = d_adjUd_.p; *bytes = n_ul * M * 4; return 0;
  }
  return fail("bad blob index");
}

int Index::blob_commit() {
  cudaSetDevice(device);
  invalidate_origin_table();
  h_level.resize(n);
  h_plevel.resize(n);
  h_origin.resize(n);
  h_upoff.resize(n);
  h_rank.resize(n);
  if (n) {
    HB_CUDA(cudaMemcpy(h_level.data(), d_level_.p, n, cudaMemcpyDeviceToHost));
    HB_CUDA(cudaMemcpy(h_plevel.data(), d_plevel_.p, n, cudaMemcpyDeviceToHost));
    HB_CUDA(cudaMemcpy(h_origin.data(), d_origin_.p, n * 8, cudaMemcpyDeviceToHost));
    HB_CUDA(cudaMemcpy(h_upoff.data(), d_upoff_.p, n * 4, cudaMemcpyDeviceToHost));
  }
  for (int l = 0; l < MAX_LAYERS; ++l) layer_count[l] = 0;
  for (size_t p = 0; p < n; ++p) h_rank[p] = (int32_t)layer_count[h_level[p]]++;
  return 0;
}

}  // namespace hb
