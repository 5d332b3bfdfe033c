// extern "C" surface of libhnsw_b200.so: the reference's libext.rs symbols (f32) + extensions.
// Declarations and the reference file:line each one replaces are in include/hnsw_b200.h.
#include <cstdlib>
#include <exception>
#include <cstring>
#include <mutex>
#include <shared_mutex>
#include <string>
#include <vector>

#include "../../include/hnsw_b200.h"
#include "index.h"

using hb::Index;
using hb::NeighbourOut;

// every typed handle of libext.rs (HnswApif32, HnswApii32, HnswApiu32, HnswApiu16, HnswApiu8) has this layout
struct HnswApif32 { Index* ix; };
struct HnswApii32 { Index* ix; };
struct HnswApiu32 { Index* ix; };
struct HnswApiu16 { Index* ix; };
struct HnswApiu8 { Index* ix; };
struct AnyApi { Index* ix; };

static thread_local std::string g_err;
static int g_device = 0;

static_assert(sizeof(Neighbour_api) == 16, "Neighbour_api must match #[repr(C)] {usize, f32}");
static_assert(sizeof(NeighbourOut) == sizeof(Neighbour_api), "device answer slot must alias Neighbour_api");
static_assert(sizeof(Neighbourhood_api) == 16 && sizeof(Vec_api_Neighbourhood_api) == 16, "libext.rs struct layouts");

static int set_err(const std::string& m) {
  g_err = m;
  return -1;
}
static int pass(Index* ix, int r) {
  if (r) g_err = ix->err();
  return r;
}

// HB_H: exclusive access (anything that may change the index); HB_HS: shared access (searches, read-only queries)
#define HB_H(h) \
  if (!(h)) return set_err("NULL handle"); \
  Index* ix = ((const AnyApi*)(h))->ix;    \
  std::unique_lock<std::shared_mutex> g__(ix->mu); \
  ix->drain_pending()
#define HB_HS(h) \
  if (!(h)) return set_err("NULL handle"); \
  Index* ix = ((const AnyApi*)(h))->ix;    \
  std::shared_lock<std::shared_mutex> g__(ix->mu)

static int metric_from_name(const uint8_t* name, size_t len) {
  std::string s((const char*)name, len);
  if (s == "DistL1") return hb::METRIC_L1;
  if (s == "DistL2") return hb::METRIC_L2;
  if (s == "DistDot") return hb::METRIC_DOT;
  if (s == "DistCosine") return hb::METRIC_COSINE;
  if (s == "DistHellinger") return hb::METRIC_HELLINGER;
  if (s == "DistJeffreys") return hb::METRIC_JEFFREYS;
  if (s == "DistJensenShannon") return hb::METRIC_JENSENSHANNON;
  if (s == "DistHamming") return hb::METRIC_HAMMING;
  if (s == "DistJaccard") return hb::METRIC_JACCARD;
  return -1;
}

static void* make_index(int dtype, size_t max_nb_conn, size_t ef_const, size_t namelen, const uint8_t* cdistname,
                        size_t max_elements, size_t max_layer) {
  if (!cdistname) {
    set_err("distance name is NULL");
    return nullptr;
  }
  const int metric = metric_from_name(cdistname, namelen);
  if (metric < 0 || !hb::metric_supported(metric, dtype)) {  // libext.rs:520-523: unknown distance => null
    set_err("unknown / unsupported distance name '" + std::string((const char*)cdistname, namelen) + "' for this element type");
    return nullptr;
  }
  if (max_nb_conn < 2 || max_nb_conn > 256) {  // hnsw.rs:784-787 caps at 256; ln(1) = 0 breaks the level law
    set_err("max_nb_connection must be in [2, 256]");
    return nullptr;
  }
  if (ef_const == 0 || max_layer == 0) {
    set_err("ef_construction and max_layer must be positive");
    return nullptr;
  }
  Index* ix = new Index((int)max_nb_conn, max_elements, (int)max_layer, (int)ef_const, metric, dtype, g_device);
  if (!ix->ok()) {
    set_err(ix->err());
    delete ix;
    return nullptr;
  }
  return new AnyApi{ix};
}

// ---- generic bodies of the reference entry points (element type = the handle's)
static void insert_any(void* hv, size_t len, const void* data, size_t id) {
  AnyApi* h = (AnyApi*)hv;
  if (!h || !data) {
    set_err("insert: NULL argument");
    return;
  }
  std::unique_lock<std::shared_mutex> g(h->ix->mu);
  h->ix->drain_pending();
  if (pass(h->ix, h->ix->set_dim((int)len))) return;
  uint64_t id64 = id;
  pass(h->ix, h->ix->insert_batch(data, 1, len, nullptr, &id64, nullptr));
}

static void parallel_insert_any(void* hv, size_t nb_vec, size_t vec_len, const void* const* datas, const size_t* ids) {
  AnyApi* h = (AnyApi*)hv;
  if (!h || !datas || !ids) {
    set_err("parallel_insert: NULL argument");
    return;
  }
  std::unique_lock<std::shared_mutex> g(h->ix->mu);
  h->ix->drain_pending();
  if (pass(h->ix, h->ix->set_dim((int)vec_len))) return;
  std::vector<uint64_t> id64(ids, ids + nb_vec);
  pass(h->ix, h->ix->insert_batch(nullptr, nb_vec, vec_len, datas, id64.data(), nullptr));
}

static const Neighbourhood_api* search_any(const void* hv, size_t len, const void* data, size_t knbn, size_t ef_search) {
  const AnyApi* h = (const AnyApi*)hv;
  if (!h || !data || knbn == 0) {
    set_err("search_neighbours: bad argument");
    return nullptr;
  }
  std::shared_lock<std::shared_mutex> g(h->ix->mu);
  Neighbour_api* nb = (Neighbour_api*)malloc(sizeof(Neighbour_api) * knbn);
  int32_t cnt = 0;
  if (pass(h->ix, h->ix->search_host(data, nullptr, 1, (int)len, knbn, ef_search, nullptr, (NeighbourOut*)nb, &cnt))) {
    free(nb);
    return nullptr;
  }
  Neighbourhood_api* out = (Neighbourhood_api*)malloc(sizeof(Neighbourhood_api));
  out->nbgh = cnt;
  out->neighbours = nb;
  return out;
}

// a batch is split over the replicas when there are any and every device gets a worthwhile share
static bool use_shards(const Index* ix, size_t nq) { return ix->replica_count() > 0 && nq >= 64 * (ix->replica_count() + 1); }

struct VecApiBox {
  Vec_api_Neighbourhood_api v;  // first member: the pointer handed to the caller
  Neighbourhood_api* hoods;
  Neighbour_api* block;
};

static const Vec_api_Neighbourhood_api* parallel_search_any(const void* hv, size_t nb_vec, int64_t vec_len,
                                                            const void* const* data, size_t knbn, size_t ef_search) {
  const AnyApi* h = (const AnyApi*)hv;
  if (!h || (!data && nb_vec) || knbn == 0) {
    set_err("parallel_search_neighbours: bad argument");
    return nullptr;
  }
  std::shared_lock<std::shared_mutex> g(h->ix->mu);
  VecApiBox* box = (VecApiBox*)malloc(sizeof(VecApiBox));
  box->hoods = (Neighbourhood_api*)malloc(sizeof(Neighbourhood_api) * (nb_vec ? nb_vec : 1));
  box->block = (Neighbour_api*)malloc(sizeof(Neighbour_api) * (nb_vec ? nb_vec * knbn : 1));
  std::vector<int32_t> cnt(nb_vec);
  int rc;
  if (use_shards(h->ix, nb_vec)) {  // replicas on other GPUs: every device answers its slice of the batch in place
    NeighbourOut* block = (NeighbourOut*)box->block;
    int32_t* cp = cnt.data();
    rc = h->ix->for_each_shard(nb_vec, [=](Index* rx, size_t first, size_t count) {
      return rx->search_host(nullptr, data + first, count, (int)vec_len, knbn, ef_search, nullptr, block + first * knbn, cp + first);
    });
  } else {
    rc = h->ix->search_host(nullptr, data, nb_vec, (int)vec_len, knbn, ef_search, nullptr, (NeighbourOut*)box->block, cnt.data());
  }
  if (pass(h->ix, rc)) {
    free(box->hoods);
    free(box->block);
    free(box);
    return nullptr;
  }
  for (size_t i = 0; i < nb_vec; ++i) {  // input order, hnsw.rs:1622-1633
    box->hoods[i].nbgh = cnt[i];
    box->hoods[i].neighbours = box->block + i * knbn;
  }
  box->v.len = (int64_t)nb_vec;
  box->v.ptr = box->hoods;
  return &box->v;
}

static void drop_any(const void* p) {
  const AnyApi* h = (const AnyApi*)p;
  if (!h) return;
  delete h->ix;
  delete h;
}

static int64_t file_dump_any(const void* hv, size_t namelen, const uint8_t* filename);

extern "C" {

// libext.rs generates one set of entry points per element type with macros (generate_insert!, ... :106-275,
// instantiated :770-771, 829-835, 898-904, 1044-1048, 1112-1116); so do we.
#define HB_TYPED_API(SUF, CT, DT)                                                                                      \
  const HnswApi##SUF* init_hnsw_##SUF(size_t max_nb_conn, size_t ef_const, size_t namelen, const uint8_t* cdistname) { \
    return (const HnswApi##SUF*)make_index(DT, max_nb_conn, ef_const, namelen, cdistname, 10000, 16);                   \
  }                                                                                                                    \
  const HnswApi##SUF* init_hnsw_ptrdist_##SUF(size_t, size_t, float (*)(const CT*, const CT*, unsigned long long)) {   \
    set_err("init_hnsw_ptrdist: a host distance callback cannot run inside a CUDA kernel; use a named distance");      \
    return nullptr;                                                                                                    \
  }                                                                                                                    \
  void insert_##SUF(HnswApi##SUF* h, size_t len, const CT* data, size_t id) { insert_any(h, len, data, id); }          \
  void parallel_insert_##SUF(HnswApi##SUF* h, size_t nb_vec, size_t vec_len, const CT** datas, const size_t* ids) {    \
    parallel_insert_any(h, nb_vec, vec_len, (const void* const*)datas, ids);                                           \
  }                                                                                                                    \
  const Neighbourhood_api* search_neighbours_##SUF(const HnswApi##SUF* h, size_t len, const CT* data, size_t knbn,     \
                                                   size_t ef_search) {                                                 \
    return search_any(h, len, data, knbn, ef_search);                                                                  \
  }                                                                                                                    \
  const Vec_api_Neighbourhood_api* parallel_search_neighbours_##SUF(const HnswApi##SUF* h, size_t nb_vec,              \
                                                                    int64_t vec_len, const CT** data, size_t knbn,     \
                                                                    size_t ef_search) {                                \
    return parallel_search_any(h, nb_vec, vec_len, (const void* const*)data, knbn, ef_search);                         \
  }                                                                                                                    \
  int64_t file_dump_##SUF(const HnswApi##SUF* h, size_t namelen, const uint8_t* filename) {                            \
    return file_dump_any(h, namelen, filename);                                                                        \
  }

HB_TYPED_API(f32, float, hb::DT_F32)
HB_TYPED_API(i32, int32_t, hb::DT_I32)
HB_TYPED_API(u32, uint32_t, hb::DT_U32)
HB_TYPED_API(u16, uint16_t, hb::DT_U16)
HB_TYPED_API(u8, uint8_t, hb::DT_U8)
#undef HB_TYPED_API

const HnswApif32* new_hnsw_f32(size_t max_nb_conn, size_t ef_const, size_t namelen, const uint8_t* cdistname,
                               size_t max_elements, size_t max_layer) {
  return (const HnswApif32*)make_index(hb::DT_F32, max_nb_conn, ef_const, namelen, cdistname, max_elements, max_layer);
}
const HnswApiu16* new_hnsw_u16(size_t max_nb_conn, size_t ef_const, size_t namelen, const uint8_t* cdistname,
                               size_t max_elements, size_t max_layer) {  // libext.rs:964-1028
  return (const HnswApiu16*)make_index(hb::DT_U16, max_nb_conn, ef_const, namelen, cdistname, max_elements, max_layer);
}
void drop_hnsw_f32(const HnswApif32* p) { drop_any(p); }  // libext.rs:626-630
void drop_hnsw_u16(const HnswApiu16* p) { drop_any(p); }  // libext.rs:636-640
void hnsw_b200_drop(const void* p) { drop_any(p); }       // upstream exports no drop for i32/u32/u8
// typed constructor with max_elements / max_layer for every element type (upstream has it for f32 and u16 only)
void* hnsw_b200_new(int dtype, size_t max_nb_conn, size_t ef_const, size_t namelen, const uint8_t* cdistname,
                    size_t max_elements, size_t max_layer) {
  if (dtype < 0 || dtype > 4) {
    set_err("dtype must be 0 f32, 1 u8, 2 u16, 3 u32, 4 i32");
    return nullptr;
  }
  return make_index(dtype, max_nb_conn, ef_const, namelen, cdistname, max_elements, max_layer);
}

}  // extern "C"

// generate_file_dump!, libext.rs:257-275: dump into "." with the given basename; 1 on success, -1 on failure
static int64_t file_dump_any(const void* hv, size_t namelen, const uint8_t* filename) {
  const AnyApi* h = (const AnyApi*)hv;
  if (!h || !filename) {
    set_err("file_dump: NULL argument");
    return -1;
  }
  std::shared_lock<std::shared_mutex> g(h->ix->mu);
  std::string used;
  // api.rs:76-78: the reference refuses to overwrite only while a dump is memory-mapped; nothing is mapped here
  if (pass(h->ix, h->ix->file_dump(".", std::string((const char*)filename, namelen), true, &used))) return -1;
  return 1;
}

// HnswIo (hnswio.rs:300-380) reduced to what the C ABI needs: directory + basename
struct HnswIo {
  std::string dir, basename;
};

static void* load_any_unguarded(HnswIo* io, int dtype, int metric);
// nothing may unwind through the C boundary: a dump that makes an allocation fail returns NULL like the reference does
static void* load_any(HnswIo* io, int dtype, int metric) {
  try {
    return load_any_unguarded(io, dtype, metric);
  } catch (const std::exception& e) {
    set_err(std::string("load_hnswdump: ") + e.what());
    return nullptr;
  }
}
static void* load_any_unguarded(HnswIo* io, int dtype, int metric) {
  if (!io) {
    set_err("load_hnswdump: NULL HnswIo");
    return nullptr;
  }
  hb::DumpDescription de;
  std::string e;
  if (hb::read_description(io->dir + "/" + io->basename + ".hnsw.graph", de, e)) {
    set_err(e);
    return nullptr;
  }
  const int M = de.max_nb_connection == 0 ? 256 : de.max_nb_connection;
  Index* ix = new Index(M, (size_t)de.nb_point, 16, (int)de.ef, metric, dtype, g_device);
  if (!ix->ok() || ix->load_dump(io->dir, io->basename)) {
    set_err(ix->err());
    delete ix;
    return nullptr;  // libext.rs:297-300: failed reload => null
  }
  return new AnyApi{ix};
}

extern "C" {

// get_hnswio, libext.rs:27-33: dump basename, files looked up in the current directory
HnswIo* get_hnswio(uint64_t flen, const uint8_t* name) {
  if (!name) return nullptr;
  return new HnswIo{".", std::string((const char*)name, (size_t)flen)};
}
HnswIo* hnsw_b200_get_hnswio(const char* dir, const char* basename) {
  if (!dir || !basename) return nullptr;
  return new HnswIo{dir, basename};
}
void hnsw_b200_free_hnswio(HnswIo* io) { delete io; }

// generate_loadhnsw!, libext.rs:280-451: one loader per (element type, distance) pair upstream instantiates
#define HB_LOADER(SUF, DIST, DT, METRIC)                                             \
  const HnswApi##SUF* load_hnswdump_##SUF##_##DIST(HnswIo* io) {                     \
    return (const HnswApi##SUF*)load_any(io, DT, METRIC);                            \
  }
HB_LOADER(f32, DistL1, hb::DT_F32, hb::METRIC_L1)
HB_LOADER(f32, DistL2, hb::DT_F32, hb::METRIC_L2)
HB_LOADER(f32, DistCosine, hb::DT_F32, hb::METRIC_COSINE)
HB_LOADER(f32, DistDot, hb::DT_F32, hb::METRIC_DOT)
HB_LOADER(f32, DistJensenShannon, hb::DT_F32, hb::METRIC_JENSENSHANNON)
HB_LOADER(f32, DistJeffreys, hb::DT_F32, hb::METRIC_JEFFREYS)
HB_LOADER(i32, DistL1, hb::DT_I32, hb::METRIC_L1)
HB_LOADER(i32, DistL2, hb::DT_I32, hb::METRIC_L2)
HB_LOADER(i32, DistHamming, hb::DT_I32, hb::METRIC_HAMMING)
HB_LOADER(u32, DistL1, hb::DT_U32, hb::METRIC_L1)
HB_LOADER(u32, DistL2, hb::DT_U32, hb::METRIC_L2)
HB_LOADER(u32, DistHamming, hb::DT_U32, hb::METRIC_HAMMING)
HB_LOADER(u32, DistJaccard, hb::DT_U32, hb::METRIC_JACCARD)
HB_LOADER(u16, DistL1, hb::DT_U16, hb::METRIC_L1)
HB_LOADER(u16, DistL2, hb::DT_U16, hb::METRIC_L2)
HB_LOADER(u16, DistHamming, hb::DT_U16, hb::METRIC_HAMMING)
HB_LOADER(u8, DistL1, hb::DT_U8, hb::METRIC_L1)
HB_LOADER(u8, DistL2, hb::DT_U8, hb::METRIC_L2)
HB_LOADER(u8, DistHamming, hb::DT_U8, hb::METRIC_HAMMING)
HB_LOADER(u8, DistJaccard, hb::DT_U8, hb::METRIC_JACCARD)
#undef HB_LOADER

// load any (element type, distance) by name: dtype 0 f32, 1 u8, 2 u16, 3 u32, 4 i32
void* hnsw_b200_load_dump(HnswIo* io, int dtype, size_t namelen, const uint8_t* cdistname) {
  if (!cdistname) return nullptr;
  const int metric = metric_from_name(cdistname, namelen);
  if (metric < 0 || !hb::metric_supported(metric, dtype)) {
    set_err("unknown / unsupported distance name for this element type");
    return nullptr;
  }
  return load_any(io, dtype, metric);
}

int hnsw_b200_file_dump(const void* h, const char* dir, const char* basename, int overwrite, char* used_basename,
                        size_t used_cap) {
  HB_H(h);
  if (!dir || !basename) return set_err("NULL path");
  std::string used;
  int r = pass(ix, ix->file_dump(dir, basename, overwrite != 0, &used));
  if (r) return r;
  if (used_basename && used_cap) {
    strncpy(used_basename, used.c_str(), used_cap - 1);
    used_basename[used_cap - 1] = 0;
  }
  return 0;
}

// load_hnsw_description, libext.rs:1170-1232.  `name` = path of the .hnsw.graph file.  Release with
// hnsw_b200_free_description (upstream leaks it).
const DescriptionFFI* load_hnsw_description(size_t flen, const uint8_t* name) {
  if (!name) return nullptr;
  hb::DumpDescription de;
  std::string e;
  if (hb::read_description(std::string((const char*)name, flen), de, e)) {
    set_err(e);
    return nullptr;
  }
  DescriptionFFI* d = (DescriptionFFI*)calloc(1, sizeof(DescriptionFFI));
  d->dumpmode = 1;  // upstream hard-codes 1 here ("CAVEAT", libext.rs:1196)
  d->max_nb_connection = de.max_nb_connection;
  d->nb_layer = de.nb_layer;
  d->ef = (size_t)de.ef;
  d->nb_point = (size_t)de.nb_point;  // upstream leaves this field at 0; filled here
  d->data_dimension = (size_t)de.dimension;
  char* dn = (char*)malloc(de.distname.size() + 1);
  memcpy(dn, de.distname.c_str(), de.distname.size() + 1);
  char* tn = (char*)malloc(de.t_name.size() + 1);
  memcpy(tn, de.t_name.c_str(), de.t_name.size() + 1);
  d->distname_len = de.distname.size();
  d->distname = (const uint8_t*)dn;
  d->t_name_len = de.t_name.size();
  d->t_name = (const uint8_t*)tn;
  return d;
}
void hnsw_b200_free_description(const DescriptionFFI* d) {
  if (!d) return;
  free((void*)d->distname);
  free((void*)d->t_name);
  free((void*)d);
}

void init_rust_log(void) {}

// ------------------------------------------------------------------ extensions
const char* hnsw_b200_last_error(void) { return g_err.c_str(); }

int hnsw_b200_device_count(void) {
  int n = 0;
  if (cudaGetDeviceCount(&n) != cudaSuccess) return 0;
  return n;
}

int hnsw_b200_set_device(int device) {
  int n = hnsw_b200_device_count();
  if (device < 0 || device >= n) return set_err("device index out of range");
  g_device = device;
  return 0;
}

void hnsw_b200_free_neighbourhood(const Neighbourhood_api* p) {
  if (!p) return;
  free((void*)p->neighbours);
  free((void*)p);
}

void hnsw_b200_free_vec_api(const Vec_api_Neighbourhood_api* p) {
  if (!p) return;
  VecApiBox* box = (VecApiBox*)p;
  free(box->hoods);
  free(box->block);
  free(box);
}


int hnsw_b200_set_extend_candidates(void* h, int flag) {
  HB_H(h);
  if (flag && ix->ef_c <= 2 * ix->M)
    return set_err("extend_candidates needs ef_construction > 2*max_nb_connection in this engine (otherwise the "
                   "extension set of hnsw.rs:1336-1362 is not provably empty)");
  ix->extend_candidates = flag != 0;
  return 0;
}
int hnsw_b200_get_extend_candidates(const void* h) {
  if (!h) return set_err("NULL handle");
  return ((const AnyApi*)h)->ix->extend_candidates ? 1 : 0;
}
int hnsw_b200_set_keeping_pruned(void* h, int flag) {
  HB_H(h);
  ix->keep_pruned = flag != 0;
  return 0;
}
int hnsw_b200_modify_level_scale(void* h, double scale) {
  HB_H(h);
  if (ix->n > 0) return set_err("modify_level_scale: index already holds points (hnsw.rs:881-888)");
  if (!(scale >= 0.2 && scale <= 1.0)) return set_err("modify_level_scale: factor must be in [0.2, 1]");  // hnsw.rs:889-900
  ix->level_scale = scale / std::log((double)ix->M);
  return 0;
}
int hnsw_b200_set_tie_mode(void* h, int mode) {
  HB_H(h);
  if (mode != 0 && mode != 1) return set_err("tie mode must be 0 (distance, id) or 1 (reference std heaps)");
  ix->tie_std_ = mode == 1;
  return 0;
}
int hnsw_b200_set_searching_mode(void* h, int flag) {
  HB_H(h);
  ix->searching = flag != 0;
  return 0;
}
int hnsw_b200_set_level_seed(void* h, uint64_t seed) {
  HB_H(h);
  ix->rng.s = seed;
  return 0;
}
uint64_t hnsw_b200_get_nb_point(const void* h) { return h ? ((const AnyApi*)h)->ix->n : 0; }
int hnsw_b200_get_max_level_observed(const void* h) { return h ? std::max(((const AnyApi*)h)->ix->entry_level, 0) : 0; }
int hnsw_b200_get_dim(const void* h) { return h ? ((const AnyApi*)h)->ix->dim : 0; }
int hnsw_b200_set_insert_batching(void* h, uint32_t ratio, uint32_t max_batch) {
  HB_H(h);
  if (ratio == 0 || max_batch == 0) return set_err("ratio and max_batch must be positive");
  ix->batch_ratio = ratio;
  ix->batch_max = max_batch;
  return 0;
}

int hnsw_b200_insert_flat(void* h, const void* vecs, uint64_t n, uint64_t dim, const uint64_t* ids,
                          const int32_t* levels) {
  HB_H(h);
  if (n == 0) return 0;
  if (!vecs) return set_err("vecs is NULL");
  int r;
  if ((r = pass(ix, ix->set_dim((int)dim)))) return r;
  return pass(ix, ix->insert_batch(vecs, n, dim, nullptr, ids, levels));
}

// one device's answers for queries [first, first + count) into the caller's arrays.  The kernel fills the slots beyond a
// query's count with (~0, +inf, INVALID_ID): plain field copies
static void unpack_answers(const Index* rx, const NeighbourOut* tmp, const int32_t* cnts, size_t first, size_t count,
                           uint64_t knbn, uint64_t* out_ids, float* out_dist, uint32_t* out_internal, int32_t* out_pid,
                           int32_t* out_counts) {
  memcpy(out_counts + first, cnts, count * sizeof(int32_t));
  const uint64_t tot = count * knbn, o0 = first * knbn;
  for (uint64_t s = 0; s < tot; ++s) out_ids[o0 + s] = tmp[s].origin;
  for (uint64_t s = 0; s < tot; ++s) out_dist[o0 + s] = tmp[s].dist;
  if (out_internal)
    for (uint64_t s = 0; s < tot; ++s) out_internal[o0 + s] = tmp[s].internal;
  if (out_pid)  // PointId(level, rank), hnsw.rs:46
    for (uint64_t s = 0; s < tot; ++s) {
      const uint32_t it = tmp[s].internal;
      out_pid[2 * (o0 + s)] = it != hb::INVALID_ID ? (int32_t)rx->h_level[it] : -1;
      out_pid[2 * (o0 + s) + 1] = it != hb::INVALID_ID ? rx->h_rank[it] : -1;
    }
}

int hnsw_b200_search_flat(const void* h, const void* queries, uint64_t nq, uint64_t dim, uint64_t knbn,
                          uint64_t ef_search, int filter_mode, const uint64_t* filter_ids, uint64_t nfilter,
                          hnsw_b200_filter_fn fn, void* ctx, uint64_t* out_ids, float* out_dist,
                          uint32_t* out_internal, int32_t* out_pid, int32_t* out_counts) {
  HB_HS(h);
  if (nq == 0) return 0;
  if (!queries || !out_ids || !out_dist || !out_counts || knbn == 0) return set_err("bad argument");
  std::vector<uint32_t> bits;
  const uint32_t* fb = nullptr;
  if (filter_mode) {
    int r = pass(ix, ix->make_filter_bits(filter_mode, filter_ids, nfilter, fn, ctx, bits));
    if (r) return r;
    fb = bits.data();
  }
  // one device, or one contiguous shard per device: search, then unpack the shard's answers into the caller's arrays
  const size_t qrow = (size_t)dim * ix->es;
  auto run = [=](Index* rx, size_t first, size_t count) -> int {
    const NeighbourOut* tmp = nullptr;
    const int32_t* cnts = nullptr;
    Index::CtxLease lease(rx);  // the answers stay in the context's pinned buffer until they are unpacked below
    int r = rx->search_host_staged(lease.c, (const char*)queries + first * qrow, nullptr, count, (int)dim, knbn, ef_search, fb, &tmp, &cnts);
    if (r) return r;
    unpack_answers(rx, tmp, cnts, first, count, knbn, out_ids, out_dist, out_internal, out_pid, out_counts);
    return 0;
  };
  return pass(ix, use_shards(ix, nq) ? ix->for_each_shard(nq, run) : run(ix, 0, nq));
}

int hnsw_b200_search_flat_filters(const void* h, const void* queries, uint64_t nq, uint64_t dim, uint64_t knbn,
                                  uint64_t ef_search, const uint64_t* filter_offsets, const uint64_t* filter_ids,
                                  uint64_t* out_ids, float* out_dist, uint32_t* out_internal, int32_t* out_pid,
                                  int32_t* out_counts) {
  HB_HS(h);
  if (nq == 0) return 0;
  if (!queries || !out_ids || !out_dist || !out_counts || !filter_offsets) return set_err("search_flat_filters: NULL array");
  if (knbn == 0) return set_err("search_flat_filters: knbn must be positive");
  if (filter_offsets[0] != 0) return set_err("search_flat_filters: filter_offsets[0] must be 0");
  for (uint64_t i = 0; i < nq; ++i)
    if (filter_offsets[i + 1] < filter_offsets[i])
      return set_err("search_flat_filters: filter_offsets decrease at query " + std::to_string(i));
  if (filter_offsets[nq] != 0 && !filter_ids) return set_err("search_flat_filters: filter_ids is NULL");
  for (uint64_t i = 0; i < nq; ++i)
    for (uint64_t j = filter_offsets[i] + 1; j < filter_offsets[i + 1]; ++j)
      if (filter_ids[j] < filter_ids[j - 1])
        return set_err("search_flat_filters: the ids of query " + std::to_string(i) + " are not ascending");
  // translated once, on this device; replicas hold the same internal ids and read their shard's descriptors
  Index::QueryFilterSet qf;
  int r = pass(ix, ix->make_query_filters(nq, filter_offsets, filter_ids, qf));
  if (r) return r;
  const size_t qrow = (size_t)dim * ix->es;
  const hb::QueryFilter* desc = qf.desc.data();
  const uint32_t* pay = qf.payload.data();
  auto run = [=](Index* rx, size_t first, size_t count) -> int {
    const NeighbourOut* tmp = nullptr;
    const int32_t* cnts = nullptr;
    Index::CtxLease lease(rx);
    int rr = rx->search_host_staged(lease.c, (const char*)queries + first * qrow, nullptr, count, (int)dim, knbn, ef_search,
                                    nullptr, &tmp, &cnts, desc + first, pay);
    if (rr) return rr;
    unpack_answers(rx, tmp, cnts, first, count, knbn, out_ids, out_dist, out_internal, out_pid, out_counts);
    return 0;
  };
  return pass(ix, use_shards(ix, nq) ? ix->for_each_shard(nq, run) : run(ix, 0, nq));
}

// Submit / wait: the same search with the call split in two, so that one host thread keeps several batches in flight
// (batch i+1 is enqueued before batch i's answers are collected).  Unfiltered, one device.
// one device's share of a submitted batch: enqueue on a leased context of `rx`, remember where to unpack to
static int submit_on(Index* rx, int* ctx_out, const void* queries, uint64_t nq, uint64_t dim, uint64_t knbn, uint64_t ef_search,
                     uint64_t* out_ids, float* out_dist, uint32_t* out_internal, int32_t* out_pid, int32_t* out_counts) {
  const int ci = rx->acquire_ctx();
  int r = rx->search_host_begin(ci, queries, nullptr, nq, (int)dim, knbn, ef_search, nullptr);
  if (r) {
    rx->release_ctx(ci);
    return r;
  }
  Index::SearchCtx::Pending& p = rx->ctx(ci).pend;
  p.u_ids = out_ids;
  p.u_dist = out_dist;
  p.u_internal = out_internal;
  p.u_pid = out_pid;
  p.u_counts = out_counts;
  *ctx_out = ci;
  return 0;
}
static int wait_on(Index* rx, int ci) {
  const NeighbourOut* tmp = nullptr;
  const int32_t* cnts = nullptr;
  int r = rx->search_host_finish(ci, &tmp, &cnts);
  if (!r) {
    const Index::SearchCtx::Pending& p = rx->ctx(ci).pend;
    memcpy(p.u_counts, cnts, p.nq * sizeof(int32_t));
    const uint64_t tot = p.nq * p.k;
    for (uint64_t s = 0; s < tot; ++s) p.u_ids[s] = tmp[s].origin;
    for (uint64_t s = 0; s < tot; ++s) p.u_dist[s] = tmp[s].dist;
    if (p.u_internal)
      for (uint64_t s = 0; s < tot; ++s) p.u_internal[s] = tmp[s].internal;
    if (p.u_pid)
      for (uint64_t s = 0; s < tot; ++s) {
        const uint32_t it = tmp[s].internal;
        p.u_pid[2 * s] = it != hb::INVALID_ID ? (int32_t)rx->h_level[it] : -1;
        p.u_pid[2 * s + 1] = it != hb::INVALID_ID ? rx->h_rank[it] : -1;
      }
  }
  rx->release_ctx(ci);
  return r;
}

// Submit / wait: the same search with the call split in two, so that one host thread keeps several batches in flight
// (batch i+1 is enqueued before batch i's answers are collected).  Unfiltered.  With replicas (hnsw_b200_replicate) the
// batch is sharded like a search_flat call: every device gets its contiguous share enqueued at submit time.
int64_t hnsw_b200_search_flat_submit(const void* h, const void* queries, uint64_t nq, uint64_t dim, uint64_t knbn,
                                     uint64_t ef_search, uint64_t* out_ids, float* out_dist, uint32_t* out_internal,
                                     int32_t* out_pid, int32_t* out_counts) {
  HB_HS(h);
  if (!queries || !out_ids || !out_dist || !out_counts || knbn == 0 || nq == 0) return set_err("bad argument");
  Index::Ticket t;
  const size_t qrow = (size_t)dim * ix->es;
  int r = 0;
  if (use_shards(ix, nq)) {
    r = ix->for_each_shard_inline(nq, [&](Index* rx, size_t first, size_t count) {
      int ci = -1;
      int rr = submit_on(rx, &ci, (const char*)queries + first * qrow, count, dim, knbn, ef_search, out_ids + first * knbn,
                         out_dist + first * knbn, out_internal ? out_internal + first * knbn : nullptr,
                         out_pid ? out_pid + 2 * first * knbn : nullptr, out_counts + first);
      if (!rr) t.parts.push_back({rx, ci});
      return rr;
    });
  } else {
    int ci = -1;
    r = submit_on(ix, &ci, queries, nq, dim, knbn, ef_search, out_ids, out_dist, out_internal, out_pid, out_counts);
    if (!r) t.parts.push_back({ix, ci});
  }
  if (r) {
    for (auto& pr : t.parts) wait_on(pr.first, pr.second);  // collect what was enqueued before the failure
    return pass(ix, r);
  }
  ix->pending_.fetch_add(1);
  return ix->park_ticket(std::move(t));
}

int hnsw_b200_search_flat_wait(const void* h, int64_t ticket) {
  if (!h) return set_err("NULL handle");
  Index* ix = ((const AnyApi*)h)->ix;  // no lock: a writer holding the index exclusively is waiting for this very call
  hb::DeviceRestore keep;
  Index::Ticket t;
  if (!ix->take_ticket(ticket, t)) return set_err("bad ticket");
  int r = 0;
  if (t.parts.size() > 1) {  // sharded batch: every device's part is collected and unpacked by that device's worker thread
    r = ix->finish_parts(t.parts, [](Index* rx, int ci) { return wait_on(rx, ci); });
    if (r) g_err = ix->err();
  } else {
    for (auto& pr : t.parts) {
      r = wait_on(pr.first, pr.second);
      if (r) g_err = pr.first->err();
    }
  }
  ix->pending_.fetch_sub(1);
  return r;
}

int hnsw_b200_search_device(const void* h, const void* d_queries, uint64_t nq, uint64_t knbn,
                            uint64_t ef_search, void* d_out, int32_t* d_counts, int sync, float* kernel_ms) {
  HB_HS(h);
  return pass(ix, ix->search_device(d_queries, nq, knbn, ef_search, nullptr, (NeighbourOut*)d_out, d_counts, sync != 0,
                                    kernel_ms));
}

int hnsw_b200_join(void* h) {
  HB_HS(h);
  return pass(ix, ix->join());
}
int hnsw_b200_stream_wait_last(void* h, void* cuda_stream) {
  HB_HS(h);
  return pass(ix, ix->stream_wait_last((cudaStream_t)cuda_stream));
}
int hnsw_b200_set_stream(void* h, void* cuda_stream) {
  HB_H(h);
  return pass(ix, ix->set_stream((cudaStream_t)cuda_stream));
}
int hnsw_b200_check_status(void* h) {
  HB_H(h);
  int r = ix->check_status();
  if (r < 0) g_err = ix->err();
  return r;
}

int hnsw_b200_enable_stats(void* h, int enable) {
  HB_H(h);
  return ix->enable_stats(enable != 0);
}
int hnsw_b200_get_stats(const void* h, uint64_t* out4, int reset) {
  HB_H(h);
  return pass(ix, ix->get_stats(out4, reset != 0));
}

int hnsw_b200_export_points(const void* h, uint8_t* levels, int32_t* ranks, uint64_t* origin, int64_t* entry) {
  HB_H(h);
  for (size_t i = 0; i < ix->n; ++i) {
    if (levels) levels[i] = ix->h_level[i];
    if (ranks) ranks[i] = ix->h_rank[i];
    if (origin) origin[i] = ix->h_origin[i];
  }
  if (entry) *entry = ix->entry == hb::INVALID_ID ? -1 : (int64_t)ix->entry;
  return 0;
}
int hnsw_b200_export_vectors(const void* h, void* out) {
  HB_H(h);
  return pass(ix, ix->export_vectors(out));
}
// FlatNeighborhood::from(&hnsw) + get_neighbours(DataId) (flatten.rs:93-126): neighbours of `origin_id` over all
// layers, ascending distance.  Returns the number written (<= cap), -1 when the id is unknown.
int64_t hnsw_b200_flat_neighbours(const void* h, uint64_t origin_id, Neighbour_api* out, uint64_t cap) {
  if (!h) return set_err("NULL handle");
  Index* ix = ((const AnyApi*)h)->ix;
  std::shared_lock<std::shared_mutex> g(ix->mu);
  std::vector<uint64_t> off, nbo;
  std::vector<float> nbd;
  if (pass(ix, ix->flatten(off, nbo, nbd))) return -1;
  for (size_t p = 0; p < ix->n; ++p)
    if (ix->h_origin[p] == origin_id) {
      uint64_t c = 0;
      for (uint64_t j = off[p]; j < off[p + 1] && c < cap; ++j, ++c) out[c] = Neighbour_api{(size_t)nbo[j], nbd[j]};
      return (int64_t)c;
    }
  set_err("unknown origin id");
  return -1;
}
// whole flattened graph: offsets[nb_point+1] (internal-id order), neighbour origin ids and distances; pass NULL
// arrays to get the total neighbour count only
int64_t hnsw_b200_flatten(const void* h, uint64_t* offsets, uint64_t* nb_origin, float* nb_dist) {
  if (!h) return set_err("NULL handle");
  Index* ix = ((const AnyApi*)h)->ix;
  std::shared_lock<std::shared_mutex> g(ix->mu);
  std::vector<uint64_t> off, nbo;
  std::vector<float> nbd;
  if (pass(ix, ix->flatten(off, nbo, nbd))) return -1;
  if (offsets) memcpy(offsets, off.data(), off.size() * 8);
  if (nb_origin) memcpy(nb_origin, nbo.data(), nbo.size() * 8);
  if (nb_dist) memcpy(nb_dist, nbd.data(), nbd.size() * 4);
  return (int64_t)nbo.size();
}

int64_t hnsw_b200_layer_edges(const void* h, int layer) {
  if (!h) return set_err("NULL handle");
  Index* ix = ((const AnyApi*)h)->ix;
  std::shared_lock<std::shared_mutex> g(ix->mu);
  int64_t total = 0;
  if (pass(ix, ix->export_layer(layer, nullptr, nullptr, nullptr, &total))) return -1;
  return total;
}
int hnsw_b200_export_layer(const void* h, int layer, uint64_t* offsets, uint32_t* ids, float* dists) {
  HB_H(h);
  return pass(ix, ix->export_layer(layer, offsets, ids, dists, nullptr));
}
int hnsw_b200_import_graph(void* h, const void* vecs, uint64_t n, uint64_t dim, const uint64_t* origin,
                           const uint8_t* levels, int64_t entry, int nlayers, const uint64_t* const* offsets,
                           const uint32_t* const* ids, const float* const* dists) {
  HB_H(h);
  return pass(ix, ix->import_graph(vecs, n, (int)dim, origin, levels, entry, nlayers, offsets, ids, dists));
}

int hnsw_b200_blob_header(const void* h, uint64_t* header16) {
  HB_H(h);
  return ix->blob_header(header16);
}
int hnsw_b200_blob_alloc(void* h, const uint64_t* header16) {
  HB_H(h);
  return pass(ix, ix->blob_alloc(header16));
}
int hnsw_b200_blob_count(const void* h) { return h ? ((const AnyApi*)h)->ix->blob_count() : 0; }
int hnsw_b200_blob_info(const void* h, int i, void** dev_ptr, uint64_t* nbytes) {
  HB_H(h);
  return pass(ix, ix->blob_info(i, dev_ptr, nbytes));
}
int hnsw_b200_blob_commit(void* h) {
  HB_H(h);
  return pass(ix, ix->blob_commit());
}

// ---- multi-GPU (multi.cu)
int hnsw_b200_replicate(void* h, int ndev, const int* devices) {
  HB_H(h);
  return pass(ix, ix->replicate(ndev, devices));
}
int hnsw_b200_replica_count(const void* h) { return h ? (int)((const AnyApi*)h)->ix->replica_count() : 0; }
int hnsw_b200_nccl_unique_id(uint8_t* id128) {
  if (!id128) return set_err("NULL argument");
  return Index::nccl_unique_id(id128) ? set_err("NCCL is not available (libnccl.so.2)") : 0;
}
int hnsw_b200_nccl_init(void* h, int nranks, int rank, const uint8_t* id128) {
  HB_H(h);
  if (!id128) return set_err("NULL argument");
  return pass(ix, ix->nccl_init(nranks, rank, id128));
}
int hnsw_b200_nccl_broadcast_index(void* h, int root) {
  HB_H(h);
  return pass(ix, ix->nccl_broadcast_index(root));
}
int hnsw_b200_nccl_allgather(void* h, const void* d_send, void* d_recv, uint64_t bytes_per_rank, void* cuda_stream) {
  HB_H(h);
  return pass(ix, ix->nccl_allgather(d_send, d_recv, bytes_per_rank, (cudaStream_t)cuda_stream));
}

int hnsw_b200_dist_batch(const void* h, const void* queries, uint64_t nq, uint64_t dim, const uint32_t* cand,
                         uint64_t m, float* out) {
  HB_H(h);
  return pass(ix, ix->dist_batch(queries, nq, (int)dim, cand, m, out));
}
int hnsw_b200_bruteforce(const void* h, const void* queries, uint64_t nq, uint64_t dim, uint64_t k,
                         uint32_t* out_ids, float* out_dist) {
  HB_H(h);
  return pass(ix, ix->bruteforce(queries, nq, (int)dim, k, out_ids, out_dist));
}

}  // extern "C"
