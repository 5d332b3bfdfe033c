"""Host-side mirror of the reference's public interface over the C ABI of libhnsw_b200.so.

Mirrors, name for name, `Hnsw<T,D>` and the `AnnT` trait of jean-pierreBoth/hnswlib-rs
(/root/reference/src/hnsw.rs:739-905,1069-1071,1224-1238,1487-1635; /root/reference/src/api.rs:13-38)
and `FilterT` (/root/reference/src/filter.rs:7-24) for f32 data.  Every call goes through the
extern "C" symbols declared in include/hnsw_b200.h (ctypes); there is no CPU fallback — constructing
an index without a usable CUDA device raises.
"""
import ctypes as C
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_LIB_PATH = os.environ.get("HNSW_B200_LIB") or os.path.join(_HERE, "lib", "libhnsw_b200.so")  # the override serves A/B builds of scripts/
_LIB = None

FILTER_FN = C.CFUNCTYPE(C.c_int, C.c_uint64, C.c_void_p)


class Neighbour_api(C.Structure):  # libext.rs:64-71
    _fields_ = [("id", C.c_size_t), ("d", C.c_float)]


class Neighbourhood_api(C.Structure):  # libext.rs:82-87
    _fields_ = [("nbgh", C.c_int64), ("neighbours", C.POINTER(Neighbour_api))]


class Vec_api(C.Structure):  # libext.rs:58-62
    _fields_ = [("len", C.c_int64), ("ptr", C.POINTER(Neighbourhood_api))]


def lib_path():
    return _LIB_PATH


def load_library():
    """dlopen libhnsw_b200.so (fails loudly when it has not been built)."""
    global _LIB
    if _LIB is not None:
        return _LIB
    if not os.path.exists(_LIB_PATH):
        raise RuntimeError(f"{_LIB_PATH} is missing: run __graft_entry__.build() (make -C hnswlib-rs_b200/csrc)")
    L = C.CDLL(_LIB_PATH)
    vp, u64, sz, i32, i64 = C.c_void_p, C.c_uint64, C.c_size_t, C.c_int, C.c_int64
    for suf in ("f32", "i32", "u32", "u16", "u8"):   # libext.rs generates one set per element type
        f = getattr(L, "init_hnsw_" + suf); f.restype = vp; f.argtypes = [sz, sz, sz, C.c_char_p]
        f = getattr(L, "init_hnsw_ptrdist_" + suf); f.restype = vp; f.argtypes = [sz, sz, vp]
        getattr(L, "insert_" + suf).argtypes = [vp, sz, vp, sz]
        getattr(L, "parallel_insert_" + suf).argtypes = [vp, sz, sz, vp, vp]
        f = getattr(L, "search_neighbours_" + suf); f.restype = C.POINTER(Neighbourhood_api); f.argtypes = [vp, sz, vp, sz, sz]
        f = getattr(L, "parallel_search_neighbours_" + suf); f.restype = C.POINTER(Vec_api); f.argtypes = [vp, sz, i64, vp, sz, sz]
        f = getattr(L, "file_dump_" + suf); f.restype = i64; f.argtypes = [vp, sz, C.c_char_p]
    for suf in ("f32", "u16"):
        f = getattr(L, "new_hnsw_" + suf); f.restype = vp; f.argtypes = [sz, sz, sz, C.c_char_p, sz, sz]
        getattr(L, "drop_hnsw_" + suf).argtypes = [vp]
    L.get_hnswio.restype = vp
    L.get_hnswio.argtypes = [u64, C.c_char_p]
    L.hnsw_b200_get_hnswio.restype = vp
    L.hnsw_b200_get_hnswio.argtypes = [C.c_char_p, C.c_char_p]
    L.hnsw_b200_free_hnswio.argtypes = [vp]
    L.hnsw_b200_file_dump.argtypes = [vp, C.c_char_p, C.c_char_p, i32, C.c_char_p, sz]
    L.hnsw_b200_load_dump.restype = vp
    L.hnsw_b200_load_dump.argtypes = [vp, i32, sz, C.c_char_p]
    L.load_hnsw_description.restype = vp
    L.load_hnsw_description.argtypes = [sz, C.c_char_p]
    L.hnsw_b200_free_description.argtypes = [vp]
    L.hnsw_b200_new.restype = vp
    L.hnsw_b200_new.argtypes = [i32, sz, sz, sz, C.c_char_p, sz, sz]
    L.hnsw_b200_drop.argtypes = [vp]
    L.hnsw_b200_last_error.restype = C.c_char_p
    L.hnsw_b200_device_count.restype = i32
    L.hnsw_b200_set_device.argtypes = [i32]
    L.hnsw_b200_free_neighbourhood.argtypes = [vp]
    L.hnsw_b200_free_vec_api.argtypes = [vp]
    for name in ("set_extend_candidates", "set_keeping_pruned", "set_searching_mode", "enable_stats", "set_tie_mode"):
        getattr(L, "hnsw_b200_" + name).argtypes = [vp, i32]
    L.hnsw_b200_get_extend_candidates.argtypes = [vp]
    L.hnsw_b200_modify_level_scale.argtypes = [vp, C.c_double]
    L.hnsw_b200_set_level_seed.argtypes = [vp, u64]
    L.hnsw_b200_get_nb_point.restype = u64
    L.hnsw_b200_get_nb_point.argtypes = [vp]
    L.hnsw_b200_get_max_level_observed.argtypes = [vp]
    L.hnsw_b200_get_dim.argtypes = [vp]
    L.hnsw_b200_set_insert_batching.argtypes = [vp, C.c_uint32, C.c_uint32]
    L.hnsw_b200_insert_flat.argtypes = [vp, vp, u64, u64, vp, vp]
    L.hnsw_b200_search_flat.argtypes = [vp, vp, u64, u64, u64, u64, i32, vp, u64, FILTER_FN, vp, vp, vp, vp, vp, vp]
    L.hnsw_b200_search_flat_filters.argtypes = [vp, vp, u64, u64, u64, u64, vp, vp, vp, vp, vp, vp, vp]
    L.hnsw_b200_search_device.argtypes = [vp, vp, u64, u64, u64, vp, vp, i32, vp]
    L.hnsw_b200_search_flat_submit.restype = i64
    L.hnsw_b200_search_flat_submit.argtypes = [vp, vp, u64, u64, u64, u64, vp, vp, vp, vp, vp]
    L.hnsw_b200_search_flat_wait.argtypes = [vp, i64]
    L.hnsw_b200_get_stats.argtypes = [vp, vp, i32]
    L.hnsw_b200_set_stream.argtypes = [vp, vp]
    L.hnsw_b200_join.argtypes = [vp]
    L.hnsw_b200_stream_wait_last.argtypes = [vp, vp]
    L.hnsw_b200_check_status.argtypes = [vp]
    L.hnsw_b200_export_points.argtypes = [vp, vp, vp, vp, vp]
    L.hnsw_b200_export_vectors.argtypes = [vp, vp]
    L.hnsw_b200_layer_edges.restype = i64
    L.hnsw_b200_layer_edges.argtypes = [vp, i32]
    L.hnsw_b200_export_layer.argtypes = [vp, i32, vp, vp, vp]
    L.hnsw_b200_flat_neighbours.restype = i64
    L.hnsw_b200_flat_neighbours.argtypes = [vp, u64, vp, u64]
    L.hnsw_b200_flatten.restype = i64
    L.hnsw_b200_flatten.argtypes = [vp, vp, vp, vp]
    L.hnsw_b200_import_graph.argtypes = [vp, vp, u64, u64, vp, vp, i64, i32, vp, vp, vp]
    L.hnsw_b200_blob_header.argtypes = [vp, vp]
    L.hnsw_b200_blob_alloc.argtypes = [vp, vp]
    L.hnsw_b200_blob_count.argtypes = [vp]
    L.hnsw_b200_blob_info.argtypes = [vp, i32, vp, vp]
    L.hnsw_b200_blob_commit.argtypes = [vp]
    L.hnsw_b200_replicate.argtypes = [vp, i32, vp]
    L.hnsw_b200_replica_count.argtypes = [vp]
    L.hnsw_b200_nccl_unique_id.argtypes = [vp]
    L.hnsw_b200_nccl_init.argtypes = [vp, i32, i32, vp]
    L.hnsw_b200_nccl_broadcast_index.argtypes = [vp, i32]
    L.hnsw_b200_nccl_allgather.argtypes = [vp, vp, vp, u64, vp]
    L.hnsw_b200_dist_batch.argtypes = [vp, vp, u64, u64, vp, u64, vp]
    L.hnsw_b200_bruteforce.argtypes = [vp, vp, u64, u64, u64, vp, vp]
    _LIB = L
    return L


def last_error():
    return load_library().hnsw_b200_last_error().decode("utf-8", "replace")


def _p(a):
    return None if a is None else a.ctypes.data_as(C.c_void_p)


class HnswError(RuntimeError):
    pass


def pack_filters(filters, nq):
    """One FilterT (id list) per query, packed for hnsw_b200_search_flat_filters: returns (offsets u64[nq + 1], ids u64),
    query i admitting ids[offsets[i]:offsets[i + 1]].

    filters is either a sequence of nq id sequences, each sorted here (as search_flat sorts its filter), or an
    (offsets, ids) pair: a tuple of two numpy arrays whose first has nq + 1 entries.  The pair is checked to describe
    ids exactly (offsets[0] == 0, offsets never decreasing, offsets[-1] == len(ids); ValueError otherwise: the library
    cannot see the length of ids) and passed on unsorted (the library refuses a list that is not ascending).  A list is
    never taken for a pair: pass per-query filters as a list to keep two numpy filters from reading as one pair."""
    if (isinstance(filters, tuple) and len(filters) == 2 and all(isinstance(x, np.ndarray) for x in filters)
            and len(filters[0]) == nq + 1):
        offsets = np.ascontiguousarray(filters[0].reshape(-1), np.uint64)
        ids = np.ascontiguousarray(filters[1].reshape(-1), np.uint64)
        if offsets[0] != 0 or np.any(offsets[1:] < offsets[:-1]) or int(offsets[-1]) != len(ids):
            raise ValueError(f"(offsets, ids) pair: offsets must start at 0, never decrease and end at len(ids) = {len(ids)}"
                             " (to give per-query filters, pass them as a list)")
        return offsets, ids
    if len(filters) != nq:
        raise ValueError(f"{len(filters)} filters for {nq} queries")
    lists = [np.sort(np.asarray(f, np.uint64).reshape(-1)) for f in filters]
    offsets = np.zeros(nq + 1, np.uint64)
    offsets[1:] = np.cumsum([len(x) for x in lists], dtype=np.uint64)
    ids = np.concatenate(lists) if lists else np.zeros(0, np.uint64)
    return offsets, np.ascontiguousarray(ids, np.uint64)


class Neighbour:
    """hnsw.rs:98-107: d_id (DataId), distance, p_id = PointId(level, rank)."""
    __slots__ = ("d_id", "distance", "p_id")

    def __init__(self, d_id, distance, p_id):
        self.d_id, self.distance, self.p_id = d_id, distance, p_id

    def get_origin_id(self):
        return self.d_id

    def get_distance(self):
        return self.distance

    def __repr__(self):
        return f"Neighbour(d_id={self.d_id}, distance={self.distance!r}, p_id={self.p_id})"


_DT = {np.dtype(np.float32): (0, "f32"), np.dtype(np.uint8): (1, "u8"), np.dtype(np.uint16): (2, "u16"),
       np.dtype(np.uint32): (3, "u32"), np.dtype(np.int32): (4, "i32")}


class Hnsw:
    """Hnsw<T, D>: T = dtype (f32 default; i32/u32/u16/u8), D given by name ("DistL2", "DistDot", "DistCosine",
    "DistL1", "DistHamming", "DistJaccard", ...)."""

    def __init__(self, max_nb_connection, max_elements, max_layer, ef_construction, dist_name, device=None,
                 dtype=np.float32):
        L = load_library()
        if device is not None:
            if L.hnsw_b200_set_device(int(device)) != 0:
                raise HnswError(last_error())
        name = dist_name.encode()
        self._L = L
        self.dtype = np.dtype(dtype)
        code, self._suf = _DT[self.dtype]
        if self._suf in ("f32", "u16"):   # the reference's own constructor with max_elements / max_layer
            ctor = getattr(L, "new_hnsw_" + self._suf)
            self._h = ctor(int(max_nb_connection), int(ef_construction), len(name), name, int(max_elements), int(max_layer))
        else:
            self._h = L.hnsw_b200_new(code, int(max_nb_connection), int(ef_construction), len(name), name,
                                      int(max_elements), int(max_layer))
        if not self._h:
            raise HnswError("new_hnsw failed: " + last_error())
        self.dist_name = dist_name
        self.max_nb_connection = int(max_nb_connection)
        self.ef_construction = int(ef_construction)

    # ---- lifetime
    def close(self):
        if getattr(self, "_h", None):
            self._L.hnsw_b200_drop(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _chk(self, r):
        if r != 0:
            raise HnswError(last_error())

    # ---- getters / setters (hnsw.rs:810-905)
    def get_nb_point(self):
        return int(self._L.hnsw_b200_get_nb_point(self._h))

    def get_max_level_observed(self):
        return int(self._L.hnsw_b200_get_max_level_observed(self._h))

    def get_max_nb_connection(self):
        return self.max_nb_connection

    def get_ef_construction(self):
        return self.ef_construction

    def get_data_dimension(self):
        return int(self._L.hnsw_b200_get_dim(self._h))

    def set_extend_candidates(self, flag):
        self._chk(self._L.hnsw_b200_set_extend_candidates(self._h, int(bool(flag))))

    def set_keeping_pruned(self, flag):
        self._chk(self._L.hnsw_b200_set_keeping_pruned(self._h, int(bool(flag))))

    def set_searching_mode(self, flag):
        self._chk(self._L.hnsw_b200_set_searching_mode(self._h, int(bool(flag))))

    def modify_level_scale(self, scale):
        self._chk(self._L.hnsw_b200_modify_level_scale(self._h, float(scale)))

    def set_level_seed(self, seed):
        self._chk(self._L.hnsw_b200_set_level_seed(self._h, int(seed)))

    def set_insert_batching(self, ratio, max_batch):
        self._chk(self._L.hnsw_b200_set_insert_batching(self._h, int(ratio), int(max_batch)))

    # ---- insertion (hnsw.rs:1069-1071, 1224-1238; api.rs:47-56)
    def insert(self, data_with_id):
        v, i = data_with_id
        v = np.ascontiguousarray(v, self.dtype)
        before = self.get_nb_point()
        getattr(self._L, "insert_" + self._suf)(self._h, v.size, _p(v), int(i))
        if self.get_nb_point() != before + 1:
            raise HnswError("insert_f32 failed: " + last_error())

    insert_data = lambda self, data, id_: self.insert((data, id_))  # AnnT::insert_data

    def parallel_insert(self, datas):
        """datas: sequence of (vector, id) — goes through parallel_insert_f32 (row pointers)."""
        if len(datas) == 0:
            return
        rows = [np.ascontiguousarray(v, self.dtype) for v, _ in datas]
        d = rows[0].size
        ptrs = (C.c_void_p * len(rows))(*[r.ctypes.data for r in rows])
        ids = (C.c_size_t * len(rows))(*[int(i) for _, i in datas])
        before = self.get_nb_point()
        getattr(self._L, "parallel_insert_" + self._suf)(self._h, len(rows), d, ptrs, ids)
        if self.get_nb_point() != before + len(rows):
            raise HnswError("parallel_insert_f32 failed: " + last_error())

    parallel_insert_slice = parallel_insert
    parallel_insert_data = parallel_insert  # AnnT::parallel_insert_data

    def insert_flat(self, vecs, ids=None, levels=None):
        """Extension: one flat [n, d] array (no per-row pointers)."""
        vecs = np.ascontiguousarray(vecs, self.dtype)
        n, d = vecs.shape
        ids_a = None if ids is None else np.ascontiguousarray(ids, np.uint64)
        lv = None if levels is None else np.ascontiguousarray(levels, np.int32)
        self._chk(self._L.hnsw_b200_insert_flat(self._h, _p(vecs), n, d, _p(ids_a), _p(lv)))

    # ---- search (hnsw.rs:1487-1635; api.rs:51-65)
    def search(self, data, knbn, ef_arg):
        return self.search_filter(data, knbn, ef_arg, None)

    search_neighbours = search  # AnnT::search_neighbours

    def search_possible_filter(self, data, knbn, ef_arg, filter=None):
        return self.search_filter(data, knbn, ef_arg, filter)

    def search_filter(self, data, knbn, ef_arg, filter=None):
        """filter: None | sorted sequence of ids (FilterT for Vec<usize>) | callable(id)->bool."""
        if filter is None:
            v = np.ascontiguousarray(data, self.dtype)
            res = getattr(self._L, "search_neighbours_" + self._suf)(self._h, v.size, _p(v), int(knbn), int(ef_arg))
            if not res:
                raise HnswError("search_neighbours_f32 failed: " + last_error())
            n = res.contents.nbgh
            ids = [int(res.contents.neighbours[j].id) for j in range(n)]
            ds = [float(res.contents.neighbours[j].d) for j in range(n)]
            self._L.hnsw_b200_free_neighbourhood(res)
            # p_id needs the extension call; fetch lazily through search_flat when asked for
            return [Neighbour(i, d, None) for i, d in zip(ids, ds)]
        o, d, it, pid, cnt = self.search_flat(np.asarray(data, self.dtype)[None, :], knbn, ef_arg, filter=filter)
        return [Neighbour(int(o[0, j]), float(d[0, j]), (int(pid[0, j, 0]), int(pid[0, j, 1]))) for j in range(cnt[0])]

    def parallel_search(self, datas, knbn, ef):
        """Vec<Vec<Neighbour>> in input order, through parallel_search_neighbours_f32 (row pointers)."""
        rows = [np.ascontiguousarray(v, self.dtype) for v in datas]
        if not rows:
            return []
        ptrs = (C.c_void_p * len(rows))(*[r.ctypes.data for r in rows])
        res = getattr(self._L, "parallel_search_neighbours_" + self._suf)(self._h, len(rows), rows[0].size, ptrs, int(knbn), int(ef))
        if not res:
            raise HnswError("parallel_search_neighbours_f32 failed: " + last_error())
        out = []
        for i in range(res.contents.len):
            nb = res.contents.ptr[i]
            out.append([Neighbour(int(nb.neighbours[j].id), float(nb.neighbours[j].d), None) for j in range(nb.nbgh)])
        self._L.hnsw_b200_free_vec_api(res)
        return out

    parallel_search_neighbours = parallel_search  # AnnT::parallel_search_neighbours

    def search_flat(self, queries, knbn, ef, filter=None, with_internal=True, with_pid=True):
        """Extension: flat batch.  Returns (origin u64[nq,k], dist f32[nq,k], internal u32[nq,k] | None,
        pid i32[nq,k,2] | None, counts)."""
        q = np.ascontiguousarray(queries, self.dtype)
        nq, d = q.shape
        o = np.empty((nq, knbn), np.uint64)
        ds = np.empty((nq, knbn), np.float32)
        it = np.empty((nq, knbn), np.uint32) if with_internal else None
        pid = np.empty((nq, knbn, 2), np.int32) if with_pid else None
        cnt = np.empty(nq, np.int32)
        mode, fids, nf, cb = 0, None, 0, FILTER_FN(0)
        if filter is not None:
            if callable(filter):
                mode = 2
                cb = FILTER_FN(lambda i, _c: 1 if filter(int(i)) else 0)
            else:
                mode = 1
                fids = np.ascontiguousarray(np.sort(np.asarray(filter, np.uint64)))
                nf = len(fids)
        self._chk(self._L.hnsw_b200_search_flat(self._h, _p(q), nq, d, int(knbn), int(ef), mode, _p(fids), nf, cb, None,
                                                _p(o), _p(ds), _p(it), _p(pid), _p(cnt)))
        return o, ds, it, pid, cnt

    def search_flat_filters(self, queries, knbn, ef, filters, with_internal=True, with_pid=True):
        """hnsw_b200_search_flat_filters: search_flat with one id-list filter per query (pack_filters says what `filters`
        may be).  Same outputs as search_flat."""
        q = np.ascontiguousarray(queries, self.dtype)
        nq, d = q.shape
        offsets, ids = pack_filters(filters, nq)
        o = np.empty((nq, knbn), np.uint64)
        ds = np.empty((nq, knbn), np.float32)
        it = np.empty((nq, knbn), np.uint32) if with_internal else None
        pid = np.empty((nq, knbn, 2), np.int32) if with_pid else None
        cnt = np.empty(nq, np.int32)
        self._chk(self._L.hnsw_b200_search_flat_filters(self._h, _p(q), nq, d, int(knbn), int(ef), _p(offsets), _p(ids),
                                                        _p(o), _p(ds), _p(it), _p(pid), _p(cnt)))
        return o, ds, it, pid, cnt

    def parallel_search_filter(self, datas, knbn, ef, filters):
        """Batched counterpart of [search_filter(datas[i], knbn, ef, filters[i]) for i ...]: lists of Neighbour in input
        order, one id-list filter per query."""
        q = np.asarray([np.asarray(v, self.dtype) for v in datas], self.dtype)
        if len(q) == 0:
            return []
        o, d, _, pid, cnt = self.search_flat_filters(q, knbn, ef, filters, with_internal=False)
        return [[Neighbour(int(o[i, j]), float(d[i, j]), (int(pid[i, j, 0]), int(pid[i, j, 1]))) for j in range(cnt[i])]
                for i in range(len(q))]

    def submit_flat(self, queries, knbn, ef, with_internal=True, with_pid=True):
        """hnsw_b200_search_flat_submit: enqueue a batch, return a ticket for wait_flat (up to 4 outstanding)"""
        q = np.ascontiguousarray(queries, self.dtype)
        nq, d = q.shape
        o = np.empty((nq, knbn), np.uint64)
        ds = np.empty((nq, knbn), np.float32)
        it = np.empty((nq, knbn), np.uint32) if with_internal else None
        pid = np.empty((nq, knbn, 2), np.int32) if with_pid else None
        cnt = np.empty(nq, np.int32)
        t = self._L.hnsw_b200_search_flat_submit(self._h, _p(q), nq, d, int(knbn), int(ef), _p(o), _p(ds), _p(it), _p(pid), _p(cnt))
        if t < 0:
            raise HnswError(last_error())
        return (int(t), q, o, ds, it, pid, cnt)

    def wait_flat(self, ticket):
        t, _q, o, ds, it, pid, cnt = ticket
        self._chk(self._L.hnsw_b200_search_flat_wait(self._h, t))
        return o, ds, it, pid, cnt

    def file_dump(self, path, basename, overwrite=True):
        """AnnT::file_dump (api.rs:70-93): writes <basename>.hnsw.graph / .hnsw.data under `path`, returns the basename
        actually used (a unique one when overwrite is False and the data file exists)."""
        used = C.create_string_buffer(4096)
        self._chk(self._L.hnsw_b200_file_dump(self._h, str(path).encode(), basename.encode(), int(bool(overwrite)), used, 4096))
        return used.value.decode()

    def file_dump_cwd(self, basename):
        """the reference C entry point file_dump_<ty>: dumps into the current directory, returns 1 / -1"""
        name = basename.encode()
        return int(getattr(self._L, "file_dump_" + self._suf)(self._h, len(name), name))

    @classmethod
    def load(cls, path, basename, dist_name, dtype=np.float32, device=None):
        """HnswIo::load_hnsw::<T, D> (hnswio.rs:431-524) through hnsw_b200_get_hnswio + hnsw_b200_load_dump."""
        L = load_library()
        if device is not None and L.hnsw_b200_set_device(int(device)) != 0:
            raise HnswError(last_error())
        io = L.hnsw_b200_get_hnswio(str(path).encode(), basename.encode())
        name = dist_name.encode()
        h = L.hnsw_b200_load_dump(io, _DT[np.dtype(dtype)][0], len(name), name)
        L.hnsw_b200_free_hnswio(io)
        if not h:
            raise HnswError("load failed: " + last_error())
        self = cls.__new__(cls)
        self._L, self._h, self.dtype, self.dist_name = L, h, np.dtype(dtype), dist_name
        self._suf = _DT[self.dtype][1]
        self.max_nb_connection = None
        self.ef_construction = None
        return self

    # ---- statistics / graph transfer (extensions)
    def enable_stats(self, on=True):
        self._chk(self._L.hnsw_b200_enable_stats(self._h, int(on)))

    def set_tie_mode(self, mode):
        """0: ties by (distance, id); 1: the reference's std-BinaryHeap tie behaviour (hnsw_b200_set_tie_mode)"""
        self._chk(self._L.hnsw_b200_set_tie_mode(self._h, int(mode)))

    def get_stats(self, reset=True):
        out = np.zeros(4, np.uint64)
        self._chk(self._L.hnsw_b200_get_stats(self._h, _p(out), int(reset)))
        return {"evals": int(out[0]), "expansions": int(out[1]), "adj_read": int(out[2]), "queries": int(out[3])}

    def set_stream(self, cuda_stream):
        self._chk(self._L.hnsw_b200_set_stream(self._h, C.c_void_p(cuda_stream)))

    def join(self):
        """the handle's stream waits for every asynchronous search_device launch enqueued so far"""
        self._chk(self._L.hnsw_b200_join(self._h))

    def stream_wait_last(self, cuda_stream=None):
        """`cuda_stream` (None = the handle's) waits for the most recent asynchronous search_device launch"""
        self._chk(self._L.hnsw_b200_stream_wait_last(self._h, C.c_void_p(cuda_stream or 0)))

    def check_status(self):
        r = self._L.hnsw_b200_check_status(self._h)
        if r < 0:
            raise HnswError(last_error())
        return r

    def search_device(self, d_queries_ptr, nq, knbn, ef, d_out_ptr, d_counts_ptr, sync=True):
        """Device-resident search: raw device pointers in, Neighbour_api[nq][knbn] + int32 counts out.
        Returns the kernel's CUDA-event time in ms when sync is true."""
        ms = C.c_float(0.0)
        self._chk(self._L.hnsw_b200_search_device(self._h, C.c_void_p(d_queries_ptr), nq, int(knbn), int(ef),
                                                  C.c_void_p(d_out_ptr), C.c_void_p(d_counts_ptr), int(bool(sync)),
                                                  C.byref(ms) if sync else None))
        return float(ms.value)

    # ---- multi-GPU (include/hnsw_b200.h "Multi-GPU search")
    def replicate(self, devices):
        """one process, N devices: copy the index to devices[1:] (NCCL); batched searches are then sharded over them"""
        d = np.ascontiguousarray(devices, np.int32)
        self._chk(self._L.hnsw_b200_replicate(self._h, len(d), _p(d)))

    def replica_count(self):
        return int(self._L.hnsw_b200_replica_count(self._h))

    @staticmethod
    def nccl_unique_id():
        """128 bytes of ncclUniqueId (rank 0 creates it, the host hands it to the other ranks)"""
        buf = np.zeros(128, np.uint8)
        if load_library().hnsw_b200_nccl_unique_id(_p(buf)) != 0:
            raise HnswError(last_error())
        return buf

    def nccl_init(self, nranks, rank, unique_id):
        uid = np.ascontiguousarray(unique_id, np.uint8)
        self._chk(self._L.hnsw_b200_nccl_init(self._h, int(nranks), int(rank), _p(uid)))

    def nccl_broadcast_index(self, root=0):
        self._chk(self._L.hnsw_b200_nccl_broadcast_index(self._h, int(root)))

    def nccl_allgather(self, d_send_ptr, d_recv_ptr, bytes_per_rank, cuda_stream=None):
        self._chk(self._L.hnsw_b200_nccl_allgather(self._h, C.c_void_p(d_send_ptr), C.c_void_p(d_recv_ptr), int(bytes_per_rank),
                                                   C.c_void_p(cuda_stream or 0)))

    def blob_header(self):
        h16 = np.zeros(16, np.uint64)
        self._chk(self._L.hnsw_b200_blob_header(self._h, _p(h16)))
        return h16

    def blob_alloc(self, h16):
        h16 = np.ascontiguousarray(h16, np.uint64)
        self._chk(self._L.hnsw_b200_blob_alloc(self._h, _p(h16)))

    def blobs(self):
        """[(device pointer, nbytes)] of the frozen index arrays (replication over NCCL)."""
        out = []
        for i in range(self._L.hnsw_b200_blob_count(self._h)):
            ptr, nb = C.c_void_p(), C.c_uint64()
            self._chk(self._L.hnsw_b200_blob_info(self._h, i, C.byref(ptr), C.byref(nb)))
            out.append((ptr.value or 0, int(nb.value)))
        return out

    def blob_commit(self):
        self._chk(self._L.hnsw_b200_blob_commit(self._h))

    def export_points(self):
        n = self.get_nb_point()
        lv, rk, og = np.empty(n, np.uint8), np.empty(n, np.int32), np.empty(n, np.uint64)
        e = C.c_int64(-1)
        self._chk(self._L.hnsw_b200_export_points(self._h, _p(lv), _p(rk), _p(og), C.byref(e)))
        return lv, rk, og, int(e.value)

    def export_vectors(self):
        out = np.empty((self.get_nb_point(), self.get_data_dimension()), self.dtype)
        self._chk(self._L.hnsw_b200_export_vectors(self._h, _p(out)))
        return out

    def export_layer(self, layer):
        n = self.get_nb_point()
        ne = int(self._L.hnsw_b200_layer_edges(self._h, layer))
        if ne < 0:
            raise HnswError(last_error())
        off, ids, ds = np.empty(n + 1, np.uint64), np.empty(ne, np.uint32), np.empty(ne, np.float32)
        self._chk(self._L.hnsw_b200_export_layer(self._h, layer, _p(off), _p(ids), _p(ds)))
        return off, ids, ds

    def flat_neighborhood(self):
        """FlatNeighborhood::from(&hnsw) (flatten.rs:93-126): dict DataId -> [(neighbour DataId, distance)] ascending."""
        n = self.get_nb_point()
        tot = int(self._L.hnsw_b200_flatten(self._h, None, None, None))
        if tot < 0:
            raise HnswError(last_error())
        off, ids, ds = np.empty(n + 1, np.uint64), np.empty(tot, np.uint64), np.empty(tot, np.float32)
        self._L.hnsw_b200_flatten(self._h, _p(off), _p(ids), _p(ds))
        og = self.export_points()[2]
        return {int(og[p]): list(zip(ids[int(off[p]):int(off[p + 1])].tolist(), ds[int(off[p]):int(off[p + 1])].tolist()))
                for p in range(n)}

    def import_graph(self, vecs, origin, levels, entry, layers):
        """layers: list (index = layer) of (offsets u64[N+1], ids u32[], dists f32[]|None)."""
        vecs = np.ascontiguousarray(vecs, self.dtype)
        n, d = vecs.shape
        origin = np.ascontiguousarray(origin, np.uint64)
        levels = np.ascontiguousarray(levels, np.uint8)
        keep = []
        nl = len(layers)
        offs, idss, dss = (C.c_void_p * nl)(), (C.c_void_p * nl)(), (C.c_void_p * nl)()
        for l, (off, ids, ds) in enumerate(layers):
            off = np.ascontiguousarray(off, np.uint64)
            ids = np.ascontiguousarray(ids, np.uint32)
            ds = None if ds is None else np.ascontiguousarray(ds, np.float32)
            keep += [off, ids, ds]
            offs[l], idss[l] = off.ctypes.data, ids.ctypes.data
            dss[l] = None if ds is None else ds.ctypes.data
        self._chk(self._L.hnsw_b200_import_graph(self._h, _p(vecs), n, d, _p(origin), _p(levels), int(entry), nl, offs,
                                                 idss, dss))

    def dist_batch(self, queries, cand):
        q = np.ascontiguousarray(queries, self.dtype)
        c = np.ascontiguousarray(cand, np.uint32)
        out = np.empty(c.shape, np.float32)
        self._chk(self._L.hnsw_b200_dist_batch(self._h, _p(q), q.shape[0], q.shape[1], _p(c), c.shape[1], _p(out)))
        return out

    def bruteforce(self, queries, k):
        q = np.ascontiguousarray(queries, self.dtype)
        ids = np.empty((q.shape[0], k), np.uint32)
        ds = np.empty((q.shape[0], k), np.float32)
        self._chk(self._L.hnsw_b200_bruteforce(self._h, _p(q), q.shape[0], q.shape[1], k, _p(ids), _p(ds)))
        return ids, ds
