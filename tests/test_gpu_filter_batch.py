"""Per-query filters in one batch (hnsw_b200_search_flat_filters): query i searched with its own FilterT must give,
bit for bit, what a one-query search_flat(filter=L_i) gives, and what the oracle's filtered search gives on the same
graph, with both device forms of a filter (ascending internal-id list, bitmap) and the threshold between them."""
import ctypes as C

import numpy as np
import pytest

from test_gpu_search import build_pair
from util import oracle_layers

pytestmark = pytest.mark.gpu


def same(a, b):
    """the five outputs of search_flat: origin ids, distances (bit patterns), internal ids, PointIds, counts"""
    for x, y in zip(a, b):
        if x is None or y is None:
            assert x is None and y is None
        elif x.dtype == np.float32:
            assert np.array_equal(x.view(np.uint32), y.view(np.uint32))
        else:
            assert np.array_equal(x, y)


def rows(res, i):
    return tuple(None if x is None else x[i:i + 1] for x in res)


def threshold_len(n):
    return -(-n // 32)  # smallest list packed as a bitmap: 32 * len >= n


def mixed_lists(n, nq, rng):
    t = threshold_len(n)
    lists = [np.zeros(0, np.int64), np.array([1234 % n]),
             rng.choice(n, t - 1, replace=False), rng.choice(n, t, replace=False), rng.choice(n, t + 1, replace=False),
             rng.choice(n, int(0.3 * n), replace=False), np.arange(n),
             np.concatenate([rng.choice(n, 40, replace=False), 10**9 + np.arange(5)]),  # ids the index does not hold
             np.array([10**12])]
    while len(lists) < nq:
        lists.append(rng.choice(n, int(rng.integers(1, n // 4)), replace=False))
    return [np.sort(x).astype(np.uint64) for x in lists[:nq]]


@pytest.mark.parametrize("d", [16, 128])
@pytest.mark.parametrize("dense", [False, True])
def test_one_list_for_every_query_equals_batch_filter(pkg, po, d, dense):
    n = 3000
    X, o, h = build_pair(pkg, po, n, d, 8, 64, "DistL2", "clustered")
    Q = pkg.datagen.clustered(150, d, 4)
    allow = np.arange(0, n, 3 if dense else 97, dtype=np.uint64)
    assert (32 * len(allow) >= n) == dense
    want = h.search_flat(Q, 10, 48, filter=allow)
    got = h.search_flat_filters(Q, 10, 48, [allow] * len(Q))
    same(got, want)
    assert want[4].sum() > 0


def test_distinct_lists_in_one_batch(pkg, po):
    n = 3000
    X, o, h = build_pair(pkg, po, n, 16, 8, 64, "DistL2")
    Q = pkg.datagen.uniform(40, 16, 5)
    L = mixed_lists(n, len(Q), np.random.default_rng(3))
    got = h.search_flat_filters(Q, 10, 48, L)
    for i in range(len(Q)):
        same(rows(got, i), h.search_flat(Q[i:i + 1], 10, 48, filter=L[i]))
    assert got[4][0] == 0 and got[4][1] <= 1 and got[4].sum() > 0
    # the same batch as an (offsets, ids) pair
    off = np.concatenate([[0], np.cumsum([len(x) for x in L])]).astype(np.uint64)
    same(h.search_flat_filters(Q, 10, 48, (off, np.concatenate(L))), got)


def test_repeated_origin_ids_admit_every_copy(pkg):
    n, d = 2000, 16
    X = pkg.datagen.uniform(n, d, 7)
    origin = (np.arange(n) // 2).astype(np.uint64)  # points 2j and 2j + 1 share origin id j
    h = pkg.Hnsw(8, n, 16, 64, "DistL2")
    h.insert_flat(X, ids=origin)
    rng = np.random.default_rng(9)
    sel = rng.choice(n // 2, 60, replace=False)
    # query = the vector of one copy, filter = that origin id alone: the copy itself must be found at distance 0
    pts = np.concatenate([2 * sel[:30], 2 * sel[30:] + 1])
    L = [np.array([j], np.uint64) for j in np.concatenate([sel[:30], sel[30:]])]
    got = h.search_flat_filters(X[pts], 4, 64, L)
    for i in range(len(pts)):
        same(rows(got, i), h.search_flat(X[pts[i]][None, :], 4, 64, filter=L[i]))
    assert np.all(got[4] <= 2)
    assert np.mean(got[2][:, 0] == pts) >= 0.9  # both even and odd copies are admitted
    for i in range(len(pts)):
        assert set(got[0][i, :got[4][i]].tolist()) <= {int(L[i][0])}
    # mixed lists over the shared origin ids
    L2 = mixed_lists(n // 2, 30, rng)
    got2 = h.search_flat_filters(X[:30], 10, 48, L2)
    for i in range(30):
        same(rows(got2, i), h.search_flat(X[i:i + 1], 10, 48, filter=L2[i]))


def _oracle_rows(o, Q, k, ef, L):
    for i in range(len(Q)):
        yield i, o.search_batch(Q[i:i + 1], k, ef, filter_ids=L[i])


def test_matches_oracle_per_query(pkg, po):
    n = 3000
    X, o, h = build_pair(pkg, po, n, 16, 8, 64, "DistL2")
    Q = pkg.datagen.uniform(30, 16, 6)
    L = mixed_lists(n, len(Q), np.random.default_rng(4))
    for k, ef in ((10, 64), (1, 1)):
        go, gd, gi, _, gc = h.search_flat_filters(Q, k, ef, L)
        for i, (oo, od, oi, _, oc) in _oracle_rows(o, Q, k, ef, L):
            assert gc[i] == oc[0], (k, ef, i)
            assert np.array_equal(gi[i], oi[0]) and np.array_equal(go[i], oo[0]), (k, ef, i)
            assert np.array_equal(gd[i].view(np.uint32), od[0].view(np.uint32)), (k, ef, i)


def test_matches_oracle_on_tie_heavy_metric(pkg, po):
    n, d = 2000, 32
    rng = np.random.default_rng(11)
    X = rng.integers(0, 3, (n, d)).astype(np.uint8)
    Q = rng.integers(0, 3, (24, d)).astype(np.uint8)
    o = po.Oracle(8, n, 16, 64, "DistHamming", d, dtype=np.uint8, mode=po.MODE_DET, order=po.ORDER_GPU)
    o.insert_batch(X)
    lv, rk, og = o.export_points()
    h = pkg.Hnsw(8, n, 16, 64, "DistHamming", dtype=np.uint8)
    h.import_graph(X, og, lv, o.entry, oracle_layers(o))
    L = mixed_lists(n, len(Q), rng)
    for k, ef in ((10, 32), (5, 8), (1, 1)):
        go, gd, gi, _, gc = h.search_flat_filters(Q, k, ef, L)
        for i, (oo, od, oi, _, oc) in _oracle_rows(o, Q, k, ef, L):
            assert gc[i] == oc[0] and np.array_equal(gi[i], oi[0]), (k, ef, i)
            assert np.array_equal(gd[i].view(np.uint32), od[0].view(np.uint32)), (k, ef, i)


def test_traversal_counters_equal_the_single_query_calls(pkg, po):
    n = 3000
    X, o, h = build_pair(pkg, po, n, 16, 8, 64, "DistL2")
    Q = pkg.datagen.uniform(32, 16, 8)
    L = mixed_lists(n, len(Q), np.random.default_rng(5))
    # the counters include a launch that a visited-table overflow re-runs (the whole batch, or the one query, with grown
    # tables): a first call grows the tables, so that neither side below overflows
    h.search_flat_filters(Q, 10, 48, L)
    h.enable_stats(True)
    h.get_stats(reset=True)
    h.search_flat_filters(Q, 10, 48, L)
    batched = h.get_stats(reset=True)
    for i in range(len(Q)):
        h.search_filter(Q[i], 10, 48, filter=L[i].tolist())
    single = h.get_stats(reset=True)
    h.enable_stats(False)
    for key in ("evals", "expansions", "adj_read", "queries"):
        assert batched[key] == single[key], key
    assert batched["evals"] > 0


def test_reference_filter_assertions(pkg, po):
    """tests/filtertest.rs:258, 263-269 of the reference: an empty filter gives no hit; a filter admitting one id gives
    at most one hit, and it is that id"""
    n = 3000
    X, o, h = build_pair(pkg, po, n, 16, 8, 64, "DistL2")
    Q = pkg.datagen.uniform(50, 16, 9)
    admit = np.random.default_rng(6).choice(n, len(Q))
    res = h.parallel_search_filter(list(Q), 10, 64, [[] if i % 2 else [int(admit[i])] for i in range(len(Q))])
    assert len(res) == len(Q)
    for i, nb in enumerate(res):
        if i % 2:
            assert nb == []
        else:
            assert len(nb) <= 1 and all(x.d_id == admit[i] for x in nb)
    assert sum(len(nb) for nb in res) > 0
    # Neighbour fields as search_filter returns them
    one = h.search_filter(Q[0], 10, 64, filter=[int(admit[0])])
    assert [(x.d_id, x.distance, x.p_id) for x in one] == [(x.d_id, x.distance, x.p_id) for x in res[0]]


def test_translation_follows_inserts(pkg):
    n, d, extra = 2000, 16, 300
    X = pkg.datagen.uniform(n + extra, d, 12)
    h = pkg.Hnsw(8, n + extra, 16, 64, "DistL2")
    h.insert_flat(X[:n], ids=np.arange(n, dtype=np.uint64))
    Q = X[n:n + 20] + 0.001
    old = [np.arange(0, n, 5, dtype=np.uint64)] * len(Q)
    h.search_flat_filters(Q, 5, 32, old)  # builds the origin-id table
    h.insert_flat(X[n:], ids=np.arange(10**6, 10**6 + extra, dtype=np.uint64))
    new = [np.arange(10**6, 10**6 + extra, 1 + i % 3, dtype=np.uint64) for i in range(len(Q))]
    got = h.search_flat_filters(Q, 5, 32, new)
    assert np.all(got[4] > 0)
    assert np.all(got[0][got[4][:, None] > np.arange(5)[None, :]] >= 10**6)
    for i in range(len(Q)):
        same(rows(got, i), h.search_flat(Q[i:i + 1], 5, 32, filter=new[i]))


def _raw(h, Q, k, ef, off, ids):
    nq, d = Q.shape
    o = np.empty((nq, k), np.uint64)
    ds = np.empty((nq, k), np.float32)
    cnt = np.empty(nq, np.int32)
    p = lambda a: None if a is None else a.ctypes.data_as(C.c_void_p)  # noqa: E731
    return h._L.hnsw_b200_search_flat_filters(h._h, p(Q), nq, d, k, ef, p(off), p(ids), p(o), p(ds), None, None, p(cnt))


def test_bad_input_is_refused_and_the_handle_stays_usable(pkg, po):
    n = 2000
    X, o, h = build_pair(pkg, po, n, 16, 8, 40, "DistL2")
    Q = pkg.datagen.uniform(3, 16, 13)
    u = lambda *v: np.array(v, np.uint64)  # noqa: E731
    good_off, good_ids = u(0, 2, 2, 3), u(4, 9, 7)
    want = h.search_flat_filters(Q, 5, 32, (good_off, good_ids))
    bad = [(None, good_ids, "NULL"), (u(1, 2, 2, 3), good_ids, "filter_offsets[0]"), (u(0, 2, 1, 3), good_ids, "decrease"),
           (good_off, u(9, 4, 7), "not ascending"), (good_off, None, "NULL")]
    for off, ids, msg in bad:
        assert _raw(h, Q, 5, 32, off, ids) < 0
        assert msg in pkg.hnsw.last_error(), (msg, pkg.hnsw.last_error())
        same(h.search_flat_filters(Q, 5, 32, (good_off, good_ids)), want)
    with pytest.raises(pkg.HnswError, match="NULL"):
        h._chk(h._L.hnsw_b200_search_flat_filters(h._h, None, 3, 16, 5, 32, None, None, None, None, None, None, None))
    same(h.search_flat_filters(Q, 5, 32, (good_off, good_ids)), want)


def test_payload_too_large_to_address_is_refused(pkg):
    # 2^17 points sharing one origin id: a one-id list admits all of them and packs as a 4096-word bitmap, so
    # 2^20 such queries would need 2^32 words
    n, d = 1 << 17, 4
    h = pkg.Hnsw(4, n, 16, 16, "DistL2")
    h.insert_flat(pkg.datagen.uniform(n, d, 14), ids=np.zeros(n, np.uint64))
    nq = 1 << 20
    Q = np.zeros((nq, d), np.float32)
    off = np.arange(nq + 1, dtype=np.uint64)
    assert _raw(h, Q, 1, 8, off, np.zeros(nq, np.uint64)) < 0
    assert "2^32" in pkg.hnsw.last_error()
    got = h.search_flat_filters(Q[:4], 1, 8, [[0]] * 4)
    assert np.all(got[4] == 1)


def test_replicated_per_query_search_equals_one_gpu(pkg, po):
    L = pkg.load_library()
    if L.hnsw_b200_device_count() < 2:
        pytest.skip("needs two GPUs")
    ndev = min(4, L.hnsw_b200_device_count())
    n = 20000
    X, o, h = build_pair(pkg, po, n, 32, 16, 100, "DistL2", "clustered")
    Q = pkg.datagen.clustered(64 * ndev + 37, 32, 9)
    lists = mixed_lists(n, len(Q), np.random.default_rng(10))
    want = h.search_flat_filters(Q, 10, 64, lists)
    h.replicate(list(range(ndev)))
    assert h.replica_count() == ndev - 1
    same(h.search_flat_filters(Q, 10, 64, lists), want)
    h.replicate([0])
