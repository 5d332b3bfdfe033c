"""Replication paths of the C ABI (include/hnsw_b200.h "Multi-GPU search" and hnsw_b200_blob_*).

On a one-GPU box: the blob protocol (header -> alloc -> copy every blob -> commit) must reproduce the index exactly,
and the NCCL entry points are exercised with a communicator of one rank.  With two or more GPUs:
hnsw_b200_replicate + sharded search_flat / parallel_search_neighbours_f32 must return what one GPU returns."""
import ctypes

import numpy as np
import pytest

from test_gpu_search import build_pair

pytestmark = pytest.mark.gpu


def _cudart():
    import torch  # noqa: F401  (loads libcudart)
    for name in ("libcudart.so.12", "libcudart.so"):
        try:
            return ctypes.CDLL(name)
        except OSError:
            continue
    pytest.skip("libcudart not loadable")


def test_blob_roundtrip_reproduces_the_index(pkg, po):
    X, o, h = build_pair(pkg, po, 3000, 24, 12, 64, "DistL2", "clustered")
    Q = pkg.datagen.clustered(200, 24, 5)
    want = h.search_flat(Q, 8, 48)
    h2 = pkg.Hnsw(12, 3000, 16, 64, "DistL2")
    h2.blob_alloc(h.blob_header())
    rt = _cudart()
    rt.cudaMemcpy.argtypes = [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_size_t, ctypes.c_int]
    src, dst = h.blobs(), h2.blobs()
    assert len(src) == len(dst) == 9
    for (sp, sn), (dp, dn) in zip(src, dst):
        assert sn == dn
        if sn:
            assert rt.cudaMemcpy(dp, sp, sn, 3) == 0  # cudaMemcpyDeviceToDevice
    h2.blob_commit()
    assert h2.get_nb_point() == h.get_nb_point()
    got = h2.search_flat(Q, 8, 48)
    for a, b in zip(want, got):
        assert np.array_equal(a, b)  # origin ids, distances (bits), internal ids, PointIds, counts
    # the copy is a full index: its graph exports like the source's, and it accepts inserts
    for l in range(3):
        for a, b in zip(h.export_layer(l), h2.export_layer(l)):
            assert np.array_equal(a, b)
    h2.insert_flat(pkg.datagen.clustered(50, 24, 6), ids=np.arange(3000, 3050, dtype=np.uint64))
    assert h2.get_nb_point() == 3050


def test_nccl_entry_points_with_one_rank(pkg, po):
    import torch
    X, o, h = build_pair(pkg, po, 2000, 16, 8, 40, "DistL2")
    Q = pkg.datagen.uniform(64, 16, 3)
    want = h.search_flat(Q, 5, 32)
    uid = pkg.Hnsw.nccl_unique_id()
    assert uid.shape == (128,) and uid.any()
    h.nccl_init(1, 0, uid)
    h.nccl_broadcast_index(0)  # root == only rank: the index stays what it is
    got = h.search_flat(Q, 5, 32)
    for a, b in zip(want, got):
        assert np.array_equal(a, b)
    send = torch.arange(4096, dtype=torch.uint8, device="cuda")
    recv = torch.zeros(4096, dtype=torch.uint8, device="cuda")
    h.nccl_allgather(send.data_ptr(), recv.data_ptr(), 4096)
    h.check_status()  # synchronises the handle's stream
    assert torch.equal(send, recv)
    with pytest.raises(pkg.HnswError):
        pkg.Hnsw(8, 10, 16, 40, "DistL2").nccl_broadcast_index(0)  # no communicator on that handle


def test_replicate_on_one_device_is_a_no_op(pkg, po):
    X, o, h = build_pair(pkg, po, 500, 8, 8, 40, "DistL2")
    h.replicate([0])
    assert h.replica_count() == 0
    with pytest.raises(pkg.HnswError):
        h.replicate([0, 0])
    with pytest.raises(pkg.HnswError):
        h.replicate([0, 99])


def test_replicated_search_equals_one_gpu(pkg, po):
    L = pkg.load_library()
    if L.hnsw_b200_device_count() < 2:
        pytest.skip("needs two GPUs")
    ndev = min(4, L.hnsw_b200_device_count())
    X, o, h = build_pair(pkg, po, 20000, 32, 16, 100, "DistL2", "clustered")
    Q = pkg.datagen.clustered(3001, 32, 9)  # odd size: the shards differ by one
    want = h.search_flat(Q, 10, 64)
    want_f = h.search_flat(Q, 10, 64, filter=np.arange(0, 20000, 3, dtype=np.uint64))
    h.replicate(list(range(ndev)))
    assert h.replica_count() == ndev - 1
    for a, b in zip(want, h.search_flat(Q, 10, 64)):
        assert np.array_equal(a, b)
    for a, b in zip(want_f, h.search_flat(Q, 10, 64, filter=np.arange(0, 20000, 3, dtype=np.uint64))):
        assert np.array_equal(a, b)
    # submit / wait shards too: two batches in flight over all the devices
    t1 = h.submit_flat(Q, 10, 64)
    t2 = h.submit_flat(Q[::-1].copy(), 10, 64)
    for a, b in zip(want, h.wait_flat(t1)):
        assert np.array_equal(a, b)
    assert np.array_equal(h.wait_flat(t2)[2], want[2][::-1])
    par = h.parallel_search([q for q in Q], 10, 64)   # the reference's entry point, row pointers
    assert [[x.d_id for x in nb] for nb in par] == [want[0][i, :want[4][i]].tolist() for i in range(len(Q))]
    # inserting makes the copies stale; the next sharded search re-broadcasts first
    extra = pkg.datagen.clustered(500, 32, 11)
    h.insert_flat(extra, ids=np.arange(20000, 20500, dtype=np.uint64))
    got = h.search_flat(Q, 10, 64)
    h.replicate([0])
    assert h.replica_count() == 0
    for a, b in zip(h.search_flat(Q, 10, 64), got):
        assert np.array_equal(a, b)


def test_calls_leave_the_current_device_alone(pkg, po):
    """a host that tracks the current device itself (torch) must find it unchanged after replicate / search / drop"""
    import torch
    L = pkg.load_library()
    if L.hnsw_b200_device_count() < 2:
        pytest.skip("needs two GPUs")
    X, o, h = build_pair(pkg, po, 5000, 16, 8, 40, "DistL2")
    Q = pkg.datagen.uniform(512, 16, 3)
    torch.cuda.set_device(0)
    rt = _cudart()
    cur = ctypes.c_int(-1)

    def current():
        assert rt.cudaGetDevice(ctypes.byref(cur)) == 0
        return cur.value
    assert current() == 0
    h.replicate([0, 1])
    assert current() == 0
    h.search_flat(Q, 5, 32)
    assert current() == 0
    h.replicate([0])
    assert current() == 0
    del h
    assert current() == 0
