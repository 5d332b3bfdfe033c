"""CPU checks of pack_filters, the Python side of hnsw_b200_search_flat_filters: one id list per query packed as
(offsets[nq + 1], ids), every list sorted, or an (offsets, ids) pair passed on unchanged."""
import importlib

import numpy as np
import pytest


@pytest.fixture(scope="module")
def pack():
    return importlib.import_module("hnswlib-rs_b200.hnsw").pack_filters


def test_lists_are_sorted_and_concatenated(pack):
    off, ids = pack([[5, 1, 3], [], [7], np.array([9, 2], np.int64), (4, 4, 0)], 5)
    assert off.dtype == np.uint64 and ids.dtype == np.uint64
    assert off.tolist() == [0, 3, 3, 4, 6, 9]
    assert ids.tolist() == [1, 3, 5, 7, 2, 9, 0, 4, 4]  # repeats kept: the library allows them
    assert off.flags.c_contiguous and ids.flags.c_contiguous


def test_no_queries_and_empty_lists(pack):
    off, ids = pack([], 0)
    assert off.tolist() == [0] and len(ids) == 0
    off, ids = pack([[], []], 2)
    assert off.tolist() == [0, 0, 0] and len(ids) == 0


def test_csr_pair_is_passed_on_unchanged(pack):
    o = np.array([0, 2, 2, 5], np.int64)
    i = np.array([3, 1, 9, 8, 7], np.int64)  # not ascending: the library, not the packer, refuses it
    off, ids = pack((o, i), 3)
    assert off.dtype == np.uint64 and ids.dtype == np.uint64
    assert off.tolist() == [0, 2, 2, 5] and ids.tolist() == [3, 1, 9, 8, 7]


def test_tuple_of_lists_is_a_sequence_of_filters(pack):
    # two per-query lists given as a tuple (not numpy arrays): each list is one query's filter
    off, ids = pack(([3, 1, 2], [0]), 2)
    assert off.tolist() == [0, 3, 4] and ids.tolist() == [1, 2, 3, 0]


def test_wrong_number_of_filters_is_refused(pack):
    with pytest.raises(ValueError):
        pack([[1], [2]], 3)


@pytest.mark.parametrize("offsets,nids", [([0, 2, 2, 6], 5), ([0, 2, 2, 4], 5), ([1, 2, 2, 5], 5), ([0, 3, 2, 5], 5)])
def test_pair_that_does_not_describe_ids_is_refused(pack, offsets, nids):
    # the library cannot see len(ids): an offset past the end would make it read beyond the array
    with pytest.raises(ValueError, match="offsets"):
        pack((np.array(offsets, np.uint64), np.arange(nids, dtype=np.uint64)), 3)


def test_a_list_is_never_a_pair(pack):
    # two numpy filters of which the first holds nq + 1 = 3 ids: as a list they are two filters
    off, ids = pack([np.array([0, 2, 9], np.uint64), np.array([4, 1], np.uint64)], 2)
    assert off.tolist() == [0, 3, 5] and ids.tolist() == [0, 2, 9, 1, 4]
