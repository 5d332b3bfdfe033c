"""bench.py host logic that needs no GPU: presets, workload naming, shard arithmetic, the committed ncu CSV reader."""
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def _parse(argv):
    import bench
    old = sys.argv
    sys.argv = ["bench.py"] + argv
    try:
        return bench, bench.parse()
    finally:
        sys.argv = old


def test_presets_match_baseline_configs():
    bench, a = _parse([])
    assert (a.config, a.n, a.d, a.nq, a.M, a.efc, a.k, a.ef, a.metric, a.custom) == ("c2", 1000000, 128, 10000, 16, 200, 10, 64, "DistL2", False)
    assert a.steps == 100 and a.warmup >= 3 and not a.strong
    assert "C2" in bench.workload_name(a) and "10000 queries/step/GPU" in bench.workload_name(a)
    _, c5 = _parse(["--config", "c5", "--gpus", "8"])
    assert c5.strong and c5.nq == 1000000 and "over 8 GPU(s) (125000/GPU)" in bench.workload_name(c5, 8)
    _, c3 = _parse(["--config", "c3"])
    assert (c3.n, c3.d, c3.M, c3.ef, c3.metric, c3.data) == (1183514, 25, 24, 128, "DistCosine", "unit")
    _, c4 = _parse(["--config", "c4"])
    assert (c4.n, c4.d, c4.M, c4.ef) == (60000, 784, 32, 200)
    _, cu = _parse(["--config", "c1", "--ef", "48"])
    assert cu.custom and "custom" in bench.workload_name(cu)


def test_steps_and_dump_arguments():
    import pytest
    _, a = _parse(["--steps", "7", "--warmup", "0", "--dump-outputs", "out"])
    assert (a.steps, a.warmup, a.dump_outputs) == (7, 0, "out")
    with pytest.raises(SystemExit):
        _parse(["--steps", "0"])


def _dump_size(d):
    return sum(f.stat().st_size for f in d.iterdir())


def test_decode_records_reads_the_kernel_layout():
    import struct
    import numpy as np
    import bench
    nq, k = 3, 2
    # Neighbour_api as the kernels write it: u64 origin id, f32 distance, the internal id in the tail padding
    raw = b"".join(struct.pack("<QfI", 1000 * q + j, q + j / 4, 7) for q in range(nq) for j in range(k))
    rec =np.frombuffer(raw, np.uint8).reshape(nq, k, 16)
    ids, ds = bench.decode_records(rec)
    assert ids.tolist() == [[1000 * q + j for j in range(k)] for q in range(nq)]
    assert ds.tolist() == [[q + j / 4 for j in range(k)] for q in range(nq)]
    pad = np.frombuffer(struct.pack("<QfI", 2 ** 64 - 1, float("inf"), 0xFFFFFFFF) * 2, np.uint8).reshape(1, 2, 16)
    ids, ds = bench.decode_records(pad)                 # the kernels' fill for slots beyond the answer count
    assert ids.tolist() == [[2 ** 64 - 1] * 2] and np.all(np.isinf(ds))


def test_step_slot_is_the_last_writer_of_its_buffer():
    import bench
    gstep, ngrp = 2, 3
    assert [bench.step_slot(i, gstep, ngrp) for i in range(7)] == [(0, 0), (0, 1), (1, 0), (1, 1), (2, 0), (2, 1), (0, 0)]
    for steps in range(1, 20):                          # no later step of the run writes the last step's slot again
        last = bench.step_slot(steps - 1, gstep, ngrp)
        assert all(bench.step_slot(i, gstep, ngrp) != last for i in range(max(0, steps - gstep * ngrp), steps - 1))


def test_dump_outputs_writes_all_rows_when_they_fit(tmp_path):
    import numpy as np
    import bench
    nq, k = 50, 4
    ids = np.arange(nq * k, dtype=np.uint64).reshape(nq, k)
    ds = np.arange(nq * k, dtype=np.float32).reshape(nq, k) / 8
    bench.dump_outputs(str(tmp_path), ids, ds, np.full(nq, k, np.int32))
    got = np.load(tmp_path / "ids.npy")
    assert got.dtype == np.float64 and np.array_equal(got, ids)
    d = np.load(tmp_path / "distances.npy")
    assert d.dtype == np.float32 and np.array_equal(d, ds)
    assert np.array_equal(np.load(tmp_path / "counts.npy"), np.full(nq, k))
    assert np.array_equal(np.load(tmp_path / "rows.npy"), np.arange(nq))


def test_dump_outputs_never_exceeds_the_limit(tmp_path, monkeypatch):
    import numpy as np
    import bench
    nq, k = 500, 4
    row = k * 8 + k * 4 + 4 + 8
    ids = np.arange(nq * k, dtype=np.uint64).reshape(nq, k)
    ds = np.arange(nq * k, dtype=np.float32).reshape(nq, k)
    cnt = np.full(nq, k, np.int32)
    monkeypatch.setattr(bench, "DUMP_LIMIT", nq * row)  # the payload alone lands exactly on the limit
    for d in ("s1", "s2"):
        bench.dump_outputs(str(tmp_path / d), ids, ds, cnt)
        assert _dump_size(tmp_path / d) <= bench.DUMP_LIMIT
    rows = np.load(tmp_path / "s1" / "rows.npy")
    assert 0 < len(rows) < nq and np.array_equal(rows, np.load(tmp_path / "s2" / "rows.npy"))   # fixed sample
    assert np.array_equal(np.load(tmp_path / "s1" / "ids.npy"), ids[rows.astype(int)])
    monkeypatch.undo()
    assert bench.DUMP_LIMIT == 64_000_000
    nq, k = 1000000, 10                                 # --config c5 on one GPU: 1 M queries in the step
    bench.dump_outputs(str(tmp_path / "c5"), np.zeros((nq, k), np.uint64), np.zeros((nq, k), np.float32),
                       np.full(nq, k, np.int32))
    assert _dump_size(tmp_path / "c5") <= 64_000_000


def test_shard_bounds_cover_the_batch():
    import bench
    for n in (0, 1, 9, 1000001):
        for w in (1, 2, 3, 8):
            b = [bench.shard_bounds(n, r, w) for r in range(w)]
            assert b[0][0] == 0 and b[-1][1] == n and all(b[i][1] == b[i + 1][0] for i in range(w - 1))
            assert max(hi - lo for lo, hi in b) - min(hi - lo for lo, hi in b) <= 1


def test_traffic_comes_from_the_committed_ncu_summary():
    bench, a = _parse([])
    t, src = bench.committed_traffic(a)
    assert src == os.path.join("profiles", "r2_search_lean_kernel_ncu_full_selected.csv")
    assert 5.4e9 < t < 7.0e9          # dram read + write of one launch, a little above the algorithmic 5.45 GB
    _, c1 = _parse(["--config", "c1"])
    assert bench.committed_traffic(c1) == (None, None)
