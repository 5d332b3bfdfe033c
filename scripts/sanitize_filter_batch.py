"""Small per-query-filtered batch for compute-sanitizer (memcheck / racecheck): list-form and bitmap-form filters, empty
lists, ids the index does not hold, a shared-origin-id index; sizes kept tiny because the tools slow kernels down."""
import importlib, os, sys
import numpy as np
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
pkg = importlib.import_module("hnswlib-rs_b200")
n = 3000
X = pkg.datagen.clustered(n, 128, 1)
h = pkg.Hnsw(16, n, 16, 64, "DistL2")
h.insert_flat(X, ids=(np.arange(n) // 2).astype(np.uint64))
Q = pkg.datagen.clustered(64, 128, 2)
rng = np.random.default_rng(0)
lists = [[], [7], np.arange(0, n // 2, 2), rng.choice(n // 2, 46, replace=False), rng.choice(n // 2, 47, replace=False),
         np.concatenate([rng.choice(n // 2, 30, replace=False), [10**9]])]
lists += [rng.choice(n // 2, int(rng.integers(1, 400)), replace=False) for _ in range(len(Q) - len(lists))]
r = h.search_flat_filters(Q, 10, 32, lists)
assert r[4][0] == 0 and r[4][1] <= 2
for i in (2, 3, 4, 5, 40):
    s = h.search_flat(Q[i:i + 1], 10, 32, filter=lists[i])
    assert np.array_equal(s[2][0], r[2][i]) and s[4][0] == r[4][i]
d16 = pkg.Hnsw(8, 1000, 16, 40, "DistL2")
d16.insert_flat(pkg.datagen.uniform(1000, 16, 3))
d16.search_flat_filters(pkg.datagen.uniform(32, 16, 4), 5, 16, [rng.choice(1000, 20) for _ in range(32)])
print("sanitize_filter_batch ok")
