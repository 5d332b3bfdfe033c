"""Per-query filters on a C2-shape graph (1 M x 128 f32 L2 clustered, M=16, ef_c=200, built on the GPU; k=10, ef=64),
at three selectivities (30 %, 3 %, 0.3 % of the points):
  (a) hnsw_b200_search_flat_filters, a distinct random list per query (1 000 queries at 30 %, 10 000 otherwise);
  (b) hnsw_b200_search_flat with ONE list shared by all queries (the batch filter path), same queries;
  (c) one hnsw_b200_search_flat(filter=L_i) call per query, on 100 queries (what per-query filtering cost before).
A list holds frac * n ids drawn uniformly WITH replacement, sorted (repeats are allowed), so it admits slightly fewer
distinct points than frac * n.  Wall-clock is the best of 3 calls (pinned queries); kernel and host-to-device copy times
come from torch.profiler over one more call; "host" = wall - kernel: origin-id translation, packing, upload and the
unpacking of the answers.  Counters (E = evaluations, X = expansions, A = adjacency ids read, per query) from
hnsw_b200_get_stats.  Writes one JSON file (argument 1, default filter_batch.json)."""
import importlib, json, os, subprocess, sys, time
import numpy as np, torch
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
pkg = importlib.import_module("hnswlib-rs_b200")

K, EF, N, D = 10, 64, 1000000, 128


def best(fn, reps=3):
    fn()
    ts = []
    for _ in range(reps):
        t = time.perf_counter(); fn(); ts.append(time.perf_counter() - t)
    return min(ts)


def device_times(fn):
    """(search kernel ms, host-to-device copy ms) of one call, from the CUDA activity torch.profiler records"""
    from torch.profiler import ProfilerActivity, profile
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CPU, ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    kern = h2d = 0.0
    for e in prof.events():
        dt = getattr(e, "device_type", None)
        if dt is None or "CUDA" not in str(dt):
            continue
        us = e.device_time_total if hasattr(e, "device_time_total") else e.cuda_time_total
        if "search_filter_kernel" in e.name:
            kern += us
        elif "HtoD" in e.name or "Memcpy HtoD" in e.name:
            h2d += us
    return kern / 1e3, h2d / 1e3


def stats(h, fn, nq):
    h.enable_stats(True); h.get_stats(); fn(); st = h.get_stats(); h.enable_stats(False)
    return {"E": st["evals"] / nq, "X": st["expansions"] / nq, "A": st["adj_read"] / nq}


def gpu_info():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                             text=True, timeout=30).stdout.strip().splitlines()[0]
    except Exception as ex:  # noqa: BLE001
        out = f"unavailable ({ex})"
    return out


def main():
    out_path = sys.argv[1] if len(sys.argv) > 1 else "filter_batch.json"
    X = pkg.datagen.clustered(N, D, 1)
    h = pkg.Hnsw(16, N, 16, 200, "DistL2")
    t0 = time.perf_counter(); h.insert_flat(X); build_s = time.perf_counter() - t0
    del X
    Qall = torch.from_numpy(pkg.datagen.clustered(10000, D, 2)).pin_memory().numpy()
    res = {"gpu": gpu_info(), "graph": {"n": N, "d": D, "M": 16, "ef_c": 200, "metric": "DistL2", "data": "clustered",
                                        "build_s": round(build_s, 2)}, "k": K, "ef": EF, "arms": []}
    print(json.dumps(res), flush=True)
    rng = np.random.default_rng(0)
    for frac in (0.3, 0.03, 0.003):
        nq = 1000 if frac >= 0.3 else 10000
        m = int(frac * N)
        Q = Qall[:nq]
        ids = np.empty((nq, m), np.uint64)
        for b in range(0, nq, 500):
            blk = rng.integers(0, N, (min(500, nq - b), m), dtype=np.int64)
            blk.sort(axis=1)
            ids[b:b + len(blk)] = blk
        distinct = np.array([np.count_nonzero(np.diff(r.astype(np.int64)) != 0) + 1 for r in ids])
        bitmap_queries = int(np.count_nonzero(32 * distinct >= N))
        off = (np.arange(nq + 1, dtype=np.uint64) * np.uint64(m))
        flat = ids.reshape(-1)
        pair = (off, flat)
        row = {"admitted_frac": frac, "ids_per_list": m, "mean_distinct_per_list": float(distinct.mean()),
               "queries": nq, "bitmap_form_queries": bitmap_queries, "list_form_queries": nq - bitmap_queries}
        # (a) one distinct list per query
        fa = lambda: h.search_flat_filters(Q, K, EF, pair, with_pid=False)  # noqa: E731
        ra = fa()
        ta = best(fa)
        ka, ca = device_times(fa)
        row["a_per_query"] = {"wall_ms": ta * 1e3, "qps": nq / ta, "kernel_ms": ka, "h2d_ms": ca,
                              "host_ms": ta * 1e3 - ka, "mean_hits": float(ra[4].mean()), **stats(h, fa, nq)}
        print(json.dumps(row), flush=True)
        # (b) one list shared by all queries (the batch bitmap path)
        shared = ids[0].copy()
        fb = lambda: h.search_flat(Q, K, EF, filter=shared, with_pid=False)  # noqa: E731
        rb = fb()
        tb = best(fb)
        kb, cb = device_times(fb)
        row["b_shared"] = {"wall_ms": tb * 1e3, "qps": nq / tb, "kernel_ms": kb, "h2d_ms": cb, "host_ms": tb * 1e3 - kb,
                           "mean_hits": float(rb[4].mean()), **stats(h, fb, nq)}
        print(json.dumps(row["b_shared"]), flush=True)
        # (c) one search_flat(filter=L_i) call per query, 100 queries; the answers must equal (a)'s rows
        nc = 100
        t = time.perf_counter()
        rc = [h.search_flat(Q[i:i + 1], K, EF, filter=ids[i], with_pid=False) for i in range(nc)]
        tc = time.perf_counter() - t
        same = all(np.array_equal(rc[i][2][0], ra[2][i]) and np.array_equal(rc[i][1][0].view(np.uint32), ra[1][i].view(np.uint32))
                   and rc[i][4][0] == ra[4][i] for i in range(nc))
        row["c_one_call_per_query"] = {"queries": nc, "wall_ms": tc * 1e3, "qps": nc / tc, "answers_equal_a": bool(same)}
        print(json.dumps(row["c_one_call_per_query"]), flush=True)
        res["arms"].append(row)
        del ids, flat, pair
        with open(out_path, "w") as f:  # after every selectivity, so that a long run keeps what it measured
            json.dump(res, f, indent=1)
    print("wrote", out_path)


if __name__ == "__main__":
    main()
