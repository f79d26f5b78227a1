#!/usr/bin/env python3
"""BoW database query (DBoW2 L1, sfe_bowdb_query) on one GPU against the C oracle (tests/cpp/bow_oracle.c) on the host cores.

Vectors are shaped like ORBvoc.txt output: word ids from a 10^6-word space, about 1000 words per vector, L1-normalised
values (default_rng).  Two workloads:
  (a) one query against 5 000 and 100 000 resident entries (loop-candidate query of a keyframe), ms per query;
  (b) 4096 queries x 4096 entries with the dense similarity matrix (offline loop-detection evaluation): ms per call and
      word comparisons per second, counted as queries x the words of all entries (each entry word is looked up in the
      query once).
GPU times are CUDA events on the matcher's stream around whole host calls: query upload, kernels, result download.  The
5 000-entry database (60 MB) fits the 126 MB L2, the 100 000-entry one (1.2 GB) does not.  The oracle keeps DBoW2's
inverted file resident, as the reference's Database does, and times queryL1 alone; (b) runs it on every host core.
Prints the card's name and power limit; ends with one JSON line."""
import argparse
import concurrent.futures as cf
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
from slam_toolkit_b200 import api  # noqa: E402
import bow_oracle  # noqa: E402

N_WORDS = 1_000_000


def vectors(rng, count, words=1000):
    out = []
    for _ in range(count):
        ids = np.unique(rng.integers(0, N_WORDS, int(words * 1.1)))[:int(rng.integers(words - 100, words + 100))]
        w = rng.uniform(0.05, 1.0, len(ids))
        out.append((ids.astype(np.int32), w / w.sum()))
    return out


def card():
    try:
        return subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                              text=True, timeout=30).stdout.strip().splitlines()[0]
    except Exception as e:  # noqa: BLE001 -- reported, not fatal
        return f"unknown ({e})"


def gpu_ms(m, fn, reps):
    fn()
    e0, e1 = api.Event(0), api.Event(0)
    e0.record(m)
    for _ in range(reps):
        fn()
    e1.record(m)
    return e0.elapsed_ms(e1) / reps


def same(gpu_res, want):
    return all(np.array_equal(g[0], w[0]) and np.array_equal(g[1].view(np.uint64), w[1].view(np.uint64)) for g, w in zip(gpu_res, want))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--k", type=int, default=10, help="max_results of the ranked query")
    args = ap.parse_args()
    if api.device_count() < 1:
        sys.exit("no CUDA device")
    print("card:", card())
    rng = np.random.default_rng(2024)
    t0 = time.time()
    db = vectors(rng, 100_000)
    queries = vectors(rng, 4096)
    print(f"vectors generated in {time.time() - t0:.1f} s; {sum(len(v[0]) for v in db) / len(db):.0f} words per entry")
    m = api.Matcher(0)
    out = {"card": card(), "k": args.k}

    for n in (5000, 100_000):
        bdb = api.BowDatabase(m, N_WORDS)
        bdb.add(db[:n])
        q = [queries[0]]
        ms = gpu_ms(m, lambda: bdb.query(q, args.k), args.reps)
        ifile = bow_oracle.BowIfile(db[:n], N_WORDS)
        ifile.query(q[0], args.k)
        t = time.perf_counter()
        for _ in range(args.reps):
            want = ifile.query(q[0], args.k)
        host_ms = (time.perf_counter() - t) * 1e3 / args.reps
        ok = same(bdb.query(q, args.k), [want])
        print(f"(a) 1 query x {n:6d} entries: GPU {ms:8.3f} ms/query   oracle (1 host thread) {host_ms:8.3f} ms/query   "
              f"bit-exact {ok}")
        out[f"a_{n}"] = {"gpu_ms": round(ms, 4), "oracle_ms": round(host_ms, 4), "bit_exact": ok}
        bdb.close()

    n = 4096
    bdb = api.BowDatabase(m, N_WORDS)
    bdb.add(db[:n])
    comparisons = len(queries) * sum(len(v[0]) for v in db[:n])
    ms = gpu_ms(m, lambda: bdb.query(queries, args.k, dense=True), max(2, args.reps // 4))
    res, dense = bdb.query(queries, args.k, dense=True)
    ifile = bow_oracle.BowIfile(db[:n], N_WORDS)
    threads = os.cpu_count() or 1
    t = time.perf_counter()
    with cf.ThreadPoolExecutor(threads) as ex:  # ctypes releases the GIL: one query per host core at a time
        want = list(ex.map(lambda v: ifile.query(v, args.k, -1, dense=True), queries))
    host_ms = (time.perf_counter() - t) * 1e3
    ok = same(res, want) and all(np.array_equal(dense[i].view(np.uint64), w[2].view(np.uint64)) for i, w in enumerate(want))
    print(f"(b) {len(queries)} queries x {n} entries, dense: GPU {ms:8.2f} ms ({comparisons / (ms / 1e3) / 1e9:.1f} G word "
          f"comparisons/s, {comparisons:.3g} per call)   oracle ({threads} host threads) {host_ms:8.1f} ms   bit-exact {ok}")
    out["b_4096x4096_dense"] = {"gpu_ms": round(ms, 3), "word_comparisons": comparisons,
                                "gpu_word_comparisons_per_s": round(comparisons / (ms / 1e3)), "oracle_ms": round(host_ms, 1),
                                "oracle_threads": threads, "bit_exact": ok}
    print(json.dumps(out))
    if not all(v["bit_exact"] for k, v in out.items() if isinstance(v, dict)):
        sys.exit(1)


if __name__ == "__main__":
    main()
