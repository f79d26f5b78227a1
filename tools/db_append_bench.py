#!/usr/bin/env python3
"""Growing a resident descriptor map in place (sfe_db_append / sfe_db_append_dev) against rebuilding it, on one GPU.

The map holds 10 M random rows (BASELINE config 4) and its tensor-core tiles are built (a 2000-query search) before any
append is timed.  Legs:
  (1) appending one keyframe (2000 rows) and a batch of 128 keyframes (128 sets of 1900..2100 rows at a row stride of
      2128, ~256 k rows), from host memory and from device memory in the extractor's cap-strided layout:
      - into spare capacity (the map has grown once before), and
      - with growth (a fresh 10 M-row map whose capacity is exactly its rows: rows and tiles move to twice the capacity);
  (2) what a caller does without append: destroy the map, create it again from all rows in host memory, and run the first
      2000-query search, which rebuilds the tiles;
  (3) knn2_dev with 2000 queries on a map grown from 9 M to the 10 M rows by four appends (tiles built at 9 M rows) against
      the same search on the map created from the 10 M rows, alternated; the keys must be identical.
Append calls are synchronous; their times are CUDA events on the appending matcher's stream around whole calls (the
host-side allocations of a growing append fall between the events).  (2) is a host clock around synchronous calls.
Prints the card's name and power limit; ends with one JSON line."""
import argparse
import json
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))
from slam_toolkit_b200 import api, synth  # noqa: E402
from bow_bench import card  # noqa: E402

MAP, Q, KF, SETS, STRIDE = 10_000_000, 2000, 2000, 128, 2128


def event_ms(m, fn):
    e0, e1 = api.Event(0), api.Event(0)
    e0.record(m)
    r = fn()
    e1.record(m)
    m.wait()
    return e0.elapsed_ms(e1), r


def median(xs):
    return float(np.median(xs))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--growth-reps", type=int, default=3)
    args = ap.parse_args()
    if api.device_count() < 1:
        sys.exit("no CUDA device")
    print("card:", card())
    out = {"card": card(), "map_rows": MAP}
    rng = np.random.default_rng(11)
    m = api.Matcher(0)
    base = synth.knn_database(MAP, seed=12)
    queries, _ = synth.knn_queries(base, Q, seed=13, hard_fraction=0.2)
    d_q = api.DeviceBuffer(queries.nbytes).upload(queries)
    keys = api.DeviceBuffer(Q * 2 * 8)
    kf = rng.integers(0, 256, (KF, 32), dtype=np.uint8)
    batch = rng.integers(0, 256, (SETS * STRIDE, 32), dtype=np.uint8)
    n = rng.integers(1900, 2101, SETS).astype(np.int32)
    batch_rows = np.concatenate([batch[i * STRIDE:i * STRIDE + n[i]] for i in range(SETS)])
    d_kf = api.DeviceBuffer(kf.nbytes).upload(kf)
    d_batch, d_n = api.DeviceBuffer(batch.nbytes).upload(batch), api.DeviceBuffer(n.nbytes).upload(n)
    print(f"map {MAP} rows, keyframe {KF} rows, batch {SETS} sets = {len(batch_rows)} rows")

    appends = {  # name -> (host rows it adds, call)
        "kf_host": (kf, lambda db: db.append(kf)),
        "kf_dev": (kf, lambda db: db.append_dev(d_kf.ptr, None, 1, KF)),
        "batch_host": (batch_rows, lambda db: db.append(batch_rows)),
        "batch_dev": (batch_rows, lambda db: db.append_dev(d_batch.ptr, d_n.ptr, SETS, STRIDE)),
    }

    def fresh_map():
        db = m.create_db(base)
        m.knn2_dev(db, d_q.ptr, Q, keys.ptr)  # builds the tiles
        return db

    # ---- (1) appends with growth: each on a fresh map whose capacity is its rows ----
    res = {}
    for name, (_, call) in appends.items():
        ts = []
        for _ in range(args.growth_reps):
            db = fresh_map()
            t, _ = event_ms(m, lambda: call(db))
            ts.append(t)
            db.close()
        res[name + "_growth_ms"] = round(median(ts), 3)
        print(f"(1) {name:10s} with growth:     {median(ts):9.3f} ms  (median of {len(ts)}: {', '.join(f'{x:.2f}' for x in ts)})")
    # ---- (1) appends into spare capacity: the grown map, alternating the four calls ----
    db = fresh_map()
    db.append(kf)  # grows once: 20 M rows of capacity
    total = MAP + KF
    ts = {k: [] for k in appends}
    for _ in range(args.reps):
        for name, (rows, call) in appends.items():
            t, _ = event_ms(m, lambda: call(db))
            ts[name].append(t)
            total += len(rows)
    for name in appends:
        res[name + "_spare_ms"] = round(median(ts[name]), 3)
        print(f"(1) {name:10s} into spare room: {median(ts[name]):9.3f} ms  (median of {len(ts[name])})")
    out["append"] = res
    assert len(db) == total

    # ---- (2) the alternative: destroy + create + first many-query search with its tile rebuild ----
    ts = []
    for _ in range(args.growth_reps):
        other = m.create_db(base)
        m.knn2_dev(other, d_q.ptr, Q, keys.ptr)
        t = time.perf_counter()
        other.close()
        other = m.create_db(np.concatenate([base, kf]))
        m.knn2_dev(other, d_q.ptr, Q, keys.ptr)
        ts.append((time.perf_counter() - t) * 1e3)
        other.close()
    out["rebuild_ms"] = round(median(ts), 3)
    print(f"(2) destroy + create_db({MAP + KF} rows) + first {Q}-query search: {median(ts):9.3f} ms (median of {len(ts)})")

    db.close()

    # ---- (3) search on a map grown to the 10 M rows by appends against the map created from them ----
    db = m.create_db(base[:MAP - 1_000_000])
    m.knn2_dev(db, d_q.ptr, Q, keys.ptr)  # tiles, then the appends keep them current
    for i in range(4):
        db.append(base[MAP - 1_000_000 + 250_000 * i:MAP - 750_000 + 250_000 * i])
    assert len(db) == MAP
    all_rows = base
    fresh = m.create_db(base)
    k_g, k_f = api.DeviceBuffer(Q * 16), api.DeviceBuffer(Q * 16)
    m.knn2_dev(fresh, d_q.ptr, Q, k_f.ptr)
    m.knn2_dev(db, d_q.ptr, Q, k_g.ptr)
    same = bool(np.array_equal(k_g.download((Q, 2), np.uint64), k_f.download((Q, 2), np.uint64)))
    tg, tf = [], []
    for _ in range(args.reps):
        tg.append(event_ms(m, lambda: m.knn2_dev(db, d_q.ptr, Q, k_g.ptr))[0])
        tf.append(event_ms(m, lambda: m.knn2_dev(fresh, d_q.ptr, Q, k_f.ptr))[0])
    out["knn2_dev_2000q"] = {"rows": int(len(all_rows)), "grown_ms": round(median(tg), 4), "fresh_ms": round(median(tf), 4),
                             "identical": same}
    print(f"(3) knn2_dev {Q} queries x {len(all_rows)} rows: grown map {median(tg):.4f} ms, fresh map {median(tf):.4f} ms "
          f"(medians of {args.reps}), keys identical: {same}")
    print(json.dumps(out))
    if not same:
        sys.exit("grown and fresh maps disagree")


if __name__ == "__main__":
    main()
