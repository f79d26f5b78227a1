#!/usr/bin/env python3
"""The resident BoW path (sfe_bow_assemble_dev, sfe_bowdb_query_dev, sfe_bowdb_add_dev) on one GPU, beside the host calls
it replaces.  Three legs, every result checked bit for bit:
  (1) BowVector assembly of 128 sets of ~2000 features whose words come from a synth.vocabulary k=12, L=5 tree
      (~2.2 x 10^5 words): sfe_bow_assemble_dev against sfe_bow_assemble on one host thread, set after set.
  (2) tools/bow_bench.py's workload (b): 4096 queries x 4096 entries with the dense matrix, through query_dev (vectors,
      results and matrix in device memory) and through the host query (upload, kernels, 128 MB download into pageable
      memory), alternated in one run.
  (3) A batch of 128 keyframes from resident descriptors to top-10 loop candidates against a database of 4096 entries,
      then added to it: transform_dev + bow_assemble_dev + query_dev + add_dev, against the host round trip
      (descriptors downloaded, Vocabulary.transform per keyframe, host query, host add).
  (1w) The worst case of assembly's serial sums: one set whose 16384 rows (the largest stride) all hold one word, beside
      a set of 16384 distinct words.
Descriptors are random (default_rng); through a random tree they fall on words much as image descriptors do on ORBvoc.
Call times are CUDA events on the matcher's stream around whole calls (bow_bench.gpu_ms).  query_dev's call span covers
the validation kernel, its status readback, the scoring and ranking kernels and the device-to-device copy of the dense
matrix out of scratch; the scoring and ranking kernels alone are summed from a torch.profiler trace in a separate pass.
Prints the card's name and power limit; ends with one JSON line."""
import argparse
import json
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
sys.path.insert(0, os.path.join(ROOT, "tools"))
from slam_toolkit_b200 import api, synth  # noqa: E402
import bow_oracle  # noqa: E402
from bow_bench import N_WORDS, card, gpu_ms, vectors  # noqa: E402

SETS, FEATURES = 128, 2000


def kernel_ms(fn, names, reps):
    """-> ms per call spent in the kernels whose names contain one of `names`, from a torch.profiler trace of reps calls"""
    import torch
    from torch.profiler import ProfilerActivity, profile
    torch.cuda.init()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(reps):
            fn()
        torch.cuda.synchronize()
    us = sum(e.device_time_total for e in prof.key_averages() if any(n in e.key for n in names))
    return us / 1e3 / reps


def bits_equal(a, b):
    return np.array_equal(np.asarray(a, np.float64).view(np.uint64), np.asarray(b, np.float64).view(np.uint64))


def same(res, want):
    return len(res) == len(want) and all(np.array_equal(g[0], w[0]) and bits_equal(g[1], w[1]) for g, w in zip(res, want))


def results(ent, sc, nres, q, k):
    e, s, n = ent.download((q, k), np.int32), sc.download((q, k), np.float64), nres.download((q,), np.int32)
    return [(e[i, :n[i]], s[i, :n[i]]) for i in range(q)]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=20)
    args = ap.parse_args()
    if api.device_count() < 1:
        sys.exit("no CUDA device")
    print("card:", card())
    out = {"card": card()}
    m = api.Matcher(0)
    rng = np.random.default_rng(77)
    parent, is_leaf, ndesc, weight, L = synth.vocabulary(k=12, L=5, seed=3)
    voc = api.Vocabulary(m, parent, is_leaf, ndesc, weight, L)
    n_words = voc.words()
    print(f"vocabulary: {n_words} words")

    # ---- (1) assembly ----
    stride = FEATURES + 128  # the row stride of each set, as an extractor capacity leaves it
    n = rng.integers(FEATURES - 100, FEATURES + 100, SETS).astype(np.int32)
    desc = rng.integers(0, 256, (SETS * stride, 32), dtype=np.uint8)
    d_desc, d_n = api.DeviceBuffer(desc.nbytes).upload(desc), api.DeviceBuffer(n.nbytes).upload(n)
    rows = SETS * stride
    d_wid, d_w, d_nid = api.DeviceBuffer(4 * rows), api.DeviceBuffer(8 * rows), api.DeviceBuffer(4 * rows)
    api._check(api.lib().sfe_vocab_transform_dev(m.h, voc.h, api._p(d_desc.ptr), rows, 4, api._p(d_wid.ptr), api._p(d_w.ptr),
                                                 api._p(d_nid.ptr)))
    wid, w = d_wid.download((rows,), np.int32), d_w.download((rows,), np.float64)
    d_off, d_ids, d_val = api.DeviceBuffer(8 * (SETS + 1)), api.DeviceBuffer(4 * rows), api.DeviceBuffer(8 * rows)
    dev_ms = gpu_ms(m, lambda: api.bow_assemble_dev(m, d_wid.ptr, d_w.ptr, d_n.ptr, SETS, stride, d_off.ptr, d_ids.ptr, d_val.ptr),
                    args.reps)
    t = time.perf_counter()
    for _ in range(max(1, args.reps // 4)):
        host = [api.bow_assemble(wid[i * stride:i * stride + n[i]], w[i * stride:i * stride + n[i]]) for i in range(SETS)]
    host_ms = (time.perf_counter() - t) * 1e3 / max(1, args.reps // 4)
    o = d_off.download((SETS + 1,), np.int64)
    ids, vals = d_ids.download((rows,), np.int32), d_val.download((rows,), np.float64)
    ok = bool(o[0] == 0) and same([(ids[o[i]:o[i + 1]], vals[o[i]:o[i + 1]]) for i in range(SETS)], host)
    words = int(o[-1]) / SETS
    print(f"(1) assembly, {SETS} sets x {n.mean():.0f} features ({words:.0f} words each): sfe_bow_assemble_dev {dev_ms:.3f} ms "
          f"(events)   sfe_bow_assemble, 1 host thread {host_ms:.2f} ms   bit-exact {ok}")
    out["assemble_128"] = {"dev_ms": round(dev_ms, 4), "host_1thread_ms": round(host_ms, 3),
                           "features_per_set": round(float(n.mean())), "words_per_set": round(words), "bit_exact": ok}

    # ---- (1w) one word filling the largest stride: one thread's serial chain of 16384 additions ----
    S = api.BOW_ASSEMBLE_MAX_STRIDE
    ww = rng.uniform(0.5, 1.0, S) * 10.0 ** rng.integers(-8, 8, S)
    d_ww = api.DeviceBuffer(8 * S).upload(ww)
    d_ns = api.DeviceBuffer(4).upload(np.array([S], np.int32))
    w_off, w_ids, w_val = api.DeviceBuffer(16), api.DeviceBuffer(4 * S), api.DeviceBuffer(8 * S)
    wcase, okw = {}, True
    for name, wids in (("one_word", np.full(S, 7, np.int32)), ("distinct_words", rng.permutation(S).astype(np.int32))):
        d_wi = api.DeviceBuffer(4 * S).upload(wids)
        wcase[name] = gpu_ms(m, lambda: api.bow_assemble_dev(m, d_wi.ptr, d_ww.ptr, d_ns.ptr, 1, S, w_off.ptr, w_ids.ptr, w_val.ptr),
                             args.reps)
        hi, hv = api.bow_assemble(wids, ww)
        nw = int(w_off.download((2,), np.int64)[1])
        okw &= nw == len(hi) and np.array_equal(w_ids.download((nw,), np.int32), hi) and bits_equal(w_val.download((nw,), np.float64), hv)
    print(f"(1w) one set of {S} rows: one word {wcase['one_word']:.3f} ms, {S} distinct words {wcase['distinct_words']:.3f} ms "
          f"(events)   bit-exact {okw}")
    out["assemble_worst_16384"] = {"one_word_ms": round(wcase["one_word"], 4), "distinct_words_ms": round(wcase["distinct_words"], 4),
                                   "bit_exact": bool(okw)}

    # ---- (2) workload (b) through query_dev ----
    brng = np.random.default_rng(2024)
    db = vectors(brng, 4096)
    queries = vectors(brng, 4096)
    k, q = 10, len(queries)
    bdb = api.BowDatabase(m, N_WORDS)
    bdb.add(db)
    off, qids, qvals = api.bow_csr(queries)
    c_off, c_ids, c_val = (api.DeviceBuffer(a.nbytes).upload(a) for a in (off, qids, qvals))
    ent, sc, nres = api.DeviceBuffer(4 * q * k), api.DeviceBuffer(8 * q * k), api.DeviceBuffer(4 * q)
    dense = api.DeviceBuffer(8 * q * len(db))

    def qdev():
        bdb.query_dev(c_off.ptr, c_ids.ptr, c_val.ptr, q, k, ent.ptr, sc.ptr, nres.ptr, -1, dense.ptr, len(db))

    reps_b = max(2, args.reps // 4)
    dev_b, host_b = [], []
    for _ in range(2):  # alternated: the host call and query_dev share the card's state
        dev_b.append(gpu_ms(m, qdev, reps_b))
        host_b.append(gpu_ms(m, lambda: bdb.query(queries, k, dense=True), reps_b))
    kern = kernel_ms(qdev, ("bow_score_kernel", "bow_topk_kernel"), reps_b)
    check = kernel_ms(qdev, ("bow_check_kernel",), reps_b)
    hres, hd = bdb.query(queries, k, dense=True)
    qdev()
    ifile = bow_oracle.BowIfile(db, N_WORDS)
    want = [ifile.query(v, k, -1) for v in queries[:64]]
    ok = same(results(ent, sc, nres, q, k), hres) and bits_equal(dense.download((q, len(db)), np.float64), hd) and \
        same(hres[:64], want)
    dmin, hmin = min(dev_b), min(host_b)
    print(f"(b) {q} queries x {len(db)} entries, dense: scoring + ranking kernels {kern:.2f} ms (profiler), validation kernel "
          f"{check:.3f} ms   query_dev call {dmin:.2f} ms (events; runs {[round(d, 2) for d in dev_b]})   "
          f"host query call {hmin:.2f} ms (runs {[round(d, 2) for d in host_b]})   bit-exact {ok}")
    out["b_4096x4096_dense"] = {"kernels_ms": round(kern, 3), "check_kernel_ms": round(check, 4), "query_dev_ms": round(dmin, 3),
                                "host_query_ms": round(hmin, 3), "bit_exact": ok}
    bdb.close()

    # ---- (3) 128 keyframes: resident descriptors -> top-10 candidates, then added ----
    vrng = np.random.default_rng(5)
    base = []
    for _ in range(4096):  # ~1000 distinct words of the tree per entry, L1-normalised
        ids = np.unique(vrng.integers(0, n_words, 1000)).astype(np.int32)
        v = vrng.uniform(0.05, 1.0, len(ids))
        base.append((ids, v / v.sum()))
    res3, ok3 = {}, True
    want_res = None
    for mode in ("resident", "host", "resident", "host"):
        bdb = api.BowDatabase(m, n_words)
        bdb.add(base)
        if mode == "resident":
            c_ids, c_val = api.DeviceBuffer(4 * rows), api.DeviceBuffer(8 * rows)

            def run():
                voc.transform_dev(d_desc.ptr, d_n.ptr, SETS, stride, 4, d_wid.ptr, d_w.ptr, d_nid.ptr, d_off.ptr, c_ids.ptr, c_val.ptr)
                bdb.query_dev(d_off.ptr, c_ids.ptr, c_val.ptr, SETS, k, ent.ptr, sc.ptr, nres.ptr)
                bdb.add_dev(d_off.ptr, c_ids.ptr, c_val.ptr, SETS)
        else:
            def run():
                dd = d_desc.download((SETS, stride, 32), np.uint8)
                nn = d_n.download((SETS,), np.int32)
                bows = [voc.transform(dd[i, :nn[i]])[0] for i in range(SETS)]
                r = bdb.query(bows, k)
                bdb.add(bows)
                return r
        t = time.perf_counter()
        r = run()
        ms = (time.perf_counter() - t) * 1e3
        got = results(ent, sc, nres, SETS, k) if mode == "resident" else r
        if want_res is None:
            want_res = got
        ok3 &= same(got, want_res) and len(bdb) == len(base) + SETS
        res3.setdefault(mode, []).append(ms)
        bdb.close()
    print(f"(3) {SETS} keyframes -> top-{k} of {len(base)} entries + add: resident chain {min(res3['resident']):.2f} ms "
          f"(runs {[round(x, 2) for x in res3['resident']]})   host round trip {min(res3['host']):.2f} ms "
          f"(runs {[round(x, 2) for x in res3['host']]})   bit-exact {ok3}")
    out["keyframes_128_top10"] = {"resident_ms": round(min(res3["resident"]), 3), "host_ms": round(min(res3["host"]), 3),
                                  "bit_exact": bool(ok3)}
    print(json.dumps(out))
    if not all(v["bit_exact"] for v in out.values() if isinstance(v, dict)):
        sys.exit(1)


if __name__ == "__main__":
    main()
