"""The keyframe BoW database: DBoW2's L1 query (TemplatedDatabase::queryL1) and L1Scoring::score, bit for bit.

CPU: the C oracle (tests/cpp/bow_oracle.c: orc_bow_query_l1 / orc_bow_score_l1) against a plain-Python restatement of queryL1 and
L1Scoring::score over dicts.  GPU: sfe_bowdb_* through the Python binding and through include/sfe_adapter.hpp
(tests/cpp/bow_values.cpp), every score compared with the oracle by its bits.
"""
import atexit
import functools
import os
import shutil
import subprocess
import tempfile
import threading

import numpy as np
import pytest

from slam_toolkit_b200 import api, synth

import bow_oracle

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
DRIVER_SRC = os.path.join(ROOT, "tests", "cpp", "bow_values.cpp")
needs_gpu = pytest.mark.gpu


# ---- literal restatements (thirdparty/DBoW2/DBoW2/TemplatedDatabase.h queryL1, GeneralScoring.cpp L1Scoring::score) --

def _query_literal(db_vectors, v, max_results, max_id):
    """queryL1 over DBoW2's inverted file (word -> [(entry, value)] in add order), with Python floats (IEEE doubles);
    sorted by raw sum with equal sums in ascending entry id (T8)."""
    ifile = {}
    for e, (ids, vals) in enumerate(db_vectors):
        for w, d in zip(ids, vals):
            ifile.setdefault(int(w), []).append((e, float(d)))
    pairs = {}
    for w, qvalue in zip(v[0], v[1]):
        qvalue = float(qvalue)
        for e, dvalue in ifile.get(int(w), []):
            if e < max_id or max_id == -1:
                value = abs(qvalue - dvalue) - abs(qvalue) - abs(dvalue)
                if e in pairs:
                    pairs[e] = pairs[e] + value
                else:
                    pairs[e] = value
    ret = sorted(pairs.items(), key=lambda kv: (kv[1], kv[0]))
    if max_results > 0 and len(ret) > max_results:
        ret = ret[:max_results]
    return [(e, -s / 2.0) for e, s in ret]


def _score_literal(a, b):
    da = {int(w): float(x) for w, x in zip(*a)}
    score = 0.0
    for w, wi in zip(b[0], b[1]):
        if int(w) in da:
            vi = da[int(w)]
            wi = float(wi)
            score = score + (abs(vi - wi) - abs(vi) - abs(wi))
    return -score / 2.0


def _bits(x):
    return np.asarray(x, np.float64).view(np.uint64)


def _rand_bow(rng, n_words, n):
    ids = np.sort(rng.choice(n_words, size=n, replace=False)).astype(np.int32)
    w = rng.uniform(0.05, 1.0, n)
    return ids, w / w.sum()


def _near_copy(rng, v):
    ids, vals = v
    w = vals * rng.uniform(0.8, 1.2, len(vals))
    return ids.copy(), w / w.sum()


def _small_case(seed=0):
    """35 entries over 50 words: empty entries, duplicated entries, and queries that are empty, share no word, copy an
    entry or are random"""
    rng = np.random.default_rng(seed)
    db = [_rand_bow(rng, 50, int(rng.integers(1, 12))) for _ in range(30)]
    db[3] = (np.zeros(0, np.int32), np.zeros(0))
    db[17] = (np.zeros(0, np.int32), np.zeros(0))
    for i in (5, 9, 22, 31, 34):  # duplicates of entry 2: equal raw sums for every query
        db.insert(i, (db[2][0].copy(), db[2][1].copy()))
    queries = [(np.zeros(0, np.int32), np.zeros(0)),
               (np.array([50, 55, 59], np.int32), np.array([0.2, 0.3, 0.5])),  # no word in common with any entry
               (db[2][0].copy(), db[2][1].copy()), _near_copy(rng, db[7])]
    queries += [_rand_bow(rng, 60, int(rng.integers(1, 15))) for _ in range(8)]
    return db, queries


def _check_results(got, want):
    """got = (entries, scores) arrays, want = [(entry, score)]: ids equal, scores equal by bits"""
    ge, gs = got
    assert list(ge) == [e for e, _ in want]
    assert np.array_equal(_bits(gs), _bits([s for _, s in want]))


# ---- CPU: the oracle against the literal restatement -----------------------------------------------------------------

@pytest.mark.parametrize("max_results", [1, 3, "size", "over"])
@pytest.mark.parametrize("max_id", [-1, 0, 1, "mid", "size", -2])
def test_oracle_query_matches_literal(max_id, max_results):
    db, queries = _small_case()
    size = len(db)
    max_id = {"mid": size // 2, "size": size}.get(max_id, max_id)
    max_results = {"size": size, "over": size + 7}.get(max_results, max_results)
    ifile = bow_oracle.BowIfile(db, 60)
    for v in queries:
        _check_results(ifile.query(v, max_results, max_id), _query_literal(db, v, max_results, max_id))


def test_oracle_query_without_a_cut_matches_literal():
    """max_results <= 0: every entry that shares a word, as in DBoW2"""
    db, queries = _small_case(1)
    ifile = bow_oracle.BowIfile(db, 60)
    for v in queries:
        for k in (0, -1):
            _check_results(ifile.query(v, k, -1), _query_literal(db, v, k, -1))


def test_oracle_ties_follow_entry_order():
    db, queries = _small_case(2)
    got = bow_oracle.BowIfile(db, 60).query(queries[2], 0, -1)  # a copy of entry 2, which is duplicated five times
    assert list(got[0][:6]) == [2, 5, 9, 22, 31, 34]
    assert len(set(_bits(got[1][:6]).tolist())) == 1


def test_oracle_score_matches_literal():
    db, queries = _small_case(3)
    for a in queries:
        for b in db:
            want = _score_literal(a, b)
            got = bow_oracle.bow_score_l1(a, b)
            assert _bits(got) == _bits(want)
            if not set(a[0].tolist()) & set(b[0].tolist()):
                assert _bits(got) == _bits(-0.0)  # no common word: -0.0, sign bit included


def test_oracle_dense_row_is_the_pairwise_score():
    """the dense row of a query equals L1Scoring::score against every entry, whatever max_id"""
    db, queries = _small_case(4)
    ifile = bow_oracle.BowIfile(db, 60)
    for v in queries:
        for max_id in (-1, 0, 7):
            _, _, dense = ifile.query(v, 3, max_id, dense=True)
            want = [bow_oracle.bow_score_l1(v, b) for b in db]
            assert np.array_equal(_bits(dense), _bits(want))


# ---- GPU -------------------------------------------------------------------------------------------------------------

@pytest.fixture(scope="module")
def dev():
    if api.device_count() < 1:
        pytest.fail("no CUDA device: the product has no CPU fallback")
    return 0


@pytest.fixture(scope="module")
def matcher(dev):
    return api.Matcher(dev)


def _check_against_oracle(oracle, bdb, ifile, queries, max_results, max_id, dense=True):
    got = bdb.query(queries, max_results, max_id, dense=dense)
    res, d = got if dense else (got, None)
    for i, v in enumerate(queries):
        want = ifile.query(v, max_results, max_id, dense=dense)
        assert np.array_equal(res[i][0], want[0]), (i, max_results, max_id)
        assert np.array_equal(_bits(res[i][1]), _bits(want[1])), (i, max_results, max_id)
        if dense:
            assert np.array_equal(_bits(d[i]), _bits(want[2])), (i, max_results, max_id)


@functools.lru_cache(maxsize=None)
def _real_bows():
    """32 BowVectors of synth.stereo_pair left images through extract -> Vocabulary.transform on a k=10, L=4 vocabulary"""
    parent, is_leaf, desc, weight, L = synth.vocabulary(k=10, L=4)
    m = api.Matcher(0)
    voc = api.Vocabulary(m, parent, is_leaf, desc, weight, L)
    ex = api.ORBextractor()
    bows, descs = [], []
    for s in range(32):
        left, _ = synth.stereo_pair(s)
        _, d = ex.extract(left)
        descs.append(d)
        bows.append(voc.transform(d)[0])
    return bows, descs, voc.words(), (parent, is_leaf, desc, weight, L)


@needs_gpu
def test_real_bow_vectors(dev, matcher, oracle):
    bows, _, n_words, _ = _real_bows()
    assert min(len(b[0]) for b in bows) > 100
    bdb = api.BowDatabase(matcher, n_words)
    assert bdb.add(bows[:20]) == 0
    assert bdb.add(bows[20:]) == 20
    assert len(bdb) == 32
    ifile = bow_oracle.BowIfile(bows, n_words)
    for k in (1, 10, 32):
        for max_id in (-1, 0, 1, 16, 32, 40, -2):
            _check_against_oracle(oracle, bdb, ifile, bows, k, max_id)


@needs_gpu
def test_orbvoc_shaped_scale(dev, matcher, oracle):
    """20 000 entries of ~300 words from a 10^6-word space, 200 queries of which half are near-copies of entries"""
    rng = np.random.default_rng(11)
    n_words = 1_000_000
    db = [_rand_bow(rng, n_words, int(rng.integers(200, 400))) for _ in range(20000)]
    queries = [_rand_bow(rng, n_words, int(rng.integers(200, 400))) for _ in range(100)]
    queries += [_near_copy(rng, db[int(i)]) for i in rng.integers(0, len(db), 100)]
    queries.append(_rand_bow(rng, n_words, 6000))  # longer than the shared-memory staging of the scoring kernel
    bdb = api.BowDatabase(matcher, n_words)
    bdb.add(db)
    ifile = bow_oracle.BowIfile(db, n_words)
    _check_against_oracle(oracle, bdb, ifile, queries, 50, -1)
    _check_against_oracle(oracle, bdb, ifile, queries[::7], 1024, 12345, dense=False)


@needs_gpu
def test_ties_come_back_in_entry_order(dev, matcher, oracle):
    rng = np.random.default_rng(5)
    n_words = 2000
    v = _rand_bow(rng, n_words, 50)
    db = []
    for i in range(300):
        db.append(_rand_bow(rng, n_words, 40))
        if i % 3 == 0 and sum(1 for x in db if x[0] is v[0]) < 100:
            db.append(v)
    copies = [i for i, x in enumerate(db) if x[0] is v[0]]
    assert len(copies) == 100
    bdb = api.BowDatabase(matcher, n_words)
    bdb.add(db)
    ifile = bow_oracle.BowIfile(db, n_words)
    for k in (1, 10, 99, 100, 101, 256):
        res = bdb.query([v], k)[0]
        assert list(res[0][:min(k, 100)]) == copies[:min(k, 100)]
        _check_against_oracle(oracle, bdb, ifile, [v], k, -1)
    for max_id in (copies[40], copies[40] + 1):
        _check_against_oracle(oracle, bdb, ifile, [v], 30, max_id)
    # more candidates than SFE_BOWDB_MAX_RESULTS, all tied: the selection cuts inside the tie group
    big = api.BowDatabase(matcher, n_words)
    big.add([v] * 1500 + db)
    res = big.query([v], 1024)[0]
    assert list(res[0]) == list(range(1024))
    _check_against_oracle(oracle, big, bow_oracle.BowIfile([v] * 1500 + db, n_words), [v, db[0]], 1024, -1)


@needs_gpu
def test_growth_one_entry_at_a_time(dev, matcher, oracle):
    """past several capacity doublings of the entry and word buffers; every answer equals the oracle on that prefix"""
    rng = np.random.default_rng(9)
    n_words = 500
    db = [_rand_bow(rng, n_words, int(rng.integers(0, 60))) for _ in range(300)]
    queries = [_rand_bow(rng, n_words, 40), _near_copy(rng, db[0]), _near_copy(rng, db[150])]
    bdb = api.BowDatabase(matcher, n_words)
    for i, v in enumerate(db):
        assert bdb.add([v]) == i
        _check_against_oracle(oracle, bdb, bow_oracle.BowIfile(db[:i + 1], n_words), queries, 5, -1)


def _raw_query(m, bdb, off, ids, vals, q, max_id=-1, k=5, dense_entries=0, dense=False):
    ent = np.zeros(max(q, 1) * 1100, np.int32)
    sc = np.zeros(max(q, 1) * 1100, np.float64)
    n = np.zeros(max(q, 1), np.int32)
    d = np.zeros(max(q, 1) * max(dense_entries, 1), np.float64) if dense else None
    return api.lib().sfe_bowdb_query(m.h, bdb.h, api._p(off), api._p(ids), api._p(vals), q, max_id, k, api._p(ent), api._p(sc),
                                     api._p(n), api._p(d), dense_entries)


@needs_gpu
def test_bad_input_is_rejected_and_leaves_the_database_unchanged(dev, matcher, oracle):
    rng = np.random.default_rng(3)
    n_words = 100
    db = [_rand_bow(rng, n_words, 20) for _ in range(10)]
    bdb = api.BowDatabase(matcher, n_words)
    bdb.add(db)
    probe = [_rand_bow(rng, n_words, 30), db[4]]
    before = bdb.query(probe, 10, dense=True)
    good = _rand_bow(rng, n_words, 5)
    bad = [(np.array([3, 1, 7], np.int32), np.ones(3) / 3),            # unsorted
           (np.array([1, 3, 3], np.int32), np.ones(3) / 3),            # duplicate
           (np.array([1, 3, n_words], np.int32), np.ones(3) / 3),      # out of range
           (np.array([-1, 3, 5], np.int32), np.ones(3) / 3),           # negative
           (np.array([1, 3, 5], np.int32), np.array([0.5, np.nan, 0.5]))]  # not finite
    for v in bad:
        for vectors in ([v], [good, v]):
            with pytest.raises(api.SfeError) as e:
                bdb.add(vectors)
            assert e.value.status == api.SFE_ERR_BAD_ARG
            with pytest.raises(api.SfeError) as e:
                bdb.query(vectors, 3)
            assert e.value.status == api.SFE_ERR_BAD_ARG
    off, ids, vals = api.bow_csr([good])
    assert _raw_query(matcher, bdb, off, ids, vals, -1) == api.SFE_ERR_BAD_ARG
    assert _raw_query(matcher, bdb, off, ids, vals, 1, k=0) == api.SFE_ERR_BAD_ARG
    assert _raw_query(matcher, bdb, off, ids, vals, 1, k=-3) == api.SFE_ERR_BAD_ARG
    assert _raw_query(matcher, bdb, off, ids, vals, 1, k=1025) == api.SFE_ERR_UNSUPPORTED
    assert _raw_query(matcher, bdb, off, ids, vals, 1, k=1024) == api.SFE_OK
    assert _raw_query(matcher, bdb, off, ids, vals, 1, dense=True, dense_entries=11) == api.SFE_ERR_BAD_ARG
    assert _raw_query(matcher, bdb, off, ids, vals, 1, dense=True, dense_entries=-1) == api.SFE_ERR_BAD_ARG
    bad_off = np.array([0, 3, 2], np.int64)
    assert api.lib().sfe_bowdb_add(matcher.h, bdb.h, api._p(bad_off), api._p(ids), api._p(vals), 2, None) == api.SFE_ERR_BAD_ARG
    assert api.lib().sfe_bowdb_add(matcher.h, bdb.h, api._p(off), api._p(ids), api._p(vals), -1, None) == api.SFE_ERR_BAD_ARG
    assert len(bdb) == 10
    after = bdb.query(probe, 10, dense=True)
    assert np.array_equal(_bits(after[1]), _bits(before[1]))
    for (e0, s0), (e1, s1) in zip(before[0], after[0]):
        assert np.array_equal(e0, e1) and np.array_equal(_bits(s0), _bits(s1))
    _check_against_oracle(oracle, bdb, bow_oracle.BowIfile(db, n_words), probe, 10, -1)


@needs_gpu
def test_two_matchers_on_two_threads_share_one_database(dev, oracle):
    """thread A adds batches (growing the buffers) while thread B queries with max_id = the count it last observed"""
    rng = np.random.default_rng(21)
    n_words = 20000
    db = [_rand_bow(rng, n_words, int(rng.integers(100, 300))) for _ in range(1200)]
    queries = [_near_copy(rng, db[int(i)]) for i in rng.integers(0, 1200, 6)] + [_rand_bow(rng, n_words, 200)]
    ma, mb = api.Matcher(dev), api.Matcher(dev)
    bdb = api.BowDatabase(ma, n_words)
    bdb.add(db[:10])
    seen, errors = [], []

    def adder():
        try:
            for i in range(10, len(db), 37):
                bdb.add(db[i:i + 37], matcher=ma)
        except Exception as e:  # noqa: BLE001 -- reported below
            errors.append(e)

    def querier():
        try:
            while True:
                n = len(bdb)
                res, d = bdb.query(queries, 8, max_id=n, dense=True, dense_entries=n, matcher=mb)
                seen.append((n, res, d))
                if n == len(db):
                    break
        except Exception as e:  # noqa: BLE001
            errors.append(e)

    ta, tb = threading.Thread(target=adder), threading.Thread(target=querier)
    ta.start(); tb.start()
    ta.join(); tb.join()
    assert not errors, errors
    assert len(seen) >= 2 and len(bdb) == len(db)
    for n, res, d in seen[:: max(1, len(seen) // 12)] + [seen[-1]]:
        ifile = bow_oracle.BowIfile(db[:n], n_words)
        for i, v in enumerate(queries):
            want = ifile.query(v, 8, n, dense=True)
            assert np.array_equal(res[i][0], want[0]) and np.array_equal(_bits(res[i][1]), _bits(want[1])), n
            assert np.array_equal(_bits(d[i]), _bits(want[2])), n


# ---- the C++ adapter -------------------------------------------------------------------------------------------------

@functools.lru_cache(maxsize=None)
def _driver() -> str:
    """tests/cpp/bow_values.cpp compiled into a temporary directory, linked against the in-tree libsfe.so"""
    import __graft_entry__ as g
    if not os.path.exists(api.LIB_PATH):
        g.build()
    out = tempfile.mkdtemp(prefix="sfe_bow_values_")
    atexit.register(shutil.rmtree, out, True)
    exe = os.path.join(out, "bow_values")
    libdir = os.path.dirname(os.path.abspath(api.LIB_PATH))
    subprocess.check_call(["g++", "-std=c++14", "-O1", "-Wall", "-pthread", "-o", exe, DRIVER_SRC, api.LIB_PATH,
                           f"-Wl,-rpath,{libdir}"])
    return exe


def _write_voc(path, voc, scoring=0):
    parent, is_leaf, desc, weight, L = voc
    with open(path, "w") as f:
        f.write(f"10 {L} {scoring} 0\n")
        for i in range(1, len(parent)):
            f.write(f"{parent[i]} {int(is_leaf[i])} " + " ".join(str(int(b)) for b in desc[i]) + f" {float(weight[i])!r}\n")


def _oracle_bow(oracle, voc, d):
    """transform() + BowVector assembly (TF-IDF, L1 norm) of the oracle, in the reference's order of operations"""
    parent, is_leaf, desc, weight, L = voc
    wid, w, _ = oracle.vocab_transform(parent, is_leaf, desc, weight, L, d, 4)
    v = {}
    for k, x in zip(wid.tolist(), w.tolist()):
        if x > 0:
            v[k] = v[k] + x if k in v else x
    s = 0.0
    for k in sorted(v):
        s = s + abs(v[k])
    ids = sorted(v)
    return np.array(ids, np.int32), np.array([v[k] / s for k in ids], np.float64)


@needs_gpu
def test_adapter_database_add_and_query(dev, oracle, tmp_path):
    _, descs, n_words, voc = _real_bows()
    _write_voc(tmp_path / "voc.txt", voc)
    with open(tmp_path / "desc.bin", "wb") as f:
        f.write(np.int32(len(descs)).tobytes())
        for d in descs:
            f.write(np.int32(len(d)).tobytes() + np.ascontiguousarray(d, np.uint8).tobytes())
    params = [(1, -1), (10, -1), (32, -1), (5, 0), (5, 16), (3, -2), (40, 33)]
    (tmp_path / "queries.txt").write_text("".join(f"{k} {m}\n" for k, m in params))
    p = subprocess.run([_driver(), "query", str(tmp_path)], capture_output=True, text=True, timeout=600)
    assert p.returncode == 0, p.stdout + p.stderr
    bows = []
    for i, line in enumerate((tmp_path / "bow.txt").read_text().splitlines()):
        t = line.split()
        n = int(t[0])
        ids = np.array([int(x) for x in t[1::2]], np.int32)
        vals = np.array([int(x, 16) for x in t[2::2]], np.uint64).view(np.float64)
        assert n == len(ids)
        want = _oracle_bow(oracle, voc, descs[i])
        assert np.array_equal(ids, want[0]) and np.array_equal(_bits(vals), _bits(want[1])), i
        bows.append((ids, vals))
    ifile = bow_oracle.BowIfile(bows, n_words)
    lines = (tmp_path / "results.txt").read_text().splitlines()
    assert len(lines) == len(bows) * len(params)
    for line in lines:
        t = line.split()
        i, k, max_id, n = (int(x) for x in t[:4])
        ent = [int(x) for x in t[4::2]]
        sc = np.array([int(x, 16) for x in t[5::2]], np.uint64)
        want = ifile.query(bows[i], k, max_id)
        assert n == len(want[0]) and ent == list(want[0]), line[:80]
        assert np.array_equal(sc, _bits(want[1])), line[:80]


@needs_gpu
def test_adapter_rejects_scoring_other_than_l1(dev, tmp_path):
    _, _, _, voc = _real_bows()
    for scoring in (1, 2, 3, 4, 5):  # L2, chi-square, KL, Bhattacharyya, dot product
        _write_voc(tmp_path / "voc.txt", voc, scoring)
        p = subprocess.run([_driver(), "reject", str(tmp_path / "voc.txt")], capture_output=True, text=True, timeout=300)
        assert p.returncode == 0, p.stdout + p.stderr
        assert p.stdout.startswith("rejected=") and api.lib().sfe_status_string(api.SFE_ERR_UNSUPPORTED).decode() in p.stdout
    _write_voc(tmp_path / "voc.txt", voc, 0)
    p = subprocess.run([_driver(), "reject", str(tmp_path / "voc.txt")], capture_output=True, text=True, timeout=300)
    assert p.stdout.strip() == "accepted", p.stdout + p.stderr
