"""The resident BoW path: BowVector assembly on the device (sfe_bow_assemble_dev) and the BoW database fed and queried from
device memory (sfe_bowdb_add_dev / sfe_bowdb_query_dev).

Assembly is compared with the host sfe_bow_assemble set by set, offsets included; the database calls with the host calls
and with the C oracle (tests/cpp/bow_oracle.c).  Every double is compared by its bits.
"""
import threading

import numpy as np
import pytest

from slam_toolkit_b200 import api, synth

import bow_oracle
from test_bow_database import _bits, _near_copy, _rand_bow, _small_case

needs_gpu = pytest.mark.gpu
F = 16  # KITTI-shaped stereo frames of the resident pipeline tests


@pytest.fixture(scope="module")
def dev():
    if api.device_count() < 1:
        pytest.fail("no CUDA device: the product has no CPU fallback")
    return 0


@pytest.fixture(scope="module")
def matcher(dev):
    return api.Matcher(dev)


@pytest.fixture(scope="module")
def frames(dev):
    """F synth.stereo_pair frames through stereo_frames_dev: the device buffers, the downloaded left descriptors / counts and
    the extractor's row stride (cap)"""
    ex = api.ORBextractor(max_images=2 * F)
    pairs = [synth.stereo_pair(s) for s in range(F)]
    L = np.stack([p[0] for p in pairs])
    R = np.stack([p[1] for p in pairs])
    h, w = L.shape[1:]
    cap = ex.cap
    dl, dr = api.DeviceBuffer(L.nbytes).upload(L), api.DeviceBuffer(R.nbytes).upload(R)
    spec = {"kps_l": 28 * cap * F, "desc_l": 32 * cap * F, "n_l": 4 * F, "kps_r": 28 * cap * F, "desc_r": 32 * cap * F,
            "n_r": 4 * F, "stereo_idx": 4 * cap * F, "stereo_dist": 4 * cap * F}
    bufs = {k: api.DeviceBuffer(v) for k, v in spec.items()}
    ex.stereo_frames_dev(dl.ptr, dr.ptr, F, w, h, {k: b.ptr for k, b in bufs.items()})
    n = bufs["n_l"].download((F,), np.int32)
    desc = bufs["desc_l"].download((F, cap, 32), np.uint8)
    assert n.min() > 500
    return {"bufs": bufs, "n": n, "desc": desc, "cap": cap, "L": L, "R": R, "ex": ex}


TREES = ((10, 4, 7), (3, 6, 8), (20, 2, 9))  # the trees of test_gpu_parity.py::test_bow_transform_vs_oracle


# ---- helpers ---------------------------------------------------------------------------------------------------------

def _assemble_dev(m, wid_ptr, w_ptr, n_ptr, count, stride, weighting, norm):
    """sfe_bow_assemble_dev -> (offsets, ids, values) downloaded"""
    off = api.DeviceBuffer(8 * (count + 1))
    ids, vals = api.DeviceBuffer(4 * count * stride), api.DeviceBuffer(8 * count * stride)
    api.bow_assemble_dev(m, wid_ptr, w_ptr, n_ptr, count, stride, off.ptr, ids.ptr, vals.ptr, weighting, norm)
    o = off.download((count + 1,), np.int64)
    return o, ids.download((count * stride,), np.int32)[:o[-1]], vals.download((count * stride,), np.float64)[:o[-1]]


def _check_assembly(got, wid, w, n, stride, weighting, norm):
    """the device CSR equals api.bow_assemble over each set's rows, offsets included"""
    off, ids, vals = got
    assert off[0] == 0
    for i in range(len(n)):
        a = i * stride
        hi, hv = api.bow_assemble(wid[a:a + n[i]], w[a:a + n[i]], weighting, norm)
        assert off[i + 1] - off[i] == len(hi), (i, weighting, norm)
        assert np.array_equal(ids[off[i]:off[i + 1]], hi), (i, weighting, norm)
        assert np.array_equal(_bits(vals[off[i]:off[i + 1]]), _bits(hv)), (i, weighting, norm)


def _assemble_all(m, wid, w, n, stride):
    """uploads one strided input and checks all 4 weightings x 3 norms against the host"""
    d_wid, d_w = api.DeviceBuffer(wid.nbytes).upload(wid), api.DeviceBuffer(w.nbytes).upload(w)
    d_n = api.DeviceBuffer(4 * len(n)).upload(np.asarray(n, np.int32))
    for weighting in range(4):
        for norm in range(3):
            got = _assemble_dev(m, d_wid.ptr, d_w.ptr, d_n.ptr, len(n), stride, weighting, norm)
            _check_assembly(got, wid, w, n, stride, weighting, norm)


class DevCsr:
    """BowVectors uploaded as one device CSR"""

    def __init__(self, vectors):
        off, ids, vals = api.bow_csr(vectors)
        self.count = len(off) - 1
        self.off = api.DeviceBuffer(off.nbytes).upload(off)
        self.ids = api.DeviceBuffer(ids.nbytes).upload(ids)
        self.val = api.DeviceBuffer(vals.nbytes).upload(vals)


def _add_dev(bdb, vectors, matcher=None):
    c = DevCsr(vectors)
    return bdb.add_dev(c.off.ptr, c.ids.ptr, c.val.ptr, c.count, matcher=matcher)


def _query_dev(bdb, vectors, k, max_id=-1, dense_entries=None, matcher=None, csr=None):
    """query_dev with every output in device memory -> (results, dense) shaped as BowDatabase.query's"""
    c = csr or DevCsr(vectors)
    q = c.count
    ent, sc, n = api.DeviceBuffer(4 * q * k), api.DeviceBuffer(8 * q * k), api.DeviceBuffer(4 * q)
    d = api.DeviceBuffer(8 * q * max(dense_entries, 1)) if dense_entries is not None else None
    bdb.query_dev(c.off.ptr, c.ids.ptr, c.val.ptr, q, k, ent.ptr, sc.ptr, n.ptr, max_id, d.ptr if d else None, dense_entries or 0,
                  matcher=matcher)
    e, s, nn = ent.download((q, k), np.int32), sc.download((q, k), np.float64), n.download((q,), np.int32)
    for i in range(q):  # the rest of a row is -1 / 0.0, as in the host call
        assert (e[i, nn[i]:] == -1).all() and (_bits(s[i, nn[i]:]) == 0).all()
    res = [(e[i, :nn[i]].copy(), s[i, :nn[i]].copy()) for i in range(q)]
    return res, (d.download((q, dense_entries), np.float64) if d else None)


def _same_results(a, b, ctx=None):
    assert len(a) == len(b)
    for (e0, s0), (e1, s1) in zip(a, b):
        assert np.array_equal(e0, e1), ctx
        assert np.array_equal(_bits(s0), _bits(s1)), ctx


def _check_query(dev_db, host_db, ifile, queries, k, max_id, dense=True):
    """query_dev on dev_db == host query on host_db == the oracle, dense matrix included"""
    n = len(dev_db)
    got, gd = _query_dev(dev_db, queries, k, max_id, dense_entries=n if dense else None)
    hq = host_db.query(queries, k, max_id, dense=dense)
    hres, hd = hq if dense else (hq, None)
    _same_results(got, hres, (k, max_id))
    for i, v in enumerate(queries):
        want = ifile.query(v, k, max_id, dense=dense)
        _same_results([got[i]], [(want[0], want[1])], (i, k, max_id))
        if dense:
            assert np.array_equal(_bits(gd[i]), _bits(want[2])), (i, k, max_id)
            assert np.array_equal(_bits(gd[i]), _bits(hd[i])), (i, k, max_id)


# ---- 1, 2: assembly --------------------------------------------------------------------------------------------------

@needs_gpu
def test_assembly_matches_host_on_real_descriptors(matcher, frames):
    """stereo_frames_dev descriptors -> sfe_vocab_transform_dev -> sfe_bow_assemble_dev == api.bow_assemble on the
    downloaded transform, for the three trees and all 12 weighting x norm pairs"""
    cap, n = frames["cap"], frames["n"]
    rows = F * cap
    d_wid, d_w, d_nid = api.DeviceBuffer(4 * rows), api.DeviceBuffer(8 * rows), api.DeviceBuffer(4 * rows)
    for (k, L, seed) in TREES:
        parent, is_leaf, ndesc, weight, L = synth.vocabulary(k=k, L=L, seed=seed)
        voc = api.Vocabulary(matcher, parent, is_leaf, ndesc, weight, L)
        assert api.lib().sfe_vocab_transform_dev(matcher.h, voc.h, api._p(frames["bufs"]["desc_l"].ptr), rows, 4,
                                                 api._p(d_wid.ptr), api._p(d_w.ptr), api._p(d_nid.ptr)) == api.SFE_OK
        wid, w = d_wid.download((rows,), np.int32), d_w.download((rows,), np.float64)
        assert (w[:n[0]] > 0).sum() > 100
        for weighting in range(4):
            for norm in range(3):
                got = _assemble_dev(matcher, d_wid.ptr, d_w.ptr, frames["bufs"]["n_l"].ptr, F, cap, weighting, norm)
                _check_assembly(got, wid, w, n, cap, weighting, norm)


def _order_sensitive_weights(rng, size):
    """weights over 16 decades: any change in the order of the additions changes bits"""
    return rng.uniform(0.5, 1.0, size) * 10.0 ** rng.integers(-8, 8, size)


@needs_gpu
def test_assembly_edge_cases(matcher):
    rng = np.random.default_rng(17)
    stride = 600
    sets = []
    sets.append((np.zeros(0, np.int32), np.zeros(0)))                                           # empty
    w = -_order_sensitive_weights(rng, 300)
    w[::3] = 0.0
    w[1::7] = np.nan
    sets.append((rng.integers(0, 50, 300).astype(np.int32), w))                                 # nothing accepted
    sets.append((np.full(stride, 42, np.int32), _order_sensitive_weights(rng, stride)))         # one word, full set
    neg = rng.integers(-40, 40, 500).astype(np.int32)
    neg[:4] = [np.iinfo(np.int32).min, np.iinfo(np.int32).max, -1, 0]
    sets.append((neg, _order_sensitive_weights(rng, 500)))                                      # negative ids
    w = _order_sensitive_weights(rng, stride)
    w[rng.integers(0, stride, 60)] = np.nan
    w[rng.integers(0, stride, 60)] = -1.0
    sets.append((rng.integers(0, 300, stride).astype(np.int32), w))                             # fills stride, mixed
    sets.append((rng.integers(0, 10 ** 6, 1).astype(np.int32), np.array([0.25])))                # one feature
    sets.append((np.zeros(0, np.int32), np.zeros(0)))                                           # empty, last
    wid = np.full(len(sets) * stride, -7, np.int32)  # rows past n[i] hold junk that must be ignored
    wts = np.full(len(sets) * stride, 3.0)
    for i, (a, b) in enumerate(sets):
        wid[i * stride:i * stride + len(a)] = a
        wts[i * stride:i * stride + len(b)] = b
    _assemble_all(matcher, wid, wts, [len(a) for a, _ in sets], stride)


@needs_gpu
def test_assembly_stride_limit_and_bad_counts(matcher):
    rng = np.random.default_rng(23)
    S = api.BOW_ASSEMBLE_MAX_STRIDE
    wid = np.concatenate([rng.integers(0, 700, S), rng.permutation(S) - S // 2, rng.integers(0, 5, S)]).astype(np.int32)
    w = _order_sensitive_weights(rng, 3 * S)
    w[rng.integers(0, 3 * S, 500)] = 0.0
    _assemble_all(matcher, wid, w, [S, S, S - 1], S)  # the largest stride, sets filling it
    d_wid, d_w = api.DeviceBuffer(4 * 2 * (S + 1)), api.DeviceBuffer(8 * 2 * (S + 1))
    d_n = api.DeviceBuffer(8)
    off, ids, vals = api.DeviceBuffer(24), api.DeviceBuffer(4 * 2 * (S + 1)), api.DeviceBuffer(8 * 2 * (S + 1))

    def call(n, count=2, stride=S, weighting=0, norm=1, wid_ptr=d_wid.ptr):
        d_n.upload(np.asarray(n, np.int32))
        return api.lib().sfe_bow_assemble_dev(matcher.h, api._p(wid_ptr), api._p(d_w.ptr), api._p(d_n.ptr), count, stride,
                                              weighting, norm, api._p(off.ptr), api._p(ids.ptr), api._p(vals.ptr))

    d_wid.upload(np.zeros(2 * (S + 1), np.int32))
    d_w.upload(np.ones(2 * (S + 1)))
    assert call([S, 1]) == api.SFE_OK
    assert call([S + 1, 1], stride=S + 1) == api.SFE_ERR_UNSUPPORTED
    assert call([10, S + 1]) == api.SFE_ERR_BAD_ARG
    assert call([-1, 10]) == api.SFE_ERR_BAD_ARG
    assert call([5, 5], weighting=4) == api.SFE_ERR_BAD_ARG
    assert call([5, 5], norm=3) == api.SFE_ERR_BAD_ARG
    assert call([5, 5], wid_ptr=None) == api.SFE_ERR_BAD_ARG
    assert call([5, 5], count=-1) == api.SFE_ERR_BAD_ARG
    assert call([5, 5]) == api.SFE_OK  # the handle is usable after the rejected calls
    assert list(off.download((3,), np.int64)) == [0, 1, 2]
    assert call([5, 5], count=0) == api.SFE_OK
    assert off.download((1,), np.int64)[0] == 0


# ---- 3, 4, 5: the database from device memory ------------------------------------------------------------------------

@needs_gpu
@pytest.mark.parametrize("max_results", [1, 3, "size", "over"])
def test_device_add_and_query_match_host_and_oracle(matcher, max_results):
    db, queries = _small_case()
    size = len(db)
    k = {"size": size, "over": size + 7}.get(max_results, max_results)
    dev_db, host_db = api.BowDatabase(matcher, 60), api.BowDatabase(matcher, 60)
    assert _add_dev(dev_db, db[:10]) == 0
    assert dev_db.add(db[10:20]) == 10    # host and device adds mixed
    assert _add_dev(dev_db, db[20:]) == 20
    assert _add_dev(dev_db, []) == size   # an empty batch: nothing added
    host_db.add(db)
    ifile = bow_oracle.BowIfile(db, 60)
    for max_id in (-1, 0, 1, size // 2, size, -2):
        _check_query(dev_db, host_db, ifile, queries, k, max_id)
    # the host query on the device-built database, and a query without dense output
    _same_results(host_db.query(queries, k), dev_db.query(queries, k))
    _same_results(_query_dev(host_db, queries, k)[0], host_db.query(queries, k))
    assert _query_dev(dev_db, [], k)[0] == []


@needs_gpu
def test_device_growth_one_entry_at_a_time(matcher):
    rng = np.random.default_rng(9)
    n_words = 500
    db = [_rand_bow(rng, n_words, int(rng.integers(0, 60))) for _ in range(200)]
    queries = [_rand_bow(rng, n_words, 40), _near_copy(rng, db[0]), _near_copy(rng, db[150])]
    q = DevCsr(queries)
    bdb = api.BowDatabase(matcher, n_words)
    for i, v in enumerate(db):
        assert _add_dev(bdb, [v]) == i
        got, d = _query_dev(bdb, None, 5, dense_entries=i + 1, csr=q)
        ifile = bow_oracle.BowIfile(db[:i + 1], n_words)
        for j, v in enumerate(queries):
            want = ifile.query(v, 5, -1, dense=True)
            _same_results([got[j]], [(want[0], want[1])], i)
            assert np.array_equal(_bits(d[j]), _bits(want[2])), i


@needs_gpu
def test_device_query_longer_than_the_staging(matcher):
    """queries of 6000 and 4100 words: past the 4096-word shared-memory staging of the scoring kernel"""
    rng = np.random.default_rng(31)
    n_words = 1_000_000
    db = [_rand_bow(rng, n_words, int(rng.integers(200, 400))) for _ in range(2000)]
    db.append(_rand_bow(rng, n_words, 5000))
    queries = [_rand_bow(rng, n_words, 6000), _near_copy(rng, db[-1]), _rand_bow(rng, n_words, 4100), _near_copy(rng, db[7])]
    dev_db, host_db = api.BowDatabase(matcher, n_words), api.BowDatabase(matcher, n_words)
    _add_dev(dev_db, db)
    host_db.add(db)
    ifile = bow_oracle.BowIfile(db, n_words)
    _check_query(dev_db, host_db, ifile, queries, 50, -1)
    _check_query(dev_db, host_db, ifile, queries, 1024, 1500, dense=False)


@needs_gpu
def test_bad_device_input_is_rejected_and_leaves_the_database_unchanged(matcher):
    rng = np.random.default_rng(3)
    n_words = 100
    db = [_rand_bow(rng, n_words, 20) for _ in range(10)]
    bdb = api.BowDatabase(matcher, n_words)
    _add_dev(bdb, db)
    probe = [_rand_bow(rng, n_words, 30), db[4]]
    before = _query_dev(bdb, probe, 10, dense_entries=10)
    good = _rand_bow(rng, n_words, 5)
    bad = [(np.array([3, 1, 7], np.int32), np.ones(3) / 3),            # unsorted
           (np.array([1, 3, 3], np.int32), np.ones(3) / 3),            # duplicate
           (np.array([1, 3, n_words], np.int32), np.ones(3) / 3),      # out of range
           (np.array([-1, 3, 5], np.int32), np.ones(3) / 3),           # negative
           (np.array([1, 3, 5], np.int32), np.array([0.5, np.nan, 0.5])),  # not finite
           (np.array([1, 3, 5], np.int32), np.array([0.5, np.inf, 0.5]))]
    for v in bad:
        for vectors in ([v], [good, v], [v, good]):
            with pytest.raises(api.SfeError) as e:
                _add_dev(bdb, vectors)
            assert e.value.status == api.SFE_ERR_BAD_ARG
            with pytest.raises(api.SfeError) as e:
                _query_dev(bdb, vectors, 3)
            assert e.value.status == api.SFE_ERR_BAD_ARG
    c = DevCsr([good, good])
    ent, sc, n = api.DeviceBuffer(4 * 2 * 1100), api.DeviceBuffer(8 * 2 * 1100), api.DeviceBuffer(8)
    dense = api.DeviceBuffer(8 * 2 * 11)
    lib = api.lib()

    def add(off_ptr, ids_ptr=c.ids.ptr, count=2):
        return lib.sfe_bowdb_add_dev(matcher.h, bdb.h, api._p(off_ptr), api._p(ids_ptr), api._p(c.val.ptr), count, None)

    def query(off_ptr, ids_ptr=c.ids.ptr, q=2, k=5, dense_ptr=None, dense_entries=0):
        return lib.sfe_bowdb_query_dev(matcher.h, bdb.h, api._p(off_ptr), api._p(ids_ptr), api._p(c.val.ptr), q, -1, k,
                                       api._p(ent.ptr), api._p(sc.ptr), api._p(n.ptr), api._p(dense_ptr), dense_entries)

    for off in ([0, 3, 2], [1, 5, 10], [0, 5, 4], [-5, 0, 5]):  # decreasing, not starting at 0
        d_off = api.DeviceBuffer(24).upload(np.array(off, np.int64))
        assert add(d_off.ptr) == api.SFE_ERR_BAD_ARG, off
        assert query(d_off.ptr) == api.SFE_ERR_BAD_ARG, off
    assert add(None) == api.SFE_ERR_BAD_ARG
    assert add(c.off.ptr, ids_ptr=None) == api.SFE_ERR_BAD_ARG        # null ids with words to add
    assert add(c.off.ptr, count=-1) == api.SFE_ERR_BAD_ARG
    assert query(c.off.ptr, ids_ptr=None) == api.SFE_ERR_BAD_ARG
    assert query(c.off.ptr, q=-1) == api.SFE_ERR_BAD_ARG
    assert query(c.off.ptr, k=0) == api.SFE_ERR_BAD_ARG
    assert query(c.off.ptr, k=1025) == api.SFE_ERR_UNSUPPORTED
    assert query(c.off.ptr, dense_ptr=dense.ptr, dense_entries=11) == api.SFE_ERR_BAD_ARG
    assert query(c.off.ptr, dense_ptr=dense.ptr, dense_entries=-1) == api.SFE_ERR_BAD_ARG
    assert query(c.off.ptr, k=1024) == api.SFE_OK
    assert query(c.off.ptr, dense_ptr=dense.ptr, dense_entries=10) == api.SFE_OK
    assert len(bdb) == 10
    after = _query_dev(bdb, probe, 10, dense_entries=10)
    _same_results(after[0], before[0])
    assert np.array_equal(_bits(after[1]), _bits(before[1]))
    ifile = bow_oracle.BowIfile(db, n_words)
    for i, v in enumerate(probe):
        want = ifile.query(v, 10, -1, dense=True)
        _same_results([after[0][i]], [(want[0], want[1])])
        assert np.array_equal(_bits(after[1][i]), _bits(want[2]))


@needs_gpu
def test_two_matchers_on_two_threads_add_dev_and_query_dev(dev):
    """thread A grows the database with add_dev while thread B runs query_dev with max_id = the count it last observed"""
    rng = np.random.default_rng(21)
    n_words = 20000
    db = [_rand_bow(rng, n_words, int(rng.integers(100, 300))) for _ in range(1200)]
    queries = [_near_copy(rng, db[int(i)]) for i in rng.integers(0, 1200, 6)] + [_rand_bow(rng, n_words, 200)]
    ma, mb = api.Matcher(dev), api.Matcher(dev)
    bdb = api.BowDatabase(ma, n_words)
    _add_dev(bdb, db[:10], matcher=ma)
    batches = [DevCsr(db[i:i + 37]) for i in range(10, len(db), 37)]
    qcsr = DevCsr(queries)
    k = 8
    q = len(queries)
    ent, sc, nres = api.DeviceBuffer(4 * q * k), api.DeviceBuffer(8 * q * k), api.DeviceBuffer(4 * q)
    dense = api.DeviceBuffer(8 * q * len(db))
    seen, errors = [], []

    def adder():
        try:
            for b in batches:
                bdb.add_dev(b.off.ptr, b.ids.ptr, b.val.ptr, b.count, matcher=ma)
        except Exception as e:  # noqa: BLE001 -- reported below
            errors.append(e)

    def querier():
        try:
            while True:
                n = len(bdb)
                bdb.query_dev(qcsr.off.ptr, qcsr.ids.ptr, qcsr.val.ptr, q, k, ent.ptr, sc.ptr, nres.ptr, n, dense.ptr, n,
                              matcher=mb)
                seen.append((n, ent.download((q, k), np.int32), sc.download((q, k), np.float64),
                             nres.download((q,), np.int32), dense.download((q, n), np.float64)))
                if n == len(db):
                    break
        except Exception as e:  # noqa: BLE001
            errors.append(e)

    ta, tb = threading.Thread(target=adder), threading.Thread(target=querier)
    ta.start(); tb.start()
    ta.join(); tb.join()
    assert not errors, errors
    assert len(seen) >= 2 and len(bdb) == len(db)
    for n, e, s, nn, d in seen[:: max(1, len(seen) // 12)] + [seen[-1]]:
        ifile = bow_oracle.BowIfile(db[:n], n_words)
        for i, v in enumerate(queries):
            want = ifile.query(v, k, n, dense=True)
            assert np.array_equal(e[i, :nn[i]], want[0]) and np.array_equal(_bits(s[i, :nn[i]]), _bits(want[1])), n
            assert np.array_equal(_bits(d[i]), _bits(want[2])), n


# ---- 6: pixels to loop candidates without a vector crossing PCIe --------------------------------------------------------

@needs_gpu
def test_resident_keyframes_to_loop_candidates_equal_the_host_path(matcher, frames):
    cap, bufs = frames["cap"], frames["bufs"]
    parent, is_leaf, ndesc, weight, L = synth.vocabulary(k=10, L=4, seed=7)
    voc = api.Vocabulary(matcher, parent, is_leaf, ndesc, weight, L)
    n_words = voc.words()
    rows = F * cap
    d_wid, d_w, d_nid = api.DeviceBuffer(4 * rows), api.DeviceBuffer(8 * rows), api.DeviceBuffer(4 * rows)
    csr = [(api.DeviceBuffer(8 * (c + 1)), api.DeviceBuffer(4 * c * cap), api.DeviceBuffer(8 * c * cap)) for c in (12, 4)]
    for (f0, c), (off, ids, val) in zip(((0, 12), (12, 4)), csr):  # keyframes 0..11 -> database, 12..15 -> queries
        voc.transform_dev(bufs["desc_l"].ptr + 32 * cap * f0, bufs["n_l"].ptr + 4 * f0, c, cap, 4, d_wid.ptr + 4 * cap * f0,
                          d_w.ptr + 8 * cap * f0, d_nid.ptr + 4 * cap * f0, off.ptr, ids.ptr, val.ptr)
    bdb = api.BowDatabase(matcher, n_words)
    assert bdb.add_dev(csr[0][0].ptr, csr[0][1].ptr, csr[0][2].ptr, 12) == 0
    k = 10
    ent, sc, nres, dense = api.DeviceBuffer(4 * 4 * k), api.DeviceBuffer(8 * 4 * k), api.DeviceBuffer(16), api.DeviceBuffer(8 * 4 * 12)
    bdb.query_dev(csr[1][0].ptr, csr[1][1].ptr, csr[1][2].ptr, 4, k, ent.ptr, sc.ptr, nres.ptr, -1, dense.ptr, 12)
    # the all-host path on the same frames
    ex = frames["ex"]
    host = ex.stereo_frames(frames["L"], frames["R"])
    bows = [voc.transform(host["desc_l"][f, :host["n_l"][f]])[0] for f in range(F)]
    hdb = api.BowDatabase(matcher, n_words)
    hdb.add(bows[:12])
    want, wd = hdb.query(bows[12:], k, dense=True)
    e, s, nn = ent.download((4, k), np.int32), sc.download((4, k), np.float64), nres.download((4,), np.int32)
    _same_results([(e[i, :nn[i]], s[i, :nn[i]]) for i in range(4)], want)
    assert np.array_equal(_bits(dense.download((4, 12), np.float64)), _bits(wd))
    assert all(len(w[0]) > 0 for w in want)
    # and the resident BowVectors themselves equal Vocabulary.transform's
    o = csr[0][0].download((13,), np.int64)
    ids, vals = csr[0][1].download((o[-1],), np.int32), csr[0][2].download((o[-1],), np.float64)
    for f in range(12):
        assert np.array_equal(ids[o[f]:o[f + 1]], bows[f][0]) and np.array_equal(_bits(vals[o[f]:o[f + 1]]), _bits(bows[f][1]))


@needs_gpu
def test_assembly_on_two_threads_with_different_strides(dev):
    """two matchers assemble concurrently, one at the largest stride and one at a small one: the kernel's shared-memory
    opt-in is per device, and neither call may fail or disturb the other"""
    rng = np.random.default_rng(41)
    cases = []
    for stride in (api.BOW_ASSEMBLE_MAX_STRIDE, 2000):
        n = [stride, stride // 2, 0, stride - 3]
        wid = rng.integers(-50, 3000, 4 * stride).astype(np.int32)
        w = _order_sensitive_weights(rng, 4 * stride)
        d = (api.DeviceBuffer(wid.nbytes).upload(wid), api.DeviceBuffer(w.nbytes).upload(w),
             api.DeviceBuffer(16).upload(np.asarray(n, np.int32)))
        want = [api.bow_assemble(wid[i * stride:i * stride + n[i]], w[i * stride:i * stride + n[i]], 0, 1) for i in range(4)]
        cases.append((api.Matcher(dev), stride, d, want))
    errors = []

    def worker(m, stride, d, want):
        try:
            for _ in range(20):
                off, ids, vals = _assemble_dev(m, d[0].ptr, d[1].ptr, d[2].ptr, 4, stride, 0, 1)
                _same_results([(ids[off[i]:off[i + 1]], vals[off[i]:off[i + 1]]) for i in range(4)], want, stride)
        except Exception as e:  # noqa: BLE001 -- reported below
            errors.append(e)

    ts = [threading.Thread(target=worker, args=c) for c in cases]
    for t in ts:
        t.start()
    for t in ts:
        t.join()
    assert not errors, errors


@needs_gpu
def test_transform_dev_rejects_a_stride_above_the_limit_before_writing(matcher):
    parent, is_leaf, ndesc, weight, L = synth.vocabulary(k=3, L=3, seed=2)
    voc = api.Vocabulary(matcher, parent, is_leaf, ndesc, weight, L)
    S = api.BOW_ASSEMBLE_MAX_STRIDE + 1
    sentinel = np.full(S, 12345, np.int32)
    d_desc, d_n = api.DeviceBuffer(32 * S), api.DeviceBuffer(4).upload(np.array([5], np.int32))
    d_wid, d_w, d_nid = api.DeviceBuffer(4 * S).upload(sentinel), api.DeviceBuffer(8 * S), api.DeviceBuffer(4 * S)
    off, ids, vals = api.DeviceBuffer(16), api.DeviceBuffer(4 * S), api.DeviceBuffer(8 * S)
    with pytest.raises(api.SfeError) as e:
        voc.transform_dev(d_desc.ptr, d_n.ptr, 1, S, 4, d_wid.ptr, d_w.ptr, d_nid.ptr, off.ptr, ids.ptr, vals.ptr)
    assert e.value.status == api.SFE_ERR_UNSUPPORTED
    assert np.array_equal(d_wid.download((S,), np.int32), sentinel)
