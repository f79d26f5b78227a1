"""Growing a resident descriptor database in place: sfe_db_append (host rows), sfe_db_append_dev (the extractor's
cap-strided device layout) and sfe_db_rows.

Every search result is compared with the oracle's knn2 over the concatenated rows (np.array_equal); where it matters, also
with a database freshly created from the same rows.  The cases cross the 128-row tile edges, the 65536-row threshold of the
tensor-core tiles and several capacity doublings; they plant appended rows as copies of queries, so that the appended rows
must enter the top-2; and they append while other matchers search, from another thread or with a search still queued.
"""
import os
import threading

import numpy as np
import pytest

from slam_toolkit_b200 import api, synth

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLDEN = os.path.join(ROOT, "tests", "golden")
NTHREADS = os.cpu_count() or 4
W, H = synth.KITTI_W, synth.KITTI_H
QS = (1, 33, 129, 300, 512)  # knn2_rows_kernel, knn2_partial_kernel or the tensor-core kernel, with and without tiles
F = 16  # KITTI-shaped stereo frames


@pytest.fixture(scope="module")
def gpu():
    if api.device_count() < 1:
        pytest.fail("no CUDA device: the product has no CPU fallback")
    return 0


def _status(call):
    with pytest.raises(api.SfeError) as e:
        call()
    return e.value.status


def _planted(rng, queries, n, flips=3):
    """n rows that are copies of random queries with 0..flips bits flipped: they must enter those queries' top-2"""
    out = queries[rng.integers(0, len(queries), n)].copy()
    for i in range(n):
        for b in rng.choice(256, int(rng.integers(0, flips + 1)), replace=False):
            out[i, b >> 3] ^= np.uint8(1 << (b & 7))
    return out


def _keys_to_quad(m, keys, shards, q):
    out = api.DeviceBuffer(q * 16)
    m.knn2_merge_dev(keys.ptr, shards, q, out.ptr)
    return out.download((q, 4), np.int32)


# ---- 1. host appends across every boundary --------------------------------------------------------------------------
PIECES = (1, 127, 128, 129, 1000, 70_000, 3, 200_000)


@pytest.mark.gpu
@pytest.mark.parametrize("start", [0, 1000])
def test_host_appends_across_boundaries(gpu, oracle, start):
    rng = np.random.default_rng(1000 + start)
    total = start + sum(PIECES)
    rows = synth.knn_database(total, seed=1001 + start)
    queries, _ = synth.knn_queries(rows, max(QS), seed=1100, hard_fraction=0.2)
    # a share of every piece copies the queries: the search must find the appended rows
    off = start
    for p in PIECES:
        k = min(p, 64)
        rows[off:off + k] = _planted(rng, queries, k)
        off += p
    m = api.Matcher(0)
    db = m.create_db(rows[:start])
    assert len(db) == start and db.rows == start
    n = start
    for p in PIECES:
        assert db.append(rows[n:n + p]) == n
        n += p
        assert len(db) == n and db.rows == n
        fresh = m.create_db(rows[:n])
        want = oracle.knn2(queries, rows[:n], nthreads=NTHREADS)
        for q in QS:
            got = m.knn2(db, queries[:q])
            assert np.array_equal(got, want[:q]), (start, n, q, int((got != want[:q]).any(axis=1).sum()))
            assert np.array_equal(m.knn2(fresh, queries[:q]), want[:q]), (start, n, q)
        fresh.close()
    assert n == total


# ---- 2. the tensor-core tiles kept current --------------------------------------------------------------------------
R4 = 4_000_000 - 50  # a partial last tile (78 of 128 rows)


@pytest.mark.gpu
@pytest.mark.parametrize("budget_gb", [None, 1.5])
def test_tiles_kept_current(gpu, oracle, budget_gb, monkeypatch):
    """A 4 M-row map whose tiles a 512-query search built; then an append that grows the capacity (the tiles follow it,
    or with a 1.5 GB budget no longer fit and are released, and a second matcher's first many-query search builds them
    again), one inside the partial last tile and one across several tiles.  The appended rows are copies of queries."""
    if budget_gb is not None:
        monkeypatch.setenv("SFE_KNN_TILES_MAX_GB", str(budget_gb))  # read when the matcher is created
    rng = np.random.default_rng(2001)
    base = synth.knn_database(R4, seed=2002)
    q, _ = synth.knn_queries(base, 512, seed=2003, hard_fraction=0.2)
    m = api.Matcher(0)
    monkeypatch.delenv("SFE_KNN_TILES_MAX_GB", raising=False)
    m2 = api.Matcher(0)
    db = m.create_db(base)
    assert np.array_equal(m.knn2(db, q), oracle.knn2(q, base, nthreads=NTHREADS))  # builds the tiles (1 GB)
    rows = base
    # growth: (R4 + 60) % 128 = 10, then 20 rows inside that tile, then 1000 rows over 8 tiles
    for piece in (60, 20, 1000):
        add = _planted(rng, q, piece, flips=2)
        assert db.append(add) == len(rows)
        rows = np.concatenate([rows, add])
        want = oracle.knn2(q, rows, nthreads=NTHREADS)
        for mm, qq in ((m2, 512), (m, 300), (m, 129)):
            got = mm.knn2(db, q[:qq])
            assert np.array_equal(got, want[:qq]), (budget_gb, len(rows), qq, int((got != want[:qq]).any(axis=1).sum()))
    assert len(db) == R4 + 1080 and db.rows == R4 + 1080


# ---- 3. device appends from the front end ---------------------------------------------------------------------------
@pytest.fixture(scope="module")
def frames(gpu):
    """F synth.stereo_pair frames through stereo_frames_dev: the device buffers, the left descriptors / counts downloaded,
    the row stride (cap)"""
    ex = api.ORBextractor(max_images=2 * F)
    pairs = [synth.stereo_pair(s) for s in range(F)]
    L = np.stack([p[0] for p in pairs])
    R = np.stack([p[1] for p in pairs])
    cap = ex.cap
    dl, dr = api.DeviceBuffer(L.nbytes).upload(L), api.DeviceBuffer(R.nbytes).upload(R)
    spec = {"kps_l": 28 * cap * F, "desc_l": 32 * cap * F, "n_l": 4 * F, "kps_r": 28 * cap * F, "desc_r": 32 * cap * F,
            "n_r": 4 * F, "stereo_idx": 4 * cap * F, "stereo_dist": 4 * cap * F}
    bufs = {k: api.DeviceBuffer(v) for k, v in spec.items()}
    ex.stereo_frames_dev(dl.ptr, dr.ptr, F, W, H, {k: b.ptr for k, b in bufs.items()})
    n = bufs["n_l"].download((F,), np.int32)
    desc = bufs["desc_l"].download((F, cap, 32), np.uint8)
    assert n.min() > 500
    return {"bufs": bufs, "n": n, "desc": desc, "cap": cap}


def _check_db(oracle, m, db, rows, seed):
    """len(db) and searches equal the oracle over `rows`: every row as a query (each must be found at its index) and a
    many-query batch"""
    assert len(db) == len(rows)
    q, _ = synth.knn_queries(rows, 512, seed=seed, hard_fraction=0.2)
    for qq in (rows, q, q[:33]):
        got = m.knn2(db, qq)
        want = oracle.knn2(qq, rows, nthreads=NTHREADS)
        assert np.array_equal(got, want), (len(rows), len(qq), int((got != want).any(axis=1).sum()))


@pytest.mark.gpu
def test_append_dev_front_end_frames(gpu, oracle, frames):
    m = api.Matcher(0)
    d, n, cap = frames["desc"], frames["n"], frames["cap"]
    pre = synth.knn_database(1000, seed=3001)
    host = np.concatenate([pre] + [d[f, :n[f]] for f in range(F)])
    # one call for the 16 frames
    db = m.create_db(pre)
    assert db.append_dev(frames["bufs"]["desc_l"].ptr, frames["bufs"]["n_l"].ptr, F, cap) == 1000
    assert db.rows == len(host)
    _check_db(oracle, m, db, host, 3002)
    # one call per frame: first_row is the rows of the frames before it
    db2 = m.create_db(pre)
    for f in range(F):
        first = db2.append_dev(frames["bufs"]["desc_l"].ptr + 32 * cap * f, frames["bufs"]["n_l"].ptr + 4 * f, 1, cap)
        assert first == 1000 + int(n[:f].sum()), f
    _check_db(oracle, m, db2, host, 3003)


@pytest.mark.gpu
def test_append_dev_layouts(gpu, oracle, frames):
    m = api.Matcher(0)
    d, cap = frames["desc"], frames["cap"]
    db = m.create_db(np.zeros((0, 32), np.uint8))
    # n_dev == NULL: 3 whole strides, rows past each frame's count included
    assert db.append_dev(frames["bufs"]["desc_l"].ptr, None, 3, cap) == 0
    rows = d[:3].reshape(-1, 32)
    _check_db(oracle, m, db, rows, 3101)
    # sets with n = 0 and n = stride, an odd stride
    rng = np.random.default_rng(3102)
    stride = 67
    src = rng.integers(0, 256, (5 * stride, 32), dtype=np.uint8)
    cnt = np.array([0, stride, 17, 0, stride], np.int32)
    d_src, d_cnt = api.DeviceBuffer(src.nbytes).upload(src), api.DeviceBuffer(cnt.nbytes).upload(cnt)
    assert db.append_dev(d_src.ptr, d_cnt.ptr, 5, stride) == len(rows)
    rows = np.concatenate([rows] + [src[i * stride:i * stride + cnt[i]] for i in range(5)])
    _check_db(oracle, m, db, rows, 3103)
    # count = 0 and all-empty sets: nothing changes
    assert db.append_dev(d_src.ptr, d_cnt.ptr, 0, stride) == len(rows)
    assert db.append_dev(d_src.ptr, d_cnt.ptr, 1, stride) == len(rows)  # cnt[0] = 0
    assert db.append(np.zeros((0, 32), np.uint8)) == len(rows)
    assert len(db) == len(rows)
    _check_db(oracle, m, db, rows, 3104)


@pytest.mark.gpu
def test_append_bad_arguments_leave_the_database_unchanged(gpu, oracle):
    m = api.Matcher(0)
    rows = synth.knn_database(70_000, seed=3201)
    q, _ = synth.knn_queries(rows, 300, seed=3202, hard_fraction=0.2)
    db = m.create_db(rows)
    before = m.knn2(db, q)
    assert np.array_equal(before, oracle.knn2(q, rows, nthreads=NTHREADS))
    stride = 64
    src = synth.knn_database(4 * stride, seed=3203)
    d_src = api.DeviceBuffer(src.nbytes + 16).upload(src)
    L = api.lib()
    for bad in (-1, stride + 1):
        cnt = np.array([stride, 5, bad, 0], np.int32)
        d_cnt = api.DeviceBuffer(cnt.nbytes).upload(cnt)
        assert _status(lambda: db.append_dev(d_src.ptr, d_cnt.ptr, 4, stride)) == api.SFE_ERR_BAD_ARG
    assert _status(lambda: db.append_dev(d_src.ptr + 8, None, 1, stride)) == api.SFE_ERR_BAD_ARG  # misaligned
    assert _status(lambda: db.append_dev(d_src.ptr, None, 1, 0)) == api.SFE_ERR_BAD_ARG           # stride < 1
    assert _status(lambda: db.append_dev(d_src.ptr, None, -1, stride)) == api.SFE_ERR_BAD_ARG     # count < 0
    assert _status(lambda: db.append_dev(None, None, 1, stride)) == api.SFE_ERR_BAD_ARG           # null rows
    assert L.sfe_db_append(m.h, db.h, None, 1, None) == api.SFE_ERR_BAD_ARG
    assert L.sfe_db_append(m.h, db.h, api._p(src), -1, None) == api.SFE_ERR_BAD_ARG
    assert L.sfe_db_append(None, db.h, api._p(src), 1, None) == api.SFE_ERR_BAD_ARG
    assert L.sfe_db_rows(None, None) == api.SFE_ERR_BAD_ARG
    assert len(db) == len(rows) and db.rows == len(rows)
    assert np.array_equal(m.knn2(db, q), before)
    # idx_base + rows would reach 2^31
    top = m.create_db(rows[:1000], idx_base=(1 << 31) - 1000 - 10)
    want_top = m.knn2(top, q)
    assert _status(lambda: top.append(src[:10])) == api.SFE_ERR_UNSUPPORTED
    assert _status(lambda: top.append_dev(d_src.ptr, None, 1, 10)) == api.SFE_ERR_UNSUPPORTED
    assert len(top) == 1000 and np.array_equal(m.knn2(top, q), want_top)
    assert top.append(src[:9]) == 1000  # idx_base + rows = 2^31 - 1: still fits
    assert len(top) == 1009


# ---- 4. global indices of a sharded map ----------------------------------------------------------------------------
@pytest.mark.gpu
def test_append_to_the_last_shard(gpu, oracle):
    rows = synth.knn_database(300_000, seed=4001)
    a, b = 120_000, 250_000
    q, _ = synth.knn_queries(rows, 512, seed=4002, hard_fraction=0.2)
    rows[b:b + 200] = _planted(np.random.default_rng(4003), q, 200)
    m = api.Matcher(0)
    s0, s1 = m.create_db(rows[:a], idx_base=0), m.create_db(rows[a:b], idx_base=a)
    assert s1.append(rows[b:b + 30_000]) == b - a
    d_tail = api.DeviceBuffer(32 * (len(rows) - b - 30_000)).upload(rows[b + 30_000:])
    assert s1.append_dev(d_tail.ptr, None, 1, len(rows) - b - 30_000) == b + 30_000 - a
    for qq in (33, 300, 512):
        d_q = api.DeviceBuffer(32 * qq).upload(q[:qq])
        keys = api.DeviceBuffer(2 * qq * 2 * 8)
        m.knn2_dev(s0, d_q.ptr, qq, keys.ptr)
        m.knn2_dev(s1, d_q.ptr, qq, keys.ptr + qq * 2 * 8)
        got = _keys_to_quad(m, keys, 2, qq)
        want = oracle.knn2(q[:qq], rows, nthreads=NTHREADS)
        assert np.array_equal(got, want), (qq, int((got != want).any(axis=1).sum()))


# ---- 5. concurrency --------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_append_while_another_thread_searches(gpu, oracle):
    """Thread 1 appends (matcher A) while thread 2 searches (matcher B).  Each search equals the oracle on one of the
    append boundaries between len(db) read before the call and after it."""
    rng = np.random.default_rng(5001)
    start = 70_000
    pieces = [int(p) for p in rng.integers(1, 20_000, 40)]
    rows = synth.knn_database(start + sum(pieces), seed=5002)
    q, _ = synth.knn_queries(rows[:start], 300, seed=5003, hard_fraction=0.2)
    bounds = [start]
    for p in pieces:  # every piece brings rows that beat some queries' current top-2
        rows[bounds[-1]:bounds[-1] + min(p, 8)] = _planted(rng, q, min(p, 8), flips=0)
        bounds.append(bounds[-1] + p)
    a, b = api.Matcher(0), api.Matcher(0)
    db = a.create_db(rows[:start])
    done = threading.Event()
    seen = []
    errors = []

    def appender():
        try:
            for i, p in enumerate(pieces):
                db.append(rows[bounds[i]:bounds[i + 1]], matcher=a)
        except Exception as e:  # noqa: BLE001 -- reported by the main thread
            errors.append(e)
        finally:
            done.set()

    def searcher():
        try:
            while not done.is_set() or len(seen) < 3:
                n0 = len(db)
                got = b.knn2(db, q)
                seen.append((n0, got, len(db)))
        except Exception as e:  # noqa: BLE001
            errors.append(e)

    ts = [threading.Thread(target=appender), threading.Thread(target=searcher)]
    for t in ts:
        t.start()
    for t in ts:
        t.join()
    assert not errors, errors
    assert len(db) == bounds[-1]
    want = {}
    for n0, got, n1 in seen:
        cands = [p for p in bounds if n0 <= p <= n1]
        assert cands, (n0, n1)
        ok = False
        for p in cands:
            if p not in want:
                want[p] = oracle.knn2(q, rows[:p], nthreads=NTHREADS)
            ok = ok or np.array_equal(got, want[p])
        assert ok, (n0, n1)
    print(f"{len(seen)} searches during {len(pieces)} appends")


IDENT = np.array([0, 0, 0, 1, 0, 0, 0], np.float64)
DIST = (-0.05, 0.01, 0.001, -0.002)


@pytest.mark.gpu
def test_append_behind_a_queued_search(gpu, oracle):
    """Matcher A queues a many-query knn2_dev behind >= 1 ms of unrelated work (ProjectionMatch calls); matcher B then
    appends: first an append that grows the buffers (rows and tiles move), then, behind a second queued search, one into
    spare capacity that rewrites the tile holding the old last row.  A's results are the oracle's on the rows from before
    each append."""
    rng = np.random.default_rng(5101)
    rows = synth.knn_database(R4, seed=5102)
    q, _ = synth.knn_queries(rows, 512, seed=5103, hard_fraction=0.2)
    a, b = api.Matcher(0), api.Matcher(0)
    db = a.create_db(rows)
    g = np.load(os.path.join(GOLDEN, "golden_seed0.npz"))
    n = 6_000_000
    z = rng.uniform(2, 80, n)
    xw = np.stack([(rng.uniform(0, W, n) - synth.KITTI_CX) / synth.KITTI_FX * z,
                   (rng.uniform(0, H, n) - synth.KITTI_CY) / synth.KITTI_FY * z, z], 1)
    d_xw = api.DeviceBuffer(xw.nbytes).upload(xw)
    d_md = api.DeviceBuffer(n * 32).upload(rng.integers(0, 256, (n, 32), dtype=np.uint8))
    mk = len(g["kl"])
    d_kp = api.DeviceBuffer(mk * 28).upload(g["kl"])
    d_kd = api.DeviceBuffer(mk * 32).upload(g["dl"])
    d_tq, d_td = api.DeviceBuffer(mk * 4), api.DeviceBuffer(mk * 4)
    d_q = api.DeviceBuffer(q.nbytes).upload(q)
    keys = api.DeviceBuffer(512 * 2 * 8)
    cam = api.Camera.make(synth.KITTI_FX, synth.KITTI_FY, synth.KITTI_CX, synth.KITTI_CY, DIST, W, H)
    # every buffer either matcher needs is allocated ahead (a device allocation may wait for the work queued so far)
    warm = synth.knn_database(R4 + 2000, seed=5104)
    for mm in (a, b):
        w = mm.create_db(warm)
        mm.knn2(w, q)
        w.close()
    a.projection_match_dev(d_xw.ptr, d_md.ptr, None, n, IDENT, cam, d_kp.ptr, d_kd.ptr, mk, 100.0, d_tq.ptr, d_td.ptr)
    assert np.array_equal(a.knn2(db, q), oracle.knn2(q, rows, nthreads=NTHREADS))  # the tiles (1 GB) are built
    # (R4 + 60) % 128 = 10: the second append writes into that tile
    for piece in (60, 40):
        add = _planted(rng, q, piece, flips=0)
        want = oracle.knn2(q, rows, nthreads=NTHREADS)
        a.set_async(True)
        e0, e1 = api.Event(0), api.Event(0)
        e0.record(a)
        for _ in range(10):
            a.projection_match_dev(d_xw.ptr, d_md.ptr, None, n, IDENT, cam, d_kp.ptr, d_kd.ptr, mk, 100.0, d_tq.ptr, d_td.ptr)
        e1.record(a)
        a.knn2_dev(db, d_q.ptr, 512, keys.ptr)
        assert db.append(add, matcher=b) == len(rows)  # on B's stream, while A's search is still queued
        a.wait()
        delay = e0.elapsed_ms(e1)
        a.set_async(False)
        got = _keys_to_quad(a, keys, 1, 512)
        print(f"append of {piece} rows behind {delay:.3f} ms of unrelated work on A's stream")
        assert np.array_equal(got, want), (piece, int((got != want).any(axis=1).sum()))
        assert delay >= 1.0, delay  # the check above only means something if B's append could overtake A's search
        rows = np.concatenate([rows, add])
        assert np.array_equal(b.knn2(db, q), oracle.knn2(q, rows, nthreads=NTHREADS)), piece
