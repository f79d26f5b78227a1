"""sfe_stereo_sequence_plan[_dev]: a motion prior per frame pair and the tracker's wide-radius retry, against the oracle's
GetDepth + ProjectionMatch run pair by pair with that pair's own prior and the two-step rule (first pass at tp.radius; fewer
than retry_below matched keypoints: again at retry_radius, which replaces it)."""
import ctypes as C

import numpy as np
import pytest

from slam_toolkit_b200 import api, synth

pytestmark = pytest.mark.gpu

B = synth.KITTI_BASELINE
INT32_MAX = 2 ** 31 - 1
# frames of synth.stereo_sequence(seed, n, step=1) at uneven canvas offsets: image shifts of 2, 9, 1, 30 and 5 px
IRREGULAR = [0, 2, 11, 12, 42, 47]
# one jump of 70 px: at radius 50 with the identity prior the oracle matches 0-2 keypoints of that pair (seeds 0-2), at
# radius 100 several hundred; the 4-px pairs match over 800 at either radius
JUMP = [0, 4, 74, 78]


@pytest.fixture(scope="module")
def gpu():
    if api.device_count() < 1:
        pytest.fail("no CUDA device: the product has no CPU fallback")
    return 0


@pytest.fixture(scope="module")
def cams(oracle):
    args = (synth.KITTI_FX, synth.KITTI_FY, synth.KITTI_CX, synth.KITTI_CY, (0, 0, 0, 0), synth.KITTI_W, synth.KITTI_H)
    return api.Camera.make(*args), oracle.make_camera(*args[:4], list(args[4]), *args[5:])


def _frames(seed, idx):
    L, R = synth.stereo_sequence(seed, max(idx) + 1, step=1)
    return np.ascontiguousarray(L[idx]), np.ascontiguousarray(R[idx])


def _shift_rt(s):
    """Tcw of an image shift of s px at the scene's uniform 24-px disparity (depth fx * B / 24)."""
    T = np.eye(4)
    T[0, 3] = -s * B / 24.0
    return T


def _shift_se3(s):
    return np.array([0.0, 0.0, 0.0, 1.0, -s * B / 24.0, 0.0, 0.0])


def _exact_priors(idx, se3=False):
    shifts = [0] + [idx[f] - idx[f - 1] for f in range(1, len(idx))]
    return np.stack([_shift_se3(s) if se3 else _shift_rt(s) for s in shifts])


def _oracle_pass(oracle, ocam, prior, radius, kl, dl, kr, si, kc, dc):
    """One ProjectionMatch of frame f-1's stereo points into frame f.  An SE3 prior goes through the parts orc_track_pair is
    made of (NormalizedUndistort, GetDepth, ProjectionMatch with the no-depth points skipped)."""
    prior = np.asarray(prior, np.float64)
    if prior.size == 7:
        xc, valid = oracle.stereo_depth(ocam, B, kl, oracle.normalized_undistort(ocam, kl), kr, si)
        return oracle.projection_match(xc, dl, valid != 1, prior, ocam, kc, dc, radius)
    return oracle.track_pair(ocam, B, prior, radius, kl, dl, kr, si, kc, dc)


def _oracle_plan(oracle, ocam, out, priors, radius, retry_radius=100.0, retry_below=0):
    """-> per pair f >= 1: (track_idx, track_dist, first-pass matches, retried) from the device's own extraction outputs."""
    res = {}
    for f in range(1, len(out["n_l"])):
        npv, nrp, nl = int(out["n_l"][f - 1]), int(out["n_r"][f - 1]), int(out["n_l"][f])
        parts = (out["kps_l"][f - 1, :npv], out["desc_l"][f - 1, :npv], out["kps_r"][f - 1, :nrp],
                 out["stereo_idx"][f - 1, :npv], out["kps_l"][f, :nl], out["desc_l"][f, :nl])
        ti, td = _oracle_pass(oracle, ocam, priors[f], radius, *parts)
        first = int((ti >= 0).sum())
        retried = first < retry_below
        if retried:
            ti, td = _oracle_pass(oracle, ocam, priors[f], retry_radius, *parts)
        res[f] = (ti, td, first, retried)
    return res


def _assert_tracks(out, ref, what=""):
    assert (out["track_idx"][0] == -1).all() and (out["track_dist"][0] == -1).all()
    for f, (ti, td, _, _) in ref.items():
        nl = int(out["n_l"][f])
        assert np.array_equal(out["track_idx"][f, :nl], ti), f"{what} pair {f}: {(out['track_idx'][f, :nl] != ti).sum()} differ"
        assert np.array_equal(out["track_dist"][f, :nl], td), f"{what} pair {f}"
        assert (out["track_idx"][f, nl:] == -1).all()


def _assert_same(a, b):
    for k in a:
        assert np.array_equal(a[k], b[k]), k


_SPEC = {"kps_l": (api.KP_DTYPE, ()), "desc_l": (np.uint8, (32,)), "n_l": (np.int32, None), "kps_r": (api.KP_DTYPE, ()),
         "desc_r": (np.uint8, (32,)), "n_r": (np.int32, None), "stereo_idx": (np.int32, ()), "stereo_dist": (np.int32, ()),
         "track_idx": (np.int32, ()), "track_dist": (np.int32, ())}


class _Resident:
    """Images and the ten output arrays of one resident call, in device memory."""

    def __init__(self, L, R, cap):
        self.F, self.h, self.w = L.shape
        self.cap = cap
        self.dl, self.dr = api.DeviceBuffer(L.nbytes).upload(L), api.DeviceBuffer(R.nbytes).upload(R)
        self.shapes = {k: ((self.F,) if tail is None else (self.F, cap) + tail, dt) for k, (dt, tail) in _SPEC.items()}
        self.bufs = {k: api.DeviceBuffer(int(np.prod(s)) * np.dtype(dt).itemsize) for k, (s, dt) in self.shapes.items()}
        self.ptrs = {k: b.ptr for k, b in self.bufs.items()}

    def run(self, ex, tp, **plan):
        ex.stereo_sequence_dev(self.dl.ptr, self.dr.ptr, self.F, self.w, self.h, self.ptrs, tp, **plan)
        return self

    def fetch(self):
        return {k: self.bufs[k].download(s, dt) for k, (s, dt) in self.shapes.items()}


def test_se3_composition_is_orc_track_pair(oracle, cams):
    """The oracle of an SE3 prior (NormalizedUndistort + GetDepth + ProjectionMatch, no-depth points skipped) is orc_track_pair
    when given the 3x4 form, and a pure translation gives the same matches in either form."""
    _, ocam = cams
    L, R = _frames(0, IRREGULAR[1:3])
    ref = oracle.Extractor()
    kl, dl = ref.extract(L[0])
    kr, dr = ref.extract(R[0])
    si, _ = oracle.stereo_match(kl, dl, kr, dr)
    kc, dc = ref.extract(L[1])
    for radius in (8.0, 50.0):
        T = _shift_rt(9)
        want = oracle.track_pair(ocam, B, T, radius, kl, dl, kr, si, kc, dc)
        xc, valid = oracle.stereo_depth(ocam, B, kl, oracle.normalized_undistort(ocam, kl), kr, si)
        got = oracle.projection_match(xc, dl, valid != 1, T[:3, :4], ocam, kc, dc, radius)
        assert np.array_equal(got[0], want[0]) and np.array_equal(got[1], want[1])
        se3 = _oracle_pass(oracle, ocam, _shift_se3(9), radius, kl, dl, kr, si, kc, dc)
        assert np.array_equal(se3[0], want[0]) and np.array_equal(se3[1], want[1])
        assert (want[0] >= 0).sum() > 500


def test_plan_without_priors_or_retry_is_sfe_stereo_sequence(gpu, cams):
    """A plan whose priors are all tp's (3x4 or SE3 form) or both NULL, without a retry, gives what sfe_stereo_sequence gives,
    bit for bit, on the host and the resident entry points, and launches the same number of kernels."""
    cam, _ = cams
    L, R = _frames(1, IRREGULAR)
    F = len(IRREGULAR)
    ex = api.ORBextractor(max_images=2 * F)
    dev = _Resident(L, R, ex.cap)
    for prior in (_shift_rt(3), _shift_se3(3)):
        tp = api.TrackParams.make(cam, B, prior, 20.0)
        n0 = ex.launches()
        base = ex.stereo_sequence(L, R, tp)
        per_call = ex.launches() - n0
        assert (base["track_idx"][1:] >= 0).sum() > 1000
        for plan in ({"retry_below": 0}, {"priors": np.stack([prior] * F)}, {"priors": np.stack([prior] * F), "retry_radius": 5.0}):
            n0 = ex.launches()
            _assert_same(ex.stereo_sequence(L, R, tp, **plan), base)
            assert ex.launches() - n0 == per_call
            _assert_same(dev.run(ex, tp, **plan).fetch(), base)
        _assert_same(dev.run(ex, tp).fetch(), base)


def test_pair_priors_on_irregular_motion(gpu, oracle, cams):
    """Image shifts of 2, 9, 1, 30 and 5 px between consecutive frames, each pair with its exact prior and a radius of 8 px:
    every pair equals the oracle under its own prior (entry f = pair (f-1, f)).  The same sequence with one shared prior finds
    far fewer matches where the motion differs from it."""
    cam, ocam = cams
    L, R = _frames(0, IRREGULAR)
    F = len(IRREGULAR)
    ex = api.ORBextractor(max_images=2 * F)
    tp = api.TrackParams.make(cam, B, _shift_rt(2), 8.0)
    for se3 in (False, True):
        priors = _exact_priors(IRREGULAR, se3)
        priors[0] = np.nan  # entry 0 is never read
        out = ex.stereo_sequence(L, R, tp, priors=priors)
        ref = _oracle_plan(oracle, ocam, out, priors, 8.0)
        _assert_tracks(out, ref, f"host se3={se3}")
        assert all(ref[f][2] > 500 for f in ref), [ref[f][2] for f in ref]
        _assert_tracks(_Resident(L, R, ex.cap).run(ex, tp, priors=priors).fetch(), ref, f"resident se3={se3}")
    shared = ex.stereo_sequence(L, R, tp)
    counts = [int((shared["track_idx"][f] >= 0).sum()) for f in range(1, F)]
    exact = [ref[f][2] for f in range(1, F)]
    assert min(c / e for c, e in zip(counts, exact)) < 0.25, (counts, exact)


def test_wide_radius_retry(gpu, oracle, cams):
    """The tracker's rule (radius 50, identity prior; fewer than 8 matches: radius 100) on a sequence with one 70-px jump: the
    jump pair is matched again and its second result kept, the 4-px pairs keep their first.  retry_below = INT32_MAX retries
    every pair, retry_below = 0 none.  The retry costs two launches (retry flags, second pass) on top of the plan call."""
    cam, ocam = cams
    L, R = _frames(0, JUMP)
    F = len(JUMP)
    ident = np.stack([np.eye(4)] * F)
    tp = api.TrackParams.make(cam, B, None, 50.0)
    ex = api.ORBextractor(max_images=2 * F)
    dev = _Resident(L, R, ex.cap)
    launches = {}
    for below in (8, INT32_MAX, 0):
        n0 = ex.launches()
        out = ex.stereo_sequence(L, R, tp, retry_radius=100.0, retry_below=below)
        launches[below] = ex.launches() - n0
        ref = _oracle_plan(oracle, ocam, out, ident, 50.0, 100.0, below)
        _assert_tracks(out, ref, f"host retry_below={below}")
        _assert_tracks(dev.run(ex, tp, priors=ident, retry_radius=100.0, retry_below=below).fetch(), ref,
                       f"resident retry_below={below}")
        retried = [f for f in ref if ref[f][3]]
        if below == 8:
            assert retried == [2], [(f, ref[f][2]) for f in ref]
            assert (ref[2][0] >= 0).sum() > 200
        else:
            assert retried == ([] if below == 0 else [1, 2, 3])
    assert launches[8] == launches[INT32_MAX] == launches[0] + 2
    n0 = ex.launches()
    ex.stereo_sequence(L, R, tp)
    assert ex.launches() - n0 == launches[0]


def test_plan_on_the_pipelined_host_path_and_a_split_resident_batch(gpu, oracle, cams, monkeypatch):
    """One frame per host sub-batch (consecutive frames in different chunks) gives the single-chunk result; a resident batch of
    48 frames (three sub-batches on three streams) equals the oracle pair by pair.  The batch strings together sequences of
    several scenes: a pair inside a scene gets its exact prior and matches over 700 keypoints at 8 px (oracle, on the CPU),
    a pair across a cut (identity prior) under 100, so with retry_below = 300 exactly the cuts are matched again at 100."""
    cam, ocam = cams
    L, R = _frames(2, IRREGULAR)
    F = len(IRREGULAR)
    tp = api.TrackParams.make(cam, B, None, 8.0)
    plan = {"priors": _exact_priors(IRREGULAR), "retry_radius": 100.0, "retry_below": 8}
    one = api.ORBextractor(max_images=2 * F).stereo_sequence(L, R, tp, **plan)
    monkeypatch.setenv("SFE_PIPELINE_CHUNKS", str(F))
    _assert_same(api.ORBextractor(max_images=2 * F).stereo_sequence(L, R, tp, **plan), one)
    monkeypatch.delenv("SFE_PIPELINE_CHUNKS")

    parts = [(_frames(s, IRREGULAR), IRREGULAR) for s in range(4)] + [(_frames(s, JUMP), JUMP) for s in range(6)]
    L = np.concatenate([p[0][0] for p in parts])
    R = np.concatenate([p[0][1] for p in parts])
    priors = np.concatenate([_exact_priors(idx) for _, idx in parts])  # a scene's entry 0 (the cut) is its identity
    F = len(L)
    assert F == 48
    ex = api.ORBextractor(max_images=2 * F)
    out = _Resident(L, R, ex.cap).run(ex, tp, priors=priors, retry_radius=100.0, retry_below=300).fetch()
    ref = _oracle_plan(oracle, ocam, out, priors, 8.0, 100.0, 300)
    _assert_tracks(out, ref, "48 resident frames")
    cuts = set(np.cumsum([len(idx) for _, idx in parts])[:-1].tolist())
    assert {f for f in ref if ref[f][3]} == cuts, [(f, ref[f][2]) for f in ref]


def test_asynchronous_plan_calls_keep_their_own_priors(gpu, oracle, cams):
    """Two resident plan calls queued back to back on an asynchronous handle, with different priors and retry settings and
    their own output arrays: the second call's priors and retry keys must not reach the first call's tracking, which still
    runs on the side stream when the second call is enqueued."""
    cam, ocam = cams
    L, R = _frames(1, IRREGULAR)
    F = len(IRREGULAR)
    tp = api.TrackParams.make(cam, B, None, 8.0)
    ex = api.ORBextractor(max_images=2 * F)
    a_prm = {"priors": _exact_priors(IRREGULAR, se3=True)}
    b_prm = {"priors": np.stack([np.eye(4)] * F), "retry_radius": 40.0, "retry_below": INT32_MAX}
    a, b = _Resident(L, R, ex.cap), _Resident(L, R, ex.cap)
    ex.set_async(True)
    for _ in range(2):
        a.run(ex, tp, **a_prm)
        b.run(ex, tp, **b_prm)
    ex.wait()
    ex.set_async(False)
    got_a, got_b = a.fetch(), b.fetch()
    ref_a = _oracle_plan(oracle, ocam, got_a, a_prm["priors"], 8.0)
    ref_b = _oracle_plan(oracle, ocam, got_b, b_prm["priors"], 8.0, 40.0, INT32_MAX)
    _assert_tracks(got_a, ref_a, "call a")
    _assert_tracks(got_b, ref_b, "call b")
    assert any(not np.array_equal(ref_a[f][0], ref_b[f][0]) for f in ref_a)


def test_bad_plans_are_rejected(gpu, cams):
    """Every rule of sfe_track_plan's validation returns SFE_ERR_BAD_ARG from both entry points; a non-finite entry 0 is
    ignored."""
    cam, _ = cams
    L, R = _frames(0, IRREGULAR[:3])
    F, h, w = L.shape
    tp = api.TrackParams.make(cam, B, None, 20.0)
    ex = api.ORBextractor(max_images=2 * F)
    out = ex.alloc_stereo_out(F, track=True)
    dev = _Resident(L, R, ex.cap)
    host_args = [out[k].ctypes.data_as(C.c_void_p) for k in _SPEC]
    dev_args = [C.c_void_p(dev.ptrs[k]) for k in _SPEC]
    rt = np.stack([np.eye(4)[:3, :4].reshape(12)] * F)
    se3 = np.stack([[0.0, 0.0, 0.0, 1.0, 0.0, 0.0, 0.0]] * F)

    def plan(rt_=None, se3_=None, radius=100.0, below=8):
        p = api.TrackPlan(None, None, radius, below)
        if rt_ is not None:
            p.rt = rt_.ctypes.data_as(C.POINTER(C.c_double))
        if se3_ is not None:
            p.se3 = se3_.ctypes.data_as(C.POINTER(api.SE3))
        return p

    def status(p):
        ref = C.byref(p) if p is not None else None
        a = api.lib().sfe_stereo_sequence_plan(ex.h, L.ctypes.data_as(C.c_void_p), R.ctypes.data_as(C.c_void_p), w * h, F, w, h, w,
                                               None, C.byref(tp), ref, *host_args, ex.cap)
        b = api.lib().sfe_stereo_sequence_plan_dev(ex.h, C.c_void_p(dev.dl.ptr), C.c_void_p(dev.dr.ptr), w * h, F, w, h, w, None,
                                                   C.byref(tp), ref, *dev_args, ex.cap)
        return a, b

    def with_value(a, row, col, v):
        a = a.copy()
        a[row, col] = v
        return a

    ok = api.SFE_OK, api.SFE_OK
    bad = api.SFE_ERR_BAD_ARG, api.SFE_ERR_BAD_ARG
    assert status(plan(rt)) == ok and status(plan(se3_=se3)) == ok
    assert status(plan(with_value(rt, 0, 3, np.nan))) == ok and status(plan(se3_=with_value(se3, 0, 6, np.inf))) == ok
    assert status(None) == bad
    assert status(plan(rt, se3)) == bad
    for row, col, v in ((1, 0, np.nan), (F - 1, 11, np.inf), (1, 7, -np.inf)):
        assert status(plan(with_value(rt, row, col, v))) == bad, (row, col, v)
    for row, col, v in ((1, 3, np.nan), (F - 1, 4, np.inf)):
        assert status(plan(se3_=with_value(se3, row, col, v))) == bad, (row, col, v)
    assert status(plan(radius=-1.0)) == bad and status(plan(radius=np.nan)) == bad
    assert status(plan(below=-1)) == bad
    assert status(plan(radius=0.0, below=0)) == ok
    with pytest.raises(ValueError):
        ex.stereo_sequence(L, R, tp, priors=np.zeros((F + 1, 7)))
