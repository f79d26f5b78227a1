"""Pins the C oracle (oracle/orb_oracle.c) to the REFERENCE'S OWN CODE: oracle/_ref = geonuklee/slam-toolkit's
src/orb_extractor.cpp, src/matcher.cpp and src/camera.cpp compiled unmodified (oracle/ref_build/Makefile) against
stand-in third-party headers whose five image primitives are the cv2-pinned models (tests/test_oracle_vs_cv2.py).

With the monotonic heap (list nodes get increasing addresses, so the reference's `sort` by (count, node address),
src/orb_extractor.cpp:684, orders equal counts by creation = the oracle's declared rule T1) every byte must agree:
tables, pyramid, the 19-px ring, FAST candidates, quadtree survivors and their order, angles, blurred planes,
descriptors, StereoMatch, ProjectionMatch.  With glibc's heap the reference itself moves; there the test asserts equality
on every level whose quadtree did NOT stop inside a group of equally-full nodes and reports the rest.

The reference's side of each comparison comes from oracle/_ref when that library is built (it needs the reference's
sources, which are not part of this repository), else from tests/golden/ref_pinning.json: the SHA-256 of every array the
reference returned here (and the quaternions its SE3Quat holds, which feed later calls).  With the library present
every live value must also equal its recorded digest; SFE_RECORD_REF_PINS=1 rewrites the file from the live library
instead.  Only the glibc-heap test needs the library itself.  CPU only."""
import hashlib
import json
import os

import numpy as np
import pytest

from slam_toolkit_b200 import synth

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PINS = os.path.join(ROOT, "tests", "golden", "ref_pinning.json")


def _digest(a):
    a = np.ascontiguousarray(a)
    return hashlib.sha256(f"{a.dtype.str}{a.shape}".encode() + a.tobytes()).hexdigest()[:32]


class Pins:
    """The reference's side of the comparisons of one test: `ref` is the live oracle/_ref binding or None."""

    def __init__(self, ref, stored, record, test):
        self.ref, self.stored, self.record, self.test = ref, stored, record, test

    def _key(self, key):
        return f"{self.test}/{key}"

    def equal(self, key, got, want):
        """got (the oracle's value) equals want() (the reference's), byte for byte"""
        k = self._key(key)
        got = np.asarray(got)
        if self.ref is None:
            assert k in self.stored["digests"], f"no recorded reference value for {k}"
            assert _digest(got) == self.stored["digests"][k], k
            return
        w = np.asarray(want())
        assert got.dtype == w.dtype and got.shape == w.shape and got.tobytes() == w.tobytes(), k
        if self.record:
            self.stored["digests"][k] = _digest(w)
        else:
            assert self.stored["digests"].get(k) == _digest(w), f"{k}: the live reference differs from its recorded digest"

    def value(self, key, want):
        """a float64 vector the reference computed (used as an input of later calls)"""
        k = self._key(key)
        if self.ref is None:
            return np.array(self.stored["values"][k], np.float64)
        w = np.asarray(want(), np.float64)
        if self.record:
            self.stored["values"][k] = w.tolist()
        else:
            assert np.array_equal(np.array(self.stored["values"].get(k, []), np.float64).view(np.uint64), w.view(np.uint64)), k
        return w


@pytest.fixture(scope="module")
def pins_store():
    import ref_c
    live = ref_c if ref_c.available() else None
    record = live is not None and os.environ.get("SFE_RECORD_REF_PINS") == "1"
    if record:
        stored = {"digests": {}, "values": {}}
    else:
        with open(PINS) as f:
            stored = json.load(f)
    if live is not None:
        live.set_heap_mode(live.HEAP_MONOTONIC)
    yield live, stored, record
    if live is not None:
        live.set_heap_mode(live.HEAP_MONOTONIC)
    if record:
        stored["generator"] = ("oracle/_ref: the reference's own src/orb_extractor.cpp, src/matcher.cpp, src/camera.cpp compiled "
                               "unmodified (oracle/ref_build), monotonic heap; written by SFE_RECORD_REF_PINS=1 pytest "
                               "tests/test_ref_pinning.py")
        with open(PINS, "w") as f:
            json.dump(stored, f, indent=0, sort_keys=True)


@pytest.fixture
def pin(pins_store, request):
    live, stored, record = pins_store
    return Pins(live, stored, record, request.node.name)


def _cam(oracle, d=(0, 0, 0, 0), w=synth.KITTI_W, h=synth.KITTI_H):
    return oracle.make_camera(synth.KITTI_FX, synth.KITTI_FY, synth.KITTI_CX, synth.KITTI_CY, list(d), w, h)


def _reflect101_ring(img, e=19):
    return np.pad(img, e, mode="reflect")


def _or_empty(plane):
    return np.zeros(0, np.int8) if plane is None else plane


def _compare_extraction(oracle, pin, o, r, img, tag):
    """o: oracle extractor; r: the reference's extractor with the same parameters (None without the library)"""
    ko, do = o.extract(img)
    if r is not None:
        kr, dr = r.extract(img)
    for l in range(o.nlevels):
        lo = o.level(l)
        pin.equal(f"{tag}/level{l}", lo, lambda: r.level(l))
        pin.equal(f"{tag}/ring{l}", _reflect101_ring(lo), lambda: r.level(l, ring=True))
        co = o.candidates(l)
        pin.equal(f"{tag}/candidates{l}", co, lambda: r.candidates(l))       # set and order
        if len(co):
            quota = int(o.tables()["per_level"][l])
            h, w = lo.shape
            pin.equal(f"{tag}/quadtree{l}", o.distributed(l), lambda: r.distribute(co, 16, w - 16, 16, h - 16, quota, l))
        ob = o.blur(l)
        pin.equal(f"{tag}/blur{l}", _or_empty(ob), lambda: _or_empty(r.blur(l)))   # only levels that kept keypoints are blurred
        if ob is None:
            assert len(o.distributed(l)) == 0
    for f in ko.dtype.names:  # angle compared by bits: fastAtan2 output
        pin.equal(f"{tag}/kp.{f}", ko[f], lambda: kr[f])
    pin.equal(f"{tag}/descriptors", do, lambda: dr)
    return ko, do


def _ref_extractor(pin, *params):
    return pin.ref.Extractor(*params) if pin.ref is not None else None


def test_ctor_tables_equal_the_reference(oracle, pin):
    for nf, sf, nl in [(2000, 1.2, 8), (500, 1.2, 4), (300, 1.5, 3), (1000, 1.2, 8), (50, 1.2, 2), (20, 1.2, 8), (1500, 1.1, 12),
                       (4000, 2.0, 5), (1, 1.2, 8), (777, 1.33, 7)]:
        to = oracle.Extractor(nf, sf, nl, 20, 7).tables()
        tr = _ref_extractor(pin, nf, sf, nl, 20, 7)
        for k in to:
            pin.equal(f"{nf},{sf},{nl}/{k}", to[k], lambda: tr.tables()[k])


@pytest.mark.parametrize("seed", range(8))
def test_kitti_frames_every_stage(oracle, pin, seed):
    o, r = oracle.Extractor(), _ref_extractor(pin)
    L, R = synth.stereo_pair(seed)
    kl, dl = _compare_extraction(oracle, pin, o, r, L, "L")
    kr, dr = _compare_extraction(oracle, pin, o, r, R, "R")
    si, _ = oracle.stereo_match(kl, dl, kr, dr)
    pin.equal("stereo", si, lambda: pin.ref.stereo_match(kl, dl, kr, dr, _cam(oracle)))
    assert (si >= 0).sum() > 1000


@pytest.mark.parametrize("case", [(320, 240, 500, 1.2, 4, 20, 7), (161, 131, 300, 1.5, 3, 20, 7), (640, 200, 1000, 1.2, 8, 30, 10),
                                  (97, 95, 50, 1.2, 2, 20, 7), (1241, 376, 20, 1.2, 8, 20, 7), (800, 600, 3000, 1.2, 8, 20, 7),
                                  (333, 500, 700, 1.3, 6, 25, 5), (1920, 1080, 2000, 1.2, 8, 20, 7)])
def test_other_geometries(oracle, pin, case):
    w, h, nf, sf, nl, it, mt = case
    img, _ = synth.stereo_pair(100 + w % 7, w, h)
    _compare_extraction(oracle, pin, oracle.Extractor(nf, sf, nl, it, mt), _ref_extractor(pin, nf, sf, nl, it, mt), img, "img")


def test_noise_flat_and_retry_images(oracle, pin):
    """noise (every level far over quota, very long careful phase), flat (nothing), low contrast (20 -> 7 retry)"""
    rng = np.random.default_rng(3)
    o, r = oracle.Extractor(), _ref_extractor(pin)
    noise = rng.integers(0, 256, (376, 1241), dtype=np.uint8)
    k, _ = _compare_extraction(oracle, pin, o, r, noise, "noise")
    assert len(k) >= 2000
    k, _ = _compare_extraction(oracle, pin, o, r, np.full((376, 1241), 77, np.uint8), "flat")
    assert len(k) == 0
    soft = (synth.stereo_pair(11)[0].astype(np.float32) * 0.12 + 100).astype(np.uint8)   # contrast below iniThFAST
    k, _ = _compare_extraction(oracle, pin, o, r, soft, "soft")
    assert len(k) > 0
    mixed = synth.stereo_pair(12)[0].copy()
    mixed[:, 600:] = (mixed[:, 600:].astype(np.float32) * 0.1 + 90).astype(np.uint8)
    _compare_extraction(oracle, pin, o, r, mixed, "mixed")


def test_distribute_random_candidate_sets(oracle, pin):
    """DistributeOctTree + DivideNode (src/orb_extractor.cpp:481-763) on synthetic candidate lists with many equal counts"""
    r = _ref_extractor(pin)
    rng = np.random.default_rng(5)
    for t in range(60):
        W, H = int(rng.integers(40, 1300)), int(rng.integers(40, 500))
        if round(W / H) < 1:
            continue
        n = int(rng.integers(1, 4000))
        xs = rng.integers(0, W - 3, n).astype(np.float32)
        ys = rng.integers(0, H - 3, n).astype(np.float32)
        if t % 3 == 0:   # duplicates and clusters
            xs[: n // 2] = xs[0]
            ys[: n // 3] = ys[0]
        resp = rng.integers(8, 120, n).astype(np.float32)
        xyr = np.stack([xs, ys, resp], 1)
        want = int(rng.integers(1, 2500))
        a = oracle.distribute(xyr, 16, 16 + W, 16, 16 + H, want)
        pin.equal(f"{t}", a, lambda: r.distribute(xyr, 16, 16 + W, 16, 16 + H, want))


def test_glibc_heap_moves_only_levels_cut_inside_a_tie_group(oracle, pin):
    """The reference as it runs on this machine (glibc malloc): equal to the oracle as a SET on every level whose careful
    phase did not stop between two equally-full nodes; the others are where the heap-address order decides (T1)."""
    if pin.ref is None:
        pytest.skip("glibc's heap order is the live reference library's own, and oracle/_ref is not built")
    ref = pin.ref
    o, r = oracle.Extractor(), ref.Extractor()
    total = moved = cut_levels = levels = 0
    for seed in range(8):
        img, _ = synth.stereo_pair(seed)
        ref.set_heap_mode(ref.HEAP_MALLOC)
        kr, dr = r.extract(img)
        ref.set_heap_mode(ref.HEAP_MONOTONIC)
        ko, do = o.extract(img)
        for l in range(8):
            so = {kp.tobytes() + d.tobytes() for kp, d in zip(ko[ko["octave"] == l], do[ko["octave"] == l])}
            sr = {kp.tobytes() + d.tobytes() for kp, d in zip(kr[kr["octave"] == l], dr[kr["octave"] == l])}
            levels += 1
            if o.tie_cut(l):
                cut_levels += 1
                moved += len(so - sr)
            else:
                assert so == sr, f"seed {seed} level {l}: no tie at the cut, yet the keypoint sets differ"
        total += len(ko)
    print(f"glibc heap: {moved} of {total} keypoints differ, all on the {cut_levels} of {levels} levels cut inside a tie group")
    assert moved < 0.05 * total


def test_descriptor_distance_and_atan2(oracle, pin):
    rng = np.random.default_rng(9)
    d = rng.integers(0, 256, (300, 32), dtype=np.uint8)
    got = np.array([oracle.hamming256(d[i], d[i + 1]) for i in range(0, 300, 2)], np.int32)
    assert np.array_equal(got, [int(np.unpackbits(d[i] ^ d[i + 1]).sum()) for i in range(0, 300, 2)])
    pin.equal("hamming", got, lambda: np.array([pin.ref.hamming256(d[i], d[i + 1]) for i in range(0, 300, 2)], np.int32))


def test_se3_and_camera_primitives(oracle, pin):
    """predicted_Tcw * Xw (g2o::SE3Quat, quaternion product), Camera::Project / IsInImage / NormalizedUndistort by bits"""
    rng = np.random.default_rng(0)
    for t in range(100):
        q = rng.normal(size=4)
        q /= np.linalg.norm(q)
        if t % 3 == 0:
            q = np.array([0, 0, 0, 1.0]) + rng.normal(size=4) * 1e-2
        qt = np.concatenate([q, rng.normal(size=3)])
        x = rng.normal(size=(300, 3)) * rng.uniform(0.1, 100)
        qh = pin.value(f"{t}/q", lambda: pin.ref.se3_apply(qt, x)[1])
        assert abs(np.linalg.norm(qh) - 1) < 1e-15 and qh[3] >= 0
        yo = oracle.se3_apply(np.concatenate([qh, qt[4:]]), x)
        pin.equal(f"{t}/xc", yo, lambda: pin.ref.se3_apply(qt, x)[0])
    cam = _cam(oracle, (-0.1, 0.02, 0.001, -0.0005))
    kps = np.zeros(500, oracle.KP_DTYPE)
    kps["x"], kps["y"] = rng.uniform(0, 1241, 500), rng.uniform(0, 376, 500)
    pin.equal("undistort", oracle.normalized_undistort(cam, kps), lambda: pin.ref.normalized_undistort(cam, kps))


def _projection_inputs(seed, kl, dl, n=3000):
    rng = np.random.default_rng(seed)
    z = rng.uniform(2, 80, n)
    u, v = rng.uniform(-50, 1291, n), rng.uniform(-30, 406, n)
    xw = np.stack([(u - synth.KITTI_CX) / synth.KITTI_FX * z, (v - synth.KITTI_CY) / synth.KITTI_FY * z, z], 1)
    xw[::17, 2] *= -1
    md = rng.integers(0, 256, (n, 32), dtype=np.uint8)
    pick = rng.integers(0, len(kl), n)
    cp = rng.random(n) < 0.5
    md[cp] = dl[pick[cp]]
    for i in np.nonzero(cp)[0]:
        for b in rng.integers(0, 256, 3):
            md[i, b // 8] ^= np.uint8(1 << (b % 8))
    # two queries with the same descriptor landing on one keypoint: equal distance, the later one must win (:197-204)
    md[n - 1], xw[n - 1] = md[np.nonzero(cp)[0][0]], xw[np.nonzero(cp)[0][0]]
    skip = (rng.random(n) < 0.05).astype(np.uint8)
    return xw, md, skip


@pytest.mark.parametrize("seed", range(3))
def test_projection_match_equals_the_reference(oracle, pin, seed):
    img = synth.stereo_pair(seed)[0]
    kl, dl = oracle.Extractor().extract(img)          # the frame: the reference's keypoints, pinned right here
    r = _ref_extractor(pin)
    if r is not None:
        kr, dr = r.extract(img)
    pin.equal("kps", kl, lambda: kr)
    pin.equal("desc", dl, lambda: dr)
    xw, md, skip = _projection_inputs(seed, kl, dl)
    for d4 in ((0, 0, 0, 0), (-0.1, 0.02, 0.001, -0.0005)):
        cam = _cam(oracle, d4)
        for qt_in in ([0, 0, 0, 1, 0, 0, 0], [0.01, -0.02, 0.005, 0.9997, 0.1, -0.05, 0.2], [0.3, -0.1, 0.2, -0.9, 1.0, 0.5, 4.0]):
            q = pin.value(f"{qt_in}/q", lambda: pin.ref.se3_apply(np.array(qt_in, float), xw[:1])[1])
            qt = np.concatenate([q, np.array(qt_in[4:], float)])
            for radius in (50.0, 10.0, 100.0):
                for grid in (False, True):
                    got, dist = oracle.projection_match(xw, md, skip, qt, cam, kl, dl, radius, grid=grid)
                    pin.equal(f"{d4}/{qt_in}/{radius}", got, lambda: pin.ref.projection_match(xw, md, skip, qt, cam, kl, dl, radius))
                    ok = got >= 0
                    assert all(dist[j] == oracle.hamming256(md[got[j]], dl[j]) for j in np.nonzero(ok)[0])


def test_projection_golden_fixture(oracle):
    """the committed ProjectionMatch result of the reference (tools/gen_golden.py)"""
    z = np.load(os.path.join(ROOT, "tests/golden/golden_proj.npz"))
    g = np.load(os.path.join(ROOT, "tests/golden/golden_seed0.npz"))
    cam = _cam(oracle, z["dist4"])
    assert np.array_equal(oracle.se3_apply(z["qt"], z["xw"]).view(np.uint64), z["xc"].view(np.uint64))
    for radius in (50, 10):
        got, _ = oracle.projection_match(z["xw"], z["mp_desc"], z["skip"], z["qt"], cam, g["kl"], g["dl"], float(radius))
        assert np.array_equal(got, z[f"to_query_r{radius}"])
        assert (got >= 0).sum() > 10


def test_stereo_match_edge_cases_equal_the_reference(oracle, pin):
    """hand-built rows: single candidate (accepted, dist1 = 999999999), tie for best (rejected), dy = +-3 exactly,
    dx = 0 / 100 / just outside, negative dx, bucket borders (y multiples of 10), an empty right set"""
    rng = np.random.default_rng(21)
    cam = _cam(oracle)
    for trial in range(30):
        nl, nr = int(rng.integers(1, 200)), int(rng.integers(0, 200))
        kl, kr = np.zeros(nl, oracle.KP_DTYPE), np.zeros(nr, oracle.KP_DTYPE)
        kl["x"], kl["y"] = rng.integers(0, 1241, nl), rng.integers(0, 40, nl)   # few rows: many candidates per keypoint
        kr["x"] = rng.integers(0, 1241, nr)
        kr["y"] = rng.integers(0, 40, nr) + rng.choice([0.0, 0.5, -0.25], nr)
        dl = rng.integers(0, 256, (nl, 32), dtype=np.uint8)
        dr = rng.integers(0, 256, (nr, 32), dtype=np.uint8)
        if nr > 4:
            dr[1] = dr[0]                               # exact tie -> rejected wherever both are candidates
            kr[1] = kr[0]
            kl[0]["x"], kl[0]["y"] = kr[0]["x"] + 100, kr[0]["y"] + 3     # on both limits
            dl[0] = dr[2]
            kr[2]["x"], kr[2]["y"] = kl[0]["x"], kl[0]["y"] - 3           # dx = 0, dy = 3
        got, _ = oracle.stereo_match(kl, dl, kr, dr)
        pin.equal(f"{trial}", got, lambda: pin.ref.stereo_match(kl, dl, kr, dr, cam))
