"""The matchers at the shapes that select their other kernel variants and kernel-side branches, against the C oracle.

Every matcher launcher picks a kernel variant, or a branch inside the kernel, from the call's shape: StereoMatch's
lanes-per-keypoint and keypoints-per-thread instantiations, ProjectionMatch's bucket grid (sized from the camera) and its
sorted path for large maps, SearchRadius' truncated rows, the multi-round child loop of the vocabulary descent and the
SE3Quat motion prior of the tracker.  Each scene plants the ties and exact boundaries where a variant could go wrong, checks
that the oracle really sees them, and compares every index, distance and double by its bits."""
import os
from concurrent.futures import ThreadPoolExecutor

import numpy as np
import pytest

from slam_toolkit_b200 import api, synth

pytestmark = pytest.mark.gpu
NCPU = os.cpu_count() or 1
F32 = np.float32


@pytest.fixture(scope="module")
def gpu():
    if api.device_count() < 1:
        pytest.fail("no CUDA device: the product has no CPU fallback")
    return 0


@pytest.fixture(scope="module")
def matcher(gpu):
    return api.Matcher()


def _kps(x, y):
    k = np.zeros(len(x), api.KP_DTYPE)
    k["x"], k["y"] = x, y
    return k


def _flipped(d, nbits, rng):
    """d with exactly nbits distinct bits flipped: Hamming distance nbits from d"""
    out = d.copy()
    for b in rng.choice(256, nbits, replace=False):
        out[b >> 3] ^= np.uint8(1 << (b & 7))
    return out


def _div_up(a, b):
    return (a + b - 1) // b


def _threaded(fn, n, *args):
    """fn(lo, hi, *args) over n rows split across the CPUs (the oracle's ctypes calls release the GIL)"""
    bounds = np.linspace(0, n, NCPU + 1).astype(int)
    with ThreadPoolExecutor(NCPU) as pool:
        return list(pool.map(lambda k: fn(bounds[k], bounds[k + 1], *args), range(NCPU)))


# ---- StereoMatch ------------------------------------------------------------------------------------------------------
def _oracle_stereo(oracle, kl, dl, kr, dr, sp):
    parts = _threaded(lambda lo, hi: oracle.stereo_match(kl[lo:hi], dl[lo:hi], kr, dr, sp.y_threshold, sp.max_dx,
                                                         sp.best12_threshold), len(kl))
    return np.concatenate([p[0] for p in parts]), np.concatenate([p[1] for p in parts])


def _stereo_variant(frames, cap):
    """the instantiation launch_stereo_match picks: (keypoints per thread, lanes per keypoint)"""
    if frames * _div_up(cap, 64) <= 2 * 148:
        return (1, 4)
    return (1, 1) if frames * _div_up(cap, 512) < 64 else (2, 1)


def _stereo_scene(n_l, n_r, seed):
    """Random right keypoints on clustered rows over [-20, 2100) x [-6, 1080] (beyond the last bucket row and column),
    left keypoints = shifted copies with 16-64 bits flipped; then planted cases at known positions.  Returns the scene and
    the planted left indices with their expected (index, distance) under ratio 0.5 and under ratio 1.5."""
    rng = np.random.default_rng(seed)
    xr = rng.uniform(-20, 2100, n_r).astype(F32)
    yr = (rng.integers(-5, 900, n_r) * 1.2).astype(F32)
    dr = rng.integers(0, 256, (n_r, 32), dtype=np.uint8)
    sel = rng.integers(0, n_r, n_l)
    xl = (xr[sel] + rng.uniform(-5, 110, n_l)).astype(F32)
    yl = (yr[sel] + rng.integers(-4, 5, n_l)).astype(F32)
    masks = [rng.integers(0, 256, (n_l, 32), dtype=np.uint8) for _ in range(4)]
    k = rng.integers(2, 5, n_l)[:, None]
    flip = masks[0] & masks[1] & np.where(k >= 3, masks[2], 0xFF).astype(np.uint8) & np.where(k >= 4, masks[3], 0xFF).astype(np.uint8)
    dl = dr[sel] ^ flip
    up = lambda v: np.nextafter(F32(v), F32(np.inf))
    down = lambda v: np.nextafter(F32(v), F32(-np.inf))
    # case: (left x, left y, [(right index or None, right x, right y, Hamming distance)], expected at 0.5, expected at 1.5);
    # an expectation is a position in the case's right list, or -1.  Right keypoints at other than the expected position
    # are either rejected by a filter or lose; nothing else within reach is closer than ~60 bits.
    cases = [
        (300.0, 100.0, [(None, 290.0, 100.0, 4), (None, 280.0, 101.0, 4)], -1, "min"),           # tie for best
        (600.0, 100.0, [(33000, 590.0, 100.0, 4), (2100, 580.0, 99.0, 4)], -1, 1),                # ... across chunks
        (900.0, 100.0, [(None, 890.0, 100.0, 3), (None, 880.0, 100.0, 9), (None, 870.0, 100.0, 9)], 0, 0),  # tie for 2nd
        (1200.0, 100.0, [(None, 1190.0, 100.0, 8), (None, 1180.0, 100.0, 16)], -1, 0),            # d0 == d1 * ratio
        (1500.0, 100.0, [(None, 1490.0, 100.0, 7), (None, 1480.0, 100.0, 16)], 0, 0),             # just below it
        (300.0, 300.0, [(None, 290.0, 303.0, 6), (None, 280.0, up(303.0), 1)], 0, 0),             # dy = -3 / beyond
        (600.0, 300.0, [(None, 590.0, 297.0, 6), (None, 580.0, down(297.0), 1)], 0, 0),           # dy = +3 / beyond
        (900.5, 300.0, [(None, 900.5, 300.0, 6), (None, up(900.5), 300.0, 1)], 0, 0),             # dx = 0 / dx < 0
        (1200.5, 300.0, [(None, 1100.5, 300.0, 6), (None, down(1100.5), 300.0, 1)], 0, 0),        # dx = max_dx / beyond
        (2050.25, 1040.5, [(None, 2040.0, 1041.0, 6), (None, 2000.0, 1039.0, 20)], 0, 0),         # clamped row and column
        (2080.0, 500.0, [(None, 1995.0, 502.0, 5)], 0, 0),                                        # clamped column
        (700.0, 1070.0, [(None, 650.0, 1068.0, 5)], 0, 0),                                        # clamped row
        (-30.5, -7.25, [(None, -60.0, -6.0, 6), (None, -20.0, -7.25, 1)], 0, 0),                  # negative coordinates
        (1500.0, 500.0, [(2500, 1450.0, 500.0, 2)], 0, 0),                                        # later chunks
        (1500.0, 700.0, [(32800, 1450.0, 700.0, 2), (None, 1470.0, 701.0, 9)], 0, 0),
        (1800.0, 700.0, [(65010, 1750.0, 700.0, 3), (10, 1760.0, 702.0, 9)], 0, 0),
        (1000.0, 900.0, [(40000, 950.0, 900.0, 5), (None, 960.0, 900.0, 5)], -1, "min"),         # tie, far chunk vs pool
    ]
    cases = [c for c in cases if all(r[0] is None or r[0] < n_r for r in c[2])]
    special = [r[0] for c in cases for r in c[2] if r[0] is not None]
    assert len(set(special)) == len(special)
    n_pool = sum(r[0] is None for c in cases for r in c[2])
    pool = [int(j) for j in rng.permutation(n_r) if int(j) not in special][:n_pool]
    lefts = np.linspace(0, n_l - 1, len(cases)).astype(int)
    assert len(set(lefts.tolist())) == len(cases)
    expect = {}
    for (lx, ly, rights, e05, e15), i in zip(cases, lefts):
        D = rng.integers(0, 256, 32, dtype=np.uint8)
        xl[i], yl[i], dl[i] = lx, ly, D
        js = []
        for (j, rx, ry, d) in rights:
            j = pool.pop() if j is None else j
            xr[j], yr[j], dr[j] = rx, ry, _flipped(D, d, rng)
            js.append(j)

        def val(e):
            if e == -1:
                return (-1, -1)
            p = int(np.argmin(js)) if e == "min" else e
            return (js[p], rights[p][3])
        expect[int(i)] = (val(e05), val(e15))
    return (_kps(xl, yl), dl, _kps(xr, yr), dr), expect


@pytest.mark.parametrize("cap", [18944, 18945, 32256, 32257, 65535])
def test_stereo_match_variant_boundaries(matcher, oracle, cap):
    """sfe_stereo_match (frames = 1, cap = max(n_l, n_r)) on both sides of each variant boundary: <1,4> up to 18944,
    <1,1> from 18945 to 32256, <2,1> from 32257; each cap with n_l == n_r, with few left and with few right keypoints."""
    sp05, sp15 = api.StereoParams(3.0, 100.0, 0.5), api.StereoParams(3.0, 100.0, 1.5)
    for shape, (n_l, n_r) in enumerate(((cap, cap), (200, cap), (cap, 200))):
        (kl, dl, kr, dr), expect = _stereo_scene(n_l, n_r, seed=cap + shape)
        assert max(n_l, n_r) == cap
        for sp, which in ((sp05, 0), (sp15, 1)) if shape == 1 else ((sp05, 0),):
            ri, rd = _oracle_stereo(oracle, kl, dl, kr, dr, sp)
            for i, e in expect.items():   # the planted cases occur as planned
                assert (ri[i], rd[i]) == e[which], (cap, shape, i, (ri[i], rd[i]), e[which])
            gi, gd = matcher.StereoMatch(kl, dl, kr, dr, sp)
            bad = np.nonzero((gi != ri) | (gd != rd))[0]
            assert len(bad) == 0, f"cap {cap} {(n_l, n_r)} ratio {sp.best12_threshold}: {len(bad)} rows differ, first {bad[:5]}"
            if shape == 0:
                assert (ri >= 0).sum() > n_l // 4 and (ri > 2047).sum() > 0


@pytest.fixture(scope="module")
def hd_pairs(oracle):
    """16 stereo pairs of 1920 x 1080 and their oracle extraction with nfeatures = 3000"""
    pairs = [synth.stereo_pair(s, 1920, 1080) for s in range(16)]

    def extract(lo, hi):
        ex = oracle.Extractor(3000)
        return [(ex.extract(L), ex.extract(R)) for L, R in pairs[lo:hi]]
    ref = [r for part in _threaded(extract, len(pairs)) for r in part]
    return np.stack([p[0] for p in pairs]), np.stack([p[1] for p in pairs]), ref


@pytest.mark.parametrize("frames", [10, 16])
def test_batched_stereo_frames_in_the_one_lane_variants(gpu, oracle, hd_pairs, monkeypatch, frames):
    """sfe_stereo_frames over 10 (<1,1>) and 16 (<2,1>) pairs of 1920 x 1080 with 3000 features in one launch: right
    frames with more than one 2048-keypoint chunk, every frame equal to the oracle's extraction and StereoMatch."""
    monkeypatch.setenv("SFE_PIPELINE_CHUNKS", "1")
    L, R, ref = hd_pairs
    ex = api.ORBextractor(3000, max_images=2 * frames)
    out = ex.stereo_frames(L[:frames], R[:frames])
    cap = out["kps_l"].shape[1]
    assert _stereo_variant(frames, cap) == ((1, 1) if frames == 10 else (2, 1)), cap
    assert (out["n_r"][:frames] > 2048).sum() >= frames // 2
    si = _threaded(lambda lo, hi: [oracle.stereo_match(*ref[f][0], *ref[f][1]) for f in range(lo, hi)], frames)
    si = [r for part in si for r in part]
    for f in range(frames):
        (kl, dl), (kr, dr) = ref[f]
        nl, nr = int(out["n_l"][f]), int(out["n_r"][f])
        assert (nl, nr) == (len(kl), len(kr)), f
        assert np.array_equal(out["kps_l"][f, :nl], kl) and np.array_equal(out["desc_l"][f, :nl], dl), f
        assert np.array_equal(out["kps_r"][f, :nr], kr) and np.array_equal(out["desc_r"][f, :nr], dr), f
        assert np.array_equal(out["stereo_idx"][f, :nl], si[f][0]) and np.array_equal(out["stereo_dist"][f, :nl], si[f][1]), f
        assert (si[f][0] > 2047).sum() > 0, f


# ---- ProjectionMatch on other cameras -------------------------------------------------------------------------------
SE3_ID = np.array([0, 0, 0, 1, 0, 0, 0], np.float64)


def _proj_entry_points(m, oracle, xw, mpd, skip, pose, cam, ocam, kps, desc, radius, grid):
    """Matcher.ProjectionMatch, the _dev call, Frame.ProjectionMatch and three keys_dev shards + merge, each against the
    oracle; -> the oracle's result"""
    ref = oracle.projection_match(xw, mpd, skip, pose, ocam, kps, desc, radius, grid=grid)
    n, mk = len(xw), len(kps)
    tag = f"n={n} m={mk} r={radius} pose={len(np.ravel(pose))} {cam.width}x{cam.height}"
    got = m.ProjectionMatch(xw, mpd, skip, pose, cam, kps, desc, radius)
    assert np.array_equal(got[0], ref[0]) and np.array_equal(got[1], ref[1]), f"host {tag}: {(got[0] != ref[0]).sum()} differ"
    d_xw, d_mpd = api.DeviceBuffer(xw.nbytes).upload(xw), api.DeviceBuffer(mpd.nbytes).upload(mpd)
    d_skip = None if skip is None else api.DeviceBuffer(skip.nbytes).upload(skip)
    d_kps, d_desc = api.DeviceBuffer(kps.nbytes).upload(kps), api.DeviceBuffer(desc.nbytes).upload(desc)
    d_q, d_d, d_keys = api.DeviceBuffer(4 * mk), api.DeviceBuffer(4 * mk), api.DeviceBuffer(8 * 3 * mk)
    m.projection_match_dev(d_xw.ptr, d_mpd.ptr, None if skip is None else d_skip.ptr, n, pose, cam, d_kps.ptr, d_desc.ptr, mk,
                           radius, d_q.ptr, d_d.ptr)
    assert np.array_equal(d_q.download(mk, np.int32), ref[0]) and np.array_equal(d_d.download(mk, np.int32), ref[1]), f"dev {tag}"
    fr = api.Frame(m, kps, desc, cam)
    got = fr.ProjectionMatch(xw, mpd, skip, pose, radius)
    assert np.array_equal(got[0], ref[0]) and np.array_equal(got[1], ref[1]), f"frame {tag}"
    fr.close()
    cuts = [0, n // 3, (2 * n) // 3 + 1, n]
    for s in range(3):
        lo, cnt = cuts[s], cuts[s + 1] - cuts[s]
        m.projection_match_keys_dev(d_xw.ptr + 24 * lo, d_mpd.ptr + 32 * lo, None if skip is None else d_skip.ptr + lo, cnt, lo,
                                    pose, cam, d_kps.ptr, d_desc.ptr, mk, radius, d_keys.ptr + 8 * mk * s)
    d_q2, d_d2 = api.DeviceBuffer(4 * mk), api.DeviceBuffer(4 * mk)
    m.projection_merge_dev(d_keys.ptr, 3, mk, d_q2.ptr, d_d2.ptr)
    assert np.array_equal(d_q2.download(mk, np.int32), ref[0]) and np.array_equal(d_d2.download(mk, np.int32), ref[1]), f"shards {tag}"
    return ref


def _pinhole_scene(w, h, m, n, radius, seed):
    """Camera fx = fy = 1, c = 0, no distortion: under the identity pose map point (u, v, 1) projects exactly to (u, v).
    Keypoints over [-8, w + 8] x [-8, h + 8] (some outside the image), map points near keypoints with their descriptor
    lightly perturbed, plus planted points: keypoints exactly on the search circle (excluded, T4) that would win if they
    counted, and map points exactly at u == width, v == height with their keypoints just outside the image."""
    rng = np.random.default_rng(seed)
    kx, ky = rng.uniform(-8, w + 8, m).astype(F32), rng.uniform(-8, h + 8, m).astype(F32)
    desc = rng.integers(0, 256, (m, 32), dtype=np.uint8)
    src = rng.integers(0, m, n)
    ang, rad = rng.uniform(0, 2 * np.pi, n), rng.uniform(0, 0.9 * min(radius, 40.0), n)
    u, v = kx[src] + rad * np.cos(ang), ky[src] + rad * np.sin(ang)
    mpd = desc[src] ^ (rng.integers(0, 256, (n, 32), dtype=np.uint8) & rng.integers(0, 256, (n, 32), dtype=np.uint8)
                       & rng.integers(0, 256, (n, 32), dtype=np.uint8))
    far = rng.uniform(size=n) < 0.3
    u[far], v[far] = rng.uniform(-3, w + 3, far.sum()), rng.uniform(-3, h + 3, far.sum())
    mpd[far] = rng.integers(0, 256, (far.sum(), 32), dtype=np.uint8)
    skip = (rng.uniform(size=n) < 0.05).astype(np.uint8)
    # planted (query q, keypoints); the keypoint index at the end of the list, which the oracle must confirm
    r = float(radius)
    spots = [(0.5 * w, 0.5 * h), (float(w), float(h)), (0.0, 0.0), (float(w), 0.0)]
    expect = {}
    kslots = [int(j) for j in rng.permutation(m)[:3 * len(spots)]]
    qslots = [int(q) for q in rng.permutation(n)[:len(spots)]]
    for (pu, pv), q in zip(spots, qslots):
        D = rng.integers(0, 256, 32, dtype=np.uint8)
        a, b, c = kslots.pop(), kslots.pop(), kslots.pop()
        u[q], v[q], mpd[q], skip[q] = pu, pv, D, 0
        sx = -1.0 if pu > 0 else 1.0
        sy = -1.0 if pv > 0 else 1.0
        if r == 5.0:   # on the circle: 3-4-5 offsets, d^2 == r^2 exactly; distance 0 but excluded
            kx[a], ky[a], desc[a] = pu + 3 * sx, pv + 4 * sy, D
        else:
            kx[a], ky[a], desc[a] = pu + sx * r, pv, _flipped(D, 40, rng)
        kx[b], ky[b], desc[b] = pu - 1.5 * sx, pv - 1.0 * sy, _flipped(D, 5, rng)      # outside the image: wins
        kx[c], ky[c], desc[c] = pu + 0.5 * sx, pv + 0.5 * sy, _flipped(D, 30, rng)
        expect[b] = q
    xw = np.stack([u, v, np.ones(n)], 1)
    return xw, mpd, skip, _kps(kx, ky), desc, expect


@pytest.mark.parametrize("w,h,m,n,radius", [(20, 10, 60, 200, 5.0), (20, 10, 60, 200, 50.0),
                                            (1280, 720, 65535, 32767, 5.0), (1280, 720, 65535, 32768, 5.0),
                                            (1280, 720, 300, 32768, 2000.0)])
def test_projection_match_pinhole_cameras(matcher, oracle, w, h, m, n, radius):
    """A 1 x 1 bucket grid (20 x 10), a width that is a multiple of 32 (u == width falls into the grid's extra column),
    radii on and beyond the image diagonal, 32767 / 32768 map points (the two sides of the sorted path) and 65535
    keypoints with winners above index 32767 (the 16 key bits that carry the keypoint index)."""
    xw, mpd, skip, kps, desc, expect = _pinhole_scene(w, h, m, n, radius, seed=w + n + int(radius))
    cam = api.Camera.make(1.0, 1.0, 0.0, 0.0, [0, 0, 0, 0], w, h)
    ocam = oracle.make_camera(1.0, 1.0, 0.0, 0.0, [0, 0, 0, 0], w, h)
    grid = m * n > 10 ** 6
    for pose in (np.eye(3, 4), SE3_ID):
        for sk in (None, skip):
            ref = _proj_entry_points(matcher, oracle, xw, mpd, sk, pose, cam, ocam, kps, desc, radius, grid)
            if radius == 5.0:
                for b, q in expect.items():
                    assert ref[0][b] == q and ref[1][b] == 5, (b, q, ref[0][b], ref[1][b])
            assert (ref[0] >= 0).sum() >= min(m, n) // 20
            if m == 65535:
                assert (ref[0][32768:] >= 0).sum() > 100


def test_projection_match_distorted_4k_camera(matcher, oracle):
    """3840 x 2160 with distortion: 8228 bucket cells, more than the sorted path's 1024 bins; keypoints beyond every
    image border; a real pose as a 3 x 4 matrix and as an SE3Quat; map points on both sides of the sorted path."""
    rng = np.random.default_rng(41)
    w, h, m = 3840, 2160, 20000
    fx, cx, cy, dist = 1800.0, 1920.0, 1080.0, [-0.05, 0.01, 0.001, -0.002]
    cam = api.Camera.make(fx, fx, cx, cy, dist, w, h)
    ocam = oracle.make_camera(fx, fx, cx, cy, dist, w, h)
    kps = _kps(rng.uniform(-20, w + 20, m).astype(F32), rng.uniform(-20, h + 20, m).astype(F32))
    desc = rng.integers(0, 256, (m, 32), dtype=np.uint8)
    nrm = oracle.normalized_undistort(ocam, kps)
    th = 0.01
    R = np.array([[np.cos(th), 0, np.sin(th)], [0, 1, 0], [-np.sin(th), 0, np.cos(th)]])
    t = np.array([0.05, -0.02, 0.1])
    qt = np.array([0, np.sin(th / 2), 0, np.cos(th / 2), *t])
    for n in (30000, 40000):
        src = rng.integers(0, m, n)
        z = rng.uniform(2, 60, n)
        xc = np.stack([nrm[src, 0] * z, nrm[src, 1] * z, z], 1) + rng.normal(0, 0.01, (n, 3))
        xw = (xc - t) @ R           # Xw = R^T (Xc - t): projects back near the source keypoint
        mpd = desc[src] ^ (rng.integers(0, 256, (n, 32), dtype=np.uint8) & rng.integers(0, 256, (n, 32), dtype=np.uint8)
                           & rng.integers(0, 256, (n, 32), dtype=np.uint8))
        for pose in (np.concatenate([R, t[:, None]], 1), qt):
            ref = _proj_entry_points(matcher, oracle, xw, mpd, None, pose, cam, ocam, kps, desc, 30.0, True)
            assert (ref[0] >= 0).sum() > m // 4


# ---- frame glue on a dense, degenerate frame -------------------------------------------------------------------------
def test_frame_search_on_dense_frame_with_duplicates(matcher, oracle):
    """About 5000 keypoints, 1200 of them in one 32-px cell, 500 exact duplicates and 800 on an integer lattice, indices
    shuffled so that index order is not cell order: SearchNeareast's tie rule (T6), SearchRadius on and inside the radius,
    and truncated rows holding the cap smallest indices."""
    rng = np.random.default_rng(17)
    xs = [rng.uniform(-10, 1250, 2500), rng.uniform(320, 352, 1200), rng.integers(0, 1241, 800).astype(np.float64)]
    ys = [rng.uniform(-10, 385, 2500), rng.uniform(160, 192, 1200), rng.integers(0, 376, 800).astype(np.float64)]
    x, y = np.concatenate(xs).astype(F32), np.concatenate(ys).astype(F32)
    dup = rng.integers(0, len(x), 500)
    dup_xy = np.stack([x[dup], y[dup]], 1).astype(np.float64)
    x, y = np.concatenate([x, x[dup]]), np.concatenate([y, y[dup]])
    perm = rng.permutation(len(x))
    kps = _kps(x[perm], y[perm])
    desc = rng.integers(0, 256, (len(kps), 32), dtype=np.uint8)
    cam = api.Camera.make(synth.KITTI_FX, synth.KITTI_FY, synth.KITTI_CX, synth.KITTI_CY, [0] * 4, 1241, 376)
    fr = api.Frame(matcher, kps, desc, cam)
    lattice = np.nonzero((kps["x"] == np.round(kps["x"])) & (kps["y"] == np.round(kps["y"])))[0][:100]
    assert len(lattice) == 100
    uv = np.concatenate([
        dup_xy[:150],                                                                           # on duplicated keypoints
        np.stack([kps["x"], kps["y"]], 1)[rng.integers(0, len(kps), 100)],                     # on keypoints
        np.stack([kps["x"][lattice] - 3.0, kps["y"][lattice] - 4.0], 1),                        # 3-4-5 from a lattice point
        np.stack([rng.uniform(300, 372, 100), rng.uniform(140, 212, 100)], 1),                  # in and around the dense cell
        np.stack([rng.uniform(-30, 1270, 100), rng.uniform(-30, 400, 100)], 1)]).astype(np.float64)
    gi, gd = fr.SearchNeareast(uv)
    ties = 0
    for i in range(len(uv)):
        ri, rd = oracle.search_nearest(kps, uv[i, 0], uv[i, 1])
        assert gi[i] == ri and gd[i].tobytes() == np.float64(rd).tobytes(), (i, gi[i], ri)
        d2 = (uv[i, 0] - kps["x"].astype(np.float64)) ** 2 + (uv[i, 1] - kps["y"].astype(np.float64)) ** 2
        ties += (d2 == rd).sum() > 1
    assert ties >= 150
    on_circle = 0
    for radius in (5.0, 12.0):
        got = fr.SearchRadius(uv, radius, cap=2048)
        for i in range(len(uv)):
            ref, cnt = oracle.search_radius(kps, uv[i, 0], uv[i, 1], radius)
            assert cnt == len(got[i]) and np.array_equal(got[i], ref), (radius, i)
            d2 = (uv[i, 0] - kps["x"].astype(np.float64)) ** 2 + (uv[i, 1] - kps["y"].astype(np.float64)) ** 2
            on_circle += (d2 == radius * radius).sum()
    assert on_circle > 50
    # truncated rows: counts hold the full count, each row the cap smallest indices (sfe.h)
    cap, radius = 4, 20.0
    idx = np.full((len(uv), cap), -7, np.int32)
    counts = np.zeros(len(uv), np.int32)
    api._check(api.lib().sfe_frame_search_radius(matcher.h, fr.h, api._p(uv), len(uv), radius, api._p(idx), cap,
                                                 api._p(counts)))
    truncated = 0
    for i in range(len(uv)):
        ref, cnt = oracle.search_radius(kps, uv[i, 0], uv[i, 1], radius)
        assert counts[i] == cnt, i
        k = min(cnt, cap)
        assert np.array_equal(idx[i, :k], ref[:k]), (i, idx[i, :k], ref[:k])
        truncated += cnt > cap
    assert truncated > 200


# ---- vocabulary descent with wide nodes ------------------------------------------------------------------------------
def _tree(branching, L, seed):
    """Breadth-first vocabulary; branching(level, ordinal) = children of the ordinal-th node of that level (0 = leaf).
    Children share most bits with their parent, as in synth.vocabulary."""
    rng = np.random.default_rng(seed)
    parent, is_leaf, desc, depth = [0], [0], [np.zeros(32, np.uint8)], [0]
    frontier = [0]
    for level in range(1, L + 1):
        nxt = []
        for o, p in enumerate(frontier):
            for _ in range(branching(level, o)):
                parent.append(p)
                desc.append(_flipped(desc[p], 24 if level > 1 else 128, rng))
                kids = branching(level + 1, len(nxt)) if level < L else 0
                is_leaf.append(0 if kids else 1)
                if kids:
                    nxt.append(len(parent) - 1)
        frontier = nxt
    weight = np.where(np.array(is_leaf) == 1, rng.uniform(0.1, 9.0, len(parent)), 0.0)
    return np.array(parent, np.int32), np.array(is_leaf, np.uint8), np.stack(desc).astype(np.uint8), weight


def _transform_both(voc, feats, levelsup):
    host = voc.transform_features(feats, levelsup)
    n = len(feats)
    d_f, d_n = api.DeviceBuffer(feats.nbytes).upload(feats), api.DeviceBuffer(4).upload(np.array([n], np.int32))
    d_w, d_wt, d_nid = api.DeviceBuffer(4 * n), api.DeviceBuffer(8 * n), api.DeviceBuffer(4 * n)
    d_off, d_ids, d_val = api.DeviceBuffer(16), api.DeviceBuffer(4 * n), api.DeviceBuffer(8 * n)
    voc.transform_dev(d_f.ptr, d_n.ptr, 1, n, levelsup, d_w.ptr, d_wt.ptr, d_nid.ptr, d_off.ptr, d_ids.ptr, d_val.ptr)
    dev = (d_w.download(n, np.int32), d_wt.download(n, np.float64), d_nid.download(n, np.int32))
    return host, dev


def _check_transform(m, oracle, tree, L, feats, levelsups):
    parent, is_leaf, ndesc, weight = tree
    voc = api.Vocabulary(m, parent, is_leaf, ndesc, weight, L)
    for levelsup in levelsups:
        ref = oracle.vocab_transform(parent, is_leaf, ndesc, weight, L, feats, levelsup)
        for got in _transform_both(voc, feats, levelsup):
            assert np.array_equal(got[0], ref[0]) and np.array_equal(got[2], ref[2]), levelsup
            assert np.array_equal(got[1].view(np.uint64), ref[1].view(np.uint64)), levelsup
    voc.close()
    return ref


def _plant_ties(tree, p, rng):
    """Features that reach node p (a few bits from its descriptor) and whose best children of p sit in different lane
    rounds: for each far rank r >= 32, an exact tie between r and a partner 32 ranks earlier (rank 0 for the first),
    which the partner must win, and a unique best at r.  Edits the descriptors of p's children in place.
    -> (features, the child each must reach)"""
    parent, _, ndesc, _ = tree
    kids = np.nonzero(parent == p)[0]
    kids = kids[kids > 0]
    feats, want = [], []
    for r, partner in _tie_ranks(len(kids)):
        X = _flipped(ndesc[p], 4, rng)
        a, b = rng.choice(256, 2, replace=False)
        F = X.copy()
        F[a >> 3] ^= np.uint8(1 << (a & 7))
        ndesc[kids[r]] = X
        ndesc[kids[partner]] = F.copy()
        ndesc[kids[partner]][b >> 3] ^= np.uint8(1 << (b & 7))
        feats += [F, X]                      # F: distance 1 to both (partner wins); X: distance 0 to r, 2 to the partner
        want += [kids[partner], kids[r]]
    return feats, want


def _tie_ranks(nk):
    far = sorted({32, nk - 1} | ({40} if nk > 41 else set()))
    return list(zip(far, [0] + [r - 32 for r in far[1:]]))


def _ancestors(parent, node):
    out = []
    while node:
        node = int(parent[node])
        out.append(node)
    return out


@pytest.mark.parametrize("root_k", [33, 64, 100, "uneven"])
def test_vocab_descent_with_wide_nodes(matcher, oracle, root_k):
    """Nodes with more than 32 children take several lane rounds: ties across rounds go to the earlier child, winners at
    rank >= 32 keep their rank; node ids at levelsup 0, 1, L and L + 2."""
    rng = np.random.default_rng(5 if root_k == "uneven" else root_k)
    if root_k == "uneven":   # 40 children at the root, then nodes of 40 and of 3 children, alternating
        L = 3
        tree = _tree(lambda level, o: 40 if level == 1 else (40 if o % 2 else 3), L, seed=3)
    else:
        L = 2
        tree = _tree(lambda level, o: root_k if level == 1 else 4, L, seed=root_k)
    parent, ndesc = tree[0], tree[2]
    counts = np.bincount(parent[1:], minlength=len(parent))
    wide = [int(p) for p in np.nonzero(counts > 32)[0]]
    # the root last, deeper nodes first; a node is planted only where no planting edits its ancestors' descriptors
    root_kids = np.nonzero(parent == 0)[0][1:]
    edited = {int(root_kids[r]) for pair in _tie_ranks(len(root_kids)) for r in pair}
    deeper = [p for p in wide[1:] if not edited & set(_ancestors(parent, p)) and p not in edited]
    planted, want = [], []
    for p in deeper[:2] + deeper[-2:] + [0]:
        f, w = _plant_ties(tree, p, rng)
        planted += f
        want += w
    feats = np.concatenate([np.stack(planted), ndesc[rng.integers(1, len(ndesc), 400)],
                            rng.integers(0, 256, (200, 32), dtype=np.uint8)]).astype(np.uint8)
    ref = _check_transform(matcher, oracle, tree, L, feats, (0, 1, L, L + 2))
    assert len(np.unique(ref[0])) > 20
    # each planted feature reaches the child it was planted for (the node id at that child's level)
    for level in sorted({len(_ancestors(parent, w)) for w in want}):
        nid = oracle.vocab_transform(*tree, L, np.stack(planted), L - level)[2]
        for i, w in enumerate(want):
            if len(_ancestors(parent, w)) == level:
                assert nid[i] == w, (root_k, i, nid[i], w)


def test_vocab_child_rank_limit(matcher, oracle):
    """The descent ranks a node's children in 20 bits: a root with 2^20 children is refused, one with 2^20 - 1 children
    descends like the oracle, ties between rank 0 and the last ranks included."""
    n = 1 << 20
    rng = np.random.default_rng(23)
    for n_nodes, ok in ((n + 1, False), (n, True)):
        parent = np.zeros(n_nodes, np.int32)
        is_leaf = np.ones(n_nodes, np.uint8)
        is_leaf[0] = 0
        ndesc = rng.integers(0, 256, (n_nodes, 32), dtype=np.uint8)
        weight = rng.uniform(0.1, 9.0, n_nodes)
        if not ok:
            with pytest.raises(api.SfeError) as e:
                api.Vocabulary(matcher, parent, is_leaf, ndesc, weight, 1)
            assert e.value.status == api.SFE_ERR_UNSUPPORTED
            continue
        ndesc[n - 1] = ndesc[1]                  # exact tie between the first and the last child: rank 0 wins
        feats = np.stack([ndesc[1], ndesc[n - 2], ndesc[700001], _flipped(ndesc[n - 3], 1, rng),
                          *rng.integers(0, 256, (4, 32), dtype=np.uint8)])
        ref = _check_transform(matcher, oracle, (parent, is_leaf, ndesc, weight), 1, feats, (0, 1))
        assert ref[0][:4].tolist() == [0, n - 3, 700000, n - 4]


# ---- tracking with an SE3Quat motion prior ---------------------------------------------------------------------------
def _oracle_track(oracle, out, frames, ocam, baseline, pose, radius):
    res = []
    for f in range(1, frames):
        npv, nrp, nl = int(out["n_l"][f - 1]), int(out["n_r"][f - 1]), int(out["n_l"][f])
        kl, dl, kr = out["kps_l"][f - 1, :npv], out["desc_l"][f - 1, :npv], out["kps_r"][f - 1, :nrp]
        sidx = out["stereo_idx"][f - 1, :npv]
        xc, valid = oracle.stereo_depth(ocam, baseline, kl, oracle.normalized_undistort(ocam, kl), kr, sidx)
        rows = np.nonzero(valid == 1)[0]
        to_q, dist = oracle.projection_match(xc[rows], dl[rows], None, pose, ocam, out["kps_l"][f, :nl], out["desc_l"][f, :nl],
                                             radius)
        res.append((np.where(to_q >= 0, rows[np.maximum(to_q, 0)], -1).astype(np.int32), dist))
    return res


def test_tracking_with_se3_motion_prior(gpu, oracle):
    """sfe_stereo_sequence and its resident form with a 7-value SE3Quat prior that is not the identity, on a distorted
    camera: GetDepth of frame f - 1, then ProjectionMatch of its stereo points under the prior into frame f."""
    F, radius = 4, 12.0
    L, R = synth.stereo_sequence(6, F, step=4)
    dist = [-0.05, 0.01, 0.001, -0.002]
    cam = api.Camera.make(synth.KITTI_FX, synth.KITTI_FY, synth.KITTI_CX, synth.KITTI_CY, dist, synth.KITTI_W, synth.KITTI_H)
    ocam = oracle.make_camera(synth.KITTI_FX, synth.KITTI_FY, synth.KITTI_CX, synth.KITTI_CY, dist, synth.KITTI_W, synth.KITTI_H)
    th = 0.006
    qt = np.array([0.0, np.sin(th / 2), 0.0, np.cos(th / 2), -0.08, 0.01, 0.02])
    tp = api.TrackParams.make(cam, synth.KITTI_BASELINE, qt, radius)
    assert tp.use_se3 == 1
    ex = api.ORBextractor(max_images=2 * F)
    out = ex.stereo_sequence(L, R, tp)
    ref = _oracle_track(oracle, out, F, ocam, synth.KITTI_BASELINE, qt, radius)
    ident = _oracle_track(oracle, out, F, ocam, synth.KITTI_BASELINE, SE3_ID, radius)
    for f in range(1, F):
        nl = int(out["n_l"][f])
        assert np.array_equal(out["track_idx"][f, :nl], ref[f - 1][0]), f"frame {f}: {(out['track_idx'][f, :nl] != ref[f - 1][0]).sum()} differ"
        assert np.array_equal(out["track_dist"][f, :nl], ref[f - 1][1]), f
        assert (ref[f - 1][0] >= 0).sum() > 100 and not np.array_equal(ref[f - 1][0], ident[f - 1][0]), f
    cap, h, w = ex.cap, *L.shape[1:]
    dl, dr = api.DeviceBuffer(L.nbytes).upload(L), api.DeviceBuffer(R.nbytes).upload(R)
    spec = {"kps_l": (28, api.KP_DTYPE, (F, cap)), "desc_l": (32, np.uint8, (F, cap, 32)), "n_l": (0, np.int32, (F,)),
            "kps_r": (28, api.KP_DTYPE, (F, cap)), "desc_r": (32, np.uint8, (F, cap, 32)), "n_r": (0, np.int32, (F,)),
            "stereo_idx": (4, np.int32, (F, cap)), "stereo_dist": (4, np.int32, (F, cap)), "track_idx": (4, np.int32, (F, cap)),
            "track_dist": (4, np.int32, (F, cap))}
    bufs = {k: api.DeviceBuffer(max(b * cap * F, 4 * F)) for k, (b, _, _) in spec.items()}
    ex.stereo_sequence_dev(dl.ptr, dr.ptr, F, w, h, {k: b.ptr for k, b in bufs.items()}, tp)
    dev = {k: bufs[k].download(shape, dt) for k, (_, dt, shape) in spec.items()}
    for f in range(F):
        nl = int(out["n_l"][f])
        assert int(dev["n_l"][f]) == nl and np.array_equal(dev["stereo_idx"][f, :nl], out["stereo_idx"][f, :nl])
        assert np.array_equal(dev["track_idx"][f, :nl], out["track_idx"][f, :nl])
        assert np.array_equal(dev["track_dist"][f, :nl], out["track_dist"][f, :nl])
