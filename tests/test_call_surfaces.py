"""The host call surfaces a user links, checked value by value against the oracle.

- include/sfe_adapter.hpp driven by tests/cpp/adapter_values.cpp: ProjectionMatch with a real SE3, a distorted camera,
  skips reported through Frame::GetIndex and a std::set whose iteration order is not the creation order; extract and
  extractStereo on cv::Mats with padded rows and on an image wide enough to grow the adapter's capacity.
- sfe_extract_batch / sfe_stereo_frames on host images with padded rows and gaps between images.
- the Python API with caller-allocated `out` arrays whose capacity differs from the extractor's.
- several matcher handles searching one database at once (its tensor-core tiles are built by whichever search comes
  first), and the adapter used from two threads with one handle each.
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

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
DRIVER_SRC = os.path.join(ROOT, "tests", "cpp", "adapter_values.cpp")
GOLDEN = os.path.join(ROOT, "tests", "golden")
W, H = synth.KITTI_W, synth.KITTI_H
DIST = (-0.05, 0.01, 0.001, -0.002)
NTHREADS = os.cpu_count() or 4


@functools.lru_cache(maxsize=None)
def _driver() -> str:
    """tests/cpp/adapter_values.cpp compiled into a temporary directory (the source tree may be read-only), linked
    against the in-tree libsfe.so"""
    import __graft_entry__ as g
    if not os.path.exists(api.LIB_PATH):
        g.build()
    out = tempfile.mkdtemp(prefix="sfe_adapter_values_")
    atexit.register(shutil.rmtree, out, True)
    exe = os.path.join(out, "adapter_values")
    libdir = os.path.dirname(os.path.abspath(api.LIB_PATH))
    subprocess.check_call(["g++", "-std=c++14", "-O1", "-Wall", "-pthread", "-o", exe, DRIVER_SRC, api.LIB_PATH,
                           f"-Wl,-rpath,{libdir}"])
    return exe


@pytest.fixture(scope="module")
def gpu():
    if api.device_count() < 1:
        pytest.fail("no CUDA device: the product has no CPU fallback")
    _driver()
    return 0


def _run(*args, timeout=600):
    p = subprocess.run([_driver()] + [str(a) for a in args], capture_output=True, text=True, timeout=timeout)
    assert p.returncode == 0, p.stdout + p.stderr
    return dict(kv.split("=") for kv in p.stdout.split())


# ---- adapter driver I/O --------------------------------------------------------------------------------------------
def _write_proj(d, xw, mpd, inframe, slot, kps, kdesc, cam, calls):
    """cam = (fx, fy, cx, cy, d[4], width, height); calls = [(qt[7], radius)]"""
    os.makedirs(d, exist_ok=True)
    n, m = len(xw), len(kps)
    fx, fy, cx, cy, dist, w, h = cam
    with open(os.path.join(d, "meta.txt"), "w") as f:
        f.write(f"{n} {m} {w} {h} {fx!r} {fy!r} {cx!r} {cy!r} " + " ".join(repr(float(v)) for v in dist) + f" {len(calls)}\n")
        for qt, r in calls:
            f.write(" ".join(repr(float(v)) for v in qt) + f" {float(r)!r}\n")
    np.ascontiguousarray(xw, "<f8").tofile(os.path.join(d, "xw.f64"))
    np.ascontiguousarray(mpd, np.uint8).tofile(os.path.join(d, "mpdesc.u8"))
    np.ascontiguousarray(inframe, np.uint8).tofile(os.path.join(d, "inframe.u8"))
    np.ascontiguousarray(slot, "<i4").tofile(os.path.join(d, "slot.i32"))
    np.ascontiguousarray(kps, api.KP_DTYPE).tofile(os.path.join(d, "kps.kp"))
    np.ascontiguousarray(kdesc, np.uint8).tofile(os.path.join(d, "kdesc.u8"))


def _read_proj(d, calls, m):
    return np.fromfile(os.path.join(d, "out.i32"), "<i4").reshape(calls, m)


def _adapter_proj(d, *case):
    _write_proj(d, *case)
    _run("proj", d)
    return _read_proj(d, len(case[-1]), len(case[4]))


def _write_extract(d, L, R, step, params=(2000, 1.2, 8, 20, 7)):
    os.makedirs(d, exist_ok=True)
    h, w = L.shape
    with open(os.path.join(d, "meta.txt"), "w") as f:
        f.write(f"{w} {h} {step} " + " ".join(str(p) for p in params) + "\n")
    np.ascontiguousarray(L, np.uint8).tofile(os.path.join(d, "l.u8"))
    np.ascontiguousarray(R, np.uint8).tofile(os.path.join(d, "r.u8"))


def _read_extract(d):
    """-> [(kps, desc)] for extract(L), extract(R), extractStereo left, extractStereo right; + stereo indices"""
    b = np.fromfile(os.path.join(d, "out.bin"), np.uint8)
    o, feats = 0, []
    for _ in range(4):
        n = int(b[o:o + 4].view("<i4")[0])
        o += 4
        k = b[o:o + 28 * n].copy().view(api.KP_DTYPE)
        o += 28 * n
        feats.append((k, b[o:o + 32 * n].reshape(n, 32).copy()))
        o += 32 * n
    n = int(b[o:o + 4].view("<i4")[0])
    sidx = b[o + 4:o + 4 + 4 * n].copy().view("<i4")
    assert o + 4 + 4 * n == len(b)
    return feats, sidx


@functools.lru_cache(maxsize=None)
def _oracle_frame(seed, w=W, h=H, params=(2000, 1.2, 8, 20, 7)):
    import oracle_c
    oracle_c.build()
    L, R = synth.stereo_pair(seed, w, h)
    ref = oracle_c.Extractor(*params)
    kl, dl = ref.extract(L)
    kr, dr = ref.extract(R)
    si, _ = oracle_c.stereo_match(kl, dl, kr, dr)
    return L, R, kl, dl, kr, dr, si


def _check_extract(d, seed, w=W, h=H, params=(2000, 1.2, 8, 20, 7)):
    L, R, kl, dl, kr, dr, si = _oracle_frame(seed, w, h, params)
    feats, sidx = _read_extract(d)
    for (k, desc), (rk, rd), what in zip(feats, [(kl, dl), (kr, dr), (kl, dl), (kr, dr)],
                                         ["extract(L)", "extract(R)", "extractStereo L", "extractStereo R"]):
        assert len(k) == len(rk), what
        assert k.tobytes() == rk.tobytes() and np.array_equal(desc, rd), what
    assert np.array_equal(sidx, si)


# ---- the ProjectionMatch scenes ------------------------------------------------------------------------------------
def _quat(axis, angle):
    a = np.asarray(axis, np.float64)
    a = a / np.linalg.norm(a)
    return np.concatenate([a * np.sin(angle / 2), [np.cos(angle / 2)]])


def _rot(q):
    x, y, z, w = q
    return np.array([[1 - 2 * (y * y + z * z), 2 * (x * y - z * w), 2 * (x * z + y * w)],
                     [2 * (x * y + z * w), 1 - 2 * (x * x + z * z), 2 * (y * z - x * w)],
                     [2 * (x * z - y * w), 2 * (y * z + x * w), 1 - 2 * (x * x + y * y)]])


IDENT = np.array([0, 0, 0, 1, 0, 0, 0], np.float64)
# a real SE3: 3 degrees about a tilted axis, 4.5 m backwards -- the near points (z < ~4.5 m) end up behind the camera
SE3_POSE = np.concatenate([_quat([0.3, -1.0, 0.2], np.deg2rad(3.0)), [0.4, -0.15, -4.5]])
SE3_NEG = np.concatenate([-SE3_POSE[:4], SE3_POSE[4:]])


@functools.lru_cache(maxsize=None)
def _conflict_scene():
    """Seed-0 frame; for 160 keypoints per pose (identity and SE3_POSE) a cluster of 2-4 map points that project within 2 px
    of the keypoint under that pose and carry its descriptor with the same k <= 4 bits flipped (distinct bits per point), so
    their distances tie and the later query in set order takes the keypoint (src/matcher.cpp:197-204); 3000 background
    points (synth.projection_scene); ~5 % of all points are reported in-frame by GetIndex.  Returns
    (xw, mp_desc, inframe, slot, kps, kdesc)."""
    g = np.load(os.path.join(GOLDEN, "golden_seed0.npz"))
    kl, dl = g["kl"], g["dl"]
    rng = np.random.default_rng(2024)
    xw, md = [], []
    for pose in (IDENT, SE3_POSE):
        R, t = _rot(pose[:4]), pose[4:]
        for j in rng.choice(len(kl), 160, replace=False):
            npts, k = int(rng.integers(2, 5)), int(rng.integers(1, 5))
            z = rng.uniform(2.5, 40.0)
            bits = rng.choice(256, npts * k, replace=False).reshape(npts, k)
            for p in range(npts):
                u = kl["x"][j] + rng.uniform(-2, 2)
                v = kl["y"][j] + rng.uniform(-2, 2)
                xc = np.array([(u - synth.KITTI_CX) / synth.KITTI_FX * z, (v - synth.KITTI_CY) / synth.KITTI_FY * z, z])
                xw.append(R.T @ (xc - t))  # Xc = R Xw + t
                d = dl[j].copy()
                for b in bits[p]:
                    d[b >> 3] ^= np.uint8(1 << (b & 7))
                md.append(d)
    bx, bd = synth.projection_scene(np.stack([kl["x"], kl["y"]], 1).astype(np.float64), dl, 3000, seed=7)
    xw = np.concatenate([np.array(xw), bx])
    md = np.concatenate([np.array(md, np.uint8), bd])
    n = len(xw)
    inframe = (rng.random(n) < 0.05).astype(np.uint8)
    slot = rng.permutation(n).astype(np.int32)
    return xw, md, inframe, slot, kl, dl


def _cam_tuple(dist):
    return (synth.KITTI_FX, synth.KITTI_FY, synth.KITTI_CX, synth.KITTI_CY, tuple(dist), W, H)


def _oracle_in_order(order, xw, md, inframe, kps, kdesc, qt, cam, radius):
    """oracle ProjectionMatch with the map points queried in `order`, mapped back to the caller's point indices"""
    import oracle_c
    oc = oracle_c.make_camera(*cam[:4], list(cam[4]), cam[5], cam[6])
    to_q, _ = oracle_c.projection_match(xw[order], md[order], inframe[order], qt, oc, kps, kdesc, float(radius), grid=True)
    return np.where(to_q >= 0, order[np.maximum(to_q, 0)], -1).astype(np.int32)


RADII = (10, 50, 100)
POSES = (IDENT, SE3_POSE, SE3_NEG)


# ---- the driver without a device -----------------------------------------------------------------------------------
def test_adapter_values_compiles_and_has_no_cpu_fallback(tmp_path):
    exe = _driver()
    if api.device_count() > 0:
        pytest.skip("a CUDA device is present")
    L, R = synth.stereo_pair(0, 160, 120)
    _write_extract(tmp_path, L, R, 173)
    p = subprocess.run([exe, "extract", str(tmp_path)], capture_output=True, text=True, timeout=120)
    assert p.returncode == 1 and "exception" in p.stdout and "sfe_extractor_create" in p.stdout


# ---- B: the adapter, value by value --------------------------------------------------------------------------------
@pytest.mark.gpu
def test_adapter_projection_match_golden_fixture(gpu, tmp_path):
    """golden_proj.npz (the reference's own result) through sfe_adapter::ProjectionMatch: distorted camera, real SE3,
    skips via Frame::GetIndex.  Identity slots: set order = the fixture's array order."""
    z = np.load(os.path.join(GOLDEN, "golden_proj.npz"))
    g = np.load(os.path.join(GOLDEN, "golden_seed0.npz"))
    n = len(z["xw"])
    got = _adapter_proj(tmp_path, z["xw"], z["mp_desc"], z["skip"], np.arange(n, dtype=np.int32), g["kl"], g["dl"],
                        _cam_tuple(z["dist4"]), [(z["qt"], 50), (z["qt"], 10)])
    assert np.array_equal(got[0], z["to_query_r50"])
    assert np.array_equal(got[1], z["to_query_r10"])


@pytest.mark.gpu
@pytest.mark.parametrize("dist", [(0, 0, 0, 0), DIST], ids=["pinhole", "distorted"])
def test_adapter_projection_match_follows_set_order(gpu, oracle, tmp_path, dist):
    xw, md, inframe, slot, kps, kdesc = _conflict_scene()
    cam = _cam_tuple(dist)
    calls = [(qt, r) for qt in POSES for r in RADII]
    got = _adapter_proj(tmp_path, xw, md, inframe, slot, kps, kdesc, cam, calls)
    slot_order = np.argsort(slot)  # slot_order[s] = the point at slot s = the s-th point std::set visits
    creation = np.arange(len(xw))
    teeth = 0
    for c, (qt, r) in enumerate(calls):
        want = _oracle_in_order(slot_order, xw, md, inframe, kps, kdesc, qt, cam, r)
        assert np.array_equal(got[c], want), (qt.tolist(), r, int((got[c] != want).sum()))
        if c < 3:  # identity pose: the conflicts were placed for it
            teeth += int((_oracle_in_order(creation, xw, md, inframe, kps, kdesc, qt, cam, r) != want).sum())
    for i in range(3):  # the quaternion negated (w < 0) is the same rotation, evaluated to the same bits
        assert np.array_equal(got[3 + i], got[6 + i])
    assert (got >= 0).sum() > 1000
    # the slot order decides the conflicts: the creation order would give a different map
    assert teeth >= 20, teeth


@pytest.mark.gpu
def test_adapter_projection_match_degenerate_calls(gpu, tmp_path):
    xw, md, inframe, slot, kps, kdesc = _conflict_scene()
    cam, calls = _cam_tuple(DIST), [(SE3_POSE, 50), (IDENT, 100)]
    e = np.zeros((0, 3)), np.zeros((0, 32), np.uint8), np.zeros(0, np.uint8), np.zeros(0, np.int32)
    got = _adapter_proj(tmp_path / "no_points", *e, kps, kdesc, cam, calls)  # empty set
    assert got.shape == (2, len(kps)) and (got == -1).all()
    got = _adapter_proj(tmp_path / "no_keypoints", xw, md, inframe, slot, kps[:0], kdesc[:0], cam, calls)
    assert got.shape == (2, 0)
    got = _adapter_proj(tmp_path / "all_in_frame", xw, md, np.ones(len(xw), np.uint8), slot, kps, kdesc, cam, calls)
    assert (got == -1).all()


@pytest.mark.gpu
@pytest.mark.parametrize("pad", [13, 64])
def test_adapter_extract_on_padded_rows(gpu, oracle, tmp_path, pad):
    """cv::Mat with step = width + pad (an ROI or padded image): ORBextractor::extract and extractStereo == oracle"""
    L, R = _oracle_frame(1)[:2]
    _write_extract(tmp_path, L, R, W + pad)
    _run("extract", tmp_path)
    _check_extract(tmp_path, 1)


@pytest.mark.gpu
def test_adapter_extract_grows_its_capacity_on_a_wide_image(gpu, oracle, tmp_path):
    params, w, h = (20, 1.2, 8, 20, 7), W, 200
    ex = api.ORBextractor(*params)
    assert ex.cap_for(w, h) > ex.cap  # the adapter's `need > cap_` branch runs
    ex.close()
    L, R = _oracle_frame(5, w, h, params)[:2]
    _write_extract(tmp_path, L, R, w + 13, params)
    _run("extract", tmp_path)
    _check_extract(tmp_path, 5, w, h, params)


# ---- B5: strided host input below the adapter ----------------------------------------------------------------------
def _padded(images, stride, image_stride):
    """images (count x h x w) -> one buffer with rows `stride` bytes apart and images `image_stride` bytes apart; every
    byte outside the images is garbage"""
    count, h, w = images.shape
    buf = np.random.default_rng(count * stride).integers(0, 256, image_stride * count, dtype=np.uint8)
    for i in range(count):
        view = buf[i * image_stride:i * image_stride + stride * h].reshape(h, stride)
        view[:, :w] = images[i]
    return buf


def _raw_extract_batch(ex, images, stride, image_stride):
    count, h, w = images.shape
    buf = _padded(images, stride, image_stride)
    cap = ex.cap_for(w, h)
    kps, desc, n = np.zeros((count, cap), api.KP_DTYPE), np.zeros((count, cap, 32), np.uint8), np.zeros(count, np.int32)
    api._check(api.lib().sfe_extract_batch(ex.h, api._p(buf), image_stride, count, w, h, stride, api._p(kps), api._p(desc),
                                           cap, api._p(n)))
    return [(kps[i, :n[i]].copy(), desc[i, :n[i]].copy()) for i in range(count)]


def _raw_stereo_frames(ex, left, right, stride, image_stride):
    f, h, w = left.shape
    bl, br = _padded(left, stride, image_stride), _padded(right, stride, image_stride + 1)[:image_stride * f]
    cap = ex.cap_for(w, h)
    o = {k: np.zeros((f, cap), api.KP_DTYPE) for k in ("kps_l", "kps_r")}
    o.update({k: np.zeros((f, cap, 32), np.uint8) for k in ("desc_l", "desc_r")})
    o.update({k: np.zeros((f, cap), np.int32) for k in ("stereo_idx", "stereo_dist")})
    o.update({k: np.zeros(f, np.int32) for k in ("n_l", "n_r")})
    api._check(api.lib().sfe_stereo_frames(ex.h, api._p(bl), api._p(br), image_stride, f, w, h, stride, None,
                                           *[api._p(o[k]) for k in ("kps_l", "desc_l", "n_l", "kps_r", "desc_r", "n_r",
                                                                     "stereo_idx", "stereo_dist")], cap))
    return o


@pytest.mark.gpu
def test_strided_host_images_one_image_and_one_pair(gpu, oracle):
    """sfe_extract_batch / sfe_stereo_frames with stride > w and gaps between images: three calls each (eager, graph
    capture, graph replay), byte-equal to the contiguous calls and to the oracle"""
    L, R, kl, dl, kr, dr, si = _oracle_frame(2)
    ex = api.ORBextractor(max_images=2)
    stride = W + 13
    ck, cd, cn = ex.extract_batch(L[None])
    assert cn[0] == len(kl) and ck[0, :cn[0]].tobytes() == kl.tobytes() and np.array_equal(cd[0, :cn[0]], dl)
    for call in range(3):
        (k, d), = _raw_extract_batch(ex, L[None], stride, stride * H + 77)
        assert k.tobytes() == kl.tobytes() and np.array_equal(d, dl), call
    cont = ex.stereo_frames(L[None], R[None])
    for call in range(3):
        o = _raw_stereo_frames(ex, L[None], R[None], stride + 3, (stride + 3) * H + 4096)
        nl, nr = int(o["n_l"][0]), int(o["n_r"][0])
        assert (nl, nr) == (len(kl), len(kr)) == (int(cont["n_l"][0]), int(cont["n_r"][0])), call
        assert o["kps_l"][0, :nl].tobytes() == kl.tobytes() and np.array_equal(o["desc_l"][0, :nl], dl), call
        assert o["kps_r"][0, :nr].tobytes() == kr.tobytes() and np.array_equal(o["desc_r"][0, :nr], dr), call
        assert np.array_equal(o["stereo_idx"][0, :nl], si) and np.array_equal(o["stereo_idx"][0, :nl], cont["stereo_idx"][0, :nl])
        assert np.array_equal(o["stereo_dist"][0, :nl], cont["stereo_dist"][0, :nl]), call


@pytest.mark.gpu
def test_strided_host_images_pipelined_batch(gpu, oracle):
    """9 images: the host call is cut into pipelined sub-batches; every image lands in its own slot"""
    seq_l, seq_r = synth.stereo_sequence(6, 5, step=8)
    images = np.concatenate([seq_l, seq_r])[:9]
    ex = api.ORBextractor(max_images=9)
    ck, cd, cn = ex.extract_batch(images)
    got = _raw_extract_batch(ex, images, W + 64, (W + 64) * H + 333)
    ref = oracle.Extractor()
    for i in range(9):
        rk, rd = ref.extract(images[i])
        k, d = got[i]
        assert k.tobytes() == rk.tobytes() and np.array_equal(d, rd), i
        assert ck[i, :cn[i]].tobytes() == rk.tobytes() and np.array_equal(cd[i, :cn[i]], rd), i


# ---- B6: caller-allocated `out` ------------------------------------------------------------------------------------
def _stereo_out(frames, cap, track=False):
    keys = ["kps_l", "desc_l", "n_l", "kps_r", "desc_r", "n_r", "stereo_idx", "stereo_dist"] + (["track_idx", "track_dist"] if track else [])
    spec = {"kps": ((frames, cap), api.KP_DTYPE), "desc": ((frames, cap, 32), np.uint8), "n": ((frames,), np.int32),
            "stereo": ((frames, cap), np.int32), "track": ((frames, cap), np.int32)}
    return {k: np.zeros(*spec[k.split("_")[0]]) for k in keys}


def _check_stereo_out(out, want, frames, cap):
    for f in range(frames):
        nl, nr = int(want["n_l"][f]), int(want["n_r"][f])
        assert (int(out["n_l"][f]), int(out["n_r"][f])) == (nl, nr), f
        for k in want:
            if k.startswith("n_"):
                continue
            n = nr if k.endswith("_r") else nl
            assert out[k].shape[1] == cap
            assert out[k][f, :n].tobytes() == want[k][f, :n].tobytes(), (k, f)


@pytest.mark.gpu
def test_caller_out_arrays_use_their_own_capacity(gpu, oracle):
    seq_l, seq_r = synth.stereo_sequence(8, 2)
    ex = api.ORBextractor(max_images=4)
    want = ex.stereo_frames(seq_l, seq_r)
    cam = api.Camera.make(synth.KITTI_FX, synth.KITTI_FY, synth.KITTI_CX, synth.KITTI_CY, (0, 0, 0, 0), W, H)
    tp = api.TrackParams.make(cam, synth.KITTI_BASELINE, None, 30.0)
    want_t = ex.stereo_sequence(seq_l, seq_r, tp)
    wk, wd, wn = ex.extract_batch(seq_l)
    ref = oracle.Extractor()
    for f in range(2):
        rk, rd = ref.extract(seq_l[f])
        assert want["kps_l"][f, :want["n_l"][f]].tobytes() == rk.tobytes() and np.array_equal(want["desc_l"][f, :want["n_l"][f]], rd)
    # 1. out larger than ex.cap: frame 1 must land at out's stride
    big = ex.cap + 300
    out = ex.stereo_frames(seq_l, seq_r, out=_stereo_out(2, big))
    _check_stereo_out(out, want, 2, big)
    out = ex.stereo_sequence(seq_l, seq_r, tp, out=_stereo_out(2, big, track=True))
    _check_stereo_out(out, want_t, 2, big)
    bk, bd, bn = ex.extract_batch(seq_l, out=(np.zeros((2, big), api.KP_DTYPE), np.zeros((2, big, 32), np.uint8), np.zeros(2, np.int32)))
    assert np.array_equal(bn, wn)
    for f in range(2):
        assert bk[f, :bn[f]].tobytes() == wk[f, :wn[f]].tobytes() and np.array_equal(bd[f, :bn[f]], wd[f, :wn[f]])
    # 2. an earlier wide call grows ex.cap past the out arrays: results still land at out's stride
    cap0 = ex.cap_for(W, H)
    ex.extract(synth.stereo_pair(5, 4000, 160)[0])
    assert ex.cap > cap0
    out = ex.stereo_frames(seq_l, seq_r, out=_stereo_out(2, cap0))
    _check_stereo_out(out, want, 2, cap0)
    out = ex.stereo_sequence(seq_l, seq_r, tp, out=_stereo_out(2, cap0, track=True))
    _check_stereo_out(out, want_t, 2, cap0)
    bk, bd, bn = ex.extract_batch(seq_l, out=(np.zeros((2, cap0), api.KP_DTYPE), np.zeros((2, cap0, 32), np.uint8), np.zeros(2, np.int32)))
    assert np.array_equal(bn, wn) and all(bk[f, :bn[f]].tobytes() == wk[f, :wn[f]].tobytes() for f in range(2))
    # 3. out smaller than one image can return: refused before any device work
    launches = ex.launches()
    for call in (lambda: ex.stereo_frames(seq_l, seq_r, out=_stereo_out(2, cap0 - 1)),
                 lambda: ex.stereo_sequence(seq_l, seq_r, tp, out=_stereo_out(2, cap0 - 1, track=True)),
                 lambda: ex.extract_batch(seq_l, out=(np.zeros((2, cap0 - 1), api.KP_DTYPE), np.zeros((2, cap0 - 1, 32), np.uint8),
                                                      np.zeros(2, np.int32)))):
        with pytest.raises(api.SfeError) as e:
            call()
        assert e.value.status == api.SFE_ERR_CAPACITY
    assert ex.launches() == launches


# ---- C: several handles on one database ----------------------------------------------------------------------------
ROWS = 4_000_000  # >= 65536 rows and >= 256 queries: the first search unpacks the tensor-core tiles (1 GB)


def _keys_to_quad(m, keys, q):
    out = api.DeviceBuffer(q * 16)
    m.knn2_merge_dev(keys.ptr, 1, q, out.ptr)
    return out.download((q, 4), np.int32)


@pytest.mark.gpu
def test_shared_database_tiles_built_on_another_matchers_stream(gpu, oracle):
    """Matcher A builds the database's tiles on its own stream behind >= 1 ms of unrelated work; matcher B searches the
    same database right away.  B must wait for the tiles, not read them before they are written."""
    db = synth.knn_database(ROWS, seed=901)
    q, _ = synth.knn_queries(db, 512, seed=902, hard_fraction=0.2)
    want = oracle.knn2(q, db, nthreads=NTHREADS)
    a, b = api.Matcher(0), api.Matcher(0)
    dbh = a.create_db(db)
    # the unrelated work: ten resident ProjectionMatch calls of 6 M map points against the seed-0 frame
    g = np.load(os.path.join(GOLDEN, "golden_seed0.npz"))
    n = 6_000_000
    rng = np.random.default_rng(903)
    z = rng.uniform(2, 80, n)
    xw = np.stack([(rng.uniform(0, W, n) - synth.KITTI_CX) / synth.KITTI_FX * z,
                   (rng.uniform(0, H, n) - synth.KITTI_CY) / synth.KITTI_FY * z, z], 1)
    d_xw = api.DeviceBuffer(xw.nbytes).upload(xw)
    d_md = api.DeviceBuffer(n * 32).upload(rng.integers(0, 256, (n, 32), dtype=np.uint8))
    m = len(g["kl"])
    d_kp = api.DeviceBuffer(m * 28).upload(g["kl"])
    d_kd = api.DeviceBuffer(m * 32).upload(g["dl"])
    d_tq, d_td = api.DeviceBuffer(m * 4), api.DeviceBuffer(m * 4)
    d_q = api.DeviceBuffer(q.nbytes).upload(q)
    keys = api.DeviceBuffer(512 * 2 * 8)
    cam = api.Camera.make(synth.KITTI_FX, synth.KITTI_FY, synth.KITTI_CX, synth.KITTI_CY, DIST, W, H)
    # every buffer either matcher needs is allocated ahead (a device allocation may wait for the work queued so far):
    # in the window below the only allocation is the tile buffer of the search that builds the tiles
    warm = synth.knn_database(ROWS, seed=904)
    for mm in (a, b):
        w = mm.create_db(warm)
        mm.knn2(w, q)
        w.close()
    a.projection_match_dev(d_xw.ptr, d_md.ptr, None, n, IDENT, cam, d_kp.ptr, d_kd.ptr, m, 100.0, d_tq.ptr, d_td.ptr)
    a.set_async(True)
    e0, e1 = api.Event(0), api.Event(0)
    e0.record(a)
    for _ in range(10):
        a.projection_match_dev(d_xw.ptr, d_md.ptr, None, n, IDENT, cam, d_kp.ptr, d_kd.ptr, m, 100.0, d_tq.ptr, d_td.ptr)
    e1.record(a)
    a.knn2_dev(dbh, d_q.ptr, 512, keys.ptr)  # A's first many-query search: the tiles are built on A's stream
    got_b = b.knn2(dbh, q)  # at once, on B's stream
    a.wait()
    delay = e0.elapsed_ms(e1)
    a.set_async(False)
    got_a = _keys_to_quad(a, keys, 512)
    print(f"unrelated work ahead of the tile build on A's stream: {delay:.3f} ms")
    assert np.array_equal(got_b, want), int((got_b != want).any(axis=1).sum())
    assert np.array_equal(got_a, want), int((got_a != want).any(axis=1).sum())
    assert delay >= 1.0, delay  # the check above only means something if B had time to overtake the tile build


@pytest.mark.gpu
def test_shared_database_first_searches_from_two_threads(gpu, oracle):
    """Two host threads, one matcher each, start their first search of the same database at once (ctypes releases the
    GIL); both results are the oracle's.  A few fresh databases, so that the tile build is raced each time."""
    db = synth.knn_database(ROWS, seed=911)
    qs = [synth.knn_queries(db, 512, seed=912 + i, hard_fraction=0.2)[0] for i in range(2)]
    want = [oracle.knn2(q, db, nthreads=NTHREADS) for q in qs]
    ms = [api.Matcher(0), api.Matcher(0)]
    for rnd in range(3):
        dbh = ms[0].create_db(db)
        got = [None, None]
        start = threading.Barrier(2)

        def search(i):
            start.wait()
            got[i] = ms[i].knn2(dbh, qs[i])

        ts = [threading.Thread(target=search, args=(i,)) for i in range(2)]
        for t in ts:
            t.start()
        for t in ts:
            t.join()
        for i in range(2):
            assert got[i] is not None and np.array_equal(got[i], want[i]), (rnd, i)
        dbh.close()


@pytest.mark.gpu
def test_adapter_from_two_threads(gpu, oracle, tmp_path):
    """Two std::threads, each with its own thread_matcher() and ORBextractor, run the set-order ProjectionMatch case and a
    padded-row extract 20 times; every result equals the single-threaded pass, which equals the oracle."""
    xw, md, inframe, slot, kps, kdesc = _conflict_scene()
    cam = _cam_tuple(DIST)
    calls = [(SE3_POSE, 50), (IDENT, 10)]
    _write_proj(tmp_path / "proj", xw, md, inframe, slot, kps, kdesc, cam, calls)
    L, R = _oracle_frame(1)[:2]
    _write_extract(tmp_path / "ext", L, R, W + 13)
    got = _run("threads", tmp_path / "proj", tmp_path / "ext", 20, timeout=900)
    assert got["diff0"] == "0" and got["diff1"] == "0", got
    p = _read_proj(tmp_path / "proj", len(calls), len(kps))
    order = np.argsort(slot)
    for c, (qt, r) in enumerate(calls):
        assert np.array_equal(p[c], _oracle_in_order(order, xw, md, inframe, kps, kdesc, qt, cam, r)), c
    _check_extract(tmp_path / "ext", 1)
