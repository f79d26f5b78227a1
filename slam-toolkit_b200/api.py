"""Python binding of the sfe C ABI (include/sfe.h) with the reference's call surface.

The reference's host code is C++ (its adapter is include/sfe_adapter.hpp); this module is the
same surface for Python callers, tests and bench.py: ``ORBextractor.extract`` (reference
include/orb_extractor.h:51-59), ``StereoMatch`` / ``ProjectionMatch`` (include/matcher.h:33-38)
and the brute-force top-2 kNN.  Everything computes on the GPU through ``libsfe.so``; there is
no CPU fallback -- a missing library or device raises.
"""
from __future__ import annotations

import ctypes as C
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("SFE_LIB") or os.path.join(_HERE, "libsfe.so")  # SFE_LIB: an experimental build of the same library

KP_DTYPE = np.dtype([("x", "<f4"), ("y", "<f4"), ("size", "<f4"), ("angle", "<f4"),
                     ("response", "<f4"), ("octave", "<i4"), ("class_id", "<i4")])
assert KP_DTYPE.itemsize == 28  # == sizeof(cv::KeyPoint)

SFE_OK, SFE_ERR_BAD_ARG, SFE_ERR_CAPACITY, SFE_ERR_CUDA, SFE_ERR_NO_DEVICE, SFE_ERR_UNSUPPORTED = range(6)


class SfeError(RuntimeError):
    def __init__(self, status, detail):
        super().__init__(f"sfe status {status}: {detail}")
        self.status = status


class ExtractorParams(C.Structure):
    _fields_ = [("nfeatures", C.c_int32), ("scale_factor", C.c_float), ("nlevels", C.c_int32),
                ("ini_th_fast", C.c_int32), ("min_th_fast", C.c_int32)]


class StereoParams(C.Structure):
    _fields_ = [("y_threshold", C.c_double), ("max_dx", C.c_double), ("best12_threshold", C.c_double)]


class Camera(C.Structure):
    _fields_ = [("fx", C.c_double), ("fy", C.c_double), ("cx", C.c_double), ("cy", C.c_double),
                ("d", C.c_double * 4), ("width", C.c_int32), ("height", C.c_int32)]

    @staticmethod
    def make(fx, fy, cx, cy, d, width, height):
        c = Camera()
        c.fx, c.fy, c.cx, c.cy, c.width, c.height = fx, fy, cx, cy, width, height
        for i in range(4):
            c.d[i] = d[i]
        return c


class SE3(C.Structure):
    """sfe_se3: g2o::SE3Quat as the reference's ProjectionMatch receives it (unit quaternion x, y, z, w + translation)."""
    _fields_ = [("qx", C.c_double), ("qy", C.c_double), ("qz", C.c_double), ("qw", C.c_double),
                ("tx", C.c_double), ("ty", C.c_double), ("tz", C.c_double)]


def _pose(Tcw):
    """A pose argument is either 7 numbers (qx, qy, qz, qw, tx, ty, tz) = g2o::SE3Quat -> ("_se3", SE3) or a 3x4 / 4x4
    matrix [R|t] -> ("", 12 doubles)."""
    a = np.asarray(Tcw, np.float64)
    if a.ndim == 1 and a.size == 7:
        return "_se3", SE3(*[float(v) for v in a])
    return "", np.ascontiguousarray(a[:3, :4]).reshape(12)


def _pose_arg(p):
    return C.byref(p) if isinstance(p, SE3) else _p(p)


class TrackParams(C.Structure):
    """sfe_track_params: camera, stereo baseline, motion prior Tcw (3x4 matrix or SE3), ProjectionMatch radius and ratio."""
    _fields_ = [("cam", Camera), ("baseline", C.c_double), ("rt", C.c_double * 12), ("radius", C.c_double),
                ("best12_threshold", C.c_double), ("use_se3", C.c_int32), ("se3", SE3)]

    @staticmethod
    def make(cam, baseline, Tcw=None, radius=50.0, best12=0.5):
        t = TrackParams()
        t.cam, t.baseline, t.radius, t.best12_threshold = cam, baseline, radius, best12
        kind, pose = _pose(np.eye(4) if Tcw is None else Tcw)
        if kind:
            t.use_se3, t.se3 = 1, pose
            pose = np.eye(4)[:3, :4].reshape(12)
        for i, v in enumerate(pose):
            t.rt[i] = v
        return t


# every symbol include/sfe.h declares: name -> (restype, argtypes)
_vp, _i, _sz, _d, _i64 = C.c_void_p, C.c_int, C.c_size_t, C.c_double, C.c_int64
_pp = C.POINTER(C.c_void_p)
SIGNATURES = {
    "sfe_abi_version": (_i, []),
    "sfe_status_string": (C.c_char_p, [_i]),
    "sfe_last_error": (C.c_char_p, []),
    "sfe_device_count": (_i, [C.POINTER(_i)]),
    "sfe_host_alloc": (_i, [_pp, _sz]),
    "sfe_host_alloc_ex": (_i, [_pp, _sz, _i]),
    "sfe_host_free": (_i, [_vp]),
    "sfe_copy_probe": (_i, [_i, _sz, _sz, _i, _d, _i, C.POINTER(_d), C.POINTER(_d)]),
    "sfe_device_alloc": (_i, [_i, _pp, _sz]),
    "sfe_device_free": (_i, [_i, _vp]),
    "sfe_copy_to_device": (_i, [_i, _vp, _vp, _sz]),
    "sfe_copy_to_host": (_i, [_i, _vp, _vp, _sz]),
    "sfe_event_create": (_i, [_i, _pp]),
    "sfe_event_destroy": (_i, [_vp]),
    "sfe_event_record_extractor": (_i, [_vp, _vp]),
    "sfe_event_record_matcher": (_i, [_vp, _vp]),
    "sfe_event_elapsed_ms": (_i, [_vp, _vp, C.POINTER(C.c_float)]),
    "sfe_extractor_create": (_i, [C.POINTER(ExtractorParams), _i, _i, _pp]),
    "sfe_extractor_destroy": (_i, [_vp]),
    "sfe_extractor_tables": (_i, [_vp, _vp, _vp, _vp, _vp, _vp]),
    "sfe_extractor_level_size": (_i, [_vp, _i, _i, _i, C.POINTER(_i), C.POINTER(_i)]),
    "sfe_extractor_max_keypoints": (_i, [_vp, C.POINTER(_i)]),
    "sfe_extractor_max_keypoints_for": (_i, [_vp, _i, _i, C.POINTER(_i)]),
    "sfe_extract": (_i, [_vp, _vp, _i, _i, _i, _vp, _vp, _i, C.POINTER(_i)]),
    "sfe_extract_batch": (_i, [_vp, _vp, _sz, _i, _i, _i, _i, _vp, _vp, _i, _vp]),
    "sfe_extract_batch_dev": (_i, [_vp, _vp, _sz, _i, _i, _i, _i, _vp, _vp, _i, _vp]),
    "sfe_stereo_frames": (_i, [_vp, _vp, _vp, _sz, _i, _i, _i, _i, C.POINTER(StereoParams)] + [_vp] * 8 + [_i]),
    "sfe_stereo_frames_dev": (_i, [_vp, _vp, _vp, _sz, _i, _i, _i, _i, C.POINTER(StereoParams)] + [_vp] * 8 + [_i]),
    "sfe_results_size": (_i, [_i, _vp, _vp, _i, C.POINTER(_sz)]),
    "sfe_results_pack": (_i, [_vp, _sz, _i, _i, _i, _i, _i] + [_vp] * 10 + [C.POINTER(_sz)]),
    "sfe_results_info": (_i, [_vp, _sz] + [C.POINTER(_i)] * 5),
    "sfe_results_unpack": (_i, [_vp, _sz, _i] + [_vp] * 10),
    "sfe_stereo_sequence": (_i, [_vp, _vp, _vp, _sz, _i, _i, _i, _i, C.POINTER(StereoParams), C.POINTER(TrackParams)] + [_vp] * 10 + [_i]),
    "sfe_stereo_sequence_dev": (_i, [_vp, _vp, _vp, _sz, _i, _i, _i, _i, C.POINTER(StereoParams), C.POINTER(TrackParams)] + [_vp] * 10 + [_i]),
    "sfe_image_pitch": (_i, [_i]),
    "sfe_extractor_set_async": (_i, [_vp, _i]),
    "sfe_extractor_wait": (_i, [_vp]),
    "sfe_debug_level": (_i, [_vp, _i, _i, _vp]),
    "sfe_debug_blur": (_i, [_vp, _i, _i, _vp]),
    "sfe_debug_candidates": (_i, [_vp, _i, _i, _vp, _i, C.POINTER(_i)]),
    "sfe_debug_distributed": (_i, [_vp, _i, _i, _vp, _i, C.POINTER(_i)]),
    "sfe_extractor_launches": (_i, [_vp, C.POINTER(_i64)]),
    "sfe_extractor_set_profiling": (_i, [_vp, _i]),
    "sfe_extractor_stage_ms": (_i, [_vp, _vp, _i, C.POINTER(_i64)]),
    "sfe_hamming256": (_i, [_vp, _vp]),
    "sfe_matcher_create": (_i, [_i, _pp]),
    "sfe_matcher_destroy": (_i, [_vp]),
    "sfe_matcher_launches": (_i, [_vp, C.POINTER(_i64)]),
    "sfe_matcher_set_async": (_i, [_vp, _i]),
    "sfe_matcher_wait": (_i, [_vp]),
    "sfe_stereo_match": (_i, [_vp, _vp, _vp, _i, _vp, _vp, _i, C.POINTER(StereoParams), _vp, _vp]),
    "sfe_projection_match": (_i, [_vp, _vp, _vp, _vp, _i, _vp, C.POINTER(Camera), _vp, _vp, _i, _d, _d, _vp, _vp]),
    "sfe_projection_match_dev": (_i, [_vp, _vp, _vp, _vp, _i, _vp, C.POINTER(Camera), _vp, _vp, _i, _d, _d, _vp, _vp]),
    "sfe_projection_match_keys_dev": (_i, [_vp, _vp, _vp, _vp, _i, _i64, _vp, C.POINTER(Camera), _vp, _vp, _i, _d, _d, _vp]),
    "sfe_projection_merge_dev": (_i, [_vp, _vp, _i, _i, _vp, _vp]),
    "sfe_projection_match_se3": (_i, [_vp, _vp, _vp, _vp, _i, C.POINTER(SE3), C.POINTER(Camera), _vp, _vp, _i, _d, _d, _vp, _vp]),
    "sfe_projection_match_se3_dev": (_i, [_vp, _vp, _vp, _vp, _i, C.POINTER(SE3), C.POINTER(Camera), _vp, _vp, _i, _d, _d, _vp, _vp]),
    "sfe_projection_match_keys_se3_dev": (_i, [_vp, _vp, _vp, _vp, _i, _i64, C.POINTER(SE3), C.POINTER(Camera), _vp, _vp, _i, _d, _d, _vp]),
    "sfe_frame_reprojection_error_se3": (_i, [_vp, _vp, _vp, _vp, C.POINTER(SE3), _vp]),
    "sfe_frame_projection_match_se3": (_i, [_vp, _vp, _vp, _vp, _vp, _i, C.POINTER(SE3), _d, _d, _vp, _vp]),
    "sfe_frame_create": (_i, [_vp, _vp, _vp, _i, C.POINTER(Camera), _pp]),
    "sfe_frame_create_dev": (_i, [_vp, _vp, _vp, _i, C.POINTER(Camera), _pp]),
    "sfe_frame_destroy": (_i, [_vp]),
    "sfe_frame_size": (_i, [_vp, C.POINTER(_i)]),
    "sfe_frame_normalized": (_i, [_vp, _vp, _vp]),
    "sfe_frame_stereo_depth": (_i, [_vp, _vp, _vp, _i, _vp, _d, _vp, _vp]),
    "sfe_frame_reprojection_error": (_i, [_vp, _vp, _vp, _vp, _vp, _vp]),
    "sfe_frame_projection_match": (_i, [_vp, _vp, _vp, _vp, _vp, _i, _vp, _d, _d, _vp, _vp]),
    "sfe_frame_search_radius": (_i, [_vp, _vp, _vp, _i, _d, _vp, _i, _vp]),
    "sfe_frame_search_nearest": (_i, [_vp, _vp, _vp, _i, _vp, _vp]),
    "sfe_vocab_create": (_i, [_vp, _i, _vp, _vp, _vp, _vp, _i, _pp]),
    "sfe_vocab_destroy": (_i, [_vp]),
    "sfe_vocab_words": (_i, [_vp, C.POINTER(_i)]),
    "sfe_vocab_transform": (_i, [_vp, _vp, _vp, _i, _i, _vp, _vp, _vp]),
    "sfe_vocab_transform_dev": (_i, [_vp, _vp, _vp, _i, _i, _vp, _vp, _vp]),
    "sfe_bow_assemble": (_i, [_vp, _vp, _i, _i, _i, _vp, _vp, _i, C.POINTER(_i)]),
    "sfe_bow_assemble_dev": (_i, [_vp, _vp, _vp, _vp, _i, _i, _i, _i, _vp, _vp, _vp]),
    "sfe_bowdb_create": (_i, [_vp, _i, _pp]),
    "sfe_bowdb_destroy": (_i, [_vp]),
    "sfe_bowdb_size": (_i, [_vp, C.POINTER(_i)]),
    "sfe_bowdb_add": (_i, [_vp, _vp, _vp, _vp, _vp, _i, _vp]),
    "sfe_bowdb_query": (_i, [_vp, _vp, _vp, _vp, _vp, _i, _i, _i, _vp, _vp, _vp, _vp, _i]),
    "sfe_bowdb_add_dev": (_i, [_vp, _vp, _vp, _vp, _vp, _i, _vp]),
    "sfe_bowdb_query_dev": (_i, [_vp, _vp, _vp, _vp, _vp, _i, _i, _i, _vp, _vp, _vp, _vp, _i]),
    "sfe_db_create": (_i, [_vp, _vp, _i64, _i64, _pp]),
    "sfe_db_destroy": (_i, [_vp]),
    "sfe_knn2": (_i, [_vp, _vp, _vp, _i, _vp]),
    "sfe_knn2_dev": (_i, [_vp, _vp, _vp, _i, _vp]),
    "sfe_knn2_merge_dev": (_i, [_vp, _vp, _i, _i, _vp]),
    "sfe_comm_create": (_i, [_i, _i, _i, _pp]),
    "sfe_comm_export": (_i, [_vp, _vp]),
    "sfe_comm_connect": (_i, [_vp, _vp]),
    "sfe_comm_create_local": (_i, [_vp, _i, _pp]),
    "sfe_comm_destroy": (_i, [_vp]),
    "sfe_comm_status": (_i, [_vp, C.POINTER(_i)]),
    "sfe_knn2_sharded": (_i, [_vp, _vp, _vp, _vp, _i, _vp]),
    "sfe_projection_match_sharded": (_i, [_vp, _vp, _vp, _vp, _vp, _vp, _i, _i64, C.POINTER(SE3), _d, _d, _vp, _vp]),
}

_lib = None


def lib():
    """Load libsfe.so (built in-tree by __graft_entry__.build()).  No fallback."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise SfeError(SFE_ERR_CUDA, f"{LIB_PATH} is missing: run `python -c 'import __graft_entry__ as g; g.build()'` "
                                         "(there is no CPU fallback)")
        L = C.CDLL(LIB_PATH)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(L, name)
            fn.restype, fn.argtypes = res, args
        if L.sfe_abi_version() != 2:
            raise SfeError(SFE_ERR_UNSUPPORTED, "libsfe.so ABI version mismatch")
        _lib = L
    return _lib


def _check(status):
    if status != SFE_OK:
        raise SfeError(status, lib().sfe_last_error().decode() or lib().sfe_status_string(status).decode())


def _p(a):
    if a is None:
        return None
    if isinstance(a, int):
        return C.c_void_p(a)
    return a.ctypes.data_as(C.c_void_p)


def device_count() -> int:
    n = C.c_int(0)
    lib().sfe_device_count(C.byref(n))
    return n.value


def hamming256(a, b) -> int:
    """ORBextractor::DescriptorDistance (reference include/orb_extractor.h:87-103)."""
    a = np.ascontiguousarray(a, np.uint8)
    b = np.ascontiguousarray(b, np.uint8)
    return lib().sfe_hamming256(_p(a), _p(b))


def copy_probe(device, h2d_bytes, d2h_bytes, chunks=8, seconds=1.0, write_combined=False):
    """copy-only ceiling of the host path -> (h2d GB/s, d2h GB/s), both directions at once (sfe_copy_probe)"""
    a, b = C.c_double(), C.c_double()
    _check(lib().sfe_copy_probe(device, h2d_bytes, d2h_bytes, chunks, seconds, 1 if write_combined else 0, C.byref(a), C.byref(b)))
    return a.value, b.value


class PinnedArray:
    """numpy view of pinned host memory (cudaHostAlloc) for the host entry points."""

    def __init__(self, shape, dtype, write_combined=False):
        self.dtype = np.dtype(dtype)
        self.shape = tuple(int(s) for s in np.atleast_1d(shape))
        self.nbytes = max(int(np.prod(self.shape)) * self.dtype.itemsize, 1)
        ptr = C.c_void_p()
        _check(lib().sfe_host_alloc_ex(C.byref(ptr), self.nbytes, 1 if write_combined else 0))
        self.ptr = ptr.value
        buf = (C.c_uint8 * self.nbytes).from_address(self.ptr)
        self.array = np.frombuffer(buf, dtype=self.dtype, count=int(np.prod(self.shape))).reshape(self.shape)

    def free(self):
        if self.ptr:
            self.array = None
            lib().sfe_host_free(C.c_void_p(self.ptr))
            self.ptr = None

    def __del__(self):
        try:
            self.free()
        except Exception:
            pass


class DeviceBuffer:
    """Raw device allocation on `device` (resident inputs / outputs of the _dev entry points)."""

    def __init__(self, nbytes, device=0):
        self.device, self.nbytes = device, max(int(nbytes), 1)
        ptr = C.c_void_p()
        _check(lib().sfe_device_alloc(device, C.byref(ptr), self.nbytes))
        self.ptr = ptr.value

    def upload(self, arr):
        arr = np.ascontiguousarray(arr)
        assert arr.nbytes <= self.nbytes
        _check(lib().sfe_copy_to_device(self.device, C.c_void_p(self.ptr), _p(arr), arr.nbytes))
        return self

    def download(self, shape, dtype):
        out = np.empty(shape, dtype)
        assert out.nbytes <= self.nbytes
        _check(lib().sfe_copy_to_host(self.device, _p(out), C.c_void_p(self.ptr), out.nbytes))
        return out

    def free(self):
        if self.ptr:
            lib().sfe_device_free(self.device, C.c_void_p(self.ptr))
            self.ptr = None

    def __del__(self):
        try:
            self.free()
        except Exception:
            pass


class Event:
    def __init__(self, device=0):
        h = C.c_void_p()
        _check(lib().sfe_event_create(device, C.byref(h)))
        self.h = h

    def record(self, handle):
        if isinstance(handle, ORBextractor):
            _check(lib().sfe_event_record_extractor(self.h, handle.h))
        else:
            _check(lib().sfe_event_record_matcher(self.h, handle.h))

    def elapsed_ms(self, stop: "Event") -> float:
        ms = C.c_float()
        _check(lib().sfe_event_elapsed_ms(self.h, stop.h, C.byref(ms)))
        return ms.value

    def __del__(self):
        try:
            lib().sfe_event_destroy(self.h)
        except Exception:
            pass


def image_pitch(w: int) -> int:
    """Row pitch (bytes) at which resident images can be fetched with TMA."""
    return lib().sfe_image_pitch(w)


class ORBextractor:
    """ORB_SLAM2::ORBextractor (reference include/orb_extractor.h:45-133)."""

    def __init__(self, nfeatures=2000, scaleFactor=1.2, nlevels=8, iniThFAST=20, minThFAST=7, device=0, max_images=2):
        self.params = ExtractorParams(nfeatures, scaleFactor, nlevels, iniThFAST, minThFAST)
        self.device, self.max_images, self.nlevels = device, max_images, nlevels
        h = C.c_void_p()
        _check(lib().sfe_extractor_create(C.byref(self.params), device, max_images, C.byref(h)))
        self.h = h
        cap = C.c_int()
        _check(lib().sfe_extractor_max_keypoints(self.h, C.byref(cap)))
        self.cap = cap.value
        self._wh = None

    def cap_for(self, w, h) -> int:
        """upper bound of the keypoints one w x h image returns (sfe_extractor_max_keypoints_for)"""
        cap = C.c_int()
        _check(lib().sfe_extractor_max_keypoints_for(self.h, w, h, C.byref(cap)))
        return cap.value

    def _grow_cap(self, w, h):  # a very wide image can return more than the default bound: 4 * nIni nodes per level
        self.cap = max(self.cap, self.cap_for(w, h))

    def _out_cap(self, cap, w, h) -> int:
        """the row stride of caller-allocated output arrays: their own capacity, which must hold one w x h image's keypoints
        (self.cap may have grown since they were allocated)"""
        need = self.cap_for(w, h)
        if cap < need:
            raise SfeError(SFE_ERR_CAPACITY, f"out holds {cap} keypoints per image, a {w} x {h} image can return {need}")
        return cap

    def close(self):
        if getattr(self, "h", None):
            lib().sfe_extractor_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # getters: include/orb_extractor.h:63-83
    def GetLevels(self):
        return self.nlevels

    def GetScaleFactor(self):
        return self.params.scale_factor

    def _tables(self):
        n = self.nlevels
        t = [np.zeros(n, np.float32) for _ in range(4)] + [np.zeros(n, np.int32)]
        _check(lib().sfe_extractor_tables(self.h, *[_p(a) for a in t]))
        return t

    def GetScaleFactors(self):
        return self._tables()[0]

    def GetInverseScaleFactors(self):
        return self._tables()[1]

    def GetScaleSigmaSquares(self):
        return self._tables()[2]

    def GetInverseScaleSigmaSquares(self):
        return self._tables()[3]

    def features_per_level(self):
        return self._tables()[4]

    def level_size(self, w, h, level):
        lw, lh = C.c_int(), C.c_int()
        _check(lib().sfe_extractor_level_size(self.h, w, h, level, C.byref(lw), C.byref(lh)))
        return lw.value, lh.value

    def extract(self, image):
        """extract(image, mask ignored) -> (keypoints[KP_DTYPE], descriptors n x 32 u8)."""
        image = np.ascontiguousarray(image, np.uint8)
        if image.size == 0:
            return np.zeros(0, KP_DTYPE), np.zeros((0, 32), np.uint8)
        assert image.ndim == 2, "CV_8UC1 expected (reference asserts the same, src/orb_extractor.cpp:1050)"
        h, w = image.shape
        self._grow_cap(w, h)
        kps = np.zeros(self.cap, KP_DTYPE)
        desc = np.zeros((self.cap, 32), np.uint8)
        n = C.c_int()
        _check(lib().sfe_extract(self.h, _p(image), w, h, w, _p(kps), _p(desc), self.cap, C.byref(n)))
        self._wh = (w, h)
        return kps[:n.value].copy(), desc[:n.value].copy()

    def extract_batch(self, images, out=None):
        """images: count x h x w u8 (numpy or PinnedArray.array).  Returns (kps[count, cap], desc[count, cap, 32], n[count])."""
        images = np.ascontiguousarray(images, np.uint8)
        count, h, w = images.shape
        if out is None:
            self._grow_cap(w, h)
            out = (np.zeros((count, self.cap), KP_DTYPE), np.zeros((count, self.cap, 32), np.uint8), np.zeros(count, np.int32))
            cap = self.cap
        else:
            cap = self._out_cap(out[0].shape[1], w, h)
        kps, desc, n = out
        _check(lib().sfe_extract_batch(self.h, _p(images), w * h, count, w, h, w, _p(kps), _p(desc), cap, _p(n)))
        self._wh = (w, h)
        return kps, desc, n

    def extract_batch_dev(self, images_ptr, count, w, h, kps_ptr, desc_ptr, n_ptr):
        _check(lib().sfe_extract_batch_dev(self.h, _p(images_ptr), w * h, count, w, h, w, _p(kps_ptr), _p(desc_ptr), self.cap,
                                           _p(n_ptr)))
        self._wh = (w, h)

    def stereo_frames(self, left, right, out=None, stereo_params=None):
        """Keyframe path (src/pipeline.cpp:243-249): extract(left), extract(right), StereoMatch for
        `frames` pairs in one call.  left/right: frames x h x w u8."""
        left = np.ascontiguousarray(left, np.uint8)
        right = np.ascontiguousarray(right, np.uint8)
        f, h, w = left.shape
        assert right.shape == left.shape
        if out is None:
            self._grow_cap(w, h)
            out = self.alloc_stereo_out(f)
        cap = self._out_cap(out["kps_l"].shape[1], w, h)
        sp = C.byref(stereo_params) if stereo_params is not None else None
        _check(lib().sfe_stereo_frames(self.h, _p(left), _p(right), w * h, f, w, h, w, sp, _p(out["kps_l"]), _p(out["desc_l"]),
                                       _p(out["n_l"]), _p(out["kps_r"]), _p(out["desc_r"]), _p(out["n_r"]),
                                       _p(out["stereo_idx"]), _p(out["stereo_dist"]), cap))
        self._wh = (w, h)
        return out

    def stereo_sequence(self, left, right, track_params, out=None, stereo_params=None):
        """Tracking front end of a stereo sequence: stereo_frames + per frame f >= 1 the ProjectionMatch of frame f-1's
        stereo-triangulated keypoints into frame f (sfe_stereo_sequence).  out["track_idx"][f, j] = keypoint of frame
        f-1 matched to keypoint j of frame f, or -1."""
        left = np.ascontiguousarray(left, np.uint8)
        right = np.ascontiguousarray(right, np.uint8)
        f, h, w = left.shape
        assert right.shape == left.shape
        if out is None:
            self._grow_cap(w, h)
            out = self.alloc_stereo_out(f, track=True)
        cap = self._out_cap(out["kps_l"].shape[1], w, h)
        sp = C.byref(stereo_params) if stereo_params is not None else None
        _check(lib().sfe_stereo_sequence(self.h, _p(left), _p(right), w * h, f, w, h, w, sp, C.byref(track_params),
                                         _p(out["kps_l"]), _p(out["desc_l"]), _p(out["n_l"]), _p(out["kps_r"]),
                                         _p(out["desc_r"]), _p(out["n_r"]), _p(out["stereo_idx"]), _p(out["stereo_dist"]),
                                         _p(out["track_idx"]), _p(out["track_dist"]), cap))
        self._wh = (w, h)
        return out

    def stereo_sequence_dev(self, left_ptr, right_ptr, frames, w, h, ptrs, track_params, stereo_params=None, pitch=None):
        """stereo_frames_dev + tracking; ptrs additionally holds "track_idx" / "track_dist" (frames x cap int32)."""
        sp = C.byref(stereo_params) if stereo_params is not None else None
        pitch = pitch or w
        _check(lib().sfe_stereo_sequence_dev(self.h, _p(left_ptr), _p(right_ptr), pitch * h, frames, w, h, pitch, sp,
                                             C.byref(track_params), _p(ptrs["kps_l"]), _p(ptrs["desc_l"]), _p(ptrs["n_l"]),
                                             _p(ptrs["kps_r"]), _p(ptrs["desc_r"]), _p(ptrs["n_r"]), _p(ptrs["stereo_idx"]),
                                             _p(ptrs["stereo_dist"]), _p(ptrs["track_idx"]), _p(ptrs["track_dist"]), self.cap))
        self._wh = (w, h)

    def alloc_stereo_out(self, frames, pinned=False, track=False):
        spec = {"kps_l": ((frames, self.cap), KP_DTYPE), "desc_l": ((frames, self.cap, 32), np.uint8),
                "n_l": ((frames,), np.int32), "kps_r": ((frames, self.cap), KP_DTYPE),
                "desc_r": ((frames, self.cap, 32), np.uint8), "n_r": ((frames,), np.int32),
                "stereo_idx": ((frames, self.cap), np.int32), "stereo_dist": ((frames, self.cap), np.int32)}
        if track:
            spec["track_idx"] = ((frames, self.cap), np.int32)
            spec["track_dist"] = ((frames, self.cap), np.int32)
        if not pinned:
            return {k: np.zeros(s, d) for k, (s, d) in spec.items()}
        self._pinned_out = {k: PinnedArray(s, d) for k, (s, d) in spec.items()}
        return {k: v.array for k, v in self._pinned_out.items()}

    def stereo_frames_dev(self, left_ptr, right_ptr, frames, w, h, ptrs, stereo_params=None, pitch=None):
        """Resident images: row pitch `pitch` bytes (default w), images pitch*h bytes apart.  A pitch that is a
        multiple of 16 (image_pitch(w)) on a 16-byte aligned buffer lets the kernels fetch level-0 tiles with TMA."""
        sp = C.byref(stereo_params) if stereo_params is not None else None
        pitch = pitch or w
        _check(lib().sfe_stereo_frames_dev(self.h, _p(left_ptr), _p(right_ptr), pitch * h, frames, w, h, pitch, sp,
                                           _p(ptrs["kps_l"]), _p(ptrs["desc_l"]), _p(ptrs["n_l"]), _p(ptrs["kps_r"]),
                                           _p(ptrs["desc_r"]), _p(ptrs["n_r"]), _p(ptrs["stereo_idx"]),
                                           _p(ptrs["stereo_dist"]), self.cap))
        self._wh = (w, h)

    def set_async(self, enable=True):
        """_dev calls return once enqueued; errors surface at wait()."""
        _check(lib().sfe_extractor_set_async(self.h, int(enable)))

    def wait(self):
        _check(lib().sfe_extractor_wait(self.h))

    def launches(self) -> int:
        n = C.c_int64()
        _check(lib().sfe_extractor_launches(self.h, C.byref(n)))
        return n.value

    STAGES = ("pyramid", "fast_cells", "quadtree", "blur", "orient_describe", "stereo_match", "track")

    def set_profiling(self, enable=True):
        _check(lib().sfe_extractor_set_profiling(self.h, int(enable)))

    def stage_ms(self):
        """-> ({stage: accumulated ms}, calls) from CUDA events on the handle's stream."""
        ms = np.zeros(len(self.STAGES), np.float64)
        calls = C.c_int64()
        _check(lib().sfe_extractor_stage_ms(self.h, _p(ms), len(ms), C.byref(calls)))
        return dict(zip(self.STAGES, ms.tolist())), calls.value

    # stage taps (parity tests)
    def debug_level(self, image, level, blur=False):
        lw, lh = self.level_size(*self._wh, level)
        out = np.zeros((lh, lw), np.uint8)
        fn = lib().sfe_debug_blur if blur else lib().sfe_debug_level
        _check(fn(self.h, image, level, _p(out)))
        return out

    def debug_points(self, image, level, distributed=False, cap=1 << 15):
        out = np.zeros((cap, 3), np.float32)
        n = C.c_int()
        fn = lib().sfe_debug_distributed if distributed else lib().sfe_debug_candidates
        _check(fn(self.h, image, level, _p(out), cap, C.byref(n)))
        return out[:n.value].copy()


class Matcher:
    """StereoMatch / ProjectionMatch (reference include/matcher.h) + brute-force top-2."""

    def __init__(self, device=0):
        h = C.c_void_p()
        _check(lib().sfe_matcher_create(device, C.byref(h)))
        self.h, self.device = h, device

    def close(self):
        if getattr(self, "h", None):
            lib().sfe_matcher_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def launches(self) -> int:
        n = C.c_int64()
        _check(lib().sfe_matcher_launches(self.h, C.byref(n)))
        return n.value

    def set_async(self, enable=True):
        _check(lib().sfe_matcher_set_async(self.h, int(enable)))

    def wait(self):
        _check(lib().sfe_matcher_wait(self.h))

    def StereoMatch(self, kps_l, desc_l, kps_r, desc_r, params=None):
        """-> (stereo_indices, distances): right index or -1 per left keypoint (src/matcher.cpp:54-132)."""
        kps_l, kps_r = np.ascontiguousarray(kps_l, KP_DTYPE), np.ascontiguousarray(kps_r, KP_DTYPE)
        desc_l, desc_r = np.ascontiguousarray(desc_l, np.uint8), np.ascontiguousarray(desc_r, np.uint8)
        idx = np.full(len(kps_l), -1, np.int32)
        dist = np.full(len(kps_l), -1, np.int32)
        sp = C.byref(params) if params is not None else None
        _check(lib().sfe_stereo_match(self.h, _p(kps_l), _p(desc_l), len(kps_l), _p(kps_r), _p(desc_r), len(kps_r), sp,
                                      _p(idx), _p(dist)))
        return idx, dist

    def ProjectionMatch(self, xw, mp_desc, skip, Tcw, camera, kps, kp_desc, search_radius, best12=0.5):
        """-> (kp_to_query, kp_dist): for every frame keypoint the matched map-point index or -1
        (the reference's std::map<int, Mappoint*>, src/matcher.cpp:134-209).  Tcw: 7 numbers (qx, qy, qz, qw, tx, ty, tz) =
        the reference's g2o::SE3Quat, or a 3x4 [R|t] matrix."""
        xw = np.ascontiguousarray(xw, np.float64)
        mp_desc = np.ascontiguousarray(mp_desc, np.uint8)
        skip = None if skip is None else np.ascontiguousarray(skip, np.uint8)
        kind, pose = _pose(Tcw)
        kps = np.ascontiguousarray(kps, KP_DTYPE)
        kp_desc = np.ascontiguousarray(kp_desc, np.uint8)
        to_q = np.full(len(kps), -1, np.int32)
        dist = np.full(len(kps), -1, np.int32)
        _check(getattr(lib(), "sfe_projection_match" + kind)(self.h, _p(xw), _p(mp_desc), _p(skip), len(xw), _pose_arg(pose),
                                                             C.byref(camera), _p(kps), _p(kp_desc), len(kps), search_radius,
                                                             best12, _p(to_q), _p(dist)))
        return to_q, dist

    def projection_match_dev(self, xw_ptr, mp_desc_ptr, skip_ptr, n, Tcw, camera, kps_ptr, kp_desc_ptr, m, radius,
                             to_q_ptr, dist_ptr, best12=0.5):
        kind, pose = _pose(Tcw)
        _check(getattr(lib(), f"sfe_projection_match{kind}_dev")(self.h, _p(xw_ptr), _p(mp_desc_ptr), _p(skip_ptr), n,
                                                                 _pose_arg(pose), C.byref(camera), _p(kps_ptr), _p(kp_desc_ptr),
                                                                 m, radius, best12, _p(to_q_ptr), _p(dist_ptr)))

    def projection_match_keys_dev(self, xw_ptr, mp_desc_ptr, skip_ptr, n, idx_base, Tcw, camera, kps_ptr, kp_desc_ptr, m,
                                  radius, keys_ptr, best12=0.5):
        """One shard of a sharded ProjectionMatch: map points [idx_base, idx_base + n) -> m per-keypoint keys."""
        kind, pose = _pose(Tcw)
        _check(getattr(lib(), f"sfe_projection_match_keys{kind}_dev")(self.h, _p(xw_ptr), _p(mp_desc_ptr), _p(skip_ptr), n,
                                                                      idx_base, _pose_arg(pose), C.byref(camera), _p(kps_ptr),
                                                                      _p(kp_desc_ptr), m, radius, best12, _p(keys_ptr)))

    def projection_merge_dev(self, keys_ptr, shards, m, to_q_ptr, dist_ptr):
        _check(lib().sfe_projection_merge_dev(self.h, _p(keys_ptr), shards, m, _p(to_q_ptr), _p(dist_ptr)))

    def create_db(self, desc, idx_base=0):
        return DescriptorDB(self, desc, idx_base)

    def knn2(self, db, queries):
        """-> int32 q x 4 {idx0, dist0, idx1, dist1}, lexicographic (dist, idx) top-2."""
        queries = np.ascontiguousarray(queries, np.uint8)
        out = np.zeros((len(queries), 4), np.int32)
        _check(lib().sfe_knn2(self.h, db.h, _p(queries), len(queries), _p(out)))
        return out

    def knn2_dev(self, db, queries_ptr, q, keys_ptr):
        _check(lib().sfe_knn2_dev(self.h, db.h, _p(queries_ptr), q, _p(keys_ptr)))

    def knn2_sharded(self, comm: "Comm", db, queries_ptr, q, out_ptr):
        """collective over comm.world ranks; returns once enqueued (wait() completes it)"""
        _check(lib().sfe_knn2_sharded(self.h, comm.h, db.h, _p(queries_ptr), q, _p(out_ptr)))

    def projection_match_sharded(self, comm: "Comm", frame: "Frame", xw_ptr, mp_desc_ptr, skip_ptr, n, idx_base, Tcw, radius,
                                 to_q_ptr, dist_ptr, best12=0.5):
        """collective; Tcw = 7 numbers (qx, qy, qz, qw, tx, ty, tz); returns once enqueued (wait() completes it)"""
        kind, pose = _pose(Tcw)
        assert kind == "_se3", "the sharded call takes the pose as an SE3Quat"
        _check(lib().sfe_projection_match_sharded(self.h, comm.h, frame.h, _p(xw_ptr), _p(mp_desc_ptr), _p(skip_ptr), n, idx_base,
                                                  C.byref(pose), radius, best12, _p(to_q_ptr), _p(dist_ptr)))

    def knn2_merge_dev(self, keys_ptr, shards, q, out_ptr):
        _check(lib().sfe_knn2_merge_dev(self.h, _p(keys_ptr), shards, q, _p(out_ptr)))


class Comm:
    """sfe_comm: one rank's end of the NVLink peer-memory exchange behind the sharded kNN / ProjectionMatch calls."""

    def __init__(self, device=0, rank=0, world=1, _handle=None):
        self.device, self.rank, self.world = device, rank, world
        if _handle is None:
            h = C.c_void_p()
            _check(lib().sfe_comm_create(device, rank, world, C.byref(h)))
            _handle = h
        self.h = _handle

    def export(self) -> bytes:
        buf = (C.c_uint8 * 64)()
        _check(lib().sfe_comm_export(self.h, buf))
        return bytes(buf)

    def connect(self, handles):
        """handles: the export() of every rank, in rank order"""
        blob = b"".join(handles)
        assert len(blob) == 64 * self.world
        buf = (C.c_uint8 * len(blob)).from_buffer_copy(blob)
        _check(lib().sfe_comm_connect(self.h, buf))
        return self

    @staticmethod
    def create_local(devices):
        """one process driving several GPUs: a connected communicator per device"""
        n = len(devices)
        devs = (C.c_int * n)(*devices)
        hs = (C.c_void_p * n)()
        _check(lib().sfe_comm_create_local(devs, n, hs))
        return [Comm(devices[i], i, n, _handle=C.c_void_p(hs[i])) for i in range(n)]

    def status(self):
        """raises when a peer never delivered its part of a collective"""
        r = C.c_int()
        _check(lib().sfe_comm_status(self.h, C.byref(r)))

    def close(self):
        if getattr(self, "h", None):
            lib().sfe_comm_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class Frame:
    """The device-resident part of the reference's Frame (src/frame.cpp:36-69): keypoints + descriptors, normalised
    undistorted keypoints (GetNormalizedPoint) and the spatial index behind SearchRadius / SearchNeareast /
    ProjectionMatch.  Build it from host arrays or from device pointers (`dev=True`)."""

    def __init__(self, matcher: "Matcher", kps, desc, camera: Camera, n=None, dev=False):
        self.m = matcher
        h = C.c_void_p()
        if dev:
            _check(lib().sfe_frame_create_dev(matcher.h, _p(kps), _p(desc), n, C.byref(camera), C.byref(h)))
        else:
            kps = np.ascontiguousarray(kps, KP_DTYPE)
            desc = np.ascontiguousarray(desc, np.uint8)
            n = len(kps)
            _check(lib().sfe_frame_create(matcher.h, _p(kps), _p(desc), n, C.byref(camera), C.byref(h)))
        self.h, self.n = h, n

    def close(self):
        if getattr(self, "h", None):
            lib().sfe_frame_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def normalized(self):
        """-> n x 2 float64, Frame::GetNormalizedPoint for every keypoint."""
        out = np.zeros((self.n, 2), np.float64)
        _check(lib().sfe_frame_normalized(self.m.h, self.h, _p(out)))
        return out

    def reprojection_error(self, xw, has_mp, Tcw):
        """ReprojectionFilter::GetOutlier's test quantity per keypoint: |Project(Tcw Xw_i) - keypoint_i|, +inf behind the
        camera, -1 where has_mp[i] == 0."""
        xw = np.ascontiguousarray(xw, np.float64)
        has_mp = np.ascontiguousarray(has_mp, np.uint8)
        kind, pose = _pose(Tcw)
        err = np.zeros(self.n, np.float64)
        _check(getattr(lib(), "sfe_frame_reprojection_error" + kind)(self.m.h, self.h, _p(xw), _p(has_mp), _pose_arg(pose), _p(err)))
        return err

    def stereo_depth(self, kps_r, stereo_idx, baseline):
        """StereoFrame::GetDepth for every keypoint -> (Xc n x 3 float64, valid n u8)."""
        kps_r = np.ascontiguousarray(kps_r, KP_DTYPE)
        stereo_idx = np.ascontiguousarray(stereo_idx, np.int32)
        xc = np.zeros((self.n, 3), np.float64)
        valid = np.zeros(self.n, np.uint8)
        _check(lib().sfe_frame_stereo_depth(self.m.h, self.h, _p(kps_r), len(kps_r), _p(stereo_idx), baseline, _p(xc), _p(valid)))
        return xc, valid

    def ProjectionMatch(self, xw, mp_desc, skip, Tcw, search_radius, best12=0.5):
        xw = np.ascontiguousarray(xw, np.float64)
        mp_desc = np.ascontiguousarray(mp_desc, np.uint8)
        skip = None if skip is None else np.ascontiguousarray(skip, np.uint8)
        kind, pose = _pose(Tcw)
        to_q = np.full(self.n, -1, np.int32)
        dist = np.full(self.n, -1, np.int32)
        _check(getattr(lib(), "sfe_frame_projection_match" + kind)(self.m.h, self.h, _p(xw), _p(mp_desc), _p(skip), len(xw),
                                                                   _pose_arg(pose), search_radius, best12, _p(to_q), _p(dist)))
        return to_q, dist

    def SearchRadius(self, uv, radius, cap=512):
        """-> list of index arrays (ascending), one per query point (Frame::SearchRadius, batch form)."""
        uv = np.ascontiguousarray(np.atleast_2d(uv), np.float64)
        idx = np.zeros((len(uv), cap), np.int32)
        counts = np.zeros(len(uv), np.int32)
        _check(lib().sfe_frame_search_radius(self.m.h, self.h, _p(uv), len(uv), radius, _p(idx), cap, _p(counts)))
        if (counts > cap).any():
            raise SfeError(SFE_ERR_CAPACITY, "SearchRadius: more neighbours than cap")
        return [idx[i, :counts[i]].copy() for i in range(len(uv))]

    def SearchNeareast(self, uv):
        """-> (kpt_index, squared distance) arrays (Frame::SearchNeareast, batch form; the name is the reference's)."""
        uv = np.ascontiguousarray(np.atleast_2d(uv), np.float64)
        idx = np.zeros(len(uv), np.int32)
        d2 = np.zeros(len(uv), np.float64)
        _check(lib().sfe_frame_search_nearest(self.m.h, self.h, _p(uv), len(uv), _p(idx), _p(d2)))
        return idx, d2


class Vocabulary:
    """DBoW2 ORB vocabulary on the device (thirdparty/DBoW2/DBoW2/TemplatedVocabulary.h): arrays as loadFromTextFile
    reads them -- parent, is_leaf flag, 32-byte descriptor and weight per node, node 0 = root."""
    TF_IDF, TF, IDF, BINARY = range(4)
    NORM_NONE, NORM_L1, NORM_L2 = range(3)

    def __init__(self, matcher: "Matcher", parent, is_leaf, desc, weight, L, weighting=0, norm=1):
        self.m, self.L, self.weighting, self.norm = matcher, L, weighting, norm
        parent = np.ascontiguousarray(parent, np.int32)
        is_leaf = np.ascontiguousarray(is_leaf, np.uint8)
        desc = np.ascontiguousarray(desc, np.uint8)
        weight = np.ascontiguousarray(weight, np.float64)
        h = C.c_void_p()
        _check(lib().sfe_vocab_create(matcher.h, len(parent), _p(parent), _p(is_leaf), _p(desc), _p(weight), L, C.byref(h)))
        self.h = h

    def close(self):
        if getattr(self, "h", None):
            lib().sfe_vocab_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def words(self) -> int:
        n = C.c_int()
        _check(lib().sfe_vocab_words(self.h, C.byref(n)))
        return n.value

    def transform_features(self, desc, levelsup=4):
        """-> (word_id, weight, node_id) per feature: TemplatedVocabulary::transform(feature, id, w, &nid, levelsup)."""
        desc = np.ascontiguousarray(desc, np.uint8)
        n = len(desc)
        wid, w, nid = np.zeros(n, np.int32), np.zeros(n, np.float64), np.zeros(n, np.int32)
        _check(lib().sfe_vocab_transform(self.m.h, self.h, _p(desc), n, levelsup, _p(wid), _p(w), _p(nid)))
        return wid, w, nid

    def transform(self, desc, levelsup=4):
        """voc->transform(vdesc, bowvec, featvec, levelsup) (src/frame.cpp:419-427) -> (BowVector as (ids, values),
        FeatureVector as {node id: [feature indices]})."""
        wid, w, nid = self.transform_features(desc, levelsup)
        ids, vals = bow_assemble(wid, w, self.weighting, self.norm)
        fv = {}
        for i in np.nonzero(w > 0)[0]:
            fv.setdefault(int(nid[i]), []).append(int(i))
        return (ids, vals), dict(sorted(fv.items()))

    def transform_dev(self, desc_ptr, n_ptr, count, stride, levelsup, word_id_ptr, weight_ptr, node_id_ptr, off_ptr, ids_ptr,
                      val_ptr):
        """transform's BowVectors for `count` resident descriptor sets, all on the device: set i = rows [i*stride,
        i*stride + n[i]) of desc_ptr (int32 counts at n_ptr), e.g. stereo_frames_dev's desc_l / n_l with stride = cap.
        sfe_vocab_transform_dev over count * stride rows into word_id_ptr / weight_ptr / node_id_ptr, then
        sfe_bow_assemble_dev with this vocabulary's weighting and norm into the CSR off_ptr (int64, count + 1) /
        ids_ptr (int32) / val_ptr (float64), the last two sized count * stride."""
        if stride > BOW_ASSEMBLE_MAX_STRIDE:  # the assembly would reject it: do not write the caller's buffers first
            raise SfeError(SFE_ERR_UNSUPPORTED, f"stride {stride} above SFE_BOW_ASSEMBLE_MAX_STRIDE ({BOW_ASSEMBLE_MAX_STRIDE})")
        _check(lib().sfe_vocab_transform_dev(self.m.h, self.h, _p(desc_ptr), count * stride, levelsup, _p(word_id_ptr),
                                             _p(weight_ptr), _p(node_id_ptr)))
        bow_assemble_dev(self.m, word_id_ptr, weight_ptr, n_ptr, count, stride, off_ptr, ids_ptr, val_ptr, self.weighting, self.norm)


def bow_assemble(word_id, weight, weighting=0, norm=1):
    word_id = np.ascontiguousarray(word_id, np.int32)
    weight = np.ascontiguousarray(weight, np.float64)
    n = C.c_int()
    ids, vals = np.zeros(len(word_id), np.int32), np.zeros(len(word_id), np.float64)
    _check(lib().sfe_bow_assemble(_p(word_id), _p(weight), len(word_id), weighting, norm, _p(ids), _p(vals), len(ids), C.byref(n)))
    return ids[:n.value].copy(), vals[:n.value].copy()


BOW_ASSEMBLE_MAX_STRIDE = 16384  # SFE_BOW_ASSEMBLE_MAX_STRIDE


def bow_assemble_dev(matcher: "Matcher", word_id_ptr, weight_ptr, n_ptr, count, stride, off_ptr, ids_ptr, val_ptr, weighting=0,
                     norm=1):
    """bow_assemble for `count` feature sets on the device (sfe_bow_assemble_dev): set i = rows [i*stride, i*stride + n[i])
    of the int32 word ids / float64 weights -> CSR off_ptr (int64, count + 1) / ids_ptr / val_ptr (count * stride each)."""
    _check(lib().sfe_bow_assemble_dev(matcher.h, _p(word_id_ptr), _p(weight_ptr), _p(n_ptr), count, stride, weighting, norm,
                                      _p(off_ptr), _p(ids_ptr), _p(val_ptr)))


BOWDB_MAX_RESULTS = 1024  # SFE_BOWDB_MAX_RESULTS


def bow_csr(vectors):
    """BowVectors given as (ids, values) pairs -> (offsets int64[n + 1], ids int32, values float64), the CSR form the
    BoW database entry points take."""
    vs = [(np.ascontiguousarray(i, np.int32).reshape(-1), np.ascontiguousarray(v, np.float64).reshape(-1)) for i, v in vectors]
    for i, v in vs:
        if len(i) != len(v):
            raise SfeError(SFE_ERR_BAD_ARG, "a BowVector needs one value per word id")
    off = np.zeros(len(vs) + 1, np.int64)
    np.cumsum([len(i) for i, _ in vs], out=off[1:])
    ids = np.concatenate([i for i, _ in vs] + [np.zeros(0, np.int32)])
    vals = np.concatenate([v for _, v in vs] + [np.zeros(0, np.float64)])
    return off, ids, vals


class BowDatabase:
    """DBoW2's keyframe database (TemplatedDatabase) with L1 scoring, resident on the device: add() BowVectors -- the
    (ids, values) that Vocabulary.transform returns -- and query them as Database::query does, bit for bit.  Entry ids are
    0, 1, 2, ... in add order.  Several matchers of the device may share one database from several threads."""

    def __init__(self, matcher: "Matcher", n_words):
        self.m = matcher
        h = C.c_void_p()
        _check(lib().sfe_bowdb_create(matcher.h, int(n_words), C.byref(h)))
        self.h, self.n_words = h, int(n_words)

    def close(self):
        if getattr(self, "h", None):
            lib().sfe_bowdb_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def __len__(self):
        n = C.c_int()
        _check(lib().sfe_bowdb_size(self.h, C.byref(n)))
        return n.value

    def add(self, vectors, matcher=None) -> int:
        """Appends BowVectors (a list of (ids, values)) -> the entry id of the first."""
        off, ids, vals = bow_csr(vectors)
        first = C.c_int32()
        _check(lib().sfe_bowdb_add((matcher or self.m).h, self.h, _p(off), _p(ids), _p(vals), len(off) - 1, C.byref(first)))
        return first.value

    def query(self, vectors, max_results, max_id=-1, dense=False, dense_entries=None, matcher=None):
        """Database::query(v, ret, max_results, max_id) for every vector -> a list of (entry ids, scores) in DBoW2's order
        (equal scores by ascending entry id).  dense=True also returns the q x dense_entries matrix of
        L1Scoring::score(query, entry) for the first dense_entries entries (default: all of them)."""
        off, ids, vals = bow_csr(vectors)
        q = len(off) - 1
        k = int(max_results)
        ent = np.full((q, max(k, 1)), -1, np.int32)
        sc = np.zeros((q, max(k, 1)), np.float64)
        n = np.zeros(q, np.int32)
        d, de = None, 0
        if dense:
            de = len(self) if dense_entries is None else int(dense_entries)
            d = np.zeros((q, max(de, 0)), np.float64)
        _check(lib().sfe_bowdb_query((matcher or self.m).h, self.h, _p(off), _p(ids), _p(vals), q, int(max_id), k, _p(ent), _p(sc),
                                     _p(n), _p(d), de))
        res = [(ent[i, :n[i]].copy(), sc[i, :n[i]].copy()) for i in range(q)]
        return (res, d) if dense else res

    def add_dev(self, off_ptr, ids_ptr, val_ptr, count, matcher=None) -> int:
        """Appends `count` BowVectors held on the device in CSR form (e.g. bow_assemble_dev's output) -> the entry id of
        the first."""
        first = C.c_int32()
        _check(lib().sfe_bowdb_add_dev((matcher or self.m).h, self.h, _p(off_ptr), _p(ids_ptr), _p(val_ptr), count, C.byref(first)))
        return first.value

    def query_dev(self, off_ptr, ids_ptr, val_ptr, q, max_results, entry_ptr, score_ptr, n_ptr, max_id=-1, dense_ptr=None,
                  dense_entries=0, matcher=None):
        """query for `q` BowVectors held on the device in CSR form; results stay on the device: entry_ptr (int32) and
        score_ptr (float64) rows of max_results, n_ptr (int32, q) and, when dense_ptr is given, the q x dense_entries
        float64 score matrix."""
        _check(lib().sfe_bowdb_query_dev((matcher or self.m).h, self.h, _p(off_ptr), _p(ids_ptr), _p(val_ptr), q, int(max_id),
                                         int(max_results), _p(entry_ptr), _p(score_ptr), _p(n_ptr), _p(dense_ptr),
                                         int(dense_entries)))


class DescriptorDB:
    def __init__(self, matcher: Matcher, desc, idx_base=0):
        desc = np.ascontiguousarray(desc, np.uint8)
        assert desc.ndim == 2 and desc.shape[1] == 32
        h = C.c_void_p()
        _check(lib().sfe_db_create(matcher.h, _p(desc), len(desc), idx_base, C.byref(h)))
        self.h, self.rows, self.idx_base = h, len(desc), idx_base

    def close(self):
        if getattr(self, "h", None):
            lib().sfe_db_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


# ---- front-end results as one byte stream (include/sfe.h "SFER"; SURVEY §8f row 4) -------------------------------
RES_STEREO, RES_TRACK = 1, 2
_RES_KEYS = ("kps_l", "desc_l", "n_l", "kps_r", "desc_r", "n_r", "stereo_idx", "stereo_dist", "track_idx", "track_dist")


def pack_results(out, w=0, h=0) -> bytes:
    """The dict alloc_stereo_out / extract_batch style calls fill (cap-strided arrays) -> one byte string that holds
    only the valid rows.  Sections present: stereo if out has "kps_r", tracking if it has "track_idx"."""
    frames, cap = out["kps_l"].shape
    flags = (RES_STEREO if "kps_r" in out else 0) | (RES_TRACK if "track_idx" in out else 0)
    arr = {k: np.ascontiguousarray(out[k]) if k in out else None for k in _RES_KEYS}
    n = C.c_size_t()
    _check(lib().sfe_results_size(frames, _p(arr["n_l"]), _p(arr["n_r"]), flags, C.byref(n)))
    buf = np.empty(n.value, np.uint8)
    wr = C.c_size_t()
    _check(lib().sfe_results_pack(_p(buf), buf.nbytes, frames, cap, w, h, flags, *[_p(arr[k]) for k in _RES_KEYS], C.byref(wr)))
    assert wr.value == n.value
    return buf.tobytes()


def unpack_results(data: bytes):
    """-> (out dict of cap-strided arrays with cap = the largest frame, (w, h))."""
    buf = np.frombuffer(data, np.uint8)
    frames, flags, w, h, mx = C.c_int(), C.c_int(), C.c_int(), C.c_int(), C.c_int()
    _check(lib().sfe_results_info(_p(buf), buf.nbytes, C.byref(frames), C.byref(flags), C.byref(w), C.byref(h), C.byref(mx)))
    f, cap = frames.value, max(mx.value, 1)
    out = {"kps_l": np.zeros((f, cap), KP_DTYPE), "desc_l": np.zeros((f, cap, 32), np.uint8), "n_l": np.zeros(f, np.int32)}
    if flags.value & RES_STEREO:
        out.update({"kps_r": np.zeros((f, cap), KP_DTYPE), "desc_r": np.zeros((f, cap, 32), np.uint8), "n_r": np.zeros(f, np.int32),
                    "stereo_idx": np.full((f, cap), -1, np.int32), "stereo_dist": np.full((f, cap), -1, np.int32)})
    if flags.value & RES_TRACK:
        out.update({"track_idx": np.full((f, cap), -1, np.int32), "track_dist": np.full((f, cap), -1, np.int32)})
    _check(lib().sfe_results_unpack(_p(buf), buf.nbytes, cap, *[_p(out.get(k)) for k in _RES_KEYS]))
    return out, (w.value, h.value)
