/* sfe.h -- C ABI of the B200-native ORB front end ("slam front end", sfe).
 *
 * Drop-in boundary for the one data-parallel hot path of geonuklee/slam-toolkit:
 *   ORBextractor::extract            include/orb_extractor.h:51-59, src/orb_extractor.cpp:1043-1105
 *   ORBextractor::DescriptorDistance include/orb_extractor.h:87-103
 *   StereoMatch                      include/matcher.h:33,  src/matcher.cpp:54-132
 *   ProjectionMatch                  include/matcher.h:35-38, src/matcher.cpp:134-209
 *   (+ the brute-force top-2 kNN that BASELINE config 4 defines over the same inner loop)
 * The reference has no FFI layer (it is one C++ library); a maintainer binds these
 * symbols through include/sfe_adapter.hpp, which keeps the reference's own class and
 * function signatures (see INTEGRATION.md).
 *
 * Conventions
 *   - plain pointers and sizes only; no C++/torch types; every call returns an int status.
 *   - the library never allocates caller-visible memory: the caller passes capacity, gets counts.
 *   - "host" entry points take host pointers and copy to/from the device inside the call;
 *     "_dev" entry points take device pointers of the handle's device (resident data).
 *   - a handle owns one CUDA device + stream + its buffers and is NOT re-entrant (the reference's
 *     extract() is not either: it mutates mvImagePyramid, src/orb_extractor.cpp:1115);
 *     use one handle per thread / per GPU.
 *   - there is no CPU fallback: without a usable CUDA device every compute call fails with
 *     SFE_ERR_NO_DEVICE / SFE_ERR_CUDA.
 */
#ifndef SFE_H_
#define SFE_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define SFE_ABI_VERSION 2

enum {
    SFE_OK = 0,
    SFE_ERR_BAD_ARG = 1,     /* null pointer, non-positive size, unsupported geometry */
    SFE_ERR_CAPACITY = 2,    /* caller capacity too small; or one pyramid level of one image holds more than 60000 FAST
                              * corners (the quadtree's candidate index).  The reference's candidate list is unbounded
                              * (src/orb_extractor.cpp:778-779): below that limit a call whose internal candidate buffers
                              * overflow is re-run with buffers sized from its own exact count, never refused. */
    SFE_ERR_CUDA = 3,        /* a CUDA runtime call failed; see sfe_last_error() */
    SFE_ERR_NO_DEVICE = 4,   /* no CUDA device (there is no CPU fallback) */
    SFE_ERR_UNSUPPORTED = 5  /* parameters outside what the kernels were built for */
};

/* byte-identical to cv::KeyPoint (28 B: pt.x, pt.y, size, angle, response, octave, class_id),
 * so the C++ adapter fills std::vector<cv::KeyPoint> with one memcpy. */
typedef struct sfe_keypoint {
    float x, y;      /* level-0 pixel coordinates (pt *= scale, src/orb_extractor.cpp:1095-1101) */
    float size;      /* (int)(31 * scale[octave]), :837-847 */
    float angle;     /* degrees in [0,360), IC_Angle + fastAtan2, :77-104 */
    float response;  /* FAST score, cv::FAST cornerScore */
    int32_t octave;
    int32_t class_id; /* always -1 */
} sfe_keypoint;

/* the five ORBextractor constructor arguments, include/orb_extractor.h:51 */
typedef struct sfe_extractor_params {
    int32_t nfeatures;    /* 2000 in the reference pipeline (src/pipeline.cpp:46-50) */
    float scale_factor;   /* 1.2f */
    int32_t nlevels;      /* 8 */
    int32_t ini_th_fast;  /* 20 */
    int32_t min_th_fast;  /* 7 */
} sfe_extractor_params;

/* StereoMatch constants, src/matcher.cpp:60,68-70 */
typedef struct sfe_stereo_params {
    double y_threshold;      /* 3.0 */
    double max_dx;           /* 100.0 */
    double best12_threshold; /* 0.5 */
} sfe_stereo_params;

/* Camera, src/camera.cpp:26-79: pinhole + 4-coefficient radial-tangential distortion */
typedef struct sfe_camera {
    double fx, fy, cx, cy;
    double d[4];
    int32_t width, height;
} sfe_camera;

/* predicted_Tcw as the reference holds it, a g2o::SE3Quat (src/matcher.cpp:135,151): unit quaternion + translation.
 * The *_se3 entry points evaluate Xc = Tcw * Xw exactly as g2o / Eigen do (t + q * Xw with Eigen's quaternion-vector
 * product, no contraction), so a point on the z = 0, image-border or radius boundary falls on the same side as in the
 * reference.  The rt[12] entry points take a row-major 3x4 [R|t] for callers that hold a matrix (rows evaluated left to
 * right); the two agree except in the last unit of precision of Xc. */
typedef struct sfe_se3 {
    double qx, qy, qz, qw; /* Eigen::Quaterniond::x(), y(), z(), w() of SE3Quat::rotation() */
    double tx, ty, tz;     /* SE3Quat::translation() */
} sfe_se3;

typedef struct sfe_extractor sfe_extractor;
typedef struct sfe_matcher sfe_matcher;
typedef struct sfe_db sfe_db;
typedef struct sfe_event sfe_event;
typedef struct sfe_frame sfe_frame;
typedef struct sfe_vocab sfe_vocab;
typedef struct sfe_bowdb sfe_bowdb;
typedef struct sfe_comm sfe_comm;

/* ---- general -------------------------------------------------------------------------- */
int sfe_abi_version(void);
const char *sfe_status_string(int status);
const char *sfe_last_error(void); /* thread-local detail of the last failure */
int sfe_device_count(int *count);
int sfe_host_alloc(void **ptr, size_t bytes); /* pinned host memory for the host entry points */
/* flags: SFE_HOST_WRITE_COMBINED = write-combined pages for buffers the host only WRITES (input images): the device reads
 * them over PCIe without snooping the CPU caches; host reads of such memory are very slow */
#define SFE_HOST_WRITE_COMBINED 1
int sfe_host_alloc_ex(void **ptr, size_t bytes, int flags);
int sfe_host_free(void *ptr);
/* Measurement aid: the ceiling of the host entry points.  Moves h2d_bytes pinned host -> device and d2h_bytes device ->
 * pinned host per step (each split into `chunks` copies, the two directions on two streams at once) for about `seconds`,
 * no kernels, and reports the sustained GB/s of each direction.  flags as sfe_host_alloc_ex, applied to the input pages. */
int sfe_copy_probe(int device, size_t h2d_bytes, size_t d2h_bytes, int chunks, double seconds, int flags,
                   double *h2d_gbs, double *d2h_gbs);
int sfe_device_alloc(int device, void **ptr, size_t bytes);
int sfe_device_free(int device, void *ptr);
int sfe_copy_to_device(int device, void *dst_dev, const void *src_host, size_t bytes);
int sfe_copy_to_host(int device, void *dst_host, const void *src_dev, size_t bytes);
/* CUDA events on a handle's own stream (bench timing must be taken on the launching stream) */
int sfe_event_create(int device, sfe_event **ev);
int sfe_event_destroy(sfe_event *ev);
int sfe_event_record_extractor(sfe_event *ev, sfe_extractor *ex);
int sfe_event_record_matcher(sfe_event *ev, sfe_matcher *m);
int sfe_event_elapsed_ms(sfe_event *start, sfe_event *stop, float *ms); /* synchronises on stop */

/* ---- ORBextractor (include/orb_extractor.h:45-133) -------------------------------------- */
/* max_images: how many images one batched call may carry (device buffers are sized for it). */
int sfe_extractor_create(const sfe_extractor_params *params, int device, int max_images,
                         sfe_extractor **out);
int sfe_extractor_destroy(sfe_extractor *ex);
/* GetScaleFactors / GetInverseScaleFactors / GetScaleSigmaSquares / GetInverseScaleSigmaSquares
 * (:63-83) + the per-level quotas; each out array has nlevels entries, any may be NULL. */
int sfe_extractor_tables(const sfe_extractor *ex, float *scale, float *inv_scale, float *sigma2,
                         float *inv_sigma2, int32_t *features_per_level);
int sfe_extractor_level_size(const sfe_extractor *ex, int w, int h, int level, int *lw, int *lh);
/* Upper bound of the keypoints one w x h image can return: per level max(quota + 3, 4 * nIni) -- DistributeOctTree stops at
 * the first size >= N and one split adds at most 3 nodes, but its first pass over the nIni root nodes is unconditional
 * (src/orb_extractor.cpp:543,606-669).  sfe_extractor_max_keypoints uses the geometry of the last call (before any call:
 * aspect ratios up to 4.5 : 1). */
int sfe_extractor_max_keypoints_for(const sfe_extractor *ex, int w, int h, int *cap);
int sfe_extractor_max_keypoints(const sfe_extractor *ex, int *cap);

/* extract(): one 8-bit gray image in, keypoints + 256-bit descriptors out (row i <-> keypoint i).
 * An empty image (w==0 || h==0) is a silent success with *n_out = 0 (:1046-1047). */
int sfe_extract(sfe_extractor *ex, const uint8_t *image, int w, int h, int stride,
                sfe_keypoint *kps, uint8_t *desc /* cap*32 */, int cap, int *n_out);
/* count images of identical geometry, image i at images + i*image_stride bytes; outputs for image i
 * at kps + i*cap, desc + i*cap*32, n_out[i]. */
int sfe_extract_batch(sfe_extractor *ex, const uint8_t *images, size_t image_stride, int count,
                      int w, int h, int stride, sfe_keypoint *kps, uint8_t *desc, int cap,
                      int32_t *n_out);
int sfe_extract_batch_dev(sfe_extractor *ex, const uint8_t *images_dev, size_t image_stride,
                          int count, int w, int h, int stride, sfe_keypoint *kps_dev,
                          uint8_t *desc_dev, int cap, int32_t *n_out_dev);

/* Keyframe path of the reference pipeline in one call (src/pipeline.cpp:243-249,
 * src/frame.cpp:47,388): extract(left), extract(right), StereoMatch, for `frames` stereo pairs.
 * stereo_idx[f*cap + i] = right keypoint index or -1 (SetStereoCorrespond, src/matcher.cpp:130);
 * stereo_dist (optional, may be NULL) = accepted Hamming distance or -1. */
int sfe_stereo_frames(sfe_extractor *ex, const uint8_t *left, const uint8_t *right,
                      size_t image_stride, int frames, int w, int h, int stride,
                      const sfe_stereo_params *sp, sfe_keypoint *kps_l, uint8_t *desc_l,
                      int32_t *n_l, sfe_keypoint *kps_r, uint8_t *desc_r, int32_t *n_r,
                      int32_t *stereo_idx, int32_t *stereo_dist, int cap);
int sfe_stereo_frames_dev(sfe_extractor *ex, const uint8_t *left_dev, const uint8_t *right_dev,
                          size_t image_stride, int frames, int w, int h, int stride,
                          const sfe_stereo_params *sp, sfe_keypoint *kps_l_dev, uint8_t *desc_l_dev,
                          int32_t *n_l_dev, sfe_keypoint *kps_r_dev, uint8_t *desc_r_dev,
                          int32_t *n_r_dev, int32_t *stereo_idx_dev, int32_t *stereo_dist_dev,
                          int cap);

/* Tracking front end of a stereo SEQUENCE in one call: sfe_stereo_frames over `frames` consecutive stereo pairs, then
 * for every frame f >= 1 what the tracker does before pose optimisation (src/posetracker.cpp -> src/matcher.cpp:134-209):
 * the previous frame's keypoints with a stereo correspondence become map points through StereoFrame::GetDepth
 * (src/frame.cpp:391-409: Xc = (n_x, n_y, 1) * fx * baseline / dx, with the normalised keypoint of
 * Camera::NormalizedUndistort), in keypoint order, and ProjectionMatch(those points, Tcw = tp->rt, frame f, tp->radius)
 * matches them against frame f's keypoints.  tp->rt is the motion prior between consecutive frames (identity = the
 * reference's first guess).  track_idx[f*cap + j] = keypoint index in frame f-1 whose map point matched keypoint j of
 * frame f, or -1 (frame 0's row is all -1); track_dist (optional) = the accepted Hamming distance or -1. */
typedef struct sfe_track_params {
    sfe_camera cam;
    double baseline;          /* metres; depth = fx * baseline / disparity */
    double rt[12];            /* Tcw (3x4 row-major) applied to the previous frame's camera-frame points */
    double radius;            /* ProjectionMatch search radius in pixels (the tracker uses 50) */
    double best12_threshold;  /* 0.5, src/matcher.cpp:196 */
    int32_t use_se3;          /* != 0: the motion prior is `se3` (evaluated like g2o::SE3Quat), rt is ignored */
    sfe_se3 se3;
} sfe_track_params;
int sfe_stereo_sequence(sfe_extractor *ex, const uint8_t *left, const uint8_t *right,
                        size_t image_stride, int frames, int w, int h, int stride,
                        const sfe_stereo_params *sp, const sfe_track_params *tp, sfe_keypoint *kps_l,
                        uint8_t *desc_l, int32_t *n_l, sfe_keypoint *kps_r, uint8_t *desc_r,
                        int32_t *n_r, int32_t *stereo_idx, int32_t *stereo_dist, int32_t *track_idx,
                        int32_t *track_dist, int cap);
int sfe_stereo_sequence_dev(sfe_extractor *ex, const uint8_t *left_dev, const uint8_t *right_dev,
                            size_t image_stride, int frames, int w, int h, int stride,
                            const sfe_stereo_params *sp, const sfe_track_params *tp,
                            sfe_keypoint *kps_l_dev, uint8_t *desc_l_dev, int32_t *n_l_dev,
                            sfe_keypoint *kps_r_dev, uint8_t *desc_r_dev, int32_t *n_r_dev,
                            int32_t *stereo_idx_dev, int32_t *stereo_dist_dev, int32_t *track_idx_dev,
                            int32_t *track_dist_dev, int cap);

/* The tracker's per-pair behaviour for sfe_stereo_sequence_plan[_dev] (src/pipeline.cpp:158-166 predicts a pose for every
 * frame; src/posetracker.cpp:185-190 matches again at a wider radius when too few points were found -- SURVEY §3.2).
 *   rt / se3: NULL, or `frames` motion priors in host memory.  Entry f (f >= 1) is the Tcw of pair (f-1, f): it takes frame
 *             f-1's camera coordinates into frame f's, exactly what tp->rt / tp->se3 is for every pair in
 *             sfe_stereo_sequence.  Entry 0 is ignored.  rt = frames x 12 doubles (row-major 3x4, evaluated like tp->rt);
 *             se3 = sfe_se3[frames] (evaluated like g2o::SE3Quat, as tp->se3).  At most one of the two may be non-NULL; both
 *             NULL = tp's prior for every pair.  The priors are read before the call returns, also by an asynchronous _dev
 *             call.
 *   retry_radius, retry_below: a pair whose first ProjectionMatch (radius tp->radius) leaves fewer than retry_below
 *             keypoints of frame f matched (the size of the std::map ProjectionMatch returns) is matched again with the same
 *             map points, the same prior and radius retry_radius, and the second result replaces the first.
 *             retry_below = 0: no retry.  The reference tracker: 100.0 and 8 (the rule as SURVEY §3.2 records it; the
 *             reference sources are not part of this tree).
 * SFE_ERR_BAD_ARG, before anything is enqueued: plan == NULL, both rt and se3 set, a prior of entries 1..frames-1 that is
 * not finite, retry_radius negative or NaN, retry_below < 0 -- besides everything sfe_stereo_sequence[_dev] rejects. */
typedef struct sfe_track_plan {
    const double *rt;
    const sfe_se3 *se3;
    double retry_radius;
    int32_t retry_below;
} sfe_track_plan;
/* sfe_stereo_sequence[_dev] with the pair priors and the retry of `plan`; every other argument and output as there.  A plan
 * with both priors NULL (or every prior equal to tp's) and retry_below = 0 gives exactly what sfe_stereo_sequence gives. */
int sfe_stereo_sequence_plan(sfe_extractor *ex, const uint8_t *left, const uint8_t *right,
                             size_t image_stride, int frames, int w, int h, int stride,
                             const sfe_stereo_params *sp, const sfe_track_params *tp,
                             const sfe_track_plan *plan, sfe_keypoint *kps_l, uint8_t *desc_l, int32_t *n_l,
                             sfe_keypoint *kps_r, uint8_t *desc_r, int32_t *n_r, int32_t *stereo_idx,
                             int32_t *stereo_dist, int32_t *track_idx, int32_t *track_dist, int cap);
int sfe_stereo_sequence_plan_dev(sfe_extractor *ex, const uint8_t *left_dev, const uint8_t *right_dev,
                                 size_t image_stride, int frames, int w, int h, int stride,
                                 const sfe_stereo_params *sp, const sfe_track_params *tp,
                                 const sfe_track_plan *plan, sfe_keypoint *kps_l_dev, uint8_t *desc_l_dev,
                                 int32_t *n_l_dev, sfe_keypoint *kps_r_dev, uint8_t *desc_r_dev,
                                 int32_t *n_r_dev, int32_t *stereo_idx_dev, int32_t *stereo_dist_dev,
                                 int32_t *track_idx_dev, int32_t *track_dist_dev, int cap);

/* Row pitch (bytes) the _dev entry points like best for resident images of width w: the smallest multiple
 * of 16 >= w.  With such a pitch, a 16-byte aligned base and an image stride that is a multiple of 16 the
 * kernels fetch level-0 tiles with TMA; any other layout is read with ordinary loads (same results). */
int sfe_image_pitch(int w);

/* Asynchronous mode for the _dev entry points: with enable != 0 they return as soon as the kernels are
 * enqueued on the handle's stream, so a caller can queue batch after batch without a host round trip
 * (consecutive calls reuse the handle's buffers in stream order).  Capacity errors of any queued batch are
 * kept on the device and reported by the next sfe_extractor_wait(), which also synchronises the stream.
 * The matchers of an asynchronous stereo call run on a side stream beside the next call's extraction kernels; the
 * handle orders every later writer of the same output arrays behind them, and sfe_extractor_wait() /
 * sfe_event_record_extractor() cover them -- other streams must not read the outputs before one of the two.
 * The host entry points are always synchronous. */
int sfe_extractor_set_async(sfe_extractor *ex, int enable);
int sfe_extractor_wait(sfe_extractor *ex);

/* stage taps for parity tests (valid for the images of the last call on this handle) */
int sfe_debug_level(sfe_extractor *ex, int image, int level, uint8_t *out /* lw*lh */);
int sfe_debug_blur(sfe_extractor *ex, int image, int level, uint8_t *out /* lw*lh */);
/* FAST candidates in the reference's vToDistributeKeys order (x, y window-relative, response) */
int sfe_debug_candidates(sfe_extractor *ex, int image, int level, float *xyr, int cap, int *n);
/* quadtree survivors in DistributeOctTree's list order */
int sfe_debug_distributed(sfe_extractor *ex, int image, int level, float *xyr, int cap, int *n);
/* number of kernel launches the handle issued since creation (bench's gpu_launches) */
int sfe_extractor_launches(const sfe_extractor *ex, int64_t *launches);
/* per-stage device time from CUDA events recorded on the handle's own stream between the stage
 * kernels (no extra synchronisation).  Stages: 0 pyramid, 1 FAST cells, 2 quadtree, 3 blur,
 * 4 orientation+rBRIEF, 5 stereo match.  ms[i] accumulates over `calls` batched calls. */
int sfe_extractor_set_profiling(sfe_extractor *ex, int enable);
int sfe_extractor_stage_ms(const sfe_extractor *ex, double *ms, int n, int64_t *calls);

/* ---- matcher (include/matcher.h, DescriptorDistance) ------------------------------------- */
int sfe_hamming256(const void *a, const void *b); /* DescriptorDistance of two 32-byte rows */

int sfe_matcher_create(int device, sfe_matcher **out);
int sfe_matcher_destroy(sfe_matcher *m);
int sfe_matcher_launches(const sfe_matcher *m, int64_t *launches);
/* as sfe_extractor_set_async: the matcher's _dev entry points return once enqueued; sfe_matcher_wait synchronises */
int sfe_matcher_set_async(sfe_matcher *m, int enable);
int sfe_matcher_wait(sfe_matcher *m);

/* StereoMatch on one frame's keypoints (host buffers) */
int sfe_stereo_match(sfe_matcher *m, const sfe_keypoint *kps_l, const uint8_t *desc_l, int n_l,
                     const sfe_keypoint *kps_r, const uint8_t *desc_r, int n_r,
                     const sfe_stereo_params *sp, int32_t *out_idx /* n_l */,
                     int32_t *out_dist /* n_l, optional */);

/* ProjectionMatch: n map points (world xyz double[3], 32-B descriptor, optional skip byte = the
 * host-side prefilter curr_frame->GetIndex(mp) >= 0, src/matcher.cpp:144) against a frame's m
 * keypoints.  rt = row-major 3x4 [R|t] of predicted_Tcw.  Map points are visited in array order
 * (the reference iterates a std::set<Mappoint*>, i.e. pointer order).
 * kp_to_query[j] = index of the map point matched to keypoint j or -1 (the reference's
 * std::map<int, Mappoint*>), kp_dist[j] = its Hamming distance or -1. */
int sfe_projection_match(sfe_matcher *m, const double *xw, const uint8_t *mp_desc,
                         const uint8_t *skip, int n, const double rt[12], const sfe_camera *cam,
                         const sfe_keypoint *kps, const uint8_t *kp_desc, int m_kps, double radius,
                         double best12_threshold, int32_t *kp_to_query, int32_t *kp_dist);
int sfe_projection_match_dev(sfe_matcher *m, const double *xw_dev, const uint8_t *mp_desc_dev,
                             const uint8_t *skip_dev, int n, const double rt[12],
                             const sfe_camera *cam, const sfe_keypoint *kps_dev,
                             const uint8_t *kp_desc_dev, int m_kps, double radius,
                             double best12_threshold, int32_t *kp_to_query_dev,
                             int32_t *kp_dist_dev);

/* the same with the pose as a g2o::SE3Quat: what the adapter's ProjectionMatch calls */
int sfe_projection_match_se3(sfe_matcher *m, const double *xw, const uint8_t *mp_desc,
                             const uint8_t *skip, int n, const sfe_se3 *Tcw, const sfe_camera *cam,
                             const sfe_keypoint *kps, const uint8_t *kp_desc, int m_kps, double radius,
                             double best12_threshold, int32_t *kp_to_query, int32_t *kp_dist);
int sfe_projection_match_se3_dev(sfe_matcher *m, const double *xw_dev, const uint8_t *mp_desc_dev,
                                 const uint8_t *skip_dev, int n, const sfe_se3 *Tcw,
                                 const sfe_camera *cam, const sfe_keypoint *kps_dev,
                                 const uint8_t *kp_desc_dev, int m_kps, double radius,
                                 double best12_threshold, int32_t *kp_to_query_dev,
                                 int32_t *kp_dist_dev);

/* ---- resident frames: the work of Frame::Frame after extract() (src/frame.cpp:50-69) ----------------------
 * A frame keeps its keypoints + descriptors on the device, with the normalised undistorted keypoints
 * (Camera::NormalizedUndistort, src/camera.cpp:95-109: what Frame::GetNormalizedPoint returns) and the spatial index
 * that replaces the per-frame FLANN kd-tree, so matching against it never re-uploads or re-indexes it. */
int sfe_frame_create(sfe_matcher *m, const sfe_keypoint *kps, const uint8_t *desc, int n,
                     const sfe_camera *cam, sfe_frame **out);
/* same from device arrays (e.g. one image's rows of sfe_extract_batch_dev outputs); copied device to device */
int sfe_frame_create_dev(sfe_matcher *m, const sfe_keypoint *kps_dev, const uint8_t *desc_dev, int n,
                         const sfe_camera *cam, sfe_frame **out);
int sfe_frame_destroy(sfe_frame *f);
int sfe_frame_size(const sfe_frame *f, int *n);
int sfe_frame_normalized(sfe_matcher *m, const sfe_frame *f, double *xy /* n x 2 */);
/* StereoFrame::GetDepth (src/frame.cpp:391-409) for every keypoint: xc[i] = (n_x, n_y, 1) * fx * baseline / dx;
 * valid[i] = 1, 0 (no stereo correspondence) or 2 (dx < 0: the reference throws). */
int sfe_frame_stereo_depth(sfe_matcher *m, const sfe_frame *f, const sfe_keypoint *kps_r, int n_r,
                           const int32_t *stereo_idx, double baseline, double *xc /* n x 3 */,
                           uint8_t *valid /* n */);
/* ReprojectionFilter::GetOutlier's per-keypoint test quantity (src/posetracker.cpp:106-137): xw[i] = the map point of
 * keypoint i (has_mp[i] != 0), err[i] = |Project(Tcw Xw) - keypoint| in pixels, +inf when the point is behind the camera
 * (an outlier whatever the threshold), -1 without a map point.  The caller compares with max_reprojection_error.  (As
 * written, the reference's own loop skips every map point the frame holds -- `GetIndex(mp) >= 0`, :118-119 -- so its
 * filter never fires; the quantity is what the comparison at :131-133 would see.) */
int sfe_frame_reprojection_error(sfe_matcher *m, const sfe_frame *f, const double *xw /* n x 3 */,
                                 const uint8_t *has_mp /* n */, const double rt[12], double *err /* n */);
int sfe_frame_reprojection_error_se3(sfe_matcher *m, const sfe_frame *f, const double *xw /* n x 3 */,
                                     const uint8_t *has_mp /* n */, const sfe_se3 *Tcw, double *err /* n */);
/* ProjectionMatch against a resident frame (map points from host memory) */
int sfe_frame_projection_match(sfe_matcher *m, const sfe_frame *f, const double *xw,
                               const uint8_t *mp_desc, const uint8_t *skip, int n, const double rt[12],
                               double radius, double best12_threshold, int32_t *kp_to_query,
                               int32_t *kp_dist);
int sfe_frame_projection_match_se3(sfe_matcher *m, const sfe_frame *f, const double *xw,
                                   const uint8_t *mp_desc, const uint8_t *skip, int n, const sfe_se3 *Tcw,
                                   double radius, double best12_threshold, int32_t *kp_to_query,
                                   int32_t *kp_dist);
/* Frame::SearchRadius (src/frame.cpp:157-178) for q points: idx[i*cap ..] = the keypoints with d^2 < radius^2 in
 * ascending index order, counts[i] = how many there are.  When counts[i] > cap the row holds the cap SMALLEST indices
 * (call again with cap >= counts[i] for all of them). */
int sfe_frame_search_radius(sfe_matcher *m, const sfe_frame *f, const double *uv /* q x 2 */, int q,
                            double radius, int32_t *idx /* q x cap */, int cap, int32_t *counts);
/* Frame::SearchNeareast (src/frame.cpp:180-193): nearest keypoint and SQUARED distance (FLANN L2), ties towards
 * the smaller index; -1 for an empty frame. */
int sfe_frame_search_nearest(sfe_matcher *m, const sfe_frame *f, const double *uv /* q x 2 */, int q,
                             int32_t *kpt_index, double *dist2);

/* ---- BoW transform (Frame::ComputeBoW, src/frame.cpp:419-427 -> DBoW2 TemplatedVocabulary::transform) ----------
 * The vocabulary as TemplatedVocabulary::loadFromTextFile holds it (thirdparty/DBoW2/DBoW2/TemplatedVocabulary.h:
 * 1338-1421): node 0 = root, node i >= 1 has parent[i] < i, a flag is_leaf[i], a 32-byte descriptor and a weight; the
 * children of a node are the nodes naming it as parent, in id order; words are numbered over the flagged nodes in
 * id order.  L = the header's depth (the `nid` level is counted from it).  A node may have at most 2^20 - 1 children
 * (the descent ranks a node's children in 20 bits); a vocabulary with a wider node returns SFE_ERR_UNSUPPORTED. */
int sfe_vocab_create(sfe_matcher *m, int n_nodes, const int32_t *parent, const uint8_t *is_leaf,
                     const uint8_t *desc /* n_nodes x 32 */, const double *weight, int L, sfe_vocab **out);
int sfe_vocab_destroy(sfe_vocab *v);
int sfe_vocab_words(const sfe_vocab *v, int *n_words);
/* per feature: transform(feature, word_id, weight, nid, levelsup) (:1218-1259): word, its weight and the node at
 * level L - levelsup on the way down (0 when the descent ends above that level; the reference leaves it unwritten). */
int sfe_vocab_transform(sfe_matcher *m, const sfe_vocab *v, const uint8_t *desc /* n x 32 */, int n,
                        int levelsup, int32_t *word_id, double *weight, int32_t *node_id);
int sfe_vocab_transform_dev(sfe_matcher *m, const sfe_vocab *v, const uint8_t *desc_dev, int n, int levelsup,
                            int32_t *word_id_dev, double *weight_dev, int32_t *node_id_dev);
/* Host-side BowVector assembly in the reference's order of operations (:1127-1194, BowVector.cpp:34-84).
 * weighting: 0 TF_IDF, 1 TF, 2 IDF, 3 BINARY; norm: 0 none, 1 L1, 2 L2 (what the scoring object's mustNormalize says;
 * ORBvoc.txt is "10 6 0 0": L1_NORM scoring -> norm 1, TF_IDF).  ids ascending; *n_out entries (ids/values may be
 * NULL to query the size).  The FeatureVector is node_id -> the feature indices with weight > 0, in feature order. */
int sfe_bow_assemble(const int32_t *word_id, const double *weight, int n, int weighting, int norm,
                     int32_t *ids, double *values, int cap, int *n_out);
/* sfe_bow_assemble for `count` feature sets at once on the device, bit for bit the same vectors.  Input in the
 * cap-strided layout of the extractor's _dev outputs: set i = rows [i*stride, i*stride + n_dev[i]) of word_id_dev /
 * weight_dev (e.g. sfe_vocab_transform_dev run over count * stride rows, n_dev = sfe_stereo_frames_dev's n_l); rows past
 * n_dev[i] are ignored.  Output: compact CSR on the device, the form sfe_bowdb_add_dev / sfe_bowdb_query_dev take --
 * bow_off_dev[count + 1] (bow_off_dev[0] = 0), set i's BowVector = bow_ids_dev / bow_val_dev [bow_off_dev[i],
 * bow_off_dev[i+1]), ids ascending.  Size bow_ids_dev / bow_val_dev for count * stride elements, which always suffices.
 * stride <= SFE_BOW_ASSEMBLE_MAX_STRIDE (above: SFE_ERR_UNSUPPORTED).  Unknown weighting / norm, null pointers, or an
 * n_dev[i] outside [0, stride] (found on the device; the outputs are then undefined): SFE_ERR_BAD_ARG.  Synchronous: the
 * call reads back one status word at its end.  Scratch of count * stride ids and values is kept in the matcher. */
#define SFE_BOW_ASSEMBLE_MAX_STRIDE 16384
int sfe_bow_assemble_dev(sfe_matcher *m, const int32_t *word_id_dev, const double *weight_dev, const int32_t *n_dev,
                         int count, int stride, int weighting, int norm, int64_t *bow_off_dev, int32_t *bow_ids_dev,
                         double *bow_val_dev);

/* ---- BoW database (DBoW2 TemplatedDatabase with L1 scoring: queryL1, L1Scoring::score in GeneralScoring.cpp) ----------
 * Keyframe BowVectors kept on the device as a forward file (entry offsets, word ids, values), scored against query
 * BowVectors exactly as DBoW2 does, bit for bit.  Only L1 scoring exists (ORBvoc.txt is "10 6 0 0").
 * Vectors travel in CSR form: vector i = ids / values [offsets[i], offsets[i+1]); ids must lie in [0, n_words) and ascend
 * strictly within a vector (a BowVector is a std::map), values must be finite; an empty vector is legal.  Anything else is
 * SFE_ERR_BAD_ARG and leaves the database unchanged.
 * Entry ids are 0, 1, 2, ... in add order, as Database::add returns them.
 * Threads: one database may be used by several matchers of its device, from several threads.  add and query take the
 * database's lock; a query sees exactly the entries added before it was called.  add is synchronous: when it returns its
 * vectors are on the device, and before a growing add frees the buffers it outgrew it waits for the queries already
 * enqueued on any stream. */
#define SFE_BOWDB_MAX_RESULTS 1024
int sfe_bowdb_create(sfe_matcher *m, int n_words, sfe_bowdb **out);
int sfe_bowdb_destroy(sfe_bowdb *db);
int sfe_bowdb_size(const sfe_bowdb *db, int *entries);
/* appends `count` vectors; *first_entry (optional) = the id of the first.  Storage grows by doubling. */
int sfe_bowdb_add(sfe_matcher *m, sfe_bowdb *db, const int64_t *offsets /* count + 1 */, const int32_t *ids,
                  const double *values, int count, int32_t *first_entry);
/* q queries.  For query i: entry[i*max_results + j], score[i*max_results + j] for j < n_results[i] = the entries that share
 * at least one word with it and satisfy (e < max_id || max_id == -1), ordered by DBoW2's raw L1 sum with equal sums in
 * ascending entry id, cut to max_results, score = -sum / 2.0 (Database::query's QueryResults); the rest of the row is
 * -1 / 0.0.  1 <= max_results <= SFE_BOWDB_MAX_RESULTS (above: SFE_ERR_UNSUPPORTED).  dense (optional, q x dense_entries):
 * dense[i*dense_entries + e] = L1Scoring::score(query i, entry e) for the entries e < dense_entries whatever max_id, -0.0
 * where no word is shared -- the similarity matrix.  dense_entries may not exceed the entry count (SFE_ERR_BAD_ARG): a
 * caller that shares the database with an adding thread passes the count it last observed, as it does for max_id. */
int sfe_bowdb_query(sfe_matcher *m, const sfe_bowdb *db, const int64_t *offsets /* q + 1 */, const int32_t *ids,
                    const double *values, int q, int max_id, int max_results, int32_t *entry, double *score,
                    int32_t *n_results, double *dense, int dense_entries);
/* add / query with offsets, ids and values in device memory of the matcher's device (e.g. sfe_bow_assemble_dev's
 * output); query_dev writes entry, score, n_results and the optional dense matrix to device arrays of the same shapes.
 * Everything else is the host calls' contract: the same rules (checked on the device by one kernel before anything
 * changes; a broken rule is SFE_ERR_BAD_ARG and leaves the database unchanged), max_id / max_results / dense_entries,
 * ties, lock and reader events.  Both read the check's result back once and are synchronous: add_dev's vectors are on
 * the device (copied device to device) and query_dev's results written when they return.  *first_entry is host memory. */
int sfe_bowdb_add_dev(sfe_matcher *m, sfe_bowdb *db, const int64_t *offsets_dev /* count + 1 */, const int32_t *ids_dev,
                      const double *values_dev, int count, int32_t *first_entry);
int sfe_bowdb_query_dev(sfe_matcher *m, const sfe_bowdb *db, const int64_t *offsets_dev /* q + 1 */,
                        const int32_t *ids_dev, const double *values_dev, int q, int max_id, int max_results,
                        int32_t *entry_dev, double *score_dev, int32_t *n_results_dev, double *dense_dev,
                        int dense_entries);

/* Sharded ProjectionMatch (map points partitioned over GPUs, frame replicated): each shard emits per keypoint
 * the key (dist << 32 | ~global map-point index) of its best accepted query -- the minimum over shards is the
 * reference's "smaller distance, later query wins ties" (src/matcher.cpp:197-204) -- keys are exchanged with an
 * all-gather and merged + decoded by sfe_projection_merge_dev (keys_dev: shards x m_kps). */
int sfe_projection_match_keys_dev(sfe_matcher *m, const double *xw_dev, const uint8_t *mp_desc_dev,
                                  const uint8_t *skip_dev, int n, int64_t idx_base, const double rt[12],
                                  const sfe_camera *cam, const sfe_keypoint *kps_dev,
                                  const uint8_t *kp_desc_dev, int m_kps, double radius,
                                  double best12_threshold, uint64_t *keys_dev /* m_kps */);
int sfe_projection_match_keys_se3_dev(sfe_matcher *m, const double *xw_dev, const uint8_t *mp_desc_dev,
                                      const uint8_t *skip_dev, int n, int64_t idx_base, const sfe_se3 *Tcw,
                                      const sfe_camera *cam, const sfe_keypoint *kps_dev,
                                      const uint8_t *kp_desc_dev, int m_kps, double radius,
                                      double best12_threshold, uint64_t *keys_dev /* m_kps */);
int sfe_projection_merge_dev(sfe_matcher *m, const uint64_t *keys_dev, int shards, int m_kps,
                             int32_t *kp_to_query_dev, int32_t *kp_dist_dev);

/* Brute-force top-2 over a resident descriptor database shard.
 * idx_base = global index of the shard's first row (multi-GPU sharding).
 * Device memory: 32 B per row; a shard of >= 65536 rows that is searched with >= 256 queries at a time
 * additionally keeps its rows as int8 operand tiles of the tensor-core kernel (256 B per row, built at
 * the first such search when that fits SFE_KNN_TILES_MAX_GB -- default 16 -- and a quarter of the free
 * memory; 0 disables it). */
int sfe_db_create(sfe_matcher *m, const uint8_t *desc_host, int64_t rows, int64_t idx_base,
                  sfe_db **out);
int sfe_db_destroy(sfe_db *db);
/* Growing a database in place, e.g. by each keyframe's descriptors.
 * Indices: appended rows continue the numbering: row r has global index idx_base + r.  An append that would take
 * idx_base + rows to 2^31 returns SFE_ERR_UNSUPPORTED and leaves the database unchanged.  The library knows nothing of
 * other shards: a caller that appends to one shard of a row-sharded map keeps the shards' global ranges disjoint itself
 * (e.g. by appending only to the shard with the highest idx_base).
 * Arguments: null pointers, rows < 0, count < 0, stride < 1 or a desc_dev that is not 16-byte aligned (every allocation of
 * the library or torch is) return SFE_ERR_BAD_ARG.  An n_dev[i] outside [0, stride] is found on the device before anything
 * changes: SFE_ERR_BAD_ARG, the database unchanged.  Appending zero rows succeeds and changes nothing.
 * Synchronous: when an append returns, its rows (and their tensor-core tiles, where the database keeps them) are on the
 * device.  append_dev reads one word (the checked total) back.
 * Threads: several matchers of the device may append to and search one database from several threads.  Appends and every
 * search (sfe_knn2, sfe_knn2_dev, sfe_knn2_sharded) take the database's lock; a search sees exactly the rows appended
 * before it was called, also when it is still queued when a later append runs: an append waits for the queued searches
 * before it frees the buffers it outgrew or rewrites the tile that holds the old last row.
 * Storage grows by capacity doubling (sfe_db_create allocates exactly `rows`); the tiles follow the capacity under the
 * budget above, and are released when they no longer fit it (a later many-query search may build them again). */
int sfe_db_rows(const sfe_db *db, int64_t *rows); /* rows the next search sees */
/* appends `rows` host rows (32 B each); *first_row (optional, host) = local row index of the first appended row */
int sfe_db_append(sfe_matcher *m, sfe_db *db, const uint8_t *desc_host, int64_t rows, int64_t *first_row);
/* appends from device memory of the matcher's device, in the extractor's cap-strided layout (sfe_stereo_frames_dev's
 * desc_l and n_l): set i = rows [i*stride, i*stride + n_dev[i]) of desc_dev, appended in set order, rows in order.
 * n_dev == NULL: every set holds `stride` rows (one contiguous block of count*stride rows). */
int sfe_db_append_dev(sfe_matcher *m, sfe_db *db, const uint8_t *desc_dev, const int32_t *n_dev, int count, int stride,
                      int64_t *first_row);
/* out[q*4] = {idx0, dist0, idx1, dist1}: lexicographic (dist, idx) smallest two; -1/999999999
 * when the shard holds fewer rows.  The ratio test is (2*dist0 < dist1) on the caller's side. */
int sfe_knn2(sfe_matcher *m, const sfe_db *db, const uint8_t *queries, int q, int32_t *out);
/* resident variant: keys_dev[q*2 + r] = (uint64)dist << 32 | global idx (r-th best);
 * this is what one rank contributes to the all-gather. */
int sfe_knn2_dev(sfe_matcher *m, const sfe_db *db, const uint8_t *queries_dev, int q,
                 uint64_t *keys_dev);
/* merge `shards` gathered key arrays (shards x q x 2) into out_dev[q*4] */
int sfe_knn2_merge_dev(sfe_matcher *m, const uint64_t *keys_dev, int shards, int q,
                       int32_t *out_dev);

/* ---- multi-GPU: sharded database / sharded local map (SURVEY §8e) -----------------------------------------------
 * A communicator is one rank's end of an exchange between `world` GPUs of one box.  The data path is ONE step: every rank's
 * kernel stores its per-query top-2 keys (kNN) or per-keypoint best keys (ProjectionMatch) straight into every peer's
 * inbox over NVLink peer memory and raises a flag; the merge kernel of each rank waits on its own flags.  No host
 * round trip, no NCCL call and no extra copy between the local kernels, the exchange and the merge; every rank ends up
 * with the full merged result (all-gather semantics).  Results are exact and independent of the shard boundaries
 * (ties break on the global index / the global query order).
 *   - one process per GPU (torchrun, MPI): sfe_comm_create on every rank, exchange the 64-byte handles of
 *     sfe_comm_export by any means (one all-gather at set-up time), sfe_comm_connect with all of them;
 *   - one process driving several GPUs: sfe_comm_create_local fills one connected communicator per device.
 * The sharded calls are COLLECTIVE: every rank must issue the same sequence of them, with its own shard.  They return
 * as soon as their kernels are enqueued on the matcher's stream (whatever the matcher's async mode: a host thread that
 * drives several ranks could not otherwise enqueue rank 1 while rank 0 waits for it); sfe_matcher_wait completes them.
 * Use one communicator per matcher.  A rank that never shows up is detected by its peers after 5 s: their results are
 * invalid and sfe_comm_status reports it. */
#define SFE_COMM_HANDLE_BYTES 64
int sfe_comm_create(int device, int rank, int world, sfe_comm **out); /* world <= 16 */
int sfe_comm_export(sfe_comm *c, uint8_t handle[SFE_COMM_HANDLE_BYTES]);
int sfe_comm_connect(sfe_comm *c, const uint8_t *handles /* world x SFE_COMM_HANDLE_BYTES, rank order */);
int sfe_comm_create_local(const int *devices, int n, sfe_comm **out /* n handles */);
int sfe_comm_destroy(sfe_comm *c);
int sfe_comm_status(sfe_comm *c, int *stalled_rank /* optional: -1 = none */);
/* Brute-force top-2 of q resident queries (the same on every rank) against the row-sharded map: `shard` = this rank's
 * rows (sfe_db_create with idx_base = global index of its first row).  out_dev[q*4] = {idx0, dist0, idx1, dist1} over
 * the WHOLE map, on every rank.  q <= 32768. */
int sfe_knn2_sharded(sfe_matcher *m, sfe_comm *c, const sfe_db *shard, const uint8_t *queries_dev, int q,
                     int32_t *out_dev);
/* ProjectionMatch of a local map sharded by map points against one resident frame (the same on every rank): this rank's
 * n points are the global map points [idx_base, idx_base + n) of the caller's order.  kp_to_query_dev[j] = GLOBAL index of
 * the map point matched to keypoint j or -1, kp_dist_dev[j] (optional) = its distance, on every rank. */
int sfe_projection_match_sharded(sfe_matcher *m, sfe_comm *c, const sfe_frame *f, const double *xw_dev,
                                 const uint8_t *mp_desc_dev, const uint8_t *skip_dev, int n, int64_t idx_base,
                                 const sfe_se3 *Tcw, double radius, double best12_threshold,
                                 int32_t *kp_to_query_dev, int32_t *kp_dist_dev);

/* ---- Front-end results as one byte stream (SURVEY §8f row 4) -------------------------------------------------
 * The reference has no on-disk form of a frame (Memento save is `#if 0`, src/pipeline.cpp:231-241); this is the one
 * the batched front end hands to an unchanged back end or another process.  Host-only, little-endian, packed:
 *   header (48 B): "SFER", u32 version = 1, u32 frames, u32 flags (SFE_RES_*), u32 w, u32 h, u64 payload bytes,
 *                  u64 FNV-1a-64 of the payload, 8 B reserved
 *   per frame    : u32 n_l, u32 n_r, kps_l[n_l] (28 B each = cv::KeyPoint), desc_l[n_l][32],
 *                  if STEREO: kps_r[n_r], desc_r[n_r][32], stereo_idx[n_l] i32, stereo_dist[n_l] i32
 *                  if TRACK : track_idx[n_l] i32, track_dist[n_l] i32
 * Arrays are the cap-strided ones sfe_stereo_frames / sfe_stereo_sequence fill; only the n valid rows travel. */
enum { SFE_RES_STEREO = 1, SFE_RES_TRACK = 2 };
int sfe_results_size(int frames, const int32_t *n_l, const int32_t *n_r, int flags, size_t *bytes);
int sfe_results_pack(void *buf, size_t buf_bytes, int frames, int cap, int w, int h, int flags,
                     const sfe_keypoint *kps_l, const uint8_t *desc_l, const int32_t *n_l,
                     const sfe_keypoint *kps_r, const uint8_t *desc_r, const int32_t *n_r,
                     const int32_t *stereo_idx, const int32_t *stereo_dist, const int32_t *track_idx,
                     const int32_t *track_dist, size_t *written);
/* header fields + the largest per-frame keypoint count (the cap an unpack needs); verifies magic, sizes, checksum */
int sfe_results_info(const void *buf, size_t bytes, int *frames, int *flags, int *w, int *h, int *max_n);
/* inverse of pack into cap-strided arrays; rows past n are left untouched; absent sections may be NULL */
int sfe_results_unpack(const void *buf, size_t bytes, int cap, sfe_keypoint *kps_l, uint8_t *desc_l, int32_t *n_l,
                       sfe_keypoint *kps_r, uint8_t *desc_r, int32_t *n_r, int32_t *stereo_idx,
                       int32_t *stereo_dist, int32_t *track_idx, int32_t *track_dist);

#ifdef __cplusplus
}
#endif
#endif /* SFE_H_ */
