// Hamming matchers for sm_100a behind the sfe C ABI: StereoMatch (reference src/matcher.cpp:54-132),
// ProjectionMatch (:134-209) and the brute-force top-2 that BASELINE config 4 defines over the same
// inner loop.  XOR + __popc over 8 words; best / second-best kept as packed (dist, index) keys so
// "strict < in ascending index order" (:114-123) becomes a plain unsigned min.
#include <algorithm>
#include <cmath>

#include <mutex>

#include "sfe_extract.cuh"

namespace sfe {

constexpr uint32_t kNoKey = 0xFFFFFFFFu;

__device__ __forceinline__ void top2_insert(uint32_t &k0, uint32_t &k1, uint32_t key) {
    k1 = min(k1, max(k0, key));
    k0 = min(k0, key);
}

__device__ __forceinline__ void load_desc(const uint8_t *p, uint32_t d[8]) {
    const uint4 a = __ldg((const uint4 *)p), b = __ldg((const uint4 *)p + 1);
    d[0] = a.x; d[1] = a.y; d[2] = a.z; d[3] = a.w;
    d[4] = b.x; d[5] = b.y; d[6] = b.z; d[7] = b.w;
}

// ---------------------------------------------------------------------------------------------
// StereoMatch.  The reference's int(y/10) row buckets (:60-66,83-95) only pre-select: |dy| <= 3 < 10 keeps
// every passing candidate inside buckets b-1..b+1, so the candidate set is every right keypoint passing the
// dy / dx filters (:103-110).  Here: one CTA = 512 left keypoints of one frame.  The CTA counting-sorts the
// right keypoints of its frame into a 2-D bucket grid in shared memory (8-px rows x 64-px columns: the dx window
// [0, max_dx] is as selective as the dy one), then one thread per left keypoint walks the few buckets that can hold
// a candidate -- per bucket row a contiguous range of the sorted order -- applies the reference's exact float
// filters and fetches descriptors only for the survivors (about ten candidates instead of the ~90 of a row-only
// index).  Visiting order is free: best / second best are packed (dist << 16 | index) keys, so "strict < in
// ascending index order" (:114-123) is a plain unsigned min.
// ---------------------------------------------------------------------------------------------
constexpr int kStereoChunk = 2048;    // right keypoints indexed in shared memory at a time
constexpr int kStereoPerThreadMax = 2; // left keypoints per thread: 2 (512 per CTA) for batches, 1 when a call carries so few
                                       // frames that more CTAs shorten it
constexpr int kRowShift = 3, kRowBuckets = 128;  // 8-px rows; y >= 1016 shares the last row of buckets
constexpr int kColShift = 6, kColBuckets = 32;   // 64-px columns; x >= 1984 shares the last column
constexpr int kStereoCells = kRowBuckets * kColBuckets;

__device__ __forceinline__ int row_bucket(float y) {
    return min(max((int)floorf(y) >> kRowShift, 0), kRowBuckets - 1);  // monotone in y
}
__device__ __forceinline__ int col_bucket(float x) {
    return min(max((int)floorf(x) >> kColShift, 0), kColBuckets - 1);  // monotone in x
}

// thr_y / thr_dx: the largest floats <= y_threshold / max_dx, so that for a float d the reference's double
// comparison (double)d > T is exactly d > thr (no float lies strictly between thr and T).  reach_y / reach_dx:
// |float(a - b)| <= T implies |a - b| < T + 1 for coordinates < 2^13, which bounds the buckets worth visiting.
// kLanes lanes share one left keypoint (candidate positions t = lane, lane + kLanes, ... of every bucket range, merged by
// shuffles): a one-pair call is bound by the longest walk in each warp, and four lanes per keypoint cut that walk fourfold
// and spread the frame over four times as many CTAs.
template <int kStereoPerThread, int kLanes>
__global__ void __launch_bounds__(256) stereo_match_kernel(int cap, const sfe_keypoint *__restrict__ kl,
                                                           const uint8_t *__restrict__ dl, const int32_t *__restrict__ nl,
                                                           const sfe_keypoint *__restrict__ kr,
                                                           const uint8_t *__restrict__ dr, const int32_t *__restrict__ nr,
                                                           float thr_y, float thr_dx, float reach_y, float reach_dx, double ratio,
                                                           int32_t *__restrict__ out_idx, int32_t *__restrict__ out_dist) {
    pdl_enter();
    __shared__ float2 rxy[kStereoChunk];            // right keypoints of the chunk, in bucket order
    __shared__ uint16_t order[kStereoChunk];        // their indices inside the chunk
    __shared__ uint16_t start[kStereoCells + 1];    // bucket c = positions start[c] .. start[c + 1]
    __shared__ __align__(16) uint16_t fill[kStereoCells];
    __shared__ int warp_tot[8];
    const int f = blockIdx.y, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int n_l = min(nl[f], cap), n_r = min(nr[f], cap);
    const size_t base = (size_t)f * cap;
    constexpr int kSlots = 256 / kLanes, kStereoPerCta = kSlots * kStereoPerThread;
    const int i0 = blockIdx.x * kStereoPerCta, sub = tid % kLanes, slot = tid / kLanes;
    uint32_t k0[kStereoPerThread], k1[kStereoPerThread];
#pragma unroll
    for (int k = 0; k < kStereoPerThread; k++) k0[k] = k1[k] = kNoKey;
    const bool block_has_work = i0 < n_l;
    for (int c0 = 0; c0 < n_r && block_has_work; c0 += kStereoChunk) {
        const int cn = min(kStereoChunk, n_r - c0);
        __syncthreads();
        for (int c = tid; c < kStereoCells; c += 256) fill[c] = 0;
        __syncthreads();
        // count: the shared-memory atomics work on 32-bit words, two 16-bit counters per word
        uint32_t *fill32 = (uint32_t *)fill;
        // the thread's right keypoints of this chunk: loaded once, all loads in flight together, used by the count and the scatter
        constexpr int kPerThread = kStereoChunk / 256;
        float2 rk[kPerThread];
#pragma unroll
        for (int k = 0; k < kPerThread; k++) {
            const int j = tid + 256 * k;
            if (j < cn) {
                const sfe_keypoint &q = kr[base + c0 + j];
                rk[k] = make_float2(q.x, q.y);
            }
        }
#pragma unroll
        for (int k = 0; k < kPerThread; k++) {
            if (tid + 256 * k < cn) {
                const int c = row_bucket(rk[k].y) * kColBuckets + col_bucket(rk[k].x);
                atomicAdd(&fill32[c >> 1], 1u << (16 * (c & 1)));
            }
        }
        __syncthreads();
        {   // exclusive scan of the bucket counts: 16 consecutive buckets per thread
            constexpr int kPer = kStereoCells / 256;
            int cnt[kPer], tot = 0;
#pragma unroll
            for (int k = 0; k < kPer; k++) {
                cnt[k] = fill[tid * kPer + k];
                tot += cnt[k];
            }
            int inc = tot;
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
                const int u = __shfl_up_sync(0xffffffffu, inc, o);
                if (lane >= o) inc += u;
            }
            if (lane == 31) warp_tot[warp] = inc;
            __syncthreads();
            int run = inc - tot;
#pragma unroll
            for (int w2 = 0; w2 < 8; w2++) run += w2 < warp ? warp_tot[w2] : 0;
#pragma unroll
            for (int k = 0; k < kPer; k++) {
                start[tid * kPer + k] = (uint16_t)run;
                fill[tid * kPer + k] = (uint16_t)run;  // becomes the bucket's write cursor
                run += cnt[k];
            }
            if (tid == 255) start[kStereoCells] = (uint16_t)run;
        }
        __syncthreads();
#pragma unroll
        for (int k = 0; k < kPerThread; k++) {
            const int j = tid + 256 * k;
            if (j < cn) {
                const float x = rk[k].x, y = rk[k].y;
                const int c = row_bucket(y) * kColBuckets + col_bucket(x);
                const uint32_t old = atomicAdd(&fill32[c >> 1], 1u << (16 * (c & 1)));
                const int t = (old >> (16 * (c & 1))) & 0xFFFF;
                order[t] = (uint16_t)j;
                rxy[t] = make_float2(x, y);
            }
        }
        __syncthreads();
#pragma unroll
        for (int k = 0; k < kStereoPerThread; k++) {
            const int i = i0 + k * kSlots + slot;
            if (i >= n_l) continue;
            const float lx = kl[base + i].x, ly = kl[base + i].y;
            uint32_t a[8];
            load_desc(dl + (base + i) * 32, a);
            const int yb0 = row_bucket(ly - reach_y), yb1 = row_bucket(ly + reach_y);
            const int xb0 = col_bucket(lx - reach_dx), xb1 = col_bucket(lx + 1.f);
            uint32_t q0 = k0[k], q1 = k1[k];
            for (int yb = yb0; yb <= yb1; yb++) {
                const int t1 = start[yb * kColBuckets + xb1 + 1];
                for (int t = start[yb * kColBuckets + xb0] + sub; t < t1; t += kLanes) {
                    const float2 r = rxy[t];
                    const float dx = __fsub_rn(lx, r.x), dy = __fsub_rn(ly, r.y);  // float subtraction, as in the reference
                    if (fabsf(dy) > thr_y || dx < 0.f || dx > thr_dx) continue;   // :103-110
                    const int j = c0 + order[t];
                    const uint4 *d = (const uint4 *)(dr + (base + j) * 32);
                    const uint4 b0 = __ldg(d), b1 = __ldg(d + 1);
                    top2_insert(q0, q1, (uint32_t)hamming8_csa(a, b0.x, b0.y, b0.z, b0.w, b1.x, b1.y, b1.z, b1.w) << 16 | (uint32_t)j);
                }
            }
            k0[k] = q0;
            k1[k] = q1;
        }
    }
#pragma unroll
    for (int k = 0; k < kStereoPerThread; k++) {
        const int i = i0 + k * kSlots + slot;
        uint32_t q0 = k0[k], q1 = k1[k];
#pragma unroll
        for (int o = 1; o < kLanes; o <<= 1) {  // the lanes of a keypoint hold disjoint candidates: merge their top-2 (kNoKey never enters)
            const uint32_t u0 = __shfl_xor_sync(0xffffffffu, q0, o), u1 = __shfl_xor_sync(0xffffffffu, q1, o);
            top2_insert(q0, q1, u0);
            top2_insert(q0, q1, u1);
        }
        if (i >= cap || sub != 0) continue;
        int idx = -1, dist = -1;
        if (i < n_l && q0 != kNoKey) {
            const double d0 = (double)(q0 >> 16), d1 = q1 == kNoKey ? 999999999. : (double)(q1 >> 16);
            if (d0 < d1 * ratio) {  // :125-128
                idx = (int)(q0 & 0xFFFF);
                dist = (int)(q0 >> 16);
            }
        }
        out_idx[base + i] = idx;
        if (out_dist) out_dist[base + i] = dist;
    }
}

static float float_at_most(double v) {  // largest float <= v
    float f = (float)v;
    if ((double)f > v) f = nextafterf(f, -INFINITY);
    return f;
}

void launch_stereo_match(cudaStream_t st, int frames, int cap, const sfe_keypoint *kl, const uint8_t *dl, const int32_t *nl,
                         const sfe_keypoint *kr, const uint8_t *dr, const int32_t *nr, double y_thr, double max_dx,
                         double ratio, int32_t *out_idx, int32_t *out_dist, bool pdl) {
    // rows a candidate can sit in: |float(ly - ry)| <= y_thr implies |ly - ry| < y_thr + 1 for coordinates < 2^13
    const float reach = (float)(std::max(y_thr, 0.0) + 1.0), reach_dx = (float)(std::max(max_dx, 0.0) + 1.0);
    if (frames * div_up(cap, 64) <= 2 * 148)  // a few frames (two CTAs per SM of a B200 at most): four lanes per keypoint, 64 keypoints per CTA
        launch_k(stereo_match_kernel<1, 4>, dim3(div_up(cap, 64), frames), 256, 0, st, pdl, cap, kl, dl, nl, kr, dr, nr, float_at_most(y_thr),
                 float_at_most(max_dx), reach, reach_dx, ratio, out_idx, out_dist);
    else if (frames * div_up(cap, 512) < 64)
        launch_k(stereo_match_kernel<1, 1>, dim3(div_up(cap, 256), frames), 256, 0, st, pdl, cap, kl, dl, nl, kr, dr, nr, float_at_most(y_thr),
                 float_at_most(max_dx), reach, reach_dx, ratio, out_idx, out_dist);
    else
        launch_k(stereo_match_kernel<kStereoPerThreadMax, 1>, dim3(div_up(cap, 256 * kStereoPerThreadMax), frames), 256, 0, st, pdl, cap, kl, dl,
                 nl, kr, dr, nr, float_at_most(y_thr), float_at_most(max_dx), reach, reach_dx, ratio, out_idx, out_dist);
}

// ---------------------------------------------------------------------------------------------
// ProjectionMatch.  The per-frame FLANN kd-tree (src/frame.cpp:59-68,170-178) is replaced by a
// uniform 32-px bucket grid over the frame's keypoints, rebuilt per call on the device; the
// candidate set "all keypoints with d^2 < r^2" is identical, and candidate order does not matter
// (SURVEY §8a invariants).
// ---------------------------------------------------------------------------------------------
constexpr int kGridShift = 5;

struct KpGrid {
    int gw, gh, m;
    int *cell_start;   // gw*gh + 1
    int *cell_fill;    // gw*gh
    int *order;        // m: keypoint indices sorted by cell
    double2 *sxy;      // m: keypoint coordinates as doubles, in cell order (the matcher's distance test is in double)
    uint4 *sdesc;      // 2 m: descriptors in cell order
};

__device__ __forceinline__ int grid_cell(const KpGrid &G, float x, float y) {
    int cx = (int)floorf(x) >> kGridShift, cy = (int)floorf(y) >> kGridShift;
    cx = min(max(cx, 0), G.gw - 1);
    cy = min(max(cy, 0), G.gh - 1);
    return cy * G.gw + cx;
}

__global__ void grid_count_kernel(KpGrid G, const sfe_keypoint *__restrict__ kps) {
    const int j = blockIdx.x * blockDim.x + threadIdx.x;
    if (j < G.m) atomicAdd(&G.cell_start[grid_cell(G, kps[j].x, kps[j].y) + 1], 1);
}

__global__ void __launch_bounds__(256) grid_scan_kernel(KpGrid G) {  // one CTA: inclusive scan of cell_start[0 .. cells]
    __shared__ int chunk_sum[256];
    const int n = G.gw * G.gh, tid = threadIdx.x;
    const int per = (n + 1 + 255) / 256, c0 = min(tid * per, n + 1), c1 = min(c0 + per, n + 1);
    int acc = 0;
    for (int c = c0; c < c1; c++) acc += G.cell_start[c];
    chunk_sum[tid] = acc;
    __syncthreads();
    if (tid < 32) {  // exclusive scan of the 256 chunk totals by one warp, 8 per lane
        int v[8], tot = 0;
#pragma unroll
        for (int k = 0; k < 8; k++) {
            v[k] = chunk_sum[tid * 8 + k];
            tot += v[k];
        }
        int inc = tot;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const int x = __shfl_up_sync(0xffffffffu, inc, o);
            if (tid >= o) inc += x;
        }
        int run = inc - tot;
#pragma unroll
        for (int k = 0; k < 8; k++) {
            chunk_sum[tid * 8 + k] = run;
            run += v[k];
        }
    }
    __syncthreads();
    acc = chunk_sum[tid];
    for (int c = c0; c < c1; c++) {
        acc += G.cell_start[c];
        G.cell_start[c] = acc;
    }
    for (int i = tid; i < n; i += 256) G.cell_fill[i] = 0;
}

__global__ void grid_fill_kernel(KpGrid G, const sfe_keypoint *__restrict__ kps, const uint8_t *__restrict__ desc) {
    const int j = blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= G.m) return;
    const float x = kps[j].x, y = kps[j].y;
    const int c = grid_cell(G, x, y), t = G.cell_start[c] + atomicAdd(&G.cell_fill[c], 1);
    G.order[t] = j;
    G.sxy[t] = make_double2((double)x, (double)y);
    if (desc) {
        const uint4 *d = (const uint4 *)(desc + (size_t)j * 32);
        G.sdesc[2 * t] = __ldg(d);
        G.sdesc[2 * t + 1] = __ldg(d + 1);
    }
}

// predicted_Tcw as the caller holds it.  quat != 0: v = {qx, qy, qz, qw, tx, ty, tz}, a g2o::SE3Quat (the reference,
// src/matcher.cpp:151); quat == 0: v = row-major 3x4 [R|t].
struct Pose {
    double v[12];
    int quat;
};
static Pose pose_from_rt(const double rt[12]) {
    Pose T{};
    memcpy(T.v, rt, sizeof(double) * 12);
    return T;
}
static Pose pose_from_se3(const sfe_se3 *q) {
    Pose T{};
    T.v[0] = q->qx; T.v[1] = q->qy; T.v[2] = q->qz; T.v[3] = q->qw; T.v[4] = q->tx; T.v[5] = q->ty; T.v[6] = q->tz;
    T.quat = 1;
    return T;
}

struct ProjParams {
    Pose T;
    sfe_camera cam;
    double radius, ratio;
};

// Xc = Tcw Xw, Camera::Project, IsInImage: false when the point is behind the camera, outside the image or not a number
// Xc = Tcw Xw and Camera::Project (with distortion); false when the point is behind the camera (z < 0)
__device__ __forceinline__ bool project_uv(const Pose &T, const sfe_camera &cam, double X, double Y, double Z, double &u, double &v);

__device__ __forceinline__ bool project_point(const ProjParams &P, double X, double Y, double Z, double &u, double &v) {
    if (!project_uv(P.T, P.cam, X, Y, Z, u, v)) return false;  // :151-153
    if (u < 0. || v < 0. || u > (double)P.cam.width || v > (double)P.cam.height) return false;  // IsInImage, :26-36
    return u == u && v == v;  // NaN: the radius search finds nothing
}

__device__ __forceinline__ bool project_uv(const Pose &T, const sfe_camera &cam, double X, double Y, double Z, double &u, double &v) {
    // Xc = Tcw * Xw without contraction (:151)
    double xc, yc, zc;
    if (T.quat) {
        // g2o::SE3Quat::operator*: _t + _r * v, with Eigen's quaternion-vector product (Quaternion.h, _transformVector):
        // uv = q.vec x v; uv += uv; (v + q.w * uv) + q.vec x uv
        const double qx = T.v[0], qy = T.v[1], qz = T.v[2], qw = T.v[3];
        double ux = __dsub_rn(__dmul_rn(qy, Z), __dmul_rn(qz, Y));
        double uy = __dsub_rn(__dmul_rn(qz, X), __dmul_rn(qx, Z));
        double uz = __dsub_rn(__dmul_rn(qx, Y), __dmul_rn(qy, X));
        ux = __dadd_rn(ux, ux); uy = __dadd_rn(uy, uy); uz = __dadd_rn(uz, uz);
        const double cx = __dsub_rn(__dmul_rn(qy, uz), __dmul_rn(qz, uy));
        const double cy = __dsub_rn(__dmul_rn(qz, ux), __dmul_rn(qx, uz));
        const double cz = __dsub_rn(__dmul_rn(qx, uy), __dmul_rn(qy, ux));
        xc = __dadd_rn(T.v[4], __dadd_rn(__dadd_rn(X, __dmul_rn(qw, ux)), cx));
        yc = __dadd_rn(T.v[5], __dadd_rn(__dadd_rn(Y, __dmul_rn(qw, uy)), cy));
        zc = __dadd_rn(T.v[6], __dadd_rn(__dadd_rn(Z, __dmul_rn(qw, uz)), cz));
    } else {
        const double *rt = T.v;  // rows left to right
        xc = __dadd_rn(__dadd_rn(__dadd_rn(__dmul_rn(rt[0], X), __dmul_rn(rt[1], Y)), __dmul_rn(rt[2], Z)), rt[3]);
        yc = __dadd_rn(__dadd_rn(__dadd_rn(__dmul_rn(rt[4], X), __dmul_rn(rt[5], Y)), __dmul_rn(rt[6], Z)), rt[7]);
        zc = __dadd_rn(__dadd_rn(__dadd_rn(__dmul_rn(rt[8], X), __dmul_rn(rt[9], Y)), __dmul_rn(rt[10], Z)), rt[11]);
    }
    if (zc < 0.) return false;
    // Camera::Project + Distort, src/camera.cpp:50-79
    const double x = __ddiv_rn(xc, zc), y = __ddiv_rn(yc, zc);
    const double r2 = __dadd_rn(__dmul_rn(x, x), __dmul_rn(y, y)), r4 = __dmul_rn(r2, r2);
    const double a1 = __dmul_rn(__dmul_rn(2., x), y);
    const double a2 = __dadd_rn(r2, __dmul_rn(__dmul_rn(2., x), x));
    const double a3 = __dadd_rn(r2, __dmul_rn(__dmul_rn(2., y), y));
    const double cdist = __dadd_rn(__dadd_rn(1., __dmul_rn(cam.d[0], r2)), __dmul_rn(cam.d[1], r4));
    const double xd = __dadd_rn(__dadd_rn(__dmul_rn(x, cdist), __dmul_rn(cam.d[2], a1)), __dmul_rn(cam.d[3], a2));
    const double yd = __dadd_rn(__dadd_rn(__dmul_rn(y, cdist), __dmul_rn(cam.d[2], a3)), __dmul_rn(cam.d[3], a1));
    u = __dadd_rn(__dmul_rn(cam.fx, xd), cam.cx);
    v = __dadd_rn(__dmul_rn(cam.fy, yd), cam.cy);
    return true;
}

// One projected map point against the frame behind G: radius search over the bucket grid, best / second-best Hamming,
// ratio test, then the conflict rule as an atomicMin on the winning keypoint's key.  `query` is the point's position in
// the caller's order (the later query wins a distance tie, :197-204).
__device__ __forceinline__ void match_projected(const KpGrid &G, const ProjParams &P, double u, double v, const uint32_t a[8],
                                                uint32_t query, unsigned long long *__restrict__ best) {
    const double r2max = __dmul_rn(P.radius, P.radius);
    const int cy0 = min(max((int)floor(v - P.radius) >> kGridShift, 0), G.gh - 1);
    const int cy1 = min(max((int)floor(v + P.radius) >> kGridShift, 0), G.gh - 1);
    uint32_t k0 = kNoKey, k1 = kNoKey;
    for (int cy = cy0; cy <= cy1; cy++) {
        // keypoints of cell row cy have y in [32 cy, 32 cy + 32) (the border rows also hold what was clamped into them):
        // the circle's half-width on that band bounds the cells worth visiting -- a superset of the d^2 < r^2 set
        const double lo = cy == 0 ? -1e300 : (double)(cy << kGridShift), hi = cy == G.gh - 1 ? 1e300 : (double)((cy + 1) << kGridShift);
        const double dy = fmax(fmax(lo - v, v - hi), 0.);
        const double h2 = r2max - dy * dy;
        if (!(h2 > 0.)) continue;
        const double hw = sqrt(h2) + 1.;
        const int cx0 = min(max((int)floor(u - hw) >> kGridShift, 0), G.gw - 1);
        const int cx1 = min(max((int)floor(u + hw) >> kGridShift, 0), G.gw - 1);
        const int s = G.cell_start[cy * G.gw + cx0], e = G.cell_start[cy * G.gw + cx1 + 1];  // cells of a row are contiguous
        for (int t = s; t < e; t++) {
            const double2 p = G.sxy[t];
            const double ddx = u - p.x, ddy = v - p.y;
            const double d2 = __dadd_rn(__dmul_rn(ddx, ddx), __dmul_rn(ddy, ddy));
            if (!(d2 < r2max)) continue;  // FLANN radius search: strict <
            const uint4 b0 = G.sdesc[2 * t], b1 = G.sdesc[2 * t + 1];
            top2_insert(k0, k1, (uint32_t)hamming8_csa(a, b0.x, b0.y, b0.z, b0.w, b1.x, b1.y, b1.z, b1.w) << 16 | (uint32_t)G.order[t]);
        }
    }
    if (k0 == kNoKey) return;
    const double d0 = (double)(k0 >> 16), d1 = k1 == kNoKey ? 999999999. : (double)(k1 >> 16);
    if (d0 < d1 * P.ratio) {
        // :197-204 processed sequentially keeps the smaller distance and lets the LATER query win a
        // tie: that is the minimum of (dist, -query) over all accepted queries of a keypoint
        const unsigned long long key = (unsigned long long)(k0 >> 16) << 32 | (0xFFFFFFFFu - query);
        atomicMin(&best[k0 & 0xFFFF], key);
    }
}

__device__ __forceinline__ void project_and_match(const KpGrid &G, const ProjParams &P, double X, double Y, double Z,
                                                  const uint32_t a[8], uint32_t query, unsigned long long *__restrict__ best) {
    double u, v;
    if (project_point(P, X, Y, Z, u, v)) match_projected(G, P, u, v, a, query, best);
}

__global__ void __launch_bounds__(128) projection_match_kernel(KpGrid G, ProjParams P, int n, uint32_t idx_base,
                                                               const double *__restrict__ xw,
                                                               const uint8_t *__restrict__ mp_desc,
                                                               const uint8_t *__restrict__ skip,
                                                               unsigned long long *__restrict__ best) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    if (skip && skip[i]) return;  // curr_frame->GetIndex(mp) >= 0, :144
    uint32_t a[8];
    load_desc(mp_desc + (size_t)i * 32, a);
    project_and_match(G, P, xw[3 * (size_t)i], xw[3 * (size_t)i + 1], xw[3 * (size_t)i + 2], a, idx_base + (uint32_t)i, best);
}

// Large local maps: the lanes of a warp walk the bucket grid in lock step, so a warp costs as much as its longest
// candidate list, and with the points in the caller's order that is 3x the average (ncu: 11 of 32 lanes active).  The
// points are therefore counting-sorted by the grid cell they project into (1024 row-major bins; points that project
// nowhere are dropped) and matched in that order: neighbouring lanes see the same cells and about the same number of
// candidates.  Results do not depend on the order -- a point's key carries its own index.
//   proj_bin_kernel      per chunk of 2048 points: bin of every point + the chunk's histogram
//   proj_offsets_kernel  per bin: exclusive prefix of the chunk counts, bin total
//   proj_scan_kernel     exclusive scan of the 1024 bin totals
//   proj_scatter_kernel  per chunk: positions from shared-memory cursors -> perm
//   proj_match_sorted_kernel  thread e handles point perm[e]
constexpr int kProjChunk = 2048, kProjBins = 1024;
constexpr int kProjSortMin = 32768;  // below this many map points the five extra launches cost more than the divergence

__global__ void __launch_bounds__(256) proj_bin_kernel(int gw, int gh, ProjParams P, int n, const double *__restrict__ xw,
                                                       const uint8_t *__restrict__ skip, uint16_t *__restrict__ bins,
                                                       int *__restrict__ hist) {
    __shared__ int h[kProjBins];
    const int tid = threadIdx.x, base = blockIdx.x * kProjChunk, cn = min(kProjChunk, n - base), cells = gw * gh;
    for (int b = tid; b < kProjBins; b += 256) h[b] = 0;
    __syncthreads();
    for (int k = tid; k < cn; k += 256) {
        const int i = base + k;
        uint16_t bin = 0xFFFF;  // dropped
        double u, v;
        if (!(skip && skip[i]) && project_point(P, xw[3 * (size_t)i], xw[3 * (size_t)i + 1], xw[3 * (size_t)i + 2], u, v)) {
            const int cx = min(max((int)floor(u) >> kGridShift, 0), gw - 1), cy = min(max((int)floor(v) >> kGridShift, 0), gh - 1);
            bin = (uint16_t)(((long long)(cy * gw + cx) * kProjBins) / cells);
            atomicAdd(&h[bin], 1);
        }
        bins[i] = bin;
    }
    __syncthreads();
    for (int b = tid; b < kProjBins; b += 256) hist[(size_t)blockIdx.x * kProjBins + b] = h[b];
}

// warp = bin: hist[c][bin] becomes the number of the bin's points in chunks before c; tot[bin] = the bin's size
__global__ void __launch_bounds__(256) proj_offsets_kernel(int chunks, int *__restrict__ hist, int *__restrict__ tot) {
    const int bin = blockIdx.x * 8 + (threadIdx.x >> 5), lane = threadIdx.x & 31;
    int run = 0;
    for (int c0 = 0; c0 < chunks; c0 += 32) {
        const int c = c0 + lane;
        const int v = c < chunks ? hist[(size_t)c * kProjBins + bin] : 0;
        int inc = v;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const int x = __shfl_up_sync(0xffffffffu, inc, o);
            if (lane >= o) inc += x;
        }
        if (c < chunks) hist[(size_t)c * kProjBins + bin] = run + inc - v;
        run += __shfl_sync(0xffffffffu, inc, 31);
    }
    if (lane == 0) tot[bin] = run;
}

__global__ void __launch_bounds__(kProjBins) proj_scan_kernel(int *__restrict__ tot) {  // tot[b] -> first position of bin b; tot[1024] = all
    __shared__ int wsum[32];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int v = tot[tid];
    int inc = v;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const int x = __shfl_up_sync(0xffffffffu, inc, o);
        if (lane >= o) inc += x;
    }
    if (lane == 31) wsum[warp] = inc;
    __syncthreads();
    if (warp == 0) {
        const int w = wsum[lane];
        int winc = w;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const int x = __shfl_up_sync(0xffffffffu, winc, o);
            if (lane >= o) winc += x;
        }
        wsum[lane] = winc - w;
    }
    __syncthreads();
    tot[tid] = wsum[warp] + inc - v;
    if (tid == kProjBins - 1) tot[kProjBins] = wsum[warp] + inc;
}

__global__ void __launch_bounds__(256) proj_scatter_kernel(int n, const uint16_t *__restrict__ bins, const int *__restrict__ hist,
                                                           const int *__restrict__ tot, uint32_t *__restrict__ perm) {
    __shared__ int cur[kProjBins];
    const int tid = threadIdx.x, base = blockIdx.x * kProjChunk, cn = min(kProjChunk, n - base);
    for (int b = tid; b < kProjBins; b += 256) cur[b] = tot[b] + hist[(size_t)blockIdx.x * kProjBins + b];
    __syncthreads();
    for (int k = tid; k < cn; k += 256) {
        const int bin = bins[base + k];
        if (bin != 0xFFFF) perm[atomicAdd(&cur[bin], 1)] = (uint32_t)(base + k);
    }
}

__global__ void __launch_bounds__(128) proj_match_sorted_kernel(KpGrid G, ProjParams P, uint32_t idx_base, const int *__restrict__ n_valid,
                                                                const uint32_t *__restrict__ perm, const double *__restrict__ xw,
                                                                const uint8_t *__restrict__ mp_desc,
                                                                unsigned long long *__restrict__ best) {
    const int e = blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= *n_valid) return;
    const uint32_t i = perm[e];
    uint32_t a[8];
    load_desc(mp_desc + (size_t)i * 32, a);
    project_and_match(G, P, xw[3 * (size_t)i], xw[3 * (size_t)i + 1], xw[3 * (size_t)i + 2], a, idx_base + i, best);
}

// keys of `shards` map-point shards (shards x m) -> per keypoint the minimum (dist, -query) key, decoded
__global__ void projection_decode_kernel(int m, int shards, const unsigned long long *__restrict__ best,
                                         int32_t *__restrict__ to_query, int32_t *__restrict__ dist) {
    const int j = blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= m) return;
    unsigned long long k = best[j];
    for (int s = 1; s < shards; s++) k = min(k, best[(size_t)s * m + j]);
    const bool none = k == ~0ull;
    to_query[j] = none ? -1 : (int32_t)(0xFFFFFFFFu - (uint32_t)(k & 0xFFFFFFFFu));
    if (dist) dist[j] = none ? -1 : (int32_t)(k >> 32);
}

// ---------------------------------------------------------------------------------------------
// Brute-force top-2: thread = query (descriptor + its two best keys in registers), CTA streams a
// chunk of database rows through shared memory with broadcast reads.
// ---------------------------------------------------------------------------------------------
constexpr int kKnnThreads = 256;
constexpr int kKnnTile = 256;  // database rows per shared-memory tile

__global__ void __launch_bounds__(kKnnThreads) knn2_partial_kernel(const uint8_t *__restrict__ db, long long rows,
                                                                   long long idx_base, int chunk_rows,
                                                                   const uint8_t *__restrict__ queries, int q,
                                                                   unsigned long long *__restrict__ part) {
    __shared__ uint4 tile[kKnnTile * 2];
    const int tid = threadIdx.x, qi = blockIdx.y * kKnnThreads + tid;
    const long long c0 = (long long)blockIdx.x * chunk_rows, c1 = min(c0 + (long long)chunk_rows, rows);
    uint32_t a[8] = {0, 0, 0, 0, 0, 0, 0, 0};
    if (qi < q) load_desc(queries + (size_t)qi * 32, a);
    uint32_t k0 = kNoKey, k1 = kNoKey;  // dist << 22 | row within the chunk
    for (long long t0 = c0; t0 < c1; t0 += kKnnTile) {
        const int tn = (int)min((long long)kKnnTile, c1 - t0);
        __syncthreads();
        if (tid < tn) {
            const uint4 *src = (const uint4 *)(db + (size_t)(t0 + tid) * 32);
            tile[2 * tid] = __ldg(src);
            tile[2 * tid + 1] = __ldg(src + 1);
        }
        __syncthreads();
        const uint32_t rbase = (uint32_t)(t0 - c0);
        // four rows per step; a row only reaches the top-2 update when it beats the current second best, which after
        // the first few hundred rows is rare: one compare + branch per four rows instead of three min/max per row
        int r = 0;
        for (; r + 4 <= tn; r += 4) {
            uint32_t key[4];
#pragma unroll
            for (int j = 0; j < 4; j++) {
                const uint4 u = tile[2 * (r + j)], w = tile[2 * (r + j) + 1];
                key[j] = (uint32_t)hamming8_csa(a, u.x, u.y, u.z, u.w, w.x, w.y, w.z, w.w) << 22 | (rbase + r + j);
            }
            if (min(min(key[0], key[1]), min(key[2], key[3])) < k1) {
#pragma unroll
                for (int j = 0; j < 4; j++) top2_insert(k0, k1, key[j]);
            }
        }
        for (; r < tn; r++) {
            const uint4 u = tile[2 * r], w = tile[2 * r + 1];
            top2_insert(k0, k1, (uint32_t)hamming8_csa(a, u.x, u.y, u.z, u.w, w.x, w.y, w.z, w.w) << 22 | (rbase + r));
        }
    }
    if (qi < q) {
        unsigned long long *o = part + ((size_t)blockIdx.x * q + qi) * 2;
        const unsigned long long gb = (unsigned long long)(idx_base + c0);
        o[0] = k0 == kNoKey ? ~0ull : ((unsigned long long)(k0 >> 22) << 32 | (gb + (k0 & 0x3FFFFF)));
        o[1] = k1 == kNoKey ? ~0ull : ((unsigned long long)(k1 >> 22) << 32 | (gb + (k1 & 0x3FFFFF)));
    }
}

// Few queries (q <= 128): thread = database row.  A warp streams 64 rows per step with coalesced 128-bit loads
// (HBM-bound when q <= 2: 32 B per row against 26 instructions per row-query pair), every lane scores its
// two rows against each query (broadcast from shared memory) and the warp keeps the running top-2 of query
// g*32 + j in lane j.  A row only enters the reduction when it beats that query's current second best --
// after the first few thousand rows almost never -- so the steady state is XOR + POPC + one vote per pair.
constexpr int kRowsQMax = 128;
constexpr int kKnnTcMinQ = 64;  // from here on the tensor-core kernel wins on a large map (10 M rows: 0.91 ms vs 1.04 ms at 64 queries, 0.91 vs 3.0 at 129); it always works on groups of 512 queries

template <int QPL>  // queries per lane: q <= 32 * QPL
__global__ void __launch_bounds__(256) knn2_rows_kernel(const uint8_t *__restrict__ db, long long rows, long long idx_base,
                                                        int chunk_rows, const uint8_t *__restrict__ queries, int q,
                                                        unsigned long long *__restrict__ part) {
    __shared__ uint4 sq[kRowsQMax * 2];
    __shared__ uint32_t sk[8][kRowsQMax][2];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    for (int i = tid; i < q * 2; i += 256) sq[i] = __ldg((const uint4 *)queries + i);
    __syncthreads();
    const long long c0 = (long long)blockIdx.x * chunk_rows, c1 = min(c0 + (long long)chunk_rows, rows);
    uint32_t k0[QPL], k1[QPL];
#pragma unroll
    for (int g = 0; g < QPL; g++) k0[g] = k1[g] = kNoKey;
    // the rows of the next step are fetched before this step's distances are computed: two steps of loads in flight per warp
    uint32_t a[2][8], nx[2][8];
    bool valid[2], nvalid[2];
    auto fetch = [&](long long r, uint32_t (&dst)[2][8], bool (&ok)[2]) {
#pragma unroll
        for (int h = 0; h < 2; h++) {
            const long long row = r + h * 32 + lane;
            ok[h] = row < c1;
            if (ok[h]) load_desc(db + (size_t)row * 32, dst[h]);
        }
    };
    fetch(c0 + warp * 64, nx, nvalid);
    for (long long r0 = c0 + warp * 64; r0 < c1; r0 += 8 * 64) {
#pragma unroll
        for (int h = 0; h < 2; h++) {
            valid[h] = nvalid[h];
#pragma unroll
            for (int k = 0; k < 8; k++) a[h][k] = nx[h][k];
        }
        fetch(r0 + 8 * 64, nx, nvalid);
        const uint32_t rel = (uint32_t)(r0 - c0) + lane;
#pragma unroll
        for (int g = 0; g < QPL; g++) {
            const int nq = min(32, q - g * 32);
#pragma unroll 2
            for (int j = 0; j < nq; j++) {
                const uint4 u = sq[2 * (g * 32 + j)], w = sq[2 * (g * 32 + j) + 1];
                const uint32_t thr = __shfl_sync(0xffffffffu, k1[g], j);
                uint32_t key[2];
#pragma unroll
                for (int h = 0; h < 2; h++) {
                    const int d = hamming8_csa(a[h], u.x, u.y, u.z, u.w, w.x, w.y, w.z, w.w);
                    key[h] = valid[h] ? (uint32_t)d << 22 | (rel + 32 * h) : kNoKey;
                }
                if (__any_sync(0xffffffffu, min(key[0], key[1]) < thr)) {
                    // the warp's two smallest keys (keys are unique: they carry the row)
                    uint32_t lo = min(key[0], key[1]), hi = max(key[0], key[1]);
                    const uint32_t m1 = __reduce_min_sync(0xffffffffu, lo);
                    if (lo == m1) lo = hi, hi = kNoKey;
                    const uint32_t m2 = __reduce_min_sync(0xffffffffu, lo);
                    if (lane == j) {
                        top2_insert(k0[g], k1[g], m1);
                        top2_insert(k0[g], k1[g], m2);
                    }
                }
            }
        }
    }
#pragma unroll
    for (int g = 0; g < QPL; g++)
        if (g * 32 + lane < q) {
            sk[warp][g * 32 + lane][0] = k0[g];
            sk[warp][g * 32 + lane][1] = k1[g];
        }
    __syncthreads();
    if (tid < q) {
        uint32_t b0 = kNoKey, b1 = kNoKey;
#pragma unroll
        for (int w2 = 0; w2 < 8; w2++) {
            top2_insert(b0, b1, sk[w2][tid][0]);
            top2_insert(b0, b1, sk[w2][tid][1]);
        }
        unsigned long long *o = part + ((size_t)blockIdx.x * q + tid) * 2;
        const unsigned long long gb = (unsigned long long)(idx_base + c0);
        o[0] = b0 == kNoKey ? ~0ull : ((unsigned long long)(b0 >> 22) << 32 | (gb + (b0 & 0x3FFFFF)));
        o[1] = b1 == kNoKey ? ~0ull : ((unsigned long long)(b1 >> 22) << 32 | (gb + (b1 & 0x3FFFFF)));
    }
}

// lexicographic (dist, global index) top-2 over `parts` candidate pairs per query: one warp per query, lanes
// stride over the parts, butterfly merge of the per-lane pairs
__global__ void __launch_bounds__(128) knn2_merge_kernel(const unsigned long long *__restrict__ part, int parts, int q,
                                                         unsigned long long *__restrict__ keys_out, int32_t *__restrict__ quad_out) {
    const int qi = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
    if (qi >= q) return;
    unsigned long long k0 = ~0ull, k1 = ~0ull;
    for (int p = lane; p < parts; p += 32) {
        const ulonglong2 k = __ldg((const ulonglong2 *)(part + ((size_t)p * q + qi) * 2));
        k1 = min(k1, max(k0, k.x));
        k0 = min(k0, k.x);
        k1 = min(k1, max(k0, k.y));
        k0 = min(k0, k.y);
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        const unsigned long long o0 = __shfl_xor_sync(0xffffffffu, k0, o), o1 = __shfl_xor_sync(0xffffffffu, k1, o);
        k1 = min(min(k1, o1), max(k0, o0));
        k0 = min(k0, o0);
    }
    if (lane != 0) return;
    if (keys_out) {
        keys_out[(size_t)qi * 2] = k0;
        keys_out[(size_t)qi * 2 + 1] = k1;
    }
    if (quad_out) {
        quad_out[4 * qi + 0] = k0 == ~0ull ? -1 : (int32_t)(k0 & 0xFFFFFFFFu);
        quad_out[4 * qi + 1] = k0 == ~0ull ? 999999999 : (int32_t)(k0 >> 32);
        quad_out[4 * qi + 2] = k1 == ~0ull ? -1 : (int32_t)(k1 & 0xFFFFFFFFu);
        quad_out[4 * qi + 3] = k1 == ~0ull ? 999999999 : (int32_t)(k1 >> 32);
    }
}

// ---------------------------------------------------------------------------------------------
// Frame glue (SURVEY §8f rows 1, 3): what Frame::Frame does after extract() (src/frame.cpp:50-69) and
// StereoFrame::GetDepth (:391-409), on the device, for a frame whose keypoints / descriptors stay resident.
// ---------------------------------------------------------------------------------------------
// Camera::NormalizedUndistort, src/camera.cpp:95-109: 5 iterations of x += x_n - Distort(D, x); one thread per keypoint
__device__ __forceinline__ double2 normalized_undistort(const sfe_camera &cam, float px, float py) {
    const double nx = __ddiv_rn(__dsub_rn((double)px, cam.cx), cam.fx), ny = __ddiv_rn(__dsub_rn((double)py, cam.cy), cam.fy);
    double x = nx, y = ny;
#pragma unroll 1
    for (int it = 0; it < 5; it++) {
        const double r2 = __dadd_rn(__dmul_rn(x, x), __dmul_rn(y, y)), r4 = __dmul_rn(r2, r2);
        const double a1 = __dmul_rn(__dmul_rn(2., x), y);
        const double a2 = __dadd_rn(r2, __dmul_rn(__dmul_rn(2., x), x));
        const double a3 = __dadd_rn(r2, __dmul_rn(__dmul_rn(2., y), y));
        const double cdist = __dadd_rn(__dadd_rn(1., __dmul_rn(cam.d[0], r2)), __dmul_rn(cam.d[1], r4));
        const double xd = __dadd_rn(__dadd_rn(__dmul_rn(x, cdist), __dmul_rn(cam.d[2], a1)), __dmul_rn(cam.d[3], a2));
        const double yd = __dadd_rn(__dadd_rn(__dmul_rn(y, cdist), __dmul_rn(cam.d[2], a3)), __dmul_rn(cam.d[3], a1));
        x = __dadd_rn(x, __dsub_rn(nx, xd));
        y = __dadd_rn(y, __dsub_rn(ny, yd));
    }
    return make_double2(x, y);
}

__global__ void normalized_undistort_kernel(sfe_camera cam, const sfe_keypoint *__restrict__ kps, int n, double2 *__restrict__ out) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) out[i] = normalized_undistort(cam, kps[i].x, kps[i].y);
}

// StereoFrame::GetDepth for every left keypoint: depth = fx * baseline / dx, dx = the FLOAT difference of the x's
__global__ void stereo_depth_kernel(double fx, double baseline, const sfe_keypoint *__restrict__ kl, const double2 *__restrict__ nrm,
                                    int n, const sfe_keypoint *__restrict__ kr, const int32_t *__restrict__ sidx,
                                    double *__restrict__ xc, uint8_t *__restrict__ valid) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    double X = 0., Y = 0., Z = 0.;
    uint8_t ok = 0;
    const int j = sidx[i];
    if (j >= 0) {
        const double dx = (double)__fsub_rn(kl[i].x, kr[j].x);
        if (dx < 0.) {
            ok = 2;  // the reference throws: StereoMatch never lets this through
        } else {
            Z = __ddiv_rn(__dmul_rn(fx, baseline), dx);
            X = __dmul_rn(nrm[i].x, Z);
            Y = __dmul_rn(nrm[i].y, Z);
            ok = 1;
        }
    }
    xc[3 * i] = X; xc[3 * i + 1] = Y; xc[3 * i + 2] = Z;
    valid[i] = ok;
}

// ---------------------------------------------------------------------------------------------
// Sequence tracking over a resident stereo batch: what the reference does per frame between extract() and the pose
// optimiser -- Frame::Frame's spatial index (src/frame.cpp:59-68), StereoFrame::GetDepth of the previous frame's
// keypoints (:391-409) and ProjectionMatch of those points into the current frame (src/matcher.cpp:134-209) -- for
// all consecutive pairs of a batch at once, straight from the extractor's cap-strided device outputs.
// ---------------------------------------------------------------------------------------------
struct TrackArrays {
    int frames, cap, gw, gh;
    const sfe_keypoint *kl, *kr;
    const uint8_t *dl;
    const int32_t *nl, *sidx;
    int *cell_start;  // frames x (cells + 1)
    int *order;       // frames x cap
    double2 *sxy;     // frames x cap
    uint4 *sdesc;     // frames x 2 cap
    int *valid;       // frames x cap: the frame's keypoints that have a stereo correspondence (any order)
    int *n_valid;     // frames
};

__device__ __forceinline__ KpGrid track_grid(const TrackArrays &A, int f) {
    KpGrid G;
    G.gw = A.gw; G.gh = A.gh;
    G.m = min(A.nl[f], A.cap);
    G.cell_start = A.cell_start + (size_t)f * (A.gw * A.gh + 1);
    G.cell_fill = nullptr;
    G.order = A.order + (size_t)f * A.cap;
    G.sxy = A.sxy + (size_t)f * A.cap;
    G.sdesc = A.sdesc + (size_t)f * 2 * A.cap;
    return G;
}

// One CTA builds one frame's bucket grid: count and scan in shared memory (cells + 1 counters, then fill cursors)
__global__ void __launch_bounds__(256) track_grids_kernel(TrackArrays A) {
    extern __shared__ int tg_smem[];
    const int f = blockIdx.x, tid = threadIdx.x, cells = A.gw * A.gh;
    int *start = tg_smem, *fill = tg_smem + cells + 1;
    __shared__ int chunk_sum[256];
    __shared__ int nv;
    const KpGrid G = track_grid(A, f);
    if (tid == 0) nv = 0;
    const sfe_keypoint *kps = A.kl + (size_t)f * A.cap;
    for (int c = tid; c <= cells; c += 256) start[c] = 0;
    __syncthreads();
    for (int j = tid; j < G.m; j += 256) atomicAdd(&start[grid_cell(G, kps[j].x, kps[j].y) + 1], 1);
    __syncthreads();
    // inclusive scan of start[0 .. cells]: a contiguous chunk per thread, then the chunk totals
    const int per = (cells + 1 + 255) / 256, c0 = min(tid * per, cells + 1), c1 = min(c0 + per, cells + 1);
    int acc = 0;
    for (int c = c0; c < c1; c++) acc += start[c];
    chunk_sum[tid] = acc;
    __syncthreads();
    if (tid < 32) {  // exclusive scan of the 256 chunk totals by one warp, 8 per lane
        int v[8], tot = 0;
#pragma unroll
        for (int k = 0; k < 8; k++) {
            v[k] = chunk_sum[tid * 8 + k];
            tot += v[k];
        }
        int inc = tot;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const int x = __shfl_up_sync(0xffffffffu, inc, o);
            if (tid >= o) inc += x;
        }
        int run = inc - tot;
#pragma unroll
        for (int k = 0; k < 8; k++) {
            chunk_sum[tid * 8 + k] = run;
            run += v[k];
        }
    }
    __syncthreads();
    acc = chunk_sum[tid];
    for (int c = c0; c < c1; c++) {
        acc += start[c];
        start[c] = acc;
        G.cell_start[c] = acc;
    }
    for (int c = tid; c < cells; c += 256) fill[c] = 0;
    __syncthreads();
    const uint8_t *desc = A.dl + (size_t)f * A.cap * 32;
    for (int j = tid; j < G.m; j += 256) {
        const float x = kps[j].x, y = kps[j].y;
        const int c = grid_cell(G, x, y), t = start[c] + atomicAdd(&fill[c], 1);
        G.order[t] = j;
        G.sxy[t] = make_double2((double)x, (double)y);
        const uint4 *d = (const uint4 *)(desc + (size_t)j * 32);
        G.sdesc[2 * t] = __ldg(d);
        G.sdesc[2 * t + 1] = __ldg(d + 1);
    }
    // the keypoints that will be projected into the next frame: compacted so that the matcher's warps are full, and in
    // the grid's cell order so that the lanes of a warp project into the same neighbourhood (the motion between
    // consecutive frames is small) and walk the same cells
    __syncthreads();  // order[] of this frame is complete
    const int32_t *sidx = A.sidx + (size_t)f * A.cap;
    int *valid = A.valid + (size_t)f * A.cap;
    __shared__ int wcount[8];
    for (int t0 = 0; t0 < G.m; t0 += 256) {
        const int t = t0 + tid, j = t < G.m ? G.order[t] : -1;
        const bool ok = j >= 0 && sidx[j] >= 0;
        const uint32_t b = __ballot_sync(0xffffffffu, ok);
        if ((tid & 31) == 0) wcount[tid >> 5] = __popc(b);
        __syncthreads();
        int base = nv;
        for (int w2 = 0; w2 < (tid >> 5); w2++) base += wcount[w2];
        if (ok) valid[base + __popc(b & ((1u << (tid & 31)) - 1))] = j;
        __syncthreads();
        if (tid == 0) {
            int tot = 0;
            for (int w2 = 0; w2 < 8; w2++) tot += wcount[w2];
            nv += tot;
        }
        __syncthreads();
    }
    if (tid == 0) A.n_valid[f] = nv;
}

// thread = keypoint i of frame f - 1 (f = blockIdx.y + 1): GetDepth, then ProjectionMatch into frame f
__global__ void __launch_bounds__(128) track_match_kernel(TrackArrays A, ProjParams P, double baseline,
                                                          unsigned long long *__restrict__ best) {
    const int f = blockIdx.y + 1, prev = f - 1, e = blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= A.n_valid[prev]) return;  // keypoints without a stereo correspondence have no depth, hence no map point
    const int i = A.valid[(size_t)prev * A.cap + e], j = A.sidx[(size_t)prev * A.cap + i];
    const sfe_keypoint kp = A.kl[(size_t)prev * A.cap + i];
    const double dx = (double)__fsub_rn(kp.x, A.kr[(size_t)prev * A.cap + j].x);  // :398, float difference
    if (dx < 0.) return;  // the reference throws (:399-402); StereoMatch never lets this through
    const double Z = __ddiv_rn(__dmul_rn(P.cam.fx, baseline), dx);
    const double2 nrm = normalized_undistort(P.cam, kp.x, kp.y);
    uint32_t a[8];
    load_desc(A.dl + ((size_t)prev * A.cap + i) * 32, a);
    const KpGrid G = track_grid(A, f);
    project_and_match(G, P, __dmul_rn(nrm.x, Z), __dmul_rn(nrm.y, Z), Z, a, (uint32_t)i, best + (size_t)f * A.cap);
}

// ReprojectionFilter::GetOutlier's per-keypoint quantity (src/posetracker.cpp:106-137): the distance between keypoint i
// and the projection of its map point under Tcw; +inf when the point is behind the camera (an outlier whatever the
// threshold), -1 when the keypoint has no map point
__global__ void reprojection_error_kernel(sfe_camera cam, ProjParams P, const sfe_keypoint *__restrict__ kps, int n,
                                          const double *__restrict__ xw, const uint8_t *__restrict__ has_mp,
                                          double *__restrict__ err) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    double e = -1.;
    if (has_mp[i]) {
        double u, v;
        if (!project_uv(P.T, cam, xw[3 * (size_t)i], xw[3 * (size_t)i + 1], xw[3 * (size_t)i + 2], u, v)) {
            e = __longlong_as_double(0x7FF0000000000000ll);
        } else {
            const double dx = __dsub_rn(u, (double)kps[i].x), dy = __dsub_rn(v, (double)kps[i].y);
            e = __dsqrt_rn(__dadd_rn(__dmul_rn(dx, dx), __dmul_rn(dy, dy)));  // Eigen's norm() of a 2-vector
        }
    }
    err[i] = e;
}

// Frame::SearchRadius / SearchNeareast over the bucket grid; one thread per query point.
__global__ void search_radius_kernel(KpGrid G, const sfe_keypoint *__restrict__ kps, const double2 *__restrict__ uv, int q,
                                     double radius, int32_t *__restrict__ idx, int cap, int32_t *__restrict__ counts) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= q) return;
    const double u = uv[i].x, v = uv[i].y, r2max = __dmul_rn(radius, radius);
    int32_t *out = idx + (size_t)i * cap;
    int n = 0;
    if (u == u && v == v) {
        const int cx0 = min(max((int)floor(u - radius) >> kGridShift, 0), G.gw - 1), cx1 = min(max((int)floor(u + radius) >> kGridShift, 0), G.gw - 1);
        const int cy0 = min(max((int)floor(v - radius) >> kGridShift, 0), G.gh - 1), cy1 = min(max((int)floor(v + radius) >> kGridShift, 0), G.gh - 1);
        for (int cy = cy0; cy <= cy1; cy++) {
            const int s = G.cell_start[cy * G.gw + cx0], e = G.cell_start[cy * G.gw + cx1 + 1];
            for (int t = s; t < e; t++) {
                const int j = G.order[t];
                const double ddx = u - (double)kps[j].x, ddy = v - (double)kps[j].y;
                if (!(__dadd_rn(__dmul_rn(ddx, ddx), __dmul_rn(ddy, ddy)) < r2max)) continue;
                // keep the row sorted by index (canonical order): insertion from the back; a full row keeps its cap
                // smallest indices whatever order the cells are visited in
                if (n < cap || j < out[cap - 1]) {
                    int p = min(n, cap - 1);
                    while (p > 0 && out[p - 1] > j) { out[p] = out[p - 1]; p--; }
                    out[p] = j;
                }
                n++;
            }
        }
    }
    counts[i] = n;
}

__global__ void search_nearest_kernel(KpGrid G, const sfe_keypoint *__restrict__ kps, const double2 *__restrict__ uv, int q,
                                      int32_t *__restrict__ idx, double *__restrict__ dist2) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= q) return;
    // exact nearest neighbour = minimum of (d^2, index) over all keypoints (T6); the frame holds ~2000 of them
    const double u = uv[i].x, v = uv[i].y;
    int best = -1;
    double bd = 0.;
    for (int j = 0; j < G.m; j++) {
        const double ddx = u - (double)kps[j].x, ddy = v - (double)kps[j].y;
        const double d2 = __dadd_rn(__dmul_rn(ddx, ddx), __dmul_rn(ddy, ddy));
        if (best < 0 || d2 < bd) { best = j; bd = d2; }
    }
    idx[i] = best;
    dist2[i] = bd;
}

// ---------------------------------------------------------------------------------------------
// BoW transform (SURVEY §8f row 2): the tree descent of DBoW2's TemplatedVocabulary::transform
// (thirdparty/DBoW2/DBoW2/TemplatedVocabulary.h:1218-1259).  One warp per feature: lane c scores child c of the
// current node (256-bit Hamming, FORB.cpp:81-101), the warp takes the minimum of (distance, child rank) -- the
// reference's strict < keeps the first child on ties -- and steps down until it reaches a node without children.
// ---------------------------------------------------------------------------------------------
struct VocabDev {
    const int *child_start;   // n_nodes + 1
    const int *child_list;    // children in id order
    const uint8_t *desc;      // n_nodes x 32
    const double *weight;
    const int *word_id;
    int n_nodes, L;
};

__global__ void __launch_bounds__(256) vocab_transform_kernel(VocabDev V, const uint8_t *__restrict__ feat, int n, int levelsup,
                                                              int32_t *__restrict__ word_id, double *__restrict__ weight,
                                                              int32_t *__restrict__ node_id) {
    const int f = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
    if (f >= n) return;
    uint32_t a[8];
    load_desc(feat + (size_t)f * 32, a);
    const int nid_level = V.L - levelsup;
    int nid = 0, cur = 0, level = 0;
    for (;;) {
        const int s = V.child_start[cur], nc = V.child_start[cur + 1] - s;
        if (nc == 0) break;  // isLeaf()
        ++level;
        uint32_t best = kNoKey;
        for (int c0 = 0; c0 < nc; c0 += 32) {  // k <= 20 in DBoW2's text format, so one round
            uint32_t key = kNoKey;
            if (c0 + lane < nc) {
                uint32_t b[8];
                load_desc(V.desc + (size_t)V.child_list[s + c0 + lane] * 32, b);
                key = (uint32_t)hamming8(a, b) << 20 | (uint32_t)(c0 + lane);
            }
            best = min(best, __reduce_min_sync(0xffffffffu, key));
        }
        cur = V.child_list[s + (best & 0xFFFFF)];
        if (level == nid_level) nid = cur;
    }
    if (lane == 0) {
        word_id[f] = V.word_id[cur];
        weight[f] = V.weight[cur];
        node_id[f] = nid;
    }
}

int launch_track_frames(cudaStream_t st, int device, TrackScratch &T, int frames, int cap, const sfe_keypoint *kl, const uint8_t *dl,
                        const int32_t *nl, const sfe_keypoint *kr, const int32_t *sidx, const sfe_track_params &tp,
                        int32_t *track_idx, int32_t *track_dist) {
    TrackArrays A{};
    A.frames = frames; A.cap = cap;
    A.gw = (std::max(tp.cam.width, 1) >> kGridShift) + 1;
    A.gh = (std::max(tp.cam.height, 1) >> kGridShift) + 1;
    const int cells = A.gw * A.gh;
    const size_t smem = sizeof(int) * (2 * (size_t)cells + 1), fc = (size_t)frames * cap;
    SFE_REQUIRE(cap < 65536, SFE_ERR_UNSUPPORTED, "more than 65535 keypoints per frame");
    SFE_REQUIRE(smem <= 200 * 1024, SFE_ERR_UNSUPPORTED, "camera image too large for the per-frame bucket grid");
    SFE_CUDA(T.cell_start.ensure((size_t)frames * (cells + 1)));
    SFE_CUDA(T.order.ensure(fc)); SFE_CUDA(T.sxy.ensure(fc)); SFE_CUDA(T.sdesc.ensure(2 * fc)); SFE_CUDA(T.best.ensure(fc));
    SFE_CUDA(T.valid.ensure(fc + frames));
    A.kl = kl; A.kr = kr; A.dl = dl; A.nl = nl; A.sidx = sidx;
    A.cell_start = T.cell_start.p; A.order = T.order.p; A.sxy = T.sxy.p; A.sdesc = T.sdesc.p;
    A.valid = T.valid.p; A.n_valid = T.valid.p + fc;
    if (smem > 48 * 1024) {  // per-function opt-in limit: only ever raise it
        static std::mutex mu;
        static size_t granted[64] = {};
        std::lock_guard<std::mutex> lock(mu);
        if (smem > granted[device & 63]) {
            SFE_CUDA(cudaFuncSetAttribute(track_grids_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
            granted[device & 63] = smem;
        }
    }
    SFE_CUDA(cudaMemsetAsync(T.best.p, 0xFF, sizeof(unsigned long long) * fc, st));
    track_grids_kernel<<<frames, 256, smem, st>>>(A);
    if (frames > 1) {
        ProjParams P;
        P.T = tp.use_se3 ? pose_from_se3(&tp.se3) : pose_from_rt(tp.rt);
        P.cam = tp.cam;
        P.radius = tp.radius;
        P.ratio = tp.best12_threshold;
        track_match_kernel<<<dim3(div_up(cap, 128), frames - 1), 128, 0, st>>>(A, P, tp.baseline, T.best.p);
    }
    projection_decode_kernel<<<div_up((int)fc, 256), 256, 0, st>>>((int)fc, 1, T.best.p, track_idx, track_dist);
    SFE_CUDA(cudaGetLastError());
    return SFE_OK;
}


// ---------------------------------------------------------------------------------------------
// Multi-GPU exchange (SURVEY §8e): every rank's kernel stores its contribution straight into every peer's inbox over
// NVLink (peer-mapped device memory: cudaIpc handles between processes, peer access inside one process), then raises a
// per-(parity, sender) flag there; the consumer kernel of each rank waits on its own flags and merges.  No NCCL, no host
// round trip between the local kernels, the exchange and the merge.
//   inbox layout (device memory of the owning rank):
//     [2 parities][world][slot_bytes] payload | u32 flags[2][kMaxWorld] | u32 push_counter | u32 status
//   flags[p][r] = sequence number of the last collective whose payload rank r finished writing into parity p.
//   Two parities suffice: a rank can be at most one collective ahead of a peer, because its merge of collective e+1
//   waits for the peer's push e+1, which the peer's stream orders behind its own merge of collective e.
// ---------------------------------------------------------------------------------------------
constexpr int kMaxWorld = 16;
constexpr size_t kCommSlotBytes = 512 * 1024;  // per sender and parity: 65535 keypoints x 8 B, or 32768 queries x 2 keys

struct CommView {
    uint8_t *base[kMaxWorld];  // inbox of every rank as mapped here; base[rank] is local memory
    int rank, world;
    uint32_t epoch;            // sequence number of this collective (>= 1), the same on every rank
};
__device__ __forceinline__ uint8_t *comm_slot(const CommView &C, int owner, int from) {
    return C.base[owner] + ((size_t)(C.epoch & 1) * C.world + from) * kCommSlotBytes;
}
__device__ __forceinline__ uint32_t *comm_flags(const CommView &C, int owner) {
    return (uint32_t *)(C.base[owner] + 2 * (size_t)C.world * kCommSlotBytes) + (C.epoch & 1) * kMaxWorld;
}
__device__ __forceinline__ uint32_t *comm_counter(const CommView &C) { return (uint32_t *)(C.base[C.rank] + 2 * (size_t)C.world * kCommSlotBytes) + 2 * kMaxWorld; }
__device__ __forceinline__ uint32_t *comm_status(const CommView &C) { return comm_counter(C) + 1; }

// end of a pushing kernel: the last CTA to get here publishes the flags.  Every CTA fences its remote stores first.
__device__ __forceinline__ void comm_publish(const CommView &C) {
    __threadfence_system();
    __syncthreads();
    if (threadIdx.x == 0) {
        const unsigned total = gridDim.x * gridDim.y * gridDim.z;
        const unsigned ticket = atomicAdd(comm_counter(C), 1u);
        if (ticket == total - 1) {
            *comm_counter(C) = 0;
            __threadfence_system();
            for (int p = 0; p < C.world; p++) {
                uint32_t *f = comm_flags(C, p) + C.rank;
                asm volatile("st.release.sys.global.u32 [%0], %1;" ::"l"(f), "r"(C.epoch) : "memory");
            }
        }
    }
}
// start of a consuming kernel: wait until every rank's payload of this collective has landed in the local inbox.
// Bounded: a peer that never arrives sets the status word instead of hanging the GPU.
__device__ __forceinline__ void comm_wait_all(const CommView &C) {
    if (threadIdx.x < C.world) {
        const uint32_t *f = comm_flags(C, C.rank) + threadIdx.x;
        unsigned long long t0 = 0;
        asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t0));
        for (;;) {
            uint32_t v;
            asm volatile("ld.acquire.sys.global.u32 %0, [%1];" : "=r"(v) : "l"(f) : "memory");
            if (v == C.epoch) break;
            __nanosleep(200);
            unsigned long long t1;
            asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t1));
            if (t1 - t0 > 5000000000ull) {  // 5 s
                atomicExch(comm_status(C), 1u + threadIdx.x);
                break;
            }
        }
    }
    __syncthreads();
}

// n16 16-byte units of the local slot (already holding this rank's payload) -> every peer's slot for this rank
__global__ void __launch_bounds__(256) comm_push_kernel(CommView C, int n16) {
    const ulonglong2 *src = (const ulonglong2 *)comm_slot(C, C.rank, C.rank);
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n16; i += gridDim.x * blockDim.x) {
        const ulonglong2 v = src[i];
        for (int p = 0; p < C.world; p++)
            if (p != C.rank) ((ulonglong2 *)comm_slot(C, p, C.rank))[i] = v;
    }
    comm_publish(C);
}

// kNN: merge of this rank's chunk partials (as knn2_merge_kernel), the query's two keys stored into every rank's inbox by
// lanes 0 .. world-1 of the warp that owns the query -- the push is the merge kernel's epilogue
__global__ void __launch_bounds__(128) knn2_merge_push_kernel(CommView C, const unsigned long long *__restrict__ part, int parts, int q) {
    const int qi = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
    if (qi < q) {
        unsigned long long k0 = ~0ull, k1 = ~0ull;
        for (int p = lane; p < parts; p += 32) {
            const ulonglong2 k = __ldg((const ulonglong2 *)(part + ((size_t)p * q + qi) * 2));
            k1 = min(k1, max(k0, k.x));
            k0 = min(k0, k.x);
            k1 = min(k1, max(k0, k.y));
            k0 = min(k0, k.y);
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            const unsigned long long o0 = __shfl_xor_sync(0xffffffffu, k0, o), o1 = __shfl_xor_sync(0xffffffffu, k1, o);
            k1 = min(min(k1, o1), max(k0, o0));
            k0 = min(k0, o0);
        }
        if (lane < C.world) ((ulonglong2 *)comm_slot(C, lane, C.rank))[qi] = make_ulonglong2(k0, k1);
    }
    comm_publish(C);
}

// kNN: wait for every shard's keys, then lexicographic top-2 of the 2 * world candidates per query, decoded
__global__ void __launch_bounds__(128) knn2_gather_merge_kernel(CommView C, int q, int32_t *__restrict__ quad_out) {
    comm_wait_all(C);
    const int qi = blockIdx.x * blockDim.x + threadIdx.x;
    if (qi >= q) return;
    unsigned long long k0 = ~0ull, k1 = ~0ull;
    for (int r = 0; r < C.world; r++) {
        const ulonglong2 k = ((const ulonglong2 *)comm_slot(C, C.rank, r))[qi];
        k1 = min(k1, max(k0, k.x));
        k0 = min(k0, k.x);
        k1 = min(k1, max(k0, k.y));
        k0 = min(k0, k.y);
    }
    quad_out[4 * qi + 0] = k0 == ~0ull ? -1 : (int32_t)(k0 & 0xFFFFFFFFu);
    quad_out[4 * qi + 1] = k0 == ~0ull ? 999999999 : (int32_t)(k0 >> 32);
    quad_out[4 * qi + 2] = k1 == ~0ull ? -1 : (int32_t)(k1 & 0xFFFFFFFFu);
    quad_out[4 * qi + 3] = k1 == ~0ull ? 999999999 : (int32_t)(k1 >> 32);
}

// ProjectionMatch: wait for every shard's per-keypoint keys, minimum = "smaller distance, later query wins" (:197-204)
__global__ void __launch_bounds__(256) projection_gather_decode_kernel(CommView C, int m, int32_t *__restrict__ to_query,
                                                                       int32_t *__restrict__ dist) {
    comm_wait_all(C);
    const int j = blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= m) return;
    unsigned long long k = ~0ull;
    for (int r = 0; r < C.world; r++) k = min(k, ((const unsigned long long *)comm_slot(C, C.rank, r))[j]);
    const bool none = k == ~0ull;
    to_query[j] = none ? -1 : (int32_t)(0xFFFFFFFFu - (uint32_t)(k & 0xFFFFFFFFu));
    if (dist) dist[j] = none ? -1 : (int32_t)(k >> 32);
}

}  // namespace sfe

using namespace sfe;

struct sfe_matcher {
    int device = 0;
    cudaStream_t stream = nullptr;
    int sm_count = 148;
    int64_t launches = 0;
    bool async_dev = false;  // _dev entry points return after enqueueing (sfe_matcher_wait)
    bool knn_tc = true;      // SFE_KNN_TC=0: brute-force top-2 with many queries stays on the XOR / POPC kernel
    int knn_tc_min_q = kKnnTcMinQ;  // SFE_KNN_TC_MINQ: query count from which the tensor-core kernel is used
    size_t knn_tiles_max_bytes = (size_t)16 << 30;  // SFE_KNN_TILES_MAX_GB: largest unpacked copy of a map (0: never unpack)
    DevBuf<sfe_keypoint> d_kl, d_kr;
    DevBuf<uint8_t> d_dl, d_dr, d_skip;
    DevBuf<int32_t> d_n, d_idx, d_dist;
    DevBuf<double> d_xw;
    DevBuf<int> d_grid;
    DevBuf<unsigned long long> d_best, d_part, d_keys;
    DevBuf<int32_t> d_quad;
    DevBuf<uint16_t> d_proj_bins;  // sorted ProjectionMatch: bin per map point,
    DevBuf<int> d_proj_hist;       // per-chunk bin histograms + bin totals,
    DevBuf<uint32_t> d_proj_perm;  // map points in bin order
    DevBuf<int64_t> d_bow_off;     // BoW database queries: CSR of the query batch,
    DevBuf<int32_t> d_bow_ids, d_bow_e, d_bow_n;
    DevBuf<double> d_bow_val, d_bow_raw, d_bow_dense, d_bow_s;  // raw L1 sums, dense scores, results
    DevBuf<uint8_t> d_bow_hit;     // 1 where a query and an entry share a word
    DevBuf<unsigned long long> d_bow_chk;  // device vectors: nnz, rule broken, longest vector / assembly status
    DevBuf<int32_t> d_bowa_cnt, d_bowa_ids;  // BowVector assembly: words per set, vectors at the input's row stride,
    DevBuf<double> d_bowa_div, d_bowa_val;   // the divisor of each set's values
};

struct sfe_db {
    int device = 0;
    uint8_t *rows_dev = nullptr;
    int64_t rows = 0, idx_base = 0;
    // the rows as ready-made int8 operand tiles of the tensor-core kernel (8 x the packed size), built at the first
    // many-query search when the policy (knn_tiles_max_bytes) allows; tiles_tried: do not try again.  Every matcher of the
    // device may search the database, from any thread: tiles_mu guards the build, which runs on the stream of the matcher
    // that comes first, and tiles_ready (recorded behind the unpack) is what every search that reads the tiles waits for.
    mutable std::mutex tiles_mu;
    mutable uint8_t *tiles_dev = nullptr;
    mutable bool tiles_tried = false;
    mutable cudaEvent_t tiles_ready = nullptr;
};

// keys_out != nullptr: leave the per-keypoint (dist << 32 | ~global query) keys there (one shard's contribution to a
// sharded match) instead of decoding them
struct sfe_vocab {
    int device = 0, n_nodes = 0, L = 0, n_words = 0;
    DevBuf<int> child_start, child_list, word_id;
    DevBuf<uint8_t> desc;
    DevBuf<double> weight;
};

struct sfe_frame {
    int device = 0;
    int n = 0;
    sfe_camera cam{};
    KpGrid grid{};
    DevBuf<sfe_keypoint> kps;
    DevBuf<uint8_t> desc;
    DevBuf<double2> nrm;
    DevBuf<int> grid_mem;
};

// bucket grid over m_kps keypoints (replaces the per-frame FLANN kd-tree, src/frame.cpp:59-68)
static int build_grid(sfe_matcher *m, DevBuf<int> &mem, KpGrid &G, const sfe_camera *cam, const sfe_keypoint *kps,
                      const uint8_t *kp_desc, int m_kps) {
    cudaStream_t st = m->stream;
    G.gw = (std::max(cam->width, 1) >> kGridShift) + 1;
    G.gh = (std::max(cam->height, 1) >> kGridShift) + 1;
    G.m = m_kps;
    const int cells = G.gw * G.gh;
    const size_t ints = ((size_t)2 * cells + 1 + std::max(m_kps, 1) + 3) & ~(size_t)3;  // what follows is 16-byte aligned
    SFE_CUDA(mem.ensure(ints + (size_t)std::max(m_kps, 1) * (4 + 8)));
    G.cell_start = mem.p;
    G.cell_fill = mem.p + cells + 1;
    G.order = mem.p + 2 * cells + 1;
    G.sxy = (double2 *)(mem.p + ints);
    G.sdesc = (uint4 *)(mem.p + ints + (size_t)std::max(m_kps, 1) * 4);
    SFE_CUDA(cudaMemsetAsync(G.cell_start, 0, sizeof(int) * (cells + 1), st));
    if (m_kps > 0) grid_count_kernel<<<div_up(m_kps, 256), 256, 0, st>>>(G, kps);
    grid_scan_kernel<<<1, 256, 0, st>>>(G);
    if (m_kps > 0) grid_fill_kernel<<<div_up(m_kps, 256), 256, 0, st>>>(G, kps, kp_desc);
    m->launches += 3;
    return SFE_OK;
}

static int projection_impl(sfe_matcher *m, const double *xw, const uint8_t *mp_desc, const uint8_t *skip, int n,
                           const Pose &T, const sfe_camera *cam, const sfe_keypoint *kps, const uint8_t *kp_desc,
                           int m_kps, double radius, double ratio, int32_t *to_query, int32_t *dist, uint32_t idx_base = 0,
                           unsigned long long *keys_out = nullptr, const KpGrid *prebuilt = nullptr) {
    cudaStream_t st = m->stream;
    if (m_kps == 0) return SFE_OK;
    KpGrid G;
    if (prebuilt) {
        G = *prebuilt;  // a resident frame brings its own index
    } else {
        int rc = build_grid(m, m->d_grid, G, cam, kps, kp_desc, m_kps);
        if (rc != SFE_OK) return rc;
    }
    SFE_CUDA(m->d_best.ensure(m_kps));
    unsigned long long *best = keys_out ? keys_out : m->d_best.p;
    SFE_CUDA(cudaMemsetAsync(best, 0xFF, sizeof(unsigned long long) * m_kps, st));
    if (n > 0) {
        ProjParams P;
        P.T = T;
        P.cam = *cam;
        P.radius = radius;
        P.ratio = ratio;
        if (n < kProjSortMin) {
            projection_match_kernel<<<div_up(n, 128), 128, 0, st>>>(G, P, n, idx_base, xw, mp_desc, skip, best);
            m->launches++;
        } else {
            const int chunks = div_up(n, kProjChunk);
            SFE_CUDA(m->d_proj_bins.ensure(n));
            SFE_CUDA(m->d_proj_hist.ensure((size_t)chunks * kProjBins + kProjBins + 1));
            SFE_CUDA(m->d_proj_perm.ensure(n));
            int *hist = m->d_proj_hist.p, *tot = hist + (size_t)chunks * kProjBins;
            proj_bin_kernel<<<chunks, 256, 0, st>>>(G.gw, G.gh, P, n, xw, skip, m->d_proj_bins.p, hist);
            proj_offsets_kernel<<<kProjBins / 8, 256, 0, st>>>(chunks, hist, tot);
            proj_scan_kernel<<<1, kProjBins, 0, st>>>(tot);
            proj_scatter_kernel<<<chunks, 256, 0, st>>>(n, m->d_proj_bins.p, hist, tot, m->d_proj_perm.p);
            proj_match_sorted_kernel<<<div_up(n, 128), 128, 0, st>>>(G, P, idx_base, tot + kProjBins, m->d_proj_perm.p, xw, mp_desc, best);
            m->launches += 5;
        }
    }
    if (!keys_out) {
        projection_decode_kernel<<<div_up(m_kps, 256), 256, 0, st>>>(m_kps, 1, best, to_query, dist);
        m->launches++;
    }
    SFE_CUDA(cudaGetLastError());
    return SFE_OK;
}

namespace sfe {
cudaError_t launch_knn2_tc(cudaStream_t st, int sm_count, const uint8_t *db, const uint8_t *tiles, long long rows, long long idx_base,
                           int chunk_rows, int chunks, const uint8_t *queries, int q, unsigned long long *part);
cudaError_t launch_knn2_unpack_tiles(cudaStream_t st, const uint8_t *db, long long rows, uint8_t *tiles);
size_t knn2_tc_tiles_bytes(long long rows);
int knn2_tc_group_queries();
}

static int knn_partial(sfe_matcher *m, const sfe_db *db, const uint8_t *q_dev, int q, unsigned long long *keys_dev,
                       int32_t *quad_dev, const CommView *push = nullptr) {
    cudaStream_t st = m->stream;
    // Below 256 queries the group of 512 is mostly padding: worth it only when the map is large enough to hide the set-up.
    if (m->knn_tc && q >= m->knn_tc_min_q && db->rows >= 1 && (q >= 256 || db->rows >= 65536)) {
        // many queries: the pair distances are an int8 GEMM on the tensor cores (sfe_knn_tc.cu), one (512-query group, chunk)
        // item per SM; the chunk partials are merged as usual
        const int groups = div_up(q, knn2_tc_group_queries());
        int chunks = std::max(1, m->sm_count / groups);
        int64_t chunk_rows = std::max<int64_t>((db->rows + chunks - 1) / chunks, 1);
        chunk_rows = (chunk_rows + 255) / 256 * 256;
        SFE_REQUIRE(chunk_rows <= (1 << 22), SFE_ERR_UNSUPPORTED, "database shard larger than 2^22 rows per chunk");
        chunks = (int)std::max<int64_t>((db->rows + chunk_rows - 1) / chunk_rows, 1);
        SFE_CUDA(m->d_part.ensure((size_t)chunks * q * 2));
        // A map that is searched with many queries keeps its rows unpacked in HBM (256 B per row instead of 32): the kernel's
        // producers then move tiles with bulk copies instead of unpacking 10 M rows once per query group.  Built on first use,
        // when it fits the budget (SFE_KNN_TILES_MAX_GB, default 16 GB and a quarter of the free memory).
        const uint8_t *tiles = nullptr;
        {
            std::lock_guard<std::mutex> lock(db->tiles_mu);
            if (!db->tiles_dev && !db->tiles_tried && q >= 256 && db->rows >= 65536) {
                db->tiles_tried = true;
                const size_t need = knn2_tc_tiles_bytes(db->rows);
                size_t free_b = 0, total_b = 0;
                uint8_t *t = nullptr;
                if (cudaMemGetInfo(&free_b, &total_b) == cudaSuccess && need <= m->knn_tiles_max_bytes && need <= free_b / 4) {
                    if (cudaMalloc((void **)&t, need) != cudaSuccess) {
                        cudaGetLastError();
                        t = nullptr;
                    }
                }
                if (t) {  // published only once the unpack and the event behind it are enqueued
                    cudaError_t e = db->tiles_ready ? cudaSuccess : cudaEventCreateWithFlags(&db->tiles_ready, cudaEventDisableTiming);
                    if (e == cudaSuccess) e = launch_knn2_unpack_tiles(st, db->rows_dev, db->rows, t);
                    if (e == cudaSuccess) e = cudaEventRecord(db->tiles_ready, st);
                    if (e != cudaSuccess) {
                        cudaFree(t);
                        set_error("knn2 tile build: %s", cudaGetErrorString(e));
                        return SFE_ERR_CUDA;
                    }
                    db->tiles_dev = t;
                    m->launches++;
                }
            }
            if (db->tiles_dev) {
                SFE_CUDA(cudaStreamWaitEvent(st, db->tiles_ready, 0));  // the unpack may run on another matcher's stream
                tiles = db->tiles_dev;
            }
        }
        SFE_CUDA(launch_knn2_tc(st, m->sm_count, db->rows_dev, tiles, db->rows, db->idx_base, (int)chunk_rows, chunks, q_dev, q,
                                m->d_part.p));
        if (push)
            knn2_merge_push_kernel<<<div_up(q, 4), 128, 0, st>>>(*push, m->d_part.p, chunks, q);
        else
            knn2_merge_kernel<<<div_up(q, 4), 128, 0, st>>>(m->d_part.p, chunks, q, keys_dev, quad_dev);
        m->launches += 2;
        SFE_CUDA(cudaGetLastError());
        return SFE_OK;
    }
    const bool by_rows = q <= kRowsQMax;  // thread = row (streaming) for few queries, thread = query otherwise
    const int qgroups = by_rows ? 1 : div_up(q, kKnnThreads);
    int chunks = std::max(1, (8 * m->sm_count) / qgroups);  // 8 CTAs of 256 threads per SM: the XOR-CSA-POPC chain needs the warps to hide its latency
    int64_t chunk_rows = std::max<int64_t>((db->rows + chunks - 1) / chunks, 1);
    const int64_t grain = by_rows ? 512 : kKnnTile;  // the streaming kernel walks 8 warps x 64 rows per step, the other one tiles of 256
    chunk_rows = (chunk_rows + grain - 1) / grain * grain;
    SFE_REQUIRE(chunk_rows <= (1 << 22), SFE_ERR_UNSUPPORTED, "database shard larger than 2^22 rows per chunk");
    chunks = (int)std::max<int64_t>((db->rows + chunk_rows - 1) / chunk_rows, 1);
    SFE_CUDA(m->d_part.ensure((size_t)chunks * q * 2));
    if (by_rows) {
        const int qpl = div_up(q, 32);
        if (qpl == 1)
            knn2_rows_kernel<1><<<chunks, 256, 0, st>>>(db->rows_dev, db->rows, db->idx_base, (int)chunk_rows, q_dev, q, m->d_part.p);
        else if (qpl == 2)
            knn2_rows_kernel<2><<<chunks, 256, 0, st>>>(db->rows_dev, db->rows, db->idx_base, (int)chunk_rows, q_dev, q, m->d_part.p);
        else
            knn2_rows_kernel<4><<<chunks, 256, 0, st>>>(db->rows_dev, db->rows, db->idx_base, (int)chunk_rows, q_dev, q, m->d_part.p);
    } else {
        knn2_partial_kernel<<<dim3(chunks, qgroups), kKnnThreads, 0, st>>>(db->rows_dev, db->rows, db->idx_base, (int)chunk_rows,
                                                                          q_dev, q, m->d_part.p);
    }
    if (push)  // sharded: the merged keys go straight into every rank's inbox
        knn2_merge_push_kernel<<<div_up(q, 4), 128, 0, st>>>(*push, m->d_part.p, chunks, q);
    else
        knn2_merge_kernel<<<div_up(q, 4), 128, 0, st>>>(m->d_part.p, chunks, q, keys_dev, quad_dev);
    m->launches += 2;
    SFE_CUDA(cudaGetLastError());
    return SFE_OK;
}

namespace sfe {
cudaError_t launch_bow_score(cudaStream_t st, const int64_t *q_off, const int32_t *q_ids, const double *q_val, int q, int max_nq,
                             const int64_t *d_off, const int32_t *d_ids, const double *d_val, int n_entries, long long stride,
                             double *raw, uint8_t *hit, double *dense);
cudaError_t launch_bow_topk(cudaStream_t st, const double *raw, const uint8_t *hit, long long stride, int q, int n, int k,
                            int32_t *out_e, double *out_s, int32_t *out_n);
cudaError_t launch_bow_check(cudaStream_t st, const int64_t *off, const int32_t *ids, const double *val, int count, int n_words,
                             unsigned long long *chk);
cudaError_t launch_bow_rebase(cudaStream_t st, const int64_t *src, int count, int64_t base, int64_t *dst);
cudaError_t launch_bow_assemble(cudaStream_t st, const int32_t *word_id, const double *weight, const int32_t *n_set, int count,
                                int stride, int weighting, int norm, int32_t *cnt, double *div, int32_t *tmp_ids, double *tmp_val,
                                unsigned long long *status, int64_t *off, int32_t *ids, double *val);
}

struct sfe_bowdb {
    int device = 0, n_words = 0;
    int size = 0;                        // entries
    int64_t nnz = 0;                     // words over all entries
    int64_t cap_entries = 0, cap_nnz = 0;
    int64_t *off = nullptr;              // forward file: entry e = ids / val [off[e], off[e+1])
    int32_t *ids = nullptr;
    double *val = nullptr;
    mutable std::mutex mu;               // guards everything above and `readers`
    // one event per stream that has queried the database, recorded behind that query's kernels: an add that outgrows the
    // buffers waits for all of them before it frees the old ones
    mutable std::vector<std::pair<cudaStream_t, cudaEvent_t>> readers;
};

extern "C" {

int sfe_matcher_create(int device, sfe_matcher **out) {
    SFE_REQUIRE(out, SFE_ERR_BAD_ARG, "null argument");
    int ndev = 0;
    SFE_CUDA(cudaGetDeviceCount(&ndev));
    SFE_REQUIRE(ndev > 0, SFE_ERR_NO_DEVICE, "no CUDA device (there is no CPU fallback)");
    SFE_REQUIRE(device >= 0 && device < ndev, SFE_ERR_BAD_ARG, "device index out of range");
    DeviceGuard g(device);
    SFE_REQUIRE(g.ok, SFE_ERR_NO_DEVICE, "cannot select the handle's device");
    sfe_matcher *m = new sfe_matcher();
    m->device = device;
    cudaError_t e = cudaStreamCreateWithFlags(&m->stream, cudaStreamNonBlocking);
    if (e != cudaSuccess) {
        set_error("cudaStreamCreate: %s", cudaGetErrorString(e));
        delete m;
        return SFE_ERR_CUDA;
    }
    cudaDeviceGetAttribute(&m->sm_count, cudaDevAttrMultiProcessorCount, device);
    if (const char *env = getenv("SFE_KNN_TC")) m->knn_tc = atoi(env) != 0;
    if (const char *env = getenv("SFE_KNN_TC_MINQ")) m->knn_tc_min_q = std::max(1, atoi(env));
    if (const char *env = getenv("SFE_KNN_TILES_MAX_GB")) m->knn_tiles_max_bytes = (size_t)(std::max(0.0, atof(env)) * (double)(1ull << 30));
    *out = m;
    return SFE_OK;
}

int sfe_matcher_destroy(sfe_matcher *m) {
    if (!m) return SFE_OK;
    DeviceGuard g(m->device);
    SFE_REQUIRE(g.ok, SFE_ERR_NO_DEVICE, "cannot select the handle's device");
    cudaStreamSynchronize(m->stream);
    m->d_kl.release(); m->d_kr.release(); m->d_dl.release(); m->d_dr.release(); m->d_skip.release();
    m->d_n.release(); m->d_idx.release(); m->d_dist.release(); m->d_xw.release(); m->d_grid.release();
    m->d_best.release(); m->d_part.release(); m->d_keys.release(); m->d_quad.release();
    m->d_proj_bins.release(); m->d_proj_hist.release(); m->d_proj_perm.release();
    m->d_bow_off.release(); m->d_bow_ids.release(); m->d_bow_e.release(); m->d_bow_n.release(); m->d_bow_val.release();
    m->d_bow_raw.release(); m->d_bow_dense.release(); m->d_bow_s.release(); m->d_bow_hit.release();
    m->d_bow_chk.release(); m->d_bowa_cnt.release(); m->d_bowa_div.release(); m->d_bowa_ids.release(); m->d_bowa_val.release();
    cudaStreamDestroy(m->stream);
    delete m;
    return SFE_OK;
}

int sfe_matcher_set_async(sfe_matcher *m, int enable) {
    SFE_REQUIRE(m, SFE_ERR_BAD_ARG, "null handle");
    DeviceGuard g(m->device);
    SFE_REQUIRE(g.ok, SFE_ERR_NO_DEVICE, "cannot select the handle's device");
    SFE_CUDA(cudaStreamSynchronize(m->stream));
    m->async_dev = enable != 0;
    return SFE_OK;
}

int sfe_matcher_wait(sfe_matcher *m) {
    SFE_REQUIRE(m, SFE_ERR_BAD_ARG, "null handle");
    DeviceGuard g(m->device);
    SFE_REQUIRE(g.ok, SFE_ERR_NO_DEVICE, "cannot select the handle's device");
    SFE_CUDA(cudaStreamSynchronize(m->stream));
    return SFE_OK;
}

int sfe_matcher_launches(const sfe_matcher *m, int64_t *launches) {
    SFE_REQUIRE(m && launches, SFE_ERR_BAD_ARG, "null argument");
    *launches = m->launches;
    return SFE_OK;
}

int sfe_event_record_matcher(sfe_event *ev, sfe_matcher *m) {
    SFE_REQUIRE(ev && m, SFE_ERR_BAD_ARG, "null argument");
    DeviceGuard g(m->device);
    SFE_REQUIRE(g.ok, SFE_ERR_NO_DEVICE, "cannot select the handle's device");
    SFE_CUDA(cudaEventRecord(ev->ev, m->stream));
    return SFE_OK;
}

int sfe_stereo_match(sfe_matcher *m, const sfe_keypoint *kps_l, const uint8_t *desc_l, int n_l, const sfe_keypoint *kps_r,
                     const uint8_t *desc_r, int n_r, const sfe_stereo_params *sp, int32_t *out_idx, int32_t *out_dist) {
    SFE_REQUIRE(m && n_l >= 0 && n_r >= 0, SFE_ERR_BAD_ARG, "bad argument");
    if (n_l == 0) return SFE_OK;
    SFE_REQUIRE(kps_l && desc_l && out_idx && (n_r == 0 || (kps_r && desc_r)), SFE_ERR_BAD_ARG, "null argument");
    SFE_REQUIRE(n_l < 65536 && n_r < 65536, SFE_ERR_UNSUPPORTED, "more than 65535 keypoints per image");
    DeviceGuard g(m->device);
    SFE_REQUIRE(g.ok, SFE_ERR_NO_DEVICE, "cannot select the handle's device");
    const sfe_stereo_params def = {3.0, 100.0, 0.5};
    if (!sp) sp = &def;
    const int cap = std::max(n_l, std::max(n_r, 1));
    cudaStream_t st = m->stream;
    SFE_CUDA(m->d_kl.ensure(cap)); SFE_CUDA(m->d_kr.ensure(cap));
    SFE_CUDA(m->d_dl.ensure((size_t)cap * 32)); SFE_CUDA(m->d_dr.ensure((size_t)cap * 32));
    SFE_CUDA(m->d_n.ensure(2)); SFE_CUDA(m->d_idx.ensure(cap)); SFE_CUDA(m->d_dist.ensure(cap));
    const int32_t nn[2] = {n_l, n_r};
    SFE_CUDA(cudaMemcpyAsync(m->d_n.p, nn, sizeof(nn), cudaMemcpyHostToDevice, st));
    SFE_CUDA(cudaMemcpyAsync(m->d_kl.p, kps_l, sizeof(sfe_keypoint) * n_l, cudaMemcpyHostToDevice, st));
    SFE_CUDA(cudaMemcpyAsync(m->d_dl.p, desc_l, (size_t)n_l * 32, cudaMemcpyHostToDevice, st));
    if (n_r > 0) {
        SFE_CUDA(cudaMemcpyAsync(m->d_kr.p, kps_r, sizeof(sfe_keypoint) * n_r, cudaMemcpyHostToDevice, st));
        SFE_CUDA(cudaMemcpyAsync(m->d_dr.p, desc_r, (size_t)n_r * 32, cudaMemcpyHostToDevice, st));
    }
    launch_stereo_match(st, 1, cap, m->d_kl.p, m->d_dl.p, m->d_n.p, m->d_kr.p, m->d_dr.p, m->d_n.p + 1, sp->y_threshold,
                        sp->max_dx, sp->best12_threshold, m->d_idx.p, m->d_dist.p);
    m->launches++;
    SFE_CUDA(cudaGetLastError());
    SFE_CUDA(cudaMemcpyAsync(out_idx, m->d_idx.p, sizeof(int32_t) * n_l, cudaMemcpyDeviceToHost, st));
    if (out_dist) SFE_CUDA(cudaMemcpyAsync(out_dist, m->d_dist.p, sizeof(int32_t) * n_l, cudaMemcpyDeviceToHost, st));
    SFE_CUDA(cudaStreamSynchronize(st));
    return SFE_OK;
}

static int projection_match_dev_pose(sfe_matcher *m, const double *xw_dev, const uint8_t *mp_desc_dev, const uint8_t *skip_dev, int n,
                             const Pose &T, const sfe_camera *cam, const sfe_keypoint *kps_dev,
                             const uint8_t *kp_desc_dev, int m_kps, double radius, double best12_threshold,
                             int32_t *kp_to_query_dev, int32_t *kp_dist_dev) {
    SFE_REQUIRE(m && cam && n >= 0 && m_kps >= 0, SFE_ERR_BAD_ARG, "bad argument");
    SFE_REQUIRE(m_kps == 0 || (kps_dev && kp_desc_dev && kp_to_query_dev), SFE_ERR_BAD_ARG, "null argument");
    SFE_REQUIRE(n == 0 || (xw_dev && mp_desc_dev), SFE_ERR_BAD_ARG, "null argument");
    SFE_REQUIRE(m_kps < 65536, SFE_ERR_UNSUPPORTED, "more than 65535 keypoints per frame");
    DeviceGuard g(m->device);
    SFE_REQUIRE(g.ok, SFE_ERR_NO_DEVICE, "cannot select the handle's device");
    int rc = projection_impl(m, xw_dev, mp_desc_dev, skip_dev, n, T, cam, kps_dev, kp_desc_dev, m_kps, radius,
                             best12_threshold, kp_to_query_dev, kp_dist_dev);
    if (rc != SFE_OK) return rc;
    if (!m->async_dev) SFE_CUDA(cudaStreamSynchronize(m->stream));
    return SFE_OK;
}
int sfe_projection_match_dev(sfe_matcher *m, const double *xw_dev, const uint8_t *mp_desc_dev, const uint8_t *skip_dev, int n,
                             const double rt[12], const sfe_camera *cam, const sfe_keypoint *kps_dev,
                             const uint8_t *kp_desc_dev, int m_kps, double radius, double best12_threshold,
                             int32_t *kp_to_query_dev, int32_t *kp_dist_dev) {
    SFE_REQUIRE(rt, SFE_ERR_BAD_ARG, "null pose");
    return projection_match_dev_pose(m, xw_dev, mp_desc_dev, skip_dev, n, pose_from_rt(rt), cam, kps_dev, kp_desc_dev, m_kps, radius, best12_threshold, kp_to_query_dev, kp_dist_dev);
}
int sfe_projection_match_se3_dev(sfe_matcher *m, const double *xw_dev, const uint8_t *mp_desc_dev, const uint8_t *skip_dev, int n,
                             const sfe_se3 *Tcw, const sfe_camera *cam, const sfe_keypoint *kps_dev,
                             const uint8_t *kp_desc_dev, int m_kps, double radius, double best12_threshold,
                             int32_t *kp_to_query_dev, int32_t *kp_dist_dev) {
    SFE_REQUIRE(Tcw, SFE_ERR_BAD_ARG, "null pose");
    return projection_match_dev_pose(m, xw_dev, mp_desc_dev, skip_dev, n, pose_from_se3(Tcw), cam, kps_dev, kp_desc_dev, m_kps, radius, best12_threshold, kp_to_query_dev, kp_dist_dev);
}

static int projection_match_pose(sfe_matcher *m, const double *xw, const uint8_t *mp_desc, const uint8_t *skip, int n,
                         const Pose &T, const sfe_camera *cam, const sfe_keypoint *kps, const uint8_t *kp_desc,
                         int m_kps, double radius, double best12_threshold, int32_t *kp_to_query, int32_t *kp_dist) {
    SFE_REQUIRE(m && cam && n >= 0 && m_kps >= 0, SFE_ERR_BAD_ARG, "bad argument");
    if (m_kps == 0) return SFE_OK;
    SFE_REQUIRE(kps && kp_desc && kp_to_query, SFE_ERR_BAD_ARG, "null argument");
    SFE_REQUIRE(n == 0 || (xw && mp_desc), SFE_ERR_BAD_ARG, "null argument");
    SFE_REQUIRE(m_kps < 65536, SFE_ERR_UNSUPPORTED, "more than 65535 keypoints per frame");
    DeviceGuard g(m->device);
    SFE_REQUIRE(g.ok, SFE_ERR_NO_DEVICE, "cannot select the handle's device");
    cudaStream_t st = m->stream;
    const int nn = std::max(n, 1);
    SFE_CUDA(m->d_xw.ensure((size_t)nn * 3)); SFE_CUDA(m->d_dl.ensure((size_t)nn * 32)); SFE_CUDA(m->d_skip.ensure(nn));
    SFE_CUDA(m->d_kr.ensure(m_kps)); SFE_CUDA(m->d_dr.ensure((size_t)m_kps * 32));
    SFE_CUDA(m->d_idx.ensure(m_kps)); SFE_CUDA(m->d_dist.ensure(m_kps));
    if (n > 0) {
        SFE_CUDA(cudaMemcpyAsync(m->d_xw.p, xw, sizeof(double) * 3 * n, cudaMemcpyHostToDevice, st));
        SFE_CUDA(cudaMemcpyAsync(m->d_dl.p, mp_desc, (size_t)n * 32, cudaMemcpyHostToDevice, st));
        if (skip) SFE_CUDA(cudaMemcpyAsync(m->d_skip.p, skip, n, cudaMemcpyHostToDevice, st));
    }
    SFE_CUDA(cudaMemcpyAsync(m->d_kr.p, kps, sizeof(sfe_keypoint) * m_kps, cudaMemcpyHostToDevice, st));
    SFE_CUDA(cudaMemcpyAsync(m->d_dr.p, kp_desc, (size_t)m_kps * 32, cudaMemcpyHostToDevice, st));
    int rc = projection_impl(m, m->d_xw.p, m->d_dl.p, skip ? m->d_skip.p : nullptr, n, T, cam, m->d_kr.p, m->d_dr.p, m_kps,
                             radius, best12_threshold, m->d_idx.p, m->d_dist.p);
    if (rc != SFE_OK) return rc;
    SFE_CUDA(cudaMemcpyAsync(kp_to_query, m->d_idx.p, sizeof(int32_t) * m_kps, cudaMemcpyDeviceToHost, st));
    if (kp_dist) SFE_CUDA(cudaMemcpyAsync(kp_dist, m->d_dist.p, sizeof(int32_t) * m_kps, cudaMemcpyDeviceToHost, st));
    SFE_CUDA(cudaStreamSynchronize(st));
    return SFE_OK;
}
int sfe_projection_match(sfe_matcher *m, const double *xw, const uint8_t *mp_desc, const uint8_t *skip, int n,
                         const double rt[12], const sfe_camera *cam, const sfe_keypoint *kps, const uint8_t *kp_desc,
                         int m_kps, double radius, double best12_threshold, int32_t *kp_to_query, int32_t *kp_dist) {
    SFE_REQUIRE(rt, SFE_ERR_BAD_ARG, "null pose");
    return projection_match_pose(m, xw, mp_desc, skip, n, pose_from_rt(rt), cam, kps, kp_desc, m_kps, radius, best12_threshold, kp_to_query, kp_dist);
}
int sfe_projection_match_se3(sfe_matcher *m, const double *xw, const uint8_t *mp_desc, const uint8_t *skip, int n,
                         const sfe_se3 *Tcw, const sfe_camera *cam, const sfe_keypoint *kps, const uint8_t *kp_desc,
                         int m_kps, double radius, double best12_threshold, int32_t *kp_to_query, int32_t *kp_dist) {
    SFE_REQUIRE(Tcw, SFE_ERR_BAD_ARG, "null pose");
    return projection_match_pose(m, xw, mp_desc, skip, n, pose_from_se3(Tcw), cam, kps, kp_desc, m_kps, radius, best12_threshold, kp_to_query, kp_dist);
}

static int projection_match_keys_dev_pose(sfe_matcher *m, const double *xw_dev, const uint8_t *mp_desc_dev, const uint8_t *skip_dev,
                                  int n, int64_t idx_base, const Pose &T, const sfe_camera *cam,
                                  const sfe_keypoint *kps_dev, const uint8_t *kp_desc_dev, int m_kps, double radius,
                                  double best12_threshold, uint64_t *keys_dev) {
    SFE_REQUIRE(m && cam && n >= 0 && m_kps >= 1 && keys_dev && kps_dev && kp_desc_dev, SFE_ERR_BAD_ARG, "bad argument");
    SFE_REQUIRE(n == 0 || (xw_dev && mp_desc_dev), SFE_ERR_BAD_ARG, "null argument");
    SFE_REQUIRE(m_kps < 65536, SFE_ERR_UNSUPPORTED, "more than 65535 keypoints per frame");
    SFE_REQUIRE(idx_base >= 0 && idx_base + n < (1ll << 31), SFE_ERR_UNSUPPORTED, "global map-point index must fit int32");
    DeviceGuard g(m->device);
    SFE_REQUIRE(g.ok, SFE_ERR_NO_DEVICE, "cannot select the handle's device");
    int rc = projection_impl(m, xw_dev, mp_desc_dev, skip_dev, n, T, cam, kps_dev, kp_desc_dev, m_kps, radius, best12_threshold,
                             nullptr, nullptr, (uint32_t)idx_base, (unsigned long long *)keys_dev);
    if (rc != SFE_OK) return rc;
    if (!m->async_dev) SFE_CUDA(cudaStreamSynchronize(m->stream));
    return SFE_OK;
}
int sfe_projection_match_keys_dev(sfe_matcher *m, const double *xw_dev, const uint8_t *mp_desc_dev, const uint8_t *skip_dev,
                                  int n, int64_t idx_base, const double rt[12], const sfe_camera *cam,
                                  const sfe_keypoint *kps_dev, const uint8_t *kp_desc_dev, int m_kps, double radius,
                                  double best12_threshold, uint64_t *keys_dev) {
    SFE_REQUIRE(rt, SFE_ERR_BAD_ARG, "null pose");
    return projection_match_keys_dev_pose(m, xw_dev, mp_desc_dev, skip_dev, n, idx_base, pose_from_rt(rt), cam, kps_dev, kp_desc_dev, m_kps, radius, best12_threshold, keys_dev);
}
int sfe_projection_match_keys_se3_dev(sfe_matcher *m, const double *xw_dev, const uint8_t *mp_desc_dev, const uint8_t *skip_dev,
                                  int n, int64_t idx_base, const sfe_se3 *Tcw, const sfe_camera *cam,
                                  const sfe_keypoint *kps_dev, const uint8_t *kp_desc_dev, int m_kps, double radius,
                                  double best12_threshold, uint64_t *keys_dev) {
    SFE_REQUIRE(Tcw, SFE_ERR_BAD_ARG, "null pose");
    return projection_match_keys_dev_pose(m, xw_dev, mp_desc_dev, skip_dev, n, idx_base, pose_from_se3(Tcw), cam, kps_dev, kp_desc_dev, m_kps, radius, best12_threshold, keys_dev);
}

int sfe_projection_merge_dev(sfe_matcher *m, const uint64_t *keys_dev, int shards, int m_kps, int32_t *kp_to_query_dev,
                             int32_t *kp_dist_dev) {
    SFE_REQUIRE(m && keys_dev && kp_to_query_dev && shards >= 1 && m_kps >= 1, SFE_ERR_BAD_ARG, "bad argument");
    DeviceGuard g(m->device);
    SFE_REQUIRE(g.ok, SFE_ERR_NO_DEVICE, "cannot select the handle's device");
    projection_decode_kernel<<<div_up(m_kps, 256), 256, 0, m->stream>>>(m_kps, shards, (const unsigned long long *)keys_dev,
                                                                         kp_to_query_dev, kp_dist_dev);
    m->launches++;
    SFE_CUDA(cudaGetLastError());
    if (!m->async_dev) SFE_CUDA(cudaStreamSynchronize(m->stream));
    return SFE_OK;
}

// ---- resident frames (SURVEY §8f rows 1, 3) ---------------------------------------------------------------
static int frame_finish(sfe_matcher *m, sfe_frame *f) {
    cudaStream_t st = m->stream;
    SFE_CUDA(f->nrm.ensure(std::max(f->n, 1)));
    if (f->n > 0) {
        normalized_undistort_kernel<<<div_up(f->n, 128), 128, 0, st>>>(f->cam, f->kps.p, f->n, f->nrm.p);
        m->launches++;
    }
    int rc = build_grid(m, f->grid_mem, f->grid, &f->cam, f->kps.p, f->desc.p, f->n);
    if (rc != SFE_OK) return rc;
    SFE_CUDA(cudaGetLastError());
    SFE_CUDA(cudaStreamSynchronize(st));
    return SFE_OK;
}

static int frame_new(sfe_matcher *m, const sfe_keypoint *kps, const uint8_t *desc, int n, const sfe_camera *cam, bool on_device,
                     sfe_frame **out) {
    SFE_REQUIRE(m && cam && out && n >= 0 && n < 65536, SFE_ERR_BAD_ARG, "bad argument");
    SFE_REQUIRE(n == 0 || (kps && desc), SFE_ERR_BAD_ARG, "null argument");
    DeviceGuard g(m->device);
    SFE_REQUIRE(g.ok, SFE_ERR_NO_DEVICE, "cannot select the handle's device");
    sfe_frame *f = new sfe_frame();
    f->device = m->device;
    f->n = n;
    f->cam = *cam;
    const cudaMemcpyKind kind = on_device ? cudaMemcpyDeviceToDevice : cudaMemcpyHostToDevice;
    cudaError_t e = f->kps.ensure(std::max(n, 1));
    if (e == cudaSuccess) e = f->desc.ensure((size_t)std::max(n, 1) * 32);
    if (e == cudaSuccess && n > 0) e = cudaMemcpyAsync(f->kps.p, kps, sizeof(sfe_keypoint) * n, kind, m->stream);
    if (e == cudaSuccess && n > 0) e = cudaMemcpyAsync(f->desc.p, desc, (size_t)n * 32, kind, m->stream);
    int rc = SFE_OK;
    if (e != cudaSuccess) {
        set_error("frame upload: %s", cudaGetErrorString(e));
        rc = SFE_ERR_CUDA;
    } else {
        rc = frame_finish(m, f);
    }
    if (rc != SFE_OK) {
        sfe_frame_destroy(f);
        return rc;
    }
    *out = f;
    return SFE_OK;
}

int sfe_frame_create(sfe_matcher *m, const sfe_keypoint *kps, const uint8_t *desc, int n, const sfe_camera *cam, sfe_frame **out) {
    return frame_new(m, kps, desc, n, cam, false, out);
}

int sfe_frame_create_dev(sfe_matcher *m, const sfe_keypoint *kps_dev, const uint8_t *desc_dev, int n, const sfe_camera *cam,
                         sfe_frame **out) {
    return frame_new(m, kps_dev, desc_dev, n, cam, true, out);
}

int sfe_frame_destroy(sfe_frame *f) {
    if (!f) return SFE_OK;
    DeviceGuard g(f->device);
    SFE_REQUIRE(g.ok, SFE_ERR_NO_DEVICE, "cannot select the handle's device");
    f->kps.release(); f->desc.release(); f->nrm.release(); f->grid_mem.release();
    delete f;
    return SFE_OK;
}

int sfe_frame_size(const sfe_frame *f, int *n) {
    SFE_REQUIRE(f && n, SFE_ERR_BAD_ARG, "null argument");
    *n = f->n;
    return SFE_OK;
}

int sfe_frame_normalized(sfe_matcher *m, const sfe_frame *f, double *xy) {
    SFE_REQUIRE(m && f && (xy || f->n == 0), SFE_ERR_BAD_ARG, "null argument");
    SFE_REQUIRE(f->device == m->device, SFE_ERR_BAD_ARG, "frame lives on another device");
    DeviceGuard g(m->device);
    SFE_REQUIRE(g.ok, SFE_ERR_NO_DEVICE, "cannot select the handle's device");
    if (f->n > 0) SFE_CUDA(cudaMemcpyAsync(xy, f->nrm.p, sizeof(double2) * f->n, cudaMemcpyDeviceToHost, m->stream));
    SFE_CUDA(cudaStreamSynchronize(m->stream));
    return SFE_OK;
}

int sfe_frame_stereo_depth(sfe_matcher *m, const sfe_frame *f, const sfe_keypoint *kps_r, int n_r, const int32_t *stereo_idx,
                           double baseline, double *xc, uint8_t *valid) {
    SFE_REQUIRE(m && f && n_r >= 0, SFE_ERR_BAD_ARG, "bad argument");
    SFE_REQUIRE(f->device == m->device, SFE_ERR_BAD_ARG, "frame lives on another device");
    if (f->n == 0) return SFE_OK;
    SFE_REQUIRE(stereo_idx && xc && valid && (kps_r || n_r == 0), SFE_ERR_BAD_ARG, "null argument");
    for (int i = 0; i < f->n; i++) SFE_REQUIRE(stereo_idx[i] < n_r, SFE_ERR_BAD_ARG, "stereo index outside the right keypoints");
    DeviceGuard g(m->device);
    SFE_REQUIRE(g.ok, SFE_ERR_NO_DEVICE, "cannot select the handle's device");
    cudaStream_t st = m->stream;
    SFE_CUDA(m->d_kr.ensure(std::max(n_r, 1)));
    SFE_CUDA(m->d_idx.ensure(f->n));
    SFE_CUDA(m->d_xw.ensure((size_t)f->n * 3));
    SFE_CUDA(m->d_skip.ensure(f->n));
    if (n_r > 0) SFE_CUDA(cudaMemcpyAsync(m->d_kr.p, kps_r, sizeof(sfe_keypoint) * n_r, cudaMemcpyHostToDevice, st));
    SFE_CUDA(cudaMemcpyAsync(m->d_idx.p, stereo_idx, sizeof(int32_t) * f->n, cudaMemcpyHostToDevice, st));
    stereo_depth_kernel<<<div_up(f->n, 128), 128, 0, st>>>(f->cam.fx, baseline, f->kps.p, f->nrm.p, f->n, m->d_kr.p, m->d_idx.p,
                                                           m->d_xw.p, m->d_skip.p);
    m->launches++;
    SFE_CUDA(cudaGetLastError());
    SFE_CUDA(cudaMemcpyAsync(xc, m->d_xw.p, sizeof(double) * 3 * f->n, cudaMemcpyDeviceToHost, st));
    SFE_CUDA(cudaMemcpyAsync(valid, m->d_skip.p, f->n, cudaMemcpyDeviceToHost, st));
    SFE_CUDA(cudaStreamSynchronize(st));
    return SFE_OK;
}

static int frame_reprojection_error_pose(sfe_matcher *m, const sfe_frame *f, const double *xw, const uint8_t *has_mp, const Pose &T,
                                 double *err) {
    SFE_REQUIRE(m && f, SFE_ERR_BAD_ARG, "bad argument");
    SFE_REQUIRE(f->device == m->device, SFE_ERR_BAD_ARG, "frame lives on another device");
    if (f->n == 0) return SFE_OK;
    SFE_REQUIRE(xw && has_mp && err, SFE_ERR_BAD_ARG, "null argument");
    DeviceGuard g(m->device);
    SFE_REQUIRE(g.ok, SFE_ERR_NO_DEVICE, "cannot select the handle's device");
    cudaStream_t st = m->stream;
    SFE_CUDA(m->d_xw.ensure((size_t)f->n * 4));  // n x 3 points, then n errors
    SFE_CUDA(m->d_skip.ensure(f->n));
    SFE_CUDA(cudaMemcpyAsync(m->d_xw.p, xw, sizeof(double) * 3 * f->n, cudaMemcpyHostToDevice, st));
    SFE_CUDA(cudaMemcpyAsync(m->d_skip.p, has_mp, f->n, cudaMemcpyHostToDevice, st));
    ProjParams P{};
    P.T = T;
    reprojection_error_kernel<<<div_up(f->n, 128), 128, 0, st>>>(f->cam, P, f->kps.p, f->n, m->d_xw.p, m->d_skip.p,
                                                                 m->d_xw.p + (size_t)f->n * 3);
    m->launches++;
    SFE_CUDA(cudaGetLastError());
    SFE_CUDA(cudaMemcpyAsync(err, m->d_xw.p + (size_t)f->n * 3, sizeof(double) * f->n, cudaMemcpyDeviceToHost, st));
    SFE_CUDA(cudaStreamSynchronize(st));
    return SFE_OK;
}
int sfe_frame_reprojection_error(sfe_matcher *m, const sfe_frame *f, const double *xw, const uint8_t *has_mp, const double rt[12],
                                 double *err) {
    SFE_REQUIRE(rt, SFE_ERR_BAD_ARG, "null pose");
    return frame_reprojection_error_pose(m, f, xw, has_mp, pose_from_rt(rt), err);
}
int sfe_frame_reprojection_error_se3(sfe_matcher *m, const sfe_frame *f, const double *xw, const uint8_t *has_mp, const sfe_se3 *Tcw,
                                 double *err) {
    SFE_REQUIRE(Tcw, SFE_ERR_BAD_ARG, "null pose");
    return frame_reprojection_error_pose(m, f, xw, has_mp, pose_from_se3(Tcw), err);
}

static int frame_projection_match_pose(sfe_matcher *m, const sfe_frame *f, const double *xw, const uint8_t *mp_desc, const uint8_t *skip,
                               int n, const Pose &T, double radius, double best12_threshold, int32_t *kp_to_query,
                               int32_t *kp_dist) {
    SFE_REQUIRE(m && f && n >= 0, SFE_ERR_BAD_ARG, "bad argument");
    SFE_REQUIRE(f->device == m->device, SFE_ERR_BAD_ARG, "frame lives on another device");
    if (f->n == 0) return SFE_OK;
    SFE_REQUIRE(kp_to_query && (n == 0 || (xw && mp_desc)), SFE_ERR_BAD_ARG, "null argument");
    DeviceGuard g(m->device);
    SFE_REQUIRE(g.ok, SFE_ERR_NO_DEVICE, "cannot select the handle's device");
    cudaStream_t st = m->stream;
    const int nn = std::max(n, 1);
    SFE_CUDA(m->d_xw.ensure((size_t)nn * 3)); SFE_CUDA(m->d_dl.ensure((size_t)nn * 32)); SFE_CUDA(m->d_skip.ensure(nn));
    SFE_CUDA(m->d_idx.ensure(f->n)); SFE_CUDA(m->d_dist.ensure(f->n));
    if (n > 0) {
        SFE_CUDA(cudaMemcpyAsync(m->d_xw.p, xw, sizeof(double) * 3 * n, cudaMemcpyHostToDevice, st));
        SFE_CUDA(cudaMemcpyAsync(m->d_dl.p, mp_desc, (size_t)n * 32, cudaMemcpyHostToDevice, st));
        if (skip) SFE_CUDA(cudaMemcpyAsync(m->d_skip.p, skip, n, cudaMemcpyHostToDevice, st));
    }
    int rc = projection_impl(m, m->d_xw.p, m->d_dl.p, skip ? m->d_skip.p : nullptr, n, T, &f->cam, f->kps.p, f->desc.p, f->n, radius,
                             best12_threshold, m->d_idx.p, m->d_dist.p, 0, nullptr, &f->grid);
    if (rc != SFE_OK) return rc;
    SFE_CUDA(cudaMemcpyAsync(kp_to_query, m->d_idx.p, sizeof(int32_t) * f->n, cudaMemcpyDeviceToHost, st));
    if (kp_dist) SFE_CUDA(cudaMemcpyAsync(kp_dist, m->d_dist.p, sizeof(int32_t) * f->n, cudaMemcpyDeviceToHost, st));
    SFE_CUDA(cudaStreamSynchronize(st));
    return SFE_OK;
}
int sfe_frame_projection_match(sfe_matcher *m, const sfe_frame *f, const double *xw, const uint8_t *mp_desc, const uint8_t *skip,
                               int n, const double rt[12], double radius, double best12_threshold, int32_t *kp_to_query,
                               int32_t *kp_dist) {
    SFE_REQUIRE(rt, SFE_ERR_BAD_ARG, "null pose");
    return frame_projection_match_pose(m, f, xw, mp_desc, skip, n, pose_from_rt(rt), radius, best12_threshold, kp_to_query, kp_dist);
}
int sfe_frame_projection_match_se3(sfe_matcher *m, const sfe_frame *f, const double *xw, const uint8_t *mp_desc, const uint8_t *skip,
                               int n, const sfe_se3 *Tcw, double radius, double best12_threshold, int32_t *kp_to_query,
                               int32_t *kp_dist) {
    SFE_REQUIRE(Tcw, SFE_ERR_BAD_ARG, "null pose");
    return frame_projection_match_pose(m, f, xw, mp_desc, skip, n, pose_from_se3(Tcw), radius, best12_threshold, kp_to_query, kp_dist);
}

int sfe_frame_search_radius(sfe_matcher *m, const sfe_frame *f, const double *uv, int q, double radius, int32_t *idx, int cap,
                            int32_t *counts) {
    SFE_REQUIRE(m && f && q >= 0 && cap >= 1, SFE_ERR_BAD_ARG, "bad argument");
    SFE_REQUIRE(f->device == m->device, SFE_ERR_BAD_ARG, "frame lives on another device");
    if (q == 0) return SFE_OK;
    SFE_REQUIRE(uv && idx && counts, SFE_ERR_BAD_ARG, "null argument");
    DeviceGuard g(m->device);
    SFE_REQUIRE(g.ok, SFE_ERR_NO_DEVICE, "cannot select the handle's device");
    cudaStream_t st = m->stream;
    SFE_CUDA(m->d_xw.ensure((size_t)q * 2));
    SFE_CUDA(m->d_quad.ensure((size_t)q * cap));
    SFE_CUDA(m->d_n.ensure(q));
    SFE_CUDA(cudaMemcpyAsync(m->d_xw.p, uv, sizeof(double) * 2 * q, cudaMemcpyHostToDevice, st));
    search_radius_kernel<<<div_up(q, 64), 64, 0, st>>>(f->grid, f->kps.p, (const double2 *)m->d_xw.p, q, radius, m->d_quad.p, cap, m->d_n.p);
    m->launches++;
    SFE_CUDA(cudaGetLastError());
    SFE_CUDA(cudaMemcpyAsync(idx, m->d_quad.p, sizeof(int32_t) * (size_t)q * cap, cudaMemcpyDeviceToHost, st));
    SFE_CUDA(cudaMemcpyAsync(counts, m->d_n.p, sizeof(int32_t) * q, cudaMemcpyDeviceToHost, st));
    SFE_CUDA(cudaStreamSynchronize(st));
    return SFE_OK;
}

int sfe_frame_search_nearest(sfe_matcher *m, const sfe_frame *f, const double *uv, int q, int32_t *kpt_index, double *dist2) {
    SFE_REQUIRE(m && f && q >= 0, SFE_ERR_BAD_ARG, "bad argument");
    SFE_REQUIRE(f->device == m->device, SFE_ERR_BAD_ARG, "frame lives on another device");
    if (q == 0) return SFE_OK;
    SFE_REQUIRE(uv && kpt_index && dist2, SFE_ERR_BAD_ARG, "null argument");
    DeviceGuard g(m->device);
    SFE_REQUIRE(g.ok, SFE_ERR_NO_DEVICE, "cannot select the handle's device");
    cudaStream_t st = m->stream;
    SFE_CUDA(m->d_xw.ensure((size_t)q * 3));
    SFE_CUDA(m->d_n.ensure(q));
    SFE_CUDA(cudaMemcpyAsync(m->d_xw.p, uv, sizeof(double) * 2 * q, cudaMemcpyHostToDevice, st));
    double *d2 = m->d_xw.p + (size_t)2 * q;
    search_nearest_kernel<<<div_up(q, 64), 64, 0, st>>>(f->grid, f->kps.p, (const double2 *)m->d_xw.p, q, m->d_n.p, d2);
    m->launches++;
    SFE_CUDA(cudaGetLastError());
    SFE_CUDA(cudaMemcpyAsync(kpt_index, m->d_n.p, sizeof(int32_t) * q, cudaMemcpyDeviceToHost, st));
    SFE_CUDA(cudaMemcpyAsync(dist2, d2, sizeof(double) * q, cudaMemcpyDeviceToHost, st));
    SFE_CUDA(cudaStreamSynchronize(st));
    return SFE_OK;
}

// ---- vocabulary (SURVEY §8f row 2) -----------------------------------------------------------------------
int sfe_vocab_create(sfe_matcher *m, int n_nodes, const int32_t *parent, const uint8_t *is_leaf, const uint8_t *desc,
                     const double *weight, int L, sfe_vocab **out) {
    SFE_REQUIRE(m && parent && is_leaf && desc && weight && out, SFE_ERR_BAD_ARG, "null argument");
    SFE_REQUIRE(n_nodes >= 2 && L >= 1, SFE_ERR_BAD_ARG, "empty vocabulary");
    std::vector<int> start(n_nodes + 1, 0), list(n_nodes, 0), fill(n_nodes, 0), wid(n_nodes, 0);
    for (int i = 1; i < n_nodes; i++) {
        SFE_REQUIRE(parent[i] >= 0 && parent[i] < i, SFE_ERR_BAD_ARG, "a node must follow its parent (loadFromTextFile order)");
        start[parent[i] + 1]++;
    }
    for (int i = 0; i < n_nodes; i++) start[i + 1] += start[i];
    int words = 0;
    for (int i = 1; i < n_nodes; i++) {
        list[start[parent[i]] + fill[parent[i]]++] = i;
        if (is_leaf[i]) wid[i] = words++;
    }
    SFE_REQUIRE(start[1] > 0, SFE_ERR_BAD_ARG, "the root has no children");
    DeviceGuard g(m->device);
    SFE_REQUIRE(g.ok, SFE_ERR_NO_DEVICE, "cannot select the handle's device");
    sfe_vocab *v = new sfe_vocab();
    v->device = m->device;
    v->n_nodes = n_nodes;
    v->L = L;
    v->n_words = words;
    cudaError_t e = v->child_start.ensure(n_nodes + 1);
    if (e == cudaSuccess) e = v->child_list.ensure(n_nodes);
    if (e == cudaSuccess) e = v->word_id.ensure(n_nodes);
    if (e == cudaSuccess) e = v->desc.ensure((size_t)n_nodes * 32);
    if (e == cudaSuccess) e = v->weight.ensure(n_nodes);
    if (e == cudaSuccess) e = cudaMemcpy(v->child_start.p, start.data(), sizeof(int) * (n_nodes + 1), cudaMemcpyHostToDevice);
    if (e == cudaSuccess) e = cudaMemcpy(v->child_list.p, list.data(), sizeof(int) * n_nodes, cudaMemcpyHostToDevice);
    if (e == cudaSuccess) e = cudaMemcpy(v->word_id.p, wid.data(), sizeof(int) * n_nodes, cudaMemcpyHostToDevice);
    if (e == cudaSuccess) e = cudaMemcpy(v->desc.p, desc, (size_t)n_nodes * 32, cudaMemcpyHostToDevice);
    if (e == cudaSuccess) e = cudaMemcpy(v->weight.p, weight, sizeof(double) * n_nodes, cudaMemcpyHostToDevice);
    if (e != cudaSuccess) {
        set_error("vocabulary upload: %s", cudaGetErrorString(e));
        sfe_vocab_destroy(v);
        return SFE_ERR_CUDA;
    }
    *out = v;
    return SFE_OK;
}

int sfe_vocab_destroy(sfe_vocab *v) {
    if (!v) return SFE_OK;
    DeviceGuard g(v->device);
    SFE_REQUIRE(g.ok, SFE_ERR_NO_DEVICE, "cannot select the handle's device");
    v->child_start.release(); v->child_list.release(); v->word_id.release(); v->desc.release(); v->weight.release();
    delete v;
    return SFE_OK;
}

int sfe_vocab_words(const sfe_vocab *v, int *n_words) {
    SFE_REQUIRE(v && n_words, SFE_ERR_BAD_ARG, "null argument");
    *n_words = v->n_words;
    return SFE_OK;
}

static int vocab_launch(sfe_matcher *m, const sfe_vocab *v, const uint8_t *feat_dev, int n, int levelsup, int32_t *wid, double *w,
                        int32_t *nid) {
    VocabDev V{v->child_start.p, v->child_list.p, v->desc.p, v->weight.p, v->word_id.p, v->n_nodes, v->L};
    vocab_transform_kernel<<<div_up(n, 8), 256, 0, m->stream>>>(V, feat_dev, n, levelsup, wid, w, nid);
    m->launches++;
    SFE_CUDA(cudaGetLastError());
    return SFE_OK;
}

int sfe_vocab_transform_dev(sfe_matcher *m, const sfe_vocab *v, const uint8_t *desc_dev, int n, int levelsup, int32_t *word_id_dev,
                            double *weight_dev, int32_t *node_id_dev) {
    SFE_REQUIRE(m && v && n >= 0 && levelsup >= 0, SFE_ERR_BAD_ARG, "bad argument");
    SFE_REQUIRE(v->device == m->device, SFE_ERR_BAD_ARG, "vocabulary lives on another device");
    if (n == 0) return SFE_OK;
    SFE_REQUIRE(desc_dev && word_id_dev && weight_dev && node_id_dev, SFE_ERR_BAD_ARG, "null argument");
    DeviceGuard g(m->device);
    SFE_REQUIRE(g.ok, SFE_ERR_NO_DEVICE, "cannot select the handle's device");
    int rc = vocab_launch(m, v, desc_dev, n, levelsup, word_id_dev, weight_dev, node_id_dev);
    if (rc != SFE_OK) return rc;
    if (!m->async_dev) SFE_CUDA(cudaStreamSynchronize(m->stream));
    return SFE_OK;
}

int sfe_vocab_transform(sfe_matcher *m, const sfe_vocab *v, const uint8_t *desc, int n, int levelsup, int32_t *word_id,
                        double *weight, int32_t *node_id) {
    SFE_REQUIRE(m && v && n >= 0 && levelsup >= 0, SFE_ERR_BAD_ARG, "bad argument");
    SFE_REQUIRE(v->device == m->device, SFE_ERR_BAD_ARG, "vocabulary lives on another device");
    if (n == 0) return SFE_OK;
    SFE_REQUIRE(desc && word_id && weight && node_id, SFE_ERR_BAD_ARG, "null argument");
    DeviceGuard g(m->device);
    SFE_REQUIRE(g.ok, SFE_ERR_NO_DEVICE, "cannot select the handle's device");
    cudaStream_t st = m->stream;
    SFE_CUDA(m->d_dl.ensure((size_t)n * 32));
    SFE_CUDA(m->d_idx.ensure(n)); SFE_CUDA(m->d_dist.ensure(n)); SFE_CUDA(m->d_xw.ensure(n));
    SFE_CUDA(cudaMemcpyAsync(m->d_dl.p, desc, (size_t)n * 32, cudaMemcpyHostToDevice, st));
    int rc = vocab_launch(m, v, m->d_dl.p, n, levelsup, m->d_idx.p, m->d_xw.p, m->d_dist.p);
    if (rc != SFE_OK) return rc;
    SFE_CUDA(cudaMemcpyAsync(word_id, m->d_idx.p, sizeof(int32_t) * n, cudaMemcpyDeviceToHost, st));
    SFE_CUDA(cudaMemcpyAsync(weight, m->d_xw.p, sizeof(double) * n, cudaMemcpyDeviceToHost, st));
    SFE_CUDA(cudaMemcpyAsync(node_id, m->d_dist.p, sizeof(int32_t) * n, cudaMemcpyDeviceToHost, st));
    SFE_CUDA(cudaStreamSynchronize(st));
    return SFE_OK;
}

// BowVector assembly on the host, in the reference's order of operations (TemplatedVocabulary.h:1127-1194,
// BowVector.cpp:34-84): ids ascending, weights accumulated in feature order, then the norm taken in id order.
int sfe_bow_assemble(const int32_t *word_id, const double *weight, int n, int weighting, int norm, int32_t *ids, double *values,
                     int cap, int *n_out) {
    SFE_REQUIRE(n >= 0 && n_out && (n == 0 || (word_id && weight)) && cap >= 0, SFE_ERR_BAD_ARG, "bad argument");
    SFE_REQUIRE(weighting >= 0 && weighting <= 3 && norm >= 0 && norm <= 2, SFE_ERR_BAD_ARG, "unknown weighting / norm");
    std::vector<std::pair<int32_t, double>> v;  // kept sorted by id: what std::map iteration yields
    v.reserve(n);
    const bool accumulate = weighting == 0 || weighting == 1;  // TF_IDF, TF: addWeight; IDF, BINARY: addIfNotExist
    for (int i = 0; i < n; i++) {
        if (!(weight[i] > 0)) continue;  // stopped word
        auto it = std::lower_bound(v.begin(), v.end(), word_id[i], [](const std::pair<int32_t, double> &a, int32_t id) { return a.first < id; });
        if (it != v.end() && it->first == word_id[i]) {
            if (accumulate) it->second += weight[i];
        } else {
            v.insert(it, std::make_pair(word_id[i], weight[i]));
        }
    }
    if (accumulate && !v.empty() && norm == 0) {  // "unnecessary when normalizing"
        const double nd = (double)v.size();
        for (auto &e : v) e.second /= nd;
    }
    if (norm != 0) {  // 1 = L1, 2 = L2
        double s = 0.0;
        if (norm == 1) for (auto &e : v) s += fabs(e.second);
        else { for (auto &e : v) s += e.second * e.second; s = sqrt(s); }
        if (s > 0.0) for (auto &e : v) e.second /= s;
    }
    *n_out = (int)v.size();
    SFE_REQUIRE((int)v.size() <= cap || (!ids && !values), SFE_ERR_CAPACITY, "BowVector larger than the caller's capacity");
    for (size_t i = 0; i < v.size() && ids && values; i++) { ids[i] = v[i].first; values[i] = v[i].second; }
    return SFE_OK;
}

// The same assembly for `count` feature sets on the device (bow_assemble_kernel, csrc/sfe_bow.cu), bit for bit.
int sfe_bow_assemble_dev(sfe_matcher *m, const int32_t *word_id_dev, const double *weight_dev, const int32_t *n_dev, int count,
                         int stride, int weighting, int norm, int64_t *bow_off_dev, int32_t *bow_ids_dev, double *bow_val_dev) {
    SFE_REQUIRE(m && count >= 0 && stride >= 0 && bow_off_dev, SFE_ERR_BAD_ARG, "bad argument");
    SFE_REQUIRE(weighting >= 0 && weighting <= 3 && norm >= 0 && norm <= 2, SFE_ERR_BAD_ARG, "unknown weighting / norm");
    SFE_REQUIRE(count == 0 || (word_id_dev && weight_dev && n_dev && bow_ids_dev && bow_val_dev), SFE_ERR_BAD_ARG, "null argument");
    SFE_REQUIRE(stride <= SFE_BOW_ASSEMBLE_MAX_STRIDE, SFE_ERR_UNSUPPORTED, "stride above SFE_BOW_ASSEMBLE_MAX_STRIDE");
    DeviceGuard g(m->device);
    SFE_REQUIRE(g.ok, SFE_ERR_NO_DEVICE, "cannot select the handle's device");
    cudaStream_t st = m->stream;
    const size_t rows = std::max<size_t>((size_t)count * stride, 1);
    SFE_CUDA(m->d_bow_chk.ensure(3));
    SFE_CUDA(m->d_bowa_cnt.ensure(std::max(count, 1)));
    SFE_CUDA(m->d_bowa_div.ensure(std::max(count, 1)));
    SFE_CUDA(m->d_bowa_ids.ensure(rows));
    SFE_CUDA(m->d_bowa_val.ensure(rows));
    SFE_CUDA(launch_bow_assemble(st, word_id_dev, weight_dev, n_dev, count, stride, weighting, norm, m->d_bowa_cnt.p, m->d_bowa_div.p,
                                 m->d_bowa_ids.p, m->d_bowa_val.p, m->d_bow_chk.p, bow_off_dev, bow_ids_dev, bow_val_dev));
    m->launches += count > 0 ? 3 : 0;
    unsigned long long status = 0;
    SFE_CUDA(cudaMemcpyAsync(&status, m->d_bow_chk.p, sizeof(status), cudaMemcpyDeviceToHost, st));
    SFE_CUDA(cudaStreamSynchronize(st));
    SFE_REQUIRE(status == 0, SFE_ERR_BAD_ARG, "a feature count n_dev[i] outside [0, stride]");
    return SFE_OK;
}

// ---- BoW database (DBoW2 TemplatedDatabase with L1 scoring) -----------------------------------------------------------
// Vectors arrive from outside the program: CSR offsets from 0, non-decreasing; ids in [0, n_words) and strictly ascending
// within a vector (a BowVector is a std::map); finite values.
static int bow_check_vectors(const int64_t *off, const int32_t *ids, const double *val, int count, int n_words) {
    SFE_REQUIRE(off, SFE_ERR_BAD_ARG, "null offsets");
    SFE_REQUIRE(off[0] == 0, SFE_ERR_BAD_ARG, "offsets[0] must be 0");
    for (int i = 0; i < count; i++) SFE_REQUIRE(off[i + 1] >= off[i], SFE_ERR_BAD_ARG, "offsets must not decrease");
    SFE_REQUIRE(off[count] == 0 || (ids && val), SFE_ERR_BAD_ARG, "null ids / values");
    for (int i = 0; i < count; i++) {
        for (int64_t j = off[i]; j < off[i + 1]; j++) {
            SFE_REQUIRE(ids[j] >= 0 && ids[j] < n_words, SFE_ERR_BAD_ARG, "word id outside [0, n_words)");
            SFE_REQUIRE(j == off[i] || ids[j] > ids[j - 1], SFE_ERR_BAD_ARG, "word ids must ascend strictly within a vector");
            SFE_REQUIRE(std::isfinite(val[j]), SFE_ERR_BAD_ARG, "values must be finite");
        }
    }
    return SFE_OK;
}

int sfe_bowdb_create(sfe_matcher *m, int n_words, sfe_bowdb **out) {
    SFE_REQUIRE(m && out && n_words >= 1, SFE_ERR_BAD_ARG, "bad argument");
    DeviceGuard g(m->device);
    SFE_REQUIRE(g.ok, SFE_ERR_NO_DEVICE, "cannot select the handle's device");
    sfe_bowdb *db = new sfe_bowdb();
    db->device = m->device;
    db->n_words = n_words;
    db->cap_entries = 64;
    cudaError_t e = cudaMalloc((void **)&db->off, sizeof(int64_t) * (db->cap_entries + 1));
    if (e == cudaSuccess) e = cudaMemset(db->off, 0, sizeof(int64_t));
    if (e == cudaSuccess) e = cudaDeviceSynchronize();
    if (e != cudaSuccess) {
        set_error("BoW database: %s", cudaGetErrorString(e));
        if (db->off) cudaFree(db->off);
        delete db;
        return SFE_ERR_CUDA;
    }
    *out = db;
    return SFE_OK;
}

int sfe_bowdb_destroy(sfe_bowdb *db) {
    if (!db) return SFE_OK;
    DeviceGuard g(db->device);
    SFE_REQUIRE(g.ok, SFE_ERR_NO_DEVICE, "cannot select the handle's device");
    for (auto &r : db->readers) {
        cudaEventSynchronize(r.second);
        cudaEventDestroy(r.second);
    }
    cudaFree(db->off);
    if (db->ids) cudaFree(db->ids);
    if (db->val) cudaFree(db->val);
    delete db;
    return SFE_OK;
}

int sfe_bowdb_size(const sfe_bowdb *db, int *entries) {
    SFE_REQUIRE(db && entries, SFE_ERR_BAD_ARG, "null argument");
    std::lock_guard<std::mutex> lock(db->mu);
    *entries = db->size;
    return SFE_OK;
}

// Room for `count` more entries of `add_nnz` more words; the caller holds db->mu.  Capacity doubling: an add costs amortised
// O(its own size).  The old buffers may still be read by queries enqueued on other streams, so they are freed only once
// those have run.  On failure the database keeps its old buffers and contents.
static int bow_reserve(sfe_bowdb *db, cudaStream_t st, int count, int64_t add_nnz) {
    const int64_t need_e = (int64_t)db->size + count, need_nnz = db->nnz + add_nnz;
    int64_t *off = db->off;
    int32_t *wid = db->ids;
    double *val = db->val;
    int64_t cap_e = db->cap_entries, cap_n = db->cap_nnz;
    if (need_e <= cap_e && need_nnz <= cap_n) return SFE_OK;
    for (auto &r : db->readers) SFE_CUDA(cudaEventSynchronize(r.second));
    if (need_e > cap_e) cap_e = std::max(need_e, 2 * cap_e);
    if (need_nnz > cap_n) cap_n = std::max(need_nnz, 2 * cap_n);
    cudaError_t e = cudaSuccess;
    if (cap_e != db->cap_entries) e = cudaMalloc((void **)&off, sizeof(int64_t) * (cap_e + 1));
    if (e == cudaSuccess && cap_n != db->cap_nnz) {
        wid = nullptr;
        val = nullptr;
        e = cudaMalloc((void **)&wid, sizeof(int32_t) * cap_n);
        if (e == cudaSuccess) e = cudaMalloc((void **)&val, sizeof(double) * cap_n);
    }
    if (e == cudaSuccess && off != db->off)
        e = cudaMemcpyAsync(off, db->off, sizeof(int64_t) * (db->size + 1), cudaMemcpyDeviceToDevice, st);
    if (e == cudaSuccess && wid != db->ids && db->nnz > 0) {
        e = cudaMemcpyAsync(wid, db->ids, sizeof(int32_t) * db->nnz, cudaMemcpyDeviceToDevice, st);
        if (e == cudaSuccess) e = cudaMemcpyAsync(val, db->val, sizeof(double) * db->nnz, cudaMemcpyDeviceToDevice, st);
    }
    if (e == cudaSuccess) e = cudaStreamSynchronize(st);
    if (e != cudaSuccess) {
        if (off != db->off) cudaFree(off);
        if (wid != db->ids && wid) cudaFree(wid);
        if (val != db->val && val) cudaFree(val);
        set_error("BoW database growth: %s", cudaGetErrorString(e));
        return SFE_ERR_CUDA;
    }
    if (off != db->off) cudaFree(db->off);
    if (wid != db->ids && db->ids) cudaFree(db->ids);
    if (val != db->val && db->val) cudaFree(db->val);
    db->off = off; db->ids = wid; db->val = val;
    db->cap_entries = cap_e; db->cap_nnz = cap_n;
    return SFE_OK;
}

// Vectors in device memory, checked there (bow_check_kernel) with the host check's rules -> their nnz and longest vector.
static int bow_check_vectors_dev(sfe_matcher *m, const int64_t *off, const int32_t *ids, const double *val, int count, int n_words,
                                 int64_t *nnz, int *max_len) {
    SFE_CUDA(m->d_bow_chk.ensure(3));
    SFE_CUDA(launch_bow_check(m->stream, off, ids, val, count, n_words, m->d_bow_chk.p));
    m->launches++;
    unsigned long long chk[3];
    SFE_CUDA(cudaMemcpyAsync(chk, m->d_bow_chk.p, sizeof(chk), cudaMemcpyDeviceToHost, m->stream));
    SFE_CUDA(cudaStreamSynchronize(m->stream));
    SFE_REQUIRE(chk[1] == 0, SFE_ERR_BAD_ARG, "offsets[0] != 0, decreasing offsets, a word id outside [0, n_words) or not "
                                              "strictly ascending within a vector, or a value that is not finite");
    *nnz = (int64_t)chk[0];
    SFE_REQUIRE(*nnz == 0 || (ids && val), SFE_ERR_BAD_ARG, "null ids / values");
    *max_len = (int)std::min<unsigned long long>(chk[2], INT32_MAX);
    return SFE_OK;
}

int sfe_bowdb_add(sfe_matcher *m, sfe_bowdb *db, const int64_t *offsets, const int32_t *ids, const double *values, int count,
                  int32_t *first_entry) {
    SFE_REQUIRE(m && db && count >= 0, SFE_ERR_BAD_ARG, "bad argument");
    SFE_REQUIRE(db->device == m->device, SFE_ERR_BAD_ARG, "database lives on another device");
    int rc = bow_check_vectors(offsets, ids, values, count, db->n_words);
    if (rc != SFE_OK) return rc;
    DeviceGuard g(m->device);
    SFE_REQUIRE(g.ok, SFE_ERR_NO_DEVICE, "cannot select the handle's device");
    std::lock_guard<std::mutex> lock(db->mu);
    SFE_REQUIRE((int64_t)db->size + count < INT32_MAX, SFE_ERR_UNSUPPORTED, "entry ids must fit int32");
    const int32_t first = db->size;
    if (count > 0) {
        cudaStream_t st = m->stream;
        const int64_t add_nnz = offsets[count];
        rc = bow_reserve(db, st, count, add_nnz);
        if (rc != SFE_OK) return rc;
        std::vector<int64_t> o(count);  // the new entries' end offsets in the database's forward file
        for (int i = 0; i < count; i++) o[i] = db->nnz + offsets[i + 1];
        SFE_CUDA(cudaMemcpyAsync(db->off + db->size + 1, o.data(), sizeof(int64_t) * count, cudaMemcpyHostToDevice, st));
        if (add_nnz > 0) {
            SFE_CUDA(cudaMemcpyAsync(db->ids + db->nnz, ids, sizeof(int32_t) * add_nnz, cudaMemcpyHostToDevice, st));
            SFE_CUDA(cudaMemcpyAsync(db->val + db->nnz, values, sizeof(double) * add_nnz, cudaMemcpyHostToDevice, st));
        }
        SFE_CUDA(cudaStreamSynchronize(st));  // synchronous: every stream's later query sees the new entries
        db->size += count;
        db->nnz += add_nnz;
    }
    if (first_entry) *first_entry = first;
    return SFE_OK;
}

// Enqueues the scoring of q query vectors (CSR in device memory, the longest max_nq words) under the database's lock: the
// top-k rows go to entry / score / n_results (device), the dense rows are copied to `dense` with `dense_kind`, and the
// stream's reader event is recorded behind them.
static int bow_query_enqueue(sfe_matcher *m, const sfe_bowdb *db, const int64_t *q_off, const int32_t *q_ids, const double *q_val,
                             int q, int max_nq, int max_id, int max_results, int32_t *entry, double *score, int32_t *n_results,
                             double *dense, int dense_entries, cudaMemcpyKind dense_kind) {
    cudaStream_t st = m->stream;
    std::lock_guard<std::mutex> lock(db->mu);  // the entry count and the buffers this query reads
    const int size = db->size;
    SFE_REQUIRE(!dense || dense_entries <= size, SFE_ERR_BAD_ARG, "dense_entries exceeds the database's entry count");
    const int n_eff = max_id == -1 ? size : (max_id < 0 ? 0 : std::min(max_id, size));  // (int)e < max_id || max_id == -1
    const int n_score = std::max(n_eff, dense ? dense_entries : 0);
    // queries in batches whose raw sums (+ hit flags, + dense scores) stay within 256 MB of scratch
    const size_t per_query = (size_t)std::max(n_score, 1) * (9 + (dense ? 8 : 0));
    const int qb = (int)std::max<size_t>(1, std::min<size_t>(std::min(q, 65535), ((size_t)256 << 20) / per_query));  // grid.y
    SFE_CUDA(m->d_bow_raw.ensure((size_t)qb * std::max(n_score, 1)));
    SFE_CUDA(m->d_bow_hit.ensure((size_t)qb * std::max(n_score, 1)));
    if (dense) SFE_CUDA(m->d_bow_dense.ensure((size_t)qb * std::max(n_score, 1)));
    for (int i0 = 0; i0 < q; i0 += qb) {
        const int nb = std::min(qb, q - i0);
        SFE_CUDA(launch_bow_score(st, q_off + i0, q_ids, q_val, nb, max_nq, db->off, db->ids, db->val, n_score, n_score,
                                  m->d_bow_raw.p, m->d_bow_hit.p, dense ? m->d_bow_dense.p : nullptr));
        SFE_CUDA(launch_bow_topk(st, m->d_bow_raw.p, m->d_bow_hit.p, n_score, nb, n_eff, max_results, entry + (size_t)i0 * max_results,
                                 score + (size_t)i0 * max_results, n_results + i0));
        m->launches += 2;
        if (dense && dense_entries > 0)
            SFE_CUDA(cudaMemcpy2DAsync(dense + (size_t)i0 * dense_entries, sizeof(double) * dense_entries, m->d_bow_dense.p,
                                       sizeof(double) * n_score, sizeof(double) * dense_entries, nb, dense_kind, st));
    }
    cudaEvent_t *ev = nullptr;
    for (auto &r : db->readers)
        if (r.first == st) ev = &r.second;
    if (!ev) {
        cudaEvent_t e = nullptr;
        SFE_CUDA(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
        db->readers.emplace_back(st, e);
        ev = &db->readers.back().second;
    }
    SFE_CUDA(cudaEventRecord(*ev, st));
    return SFE_OK;
}

int sfe_bowdb_query(sfe_matcher *m, const sfe_bowdb *db, const int64_t *offsets, const int32_t *ids, const double *values, int q,
                    int max_id, int max_results, int32_t *entry, double *score, int32_t *n_results, double *dense,
                    int dense_entries) {
    SFE_REQUIRE(m && db && q >= 0, SFE_ERR_BAD_ARG, "bad argument");
    SFE_REQUIRE(db->device == m->device, SFE_ERR_BAD_ARG, "database lives on another device");
    SFE_REQUIRE(max_results >= 1, SFE_ERR_BAD_ARG, "max_results must be >= 1 (the score against every entry is `dense`)");
    SFE_REQUIRE(max_results <= SFE_BOWDB_MAX_RESULTS, SFE_ERR_UNSUPPORTED, "max_results above SFE_BOWDB_MAX_RESULTS");
    SFE_REQUIRE(!dense || dense_entries >= 0, SFE_ERR_BAD_ARG, "negative dense_entries");
    if (q == 0) return SFE_OK;
    SFE_REQUIRE(entry && score && n_results, SFE_ERR_BAD_ARG, "null argument");
    int rc = bow_check_vectors(offsets, ids, values, q, db->n_words);
    if (rc != SFE_OK) return rc;
    DeviceGuard g(m->device);
    SFE_REQUIRE(g.ok, SFE_ERR_NO_DEVICE, "cannot select the handle's device");
    cudaStream_t st = m->stream;
    const int64_t qnnz = offsets[q];
    int max_nq = 0;
    for (int i = 0; i < q; i++) max_nq = std::max(max_nq, (int)(offsets[i + 1] - offsets[i]));
    SFE_CUDA(m->d_bow_off.ensure(q + 1));
    SFE_CUDA(m->d_bow_ids.ensure(std::max<int64_t>(qnnz, 1)));
    SFE_CUDA(m->d_bow_val.ensure(std::max<int64_t>(qnnz, 1)));
    SFE_CUDA(m->d_bow_e.ensure((size_t)q * max_results));
    SFE_CUDA(m->d_bow_s.ensure((size_t)q * max_results));
    SFE_CUDA(m->d_bow_n.ensure(q));
    SFE_CUDA(cudaMemcpyAsync(m->d_bow_off.p, offsets, sizeof(int64_t) * (q + 1), cudaMemcpyHostToDevice, st));
    if (qnnz > 0) {
        SFE_CUDA(cudaMemcpyAsync(m->d_bow_ids.p, ids, sizeof(int32_t) * qnnz, cudaMemcpyHostToDevice, st));
        SFE_CUDA(cudaMemcpyAsync(m->d_bow_val.p, values, sizeof(double) * qnnz, cudaMemcpyHostToDevice, st));
    }
    rc = bow_query_enqueue(m, db, m->d_bow_off.p, m->d_bow_ids.p, m->d_bow_val.p, q, max_nq, max_id, max_results, m->d_bow_e.p,
                           m->d_bow_s.p, m->d_bow_n.p, dense, dense_entries, cudaMemcpyDeviceToHost);
    if (rc != SFE_OK) return rc;
    SFE_CUDA(cudaMemcpyAsync(entry, m->d_bow_e.p, sizeof(int32_t) * q * max_results, cudaMemcpyDeviceToHost, st));
    SFE_CUDA(cudaMemcpyAsync(score, m->d_bow_s.p, sizeof(double) * q * max_results, cudaMemcpyDeviceToHost, st));
    SFE_CUDA(cudaMemcpyAsync(n_results, m->d_bow_n.p, sizeof(int32_t) * q, cudaMemcpyDeviceToHost, st));
    SFE_CUDA(cudaStreamSynchronize(st));
    return SFE_OK;
}

// add / query with the vectors (and query's results) in device memory: validated there, then the host calls' paths
int sfe_bowdb_add_dev(sfe_matcher *m, sfe_bowdb *db, const int64_t *offsets_dev, const int32_t *ids_dev, const double *values_dev,
                      int count, int32_t *first_entry) {
    SFE_REQUIRE(m && db && count >= 0, SFE_ERR_BAD_ARG, "bad argument");
    SFE_REQUIRE(db->device == m->device, SFE_ERR_BAD_ARG, "database lives on another device");
    SFE_REQUIRE(offsets_dev, SFE_ERR_BAD_ARG, "null offsets");
    DeviceGuard g(m->device);
    SFE_REQUIRE(g.ok, SFE_ERR_NO_DEVICE, "cannot select the handle's device");
    int64_t add_nnz = 0;
    int max_len = 0;
    int rc = bow_check_vectors_dev(m, offsets_dev, ids_dev, values_dev, count, db->n_words, &add_nnz, &max_len);
    if (rc != SFE_OK) return rc;
    std::lock_guard<std::mutex> lock(db->mu);
    SFE_REQUIRE((int64_t)db->size + count < INT32_MAX, SFE_ERR_UNSUPPORTED, "entry ids must fit int32");
    const int32_t first = db->size;
    if (count > 0) {
        cudaStream_t st = m->stream;
        rc = bow_reserve(db, st, count, add_nnz);
        if (rc != SFE_OK) return rc;
        SFE_CUDA(launch_bow_rebase(st, offsets_dev, count, db->nnz, db->off + db->size + 1));
        m->launches++;
        if (add_nnz > 0) {
            SFE_CUDA(cudaMemcpyAsync(db->ids + db->nnz, ids_dev, sizeof(int32_t) * add_nnz, cudaMemcpyDeviceToDevice, st));
            SFE_CUDA(cudaMemcpyAsync(db->val + db->nnz, values_dev, sizeof(double) * add_nnz, cudaMemcpyDeviceToDevice, st));
        }
        SFE_CUDA(cudaStreamSynchronize(st));  // synchronous: every stream's later query sees the new entries
        db->size += count;
        db->nnz += add_nnz;
    }
    if (first_entry) *first_entry = first;
    return SFE_OK;
}

int sfe_bowdb_query_dev(sfe_matcher *m, const sfe_bowdb *db, const int64_t *offsets_dev, const int32_t *ids_dev,
                        const double *values_dev, int q, int max_id, int max_results, int32_t *entry_dev, double *score_dev,
                        int32_t *n_results_dev, double *dense_dev, int dense_entries) {
    SFE_REQUIRE(m && db && q >= 0, SFE_ERR_BAD_ARG, "bad argument");
    SFE_REQUIRE(db->device == m->device, SFE_ERR_BAD_ARG, "database lives on another device");
    SFE_REQUIRE(max_results >= 1, SFE_ERR_BAD_ARG, "max_results must be >= 1 (the score against every entry is `dense`)");
    SFE_REQUIRE(max_results <= SFE_BOWDB_MAX_RESULTS, SFE_ERR_UNSUPPORTED, "max_results above SFE_BOWDB_MAX_RESULTS");
    SFE_REQUIRE(!dense_dev || dense_entries >= 0, SFE_ERR_BAD_ARG, "negative dense_entries");
    if (q == 0) return SFE_OK;
    SFE_REQUIRE(entry_dev && score_dev && n_results_dev && offsets_dev, SFE_ERR_BAD_ARG, "null argument");
    DeviceGuard g(m->device);
    SFE_REQUIRE(g.ok, SFE_ERR_NO_DEVICE, "cannot select the handle's device");
    int64_t qnnz = 0;
    int max_nq = 0;
    int rc = bow_check_vectors_dev(m, offsets_dev, ids_dev, values_dev, q, db->n_words, &qnnz, &max_nq);
    if (rc != SFE_OK) return rc;
    rc = bow_query_enqueue(m, db, offsets_dev, ids_dev, values_dev, q, max_nq, max_id, max_results, entry_dev, score_dev,
                           n_results_dev, dense_dev, dense_entries, cudaMemcpyDeviceToDevice);
    if (rc != SFE_OK) return rc;
    SFE_CUDA(cudaStreamSynchronize(m->stream));
    return SFE_OK;
}

int sfe_db_create(sfe_matcher *m, const uint8_t *desc_host, int64_t rows, int64_t idx_base, sfe_db **out) {
    SFE_REQUIRE(m && out && rows >= 0 && idx_base >= 0, SFE_ERR_BAD_ARG, "bad argument");
    SFE_REQUIRE(rows == 0 || desc_host, SFE_ERR_BAD_ARG, "null argument");
    SFE_REQUIRE(idx_base + rows < (1ll << 31), SFE_ERR_UNSUPPORTED, "global row index must fit int32");
    DeviceGuard g(m->device);
    SFE_REQUIRE(g.ok, SFE_ERR_NO_DEVICE, "cannot select the handle's device");
    sfe_db *db = new sfe_db();
    db->device = m->device;
    db->rows = rows;
    db->idx_base = idx_base;
    cudaError_t e = cudaMalloc((void **)&db->rows_dev, std::max<size_t>((size_t)rows * 32, 32));
    if (e == cudaSuccess && rows > 0) e = cudaMemcpy(db->rows_dev, desc_host, (size_t)rows * 32, cudaMemcpyHostToDevice);
    if (e != cudaSuccess) {
        set_error("database upload: %s", cudaGetErrorString(e));
        if (db->rows_dev) cudaFree(db->rows_dev);
        delete db;
        return SFE_ERR_CUDA;
    }
    *out = db;
    return SFE_OK;
}

int sfe_db_destroy(sfe_db *db) {
    if (!db) return SFE_OK;
    DeviceGuard g(db->device);
    SFE_REQUIRE(g.ok, SFE_ERR_NO_DEVICE, "cannot select the handle's device");
    cudaFree(db->rows_dev);
    if (db->tiles_dev) cudaFree(db->tiles_dev);
    if (db->tiles_ready) cudaEventDestroy(db->tiles_ready);
    delete db;
    return SFE_OK;
}

int sfe_knn2_dev(sfe_matcher *m, const sfe_db *db, const uint8_t *queries_dev, int q, uint64_t *keys_dev) {
    SFE_REQUIRE(m && db && queries_dev && keys_dev && q >= 1, SFE_ERR_BAD_ARG, "bad argument");
    SFE_REQUIRE(db->device == m->device, SFE_ERR_BAD_ARG, "database lives on another device");
    DeviceGuard g(m->device);
    SFE_REQUIRE(g.ok, SFE_ERR_NO_DEVICE, "cannot select the handle's device");
    int rc = knn_partial(m, db, queries_dev, q, (unsigned long long *)keys_dev, nullptr);
    if (rc != SFE_OK) return rc;
    if (!m->async_dev) SFE_CUDA(cudaStreamSynchronize(m->stream));
    return SFE_OK;
}

int sfe_knn2_merge_dev(sfe_matcher *m, const uint64_t *keys_dev, int shards, int q, int32_t *out_dev) {
    SFE_REQUIRE(m && keys_dev && out_dev && shards >= 1 && q >= 1, SFE_ERR_BAD_ARG, "bad argument");
    DeviceGuard g(m->device);
    SFE_REQUIRE(g.ok, SFE_ERR_NO_DEVICE, "cannot select the handle's device");
    knn2_merge_kernel<<<div_up(q, 4), 128, 0, m->stream>>>((const unsigned long long *)keys_dev, shards, q, nullptr, out_dev);
    m->launches++;
    SFE_CUDA(cudaGetLastError());
    if (!m->async_dev) SFE_CUDA(cudaStreamSynchronize(m->stream));
    return SFE_OK;
}

int sfe_knn2(sfe_matcher *m, const sfe_db *db, const uint8_t *queries, int q, int32_t *out) {
    SFE_REQUIRE(m && db && queries && out && q >= 1, SFE_ERR_BAD_ARG, "bad argument");
    SFE_REQUIRE(db->device == m->device, SFE_ERR_BAD_ARG, "database lives on another device");
    DeviceGuard g(m->device);
    SFE_REQUIRE(g.ok, SFE_ERR_NO_DEVICE, "cannot select the handle's device");
    cudaStream_t st = m->stream;
    SFE_CUDA(m->d_dl.ensure((size_t)q * 32));
    SFE_CUDA(m->d_quad.ensure((size_t)q * 4));
    SFE_CUDA(cudaMemcpyAsync(m->d_dl.p, queries, (size_t)q * 32, cudaMemcpyHostToDevice, st));
    int rc = knn_partial(m, db, m->d_dl.p, q, nullptr, m->d_quad.p);
    if (rc != SFE_OK) return rc;
    SFE_CUDA(cudaMemcpyAsync(out, m->d_quad.p, sizeof(int32_t) * 4 * q, cudaMemcpyDeviceToHost, st));
    SFE_CUDA(cudaStreamSynchronize(st));
    return SFE_OK;
}


// ---- multi-GPU exchange: handles and collectives (SURVEY §8e) ---------------------------------------------------------
struct sfe_comm {
    int device = 0, rank = 0, world = 1;
    uint8_t *inbox = nullptr;             // local inbox (cudaMalloc)
    size_t inbox_bytes = 0;
    uint8_t *base[kMaxWorld] = {};        // every rank's inbox as mapped in this process
    bool ipc_mapped[kMaxWorld] = {};
    bool connected = false;
    uint32_t epoch = 0;
};

static size_t comm_inbox_bytes(int world) { return 2 * (size_t)world * kCommSlotBytes + sizeof(uint32_t) * (2 * kMaxWorld + 2); }

static int comm_alloc(int device, int rank, int world, sfe_comm **out) {
    DeviceGuard g(device);
    SFE_REQUIRE(g.ok, SFE_ERR_NO_DEVICE, "cannot select the device");
    sfe_comm *c = new sfe_comm();
    c->device = device; c->rank = rank; c->world = world;
    c->inbox_bytes = comm_inbox_bytes(world);
    cudaError_t e = cudaMalloc((void **)&c->inbox, c->inbox_bytes);
    if (e == cudaSuccess) e = cudaMemset(c->inbox, 0, c->inbox_bytes);
    if (e != cudaSuccess) {
        set_error("sfe_comm: inbox allocation: %s", cudaGetErrorString(e));
        if (c->inbox) cudaFree(c->inbox);
        delete c;
        return SFE_ERR_CUDA;
    }
    c->base[rank] = c->inbox;
    c->connected = world == 1;
    *out = c;
    return SFE_OK;
}

static CommView comm_view(sfe_comm *c) {
    CommView V{};
    for (int r = 0; r < c->world; r++) V.base[r] = c->base[r];
    V.rank = c->rank; V.world = c->world; V.epoch = c->epoch;
    return V;
}

int sfe_comm_create(int device, int rank, int world, sfe_comm **out) {
    SFE_REQUIRE(out && world >= 1 && world <= kMaxWorld && rank >= 0 && rank < world, SFE_ERR_BAD_ARG, "bad rank / world (world <= 16)");
    int ndev = 0;
    SFE_CUDA(cudaGetDeviceCount(&ndev));
    SFE_REQUIRE(device >= 0 && device < ndev, SFE_ERR_BAD_ARG, "device index out of range");
    return comm_alloc(device, rank, world, out);
}

int sfe_comm_export(sfe_comm *c, uint8_t handle[SFE_COMM_HANDLE_BYTES]) {
    SFE_REQUIRE(c && handle, SFE_ERR_BAD_ARG, "null argument");
    static_assert(sizeof(cudaIpcMemHandle_t) <= SFE_COMM_HANDLE_BYTES, "IPC handle larger than the ABI's handle");
    DeviceGuard g(c->device);
    SFE_REQUIRE(g.ok, SFE_ERR_NO_DEVICE, "cannot select the handle's device");
    cudaIpcMemHandle_t h;
    SFE_CUDA(cudaIpcGetMemHandle(&h, c->inbox));
    memset(handle, 0, SFE_COMM_HANDLE_BYTES);
    memcpy(handle, &h, sizeof(h));
    return SFE_OK;
}

int sfe_comm_connect(sfe_comm *c, const uint8_t *handles) {
    SFE_REQUIRE(c && (handles || c->world == 1), SFE_ERR_BAD_ARG, "null argument");
    DeviceGuard g(c->device);
    SFE_REQUIRE(g.ok, SFE_ERR_NO_DEVICE, "cannot select the handle's device");
    for (int r = 0; r < c->world; r++) {
        if (r == c->rank || c->base[r]) continue;
        cudaIpcMemHandle_t h;
        memcpy(&h, handles + (size_t)r * SFE_COMM_HANDLE_BYTES, sizeof(h));
        void *p = nullptr;
        cudaError_t e = cudaIpcOpenMemHandle(&p, h, cudaIpcMemLazyEnablePeerAccess);
        if (e != cudaSuccess) {
            set_error("sfe_comm_connect: rank %d's inbox cannot be mapped (%s): the GPUs need peer access (NVLink / PCIe P2P)", r,
                      cudaGetErrorString(e));
            cudaGetLastError();
            return SFE_ERR_CUDA;
        }
        c->base[r] = (uint8_t *)p;
        c->ipc_mapped[r] = true;
    }
    c->connected = true;
    return SFE_OK;
}

int sfe_comm_create_local(const int *devices, int n, sfe_comm **out) {
    SFE_REQUIRE(devices && out && n >= 1 && n <= kMaxWorld, SFE_ERR_BAD_ARG, "bad argument (at most 16 devices)");
    for (int i = 0; i < n; i++) out[i] = nullptr;
    for (int i = 0; i < n; i++) {
        int rc = comm_alloc(devices[i], i, n, &out[i]);
        if (rc != SFE_OK) {
            for (int j = 0; j < i; j++) { sfe_comm_destroy(out[j]); out[j] = nullptr; }
            return rc;
        }
    }
    for (int i = 0; i < n; i++) {
        DeviceGuard g(devices[i]);
        for (int j = 0; j < n; j++) {
            if (devices[j] != devices[i]) {
                int can = 0;
                cudaDeviceCanAccessPeer(&can, devices[i], devices[j]);
                cudaError_t e = can ? cudaDeviceEnablePeerAccess(devices[j], 0) : cudaErrorPeerAccessUnsupported;
                if (e == cudaErrorPeerAccessAlreadyEnabled) { cudaGetLastError(); e = cudaSuccess; }
                if (e != cudaSuccess) {
                    set_error("sfe_comm_create_local: device %d cannot access device %d (%s)", devices[i], devices[j], cudaGetErrorString(e));
                    for (int k = 0; k < n; k++) { sfe_comm_destroy(out[k]); out[k] = nullptr; }
                    return SFE_ERR_UNSUPPORTED;
                }
            }
            out[i]->base[j] = out[j]->inbox;
        }
        out[i]->connected = true;
    }
    return SFE_OK;
}

int sfe_comm_destroy(sfe_comm *c) {
    if (!c) return SFE_OK;
    DeviceGuard g(c->device);
    cudaDeviceSynchronize();
    for (int r = 0; r < c->world; r++)
        if (c->ipc_mapped[r]) cudaIpcCloseMemHandle(c->base[r]);
    if (c->inbox) cudaFree(c->inbox);
    delete c;
    return SFE_OK;
}

int sfe_comm_status(sfe_comm *c, int *stalled_rank) {
    SFE_REQUIRE(c, SFE_ERR_BAD_ARG, "null handle");
    DeviceGuard g(c->device);
    SFE_REQUIRE(g.ok, SFE_ERR_NO_DEVICE, "cannot select the handle's device");
    uint32_t st = 0;
    SFE_CUDA(cudaMemcpy(&st, c->inbox + 2 * (size_t)c->world * kCommSlotBytes + sizeof(uint32_t) * (2 * kMaxWorld + 1), sizeof(st),
                        cudaMemcpyDeviceToHost));
    if (stalled_rank) *stalled_rank = st ? (int)st - 1 : -1;
    if (st) {
        set_error("sfe_comm: rank %u never delivered its part of a collective (5 s); results of that call are invalid", st - 1);
        return SFE_ERR_CUDA;
    }
    return SFE_OK;
}

static int comm_check(sfe_matcher *m, sfe_comm *c) {
    SFE_REQUIRE(m && c, SFE_ERR_BAD_ARG, "null handle");
    SFE_REQUIRE(c->connected, SFE_ERR_BAD_ARG, "sfe_comm is not connected (sfe_comm_connect)");
    SFE_REQUIRE(c->device == m->device, SFE_ERR_BAD_ARG, "communicator and matcher live on different devices");
    return SFE_OK;
}

int sfe_knn2_sharded(sfe_matcher *m, sfe_comm *c, const sfe_db *shard, const uint8_t *queries_dev, int q, int32_t *out_dev) {
    int rc = comm_check(m, c);
    if (rc != SFE_OK) return rc;
    SFE_REQUIRE(shard && queries_dev && out_dev && q >= 1, SFE_ERR_BAD_ARG, "bad argument");
    SFE_REQUIRE((size_t)q * 16 <= kCommSlotBytes, SFE_ERR_UNSUPPORTED, "more than 32768 queries per sharded call");
    SFE_REQUIRE(shard->device == m->device, SFE_ERR_BAD_ARG, "database shard lives on another device");
    DeviceGuard g(m->device);
    SFE_REQUIRE(g.ok, SFE_ERR_NO_DEVICE, "cannot select the handle's device");
    if (c->world == 1) return knn_partial(m, shard, queries_dev, q, nullptr, out_dev);  // nothing to exchange
    c->epoch++;
    const CommView V = comm_view(c);
    if ((rc = knn_partial(m, shard, queries_dev, q, nullptr, nullptr, &V)) != SFE_OK) return rc;
    knn2_gather_merge_kernel<<<div_up(q, 128), 128, 0, m->stream>>>(V, q, out_dev);
    m->launches++;
    SFE_CUDA(cudaGetLastError());
    return SFE_OK;
}

int sfe_projection_match_sharded(sfe_matcher *m, sfe_comm *c, const sfe_frame *f, const double *xw_dev, const uint8_t *mp_desc_dev,
                                 const uint8_t *skip_dev, int n, int64_t idx_base, const sfe_se3 *Tcw, double radius,
                                 double best12_threshold, int32_t *kp_to_query_dev, int32_t *kp_dist_dev) {
    int rc = comm_check(m, c);
    if (rc != SFE_OK) return rc;
    SFE_REQUIRE(f && Tcw && kp_to_query_dev && n >= 0 && (n == 0 || (xw_dev && mp_desc_dev)), SFE_ERR_BAD_ARG, "bad argument");
    SFE_REQUIRE(f->device == m->device, SFE_ERR_BAD_ARG, "frame lives on another device");
    SFE_REQUIRE(f->n >= 1, SFE_ERR_BAD_ARG, "empty frame");
    SFE_REQUIRE(idx_base >= 0 && idx_base + n < (1ll << 31), SFE_ERR_UNSUPPORTED, "global map-point index must fit int32");
    DeviceGuard g(m->device);
    SFE_REQUIRE(g.ok, SFE_ERR_NO_DEVICE, "cannot select the handle's device");
    c->epoch++;
    const CommView V = comm_view(c);
    // the shard's per-keypoint keys are built directly in this rank's own inbox slot, then pushed to the peers
    unsigned long long *own = (unsigned long long *)(c->inbox + ((size_t)(c->epoch & 1) * c->world + c->rank) * kCommSlotBytes);
    const int m16 = (f->n + 1) / 2;  // 16-byte units; the odd tail key is padding inside the slot
    if ((rc = projection_impl(m, xw_dev, mp_desc_dev, skip_dev, n, pose_from_se3(Tcw), &f->cam, f->kps.p, f->desc.p, f->n, radius,
                              best12_threshold, nullptr, nullptr, (uint32_t)idx_base, own, &f->grid)) != SFE_OK)
        return rc;
    if (c->world > 1) {
        comm_push_kernel<<<std::min(div_up(m16, 256), 64), 256, 0, m->stream>>>(V, m16);
        m->launches++;
    }
    if (c->world > 1)
        projection_gather_decode_kernel<<<div_up(f->n, 256), 256, 0, m->stream>>>(V, f->n, kp_to_query_dev, kp_dist_dev);
    else
        projection_decode_kernel<<<div_up(f->n, 256), 256, 0, m->stream>>>(f->n, 1, own, kp_to_query_dev, kp_dist_dev);
    m->launches++;
    SFE_CUDA(cudaGetLastError());
    return SFE_OK;
}

}  // extern "C"
