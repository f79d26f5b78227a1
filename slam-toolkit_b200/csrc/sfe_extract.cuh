// Internal layout shared by the extraction kernels and the extractor handle.
#pragma once
#include "sfe_common.cuh"
#include "sfe_tma.cuh"

namespace sfe {

constexpr int kMaxLevels = 16;
constexpr int kEdge = 19;          // EDGE_THRESHOLD, reference src/orb_extractor.cpp:74
constexpr int kBorder = kEdge - 3; // minBorderX/Y of the FAST window, :771-772
constexpr int kHalfPatch = 15;     // HALF_PATCH_SIZE, :73
constexpr int kMaxSub = 66;        // largest FAST cell sub-image side (wCell + 6 < 60 + 6)
constexpr int kNarrowCandCap = 60000;   // per level: up to here the quadtree indexes candidates with 16 bits (up to 3072 of them in
                                        // shared memory, 14 B each; fuller levels in a global scratch slot)
constexpr int kMaxCandCap = 1 << 22;    // hard limit of a level's candidate buffer: non-max-suppressed corners cannot be 8-neighbours,
                                        // so a 4096 x 4096 window holds at most 2^22 of them; above kNarrowCandCap the quadtree runs
                                        // its 32-bit instance
constexpr int kBlurTileW = 128, kBlurTileH = 32;
constexpr int kBlurInWords = 40;   // shared-memory row of a blur input tile: x0-16 .. x0+143 (a TMA box starts and ends on 16-byte
                                   // multiples of the row: the innermost coordinate must be 16-byte aligned)
constexpr int kBlurLead = 16;      // bytes of a tile row before output column 0

// One pyramid level's geometry for the current image size (host-built, mirrored on device).
struct LevelPlan {
    int w, h, pitch;        // level size; row pitch of levels >= 1 in the pyramid buffer
    int plane_off;          // byte offset of this level inside one image's pyramid buffer (l >= 1)
    int blur_pitch, blur_off;
    int win_w, win_h;       // FAST window maxBorder - minBorder, :773-781
    int n_cols, n_rows, w_cell, h_cell;  // :784-787
    int quota;              // mnFeaturesPerLevel, :435-446
    int n_ini;              // quadtree roots, :543
    float hx;               // root width, :545
    int ff_depth;           // quadtree passes whose outcome is written directly (octree_build_at_depth); 0 = start from the roots
    int cand_cap, cand_off; // FAST candidate slots of this level inside one image's array
    int kp_cap, kp_off;     // quadtree survivor slots
    int xtab_off, ytab_off; // resize tables that PRODUCE this level from level-1
    float scale;            // mvScaleFactor[level]
    float size;             // (int)(31 * scale), :837
};

// FAST segments.  One reference cv::FAST call = one 30-px grid cell (:789-816); cells that pass the skip rules
// (:794,803) and hold at least a 7x7 sub-image are grouped, along their cell row, into segments of up to 128 tested
// pixels (the tested regions of neighbouring cells tile the row without gaps or overlap).  One CTA runs one segment:
// the per-pixel work does not care about cells, only the non-max suppression and the 20 -> 7 retry are per cell.
struct SegRec {
    short ini_x, ini_y;            // iniX of the first cell, iniY of the cell row (level pixels)
    short tw;                      // tested pixels across the segment = sum over its cells of (sub-image width - 6)
    unsigned char sh, level;       // sub-image height handed to cv::FAST (<= kMaxSub)
    unsigned char n_cells, w_cell; // every cell tests w_cell columns, the last one of a row possibly fewer
    unsigned short inv_w;          // x / w_cell == (x * inv_w) >> 16 for x < 256
    unsigned int pad;              // 16 bytes: the kernel fetches a record with one 128-bit load
};
static_assert(sizeof(SegRec) == 16, "SegRec is loaded as one uint4");
struct FastLevel {
    int pitch, plane_off;  // level pixels (levels >= 1; level 0 is the input image)
    int cand_off, cand_cap;
};
struct FastPlan {
    FastLevel lv[kMaxLevels];
    int nlevels, n_cells, n_segs;
    int ini_th, min_th;
    int tile_rows, score_rows, list_cap;  // dynamic shared-memory carve-up, sized for the largest segment
};
constexpr int kFastThreads = 256;
constexpr int kFastCtasPerSm = 5;    // register budget: 64 K / (5 x 256) = 51 per thread (6 CTAs = 40 registers measured slower)
#ifndef SFE_FAST_TILE_PITCH
#define SFE_FAST_TILE_PITCH 176
#endif
constexpr int kFastTilePitch = SFE_FAST_TILE_PITCH;  // bytes: first tested column at 7..22, 128 tested px, 3 px + one word beyond (>= 160,
                                                     // multiple of 16: the row of a TMA box)
constexpr int kFastScorePitch = 144; // 128 tested px + 2, multiple of 16
constexpr int kFastSegPx = 128;      // tested pixels per segment row: 32 lanes x one 4-pixel word
constexpr int kFastMaxCells = 8;

struct TilePlan {  // one blur tile
    short level, x0, y0, pad;
};

// Everything a kernel needs to address one batch.  Images [0, split) read/write set A,
// [split, count) set B (left / right images of a stereo batch).
struct ImgSet {
    const uint8_t *in_a, *in_b;  // level-0 pixels
    size_t in_stride;            // bytes between consecutive images of a set
    int in_pitch;                // bytes between rows
    int split;
    int in_z0;                   // index of image 0 of this (sub-)batch inside the level-0 tensor maps
    int slot_a, slot_b;          // internal buffer slot of image 0 of set A / set B (a pipelined host call runs
                                 // the batch as chunks that share the handle's buffers)
    uint8_t *pyr;                // levels 1.. of all images
    size_t pyr_stride;
    uint8_t *blur;               // blurred levels 0.. of all images
    size_t blur_stride;
    LevelPlan lv[kMaxLevels];    // per-level geometry, read from the constant bank (kernel parameters)
    int nlevels;
    uint32_t *cand;              // packed candidates: resp << 24 | y << 12 | x (window-relative)
    int cand_stride;
    uint32_t *kpst;              // packed quadtree survivors, same packing, list order
    int kpst_stride;
    int *cand_count;             // [image][level]
    int *kp_count;               // [image][level]
    int *flags;                  // [image] error bits
};

// TMA descriptors of one box shape: lv[l] = pyramid level l over the handle's slots (l >= 1),
// lv[0] / l0b = the level-0 images of set A / set B of the current call.
struct TmaMaps {
    CUtensorMap lv[kMaxLevels];
    CUtensorMap l0b;
};

enum { kFlagCandOverflow = 1, kFlagNodeOverflow = 2, kFlagOutOverflow = 4 };

struct OutSet {  // final outputs, set A / set B
    sfe_keypoint *kps_a, *kps_b;
    uint8_t *desc_a, *desc_b;
    int32_t *n_a, *n_b;
    int cap;
};

__device__ __forceinline__ int slot_of(const ImgSet &S, int img) {
    return img < S.split ? S.slot_a + img : S.slot_b + (img - S.split);
}

__device__ __forceinline__ const uint8_t *level_pixels(const ImgSet &S, int l, int img, int &pitch) {
    if (l == 0) {
        pitch = S.in_pitch;
        return img < S.split ? S.in_a + (size_t)img * S.in_stride
                             : S.in_b + (size_t)(img - S.split) * S.in_stride;
    }
    pitch = S.lv[l].pitch;
    return S.pyr + (size_t)slot_of(S, img) * S.pyr_stride + S.lv[l].plane_off;
}

// stereo matcher launch (sfe_match.cu), used by sfe_stereo_frames on the extractor's stream
void launch_stereo_match(cudaStream_t st, int frames, int cap, const sfe_keypoint *kl,
                         const uint8_t *dl, const int32_t *nl, const sfe_keypoint *kr,
                         const uint8_t *dr, const int32_t *nr, double y_thr, double max_dx,
                         double ratio, int32_t *out_idx, int32_t *out_dist, bool pdl = false);

// sequence tracking launch (sfe_match.cu), used by sfe_stereo_sequence on the extractor's stream: per-frame bucket grids,
// GetDepth + ProjectionMatch of frame f-1's stereo points into frame f, decode.  3 launches.
struct Pose;
struct TrackScratch {
    DevBuf<int> cell_start, order, valid;
    DevBuf<double2> sxy;
    DevBuf<uint4> sdesc;
    DevBuf<unsigned long long> best;
    // sfe_stereo_sequence_plan: the pair priors, the keys of the retry pass and which pairs took it
    DevBuf<Pose> poses;
    DevBuf<unsigned long long> best2;
    DevBuf<int> redo;
    void release() {
        cell_start.release(); order.release(); valid.release(); sxy.release(); sdesc.release(); best.release();
        poses.release(); best2.release(); redo.release();
    }
};
int launch_track_frames(cudaStream_t st, int device, TrackScratch &T, int frames, int cap, const sfe_keypoint *kl, const uint8_t *dl,
                        const int32_t *nl, const sfe_keypoint *kr, const int32_t *sidx, const sfe_track_params &tp,
                        int32_t *track_idx, int32_t *track_dist);
// the same with a validated plan: the priors are copied on `st` before the call returns; 3 launches, 5 with a retry
// (grids, first pass, retry flags, retry pass, decode; 2 for a single frame), added to `launches`
int launch_track_frames_plan(cudaStream_t st, int device, TrackScratch &T, int frames, int cap, const sfe_keypoint *kl,
                             const uint8_t *dl, const int32_t *nl, const sfe_keypoint *kr, const int32_t *sidx,
                             const sfe_track_params &tp, const sfe_track_plan &plan, int32_t *track_idx, int32_t *track_dist,
                             int64_t &launches);
// would this call's tracking reallocate a buffer of T?  (an asynchronous call must not free one under a running tail)
inline bool track_scratch_grows(const TrackScratch &T, int frames, int cap, const sfe_track_plan *plan) {
    const size_t fc = (size_t)frames * cap;
    if (fc > T.best.n) return true;
    if (!plan) return false;
    return (size_t)frames > T.poses.n || (plan->retry_below > 0 && (fc > T.best2.n || (size_t)frames > T.redo.n));
}

}  // namespace sfe
