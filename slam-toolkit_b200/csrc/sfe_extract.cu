// ORB extraction for sm_100a: pyramid -> per-cell FAST -> quadtree distribution ->
// IC_Angle -> 7x7 Gaussian -> rBRIEF.  From-scratch CUDA behind the sfe C ABI; reproduces
// reference src/orb_extractor.cpp:410-853,1034-1132 bit-for-bit under the canonical rules of
// oracle/orb_oracle.h.  Compiled with -fmad=false: every float op is individually rounded, as
// in the reference build (no -march => no FMA, CMakeLists.txt:54-55).
#include <cuda_fp16.h>

#include <algorithm>
#include <cmath>
#include <mutex>
#include <type_traits>

#include "sfe_extract.cuh"

namespace sfe {

// the 32-bit little-endian word at byte address p, any alignment (reads the two aligned words around it)
__device__ __forceinline__ uint32_t ldg_word_at(const uint8_t *p) {
    const uintptr_t a = (uintptr_t)p;
    const uint32_t *w = (const uint32_t *)(a & ~(uintptr_t)3);
    return __funnelshift_r(__ldg(w), __ldg(w + 1), (uint32_t)(a & 3) * 8);
}

// integer dot products (IDP.4A / IDP.2A: full rate, on the FMA pipe beside the ALU's LOP3 / PRMT -- tools/microbench.cu)
__device__ __forceinline__ uint32_t dp4a_u8u8(uint32_t a, uint32_t b, uint32_t c) {  // c + sum_k a.byte[k] * b.byte[k]
    uint32_t d;
    asm("dp4a.u32.u32 %0, %1, %2, %3;" : "=r"(d) : "r"(a), "r"(b), "r"(c));
    return d;
}
__device__ __forceinline__ uint32_t dp2a_lo(uint32_t a, uint32_t b, uint32_t c) {  // c + a.lo16 * b.byte0 + a.hi16 * b.byte1
    uint32_t d;
    asm("dp2a.lo.u32.u32 %0, %1, %2, %3;" : "=r"(d) : "r"(a), "r"(b), "r"(c));
    return d;
}
__device__ __forceinline__ uint32_t dp2a_hi(uint32_t a, uint32_t b, uint32_t c) {  // c + a.lo16 * b.byte2 + a.hi16 * b.byte3
    uint32_t d;
    asm("dp2a.hi.u32.u32 %0, %1, %2, %3;" : "=r"(d) : "r"(a), "r"(b), "r"(c));
    return d;
}

// ---------------------------------------------------------------------------------------------
// level-0 staging: images as the host holds them (tight rows) -> rows pitched to 16 bytes, the layout TMA
// can describe.  One thread = one 16-byte chunk of a destination row.
// ---------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) realign_kernel(const uint8_t *__restrict__ src, size_t src_stride, int src_pitch,
                                                      uint8_t *__restrict__ dst, size_t dst_stride, int dst_pitch, int w, int h) {
    pdl_enter();
    const int x = (blockIdx.x * 32 + threadIdx.x) * 16, y = blockIdx.y * 8 + threadIdx.y, img = blockIdx.z;
    if (x >= dst_pitch || y >= h) return;
    const uint8_t *p = src + (size_t)img * src_stride + (size_t)y * src_pitch + x;
    uint4 v;
    if (x + 20 <= w) {  // the unaligned word reads stay inside the row
        v = make_uint4(ldg_word_at(p), ldg_word_at(p + 4), ldg_word_at(p + 8), ldg_word_at(p + 12));
    } else {
        uint32_t q[4] = {0, 0, 0, 0};
#pragma unroll
        for (int k = 0; k < 16; k++)
            if (x + k < w) q[k >> 2] |= (uint32_t)__ldg(p + k) << (8 * (k & 3));
        v = make_uint4(q[0], q[1], q[2], q[3]);
    }
    *(uint4 *)(dst + (size_t)img * dst_stride + (size_t)y * dst_pitch + x) = v;
}

// ---------------------------------------------------------------------------------------------
// pyramid: cv::resize(INTER_LINEAR) fixed-point model, level l from level l-1 (:1120)
//   out = (((b0 * (T0 >> 4)) >> 16) + ((b1 * (T1 >> 4)) >> 16) + 2) >> 2,   T = S[sx] * w0 + S[sx + 1] * w1
// Separable, so one CTA (64 x 32 outputs) first forms U = T >> 4 (<= 32640, u16) for every source row its
// outputs touch -- 1.2 source rows per output row instead of 2 -- into shared memory, then combines two
// rows per output, 4 outputs per thread and one 32-bit store.  Coefficients come from host-built tables.
// ---------------------------------------------------------------------------------------------
constexpr int kPyrTileW = 64, kPyrTileH = 64;

struct PyrStep {            // geometry of one resize launch, in the kernel parameters
    int w, h, pitch, plane_off;      // destination level
    int src_w, src_pitch, src_plane_off, src_is_input;
    int xtab_off, ytab_off;
    int src_level, box_w, box_h;     // TMA variant: source level and its box
    int wide_h;                      // TMA variant: 4 outputs per thread in the horizontal pass (their sources span <= 7 px)
};

// kTma: the source pixels of the tile (box P.box_w x P.box_h bytes, origin on the 16-byte grid of the source row)
// arrive by one TMA load, so the horizontal pass reads shared memory instead of waiting on global loads
// (the plain variant spent 56 % of its stall samples on the long scoreboard).
template <bool kTma>
__global__ void __launch_bounds__(256) pyr_resize_kernel(ImgSet S, PyrStep P, const uint2 *__restrict__ xtab,
                                                         const uint2 *__restrict__ ytab, const __grid_constant__ TmaMaps M) {
    pdl_enter();
    extern __shared__ __align__(128) uint8_t pyr_smem[];
    uint16_t *pyr_u = (uint16_t *)(pyr_smem + (kTma ? P.box_w * P.box_h : 0));  // [source row][kPyrTileW]
    __shared__ uint64_t bar;
    const int x0 = blockIdx.x * kPyrTileW, y0 = blockIdx.y * kPyrTileH, img = blockIdx.z, tid = threadIdx.x;
    const uint2 *yt = ytab + P.ytab_off;
    const int sy_first = __ldg(&yt[y0]).x & 0xFFFF;                               // rows are monotone in y
    const int n_rows = (int)(__ldg(&yt[min(y0 + kPyrTileH, P.h) - 1]).x >> 16) - sy_first + 1;
    const int slot = slot_of(S, img);
    const int xa = (int)__ldg(&xtab[P.xtab_off + x0]).x & ~15;  // source column of shared column 0 (columns are monotone in x)
    if (kTma && tid == 0) {
        mbar_init(&bar, 1);
        mbar_expect_tx(&bar, (uint32_t)(P.box_w * P.box_h));
        const bool set_a = img < S.split;
        const CUtensorMap *map = P.src_is_input ? (set_a ? &M.lv[0] : &M.l0b) : &M.lv[P.src_level];
        const int z = P.src_is_input ? S.in_z0 + (set_a ? img : img - S.split) : slot;
        tma_load_3d(pyr_smem, map, &bar, xa, sy_first, z);
    }
    {   // horizontal: thread = output column, walking the source rows
        const int ox = tid & (kPyrTileW - 1);
        const uint2 xt = __ldg(&xtab[P.xtab_off + min(x0 + ox, P.w - 1)]);
        const int sx = xt.x, d1 = min(sx + 1, P.src_w - 1) - sx;
        const uint32_t w0 = xt.y & 0xFFFF, w1 = xt.y >> 16;
        if (kTma && P.wide_h) {
            // thread = 4 adjacent output columns: their source pixels lie within 8 bytes of the first one's (host-checked),
            // so three aligned words realigned by two funnel shifts hold all four (S[sx], S[sx + 1]) pairs; a PRMT per
            // output puts its pair into the low bytes and one IDP.2A forms S[sx] * w0 + S[sx + 1] * w1 (the table packs
            // w0 | w1 << 16).  At the right border w1 = 0, so whatever byte follows the last column is harmless.
            const int g4 = (tid & 15) * 4, gi = P.xtab_off + min(x0 + g4, (P.w - 1) & ~3);  // the table is padded to whole groups
            const uint4 ta = __ldg((const uint4 *)&xtab[gi]), tb = __ldg((const uint4 *)&xtab[gi + 2]);
            const int o0 = (int)ta.x - xa;
            const uint32_t sh8 = (uint32_t)(o0 & 3) * 8;
            const uint32_t r1 = ta.z - ta.x, r2 = tb.x - ta.x, r3 = tb.z - ta.x;
            const uint32_t s0 = 0x10u, s1 = r1 | (r1 + 1) << 4, s2 = r2 | (r2 + 1) << 4, s3 = r3 | (r3 + 1) << 4;
            __syncthreads();  // barrier initialised
            mbar_wait(&bar, 0);
            const uint32_t *p = (const uint32_t *)pyr_smem + (tid >> 4) * (P.box_w >> 2) + (o0 >> 2);
            const int step = 16 * (P.box_w >> 2);
            for (int r = tid >> 4; r < n_rows; r += 16) {
                const uint32_t a = __funnelshift_r(p[0], p[1], sh8), b = __funnelshift_r(p[1], p[2], sh8);
                const uint32_t u0 = dp2a_lo(ta.y, __byte_perm(a, b, s0), 0) >> 4, u1 = dp2a_lo(ta.w, __byte_perm(a, b, s1), 0) >> 4;
                const uint32_t u2 = dp2a_lo(tb.y, __byte_perm(a, b, s2), 0) >> 4, u3 = dp2a_lo(tb.w, __byte_perm(a, b, s3), 0) >> 4;
                *(uint2 *)&pyr_u[r * kPyrTileW + g4] = make_uint2(u0 | u1 << 16, u2 | u3 << 16);
                p += step;
            }
        } else if (kTma) {
            __syncthreads();  // barrier initialised
            mbar_wait(&bar, 0);
            const uint8_t *p = pyr_smem + (tid >> 6) * P.box_w + (sx - xa);
            const int step = 4 * P.box_w;
            for (int r = tid >> 6; r < n_rows; r += 4) {
                pyr_u[r * kPyrTileW + ox] = (uint16_t)((p[0] * w0 + p[d1] * w1) >> 4);
                p += step;
            }
        } else {
            const uint8_t *src;
            if (P.src_is_input)
                src = img < S.split ? S.in_a + (size_t)img * S.in_stride : S.in_b + (size_t)(img - S.split) * S.in_stride;
            else
                src = S.pyr + (size_t)slot * S.pyr_stride + P.src_plane_off;
            const uint8_t *p = src + (size_t)(sy_first + (tid >> 6)) * P.src_pitch + sx;
            const int step = 4 * P.src_pitch;
            for (int r = tid >> 6; r < n_rows; r += 4) {
                pyr_u[r * kPyrTileW + ox] = (uint16_t)((__ldg(p) * w0 + __ldg(p + d1) * w1) >> 4);
                p += step;
            }
        }
    }
    __syncthreads();
    // vertical: thread = 4 adjacent outputs on rows ry, ry + 16, ry + 32, ry + 48
    const int cg = (tid & 15) * 4, ry = tid >> 4;
    if (x0 + cg >= P.w) return;
    uint8_t *dst = S.pyr + (size_t)slot * S.pyr_stride + P.plane_off + x0 + cg;
#pragma unroll
    for (int k = 0; k < kPyrTileH / 16; k++) {
        const int oy = y0 + ry + 16 * k;
        if (oy >= P.h) break;
        const uint2 t = __ldg(&yt[oy]);
        const int r0 = (int)(t.x & 0xFFFF) - sy_first, r1 = (int)(t.x >> 16) - sy_first;
        const uint32_t b0 = t.y << 16, b1 = t.y & 0xFFFF0000u;  // (b * u) >> 16 == __umulhi(b << 16, u)
        const uint2 A = *(const uint2 *)&pyr_u[r0 * kPyrTileW + cg], B = *(const uint2 *)&pyr_u[r1 * kPyrTileW + cg];
        const uint32_t a[4] = {A.x & 0xFFFF, A.x >> 16, A.y & 0xFFFF, A.y >> 16};
        const uint32_t b[4] = {B.x & 0xFFFF, B.x >> 16, B.y & 0xFFFF, B.y >> 16};
        uint32_t v[4];
#pragma unroll
        for (int i = 0; i < 4; i++) v[i] = (__umulhi(b0, a[i]) + __umulhi(b1, b[i]) + 2) >> 2;  // <= (2048 * 32640 >> 16) + 2 >> 2 = 255
        *(uint32_t *)(dst + (size_t)oy * P.pitch) = v[0] | v[1] << 8 | v[2] << 16 | v[3] << 24;  // pitch % 16 == 0: pad absorbs the tail
    }
}

// ---------------------------------------------------------------------------------------------
// FAST-9-16, one CTA per segment of up to 128 tested pixels along one cell row (SegRec): the tested
// regions of the reference's cv::FAST calls (one 30-px grid cell each, :789-816) tile the row, so the
// per-pixel stages run on the whole segment and only NMS and the 20 -> 7 retry look at cell borders.
//   load     the segment's sub-image into shared memory (one TMA box, or aligned words + funnel shift)
//   stage 0  pre-test on the four compass pixels, 4 pixels per lane with VABSDIFF4: any 9-arc of the
//            16-pixel circle contains a vertical and a horizontal compass pixel, so a corner needs
//            (|up - c| > t or |dn - c| > t) and (|lf - c| > t or |rt - c| > t); the cheaper superset
//            ((|up - c| | |dn - c|) > t) and ((|lf - c| | |rt - c|) > t) is what is evaluated.  One warp =
//            one row of the segment, one lane = one aligned word of 4 centre pixels; survivors go to a list
//   stage 1  exact score best(p) on the survivors, two pixels per thread in 16x2 lanes
//            (VIMNMX3.S16x2); corner iff best > t
//   stage 2  non-max suppression inside each cell (strict > over 8 neighbours, outside the cell = 0)
//   emit, then retry with minThFAST the cells where nothing survived (:811-816)
// ---------------------------------------------------------------------------------------------
// Shared column c of the tile is level column xa + c with xa = (ini_x - 4) rounded down to 16: a TMA box
// must start on a 16-byte multiple of the row, and stage 0 then works on the level's own 4-pixel words.

// best(p) = max over the 16 arcs of 9 consecutive circle pixels of max(min (v - p_k), min (p_k - v))
//         = max(v - min_arcs max_k p_k, max_arcs min_k p_k - v)                    (cv::FAST score + 1)
// for the two pixels at c0 / c1 at once: circle pixels packed as 16x2 lanes, 9 = 3 + 3 + 3 so every arc
// extremum is a 3-input extremum of 3-input extrema (VIMNMX3.S16x2).
template <int TP>
__device__ __forceinline__ void fast_best_x2(const uint8_t *c0, const uint8_t *c1, int &best0, int &best1) {
    constexpr int off[16] = {3 * TP,  3 * TP + 1,  2 * TP + 2,  TP + 3,  3,  -TP + 3, -2 * TP + 2, -3 * TP + 1,
                             -3 * TP, -3 * TP - 1, -2 * TP - 2, -TP - 3, -3, TP - 3,  2 * TP - 2,  3 * TP - 1};
    uint32_t p[16], lo3[16], hi3[16];
#pragma unroll
    for (int k = 0; k < 16; k++) p[k] = __byte_perm(c0[off[k]], c1[off[k]], 0x5410);
#pragma unroll
    for (int s = 0; s < 16; s++) {
        lo3[s] = __vimin3_s16x2(p[s], p[(s + 1) & 15], p[(s + 2) & 15]);
        hi3[s] = __vimax3_s16x2(p[s], p[(s + 1) & 15], p[(s + 2) & 15]);
    }
    uint32_t max_of_min = 0u, min_of_max = 0x7fff7fffu;
#pragma unroll
    for (int s = 0; s < 16; s += 2) {
        const uint32_t l0 = __vimin3_s16x2(lo3[s], lo3[(s + 3) & 15], lo3[(s + 6) & 15]);
        const uint32_t l1 = __vimin3_s16x2(lo3[s + 1], lo3[(s + 4) & 15], lo3[(s + 7) & 15]);
        const uint32_t h0 = __vimax3_s16x2(hi3[s], hi3[(s + 3) & 15], hi3[(s + 6) & 15]);
        const uint32_t h1 = __vimax3_s16x2(hi3[s + 1], hi3[(s + 4) & 15], hi3[(s + 7) & 15]);
        max_of_min = __vimax3_s16x2(max_of_min, l0, l1);
        min_of_max = __vimin3_s16x2(min_of_max, h0, h1);
    }
    const int v0 = c0[0], v1 = c1[0];
    best0 = max(v0 - (int)(min_of_max & 0xFFFF), (int)(max_of_min & 0xFFFF) - v0);
    best1 = max(v1 - (int)(min_of_max >> 16), (int)(max_of_min >> 16) - v1);
}

// kTma: the sub-image arrives as one TMA box (kFastTilePitch x tile_rows bytes) issued by thread 0; otherwise
// (level-0 images whose layout TMA cannot describe) the threads assemble it from aligned global words.
template <bool kTma>
__global__ void __launch_bounds__(kFastThreads, kFastCtasPerSm) fast_segments_kernel(ImgSet S, FastPlan P, const SegRec *__restrict__ segs,
                                                                     const __grid_constant__ TmaMaps M) {
    constexpr int TP = kFastTilePitch, TW = TP / 4, SP = kFastScorePitch, T = kFastThreads;
    pdl_enter();
    extern __shared__ __align__(128) uint32_t fast_smem[];
    uint32_t *tile32 = fast_smem;                              // tile_rows x TW
    uint8_t *score = (uint8_t *)(tile32 + P.tile_rows * TW);   // score_rows x SP
    uint16_t *pre = (uint16_t *)(score + P.score_rows * SP);   // y << 8 | x of pixels passing stage 0
    uint16_t *det = pre + P.list_cap;                          // corners
    __shared__ int n_pre, n_det;
    __shared__ int cell_surv[kFastMaxCells];
    __shared__ uint64_t bar;
    const uint8_t *tile = (const uint8_t *)tile32;

    const uint4 rec = __ldg((const uint4 *)segs + blockIdx.x);  // one 16-byte SegRec
    const int ini_x = (short)(rec.x & 0xFFFF), ini_y = (short)(rec.x >> 16), tw = (short)(rec.y & 0xFFFF);
    const int sh = (rec.y >> 16) & 0xFF, level = rec.y >> 24, n_cells = rec.z & 0xFF, w_cell = (rec.z >> 8) & 0xFF;
    const int inv_w = rec.z >> 16, th = sh - 6;
    const FastLevel &F = P.lv[level];
    const int img = blockIdx.y, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int xa = (ini_x - 4) & ~15;  // level column of shared column 0 (ini_x >= 16)
    const int cs = ini_x + 3 - xa;     // shared column of tested x = 0, in [7, 22]
    if (kTma) {
        // bytes outside the image arrive as zeros and are never tested
        if (tid == 0) {
            mbar_init(&bar, 1);
            mbar_expect_tx(&bar, (uint32_t)(P.tile_rows * TP));
            const bool set_a = img < S.split;
            const CUtensorMap *map = level == 0 ? (set_a ? &M.lv[0] : &M.l0b) : &M.lv[level];
            const int z = level == 0 ? S.in_z0 + (set_a ? img : img - S.split) : slot_of(S, img);
            tma_load_3d(tile32, map, &bar, xa, ini_y, z);
        }
    } else {
        const uint8_t *src;
        int pitch;
        if (level == 0) {
            pitch = S.in_pitch;
            src = img < S.split ? S.in_a + (size_t)img * S.in_stride : S.in_b + (size_t)(img - S.split) * S.in_stride;
        } else {
            pitch = F.pitch;
            src = S.pyr + (size_t)slot_of(S, img) * S.pyr_stride + F.plane_off;
        }
        src += (size_t)ini_y * pitch + xa;
        // words up to the one after the last tested pixel's; the row has >= 16 px beyond the segment
        const int nw = min(((cs + tw - 1) >> 2) + 2, TW);
        for (int r = warp; r < sh; r += T / 32)
            for (int j = lane; j < nw; j += 32) tile32[r * TW + j] = ldg_word_at(src + (size_t)r * pitch + 4 * j);
    }
    // stage-0 geometry of this lane: its word of the row, and which of the word's 4 pixels are tested ones
    const int jw = (cs >> 2) + lane, x0 = 4 * jw - cs;  // tested x of the word's first pixel (may be negative)
    uint32_t vm = 0;                                    // bit 7 of byte k: pixel k of the word is a tested one
#pragma unroll
    for (int k = 0; k < 4; k++)
        if (x0 + k >= 0 && x0 + k < tw) vm |= 0x80u << (8 * k);
    uint32_t todo = (1u << n_cells) - 1;  // cells this pass works on
    int t = P.ini_th;
    for (int i = tid; i < (th + 2) * (SP / 16); i += T) ((uint4 *)score)[i] = make_uint4(0, 0, 0, 0);
    for (int attempt = 0; attempt < 2; attempt++) {
        if (tid == 0) { n_pre = 0; n_det = 0; }
        if (tid < kFastMaxCells) cell_surv[tid] = 0;
        __syncthreads();
        if (kTma && attempt == 0) mbar_wait(&bar, 0);  // the barrier was initialised by thread 0 before the sync above
        // stage 0: one row per warp, one word of 4 centre pixels per lane
        uint32_t vm_now = vm;
        if (attempt) {
#pragma unroll
            for (int k = 0; k < 4; k++)
                if (!((todo >> ((max(x0 + k, 0) * inv_w) >> 16)) & 1)) vm_now &= ~(0x80u << (8 * k));
        }
        const uint32_t kk = (uint32_t)(0x7F - min(t, 127)) * 0x01010101u;
        if (vm_now) {
            const uint32_t *row = tile32 + (warp + 3) * TW + jw;
            for (int y = warp; y < th; y += T / 32, row += (T / 32) * TW) {
                const uint32_t c = row[0];
                const uint32_t dv0 = __vabsdiffu4(row[-3 * TW], c), dv1 = __vabsdiffu4(row[3 * TW], c);
                const uint32_t dh0 = __vabsdiffu4(__byte_perm(row[-1], c, 0x4321), c);  // pixels x-3 .. x
                const uint32_t dh1 = __vabsdiffu4(__byte_perm(c, row[1], 0x6543), c);   // pixels x+3 .. x+6
                // byte > t  <=>  bit 7 of (byte | ((byte & 0x7f) + 0x7f - t)); a | b >= max(a, b) keeps this a superset
                const uint32_t rv = (((dv0 | dv1) & 0x7F7F7F7Fu) + kk) | dv0 | dv1;
                const uint32_t rh = (((dh0 | dh1) & 0x7F7F7F7Fu) + kk) | dh0 | dh1;
                const uint32_t m = rv & rh & vm_now;
                // the list order is irrelevant downstream and only some lanes hold survivors, so a shared-memory
                // atomic per such lane costs fewer issue slots than a ballot / prefix scheme
                if (m) {
                    int pos = atomicAdd(&n_pre, __popc(m));
                    const uint16_t item = (uint16_t)((y << 8) + x0);  // pixels left of the segment are masked out
                    if (m & 0x80u) pre[pos++] = item;
                    if (m & 0x8000u) pre[pos++] = item + 1;
                    if (m & 0x800000u) pre[pos++] = item + 2;
                    if (m & 0x80000000u) pre[pos] = item + 3;
                }
            }
        }
        __syncthreads();
        // stage 1: exact score, two survivors per thread; corner at threshold t iff best > t
        const int np = n_pre, npairs = (np + 1) >> 1;
        for (int e0 = 0; e0 < npairs; e0 += T) {
            bool corner0 = false, corner1 = false;
            uint16_t yx0 = 0, yx1 = 0;
            const int e = e0 + tid;
            if (e < npairs) {
                yx0 = pre[2 * e];
                yx1 = pre[min(2 * e + 1, np - 1)];
                int best0, best1;
                fast_best_x2<TP>(&tile[((yx0 >> 8) + 3) * TP + (yx0 & 255) + cs], &tile[((yx1 >> 8) + 3) * TP + (yx1 & 255) + cs],
                                 best0, best1);
                corner0 = best0 > t;
                corner1 = best1 > t && 2 * e + 1 < np;
                if (corner0) score[((yx0 >> 8) + 1) * SP + (yx0 & 255) + 1] = (uint8_t)best0;
                if (corner1) score[((yx1 >> 8) + 1) * SP + (yx1 & 255) + 1] = (uint8_t)best1;
            }
            // one shared-memory atomic per warp reserves the slots of both corner flags
            const uint32_t c0 = __ballot_sync(0xffffffffu, corner0), c1 = __ballot_sync(0xffffffffu, corner1);
            if (c0 | c1) {
                int base = 0;
                if (lane == 0) base = atomicAdd(&n_det, __popc(c0) + __popc(c1));
                base = __shfl_sync(0xffffffffu, base, 0);
                const uint32_t lt = (1u << lane) - 1;
                if (corner0) det[base + __popc(c0 & lt)] = yx0;
                if (corner1) det[base + __popc(c0) + __popc(c1 & lt)] = yx1;
            }
        }
        __syncthreads();
        // stage 2: non-max suppression; a neighbour in another cell counts as 0 (the reference runs cv::FAST per cell).
        // Survivors go straight to the level's candidate array: one global atomic per warp reserves their slots.
        const int nd = n_det, slot = slot_of(S, img);
        uint32_t *out = S.cand + (size_t)slot * S.cand_stride + F.cand_off;
        for (int e0 = warp * 32; e0 < nd; e0 += T) {
            bool keep = false;
            uint32_t packed = 0;
            int cell = 0;
            if (e0 + lane < nd) {
                const uint16_t yx = det[e0 + lane];
                const int x = yx & 255, y = yx >> 8;
                cell = (x * inv_w) >> 16;
                const int cx0 = cell * w_cell, cx1 = min(cx0 + w_cell, tw);
                const uint8_t *sc = &score[(y + 1) * SP + x + 1];
                const int s = sc[0];
                // branch-free: the three neighbours of a side count as 0 when that side lies in another cell
                const int lft = x > cx0 ? __vimax3_s32(sc[-1], sc[-SP - 1], sc[SP - 1]) : 0;
                const int rgt = x + 1 < cx1 ? __vimax3_s32(sc[1], sc[-SP + 1], sc[SP + 1]) : 0;
                keep = s > __vimax3_s32(max(sc[-SP], sc[SP]), lft, rgt);
                // cv::FAST response = best - 1; window-relative coordinates
                packed = (uint32_t)(s - 1) << 24 | (uint32_t)(ini_y - kBorder + y + 3) << 12 | (uint32_t)(ini_x - kBorder + x + 3);
            }
            const uint32_t kept = __ballot_sync(0xffffffffu, keep);
            if (kept) {
                int base = 0;
                if (lane == 0) base = atomicAdd(&S.cand_count[slot * S.nlevels + level], __popc(kept));
                base = __shfl_sync(0xffffffffu, base, 0);
                if (keep) {
                    const int o = base + __popc(kept & ((1u << lane) - 1));
                    if (o < F.cand_cap) out[o] = packed;
                    else atomicOr(&S.flags[slot], kFlagCandOverflow);
                    cell_surv[cell] = 1;
                }
            }
        }
        __syncthreads();
        // :811-816: cells of this pass where nothing survived (lane c looks at cell c; every warp forms the same mask)
        const uint32_t retry = __ballot_sync(0xffffffffu, lane < n_cells && ((todo >> lane) & 1) && cell_surv[min(lane, kFastMaxCells - 1)] == 0);
        if (retry == 0 || P.min_th >= t) break;  // a higher threshold cannot find what the lower one did not
        t = P.min_th;
        todo = retry;
        __syncthreads();
    }
}

// ---------------------------------------------------------------------------------------------
// DistributeOctTree (:539-763) as arrays + prefix sums; one CTA per (level, image).
// Transcribes tools/octree_model.py, which tests/test_octree_model.py checks against the literal
// std::list emulation of the oracle.  Candidate order is irrelevant here: membership is a pure
// function of coordinates, and the only order-dependent step (first max response wins, :742-760)
// uses the explicit order key of the reference's cell-major / raster candidate list.
// ---------------------------------------------------------------------------------------------
// kWide = false: a level holds at most 60000 candidates and positions / counts fit 16 bits (14 B of working set per
// candidate, 12-byte nodes); kWide = true: 32-bit positions for fuller levels (dense 4K frames, noise), always on global
// scratch.  Same code, same results; the narrow instance is the one every ordinary frame runs.
template <bool kWide>
struct ONodeT {
    typedef typename std::conditional<kWide, uint32_t, unsigned short>::type pos_t;
    short x0, x1, y0, y1;
    pos_t start, cnt;
};

template <bool kWide>
struct OctSmemT {
    typedef ONodeT<kWide> ONode;
    typedef typename ONode::pos_t pos_t;
    uint32_t *pk[2];       // packed candidates, grouped by node
    uint16_t *own[2];      // list index of the node owning each position
    pos_t *qs;             // slot within the child node (the quadrant is recomputed from the coordinates)
    ONode *nd[2];
    uint16_t *eidx[2];     // creation order among expandable nodes (tie rule T1)
    uint32_t *child;       // [node][4]: child counts, then child start positions
    uint16_t *childpos;    // [node][4]: list index of each child in the next list
    int *tord;             // processing order of a split node, -1 = not split
    int *arr_a, *arr_b;    // scan scratch
    int *warp_sums;
};

__device__ int block_excl_scan(int *a, int n, int *warp_sums) {
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, nwarps = blockDim.x >> 5;
    int carry = 0;
    for (int base = 0; base < n; base += blockDim.x) {
        const int i = base + tid;
        const int v = i < n ? a[i] : 0;
        int inc = v;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const int u = __shfl_up_sync(0xffffffffu, inc, o);
            if (lane >= o) inc += u;
        }
        if (lane == 31) warp_sums[warp] = inc;
        __syncthreads();
        if (warp == 0) {
            int w = lane < nwarps ? warp_sums[lane] : 0;
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
                const int u = __shfl_up_sync(0xffffffffu, w, o);
                if (lane >= o) w += u;
            }
            warp_sums[lane] = w;
        }
        __syncthreads();
        const int woff = warp > 0 ? warp_sums[warp - 1] : 0;
        if (i < n) a[i] = carry + woff + inc - v;
        const int chunk = warp_sums[nwarps - 1];
        __syncthreads();
        carry += chunk;
    }
    return carry;
}

// Exclusive scan of one packed 64-bit value per thread (fields that never carry into each other), chunk by chunk over n items:
// scan_chunk() returns the exclusive prefix of the thread's value inside the chunk plus the running carry.  Two barriers a chunk.
__device__ __forceinline__ unsigned long long block_excl_scan64(unsigned long long v, unsigned long long *ws, unsigned long long &carry) {
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, nwarps = blockDim.x >> 5;
    unsigned long long inc = v;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const unsigned long long u = __shfl_up_sync(0xffffffffu, inc, o);
        if (lane >= o) inc += u;
    }
    if (lane == 31) ws[warp] = inc;
    __syncthreads();
    // every warp scans the warp totals itself (lane w holds warp w's)
    unsigned long long x = lane < nwarps ? ws[lane] : 0ull;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const unsigned long long u = __shfl_up_sync(0xffffffffu, x, o);
        if (lane >= o) x += u;
    }
    const unsigned long long tot = __shfl_sync(0xffffffffu, x, 31);
    const unsigned long long upto = __shfl_sync(0xffffffffu, x, max(warp - 1, 0));
    const unsigned long long woff = warp > 0 ? upto : 0ull;
    const unsigned long long r = carry + woff + inc - v;
    carry += tot;
    __syncthreads();  // ws is reused by the next chunk
    return r;
}

// Second half of a pass: write the next node list and move the points.  M.tord[i] = processing index of a split node or -1;
// M.arr_b[by_order ? tord[i] : i] = exclusive prefix (non-empty children | expandable children << 16) over the processing order;
// M.arr_a[i] = rank of an unsplit node among the unsplit ones.  C = number of children.  Returns the new list size.
template <bool kWide>
__device__ int octree_emit(OctSmemT<kWide> &M, int cur, int n, int nL, int C, int n_unsplit, bool by_order) {
    typedef ONodeT<kWide> ONode;
    typedef typename ONode::pos_t pos_t;
    const int tid = threadIdx.x, T = blockDim.x, nxt = cur ^ 1;
    const ONode *nd = M.nd[cur];
    for (int i = tid; i < nL; i += T) {
        const int t = M.tord[i];
        const ONode o = nd[i];
        if (t >= 0) {
            const int pe = M.arr_b[by_order ? t : i], pp = pe & 0xFFFF, ep = pe >> 16;
            const int mx = o.x0 + ((o.x1 - o.x0 + 1) >> 1), my = o.y0 + ((o.y1 - o.y0 + 1) >> 1);
            uint32_t cc[4];
#pragma unroll
            for (int q = 0; q < 4; q++) cc[q] = M.child[i * 4 + q];
            int k = 0, ke = 0, off = 0;
#pragma unroll
            for (int q = 0; q < 4; q++) {
                M.child[i * 4 + q] = o.start + off;  // from now on: start position of child q
                if (cc[q] > 0) {
                    const int pos = C - 1 - (pp + k);  // push_front order reversed (:606-662)
                    ONode c;
                    c.x0 = (q & 1) ? mx : o.x0;
                    c.x1 = (q & 1) ? o.x1 : mx;
                    c.y0 = (q & 2) ? my : o.y0;
                    c.y1 = (q & 2) ? o.y1 : my;
                    c.start = (pos_t)(o.start + off);
                    c.cnt = (pos_t)cc[q];
                    M.nd[nxt][pos] = c;
                    M.eidx[nxt][pos] = (uint16_t)(cc[q] > 1 ? ep + ke : 0);
                    M.childpos[i * 4 + q] = (uint16_t)pos;
                    k++;
                    ke += cc[q] > 1;
                }
                off += cc[q];
            }
        } else {
            const int pos = C + M.arr_a[i];
            M.nd[nxt][pos] = o;
            M.eidx[nxt][pos] = M.eidx[cur][i];
            M.childpos[i * 4] = (uint16_t)pos;
        }
    }
    __syncthreads();
    for (int p = tid; p < n; p += T) {
        const int i = M.own[cur][p];
        if (M.tord[i] >= 0) {
            const ONode o = nd[i];
            const uint32_t v = M.pk[cur][p];
            const int x = v & 0xFFF, y = (v >> 12) & 0xFFF;
            const int mx = o.x0 + ((o.x1 - o.x0 + 1) >> 1), my = o.y0 + ((o.y1 - o.y0 + 1) >> 1);
            const int q = (x < mx ? 0 : 1) + (y < my ? 0 : 2);  // as in the counting loop above
            const int np = M.child[i * 4 + q] + M.qs[p];
            M.pk[nxt][np] = v;
            M.own[nxt][np] = M.childpos[i * 4 + q];
        } else {
            M.pk[nxt][p] = M.pk[cur][p];
            M.own[nxt][p] = M.childpos[i * 4];
        }
    }
    __syncthreads();
    return C + n_unsplit;
}

// One pass over the node list.  careful == false: split every expandable node in list order
// (:594-665).  careful == true: split expandable nodes in descending (count, creation order)
// until the list reaches n_want (:673-738).  Returns new list size; *n_expand = new |E|.
template <bool kWide>
__device__ int octree_pass(OctSmemT<kWide> &M, int cur, int n, int nL, int n_want, bool careful, int *n_expand,
                           int *sh_misc) {
    typedef ONodeT<kWide> ONode;
    typedef typename ONode::pos_t pos_t;
    const int tid = threadIdx.x, T = blockDim.x, nxt = cur ^ 1;
    const ONode *nd = M.nd[cur];
    for (int i = tid; i < nL * 4; i += T) M.child[i] = 0;
    __syncthreads();
    for (int p = tid; p < n; p += T) {
        const int i = M.own[cur][p];
        const ONode o = nd[i];
        if (o.cnt > 1) {
            const uint32_t v = M.pk[cur][p];
            const int x = v & 0xFFF, y = (v >> 12) & 0xFFF;
            const int mx = o.x0 + ((o.x1 - o.x0 + 1) >> 1), my = o.y0 + ((o.y1 - o.y0 + 1) >> 1);
            const int q = (x < mx ? 0 : 1) + (y < my ? 0 : 2);
            M.qs[p] = (pos_t)atomicAdd(&M.child[i * 4 + q], 1u);
        }
    }
    __syncthreads();
    // processing order of expandable nodes
    int n_split;
    if (!careful) {
        // list order is processing order: one scan of (expandable, non-empty children, expandable children) per node gives the
        // processing index, the position of the children in the next list and their creation order
        __shared__ unsigned long long ws64[32];
        unsigned long long carry = 0;
        for (int base = 0; base < nL; base += T) {
            const int i = base + tid;
            unsigned long long v = 0;
            if (i < nL && nd[i].cnt > 1) {
                const uint32_t *c = &M.child[i * 4];
                const unsigned long long nz = (c[0] > 0) + (c[1] > 0) + (c[2] > 0) + (c[3] > 0);
                const unsigned long long ne = (c[0] > 1) + (c[1] > 1) + (c[2] > 1) + (c[3] > 1);
                v = 1ull | nz << 16 | ne << 32;
            }
            const unsigned long long ex = block_excl_scan64(v, ws64, carry);
            if (i < nL) {
                const int e = (int)(ex & 0xFFFF);
                M.tord[i] = v ? e : -1;
                M.arr_b[i] = (int)((ex >> 16) & 0xFFFF) | (int)((ex >> 32) & 0xFFFF) << 16;
                M.arr_a[i] = i - e;  // unsplit nodes keep their relative order behind the children
            }
        }
        n_split = (int)(carry & 0xFFFF);
        const int C = (int)((carry >> 16) & 0xFFFF);
        *n_expand = (int)((carry >> 32) & 0xFFFF);
        __syncthreads();
        return octree_emit<kWide>(M, cur, n, nL, C, nL - n_split, false);
    } else {
        // rank by (count, creation order) descending (0 = not expandable)
        int n_e_local = 0;
        if (!kWide) {  // count < 65536: one unsigned key per node
            for (int i = tid; i < nL; i += T)
                M.arr_a[i] = nd[i].cnt > 1 ? (int)((uint32_t)nd[i].cnt << 16 | M.eidx[cur][i]) : 0;
            __syncthreads();
            for (int i = tid; i < nL; i += T) {
                const uint32_t key = (uint32_t)M.arr_a[i];
                int rank = -1;
                if (key != 0) {
                    rank = 0;
                    for (int j = 0; j < nL; j++) rank += (uint32_t)M.arr_a[j] > key;
                    n_e_local++;
                }
                M.tord[i] = rank;
            }
        } else {       // count in arr_a, creation order in eidx
            for (int i = tid; i < nL; i += T) M.arr_a[i] = nd[i].cnt > 1 ? (int)nd[i].cnt : 0;
            __syncthreads();
            for (int i = tid; i < nL; i += T) {
                const int cnt_i = M.arr_a[i];
                int rank = -1;
                if (cnt_i > 0) {
                    const int e_i = M.eidx[cur][i];
                    rank = 0;
                    for (int j = 0; j < nL; j++) {
                        const int cnt_j = M.arr_a[j];
                        rank += cnt_j > cnt_i || (cnt_j == cnt_i && M.eidx[cur][j] > e_i);
                    }
                    n_e_local++;
                }
                M.tord[i] = rank;
            }
        }
        if (tid == 0) { sh_misc[0] = 0; sh_misc[1] = 0x7fffffff; }
        __syncthreads();
        if (n_e_local) atomicAdd(&sh_misc[0], n_e_local);
        // per expandable node, in processing order: non-empty children | children with > 1 points << 16.  One scan serves the
        // list growth (a split adds its non-empty children minus itself), the children's positions and their creation order.
        for (int i = tid; i < nL; i += T) {
            const int t = M.tord[i];
            if (t >= 0) {
                const uint32_t *c = &M.child[i * 4];
                const int nz = (c[0] > 0) + (c[1] > 0) + (c[2] > 0) + (c[3] > 0);
                const int ne = (c[0] > 1) + (c[1] > 1) + (c[2] > 1) + (c[3] > 1);
                M.arr_b[t] = nz | ne << 16;
            }
        }
        __syncthreads();
        const int n_e = sh_misc[0];
        const int tot = block_excl_scan(M.arr_b, n_e, M.warp_sums);
        for (int i = tid; i < nL; i += T) {
            const int t = M.tord[i];
            if (t >= 0) {
                const uint32_t *c = &M.child[i * 4];
                const int nz = (c[0] > 0) + (c[1] > 0) + (c[2] > 0) + (c[3] > 0);
                if (nL + (M.arr_b[t] & 0xFFFF) - t + nz - 1 >= n_want) atomicMin(&sh_misc[1], t + 1);  // break after this split (:730)
            }
        }
        __syncthreads();
        n_split = min(sh_misc[1], n_e);
        const int upto = n_split < n_e ? M.arr_b[n_split] : tot;  // totals over the nodes that are split
        for (int i = tid; i < nL; i += T) {
            int t = M.tord[i];
            if (t >= n_split) M.tord[i] = t = -1;
            M.arr_a[i] = t < 0 ? 1 : 0;  // unsplit nodes keep their relative order behind the children
        }
        __syncthreads();
        const int n_unsplit = block_excl_scan(M.arr_a, nL, M.warp_sums);
        *n_expand = upto >> 16;
        return octree_emit<kWide>(M, cur, n, nL, upto & 0xFFFF, n_unsplit, true);
    }
}

// The node list after `d0` full passes, written directly (tools/octree_model.py: fast_forward).  With 4 * n_ini * 4^d0 <= quota
// those passes cannot end the reference's loop through its size tests (|list| <= n_ini * 4^d, |list| + 3 |E| <= 4 |list|), and
// node boundaries do not depend on the data: the list holds the non-empty cells of the depth-d0 grid -- a cell with a single
// point stopped splitting at the depth f where it became single and sits behind every deeper node -- in the order the
// push_front passes leave: per depth f, digit i of the cell's path (root = digit 0) runs descending when the list was reversed
// an odd number of times since that digit was appended (root: f odd; q_i: f - i even).  A pass that does not grow the list
// ends the loop (:665): then the list of that depth is final (*finished).  Returns the list size; list 0 is written.
template <bool kWide>
__device__ int octree_build_at_depth(OctSmemT<kWide> &M, const uint32_t *__restrict__ cand, int n, int n_ini, float hx, int win_h, int d0,
                                     bool *finished) {
    typedef ONodeT<kWide> ONode;
    typedef typename ONode::pos_t pos_t;
    __shared__ unsigned long long ws64[32];
    __shared__ int sizes[8];
    const int tid = threadIdx.x, T = blockDim.x;
    uint32_t *cntp = M.child;  // counts of every cell of depths 0 .. d0: cell c of depth f at off(f) + c
    auto off = [n_ini](int f) { return n_ini * (((1 << (2 * f)) - 1) / 3); };
    auto cells = [n_ini](int f) { return n_ini << (2 * f); };
    const int tot = off(d0 + 1);
    for (int i = tid; i < tot; i += T) cntp[i] = 0;
    if (tid < 8) sizes[tid] = 0;
    __syncthreads();
    for (int p = tid; p < n; p += T) {
        const uint32_t v = cand[p];
        const int x = v & 0xFFF, y = (v >> 12) & 0xFFF;
        int r = (int)__fdiv_rn((float)x, hx);
        r = min(r, n_ini - 1);
        int x0 = (int)__fmul_rn(hx, (float)r), x1 = (int)__fmul_rn(hx, (float)(r + 1)), y0 = 0, y1 = win_h, cell = r;
        for (int f = 0; f < d0; f++) {
            const int mx = x0 + ((x1 - x0 + 1) >> 1), my = y0 + ((y1 - y0 + 1) >> 1);
            const bool right = x >= mx, low = y >= my;
            x0 = right ? mx : x0; x1 = right ? x1 : mx;
            y0 = low ? my : y0;   y1 = low ? y1 : my;
            cell = cell * 4 + (right ? 1 : 0) + (low ? 2 : 0);
        }
        M.own[1][p] = (uint16_t)cell;  // < quota / 4
        atomicAdd(&cntp[off(d0) + cell], 1u);
    }
    __syncthreads();
    for (int f = d0 - 1; f >= 0; f--) {
        for (int c = tid; c < cells(f); c += T) {
            const uint32_t *k = &cntp[off(f + 1) + 4 * c];
            cntp[off(f) + c] = k[0] + k[1] + k[2] + k[3];
        }
        __syncthreads();
    }
    for (int i = tid; i < tot; i += T) {
        if (cntp[i] == 0) continue;
        int f = 0;
        while (i >= off(f + 1)) f++;
        atomicAdd(&sizes[f], 1);
    }
    __syncthreads();
    int d_build = d0;
    *finished = false;
    for (int f = 1; f <= d0; f++)
        if (sizes[f] == sizes[f - 1]) { d_build = f; *finished = true; break; }
    // list order: the nodes of depth d_build, then the single-point nodes of depth d_build - 1, ..., 0
    const int totb = off(d_build + 1);
    unsigned long long carry = 0;
    for (int base = 0; base < totb; base += T) {
        const int k = base + tid;
        unsigned long long v = 0;
        int f = d_build, cell = 0;
        uint32_t here = 0;
        if (k < totb) {
            int e = k;
            while (e >= cells(f)) { e -= cells(f); f--; }
            const int re = e >> (2 * f);
            cell = (f & 1) ? n_ini - 1 - re : re;
            for (int i = 1; i <= f; i++) {
                const int q = (e >> (2 * (f - i))) & 3;
                cell = cell * 4 + (((f - i) & 1) == 0 ? 3 - q : q);
            }
            here = cntp[off(f) + cell];
            const uint32_t parent = f > 0 ? cntp[off(f - 1) + (cell >> 2)] : 2u;
            const bool node = parent > 1 && (f == d_build ? here > 0 : here == 1);
            if (node) v = 1ull | (unsigned long long)here << 32;
        }
        const unsigned long long ex = block_excl_scan64(v, ws64, carry);
        if (v) {
            const int pos = (int)(ex & 0xFFFF);
            int x0 = 0, x1 = 0, y0 = 0, y1 = win_h;
            {
                const int r = cell >> (2 * f);
                x0 = (int)__fmul_rn(hx, (float)r);
                x1 = (int)__fmul_rn(hx, (float)(r + 1));
                for (int i = 1; i <= f; i++) {
                    const int q = (cell >> (2 * (f - i))) & 3;
                    const int mx = x0 + ((x1 - x0 + 1) >> 1), my = y0 + ((y1 - y0 + 1) >> 1);
                    x0 = (q & 1) ? mx : x0; x1 = (q & 1) ? x1 : mx;
                    y0 = (q & 2) ? my : y0; y1 = (q & 2) ? y1 : my;
                }
            }
            ONode o;
            o.x0 = (short)x0; o.x1 = (short)x1; o.y0 = (short)y0; o.y1 = (short)y1;
            o.start = (pos_t)(ex >> 32);
            o.cnt = (pos_t)here;
            M.nd[0][pos] = o;
            M.eidx[0][pos] = 0;  // the next pass is a full one: it numbers its children itself
            M.arr_a[off(f) + cell] = pos;
            M.arr_b[pos] = 0;    // fill cursor of the node's segment
        }
    }
    const int nL = (int)(carry & 0xFFFF);
    __syncthreads();
    for (int p = tid; p < n; p += T) {
        const int fine = M.own[1][p];
        int f = 0, c = 0;
        for (; f <= d_build; f++) {
            c = fine >> (2 * (d0 - f));
            if (f == d_build || cntp[off(f) + c] == 1) break;
        }
        const int pos = M.arr_a[off(f) + c];
        const int np = (int)M.nd[0][pos].start + atomicAdd(&M.arr_b[pos], 1);
        M.pk[0][np] = cand[p];
        M.own[0][np] = (uint16_t)pos;
    }
    __syncthreads();
    return nL;
}

// Candidate-sized arrays (14 B per candidate) live in shared memory when the level has at most smem_cand
// candidates -- sized for the common case so that several CTAs fit an SM -- and otherwise in one of the
// handle's global scratch slots (same code, generic pointers; L2-resident).
template <bool kWide>
__device__ __forceinline__ void octree_item(const ImgSet &S, int l, int image, int smem_cand, int max_cand, int max_nodes,
                            uint8_t *__restrict__ scratch, int scratch_slots, int *scratch_next) {
    typedef ONodeT<kWide> ONode;
    typedef typename ONode::pos_t pos_t;
    constexpr int kCandBytes = 2 * 4 + 2 * 2 + (int)sizeof(pos_t);
    extern __shared__ __align__(16) uint8_t smem_raw[];
    __shared__ int sh_misc[4];
    const int img = slot_of(S, image), tid = threadIdx.x, T = blockDim.x;  // internal buffers only
    const LevelPlan &L = S.lv[l];
    int *kp_count = &S.kp_count[img * S.nlevels + l];
    const int n = min(S.cand_count[img * S.nlevels + l], L.cand_cap);
    if (n <= 0) {
        if (tid == 0) *kp_count = 0;
        return;
    }
    uint8_t *cbase = smem_raw;
    int ccap = smem_cand;
    if (n > smem_cand) {
        if (tid == 0) sh_misc[0] = atomicAdd(scratch_next, 1);
        __syncthreads();
        const int slot = sh_misc[0];
        __syncthreads();
        if (slot >= scratch_slots) {
            if (tid == 0) {
                atomicOr(&S.flags[img], kFlagNodeOverflow);
                *kp_count = 0;
            }
            return;
        }
        ccap = max_cand;
        cbase = scratch + (size_t)slot * max_cand * kCandBytes;
    }
    OctSmemT<kWide> M;
    {
        uint8_t *p = cbase;
        M.pk[0] = (uint32_t *)p; p += sizeof(uint32_t) * ccap;
        M.pk[1] = (uint32_t *)p; p += sizeof(uint32_t) * ccap;
        M.own[0] = (uint16_t *)p; p += sizeof(uint16_t) * ccap;
        M.own[1] = (uint16_t *)p; p += sizeof(uint16_t) * ccap;
        M.qs = (pos_t *)p;
        p = smem_raw + (size_t)smem_cand * kCandBytes;
        M.child = (uint32_t *)p; p += sizeof(uint32_t) * 4 * max_nodes;
        M.tord = (int *)p; p += sizeof(int) * max_nodes;
        M.arr_a = (int *)p; p += sizeof(int) * max_nodes;
        M.arr_b = (int *)p; p += sizeof(int) * max_nodes;
        M.warp_sums = (int *)p; p += sizeof(int) * 32;
        M.nd[0] = (ONode *)p; p += sizeof(ONode) * max_nodes;
        M.nd[1] = (ONode *)p; p += sizeof(ONode) * max_nodes;
        M.eidx[0] = (uint16_t *)p; p += sizeof(uint16_t) * max_nodes;
        M.eidx[1] = (uint16_t *)p; p += sizeof(uint16_t) * max_nodes;
        M.childpos = (uint16_t *)p; p += sizeof(uint16_t) * 4 * max_nodes;
    }
    const uint32_t *cand = S.cand + (size_t)img * S.cand_stride + L.cand_off;
    const int n_ini = L.n_ini, n_want = L.quota;
    const float hx = L.hx;
    int nL;
    bool finished = false;
    if (L.ff_depth > 0) {
        nL = octree_build_at_depth<kWide>(M, cand, n, n_ini, hx, L.win_h, L.ff_depth, &finished);
    } else {
    // roots (:543-585): point -> root (int)(x / hX); empty roots are dropped
    for (int i = tid; i < n_ini; i += T) M.child[i] = 0;
    __syncthreads();
    for (int p = tid; p < n; p += T) {
        const uint32_t v = cand[p];
        int r = (int)__fdiv_rn((float)(v & 0xFFF), hx);
        r = min(r, n_ini - 1);
        M.own[1][p] = (uint16_t)r;
        M.qs[p] = (pos_t)atomicAdd(&M.child[r], 1u);
    }
    __syncthreads();
    if (n_ini <= 32) {  // the usual handful of roots: one warp scans them
        if (tid < 32) {
            const int c = tid < n_ini ? (int)M.child[tid] : 0;
            int a = c, b = c > 0;
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
                const int ua = __shfl_up_sync(0xffffffffu, a, o), ub = __shfl_up_sync(0xffffffffu, b, o);
                if (tid >= o) { a += ua; b += ub; }
            }
            if (tid < n_ini) {
                M.arr_a[tid] = a - c;
                M.arr_b[tid] = b - (c > 0);
            }
            if (tid == 31) sh_misc[1] = b;
        }
        __syncthreads();
        nL = sh_misc[1];
    } else {
        for (int i = tid; i < n_ini; i += T) {
            M.arr_a[i] = M.child[i];
            M.arr_b[i] = M.child[i] > 0;
        }
        __syncthreads();
        block_excl_scan(M.arr_a, n_ini, M.warp_sums);
        nL = block_excl_scan(M.arr_b, n_ini, M.warp_sums);
    }
    for (int i = tid; i < n_ini; i += T) {
        const int c = M.child[i];
        if (c > 0) {
            ONode o;
            o.x0 = (short)(int)__fmul_rn(hx, (float)i);
            o.x1 = (short)(int)__fmul_rn(hx, (float)(i + 1));
            o.y0 = 0;
            o.y1 = (short)L.win_h;
            o.start = (pos_t)M.arr_a[i];
            o.cnt = (pos_t)c;
            M.nd[0][M.arr_b[i]] = o;
            M.eidx[0][M.arr_b[i]] = 0;
        }
    }
    __syncthreads();
    for (int p = tid; p < n; p += T) {
        const int r = M.own[1][p];
        const int np = M.arr_a[r] + M.qs[p];
        M.pk[0][np] = cand[p];
        M.own[0][np] = (uint16_t)M.arr_b[r];
    }
    __syncthreads();
    }
    // main loop (:587-739)
    int cur = 0;
    const bool overflow = false;
    while (!finished) {
        // a full pass is only entered with nL <= n_ini or nL + 3 * nExpand <= quota, so the next
        // list always fits max_nodes >= max(quota + 8, 4 * n_ini + 5)
        const int prev = nL;
        int n_expand;
        nL = octree_pass(M, cur, n, nL, n_want, false, &n_expand, sh_misc);
        cur ^= 1;
        if (nL >= n_want || nL == prev) break;
        if (nL + 3 * n_expand > n_want) {
            for (;;) {
                const int prev2 = nL;
                nL = octree_pass(M, cur, n, nL, n_want, true, &n_expand, sh_misc);
                cur ^= 1;
                if (nL >= n_want || nL == prev2) break;
            }
            break;
        }
    }
    if (overflow || nL > L.kp_cap) {
        if (tid == 0) {
            atomicOr(&S.flags[img], kFlagNodeOverflow);
            *kp_count = 0;
        }
        return;
    }
    // retain the best point of every node (:742-760): max response, earliest in the reference's
    // candidate order (cell-row-major, raster inside the cell) on ties
    uint32_t *out = S.kpst + (size_t)img * S.kpst_stride + L.kp_off;
    for (int i = tid; i < nL; i += T) {
        const ONode o = M.nd[cur][i];
        uint32_t best = 0;
        unsigned long long best_key = 0;
        for (int p = (int)o.start; p < (int)(o.start + o.cnt); p++) {
            const uint32_t v = M.pk[cur][p];
            const uint32_t x = v & 0xFFF, y = (v >> 12) & 0xFFF, r = v >> 24;
            const uint32_t ci = (y - 3) / L.h_cell, cj = (x - 3) / L.w_cell;
            const unsigned long long ord = (((unsigned long long)ci * 4096 + cj) * 4096 + y) * 4096 + x;
            const unsigned long long key = (unsigned long long)r << 48 | (0xFFFFFFFFFFFFull - ord);
            if (p == (int)o.start || key > best_key) { best_key = key; best = v; }
        }
        out[i] = best;
    }
    if (tid == 0) *kp_count = nL;
}

// (level, image) items in level-major order -- the fullest levels first -- handed out round-robin: with one CTA per item
// this is the plain launch, with fewer CTAs (SFE_OCTREE_CTAS) the kernel is persistent and leaves shared memory to a
// kernel running beside it.
template <bool kWide>
__global__ void __launch_bounds__(1024) octree_kernel(ImgSet S, int count, int level0, int level_n, int smem_cand, int max_cand, int max_nodes,
                                                     uint8_t *__restrict__ scratch, int scratch_slots, int *scratch_next) {
    pdl_enter();
    const int items = level_n * count;  // levels [level0, level0 + level_n)
    for (int w = blockIdx.x; w < items; w += gridDim.x) {
        octree_item<kWide>(S, level0 + w / count, w % count, smem_cand, max_cand, max_nodes, scratch, scratch_slots, scratch_next);
        __syncthreads();  // the next item reuses the shared arrays
    }
}

// ---------------------------------------------------------------------------------------------
// cv::GaussianBlur(7x7, sigma 2, BORDER_REFLECT_101) fixed-point model (:1085-1086)
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ int reflect101(int i, int n) {
    if (i < 0) i = -i;
    if (i >= n) i = 2 * n - 2 - i;
    return min(max(i, 0), n - 1);  // only reached by halo pixels of outputs outside the image
}

// Tile = 128 x 32 outputs, Q8 kernel [18 34 48 56 48 34 18]; sums are exact integers, the only rounding is
// the final (v + 2^15) >> 16, exactly cv::GaussianBlur's fixed-point path.
//   load        (32+6) rows x 36 words (x0-4 .. x0+139) into shared memory.  kTma: one TMA box issued by
//               thread 0, out-of-image bytes arrive as zeros and the tiles on the image border rebuild their
//               BORDER_REFLECT_101 halo from the tile itself; otherwise aligned global words (one 32-bit store
//               per 4 px), border words assembled byte by byte
//   horizontal  4 outputs x 2 rows per thread from three shared words per row: two IDP.4A per output on byte-shifted
//               windows (PRMT); the two rows' sums of a column are packed into one word (a sum never exceeds
//               255 * 256 = 65280)
//   vertical    4 columns x 4 rows per thread: four IDP.2A per output on the row pairs, the rounding constant
//               folded into the first, result bytes picked with PRMT, one 32-bit store per row
template <bool kTma>
__global__ void __launch_bounds__(256) blur_kernel(ImgSet S, const TilePlan *__restrict__ tiles,
                                                   const __grid_constant__ TmaMaps M) {
    pdl_enter();
    constexpr int IH = kBlurTileH + 6, IWW = kBlurInWords;
    static_assert(IH % 2 == 0 && kBlurTileW == 128 && kBlurTileH == 32, "the blur passes pair rows and map 32 x 8 threads onto the tile");
    __shared__ __align__(128) uint32_t in32[IH * IWW];
    __shared__ __align__(16) uint32_t hb[(IH / 2) * kBlurTileW];  // horizontal sums: word = (row 2p, row 2p + 1) of one column, u16 each
    __shared__ uint64_t bar;
    const TilePlan t = tiles[blockIdx.x];
    const int img = blockIdx.y, tid = threadIdx.x, l = t.level;
    const int slot = slot_of(S, img);
    // (the reference blurs only levels that kept keypoints, :1085; blurring all of them changes no output and lets
    // this kernel run beside FAST / quadtree instead of after them)
    const LevelPlan &L = S.lv[l];
    const int w = L.w, h = L.h, x_first = t.x0 - kBlurLead, y_first = t.y0 - 3;
    if (kTma) {
        if (tid == 0) {
            mbar_init(&bar, 1);
            mbar_expect_tx(&bar, IH * IWW * 4);
            const bool set_a = img < S.split;
            const CUtensorMap *map = l == 0 ? (set_a ? &M.lv[0] : &M.l0b) : &M.lv[l];
            const int z = l == 0 ? S.in_z0 + (set_a ? img : img - S.split) : slot;
            tma_load_3d(in32, map, &bar, x_first, y_first, z);
        }
        __syncthreads();  // barrier initialised
        mbar_wait(&bar, 0);
        // BORDER_REFLECT_101 for tiles on the image border (levels are >= 8 px per side on this path): the
        // source pixel of every missing one lies inside this tile.  Columns first, then whole rows.
        uint8_t *in8 = (uint8_t *)in32;
        if (t.x0 == 0 || t.x0 + kBlurTileW + 3 > w) {
            for (int it = tid; it < IH * 6; it += 256) {
                const int r = (it * 10923) >> 16, k = it - r * 6;  // it / 6 for it < 228
                const int x = k < 3 ? k - 3 : w + (k - 3);
                const int c = x - x_first, sc = (k < 3 ? -x : 2 * w - 2 - x) - x_first;
                if (c >= 0 && c < IWW * 4 && sc >= 0) in8[r * IWW * 4 + c] = in8[r * IWW * 4 + sc];
            }
            __syncthreads();
        }
        if (t.y0 == 0 || t.y0 + kBlurTileH + 3 > h) {
            for (int it = tid; it < 6 * IWW; it += 256) {
                const int k = (it * (65536 / IWW + 1)) >> 16, j = it - k * IWW;  // it / IWW for it < 6 * IWW
                const int y = k < 3 ? k - 3 : h + (k - 3);
                const int r = y - y_first, sr = (k < 3 ? -y : 2 * h - 2 - y) - y_first;
                if (r >= 0 && r < IH && sr >= 0) in32[r * IWW + j] = in32[sr * IWW + j];
            }
            __syncthreads();
        }
    } else {
        int pitch;
        const uint8_t *src = level_pixels(S, l, img, pitch);
        constexpr int kFirst = kBlurLead / 4 - 1, kWords = kBlurTileW / 4 + 2;  // only x0-4 .. x0+131 is ever read
        for (int it = tid; it < IH * kWords; it += 256) {
            const int r = (it * (65536 / kWords + 1)) >> 16, j = kFirst + it - r * kWords;  // exact for it < 4000
            int yy = y_first + r;
            if ((unsigned)yy >= (unsigned)h) yy = reflect101(yy, h);
            const uint8_t *row = src + (size_t)yy * pitch;
            const int x = x_first + 4 * j;
            uint32_t v;
            if (x >= 0 && x + 8 <= w) {
                v = ldg_word_at(row + x);
            } else {
                v = __ldg(row + reflect101(x, w)) | (uint32_t)__ldg(row + reflect101(x + 1, w)) << 8 |
                    (uint32_t)__ldg(row + reflect101(x + 2, w)) << 16 | (uint32_t)__ldg(row + reflect101(x + 3, w)) << 24;
            }
            in32[r * IWW + j] = v;
        }
        __syncthreads();
    }
    // horizontal: item = (row pair rp, group g of 4 outputs).  Output k of a row = taps on bytes 4g+k-3 .. 4g+k+3 = one
    // IDP.4A over the byte window starting at 4g+k-3 (taps 0..3) + one over the window at 4g+k+1 (taps 4..6); the
    // windows are byte shifts of three consecutive words.  The two rows' sums of a column share a word (u16 each, a sum
    // never exceeds 255 * 256), which is the operand layout IDP.2A wants for the vertical pass.
    constexpr uint32_t kTapLo = 18u | 34u << 8 | 48u << 16 | 56u << 24, kTapHi = 48u | 34u << 8 | 18u << 16;
    for (int it = tid; it < (IH / 2) * (kBlurTileW / 4); it += 256) {
        const int rp = it >> 5, g = it & 31;
        uint32_t hsum[2][4];
#pragma unroll
        for (int q = 0; q < 2; q++) {
            const uint32_t *wp = &in32[(2 * rp + q) * IWW + g + (kBlurLead / 4 - 1)];
            const uint32_t w0 = wp[0], w1 = wp[1], w2 = wp[2];
            hsum[q][0] = dp4a_u8u8(__byte_perm(w0, w1, 0x4321), kTapLo, dp4a_u8u8(__byte_perm(w1, w2, 0x4321), kTapHi, 0));
            hsum[q][1] = dp4a_u8u8(__byte_perm(w0, w1, 0x5432), kTapLo, dp4a_u8u8(__byte_perm(w1, w2, 0x5432), kTapHi, 0));
            hsum[q][2] = dp4a_u8u8(__byte_perm(w0, w1, 0x6543), kTapLo, dp4a_u8u8(__byte_perm(w1, w2, 0x6543), kTapHi, 0));
            hsum[q][3] = dp4a_u8u8(w1, kTapLo, dp4a_u8u8(w2, kTapHi, 0));
        }
        *(uint4 *)&hb[rp * kBlurTileW + 4 * g] =
            make_uint4(__byte_perm(hsum[0][0], hsum[1][0], 0x5410), __byte_perm(hsum[0][1], hsum[1][1], 0x5410),
                       __byte_perm(hsum[0][2], hsum[1][2], 0x5410), __byte_perm(hsum[0][3], hsum[1][3], 0x5410));
    }
    __syncthreads();
    // vertical: thread = (4 columns, strip of 4 output rows).  Output row k taps tile rows k .. k+6; with the rows paired
    // (2p, 2p+1) that is four IDP.2A per pixel, the pair coefficients depending on the parity of k.
    uint8_t *dst = S.blur + (size_t)slot * S.blur_stride + L.blur_off;
    const int cg = tid & 31, r0 = (tid >> 5) * 4;  // r0 is even: the strip starts on a pair
    const int gx = t.x0 + 4 * cg;
    if (gx >= w) return;
    uint4 pr[5];  // pairs r0/2 .. r0/2 + 4 = tile rows r0 .. r0 + 9, four columns each
#pragma unroll
    for (int p = 0; p < 5; p++) pr[p] = *(const uint4 *)&hb[(r0 / 2 + p) * kBlurTileW + 4 * cg];
    constexpr uint32_t kEvenA = 18u | 34u << 8 | 48u << 16 | 56u << 24, kEvenB = 48u | 34u << 8 | 18u << 16;   // (c0 c1)(c2 c3) (c4 c5)(c6 0)
    constexpr uint32_t kOddA = 18u << 8 | 34u << 16 | 48u << 24, kOddB = 56u | 48u << 8 | 34u << 16 | 18u << 24;  // (0 c0)(c1 c2) (c3 c4)(c5 c6)
#pragma unroll
    for (int k = 0; k < 4; k++) {
        const int gy = t.y0 + r0 + k;
        if (gy >= h) break;
        const int p = k >> 1;
        uint32_t v[4];
#pragma unroll
        for (int c = 0; c < 4; c++) {
            const uint32_t a0 = (&pr[p].x)[c], a1 = (&pr[p + 1].x)[c], a2 = (&pr[p + 2].x)[c], a3 = (&pr[p + 3].x)[c];
            v[c] = (k & 1) ? dp2a_hi(a3, kOddB, dp2a_lo(a2, kOddB, dp2a_hi(a1, kOddA, dp2a_lo(a0, kOddA, 32768u))))
                           : dp2a_hi(a3, kEvenB, dp2a_lo(a2, kEvenB, dp2a_hi(a1, kEvenA, dp2a_lo(a0, kEvenA, 32768u))));
        }
        // (v + 2^15) >> 16 <= 255 is byte 2 of each sum
        *(uint32_t *)(dst + (size_t)gy * L.blur_pitch + gx) =
            __byte_perm(__byte_perm(v[0], v[1], 0x0062), __byte_perm(v[2], v[3], 0x0062), 0x5410);  // pitch, gx multiples of 4
    }
}

// ---------------------------------------------------------------------------------------------
// IC_Angle (:77-104) + rBRIEF (:107-147), one warp per keypoint; also the final keypoint record
// ---------------------------------------------------------------------------------------------
__device__ const signed char g_pattern[1024] = {
#include "orb_pattern_data.inc"
};

// cv::fastAtan2 (degree-7 polynomial, float32)
__device__ __forceinline__ float fast_atan2_deg(float y, float x) {
    // OpenCV: atan2_pN = <coef>f * (float)(180 / CV_PI), folded at compile time in float
    constexpr float s = (float)(180.0 / 3.1415926535897932384626433832795);
    constexpr float p1 = 0.9997878412794807f * s, p3 = -0.3258083974640975f * s, p5 = 0.1555786518463281f * s,
                    p7 = -0.04432655554792128f * s;
    const float ax = fabsf(x), ay = fabsf(y);
    const float eps = 2.220446049250313e-16f;
    float a, c, c2;
    if (ax >= ay) {
        c = __fdiv_rn(ay, __fadd_rn(ax, eps));
        c2 = __fmul_rn(c, c);
        a = __fmul_rn(__fadd_rn(__fmul_rn(__fadd_rn(__fmul_rn(__fadd_rn(__fmul_rn(p7, c2), p5), c2), p3), c2), p1), c);
    } else {
        c = __fdiv_rn(ax, __fadd_rn(ay, eps));
        c2 = __fmul_rn(c, c);
        a = __fsub_rn(90.f, __fmul_rn(__fadd_rn(__fmul_rn(__fadd_rn(__fmul_rn(__fadd_rn(__fmul_rn(p7, c2), p5), c2), p3), c2), p1), c));
    }
    if (x < 0) a = __fsub_rn(180.f, a);
    if (y < 0) a = __fsub_rn(360.f, a);
    return a;
}

// The disc |u| <= umax[|dv|] is symmetric (|dv| <= umax[|u|] describes the same set), so the rows a column
// u touches are the contiguous range |dv| <= umax[|u|].  Checked at compile time against the table.
constexpr int kUmax[16] = {15, 15, 15, 15, 14, 14, 14, 13, 13, 12, 11, 10, 9, 8, 6, 3};
constexpr bool disc_is_symmetric() {
    for (int u = 0; u < 16; u++)
        for (int v = 0; v < 16; v++)
            if ((u <= kUmax[v]) != (v <= kUmax[u])) return false;
    return true;
}
static_assert(disc_is_symmetric(), "IC_Angle disc must be symmetric");
// Per disc row dv (|dv| = 0..15) the eight 4-pixel words that cover columns u = -15 .. +16: u[j] = the column
// offsets as signed bytes, zero outside the disc; in[j] = 1 per pixel inside the disc.  One IDP.4A per word then
// gives sum(u * I) and sum(I) of four pixels at once.
struct DiscTable {
    uint32_t u[16][8], in[16][8];
};
constexpr DiscTable make_disc_table() {
    DiscTable t{};
    for (int v = 0; v < 16; v++)
        for (int j = 0; j < 8; j++)
            for (int k = 0; k < 4; k++) {
                const int u = -kHalfPatch + 4 * j + k, au = u < 0 ? -u : u;
                if (au <= kUmax[v]) {
                    t.u[v][j] |= (uint32_t)(u & 0xFF) << (8 * k);
                    t.in[v][j] |= 1u << (8 * k);
                }
            }
    return t;
}
__device__ const DiscTable g_disc = make_disc_table();

__device__ __forceinline__ int dp4a_u8s8(uint32_t pix, uint32_t w, int acc) {  // acc + sum_k u8(pix.k) * s8(w.k)
    int d;
    asm("dp4a.u32.s32 %0, %1, %2, %3;" : "=r"(d) : "r"(pix), "r"(w), "r"(acc));
    return d;
}

constexpr int kPatchR = 18;      // rBRIEF pattern radius: max |(x, y)| = |(-13, -13)| = 18.4, rounds to at most 18
constexpr int kPatchRows = 2 * kPatchR + 1, kPatchWords = 10;  // 37 px + up to 3 px of word alignment = 40 bytes
constexpr signed char kPatternHost[1024] = {
#include "orb_pattern_data.inc"
};
constexpr bool pattern_within_patch() {
    for (int i = 0; i < 512; i++) {
        const int px = kPatternHost[2 * i], py = kPatternHost[2 * i + 1];
        if (4 * (px * px + py * py) >= (2 * kPatchR + 1) * (2 * kPatchR + 1)) return false;  // |p| < R + 0.5
    }
    return true;
}
static_assert(pattern_within_patch(), "a rotated pattern point could round outside the staged window");
#ifndef SFE_KP_PER_WARP
#define SFE_KP_PER_WARP 8
#endif
constexpr int kKpPerWarp = SFE_KP_PER_WARP;  // keypoints one warp handles in turn: the pattern / disc table set-up is paid once

// kTma: both windows of a keypoint -- the 31 rows x 48 bytes of the unblurred level around it for IC_Angle and the 37 rows x
// 64 bytes of the blurred level for rBRIEF, each starting on the 16-byte grid of its row -- arrive by two TMA boxes issued by
// lane 0 of the keypoint's warp; otherwise the lanes read the first with global loads and stage the second themselves.
constexpr int kIcBoxW = 48, kIcBoxH = 2 * kHalfPatch + 1, kBdBoxW = 64, kBdBoxH = kPatchRows;
constexpr int kIcBytes = 1536, kWinBytes = kIcBytes + 2432;  // per warp: IC box (1488 B) padded to 128, blurred box (2368 B) padded
struct OrientMaps {
    CUtensorMap ic[kMaxLevels], ic_l0b;  // unblurred levels (ic[0] / ic_l0b = the level-0 images of set A / set B of the call)
    CUtensorMap bd[kMaxLevels];          // blurred levels
};

template <bool kTma>
__global__ void __launch_bounds__(256, 5) orient_describe_kernel(ImgSet S, OutSet O, int kp_per_warp, const __grid_constant__ OrientMaps M) {
    __shared__ float2 pat[16 * 32];  // pat[s * 32 + lane] = sample s of descriptor byte `lane` (floats: no conversion in the loop)
    __shared__ __align__(128) uint8_t win_all[8][kTma ? kWinBytes : kPatchRows * kPatchWords * 4];  // per warp: the windows
    __shared__ uint64_t bars[8];
    pdl_enter();
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, img = blockIdx.y, slot = slot_of(S, img);
    uint32_t *patch = (uint32_t *)win_all[warp];
    uint32_t phase = 0;
    if (kTma && lane == 0) mbar_init(&bars[warp], 1);
    for (int i = tid; i < 512; i += 256) {
        const int byte = i >> 4, s = i & 15;
        pat[s * 32 + byte] = make_float2((float)g_pattern[2 * i], (float)g_pattern[2 * i + 1]);
    }
    // IC_Angle: the 31 x 32-byte window is 31 rows x 8 words; lane = word (lane & 7) of the rows ic_row(t), t = 0..7: step t
    // covers rows b, b + 2, b + 4, b + 6 with b = 8 (t / 2) + t % 2, so one warp-wide load touches 4 rows (4-8 cache
    // lines) and, in the TMA box with its 12-word rows, 32 different banks.  The lane's weights stay in registers.
    const int wj = lane & 7, wr0 = 2 * (lane >> 3);
    auto ic_row = [wr0](int t) { return 8 * (t >> 1) + (t & 1) + wr0; };
    uint32_t wu[8], win[8];
#pragma unroll
    for (int t = 0; t < 8; t++) {
        const int r = ic_row(t), adv = r < 31 ? (r < kHalfPatch ? kHalfPatch - r : r - kHalfPatch) : 0;
        wu[t] = r < 31 ? __ldg(&g_disc.u[adv][wj]) : 0u;
        win[t] = r < 31 ? __ldg(&g_disc.in[adv][wj]) : 0u;
    }
    __syncthreads();
    // keypoints are the levels' survivors concatenated 0..L-1 (:1076-1104); lane k holds level k's count
    const int cnt = lane < S.nlevels ? min(S.kp_count[slot * S.nlevels + lane], S.lv[lane].kp_cap) : 0;
    int inc = cnt;
#pragma unroll
    for (int o = 1; o < kMaxLevels; o <<= 1) {
        const int u = __shfl_up_sync(0xffffffffu, inc, o);
        if (lane >= o) inc += u;
    }
    const int total = __shfl_sync(0xffffffffu, inc, kMaxLevels - 1);
    const bool set_a = img < S.split;
    const int oi = set_a ? img : img - S.split;
    if (blockIdx.x == 0 && tid == 0) {
        (set_a ? O.n_a : O.n_b)[oi] = min(total, O.cap);
        if (total > O.cap) atomicOr(&S.flags[slot], kFlagOutOverflow);
    }
    const int g0 = (blockIdx.x * 8 + warp) * kp_per_warp;
    for (int g = g0; g < g0 + kp_per_warp; g++) {
        if (g >= total || g >= O.cap) return;
        const int l = __popc(__ballot_sync(0xffffffffu, lane < S.nlevels && inc <= g));  // first level whose prefix exceeds g
        const int local = g - __shfl_sync(0xffffffffu, inc - cnt, min(l, 31));
        const LevelPlan &L = S.lv[l];
        const uint32_t v = S.kpst[(size_t)slot * S.kpst_stride + L.kp_off + local];
        const int x = (v & 0xFFF) + kBorder, y = ((v >> 12) & 0xFFF) + kBorder;
        int pitch;
        const uint8_t *lvl = level_pixels(S, l, img, pitch);
        // intensity centroid over the 31-px disc on the UNBLURRED level (:77-104): m_10 = sum u * I, m_01 = sum dv * I.
        // Word j of a row = pixels x - 15 + 4 j .. + 3, assembled from the two aligned words around it (rows may
        // start at any byte); the last word reaches x + 20 at most: keypoints keep 19 px from the border, so that
        // stays inside the row or spills 2 bytes into the next one.  Four pixels per IDP.4A.
        int m10 = 0, m01 = 0;
        const int xl = x - kPatchR, xb0 = xl & ~15;  // blurred window: first column, and the 16-byte grid column before it
        if (kTma) {
            const int xi = x - kHalfPatch, xi0 = xi & ~15;
            __syncwarp();  // the previous keypoint's reads of both windows are done
            if (lane == 0) {
                mbar_expect_tx(&bars[warp], kIcBoxW * kIcBoxH + kBdBoxW * kBdBoxH);
                const bool sa = img < S.split;
                const CUtensorMap *mi = l == 0 ? (sa ? &M.ic[0] : &M.ic_l0b) : &M.ic[l];
                tma_load_3d(win_all[warp], mi, &bars[warp], xi0, y - kHalfPatch, l == 0 ? S.in_z0 + (sa ? img : img - S.split) : slot);
                tma_load_3d(win_all[warp] + kIcBytes, &M.bd[l], &bars[warp], xb0, y - kPatchR, slot);
            }
            mbar_wait(&bars[warp], phase);
            phase ^= 1;
            const int o = xi - xi0;  // 0..15: byte offset of the window's first pixel inside the box row
            const uint32_t *w0 = (const uint32_t *)(win_all[warp] + (o & ~3) + 4 * wj);
            const uint32_t sh8 = (uint32_t)(o & 3) * 8;
#pragma unroll
            for (int t = 0; t < 8; t++) {
                const int r = ic_row(t);
                if (r < 31) {
                    const uint32_t *wp = w0 + r * (kIcBoxW / 4);
                    const uint32_t px = __funnelshift_r(wp[0], wp[1], sh8);
                    m10 = dp4a_u8s8(px, wu[t], m10);
                    m01 += (r - kHalfPatch) * dp4a_u8s8(px, win[t], 0);
                }
            }
        } else {
            const uint8_t *r0p = lvl + (size_t)(y - kHalfPatch) * pitch + (x - kHalfPatch + 4 * wj);
#pragma unroll
            for (int t = 0; t < 8; t++) {
                const int r = ic_row(t);
                if (r < 31) {
                    const uint8_t *rp = r0p + (size_t)r * pitch;
                    const uint32_t *wp = (const uint32_t *)((uintptr_t)rp & ~(uintptr_t)3);
                    const uint32_t px = __funnelshift_r(__ldg(wp), __ldg(wp + 1), ((uint32_t)(uintptr_t)rp & 3) * 8);
                    m10 = dp4a_u8s8(px, wu[t], m10);
                    m01 += (r - kHalfPatch) * dp4a_u8s8(px, win[t], 0);
                }
            }
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            m01 += __shfl_xor_sync(0xffffffffu, m01, o);
            m10 += __shfl_xor_sync(0xffffffffu, m10, o);
        }
        const float angle = fast_atan2_deg((float)m01, (float)m10);
        // rotated pattern lookups on the blurred level; float ops rounded one by one (T2)
        float a = 0.f, b = 0.f;
        if (lane == 0) {
            const float factor_pi = (float)(3.1415926535897932384626433832795 / 180.0);
            const float rad = __fmul_rn(angle, factor_pi);
            double sn, cs;
            sincos((double)rad, &sn, &cs);
            a = (float)cs;
            b = (float)sn;
        }
        a = __shfl_sync(0xffffffffu, a, 0);
        b = __shfl_sync(0xffffffffu, b, 0);
        // The 512 pattern points lie within 18.4 px of the centre, so every rotated sample falls in the 37 x 37 window
        // around the keypoint: the warp copies it to shared memory with row-coalesced word loads (3 rows of 10 aligned
        // words per step; blurred planes have 16-byte pitches, so all rows share one alignment) and gathers from there
        // instead of sending 16 scattered loads per lane through L1.
        const uint8_t *pc;  // the keypoint's pixel inside the staged blurred window
        int wpitch;
        if (kTma) {
            wpitch = kBdBoxW;
            pc = win_all[warp] + kIcBytes + kPatchR * kBdBoxW + (xl - xb0) + kPatchR;
        } else {
            const int bp = L.blur_pitch;
            const uint8_t *bl = S.blur + (size_t)slot * S.blur_stride + L.blur_off;
            const int al = xl & 3;        // the window's first column inside an aligned word
            __syncwarp();                 // the previous keypoint's gathers are done
            if (lane < 3 * kPatchWords) {
                const int rs = lane / kPatchWords, c = lane - rs * kPatchWords;
                const uint32_t *src = (const uint32_t *)(bl + (size_t)(y - kPatchR + rs) * bp + (xl - al)) + c;
                uint32_t *dst = patch + rs * kPatchWords + c;
#pragma unroll
                for (int r = rs; r < kPatchRows; r += 3, src += 3 * (bp >> 2), dst += 3 * kPatchWords) *dst = __ldg(src);
            }
            __syncwarp();
            wpitch = kPatchWords * 4;
            pc = (const uint8_t *)patch + kPatchR * (kPatchWords * 4) + kPatchR + al;
        }
        uint32_t byte = 0;
#pragma unroll
        for (int k = 0; k < 8; k++) {
            int tv[2];
#pragma unroll
            for (int s = 0; s < 2; s++) {
                const float2 pp = pat[(2 * k + s) * 32 + lane];
                const int ry = __float2int_rn(__fadd_rn(__fmul_rn(pp.x, b), __fmul_rn(pp.y, a)));
                const int rx = __float2int_rn(__fsub_rn(__fmul_rn(pp.x, a), __fmul_rn(pp.y, b)));
                tv[s] = pc[ry * wpitch + rx];
            }
            byte |= (uint32_t)(tv[0] < tv[1]) << k;
        }
        uint8_t *desc = (set_a ? O.desc_a : O.desc_b) + ((size_t)oi * O.cap + g) * 32;
        desc[lane] = (uint8_t)byte;
        if (lane == 0) {
            sfe_keypoint kp;
            kp.x = (float)x;
            kp.y = (float)y;
            if (l != 0) {  // :1095-1101
                kp.x = __fmul_rn(kp.x, L.scale);
                kp.y = __fmul_rn(kp.y, L.scale);
            }
            kp.size = L.size;
            kp.angle = angle;
            kp.response = (float)(v >> 24);
            kp.octave = l;
            kp.class_id = -1;
            (set_a ? O.kps_a : O.kps_b)[(size_t)oi * O.cap + g] = kp;
        }
    }
}

}  // namespace sfe

// =============================================================================================
// host side: the extractor handle
// =============================================================================================
using namespace sfe;

enum { kStagePyramid, kStageFast, kStageQuadtree, kStageBlur, kStageDescribe, kStageStereo, kStageTrack, kNumStages };
constexpr int kOctreeSmemCand = 3072;
constexpr int kComputeStreams = 4;
constexpr int kMaxChunks = 16;  // sub-batches one pipelined host call is cut into

struct sfe_extractor {
    int device = 0;
    cudaStream_t stream = nullptr;                  // compute (and everything, for unpipelined calls)
    cudaStream_t s_h2d = nullptr, s_d2h = nullptr;  // copy streams of the pipelined host entry points
    cudaStream_t extra[kComputeStreams - 1] = {};   // further compute streams: sub-batch c runs on stream c % n_compute, so the
                                                    // kernels of one sub-batch fill the tail waves / latency-bound stages of others
    int n_compute = 3;                              // SFE_COMPUTE_STREAMS
    cudaStream_t aux[3] = {nullptr, nullptr, nullptr};  // [0] the blur beside FAST + quadtree, [1] the matchers of an asynchronous call beside the next
                                                        // call, [2] FAST + quadtree of levels 0-1 of a few-image call beside the rest of the pyramid
    cudaEvent_t ev_fork[3] = {}, ev_join[3] = {};
    int dev_split = 3;                              // SFE_DEV_SPLIT=n: a resident stereo batch runs as n sub-batches on n streams
    bool split_small = false;                       // SFE_SPLIT_SMALL=1: few-image calls run FAST + quadtree of levels 0-1 beside the pyramid tail
                                                    // (measured: no gain, 195 vs 198 us per stereo pair; DESIGN.md §9)
    int octree_ctas = 0;    // SFE_OCTREE_CTAS: > 0 = persistent quadtree kernel with that many CTAs
    int sm_count = 148;
    bool piped_now = false; // a pipelined host call is enqueueing its sub-batches
    bool orient_tma = true; // SFE_ORIENT_TMA=0: the orientation / descriptor kernel stages its windows with plain loads
    bool overlap_tail = true;   // SFE_OVERLAP_TAIL=0 turns it off: asynchronous resident stereo calls run StereoMatch + tracking on
    bool tail_pending = false;  // aux[1], beside the next call's pyramid / FAST (the next call's descriptor kernel, the first
                                // writer of the caller's output arrays, waits for it: ev_join[1])
    int overlap_blur = 2;   // SFE_OVERLAP_BLUR: 0 off, 1 = blur forks before FAST (no gain: both kernels fill the machine on their
                            // own), 2 = blur forks after FAST and runs beside the latency-bound quadtree (default)
    cudaEvent_t ev_start = nullptr;
    bool async_dev = false;                         // _dev entry points return after enqueueing (sfe_extractor_wait)
    cudaEvent_t ev_in[kMaxChunks] = {}, ev_done[kMaxChunks] = {};
    int chunks_override = 0;                        // SFE_PIPELINE_CHUNKS
    bool trace = false;                             // SFE_TRACE=1: per-sub-batch timeline of the host pipeline on stderr
    cudaEvent_t tr_ev[3 * kMaxChunks + 1] = {};
    sfe_extractor_params prm{};
    float scale[kMaxLevels], inv_scale[kMaxLevels], sigma2[kMaxLevels], inv_sigma2[kMaxLevels];
    int quota[kMaxLevels];
    int max_images = 0;
    // geometry-dependent plan
    int w = 0, h = 0;
    LevelPlan lv[kMaxLevels];
    FastPlan fast{};
    // TMA descriptors (fast: TP x tile_rows boxes, blur: 144 x 38 boxes); level >= 1 entries follow the plan,
    // level-0 entries follow the images of the current call
    alignas(64) TmaMaps fast_maps{}, blur_maps{}, pyr_maps{};  // pyr_maps.lv[l] = level l as the SOURCE of level l + 1
    alignas(64) OrientMaps orient_maps{};                      // per-keypoint windows of the orientation / descriptor kernel
    int pyr_box_w = 0, pyr_box_h = 0;
    bool tma_plan_ok = false, tma_disabled = false, tma_now = false;
    const void *l0_key[2] = {nullptr, nullptr};
    size_t l0_geom[4] = {0, 0, 0, 0};
    int pitch0 = 0;       // row pitch of the host-path staging buffer
    std::vector<SegRec> segs;
    int seg_level_start[kMaxLevels + 1] = {};  // segments are stored level by level: level l = [start[l], start[l + 1])
    DevBuf<SegRec> d_segs;
    size_t fast_smem = 0, pyr_smem = 0;
    int pyr_wide_h[kMaxLevels] = {};
    std::vector<TilePlan> tiles;
    size_t pyr_stride = 0, blur_stride = 0;
    int cand_stride = 0, kpst_stride = 0, max_cand = 0, max_nodes = 0;
    size_t octree_smem = 0;
    int octree_smem_cand = 0, octree_slots = 0, octree_cand_override = 0;  // SFE_OCTREE_SMEM_CAND (tests)
    // CUDA graphs of the kernel sequence of small unpipelined host calls (one image, one stereo pair: the reference-shaped
    // calls): the second call with a signature captures it, later ones replay it with one launch
    struct GraphEntry {
        uint64_t plan_gen = 0;
        int frames = 0, cap = 0, stereo = 0, seen = 0;
        double sp[3] = {0, 0, 0};
        const void *ptr[7] = {};
        cudaGraphExec_t exec = nullptr;
        int64_t launches = 0;
        uint64_t used = 0;
    };
    std::vector<GraphEntry> graphs;
    uint64_t plan_gen = 0, graph_clock = 0;
    bool use_graphs = true;           // SFE_GRAPHS=0 turns it off
    bool use_pdl = true;              // SFE_PDL=0: no programmatic dependent launches in small host calls
    bool octree_ff = true;            // SFE_OCTREE_FF=0: the quadtree starts from its roots and makes every pass
    bool pdl_now = false;             // this call's kernels are launched with programmatic stream serialization
    bool octree_wide = false;         // some level's candidate buffer exceeds 16-bit positions: the quadtree runs its 32-bit instance
    int cand_floor[kMaxLevels] = {};  // per-level candidate capacity learnt from an overflow (the reference's list is unbounded,
                                      // src/orb_extractor.cpp:778-779: a call that overflows is re-run with room for what it counted)
    int cand_cap_override = 0;        // SFE_CAND_CAP (tests): initial per-level capacity instead of tested / 12
    DevBuf<uint8_t> d_octree_scratch;
    DevBuf<uint8_t> d_pyr, d_blur, d_in, d_l0, d_desc;  // d_in: images as uploaded (tight), d_l0: pitched level 0
    DevBuf<uint32_t> d_cand, d_kpst;
    DevBuf<int> d_counts;  // cand_count | kp_count | flags
    DevBuf<TilePlan> d_tiles;
    DevBuf<uint2> d_xtab, d_ytab;
    DevBuf<sfe_keypoint> d_kps;
    DevBuf<int32_t> d_nout, d_sidx, d_sdist, d_tidx, d_tdist;
    std::vector<int> h_flags;
    int *h_flags_pinned = nullptr;    // kGraphMaxImages flags written by copy_out_kernel
    uint8_t *h_stage = nullptr;       // pinned staging for the results of small calls whose output arrays are pageable
    size_t h_stage_bytes = 0;
    bool use_copy_kernel = true;      // SFE_COPY_KERNEL=0: small host calls download with cudaMemcpyAsync like large ones
    int64_t launches = 0;
    // optional per-stage CUDA-event timing on the handle's own stream (bench roofline)
    bool profiling = false;
    cudaEvent_t prof_ev[kNumStages + 1] = {};
    bool prof_pending = false, prof_has_stereo = false, prof_has_track = false;
    TrackScratch track;  // sfe_stereo_sequence: per-frame bucket grids + keys
    double stage_ms[kNumStages] = {};
    int64_t stage_calls = 0;
    // what the last call processed (stage taps)
    ImgSet last{};
    int last_count = 0;
};

static inline int cv_round_f(float v) { return (int)nearbyintf(v); }

static inline void prof_mark(sfe_extractor *ex, int i) {
    if (ex->profiling) cudaEventRecord(ex->prof_ev[i], ex->stream);
}

// ctor tables, reference src/orb_extractor.cpp:410-446
static void build_tables(sfe_extractor *ex) {
    const int nl = ex->prm.nlevels;
    const double sf = (double)ex->prm.scale_factor;  // the member is a double initialised from float
    ex->scale[0] = 1.0f;
    ex->sigma2[0] = 1.0f;
    for (int i = 1; i < nl; i++) {
        ex->scale[i] = (float)((double)ex->scale[i - 1] * sf);
        ex->sigma2[i] = ex->scale[i] * ex->scale[i];
    }
    for (int i = 0; i < nl; i++) {
        ex->inv_scale[i] = 1.0f / ex->scale[i];
        ex->inv_sigma2[i] = 1.0f / ex->sigma2[i];
    }
    const float factor = (float)(1.0 / sf);
    const float denom = 1 - (float)pow((double)factor, (double)nl);
    float want = (float)ex->prm.nfeatures * (1 - factor) / denom;
    int sum = 0;
    for (int l = 0; l < nl - 1; l++) {
        ex->quota[l] = cv_round_f(want);
        sum += ex->quota[l];
        want *= factor;
    }
    ex->quota[nl - 1] = std::max(ex->prm.nfeatures - sum, 0);
}

// geometry plan for a w x h input: level sizes (:1111-1112), FAST cells (:771-806), quadtree roots
// (:543-545), buffer layout, resize tables (cv::resize INTER_LINEAR coefficient tables)
static void drop_graphs(sfe_extractor *ex) {
    for (auto &g : ex->graphs)
        if (g.exec) cudaGraphExecDestroy(g.exec);
    ex->graphs.clear();
}

static int build_plan(sfe_extractor *ex, int w, int h) {
    const int nl = ex->prm.nlevels;
    drop_graphs(ex);  // they hold the old buffers and geometry
    ex->plan_gen++;
    std::vector<uint2> xtab, ytab;
    int max_src_rows = 1, max_src_cols = 1;
    memset(&ex->fast, 0, sizeof(ex->fast));
    ex->segs.clear();
    int max_sh = 7, max_list = 8;
    ex->tiles.clear();
    size_t pyr_off = 0, blur_off = 0;
    int cand_off = 0, kp_off = 0, max_cand = 0, max_nodes = 8;
    for (int l = 0; l < nl; l++) {
        LevelPlan &L = ex->lv[l];
        memset(&L, 0, sizeof(L));
        L.w = cv_round_f((float)w * ex->inv_scale[l]);
        L.h = cv_round_f((float)h * ex->inv_scale[l]);
        SFE_REQUIRE(L.w >= 1 && L.h >= 1, SFE_ERR_UNSUPPORTED, "pyramid level collapses to zero size");
        SFE_REQUIRE(L.w <= 4096 + 2 * kBorder && L.h <= 4096 + 2 * kBorder, SFE_ERR_UNSUPPORTED,
                    "image larger than 4128 px per side");
        L.pitch = (int)align_up((size_t)L.w, 16);
        L.blur_pitch = L.pitch;
        if (l > 0) {
            L.plane_off = (int)pyr_off;
            pyr_off += align_up((size_t)L.pitch * L.h, 128);
        }
        L.blur_off = (int)blur_off;
        blur_off += align_up((size_t)L.blur_pitch * L.h, 128);
        L.scale = ex->scale[l];
        L.size = (float)(int)(31 * ex->scale[l]);
        L.quota = ex->quota[l];
        // FAST window and cells
        const int max_bx = L.w - kBorder, max_by = L.h - kBorder;
        L.win_w = max_bx - kBorder;
        L.win_h = max_by - kBorder;
        const float width = (float)L.win_w, height = (float)L.win_h;
        L.n_cols = L.win_w > 0 ? (int)(width / 30.f) : 0;
        L.n_rows = L.win_h > 0 ? (int)(height / 30.f) : 0;
        L.w_cell = L.h_cell = 1;
        int tested = 0, n_level_cells = 0;
        if (L.n_cols >= 1 && L.n_rows >= 1) {  // else: reference divides by zero; canonical = no keypoints (T5)
            L.w_cell = (int)ceilf(width / L.n_cols);
            L.h_cell = (int)ceilf(height / L.n_rows);
            // rows / columns that pass the skip rules (:794,803) and hold a >= 7 px sub-image (cv::FAST tests
            // nothing on a smaller one) form a prefix of the nominal grid
            int rows_eff = 0, cols_eff = 0;
            for (int i = 0; i < L.n_rows; i++)
                if (kBorder + i * L.h_cell < max_by - 3 && max_by - (kBorder + i * L.h_cell) >= 7) rows_eff = i + 1;
            for (int j = 0; j < L.n_cols; j++)
                if (kBorder + j * L.w_cell < max_bx - 6) cols_eff = j + 1;
            SFE_REQUIRE(L.w_cell + 6 <= kMaxSub && L.h_cell + 6 <= kMaxSub, SFE_ERR_UNSUPPORTED, "FAST cell larger than 66 px");
            if (rows_eff > 0 && cols_eff > 0) {
                FastLevel &F = ex->fast.lv[l];
                F.pitch = L.pitch;
                F.plane_off = L.plane_off;
                n_level_cells = rows_eff * cols_eff;
                const int inv_w = 65536 / L.w_cell + 1;  // x / w_cell == (x * inv_w) >> 16 for x < 256 (w_cell in [30, 60])
                for (int x = 0; x < 256; x++) SFE_REQUIRE(((x * inv_w) >> 16) == x / L.w_cell && inv_w < 65536, SFE_ERR_UNSUPPORTED, "cell reciprocal");
                for (int i = 0; i < rows_eff; i++) {
                    const int ini_y = kBorder + i * L.h_cell, sh = std::min(ini_y + L.h_cell + 6, max_by) - ini_y;
                    max_sh = std::max(max_sh, sh);
                    // greedy segments: as many cells as keep the tested pixels inside 32 of the level's 4-pixel words
                    for (int j = 0; j < cols_eff;) {
                        const int ini_x = kBorder + j * L.w_cell, cs = ini_x + 3 - ((ini_x - 4) & ~15);
                        int tw = 0, nc = 0;
                        while (j + nc < cols_eff && nc < kFastMaxCells) {
                            const int cx = kBorder + (j + nc) * L.w_cell, sw = std::min(cx + L.w_cell + 6, max_bx) - cx;
                            const int tw2 = tw + sw - 6;
                            if (nc > 0 && (tw2 > kFastSegPx || ((cs + tw2 - 1) >> 2) - (cs >> 2) + 1 > 32)) break;
                            tw = tw2;
                            nc++;
                        }
                        SFE_REQUIRE(tw >= 1 && tw <= kFastSegPx && ((cs + tw - 1) >> 2) - (cs >> 2) + 1 <= 32, SFE_ERR_UNSUPPORTED, "FAST segment");
                        ex->segs.push_back(SegRec{(short)ini_x, (short)ini_y, (short)tw, (unsigned char)sh, (unsigned char)l,
                                                  (unsigned char)nc, (unsigned char)L.w_cell, (unsigned short)inv_w, 0});
                        tested += tw * (sh - 6);
                        max_list = std::max(max_list, tw * (sh - 6));
                        j += nc;
                    }
                }
            }
        }
        ex->fast.n_cells += n_level_cells;
        ex->seg_level_start[l + 1] = (int)ex->segs.size();
        // quadtree roots
        L.n_ini = 1;
        L.hx = 1.f;
        if (tested > 0) {
            L.n_ini = (int)roundf((float)L.win_w / (float)L.win_h);
            SFE_REQUIRE(L.n_ini >= 1, SFE_ERR_UNSUPPORTED,
                        "portrait level (W/H < 0.5): the reference divides by nIni == 0");
            L.hx = (float)L.win_w / (float)L.n_ini;
        }
        // 4 * n_ini * 4^d <= quota: the first d full passes cannot end through the list-size tests (see octree_build_at_depth)
        L.ff_depth = 0;
        while (ex->octree_ff && L.ff_depth < 6 && 4ll * L.n_ini * (1ll << (2 * (L.ff_depth + 1))) <= L.quota) L.ff_depth++;
        // NMS'd FAST corners reach ~1 per 30 px on the small pyramid levels of textured frames
        // first guess: one corner per 12 tested pixels, within the quadtree's 16-bit instance; a level that really holds more
        // teaches the handle its floor (grow_candidate_buffers)
        L.cand_cap = tested > 0 ? std::max(std::min(ex->cand_cap_override > 0 ? ex->cand_cap_override : std::max(tested / 12, 1024), kNarrowCandCap),
                                           std::min(ex->cand_floor[l], kMaxCandCap)) : 0;
        L.cand_off = cand_off;
        cand_off += L.cand_cap;
        ex->fast.lv[l].cand_off = L.cand_off;
        ex->fast.lv[l].cand_cap = L.cand_cap;
        L.kp_cap = tested > 0 ? std::max(L.quota + 3, 4 * L.n_ini) + 1 : 0;
        L.kp_off = kp_off;
        kp_off += L.kp_cap;
        max_cand = std::max(max_cand, L.cand_cap);
        max_nodes = std::max(max_nodes, std::max(L.kp_cap + 4, L.n_ini));
        if (tested > 0)
            for (int y0 = 0; y0 < L.h; y0 += kBlurTileH)
                for (int x0 = 0; x0 < L.w; x0 += kBlurTileW) ex->tiles.push_back(TilePlan{(short)l, (short)x0, (short)y0, 0});
        // resize coefficient tables producing level l from level l-1
        if (l > 0) {
            const int sw = ex->lv[l - 1].w, sh = ex->lv[l - 1].h;
            while (xtab.size() % 4) xtab.push_back(xtab.back());  // 16-byte aligned uint4 loads, 4 px per thread
            L.xtab_off = (int)xtab.size();
            L.ytab_off = (int)ytab.size();
            const double scale_x = 1.0 / ((double)L.w / sw), scale_y = 1.0 / ((double)L.h / sh);
            for (int dx = 0; dx < L.w; dx++) {
                float fx = (float)((dx + 0.5) * scale_x - 0.5);
                int sx = (int)floorf(fx);
                fx -= sx;
                if (sx < 0) { fx = 0; sx = 0; }
                if (sx >= sw - 1) { fx = 0; sx = sw - 1; }
                const int w0 = cv_round_f((1.f - fx) * 2048), w1 = cv_round_f(fx * 2048);
                xtab.push_back(make_uint2((unsigned)sx, (unsigned)w0 | (unsigned)w1 << 16));
            }
            while (xtab.size() % 4) xtab.push_back(xtab.back());
            // 4-outputs-per-thread horizontal pass: the 4 source pairs of every aligned group must fit 8 bytes
            ex->pyr_wide_h[l] = 1;
            for (int gx = 0; gx < L.w; gx += 4)
                if (xtab[L.xtab_off + gx + 3].x - xtab[L.xtab_off + gx].x > 6) ex->pyr_wide_h[l] = 0;
            for (int dy = 0; dy < L.h; dy++) {
                float fy = (float)((dy + 0.5) * scale_y - 0.5);
                int sy = (int)floorf(fy);
                fy -= sy;
                const int b0 = cv_round_f((1.f - fy) * 2048), b1 = cv_round_f(fy * 2048);
                const int y0 = std::min(std::max(sy, 0), sh - 1), y1 = std::min(std::max(sy + 1, 0), sh - 1);
                ytab.push_back(make_uint2((unsigned)y0 | (unsigned)y1 << 16, (unsigned)b0 | (unsigned)b1 << 16));
            }
            for (int tx = 0; tx < L.w; tx += kPyrTileW) {  // source columns one output tile touches, from the 16-byte grid
                const int last = std::min(tx + kPyrTileW, L.w) - 1;
                const int first_sx = (int)xtab[L.xtab_off + tx].x & ~15;
                max_src_cols = std::max(max_src_cols, std::min((int)xtab[L.xtab_off + last].x + 1, sw - 1) - first_sx + 1);
            }
            for (int ty = 0; ty < L.h; ty += kPyrTileH) {  // source rows one output tile touches
                const int last = std::min(ty + kPyrTileH, L.h) - 1;
                const int span = (int)(ytab[L.ytab_off + last].x >> 16) - (int)(ytab[L.ytab_off + ty].x & 0xFFFF) + 1;
                max_src_rows = std::max(max_src_rows, span);
            }
        }
    }
    ex->pyr_stride = std::max<size_t>(pyr_off, 128);
    ex->blur_stride = std::max<size_t>(blur_off, 128);
    ex->cand_stride = std::max(cand_off, 1);
    ex->kpst_stride = std::max(kp_off, 1);
    ex->max_cand = (std::max(max_cand, 1) + 7) & ~7;
    ex->max_nodes = max_nodes;
    ex->pyr_smem = (size_t)max_src_rows * kPyrTileW * sizeof(uint16_t);
    ex->pyr_box_w = (int)align_up((size_t)max_src_cols, 16);
    ex->pyr_box_h = max_src_rows;
    SFE_REQUIRE(ex->pyr_smem + (size_t)ex->pyr_box_w * ex->pyr_box_h <= 48 * 1024 && ex->pyr_box_w <= 256 && ex->pyr_box_h <= 256,
                SFE_ERR_UNSUPPORTED, "scale factor too large for the pyramid tile");
    ex->fast.nlevels = nl;
    ex->fast.ini_th = ex->prm.ini_th_fast;
    ex->fast.min_th = ex->prm.min_th_fast;
    ex->fast.n_segs = (int)ex->segs.size();
    ex->fast.tile_rows = (max_sh + 1) & ~1;  // even: tile_rows * pitch keeps the score array 16-byte aligned
    ex->fast.score_rows = max_sh - 4;
    ex->fast.list_cap = (max_list + 7) & ~7;
    ex->fast_smem = (size_t)ex->fast.tile_rows * kFastTilePitch + (size_t)ex->fast.score_rows * kFastScorePitch + 2 * 2 * (size_t)ex->fast.list_cap;
    SFE_REQUIRE(ex->fast_smem <= 200 * 1024, SFE_ERR_UNSUPPORTED, "FAST segment working set exceeds shared memory");
    // candidate arrays for up to kOctreeSmemCand points in shared memory (3 CTAs per SM at the KITTI config); fuller
    // levels spill to global scratch slots
    ex->octree_smem_cand = std::min(ex->max_cand, ex->octree_cand_override > 0 ? ex->octree_cand_override : kOctreeSmemCand) & ~7;
    if (ex->octree_smem_cand < 8) ex->octree_smem_cand = 8;
    ex->octree_wide = ex->max_cand > kNarrowCandCap;
    const size_t oct_cand_bytes = ex->octree_wide ? 16 : 14, oct_node_bytes = ex->octree_wide ? sizeof(ONodeT<true>) : sizeof(ONodeT<false>);
    ex->octree_smem = (size_t)ex->octree_smem_cand * oct_cand_bytes + (size_t)max_nodes * (16 + 3 * 4 + 2 * oct_node_bytes + 2 * 2 + 8) + 32 * 4 + 64;
    SFE_REQUIRE(ex->octree_smem <= 227 * 1024, SFE_ERR_UNSUPPORTED, "quadtree working set exceeds shared memory");
    {   // one global scratch slot for every (level, image) whose candidate buffer can outgrow the shared-memory arrays
        int big_levels = 0;
        for (int l = 0; l < nl; l++) big_levels += ex->lv[l].cand_cap > ex->octree_smem_cand;
        ex->octree_slots = big_levels * ex->max_images;
    }
    SFE_CUDA(ex->d_octree_scratch.ensure(std::max<size_t>((size_t)ex->octree_slots * ex->max_cand * oct_cand_bytes, 16)));
    const int n = ex->max_images;
    SFE_CUDA(ex->d_pyr.ensure(ex->pyr_stride * n));
    SFE_CUDA(ex->d_blur.ensure(ex->blur_stride * n));
    SFE_CUDA(ex->d_cand.ensure((size_t)ex->cand_stride * n));
    SFE_CUDA(ex->d_kpst.ensure((size_t)ex->kpst_stride * n));
    SFE_CUDA(ex->d_counts.ensure((size_t)n * (2 * nl + 1) + 1));  // cand_count | kp_count | scratch_next | flags
    // (an asynchronous handle only clears its error flags at sfe_extractor_wait: they must not start as whatever the
    // allocation held)
    SFE_CUDA(cudaMemsetAsync(ex->d_counts.p, 0, sizeof(int) * ex->d_counts.n, ex->stream));
    SFE_CUDA(ex->d_tiles.ensure(std::max<size_t>(ex->tiles.size(), 1)));
    SFE_CUDA(ex->d_segs.ensure(std::max<size_t>(ex->segs.size(), 1)));
    if (!ex->segs.empty())
        SFE_CUDA(cudaMemcpyAsync(ex->d_segs.p, ex->segs.data(), sizeof(SegRec) * ex->segs.size(), cudaMemcpyHostToDevice, ex->stream));
    SFE_CUDA(ex->d_xtab.ensure(std::max<size_t>(xtab.size(), 1)));
    SFE_CUDA(ex->d_ytab.ensure(std::max<size_t>(ytab.size(), 1)));
    if (!ex->tiles.empty())
        SFE_CUDA(cudaMemcpyAsync(ex->d_tiles.p, ex->tiles.data(), sizeof(TilePlan) * ex->tiles.size(), cudaMemcpyHostToDevice, ex->stream));
    if (!xtab.empty()) {
        SFE_CUDA(cudaMemcpyAsync(ex->d_xtab.p, xtab.data(), sizeof(uint2) * xtab.size(), cudaMemcpyHostToDevice, ex->stream));
        SFE_CUDA(cudaMemcpyAsync(ex->d_ytab.p, ytab.data(), sizeof(uint2) * ytab.size(), cudaMemcpyHostToDevice, ex->stream));
    }
    SFE_CUDA(cudaStreamSynchronize(ex->stream));  // the std::vectors above die at return
    // tensor maps of the pyramid levels (the reflect patch-up of the TMA blur needs >= 8 px per side)
    ex->tma_plan_ok = !ex->tma_disabled;
    for (int l = 0; l < nl && ex->tma_plan_ok; l++) {
        const LevelPlan &L = ex->lv[l];
        if (L.w < 8 || L.h < 8) ex->tma_plan_ok = false;
        if (l == 0 || !ex->tma_plan_ok) continue;
        ex->tma_plan_ok = tma_encode_u8_3d(&ex->fast_maps.lv[l], ex->d_pyr.p + L.plane_off, L.w, L.h, n, L.pitch, ex->pyr_stride,
                                           kFastTilePitch, ex->fast.tile_rows) &&
                          tma_encode_u8_3d(&ex->blur_maps.lv[l], ex->d_pyr.p + L.plane_off, L.w, L.h, n, L.pitch, ex->pyr_stride,
                                           kBlurInWords * 4, kBlurTileH + 6) &&
                          (nl < 2 || tma_encode_u8_3d(&ex->pyr_maps.lv[l], ex->d_pyr.p + L.plane_off, L.w, L.h, n, L.pitch, ex->pyr_stride,
                                                      ex->pyr_box_w, ex->pyr_box_h)) &&
                          tma_encode_u8_3d(&ex->orient_maps.ic[l], ex->d_pyr.p + L.plane_off, L.w, L.h, n, L.pitch, ex->pyr_stride,
                                           kIcBoxW, kIcBoxH);
    }
    for (int l = 0; l < nl && ex->tma_plan_ok; l++) {
        const LevelPlan &L = ex->lv[l];
        ex->tma_plan_ok = tma_encode_u8_3d(&ex->orient_maps.bd[l], ex->d_blur.p + L.blur_off, L.w, L.h, n, L.blur_pitch, ex->blur_stride,
                                           kBdBoxW, kBdBoxH);
    }
    ex->l0_key[0] = ex->l0_key[1] = nullptr;
    ex->pitch0 = (int)align_up((size_t)w, 16);
    ex->w = w;
    ex->h = h;
    return SFE_OK;
}

// The batch-wide view of the handle's buffers: set A = images [0, split) of the call at internal slots
// [0, split), set B behind them.
static ImgSet make_imgset(sfe_extractor *ex, const uint8_t *in_a, const uint8_t *in_b, int split, size_t in_stride,
                          int in_pitch) {
    const int nl = ex->prm.nlevels;
    ImgSet S{};
    S.in_a = in_a;
    S.in_b = in_b;
    S.split = split;
    S.slot_a = 0;
    S.slot_b = split;
    S.in_stride = in_stride;
    S.in_pitch = in_pitch;
    S.pyr = ex->d_pyr.p;
    S.pyr_stride = ex->pyr_stride;
    S.blur = ex->d_blur.p;
    S.blur_stride = ex->blur_stride;
    memcpy(S.lv, ex->lv, sizeof(LevelPlan) * nl);
    S.nlevels = nl;
    S.cand = ex->d_cand.p;
    S.cand_stride = ex->cand_stride;
    S.kpst = ex->d_kpst.p;
    S.kpst_stride = ex->kpst_stride;
    S.cand_count = ex->d_counts.p;
    S.kp_count = ex->d_counts.p + (size_t)ex->max_images * nl;
    S.flags = ex->d_counts.p + (size_t)ex->max_images * nl * 2 + 1;
    return S;
}

// frames [f0, f1) of a batch as a self-contained sub-batch (set A first, then set B if the batch has one)
static ImgSet chunk_of(const ImgSet &B, int f0, int f1, bool has_b) {
    ImgSet S = B;
    S.in_a = B.in_a + (size_t)f0 * B.in_stride;
    S.in_b = B.in_b + (size_t)f0 * B.in_stride;
    S.split = f1 - f0;
    S.in_z0 = B.in_z0 + f0;
    S.slot_a = B.slot_a + f0;
    S.slot_b = has_b ? B.slot_b + f0 : 0;
    return S;
}
static OutSet chunk_of(const OutSet &O, int f0) {
    OutSet C = O;
    C.kps_a += (size_t)f0 * O.cap; C.kps_b += (size_t)f0 * O.cap;
    C.desc_a += (size_t)f0 * O.cap * 32; C.desc_b += (size_t)f0 * O.cap * 32;
    C.n_a += f0; C.n_b += f0;
    return C;
}

// Results of a small host call whose output arrays are pinned (device-mapped) host memory: one kernel stores every array
// straight into the caller's buffers over PCIe -- one launch instead of nine DMA copies of 4 - 80 KB each, which cost the
// one-pair call 43 us of its 200.
constexpr int kMaxCopySegs = 12;
struct CopySeg { const void *src; void *dst; uint32_t bytes; };
struct CopyPlan { CopySeg seg[kMaxCopySegs]; int n; };
__global__ void __launch_bounds__(256) copy_out_kernel(const __grid_constant__ CopyPlan P) {
    pdl_enter();
    const uint32_t t = blockIdx.x * blockDim.x + threadIdx.x, T = gridDim.x * blockDim.x;
    for (int s = 0; s < P.n; s++) {
        const CopySeg &g = P.seg[s];
        if ((((uintptr_t)g.src | (uintptr_t)g.dst | g.bytes) & 15) == 0) {
            const uint4 *a = (const uint4 *)g.src;
            uint4 *b = (uint4 *)g.dst;
            for (uint32_t i = t; i < g.bytes / 16; i += T) b[i] = a[i];
        } else {  // every array here is made of 4-byte items
            const uint32_t *a = (const uint32_t *)g.src;
            uint32_t *b = (uint32_t *)g.dst;
            for (uint32_t i = t; i < g.bytes / 4; i += T) b[i] = a[i];
        }
    }
}

// device address of a host pointer a kernel may store to (pinned or registered memory), or nullptr
static void *mapped_host_pointer(const void *p) {
    cudaPointerAttributes a;
    if (cudaPointerGetAttributes(&a, p) != cudaSuccess) { cudaGetLastError(); return nullptr; }
    return a.type == cudaMemoryTypeHost ? a.devicePointer : nullptr;
}

static int reset_counters(sfe_extractor *ex) {
    // layout: cand_count | kp_count | scratch_next | flags.  An asynchronous handle keeps the error flags until sfe_extractor_wait.
    const size_t n = (size_t)ex->max_images * (2 * ex->prm.nlevels + (ex->async_dev ? 0 : 1)) + 1;
    SFE_CUDA(cudaMemsetAsync(ex->d_counts.p, 0, sizeof(int) * n, ex->stream));
    return SFE_OK;
}

// Level-0 tensor maps for the images of this call (set A: n_a images at `a`, set B: n_b at `b`).  Sets
// ex->tma_now: whether this call's kernels load their tiles with TMA.
static void prepare_l0_maps(sfe_extractor *ex, const uint8_t *a, const uint8_t *b, int n_a, int n_b, size_t stride, int pitch) {
    ex->tma_now = false;
    if (!ex->tma_plan_ok || !tma_layout_ok(a, pitch, stride) || !tma_layout_ok(b, pitch, stride)) return;
    const size_t geom[4] = {(size_t)n_a, (size_t)n_b, stride, (size_t)pitch};
    if (ex->l0_key[0] != a || ex->l0_key[1] != b || memcmp(geom, ex->l0_geom, sizeof(geom)) != 0) {
        const LevelPlan &L = ex->lv[0];
        const bool ok = tma_encode_u8_3d(&ex->fast_maps.lv[0], a, L.w, L.h, n_a, pitch, stride, kFastTilePitch, ex->fast.tile_rows) &&
                        tma_encode_u8_3d(&ex->fast_maps.l0b, b, L.w, L.h, n_b, pitch, stride, kFastTilePitch, ex->fast.tile_rows) &&
                        tma_encode_u8_3d(&ex->blur_maps.lv[0], a, L.w, L.h, n_a, pitch, stride, kBlurInWords * 4, kBlurTileH + 6) &&
                        tma_encode_u8_3d(&ex->blur_maps.l0b, b, L.w, L.h, n_b, pitch, stride, kBlurInWords * 4, kBlurTileH + 6) &&
                        (ex->prm.nlevels < 2 ||
                         (tma_encode_u8_3d(&ex->pyr_maps.lv[0], a, L.w, L.h, n_a, pitch, stride, ex->pyr_box_w, ex->pyr_box_h) &&
                          tma_encode_u8_3d(&ex->pyr_maps.l0b, b, L.w, L.h, n_b, pitch, stride, ex->pyr_box_w, ex->pyr_box_h))) &&
                        tma_encode_u8_3d(&ex->orient_maps.ic[0], a, L.w, L.h, n_a, pitch, stride, kIcBoxW, kIcBoxH) &&
                        tma_encode_u8_3d(&ex->orient_maps.ic_l0b, b, L.w, L.h, n_b, pitch, stride, kIcBoxW, kIcBoxH);
        ex->l0_key[0] = ok ? a : nullptr;
        ex->l0_key[1] = ok ? b : nullptr;
        memcpy(ex->l0_geom, geom, sizeof(geom));
        if (!ok) return;
    }
    ex->tma_now = true;
}

constexpr bool kFastTma = true;

static int launch_fast(sfe_extractor *ex, cudaStream_t st, const ImgSet &S, int count, int level0 = 0, int level1 = kMaxLevels) {
    level1 = std::min(level1, ex->prm.nlevels);
    const int seg0 = ex->seg_level_start[level0], nseg = ex->seg_level_start[level1] - seg0;  // the segments of levels [level0, level1)
    if (nseg <= 0) return SFE_OK;
    const dim3 grid((unsigned)nseg, count);
    if (ex->fast_smem > 48 * 1024) {  // the opt-in shared-memory limit is a per-function attribute: only ever raise it
        static std::mutex mu;
        static size_t granted[64] = {};
        std::lock_guard<std::mutex> lock(mu);
        if (ex->fast_smem > granted[ex->device & 63]) {
            SFE_CUDA(cudaFuncSetAttribute(fast_segments_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)ex->fast_smem));
            SFE_CUDA(cudaFuncSetAttribute(fast_segments_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)ex->fast_smem));
            granted[ex->device & 63] = ex->fast_smem;
        }
    }
    {   // ask for the largest shared-memory carve-out (the default heuristic leaves the kernel at 4 CTAs per SM)
        static std::once_flag once[64];
        std::call_once(once[ex->device & 63], [] {
            cudaFuncSetAttribute(fast_segments_kernel<true>, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared);
            cudaFuncSetAttribute(fast_segments_kernel<false>, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared);
        });
    }
    if (ex->tma_now && kFastTma)
        launch_k(fast_segments_kernel<true>, grid, kFastThreads, ex->fast_smem, st, ex->pdl_now, S, ex->fast, ex->d_segs.p + seg0, ex->fast_maps);
    else
        launch_k(fast_segments_kernel<false>, grid, kFastThreads, ex->fast_smem, st, ex->pdl_now, S, ex->fast, ex->d_segs.p + seg0, ex->fast_maps);
    return SFE_OK;
}

constexpr int kSplitMaxImages = 4;  // calls with at most this many images run levels 0-1 beside the rest of the pyramid

// Order the handle's main stream behind a matching tail still running on the side stream.
static int join_tail(sfe_extractor *ex) {
    if (ex->tail_pending) {
        SFE_CUDA(cudaStreamWaitEvent(ex->stream, ex->ev_join[1], 0));
        ex->tail_pending = false;
    }
    return SFE_OK;
}

static int enqueue_extract(sfe_extractor *ex, cudaStream_t st, const ImgSet &S, int count, const OutSet &O) {
    const int nl = ex->prm.nlevels;
    prof_mark(ex, 0);
    auto launch_pyr = [&](int l) {  // level l from level l - 1
        const LevelPlan &D = ex->lv[l], &Q = ex->lv[l - 1];
        const PyrStep P{D.w, D.h, D.pitch, D.plane_off, Q.w, l == 1 ? S.in_pitch : Q.pitch, Q.plane_off, l == 1, D.xtab_off, D.ytab_off,
                        l - 1, ex->pyr_box_w, ex->pyr_box_h, ex->pyr_wide_h[l]};
        dim3 grid(div_up(D.w, kPyrTileW), div_up(D.h, kPyrTileH), count);
        if (ex->tma_now)
            launch_k(pyr_resize_kernel<true>, grid, 256, ex->pyr_smem + (size_t)ex->pyr_box_w * ex->pyr_box_h, st, ex->pdl_now, S, P, ex->d_xtab.p,
                     ex->d_ytab.p, ex->pyr_maps);
        else
            launch_k(pyr_resize_kernel<false>, grid, 256, ex->pyr_smem, st, ex->pdl_now, S, P, ex->d_xtab.p, ex->d_ytab.p, ex->pyr_maps);
        ex->launches++;
    };
    const bool has_cells = ex->fast.n_cells > 0;
    {   // every kernel of the sequence asks for the same (largest) shared-memory carve-out as FAST: kernels that want different
        // L1 / shared splits cannot share an SM, which serialised the branches of a few-image call
        static std::once_flag once[64];
        std::call_once(once[ex->device & 63], [] {
            const void *fns[] = {(const void *)pyr_resize_kernel<true>, (const void *)pyr_resize_kernel<false>, (const void *)blur_kernel<true>,
                                 (const void *)blur_kernel<false>, (const void *)octree_kernel<true>, (const void *)octree_kernel<false>,
                                 (const void *)orient_describe_kernel<true>, (const void *)orient_describe_kernel<false>,
                                 (const void *)realign_kernel};
            for (const void *f : fns) cudaFuncSetAttribute(f, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared);
        });
    }
    if (has_cells) {  // the opt-in shared-memory limit is a per-function (not per-handle) attribute: only ever raise it
        static std::mutex mu;
        static size_t granted[64] = {};
        std::lock_guard<std::mutex> lock(mu);
        if (ex->octree_smem > granted[ex->device & 63]) {
            SFE_CUDA(cudaFuncSetAttribute(octree_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)ex->octree_smem));
            SFE_CUDA(cudaFuncSetAttribute(octree_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)ex->octree_smem));
            granted[ex->device & 63] = ex->octree_smem;
        }
    }
    int *scratch_next = ex->d_counts.p + (size_t)ex->max_images * nl * 2;
    auto launch_octree = [&](cudaStream_t so, int level0, int level_n, int ctas) {
        const int items = level_n * count;
        const int grid = ctas > 0 ? std::min(items, ctas) : items;
        // a call with few images cannot fill the machine with (level, image) items: their latency is what counts, and a
        // 1024-thread CTA walks a level's candidates in a quarter of the iterations
        const int threads = nl * count <= ex->sm_count / 2 ? 1024 : 256;
        if (ex->octree_wide)
            launch_k(octree_kernel<true>, grid, threads, ex->octree_smem, so, ex->pdl_now, S, count, level0, level_n, ex->octree_smem_cand,
                     ex->max_cand, ex->max_nodes, ex->d_octree_scratch.p, ex->octree_slots, scratch_next);
        else
            launch_k(octree_kernel<false>, grid, threads, ex->octree_smem, so, ex->pdl_now, S, count, level0, level_n, ex->octree_smem_cand,
                     ex->max_cand, ex->max_nodes, ex->d_octree_scratch.p, ex->octree_slots, scratch_next);
        ex->launches++;
    };
    const bool fork_ok = !ex->profiling && !ex->piped_now && st == ex->stream;
    // Few images (the reference-shaped single call): the chain pyramid -> FAST -> quadtree is pure latency, and its longest link is
    // the quadtree of level 0.  Levels 0 and 1 only need the first pyramid launch, so their FAST + quadtree run on a side stream
    // beside the rest of the pyramid, the FAST + quadtree of the small levels and the blur.
    const bool split = fork_ok && has_cells && ex->split_small && count <= kSplitMaxImages && nl >= 3;
    if (split) {
        launch_pyr(1);
        cudaStream_t sa = ex->aux[2];
        SFE_CUDA(cudaEventRecord(ex->ev_fork[2], st));
        SFE_CUDA(cudaStreamWaitEvent(sa, ex->ev_fork[2], 0));
        if (int rc = launch_fast(ex, sa, S, count, 0, 2)) return rc;
        launch_octree(sa, 0, 2, 0);
        SFE_CUDA(cudaEventRecord(ex->ev_join[2], sa));
        for (int l = 2; l < nl; l++) launch_pyr(l);
        cudaStream_t sb = ex->aux[0];
        SFE_CUDA(cudaEventRecord(ex->ev_fork[0], st));
        SFE_CUDA(cudaStreamWaitEvent(sb, ex->ev_fork[0], 0));
        if (ex->tma_now)
            blur_kernel<true><<<dim3((unsigned)ex->tiles.size(), count), 256, 0, sb>>>(S, ex->d_tiles.p, ex->blur_maps);
        else
            blur_kernel<false><<<dim3((unsigned)ex->tiles.size(), count), 256, 0, sb>>>(S, ex->d_tiles.p, ex->blur_maps);
        SFE_CUDA(cudaEventRecord(ex->ev_join[0], sb));
        if (int rc = launch_fast(ex, st, S, count, 2, nl)) return rc;
        launch_octree(st, 2, nl - 2, 0);
        SFE_CUDA(cudaStreamWaitEvent(st, ex->ev_join[2], 0));
        SFE_CUDA(cudaStreamWaitEvent(st, ex->ev_join[0], 0));
        ex->launches += 3;
    } else {
        for (int l = 1; l < nl; l++) launch_pyr(l);
        prof_mark(ex, 1);
        if (has_cells) {
            // The blur only needs the pyramid, so it runs on a side stream beside the quadtree (which is latency-bound: 35 %
            // issue-active) and joins before the descriptors.  Serial when stages are timed and on the pipelined host path,
            // whose sub-batches already overlap across compute streams.
            const int si = 0;
            const bool fork = ex->overlap_blur && fork_ok, late = ex->overlap_blur == 2;
            cudaStream_t sb = fork ? ex->aux[si] : st;
            auto launch_blur = [&]() {
                if (ex->tma_now)
                    blur_kernel<true><<<dim3((unsigned)ex->tiles.size(), count), 256, 0, sb>>>(S, ex->d_tiles.p, ex->blur_maps);
                else
                    blur_kernel<false><<<dim3((unsigned)ex->tiles.size(), count), 256, 0, sb>>>(S, ex->d_tiles.p, ex->blur_maps);
            };
            auto fork_blur = [&]() -> int {
                SFE_CUDA(cudaEventRecord(ex->ev_fork[si], st));
                SFE_CUDA(cudaStreamWaitEvent(sb, ex->ev_fork[si], 0));
                launch_blur();
                SFE_CUDA(cudaEventRecord(ex->ev_join[si], sb));
                return SFE_OK;
            };
            if (fork && !late)
                if (int rc = fork_blur()) return rc;
            if (int rc = launch_fast(ex, st, S, count)) return rc;
            prof_mark(ex, 2);
            if (fork && late)
                if (int rc = fork_blur()) return rc;
            // beside the forked blur the quadtree runs persistent with 2 CTAs per SM: its ~60 KB of shared memory per CTA would
            // otherwise leave the blur one CTA per SM (measured: 2.12 -> 2.06 ms per 128-frame step; alone, fewer CTAs are slower)
            launch_octree(st, 0, nl, ex->octree_ctas > 0 ? ex->octree_ctas : (fork && late ? 2 * ex->sm_count : 0));
            prof_mark(ex, 3);
            if (fork) SFE_CUDA(cudaStreamWaitEvent(st, ex->ev_join[si], 0));
            else launch_blur();
            prof_mark(ex, 4);
            ex->launches += 2;
        } else {
            prof_mark(ex, 2); prof_mark(ex, 3); prof_mark(ex, 4);
        }
    }
    if (st == ex->stream) {  // the previous call's matchers may still be reading the output arrays this kernel writes
        if (int rc = join_tail(ex)) return rc;
    } else if (ex->tail_pending) {
        SFE_CUDA(cudaStreamWaitEvent(st, ex->ev_join[1], 0));
    }
    // keypoints per warp: kKpPerWarp amortises the table set-up of a CTA in a batch; a call with few images instead spreads its
    // keypoints over every warp the machine holds (5 CTAs x 8 warps per SM) -- one pair: one keypoint per warp, 21 -> 9 us
    const int kpw = std::max(1, std::min(kKpPerWarp, div_up(O.cap * count, ex->sm_count * 5 * 8)));
    if (ex->tma_now && ex->orient_tma)
        launch_k(orient_describe_kernel<true>, dim3(div_up(O.cap, 8 * kpw), count), 256, 0, st, ex->pdl_now, S, O, kpw, ex->orient_maps);
    else
        launch_k(orient_describe_kernel<false>, dim3(div_up(O.cap, 8 * kpw), count), 256, 0, st, ex->pdl_now, S, O, kpw, ex->orient_maps);
    prof_mark(ex, 5);
    ex->prof_pending = ex->profiling;
    ex->prof_has_stereo = ex->prof_has_track = false;
    ex->launches++;
    SFE_CUDA(cudaGetLastError());
    return SFE_OK;
}

// Internal status of a finished call whose FAST candidate buffers overflowed: the buffers have been enlarged to what the
// call counted (the counters are exact even when stores were dropped) and the caller re-runs the batch.
constexpr int kStatusRerun = -1000;

// After a candidate overflow: raise the per-level capacities to what the flagged images counted and drop the plan so that
// the next prepare() rebuilds the buffers.  SFE_ERR_CAPACITY only when a level holds more corners than the quadtree's
// 16-bit candidate index can address.
static int grow_candidate_buffers(sfe_extractor *ex, int count) {
    const int nl = ex->prm.nlevels;
    std::vector<int> cnt((size_t)count * nl);
    SFE_CUDA(cudaMemcpy(cnt.data(), ex->d_counts.p, sizeof(int) * cnt.size(), cudaMemcpyDeviceToHost));
    bool grew = false;
    for (int l = 0; l < nl; l++) {
        int most = 0, who = 0;
        for (int i = 0; i < count; i++)
            if (cnt[(size_t)i * nl + l] > most) { most = cnt[(size_t)i * nl + l]; who = i; }
        if (most <= ex->lv[l].cand_cap) continue;
        if (most > kMaxCandCap) {
            set_error("image slot %d, level %d: %d FAST corners, more than the %d a level may hold", who, l, most, kMaxCandCap);
            return SFE_ERR_CAPACITY;
        }
        ex->cand_floor[l] = std::min(kMaxCandCap, most + most / 8 + 64);
        grew = true;
    }
    if (!grew)  // asynchronous handle: a later call already reset the counters of the one that overflowed
        for (int l = 0; l < nl; l++) {
            if (ex->lv[l].cand_cap >= kMaxCandCap) continue;
            ex->cand_floor[l] = std::min(kMaxCandCap, 2 * std::max(ex->lv[l].cand_cap, 1024));
            grew = true;
        }
    if (!grew) { set_error("FAST candidate buffers are at their maximum (%d per level)", kMaxCandCap); return SFE_ERR_CAPACITY; }
    if (ex->tail_pending) { cudaStreamSynchronize(ex->aux[1]); ex->tail_pending = false; }
    ex->w = ex->h = 0;  // forces build_plan
    ex->last_count = 0;
    return kStatusRerun;
}

// flags_here: the flags of this call already sit in ex->h_flags_pinned behind `st` (copy_out_kernel)
static int check_flags(sfe_extractor *ex, cudaStream_t st, int count, bool flags_here = false) {
    ex->h_flags.resize(count);
    if (!flags_here) SFE_CUDA(cudaMemcpyAsync(ex->h_flags.data(), ex->last.flags, sizeof(int) * count, cudaMemcpyDeviceToHost, st));
    SFE_CUDA(cudaStreamSynchronize(st));
    if (flags_here) memcpy(ex->h_flags.data(), ex->h_flags_pinned, sizeof(int) * count);
    if (ex->prof_pending) {
        const int ns = ex->prof_has_track ? kNumStages : ex->prof_has_stereo ? kNumStages - 1 : kNumStages - 2;
        for (int i = 0; i < ns; i++) {
            float ms = 0.f;
            if (cudaEventElapsedTime(&ms, ex->prof_ev[i], ex->prof_ev[i + 1]) == cudaSuccess) ex->stage_ms[i] += ms;
        }
        ex->stage_calls++;
        ex->prof_pending = false;
    }
    bool cand = false;
    for (int i = 0; i < count; i++) {
        if (ex->h_flags[i] & kFlagNodeOverflow) { set_error("image %d: quadtree node buffer overflow", i); return SFE_ERR_CAPACITY; }
        cand = cand || (ex->h_flags[i] & kFlagCandOverflow);
    }
    if (cand) return grow_candidate_buffers(ex, count);
    for (int i = 0; i < count; i++)
        if (ex->h_flags[i] & kFlagOutOverflow) { set_error("image %d: more keypoints than the caller's capacity", i); return SFE_ERR_CAPACITY; }
    return SFE_OK;
}

// end of a _dev call: synchronous handles wait and report now; asynchronous ones leave both to sfe_extractor_wait
static int finish_dev(sfe_extractor *ex, int count) {
    if (ex->async_dev) return SFE_OK;
    return check_flags(ex, ex->stream, count);
}

static int prepare(sfe_extractor *ex, int count, int w, int h, int stride, int cap) {
    SFE_REQUIRE(ex != nullptr, SFE_ERR_BAD_ARG, "null handle");
    SFE_REQUIRE(count >= 1 && count <= ex->max_images, SFE_ERR_BAD_ARG, "count outside [1, max_images]");
    SFE_REQUIRE(w > 0 && h > 0 && stride >= w, SFE_ERR_BAD_ARG, "bad image geometry");
    SFE_REQUIRE(cap >= 1 && cap < 65536, SFE_ERR_BAD_ARG, "capacity must be in [1, 65535]");
    if (w != ex->w || h != ex->h) {
        if (ex->tail_pending) SFE_CUDA(cudaStreamSynchronize(ex->aux[1]));  // buffers are about to be reallocated
        int rc = build_plan(ex, w, h);
        if (rc != SFE_OK) { ex->w = ex->h = 0; return rc; }
    }
    return SFE_OK;
}

// upload `count` host images into the tight staging buffer at slot `first`
static int upload_images(sfe_extractor *ex, cudaStream_t st, const uint8_t *images, size_t image_stride, int count, int w,
                         int h, int stride, int first) {
    uint8_t *dst = ex->d_in.p + (size_t)first * w * h;
    if (stride == w && image_stride == (size_t)w * h) {
        SFE_CUDA(cudaMemcpyAsync(dst, images, (size_t)count * w * h, cudaMemcpyHostToDevice, st));
    } else {  // (a 2-D copy of 1241-byte rows runs at a third of the 1-D rate: only for callers with padded rows)
        for (int i = 0; i < count; i++)
            SFE_CUDA(cudaMemcpy2DAsync(dst + (size_t)i * w * h, w, images + (size_t)i * image_stride, stride, w, h,
                                       cudaMemcpyHostToDevice, st));
    }
    return SFE_OK;
}

// tight staging slots [first, first + count) -> pitched level-0 planes (same slots) on stream st
static void realign_images(sfe_extractor *ex, cudaStream_t st, int first, int count, int w, int h) {
    const size_t p0 = ex->pitch0;
    launch_k(realign_kernel, dim3(div_up((int)p0 / 16, 32), div_up(h, 8), count), dim3(32, 8), 0, st, false,
             (const uint8_t *)(ex->d_in.p + (size_t)first * w * h), (size_t)w * h, w, ex->d_l0.p + (size_t)first * p0 * h, p0 * h, (int)p0, w, h);
    ex->launches++;
}

// How many sub-batches a host call of `units` frames is cut into: the copies of one sub-batch overlap the
// kernels of its neighbours (H2D, compute and D2H each on their own stream).
static int pipeline_chunks(const sfe_extractor *ex, int units) {
    // measured on B200 (gpurun_out r22): sub-batches of ~16 stereo frames keep every stream busy
    int n = ex->chunks_override > 0 ? ex->chunks_override : (units >= 8 ? (units + 8) / 16 + (units < 24) : 1);
    return std::max(1, std::min(std::min(n, units), kMaxChunks));
}

static const sfe_stereo_params k_default_stereo = {3.0, 100.0, 0.5};  // src/matcher.cpp:68-70
constexpr int kGraphMaxImages = 8;  // host calls with at most this many images replay their kernels as a CUDA graph

// Host-buffer batch: `frames` images (right == nullptr) or stereo pairs, pinned or pageable host memory in and out.
// Sub-batch c: upload on s_h2d -> kernels on the compute stream -> results on s_d2h, chained with events.
// inside the sub-batch loop an error must not return past the clean-up that waits for the copies already queued into the
// caller's buffers: record it and leave the loop
#define SFE_CUDA_BREAK(call)                                                                            \
    {                                                                                                   \
        cudaError_t e_ = (call);                                                                        \
        if (e_ != cudaSuccess) {                                                                        \
            ::sfe::set_error("%s:%d: %s -> %s", __FILE__, __LINE__, #call, cudaGetErrorString(e_));     \
            rc = SFE_ERR_CUDA;                                                                          \
            break;                                                                                      \
        }                                                                                               \
    }
#define SFE_CUDA_DRAIN(call)                                                                            \
    {                                                                                                   \
        cudaError_t e_ = (call);                                                                        \
        if (e_ != cudaSuccess) {                                                                        \
            ::sfe::set_error("%s:%d: %s -> %s", __FILE__, __LINE__, #call, cudaGetErrorString(e_));     \
            return drain(SFE_ERR_CUDA);                                                                 \
        }                                                                                               \
    }
static int run_host_batch_once(sfe_extractor *ex, const uint8_t *left, const uint8_t *right, size_t image_stride, int frames, int w,
                               int h, int stride, const sfe_stereo_params *sp, sfe_keypoint *kps_l, uint8_t *desc_l, int32_t *n_l,
                               sfe_keypoint *kps_r, uint8_t *desc_r, int32_t *n_r, int32_t *stereo_idx, int32_t *stereo_dist,
                               int cap, const sfe_track_params *tp, const sfe_track_plan *plan, int32_t *track_idx,
                               int32_t *track_dist) {
    const bool stereo = right != nullptr;
    const int images = stereo ? 2 * frames : frames;
    int rc = join_tail(ex);  // an asynchronous resident call may still be matching on the side stream
    if (rc != SFE_OK) return rc;
    if ((rc = prepare(ex, images, w, h, stride, cap)) != SFE_OK) return rc;
    const size_t F = frames, wh = (size_t)ex->pitch0 * h;  // level 0 as the kernels see it: pitched rows, images back to back
    SFE_CUDA(ex->d_in.ensure((size_t)ex->max_images * w * h + 32));
    SFE_CUDA(ex->d_l0.ensure((size_t)ex->max_images * wh + 32));
    SFE_CUDA(ex->d_kps.ensure((size_t)ex->max_images * cap));
    SFE_CUDA(ex->d_desc.ensure((size_t)ex->max_images * cap * 32));
    SFE_CUDA(ex->d_nout.ensure(ex->max_images));
    if (stereo) {
        SFE_CUDA(ex->d_sidx.ensure((size_t)ex->max_images * cap));
        SFE_CUDA(ex->d_sdist.ensure((size_t)ex->max_images * cap));
    }
    sfe_keypoint *kl = ex->d_kps.p, *kr = ex->d_kps.p + F * cap;
    uint8_t *dl = ex->d_desc.p, *dr = ex->d_desc.p + F * cap * 32;
    int32_t *nl = ex->d_nout.p, *nr = ex->d_nout.p + F;
    const ImgSet B = make_imgset(ex, ex->d_l0.p, ex->d_l0.p + F * wh, frames, wh, ex->pitch0);
    prepare_l0_maps(ex, B.in_a, stereo ? B.in_b : B.in_a, frames, frames, wh, ex->pitch0);
    const OutSet O{kl, stereo ? kr : kl, dl, stereo ? dr : dl, nl, stereo ? nr : nl, cap};
    if ((rc = reset_counters(ex)) != SFE_OK) return rc;
    const int nch = pipeline_chunks(ex, frames);
    const bool piped = nch > 1;
    cudaStream_t sin = piped ? ex->s_h2d : ex->stream, sout = piped ? ex->s_d2h : ex->stream;
    const bool prof = ex->profiling;
    struct Restore {  // every exit puts the handle's mode switches back
        sfe_extractor *ex; bool prof;
        ~Restore() { ex->profiling = prof; ex->piped_now = false; ex->pdl_now = false; }
    } restore{ex, prof};
    ex->piped_now = piped;
    // a one-image / one-pair call is a chain of small dependent kernels: let each be scheduled under its predecessor's tail
    ex->pdl_now = ex->use_pdl && !piped && images <= kGraphMaxImages && !prof;
    if (piped) {
        ex->profiling = false;  // per-stage events describe one unpipelined batch
        SFE_CUDA(cudaEventRecord(ex->ev_start, ex->stream));  // the counter reset precedes every sub-batch
        for (int i = 0; i + 1 < ex->n_compute; i++) SFE_CUDA(cudaStreamWaitEvent(ex->extra[i], ex->ev_start, 0));
    }
    int bound[kMaxChunks + 1];  // sub-batch boundaries (an uneven split -- small first sub-batch -- measured slower)
    for (int c = 0; c <= nch; c++) bound[c] = (int)((long long)frames * c / nch);
    if (ex->trace) cudaEventRecord(ex->tr_ev[3 * kMaxChunks], sin);
    // small calls: arrays in pinned host memory are stored by one kernel (with the counts and the flags) instead of DMA copies
    const bool small_out = ex->use_copy_kernel && !piped && images <= kGraphMaxImages && !(tp && stereo);
    CopyPlan out_plan;
    out_plan.n = 0;
    struct Staged { void *dst; size_t off, bytes; };  // pageable destinations: stored into ex->h_stage, copied out after the wait
    Staged staged[kMaxCopySegs];
    int n_staged = 0;
    size_t stage_used = 0;
    if (small_out) {  // room for every array of the call (grow-only)
        const size_t need = (size_t)images * cap * (sizeof(sfe_keypoint) + 32 + 2 * sizeof(int32_t)) + 16 * kMaxCopySegs + sizeof(int32_t) * 2 * F;
        if (need > ex->h_stage_bytes) {
            if (ex->h_stage) cudaFreeHost(ex->h_stage);
            ex->h_stage = nullptr;
            ex->h_stage_bytes = 0;
            if (cudaHostAlloc((void **)&ex->h_stage, need, cudaHostAllocDefault) == cudaSuccess) ex->h_stage_bytes = need;
            else cudaGetLastError();
        }
    }
    // destination of one result array inside the copy kernel's plan: the caller's pages when they are pinned, else the staging buffer
    auto plan_out = [&](const void *src, void *dst, size_t bytes) -> bool {
        if (!small_out || bytes >= (1u << 31) || out_plan.n >= kMaxCopySegs - 1) return false;
        void *target = mapped_host_pointer(dst);
        if (!target) {
            const size_t room = (bytes + 15) & ~(size_t)15;
            if (!ex->h_stage || stage_used + room > ex->h_stage_bytes) return false;
            target = ex->h_stage + stage_used;
            staged[n_staged++] = Staged{dst, stage_used, bytes};
            stage_used += room;
        }
        out_plan.seg[out_plan.n++] = CopySeg{src, target, (uint32_t)bytes};
        return true;
    };
    if (small_out && !ex->h_flags_pinned && cudaHostAlloc((void **)&ex->h_flags_pinned, sizeof(int) * kGraphMaxImages, cudaHostAllocDefault) != cudaSuccess) {
        cudaGetLastError();
        ex->h_flags_pinned = nullptr;
    }
    // SFE_TRACE_SMALL=1 (diagnostic, one thread): wait after the upload, the kernels and the downloads of an unpipelined call and
    // print the mean host time of each phase every 100 calls
    static const bool trs = getenv("SFE_TRACE_SMALL") != nullptr;
    static double tr_acc[6]; static int tr_n;
    auto now_us = [] { timespec ts; clock_gettime(CLOCK_MONOTONIC, &ts); return ts.tv_sec * 1e6 + ts.tv_nsec * 1e-3; };
    double tr_t[6] = {now_us()};
    for (int c = 0; c < nch && rc == SFE_OK; c++) {
        const int f0 = bound[c], f1 = bound[c + 1], fc = f1 - f0;
        if (fc <= 0) continue;
        cudaStream_t sc = piped && c % ex->n_compute ? ex->extra[c % ex->n_compute - 1] : ex->stream;
        if ((rc = upload_images(ex, sin, left + (size_t)f0 * image_stride, image_stride, fc, w, h, stride, f0)) != SFE_OK) break;
        if (stereo && (rc = upload_images(ex, sin, right + (size_t)f0 * image_stride, image_stride, fc, w, h, stride,
                                          frames + f0)) != SFE_OK)
            break;
        if (ex->trace) cudaEventRecord(ex->tr_ev[3 * c], sin);
        if (trs) { tr_t[1] = now_us(); cudaStreamSynchronize(sin); tr_t[2] = now_us(); }
        if (piped) {
            SFE_CUDA_BREAK(cudaEventRecord(ex->ev_in[c], sin));
            SFE_CUDA_BREAK(cudaStreamWaitEvent(sc, ex->ev_in[c], 0));
        }
        auto compute = [&]() -> int {  // the kernels of this sub-batch, on stream sc
            if (stereo && fc == frames) {  // the whole call in one sub-batch: left and right slots are adjacent
                realign_images(ex, sc, 0, 2 * fc, w, h);
            } else {
                realign_images(ex, sc, f0, fc, w, h);
                if (stereo) realign_images(ex, sc, frames + f0, fc, w, h);
            }
            const OutSet Oc = chunk_of(O, f0);
            if (int r = enqueue_extract(ex, sc, chunk_of(B, f0, f1, stereo), stereo ? 2 * fc : fc, Oc)) return r;
            if (stereo) {
                launch_stereo_match(sc, fc, cap, Oc.kps_a, Oc.desc_a, Oc.n_a, Oc.kps_b, Oc.desc_b, Oc.n_b, sp->y_threshold, sp->max_dx,
                                    sp->best12_threshold, ex->d_sidx.p + (size_t)f0 * cap, ex->d_sdist.p + (size_t)f0 * cap, ex->pdl_now);
                if (!piped) prof_mark(ex, 6);
                ex->prof_has_stereo = true;
                ex->launches++;
                SFE_CUDA(cudaGetLastError());
            }
            return SFE_OK;
        };
        // Reference-shaped calls (one image, one stereo pair) are launch-bound: their kernel sequence is replayed as a CUDA
        // graph.  First sighting of a signature: run eagerly (every buffer gets allocated); second: capture + instantiate.
        sfe_extractor::GraphEntry *ge = nullptr;
        if (ex->use_graphs && !piped && images <= kGraphMaxImages && !prof && !ex->trace) {
            sfe_extractor::GraphEntry key;
            key.plan_gen = ex->plan_gen; key.frames = frames; key.cap = cap; key.stereo = stereo;
            key.sp[0] = sp->y_threshold; key.sp[1] = sp->max_dx; key.sp[2] = sp->best12_threshold;
            const void *ptrs[7] = {ex->d_in.p, ex->d_l0.p, ex->d_kps.p, ex->d_desc.p, ex->d_nout.p, stereo ? ex->d_sidx.p : nullptr,
                                   stereo ? ex->d_sdist.p : nullptr};
            memcpy(key.ptr, ptrs, sizeof(ptrs));
            for (auto &g : ex->graphs)
                if (g.plan_gen == key.plan_gen && g.frames == key.frames && g.cap == key.cap && g.stereo == key.stereo &&
                    !memcmp(g.sp, key.sp, sizeof(key.sp)) && !memcmp(g.ptr, key.ptr, sizeof(key.ptr)))
                    ge = &g;
            if (!ge) {
                if (ex->graphs.size() >= 4) {  // evict the least recently used signature
                    size_t lru = 0;
                    for (size_t i = 1; i < ex->graphs.size(); i++)
                        if (ex->graphs[i].used < ex->graphs[lru].used) lru = i;
                    if (ex->graphs[lru].exec) cudaGraphExecDestroy(ex->graphs[lru].exec);
                    ex->graphs.erase(ex->graphs.begin() + lru);
                }
                ex->graphs.push_back(key);
                ge = &ex->graphs.back();
            }
            ge->used = ++ex->graph_clock;
        }
        if (ge && ge->exec) {
            SFE_CUDA_BREAK(cudaGraphLaunch(ge->exec, sc));
            ex->launches += ge->launches;
            ex->prof_has_stereo = stereo;
        } else if (ge && ge->seen) {
            const int64_t l0 = ex->launches;
            SFE_CUDA_BREAK(cudaStreamBeginCapture(sc, cudaStreamCaptureModeRelaxed));
            rc = compute();
            cudaGraph_t graph = nullptr;
            const cudaError_t ce = cudaStreamEndCapture(sc, &graph);
            if (rc == SFE_OK && ce != cudaSuccess) {
                set_error("graph capture of a small host call failed: %s", cudaGetErrorString(ce));
                rc = SFE_ERR_CUDA;
            }
            if (rc == SFE_OK) {
                const cudaError_t ie = cudaGraphInstantiate(&ge->exec, graph, 0);
                if (ie != cudaSuccess) { set_error("cudaGraphInstantiate: %s", cudaGetErrorString(ie)); ge->exec = nullptr; rc = SFE_ERR_CUDA; }
            }
            if (graph) cudaGraphDestroy(graph);
            if (rc != SFE_OK) { cudaGetLastError(); break; }
            ge->launches = ex->launches - l0;
            SFE_CUDA_BREAK(cudaGraphLaunch(ge->exec, sc));
        } else {
            if ((rc = compute()) != SFE_OK) break;
            if (ge) ge->seen = 1;
        }
        if (ex->trace) cudaEventRecord(ex->tr_ev[3 * c + 1], sc);
        if (trs) { tr_t[3] = now_us(); cudaStreamSynchronize(sc); tr_t[4] = now_us(); }
        if (piped) {
            SFE_CUDA_BREAK(cudaEventRecord(ex->ev_done[c], sc));
            SFE_CUDA_BREAK(cudaStreamWaitEvent(sout, ex->ev_done[c], 0));
        }
        const size_t o = (size_t)f0 * cap, nk = (size_t)fc * cap;
        struct Out { const void *src; void *dst; size_t bytes; };
        const Out outs[6] = {{kl + o, kps_l + o, sizeof(sfe_keypoint) * nk},
                             {dl + o * 32, desc_l + o * 32, nk * 32},
                             {kr + o, stereo ? kps_r + o : nullptr, sizeof(sfe_keypoint) * nk},
                             {dr + o * 32, stereo ? desc_r + o * 32 : nullptr, nk * 32},
                             {ex->d_sidx.p + o, stereo ? stereo_idx + o : nullptr, sizeof(int32_t) * nk},
                             {ex->d_sdist.p + o, stereo && stereo_dist ? stereo_dist + o : nullptr, sizeof(int32_t) * nk}};
        for (const Out &g : outs) {
            if (!g.dst) continue;
            if (!plan_out(g.src, g.dst, g.bytes)) {
                cudaError_t e_ = cudaMemcpyAsync(g.dst, g.src, g.bytes, cudaMemcpyDeviceToHost, sout);
                if (e_ != cudaSuccess) { set_error("download: %s", cudaGetErrorString(e_)); rc = SFE_ERR_CUDA; break; }
            }
        }
        if (rc != SFE_OK) break;
        if (ex->trace) cudaEventRecord(ex->tr_ev[3 * c + 2], sout);
    }
    ex->profiling = prof;
    ex->piped_now = false;
    auto drain = [&](int status) {  // nothing may still be writing into the caller's buffers once the call has returned
        cudaStreamSynchronize(sin); cudaStreamSynchronize(ex->stream);
        for (auto &e : ex->extra) cudaStreamSynchronize(e);
        cudaStreamSynchronize(sout);
        return status;
    };
    if (rc != SFE_OK) return drain(rc);
    if (tp && stereo) {
        // tracking needs consecutive frames, which may sit in different sub-batches: it runs once, behind all of them
        // (sout already waits for every sub-batch), on the D2H stream's tail
        SFE_CUDA_DRAIN(ex->d_tidx.ensure((size_t)ex->max_images * cap));
        SFE_CUDA_DRAIN(ex->d_tdist.ensure((size_t)ex->max_images * cap));
        if (plan) {
            rc = launch_track_frames_plan(sout, ex->device, ex->track, frames, cap, kl, dl, nl, kr, ex->d_sidx.p, *tp, *plan,
                                          ex->d_tidx.p, ex->d_tdist.p, ex->launches);
        } else {
            rc = launch_track_frames(sout, ex->device, ex->track, frames, cap, kl, dl, nl, kr, ex->d_sidx.p, *tp, ex->d_tidx.p,
                                     ex->d_tdist.p);
            ex->launches += 3;
        }
        if (rc != SFE_OK) return drain(rc);
        SFE_CUDA_DRAIN(cudaMemcpyAsync(track_idx, ex->d_tidx.p, sizeof(int32_t) * F * cap, cudaMemcpyDeviceToHost, sout));
        if (track_dist) SFE_CUDA_DRAIN(cudaMemcpyAsync(track_dist, ex->d_tdist.p, sizeof(int32_t) * F * cap, cudaMemcpyDeviceToHost, sout));
    }
    if (!plan_out(nl, n_l, sizeof(int32_t) * F))
        SFE_CUDA_DRAIN(cudaMemcpyAsync(n_l, nl, sizeof(int32_t) * F, cudaMemcpyDeviceToHost, sout));  // after the last sub-batch
    if (stereo && !plan_out(nr, n_r, sizeof(int32_t) * F))
        SFE_CUDA_DRAIN(cudaMemcpyAsync(n_r, nr, sizeof(int32_t) * F, cudaMemcpyDeviceToHost, sout));
    const bool flags_here = small_out && ex->h_flags_pinned && out_plan.n > 0;
    if (flags_here) out_plan.seg[out_plan.n++] = CopySeg{B.flags, ex->h_flags_pinned, (uint32_t)(sizeof(int) * images)};
    if (out_plan.n > 0) {
        // (an ordinary launch: what precedes it on the stream is a graph launch, not a kernel it could be serialized under)
        SFE_CUDA_DRAIN(launch_k(copy_out_kernel, dim3(64), dim3(256), 0, sout, false, out_plan));
        ex->launches++;
    }
    ex->last = B;
    if (!stereo) ex->last.split = images;  // one set: every image reads in_a
    ex->last_count = images;
    if (trs) tr_t[5] = now_us();
    rc = check_flags(ex, sout, images, flags_here);  // sout is behind every sub-batch
    for (int i = 0; i < n_staged; i++) memcpy(staged[i].dst, ex->h_stage + staged[i].off, staged[i].bytes);
    if (trs) {
        const double e = now_us();
        const double d[6] = {tr_t[1] - tr_t[0], tr_t[2] - tr_t[1], tr_t[3] - tr_t[2], tr_t[4] - tr_t[3], tr_t[5] - tr_t[4], e - tr_t[5]};
        for (int i = 0; i < 6; i++) tr_acc[i] += d[i];
        if (++tr_n % 100 == 0) {
            fprintf(stderr, "sfe small-call trace (us, mean of 100): enqueue upload %.1f | upload done %.1f | enqueue kernels %.1f | kernels done %.1f | enqueue downloads %.1f | downloads done %.1f\n",
                    tr_acc[0] / 100, tr_acc[1] / 100, tr_acc[2] / 100, tr_acc[3] / 100, tr_acc[4] / 100, tr_acc[5] / 100);
            for (double &a : tr_acc) a = 0;
        }
    }
    if (ex->trace) {
        fprintf(stderr, "sfe trace: %d frames in %d sub-batches (ms since the first upload was queued)\n", frames, nch);
        for (int c = 0; c < nch; c++) {
            float a = 0, b = 0, d = 0;
            cudaEventElapsedTime(&a, ex->tr_ev[3 * kMaxChunks], ex->tr_ev[3 * c]);
            cudaEventElapsedTime(&b, ex->tr_ev[3 * kMaxChunks], ex->tr_ev[3 * c + 1]);
            cudaEventElapsedTime(&d, ex->tr_ev[3 * kMaxChunks], ex->tr_ev[3 * c + 2]);
            fprintf(stderr, "  sub-batch %2d frames [%3d,%3d): uploaded %.3f  computed %.3f  downloaded %.3f\n", c, bound[c], bound[c + 1], a, b, d);
        }
    }
    return rc;
}

static int run_host_batch(sfe_extractor *ex, const uint8_t *left, const uint8_t *right, size_t image_stride, int frames, int w,
                          int h, int stride, const sfe_stereo_params *sp, sfe_keypoint *kps_l, uint8_t *desc_l, int32_t *n_l,
                          sfe_keypoint *kps_r, uint8_t *desc_r, int32_t *n_r, int32_t *stereo_idx, int32_t *stereo_dist,
                          int cap, const sfe_track_params *tp = nullptr, const sfe_track_plan *plan = nullptr,
                          int32_t *track_idx = nullptr, int32_t *track_dist = nullptr) {
    int rc = kStatusRerun;
    for (int attempt = 0; attempt < 3 && rc == kStatusRerun; attempt++)  // one re-run suffices: the first pass counted exactly
        rc = run_host_batch_once(ex, left, right, image_stride, frames, w, h, stride, sp, kps_l, desc_l, n_l, kps_r, desc_r, n_r,
                                 stereo_idx, stereo_dist, cap, tp, plan, track_idx, track_dist);
    if (rc == kStatusRerun) { set_error("FAST candidate buffers still overflow after two re-runs"); rc = SFE_ERR_CAPACITY; }
    return rc;
}

extern "C" {

int sfe_extractor_create(const sfe_extractor_params *p, int device, int max_images, sfe_extractor **out) {
    SFE_REQUIRE(p && out, SFE_ERR_BAD_ARG, "null argument");
    SFE_REQUIRE(p->nlevels >= 1 && p->nlevels <= kMaxLevels, SFE_ERR_BAD_ARG, "nlevels outside [1,16]");
    SFE_REQUIRE(p->nfeatures >= 1 && p->nfeatures <= 60000, SFE_ERR_BAD_ARG, "nfeatures outside [1,60000]");
    SFE_REQUIRE(p->scale_factor > 1.0f, SFE_ERR_BAD_ARG, "scale_factor must be > 1");
    SFE_REQUIRE(p->ini_th_fast >= 1 && p->min_th_fast >= 1 && p->ini_th_fast < 255 && p->min_th_fast < 255, SFE_ERR_BAD_ARG,
                "FAST thresholds outside [1,254]");
    SFE_REQUIRE(max_images >= 1 && max_images <= 65535, SFE_ERR_BAD_ARG, "max_images outside [1,65535]");
    int ndev = 0;
    SFE_CUDA(cudaGetDeviceCount(&ndev));
    SFE_REQUIRE(ndev > 0, SFE_ERR_NO_DEVICE, "no CUDA device (there is no CPU fallback)");
    SFE_REQUIRE(device >= 0 && device < ndev, SFE_ERR_BAD_ARG, "device index out of range");
    DeviceGuard g(device);
    SFE_REQUIRE(g.ok, SFE_ERR_NO_DEVICE, "cannot select the handle's device");
    sfe_extractor *ex = new sfe_extractor();
    ex->device = device;
    ex->prm = *p;
    ex->max_images = max_images;
    cudaError_t e = cudaStreamCreateWithFlags(&ex->stream, cudaStreamNonBlocking);
    if (e != cudaSuccess) {
        set_error("cudaStreamCreate: %s", cudaGetErrorString(e));
        delete ex;
        return SFE_ERR_CUDA;
    }
    bool ok = cudaStreamCreateWithFlags(&ex->s_h2d, cudaStreamNonBlocking) == cudaSuccess &&
              cudaStreamCreateWithFlags(&ex->s_d2h, cudaStreamNonBlocking) == cudaSuccess &&
              cudaEventCreateWithFlags(&ex->ev_start, cudaEventDisableTiming) == cudaSuccess;
    for (int i = 0; i < kComputeStreams - 1 && ok; i++) ok = cudaStreamCreateWithFlags(&ex->extra[i], cudaStreamNonBlocking) == cudaSuccess;
    for (int i = 0; i < 3 && ok; i++)
        ok = cudaStreamCreateWithFlags(&ex->aux[i], cudaStreamNonBlocking) == cudaSuccess &&
             cudaEventCreateWithFlags(&ex->ev_fork[i], cudaEventDisableTiming) == cudaSuccess &&
             cudaEventCreateWithFlags(&ex->ev_join[i], cudaEventDisableTiming) == cudaSuccess;
    for (int i = 0; i < kMaxChunks && ok; i++)
        ok = cudaEventCreateWithFlags(&ex->ev_in[i], cudaEventDisableTiming) == cudaSuccess &&
             cudaEventCreateWithFlags(&ex->ev_done[i], cudaEventDisableTiming) == cudaSuccess;
    if (!ok) {
        set_error("stream/event creation: %s", cudaGetErrorString(cudaGetLastError()));
        sfe_extractor_destroy(ex);
        return SFE_ERR_CUDA;
    }
    if (const char *env = getenv("SFE_PIPELINE_CHUNKS")) ex->chunks_override = atoi(env);
    if (const char *env = getenv("SFE_NO_TMA")) ex->tma_disabled = atoi(env) != 0;
    if (const char *env = getenv("SFE_OVERLAP_BLUR")) ex->overlap_blur = atoi(env);
    cudaDeviceGetAttribute(&ex->sm_count, cudaDevAttrMultiProcessorCount, device);
    if (const char *env = getenv("SFE_OCTREE_CTAS")) ex->octree_ctas = atoi(env);
    if (const char *env = getenv("SFE_ORIENT_TMA")) ex->orient_tma = atoi(env) != 0;
    if (const char *env = getenv("SFE_OVERLAP_TAIL")) ex->overlap_tail = atoi(env) != 0;
    if (const char *env = getenv("SFE_TRACE")) ex->trace = atoi(env) != 0;
    if (const char *env = getenv("SFE_COMPUTE_STREAMS")) ex->n_compute = std::max(1, std::min(atoi(env), kComputeStreams));
    if (ex->trace)
        for (auto &e : ex->tr_ev) cudaEventCreate(&e);
    if (const char *env = getenv("SFE_OCTREE_SMEM_CAND")) ex->octree_cand_override = atoi(env);
    if (const char *env = getenv("SFE_CAND_CAP")) ex->cand_cap_override = std::max(8, atoi(env));
    if (const char *env = getenv("SFE_GRAPHS")) ex->use_graphs = atoi(env) != 0;
    if (const char *env = getenv("SFE_PDL")) ex->use_pdl = atoi(env) != 0;
    if (const char *env = getenv("SFE_OCTREE_FF")) ex->octree_ff = atoi(env) != 0;
    if (const char *env = getenv("SFE_COPY_KERNEL")) ex->use_copy_kernel = atoi(env) != 0;
    if (const char *env = getenv("SFE_SPLIT_SMALL")) ex->split_small = atoi(env) != 0;
    if (const char *env = getenv("SFE_DEV_SPLIT")) ex->dev_split = std::max(1, std::min(atoi(env), kComputeStreams));
    build_tables(ex);
    *out = ex;
    return SFE_OK;
}

int sfe_extractor_destroy(sfe_extractor *ex) {
    if (!ex) return SFE_OK;
    drop_graphs(ex);
    if (ex->h_flags_pinned) cudaFreeHost(ex->h_flags_pinned);
    if (ex->h_stage) cudaFreeHost(ex->h_stage);
    DeviceGuard g(ex->device);
    SFE_REQUIRE(g.ok, SFE_ERR_NO_DEVICE, "cannot select the handle's device");
    cudaStreamSynchronize(ex->stream);
    ex->d_pyr.release(); ex->d_blur.release(); ex->d_in.release(); ex->d_l0.release(); ex->d_octree_scratch.release(); ex->d_desc.release();
    ex->d_cand.release(); ex->d_kpst.release(); ex->d_counts.release();
    ex->d_tiles.release(); ex->d_segs.release(); ex->d_xtab.release(); ex->d_ytab.release();
    ex->d_kps.release(); ex->d_nout.release(); ex->d_sidx.release(); ex->d_sdist.release(); ex->d_tidx.release(); ex->d_tdist.release();
    ex->track.release();
    for (int i = 0; i <= kNumStages; i++)
        if (ex->prof_ev[i]) cudaEventDestroy(ex->prof_ev[i]);
    for (int i = 0; i < kMaxChunks; i++) {
        if (ex->ev_in[i]) cudaEventDestroy(ex->ev_in[i]);
        if (ex->ev_done[i]) cudaEventDestroy(ex->ev_done[i]);
    }
    for (auto &e : ex->tr_ev)
        if (e) cudaEventDestroy(e);
    for (int i = 0; i < 3; i++) {
        if (ex->ev_fork[i]) cudaEventDestroy(ex->ev_fork[i]);
        if (ex->ev_join[i]) cudaEventDestroy(ex->ev_join[i]);
        if (ex->aux[i]) cudaStreamDestroy(ex->aux[i]);
    }
    if (ex->ev_start) cudaEventDestroy(ex->ev_start);
    for (auto &e : ex->extra)
        if (e) cudaStreamDestroy(e);
    if (ex->s_h2d) cudaStreamDestroy(ex->s_h2d);
    if (ex->s_d2h) cudaStreamDestroy(ex->s_d2h);
    cudaStreamDestroy(ex->stream);
    delete ex;
    return SFE_OK;
}

int sfe_extractor_tables(const sfe_extractor *ex, float *scale, float *inv_scale, float *sigma2, float *inv_sigma2,
                         int32_t *per_level) {
    SFE_REQUIRE(ex, SFE_ERR_BAD_ARG, "null handle");
    for (int i = 0; i < ex->prm.nlevels; i++) {
        if (scale) scale[i] = ex->scale[i];
        if (inv_scale) inv_scale[i] = ex->inv_scale[i];
        if (sigma2) sigma2[i] = ex->sigma2[i];
        if (inv_sigma2) inv_sigma2[i] = ex->inv_sigma2[i];
        if (per_level) per_level[i] = ex->quota[i];
    }
    return SFE_OK;
}

int sfe_extractor_level_size(const sfe_extractor *ex, int w, int h, int level, int *lw, int *lh) {
    SFE_REQUIRE(ex && lw && lh && level >= 0 && level < ex->prm.nlevels, SFE_ERR_BAD_ARG, "bad argument");
    *lw = cv_round_f((float)w * ex->inv_scale[level]);
    *lh = cv_round_f((float)h * ex->inv_scale[level]);
    return SFE_OK;
}

// A level returns at most max(quota + 2, 4 * nIni) keypoints: DistributeOctTree stops at the first size >= N and one split adds
// at most 3 nodes (:669,730), but the first pass over the nIni roots is unconditional (:606-665) and may leave 4 * nIni nodes
// even when that exceeds N (small nfeatures on a wide image).
int sfe_extractor_max_keypoints_for(const sfe_extractor *ex, int w, int h, int *cap) {
    SFE_REQUIRE(ex && cap, SFE_ERR_BAD_ARG, "null argument");
    int total = 0;
    for (int l = 0; l < ex->prm.nlevels; l++) {
        int n_ini = 4;  // without a geometry: aspect ratios up to 4.5 : 1
        if (w > 0 && h > 0) {
            const int ww = cv_round_f((float)w * ex->inv_scale[l]) - 2 * kBorder, wh = cv_round_f((float)h * ex->inv_scale[l]) - 2 * kBorder;
            n_ini = ww > 0 && wh > 0 ? std::max(1, (int)roundf((float)ww / (float)wh)) : 1;
        }
        total += std::max(ex->quota[l] + 3, 4 * n_ini);
    }
    *cap = total;
    return SFE_OK;
}
int sfe_extractor_max_keypoints(const sfe_extractor *ex, int *cap) {
    SFE_REQUIRE(ex, SFE_ERR_BAD_ARG, "null argument");
    return sfe_extractor_max_keypoints_for(ex, ex->w, ex->h, cap);
}

int sfe_extractor_launches(const sfe_extractor *ex, int64_t *launches) {
    SFE_REQUIRE(ex && launches, SFE_ERR_BAD_ARG, "null argument");
    *launches = ex->launches;
    return SFE_OK;
}

static int extract_batch_dev_once(sfe_extractor *ex, const uint8_t *images_dev, size_t image_stride, int count, int w, int h,
                                  int stride, sfe_keypoint *kps_dev, uint8_t *desc_dev, int cap, int32_t *n_out_dev) {
    int rc = prepare(ex, count, w, h, stride, cap);
    if (rc != SFE_OK) return rc;
    const OutSet O{kps_dev, kps_dev, desc_dev, desc_dev, n_out_dev, n_out_dev, cap};
    const ImgSet S = make_imgset(ex, images_dev, images_dev, count, image_stride, stride);
    prepare_l0_maps(ex, images_dev, images_dev, count, count, image_stride, stride);
    if ((rc = reset_counters(ex)) != SFE_OK) return rc;
    const int nsplit = !ex->profiling && count >= 32 * ex->dev_split ? std::min(ex->dev_split, ex->n_compute) : 1;
    if (nsplit <= 1) {
        if ((rc = enqueue_extract(ex, ex->stream, S, count, O)) != SFE_OK) return rc;
    } else {  // sub-batches on as many streams, as in stereo_frames_dev_once
        SFE_CUDA(cudaEventRecord(ex->ev_start, ex->stream));
        for (int c = 1; c < nsplit; c++) SFE_CUDA(cudaStreamWaitEvent(ex->extra[c - 1], ex->ev_start, 0));
        for (int c = nsplit - 1; c >= 0; c--) {
            const int f0 = (int)((long long)count * c / nsplit), f1 = (int)((long long)count * (c + 1) / nsplit);
            cudaStream_t sc = c == 0 ? ex->stream : ex->extra[c - 1];
            if ((rc = enqueue_extract(ex, sc, chunk_of(S, f0, f1, false), f1 - f0, chunk_of(O, f0))) != SFE_OK) return rc;
            if (c > 0) SFE_CUDA(cudaEventRecord(ex->ev_done[c], sc));
        }
        for (int c = 1; c < nsplit; c++) SFE_CUDA(cudaStreamWaitEvent(ex->stream, ex->ev_done[c], 0));
    }
    ex->last = S;
    ex->last_count = count;
    return finish_dev(ex, count);
}

// a synchronous _dev call whose candidate buffers overflowed is run again with the enlarged buffers (the inputs are resident)
#define SFE_RERUN(call)                                                                                          \
    int rc = kStatusRerun;                                                                                       \
    for (int attempt = 0; attempt < 3 && rc == kStatusRerun; attempt++) rc = (call);                             \
    if (rc == kStatusRerun) { set_error("FAST candidate buffers still overflow after two re-runs"); rc = SFE_ERR_CAPACITY; } \
    return rc;

int sfe_extract_batch_dev(sfe_extractor *ex, const uint8_t *images_dev, size_t image_stride, int count, int w, int h,
                          int stride, sfe_keypoint *kps_dev, uint8_t *desc_dev, int cap, int32_t *n_out_dev) {
    SFE_REQUIRE(ex && images_dev && kps_dev && desc_dev && n_out_dev, SFE_ERR_BAD_ARG, "null argument");
    DeviceGuard g(ex->device);
    SFE_REQUIRE(g.ok, SFE_ERR_NO_DEVICE, "cannot select the handle's device");
    SFE_RERUN(extract_batch_dev_once(ex, images_dev, image_stride, count, w, h, stride, kps_dev, desc_dev, cap, n_out_dev));
}

int sfe_extract_batch(sfe_extractor *ex, const uint8_t *images, size_t image_stride, int count, int w, int h, int stride,
                      sfe_keypoint *kps, uint8_t *desc, int cap, int32_t *n_out) {
    SFE_REQUIRE(ex && kps && desc && n_out, SFE_ERR_BAD_ARG, "null argument");
    if (w == 0 || h == 0 || images == nullptr) {  // empty image: silent return (:1046-1047)
        for (int i = 0; i < count; i++) n_out[i] = 0;
        return SFE_OK;
    }
    DeviceGuard g(ex->device);
    SFE_REQUIRE(g.ok, SFE_ERR_NO_DEVICE, "cannot select the handle's device");
    return run_host_batch(ex, images, nullptr, image_stride, count, w, h, stride, &k_default_stereo, kps, desc, n_out, nullptr,
                          nullptr, nullptr, nullptr, nullptr, cap);
}

int sfe_extract(sfe_extractor *ex, const uint8_t *image, int w, int h, int stride, sfe_keypoint *kps, uint8_t *desc, int cap,
                int *n_out) {
    SFE_REQUIRE(n_out, SFE_ERR_BAD_ARG, "null argument");
    int32_t n = 0;
    int rc = sfe_extract_batch(ex, image, (size_t)stride * (h > 0 ? h : 0), 1, w, h, stride, kps, desc, cap, &n);
    *n_out = n;
    return rc;
}

static int stereo_frames_dev_once(sfe_extractor *ex, const uint8_t *left_dev, const uint8_t *right_dev, size_t image_stride,
                                  int frames, int w, int h, int stride, const sfe_stereo_params *sp, const sfe_track_params *tp,
                                  const sfe_track_plan *plan, sfe_keypoint *kps_l_dev, uint8_t *desc_l_dev, int32_t *n_l_dev,
                                  sfe_keypoint *kps_r_dev, uint8_t *desc_r_dev, int32_t *n_r_dev, int32_t *stereo_idx_dev,
                                  int32_t *stereo_dist_dev, int32_t *track_idx_dev, int32_t *track_dist_dev, int cap) {
    int rc = prepare(ex, 2 * frames, w, h, stride, cap);
    if (rc != SFE_OK) return rc;
    if (!sp) sp = &k_default_stereo;
    const OutSet O{kps_l_dev, kps_r_dev, desc_l_dev, desc_r_dev, n_l_dev, n_r_dev, cap};
    const ImgSet S = make_imgset(ex, left_dev, right_dev, frames, image_stride, stride);
    prepare_l0_maps(ex, left_dev, right_dev, frames, frames, image_stride, stride);
    if ((rc = reset_counters(ex)) != SFE_OK) return rc;
    const int nsplit = !ex->profiling && frames >= 16 * ex->dev_split ? std::min(ex->dev_split, ex->n_compute) : 1;
    if (nsplit <= 1) {
        if ((rc = enqueue_extract(ex, ex->stream, S, 2 * frames, O)) != SFE_OK) return rc;
    } else {
        // A large resident batch runs as nsplit sub-batches on as many streams: while one is in a latency-bound stage (quadtree,
        // the tail of a launch) the issue slots it leaves idle go to the FAST / blur / descriptor kernels of another.
        SFE_CUDA(cudaEventRecord(ex->ev_start, ex->stream));  // the counter reset precedes every sub-batch
        for (int c = 1; c < nsplit; c++) SFE_CUDA(cudaStreamWaitEvent(ex->extra[c - 1], ex->ev_start, 0));
        // (the side streams first: while a previous asynchronous call's matchers are still pending, each of them waits for that
        // tail before its descriptor kernel overwrites the arrays the matchers read; the main stream's join clears the flag)
        for (int c = nsplit - 1; c >= 0; c--) {
            const int f0 = (int)((long long)frames * c / nsplit), f1 = (int)((long long)frames * (c + 1) / nsplit);
            cudaStream_t sc = c == 0 ? ex->stream : ex->extra[c - 1];
            if ((rc = enqueue_extract(ex, sc, chunk_of(S, f0, f1, true), 2 * (f1 - f0), chunk_of(O, f0))) != SFE_OK) return rc;
            if (c > 0) SFE_CUDA(cudaEventRecord(ex->ev_done[c], sc));
        }
        for (int c = 1; c < nsplit; c++) SFE_CUDA(cudaStreamWaitEvent(ex->stream, ex->ev_done[c], 0));
    }
    // asynchronous calls: the matchers are small latency-bound kernels, so they go to a side stream and run beside the
    // next call's pyramid and FAST kernels
    const bool tail = ex->async_dev && ex->overlap_tail && !ex->profiling;
    cudaStream_t sm = tail ? ex->aux[1] : ex->stream;
    if (!tail) {
        if ((rc = join_tail(ex)) != SFE_OK) return rc;
    } else if (tp && ex->tail_pending && track_scratch_grows(ex->track, frames, cap, plan)) {
        SFE_CUDA(cudaStreamSynchronize(ex->aux[1]));  // the tracking scratch is about to grow under a running tail
    }
    if (tail) {
        SFE_CUDA(cudaEventRecord(ex->ev_fork[1], ex->stream));
        SFE_CUDA(cudaStreamWaitEvent(sm, ex->ev_fork[1], 0));
    }
    launch_stereo_match(sm, frames, cap, kps_l_dev, desc_l_dev, n_l_dev, kps_r_dev, desc_r_dev, n_r_dev, sp->y_threshold,
                        sp->max_dx, sp->best12_threshold, stereo_idx_dev, stereo_dist_dev);
    prof_mark(ex, 6);
    ex->prof_has_stereo = true;
    ex->launches++;
    SFE_CUDA(cudaGetLastError());
    if (tp && plan) {
        if ((rc = launch_track_frames_plan(sm, ex->device, ex->track, frames, cap, kps_l_dev, desc_l_dev, n_l_dev, kps_r_dev,
                                           stereo_idx_dev, *tp, *plan, track_idx_dev, track_dist_dev, ex->launches)) != SFE_OK)
            return rc;
        prof_mark(ex, 7);
        ex->prof_has_track = true;
    } else if (tp) {
        if ((rc = launch_track_frames(sm, ex->device, ex->track, frames, cap, kps_l_dev, desc_l_dev, n_l_dev, kps_r_dev,
                                      stereo_idx_dev, *tp, track_idx_dev, track_dist_dev)) != SFE_OK)
            return rc;
        prof_mark(ex, 7);
        ex->prof_has_track = true;
        ex->launches += 3;
    }
    if (tail) {
        SFE_CUDA(cudaEventRecord(ex->ev_join[1], sm));
        ex->tail_pending = true;
    }
    ex->last = S;
    ex->last_count = 2 * frames;
    return finish_dev(ex, 2 * frames);
}

static int check_track_params(const sfe_track_params *tp, const int32_t *track_idx) {
    SFE_REQUIRE(tp && track_idx, SFE_ERR_BAD_ARG, "null argument");
    SFE_REQUIRE(tp->cam.width >= 1 && tp->cam.height >= 1 && tp->cam.fx != 0. && tp->cam.fy != 0., SFE_ERR_BAD_ARG, "bad camera");
    SFE_REQUIRE(tp->radius >= 0. && tp->radius == tp->radius, SFE_ERR_BAD_ARG, "bad radius");
    return SFE_OK;
}

// a plan's contents, once `frames` is known to be valid (its priors are read for entries 1..frames-1)
static int check_track_plan(const sfe_track_plan *plan, int frames) {
    SFE_REQUIRE(!(plan->rt && plan->se3), SFE_ERR_BAD_ARG, "a track plan takes rt or se3 priors, not both");
    SFE_REQUIRE(plan->retry_radius >= 0., SFE_ERR_BAD_ARG, "bad retry radius");
    SFE_REQUIRE(plan->retry_below >= 0, SFE_ERR_BAD_ARG, "negative retry_below");
    const int per = plan->rt ? 12 : 7;
    const double *v = plan->rt ? plan->rt : plan->se3 ? &plan->se3->qx : nullptr;
    static_assert(sizeof(sfe_se3) == 7 * sizeof(double), "sfe_se3 is read as 7 doubles");
    for (size_t i = per; v && i < (size_t)frames * per; i++)
        SFE_REQUIRE(std::isfinite(v[i]), SFE_ERR_BAD_ARG, "a motion prior is not finite");
    return SFE_OK;
}

static int stereo_frames_dev_impl(sfe_extractor *ex, const uint8_t *left_dev, const uint8_t *right_dev, size_t image_stride,
                                  int frames, int w, int h, int stride, const sfe_stereo_params *sp, const sfe_track_params *tp,
                                  const sfe_track_plan *plan, sfe_keypoint *kps_l_dev, uint8_t *desc_l_dev, int32_t *n_l_dev,
                                  sfe_keypoint *kps_r_dev, uint8_t *desc_r_dev, int32_t *n_r_dev, int32_t *stereo_idx_dev,
                                  int32_t *stereo_dist_dev, int32_t *track_idx_dev, int32_t *track_dist_dev, int cap) {
    SFE_REQUIRE(ex && left_dev && right_dev && kps_l_dev && desc_l_dev && n_l_dev && kps_r_dev && desc_r_dev && n_r_dev &&
                    stereo_idx_dev,
                SFE_ERR_BAD_ARG, "null argument");
    SFE_REQUIRE(frames >= 1 && 2 * frames <= ex->max_images, SFE_ERR_BAD_ARG, "2*frames exceeds max_images");
    if (plan)
        if (int rc = check_track_plan(plan, frames)) return rc;
    DeviceGuard g(ex->device);
    SFE_REQUIRE(g.ok, SFE_ERR_NO_DEVICE, "cannot select the handle's device");
    SFE_RERUN(stereo_frames_dev_once(ex, left_dev, right_dev, image_stride, frames, w, h, stride, sp, tp, plan, kps_l_dev,
                                     desc_l_dev, n_l_dev, kps_r_dev, desc_r_dev, n_r_dev, stereo_idx_dev, stereo_dist_dev,
                                     track_idx_dev, track_dist_dev, cap));
}

int sfe_stereo_frames_dev(sfe_extractor *ex, const uint8_t *left_dev, const uint8_t *right_dev, size_t image_stride,
                          int frames, int w, int h, int stride, const sfe_stereo_params *sp, sfe_keypoint *kps_l_dev,
                          uint8_t *desc_l_dev, int32_t *n_l_dev, sfe_keypoint *kps_r_dev, uint8_t *desc_r_dev,
                          int32_t *n_r_dev, int32_t *stereo_idx_dev, int32_t *stereo_dist_dev, int cap) {
    return stereo_frames_dev_impl(ex, left_dev, right_dev, image_stride, frames, w, h, stride, sp, nullptr, nullptr, kps_l_dev,
                                  desc_l_dev, n_l_dev, kps_r_dev, desc_r_dev, n_r_dev, stereo_idx_dev, stereo_dist_dev, nullptr,
                                  nullptr, cap);
}

int sfe_stereo_sequence_dev(sfe_extractor *ex, const uint8_t *left_dev, const uint8_t *right_dev, size_t image_stride, int frames,
                            int w, int h, int stride, const sfe_stereo_params *sp, const sfe_track_params *tp,
                            sfe_keypoint *kps_l_dev, uint8_t *desc_l_dev, int32_t *n_l_dev, sfe_keypoint *kps_r_dev,
                            uint8_t *desc_r_dev, int32_t *n_r_dev, int32_t *stereo_idx_dev, int32_t *stereo_dist_dev,
                            int32_t *track_idx_dev, int32_t *track_dist_dev, int cap) {
    if (int rc = check_track_params(tp, track_idx_dev)) return rc;
    return stereo_frames_dev_impl(ex, left_dev, right_dev, image_stride, frames, w, h, stride, sp, tp, nullptr, kps_l_dev,
                                  desc_l_dev, n_l_dev, kps_r_dev, desc_r_dev, n_r_dev, stereo_idx_dev, stereo_dist_dev,
                                  track_idx_dev, track_dist_dev, cap);
}

int sfe_stereo_sequence_plan_dev(sfe_extractor *ex, const uint8_t *left_dev, const uint8_t *right_dev, size_t image_stride,
                                 int frames, int w, int h, int stride, const sfe_stereo_params *sp, const sfe_track_params *tp,
                                 const sfe_track_plan *plan, sfe_keypoint *kps_l_dev, uint8_t *desc_l_dev, int32_t *n_l_dev,
                                 sfe_keypoint *kps_r_dev, uint8_t *desc_r_dev, int32_t *n_r_dev, int32_t *stereo_idx_dev,
                                 int32_t *stereo_dist_dev, int32_t *track_idx_dev, int32_t *track_dist_dev, int cap) {
    if (int rc = check_track_params(tp, track_idx_dev)) return rc;
    SFE_REQUIRE(plan, SFE_ERR_BAD_ARG, "null track plan");
    return stereo_frames_dev_impl(ex, left_dev, right_dev, image_stride, frames, w, h, stride, sp, tp, plan, kps_l_dev,
                                  desc_l_dev, n_l_dev, kps_r_dev, desc_r_dev, n_r_dev, stereo_idx_dev, stereo_dist_dev,
                                  track_idx_dev, track_dist_dev, cap);
}

int sfe_stereo_frames(sfe_extractor *ex, const uint8_t *left, const uint8_t *right, size_t image_stride, int frames, int w,
                      int h, int stride, const sfe_stereo_params *sp, sfe_keypoint *kps_l, uint8_t *desc_l, int32_t *n_l,
                      sfe_keypoint *kps_r, uint8_t *desc_r, int32_t *n_r, int32_t *stereo_idx, int32_t *stereo_dist,
                      int cap) {
    SFE_REQUIRE(ex && left && right && kps_l && desc_l && n_l && kps_r && desc_r && n_r && stereo_idx, SFE_ERR_BAD_ARG,
                "null argument");
    SFE_REQUIRE(frames >= 1 && 2 * frames <= ex->max_images, SFE_ERR_BAD_ARG, "2*frames exceeds max_images");
    DeviceGuard g(ex->device);
    SFE_REQUIRE(g.ok, SFE_ERR_NO_DEVICE, "cannot select the handle's device");
    return run_host_batch(ex, left, right, image_stride, frames, w, h, stride, sp ? sp : &k_default_stereo, kps_l, desc_l, n_l,
                          kps_r, desc_r, n_r, stereo_idx, stereo_dist, cap);
}

int sfe_stereo_sequence(sfe_extractor *ex, const uint8_t *left, const uint8_t *right, size_t image_stride, int frames, int w,
                        int h, int stride, const sfe_stereo_params *sp, const sfe_track_params *tp, sfe_keypoint *kps_l,
                        uint8_t *desc_l, int32_t *n_l, sfe_keypoint *kps_r, uint8_t *desc_r, int32_t *n_r, int32_t *stereo_idx,
                        int32_t *stereo_dist, int32_t *track_idx, int32_t *track_dist, int cap) {
    SFE_REQUIRE(ex && left && right && kps_l && desc_l && n_l && kps_r && desc_r && n_r && stereo_idx, SFE_ERR_BAD_ARG,
                "null argument");
    if (int rc = check_track_params(tp, track_idx)) return rc;
    SFE_REQUIRE(frames >= 1 && 2 * frames <= ex->max_images, SFE_ERR_BAD_ARG, "2*frames exceeds max_images");
    DeviceGuard g(ex->device);
    SFE_REQUIRE(g.ok, SFE_ERR_NO_DEVICE, "cannot select the handle's device");
    return run_host_batch(ex, left, right, image_stride, frames, w, h, stride, sp ? sp : &k_default_stereo, kps_l, desc_l, n_l,
                          kps_r, desc_r, n_r, stereo_idx, stereo_dist, cap, tp, nullptr, track_idx, track_dist);
}

int sfe_stereo_sequence_plan(sfe_extractor *ex, const uint8_t *left, const uint8_t *right, size_t image_stride, int frames, int w,
                             int h, int stride, const sfe_stereo_params *sp, const sfe_track_params *tp, const sfe_track_plan *plan,
                             sfe_keypoint *kps_l, uint8_t *desc_l, int32_t *n_l, sfe_keypoint *kps_r, uint8_t *desc_r,
                             int32_t *n_r, int32_t *stereo_idx, int32_t *stereo_dist, int32_t *track_idx, int32_t *track_dist,
                             int cap) {
    SFE_REQUIRE(ex && left && right && kps_l && desc_l && n_l && kps_r && desc_r && n_r && stereo_idx, SFE_ERR_BAD_ARG,
                "null argument");
    if (int rc = check_track_params(tp, track_idx)) return rc;
    SFE_REQUIRE(plan, SFE_ERR_BAD_ARG, "null track plan");
    SFE_REQUIRE(frames >= 1 && 2 * frames <= ex->max_images, SFE_ERR_BAD_ARG, "2*frames exceeds max_images");
    if (int rc = check_track_plan(plan, frames)) return rc;
    DeviceGuard g(ex->device);
    SFE_REQUIRE(g.ok, SFE_ERR_NO_DEVICE, "cannot select the handle's device");
    return run_host_batch(ex, left, right, image_stride, frames, w, h, stride, sp ? sp : &k_default_stereo, kps_l, desc_l, n_l,
                          kps_r, desc_r, n_r, stereo_idx, stereo_dist, cap, tp, plan, track_idx, track_dist);
}

int sfe_image_pitch(int w) { return w > 0 ? (int)align_up((size_t)w, 16) : 0; }

int sfe_extractor_set_async(sfe_extractor *ex, int enable) {
    SFE_REQUIRE(ex, SFE_ERR_BAD_ARG, "null handle");
    DeviceGuard g(ex->device);
    SFE_REQUIRE(g.ok, SFE_ERR_NO_DEVICE, "cannot select the handle's device");
    if (int rc = join_tail(ex)) return rc;
    SFE_CUDA(cudaStreamSynchronize(ex->stream));
    ex->async_dev = enable != 0;
    if (ex->d_counts.p)  // start from clean flags
        SFE_CUDA(cudaMemset(ex->d_counts.p + (size_t)ex->max_images * ex->prm.nlevels * 2 + 1, 0, sizeof(int) * ex->max_images));
    return SFE_OK;
}

int sfe_extractor_wait(sfe_extractor *ex) {
    SFE_REQUIRE(ex, SFE_ERR_BAD_ARG, "null handle");
    DeviceGuard g(ex->device);
    SFE_REQUIRE(g.ok, SFE_ERR_NO_DEVICE, "cannot select the handle's device");
    if (int rc = join_tail(ex)) return rc;
    if (ex->last_count <= 0) {
        SFE_CUDA(cudaStreamSynchronize(ex->stream));
        return SFE_OK;
    }
    int rc = check_flags(ex, ex->stream, ex->max_images);
    if (rc == kStatusRerun) {  // the inputs of a queued batch are the caller's: it has to be submitted again
        set_error("a queued batch overflowed its FAST candidate buffers; they have been enlarged, submit the batch again");
        rc = SFE_ERR_CAPACITY;
    }
    if (ex->async_dev && ex->d_counts.p)
        SFE_CUDA(cudaMemset(ex->d_counts.p + (size_t)ex->max_images * ex->prm.nlevels * 2 + 1, 0, sizeof(int) * ex->max_images));
    return rc;
}

// ---- stage taps ---------------------------------------------------------------------------------
static int tap_check(sfe_extractor *ex, int image, int level) {
    SFE_REQUIRE(ex, SFE_ERR_BAD_ARG, "null handle");
    SFE_REQUIRE(ex->last_count > 0 && image >= 0 && image < ex->last_count, SFE_ERR_BAD_ARG, "image index outside the last call");
    SFE_REQUIRE(level >= 0 && level < ex->prm.nlevels, SFE_ERR_BAD_ARG, "level out of range");
    return SFE_OK;
}

int sfe_debug_level(sfe_extractor *ex, int image, int level, uint8_t *out) {
    int rc = tap_check(ex, image, level);
    if (rc != SFE_OK) return rc;
    SFE_REQUIRE(out, SFE_ERR_BAD_ARG, "null argument");
    DeviceGuard g(ex->device);
    SFE_REQUIRE(g.ok, SFE_ERR_NO_DEVICE, "cannot select the handle's device");
    const LevelPlan &L = ex->lv[level];
    const ImgSet &S = ex->last;
    const uint8_t *src;
    int pitch;
    if (level == 0) {
        pitch = S.in_pitch;
        src = image < S.split ? S.in_a + (size_t)image * S.in_stride : S.in_b + (size_t)(image - S.split) * S.in_stride;
    } else {
        pitch = L.pitch;
        src = S.pyr + (size_t)image * S.pyr_stride + L.plane_off;
    }
    SFE_CUDA(cudaStreamSynchronize(ex->stream));
    SFE_CUDA(cudaMemcpy2D(out, L.w, src, pitch, L.w, L.h, cudaMemcpyDeviceToHost));
    return SFE_OK;
}

int sfe_debug_blur(sfe_extractor *ex, int image, int level, uint8_t *out) {
    int rc = tap_check(ex, image, level);
    if (rc != SFE_OK) return rc;
    SFE_REQUIRE(out, SFE_ERR_BAD_ARG, "null argument");
    DeviceGuard g(ex->device);
    SFE_REQUIRE(g.ok, SFE_ERR_NO_DEVICE, "cannot select the handle's device");
    const LevelPlan &L = ex->lv[level];
    SFE_CUDA(cudaStreamSynchronize(ex->stream));
    SFE_CUDA(cudaMemcpy2D(out, L.w, ex->last.blur + (size_t)image * ex->last.blur_stride + L.blur_off, L.blur_pitch, L.w, L.h,
                          cudaMemcpyDeviceToHost));
    return SFE_OK;
}

static int tap_points(sfe_extractor *ex, int image, int level, bool distributed, float *xyr, int cap, int *n) {
    int rc = tap_check(ex, image, level);
    if (rc != SFE_OK) return rc;
    SFE_REQUIRE(xyr && n && cap >= 0, SFE_ERR_BAD_ARG, "null argument");
    DeviceGuard g(ex->device);
    SFE_REQUIRE(g.ok, SFE_ERR_NO_DEVICE, "cannot select the handle's device");
    const LevelPlan &L = ex->lv[level];
    const ImgSet &S = ex->last;
    SFE_CUDA(cudaStreamSynchronize(ex->stream));
    int cnt = 0;
    const int *cp = (distributed ? S.kp_count : S.cand_count) + image * S.nlevels + level;
    SFE_CUDA(cudaMemcpy(&cnt, cp, sizeof(int), cudaMemcpyDeviceToHost));
    cnt = std::min(cnt, distributed ? L.kp_cap : L.cand_cap);
    std::vector<uint32_t> v(std::max(cnt, 1));
    const uint32_t *src = distributed ? S.kpst + (size_t)image * S.kpst_stride + L.kp_off
                                      : S.cand + (size_t)image * S.cand_stride + L.cand_off;
    if (cnt > 0) SFE_CUDA(cudaMemcpy(v.data(), src, sizeof(uint32_t) * cnt, cudaMemcpyDeviceToHost));
    v.resize(cnt);
    if (!distributed) {  // device order is arbitrary; present the reference's cell-major raster order
        const int wc = L.w_cell, hc = L.h_cell;
        auto key = [wc, hc](uint32_t p) {
            const uint64_t x = p & 0xFFF, y = (p >> 12) & 0xFFF;
            return ((((y - 3) / hc) * 4096 + (x - 3) / wc) * 4096 + y) * 4096 + x;
        };
        std::sort(v.begin(), v.end(), [&](uint32_t a, uint32_t b) { return key(a) < key(b); });
    }
    for (int i = 0; i < cnt && i < cap; i++) {
        xyr[3 * i] = (float)(v[i] & 0xFFF);
        xyr[3 * i + 1] = (float)((v[i] >> 12) & 0xFFF);
        xyr[3 * i + 2] = (float)(v[i] >> 24);
    }
    *n = cnt;
    return SFE_OK;
}

int sfe_debug_candidates(sfe_extractor *ex, int image, int level, float *xyr, int cap, int *n) {
    return tap_points(ex, image, level, false, xyr, cap, n);
}
int sfe_debug_distributed(sfe_extractor *ex, int image, int level, float *xyr, int cap, int *n) {
    return tap_points(ex, image, level, true, xyr, cap, n);
}

int sfe_extractor_set_profiling(sfe_extractor *ex, int enable) {
    SFE_REQUIRE(ex, SFE_ERR_BAD_ARG, "null handle");
    DeviceGuard g(ex->device);
    SFE_REQUIRE(g.ok, SFE_ERR_NO_DEVICE, "cannot select the handle's device");
    if (enable && !ex->prof_ev[0])
        for (int i = 0; i <= kNumStages; i++) SFE_CUDA(cudaEventCreate(&ex->prof_ev[i]));
    ex->profiling = enable != 0;
    for (int i = 0; i < kNumStages; i++) ex->stage_ms[i] = 0.0;
    ex->stage_calls = 0;
    return SFE_OK;
}

int sfe_extractor_stage_ms(const sfe_extractor *ex, double *ms, int n, int64_t *calls) {
    SFE_REQUIRE(ex && ms && calls && n >= 1, SFE_ERR_BAD_ARG, "bad argument");
    for (int i = 0; i < n; i++) ms[i] = i < kNumStages ? ex->stage_ms[i] : 0.0;
    *calls = ex->stage_calls;
    return SFE_OK;
}

int sfe_event_record_extractor(sfe_event *ev, sfe_extractor *ex) {
    SFE_REQUIRE(ev && ex, SFE_ERR_BAD_ARG, "null argument");
    DeviceGuard g(ex->device);
    SFE_REQUIRE(g.ok, SFE_ERR_NO_DEVICE, "cannot select the handle's device");
    if (int rc = join_tail(ex)) return rc;  // the event marks the end of everything enqueued so far
    SFE_CUDA(cudaEventRecord(ev->ev, ex->stream));
    return SFE_OK;
}

}  // extern "C"
