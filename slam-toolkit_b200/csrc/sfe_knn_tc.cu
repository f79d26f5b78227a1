// Brute-force Hamming top-2 for MANY queries on the 5th-generation tensor cores (tcgen05, sm_100a).
//
// For 256-bit descriptors a, b:  hamming(a, b) = |a| + |b| - 2 <a, b> = |a| + sum_k b_k (1 - 2 a_k).  With the query bits
// unpacked to int8 {+1, -1} (= 1 - 2 a_k) and the database bits to int8 {0, 1}, the Q x M values  D' = hamming - |a|  are an
// int8 GEMM with K = 256 whose int32 accumulators are exact, so the distances -- and the lexicographic (distance, row) top-2
// the matchers of the reference keep (src/matcher.cpp:114-123) -- are bit-identical to the XOR / POPC kernels
// (knn2_partial_kernel), at a fraction of their integer-pipe cost: the pair loop shrinks from 16 LOP3 + 4 POPC + 3 min/max
// per pair to half a min per pair in the epilogue, which only looks closer at the rare accumulator that can still enter a
// query's top-2 (BASELINE config 4: 2000 queries x 10 M rows).
//
// One persistent CTA per SM works on one (query group of 512, chunk of database rows) item:
//   * the group's 4 x 128 queries are unpacked once into shared memory as four A tiles (K-major, no swizzle: 8-row x 16-byte
//     core matrices, LBO = 128 B between K chunks, SBO = 2048 B between 8-row groups);
//   * the chunk's database rows arrive 128 at a time as B tiles of the same layout: ready-made from HBM by one bulk copy per
//     tile (cp.async.bulk, three in flight) when the map keeps an unpacked copy (256 B per row, built at the first many-query
//     search if it fits the budget), else unpacked by 2 producer warps into one of two B tiles;
//   * two issuer warps, one per TMEM stage (an elected lane each), issue tcgen05.mma.kind::i8 (M = 128, N = 128, K = 32, 8 per
//     tile pair) into TMEM: two stages of two 128-column accumulators each fill the 512 columns;
//   * 16 epilogue warps, 8 per TMEM stage, drain their stage with tcgen05.ld.pack::16b (thread = query row; the accumulators lie
//     in [-256, 256], so two of them travel in one register: 128 columns = two loads of 32 registers, both in flight) and give
//     the stage back before looking at the values: packed 16x2 minima are compared with the query's current second-best D';
//     only a group of 8 that can still matter is turned into keys ((D' + 512) << 22 | row in chunk) and inserted;
//   * mbarriers carry the B-tile full / empty and TMEM full / empty hand-offs; tcgen05.commit arrives on them.
// Output = the same per-(chunk, query) pair of 64-bit keys (distance << 32 | global row) the other partial kernels
// write, so knn2_merge_kernel / knn2_merge_push_kernel finish the job.
#include <algorithm>
#include <mutex>

#include "sfe_common.cuh"
#include "sfe_tma.cuh"

namespace sfe {

namespace {

constexpr int kTileN = 128;                   // database rows per B tile = N of one MMA (N = 256 tiles measured slower, DESIGN.md §9)
constexpr int kGroupTiles = 4, kGroupQ = 128 * kGroupTiles;  // query tiles / queries per work item: one 128-column accumulator each
constexpr int kEpiWarps = 16;  // 8 per TMEM stage: one per (lane quadrant, half of the stage's 256 columns); a stage's warps examine
                               // their registers while the other stage's warps wait for theirs
#ifndef SFE_TC_PRODUCERS
#define SFE_TC_PRODUCERS 2
#endif
constexpr int kProdWarps = SFE_TC_PRODUCERS;           // 2: 20 warps in all = 640 threads, which leaves 96 registers per thread
constexpr int kTcThreads = (2 + kProdWarps + kEpiWarps) * 32;  // warps 0-1: MMA issuers (one per TMEM stage), then the producers, then the epilogue
constexpr int kATileBytes = 128 * 256, kBTileBytes = kTileN * 256;  // operand tiles: rows x 256 int8
constexpr uint32_t kSBO = 2048, kLBO = 128;  // bytes: between 8-row groups / between 16-byte K chunks
constexpr int kKeyOffset = 512;              // keeps D' = |b| - 2 dot non-negative in the key (D' >= -256)
constexpr uint32_t kNoKey32 = 0xFFFFFFFFu;
#ifndef SFE_TC_PREFETCH
#define SFE_TC_PREFETCH 0
#endif
constexpr bool kPrefetchB = SFE_TC_PREFETCH != 0;  // fetch the next tile's bits before writing this one (measured: slower, DESIGN.md §9)

// ---- PTX wrappers ------------------------------------------------------------------------------------------------
__device__ __forceinline__ void fence_async_smem() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void mbar_arrive(uint64_t *bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
// tcgen05.commit: the barrier gets one arrival once every MMA issued so far by this thread has completed
__device__ __forceinline__ void tc_commit(uint64_t *bar) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar)) : "memory");
}
// shared-memory matrix descriptor, K-major, no swizzle (cute::UMMA::SmemDescriptor): start >> 4 | LBO >> 4 << 16 |
// SBO >> 4 << 32 | version 1 << 46
__device__ __forceinline__ uint64_t smem_desc(uint32_t addr) {
    return (uint64_t)((addr & 0x3FFFF) >> 4) | (uint64_t)(kLBO >> 4) << 16 | (uint64_t)(kSBO >> 4) << 32 | 1ull << 46;
}
// instruction descriptor (cute::UMMA::InstrDescriptor): D = S32, A = B = signed 8-bit, both K-major, N >> 3, M >> 4
constexpr uint32_t kIdesc = (2u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(kTileN >> 3) << 17) | ((128u >> 4) << 24);  // M = 128, N = kTileN
__device__ __forceinline__ void mma_i8(uint32_t d_tmem, uint64_t a_desc, uint64_t b_desc, bool accumulate) {
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "setp.ne.b32 p, %4, 0;\n"
        "tcgen05.mma.cta_group::1.kind::i8 [%0], %1, %2, %3, {%5, %5, %5, %5}, p;\n"
        "}\n" ::"r"(d_tmem),
        "l"(a_desc), "l"(b_desc), "r"(kIdesc), "r"((uint32_t)accumulate), "r"(0u)
        : "memory");
}
// TMEM loads are asynchronous: tmem_ld_wait2 makes the registers valid (they are operands of the wait so that no use moves above it).
#define SFE_R32(v) "+r"(v[0]), "+r"(v[1]), "+r"(v[2]), "+r"(v[3]), "+r"(v[4]), "+r"(v[5]), "+r"(v[6]), "+r"(v[7]), "+r"(v[8]), "+r"(v[9]), \
                   "+r"(v[10]), "+r"(v[11]), "+r"(v[12]), "+r"(v[13]), "+r"(v[14]), "+r"(v[15]), "+r"(v[16]), "+r"(v[17]), "+r"(v[18]),   \
                   "+r"(v[19]), "+r"(v[20]), "+r"(v[21]), "+r"(v[22]), "+r"(v[23]), "+r"(v[24]), "+r"(v[25]), "+r"(v[26]), "+r"(v[27]),   \
                   "+r"(v[28]), "+r"(v[29]), "+r"(v[30]), "+r"(v[31])
__device__ __forceinline__ void tmem_ld_wait2(int (&v)[32], int (&w)[32]) {  // two loads in flight: both register sets hang on the wait
    asm volatile("tcgen05.wait::ld.sync.aligned;" : SFE_R32(v)::"memory");
    asm volatile("" : SFE_R32(w)::"memory");
}

// The same load with .pack::16b: 64 consecutive columns, the low halves of columns 2 i and 2 i + 1 in register i (the accumulators
// D' lie in [-256, 256]: their low 16 bits are the value).  Half the bytes cross from tensor memory to the register file, and the
// epilogue's minima work on two accumulators per instruction (tools/tc_pack_probe.cu, tools/tc_tmem_ld_rate.cu).
__device__ __forceinline__ void tmem_ld64p_issue(uint32_t addr, int (&v)[32]) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x32.pack::16b.b32 {%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16, %17, "
        "%18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
        : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]), "=r"(v[8]), "=r"(v[9]),
          "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15]), "=r"(v[16]), "=r"(v[17]), "=r"(v[18]),
          "=r"(v[19]), "=r"(v[20]), "=r"(v[21]), "=r"(v[22]), "=r"(v[23]), "=r"(v[24]), "=r"(v[25]), "=r"(v[26]), "=r"(v[27]),
          "=r"(v[28]), "=r"(v[29]), "=r"(v[30]), "=r"(v[31])
        : "r"(addr)
        : "memory");
}

// 16 descriptor bits -> 16 bytes of {0, 1}: bit k of the half-word goes to byte k (any fixed order works: both operands use it);
// unpack16_pm turns them into {+1, -1} = 1 - 2 bit
__device__ __forceinline__ uint4 unpack16(uint32_t bits) {
    uint4 o;
    o.x = ((bits & 0xFu) * 0x00204081u) & 0x01010101u;
    o.y = (((bits >> 4) & 0xFu) * 0x00204081u) & 0x01010101u;
    o.z = (((bits >> 8) & 0xFu) * 0x00204081u) & 0x01010101u;
    o.w = (((bits >> 12) & 0xFu) * 0x00204081u) & 0x01010101u;
    return o;
}
__device__ __forceinline__ uint4 unpack16_pm(uint32_t bits) {
    uint4 o = unpack16(bits);
    o.x = 0x01010101u | (o.x * 0xFEu);  // byte 0 -> 0x01, byte 1 -> 0xFF; no carry crosses a byte
    o.y = 0x01010101u | (o.y * 0xFEu);
    o.z = 0x01010101u | (o.z * 0xFEu);
    o.w = 0x01010101u | (o.w * 0xFEu);
    return o;
}
// byte offset of (row, 16-byte K chunk) inside an operand tile
__device__ __forceinline__ uint32_t tile_off(int row, int chunk) { return (uint32_t)(row >> 3) * kSBO + (uint32_t)chunk * kLBO + (uint32_t)(row & 7) * 16; }

// the two smallest of {k0 <= k1, x, y}
__device__ __forceinline__ void top2_pair(uint32_t &k0, uint32_t &k1, uint32_t x, uint32_t y) {
    const uint32_t lo = min(x, y), hi = max(x, y);
    k1 = min(min(k1, hi), max(k0, lo));
    k0 = min(k0, lo);
}
__device__ __forceinline__ void top2_one(uint32_t &k0, uint32_t &k1, uint32_t x) {
    k1 = min(k1, max(k0, x));
    k0 = min(k0, x);
}

// 8 accumulators of which at least one can still enter the query's top-2: key and insert the valid ones (a few percent of
// the groups; kept inline: out of line, the running top-2 would live in local memory around every call)
__device__ __forceinline__ void insert8(int v0, int v1, int v2, int v3, int v4, int v5, int v6, int v7, uint32_t idx, uint32_t chunk_n,
                                     uint32_t &k0, uint32_t &k1, int &thr) {
    const int v[8] = {v0, v1, v2, v3, v4, v5, v6, v7};
#pragma unroll
    for (int e = 0; e < 8; e++)
        if (v[e] <= thr && idx + e < chunk_n) top2_one(k0, k1, (uint32_t)(v[e] + kKeyOffset) << 22 | (idx + e));
    thr = (int)(k1 >> 22) - kKeyOffset;  // 511 while fewer than two rows have been seen: everything passes
}

// 64 accumulators of one query as 32 packed pairs (rows idx0 .. idx0 + 63 of the chunk; register i = rows 2 i, 2 i + 1): one
// test of their minimum against the query's second-best distance drops them all; otherwise the groups of 8 whose own minimum
// passes are unpacked, keyed and inserted
__device__ __forceinline__ void examine64p(const int (&v)[32], uint32_t &k0, uint32_t &k1, int &thr, uint32_t idx0, uint32_t chunk_n) {
    uint32_t g[8];  // packed minima of 4 registers = 8 accumulators
#pragma unroll
    for (int j = 0; j < 8; j++)
        g[j] = __vmins2(__vimin3_s16x2((uint32_t)v[4 * j], (uint32_t)v[4 * j + 1], (uint32_t)v[4 * j + 2]), (uint32_t)v[4 * j + 3]);
    const uint32_t m = __vimin3_s16x2(__vimin3_s16x2(g[0], g[1], g[2]), __vimin3_s16x2(g[3], g[4], g[5]), __vmins2(g[6], g[7]));
    if (min((int)(short)(m & 0xFFFF), (int)(short)(m >> 16)) <= thr) {
#pragma unroll
        for (int j = 0; j < 8; j++)
            if (min((int)(short)(g[j] & 0xFFFF), (int)(short)(g[j] >> 16)) <= thr)
                insert8((short)(v[4 * j] & 0xFFFF), (short)((uint32_t)v[4 * j] >> 16), (short)(v[4 * j + 1] & 0xFFFF),
                        (short)((uint32_t)v[4 * j + 1] >> 16), (short)(v[4 * j + 2] & 0xFFFF), (short)((uint32_t)v[4 * j + 2] >> 16),
                        (short)(v[4 * j + 3] & 0xFFFF), (short)((uint32_t)v[4 * j + 3] >> 16), idx0 + 8 * j, chunk_n, k0, k1, thr);
    }
}

// kBStages database tiles in flight: 2 when the producer warps unpack them, 3 when they arrive ready-made by bulk copies (whose
// latency is longer than the microsecond a tile lasts)
template <int kBStages>
struct TcSmemT {
    uint8_t a[kGroupTiles][kATileBytes];  // query tiles of the group
    uint8_t b[kBStages][kBTileBytes];     // database tiles
    uint64_t b_full[kBStages], b_empty[kBStages], d_full[kGroupTiles], d_empty[kGroupTiles];  // one hand-off per accumulator
    uint32_t tmem_base;
};
constexpr int kBulkStages = 3;

// 1-D bulk copy global -> shared memory, completion in bytes on an mbarrier (TMA engine, no tensor map)
__device__ __forceinline__ void bulk_load(void *dst, const void *src, uint32_t bytes, uint64_t *bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(smem_u32(dst)), "l"(src),
                 "r"(bytes), "r"(smem_u32(bar))
                 : "memory");
}

}  // namespace

// part[(chunk * q + query) * 2 + r] = r-th smallest (distance << 32 | global row) of the chunk, ~0 when there is none
// kBulk: `db` holds the rows already unpacked, one 32 KB operand tile per 128 rows (knn2_unpack_tiles_kernel): a database
// tile is one bulk copy issued by one thread instead of 2048 unpack + store steps of the producer warps.
template <bool kBulk>
__global__ void __launch_bounds__(kTcThreads, 1)
knn2_tc_kernel(const uint8_t *__restrict__ db, long long rows, long long idx_base, int chunk_rows, int chunks, const uint8_t *__restrict__ queries,
               int q, unsigned long long *__restrict__ part_out) {
    constexpr int kBStages = kBulk ? kBulkStages : 2;
    extern __shared__ __align__(128) uint8_t tc_smem_raw[];
    TcSmemT<kBStages> &S = *(TcSmemT<kBStages> *)tc_smem_raw;
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int groups = (q + kGroupQ - 1) / kGroupQ;
    if (warp == 0) {  // TMEM: all 512 columns (one CTA per SM: the shared memory footprint sees to that)
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(&S.tmem_base)), "r"(512u) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    if (tid == 64) {
        for (int i = 0; i < kBStages; i++) {
            mbar_init(&S.b_full[i], kBulk ? 1 : kProdWarps);  // one arrival per producer warp / the expect_tx of the bulk copy
            mbar_init(&S.b_empty[i], 2);  // tcgen05.commit of either MMA issuer
        }
        for (int i = 0; i < kGroupTiles; i++) {
            mbar_init(&S.d_full[i], 1);   // tcgen05.commit
            mbar_init(&S.d_empty[i], kEpiWarps / kGroupTiles);  // one arrival per epilogue warp of the accumulator
        }
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem = S.tmem_base;
    uint32_t tb = 0;  // database tiles this thread's role has gone through so far: tile tb uses buffer tb % kBStages in phase
                      // tb / kBStages, and every accumulator hand-off is in phase tb & 1

    for (int item = blockIdx.x; item < groups * chunks; item += gridDim.x) {
        const int g = item / chunks, chunk = item % chunks;
        const long long r0 = (long long)chunk * chunk_rows, r1 = min(r0 + (long long)chunk_rows, rows);
        const int q0 = g * kGroupQ, ntiles = r1 > r0 ? (int)((r1 - r0 + kTileN - 1) / kTileN) : 0;
        // ---- A tiles: the group's queries as +1 / -1, unpacked by every thread (rows past q are ignored later) -----------
        __syncthreads();  // the previous item's MMAs no longer read the A tiles (its epilogue has drained every accumulator)
        for (int u = tid; u < kGroupQ * 16; u += kTcThreads) {
            const int row = u >> 4, chunk16 = u & 15, qi = q0 + row;
            const uint32_t bits = qi < q ? __ldg((const uint16_t *)(queries + (size_t)qi * 32) + chunk16) : 0u;
            *(uint4 *)(S.a[row >> 7] + tile_off(row & 127, chunk16)) = unpack16_pm(bits);
        }
        fence_async_smem();
        __syncthreads();

        if (warp <= 1) {
            // ===== MMA issuers: warp h feeds TMEM stage h (query tiles kTilesPerStage h ..), so the wait -> issue -> commit chains
            // of the two stages run side by side ==========================================================================
            const int h = warp;  // accumulators 2 h and 2 h + 1: columns [256 h, 256 h + 256)
            for (int n = 0; n < ntiles; n++, tb++) {
                const int bi = (int)(tb % kBStages);
                mbar_wait(&S.b_full[bi], (tb / kBStages) & 1);
                const uint32_t b_addr = smem_u32(S.b[bi]);
                for (int t = 0; t < 2; t++) {  // each accumulator is handed over on its own: its warps start after 8 MMAs, not 16
                    const int acc = 2 * h + t;
                    mbar_wait(&S.d_empty[acc], (tb & 1) ^ 1);  // first use passes: the barrier starts in phase 0
                    tc_fence_after();
                    if (lane == 0) {
                        const uint32_t a_addr = smem_u32(S.a[acc]), d = tmem + (uint32_t)(128 * acc);
#pragma unroll
                        for (int k = 0; k < 8; k++)  // K = 32 per instruction: two 16-byte chunks
                            mma_i8(d, smem_desc(a_addr + k * 2 * kLBO), smem_desc(b_addr + k * 2 * kLBO), k > 0);
                        tc_commit(&S.d_full[acc]);
                    }
                    __syncwarp();
                }
                if (lane == 0) tc_commit(&S.b_empty[bi]);
                __syncwarp();
            }
        } else if (warp < 2 + kProdWarps) {
            // ===== producers: database rows -> B tile ================================================================
            const int pw = warp - 2, pt = pw * 32 + lane;  // producer thread
            // thread = kPasses (row, chunk) cells of a tile, one 16-byte store each, which a warp lays down as 8 rows x 4 chunks =
            // 512 contiguous bytes.  The descriptor bits of the NEXT tile are fetched before this one is written, so the global
            // latency never sits between "buffer free" and "buffer full".
            constexpr int kPasses = kTileN * 16 / (kProdWarps * 32);  // 16-byte stores per producer thread and tile
            uint32_t bits[kPasses];
            auto fetch = [&](int n) {
                const long long t0 = r0 + (long long)n * kTileN;
#pragma unroll
                for (int pass = 0; pass < kPasses; pass++) {
                    const int row = (pt & 7) + 8 * ((pt >> 5) + kProdWarps * (pass >> 2)), chunk16 = ((pt >> 3) & 3) + 4 * (pass & 3);
                    const long long gr = t0 + row;
                    bits[pass] = gr < r1 ? __ldg((const uint16_t *)(db + (size_t)gr * 32) + chunk16) : 0u;
                }
            };
            if (kBulk) {
                // the tiles are ready-made in global memory: one elected thread keeps kBStages bulk copies in flight
                if (pw == 0 && lane == 0) {
                    const uint8_t *src = db + (size_t)(r0 / kTileN) * kBTileBytes;
                    for (int n = 0; n < ntiles; n++, tb++) {
                        const int bi = (int)(tb % kBStages);
                        mbar_wait(&S.b_empty[bi], ((tb / kBStages) & 1) ^ 1);
                        mbar_expect_tx(&S.b_full[bi], kBTileBytes);
                        bulk_load(S.b[bi], src + (size_t)n * kBTileBytes, kBTileBytes, &S.b_full[bi]);
                    }
                }
            } else {
            if (kPrefetchB && ntiles > 0) fetch(0);
            for (int n = 0; n < ntiles; n++, tb++) {
                const int bi = (int)(tb % kBStages);
                mbar_wait(&S.b_empty[bi], ((tb / kBStages) & 1) ^ 1);
                if (!kPrefetchB) fetch(n);
#pragma unroll
                for (int pass = 0; pass < kPasses; pass++) {
                    const int row = (pt & 7) + 8 * ((pt >> 5) + kProdWarps * (pass >> 2)), chunk16 = ((pt >> 3) & 3) + 4 * (pass & 3);
                    *(uint4 *)(S.b[bi] + tile_off(row, chunk16)) = unpack16(bits[pass]);
                }
                fence_async_smem();
                __syncwarp();
                if (lane == 0) mbar_arrive(&S.b_full[bi]);
                if (kPrefetchB && n + 1 < ntiles) fetch(n + 1);
            }
            }
        } else {
            // ===== epilogue: TMEM -> keys -> running top-2 per query ====================================================
            const int ew = warp - 2 - kProdWarps, quad = warp & 3;  // a warp reads the TMEM lanes of quadrant warp % 4
            const int tile = ew >> 2;                   // the query tile = accumulator this warp serves (4 warps each: one per quadrant)
            const int row = quad * 32 + lane;           // query row inside the tile
            uint32_t k0 = kNoKey32, k1 = kNoKey32;
            int thr = (int)(kNoKey32 >> 22) - kKeyOffset;
            const uint32_t chunk_n = (uint32_t)(r1 - r0);
            const uint32_t lane_addr = tmem + ((uint32_t)(quad * 32) << 16) + (uint32_t)(128 * tile);
            for (int n = 0; n < ntiles; n++, tb++) {
                const uint32_t idx0 = (uint32_t)n * kTileN;
                mbar_wait(&S.d_full[tile], tb & 1);
                tc_fence_after();
                // 128 columns as two packed loads of 64, both in flight: the accumulator goes back to its issuer one load latency
                // after the commit
                int buf[2][32];
                tmem_ld64p_issue(lane_addr, buf[0]);
                tmem_ld64p_issue(lane_addr + 64u, buf[1]);
                tmem_ld_wait2(buf[0], buf[1]);
                tc_fence_before();
                __syncwarp();
                if (lane == 0) mbar_arrive(&S.d_empty[tile]);
                examine64p(buf[0], k0, k1, thr, idx0, chunk_n);
                examine64p(buf[1], k0, k1, thr, idx0 + 64, chunk_n);
            }
            {
                const int qi = q0 + tile * 128 + row;
                if (qi < q) {
                    const uint4 *p = (const uint4 *)(queries + (size_t)qi * 32);
                    const uint4 u = __ldg(p), w = __ldg(p + 1);
                    const int pa = __popc(u.x) + __popc(u.y) + __popc(u.z) + __popc(u.w) + __popc(w.x) + __popc(w.y) + __popc(w.z) + __popc(w.w);
                    unsigned long long o[2];
                    const uint32_t kk[2] = {k0, k1};
#pragma unroll
                    for (int r = 0; r < 2; r++) {
                        if (kk[r] == kNoKey32) { o[r] = ~0ull; continue; }
                        const unsigned long long dist = (unsigned long long)((int)(kk[r] >> 22) - kKeyOffset + pa);  // D' + |a|
                        o[r] = dist << 32 | (unsigned long long)(idx_base + r0 + (long long)(kk[r] & 0x3FFFFFu));
                    }
                    unsigned long long *dst = part_out + ((size_t)chunk * q + qi) * 2;
                    dst[0] = o[0];
                    dst[1] = o[1];
                }
            }
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 0) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem), "r"(512u) : "memory");
}

// Database rows -> ready-made operand tiles: tile t = rows 128 t .. 128 t + 127 as int8 {0, 1} in the K-major core-matrix layout
// the MMA reads (32 KB per tile, 256 B per row: 8 x the packed map; rows past the end are zeros, which the epilogue never keys).
__global__ void __launch_bounds__(256) knn2_unpack_tiles_kernel(const uint8_t *__restrict__ db, long long rows, long long first_tile,
                                                                uint8_t *__restrict__ tiles) {
    const long long t = first_tile + blockIdx.x;
    const long long t0 = t * kTileN;
    uint8_t *dst = tiles + (size_t)t * kBTileBytes;
    for (int u = threadIdx.x; u < kTileN * 16; u += 256) {
        const int row = u >> 4, chunk16 = u & 15;
        const long long gr = t0 + row;
        const uint32_t bits = gr < rows ? __ldg((const uint16_t *)(db + (size_t)gr * 32) + chunk16) : 0u;
        *(uint4 *)(dst + tile_off(row, chunk16)) = unpack16(bits);
    }
}

size_t knn2_tc_smem_bytes() { return sizeof(TcSmemT<2>) + 128; }
int knn2_tc_group_queries() { return kGroupQ; }  // queries per work item: the caller sizes its chunks with it
size_t knn2_tc_tiles_bytes(long long rows) { return (size_t)((rows + kTileN - 1) / kTileN) * kBTileBytes; }

// (re)writes tiles first_tile .. the one holding row rows - 1: 0 for a full build; an append into spare capacity starts at the
// tile of its first new row, whose zero padding becomes real rows
cudaError_t launch_knn2_unpack_tiles(cudaStream_t st, const uint8_t *db, long long rows, long long first_tile, uint8_t *tiles) {
    const long long n = (rows + kTileN - 1) / kTileN - first_tile;
    if (n > 0) knn2_unpack_tiles_kernel<<<(unsigned)n, 256, 0, st>>>(db, rows, first_tile, tiles);
    return cudaGetLastError();
}

// chunks x q x 2 keys into `part`; chunk_rows must be a multiple of 128 and at most 2^22.  tiles != nullptr: the map's
// ready-made operand tiles (launch_knn2_unpack_tiles), fetched by bulk copies instead of being unpacked by the producer warps.
cudaError_t launch_knn2_tc(cudaStream_t st, int sm_count, const uint8_t *db, const uint8_t *tiles, long long rows, long long idx_base,
                           int chunk_rows, int chunks, const uint8_t *queries, int q, unsigned long long *part) {
    static std::once_flag once[64];  // matchers of one device may search from several threads at once
    static cudaError_t configured[64];
    int dev = 0;
    cudaGetDevice(&dev);
    const size_t smem = knn2_tc_smem_bytes(), smem_bulk = sizeof(TcSmemT<kBulkStages>) + 128;
    std::call_once(once[dev & 63], [&] {
        cudaError_t e = cudaFuncSetAttribute(knn2_tc_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (e == cudaSuccess) e = cudaFuncSetAttribute(knn2_tc_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_bulk);
        configured[dev & 63] = e;
    });
    if (configured[dev & 63] != cudaSuccess) return configured[dev & 63];
    const int groups = (q + kGroupQ - 1) / kGroupQ;
    const int grid = std::min(sm_count, groups * chunks);
    if (tiles)
        knn2_tc_kernel<true><<<grid, kTcThreads, smem_bulk, st>>>(tiles, rows, idx_base, chunk_rows, chunks, queries, q, part);
    else
        knn2_tc_kernel<false><<<grid, kTcThreads, smem, st>>>(db, rows, idx_base, chunk_rows, chunks, queries, q, part);
    return cudaGetLastError();
}

}  // namespace sfe
