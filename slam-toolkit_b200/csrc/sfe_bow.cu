// BoW database scoring kernels: DBoW2's L1 query (TemplatedDatabase::queryL1, L1Scoring::score), bit for bit; the
// validation of vectors that arrive in device memory; BowVector assembly on the device.
//
// Every score is a double sum of fabs(q - d) - fabs(q) - fabs(d) over the words a query and an entry share, taken in
// ascending word order.  The kernels therefore never reduce as a tree: the lanes of a warp find the common words in
// parallel, and one ordered chain of additions per (query, entry) pair consumes them in word order.
#include <algorithm>
#include <cstdint>
#include <mutex>

#include "sfe_common.cuh"

namespace sfe {

constexpr int kBowWarps = 8;                 // warps per CTA of the scoring kernel
constexpr int kBowEntriesPerCta = 256;       // entries one scoring CTA walks (32 per warp): the staged query is reused
constexpr int kBowSmemWords = 4096;          // queries up to this many words are staged in shared memory (48 KB)
constexpr int kBowTopkThreads = 1024;        // = SFE_BOWDB_MAX_RESULTS: the selected results are sorted in one CTA

// Forward file of the database / of a batch of queries: vector i = ids / values [off[i], off[i+1]).
struct BowCsr {
    const int64_t *off;
    const int32_t *ids;
    const double *val;
};

// raw[qi*stride + e] = the ordered L1 sum of query qi against entry e (0.0 when they share no word), hit[..] = 1 when they
// share one; dense (optional) = -raw / 2.0, L1Scoring::score.  Grid (entry blocks, queries); warp w of a CTA takes entries
// blockIdx.x * 256 + w, + 8, ...
template <bool kStaged>
__global__ void __launch_bounds__(kBowWarps * 32) bow_score_kernel(BowCsr Q, BowCsr D, int stage_cap, int n_entries, long long stride,
                                                                  double *__restrict__ raw, uint8_t *__restrict__ hit,
                                                                  double *__restrict__ dense) {
    extern __shared__ __align__(16) unsigned char bow_smem[];
    const int qi = blockIdx.y;
    const int64_t q0 = Q.off[qi];
    const int nq = (int)(Q.off[qi + 1] - q0);
    const int32_t *qid = Q.ids + q0;
    const double *qval = Q.val + q0;
    if (kStaged) {
        double *sv = (double *)bow_smem;
        int32_t *si = (int32_t *)(sv + stage_cap);
        for (int i = threadIdx.x; i < nq; i += blockDim.x) {
            si[i] = qid[i];
            sv[i] = qval[i];
        }
        qid = si;
        qval = sv;
        __syncthreads();
    }
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int e_end = min(n_entries, (blockIdx.x + 1) * kBowEntriesPerCta);
    for (int e = blockIdx.x * kBowEntriesPerCta + warp; e < e_end; e += kBowWarps) {
        const int64_t b = D.off[e];
        const int64_t ne = D.off[e + 1] - b;
        double acc = 0.0;
        bool any = false;
        int lo = 0;  // the query words below `lo` are smaller than every entry word still to come
        for (int64_t base = 0; base < ne && lo < nq; base += 32) {
            const int64_t j = base + lane;
            const bool valid = j < ne;
            const int w = valid ? __ldg(D.ids + b + j) : 0x7FFFFFFF;
            int l = lo, h = nq;  // lower_bound of w in qid[lo, nq)
            while (l < h) {
                const int mid = (l + h) >> 1;
                if (qid[mid] < w) l = mid + 1; else h = mid;
            }
            const bool found = valid && l < nq && qid[l] == w;
            double v = 0.0;
            if (found) {
                const double qv = qval[l], d = __ldg(D.val + b + j);
                v = __dsub_rn(__dsub_rn(fabs(__dsub_rn(qv, d)), fabs(qv)), fabs(d));
            }
            unsigned m = __ballot_sync(0xFFFFFFFFu, found);
            any |= m != 0;
            while (m) {  // lane order = ascending word order: the additions stay in DBoW2's sequence
                const double x = __shfl_sync(0xFFFFFFFFu, v, __ffs(m) - 1);
                acc = __dadd_rn(acc, x);
                m &= m - 1;
            }
            lo = __shfl_sync(0xFFFFFFFFu, l, 31);
        }
        if (lane == 0) {
            const size_t o = (size_t)qi * stride + e;
            raw[o] = acc;
            hit[o] = any ? 1 : 0;
            if (dense) dense[o] = -acc / 2.0;
        }
    }
}

// Total order of doubles as unsigned integers (+0.0 and -0.0 are made equal first, as the reference's < sees them).
__device__ __forceinline__ unsigned long long bow_key(double x) {
    const long long b = __double_as_longlong(x == 0.0 ? 0.0 : x);
    return b < 0 ? ~(unsigned long long)b : (unsigned long long)b | 0x8000000000000000ull;
}
__device__ __forceinline__ double bow_unkey(unsigned long long k) {
    return __longlong_as_double((long long)((k & 0x8000000000000000ull) ? (k & 0x7FFFFFFFFFFFFFFFull) : ~k));
}

// Block-wide sum of one int per thread (kBowTopkThreads threads); every thread gets the total.
__device__ __forceinline__ int bow_block_sum(int v, int *red) {
    for (int o = 16; o; o >>= 1) v += __shfl_xor_sync(0xFFFFFFFFu, v, o);
    __syncthreads();
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = v;
    __syncthreads();
    int t = 0;
    for (int i = 0; i < kBowTopkThreads / 32; i++) t += red[i];
    return t;
}

// Per query (one CTA): the k results of queryL1 among the entries e < n with hit[e] -- ascending (raw sum, entry id), which
// is DBoW2's order with T8 -- as entry ids and scores -raw / 2.0.  With more than k candidates the k-th smallest sum is
// found by an MSB radix select over the 64-bit keys (8 passes of 8 bits); the entries below it are all taken and the
// entries equal to it in ascending id until k are reached.  The at most k chosen pairs are then bitonic-sorted.
__global__ void __launch_bounds__(kBowTopkThreads) bow_topk_kernel(const double *__restrict__ raw, const uint8_t *__restrict__ hit,
                                                                  long long stride, int n, int k, int32_t *__restrict__ out_e,
                                                                  double *__restrict__ out_s, int32_t *__restrict__ out_n) {
    __shared__ unsigned long long skey[kBowTopkThreads];
    __shared__ int sidx[kBowTopkThreads];
    __shared__ int hist[256];
    __shared__ int red[kBowTopkThreads / 32];
    __shared__ unsigned long long s_prefix;
    __shared__ int s_rem, s_fill;
    const int qi = blockIdx.x, t = threadIdx.x;
    raw += (size_t)qi * stride;
    hit += (size_t)qi * stride;
    int c = 0;
    for (int e = t; e < n; e += kBowTopkThreads) c += hit[e];
    c = bow_block_sum(c, red);
    unsigned long long T = ~0ull;  // take every key <= T ...
    int ties = 0x7FFFFFFF;         // ... but at most this many keys == T, in ascending entry order
    if (c > k) {
        unsigned long long prefix = 0, mask = 0;
        int rem = k;  // rank of the wanted key among those matching `prefix`
        for (int shift = 56; shift >= 0; shift -= 8) {
            if (t < 256) hist[t] = 0;
            __syncthreads();
            for (int e = t; e < n; e += kBowTopkThreads) {
                if (!hit[e]) continue;
                const unsigned long long key = bow_key(raw[e]);
                if ((key & mask) == prefix) atomicAdd(&hist[(key >> shift) & 255], 1);
            }
            __syncthreads();
            if (t == 0) {
                int cum = 0, bin = 0;
                while (cum + hist[bin] < rem) cum += hist[bin++];
                s_rem = rem - cum;
                s_prefix = prefix | ((unsigned long long)bin << shift);
            }
            __syncthreads();
            rem = s_rem;
            prefix = s_prefix;
            mask |= 255ull << shift;
        }
        T = prefix;
        ties = rem;
    }
    // strictly below T: unordered slots; T itself (or, when c <= k, nothing: every hit is below ~0) in entry order
    if (t == 0) s_fill = 0;
    __syncthreads();
    for (int e = t; e < n; e += kBowTopkThreads) {
        if (!hit[e]) continue;
        const unsigned long long key = bow_key(raw[e]);
        if (key < T || (c <= k)) {
            const int s = atomicAdd(&s_fill, 1);
            skey[s] = key;
            sidx[s] = e;
        }
    }
    __syncthreads();
    const int below = s_fill;
    if (c > k) {
        int taken = 0;
        for (int base = 0; base < n && taken < ties; base += kBowTopkThreads) {  // uniform: taken is block-wide
            const int e = base + t;
            const bool tie = e < n && hit[e] && bow_key(raw[e]) == T;
            const unsigned bal = __ballot_sync(0xFFFFFFFFu, tie);
            __syncthreads();
            if ((t & 31) == 0) red[t >> 5] = __popc(bal);
            __syncthreads();
            int before = 0, total = 0;
            for (int i = 0; i < kBowTopkThreads / 32; i++) {
                if (i < (t >> 5)) before += red[i];
                total += red[i];
            }
            const int pos = taken + before + __popc(bal & ((1u << (t & 31)) - 1));
            if (tie && pos < ties) {
                skey[below + pos] = T;
                sidx[below + pos] = e;
            }
            taken += total;
        }
    }
    const int cnt = c > k ? k : c;
    int P = 1;
    while (P < cnt) P <<= 1;
    for (int s = cnt + t; s < P; s += kBowTopkThreads) {
        skey[s] = ~0ull;
        sidx[s] = 0x7FFFFFFF;
    }
    __syncthreads();
    for (int size = 2; size <= P; size <<= 1) {
        for (int stride2 = size >> 1; stride2 > 0; stride2 >>= 1) {
            const int i = t, j = t ^ stride2;
            if (i < P && j > i) {
                const bool up = (i & size) == 0;
                const unsigned long long ki = skey[i], kj = skey[j];
                const int ii = sidx[i], ij = sidx[j];
                const bool gt = ki > kj || (ki == kj && ii > ij);
                if (gt == up) {
                    skey[i] = kj; skey[j] = ki;
                    sidx[i] = ij; sidx[j] = ii;
                }
            }
            __syncthreads();
        }
    }
    for (int s = t; s < k; s += kBowTopkThreads) {
        const bool ok = s < cnt;
        out_e[(size_t)qi * k + s] = ok ? sidx[s] : -1;
        out_s[(size_t)qi * k + s] = ok ? -bow_unkey(skey[s]) / 2.0 : 0.0;
    }
    if (t == 0) out_n[qi] = cnt;
}

// Scores queries [0, q) of Q against entries [0, n_entries) of D into rows of `stride` (see bow_score_kernel).
cudaError_t launch_bow_score(cudaStream_t st, const int64_t *q_off, const int32_t *q_ids, const double *q_val, int q, int max_nq,
                             const int64_t *d_off, const int32_t *d_ids, const double *d_val, int n_entries, long long stride,
                             double *raw, uint8_t *hit, double *dense) {
    if (q == 0 || n_entries == 0) return cudaSuccess;
    const BowCsr Q{q_off, q_ids, q_val}, D{d_off, d_ids, d_val};
    const dim3 grid((n_entries + kBowEntriesPerCta - 1) / kBowEntriesPerCta, q);
    const int stage_cap = (max_nq + 31) / 32 * 32;  // sized to the longest query: short queries leave room for more CTAs
    if (stage_cap <= kBowSmemWords)
        bow_score_kernel<true><<<grid, kBowWarps * 32, (size_t)stage_cap * 12, st>>>(Q, D, stage_cap, n_entries, stride, raw, hit, dense);
    else
        bow_score_kernel<false><<<grid, kBowWarps * 32, 0, st>>>(Q, D, 0, n_entries, stride, raw, hit, dense);
    return cudaGetLastError();
}

cudaError_t launch_bow_topk(cudaStream_t st, const double *raw, const uint8_t *hit, long long stride, int q, int n, int k,
                            int32_t *out_e, double *out_s, int32_t *out_n) {
    if (q == 0) return cudaSuccess;
    bow_topk_kernel<<<q, kBowTopkThreads, 0, st>>>(raw, hit, stride, n, k, out_e, out_s, out_n);
    return cudaGetLastError();
}

// ---- vectors from device memory: validation and rebasing ---------------------------------------------------------------

// chk[0] = nnz (offsets[count]), chk[1] != 0 when a rule is broken, chk[2] = the longest vector.  The rules are the host
// check's: offsets[0] == 0 and never decreasing, ids in [0, n_words) and strictly ascending within a vector, values finite.
// One warp per vector; every read stays inside [0, offsets[count]), the extent the CSR itself declares, so inconsistent
// offsets are reported rather than followed.  Null ids / values skip the content checks (the host rejects them when nnz > 0).
__global__ void __launch_bounds__(256) bow_check_kernel(const int64_t *__restrict__ off, const int32_t *__restrict__ ids,
                                                        const double *__restrict__ val, int count, int n_words,
                                                        unsigned long long *__restrict__ chk) {
    const int64_t end = off[count];
    const int lane = threadIdx.x & 31;
    const int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, n_warps = (gridDim.x * blockDim.x) >> 5;
    if (warp == 0 && lane == 0) {
        chk[0] = (unsigned long long)end;
        if (off[0] != 0) atomicOr(&chk[1], 1ull);
    }
    for (int i = warp; i < count; i += n_warps) {
        const int64_t lo = off[i], hi = off[i + 1];
        bool bad = hi < lo;
        if (!bad && ids && val) {
            const int64_t a = lo > 0 ? lo : 0, b = hi < end ? hi : end;
            for (int64_t j = a + lane; j < b; j += 32) {
                const int32_t w = ids[j];
                bad |= w < 0 || w >= n_words || (j > a && w <= ids[j - 1]) || !isfinite(val[j]);
            }
        }
        bad = __any_sync(0xFFFFFFFFu, bad);
        if (lane == 0) {
            if (bad) atomicOr(&chk[1], 1ull);
            else atomicMax(&chk[2], (unsigned long long)(hi - lo));
        }
    }
}

__global__ void bow_rebase_kernel(const int64_t *__restrict__ src, int count, int64_t base, int64_t *__restrict__ dst) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < count) dst[i] = base + src[i + 1];
}

cudaError_t launch_bow_check(cudaStream_t st, const int64_t *off, const int32_t *ids, const double *val, int count, int n_words,
                             unsigned long long *chk) {
    cudaError_t e = cudaMemsetAsync(chk, 0, sizeof(unsigned long long) * 3, st);
    if (e != cudaSuccess) return e;
    const int blocks = std::max(1, std::min((count + 7) / 8, 4096));
    bow_check_kernel<<<blocks, 256, 0, st>>>(off, ids, val, count, n_words, chk);
    return cudaGetLastError();
}

// dst[i] = base + src[i + 1], i < count: a batch's end offsets moved into a forward file that already holds `base` words
cudaError_t launch_bow_rebase(cudaStream_t st, const int64_t *src, int count, int64_t base, int64_t *dst) {
    if (count == 0) return cudaSuccess;
    bow_rebase_kernel<<<(count + 255) / 256, 256, 0, st>>>(src, count, base, dst);
    return cudaGetLastError();
}

// ---- BowVector assembly (TemplatedVocabulary::transform's BowVector half, BowVector.cpp:34-84) ---------------------------
//
// The host sfe_bow_assemble's order of operations, one CTA per feature set: the accepted features (weight > 0, so NaN is
// skipped) become keys (word id with the sign bit flipped << 32 | feature index), which a bitonic sort puts in ascending
// signed word order with each word's features in feature order -- the order std::map insertion sees them.  The first key
// of each run owns the word: TF_IDF / TF (addWeight) add the run's weights serially in that order, IDF / BINARY
// (addIfNotExist) keep the first.  The norm is one chain of additions in word order, on one warp.

constexpr int kBowAsmThreads = 1024;

__device__ __forceinline__ int32_t bow_asm_word(unsigned long long key) { return (int32_t)((uint32_t)(key >> 32) ^ 0x80000000u); }

// Set i = rows [i*stride, i*stride + n[i]) of word_id / weight.  Its BowVector goes to rows [i*stride, + cnt[i]) of
// out_ids / out_val, each value still to be divided by div_out[i] when that is > 0.0.  A count outside [0, stride] sets
// *status and leaves the set empty.  (The division sits in the compaction: its slow path makes this kernel spill.)
__global__ void __launch_bounds__(kBowAsmThreads) bow_assemble_kernel(const int32_t *__restrict__ word_id,
                                                                      const double *__restrict__ weight,
                                                                      const int32_t *__restrict__ n_set, int stride, int weighting,
                                                                      int norm, int32_t *__restrict__ cnt,
                                                                      double *__restrict__ div_out, int32_t *out_ids, double *out_val,
                                                                      unsigned long long *__restrict__ status) {
    extern __shared__ __align__(16) unsigned char bow_asm_smem[];
    unsigned long long *key = (unsigned long long *)bow_asm_smem;
    __shared__ int wsum[kBowAsmThreads / 32];
    __shared__ double s_norm;
    const int set = blockIdx.x, t = threadIdx.x, lane = t & 31, warp = t >> 5;
    const int n = n_set[set];
    if (n < 0 || n > stride) {  // uniform
        if (t == 0) {
            atomicOr(status, 1ull);
            cnt[set] = 0;
            div_out[set] = 0.0;
        }
        return;
    }
    const size_t row0 = (size_t)set * stride;
    word_id += row0;
    weight += row0;
    out_ids += row0;
    out_val += row0;
    int P = 1;
    while (P < n) P <<= 1;
    int c = 0;  // accepted features
    for (int f0 = 0; f0 < P; f0 += kBowAsmThreads) {
        const int f = f0 + t;
        bool ok = false;
        if (f < P) {
            ok = f < n && weight[f] > 0.0;
            key[f] = ok ? ((unsigned long long)((uint32_t)word_id[f] ^ 0x80000000u) << 32) | (unsigned)f : ~0ull;
        }
        c += __syncthreads_count(ok);
    }
    for (int size = 2; size <= P; size <<= 1) {
        for (int j = size >> 1; j > 0; j >>= 1) {
            for (int x = t; x < P / 2; x += kBowAsmThreads) {
                const int lo = (x / j) * 2 * j + (x & (j - 1)), hi = lo + j;
                const unsigned long long a = key[lo], b = key[hi];
                if ((a > b) == ((lo & size) == 0)) {
                    key[lo] = b;
                    key[hi] = a;
                }
            }
            __syncthreads();
        }
    }
    const bool accumulate = weighting == 0 || weighting == 1;
    int u = 0;  // words so far
    for (int p0 = 0; p0 < c; p0 += kBowAsmThreads) {  // uniform
        const int p = p0 + t;
        const bool head = p < c && (p == 0 || (key[p] >> 32) != (key[p - 1] >> 32));
        const unsigned bal = __ballot_sync(0xFFFFFFFFu, head);
        if (lane == 0) wsum[warp] = __popc(bal);
        __syncthreads();
        int before = 0, total = 0;
        for (int w = 0; w < kBowAsmThreads / 32; w++) {
            if (w < warp) before += wsum[w];
            total += wsum[w];
        }
        if (head) {
            const unsigned long long k0 = key[p];
            double v = weight[(uint32_t)k0];
            if (accumulate)
                for (int q = p + 1; q < c && (key[q] >> 32) == (k0 >> 32); q++) v = __dadd_rn(v, weight[(uint32_t)key[q]]);
            const int r = u + before + __popc(bal & ((1u << lane) - 1));
            out_ids[r] = bow_asm_word(k0);
            out_val[r] = v;
        }
        u += total;
        __syncthreads();  // wsum is rewritten by the next chunk
    }
    // every value is then divided (by bow_compact_kernel) by the word count -- TF_IDF / TF without a norm: "unnecessary when
    // normalizing" -- or by the norm when it is > 0.0; never both
    double div = accumulate && norm == 0 ? (double)u : 0.0;
    if (norm != 0) {
        if (warp == 0) {  // one serial chain in word order: the lanes fetch 32 terms, the additions consume them in lane order
            double s = 0.0;
            for (int r0 = 0; r0 < u; r0 += 32) {
                const int r = r0 + lane;
                double x = 0.0;
                if (r < u) {
                    const double v = out_val[r];
                    x = norm == 1 ? fabs(v) : __dmul_rn(v, v);
                }
                const int m = min(32, u - r0);
                for (int l = 0; l < m; l++) s = __dadd_rn(s, __shfl_sync(0xFFFFFFFFu, x, l));
            }
            if (lane == 0) s_norm = norm == 2 ? __dsqrt_rn(s) : s;
        }
        __syncthreads();
        div = s_norm;
    }
    if (t == 0) {
        cnt[set] = u;
        div_out[set] = div;
    }
}

// off[0] = 0, off[i + 1] = off[i] + cnt[i]: one CTA, a block-wide scan per chunk of kBowAsmThreads sets
__global__ void __launch_bounds__(kBowAsmThreads) bow_offsets_kernel(const int32_t *__restrict__ cnt, int count,
                                                                     int64_t *__restrict__ off) {
    __shared__ long long wsum[kBowAsmThreads / 32];
    const int t = threadIdx.x, lane = t & 31, warp = t >> 5;
    long long base = 0;
    if (t == 0) off[0] = 0;
    for (int i0 = 0; i0 < count; i0 += kBowAsmThreads) {
        const int i = i0 + t;
        long long v = i < count ? cnt[i] : 0;
        for (int o = 1; o < 32; o <<= 1) {  // inclusive warp scan
            const long long y = __shfl_up_sync(0xFFFFFFFFu, v, o);
            if (lane >= o) v += y;
        }
        if (lane == 31) wsum[warp] = v;
        __syncthreads();
        long long before = 0, total = 0;
        for (int w = 0; w < kBowAsmThreads / 32; w++) {
            if (w < warp) before += wsum[w];
            total += wsum[w];
        }
        if (i < count) off[i + 1] = base + before + v;
        base += total;
        __syncthreads();
    }
}

// rows [set*stride, + cnt[set]) of the strided vectors -> [off[set], off[set + 1]) of the compact CSR, values divided by
// div[set] when that is > 0.0
__global__ void __launch_bounds__(256) bow_compact_kernel(const int32_t *__restrict__ cnt, const double *__restrict__ div,
                                                          const int64_t *__restrict__ off, int stride,
                                                          const int32_t *__restrict__ src_ids, const double *__restrict__ src_val,
                                                          int32_t *__restrict__ dst_ids, double *__restrict__ dst_val) {
    const int set = blockIdx.x;
    const int u = cnt[set];
    const double d = div[set];
    const size_t s0 = (size_t)set * stride;
    const int64_t d0 = off[set];
    for (int r = threadIdx.x; r < u; r += blockDim.x) {
        const double v = src_val[s0 + r];
        dst_ids[d0 + r] = src_ids[s0 + r];
        dst_val[d0 + r] = d > 0.0 ? __ddiv_rn(v, d) : v;
    }
}

// count sets of at most stride (<= SFE_BOW_ASSEMBLE_MAX_STRIDE) features -> compact CSR; cnt / div / tmp_ids / tmp_val:
// scratch of count, count, count * stride, count * stride elements.  *status is set when a set's feature count lies outside [0, stride].
cudaError_t launch_bow_assemble(cudaStream_t st, const int32_t *word_id, const double *weight, const int32_t *n_set, int count,
                                int stride, int weighting, int norm, int32_t *cnt, double *div, int32_t *tmp_ids, double *tmp_val,
                                unsigned long long *status, int64_t *off, int32_t *ids, double *val) {
    cudaError_t e = cudaMemsetAsync(status, 0, sizeof(unsigned long long), st);
    if (e != cudaSuccess) return e;
    if (count == 0) return cudaMemsetAsync(off, 0, sizeof(int64_t), st);
    // the opt-in limit belongs to the function on the device, shared by every matcher: set once per device, to what the
    // largest stride needs, so no call ever lowers it under another thread's launch
    static std::once_flag once[64];
    static cudaError_t configured[64];
    int dev = 0;
    e = cudaGetDevice(&dev);
    if (e != cudaSuccess) return e;
    std::call_once(once[dev & 63], [&] {
        configured[dev & 63] = cudaFuncSetAttribute(bow_assemble_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                                    (int)(sizeof(unsigned long long) * SFE_BOW_ASSEMBLE_MAX_STRIDE));
    });
    if (configured[dev & 63] != cudaSuccess) return configured[dev & 63];
    int P = 1;
    while (P < stride) P <<= 1;
    const size_t smem = sizeof(unsigned long long) * P;
    bow_assemble_kernel<<<count, kBowAsmThreads, smem, st>>>(word_id, weight, n_set, stride, weighting, norm, cnt, div, tmp_ids,
                                                             tmp_val, status);
    e = cudaGetLastError();  // the scan and the compaction read what the assembly wrote: never enqueue them behind a failure
    if (e != cudaSuccess) return e;
    bow_offsets_kernel<<<1, kBowAsmThreads, 0, st>>>(cnt, count, off);
    bow_compact_kernel<<<count, 256, 0, st>>>(cnt, div, off, stride, tmp_ids, tmp_val, ids, val);
    return cudaGetLastError();
}

}  // namespace sfe
