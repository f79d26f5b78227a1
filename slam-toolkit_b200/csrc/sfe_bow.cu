// BoW database scoring kernels: DBoW2's L1 query (TemplatedDatabase::queryL1, L1Scoring::score), bit for bit.
//
// Every score is a double sum of fabs(q - d) - fabs(q) - fabs(d) over the words a query and an entry share, taken in
// ascending word order.  The kernels therefore never reduce as a tree: the lanes of a warp find the common words in
// parallel, and one ordered chain of additions per (query, entry) pair consumes them in word order.
#include <cstdint>

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

}  // namespace sfe
