// Evaluation metrics on the device, sm_100a: full-sort metrics from a top-K index matrix and the by-user
// metrics of candidate score segments.  Replaces the host numpy step after `evaluate_full_sort` /
// `evaluate_by_user` (metrics.topk_metrics / metrics.by_user_metrics; FoodRec/utils/topk_evaluator.py:68-115,
// FoodRec/common/matrics.py:9-102, FoodRec/common/trainer.py:49-69,231-282).
//
// Both kernels are latency bound (a few dependent loads per row); each block folds its users' per-user values into
// fp64 partials and the last block to arrive (atomic ticket, reset by that block) folds the block partials in a
// fixed order, so the sums are bit-reproducible from run to run on a given device.
#include <algorithm>

#include "common.cuh"

namespace {

constexpr int kMaxCut = FR_EVAL_MAX_CUTOFFS;
constexpr int kTopkEntries = FR_TOPK_METRICS * kMaxCut + 1;   // [metric][cutoff] + sum of pos_len
constexpr int kUserEntries = 1 + 2 * kMaxCut;                   // AUC, recall[cutoff], ndcg[cutoff]
constexpr int kTopkWarps = 8;
constexpr int kUserThreads = 256;
constexpr int kStage = 4096;                                    // candidate scores staged in shared memory per user

struct Cutoffs {
    int c[kMaxCut];
    int n;
};

// Fixed-order fold of `part` ([E][grid] doubles) by one block: warp w owns entries w, w + nwarps, ...; lane l sums
// blocks l, l + 32, ... in order, then a fixed butterfly combines the lanes.
template <int kPerWarp>
__device__ void fold_partials(const double *__restrict__ part, int E, int grid, double *__restrict__ out) {
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5, nw = blockDim.x >> 5;
    double acc[kPerWarp];
#pragma unroll
    for (int q = 0; q < kPerWarp; ++q) acc[q] = 0.0;
#pragma unroll 2
    for (int b = lane; b < grid; b += 32) {
#pragma unroll
        for (int q = 0; q < kPerWarp; ++q) {
            const int e = w + q * nw;
            if (e < E) acc[q] += __ldcg(part + (size_t)e * grid + b);
        }
    }
#pragma unroll
    for (int q = 0; q < kPerWarp; ++q) {
        double v = acc[q];
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
        const int e = w + q * nw;
        if (lane == 0 && e < E) out[e] = v;
    }
}

// Ticket: true in the last block of the grid to finish (its partials and everyone else's are then visible).
__device__ __forceinline__ bool last_block(unsigned *ticket) {
    __shared__ int last;
    __threadfence();
    __syncthreads();
    if (threadIdx.x == 0) last = (atomicAdd(ticket, 1u) == gridDim.x - 1);
    __syncthreads();
    if (last) __threadfence();
    return last;
}

// Binary search in the sorted row a[lo, hi).
__device__ __forceinline__ bool contains(const int32_t *__restrict__ a, int64_t lo, int64_t hi, long long x) {
    if (x < 0 || x > 0x7fffffffLL) return false;
    const int v = (int)x;
    const int64_t end = hi;
    while (lo < hi) {
        const int64_t mid = (lo + hi) >> 1;
        if (__ldg(a + mid) < v) lo = mid + 1;
        else hi = mid;
    }
    return lo < end && __ldg(a + lo) == v;
}

template <typename IdxT>
__device__ __forceinline__ long long load_idx(const IdxT *p) {
    return (long long)__ldcs(p);
}

// One warp per row, grid-stride over rows.  Lane l tests columns l and l + 32; two ballots give the row's 64-bit
// hit mask.  Lane i < n_cut then walks the hits below cutoff i in rank order with the host's dtypes and summation
// order (module comment of metrics.topk_metrics_device) and keeps the running per-cutoff sums.
template <typename IdxT>
__global__ void __launch_bounds__(kTopkWarps * 32, 4)
topk_metrics_kernel(const IdxT *__restrict__ top, long long n, int K, const int64_t *__restrict__ pos_ptr,
                    const int32_t *__restrict__ pos_idx, const int32_t *__restrict__ pos_len, Cutoffs cut,
                    const float *__restrict__ disc, const float *__restrict__ ideal, double *__restrict__ sums,
                    double *__restrict__ per_user, unsigned *__restrict__ ticket, double *__restrict__ part) {
    __shared__ double sh[kTopkWarps][kTopkEntries];
    const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
    const long long stride = (long long)gridDim.x * kTopkWarps;
    const int my_c = lane < cut.n ? cut.c[lane] : 0;
    const unsigned long long below = my_c >= 64 ? ~0ull : ((1ull << my_c) - 1);
    double acc[FR_TOPK_METRICS];
#pragma unroll
    for (int m = 0; m < FR_TOPK_METRICS; ++m) acc[m] = 0.0;
    double len_sum = 0.0;

    long long r = (long long)blockIdx.x * kTopkWarps + wib;
    // software pipeline: the next row's indices, CSR bounds and length are in flight while this row searches
    long long v0 = -1, v1 = -1;
    int64_t lo = 0, hi = 0;
    int pl = 0;
    if (r < n) {
        if (lane < K) v0 = load_idx(top + r * K + lane);
        if (lane + 32 < K) v1 = load_idx(top + r * K + lane + 32);
        lo = __ldg(pos_ptr + r);
        hi = __ldg(pos_ptr + r + 1);
        pl = __ldg(pos_len + r);
    }
    for (; r < n; r += stride) {
        const long long rn = r + stride;
        long long n0 = -1, n1 = -1;
        int64_t nlo = 0, nhi = 0;
        int npl = 0;
        if (rn < n) {
            if (lane < K) n0 = load_idx(top + rn * K + lane);
            if (lane + 32 < K) n1 = load_idx(top + rn * K + lane + 32);
            nlo = __ldg(pos_ptr + rn);
            nhi = __ldg(pos_ptr + rn + 1);
            npl = __ldg(pos_len + rn);
        }
        const bool h0 = contains(pos_idx, lo, hi, v0);
        const bool h1 = contains(pos_idx, lo, hi, v1);
        const unsigned long long mask =
            (unsigned long long)__ballot_sync(0xffffffffu, h0) | ((unsigned long long)__ballot_sync(0xffffffffu, h1) << 32);
        if (lane < cut.n) {
            unsigned long long bits = mask & below;
            int cnt = 0;
            float dcg = 0.f;          // numpy: fp32 cumsum of where(hits, disc, 0); adding +0.0 is exact
            double ap = 0.0;          // numpy: fp64 cumsum of (cum / rank) * hit
            while (bits) {
                const int j = __ffsll((long long)bits) - 1;
                bits &= bits - 1;
                ++cnt;
                dcg = dcg + __ldg(disc + j);
                ap = ap + (double)cnt / (double)(j + 1);
            }
            double val[FR_TOPK_METRICS];
            if (pl >= 1) {
                const int den = min(my_c, pl);
                val[0] = (double)cnt / (double)pl;                          // recall
                val[1] = (double)cnt;                                       // recall2 numerator
                val[2] = (double)(dcg / __ldg(ideal + den - 1));            // ndcg (fp32 quotient)
                val[3] = (double)cnt / (double)my_c;                        // precision
                val[4] = (double)__double2float_rn(ap / (double)den);       // map (fp64 quotient cast to fp32)
            } else {
#pragma unroll
                for (int m = 0; m < FR_TOPK_METRICS; ++m) val[m] = __longlong_as_double(0x7ff8000000000000LL);
            }
#pragma unroll
            for (int m = 0; m < FR_TOPK_METRICS; ++m) {
                acc[m] += val[m];
                if (per_user) per_user[((size_t)r * FR_TOPK_METRICS + m) * cut.n + lane] = val[m];
            }
        }
        if (lane == 0) len_sum += (double)pl;
        v0 = n0; v1 = n1; lo = nlo; hi = nhi; pl = npl;
    }
    if (lane < kMaxCut) {
#pragma unroll
        for (int m = 0; m < FR_TOPK_METRICS; ++m) sh[wib][m * kMaxCut + lane] = acc[m];
    }
    if (lane == 0) sh[wib][kTopkEntries - 1] = len_sum;
    __syncthreads();
    if (threadIdx.x < kTopkEntries) {
        double s = 0.0;
        for (int w = 0; w < kTopkWarps; ++w) s += sh[w][threadIdx.x];
        __stcg(part + (size_t)threadIdx.x * gridDim.x + blockIdx.x, s);
    }
    if (!last_block(ticket)) return;
    fold_partials<(kTopkEntries + kTopkWarps - 1) / kTopkWarps>(part, kTopkEntries, gridDim.x, &sh[0][0]);
    __syncthreads();
    // compact [metric][kMaxCut] -> [metric][n_cut], then the pos_len sum
    if (threadIdx.x < FR_TOPK_METRICS * cut.n) {
        const int m = threadIdx.x / cut.n, i = threadIdx.x % cut.n;
        sums[threadIdx.x] = (&sh[0][0])[m * kMaxCut + i];
    }
    if (threadIdx.x == 0) {
        sums[FR_TOPK_METRICS * cut.n] = (&sh[0][0])[kTopkEntries - 1];
        *ticket = 0u;
    }
}

// One CTA per user (grid-stride over users).  The segment is staged in shared memory when it fits, otherwise read
// from global memory.  Warp w handles positives w, w + 8, ...: its lanes count, over the whole segment, the
// candidates that rank above the positive in the order of np.argsort(pred, kind="stable")[::-1] (greater score, or
// equal score at a later position) and the negatives with a strictly smaller score (AUC).  Positive ranks below 64
// set bits of a per-user hit mask; thread 0 turns mask and count into the user's values.
__global__ void __launch_bounds__(kUserThreads)
by_user_metrics_kernel(const float *__restrict__ scores, const int64_t *__restrict__ ptr,
                       const int32_t *__restrict__ n_pos, long long n, int neg_num, Cutoffs cut,
                       double *__restrict__ sums, double *__restrict__ per_user, unsigned *__restrict__ ticket,
                       double *__restrict__ part) {
    __shared__ float stage[kStage];
    __shared__ double disc[64];
    __shared__ double acc[kUserEntries];
    __shared__ unsigned long long hitmask, auc_cnt;
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    constexpr int kW = kUserThreads / 32;
    if (threadIdx.x < 64) disc[threadIdx.x] = 1.0 / log2((double)threadIdx.x + 2.0);
    if (threadIdx.x < kUserEntries) acc[threadIdx.x] = 0.0;
    const int n_out = 1 + 2 * cut.n;

    for (long long u = blockIdx.x; u < n; u += gridDim.x) {
        const int64_t lo = __ldg(ptr + u);
        const long long L = __ldg(ptr + u + 1) - lo;
        const int p = __ldg(n_pos + u);
        const bool staged = L <= kStage;
        if (staged)
            for (int j = threadIdx.x; j < L; j += kUserThreads) stage[j] = __ldcs(scores + lo + j);
        if (threadIdx.x == 0) {
            hitmask = 0ull;
            auc_cnt = 0ull;
        }
        __syncthreads();
        const bool valid = p >= 1 && p <= L;
        if (valid) {
            const float *s = staged ? stage : scores + lo;
            for (int i = w; i < p; i += kW) {
                const float si = s[i];
                unsigned above = 0, below_neg = 0;
                for (long long j = lane; j < L; j += 32) {
                    const float v = s[j];
                    above += (v > si) | ((v == si) & (j > i));
                    below_neg += (j >= p) & (v < si);
                }
                above = __reduce_add_sync(0xffffffffu, above);
                below_neg = __reduce_add_sync(0xffffffffu, below_neg);
                if (lane == 0) {
                    if (above < 64u) atomicOr(&hitmask, 1ull << above);
                    atomicAdd(&auc_cnt, (unsigned long long)below_neg);
                }
            }
        }
        __syncthreads();
        if (threadIdx.x == 0) {
            double val[kUserEntries];
            if (valid) {
                val[0] = (double)auc_cnt / ((double)p * (double)neg_num);
                const unsigned long long mask = hitmask;
                for (int i = 0; i < cut.n; ++i) {
                    const int c = cut.c[i];
                    unsigned long long bits = mask & (c >= 64 ? ~0ull : ((1ull << c) - 1));
                    val[1 + i] = (double)__popcll(bits) / (double)p;
                    double dcg = 0.0, idcg = 0.0;
                    while (bits) {
                        dcg += disc[__ffsll((long long)bits) - 1];
                        bits &= bits - 1;
                    }
                    const long long m = min((long long)min(c, p), L);
                    for (int t = 0; t < m; ++t) idcg += disc[t];
                    val[1 + cut.n + i] = dcg / idcg;
                }
            } else {
                for (int e = 0; e < n_out; ++e) val[e] = __longlong_as_double(0x7ff8000000000000LL);
            }
            for (int e = 0; e < n_out; ++e) {
                const int slot = e == 0 ? 0 : (e <= cut.n ? e : kMaxCut + e - cut.n);
                acc[slot] += val[e];
                if (per_user) per_user[(size_t)u * n_out + e] = val[e];
            }
        }
    }
    __syncthreads();
    if (threadIdx.x < kUserEntries) __stcg(part + (size_t)threadIdx.x * gridDim.x + blockIdx.x, acc[threadIdx.x]);
    if (!last_block(ticket)) return;
    __shared__ double folded[kUserEntries];
    fold_partials<(kUserEntries + kW - 1) / kW>(part, kUserEntries, gridDim.x, folded);
    __syncthreads();
    if (threadIdx.x < n_out) {
        const int e = threadIdx.x;
        sums[e] = folded[e == 0 ? 0 : (e <= cut.n ? e : kMaxCut + e - cut.n)];
    }
    if (threadIdx.x == 0) *ticket = 0u;
}

// Resident blocks of a kernel on the whole device (the grid of the persistent launches; at most this many partials).
template <typename Kern>
int resident_blocks(Kern k, int threads) {
    int per_sm = 0;
    if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, k, threads, 0) != cudaSuccess || per_sm < 1) per_sm = 1;
    return per_sm * fr::num_sms();
}

int grid_topk(bool idx64) {
    static int g32 = 0, g64 = 0;
    int &g = idx64 ? g64 : g32;
    if (!g) g = idx64 ? resident_blocks(topk_metrics_kernel<long long>, kTopkWarps * 32)
                      : resident_blocks(topk_metrics_kernel<int>, kTopkWarps * 32);
    return g;
}

int grid_by_user() {
    static int g = 0;
    if (!g) g = resident_blocks(by_user_metrics_kernel, kUserThreads);
    return g;
}

int max_grid() { return std::max(std::max(grid_topk(false), grid_topk(true)), grid_by_user()); }

}  // namespace

extern "C" int64_t fr_eval_metrics_ws_bytes(void) {
    return 16 + (int64_t)std::max(kTopkEntries, kUserEntries) * max_grid() * (int64_t)sizeof(double);
}

extern "C" int fr_topk_metrics(const void *top, int32_t idx64, int64_t n, int32_t K, const int64_t *pos_ptr,
                               const int32_t *pos_idx, const int32_t *pos_len, const int32_t *cutoffs_host,
                               int32_t n_cut, const float *disc, const float *ideal, double *sums, double *per_user,
                               void *ws, void *stream) {
    FR_REQUIRE(top && pos_ptr && pos_idx && pos_len && cutoffs_host && disc && ideal && sums && ws,
               "fr_topk_metrics: null pointer");
    FR_REQUIRE(n >= 1, "fr_topk_metrics: n=%lld", (long long)n);
    FR_REQUIRE(K >= 1 && K <= 64, "fr_topk_metrics: K=%d outside [1, 64]", K);
    FR_REQUIRE(n_cut >= 1 && n_cut <= kMaxCut, "fr_topk_metrics: %d cutoffs (1..%d allowed)", n_cut, kMaxCut);
    FR_REQUIRE(((uintptr_t)ws & 15) == 0, "fr_topk_metrics: ws must be 16-byte aligned");
    Cutoffs cut{};
    cut.n = n_cut;
    for (int i = 0; i < n_cut; ++i) {
        FR_REQUIRE(cutoffs_host[i] >= 1 && cutoffs_host[i] <= K, "fr_topk_metrics: cutoff %d outside [1, K=%d]",
                   cutoffs_host[i], K);
        cut.c[i] = cutoffs_host[i];
    }
    const int grid = (int)std::min<long long>((n + kTopkWarps - 1) / kTopkWarps, grid_topk(idx64 != 0));
    unsigned *ticket = reinterpret_cast<unsigned *>(ws);
    double *part = reinterpret_cast<double *>(ws) + 2;
    cudaStream_t st = (cudaStream_t)stream;
    fr::LaunchTimer _lt("topk_metrics_kernel", st);
    if (idx64)
        topk_metrics_kernel<long long><<<grid, kTopkWarps * 32, 0, st>>>(
            static_cast<const long long *>(top), n, K, pos_ptr, pos_idx, pos_len, cut, disc, ideal, sums, per_user,
            ticket, part);
    else
        topk_metrics_kernel<int><<<grid, kTopkWarps * 32, 0, st>>>(
            static_cast<const int *>(top), n, K, pos_ptr, pos_idx, pos_len, cut, disc, ideal, sums, per_user, ticket,
            part);
    return fr::check_launch("fr_topk_metrics");
}

extern "C" int fr_by_user_metrics(const float *scores, const int64_t *ptr, const int32_t *n_pos, int64_t n,
                                  int32_t neg_num, const int32_t *cutoffs_host, int32_t n_cut, double *sums,
                                  double *per_user, void *ws, void *stream) {
    FR_REQUIRE(scores && ptr && n_pos && cutoffs_host && sums && ws, "fr_by_user_metrics: null pointer");
    FR_REQUIRE(n >= 1, "fr_by_user_metrics: n=%lld", (long long)n);
    FR_REQUIRE(neg_num >= 1, "fr_by_user_metrics: neg_num=%d", neg_num);
    FR_REQUIRE(n_cut >= 1 && n_cut <= kMaxCut, "fr_by_user_metrics: %d cutoffs (1..%d allowed)", n_cut, kMaxCut);
    FR_REQUIRE(((uintptr_t)ws & 15) == 0, "fr_by_user_metrics: ws must be 16-byte aligned");
    Cutoffs cut{};
    cut.n = n_cut;
    for (int i = 0; i < n_cut; ++i) {
        FR_REQUIRE(cutoffs_host[i] >= 1 && cutoffs_host[i] <= 64, "fr_by_user_metrics: cutoff %d outside [1, 64]",
                   cutoffs_host[i]);
        cut.c[i] = cutoffs_host[i];
    }
    const int grid = (int)std::min<long long>(n, grid_by_user());
    cudaStream_t st = (cudaStream_t)stream;
    fr::LaunchTimer _lt("by_user_metrics_kernel", st);
    by_user_metrics_kernel<<<grid, kUserThreads, 0, st>>>(scores, ptr, n_pos, n, neg_num, cut, sums, per_user,
                                                          reinterpret_cast<unsigned *>(ws),
                                                          reinterpret_cast<double *>(ws) + 2);
    return fr::check_launch("fr_by_user_metrics");
}
