// Fused BPR + embedding-regulariser loss on gathered rows (forward and backward), sm_100a.
//
// Latency-bound (B = 512 rows of 256 bytes): the point of the fusion is launch count -- the
// reference path issues ~25 small kernels for these gathers / reductions and ~15 more for their
// autograd; here it is one launch each way.  One warp per task (a BPR triple or one regularised
// row); block partials go to a workspace and the last block (atomic ticket) folds them in fixed
// order, so the loss value is bit-reproducible.
#include "common.cuh"

namespace {

constexpr int kWarps = 8;

struct Groups {
    const float *tab[FR_MAX_REG_GROUPS];
    const int64_t *idx[FR_MAX_REG_GROUPS];
    float *dtab[FR_MAX_REG_GROUPS];
    long long start[FR_MAX_REG_GROUPS + 1];  // task-id prefix (after the B triples)
    long long pad[FR_MAX_REG_GROUPS];
    int n;
};

__device__ __forceinline__ float dot_rows(const float *__restrict__ a, const float *__restrict__ b, int d, int lane) {
    float s = 0.f;
    for (int k = lane; k < d; k += 32) s = fmaf(__ldg(a + k), __ldg(b + k), s);
    return s;
}

__global__ void __launch_bounds__(kWarps * 32)
rank_loss_fwd_kernel(const float *__restrict__ emb, int d, long long item_off, const int64_t *__restrict__ u,
                     const int64_t *__restrict__ p, const int64_t *__restrict__ n, int B, float gamma, Groups g,
                     float reg_den, float *__restrict__ out, float *__restrict__ coef, float *__restrict__ gnorm,
                     float *__restrict__ ws) {
    __shared__ float sh[kWarps][1 + FR_MAX_REG_GROUPS];
    __shared__ int last;
    const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
    const long long n_tasks = B + g.start[g.n];
    const long long warps_total = (long long)gridDim.x * kWarps;
    float part[1 + FR_MAX_REG_GROUPS];
#pragma unroll
    for (int i = 0; i <= FR_MAX_REG_GROUPS; ++i) part[i] = 0.f;

    for (long long t = (long long)blockIdx.x * kWarps + wib; t < n_tasks; t += warps_total) {
        if (t < B) {
            const float *ue = emb + (size_t)u[t] * d;
            const float *pe = emb + (size_t)(item_off + p[t]) * d;
            const float *ne = emb + (size_t)(item_off + n[t]) * d;
            float x = 0.f;
            for (int k = lane; k < d; k += 32) {
                const float uv = __ldg(ue + k);
                x = fmaf(uv, __ldg(pe + k) - __ldg(ne + k), x);
            }
            x = fr::warp_sum(x);
            const float sg = 1.f / (1.f + expf(-x));
            part[0] += -logf(gamma + sg);
            if (lane == 0) coef[t] = -(sg * (1.f - sg)) / ((gamma + sg) * (float)B);
        } else {
            const long long q = t - B;
            int gi = 0;
#pragma unroll
            for (int i = 1; i < FR_MAX_REG_GROUPS; ++i)
                if (i < g.n && q >= g.start[i]) gi = i;
            const long long id = g.idx[gi][q - g.start[gi]];
            const float *row = g.tab[gi] + (size_t)id * d;
            const float s = fr::warp_sum(dot_rows(row, row, d, lane));
#pragma unroll
            for (int i = 0; i < FR_MAX_REG_GROUPS; ++i)
                if (i == gi) part[1 + i] += s;
        }
    }
    if (lane == 0) {
#pragma unroll
        for (int i = 0; i <= FR_MAX_REG_GROUPS; ++i) sh[wib][i] = part[i];
    }
    __syncthreads();
    if (threadIdx.x <= FR_MAX_REG_GROUPS) {
        float s = 0.f;
        for (int w = 0; w < kWarps; ++w) s += sh[w][threadIdx.x];
        __stcg(ws + 8 + (size_t)blockIdx.x * 8 + threadIdx.x, s);
    }
    __threadfence();
    __syncthreads();
    if (threadIdx.x == 0) last = (atomicAdd(reinterpret_cast<int *>(ws), 1) == (int)gridDim.x - 1);
    __syncthreads();
    if (!last) return;
    __threadfence();
    if (threadIdx.x <= FR_MAX_REG_GROUPS) {
        float s = 0.f;
        for (unsigned b = 0; b < gridDim.x; ++b) s += __ldcg(ws + 8 + (size_t)b * 8 + threadIdx.x);
        sh[0][threadIdx.x] = s;
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        out[0] = sh[0][0] / (float)B;
        float r = 0.f;
        for (int i = 0; i < g.n; ++i) {
            const float nr = sqrtf(sh[0][1 + i]);
            gnorm[i] = nr;
            r += nr;
        }
        out[1] = r / reg_den;
        *reinterpret_cast<int *>(ws) = 0;
    }
}

__global__ void __launch_bounds__(kWarps * 32)
rank_loss_bwd_kernel(const float *__restrict__ emb, int d, long long item_off, const int64_t *__restrict__ u,
                     const int64_t *__restrict__ p, const int64_t *__restrict__ n, int B,
                     const float *__restrict__ coef, const float *__restrict__ g_out, float *__restrict__ d_emb,
                     Groups g, float reg_den, const float *__restrict__ gnorm, unsigned char *__restrict__ emb_mask) {
    const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
    const long long n_tasks = B + g.start[g.n];
    const long long warps_total = (long long)gridDim.x * kWarps;
    const float g_mf = __ldg(g_out), g_reg = __ldg(g_out + 1);
    for (long long t = (long long)blockIdx.x * kWarps + wib; t < n_tasks; t += warps_total) {
        if (t < B) {
            if (d_emb == nullptr) continue;
            const size_t ur = (size_t)u[t] * d, pr = (size_t)(item_off + p[t]) * d, nr = (size_t)(item_off + n[t]) * d;
            const float c = coef[t] * g_mf;
            if (emb_mask != nullptr && lane < 3)      // rows of d_emb this triple touches (all others stay exactly 0)
                emb_mask[lane == 0 ? u[t] : (item_off + (lane == 1 ? p[t] : n[t]))] = 1;
            for (int k = lane; k < d; k += 32) {
                const float uv = __ldg(emb + ur + k), pv = __ldg(emb + pr + k), nv = __ldg(emb + nr + k);
                atomicAdd(d_emb + ur + k, c * (pv - nv));
                atomicAdd(d_emb + pr + k, c * uv);
                atomicAdd(d_emb + nr + k, -c * uv);
            }
        } else {
            const long long q = t - B;
            int gi = 0;
#pragma unroll
            for (int i = 1; i < FR_MAX_REG_GROUPS; ++i)
                if (i < g.n && q >= g.start[i]) gi = i;
            if (g.dtab[gi] == nullptr) continue;
            const long long id = g.idx[gi][q - g.start[gi]];
            if (id == g.pad[gi]) continue;
            const float nr = __ldg(gnorm + gi);
            const float sc = nr > 0.f ? g_reg / (reg_den * nr) : 0.f;
            const float *row = g.tab[gi] + (size_t)id * d;
            float *drow = g.dtab[gi] + (size_t)id * d;
            for (int k = lane; k < d; k += 32) atomicAdd(drow + k, sc * __ldg(row + k));
        }
    }
}

// Stand-alone forms of the two loss modules (FoodRec/common/loss.py:31-34, 44-50) for callers that already hold
// scores / gathered rows (batch-sized inputs): ONE block, fixed summation order, so the value is bit-reproducible.
__global__ void __launch_bounds__(1024)
bpr_scores_kernel(const float *__restrict__ pos, const float *__restrict__ neg, long long n, float gamma,
                  float *__restrict__ out, float *__restrict__ coef) {
    __shared__ float sh[32];
    float s = 0.f;
    for (long long i = threadIdx.x; i < n; i += blockDim.x) {
        const float x = pos[i] - neg[i];
        const float sg = 1.f / (1.f + expf(-x));
        s += -logf(gamma + sg);
        coef[i] = -(sg * (1.f - sg)) / ((gamma + sg) * (float)n);   // d out / d pos[i] = -d out / d neg[i]
    }
    s = fr::warp_sum(s);
    if ((threadIdx.x & 31) == 0) sh[threadIdx.x >> 5] = s;
    __syncthreads();
    if (threadIdx.x < 32) {
        s = fr::warp_sum(threadIdx.x < (blockDim.x >> 5) ? sh[threadIdx.x] : 0.f);
        if (threadIdx.x == 0) out[0] = s / (float)n;
    }
}

__global__ void __launch_bounds__(1024)
l2_norm_kernel(const float *__restrict__ x, long long n, float *__restrict__ out) {
    __shared__ float sh[32];
    float s = 0.f;
    for (long long i = threadIdx.x; i < n; i += blockDim.x) s = fmaf(x[i], x[i], s);
    s = fr::warp_sum(s);
    if ((threadIdx.x & 31) == 0) sh[threadIdx.x >> 5] = s;
    __syncthreads();
    if (threadIdx.x < 32) {
        s = fr::warp_sum(threadIdx.x < (blockDim.x >> 5) ? sh[threadIdx.x] : 0.f);
        if (threadIdx.x == 0) out[0] = sqrtf(s);
    }
}

int fill_groups(Groups &g, int n_groups, const float *const *tab, const int64_t *const *idx, const int64_t *cnt,
                const int64_t *pad, float *const *dtab) {
    FR_REQUIRE(n_groups >= 0 && n_groups <= FR_MAX_REG_GROUPS, "rank_loss: n_groups=%d out of range", n_groups);
    g.n = n_groups;
    g.start[0] = 0;
    for (int i = 0; i < FR_MAX_REG_GROUPS; ++i) {
        const bool on = i < n_groups;
        // an empty group (cnt 0) owns no task, so its index pointer is never read and may be NULL (an empty tensor's)
        FR_REQUIRE(!on || (tab[i] && cnt[i] >= 0 && (idx[i] || cnt[i] == 0)), "rank_loss: bad regulariser group %d", i);
        g.tab[i] = on ? tab[i] : nullptr;
        g.idx[i] = on ? idx[i] : nullptr;
        g.dtab[i] = (on && dtab) ? dtab[i] : nullptr;
        g.pad[i] = (on && pad) ? pad[i] : -1;
        g.start[i + 1] = g.start[i] + (on ? cnt[i] : 0);
    }
    return FR_OK;
}

int grid_for(long long n_tasks) {
    long long b = (n_tasks + kWarps - 1) / kWarps;
    const long long cap = (long long)fr::num_sms() * 4;
    return (int)std::max<long long>(1, std::min(b, cap));
}

}  // namespace

extern "C" int64_t fr_rank_loss_ws_floats(void) { return 8 + 8 * (int64_t)fr::num_sms() * 4; }

extern "C" int fr_rank_loss_fwd(const float *emb, int32_t d, int64_t item_off, const int64_t *u, const int64_t *p,
                                const int64_t *n, int32_t B, float gamma, int32_t n_groups,
                                const float *const *reg_tab_host, const int64_t *const *reg_idx_host,
                                const int64_t *reg_cnt_host, float reg_den, float *out, float *coef, float *gnorm,
                                float *ws, void *stream) {
    FR_REQUIRE(emb && u && p && n && out && coef && gnorm && ws, "fr_rank_loss_fwd: null pointer");
    FR_REQUIRE(B > 0 && d > 0, "fr_rank_loss_fwd: B=%d d=%d", B, d);
    Groups g;
    if (int rc = fill_groups(g, n_groups, reg_tab_host, reg_idx_host, reg_cnt_host, nullptr, nullptr)) return rc;
    const int grid = grid_for(B + g.start[g.n]);
    fr::LaunchTimer _lt("rank_loss_fwd_kernel", (cudaStream_t)stream);
    rank_loss_fwd_kernel<<<grid, kWarps * 32, 0, (cudaStream_t)stream>>>(emb, d, item_off, u, p, n, B, gamma, g,
                                                                         reg_den, out, coef, gnorm, ws);
    return fr::check_launch("fr_rank_loss_fwd");
}

extern "C" int fr_rank_loss_bwd(const float *emb, int32_t d, int64_t item_off, const int64_t *u, const int64_t *p,
                                const int64_t *n, int32_t B, const float *coef, const float *g_out, float *d_emb,
                                int32_t n_groups, const float *const *reg_tab_host,
                                const int64_t *const *reg_idx_host, const int64_t *reg_cnt_host,
                                const int64_t *reg_pad_host, float reg_den, const float *gnorm,
                                float *const *d_tab_host, uint8_t *emb_mask, void *stream) {
    FR_REQUIRE(emb && u && p && n && coef && g_out && gnorm, "fr_rank_loss_bwd: null pointer");
    FR_REQUIRE(B > 0 && d > 0, "fr_rank_loss_bwd: B=%d d=%d", B, d);
    Groups g;
    if (int rc = fill_groups(g, n_groups, reg_tab_host, reg_idx_host, reg_cnt_host, reg_pad_host, d_tab_host))
        return rc;
    const int grid = grid_for(B + g.start[g.n]);
    fr::LaunchTimer _lt("rank_loss_bwd_kernel", (cudaStream_t)stream);
    rank_loss_bwd_kernel<<<grid, kWarps * 32, 0, (cudaStream_t)stream>>>(emb, d, item_off, u, p, n, B, coef, g_out,
                                                                         d_emb, g, reg_den, gnorm, emb_mask);
    return fr::check_launch("fr_rank_loss_bwd");
}

extern "C" int fr_bpr_scores_fwd(const float *pos, const float *neg, int64_t n, float gamma, float *out, float *coef,
                                 void *stream) {
    FR_REQUIRE(pos && neg && out && coef, "fr_bpr_scores_fwd: null pointer");
    FR_REQUIRE(n > 0, "fr_bpr_scores_fwd: n=%lld", (long long)n);
    fr::LaunchTimer _lt("bpr_scores_kernel", (cudaStream_t)stream);
    bpr_scores_kernel<<<1, 1024, 0, (cudaStream_t)stream>>>(pos, neg, n, gamma, out, coef);
    return fr::check_launch("fr_bpr_scores_fwd");
}

extern "C" int fr_l2_norm_f32(const float *x, int64_t n, float *out, void *stream) {
    FR_REQUIRE(x && out, "fr_l2_norm_f32: null pointer");
    FR_REQUIRE(n > 0, "fr_l2_norm_f32: n=%lld", (long long)n);
    fr::LaunchTimer _lt("l2_norm_kernel", (cudaStream_t)stream);
    l2_norm_kernel<<<1, 1024, 0, (cudaStream_t)stream>>>(x, n, out);
    return fr::check_launch("fr_l2_norm_f32");
}
