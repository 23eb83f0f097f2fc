// SCHGN's per-pair scorer for full-sort evaluation, fused (sm_100a).
//
// Reference: FoodRec/models/schgn.py:159-206 (ingredient-level and component-level attention),
// :233-268 (compute_score), :318-345 (full_sort_predict: one user against every item, with python loops,
// an [I, Dv] upload and a full GCN per user).  Everything that does not depend on the user is computed
// once by the host side (models/schgn.py `_item_side`): final ingredient / item / image / health rows and
// their images under the attention weights.  What is left per (user, item) pair is
//
//   a_j    = h_i . tanh(ingre_key[code_j] + img_key[item] + user_key[u])          j < n_item
//   A      = softmax_j(a)                 att = sum_j A_j ingre_final[code_j]
//   l_1    = h_c . tanh(user_comp[u] + sum_j A_j ingre_comp[code_j])              (linear in att)
//   l_k    = h_c . tanh(user_comp[u] + comp_key_k[item])                          k = item, image, health
//   B      = softmax over the reference's `.view(b, -1)` grouping of the [4, I] logits (schgn.py:198)
//   x      = B_0 item + B_1 att + B_2 image + B_3 health
//   score  = w_out . relu(user_hidden[u] + W_item x + W_prod (u_final * x))
//
// Two launches per block of users because B mixes logits of different items:
//   schgn_attend_kernel: one warp per item, lanes over the 64 features, 16 users per pass so every
//     gathered ingredient row is reused 16 times from registers; writes att [nu, I, 64] and logits [nu, 4, I].
//   schgn_score_kernel: one thread per (user, 2 items); the user's 64x64 matrix
//     M_u = W_item + W_prod diag(u_final) sits in shared memory (broadcast reads), x in registers (rows are
//     loaded coalesced, 16 threads per row, and handed to their owner thread through shared memory).
// Arithmetic is fp32 throughout (scores feed a top-K that must match the reference's).
//
// tanh of a sum of a user-independent and a user-dependent term is evaluated as
//   tanh(a + b) = 1 - 2 / (1 + e^{2a} e^{2b})
// with e^{2a} computed once per (item, ingredient, feature) and reused by the 16 users of the pass, e^{2b}
// once per (user, feature) per CTA, both with the precise expf; what is left per (user, item, ingredient,
// feature) is one FFMA, one hardware reciprocal refined by a Newton step, and one FFMA into the logit --
// one MUFU op instead of tanhf's two plus its polynomial branch.  Error ~ 2e-7 absolute, the same order
// as tanhf's own 2 ulp.  Operands are clamped to +-43 before the exponential (so the product cannot be
// inf * 0); tanh is saturated in fp32 beyond |x| = 9.1.
#include "common.cuh"

namespace {

constexpr int D = 64;           // embedding width of the model (schgn.py:69-70 hard-codes 64)
constexpr int MAX_SLOTS = 32;   // ingredient slots per recipe (reference: 20)
constexpr int UB = 16;          // users per attend pass
constexpr int ATT_WARPS = 8;

struct AttendParams {
    const float *user_key, *user_comp;
    const int32_t *codes, *nums;
    const float *ingre_key, *ingre_final, *ingre_comp, *img_key, *comp_keys, *h_ingre, *h_comp;
    float *att, *logits;
    int32_t nu, n_items, slots;
};

constexpr float CLAMP = 43.0f;
// e^{2x}, x clamped so that products of two such factors stay finite or overflow cleanly to +inf
__device__ __forceinline__ float exp2x(float x) { return expf(2.0f * fminf(fmaxf(x, -CLAMP), CLAMP)); }
// 1 / (1 + ea * eb) to ~1 ulp: hardware reciprocal + one Newton step (x is in [1, 1e30])
__device__ __forceinline__ float inv1p(float ea, float eb) {
    const float x = fminf(fmaf(ea, eb, 1.0f), 1e30f);
    float r;
    asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x));
    return fmaf(r, fmaf(-x, r, 1.0f), r);
}

// Sum each of v[0..15] over the 32 lanes with 16 shuffles; lane L ends up holding the total of
// v[L >> 1] (both lanes of a pair hold the same value).
__device__ __forceinline__ float reduce16(float (&v)[UB], int lane) {
#pragma unroll
    for (int half = 8, bit = 16; half >= 1; half >>= 1, bit >>= 1) {
        const bool up = lane & bit;
#pragma unroll
        for (int i = 0; i < half; ++i) {
            const float send = up ? v[i] : v[i + half];
            const float keep = up ? v[i + half] : v[i];
            v[i] = keep + __shfl_xor_sync(0xffffffffu, send, bit);
        }
    }
    return v[0] + __shfl_xor_sync(0xffffffffu, v[0], 1);
}

__global__ void __launch_bounds__(ATT_WARPS * 32) schgn_attend_kernel(const AttendParams p) {
    __shared__ float s_ukey[UB][D];   // e^{2 user_key}
    __shared__ float s_ucomp[UB][D];  // e^{2 user_comp}
    __shared__ float s_logit[ATT_WARPS][UB][MAX_SLOTS];
    const int u0 = blockIdx.y * UB;
    for (int t = threadIdx.x; t < UB * D; t += blockDim.x) {
        const int u = min(u0 + t / D, p.nu - 1);
        s_ukey[t / D][t % D] = exp2x(p.user_key[(size_t)u * D + t % D]);
        s_ucomp[t / D][t % D] = exp2x(p.user_comp[(size_t)u * D + t % D]);
    }
    __syncthreads();
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int item = blockIdx.x * ATT_WARPS + warp;
    if (item >= p.n_items) return;
    const int n = max(0, min(p.nums[item], p.slots));
    const int code = lane < p.slots ? p.codes[(size_t)item * p.slots + lane] : 0;
    const int c2 = 2 * lane;
    const float2 pi = *reinterpret_cast<const float2 *>(p.img_key + (size_t)item * D + c2);
    const float2 hi = *reinterpret_cast<const float2 *>(p.h_ingre + c2);
    const float2 hc = *reinterpret_cast<const float2 *>(p.h_comp + c2);
    const float hi_sum = hi.x + hi.y, hc_sum = hc.x + hc.y;  // sum_d h (1 - 2 r_d) = sum h - 2 sum h r_d

    // pass 1: attention logits a[u][j]
    for (int j = 0; j < n; ++j) {
        const int c = __shfl_sync(0xffffffffu, code, j);
        const float2 pe = __ldg(reinterpret_cast<const float2 *>(p.ingre_key + (size_t)c * D + c2));
        const float ex = exp2x(pe.x + pi.x), ey = exp2x(pe.y + pi.y);
        float v[UB];
#pragma unroll
        for (int u = 0; u < UB; ++u) {
            const float2 uk = *reinterpret_cast<const float2 *>(&s_ukey[u][c2]);
            v[u] = fmaf(-2.0f, fmaf(hi.x, inv1p(ex, uk.x), hi.y * inv1p(ey, uk.y)), hi_sum);
        }
        const float tot = reduce16(v, lane);
        if (!(lane & 1)) s_logit[warp][lane >> 1][j] = tot;
    }
    __syncwarp();

    // softmax over the recipe's real ingredients (masked slots carry weight exactly 0 in the reference:
    // exp(-1e12 - max) underflows); lane j keeps A[u][j]
    float A[UB];
#pragma unroll
    for (int u = 0; u < UB; ++u) {
        const float x = lane < n ? s_logit[warp][u][lane] : -INFINITY;
        float m = x;
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, o));
        const float e = lane < n ? expf(x - m) : 0.0f;
        const float s = fr::warp_sum(e);
        A[u] = n > 0 ? e / s : 0.0f;
    }

    // pass 2: attended ingredient row and its image under W_att_comp's component half
    float2 att[UB], q[UB];
#pragma unroll
    for (int u = 0; u < UB; ++u) att[u] = q[u] = make_float2(0.0f, 0.0f);
    for (int j = 0; j < n; ++j) {
        const int c = __shfl_sync(0xffffffffu, code, j);
        const float2 ef = __ldg(reinterpret_cast<const float2 *>(p.ingre_final + (size_t)c * D + c2));
        const float2 qe = __ldg(reinterpret_cast<const float2 *>(p.ingre_comp + (size_t)c * D + c2));
#pragma unroll
        for (int u = 0; u < UB; ++u) {
            const float w = __shfl_sync(0xffffffffu, A[u], j);
            att[u].x = fmaf(w, ef.x, att[u].x);
            att[u].y = fmaf(w, ef.y, att[u].y);
            q[u].x = fmaf(w, qe.x, q[u].x);
            q[u].y = fmaf(w, qe.y, q[u].y);
        }
    }
#pragma unroll
    for (int u = 0; u < UB; ++u)
        if (u0 + u < p.nu)
            *reinterpret_cast<float2 *>(p.att + ((size_t)(u0 + u) * p.n_items + item) * D + c2) = att[u];

    // component logits, reference order: item id, attended ingredients, image, health
    const float *ck = p.comp_keys + (size_t)item * 3 * D + c2;
    float2 k_item = *reinterpret_cast<const float2 *>(ck);
    float2 k_img = *reinterpret_cast<const float2 *>(ck + D);
    float2 k_hl = *reinterpret_cast<const float2 *>(ck + 2 * D);
    k_item = make_float2(exp2x(k_item.x), exp2x(k_item.y));
    k_img = make_float2(exp2x(k_img.x), exp2x(k_img.y));
    k_hl = make_float2(exp2x(k_hl.x), exp2x(k_hl.y));
    const int my_u = u0 + (lane >> 1);
#pragma unroll
    for (int comp = 0; comp < 4; ++comp) {
        float v[UB];
#pragma unroll
        for (int u = 0; u < UB; ++u) {
            const float2 uc = *reinterpret_cast<const float2 *>(&s_ucomp[u][c2]);
            const float2 k = comp == 0   ? k_item
                             : comp == 1 ? make_float2(exp2x(q[u].x), exp2x(q[u].y))
                             : comp == 2 ? k_img
                                         : k_hl;
            v[u] = fmaf(-2.0f, fmaf(hc.x, inv1p(k.x, uc.x), hc.y * inv1p(k.y, uc.y)), hc_sum);
        }
        const float tot = reduce16(v, lane);
        if (!(lane & 1) && my_u < p.nu) p.logits[((size_t)my_u * 4 + comp) * p.n_items + item] = tot;
    }
}

struct ScoreParams {
    const float *user_final, *user_hidden, *W_item, *W_prod, *w_out, *comps, *att, *logits;
    float *scores;
    int32_t nu, n_items;
    // fused top-k mode (TOPK): instead of the dense scores, each CTA keeps the kt best of its 256 items as sortable
    // 64-bit keys [nu, n_blocks, kt]; `user_ids` + the history CSR mask training items (NULL: no mask, as the reference)
    unsigned long long *cand;
    const int64_t *user_ids, *hist_ptr;
    const int32_t *hist_idx;
    int32_t kt;
};

// (score desc, column asc) as ONE descending 64-bit key; 0 = absent
__device__ __forceinline__ unsigned long long topk_key(float score, int col) {
    const unsigned u = __float_as_uint(score);
    const unsigned ok = (u & 0x80000000u) ? ~u : (u | 0x80000000u);
    return ((unsigned long long)ok << 32) | (unsigned)(~col);
}
__device__ __forceinline__ float key_score(unsigned long long k) {
    const unsigned ok = (unsigned)(k >> 32);
    return __uint_as_float((ok & 0x80000000u) ? (ok & 0x7fffffffu) : ~ok);
}
// descending bitonic sort of `n` (power of two) keys in shared memory by the whole CTA
__device__ __forceinline__ void bitonic_desc(unsigned long long *key, int n, int tid, int nthreads) {
    for (int size = 2; size <= n; size <<= 1)
        for (int stride = size >> 1; stride > 0; stride >>= 1) {
            for (int i = tid; i < n / 2; i += nthreads) {
                const int lo = 2 * i - (i & (stride - 1)), hi = lo + stride;
                const bool desc = (lo & size) == 0;
                const unsigned long long a = key[lo], b = key[hi];
                if ((a < b) == desc) { key[lo] = b; key[hi] = a; }
            }
            __syncthreads();
        }
}

constexpr int SC_THREADS = 128;
constexpr int IPT = 2;                      // items per thread
constexpr int SC_ITEMS = SC_THREADS * IPT;  // items per CTA
constexpr int XS = D + 4;                   // row stride of the x tile (floats): conflict-free LDS.128 per quarter-warp
constexpr int SC_SMEM = (SC_ITEMS * XS + D * D + 2 * D + SC_ITEMS * 4) * (int)sizeof(float);

template <bool TOPK>
__global__ void __launch_bounds__(SC_THREADS) schgn_score_kernel(const ScoreParams p) {
    extern __shared__ __align__(16) float smem[];
    float *sX = smem;                    // [SC_ITEMS][XS]   x = B-weighted component mix, one row per item
    float *sM = sX + SC_ITEMS * XS;      // [D][D]           M_u = W_item + W_prod diag(u_final)
    float *sH = sM + D * D;              // [D]              user_hidden[u]
    float *sW = sH + D;                  // [D]              w_out
    float *sB = sW + D;                  // [SC_ITEMS][4]    component softmax weights
    const int u = blockIdx.y, tid = threadIdx.x;
    const int base = blockIdx.x * SC_ITEMS;
    for (int t = tid; t < D * D; t += SC_THREADS)
        sM[t] = fmaf(p.W_prod[t], p.user_final[(size_t)u * D + t % D], p.W_item[t]);
    if (tid < D) {
        sH[tid] = p.user_hidden[(size_t)u * D + tid];
        sW[tid] = p.w_out[tid];
    }
    // component weights: the [4, I] logits of this user read back as [I, 4] (schgn.py:198)
    const float *lg = p.logits + (size_t)u * 4 * p.n_items;
#pragma unroll
    for (int t = 0; t < IPT; ++t) {
        const int r = min(base + tid + t * SC_THREADS, p.n_items - 1);
        const float4 l = *reinterpret_cast<const float4 *>(lg + (size_t)4 * r);
        const float m = fmaxf(fmaxf(l.x, l.y), fmaxf(l.z, l.w));
        const float e0 = expf(l.x - m), e1 = expf(l.y - m), e2 = expf(l.z - m), e3 = expf(l.w - m);
        const float inv = 1.0f / (e0 + e1 + e2 + e3);
        *reinterpret_cast<float4 *>(sB + 4 * (tid + t * SC_THREADS)) = make_float4(e0 * inv, e1 * inv, e2 * inv, e3 * inv);
    }
    __syncthreads();
    // x rows, loaded coalesced: 16 threads per row (one float4 each), 8 rows per pass
    {
        const int sub = (tid & 15) * 4, rr = tid >> 4;
#pragma unroll 4
        for (int row = rr; row < SC_ITEMS; row += SC_THREADS / 16) {
            const int r = min(base + row, p.n_items - 1);
            const float4 b = *reinterpret_cast<const float4 *>(sB + 4 * row);
            const float *cr = p.comps + (size_t)r * 3 * D + sub;
            const float4 ci = fr::ldg_f4(cr), cm = fr::ldg_f4(cr + D), ch = fr::ldg_f4(cr + 2 * D);
            const float4 ca = fr::ldg_f4(p.att + ((size_t)u * p.n_items + r) * D + sub);
            float4 x;
            x.x = b.x * ci.x + b.y * ca.x + b.z * cm.x + b.w * ch.x;
            x.y = b.x * ci.y + b.y * ca.y + b.z * cm.y + b.w * ch.y;
            x.z = b.x * ci.z + b.y * ca.z + b.z * cm.z + b.w * ch.z;
            x.w = b.x * ci.w + b.y * ca.w + b.z * cm.w + b.w * ch.w;
            *reinterpret_cast<float4 *>(sX + row * XS + sub) = x;
        }
    }
    __syncthreads();
    float x[IPT][D];
#pragma unroll
    for (int t = 0; t < IPT; ++t)
#pragma unroll
        for (int d = 0; d < D; d += 4) {
            const float4 v = *reinterpret_cast<const float4 *>(sX + (tid + t * SC_THREADS) * XS + d);
            x[t][d] = v.x, x[t][d + 1] = v.y, x[t][d + 2] = v.z, x[t][d + 3] = v.w;
        }
    float score[IPT];
#pragma unroll
    for (int t = 0; t < IPT; ++t) score[t] = 0.0f;
#pragma unroll 2
    for (int e = 0; e < D; ++e) {
        float h[IPT][4];
#pragma unroll
        for (int t = 0; t < IPT; ++t) h[t][0] = sH[e], h[t][1] = h[t][2] = h[t][3] = 0.0f;
#pragma unroll
        for (int d = 0; d < D; d += 4) {
            const float4 m = *reinterpret_cast<const float4 *>(sM + e * D + d);
#pragma unroll
            for (int t = 0; t < IPT; ++t) {
                h[t][0] = fmaf(m.x, x[t][d + 0], h[t][0]);
                h[t][1] = fmaf(m.y, x[t][d + 1], h[t][1]);
                h[t][2] = fmaf(m.z, x[t][d + 2], h[t][2]);
                h[t][3] = fmaf(m.w, x[t][d + 3], h[t][3]);
            }
        }
        const float w = sW[e];
#pragma unroll
        for (int t = 0; t < IPT; ++t)
            score[t] = fmaf(w, fmaxf((h[t][0] + h[t][1]) + (h[t][2] + h[t][3]), 0.0f), score[t]);
    }
    if (!TOPK) {
#pragma unroll
        for (int t = 0; t < IPT; ++t) {
            const int r = base + tid + t * SC_THREADS;
            if (r < p.n_items) p.scores[(size_t)u * p.n_items + r] = score[t];
        }
        return;
    }
    // ---- fused top-k: this CTA's 256 scores -> the kt best as keys; the [users, items] block never reaches HBM
    __syncthreads();                                   // every thread has its x rows in registers: the tile can be reused
    unsigned long long *key = reinterpret_cast<unsigned long long *>(sX);
    long long h0 = 0, h1 = 0;
    if (p.user_ids != nullptr) {
        const long long id = p.user_ids[u];
        h0 = p.hist_ptr[id];
        h1 = p.hist_ptr[id + 1];
    }
#pragma unroll
    for (int t = 0; t < IPT; ++t) {
        const int r = base + tid + t * SC_THREADS;
        bool dead = r >= p.n_items;
        if (!dead && h1 > h0) {                        // binary search in the user's sorted training items
            long long lo = h0, hi = h1;
            while (lo < hi) {
                const long long mid = (lo + hi) >> 1;
                if (p.hist_idx[mid] < r) lo = mid + 1; else hi = mid;
            }
            dead = lo < h1 && p.hist_idx[lo] == r;
        }
        key[tid + t * SC_THREADS] = dead ? 0ull : topk_key(score[t], r);
    }
    __syncthreads();
    bitonic_desc(key, SC_ITEMS, tid, SC_THREADS);
    if (tid < p.kt) p.cand[((size_t)u * gridDim.x + blockIdx.x) * p.kt + tid] = key[tid];
}

// One CTA per user: the n_cand = n_blocks * kt block winners -> the k best, (score desc, column asc).  The running
// best stays in the first k slots of a 2048-key shared tile while the candidates stream through the rest.
constexpr int MG_TILE = 2048;
__global__ void __launch_bounds__(256)
schgn_merge_topk_kernel(const unsigned long long *__restrict__ cand, int n_cand, int k, float *__restrict__ out_val,
                        int64_t *__restrict__ out_idx) {
    __shared__ unsigned long long key[MG_TILE];
    const int u = blockIdx.x, tid = threadIdx.x;
    const unsigned long long *c = cand + (size_t)u * n_cand;
    int pos = 0, keep = 0;
    while (pos < n_cand || keep == 0) {
        const int take = min(MG_TILE - keep, n_cand - pos);
        for (int i = tid; i < MG_TILE - keep; i += 256) key[keep + i] = i < take ? c[pos + i] : 0ull;
        __syncthreads();
        bitonic_desc(key, MG_TILE, tid, 256);
        pos += take;
        keep = k;
        if (take <= 0) break;
    }
    if (tid < k) {
        const unsigned long long kv = key[tid];
        out_val[(size_t)u * k + tid] = kv ? key_score(kv) : -INFINITY;
        out_idx[(size_t)u * k + tid] = kv ? (int64_t)(int)(~(unsigned)(kv & 0xffffffffull)) : -1;
    }
}

// ------------------------------------------------------------------------------------------------ candidate lists
// By-user evaluation: user u of a block has its own candidate list; pair q = ptr[u] - ptr[0] + k is its k-th candidate
// items[q].  The same per-pair arithmetic as above, with two changes:
//   * attend runs item-major over the block's pairs grouped by candidate item (a counting sort: count, scan, scatter),
//     one warp per item and 16 of its pairs per pass, so the gathered ingredient rows and their e^{2a} factors are
//     reused across the users that hold the item, as schgn_attend_kernel reuses them across a fixed 16-user block;
//   * the component softmax groups the logits of each user's OWN list: with L = the list's length, row r reads flat
//     entries 4r .. 4r+3 of the list's component-major [4, L] logit block, which is what the reference computes when
//     the list is scored as one batch (`.view(b, -1)` with b = L, schgn.py:198).
// A pair's result does not depend on which pass or slot it lands in (the reduce16 tree is the same for every slot), so
// the atomics' ordering of the scatter leaves every score bit-reproducible.
constexpr int PL_WARPS = 8;   // users per CTA of the count / scatter passes (one warp each)

// User u's pair range [b, e), or false when it is empty or leaves [0, n_pairs) (ptr not increasing), or the last list
// does not end at n_pairs.  This check is per list: with a decreasing ptr the lists that pass it can overlap (ptr =
// [0, 4, 2, 6] passes [0, 4) and [2, 6)), and the per-item counts then exceed n_pairs.  So once the count kernel has
// set FR_PAIRS_BAD_PTR for any list, the scatter and attend launches that follow it on the stream do nothing.
__device__ __forceinline__ bool list_range(const int64_t *ptr, int u, int32_t nu, int64_t n_pairs, int64_t &b, int64_t &e) {
    b = ptr[u] - ptr[0];
    e = ptr[u + 1] - ptr[0];
    return b >= 0 && e > b && e <= n_pairs && (u < nu - 1 || e == n_pairs);
}
__device__ __forceinline__ bool item_ok(int it, int32_t n_items) { return it >= 0 && it < n_items; }

// Validation + per-item pair counts.  status |= FR_PAIRS_BAD_PTR / FR_PAIRS_BAD_ITEM.
__global__ void __launch_bounds__(PL_WARPS * 32)
pairs_count_kernel(const int64_t *__restrict__ ptr, int32_t nu, int64_t n_pairs, const int32_t *__restrict__ items,
                   int32_t n_items, int32_t *__restrict__ cnt, int32_t *__restrict__ status) {
    const int u = blockIdx.x * PL_WARPS + (threadIdx.x >> 5), lane = threadIdx.x & 31;
    if (u >= nu) return;
    int64_t b, e;
    if (!list_range(ptr, u, nu, n_pairs, b, e)) {
        if (lane == 0) atomicOr(status, FR_PAIRS_BAD_PTR);
        return;
    }
    for (int64_t q = b + lane; q < e; q += 32) {
        const int it = items[q];
        if (item_ok(it, n_items)) atomicAdd(cnt + it, 1);
        else atomicOr(status, FR_PAIRS_BAD_ITEM);
    }
}

// Exclusive scan of cnt[0, n) in one CTA -> cnt (item_ptr, with cnt[n] = total) and cursor (a copy for the scatter).
__global__ void __launch_bounds__(1024) pairs_scan_kernel(int32_t *__restrict__ cnt, int32_t *__restrict__ cursor, int32_t n) {
    __shared__ int32_t s_warp[32];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int per = (n + 1023) / 1024, lo = min(n, tid * per), hi = min(n, lo + per);
    int sum = 0;
    for (int i = lo; i < hi; ++i) sum += cnt[i];
    int x = sum;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const int y = __shfl_up_sync(0xffffffffu, x, o);
        if (lane >= o) x += y;
    }
    if (lane == 31) s_warp[warp] = x;
    __syncthreads();
    if (warp == 0) {
        int w = s_warp[lane];
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const int y = __shfl_up_sync(0xffffffffu, w, o);
            if (lane >= o) w += y;
        }
        s_warp[lane] = w;
    }
    __syncthreads();
    int run = x - sum + (warp ? s_warp[warp - 1] : 0);
    for (int i = lo; i < hi; ++i) {
        const int c = cnt[i];
        cnt[i] = cursor[i] = run;
        run += c;
    }
    if (tid == 1023) cnt[n] = run;
}

// Pairs into their item's group as (pair, user); and the user factors e^{2 user_key}, e^{2 user_comp} -> uexp [nu][2][64].
__global__ void __launch_bounds__(PL_WARPS * 32)
pairs_scatter_kernel(const int64_t *__restrict__ ptr, int32_t nu, int64_t n_pairs, const int32_t *__restrict__ items,
                     int32_t n_items, const float *__restrict__ user_key, const float *__restrict__ user_comp,
                     const int32_t *__restrict__ status, int32_t *__restrict__ cursor, int2 *__restrict__ grp,
                     float *__restrict__ uexp) {
    const int u = blockIdx.x * PL_WARPS + (threadIdx.x >> 5), lane = threadIdx.x & 31;
    if (u >= nu || (*status & FR_PAIRS_BAD_PTR)) return;     // lists may overlap: the group offsets are not valid
    const int c2 = 2 * lane;
    const float2 k = *reinterpret_cast<const float2 *>(user_key + (size_t)u * D + c2);
    const float2 c = *reinterpret_cast<const float2 *>(user_comp + (size_t)u * D + c2);
    *reinterpret_cast<float2 *>(uexp + (size_t)u * 2 * D + c2) = make_float2(exp2x(k.x), exp2x(k.y));
    *reinterpret_cast<float2 *>(uexp + (size_t)u * 2 * D + D + c2) = make_float2(exp2x(c.x), exp2x(c.y));
    int64_t b, e;
    if (!list_range(ptr, u, nu, n_pairs, b, e)) return;
    for (int64_t q = b + lane; q < e; q += 32)
        if (item_ok(items[q], n_items)) grp[atomicAdd(cursor + items[q], 1)] = make_int2((int)q, u);
}

struct AttendPairsParams {
    const int64_t *ptr;
    const int32_t *item_ptr;
    const int2 *grp;
    const float *uexp;
    const int32_t *codes, *nums;
    const float *ingre_key, *ingre_final, *ingre_comp, *img_key, *comp_keys, *h_ingre, *h_comp;
    float *att, *logits;
    const int32_t *status;
    int32_t n_items, slots;
};

// schgn_attend_kernel's two passes and component logits for the pairs of one item, 16 per pass; writes att [q] and
// the logits into each pair's list block: logits[4 (ptr[u] - ptr[0]) + comp L + k].
__global__ void __launch_bounds__(ATT_WARPS * 32, 2) schgn_attend_pairs_kernel(const AttendPairsParams p) {
    __shared__ float s_u[ATT_WARPS][UB][D];   // per warp: e^{2 user_key} of the pass's users, then their e^{2 user_comp}
    __shared__ float s_logit[ATT_WARPS][UB][MAX_SLOTS];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int item = blockIdx.x * ATT_WARPS + warp;
    if (item >= p.n_items || (*p.status & FR_PAIRS_BAD_PTR)) return;   // grp was not filled
    const int g0 = p.item_ptr[item], g1 = p.item_ptr[item + 1];
    if (g0 == g1) return;
    const int n = max(0, min(p.nums[item], p.slots));
    const int code = lane < p.slots ? p.codes[(size_t)item * p.slots + lane] : 0;
    const int c2 = 2 * lane;
    const float2 pi = *reinterpret_cast<const float2 *>(p.img_key + (size_t)item * D + c2);
    const float2 hi = *reinterpret_cast<const float2 *>(p.h_ingre + c2);
    const float2 hc = *reinterpret_cast<const float2 *>(p.h_comp + c2);
    const float hi_sum = hi.x + hi.y, hc_sum = hc.x + hc.y;
    float(&su)[UB][D] = s_u[warp];

    for (int g = g0; g < g1; g += UB) {
        // lanes 2s and 2s+1 own slot s of the pass; slots past the group's end repeat slot 0 and write nothing
        const bool valid = g + (lane >> 1) < g1;
        const int2 pr = p.grp[valid ? g + (lane >> 1) : g];
        __syncwarp();                                  // the previous pass has finished reading su
#pragma unroll
        for (int s = 0; s < UB; ++s) {
            const int us = __shfl_sync(0xffffffffu, pr.y, 2 * s);
            *reinterpret_cast<float2 *>(&su[s][c2]) = __ldg(reinterpret_cast<const float2 *>(p.uexp + (size_t)us * 2 * D + c2));
        }
        __syncwarp();

        // pass 1: attention logits a[s][j]
        for (int j = 0; j < n; ++j) {
            const int c = __shfl_sync(0xffffffffu, code, j);
            const float2 pe = __ldg(reinterpret_cast<const float2 *>(p.ingre_key + (size_t)c * D + c2));
            const float ex = exp2x(pe.x + pi.x), ey = exp2x(pe.y + pi.y);
            float v[UB];
#pragma unroll
            for (int s = 0; s < UB; ++s) {
                const float2 uk = *reinterpret_cast<const float2 *>(&su[s][c2]);
                v[s] = fmaf(-2.0f, fmaf(hi.x, inv1p(ex, uk.x), hi.y * inv1p(ey, uk.y)), hi_sum);
            }
            const float tot = reduce16(v, lane);
            if (!(lane & 1)) s_logit[warp][lane >> 1][j] = tot;
        }
        __syncwarp();
#pragma unroll
        for (int s = 0; s < UB; ++s) {
            const int us = __shfl_sync(0xffffffffu, pr.y, 2 * s);
            *reinterpret_cast<float2 *>(&su[s][c2]) =
                __ldg(reinterpret_cast<const float2 *>(p.uexp + (size_t)us * 2 * D + D + c2));
        }

        // softmax over the recipe's real ingredients; lane j keeps A[s][j]
        float A[UB];
#pragma unroll
        for (int s = 0; s < UB; ++s) {
            const float x = lane < n ? s_logit[warp][s][lane] : -INFINITY;
            float m = x;
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, o));
            const float e = lane < n ? expf(x - m) : 0.0f;
            const float sum = fr::warp_sum(e);
            A[s] = n > 0 ? e / sum : 0.0f;
        }

        // pass 2: attended ingredient row and its image under W_att_comp's component half
        float2 att[UB], q[UB];
#pragma unroll
        for (int s = 0; s < UB; ++s) att[s] = q[s] = make_float2(0.0f, 0.0f);
        for (int j = 0; j < n; ++j) {
            const int c = __shfl_sync(0xffffffffu, code, j);
            const float2 ef = __ldg(reinterpret_cast<const float2 *>(p.ingre_final + (size_t)c * D + c2));
            const float2 qe = __ldg(reinterpret_cast<const float2 *>(p.ingre_comp + (size_t)c * D + c2));
#pragma unroll
            for (int s = 0; s < UB; ++s) {
                const float w = __shfl_sync(0xffffffffu, A[s], j);
                att[s].x = fmaf(w, ef.x, att[s].x);
                att[s].y = fmaf(w, ef.y, att[s].y);
                q[s].x = fmaf(w, qe.x, q[s].x);
                q[s].y = fmaf(w, qe.y, q[s].y);
            }
        }
#pragma unroll
        for (int s = 0; s < UB; ++s) {
            const int qs = __shfl_sync(0xffffffffu, pr.x, 2 * s);
            if (g + s < g1) *reinterpret_cast<float2 *>(p.att + (size_t)qs * D + c2) = att[s];
        }
        __syncwarp();                                  // su holds e^{2 user_comp} for every lane

        // component logits, reference order: item id, attended ingredients, image, health (the item's factors are
        // recomputed per pass: keeping them live across passes costs spills at two CTAs per SM)
        const float *ck = p.comp_keys + (size_t)item * 3 * D + c2;
        float2 k_item = *reinterpret_cast<const float2 *>(ck);
        float2 k_img = *reinterpret_cast<const float2 *>(ck + D);
        float2 k_hl = *reinterpret_cast<const float2 *>(ck + 2 * D);
        k_item = make_float2(exp2x(k_item.x), exp2x(k_item.y));
        k_img = make_float2(exp2x(k_img.x), exp2x(k_img.y));
        k_hl = make_float2(exp2x(k_hl.x), exp2x(k_hl.y));
        const int64_t ub = p.ptr[pr.y] - p.ptr[0], L = p.ptr[pr.y + 1] - p.ptr[pr.y];
        float *lg = p.logits + 4 * ub + (pr.x - ub);
#pragma unroll
        for (int comp = 0; comp < 4; ++comp) {
            float v[UB];
#pragma unroll
            for (int s = 0; s < UB; ++s) {
                const float2 uc = *reinterpret_cast<const float2 *>(&su[s][c2]);
                const float2 k = comp == 0   ? k_item
                                 : comp == 1 ? make_float2(exp2x(q[s].x), exp2x(q[s].y))
                                 : comp == 2 ? k_img
                                             : k_hl;
                v[s] = fmaf(-2.0f, fmaf(hc.x, inv1p(k.x, uc.x), hc.y * inv1p(k.y, uc.y)), hc_sum);
            }
            const float tot = reduce16(v, lane);
            if (!(lane & 1) && valid) lg[comp * L] = tot;
        }
    }
}

struct ScorePairsParams {
    const int64_t *ptr;
    const int32_t *items;
    const float *user_final, *user_hidden, *W_item, *W_prod, *w_out, *comps, *att, *logits;
    float *scores;
    int64_t n_pairs;
    int32_t nu, n_items;
};

// One CTA per user: M_u built once in shared memory, then the user's list in tiles of SC_ITEMS candidates with the
// tile body of schgn_score_kernel.  Candidate r's component weights: softmax of logits[4 (ptr[u] - ptr[0]) + 4r ..+3].
__global__ void __launch_bounds__(SC_THREADS) schgn_score_pairs_kernel(const ScorePairsParams p) {
    extern __shared__ __align__(16) float smem[];
    float *sX = smem;                    // [SC_ITEMS][XS]   x rows of the tile
    float *sM = sX + SC_ITEMS * XS;      // [D][D]           M_u = W_item + W_prod diag(u_final)
    float *sH = sM + D * D;              // [D]              user_hidden[u]
    float *sW = sH + D;                  // [D]              w_out
    float *sB = sW + D;                  // [SC_ITEMS][4]    component softmax weights
    const int u = blockIdx.x, tid = threadIdx.x;
    int64_t ub, ue;
    if (!list_range(p.ptr, u, p.nu, p.n_pairs, ub, ue)) return;      // reported by fr_schgn_attend_pairs
    const int L = (int)(ue - ub);
    for (int t = tid; t < D * D; t += SC_THREADS)
        sM[t] = fmaf(p.W_prod[t], p.user_final[(size_t)u * D + t % D], p.W_item[t]);
    if (tid < D) {
        sH[tid] = p.user_hidden[(size_t)u * D + tid];
        sW[tid] = p.w_out[tid];
    }
    const float *lg = p.logits + 4 * ub;
    const int32_t *it = p.items + ub;
    const float *att = p.att + ub * D;
    for (int base = 0; base < L; base += SC_ITEMS) {
        if (base) __syncthreads();       // every thread holds its previous x rows in registers: the tile is free
#pragma unroll
        for (int t = 0; t < IPT; ++t) {
            const int r = min(base + tid + t * SC_THREADS, L - 1);
            const float4 l = *reinterpret_cast<const float4 *>(lg + (size_t)4 * r);
            const float m = fmaxf(fmaxf(l.x, l.y), fmaxf(l.z, l.w));
            const float e0 = expf(l.x - m), e1 = expf(l.y - m), e2 = expf(l.z - m), e3 = expf(l.w - m);
            const float inv = 1.0f / (e0 + e1 + e2 + e3);
            *reinterpret_cast<float4 *>(sB + 4 * (tid + t * SC_THREADS)) = make_float4(e0 * inv, e1 * inv, e2 * inv, e3 * inv);
        }
        __syncthreads();
        {
            const int sub = (tid & 15) * 4, rr = tid >> 4;
#pragma unroll 4
            for (int row = rr; row < SC_ITEMS; row += SC_THREADS / 16) {
                const int r = min(base + row, L - 1);
                const int item = min(max(it[r], 0), p.n_items - 1);   // a bad id is reported by fr_schgn_attend_pairs
                const float4 b = *reinterpret_cast<const float4 *>(sB + 4 * row);
                const float *cr = p.comps + (size_t)item * 3 * D + sub;
                const float4 ci = fr::ldg_f4(cr), cm = fr::ldg_f4(cr + D), ch = fr::ldg_f4(cr + 2 * D);
                const float4 ca = fr::ldg_f4(att + (size_t)r * D + sub);
                float4 x;
                x.x = b.x * ci.x + b.y * ca.x + b.z * cm.x + b.w * ch.x;
                x.y = b.x * ci.y + b.y * ca.y + b.z * cm.y + b.w * ch.y;
                x.z = b.x * ci.z + b.y * ca.z + b.z * cm.z + b.w * ch.z;
                x.w = b.x * ci.w + b.y * ca.w + b.z * cm.w + b.w * ch.w;
                *reinterpret_cast<float4 *>(sX + row * XS + sub) = x;
            }
        }
        __syncthreads();
        float x[IPT][D];
#pragma unroll
        for (int t = 0; t < IPT; ++t)
#pragma unroll
            for (int d = 0; d < D; d += 4) {
                const float4 v = *reinterpret_cast<const float4 *>(sX + (tid + t * SC_THREADS) * XS + d);
                x[t][d] = v.x, x[t][d + 1] = v.y, x[t][d + 2] = v.z, x[t][d + 3] = v.w;
            }
        float score[IPT];
#pragma unroll
        for (int t = 0; t < IPT; ++t) score[t] = 0.0f;
#pragma unroll 2
        for (int e = 0; e < D; ++e) {
            float h[IPT][4];
#pragma unroll
            for (int t = 0; t < IPT; ++t) h[t][0] = sH[e], h[t][1] = h[t][2] = h[t][3] = 0.0f;
#pragma unroll
            for (int d = 0; d < D; d += 4) {
                const float4 m = *reinterpret_cast<const float4 *>(sM + e * D + d);
#pragma unroll
                for (int t = 0; t < IPT; ++t) {
                    h[t][0] = fmaf(m.x, x[t][d + 0], h[t][0]);
                    h[t][1] = fmaf(m.y, x[t][d + 1], h[t][1]);
                    h[t][2] = fmaf(m.z, x[t][d + 2], h[t][2]);
                    h[t][3] = fmaf(m.w, x[t][d + 3], h[t][3]);
                }
            }
            const float w = sW[e];
#pragma unroll
            for (int t = 0; t < IPT; ++t)
                score[t] = fmaf(w, fmaxf((h[t][0] + h[t][1]) + (h[t][2] + h[t][3]), 0.0f), score[t]);
        }
#pragma unroll
        for (int t = 0; t < IPT; ++t) {
            const int r = base + tid + t * SC_THREADS;
            if (r < L) p.scores[ub + r] = score[t];
        }
    }
}

// workspace of fr_schgn_attend_pairs: cnt [n_items + 1] | cursor [n_items] | grp [n_pairs] | uexp [nu][2][64]
struct PairsWs {
    int32_t *cnt, *cursor;
    int2 *grp;
    float *uexp;
    int64_t bytes;
};
inline int64_t align16(int64_t b) { return (b + 15) & ~int64_t(15); }
inline PairsWs pairs_ws(void *base, int32_t nu, int64_t n_pairs, int32_t n_items) {
    char *b = static_cast<char *>(base);
    PairsWs w;
    int64_t off = 0;
    w.cnt = reinterpret_cast<int32_t *>(b + off), off += align16(4 * ((int64_t)n_items + 1));
    w.cursor = reinterpret_cast<int32_t *>(b + off), off += align16(4 * (int64_t)n_items);
    w.grp = reinterpret_cast<int2 *>(b + off), off += align16(8 * n_pairs);
    w.uexp = reinterpret_cast<float *>(b + off), off += (int64_t)nu * 2 * D * 4;
    w.bytes = off;
    return w;
}

inline bool aligned16(const void *p) { return ((uintptr_t)p & 15) == 0; }

}  // namespace

extern "C" int fr_schgn_attend(const float *user_key, const float *user_comp, int32_t nu, const int32_t *codes,
                               int32_t slots, const int32_t *nums, int32_t n_items, const float *ingre_key,
                               const float *ingre_final, const float *ingre_comp, const float *img_key,
                               const float *comp_keys, const float *h_ingre, const float *h_comp, int32_t d,
                               float *att, float *logits, void *stream) {
    FR_REQUIRE(d == D, "fr_schgn_attend: embedding width %d unsupported (the model fixes 64)", d);
    FR_REQUIRE(nu >= 0 && n_items >= 0 && slots >= 1 && slots <= MAX_SLOTS,
               "fr_schgn_attend: bad extents (nu=%d, n_items=%d, slots=%d; at most %d slots)", nu, n_items, slots,
               MAX_SLOTS);
    if (nu == 0 || n_items == 0) return FR_OK;
    FR_REQUIRE(user_key && user_comp && codes && nums && ingre_key && ingre_final && ingre_comp && img_key &&
                   comp_keys && h_ingre && h_comp && att && logits,
               "fr_schgn_attend: null pointer");
    FR_REQUIRE((nu + UB - 1) / UB <= 65535, "fr_schgn_attend: at most %d users per call", 65535 * UB);
    AttendParams p{user_key, user_comp, codes,   nums, ingre_key, ingre_final, ingre_comp, img_key,
                   comp_keys, h_ingre,  h_comp, att,  logits,    nu,          n_items,    slots};
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    fr::LaunchTimer timer("schgn_attend", st);
    dim3 grid((n_items + ATT_WARPS - 1) / ATT_WARPS, (nu + UB - 1) / UB);
    schgn_attend_kernel<<<grid, ATT_WARPS * 32, 0, st>>>(p);
    return fr::check_launch("fr_schgn_attend");
}

extern "C" int fr_schgn_score(const float *user_final, const float *user_hidden, int32_t nu, const float *W_item,
                              const float *W_prod, const float *w_out, const float *comps, const float *att,
                              const float *logits, int32_t n_items, int32_t d, float *scores, void *stream) {
    FR_REQUIRE(d == D, "fr_schgn_score: embedding width %d unsupported (the model fixes 64)", d);
    FR_REQUIRE(nu >= 0 && nu <= 65535 && n_items >= 0, "fr_schgn_score: bad extents (nu=%d, n_items=%d)", nu, n_items);
    if (nu == 0 || n_items == 0) return FR_OK;
    FR_REQUIRE(user_final && user_hidden && W_item && W_prod && w_out && comps && att && logits && scores,
               "fr_schgn_score: null pointer");
    ScoreParams p{user_final, user_hidden, W_item, W_prod, w_out, comps, att, logits, scores, nu, n_items,
                  nullptr, nullptr, nullptr, nullptr, 0};
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    fr::LaunchTimer timer("schgn_score", st);
    static bool configured = false;
    if (!configured) {
        if (cudaFuncSetAttribute(schgn_score_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, SC_SMEM) != cudaSuccess)
            return fr::check_launch("fr_schgn_score (shared-memory opt-in)");
        configured = true;
    }
    dim3 grid((n_items + SC_ITEMS - 1) / SC_ITEMS, nu);
    schgn_score_kernel<false><<<grid, SC_THREADS, SC_SMEM, st>>>(p);
    return fr::check_launch("fr_schgn_score");
}

extern "C" int64_t fr_schgn_score_topk_ws_bytes(int32_t nu, int32_t n_items, int32_t k) {
    return (int64_t)nu * ((n_items + SC_ITEMS - 1) / SC_ITEMS) * k * 8;
}

extern "C" int fr_schgn_score_topk(const float *user_final, const float *user_hidden, int32_t nu, const float *W_item,
                                   const float *W_prod, const float *w_out, const float *comps, const float *att,
                                   const float *logits, int32_t n_items, int32_t d, const int64_t *user_ids,
                                   const int64_t *hist_ptr, const int32_t *hist_idx, int32_t k, void *ws, float *out_val,
                                   int64_t *out_idx, void *stream) {
    FR_REQUIRE(d == D, "fr_schgn_score_topk: embedding width %d unsupported (the model fixes 64)", d);
    FR_REQUIRE(nu >= 0 && nu <= 65535 && n_items >= 0, "fr_schgn_score_topk: bad extents (nu=%d, n_items=%d)", nu, n_items);
    FR_REQUIRE(k >= 1 && k <= 64, "fr_schgn_score_topk: k=%d out of [1, 64]", k);
    if (nu == 0) return FR_OK;
    FR_REQUIRE(n_items > 0, "fr_schgn_score_topk: no items");
    FR_REQUIRE(user_final && user_hidden && W_item && W_prod && w_out && comps && att && logits && ws && out_val && out_idx,
               "fr_schgn_score_topk: null pointer");
    FR_REQUIRE((user_ids == nullptr) == (hist_ptr == nullptr) && (user_ids == nullptr) == (hist_idx == nullptr),
               "fr_schgn_score_topk: user_ids / hist_ptr / hist_idx go together");
    FR_REQUIRE(((uintptr_t)ws & 7) == 0, "fr_schgn_score_topk: workspace must be 8-byte aligned");
    ScoreParams p{user_final, user_hidden, W_item, W_prod, w_out, comps, att, logits, nullptr, nu, n_items,
                  reinterpret_cast<unsigned long long *>(ws), user_ids, hist_ptr, hist_idx, k};
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    static bool configured = false;
    if (!configured) {
        if (cudaFuncSetAttribute(schgn_score_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, SC_SMEM) != cudaSuccess)
            return fr::check_launch("fr_schgn_score_topk (shared-memory opt-in)");
        configured = true;
    }
    const int n_blk = (n_items + SC_ITEMS - 1) / SC_ITEMS;
    {
        fr::LaunchTimer timer("schgn_score<topk>", st);
        dim3 grid(n_blk, nu);
        schgn_score_kernel<true><<<grid, SC_THREADS, SC_SMEM, st>>>(p);
        if (int rc = fr::check_launch("fr_schgn_score_topk(score)")) return rc;
    }
    fr::LaunchTimer timer("schgn_merge_topk", st);
    schgn_merge_topk_kernel<<<nu, 256, 0, st>>>(p.cand, n_blk * k, k, out_val, out_idx);
    return fr::check_launch("fr_schgn_score_topk(merge)");
}

extern "C" int64_t fr_schgn_attend_pairs_ws_bytes(int32_t nu, int64_t n_pairs, int32_t n_items) {
    if (nu < 0 || n_pairs < 0 || n_items < 0) return -1;
    return pairs_ws(nullptr, nu, n_pairs, n_items).bytes;
}

extern "C" int fr_schgn_attend_pairs(const float *user_key, const float *user_comp, int32_t nu, const int64_t *ptr,
                                     const int32_t *items, int64_t n_pairs, const int32_t *codes, int32_t slots,
                                     const int32_t *nums, int32_t n_items, const float *ingre_key,
                                     const float *ingre_final, const float *ingre_comp, const float *img_key,
                                     const float *comp_keys, const float *h_ingre, const float *h_comp, int32_t d,
                                     void *ws, int64_t ws_bytes, float *att, float *logits, int32_t *status,
                                     void *stream) {
    FR_REQUIRE(d == D, "fr_schgn_attend_pairs: embedding width %d unsupported (the model fixes 64)", d);
    FR_REQUIRE(nu >= 0 && n_items >= 1 && slots >= 1 && slots <= MAX_SLOTS,
               "fr_schgn_attend_pairs: bad extents (nu=%d, n_items=%d, slots=%d; at most %d slots)", nu, n_items, slots,
               MAX_SLOTS);
    if (nu == 0) return FR_OK;
    FR_REQUIRE(n_pairs >= nu && n_pairs <= INT32_MAX,
               "fr_schgn_attend_pairs: %lld pairs for %d users (every list non-empty, at most 2^31 - 1 pairs per call)",
               (long long)n_pairs, nu);
    FR_REQUIRE(user_key && user_comp && ptr && items && codes && nums && ingre_key && ingre_final && ingre_comp &&
                   img_key && comp_keys && h_ingre && h_comp && ws && att && logits && status,
               "fr_schgn_attend_pairs: null pointer");
    FR_REQUIRE(aligned16(user_key) && aligned16(user_comp) && aligned16(ingre_key) && aligned16(ingre_final) &&
                   aligned16(ingre_comp) && aligned16(img_key) && aligned16(comp_keys) && aligned16(h_ingre) &&
                   aligned16(h_comp) && aligned16(ws) && aligned16(att) && aligned16(logits) && ((uintptr_t)ptr & 7) == 0 &&
                   ((uintptr_t)items & 3) == 0 && ((uintptr_t)status & 3) == 0,
               "fr_schgn_attend_pairs: tables must be 16-byte aligned (ptr 8-byte, items / status 4-byte)");
    const PairsWs w = pairs_ws(ws, nu, n_pairs, n_items);
    FR_REQUIRE(ws_bytes >= w.bytes, "fr_schgn_attend_pairs: workspace of %lld bytes, %lld needed", (long long)ws_bytes,
               (long long)w.bytes);
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    const int ublocks = (nu + PL_WARPS - 1) / PL_WARPS;
    {
        fr::LaunchTimer timer("schgn_pairs_group", st);
        if (cudaMemsetAsync(w.cnt, 0, 4 * ((int64_t)n_items + 1), st) != cudaSuccess)
            return fr::check_launch("fr_schgn_attend_pairs (memset)");
        pairs_count_kernel<<<ublocks, PL_WARPS * 32, 0, st>>>(ptr, nu, n_pairs, items, n_items, w.cnt, status);
        if (int rc = fr::check_launch("fr_schgn_attend_pairs(count)")) return rc;
        pairs_scan_kernel<<<1, 1024, 0, st>>>(w.cnt, w.cursor, n_items);
        if (int rc = fr::check_launch("fr_schgn_attend_pairs(scan)")) return rc;
        pairs_scatter_kernel<<<ublocks, PL_WARPS * 32, 0, st>>>(ptr, nu, n_pairs, items, n_items, user_key, user_comp,
                                                                 status, w.cursor, w.grp, w.uexp);
        if (int rc = fr::check_launch("fr_schgn_attend_pairs(scatter)")) return rc;
    }
    AttendPairsParams p{ptr,     w.cnt,       w.grp,      w.uexp,  codes,     nums,   ingre_key, ingre_final,
                        ingre_comp, img_key, comp_keys, h_ingre, h_comp, att, logits, status, n_items, slots};
    fr::LaunchTimer timer("schgn_attend_pairs", st);
    schgn_attend_pairs_kernel<<<(n_items + ATT_WARPS - 1) / ATT_WARPS, ATT_WARPS * 32, 0, st>>>(p);
    return fr::check_launch("fr_schgn_attend_pairs");
}

extern "C" int fr_schgn_score_pairs(const float *user_final, const float *user_hidden, int32_t nu, const int64_t *ptr,
                                    const int32_t *items, int64_t n_pairs, const float *W_item, const float *W_prod,
                                    const float *w_out, const float *comps, const float *att, const float *logits,
                                    int32_t n_items, int32_t d, float *scores, void *stream) {
    FR_REQUIRE(d == D, "fr_schgn_score_pairs: embedding width %d unsupported (the model fixes 64)", d);
    FR_REQUIRE(nu >= 0 && n_items >= 1, "fr_schgn_score_pairs: bad extents (nu=%d, n_items=%d)", nu, n_items);
    if (nu == 0) return FR_OK;
    FR_REQUIRE(n_pairs >= nu && n_pairs <= INT32_MAX, "fr_schgn_score_pairs: %lld pairs for %d users", (long long)n_pairs, nu);
    FR_REQUIRE(user_final && user_hidden && ptr && items && W_item && W_prod && w_out && comps && att && logits && scores,
               "fr_schgn_score_pairs: null pointer");
    FR_REQUIRE(aligned16(user_final) && aligned16(user_hidden) && aligned16(W_item) && aligned16(W_prod) &&
                   aligned16(w_out) && aligned16(comps) && aligned16(att) && aligned16(logits) &&
                   ((uintptr_t)ptr & 7) == 0 && ((uintptr_t)items & 3) == 0 && ((uintptr_t)scores & 3) == 0,
               "fr_schgn_score_pairs: tables must be 16-byte aligned (ptr 8-byte, items / scores 4-byte)");
    ScorePairsParams p{ptr, items, user_final, user_hidden, W_item, W_prod, w_out, comps, att, logits, scores, n_pairs,
                       nu, n_items};
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    fr::LaunchTimer timer("schgn_score_pairs", st);
    static bool configured = false;
    if (!configured) {
        if (cudaFuncSetAttribute(schgn_score_pairs_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, SC_SMEM) != cudaSuccess)
            return fr::check_launch("fr_schgn_score_pairs (shared-memory opt-in)");
        configured = true;
    }
    schgn_score_pairs_kernel<<<nu, SC_THREADS, SC_SMEM, st>>>(p);
    return fr::check_launch("fr_schgn_score_pairs");
}
