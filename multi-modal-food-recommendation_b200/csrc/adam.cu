// Dense Adam over many tensors in ONE launch (SURVEY.md 8f-1).
//
// The reference trains with `optim.Adam(model.parameters())` (FoodRec/common/trainer.py:144): dense gradients, dense
// state -- a row whose gradient is zero still moves while its first moment decays, so a sparse update would change
// results.  For HealthRec the `freeze=False` raw-feature tables (cikm_model.py:83,87: [I, 2048..4096] + [I, 384..512])
// make this pass ~200 M parameters = 5.6 GB of HBM traffic per step: p, g, m, v read and p, m, v written once, 128-bit
// accesses, nothing else -- purely HBM-bound.  One persistent grid walks 4096-element chunks of all tensors (the table
// of pointers travels in the kernel parameters); the step counter lives on the device (a one-thread prologue advances
// it and derives the bias corrections in double), so the launch pair can be captured in a CUDA graph and replayed.
// Arithmetic and its order follow torch.optim.Adam (`_single_tensor_adam`, amsgrad = False, weight_decay = 0):
//   m += (1 - b1) (g - m);  v = v b2 + ((1 - b2) g) g;  p += -(lr / (1 - b1^t)) * (m / (sqrt(v) / sqrt(1 - b2^t) + eps))
#include <algorithm>

#include "common.cuh"

namespace {

constexpr int kThreads = 256;
constexpr int kChunk = kThreads * 4 * 4;      // elements per block iteration: 4 float4 per thread

struct Tensors {
    float *p[FR_ADAM_MAX_TENSORS];
    const float *g[FR_ADAM_MAX_TENSORS];
    float *m[FR_ADAM_MAX_TENSORS];
    float *v[FR_ADAM_MAX_TENSORS];
    long long chunk_end[FR_ADAM_MAX_TENSORS];  // exclusive prefix of chunk counts (tensor t owns chunks [end[t-1], end[t]))
    long long n[FR_ADAM_MAX_TENSORS];
    int count;
};

__global__ void adam_prepare_kernel(int *step, float *scal, double lr, double b1, double b2) {
    const int t = *step + 1;
    *step = t;
    const double bc1 = 1.0 - pow(b1, (double)t), bc2 = 1.0 - pow(b2, (double)t);
    scal[0] = (float)(-lr / bc1);              // -step_size
    scal[1] = (float)sqrt(bc2);                // bias_correction2_sqrt
}

__device__ __forceinline__ void adam1(float &p, float g, float &m, float &v, float neg_step, float bc2s, float omb1,
                                      float b2, float omb2, float eps) {
    m = m + omb1 * (g - m);
    v = v * b2 + (omb2 * g) * g;
    const float denom = sqrtf(v) / bc2s + eps;
    p = p + neg_step * (m / denom);
}

__global__ void __launch_bounds__(kThreads)
adam_multi_kernel(const __grid_constant__ Tensors T, const float *__restrict__ scal, float omb1, float b2, float omb2, float eps) {
    // (1 - beta) arrives rounded from DOUBLE, as torch passes it: 1 - 0.999f evaluated in fp32 is off by 1.3e-5 relative
    const float neg_step = __ldg(scal), bc2s = __ldg(scal + 1);
    const long long total = T.chunk_end[T.count - 1];
    for (long long c = blockIdx.x; c < total; c += gridDim.x) {
        int lo = 0, hi = T.count - 1;          // first tensor whose chunk range ends after c
        while (lo < hi) {
            const int mid = (lo + hi) >> 1;
            if (T.chunk_end[mid] > c) hi = mid; else lo = mid + 1;
        }
        const long long c0 = lo ? T.chunk_end[lo - 1] : 0;
        const long long base = (c - c0) * kChunk, n = T.n[lo];
        float *__restrict__ p = T.p[lo] + base;
        const float *__restrict__ g = T.g[lo] + base;
        float *__restrict__ m = T.m[lo] + base;
        float *__restrict__ v = T.v[lo] + base;
        const long long left = n - base;
        if (left >= kChunk && ((((uintptr_t)p | (uintptr_t)g | (uintptr_t)m | (uintptr_t)v) & 15) == 0)) {
            float4 P[4], G[4], M[4], V[4];
#pragma unroll
            for (int u = 0; u < 4; ++u) {       // all loads of the chunk in flight before the first use
                const int o = (u * kThreads + threadIdx.x) * 4;
                P[u] = *reinterpret_cast<const float4 *>(p + o);
                G[u] = __ldcs(reinterpret_cast<const float4 *>(g + o));      // gradients are read once: streaming
                M[u] = *reinterpret_cast<const float4 *>(m + o);
                V[u] = *reinterpret_cast<const float4 *>(v + o);
            }
#pragma unroll
            for (int u = 0; u < 4; ++u) {
                const int o = (u * kThreads + threadIdx.x) * 4;
                adam1(P[u].x, G[u].x, M[u].x, V[u].x, neg_step, bc2s, omb1, b2, omb2, eps);
                adam1(P[u].y, G[u].y, M[u].y, V[u].y, neg_step, bc2s, omb1, b2, omb2, eps);
                adam1(P[u].z, G[u].z, M[u].z, V[u].z, neg_step, bc2s, omb1, b2, omb2, eps);
                adam1(P[u].w, G[u].w, M[u].w, V[u].w, neg_step, bc2s, omb1, b2, omb2, eps);
                *reinterpret_cast<float4 *>(p + o) = P[u];
                *reinterpret_cast<float4 *>(m + o) = M[u];
                *reinterpret_cast<float4 *>(v + o) = V[u];
            }
        } else {
            for (long long i = threadIdx.x; i < min(left, (long long)kChunk); i += kThreads) {
                float pp = p[i], mm = m[i], vv = v[i];
                adam1(pp, g[i], mm, vv, neg_step, bc2s, omb1, b2, omb2, eps);
                p[i] = pp;
                m[i] = mm;
                v[i] = vv;
            }
        }
    }
}

}  // namespace

extern "C" int fr_adam_step(const fr_adam_tensor *tensors_host, int32_t n_tensors, double lr, double beta1, double beta2,
                            double eps, int32_t *step_dev, float *scalars_dev, void *stream) {
    FR_REQUIRE(n_tensors >= 0 && (n_tensors == 0 || tensors_host) && step_dev && scalars_dev, "fr_adam_step: bad argument");
    FR_REQUIRE(lr >= 0.0 && beta1 >= 0.0 && beta1 < 1.0 && beta2 >= 0.0 && beta2 < 1.0 && eps >= 0.0,
               "fr_adam_step: lr=%g betas=(%g, %g) eps=%g", lr, beta1, beta2, eps);
    // every tensor is checked before anything is launched: a rejected call leaves the parameters, the moments and the
    // step counter as they were
    for (int32_t t = 0; t < n_tensors; ++t) {
        const fr_adam_tensor &h = tensors_host[t];
        FR_REQUIRE(h.n >= 0, "fr_adam_step: tensor %d has a negative extent", t);
        FR_REQUIRE(h.n == 0 || (h.param && h.grad && h.exp_avg && h.exp_avg_sq), "fr_adam_step: tensor %d: null pointer", t);
    }
    cudaStream_t st = (cudaStream_t)stream;
    {
        fr::LaunchTimer _lt("adam_prepare_kernel", st);
        adam_prepare_kernel<<<1, 1, 0, st>>>(step_dev, scalars_dev, lr, beta1, beta2);
        if (int rc = fr::check_launch("fr_adam_step/prepare")) return rc;
    }
    // one cursor across the launches: each non-empty tensor lands in exactly one batch of <= FR_ADAM_MAX_TENSORS
    for (int32_t t = 0; t < n_tensors;) {
        Tensors T;
        T.count = 0;
        long long chunks = 0;
        for (; t < n_tensors && T.count < FR_ADAM_MAX_TENSORS; ++t) {
            const fr_adam_tensor &h = tensors_host[t];
            if (h.n == 0) continue;
            const int k = T.count++;
            T.p[k] = h.param;
            T.g[k] = h.grad;
            T.m[k] = h.exp_avg;
            T.v[k] = h.exp_avg_sq;
            T.n[k] = h.n;
            chunks += (h.n + kChunk - 1) / kChunk;
            T.chunk_end[k] = chunks;
        }
        if (T.count == 0) continue;
        for (int k = T.count; k < FR_ADAM_MAX_TENSORS; ++k) {
            T.p[k] = nullptr; T.g[k] = nullptr; T.m[k] = nullptr; T.v[k] = nullptr; T.n[k] = 0; T.chunk_end[k] = chunks;
        }
        const unsigned grid = (unsigned)std::min<long long>(chunks, (long long)fr::num_sms() * 8);
        fr::LaunchTimer _lt("adam_multi_kernel", st);
        adam_multi_kernel<<<grid, kThreads, 0, st>>>(T, scalars_dev, (float)(1.0 - beta1), (float)beta2, (float)(1.0 - beta2), (float)eps);
        if (int rc = fr::check_launch("fr_adam_step")) return rc;
    }
    return FR_OK;
}
