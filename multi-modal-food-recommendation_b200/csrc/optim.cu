// Dense optimizer steps over many tensors in ONE launch (SURVEY.md 8f-1): Adam, SGD, Adagrad and RMSprop, the learners
// of the reference trainer's optimizer factory (FoodRec/common/trainer.py:137-154).
//
// The reference trains with `optim.Adam(model.parameters())` (FoodRec/common/trainer.py:144): dense gradients, dense
// state -- a row whose gradient is zero still moves while its first moment decays, so a sparse update would change
// results.  For HealthRec the `freeze=False` raw-feature tables (cikm_model.py:83,87: [I, 2048..4096] + [I, 384..512])
// make this pass ~200 M parameters = 5.6 GB of HBM traffic per step: p, g, m, v read and p, m, v written once, 128-bit
// accesses, nothing else -- purely HBM-bound.  One persistent grid walks 4096-element chunks of all tensors (the table
// of pointers travels in the kernel parameters); the step counter and the learning rate live on the device (a
// one-thread prologue reads them and derives the step's scalars in double), so the launch pair can be captured in a
// CUDA graph and replayed, and an lr schedule reaches the replays through the device scalar.
// Arithmetic and its order follow torch 2.11's `_single_tensor_*` functions (options the factory never sets at their
// defaults); with weight decay the gradient is first replaced by g' = g + wd p (`grad.add(param, alpha=wd)`):
//   Adam     m += (1 - b1) (g' - m);  v = v b2 + ((1 - b2) g') g';  p += -(lr / (1 - b1^t)) * (m / (sqrt(v) / sqrt(1 - b2^t) + eps))
//   SGD      p += (-lr) g'
//   Adagrad  s += g' g';  p += (-lr) (g' / (sqrt(s) + eps))
//   RMSprop  a = a alpha + ((1 - alpha) g') g';  p += (-lr) (g' / (sqrt(a) + eps))
#include <algorithm>
#include <vector>

#include "common.cuh"

namespace {

constexpr int kThreads = 256;
constexpr int kChunk = kThreads * 4 * 4;      // elements per block iteration: 4 float4 per thread

struct Tensors {
    float *p[FR_ADAM_MAX_TENSORS];
    const float *g[FR_ADAM_MAX_TENSORS];
    float *s0[FR_ADAM_MAX_TENSORS];
    float *s1[FR_ADAM_MAX_TENSORS];
    long long chunk_end[FR_ADAM_MAX_TENSORS];  // exclusive prefix of chunk counts (tensor t owns chunks [end[t-1], end[t]))
    long long n[FR_ADAM_MAX_TENSORS];
    int count;
};

// Hyper-parameters rounded to fp32 where torch rounds them.  (1 - beta) arrives rounded from DOUBLE, as torch passes
// it: 1 - 0.999f evaluated in fp32 is off by 1.3e-5 relative.
struct Coef {
    float omb1;       // Adam: 1 - beta1
    float decay;      // Adam: beta2; RMSprop: alpha
    float om_decay;   // Adam: 1 - beta2; RMSprop: 1 - alpha
    float eps;
    float wd;
};

constexpr int n_state(int R) { return R == FR_OPTIM_ADAM ? 2 : R == FR_OPTIM_SGD ? 0 : 1; }

// scal[0] = the (negative) step size, scal[1] = sqrt(1 - b2^t) (Adam).  A learning rate that is negative or NaN
// rejects the call: nothing is advanced and scal[0] = NaN tells the update launches to write nothing.
template <int R>
__global__ void optim_prepare_kernel(const double *lr_dev, double lr, int *step, float *scal, double b1, double b2) {
    const int t = step ? *step + 1 : 0;       // both loads in flight before the first branch on them
    if (lr_dev) lr = *lr_dev;
    if (!(lr >= 0.0)) {
        scal[0] = __int_as_float(0x7fc00000);
        return;
    }
    if (step) *step = t;
    if (R == FR_OPTIM_ADAM) {
        const double bc1 = 1.0 - pow(b1, (double)t), bc2 = 1.0 - pow(b2, (double)t);
        scal[0] = (float)(-lr / bc1);          // -step_size
        scal[1] = (float)sqrt(bc2);            // bias_correction2_sqrt
    } else {
        scal[0] = (float)(-lr);                // Adagrad: clr = lr / (1 + (t - 1) lr_decay) = lr at lr_decay = 0
    }
}

template <int R, bool WD>
__device__ __forceinline__ void update1(float &p, float g, float &s0, float &s1, float neg_step, float bc2s, const Coef &k) {
    if (WD) g = g + k.wd * p;                                // grad.add(param, alpha=weight_decay)
    if (R == FR_OPTIM_ADAM) {
        s0 = s0 + k.omb1 * (g - s0);                         // exp_avg.lerp_(grad, 1 - beta1)
        s1 = s1 * k.decay + (k.om_decay * g) * g;            // exp_avg_sq.mul_(beta2).addcmul_(grad, grad, 1 - beta2)
        const float denom = sqrtf(s1) / bc2s + k.eps;
        p = p + neg_step * (s0 / denom);
    } else if (R == FR_OPTIM_SGD) {
        p = p + neg_step * g;                                // param.add_(grad, alpha=-lr)
    } else if (R == FR_OPTIM_ADAGRAD) {
        s0 = s0 + g * g;                                     // state_sum.addcmul_(grad, grad, value=1)
        p = p + neg_step * (g / (sqrtf(s0) + k.eps));        // param.addcdiv_(grad, std, value=-clr)
    } else {
        s0 = s0 * k.decay + (k.om_decay * g) * g;            // square_avg.mul_(alpha).addcmul_(grad, grad, 1 - alpha)
        p = p + neg_step * (g / (sqrtf(s0) + k.eps));        // param.addcdiv_(grad, avg, value=-lr)
    }
}

template <int R, bool WD>
__device__ __forceinline__ void update4(float4 &p, const float4 &g, float4 &s0, float4 &s1, float neg_step, float bc2s,
                                        const Coef &k) {
    update1<R, WD>(p.x, g.x, s0.x, s1.x, neg_step, bc2s, k);
    update1<R, WD>(p.y, g.y, s0.y, s1.y, neg_step, bc2s, k);
    update1<R, WD>(p.z, g.z, s0.z, s1.z, neg_step, bc2s, k);
    update1<R, WD>(p.w, g.w, s0.w, s1.w, neg_step, bc2s, k);
}

// WD: weight decay is on (a separate instantiation, so the kernels without it carry no per-element test)
template <int R, bool WD>
__global__ void __launch_bounds__(kThreads)
optim_multi_kernel(const __grid_constant__ Tensors T, const float *__restrict__ scal, const Coef k) {
    constexpr int NS = n_state(R);
    const float neg_step = __ldg(scal), bc2s = R == FR_OPTIM_ADAM ? __ldg(scal + 1) : 1.f;
    if (neg_step != neg_step) return;          // the prologue rejected the learning rate
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
        float *__restrict__ s0 = NS > 0 ? T.s0[lo] + base : nullptr;
        float *__restrict__ s1 = NS > 1 ? T.s1[lo] + base : nullptr;
        const long long left = n - base;
        if (left >= kChunk && ((((uintptr_t)p | (uintptr_t)g | (uintptr_t)s0 | (uintptr_t)s1) & 15) == 0)) {
            float4 P[4], G[4], S0[4], S1[4];
#pragma unroll
            for (int u = 0; u < 4; ++u) {       // all loads of the chunk in flight before the first use
                const int o = (u * kThreads + threadIdx.x) * 4;
                P[u] = *reinterpret_cast<const float4 *>(p + o);
                G[u] = __ldcs(reinterpret_cast<const float4 *>(g + o));      // gradients are read once: streaming
                if (NS > 0) S0[u] = *reinterpret_cast<const float4 *>(s0 + o);
                if (NS > 1) S1[u] = *reinterpret_cast<const float4 *>(s1 + o);
            }
#pragma unroll
            for (int u = 0; u < 4; ++u) {
                const int o = (u * kThreads + threadIdx.x) * 4;
                update4<R, WD>(P[u], G[u], S0[u], S1[u], neg_step, bc2s, k);
                *reinterpret_cast<float4 *>(p + o) = P[u];
                if (NS > 0) *reinterpret_cast<float4 *>(s0 + o) = S0[u];
                if (NS > 1) *reinterpret_cast<float4 *>(s1 + o) = S1[u];
            }
        } else {
            for (long long i = threadIdx.x; i < min(left, (long long)kChunk); i += kThreads) {
                float pp = p[i], a = NS > 0 ? s0[i] : 0.f, b = NS > 1 ? s1[i] : 0.f;
                update1<R, WD>(pp, g[i], a, b, neg_step, bc2s, k);
                p[i] = pp;
                if (NS > 0) s0[i] = a;
                if (NS > 1) s1[i] = b;
            }
        }
    }
}

const char *const kPrepareName[] = {"adam_prepare_kernel", "sgd_prepare_kernel", "adagrad_prepare_kernel",
                                    "rmsprop_prepare_kernel"};
const char *const kMultiName[] = {"adam_multi_kernel", "sgd_multi_kernel", "adagrad_multi_kernel",
                                  "rmsprop_multi_kernel"};

// Launches one validated call: the prologue, then one cursor across the launches, so each non-empty tensor lands in
// exactly one batch of <= FR_ADAM_MAX_TENSORS.  The learning rate is *lr_dev when lr_dev is set, else `lr`.
template <int R>
int launch(const fr_optim_tensor *ts, int32_t n_tensors, const fr_optim_hyper &h, const double *lr_dev, double lr,
           int32_t *step_dev, float *scalars_dev, cudaStream_t st, const char *who) {
    {
        fr::LaunchTimer _lt(kPrepareName[R], st);
        optim_prepare_kernel<R><<<1, 1, 0, st>>>(lr_dev, lr, step_dev, scalars_dev, h.beta1, R == FR_OPTIM_ADAM ? h.beta2 : 0.0);
        if (int rc = fr::check_launch(who)) return rc;
    }
    Coef k;
    k.omb1 = (float)(1.0 - h.beta1);
    k.decay = (float)(R == FR_OPTIM_ADAM ? h.beta2 : h.alpha);
    k.om_decay = (float)(1.0 - (R == FR_OPTIM_ADAM ? h.beta2 : h.alpha));
    k.eps = (float)h.eps;
    k.wd = (float)h.weight_decay;
    for (int32_t t = 0; t < n_tensors;) {
        Tensors T;
        T.count = 0;
        long long chunks = 0;
        for (; t < n_tensors && T.count < FR_ADAM_MAX_TENSORS; ++t) {
            const fr_optim_tensor &x = ts[t];
            if (x.n == 0) continue;
            const int c = T.count++;
            T.p[c] = x.param;
            T.g[c] = x.grad;
            T.s0[c] = n_state(R) > 0 ? x.state0 : nullptr;
            T.s1[c] = n_state(R) > 1 ? x.state1 : nullptr;
            T.n[c] = x.n;
            chunks += (x.n + kChunk - 1) / kChunk;
            T.chunk_end[c] = chunks;
        }
        if (T.count == 0) continue;
        for (int c = T.count; c < FR_ADAM_MAX_TENSORS; ++c) {
            T.p[c] = nullptr; T.g[c] = nullptr; T.s0[c] = nullptr; T.s1[c] = nullptr; T.n[c] = 0; T.chunk_end[c] = chunks;
        }
        const unsigned grid = (unsigned)std::min<long long>(chunks, (long long)fr::num_sms() * 8);
        fr::LaunchTimer _lt(kMultiName[R], st);
        if (k.wd != 0.f) optim_multi_kernel<R, true><<<grid, kThreads, 0, st>>>(T, scalars_dev, k);
        else optim_multi_kernel<R, false><<<grid, kThreads, 0, st>>>(T, scalars_dev, k);
        if (int rc = fr::check_launch(who)) return rc;
    }
    return FR_OK;
}

int dispatch(int32_t rule, const fr_optim_tensor *ts, int32_t n_tensors, const fr_optim_hyper &h, const double *lr_dev,
             double lr, int32_t *step_dev, float *scalars_dev, void *stream, const char *who) {
    cudaStream_t st = (cudaStream_t)stream;
    switch (rule) {
        case FR_OPTIM_ADAM: return launch<FR_OPTIM_ADAM>(ts, n_tensors, h, lr_dev, lr, step_dev, scalars_dev, st, who);
        case FR_OPTIM_SGD: return launch<FR_OPTIM_SGD>(ts, n_tensors, h, lr_dev, lr, step_dev, scalars_dev, st, who);
        case FR_OPTIM_ADAGRAD: return launch<FR_OPTIM_ADAGRAD>(ts, n_tensors, h, lr_dev, lr, step_dev, scalars_dev, st, who);
        default: return launch<FR_OPTIM_RMSPROP>(ts, n_tensors, h, lr_dev, lr, step_dev, scalars_dev, st, who);
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
    std::vector<fr_optim_tensor> ts(n_tensors);
    for (int32_t t = 0; t < n_tensors; ++t) {
        const fr_adam_tensor &h = tensors_host[t];
        FR_REQUIRE(h.n >= 0, "fr_adam_step: tensor %d has a negative extent", t);
        FR_REQUIRE(h.n == 0 || (h.param && h.grad && h.exp_avg && h.exp_avg_sq), "fr_adam_step: tensor %d: null pointer", t);
        ts[t] = fr_optim_tensor{h.param, h.grad, h.exp_avg, h.exp_avg_sq, h.n};
    }
    const fr_optim_hyper hyper{beta1, beta2, 0.0, eps, 0.0};
    return dispatch(FR_OPTIM_ADAM, ts.data(), n_tensors, hyper, nullptr, lr, step_dev, scalars_dev, stream, "fr_adam_step");
}

extern "C" int fr_optim_step(int32_t rule, const fr_optim_tensor *tensors_host, int32_t n_tensors,
                             const fr_optim_hyper *hyper, const double *lr_dev, int32_t *step_dev, float *scalars_dev,
                             void *stream) {
    FR_REQUIRE(rule == FR_OPTIM_ADAM || rule == FR_OPTIM_SGD || rule == FR_OPTIM_ADAGRAD || rule == FR_OPTIM_RMSPROP,
               "fr_optim_step: unknown rule %d", rule);
    FR_REQUIRE(n_tensors >= 0 && (n_tensors == 0 || tensors_host) && hyper && lr_dev && scalars_dev,
               "fr_optim_step: bad argument");
    const fr_optim_hyper &h = *hyper;
    const int ns = rule == FR_OPTIM_ADAM ? 2 : rule == FR_OPTIM_SGD ? 0 : 1;
    FR_REQUIRE(step_dev || !(rule == FR_OPTIM_ADAM || rule == FR_OPTIM_ADAGRAD), "fr_optim_step: rule %d needs step_dev", rule);
    FR_REQUIRE(h.eps >= 0.0 && h.weight_decay >= 0.0, "fr_optim_step: eps=%g weight_decay=%g", h.eps, h.weight_decay);
    FR_REQUIRE(rule != FR_OPTIM_ADAM || (h.beta1 >= 0.0 && h.beta1 < 1.0 && h.beta2 >= 0.0 && h.beta2 < 1.0),
               "fr_optim_step: betas=(%g, %g)", h.beta1, h.beta2);
    FR_REQUIRE(rule != FR_OPTIM_RMSPROP || h.alpha >= 0.0, "fr_optim_step: alpha=%g", h.alpha);
    // every tensor is checked before anything is launched: a rejected call changes nothing
    for (int32_t t = 0; t < n_tensors; ++t) {
        const fr_optim_tensor &x = tensors_host[t];
        FR_REQUIRE(x.n >= 0, "fr_optim_step: tensor %d has a negative extent", t);
        FR_REQUIRE(x.n == 0 || (x.param && x.grad && (ns < 1 || x.state0) && (ns < 2 || x.state1)),
                   "fr_optim_step: tensor %d: null pointer", t);
    }
    return dispatch(rule, tensors_host, n_tensors, h, lr_dev, 0.0, step_dev, scalars_dev, stream, "fr_optim_step");
}
