// Adam update of every parameter tensor of a model in (normally) one launch.
// Replaces `optimizer.step()` of the reference's trainer (contrastive_estimation_training.py:162 with
// optimizer = torch.optim.Adam, :41): p, exp_avg, exp_avg_sq are read and written once, the gradient read once
// (28 B per parameter), instead of the ~12 whole-model passes of the per-op implementation.
//   g  = grad_scale * grad (+ weight_decay * p)            [maximize: g = -g]
//   m  = m + (1 - beta1) (g - m);   v = beta2 v + (1 - beta2) g^2
//   p -= lr / (1 - beta1^t) * m / (sqrt(v) / sqrt(1 - beta2^t) + eps)
// The step count t lives on the device (CUDA-graph replays advance it); the bias corrections are evaluated in
// double precision by a one-thread kernel in front of the update.
// An optional device flag `skip` is read by both kernels when they run: a non-zero flag turns the launch into a no-op
// (parameters, moments, step count and bias corrections untouched), so a captured step can decide per replay.
#include "common.cuh"

namespace cpc {

constexpr int ADAM_MAX_TENSORS = 48;      // per launch: the tables travel as kernel parameters (<= 4 KB)
constexpr int ADAM_BLOCK_ELEMS = 4096;    // 256 threads x 4 float4

struct AdamTable {
    float* p[ADAM_MAX_TENSORS];
    const float* g[ADAM_MAX_TENSORS];
    float* m[ADAM_MAX_TENSORS];
    float* v[ADAM_MAX_TENSORS];
    int n[ADAM_MAX_TENSORS];
    int block_start[ADAM_MAX_TENSORS + 1];
    int count;
};

// state[0] = t (advanced here), state[1] = lr / (1 - beta1^t), state[2] = 1 / sqrt(1 - beta2^t)
__global__ void adam_tick_kernel(float* state, const float* skip, double lr, double beta1, double beta2) {
    if (skip && *skip != 0.f) return;
    const double t = (double)state[0] + 1.0;
    state[0] = (float)t;
    state[1] = (float)(lr / (1.0 - pow(beta1, t)));
    state[2] = (float)(1.0 / sqrt(1.0 - pow(beta2, t)));
}

// hyper-parameters rounded to fp32 once, on the host
struct AdamScalars { float beta2, one_minus_beta1, one_minus_beta2, eps, weight_decay, grad_scale; int maximize; };

__device__ __forceinline__ void adam_one(float& p, float g, float& m, float& v, float step_size, float inv_bc2_sqrt,
                                         const AdamScalars& a) {
    g *= a.grad_scale;
    if (a.maximize) g = -g;
    if (a.weight_decay != 0.f) g = fmaf(a.weight_decay, p, g);
    m = fmaf(a.one_minus_beta1, g - m, m);
    v = fmaf(a.one_minus_beta2, g * g, a.beta2 * v);
    const float denom = fmaf(sqrtf(v), inv_bc2_sqrt, a.eps);
    p -= step_size * (m / denom);
}

__global__ void __launch_bounds__(256) adam_update_kernel(const __grid_constant__ AdamTable tab,
                                                         const float* __restrict__ state, const float* skip,
                                                         const AdamScalars a) {
    if (skip && *skip != 0.f) return;
    // which tensor does this block work on? (block_start is ascending; <= 48 entries in the constant bank)
    int lo = 0, hi = tab.count - 1;
    while (lo < hi) {
        const int mid = (lo + hi + 1) >> 1;
        if (tab.block_start[mid] <= (int)blockIdx.x) lo = mid; else hi = mid - 1;
    }
    const int t = lo;
    const int n = tab.n[t];
    const int base = ((int)blockIdx.x - tab.block_start[t]) * ADAM_BLOCK_ELEMS;
    float* __restrict__ p = tab.p[t];
    const float* __restrict__ g = tab.g[t];
    float* __restrict__ m = tab.m[t];
    float* __restrict__ v = tab.v[t];
    const float step_size = state[1], inv_bc2_sqrt = state[2];
    const bool vec = ((reinterpret_cast<uintptr_t>(p) | reinterpret_cast<uintptr_t>(g) | reinterpret_cast<uintptr_t>(m) |
                       reinterpret_cast<uintptr_t>(v)) & 15) == 0;
    if (vec && base + ADAM_BLOCK_ELEMS <= n) {
        float4 pv[4], gv[4], mv[4], vv[4];
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            const int e = base + (i * 256 + threadIdx.x) * 4;
            pv[i] = *reinterpret_cast<const float4*>(p + e);
            gv[i] = *reinterpret_cast<const float4*>(g + e);
            mv[i] = *reinterpret_cast<const float4*>(m + e);
            vv[i] = *reinterpret_cast<const float4*>(v + e);
        }
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            const int e = base + (i * 256 + threadIdx.x) * 4;
            adam_one(pv[i].x, gv[i].x, mv[i].x, vv[i].x, step_size, inv_bc2_sqrt, a);
            adam_one(pv[i].y, gv[i].y, mv[i].y, vv[i].y, step_size, inv_bc2_sqrt, a);
            adam_one(pv[i].z, gv[i].z, mv[i].z, vv[i].z, step_size, inv_bc2_sqrt, a);
            adam_one(pv[i].w, gv[i].w, mv[i].w, vv[i].w, step_size, inv_bc2_sqrt, a);
            *reinterpret_cast<float4*>(p + e) = pv[i];
            *reinterpret_cast<float4*>(m + e) = mv[i];
            *reinterpret_cast<float4*>(v + e) = vv[i];
        }
        return;
    }
    const int end = min(n, base + ADAM_BLOCK_ELEMS);
    for (int e = base + threadIdx.x; e < end; e += 256) {
        float pe = p[e], me = m[e], ve = v[e];
        adam_one(pe, g[e], me, ve, step_size, inv_bc2_sqrt, a);
        p[e] = pe; m[e] = me; v[e] = ve;
    }
}

}  // namespace cpc

using namespace cpc;

extern "C" int cpc_adam_step_ex(int32_t n_tensors, void* const* params, const void* const* grads, void* const* exp_avg,
                                void* const* exp_avg_sq, const int64_t* numel, float* step_state, const float* skip,
                                const cpc_adam_params* a, void* stream) {
    if (!a || !step_state || (n_tensors > 0 && (!params || !grads || !exp_avg || !exp_avg_sq || !numel))) return CPC_ERR_NULL;
    if (n_tensors < 0 || !(a->beta1 >= 0. && a->beta1 < 1.) || !(a->beta2 >= 0. && a->beta2 < 1.) || !(a->eps >= 0.))
        return CPC_ERR_BAD_SHAPE;
    for (int i = 0; i < n_tensors; ++i) {
        if (numel[i] < 0 || numel[i] > (int64_t)1 << 30) return CPC_ERR_BAD_SHAPE;
        if (numel[i] > 0 && (!params[i] || !grads[i] || !exp_avg[i] || !exp_avg_sq[i])) return CPC_ERR_NULL;
        if ((reinterpret_cast<uintptr_t>(params[i]) | reinterpret_cast<uintptr_t>(grads[i]) |
             reinterpret_cast<uintptr_t>(exp_avg[i]) | reinterpret_cast<uintptr_t>(exp_avg_sq[i])) & 3)
            return CPC_ERR_ALIGNMENT;
    }
    const int st = check_device();
    if (st != CPC_OK) return st;
    cudaStream_t s = reinterpret_cast<cudaStream_t>(stream);
    const AdamScalars sc{(float)a->beta2, (float)(1.0 - a->beta1), (float)(1.0 - a->beta2), (float)a->eps,
                         (float)a->weight_decay, a->grad_scale, a->maximize};
    adam_tick_kernel<<<1, 1, 0, s>>>(step_state, skip, a->lr, a->beta1, a->beta2);
    CPC_LAUNCH_CHECK();
    count_launch();
    int i = 0;
    while (i < n_tensors) {
        AdamTable tab{};
        int blocks = 0;
        while (i < n_tensors && tab.count < ADAM_MAX_TENSORS) {
            if (numel[i] > 0) {
                const int c = tab.count++;
                tab.p[c] = reinterpret_cast<float*>(params[i]);
                tab.g[c] = reinterpret_cast<const float*>(grads[i]);
                tab.m[c] = reinterpret_cast<float*>(exp_avg[i]);
                tab.v[c] = reinterpret_cast<float*>(exp_avg_sq[i]);
                tab.n[c] = (int)numel[i];
                tab.block_start[c] = blocks;
                blocks += (int)((numel[i] + ADAM_BLOCK_ELEMS - 1) / ADAM_BLOCK_ELEMS);
            }
            ++i;
        }
        if (tab.count == 0) break;
        tab.block_start[tab.count] = blocks;
        adam_update_kernel<<<blocks, 256, 0, s>>>(tab, step_state, skip, sc);
        CPC_LAUNCH_CHECK();
        count_launch();
    }
    return CPC_OK;
}

extern "C" int cpc_adam_step(int32_t n_tensors, void* const* params, const void* const* grads, void* const* exp_avg,
                             void* const* exp_avg_sq, const int64_t* numel, float* step_state,
                             const cpc_adam_params* a, void* stream) {
    return cpc_adam_step_ex(n_tensors, params, grads, exp_avg, exp_avg_sq, numel, step_state, nullptr, a, stream);
}
