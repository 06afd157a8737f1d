// Optimizer side of the training step (SURVEY.md §8f N1): torch.nn.utils.clip_grad_norm_(model.parameters(), 3) +
// torch.optim.Adam.step() (trainer.py:159-160) as two multi-tensor launches with no host synchronisation:
//   1. grad_sqnorm_kernel: sum of squares of every clipped gradient (fp64 atomics)
//   2. adam_clip_kernel:   clip coefficient from that norm (computed on the device), exp_avg / exp_avg_sq update,
//                          bias-corrected parameter update -- the exact op order of torch's _single_tensor_adam.
#include <cuda_runtime.h>
#include <math.h>
#include <stdint.h>

#include "../../include/monoloco_b200.h"
#include "host_error.h"

namespace mlb {

struct TensorList {
    float* p[64];
    const float* g[64];
    float* m[64];
    float* v[64];
    long long n[64];
    int clip[64];
    int count;
};

__global__ void grad_sqnorm_kernel(const __grid_constant__ TensorList tl, double* out) {
    double acc = 0.0;
    for (int t = 0; t < tl.count; ++t) {
        if (!tl.clip[t]) continue;
        const float* g = tl.g[t];
        for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < tl.n[t]; i += (long long)gridDim.x * blockDim.x) {
            const float x = g[i];
            acc += (double)x * (double)x;
        }
    }
    for (int s = 16; s > 0; s >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, s);
    __shared__ double ws[32];
    if ((threadIdx.x & 31) == 0) ws[threadIdx.x >> 5] = acc;
    __syncthreads();
    if (threadIdx.x < 32) {
        double v = threadIdx.x < (blockDim.x >> 5) ? ws[threadIdx.x] : 0.0;
        for (int s = 16; s > 0; s >>= 1) v += __shfl_xor_sync(0xffffffffu, v, s);
        if (threadIdx.x == 0) atomicAdd(out, v);
    }
}

__global__ void adam_clip_kernel(const __grid_constant__ TensorList tl, const double* sqnorm, float max_norm, float lr, float beta1,
                                 float beta2, float eps, float weight_decay, float bc1, float bc2_sqrt) {
    float coef = 1.0f;
    if (max_norm > 0.f) {
        const float total = (float)sqrt(*sqnorm);
        coef = fminf(max_norm / (total + 1e-6f), 1.0f);  // torch: clip_coef = max_norm / (total_norm + 1e-6), clamped to 1
    }
    const float step_size = lr / bc1;
    for (int t = 0; t < tl.count; ++t) {
        float* p = tl.p[t];
        const float* g = tl.g[t];
        float* m = tl.m[t];
        float* v = tl.v[t];
        const float c = tl.clip[t] ? coef : 1.0f;
        for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < tl.n[t]; i += (long long)gridDim.x * blockDim.x) {
            float gi = g[i] * c;
            if (weight_decay != 0.f) gi = fmaf(weight_decay, p[i], gi);
            const float mi = m[i] + (gi - m[i]) * (1.0f - beta1);            // exp_avg.lerp_(grad, 1 - beta1)
            const float vi = beta2 * v[i] + (1.0f - beta2) * gi * gi;        // exp_avg_sq.mul_(beta2).addcmul_(grad, grad, 1 - beta2)
            m[i] = mi;
            v[i] = vi;
            const float denom = sqrtf(vi) / bc2_sqrt + eps;
            p[i] = p[i] - step_size * (mi / denom);                          // param.addcdiv_(exp_avg, denom, value=-step_size)
        }
    }
}

}  // namespace mlb

using namespace mlb;

extern "C" int mlb_adam_clip_step(int n_tensors, float* const* params, const float* const* grads, float* const* exp_avg,
                                  float* const* exp_avg_sq, const int64_t* sizes, const int32_t* clip_mask, float max_norm,
                                  float lr, float beta1, float beta2, float eps, float weight_decay, int64_t step,
                                  double* sqnorm_scratch_dev, void* stream) {
    if (n_tensors < 1 || !params || !grads || !exp_avg || !exp_avg_sq || !sizes || !sqnorm_scratch_dev || step < 1)
        return mlb_fail("mlb_adam_clip_step: bad argument");
    cudaStream_t st = (cudaStream_t)stream;
    const float bc1 = 1.0f - powf(beta1, (float)step);
    const float bc2_sqrt = sqrtf(1.0f - powf(beta2, (float)step));
    cudaError_t e = cudaMemsetAsync(sqnorm_scratch_dev, 0, sizeof(double), st);
    for (int base = 0; base < n_tensors && e == cudaSuccess; base += 64) {
        TensorList tl;
        tl.count = n_tensors - base < 64 ? n_tensors - base : 64;
        for (int i = 0; i < tl.count; ++i) {
            tl.p[i] = params[base + i], tl.g[i] = grads[base + i], tl.m[i] = exp_avg[base + i], tl.v[i] = exp_avg_sq[base + i];
            tl.n[i] = sizes[base + i], tl.clip[i] = clip_mask ? clip_mask[base + i] : 1;
        }
        if (max_norm > 0.f) {
            grad_sqnorm_kernel<<<296, 256, 0, st>>>(tl, sqnorm_scratch_dev);
            mlb_count_launch();
        }
        e = cudaGetLastError();
    }
    for (int base = 0; base < n_tensors && e == cudaSuccess; base += 64) {
        TensorList tl;
        tl.count = n_tensors - base < 64 ? n_tensors - base : 64;
        for (int i = 0; i < tl.count; ++i) {
            tl.p[i] = params[base + i], tl.g[i] = grads[base + i], tl.m[i] = exp_avg[base + i], tl.v[i] = exp_avg_sq[base + i];
            tl.n[i] = sizes[base + i], tl.clip[i] = clip_mask ? clip_mask[base + i] : 1;
        }
        adam_clip_kernel<<<592, 256, 0, st>>>(tl, sqnorm_scratch_dev, max_norm, lr, beta1, beta2, eps, weight_decay, bc1, bc2_sqrt);
        mlb_count_launch();
        e = cudaGetLastError();
    }
    if (e != cudaSuccess) return mlb_fail(std::string("mlb_adam_clip_step: ") + cudaGetErrorString(e));
    return 0;
}
