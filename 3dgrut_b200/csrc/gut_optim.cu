// 3dgrut_b200/csrc/gut_optim.cu -- optimizer step of the Gaussian parameters (SURVEY.md section 8f row 2, "next" row).
//
//   selective_adam_kernel   drop-in for selective_adam_update_kernel of the reference plugin
//                           (threedgrut/optimizers/optimizers.cu:49-83): Adam without bias correction on the rows whose
//                           visibility flag is set, one launch per parameter tensor.
//   gaussian_adam_kernel    ours: ONE launch for all six parameter tensors of the SH model, taking the renderer's gradients
//                           ([N,12] w.r.t. post-activation position/density/quaternion/scale and [N,48] w.r.t. the SH coefficients,
//                           i.e. after the view-parallel exchange) and applying the activation chain rule the reference leaves to
//                           autograd (threedgrut/model/model.py:102-118 with utils/misc.py:46-50: density = sigmoid(raw),
//                           scale = exp(raw), rotation = normalize(raw)) followed by the Adam update, either torch.optim.Adam's
//                           (bias-corrected, model.py:807-810) or the selective one.
//                           The REG instantiation also adds the opacity and scale regularisers of the reference's loss
//                           (threedgrut/trainer.py:722-739) to the density and scale gradients, and can report their values.
// Both are streaming kernels: every byte is read and written once, coalesced (element-wise index space; the quaternion rows as
// float4).  Algorithmic bytes per Gaussian of the fused step: 59 x (4 param r + 4 param w + 8 moments r + 8 moments w) + 240
// gradient + 4 visibility = 1660 B.
#include <cuda_runtime.h>
#include <stdint.h>

#include "../../include/gut_b200.h"

namespace gutb200 {

namespace {

struct AdamHyper {
    float b1, b2, eps;
    float bc1, bc2_sqrt;  // bias corrections 1 - b1^t and sqrt(1 - b2^t); both 1 in selective mode
    int selective;
};

__device__ __forceinline__ float adam_update(float p, float g, float& m, float& v, float lr, const AdamHyper& h) {
    m = h.b1 * m + (1.0f - h.b1) * g;
    v = h.b2 * v + (1.0f - h.b2) * g * g;
    // selective: step = -lr m / (sqrt(v) + eps)                                   (optimizers.cu:74)
    // adam:      step = -(lr / bc1) m / (sqrt(v) / sqrt(bc2) + eps)               (torch.optim.Adam, single-tensor path)
    const float denom = sqrtf(v) / h.bc2_sqrt + h.eps;
    return p - (lr / h.bc1) * m / denom;
}

__global__ void __launch_bounds__(256) selective_adam_kernel(float* __restrict__ param, const float* __restrict__ grad, float* __restrict__ m,
                                                             float* __restrict__ v, const uint8_t* __restrict__ visibility, float lr,
                                                             AdamHyper h, int64_t total, int width) {
    const int64_t i = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x;
    if (i >= total) return;
    if (visibility && !visibility[i / width]) return;
    float mi = m[i], vi = v[i];
    param[i] = adam_update(param[i], grad[i], mi, vi, lr, h);
    m[i] = mi;
    v[i] = vi;
}

struct GaussianAdamArgs {
    float* param[6];        // positions [N,3], density [N,1], rotation [N,4], scale [N,3], albedo [N,3], specular [N,45] (raw, pre-activation)
    float* m[6];
    float* v[6];
    float lr[6];
    unsigned block_end[6];     // exclusive prefix of the blocks of each group: a block works on ONE group (no divergence)
    const float* d_particles;  // [N,12] dL/d(pos3, density, quat4 (wxyz), scale3, pad) w.r.t. the ACTIVATED values
    const float* d_sph;        // [N,48]
    const float* visibility;   // [N] float bits (the renderer's output) or nullptr
    int64_t n;
    AdamHyper h;
    // REG instantiation only: d(lambda_opacity mean|sigmoid(raw)|) / d sigmoid = lambda_opacity / N * sign and
    // d(lambda_scale mean|exp(raw)|) / d exp = lambda_scale / (3N) * sign; reg_loss [2] (or nullptr) accumulates the two means
    float reg_density, reg_scale;
    float inv_count[2];  // 1 / N, 1 / (3N)
    float* reg_loss;
};

__device__ __forceinline__ float sign_of(float x) { return x > 0.0f ? 1.0f : (x < 0.0f ? -1.0f : 0.0f); }

// activated value of a raw density (G = 1) or scale (G = 3) element
template <int G>
__device__ __forceinline__ float activation(float p) {
    return G == 1 ? 1.0f / (1.0f + expf(-p)) : expf(p);
}

// gradient of element (row, col) of group G w.r.t. the RAW parameter value p
template <int G, bool REG>
__device__ __forceinline__ float raw_gradient(const GaussianAdamArgs& a, int64_t row, int col, float p) {
    if (G == 0) return a.d_particles[row * 12 + col];
    if (G == 1) {
        const float s = activation<1>(p);   // density = sigmoid(raw)
        float g = a.d_particles[row * 12 + 3];
        if (REG) g += a.reg_density * sign_of(s);  // sign, not 1: an underflowed sigmoid gets torch's abs'(0) = 0
        return g * s * (1.0f - s);
    }
    if (G == 3) {
        const float e = activation<3>(p);   // scale = exp(raw)
        float g = a.d_particles[row * 12 + 8 + col];
        if (REG) g += a.reg_scale * sign_of(e);
        return g * e;
    }
    if (G == 4) return a.d_sph[row * 48 + col];                        // features = cat(albedo [N,3], specular [N,45])  (model.py:94-96)
    return a.d_sph[row * 48 + 3 + col];
}

// flat groups: a thread owns 4 consecutive floats of the [N*W] array (16-byte loads and stores of param / moments).
// Returns the sum of the activated values of those floats BEFORE the update when the regularisers' loss is reported (every row,
// visible or not, as the reference's mean over the whole tensor), else 0.
template <int G, int W, bool REG>
__device__ __forceinline__ float flat_group(const GaussianAdamArgs& a, int64_t t) {
    const bool report = REG && (G == 1 || G == 3) && a.reg_loss;
    const int64_t total = a.n * W, e0 = t * 4;
    if (e0 >= total) return 0.0f;
    float* P = a.param[G] + e0;
    float* M = a.m[G] + e0;
    float* V = a.v[G] + e0;
    const float lr = a.lr[G];
    const bool masked = a.h.selective && a.visibility;
    if (e0 + 3 < total) {
        float4 p = *reinterpret_cast<float4*>(P), m = *reinterpret_cast<float4*>(M), v = *reinterpret_cast<float4*>(V);
        float pe[4] = {p.x, p.y, p.z, p.w}, me[4] = {m.x, m.y, m.z, m.w}, ve[4] = {v.x, v.y, v.z, v.w};
        float act = 0.0f;
        if (report) {
#pragma unroll
            for (int k = 0; k < 4; ++k) act += activation<G>(pe[k]);
        }
        bool any = false;
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            const int64_t e = e0 + k, row = e / W;
            const int col = static_cast<int>(e - row * W);
            if (masked && (__float_as_uint(a.visibility[row]) == 0u)) continue;
            any = true;
            pe[k] = adam_update(pe[k], raw_gradient<G, REG>(a, row, col, pe[k]), me[k], ve[k], lr, a.h);
        }
        if (!any) return act;  // nothing visible: leave the 48 bytes alone
        *reinterpret_cast<float4*>(P) = make_float4(pe[0], pe[1], pe[2], pe[3]);
        *reinterpret_cast<float4*>(M) = make_float4(me[0], me[1], me[2], me[3]);
        *reinterpret_cast<float4*>(V) = make_float4(ve[0], ve[1], ve[2], ve[3]);
        return act;
    }
    float act = 0.0f;
    for (int64_t e = e0; e < total; ++e) {
        const int64_t row = e / W;
        const int col = static_cast<int>(e - row * W);
        if (report) act += activation<G>(a.param[G][e]);
        if (masked && (__float_as_uint(a.visibility[row]) == 0u)) continue;
        float m = a.m[G][e], v = a.v[G][e];
        const float p = a.param[G][e];
        a.param[G][e] = adam_update(p, raw_gradient<G, REG>(a, row, col, p), m, v, lr, a.h);
        a.m[G][e] = m;
        a.v[G][e] = v;
    }
    return act;
}

// sum over the block (blockDim.x == 256), valid in thread 0
__device__ __forceinline__ float block_sum(float x) {
    __shared__ float warp_sums[8];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) x += __shfl_xor_sync(0xffffffffu, x, o);
    if ((threadIdx.x & 31) == 0) warp_sums[threadIdx.x >> 5] = x;
    __syncthreads();
    x = threadIdx.x < 8 ? warp_sums[threadIdx.x] : 0.0f;
    if (threadIdx.x < 32) {
#pragma unroll
        for (int o = 4; o > 0; o >>= 1) x += __shfl_xor_sync(0xffffffffu, x, o);
    }
    return x;
}

template <bool REG>
__global__ void __launch_bounds__(256, 4) gaussian_adam_kernel(GaussianAdamArgs a) {
    const unsigned blk = blockIdx.x;
    int group = 0;
#pragma unroll
    for (int k = 0; k < 5; ++k) group += blk >= a.block_end[k] ? 1 : 0;
    const unsigned first = group == 0 ? 0u : a.block_end[group - 1];
    const int64_t t = static_cast<int64_t>(blk - first) * blockDim.x + threadIdx.x;
    float act = 0.0f;
    switch (group) {
        case 0: flat_group<0, 3, REG>(a, t); break;
        case 1: act = flat_group<1, 1, REG>(a, t); break;
        case 3: act = flat_group<3, 3, REG>(a, t); break;
        case 4: flat_group<4, 3, REG>(a, t); break;
        case 5: flat_group<5, 45, REG>(a, t); break;
        default: {
            // rotation = normalize(raw): d raw = (g - q (q . g)) / max(|raw|, 1e-12)   (torch.nn.functional.normalize, eps 1e-12)
            const int64_t row = t;
            if (row >= a.n) return;
            if (a.h.selective && a.visibility && (__float_as_uint(a.visibility[row]) == 0u)) return;
            const float lr = a.lr[2];
            float4* P = reinterpret_cast<float4*>(a.param[2]) + row;
            float4* M = reinterpret_cast<float4*>(a.m[2]) + row;
            float4* V = reinterpret_cast<float4*>(a.v[2]) + row;
            const float4 r = *P;
            const float4 g = *reinterpret_cast<const float4*>(a.d_particles + row * 12 + 4);
            const float len = fmaxf(sqrtf(r.x * r.x + r.y * r.y + r.z * r.z + r.w * r.w), 1e-12f);
            const float il = 1.0f / len;
            const float qx = r.x * il, qy = r.y * il, qz = r.z * il, qw = r.w * il;
            const float dot = qx * g.x + qy * g.y + qz * g.z + qw * g.w;
            float4 m = *M, v = *V, out;
            out.x = adam_update(r.x, (g.x - qx * dot) * il, m.x, v.x, lr, a.h);
            out.y = adam_update(r.y, (g.y - qy * dot) * il, m.y, v.y, lr, a.h);
            out.z = adam_update(r.z, (g.z - qz * dot) * il, m.z, v.z, lr, a.h);
            out.w = adam_update(r.w, (g.w - qw * dot) * il, m.w, v.w, lr, a.h);
            *P = out;
            *M = m;
            *V = v;
        }
    }
    // a block works on one group, so the whole block takes this branch or none of it; the order of the atomics makes only the
    // reported loss nondeterministic, never the parameters
    if (REG && a.reg_loss && (group == 1 || group == 3)) {
        const int slot = group == 1 ? 0 : 1;
        const float sum = block_sum(act);
        if (threadIdx.x == 0) atomicAdd(a.reg_loss + slot, sum * a.inv_count[slot]);
    }
}

AdamHyper make_hyper(float b1, float b2, float eps, int64_t step, int selective) {
    AdamHyper h;
    h.b1 = b1; h.b2 = b2; h.eps = eps; h.selective = selective;
    h.bc1 = 1.f; h.bc2_sqrt = 1.f;
    if (!selective) {
        double p1 = 1.0, p2 = 1.0;
        for (int64_t k = 0; k < step; ++k) { p1 *= b1; p2 *= b2; if (p1 < 1e-300 && p2 < 1e-300) break; }
        h.bc1 = static_cast<float>(1.0 - p1);
        h.bc2_sqrt = static_cast<float>(sqrt(1.0 - p2));
    }
    return h;
}

// argument checks and launch geometry shared by both entry points; blocks == 0 means there is nothing to do (n == 0)
int make_gaussian_adam_args(int64_t n, float* const* params6, float* const* exp_avg6, float* const* exp_avg_sq6, const float* lr6, float b1,
                            float b2, float eps, int64_t step, int32_t selective, const float* d_particles, const float* d_sph,
                            const float* visibility, GaussianAdamArgs& a, unsigned& blocks) {
    blocks = 0;
    if (n < 0 || !params6 || !exp_avg6 || !exp_avg_sq6 || !lr6 || !d_particles || !d_sph) return 1;
    if (!selective && step < 1) return 1;
    if (n == 0) return 0;
    for (int k = 0; k < 6; ++k) {
        if (!params6[k] || !exp_avg6[k] || !exp_avg_sq6[k]) return 1;
        a.param[k] = params6[k];
        a.m[k] = exp_avg6[k];
        a.v[k] = exp_avg_sq6[k];
        a.lr[k] = lr6[k];
    }
    for (int k = 0; k < 6; ++k) {  // parameters and moments are accessed 16 bytes at a time
        if ((reinterpret_cast<uintptr_t>(a.param[k]) | reinterpret_cast<uintptr_t>(a.m[k]) | reinterpret_cast<uintptr_t>(a.v[k])) & 15) return 3;
    }
    if (reinterpret_cast<uintptr_t>(d_particles) & 15) return 3;
    a.d_particles = d_particles;
    a.d_sph = d_sph;
    a.visibility = visibility;
    a.n = n;
    a.h = make_hyper(b1, b2, eps, step, selective);
    a.reg_density = a.reg_scale = 0.0f;
    a.inv_count[0] = a.inv_count[1] = 0.0f;
    a.reg_loss = nullptr;
    const int widths[6] = {3, 1, 4, 3, 3, 45};
    unsigned total = 0;
    for (int k = 0; k < 6; ++k) {
        const int64_t threads = k == 2 ? n : (n * widths[k] + 3) / 4;  // rotation: one row per thread; flat groups: 4 floats per thread
        total += static_cast<unsigned>((threads + 255) / 256);
        a.block_end[k] = total;
    }
    blocks = total;
    return 0;
}

}  // namespace

}  // namespace gutb200

extern "C" {

int gutb200_selective_adam_update(void* stream, float* param, const float* grad, float* exp_avg, float* exp_avg_sq,
                                  const uint8_t* visibility, float lr, float b1, float b2, float eps, int64_t n, int64_t m) {
    using namespace gutb200;
    if (n < 0 || m <= 0 || !param || !grad || !exp_avg || !exp_avg_sq) return 1;
    const int64_t total = n * m;
    if (total == 0) return 0;
    if (m > 0x7FFFFFFF) return 1;
    const AdamHyper h = make_hyper(b1, b2, eps, 0, 1);
    const unsigned blocks = static_cast<unsigned>((total + 255) / 256);
    selective_adam_kernel<<<blocks, 256, 0, static_cast<cudaStream_t>(stream)>>>(param, grad, exp_avg, exp_avg_sq, visibility, lr, h, total,
                                                                                 static_cast<int>(m));
    return cudaGetLastError() == cudaSuccess ? 0 : 2;
}

int gutb200_gaussian_adam_step(void* stream, int64_t n, float* const* params6, float* const* exp_avg6, float* const* exp_avg_sq6,
                               const float* lr6, float b1, float b2, float eps, int64_t step, int32_t selective, const float* d_particles,
                               const float* d_sph, const float* visibility) {
    using namespace gutb200;
    GaussianAdamArgs a;
    unsigned blocks = 0;
    const int rc = make_gaussian_adam_args(n, params6, exp_avg6, exp_avg_sq6, lr6, b1, b2, eps, step, selective, d_particles, d_sph, visibility,
                                           a, blocks);
    if (rc != 0 || blocks == 0) return rc;
    gaussian_adam_kernel<false><<<blocks, 256, 0, static_cast<cudaStream_t>(stream)>>>(a);
    return cudaGetLastError() == cudaSuccess ? 0 : 2;
}

int gutb200_gaussian_adam_step_reg(void* stream, int64_t n, float* const* params6, float* const* exp_avg6, float* const* exp_avg_sq6,
                                   const float* lr6, float b1, float b2, float eps, int64_t step, int32_t selective, const float* d_particles,
                                   const float* d_sph, const float* visibility, float lambda_opacity, float lambda_scale, float* reg_loss2) {
    using namespace gutb200;
    GaussianAdamArgs a;
    unsigned blocks = 0;
    const int rc = make_gaussian_adam_args(n, params6, exp_avg6, exp_avg_sq6, lr6, b1, b2, eps, step, selective, d_particles, d_sph, visibility,
                                           a, blocks);
    if (rc != 0) return rc;
    const cudaStream_t s = static_cast<cudaStream_t>(stream);
    if (reg_loss2 && cudaMemsetAsync(reg_loss2, 0, 2 * sizeof(float), s) != cudaSuccess) return 2;
    if (blocks == 0) return 0;
    a.reg_density = static_cast<float>(static_cast<double>(lambda_opacity) / static_cast<double>(n));
    a.reg_scale = static_cast<float>(static_cast<double>(lambda_scale) / (3.0 * static_cast<double>(n)));
    a.inv_count[0] = static_cast<float>(1.0 / static_cast<double>(n));
    a.inv_count[1] = static_cast<float>(1.0 / (3.0 * static_cast<double>(n)));
    a.reg_loss = reg_loss2;
    gaussian_adam_kernel<true><<<blocks, 256, 0, s>>>(a);
    return cudaGetLastError() == cudaSuccess ? 0 : 2;
}

}  // extern "C"
