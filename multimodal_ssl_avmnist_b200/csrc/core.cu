// Library plumbing + the flat-arena kernels: teacher EMA, Adam, scaling, dropout masks.
#include <stdarg.h>
#include <string.h>

#include <stdlib.h>

#include "common.cuh"

namespace b200 {

static thread_local char g_err[512] = "";

void set_error(const char* fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
}

int sm_count() {
    static int cached = 0;
    if (cached == 0) {
        int dev = 0, n = 0;
        if (cudaGetDevice(&dev) == cudaSuccess &&
            cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev) == cudaSuccess && n > 0)
            cached = n;
        else
            return 148;
    }
    return cached;
}

// ---------------------------------------------------------------------------------------------------------
// EMA: t <- RN(RN(m*t) + RN(om*s)).  __fmul_rn/__fadd_rn are never contracted into an FMA (SURVEY A7).
// HBM-bound: 12 B per element.  float4 loads, 4 independent vectors in flight per thread, grid = SMs x 8.
// ---------------------------------------------------------------------------------------------------------
__device__ __forceinline__ float ema1(float t, float s, float m, float om) {
    return __fadd_rn(__fmul_rn(m, t), __fmul_rn(om, s));
}
__device__ __forceinline__ float4 ema4(float4 t, float4 s, float m, float om) {
    return make_float4(ema1(t.x, s.x, m, om), ema1(t.y, s.y, m, om), ema1(t.z, s.z, m, om), ema1(t.w, s.w, m, om));
}

__global__ void __launch_bounds__(256) ema_flat_kernel(float* __restrict__ t, const float* __restrict__ s, int64_t n,
                                                       float m, float om) {
    const int64_t n4 = n >> 2;
    float4* t4 = reinterpret_cast<float4*>(t);
    const float4* s4 = reinterpret_cast<const float4*>(s);
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    for (; i + 3 * stride < n4; i += 4 * stride) {
        float4 a0 = t4[i], a1 = t4[i + stride], a2 = t4[i + 2 * stride], a3 = t4[i + 3 * stride];
        float4 b0 = __ldg(s4 + i), b1 = __ldg(s4 + i + stride), b2 = __ldg(s4 + i + 2 * stride),
               b3 = __ldg(s4 + i + 3 * stride);
        t4[i] = ema4(a0, b0, m, om);
        t4[i + stride] = ema4(a1, b1, m, om);
        t4[i + 2 * stride] = ema4(a2, b2, m, om);
        t4[i + 3 * stride] = ema4(a3, b3, m, om);
    }
    for (; i < n4; i += stride) t4[i] = ema4(t4[i], __ldg(s4 + i), m, om);
    // tail (n % 4)
    int64_t k = (n4 << 2) + (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (k < n) t[k] = ema1(t[k], s[k], m, om);
}

// Multi-tensor variant: CTA `c` owns elements [c*CHUNK, (c+1)*CHUNK) of the virtual concatenation and finds the
// tensors it overlaps by binary search in the prefix-offset table.
constexpr int EMA_CHUNK = 4096;
__global__ void __launch_bounds__(256) ema_multi_kernel(float* const* __restrict__ tp, const float* const* __restrict__ sp,
                                                        const int64_t* __restrict__ off, int nt, int64_t total, float m,
                                                        float om) {
    for (int64_t base = (int64_t)blockIdx.x * EMA_CHUNK; base < total; base += (int64_t)gridDim.x * EMA_CHUNK) {
        int lo = 0, hi = nt - 1;
        while (lo < hi) {  // last tensor with off[k] <= base
            int mid = (lo + hi + 1) >> 1;
            if (off[mid] <= base) lo = mid; else hi = mid - 1;
        }
        int k = lo;
        int64_t end = min(base + EMA_CHUNK, total);
        for (int64_t e = base + threadIdx.x; e < end; e += blockDim.x) {
            while (e >= off[k + 1]) ++k;
            int64_t j = e - off[k];
            float* t = tp[k];
            t[j] = ema1(t[j], __ldg(sp[k] + j), m, om);
        }
    }
}

// ---------------------------------------------------------------------------------------------------------
// Adam over a flat arena (torch.optim.Adam semantics: g += wd*p; m,v EMAs; p -= lr/bc1 * m / (sqrt(v)/sqrt(bc2) + eps))
// 28 B per element.  grad_scale multiplies the incoming gradient (DP mean, AMP unscale).
// ---------------------------------------------------------------------------------------------------------
__device__ __forceinline__ void adam_one(float& pi, float gi_raw, float& mi, float& vi, float step, float b1, float b2, float eps, float wd,
                                         float bc2s, float gs) {
    const float gi = gi_raw * gs + wd * pi;
    mi = mi * b1 + (1.0f - b1) * gi;
    vi = vi * b2 + (1.0f - b2) * gi * gi;
    const float denom = sqrtf(vi) / bc2s + eps;
    pi = pi - step * (mi / denom);
}

// DECOUPLED (torch.optim.AdamW): p <- p * (1 - lr*wd) first, and no L2 term in the gradient; the rest is adam_one unchanged, so
// with wd = 0 the update is bit-identical to Adam's.  `decay` is 1 - lr*wd rounded from double like torch's Python scalar (the
// kernel recomputes it only when the learning rate comes from bc_dev).
template <bool DECOUPLED>
__global__ void __launch_bounds__(256) adam_flat_kernel(float* __restrict__ p, const float* __restrict__ g,
                                                        float* __restrict__ m, float* __restrict__ v, int64_t n, float lr,
                                                        float b1, float b2, float eps, float wd, float bc1, float bc2s,
                                                        float gs, const float* __restrict__ bc_dev, float decay = 1.f) {
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    if (bc_dev != nullptr) {          // CUDA-graph replay: the bias corrections (and the learning rate) of this step live on the device
        bc1 = __ldg(bc_dev);
        bc2s = __ldg(bc_dev + 1);
        if (lr < 0.f) {
            lr = __ldg(bc_dev + 2);
            if (DECOUPLED) decay = (float)(1.0 - (double)lr * (double)wd);
        }
    }
    if (DECOUPLED) wd = 0.f;
    const float step = lr / bc1;
    // 128-bit accesses over the aligned body (the arenas are 16-byte aligned and padded; same arithmetic per element either way)
    const bool vec = ((reinterpret_cast<uintptr_t>(p) | reinterpret_cast<uintptr_t>(g) | reinterpret_cast<uintptr_t>(m) |
                       reinterpret_cast<uintptr_t>(v)) & 15) == 0;
    const int64_t n4 = vec ? n / 4 : 0;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n4; i += stride) {
        float4 pp = reinterpret_cast<float4*>(p)[i], mm = reinterpret_cast<float4*>(m)[i], vv = reinterpret_cast<float4*>(v)[i];
        const float4 gg = __ldg(reinterpret_cast<const float4*>(g) + i);
        if (DECOUPLED) {
            pp.x *= decay;
            pp.y *= decay;
            pp.z *= decay;
            pp.w *= decay;
        }
        adam_one(pp.x, gg.x, mm.x, vv.x, step, b1, b2, eps, wd, bc2s, gs);
        adam_one(pp.y, gg.y, mm.y, vv.y, step, b1, b2, eps, wd, bc2s, gs);
        adam_one(pp.z, gg.z, mm.z, vv.z, step, b1, b2, eps, wd, bc2s, gs);
        adam_one(pp.w, gg.w, mm.w, vv.w, step, b1, b2, eps, wd, bc2s, gs);
        reinterpret_cast<float4*>(m)[i] = mm;
        reinterpret_cast<float4*>(v)[i] = vv;
        reinterpret_cast<float4*>(p)[i] = pp;
    }
    for (int64_t i = n4 * 4 + (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) {
        float pi = p[i], mi = m[i], vi = v[i];
        if (DECOUPLED) pi *= decay;
        adam_one(pi, __ldg(g + i), mi, vi, step, b1, b2, eps, wd, bc2s, gs);
        m[i] = mi;
        v[i] = vi;
        p[i] = pi;
    }
}

__global__ void __launch_bounds__(256) scale_flat_kernel(float* __restrict__ y, int64_t n, float a) {
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) y[i] *= a;
}

// bias corrections of Adam step t = *step_dev + 1, in double like the host path (1 - beta^t, sqrt(1 - beta2^t)), rounded to fp32
__global__ void adam_bias_kernel(const int64_t* __restrict__ step_dev, double b1, double b2, float* __restrict__ out) {
    const double t = (double)(*step_dev + 1);
    out[0] = (float)(1.0 - pow(b1, t));
    out[1] = (float)sqrt(1.0 - pow(b2, t));
}

__global__ void counters_advance_kernel(int64_t* __restrict__ ctr, int n) {
    if ((int)threadIdx.x < n) ctr[threadIdx.x] += 1;
}

__global__ void __launch_bounds__(256) dropout_mask_kernel(uint8_t* __restrict__ mask, int64_t n, float p, uint64_t seed,
                                                           uint64_t offset, const int64_t* __restrict__ step_dev) {
    if (step_dev != nullptr) offset += 4ull * (uint64_t)__ldg(step_dev);      // the engine's offsets are 4*step + k
    Philox rng(seed);
    const int64_t n4 = (n + 3) >> 2;
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n4; i += stride) {
        uint4 r = rng((uint64_t)i, offset);
        uint32_t w[4] = {r.x, r.y, r.z, r.w};
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            int64_t e = i * 4 + k;
            if (e < n) mask[e] = u01(w[k]) >= p ? 1 : 0;
        }
    }
}

static int flat_grid(int64_t n, int per_thread) {
    int64_t want = (n + (int64_t)256 * per_thread - 1) / ((int64_t)256 * per_thread);
    int64_t cap = (int64_t)sm_count() * 8;
    if (want < 1) want = 1;
    return (int)(want < cap ? want : cap);
}

}  // namespace b200

using namespace b200;

extern "C" {

const char* b200_last_error(void) { return g_err; }
int b200_abi_version(void) { return 1; }

// Node census of a captured CUDA graph (cudaGraph_t): counts[0..3] = kernel, memset, memcpy, other nodes.  The engine uses it to
// COUNT the kernel launches of one training step instead of tallying them by hand.
int b200_graph_node_counts(void* graph, int64_t* counts) {
    B200_REQUIRE(graph && counts, B200_E_ARG, "graph_node_counts: null pointer");
    cudaGraph_t g = reinterpret_cast<cudaGraph_t>(graph);
    size_t n = 0;
    cudaError_t e = cudaGraphGetNodes(g, nullptr, &n);
    if (e != cudaSuccess) {
        set_error("graph_node_counts: %s", cudaGetErrorString(e));
        return (int)e;
    }
    cudaGraphNode_t* nodes = n ? (cudaGraphNode_t*)malloc(n * sizeof(cudaGraphNode_t)) : nullptr;
    if (n) e = cudaGraphGetNodes(g, nodes, &n);
    counts[0] = counts[1] = counts[2] = counts[3] = 0;
    for (size_t i = 0; e == cudaSuccess && i < n; ++i) {
        cudaGraphNodeType t;
        e = cudaGraphNodeGetType(nodes[i], &t);
        if (e != cudaSuccess) break;
        if (t == cudaGraphNodeTypeKernel) ++counts[0];
        else if (t == cudaGraphNodeTypeMemset) ++counts[1];
        else if (t == cudaGraphNodeTypeMemcpy) ++counts[2];
        else ++counts[3];
    }
    free(nodes);
    if (e != cudaSuccess) {
        set_error("graph_node_counts: %s", cudaGetErrorString(e));
        return (int)e;
    }
    return 0;
}
int b200_device_sm_count(int device) {
    int n = 0;
    if (cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, device) != cudaSuccess) return -1;
    return n;
}

int b200_ema_flat(float* teacher, const float* student, int64_t n, float m, float one_minus_m, void* stream) {
    B200_REQUIRE(teacher && student && n > 0, B200_E_ARG, "ema_flat: null pointer or n <= 0");
    B200_REQUIRE((((uintptr_t)teacher | (uintptr_t)student) & 15) == 0, B200_E_ARG, "ema_flat: pointers must be 16-byte aligned");
    ema_flat_kernel<<<flat_grid(n, 16), 256, 0, as_stream(stream)>>>(teacher, student, n, m, one_minus_m);
    return launch_status("ema_flat");
}

int b200_ema_multi(float* const* t_ptrs, const float* const* s_ptrs, const int64_t* offsets, int n_tensors,
                   int64_t total, float m, float one_minus_m, void* stream) {
    B200_REQUIRE(t_ptrs && s_ptrs && offsets && n_tensors > 0 && total > 0, B200_E_ARG, "ema_multi: bad arguments");
    int64_t chunks = (total + EMA_CHUNK - 1) / EMA_CHUNK;
    int64_t cap = (int64_t)sm_count() * 8;
    ema_multi_kernel<<<(int)(chunks < cap ? chunks : cap), 256, 0, as_stream(stream)>>>(t_ptrs, s_ptrs, offsets, n_tensors,
                                                                                          total, m, one_minus_m);
    return launch_status("ema_multi");
}

int b200_adam_flat(float* param, const float* grad, float* exp_avg, float* exp_avg_sq, int64_t n, float lr, float beta1,
                   float beta2, float eps, float weight_decay, float bias_correction1, float bias_correction2_sqrt,
                   float grad_scale, void* stream) {
    B200_REQUIRE(param && grad && exp_avg && exp_avg_sq && n > 0, B200_E_ARG, "adam_flat: null pointer or n <= 0");
    adam_flat_kernel<false><<<flat_grid(n, 4), 256, 0, as_stream(stream)>>>(param, grad, exp_avg, exp_avg_sq, n, lr, beta1, beta2,
                                                                     eps, weight_decay, bias_correction1,
                                                                     bias_correction2_sqrt, grad_scale, nullptr);
    return launch_status("adam_flat");
}

int b200_adam_bias_dev(const int64_t* step_dev, double beta1, double beta2, float* bc_out, void* stream) {
    B200_REQUIRE(step_dev && bc_out, B200_E_ARG, "adam_bias_dev: null pointer");
    adam_bias_kernel<<<1, 1, 0, as_stream(stream)>>>(step_dev, beta1, beta2, bc_out);
    return launch_status("adam_bias_dev");
}

int b200_adam_flat_dev(float* param, const float* grad, float* exp_avg, float* exp_avg_sq, int64_t n, float lr, float beta1,
                       float beta2, float eps, float weight_decay, const float* bc_dev, float grad_scale, void* stream) {
    B200_REQUIRE(param && grad && exp_avg && exp_avg_sq && bc_dev && n > 0, B200_E_ARG, "adam_flat_dev: null pointer or n <= 0");
    adam_flat_kernel<false><<<flat_grid(n, 4), 256, 0, as_stream(stream)>>>(param, grad, exp_avg, exp_avg_sq, n, lr, beta1, beta2,
                                                                     eps, weight_decay, 1.f, 1.f, grad_scale, bc_dev);
    return launch_status("adam_flat_dev");
}

int b200_adamw_flat(float* param, const float* grad, float* exp_avg, float* exp_avg_sq, int64_t n, float lr, float beta1,
                    float beta2, float eps, float weight_decay, float bias_correction1, float bias_correction2_sqrt, void* stream) {
    B200_REQUIRE(param && grad && exp_avg && exp_avg_sq && n > 0 && lr >= 0.f, B200_E_ARG, "adamw_flat: null pointer, n <= 0 or lr < 0");
    const float decay = (float)(1.0 - (double)lr * (double)weight_decay);
    adam_flat_kernel<true><<<flat_grid(n, 4), 256, 0, as_stream(stream)>>>(param, grad, exp_avg, exp_avg_sq, n, lr, beta1, beta2, eps,
                                                                           weight_decay, bias_correction1, bias_correction2_sqrt, 1.f,
                                                                           nullptr, decay);
    return launch_status("adamw_flat");
}

int b200_adamw_flat_dev(float* param, const float* grad, float* exp_avg, float* exp_avg_sq, int64_t n, float lr, float beta1,
                        float beta2, float eps, float weight_decay, const float* bc_dev, void* stream) {
    B200_REQUIRE(param && grad && exp_avg && exp_avg_sq && bc_dev && n > 0, B200_E_ARG, "adamw_flat_dev: null pointer or n <= 0");
    const float decay = (float)(1.0 - (double)lr * (double)weight_decay);     // replaced on the device when lr < 0
    adam_flat_kernel<true><<<flat_grid(n, 4), 256, 0, as_stream(stream)>>>(param, grad, exp_avg, exp_avg_sq, n, lr, beta1, beta2, eps,
                                                                           weight_decay, 1.f, 1.f, 1.f, bc_dev, decay);
    return launch_status("adamw_flat_dev");
}

int b200_counters_advance(int64_t* counters, int n, void* stream) {
    B200_REQUIRE(counters && n > 0 && n <= 32, B200_E_ARG, "counters_advance: bad arguments");
    counters_advance_kernel<<<1, 32, 0, as_stream(stream)>>>(counters, n);
    return launch_status("counters_advance");
}

int b200_scale_flat(float* y, int64_t n, float alpha, void* stream) {
    B200_REQUIRE(y && n > 0, B200_E_ARG, "scale_flat: null pointer or n <= 0");
    scale_flat_kernel<<<flat_grid(n, 4), 256, 0, as_stream(stream)>>>(y, n, alpha);
    return launch_status("scale_flat");
}

int b200_dropout_mask(uint8_t* mask, int64_t n, float p, uint64_t seed, uint64_t offset, void* stream) {
    return b200_dropout_mask_dev(mask, n, p, seed, offset, nullptr, stream);
}

int b200_dropout_mask_dev(uint8_t* mask, int64_t n, float p, uint64_t seed, uint64_t offset, const int64_t* step_dev, void* stream) {
    B200_REQUIRE(mask && n > 0 && p >= 0.f && p < 1.f, B200_E_ARG, "dropout_mask: bad arguments");
    dropout_mask_kernel<<<flat_grid((n + 3) / 4, 4), 256, 0, as_stream(stream)>>>(mask, n, p, seed, offset, step_dev);
    return launch_status("dropout_mask");
}

}  // extern "C"
