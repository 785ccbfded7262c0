// Downstream MLP probe on frozen features (train_downstream): Linear(O, 128) -> ReLU -> Linear(128, C) -> softmax cross-entropy,
// forward + backward in two launches, fp32, deterministic.
//
//   probe_rows_kernel : one CTA per PROBE_R rows.  hidden = ReLU(x W1^T + b1) (x / W1 tiles through shared memory, each thread one
//                       hidden unit for all rows), logits, log-sum-exp, loss, argmax, d_logits = (softmax - onehot) / B and
//                       d_hidden = (d_logits W2) * (hidden > 0).  hidden / d_hidden / d_logits go to the work buffer; the CTA's loss
//                       sum (fp64, row order) to its partial slot; the correct count and confusion entries are integer atomics.
//   probe_grads_kernel: every weight / bias gradient is one thread's sum over the batch in row order (no float atomics):
//                       dW1 in 32 x 32 tiles, dW2 one CTA per class, db1 / db2 / the loss-partial sum in the last CTA.
// The backward CTAs exist only for train = 1; with train = 0 the second launch is the single loss-reduction CTA.
#include <math.h>

#include "common.cuh"

namespace b200 {

constexpr int PROBE_H = 128;     // DownstreamClassifier's hidden width
constexpr int PROBE_R = 16;      // rows per CTA of the row kernel
constexpr int PROBE_KT = 32;     // k tile of the hidden GEMM
constexpr int PROBE_CMAX = 16;
constexpr int PROBE_T = 32;      // dW1 tile (hidden units x feature columns)

struct ProbeWork {
    double* part;     // [n_row_blocks] loss partials
    float* h;         // [B, 128]
    float* dh;        // [B, 128]
    float* dlog;      // [B, C]
};

static inline int probe_row_blocks(int B) { return (B + PROBE_R - 1) / PROBE_R; }

static inline int64_t probe_part_floats(int B) { return ((int64_t)probe_row_blocks(B) * 2 + 3) / 4 * 4; }

static inline ProbeWork probe_work(float* work, int B) {
    ProbeWork w;
    w.part = reinterpret_cast<double*>(work);
    w.h = work + probe_part_floats(B);
    w.dh = w.h + (int64_t)B * PROBE_H;
    w.dlog = w.dh + (int64_t)B * PROBE_H;
    return w;
}

template <bool TRAIN>
__global__ void __launch_bounds__(PROBE_H) probe_rows_kernel(const float* __restrict__ x, const float* __restrict__ w1,
                                                             const float* __restrict__ b1, const float* __restrict__ w2,
                                                             const float* __restrict__ b2, const int64_t* __restrict__ labels,
                                                             int B, int O, int C, ProbeWork w, unsigned long long* __restrict__ correct,
                                                             int64_t* __restrict__ preds, unsigned long long* __restrict__ confusion) {
    __shared__ __align__(16) float xs[PROBE_R][PROBE_KT];
    __shared__ float w1s[PROBE_H][PROBE_KT + 1];
    __shared__ float hs[PROBE_R][PROBE_H + 1];
    __shared__ float w2s[PROBE_CMAX][PROBE_H + 1];
    __shared__ float ls[PROBE_R][PROBE_CMAX];
    __shared__ double row_loss[PROBE_R];
    __shared__ int row_ok[PROBE_R];
    const int t = threadIdx.x;
    const int row0 = blockIdx.x * PROBE_R;
    const int nr = min(PROBE_R, B - row0);

    float acc[PROBE_R];
#pragma unroll
    for (int r = 0; r < PROBE_R; ++r) acc[r] = 0.f;
    for (int k0 = 0; k0 < O; k0 += PROBE_KT) {
        const int kw = min(PROBE_KT, O - k0);          // a multiple of 4
        // W1[:, k0:k0+kw] -> w1s (float4 loads along k)
        for (int i = t; i < PROBE_H * (PROBE_KT / 4); i += PROBE_H) {
            const int j = i / (PROBE_KT / 4), q = (i % (PROBE_KT / 4)) * 4;
            float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
            if (q < kw) v = __ldg(reinterpret_cast<const float4*>(w1 + (int64_t)j * O + k0 + q));
            w1s[j][q] = v.x;
            w1s[j][q + 1] = v.y;
            w1s[j][q + 2] = v.z;
            w1s[j][q + 3] = v.w;
        }
        for (int i = t; i < PROBE_R * (PROBE_KT / 4); i += PROBE_H) {
            const int r = i / (PROBE_KT / 4), q = (i % (PROBE_KT / 4)) * 4;
            float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
            if (r < nr && q < kw) v = __ldg(reinterpret_cast<const float4*>(x + (int64_t)(row0 + r) * O + k0 + q));
            *reinterpret_cast<float4*>(&xs[r][q]) = v;
        }
        __syncthreads();
        for (int kk = 0; kk < kw; ++kk) {
            const float wv = w1s[t][kk];
#pragma unroll
            for (int r = 0; r < PROBE_R; ++r) acc[r] = fmaf(xs[r][kk], wv, acc[r]);
        }
        __syncthreads();
    }
    const float bj = __ldg(b1 + t);
#pragma unroll
    for (int r = 0; r < PROBE_R; ++r) {
        const float h = fmaxf(acc[r] + bj, 0.f);
        hs[r][t] = h;
        if (TRAIN && r < nr) w.h[(int64_t)(row0 + r) * PROBE_H + t] = h;
    }
    for (int c = 0; c < C; ++c) w2s[c][t] = __ldg(w2 + c * PROBE_H + t);
    __syncthreads();

    // logits: PROBE_R x C dot products of length 128, fixed order
    for (int i = t; i < PROBE_R * C; i += PROBE_H) {
        const int r = i / C, c = i % C;
        float s = 0.f;
        for (int j = 0; j < PROBE_H; ++j) s = fmaf(hs[r][j], w2s[c][j], s);
        ls[r][c] = s + __ldg(b2 + c);
    }
    __syncthreads();

    // per row: loss, argmax, d_logits
    if (t < PROBE_R) {
        const int r = t;
        double loss = 0.0;
        int ok = 0;
        if (r < nr) {
            const int64_t lab = labels[row0 + r];
            float mx = ls[r][0];
            int am = 0;
            for (int c = 1; c < C; ++c)
                if (ls[r][c] > mx) {
                    mx = ls[r][c];
                    am = c;
                }
            float se = 0.f;
            for (int c = 0; c < C; ++c) se += expf(ls[r][c] - mx);
            const float lse = mx + logf(se);
            const bool valid = lab >= 0 && lab < C;
            loss = valid ? (double)(lse - ls[r][(int)lab]) : (double)NAN;
            ok = valid && am == (int)lab;
            if (TRAIN) {
                const float inv_b = 1.f / (float)B;
                for (int c = 0; c < C; ++c) {
                    const float p = expf(ls[r][c] - lse);
                    const float d = (p - (c == lab ? 1.f : 0.f)) * inv_b;
                    ls[r][c] = d;
                    w.dlog[(int64_t)(row0 + r) * C + c] = d;
                }
            } else {
                if (preds) preds[row0 + r] = am;
                if (confusion && valid) atomicAdd(confusion + lab * C + am, 1ull);
            }
        }
        row_loss[r] = loss;
        row_ok[r] = ok;
    }
    __syncthreads();
    if (t == 0) {
        double s = 0.0;
        int n_ok = 0;
        for (int r = 0; r < PROBE_R; ++r) {
            s += row_loss[r];
            n_ok += row_ok[r];
        }
        w.part[blockIdx.x] = s;
        if (n_ok) atomicAdd(correct, (unsigned long long)n_ok);
    }
    if (TRAIN) {
        for (int r = 0; r < nr; ++r) {
            float d = 0.f;
            for (int c = 0; c < C; ++c) d = fmaf(ls[r][c], w2s[c][t], d);
            w.dh[(int64_t)(row0 + r) * PROBE_H + t] = hs[r][t] > 0.f ? d : 0.f;
        }
    }
}

// blockIdx.x < n_tiles: a 32 x 32 tile of dW1 = d_hidden^T x (thread: one hidden unit x 4 feature columns);
// n_tiles <= blockIdx.x < n_tiles + n_w2 (= C, or 0 without a backward): row c of dW2 = d_logits[:, c]^T hidden; the last CTA: db1, db2 and the loss sum.
__global__ void __launch_bounds__(256) probe_grads_kernel(const float* __restrict__ x, int B, int O, int C, ProbeWork w, int n_tiles,
                                                          int n_w2, int n_row_blocks, float* __restrict__ grad, double* __restrict__ loss_sum) {
    const int t = threadIdx.x;
    const int bid = blockIdx.x;
    if (bid < n_tiles) {
        __shared__ float dhs[PROBE_T][PROBE_T];
        __shared__ __align__(16) float xs[PROBE_T][PROBE_T];
        const int tiles_k = (O + PROBE_T - 1) / PROBE_T;
        const int j0 = (bid / tiles_k) * PROBE_T, kt0 = (bid % tiles_k) * PROBE_T;
        const int tj = t / 8, tk = (t % 8) * 4;
        const int kw = min(PROBE_T, O - kt0);
        float a0 = 0.f, a1 = 0.f, a2 = 0.f, a3 = 0.f;
        for (int r0 = 0; r0 < B; r0 += PROBE_T) {
            const int nr = min(PROBE_T, B - r0);
            for (int i = t; i < PROBE_T * PROBE_T; i += 256) {
                const int r = i / PROBE_T, c = i % PROBE_T;
                dhs[r][c] = r < nr ? w.dh[(int64_t)(r0 + r) * PROBE_H + j0 + c] : 0.f;
                xs[r][c] = (r < nr && c < kw) ? __ldg(x + (int64_t)(r0 + r) * O + kt0 + c) : 0.f;
            }
            __syncthreads();
            for (int r = 0; r < nr; ++r) {
                const float d = dhs[r][tj];
                const float4 xv = *reinterpret_cast<const float4*>(&xs[r][tk]);
                a0 = fmaf(d, xv.x, a0);
                a1 = fmaf(d, xv.y, a1);
                a2 = fmaf(d, xv.z, a2);
                a3 = fmaf(d, xv.w, a3);
            }
            __syncthreads();
        }
        if (tk < kw) {       // kw is a multiple of 4
            float* g = grad + (int64_t)(j0 + tj) * O + kt0 + tk;
            g[0] = a0;
            g[1] = a1;
            g[2] = a2;
            g[3] = a3;
        }
        return;
    }
    float* gb1 = grad + (int64_t)PROBE_H * O;
    float* gw2 = gb1 + PROBE_H;
    float* gb2 = gw2 + PROBE_H * C;
    if (bid < n_tiles + n_w2) {
        const int c = bid - n_tiles;
        if (t < PROBE_H) {
            float s = 0.f;
            for (int r = 0; r < B; ++r) s = fmaf(w.dlog[(int64_t)r * C + c], w.h[(int64_t)r * PROBE_H + t], s);
            gw2[c * PROBE_H + t] = s;
        }
        return;
    }
    if (grad != nullptr) {
        if (t < PROBE_H) {
            float s = 0.f;
            for (int r = 0; r < B; ++r) s += w.dh[(int64_t)r * PROBE_H + t];
            gb1[t] = s;
        } else if (t - PROBE_H < C) {
            const int c = t - PROBE_H;
            float s = 0.f;
            for (int r = 0; r < B; ++r) s += w.dlog[(int64_t)r * C + c];
            gb2[c] = s;
        }
    }
    if (t == 0) {
        double s = 0.0;
        for (int b = 0; b < n_row_blocks; ++b) s += w.part[b];
        *loss_sum += s;
    }
}

}  // namespace b200

using namespace b200;

extern "C" {

int64_t b200_probe_work_floats(int B, int C) {
    if (B < 1 || C < 1 || C > PROBE_CMAX) return B200_E_SHAPE;
    return probe_part_floats(B) + (int64_t)B * (2 * PROBE_H + C);
}

int b200_probe_mlp_fwd_bwd(const float* x, const float* w1, const float* b1, const float* w2, const float* b2, const int64_t* labels,
                           int B, int O, int C, int train, float* grad, float* work, double* loss_sum, int64_t* correct,
                           int64_t* preds, int64_t* confusion, void* stream) {
    B200_REQUIRE(x && w1 && b1 && w2 && b2 && labels && work && loss_sum && correct, B200_E_ARG, "probe_mlp_fwd_bwd: null pointer");
    B200_REQUIRE(!train || grad, B200_E_ARG, "probe_mlp_fwd_bwd: train = 1 needs the gradient arena");
    B200_REQUIRE(B >= 1 && O >= 64 && O <= 1024 && O % 4 == 0 && C >= 1 && C <= PROBE_CMAX, B200_E_SHAPE,
                 "probe_mlp_fwd_bwd: need B >= 1, O in 64..1024 (multiple of 4), C in 1..16 (got B=%d O=%d C=%d)", B, O, C);
    B200_REQUIRE((((uintptr_t)x | (uintptr_t)w1 | (uintptr_t)work) & 15) == 0, B200_E_ARG,
                 "probe_mlp_fwd_bwd: x, w1 and work must be 16-byte aligned");
    const cudaStream_t s = as_stream(stream);
    const ProbeWork w = probe_work(work, B);
    const int nb = probe_row_blocks(B);
    auto* cnt = reinterpret_cast<unsigned long long*>(correct);
    auto* conf = reinterpret_cast<unsigned long long*>(confusion);
    if (train) {
        probe_rows_kernel<true><<<nb, PROBE_H, 0, s>>>(x, w1, b1, w2, b2, labels, B, O, C, w, cnt, nullptr, nullptr);
        const int n_tiles = (PROBE_H / PROBE_T) * ((O + PROBE_T - 1) / PROBE_T);
        probe_grads_kernel<<<n_tiles + C + 1, 256, 0, s>>>(x, B, O, C, w, n_tiles, C, nb, grad, loss_sum);
    } else {
        probe_rows_kernel<false><<<nb, PROBE_H, 0, s>>>(x, w1, b1, w2, b2, labels, B, O, C, w, cnt, preds, conf);
        probe_grads_kernel<<<1, 256, 0, s>>>(x, B, O, C, w, 0, 0, nb, nullptr, loss_sum);
    }
    return launch_status("probe_mlp_fwd_bwd");
}

}  // extern "C"
