// Fused multi-crop augmentation for AVMNIST: one CTA stages one (sample, view) in shared memory, runs the whole
// op chain there (ping-pong buffers, every op in the reference's own order and fp32 arithmetic) and writes the
// finished view once.  HBM traffic = source read (re-reads by the other views hit L2) + one write per view:
// the algorithmic minimum of SURVEY §8(d) (373,184 B / sample for 2 global + 4 local views of both modalities).
//
// Arithmetic restated from the third-party transforms the reference calls (SURVEY Appendix A1-A5), pinned
// against torch 2.11 / torchvision 0.26 / torchaudio 2.11 CPU through oracle/augment_ref.py:
//   * nearest rotate/affine: integer gather, grid = fma(y, r1, x*r0) + r2 (ATen's bmm order), round-half-even;
//   * antialiased bilinear resize: ATen's separable weight tables (fp32 weights, double index math), FMA sums;
//   * time warp: linear interpolation of |x| at torch.arange(0, W, rate) time steps (vectorised-arange rounding);
//   * frequency/time masks, grouped 4x4 masking, erasing, additive gaussian noise.
#include <cuda_bf16.h>

#include "common.cuh"

namespace b200 {

enum { OP_NOP = 0, OP_CROP_RESIZE, OP_AFFINE, OP_ERASE, OP_FREQ_MASK, OP_TIME_MASK, OP_NOISE, OP_GROUP_MASK, OP_TIME_WARP, OP_BLUR3, OP_ELASTIC };
enum { SPEC_RRC = 1, SPEC_ROTATE, SPEC_AFFINE, SPEC_ERASE, SPEC_FREQ_MASK, SPEC_TIME_MASK, SPEC_NOISE, SPEC_GROUP_MASK, SPEC_TIME_WARP, SPEC_BLUR,
       SPEC_ELASTIC };

struct AATable {  // per output index: first source index, tap count, up to 3 weights
    int lo;
    int n;
    float w[3];
};

__device__ __forceinline__ void aa_entry(int i, int in_size, int out_size, AATable& e) {
    const float scale = __fdiv_rn((float)in_size, (float)out_size);
    const float support = (scale >= 1.0f) ? scale : 1.0f;
    const float invscale = (scale >= 1.0f) ? (float)(1.0 / (double)scale) : 1.0f;
    const float center = (float)((double)scale * ((double)i + 0.5));
    int lo = (int)((double)center - (double)support + 0.5);
    lo = lo < 0 ? 0 : lo;
    int hi = (int)((double)center + (double)support + 0.5);
    hi = hi > in_size ? in_size : hi;
    int n = hi - lo;
    n = n < 0 ? 0 : (n > 3 ? 3 : n);
    float total = 0.f;
    float w[3] = {0.f, 0.f, 0.f};
    for (int j = 0; j < n; ++j) {
        float t = (float)(((double)(j + lo) - (double)center + 0.5) * (double)invscale);
        t = fabsf(t);
        w[j] = t < 1.0f ? __fsub_rn(1.0f, t) : 0.f;
        total = __fadd_rn(total, w[j]);
    }
    if (total != 0.f) {
        const float norm = (float)(1.0 / (double)total);
        for (int j = 0; j < n; ++j) w[j] = __fmul_rn(w[j], norm);
    }
    e.lo = lo;
    e.n = n;
    e.w[0] = w[0];
    e.w[1] = w[1];
    e.w[2] = w[2];
}

// torch.arange(0, stop, step, float32)[k] as ATen's CPU kernel rounds it (see oracle/augment_ref.py arange_f32)
__device__ __forceinline__ float arange_f32(int k, int n, double step) {
    if (k < (n / 16) * 16) {
        int i8 = k & ~7;
        float base = (float)((double)i8 * step);
        return (float)((double)base + (double)(k & 7) * step);
    }
    return (float)((double)k * step);
}

template <int S, int T>
__global__ void __launch_bounds__(T) aug_apply_kernel(const void* __restrict__ src, int src_u8, const int32_t* __restrict__ ops,
                                                      const uint32_t* __restrict__ group_bits, const float* __restrict__ noise,
                                                      uint64_t seed, float* __restrict__ out, uint4* __restrict__ out8, int pad8, int B, int V,
                                                      const int64_t* __restrict__ step_dev, const float* __restrict__ egrid) {
    constexpr int NPIX = S * S;
    if (step_dev != nullptr) seed = (seed + (uint64_t)__ldg(step_dev)) & 0xFFFFFFFFFFFFull;      // CUDA-graph replay: the step lives on the device
    extern __shared__ __align__(16) unsigned char smem_raw[];
    float* bufA = reinterpret_cast<float*>(smem_raw);
    float* bufB = bufA + NPIX;
    AATable* xtab = reinterpret_cast<AATable*>(bufB + NPIX);
    AATable* ytab = xtab + S;
    __shared__ int32_t sops[B200_AUG_MAX_OPS * 8];
    __shared__ uint32_t sbits[B200_AUG_GROUP_WORDS];
    __shared__ float u8lut[256];          // v / 255 exactly as the reference computes it (float64 division, rounded to fp32)
    __shared__ float tw_alpha[S];         // time-warp per-column tables
    __shared__ int tw_i0[S];

    const int tid = threadIdx.x;
    const int b = blockIdx.x / V, v = blockIdx.x - b * V;
    const size_t rec = (size_t)b * V + v;
    if (tid < B200_AUG_MAX_OPS * 8) sops[tid] = __ldg(ops + rec * (B200_AUG_MAX_OPS * 8) + tid);
    if (group_bits != nullptr && tid < B200_AUG_GROUP_WORDS) sbits[tid] = __ldg(group_bits + rec * B200_AUG_GROUP_WORDS + tid);

    // ---- stage the source (coalesced, vectorised) ----
    if (src_u8) {
        for (int i = tid; i < 256; i += T) u8lut[i] = (float)((double)i / 255.0);
        __syncthreads();
        const uint32_t* s4 = reinterpret_cast<const uint32_t*>(reinterpret_cast<const uint8_t*>(src) + (size_t)b * NPIX);
        for (int i = tid; i < NPIX / 4; i += T) {
            const uint32_t w = __ldg(s4 + i);
            reinterpret_cast<float4*>(bufA)[i] = make_float4(u8lut[w & 0xff], u8lut[(w >> 8) & 0xff], u8lut[(w >> 16) & 0xff], u8lut[w >> 24]);
        }
    } else {
        const float4* s4 = reinterpret_cast<const float4*>(reinterpret_cast<const float*>(src) + (size_t)b * NPIX);
        for (int i = tid; i < NPIX / 4; i += T) reinterpret_cast<float4*>(bufA)[i] = __ldg(s4 + i);
    }
    __syncthreads();

    float* cur = bufA;
    float* alt = bufB;
    for (int k = 0; k < B200_AUG_MAX_OPS; ++k) {
        const int kind = sops[k * 8];
        const int32_t* p = sops + k * 8 + 1;
        if (kind == OP_NOP) continue;
        if (kind == OP_CROP_RESIZE) {
            const int ci = p[0], cj = p[1], ch = p[2], cw = p[3];
            for (int i = tid; i < 2 * S; i += T) {
                if (i < S) aa_entry(i, cw, S, xtab[i]);
                else aa_entry(i - S, ch, S, ytab[i - S]);
            }
            __syncthreads();
            // horizontal: alt[r][o] for r < ch
            for (int e = tid; e < ch * S; e += T) {
                const int r = e / S, o = e - r * S;
                const AATable te = xtab[o];
                const float* row = cur + (ci + r) * S + cj + te.lo;
                float acc = 0.f;
                if (te.n > 0) acc = __fmul_rn(row[0], te.w[0]);
                if (te.n > 1) acc = __fmaf_rn(row[1], te.w[1], acc);
                if (te.n > 2) acc = __fmaf_rn(row[2], te.w[2], acc);
                alt[e] = acc;
            }
            __syncthreads();
            // vertical: cur[o][x]
            for (int e = tid; e < NPIX; e += T) {
                const int o = e / S, x = e - o * S;
                const AATable te = ytab[o];
                const float* col = alt + te.lo * S + x;
                float acc = 0.f;
                if (te.n > 0) acc = __fmul_rn(col[0], te.w[0]);
                if (te.n > 1) acc = __fmaf_rn(col[S], te.w[1], acc);
                if (te.n > 2) acc = __fmaf_rn(col[2 * S], te.w[2], acc);
                cur[e] = acc;
            }
            __syncthreads();
        } else if (kind == OP_AFFINE) {
            const float half = 0.5f * (float)S;
            const float r00 = __fdiv_rn(__int_as_float(p[0]), half), r10 = __fdiv_rn(__int_as_float(p[1]), half),
                        r20 = __fdiv_rn(__int_as_float(p[2]), half);
            const float r01 = __fdiv_rn(__int_as_float(p[3]), half), r11 = __fdiv_rn(__int_as_float(p[4]), half),
                        r21 = __fdiv_rn(__int_as_float(p[5]), half);
            const float off = -(float)S * 0.5f + 0.5f;
            for (int e = tid; e < NPIX; e += T) {
                const int y = e / S, x = e - y * S;
                const float xs = (float)x + off, ys = (float)y + off;
                const float gx = __fadd_rn(__fmaf_rn(ys, r10, __fmul_rn(xs, r00)), r20);
                const float gy = __fadd_rn(__fmaf_rn(ys, r11, __fmul_rn(xs, r01)), r21);
                const float ix = __fmul_rn(__fsub_rn(__fmul_rn(__fadd_rn(gx, 1.0f), (float)S), 1.0f), 0.5f);     // x/2 == x*0.5 exactly
                const float iy = __fmul_rn(__fsub_rn(__fmul_rn(__fadd_rn(gy, 1.0f), (float)S), 1.0f), 0.5f);
                const float fx = rintf(ix), fy = rintf(iy);
                float val = 0.f;
                if (fx >= 0.f && fx < (float)S && fy >= 0.f && fy < (float)S) val = cur[(int)fy * S + (int)fx];
                alt[e] = val;
            }
            __syncthreads();
            float* t = cur; cur = alt; alt = t;
        } else if (kind == OP_ERASE) {
            const int ei = p[0], ej = p[1], eh = p[2], ew = p[3];
            for (int e = tid; e < eh * ew; e += T) {
                const int r = e / ew, c = e - r * ew;
                cur[(ei + r) * S + ej + c] = 0.f;
            }
            __syncthreads();
        } else if (kind == OP_FREQ_MASK) {
            const int s0 = p[0], s1 = p[1];
            for (int e = tid; e < (s1 - s0) * S; e += T) cur[s0 * S + e] = 0.f;
            __syncthreads();
        } else if (kind == OP_TIME_MASK) {
            const int s0 = p[0], n = p[1] - p[0];
            for (int e = tid; e < n * S; e += T) {
                const int y = e / n, c = e - y * n;
                cur[y * S + s0 + c] = 0.f;
            }
            __syncthreads();
        } else if (kind == OP_NOISE) {
            const float std = __int_as_float(p[0]);
            if (noise != nullptr) {
                const float* nz = noise + rec * NPIX;
                for (int e = tid; e < NPIX; e += T) cur[e] = __fadd_rn(cur[e], __fmul_rn(__ldg(nz + e), std));
            } else {
                Philox rng(seed);
                for (int q = tid; q < NPIX / 4; q += T) {
                    uint4 r = rng((uint64_t)q, (uint64_t)rec * 4 + 1);
                    // two Box-Muller pairs
                    float u1 = 1.0f - u01(r.x), u2 = u01(r.y), u3 = 1.0f - u01(r.z), u4 = u01(r.w);
                    // device-sampled noise only has to be N(0, 1): hardware log / sin / cos approximations (2^-21 abs) are enough
                    float ra = sqrtf(-2.0f * __logf(u1)), rb = sqrtf(-2.0f * __logf(u3));
                    float s1, c1, s2, c2;
                    __sincosf(6.283185307179586f * u2, &s1, &c1);
                    __sincosf(6.283185307179586f * u4, &s2, &c2);
                    cur[4 * q + 0] += ra * c1 * std;
                    cur[4 * q + 1] += ra * s1 * std;
                    cur[4 * q + 2] += rb * c2 * std;
                    cur[4 * q + 3] += rb * s2 * std;
                }
            }
            __syncthreads();
        } else if (kind == OP_GROUP_MASK) {
            // 4 x 4 pixel groups: iterate over (group, row-in-group) = one aligned float4 each; only masked groups write
            constexpr int GW = S / 4, NG = GW * GW;
            for (int e = tid; e < NG * 4; e += T) {
                const int g = e >> 2, r = e & 3;
                if ((sbits[g >> 5] >> (g & 31)) & 1u) {
                    const int gy = g / GW, gx = g - gy * GW;
                    reinterpret_cast<float4*>(cur + (gy * 4 + r) * S)[gx] = make_float4(0.f, 0.f, 0.f, 0.f);
                }
            }
            __syncthreads();
        } else if (kind == OP_TIME_WARP) {
            const double rate = __hiloint2double(p[1], p[0]);
            const int n_frames = (int)ceil((double)S / rate);
            for (int kx = tid; kx < S; kx += T) {            // the interpolation position depends on the column only
                const float ts = kx < n_frames ? arange_f32(kx, n_frames, rate) : 0.f;
                tw_alpha[kx] = fmodf(ts, 1.0f);
                tw_i0[kx] = kx < n_frames ? (int)ts : -1;
            }
            __syncthreads();
            for (int e = tid; e < NPIX; e += T) {
                const int y = e / S, kx = e - y * S;
                float val = 0.f;
                const int i0 = tw_i0[kx];
                if (i0 >= 0) {
                    const float alpha = tw_alpha[kx];
                    const float n0 = i0 < S ? fabsf(cur[y * S + i0]) : 0.f;
                    const float n1 = (i0 + 1) < S ? fabsf(cur[y * S + i0 + 1]) : 0.f;
                    val = __fadd_rn(__fmul_rn(alpha, n1), __fmul_rn(__fsub_rn(1.0f, alpha), n0));
                }
                alt[e] = val;
            }
            __syncthreads();
            float* t = cur; cur = alt; alt = t;
        } else if (kind == OP_BLUR3) {
            // torchvision GaussianBlur(3): reflect padding, kernel2d = k (outer) k, fp32 FMA accumulation row by row (get_data.py:337)
            const float k0 = __int_as_float(p[0]), k1 = __int_as_float(p[1]), k2 = __int_as_float(p[2]);
            const float kk[3] = {k0, k1, k2};
            for (int e = tid; e < NPIX; e += T) {
                const int y = e / S, x = e - y * S;
                float acc = 0.f;
#pragma unroll
                for (int i = 0; i < 3; ++i) {
                    int yy = y + i - 1;
                    yy = yy < 0 ? -yy : (yy >= S ? 2 * S - 2 - yy : yy);
#pragma unroll
                    for (int j = 0; j < 3; ++j) {
                        int xx = x + j - 1;
                        xx = xx < 0 ? -xx : (xx >= S ? 2 * S - 2 - xx : xx);
                        acc = __fmaf_rn(cur[yy * S + xx], __fmul_rn(kk[i], kk[j]), acc);
                    }
                }
                alt[e] = acc;
            }
            __syncthreads();
            float* t = cur; cur = alt; alt = t;
        } else if (kind == OP_ELASTIC) {
            // torchvision ElasticTransform (get_data.py:330): bilinear grid_sample (zeros padding, align_corners=False) of the image and
            // of a ones mask at grid = identity + displacement, out = img * mask.  Parity mode: the grid [2,S,S] comes from the host
            // (egrid); throughput mode: the displacement field is drawn here (uniform field, separable Gaussian blur, reflect padding).
            const float* gxp = nullptr;
            const float* gyp = nullptr;
            if (egrid != nullptr) {
                gxp = egrid + rec * 2 * NPIX;
                gyp = gxp + NPIX;
            }
            if constexpr (S <= 32) {
                __shared__ float fld[3 * S * S];                   // dx, dy, scratch
                if (egrid == nullptr) {
                    const float alpha = __int_as_float(p[0]), sigma = __int_as_float(p[1]);
                    int kr = (int)(8.f * sigma + 1.f);
                    kr = (kr | 1) / 2;                              // radius of the odd kernel size
                    if (kr > S - 1) kr = S - 1;
                    Philox rng(seed);
                    for (int q = tid; q < NPIX / 2; q += T) {       // 2 * NPIX uniforms in [-1, 1)
                        const uint4 r = rng((uint64_t)q, (uint64_t)rec * 4 + 2);
                        fld[4 * q + 0] = 2.f * u01(r.x) - 1.f;
                        fld[4 * q + 1] = 2.f * u01(r.y) - 1.f;
                        fld[4 * q + 2] = 2.f * u01(r.z) - 1.f;
                        fld[4 * q + 3] = 2.f * u01(r.w) - 1.f;
                    }
                    __syncthreads();
                    const float inv2s2 = sigma > 0.f ? 0.5f / (sigma * sigma) : 0.f;
                    float norm = 0.f;
                    for (int d = -kr; d <= kr; ++d) norm += __expf(-(float)(d * d) * inv2s2);
                    for (int f = 0; f < 2 && sigma > 0.f; ++f) {    // separable blur of field f: rows into scratch, columns back
                        float* src_f = fld + f * NPIX;
                        float* tmp = fld + 2 * NPIX;
                        for (int e = tid; e < NPIX; e += T) {
                            const int y = e / S, x = e - y * S;
                            float a = 0.f;
                            for (int d = -kr; d <= kr; ++d) {
                                int xx = x + d;
                                xx = xx < 0 ? -xx : (xx >= S ? 2 * S - 2 - xx : xx);
                                a += src_f[y * S + xx] * __expf(-(float)(d * d) * inv2s2);
                            }
                            tmp[e] = a / norm;
                        }
                        __syncthreads();
                        for (int e = tid; e < NPIX; e += T) {
                            const int y = e / S, x = e - y * S;
                            float a = 0.f;
                            for (int d = -kr; d <= kr; ++d) {
                                int yy = y + d;
                                yy = yy < 0 ? -yy : (yy >= S ? 2 * S - 2 - yy : yy);
                                a += tmp[yy * S + x] * __expf(-(float)(d * d) * inv2s2);
                            }
                            src_f[e] = a / norm * alpha / (float)S;
                        }
                        __syncthreads();
                    }
                    for (int e = tid; e < NPIX; e += T) {           // + identity grid
                        const int y = e / S, x = e - y * S;
                        fld[e] += (2.f * (float)x + 1.f) / (float)S - 1.f;
                        fld[NPIX + e] += (2.f * (float)y + 1.f) / (float)S - 1.f;
                    }
                    __syncthreads();
                    gxp = fld;
                    gyp = fld + NPIX;
                }
            }
            if (gxp != nullptr) {
                for (int e = tid; e < NPIX; e += T) {
                    const float gx = gxp[e], gy = gyp[e];
                    const float ix = __fsub_rn(__fmul_rn(__fadd_rn(gx, 1.f), 0.5f * (float)S), 0.5f);
                    const float iy = __fsub_rn(__fmul_rn(__fadd_rn(gy, 1.f), 0.5f * (float)S), 0.5f);
                    const float fx = floorf(ix), fy = floorf(iy);
                    const float w = __fsub_rn(ix, fx), ee = __fsub_rn(1.f, w), n = __fsub_rn(iy, fy), sn = __fsub_rn(1.f, n);
                    const int x0 = (int)fx, y0 = (int)fy;
                    float img = 0.f, msk = 0.f;
                    const float wt[4] = {__fmul_rn(sn, ee), __fmul_rn(sn, w), __fmul_rn(n, ee), __fmul_rn(n, w)};
#pragma unroll
                    for (int c = 0; c < 4; ++c) {
                        const int xx = x0 + (c & 1), yy = y0 + (c >> 1);
                        if (xx >= 0 && xx < S && yy >= 0 && yy < S) {
                            img = __fmaf_rn(cur[yy * S + xx], wt[c], img);
                            msk = __fadd_rn(msk, wt[c]);
                        }
                    }
                    alt[e] = __fmul_rn(img, msk);
                }
                __syncthreads();
                float* t = cur; cur = alt; alt = t;
            }
        }
    }
    // ---- write the finished view (view-major layout [V,B,S,S]) ----
    if (out != nullptr) {
        float4* o4 = reinterpret_cast<float4*>(out + ((size_t)v * B + b) * NPIX);
        for (int i = tid; i < NPIX / 4; i += T) o4[i] = reinterpret_cast<const float4*>(cur)[i];
    }
    // ---- and / or the bf16 "quad8" image of the first-layer tensor-core convolution: [V,B,S,WQ,8], WQ = ceil((S + 2 pad) / 4),
    //      unit (y, xq) = the zero-padded row's pixels 4xq .. 4xq+7 (padded column c = image column c - pad); see conv_tc.cu ----
    if (out8 != nullptr) {
        const int WQ = (S + 2 * pad8 + 3) / 4;
        uint4* o8 = out8 + ((size_t)v * B + b) * S * WQ;
        for (int i = tid; i < S * WQ; i += T) {
            const int y = i / WQ, xq = i - y * WQ;
            const float* r = cur + y * S;
            float f[8];
            const int x0 = 4 * xq - pad8;
            if ((pad8 & 1) == 0 && x0 >= 0 && x0 + 8 <= S) {          // interior unit, 8-byte aligned: four 64-bit shared loads
#pragma unroll
                for (int c = 0; c < 4; ++c) {
                    const float2 v2 = *reinterpret_cast<const float2*>(r + x0 + 2 * c);
                    f[2 * c] = v2.x;
                    f[2 * c + 1] = v2.y;
                }
            } else {
#pragma unroll
                for (int c = 0; c < 8; ++c) {
                    const int xc = x0 + c;
                    f[c] = (xc >= 0 && xc < S) ? r[xc] : 0.f;
                }
            }
            __nv_bfloat162 p0 = __floats2bfloat162_rn(f[0], f[1]), p1 = __floats2bfloat162_rn(f[2], f[3]);
            __nv_bfloat162 p2 = __floats2bfloat162_rn(f[4], f[5]), p3 = __floats2bfloat162_rn(f[6], f[7]);
            o8[i] = make_uint4(*reinterpret_cast<uint32_t*>(&p0), *reinterpret_cast<uint32_t*>(&p1), *reinterpret_cast<uint32_t*>(&p2),
                               *reinterpret_cast<uint32_t*>(&p3));
        }
    }
}

// ---------------------------------------------------------------------------------------------------------
// Device-side parameter sampling (throughput mode).  Same distributions as the host sampler (augment.py), drawn
// from Philox(seed; stream = step, sample, view, modality).  One CTA per (sample, view); thread 0 walks the two
// chains, all threads cooperate on the grouped-masking subset selection.
// ---------------------------------------------------------------------------------------------------------
struct Draw {
    Philox rng;
    uint64_t stream;
    uint64_t ctr;
    __device__ Draw(uint64_t seed, uint64_t s) : rng(seed), stream(s), ctr(0) {}
    __device__ uint32_t bits() { return rng(ctr++, stream).x; }
    __device__ float uniform(float lo, float hi) { return u01(bits()) * (hi - lo) + lo; }   // torch uniform_ on float
    __device__ float rand01() { return u01(bits()); }
    __device__ int randint(int n) { return (int)(bits() % (uint32_t)n); }
};

__device__ void store_affine(int32_t* rec, double angle_deg, double tx, double ty, double scale) {
    const double rot = angle_deg * 0.017453292519943295;
    const double a = cos(rot), b = -sin(rot), c = sin(rot), d = cos(rot);
    double m[6] = {d / scale, -b / scale, 0.0, -c / scale, a / scale, 0.0};
    m[2] += m[0] * (-tx) + m[1] * (-ty);
    m[5] += m[3] * (-tx) + m[4] * (-ty);
    rec[0] = OP_AFFINE;
    for (int i = 0; i < 6; ++i) rec[1 + i] = __float_as_int((float)m[i]);
}

__device__ int sample_chain(const int32_t* spec, int S, Draw& d, int32_t* rec /*[MAX_OPS*8]*/, int* group_count) {
    int n_out = 0;
    *group_count = -1;
    for (int i = 0; i < B200_AUG_MAX_OPS * 8; ++i) rec[i] = 0;     // unused payload words are defined (zero)
    for (int k = 0; k < B200_AUG_MAX_OPS; ++k) {
        const int kind = spec[k * 8];
        if (kind == 0) continue;
        const float p = __int_as_float(spec[k * 8 + 1]);
        float a[6];
        for (int i = 0; i < 6; ++i) a[i] = __int_as_float(spec[k * 8 + 2 + i]);
        int32_t* r = rec + n_out * 8;
        if (kind == SPEC_ERASE) {
            if (!(d.rand01() < p)) continue;
            const double area = (double)S * S;
            for (int t = 0; t < 10; ++t) {
                const double ea = area * (double)d.uniform(a[0], a[1]);
                const double ar = (double)expf(d.uniform(a[2], a[3]));
                const int h = (int)rint(sqrt(ea * ar)), w = (int)rint(sqrt(ea / ar));
                if (!(h < S && w < S)) continue;
                r[0] = OP_ERASE;
                r[1] = d.randint(S - h + 1);
                r[2] = d.randint(S - w + 1);
                r[3] = h;
                r[4] = w;
                ++n_out;
                break;
            }
            continue;
        }
        if (p >= 0.f && p < d.rand01()) continue;   // RandomApply: skip iff p < r
        if (kind == SPEC_RRC) {
            const double area = (double)S * S;
            bool done = false;
            int ci = 0, cj = 0, ch = S, cw = S;
            for (int t = 0; t < 10 && !done; ++t) {
                const double target = area * (double)d.uniform(a[0], a[1]);
                const double ar = (double)expf(d.uniform(a[2], a[3]));
                const int w = (int)rint(sqrt(target * ar)), h = (int)rint(sqrt(target / ar));
                if (w > 0 && w <= S && h > 0 && h <= S) {
                    ci = d.randint(S - h + 1);
                    cj = d.randint(S - w + 1);
                    ch = h;
                    cw = w;
                    done = true;
                }
            }
            if (!done) {  // central-crop fallback (square input: in_ratio == 1)
                const float rlo = expf(a[2]), rhi = expf(a[3]);
                if (1.0f < fminf(rlo, rhi)) { cw = S; ch = (int)rint((double)S / fminf(rlo, rhi)); }
                else if (1.0f > fmaxf(rlo, rhi)) { ch = S; cw = (int)rint((double)S * fmaxf(rlo, rhi)); }
                ci = (S - ch) / 2;
                cj = (S - cw) / 2;
            }
            r[0] = OP_CROP_RESIZE; r[1] = ci; r[2] = cj; r[3] = ch; r[4] = cw;
            ++n_out;
        } else if (kind == SPEC_ROTATE) {
            const double angle = (double)d.uniform(-a[0], a[0]);
            store_affine(r, -angle, 0.0, 0.0, 1.0);
            ++n_out;
        } else if (kind == SPEC_AFFINE) {
            const double angle = (double)d.uniform(-a[0], a[0]);
            const int flags = (int)a[5];
            double tx = 0.0, ty = 0.0, sc = 1.0;
            if (flags & 2) {
                const float mdx = a[1] * (float)S, mdy = a[2] * (float)S;
                tx = rint((double)d.uniform(-mdx, mdx));
                ty = rint((double)d.uniform(-mdy, mdy));
            }
            if (flags & 1) sc = (double)d.uniform(a[3], a[4]);
            store_affine(r, angle, tx, ty, sc);
            ++n_out;
        } else if (kind == SPEC_FREQ_MASK || kind == SPEC_TIME_MASK) {
            const int param = (int)a[0];
            if (param < 1) continue;
            const float value = d.rand01() * (float)param;
            const float minv = d.rand01() * ((float)S - value);
            r[0] = kind == SPEC_FREQ_MASK ? OP_FREQ_MASK : OP_TIME_MASK;
            r[1] = (int)minv;
            r[2] = (int)minv + (int)value;
            ++n_out;
        } else if (kind == SPEC_NOISE) {
            r[0] = OP_NOISE;
            r[1] = __float_as_int(a[0]);
            ++n_out;
        } else if (kind == SPEC_GROUP_MASK) {
            r[0] = OP_GROUP_MASK;
            *group_count = (int)a[0];
            ++n_out;
        } else if (kind == SPEC_BLUR) {
            const float sigma = d.uniform(a[0], a[1]);               // GaussianBlur.get_params; taps of the 3-wide kernel
            const float e1 = expf(-0.5f / (sigma * sigma)), inv = 1.0f / (1.0f + 2.0f * e1);
            r[0] = OP_BLUR3;
            r[1] = __float_as_int(e1 * inv);
            r[2] = __float_as_int(inv);
            r[3] = __float_as_int(e1 * inv);
            ++n_out;
        } else if (kind == SPEC_ELASTIC) {
            r[0] = OP_ELASTIC;                                       // the field itself is drawn inside the apply kernel
            r[1] = __float_as_int(a[0]);
            r[2] = __float_as_int(a[1]);
            ++n_out;
        } else if (kind == SPEC_TIME_WARP) {
            const double u = u01d(d.bits(), d.bits());
            const double rate = (double)a[0] + ((double)a[1] - (double)a[0]) * u;   // random.uniform(min, max)
            r[0] = OP_TIME_WARP;
            r[1] = __double2loint(rate);
            r[2] = __double2hiint(rate);
            ++n_out;
        }
    }
    return n_out;
}

constexpr int NGROUPS = 784;
constexpr int SAMPLE_WARPS = 4;         // records per CTA (one warp each): 4 x fewer, 4 x fuller CTAs than one warp per block
__global__ void __launch_bounds__(32 * SAMPLE_WARPS) aug_sample_kernel(const int32_t* __restrict__ spec, int B, int Vg, int Vl, uint64_t seed,
                                                                       uint64_t step, int32_t* __restrict__ img_ops, int32_t* __restrict__ aud_ops,
                                                                       uint32_t* __restrict__ group_bits, const int64_t* __restrict__ step_dev) {
    if (step_dev != nullptr) step += (uint64_t)__ldg(step_dev);
    // one warp per (sample, view) record: lane 0 replays the two op chains (sequential by nature), the whole warp draws the
    // grouped-masking subset (random keys + threshold selection) and copies the records out.
    __shared__ int32_t sspec[4 * B200_AUG_MAX_OPS * 8];
    __shared__ int32_t rec_i_s[SAMPLE_WARPS][B200_AUG_MAX_OPS * 8], rec_a_s[SAMPLE_WARPS][B200_AUG_MAX_OPS * 8];
    __shared__ uint32_t bits_s[SAMPLE_WARPS][B200_AUG_GROUP_WORDS];
    const int V = Vg + Vl;
    const int warp = threadIdx.x >> 5, tid = threadIdx.x & 31;
    for (int i = threadIdx.x; i < 4 * B200_AUG_MAX_OPS * 8; i += blockDim.x) sspec[i] = __ldg(spec + i);
    __syncthreads();
    const long rec_l = (long)blockIdx.x * SAMPLE_WARPS + warp;
    if (rec_l >= (long)B * V) return;
    const int b = (int)(rec_l / V), v = (int)(rec_l - (long)b * V);
    const size_t rec = (size_t)rec_l;
    int32_t* rec_i = rec_i_s[warp];
    int32_t* rec_a = rec_a_s[warp];
    uint32_t* bits = bits_s[warp];
    if (tid < B200_AUG_GROUP_WORDS) bits[tid] = 0u;
    __syncwarp();
    const bool local = v >= Vg;
    const uint64_t stream = (step << 36) ^ ((uint64_t)rec << 4);
    int gc = -1;
    if (tid == 0) {
        Draw di(seed, stream | 2), da(seed, stream | 3);
        // the two chains draw from separate streams and only the audio chain sets gc: skipping the image records (img_ops NULL,
        // audio-only models) leaves the audio records and the group mask unchanged
        if (img_ops != nullptr) sample_chain(sspec + (local ? 1 : 0) * B200_AUG_MAX_OPS * 8, 28, di, rec_i, &gc);
        sample_chain(sspec + (local ? 3 : 2) * B200_AUG_MAX_OPS * 8, 112, da, rec_a, &gc);
        if (gc > NGROUPS) gc = NGROUPS;
    }
    gc = __shfl_sync(0xffffffffu, gc, 0);
    if (gc > 0) {
        // Uniformly random subset of gc of the 784 groups, by the whole warp: every group draws an independent 32-bit key and the gc
        // smallest keys win (i.i.d. keys: every gc-subset is equally likely; equal keys at the threshold are taken in index order).
        // Lane l owns the 32 groups of mask word l.  (Round 1-2: a 508-step Fisher-Yates chain on lane 0 -- the kernel was latency
        // bound on that one lane, 23 % warps active.)
        constexpr int NW = (NGROUPS + 31) / 32;                           // 25 words, the last one half full
        const int nvalid = tid < NW ? (NGROUPS - 32 * tid < 32 ? NGROUPS - 32 * tid : 32) : 0;
        uint32_t key[32];
        Philox rng(seed);
#pragma unroll
        for (int j = 0; j < 8; ++j) {
            uint4 r = make_uint4(0, 0, 0, 0);
            if (tid < NW) r = rng((uint64_t)(tid * 8 + j), stream | 4);
            key[4 * j + 0] = r.x; key[4 * j + 1] = r.y; key[4 * j + 2] = r.z; key[4 * j + 3] = r.w;
        }
        uint32_t lo = 0u, hi = 0xFFFFFFFFu;                                // smallest T with #(key <= T) >= gc
#pragma unroll 1
        for (int it = 0; it < 32 && lo < hi; ++it) {
            const uint32_t mid = lo + ((hi - lo) >> 1);
            int c = 0;
#pragma unroll
            for (int j = 0; j < 32; ++j) c += (j < nvalid && key[j] <= mid) ? 1 : 0;
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) c += __shfl_xor_sync(0xffffffffu, c, o);
            if (c >= gc) hi = mid; else lo = mid + 1u;
        }
        const uint32_t T = lo;
        int less = 0, eq = 0;
        uint32_t mless = 0u, meq = 0u;
#pragma unroll
        for (int j = 0; j < 32; ++j) {
            if (j < nvalid) {
                if (key[j] < T) { mless |= 1u << j; ++less; }
                else if (key[j] == T) { meq |= 1u << j; ++eq; }
            }
        }
        int tot_less = less, eq_before = eq;                               // warp total of `less`; exclusive prefix of `eq` over the lanes
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) tot_less += __shfl_xor_sync(0xffffffffu, tot_less, o);
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const int t2 = __shfl_up_sync(0xffffffffu, eq_before, o);
            if (tid >= o) eq_before += t2;
        }
        eq_before -= eq;
        int take = gc - tot_less - eq_before;                              // how many of this lane's threshold-equal keys are still needed
        take = take < 0 ? 0 : (take > eq ? eq : take);
        uint32_t m = mless;
        while (take > 0) {                                                 // lowest set bits of meq first (index order)
            const uint32_t b = meq & (0u - meq);
            m |= b;
            meq ^= b;
            --take;
        }
        if (tid < B200_AUG_GROUP_WORDS) bits[tid] = m;
    }
    __syncwarp();
    for (int i = tid; i < B200_AUG_MAX_OPS * 8; i += 32) {
        if (img_ops != nullptr) img_ops[rec * (B200_AUG_MAX_OPS * 8) + i] = rec_i[i];
        aud_ops[rec * (B200_AUG_MAX_OPS * 8) + i] = rec_a[i];
    }
    if (tid < B200_AUG_GROUP_WORDS) group_bits[rec * B200_AUG_GROUP_WORDS + tid] = bits[tid];
}

}  // namespace b200

using namespace b200;

extern "C" {

int b200_aug_apply_image(const void* src, int src_u8, const int32_t* ops, float* out, void* out_quad8, int pad, int B, int V, void* stream) {
    return b200_aug_apply_image_ex(src, src_u8, ops, nullptr, 0, out, out_quad8, pad, B, V, stream);
}

int b200_aug_apply_image_ex(const void* src, int src_u8, const int32_t* ops, const float* elastic_grid, uint64_t seed, float* out, void* out_quad8,
                            int pad, int B, int V, void* stream) {
    B200_REQUIRE(src && ops && (out || out_quad8) && B > 0 && V > 0 && pad >= 0, B200_E_ARG, "aug_apply_image: bad arguments");
    B200_REQUIRE((((uintptr_t)src | (uintptr_t)out | (uintptr_t)out_quad8) & 15) == 0, B200_E_ARG, "aug_apply_image: pointers must be 16-byte aligned");
    constexpr int S = 28, T = 128;
    const size_t smem = 2 * S * S * sizeof(float) + 2 * S * sizeof(AATable);
    aug_apply_kernel<S, T><<<B * V, T, smem, as_stream(stream)>>>(src, src_u8, ops, nullptr, nullptr, seed, out, reinterpret_cast<uint4*>(out_quad8), pad, B, V,
                                                                  nullptr, elastic_grid);
    return launch_status("aug_apply_image");
}

int b200_aug_apply_audio(const void* src, int src_u8, const int32_t* ops, const uint32_t* group_bits, const float* noise,
                         uint64_t seed, float* out, void* out_quad8, int pad, int B, int V, void* stream) {
    return b200_aug_apply_audio_dev(src, src_u8, ops, group_bits, noise, seed, nullptr, out, out_quad8, pad, B, V, stream);
}

int b200_aug_apply_audio_dev(const void* src, int src_u8, const int32_t* ops, const uint32_t* group_bits, const float* noise,
                             uint64_t seed, const int64_t* step_dev, float* out, void* out_quad8, int pad, int B, int V, void* stream) {
    B200_REQUIRE(src && ops && group_bits && (out || out_quad8) && B > 0 && V > 0 && pad >= 0, B200_E_ARG, "aug_apply_audio: bad arguments");
    B200_REQUIRE((((uintptr_t)src | (uintptr_t)out | (uintptr_t)out_quad8) & 15) == 0, B200_E_ARG, "aug_apply_audio: pointers must be 16-byte aligned");
    constexpr int S = 112, T = 512;
    const size_t smem = 2 * S * S * sizeof(float) + 2 * S * sizeof(AATable);
    static bool attr_done = false;
    if (!attr_done) {
        cudaError_t e = cudaFuncSetAttribute(aug_apply_kernel<S, T>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        B200_REQUIRE(e == cudaSuccess, B200_E_SMEM, "aug_apply_audio: cannot reserve %zu B of shared memory", smem);
        attr_done = true;
    }
    aug_apply_kernel<S, T><<<B * V, T, smem, as_stream(stream)>>>(src, src_u8, ops, group_bits, noise, seed, out, reinterpret_cast<uint4*>(out_quad8), pad, B, V,
                                                                  step_dev, nullptr);
    return launch_status("aug_apply_audio");
}

int b200_aug_sample(const int32_t* spec, int B, int Vg, int Vl, uint64_t seed, uint64_t step, int32_t* img_ops,
                    int32_t* aud_ops, uint32_t* group_bits, void* stream) {
    return b200_aug_sample_dev(spec, B, Vg, Vl, seed, step, nullptr, img_ops, aud_ops, group_bits, stream);
}

int b200_aug_sample_dev(const int32_t* spec, int B, int Vg, int Vl, uint64_t seed, uint64_t step, const int64_t* step_dev, int32_t* img_ops,
                        int32_t* aud_ops, uint32_t* group_bits, void* stream) {
    B200_REQUIRE(spec && aud_ops && group_bits && B > 0 && Vg >= 0 && Vl >= 0 && Vg + Vl > 0, B200_E_ARG,
                 "aug_sample: bad arguments");
    const long recs = (long)B * (Vg + Vl);
    aug_sample_kernel<<<(unsigned)((recs + SAMPLE_WARPS - 1) / SAMPLE_WARPS), 32 * SAMPLE_WARPS, 0, as_stream(stream)>>>(spec, B, Vg, Vl, seed, step, img_ops,
                                                                                                                     aud_ops, group_bits, step_dev);
    return launch_status("aug_sample");
}

}  // extern "C"
