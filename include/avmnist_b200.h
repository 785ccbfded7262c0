/*
 * avmnist_b200.h -- C ABI of the B200-native DINO training-step library (libavmnist_b200.so).
 *
 * The reference (wardvdnb/Multimodal-SSL-AVMNIST) is pure Python/PyTorch and has no FFI of its own; its boundary
 * for this path is the Python API in AVMNIST_Experiments/{models/dino.py, utils/get_data.py}.  Each entry point
 * below therefore cites the reference *Python* call site whose arithmetic it replaces (paths relative to
 * /root/reference/AVMNIST_Experiments/).  The Python binding a maintainer adds is a ctypes stub
 * (multimodal_ssl_avmnist_b200/_lib.py; see INTEGRATION.md).
 *
 * Conventions
 *   - plain pointers + sizes; every pointer is a DEVICE pointer unless the name ends in _host;
 *   - `stream` is a cudaStream_t passed as void*; all calls are asynchronous on it, never allocate,
 *     never synchronise; the caller owns every buffer (workspaces included);
 *   - return value: 0 = ok, <0 = argument / shape error (B200_E_*), >0 = cudaError_t of the launch;
 *     b200_last_error() returns a thread-local description of the last non-zero return;
 *   - fp32 everywhere unless stated; tensors are dense row-major in the stated shape.
 */
#ifndef AVMNIST_B200_H
#define AVMNIST_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define B200_E_ARG (-1)        /* null pointer / non-positive size / misaligned pointer */
#define B200_E_SHAPE (-2)      /* shape not supported by the compiled kernels */
#define B200_E_SMEM (-3)       /* kernel needs more shared memory than the device grants */

const char* b200_last_error(void);
int b200_abi_version(void);                      /* bumped whenever a signature below changes */
int b200_device_sm_count(int device);            /* helper for the host-side launch planner */
/* node census of a captured CUDA graph (cudaGraph_t): counts[0..3] = kernel, memset, memcpy, other nodes */
int b200_graph_node_counts(void* graph, int64_t* counts);

/* ------------------------------------------------------------------------------------------------------------
 * Teacher EMA  --  MultiModalDINO.update_teacher, models/dino.py:635-646 (UniModalDINO :1300-1311)
 *   t <- RN(RN(m*t) + RN((1-m)*s)), two products and one sum, never contracted to an FMA (bit-exact with ATen).
 * b200_ema_flat  : one contiguous arena of n floats (the layout the engine uses: all teacher params in one arena).
 * b200_ema_multi : n_tensors separate tensors in ONE launch; t_ptrs/s_ptrs are device arrays of device pointers,
 *                  offsets is a device array of n_tensors+1 exclusive prefix sums of the tensor sizes.
 * ---------------------------------------------------------------------------------------------------------- */
int b200_ema_flat(float* teacher, const float* student, int64_t n, float m, float one_minus_m, void* stream);
int b200_ema_multi(float* const* t_ptrs, const float* const* s_ptrs, const int64_t* offsets, int n_tensors,
                   int64_t total, float m, float one_minus_m, void* stream);

/* ------------------------------------------------------------------------------------------------------------
 * Fused DINO loss, forward + backward + teacher column sums
 *   -- MultiModalDINOLightning.dino_loss, models/dino.py:822-854 (variant 0)
 *   -- UniModalDINOLightning.dino_loss,   models/dino.py:1596-1635 (variant 1: needs t_colmean from
 *      b200_teacher_norm_colmean)
 *   -- the centre subtraction of MultiModalDINO.forward, models/dino.py:711-714, is folded in: `t` holds the
 *      UNcentred teacher projections and `center` is subtracted on load.
 *   s [Vs,B,D], t [Vt,B,D], center [D], grad_s [Vs,B,D] (d loss / d s, times grad_scale),
 *   part_loss [n_parts], part_colsum [n_parts, D]: per-CTA partials, n_parts = b200_dino_loss_parts(B);
 *   they are reduced in a fixed order by b200_center_update (deterministic).
 *   D must be a multiple of 32, D <= 1024.
 * ---------------------------------------------------------------------------------------------------------- */
int b200_dino_loss_parts(int B);
int b200_dino_loss_fwd_bwd(const float* s, const float* t, const float* center, const float* t_colmean,
                           int Vs, int Vt, int B, int D, float tau_s, float tau_t, float grad_scale, int variant,
                           float* grad_s, float* part_loss, float* part_colsum, void* stream);
/* column mean over the batch of the L2-normalised, centre-subtracted teacher outputs: out [Vt, D] */
int b200_teacher_norm_colmean(const float* t, const float* center, int Vt, int B, int D, float* out, void* stream);

/* Centre EMA + loss finalisation -- MultiModalDINO.update_center, models/dino.py:648-653
 *   colsum = sum over parts (fixed order);  center <- center*m_c + (colsum / n_rows) * one_minus_mc;
 *   loss_out[0] = sum over parts of part_loss.  If colsum_out != NULL the reduced column sums are also written
 *   there instead of updating the centre (data-parallel: all-reduce colsum_out, then b200_center_apply). */
int b200_center_update(float* center, const float* part_colsum, const float* part_loss, int n_parts, int D,
                       int64_t n_rows, float m_c, float one_minus_mc, float* loss_out, float* colsum_out, void* stream);
int b200_center_apply(float* center, const float* colsum, int D, int64_t n_rows, float m_c, float one_minus_mc,
                      void* stream);

/* ------------------------------------------------------------------------------------------------------------
 * Auxiliary losses, forward + backward fused (grad_scale multiplies the gradients)
 *   b200_mse_align_fwd_bwd -- MultiModalDINOWithMSELightning.mse_loss, models/dino.py:1193-1211
 *   b200_ce_fwd_bwd        -- supervised_loss, models/dino.py:1001-1025 (one call per modality; mean CE)
 *   b200_infonce_fwd_bwd   -- infoNCE_loss, models/dino.py:1091-1128: sim = normalize(a) normalize(b)^T / temp,
 *                             0.5*(CE(sim, I) + CE(sim^T, I)); the [B,B] matrix is never written to HBM.
 *                             work: float[b200_infonce_work_floats(B, D)].
 * loss_out[0] receives the scalar (written, not accumulated).  The scalar is a FIXED-ORDER sum (per-block partials added by
 * block index by the last block to finish): bit-identical from run to run, like the reference's deterministic=True
 * (run_dino.py:364).  work: float[b200_loss_work_floats(B)] scratch for those partials (contents irrelevant on entry).
 * ---------------------------------------------------------------------------------------------------------- */
int64_t b200_loss_work_floats(int B);
int b200_mse_align_fwd_bwd(const float* a, const float* b, int B, int D, float grad_scale, float* grad_a,
                           float* grad_b, float* loss_out, float* work, void* stream);
int b200_ce_fwd_bwd(const float* logits, const int64_t* labels, int B, int C, float grad_scale, float* grad_logits,
                    float* loss_out, float* work, void* stream);
int64_t b200_infonce_work_floats(int B, int D);
int b200_infonce_fwd_bwd(const float* a, const float* b, int B, int D, float temperature, float grad_scale,
                         float* grad_a, float* grad_b, float* loss_out, float* work, void* stream);
/* the same loss and gradients on the tensor cores: tcgen05 tf32 similarity GEMM with an exp / row-sum epilogue (E = exp(sim)
 * kept once in bf16), bf16 tcgen05 GEMMs for the gradients.  work: float[b200_infonce_tc_work_floats(B, D)], 16-byte aligned. */
int64_t b200_infonce_tc_work_floats(int B, int D);
int b200_infonce_fwd_bwd_tc(const float* a, const float* b, int B, int D, float temperature, float grad_scale, float* grad_a,
                            float* grad_b, float* loss_out, float* work, void* stream);
/* SimCLR NT-Xent (other_ssl/multimodal_simclr/multimodal_simclr.py:74-89): reps [N = 2B, D] = cat([z1, z2]); row-normalised
 * similarities / temperature, self-similarity masked, positive of row i = row (i + B) mod N, mean cross-entropy; forward and
 * backward in one call on the InfoNCE tile kernels.  work: float[b200_ntxent_work_floats(N, D)]. */
int64_t b200_ntxent_work_floats(int N, int D);
int b200_ntxent_fwd_bwd(const float* reps, int N, int D, float temperature, float grad_scale, float* grad, float* loss_out,
                        float* work, void* stream);
/* UniModalDINOLightning._cosine_consistency_loss, models/dino.py:1575-1594: emb [V,B,D] */
int b200_cosine_consistency_fwd_bwd(const float* emb, int V, int B, int D, float grad_scale, float* grad_emb,
                                    float* loss_out, float* work, void* stream);

/* ------------------------------------------------------------------------------------------------------------
 * Multi-crop augmentation  --  MultiModalAugmentation.__call__, utils/get_data.py:233-257 and its chains
 * :121-231 (GaussianNoise :21-27, TimeWarpWithStretch :29-58, GroupedMasking :60-108; torchvision
 * RandomResizedCrop/RandomRotation/RandomAffine/RandomErasing, torchaudio Frequency/TimeMasking restated).
 *
 * One op record = 8 int32 words: kind, then 7 payload words (ints, or float bit patterns):
 *   1 CROP_RESIZE i,j,h,w   2 AFFINE m0..m5 (fp32 inverse matrix)   3 ERASE i,j,h,w   4 FREQ_MASK start,end
 *   5 TIME_MASK start,end   6 NOISE std   7 GROUP_MASK (bits in group_bits)   8 TIME_WARP rate   0 NOP
 *   9 BLUR3 k0,k1,k2 (fp32 taps of torchvision GaussianBlur(3))   10 ELASTIC [alpha, sigma] (torchvision ElasticTransform: the
 *   sampling grid comes from elastic_grid, or is drawn in-kernel) -- the SimCLR image chain, utils/get_data.py:311-339
 * ops: int32 [B, V, B200_AUG_MAX_OPS, 8]; group_bits: uint32 [B, V, 28] (784 bits, 4x4 groups, 1 = zeroed).
 * Output is view-major: out [V, B, S, S] (S = 28 image / 112 audio) so that every view-call of the encoder
 * reads a contiguous batch.
 * ---------------------------------------------------------------------------------------------------------- */
#define B200_AUG_MAX_OPS 8
#define B200_AUG_GROUP_WORDS 28

/* Outputs (either may be NULL, not both): out fp32 [V,B,S,S]; out_quad8 bf16 [V,B,S,ceil((S+2 pad)/4),8], the first-layer
 * input image of the tensor-core convolutions (see b200_pack_quad8; pad = that convolution's padding).
 * image: src float [B,28,28] in [0,1] (src_u8 == 0) or uint8 [B,28,28] scaled by 1/255 (src_u8 == 1) */
int b200_aug_apply_image(const void* src, int src_u8, const int32_t* ops, float* out, void* out_quad8, int pad, int B,
                         int V, void* stream);
/* the same with the side inputs of the SimCLR image chain: elastic_grid = optional fp32 [B, V, 2, 28, 28] absolute sampling grid
 * (x, y in [-1, 1] units, identity + displacement: parity mode); NULL -> the displacement field of an ELASTIC op is drawn in-kernel
 * from Philox(seed, sample*V+view) */
int b200_aug_apply_image_ex(const void* src, int src_u8, const int32_t* ops, const float* elastic_grid, uint64_t seed,
                            float* out, void* out_quad8, int pad, int B, int V, void* stream);
/* audio: src uint8 [B,112,112] (scaled by 1/255, utils/get_data.py:467) or float; noise: optional injected N(0,1)
 * field [B,V,112,112] (parity mode), NULL -> Philox(seed, sample*V+view) in-kernel */
int b200_aug_apply_audio(const void* src, int src_u8, const int32_t* ops, const uint32_t* group_bits,
                         const float* noise, uint64_t seed, float* out, void* out_quad8, int pad, int B, int V,
                         void* stream);
/* device-side parameter sampling: spec tables int32 [4][B200_AUG_MAX_OPS][8] in the order
 * image-global, image-local, audio-global, audio-local (kind, p, a0..a5 as float bits; see augment.py pack_spec);
 * fills img_ops/aud_ops/group_bits for B samples x (Vg+Vl) views from Philox(seed, step).  img_ops may be NULL (audio-only
 * models): the image records are then neither drawn nor written, and the audio records and group bits are unchanged. */
int b200_aug_sample(const int32_t* spec, int B, int Vg, int Vl, uint64_t seed, uint64_t step, int32_t* img_ops,
                    int32_t* aud_ops, uint32_t* group_bits, void* stream);
/* CUDA-graph replay variants: the step counter lives in device memory (int64, advanced by b200_counters_advance inside the
 * graph), so the captured launches need no per-step host arguments.  step_dev == NULL: identical to the plain calls.
 * aug_sample: step + *step_dev; aug_apply_audio: noise seed (seed + *step_dev) & (2^48 - 1). */
int b200_aug_sample_dev(const int32_t* spec, int B, int Vg, int Vl, uint64_t seed, uint64_t step, const int64_t* step_dev,
                        int32_t* img_ops, int32_t* aud_ops, uint32_t* group_bits, void* stream);
int b200_aug_apply_audio_dev(const void* src, int src_u8, const int32_t* ops, const uint32_t* group_bits,
                             const float* noise, uint64_t seed, const int64_t* step_dev, float* out, void* out_quad8,
                             int pad, int B, int V, void* stream);

/* ------------------------------------------------------------------------------------------------------------
 * Encoder building blocks -- conv -> BatchNorm(train) -> ReLU -> MaxPool2 of CentralUnimodalImage/Audio
 * (models/unimodal.py:127-143, 185-211) and image_encoder()/ImageEncoder (models/dino.py:18-41, 483-499).
 * Activations are NCHW fp32.  A launch covers n_views view-calls at once: N = n_views*n_per_view samples,
 * BatchNorm statistics stay segmented per view-call (the reference calls the encoder once per view).
 * ---------------------------------------------------------------------------------------------------------- */
/* z = conv(x, w) + bias; stats[view][c] += {sum z, sum z^2} (double).  stats must be zeroed by the caller.
 * Supported (Cin,Cout,H,W,K,pad): see b200_conv_supported. */
int b200_conv_supported(int Cin, int Cout, int H, int W, int K, int pad);
int b200_conv_fwd(const float* x, const float* w, const float* bias, float* z, double* stats, int N,
                  int n_per_view, int Cin, int Cout, int H, int W, int K, int pad, void* stream);
/* dx = conv_transpose(dz, w)  (gradient w.r.t. the conv input) */
int b200_conv_bwd_data(const float* dz, const float* w, float* dx, int N, int Cin, int Cout, int H, int W, int K,
                       int pad, void* stream);
/* ---- tensor-core path (tcgen05 + TMEM + TMA) for the C_in >= 8 convolutions: same call sites as above ----
 * Activations are bf16 in the "act8" layout [N][C/8][H][W][8] (channel octets are planes; a pixel of a plane is one
 * 16-byte unit); accumulation is fp32.  b200_conv_tc computes z = conv(x, w) (+ bias and the BatchNorm partial
 * statistics when bias != NULL) and writes fp32 NCHW (out_bf16 = 0), bf16 act8 (1) or fp16 act8 (2).  The data
 * gradient of a convolution is the same call with (Cin, Cout) swapped, pad' = K-1-pad, H/W those of dz, and weights
 * prepared with flip = 1.  wprep: b200_conv_tc_weight_bytes(Cin, Cout, K) bytes filled by b200_conv_tc_prep_weights
 * from the fp32 OIHW weight (for flip = 1: `w` is the FORWARD weight [Cin][Cout][K][K]). */
int b200_conv_tc_supported(int Cin, int Cout, int H, int W, int K, int pad);
int64_t b200_conv_tc_weight_bytes(int Cin, int Cout, int K);
int b200_conv_tc_prep_weights(const float* w, void* wprep, int Cin, int Cout, int K, int flip, void* stream);
/* the same for n weight tensors in ONE launch: desc_dev = device array int64 [n][6] = {w pointer, out pointer, Cin, Cout, K, flip}
 * (validated like b200_conv_tc_prep_weights by the caller: the kernel trusts the table) */
int b200_conv_tc_prep_weights_multi(const int64_t* desc_dev, int n, void* stream);
int b200_conv_tc(const void* x_act8, const void* wprep, const float* bias, void* out, double* stats, int N,
                 int n_per_view, int Cin, int Cout, int H, int W, int K, int pad, int out_bf16, void* stream);
/* dw [Cout][Cin][K][K] = sum_n corr(x_n, dz_n); x and dz bf16 act8, fp32 accumulate in TMEM; per-CTA partials in work
 * (float[b200_conv_tc_wgrad_work_floats(...)]) reduced in a fixed order.  (The bias gradient sum(dz) comes from
 * b200_bn_relu_pool8_bwd_apply's dbsum.)
 * First layers (Cin = 1): b200_conv_tc takes the "quad8" image (b200_pack_quad8); the stand-alone b200_conv_tc_wgrad takes the
 * "shift8" image bf16 [N][H][W+pad][8] written by b200_pack_shift8 (unit (y,xs) = x[y][xs-pad .. xs-pad+7], zero outside the
 * row) -- the training step uses b200_conv_tc_wgrad_l0_fused (quad8) instead. */
/* Selects the weight-gradient formulation of the wide 3x3 layers: 1 (default) = one TMEM accumulator per filter tap, 0 = the
 * shift-row kernel everywhere (A/B measurements; the work size depends on it: query b200_conv_tc_wgrad_work_floats afterwards).
 * Any other value only queries.  Returns the previous setting. */
int b200_conv_tc_wgrad_variant(int tap);
int64_t b200_conv_tc_wgrad_work_floats(int N, int Cin, int Cout, int H, int W, int K, int pad);
int b200_conv_tc_wgrad(const void* x_act8, const void* dz_act8, float* dw, float* work, int N, int Cin, int Cout, int H,
                       int W, int K, int pad, void* stream);
int b200_pack_shift8(const float* x, void* out, int N, int H, int W, int pad, void* stream);
/* fp32 [N][H][W] -> bf16 "quad8" [N][H][WQ][8], WQ = ceil((W + 2 pad) / 4): unit (y, xq) = the 8 zero-padded-row pixels
 * 4 xq .. 4 xq + 7 (padded column c = image column c - pad).  The first-layer input of b200_conv_tc (C_in = 1) and of
 * b200_conv_tc_wgrad_l0_fused: four adjacent output pixels share one unit, whose 8 elements are all their kw taps. */
int b200_pack_quad8(const float* x, void* out, int N, int H, int W, int pad, void* stream);
/* First layers, fused backward: b200_bn_relu_pool8_bwd_apply + b200_conv_tc_wgrad in one kernel (the first layer needs no data
 * gradient, so dz never has to exist in HBM): x_quad8 from b200_pack_quad8 / the augmentation kernels, z8 fp16 act8 [N][Cout/8][H][W][8], dp8 bf16 act8 [N][Cout/8][H/2][W/2][8],
 * scale/shift/mean/invstd [views][Cout], sums double [views][Cout][2] (from b200_bn_pool8_bwd_reduce_p) -> dw [Cout][1][K][K],
 * dbsum double [Cout] += sum(dz) (may be NULL).  work: float[b200_conv_tc_wgrad_l0_fused_work_floats(...)], 16-byte aligned. */
int64_t b200_conv_tc_wgrad_l0_fused_work_floats(int N, int n_per_view, int Cout, int H, int W, int K, int pad);
int b200_conv_tc_wgrad_l0_fused(const void* x_quad8, const void* z8, const void* dp8, const float* scale, const float* shift,
                                const float* mean, const float* invstd, const double* sums, float* dw, double* dbsum,
                                float* work, int N, int n_per_view, int Cout, int H, int W, int K, int pad, void* stream);
/* Forward convolution with the 2x2 max-pool FUSED INTO ITS EPILOGUE (conv -> BatchNorm -> ReLU -> MaxPool2 of
 * models/unimodal.py:129-140, 186-208; models/dino.py:20-30).  Train-mode BatchNorm is a*z + b with a = gamma * invstd, so
 * ReLU(maxpool(a z + b)) = ReLU(a ext(z) + b) with ext = max where gamma >= 0 and min where gamma < 0 -- known BEFORE the batch
 * statistics are.  The epilogue therefore emits, besides the statistics, the window extreme `pool_out` (fp16 act8
 * [N][Cout/8][Ho/2][Wo/2][8], a quarter of z) and b200_bn_relu_apply8 finishes p = ReLU(a e + b) once b200_bn_finalize has run:
 * bit-identical to b200_bn_relu_pool8_fwd on the full-resolution z.  z_out (fp16 / bf16 act8, z_fmt 2 / 1) is still written for
 * the student (its backward needs the dense z) and may be NULL for the teacher and for evaluation: full-resolution z then never
 * leaves the SM.  gamma: the BatchNorm weight [Cout] (device pointer, read at kernel start). */
int b200_conv_tc_pool_supported(int Cin, int Cout, int H, int W, int K, int pad);
int b200_conv_tc_pool(const void* x_act8, const void* wprep, const float* bias, const float* gamma, void* z_out, void* pool_out,
                      double* stats, int N, int n_per_view, int Cin, int Cout, int H, int W, int K, int pad, int z_fmt,
                      void* stream);
/* Data gradient of a convolution whose output dx is the gradient dp of the layer below's pooled activation p (bf16 act8, same
 * shape as dx), with that layer's BatchNorm-backward statistics fused into the epilogue:
 *   sums[view][c] += { sum_{p>0} dp, sum_{p>0} dp * (p - beta[c]) / gamma[c] }      (what b200_bn_pool8_bwd_reduce_p computes in a
 * pass of its own; gamma / beta = the lower layer's BatchNorm weight / bias, sums zeroed by the caller).  Arguments as b200_conv_tc
 * for a data gradient: (Cin, Cout) = (channels of dz, channels of dx), H/W those of dz, pad = K-1-pad_forward, flipped weights. */
int b200_conv_tc_dgrad_bnstat_supported(int Cin, int Cout, int H, int W, int K, int pad);
int b200_conv_tc_dgrad_bnstat(const void* dz_act8, const void* wprep_flip, void* dx_act8, const void* p_act8, const float* gamma,
                              const float* beta, double* sums, int N, int n_per_view, int Cin, int Cout, int H, int W, int K,
                              int pad, void* stream);
/* e8: fp16 act8 [N][C/8][HP][WP][8] from b200_conv_tc_pool; out_fmt 0 = fp32 NCHW [N][C][HP][WP], 1 = bf16 act8 */
int b200_bn_relu_apply8(const void* e8, const float* scale, const float* shift, void* out, int N, int n_per_view, int C, int HP,
                        int WP, int out_fmt, void* stream);
/* BatchNorm-apply + ReLU + MaxPool2 on bf16 act8 activations (same reference call sites as b200_bn_relu_pool_*):
 *   z8 [N][C/8][H][W][8] bf16 (z_f16 = 0) or fp16 (z_f16 = 1) (H, W even); scale/shift/mean/invstd [views][C] from b200_bn_finalize;
 *   out_fmt / dp_fmt: 0 = fp32 NCHW [N][C][H/2][W/2], 1 = bf16 act8 [N][C/8][H/2][W/2][8];
 *   sums: double [views][C][2] = {sum g, sum g*xhat} (zeroed by the caller before _bwd_reduce); dz8: bf16 act8 like z8. */
int b200_bn_relu_pool8_fwd(const void* z8, const float* scale, const float* shift, void* out, int N, int n_per_view,
                           int C, int H, int W, int z_f16, int out_fmt, void* stream);
int b200_bn_relu_pool8_bwd_reduce(const void* z8, const void* dp, const float* scale, const float* shift,
                                  const float* mean, const float* invstd, double* sums, int N, int n_per_view, int C,
                                  int H, int W, int z_f16, int dp_fmt, void* stream);
int b200_bn_relu_pool8_bwd_apply(const void* z8, const void* dp, const float* scale, const float* shift,
                                 const float* mean, const float* invstd, const double* sums, void* dz8, double* dbsum,
                                 int N, int n_per_view, int C, int H, int W, int z_f16, int dp_fmt, void* stream);
/* The same statistics as _bwd_reduce from the POOLED tensors only (no read of z): wherever the pooled output p is > 0 it
 * equals gamma*xhat + beta at the arg-max, elsewhere the gradient is zero.  p, dp: [N][C][HP][WP] fp32 (fmt 0) or bf16 act8
 * (fmt 1); gamma, beta: the BatchNorm weight / bias [C]. */
int b200_bn_pool8_bwd_reduce_p(const void* p, const void* dp, const float* gamma, const float* beta, double* sums, int N,
                               int n_per_view, int C, int HP, int WP, int p_fmt, int dp_fmt, void* stream);
/* dbsum: double [C] (zeroed by the caller, may be NULL) += sum of dz per channel = the convolution's bias gradient */
int b200_bias_grad_finalize(const double* dbsum, float* db, int C, void* stream);
/* bf16 act8 -> fp32 NCHW */
int b200_unpack_act8(const void* x8, float* out, int N, int C, int H, int W, void* stream);
/* fp32 NCHW -> bf16 act8 */
int b200_pack_act8(const float* x, void* out, int N, int C, int H, int W, void* stream);
/* dw = sum_n corr(x_n, dz_n), db = sum dz.  work: float[b200_conv_bwd_weight_work_floats(...)] */
int64_t b200_conv_bwd_weight_work_floats(int N, int Cin, int Cout, int H, int W, int K, int pad);
int b200_conv_bwd_weight(const float* x, const float* dz, float* dw, float* db, float* work, int N, int Cin,
                         int Cout, int H, int W, int K, int pad, void* stream);

/* BatchNorm finalisation (nn.BatchNorm2d / BatchNorm1d train mode, eps 1e-5, momentum 0.1; SURVEY A6):
 *   per view v (in order) and channel c: mean, biased var -> scale[v][c] = gamma*invstd, shift = beta - mean*scale,
 *   save mean/invstd; running_mean/var updated sequentially over the views (unbiased var), nbt += n_views.
 *   train == 0: scale/shift come from the running statistics (eval mode), stats ignored. */
int b200_bn_finalize(const double* stats, const float* gamma, const float* beta, float* running_mean,
                     float* running_var, int64_t* num_batches_tracked, float* scale, float* shift, float* mean,
                     float* invstd, int n_views, int C, int64_t count, float momentum, float eps, int train,
                     void* stream);
/* out[n,c,oy,ox] = relu(max over 2x2 of scale*z+shift)   (H, W even; out is [N,C,H/2,W/2]) */
int b200_bn_relu_pool_fwd(const float* z, const float* scale, const float* shift, float* out, int N,
                          int n_per_view, int C, int H, int W, void* stream);
/* backward, pass 1: sums[view][c] += {sum dy, sum dy*xhat} (double; zeroed by caller), dy = unpool+relu' of dout */
int b200_bn_relu_pool_bwd_reduce(const float* z, const float* dout, const float* scale, const float* shift,
                                 const float* mean, const float* invstd, double* sums, int N, int n_per_view,
                                 int C, int H, int W, void* stream);
/* backward, pass 2: dz = scale*(dy - sum_dy/cnt - xhat*sum_dyxhat/cnt) */
int b200_bn_relu_pool_bwd_apply(const float* z, const float* dout, const float* scale, const float* shift,
                                const float* mean, const float* invstd, const double* sums, float* dz, int N,
                                int n_per_view, int C, int H, int W, void* stream);
/* dgamma[c] = sum_v sums[v][c].dyxhat, dbeta[c] = sum_v sums[v][c].dy  (accumulate != 0: add into dgamma/dbeta) */
int b200_bn_param_grads(const double* sums, float* dgamma, float* dbeta, int n_views, int C, int accumulate,
                        void* stream);
/* global average pool (AdaptiveAvgPool2d(1), models/dino.py:34) forward / backward over [N,C,HW] */
int b200_avgpool_fwd(const float* x, float* out, int N, int C, int HW, void* stream);
int b200_avgpool_bwd(const float* dout, float* dx, int N, int C, int HW, void* stream);

/* ------------------------------------------------------------------------------------------------------------
 * Linear layers and their fused middles -- nn.Linear of the encoders / fusion / ProjectionHead
 * (models/dino.py:223-226, 459-468, 1244-1248).
 *   b200_linear_fwd      : y[M,N] = act(x[M,K] w[N,K]^T + bias); act: 0 none, 1 relu, 2 relu + dropout keep-mask
 *                          (mask uint8 [M,N], scaled by 1/(1-p)).  ldx/ldy = row strides in floats (concat support).
 *   b200_linear_bwd_data : dx[M,K] = dy[M,N] w[N,K]            (act backward applied to dy by the caller kernels)
 *   b200_linear_bwd_weight: dw[N,K] (+)= dy^T x, db[N] (+)= column sums of dy; the reduction over M is split across
 *                          CTAs through `work` (float[b200_linear_bwd_weight_work_floats]) and summed in a fixed order
 *   b200_act_bwd         : dy <- dy * (y > 0) [* mask/(1-p)]  in place (relu / relu+dropout backward)
 * ---------------------------------------------------------------------------------------------------------- */
int b200_linear_fwd(const float* x, int64_t ldx, const float* w, const float* bias, float* y, int64_t ldy, int M,
                    int N, int K, int act, const uint8_t* mask, float drop_p, void* stream);
int b200_linear_bwd_data(const float* dy, int64_t lddy, const float* w, float* dx, int64_t lddx, int M, int N,
                         int K, void* stream);
int64_t b200_linear_bwd_weight_work_floats(int M, int N, int K);
int b200_linear_bwd_weight(const float* dy, int64_t lddy, const float* x, int64_t ldx, float* dw, float* db, float* work,
                           int M, int N, int K, int accumulate, void* stream);
/* tensor-core variants (tcgen05 kind::tf32, TMA-staged fp32 operands, fp32 TMEM accumulators): same results up to tf32
 * operand rounding; operands that TMA cannot address (row pitch not a multiple of 16 bytes) run on the SIMT kernels.
 * kind::tf32 needs K-major operands, so the two backward GEMMs transpose W (resp. dy and x) into `work` first:
 * work is REQUIRED, float[b200_linear_bwd_{data,weight}_tc_work_floats(M, N, K)], 16-byte aligned. */
int b200_linear_fwd_tc(const float* x, int64_t ldx, const float* w, const float* bias, float* y, int64_t ldy, int M, int N,
                       int K, int act, const uint8_t* mask, float drop_p, void* stream);
int64_t b200_linear_bwd_data_tc_work_floats(int M, int N, int K);
int b200_linear_bwd_data_tc(const float* dy, int64_t lddy, const float* w, float* dx, int64_t lddx, float* work, int M, int N,
                            int K, void* stream);
int64_t b200_linear_bwd_weight_tc_work_floats(int M, int N, int K);
int b200_linear_bwd_weight_tc(const float* dy, int64_t lddy, const float* x, int64_t ldx, float* dw, float* db, float* work,
                              int M, int N, int K, int accumulate, void* stream);
int b200_act_bwd(float* dy, const float* y, const uint8_t* mask, float drop_p, int64_t n, void* stream);
/* BatchNorm1d statistics over the rows of h[M,C] (double sums, zeroed by the caller): stats[c] = {sum, sum^2} */
int b200_colstats(const float* h, double* stats, int M, int C, void* stream);
/* g = dropout(gelu_erf(scale*h + shift)) ; backward pass 1 accumulates {sum dy, sum dy*xhat}, pass 2 writes dh */
int b200_bn1d_gelu_drop_fwd(const float* h, const float* scale, const float* shift, const uint8_t* mask,
                            float drop_p, float* g, int M, int C, void* stream);
int b200_bn1d_gelu_drop_bwd_reduce(const float* h, const float* dg, const float* scale, const float* shift,
                                   const float* mean, const float* invstd, const uint8_t* mask, float drop_p,
                                   double* sums, int M, int C, void* stream);
int b200_bn1d_gelu_drop_bwd_apply(const float* h, const float* dg, const float* scale, const float* shift,
                                  const float* mean, const float* invstd, const uint8_t* mask, float drop_p,
                                  const double* sums, float* dh, int M, int C, void* stream);
/* Bernoulli keep-mask from Philox(seed, offset): mask[i] = u >= p */
int b200_dropout_mask(uint8_t* mask, int64_t n, float p, uint64_t seed, uint64_t offset, void* stream);
/* offset + 4 * (*step_dev): the CUDA-graph replay variant (see b200_aug_sample_dev) */
int b200_dropout_mask_dev(uint8_t* mask, int64_t n, float p, uint64_t seed, uint64_t offset, const int64_t* step_dev,
                          void* stream);

/* ------------------------------------------------------------------------------------------------------------
 * Optimiser -- torch.optim.Adam(lr, weight_decay) as configured at models/dino.py:953-962, over one flat arena;
 * `has_grad` (uint8 per element-block of 1 << has_grad_shift elements, may be NULL = all) marks the parameters that
 * received a gradient this step (Adam skips p.grad is None: the unused fc1/fc2 heads).
 * ---------------------------------------------------------------------------------------------------------- */
int b200_adam_flat(float* param, const float* grad, float* exp_avg, float* exp_avg_sq, int64_t n, float lr,
                   float beta1, float beta2, float eps, float weight_decay, float bias_correction1,
                   float bias_correction2_sqrt, float grad_scale, void* stream);
/* CUDA-graph replay: bc_out[0] = 1 - beta1^t, bc_out[1] = sqrt(1 - beta2^t) for t = *step_dev + 1 (double arithmetic, rounded
 * to fp32 like the host path); b200_adam_flat_dev reads them from device memory -- bc_dev is float[3]: with lr < 0 the learning
 * rate is read from bc_dev[2] as well, so a per-epoch scheduler (CosineAnnealingLR, models/dino.py:959) changes it without a
 * re-capture; b200_counters_advance adds 1 to n counters. */
int b200_adam_bias_dev(const int64_t* step_dev, double beta1, double beta2, float* bc_out, void* stream);
int b200_adam_flat_dev(float* param, const float* grad, float* exp_avg, float* exp_avg_sq, int64_t n, float lr,
                       float beta1, float beta2, float eps, float weight_decay, const float* bc_dev, float grad_scale,
                       void* stream);
int b200_counters_advance(int64_t* counters, int n, void* stream);
/* y <- y * alpha (used to apply an upstream autograd scale / the 1/world_size of the gradient all-reduce) */
int b200_scale_flat(float* y, int64_t n, float alpha, void* stream);

/* ------------------------------------------------------------------------------------------------------------
 * kNN evaluation of frozen encoder features (SURVEY 8f-3) -- train_knn_classifier,
 * training_structures/dino_train.py:349-368: sklearn KNeighborsClassifier(n_neighbors=5) = Euclidean distance, uniform
 * weights, majority vote, vote ties -> smallest class label.
 *   ||a - b||^2 = ||a||^2 - 2 (a.b - ||b||^2 / 2): score(i, j) = a_i . b_j - ||b_j||^2 / 2 is ONE exact-fp32 GEMM with a bias
 *   (b200_linear_fwd with x = test features [M,D], w = train features [N,D], bias = b200_knn_neg_half_sqnorm(train));
 *   b200_knn_topk_vote picks the k largest scores of every row (equal scores -> smaller train index) and votes.
 *   scores [M, lds >= N] fp32; labels int64 [N] in [0, n_classes), n_classes <= 32; k <= 16; pred int64 [M];
 *   neighbours (optional, may be NULL) int32 [M, k] = train indices, nearest first.
 * ---------------------------------------------------------------------------------------------------------- */
int b200_knn_neg_half_sqnorm(const float* x, int64_t ldx, int N, int D, float* out, void* stream);
int b200_knn_topk_vote(const float* scores, int64_t lds, const int64_t* labels, int M, int N, int k, int n_classes,
                       int64_t* pred, int32_t* neighbours, void* stream);

/* ------------------------------------------------------------------------------------------------------------
 * Feature mixing of the "simple" multimodal encoder family (SURVEY 8f-4), between the per-modality encoders and the fusion MLP:
 *   GatedMultiModalEncoder.forward (models/dino.py:249-263): features * sigmoid(gate), gate a learnable scalar --
 *     b200_gate_apply: y[M,N] = sigmoid(*gate) * x[M,N] (forward on the features AND backward on their gradient);
 *     b200_gate_grad : dgate (+)= sigmoid'(gate) * sum(dy . x) over the [M,N] block, fixed summation order;
 *                      work: b200_gate_grad_work_floats() floats, ZERO before the first call (left zero by every call).
 *   CrossModalAttention.forward (models/dino.py:385-405): attention over the BATCH of one view-call,
 *     softmax((x1 Wq)(x2 Wk)^T * dim^-0.5) (x2 Wv) + x1.  The products are b200_linear_* calls; the rest:
 *     b200_softmax_rows     : s[M, ld >= N] <- softmax(scale * s) per row, in place;
 *     b200_softmax_rows_bwd : dp <- scale * p * (dp - sum_n dp p) per row, in place on dp;
 *     b200_add2d            : dst[M,N] += src[M,N] with row strides (residual connection, gradient sums).
 * ---------------------------------------------------------------------------------------------------------- */
int b200_gate_apply(const float* x, int64_t ldx, float* y, int64_t ldy, const float* gate, int M, int N, void* stream);
int64_t b200_gate_grad_work_floats(void);
int b200_gate_grad(const float* dy, int64_t lddy, const float* x, int64_t ldx, const float* gate, float* dgate, float* work, int M, int N,
                   int accumulate, void* stream);
int b200_softmax_rows(float* s, int64_t ld, int M, int N, float scale, void* stream);
int b200_softmax_rows_bwd(float* dp, int64_t lddp, const float* p, int64_t ldp, int M, int N, float scale, void* stream);
int b200_add2d(float* dst, int64_t ld_dst, const float* src, int64_t ld_src, int M, int N, void* stream);

/* ------------------------------------------------------------------------------------------------------------
 * Data-parallel exchange (SURVEY 8b / 8e) -- what Lightning's strategy="ddp" (run_dino.py:359) does for the reference: ONE
 * NCCL communicator per process (one process per GPU).  Rank 0 calls b200_dp_unique_id and ships the 128 bytes to the other
 * ranks by any means (the Python host uses the torch.distributed store); every rank then calls b200_dp_init with its GPU
 * current.  The two all-reduces (sum, fp32, in place) are asynchronous on `stream` and may be captured into a CUDA graph.
 *   b200_dp_allreduce_grads  -- a slice of the flat gradient arena (the 1/world average is folded into Adam's grad_scale)
 *   b200_dp_allreduce_center -- the [D] column sums of the un-centred teacher projections (then b200_center_apply)
 * NCCL is bound at run time with dlopen (no link-time dependency); return codes >= 1000 are 1000 + ncclResult_t.
 * ---------------------------------------------------------------------------------------------------------- */
int b200_dp_nccl_version(void);
int b200_dp_unique_id(char* id_out /* 128 bytes */);
int b200_dp_init(const char* id /* 128 bytes */, int rank, int world);
int b200_dp_world(void);
int b200_dp_rank(void);
int b200_dp_allreduce_grads(float* grad, int64_t n, void* stream);
int b200_dp_allreduce_center(float* colsum, int D, void* stream);
int b200_dp_destroy(void);

#ifdef __cplusplus
}
#endif
#endif /* AVMNIST_B200_H */
