"""Thin tensor-level wrappers over the C ABI (one Python function per `b200_*` entry point).

torch is used only for device memory and the current CUDA stream; every wrapper hands raw pointers to the
library and raises if the call fails.  Tensors must live on a CUDA device and be contiguous.
"""
import torch

from . import _lib


def _lib_():
    return _lib.load()


def _ptr(t, dtype=None):
    if t is None:
        return None
    if not t.is_cuda:
        raise _lib.B200Error("B200 ops need CUDA tensors (there is no CPU fallback)")
    if not t.is_contiguous():
        raise _lib.B200Error("B200 ops need contiguous tensors")
    if dtype is not None and t.dtype != dtype:
        raise _lib.B200Error(f"expected {dtype}, got {t.dtype}")
    return t.data_ptr()


_RAW_STREAM = getattr(torch._C, "_cuda_getCurrentRawStream", None)
_GET_DEVICE = getattr(torch._C, "_cuda_getDevice", None)


def _stream():
    """cudaStream_t of torch's current stream on the current device.  torch.cuda.current_stream() costs ~10 us of Python per
    call (device-index resolution, a Stream object); the raw queries are plain C calls."""
    if _RAW_STREAM is None or _GET_DEVICE is None:
        return torch.cuda.current_stream().cuda_stream
    return _RAW_STREAM(_GET_DEVICE())


F32, F64, I32, I64, U8 = torch.float32, torch.float64, torch.int32, torch.int64, torch.uint8


# ---- flat arena ops ----------------------------------------------------------------------------------------
def ema_flat(teacher, student, m):
    """teacher <- m*teacher + (1-m)*student (bit-exact with the reference's mul/mul/add, dino.py:635-646)."""
    one_minus_m = 1 - m          # Python double, rounded to fp32 by the call (SURVEY A7)
    _lib.check(_lib_().b200_ema_flat(_ptr(teacher, F32), _ptr(student, F32), teacher.numel(), m, one_minus_m, _stream()), "ema_flat")


class MultiTensorTable:
    """Device-side pointer/offset table for b200_ema_multi (built once per parameter set)."""

    def __init__(self, teacher_tensors, student_tensors):
        assert len(teacher_tensors) == len(student_tensors) and len(teacher_tensors) > 0
        dev = teacher_tensors[0].device
        sizes = [t.numel() for t in teacher_tensors]
        for t, s in zip(teacher_tensors, student_tensors):
            assert t.numel() == s.numel() and t.is_contiguous() and s.is_contiguous() and t.dtype == F32 and s.dtype == F32
        off = [0]
        for n in sizes:
            off.append(off[-1] + n)
        self.total = off[-1]
        self.n = len(sizes)
        self.t_ptrs = torch.tensor([t.data_ptr() for t in teacher_tensors], dtype=I64, device=dev)
        self.s_ptrs = torch.tensor([s.data_ptr() for s in student_tensors], dtype=I64, device=dev)
        self.offsets = torch.tensor(off, dtype=I64, device=dev)
        self._keep = (teacher_tensors, student_tensors)


def ema_multi(table, m):
    one_minus_m = 1 - m
    _lib.check(_lib_().b200_ema_multi(table.t_ptrs.data_ptr(), table.s_ptrs.data_ptr(), table.offsets.data_ptr(), table.n,
                                      table.total, m, one_minus_m, _stream()), "ema_multi")


def adam_flat(param, grad, exp_avg, exp_avg_sq, step, lr, beta1=0.9, beta2=0.999, eps=1e-8, weight_decay=0.0, grad_scale=1.0):
    bc1 = 1 - beta1 ** step
    bc2s = (1 - beta2 ** step) ** 0.5
    _lib.check(_lib_().b200_adam_flat(_ptr(param, F32), _ptr(grad, F32), _ptr(exp_avg, F32), _ptr(exp_avg_sq, F32), param.numel(),
                                      lr, beta1, beta2, eps, weight_decay, bc1, bc2s, grad_scale, _stream()), "adam_flat")


def scale_flat(y, alpha):
    _lib.check(_lib_().b200_scale_flat(_ptr(y, F32), y.numel(), alpha, _stream()), "scale_flat")


def dropout_mask(mask, p, seed, offset, step_dev=None):
    """step_dev (int64 device scalar, CUDA-graph replay): the Philox offset becomes offset + 4 * *step_dev"""
    _lib.check(_lib_().b200_dropout_mask_dev(_ptr(mask, U8), mask.numel(), p, seed, offset, _ptr(step_dev, I64), _stream()), "dropout_mask")


def adam_bias_dev(step_dev, bc_out, beta1=0.9, beta2=0.999):
    """bc_out[0:2] = (1 - beta1^t, sqrt(1 - beta2^t)) for t = *step_dev + 1, computed on the device (CUDA-graph replay)"""
    _lib.check(_lib_().b200_adam_bias_dev(_ptr(step_dev, I64), beta1, beta2, _ptr(bc_out, F32), _stream()), "adam_bias_dev")


def adam_flat_dev(param, grad, exp_avg, exp_avg_sq, bc_dev, lr, beta1=0.9, beta2=0.999, eps=1e-8, weight_decay=0.0, grad_scale=1.0):
    _lib.check(_lib_().b200_adam_flat_dev(_ptr(param, F32), _ptr(grad, F32), _ptr(exp_avg, F32), _ptr(exp_avg_sq, F32), param.numel(),
                                          lr, beta1, beta2, eps, weight_decay, _ptr(bc_dev, F32), grad_scale, _stream()), "adam_flat")


def adamw_flat(param, grad, exp_avg, exp_avg_sq, step, lr, beta1=0.9, beta2=0.999, eps=1e-8, weight_decay=1e-2):
    """torch.optim.AdamW step `step` (1-based): p *= 1 - lr*weight_decay, then the Adam update without an L2 term."""
    bc1 = 1 - beta1 ** step
    bc2s = (1 - beta2 ** step) ** 0.5
    _lib.check(_lib_().b200_adamw_flat(_ptr(param, F32), _ptr(grad, F32), _ptr(exp_avg, F32), _ptr(exp_avg_sq, F32), param.numel(),
                                       lr, beta1, beta2, eps, weight_decay, bc1, bc2s, _stream()), "adamw_flat")


def adamw_flat_dev(param, grad, exp_avg, exp_avg_sq, bc_dev, lr, beta1=0.9, beta2=0.999, eps=1e-8, weight_decay=1e-2):
    """adamw_flat with the bias corrections read from bc_dev (written by adam_bias_dev; CUDA-graph replay)."""
    _lib.check(_lib_().b200_adamw_flat_dev(_ptr(param, F32), _ptr(grad, F32), _ptr(exp_avg, F32), _ptr(exp_avg_sq, F32), param.numel(),
                                           lr, beta1, beta2, eps, weight_decay, _ptr(bc_dev, F32), _stream()), "adamw_flat_dev")


def counters_advance(counters):
    _lib.check(_lib_().b200_counters_advance(_ptr(counters, I64), counters.numel(), _stream()), "counters_advance")


# ---- losses ------------------------------------------------------------------------------------------------
def dino_loss_parts(B):
    return _lib_().b200_dino_loss_parts(B)


def dino_loss_fwd_bwd(s, t, center, tau_s, tau_t, grad_s, part_loss, part_colsum, grad_scale=1.0, variant=0, t_colmean=None):
    Vs, B, D = s.shape
    Vt = t.shape[0]
    _lib.check(_lib_().b200_dino_loss_fwd_bwd(_ptr(s, F32), _ptr(t, F32), _ptr(center, F32), _ptr(t_colmean, F32), Vs, Vt, B, D,
                                              tau_s, tau_t, grad_scale, variant, _ptr(grad_s, F32), _ptr(part_loss, F32),
                                              _ptr(part_colsum, F32), _stream()), "dino_loss_fwd_bwd")


def teacher_norm_colmean(t, center, out):
    Vt, B, D = t.shape
    _lib.check(_lib_().b200_teacher_norm_colmean(_ptr(t, F32), _ptr(center, F32), Vt, B, D, _ptr(out, F32), _stream()), "teacher_norm_colmean")


def center_update(center, part_colsum, part_loss, n_rows, m_c, loss_out, colsum_out=None):
    n_parts, D = part_colsum.shape
    _lib.check(_lib_().b200_center_update(_ptr(center, F32), _ptr(part_colsum, F32), _ptr(part_loss, F32), n_parts, D, n_rows,
                                          m_c, 1 - m_c, _ptr(loss_out, F32), _ptr(colsum_out, F32), _stream()), "center_update")


def center_apply(center, colsum, n_rows, m_c):
    _lib.check(_lib_().b200_center_apply(_ptr(center, F32), _ptr(colsum, F32), colsum.numel(), n_rows, m_c, 1 - m_c, _stream()), "center_apply")


_LOSS_WORK = {}


def _loss_work(device, B):
    """Scratch for the fixed-order loss sums (per-block partials + ticket), one per device and stream."""
    need = int(_lib_().b200_loss_work_floats(B))
    key = (device, _stream())
    work = _LOSS_WORK.get(key)
    if work is None or work.numel() < need:
        work = _LOSS_WORK[key] = torch.zeros(need, dtype=F32, device=device)
    return work


def mse_align_fwd_bwd(a, b, grad_a, grad_b, loss_out, grad_scale=1.0, work=None):
    B, D = a.shape
    work = _loss_work(a.device, B) if work is None else work
    _lib.check(_lib_().b200_mse_align_fwd_bwd(_ptr(a, F32), _ptr(b, F32), B, D, grad_scale, _ptr(grad_a, F32), _ptr(grad_b, F32),
                                              _ptr(loss_out, F32), _ptr(work, F32), _stream()), "mse_align_fwd_bwd")


def ce_fwd_bwd(logits, labels, grad_logits, loss_out, grad_scale=1.0, work=None):
    B, Cc = logits.shape
    work = _loss_work(logits.device, B) if work is None else work
    _lib.check(_lib_().b200_ce_fwd_bwd(_ptr(logits, F32), _ptr(labels, I64), B, Cc, grad_scale, _ptr(grad_logits, F32),
                                       _ptr(loss_out, F32), _ptr(work, F32), _stream()), "ce_fwd_bwd")


def infonce_work_floats(B, D, tc=False):
    return (_lib_().b200_infonce_tc_work_floats if tc else _lib_().b200_infonce_work_floats)(B, D)


def infonce_fwd_bwd(a, b, grad_a, grad_b, loss_out, work, temperature=0.07, grad_scale=1.0, tc=False):
    """InfoNCE loss + gradients; tc=True: tensor-core similarity / gradient GEMMs (work sized with infonce_work_floats(tc=True))."""
    B, D = a.shape
    fn = _lib_().b200_infonce_fwd_bwd_tc if tc else _lib_().b200_infonce_fwd_bwd
    _lib.check(fn(_ptr(a, F32), _ptr(b, F32), B, D, temperature, grad_scale, _ptr(grad_a, F32), _ptr(grad_b, F32), _ptr(loss_out, F32),
                  _ptr(work, F32), _stream()), "infonce_fwd_bwd")


def ntxent_work_floats(N, D):
    return int(_lib_().b200_ntxent_work_floats(N, D))


def ntxent_fwd_bwd(reps, grad, loss_out, work, temperature=0.07, grad_scale=1.0):
    """SimCLR NT-Xent on reps [2B, D] = cat([z1, z2]) (positives B rows apart, self-similarity masked): loss + d loss / d reps."""
    N, D = reps.shape
    _lib.check(_lib_().b200_ntxent_fwd_bwd(_ptr(reps, F32), N, D, temperature, grad_scale, _ptr(grad, F32), _ptr(loss_out, F32),
                                           _ptr(work, F32), _stream()), "ntxent_fwd_bwd")


def cosine_consistency_fwd_bwd(emb, grad_emb, loss_out, grad_scale=1.0, work=None):
    V, B, D = emb.shape
    work = _loss_work(emb.device, B) if work is None else work
    _lib.check(_lib_().b200_cosine_consistency_fwd_bwd(_ptr(emb, F32), V, B, D, grad_scale, _ptr(grad_emb, F32), _ptr(loss_out, F32),
                                                       _ptr(work, F32), _stream()), "cosine_consistency_fwd_bwd")


# ---- augmentation ------------------------------------------------------------------------------------------
def _aug_outs(out, out8, pad):
    ref = out if out is not None else out8
    if ref is None:
        raise _lib.B200Error("augmentation needs an fp32 and / or a quad8 output")
    return ref.shape[0], ref.shape[1], (_ptr(out, F32) if out is not None else None), (_ptr(out8, torch.bfloat16) if out8 is not None else None)


def aug_apply_image(src, ops, out, out8=None, pad=0, elastic_grid=None, seed=0):
    """out: fp32 [V, B, 28, 28] and / or out8: bf16 quad8 [V, B, 28, ceil((28 + 2 pad) / 4), 8] (first-layer tensor-core input).
    elastic_grid: fp32 [B, V, 2, 28, 28] sampling grids of ELASTIC ops (parity mode); None -> drawn in-kernel from Philox(seed)."""
    V, B, po, p8 = _aug_outs(out, out8, pad)
    _lib.check(_lib_().b200_aug_apply_image_ex(_ptr(src), 1 if src.dtype == U8 else 0, _ptr(ops, I32), _ptr(elastic_grid, F32), seed, po, p8, pad,
                                               B, V, _stream()), "aug_apply_image")


def aug_apply_audio(src, ops, group_bits, out, noise=None, seed=0, out8=None, pad=0, step_dev=None):
    """step_dev (int64 device scalar, CUDA-graph replay): the noise seed becomes (seed + *step_dev) mod 2^48"""
    V, B, po, p8 = _aug_outs(out, out8, pad)
    _lib.check(_lib_().b200_aug_apply_audio_dev(_ptr(src), 1 if src.dtype == U8 else 0, _ptr(ops, I32), _ptr(group_bits, I32),
                                                _ptr(noise, F32), seed, _ptr(step_dev, I64), po, p8, pad, B, V, _stream()), "aug_apply_audio")


def aug_sample(spec, B, Vg, Vl, seed, step, img_ops, aud_ops, group_bits, step_dev=None):
    """step_dev (int64 device scalar, CUDA-graph replay): the Philox stream position is step + *step_dev"""
    _lib.check(_lib_().b200_aug_sample_dev(_ptr(spec, I32), B, Vg, Vl, seed, step, _ptr(step_dev, I64), _ptr(img_ops, I32),
                                           _ptr(aud_ops, I32), _ptr(group_bits, I32), _stream()), "aug_sample")


# ---- encoder blocks ----------------------------------------------------------------------------------------
def conv_supported(Cin, Cout, H, W, K, pad):
    return bool(_lib_().b200_conv_supported(Cin, Cout, H, W, K, pad))


def conv_fwd(x, w, bias, z, stats, n_per_view, pad):
    N, Cin, H, W = x.shape
    Cout, _, K, _ = w.shape
    _lib.check(_lib_().b200_conv_fwd(_ptr(x, F32), _ptr(w, F32), _ptr(bias, F32), _ptr(z, F32), _ptr(stats, F64), N, n_per_view, Cin,
                                     Cout, H, W, K, pad, _stream()), "conv_fwd")


def conv_bwd_data(dz, w, dx, pad):
    N, Cin, H, W = dx.shape
    Cout, _, K, _ = w.shape
    _lib.check(_lib_().b200_conv_bwd_data(_ptr(dz, F32), _ptr(w, F32), _ptr(dx, F32), N, Cin, Cout, H, W, K, pad, _stream()), "conv_bwd_data")


def conv_bwd_weight_work_floats(N, Cin, Cout, H, W, K, pad):
    n = _lib_().b200_conv_bwd_weight_work_floats(N, Cin, Cout, H, W, K, pad)
    if n < 0:
        raise _lib.B200Error(f"conv_bwd_weight: shape {(Cin, Cout, H, W, K, pad)} not compiled")
    return n


def conv_bwd_weight(x, dz, dw, db, work, pad):
    N, Cin, H, W = x.shape
    Cout, _, K, _ = dw.shape
    _lib.check(_lib_().b200_conv_bwd_weight(_ptr(x, F32), _ptr(dz, F32), _ptr(dw, F32), _ptr(db, F32), _ptr(work, F32), N, Cin, Cout, H, W,
                                            K, pad, _stream()), "conv_bwd_weight")


# ---- tensor-core convolutions (tcgen05 / TMEM / TMA; bf16 "act8" activations [N][C/8][H][W][8]) -----------------
BF16 = torch.bfloat16


def conv_tc_supported(Cin, Cout, H, W, K, pad):
    return bool(_lib_().b200_conv_tc_supported(Cin, Cout, H, W, K, pad))


def conv_tc_weight_bytes(Cin, Cout, K):
    return int(_lib_().b200_conv_tc_weight_bytes(Cin, Cout, K))


def conv_tc_prep_weights(w, wprep, flip=False):
    """fp32 OIHW weight -> the bf16 operand image of b200_conv_tc.  flip=True prepares the data-gradient convolution
    (w stays the forward weight [Cout_fwd, Cin_fwd, K, K]; the call's Cin is Cout_fwd)."""
    Co, Ci, K, _ = w.shape
    cin, cout = (Co, Ci) if flip else (Ci, Co)
    _lib.check(_lib_().b200_conv_tc_prep_weights(_ptr(w, F32), _ptr(wprep), cin, cout, K, 1 if flip else 0, _stream()), "conv_tc_prep_weights")


def pack_act8(x, out):
    """fp32 NCHW -> bf16 act8 [N, C/8, H, W, 8]"""
    N, Cc, H, W = x.shape
    _lib.check(_lib_().b200_pack_act8(_ptr(x, F32), _ptr(out, BF16), N, Cc, H, W, _stream()), "pack_act8")


def conv_tc(x8, wprep, bias, out, stats, n_per_view, Cout, K, pad):
    """x8: bf16 act8 [N, Cin/8, H, W, 8] (or the quad8 image [N, H, ceil((W + 2 pad) / 4), 8] of a first layer, Cin = 1); out: fp32 NCHW
    [N, Cout, Ho, Wo] or bf16 / fp16 act8 [N, Cout/8, Ho, Wo, 8]; bias/stats may be None (data-gradient use)."""
    if x8.dim() == 4:               # first layer: quad8 image [N, H, WQ, 8]; the width follows from the output
        N, H, WQ, _ = x8.shape
        W = out.shape[-1 if out.dim() == 4 else -2] - 2 * pad + K - 1
        if WQ != quad8_width(W, pad):
            raise _lib.B200Error(f"conv_tc: quad8 input of width {WQ} does not match W={W}, pad={pad}")
        P = 0.125
    else:
        N, P, H, W, _ = x8.shape
    fmt = 1 if out.dtype == BF16 else 2 if out.dtype == torch.float16 else 0
    _lib.check(_lib_().b200_conv_tc(_ptr(x8, BF16), _ptr(wprep), _ptr(bias, F32) if bias is not None else None, _ptr(out),
                                    _ptr(stats, F64) if stats is not None else None, N, n_per_view, int(P * 8), Cout, H, W, K, pad,
                                    fmt, _stream()), "conv_tc")


def conv_tc_pool_supported(Cin, Cout, H, W, K, pad):
    return bool(_lib_().b200_conv_tc_pool_supported(Cin, Cout, H, W, K, pad))


def conv_tc_pool(x8, wprep, bias, gamma, z_out, pool_out, stats, n_per_view, Cout, K, pad):
    """Forward convolution + BatchNorm statistics + the 2x2 window extreme (max / min by sign(gamma)) in the epilogue.
    x8 as in conv_tc; pool_out: fp16 act8 [N, Cout/8, Ho/2, Wo/2, 8]; z_out: fp16 / bf16 act8 [N, Cout/8, Ho, Wo, 8] or None."""
    Wo = pool_out.shape[-2] * 2
    if x8.dim() == 4:
        N, H, WQ, _ = x8.shape
        W = Wo - 2 * pad + K - 1
        if WQ != quad8_width(W, pad):
            raise _lib.B200Error(f"conv_tc_pool: quad8 input of width {WQ} does not match W={W}, pad={pad}")
        Cin = 1
    else:
        N, P, H, W, _ = x8.shape
        Cin = P * 8
    fmt = 0 if z_out is None else (1 if z_out.dtype == BF16 else 2)
    _lib.check(_lib_().b200_conv_tc_pool(_ptr(x8, BF16), _ptr(wprep), _ptr(bias, F32), _ptr(gamma, F32), _ptr(z_out) if z_out is not None else None,
                                         _ptr(pool_out, torch.float16), _ptr(stats, F64), N, n_per_view, Cin, Cout, H, W, K, pad, fmt, _stream()),
               "conv_tc_pool")


def conv_tc_dgrad_bnstat_supported(Cin, Cout, H, W, K, pad):
    return bool(_lib_().b200_conv_tc_dgrad_bnstat_supported(Cin, Cout, H, W, K, pad))


def conv_tc_dgrad_bnstat(dz8, wprep_flip, dx8, p8, gamma, beta, sums, n_per_view, K, pad):
    """Data gradient (dz8 -> dx8, bf16 act8) + the BatchNorm-backward sums of the layer below (from its pooled output p8 and dx8 = dp)
    in the epilogue.  pad = K - 1 - pad_forward."""
    N, P, H, W, _ = dz8.shape
    Cout = dx8.shape[1] * 8
    _lib.check(_lib_().b200_conv_tc_dgrad_bnstat(_ptr(dz8, BF16), _ptr(wprep_flip), _ptr(dx8, BF16), _ptr(p8, BF16), _ptr(gamma, F32), _ptr(beta, F32),
                                                 _ptr(sums, F64), N, n_per_view, P * 8, Cout, H, W, K, pad, _stream()), "conv_tc_dgrad_bnstat")


def bn_relu_apply8(e8, scale, shift, out, n_per_view):
    """p = ReLU(scale * e + shift) on the pooled extreme e8 (fp16 act8) -> out: fp32 NCHW or bf16 act8 (by dtype)."""
    N, P, HP, WP, _ = e8.shape
    _lib.check(_lib_().b200_bn_relu_apply8(_ptr(e8, torch.float16), _ptr(scale, F32), _ptr(shift, F32), _ptr(out), N, n_per_view, P * 8, HP, WP,
                                           _fmt(out), _stream()), "bn_relu_apply8")


def conv_tc_prep_weights_multi(desc):
    """desc: int64 CUDA tensor [n, 6] = (w data_ptr, out data_ptr, Cin, Cout, K, flip) per weight image; one launch for all"""
    _lib.check(_lib_().b200_conv_tc_prep_weights_multi(_ptr(desc, torch.int64), desc.shape[0], _stream()), "conv_tc_prep_weights_multi")


def conv_tc_wgrad_variant(tap=-1):
    """1: one TMEM accumulator per filter tap for the wide 3x3 layers (default), 0: the shift-row kernel everywhere (A/B); -1 queries.
    Returns the previous setting.  Work sizes depend on it."""
    return int(_lib_().b200_conv_tc_wgrad_variant(tap))


def conv_tc_wgrad_work_floats(N, Cin, Cout, H, W, K, pad):
    n = int(_lib_().b200_conv_tc_wgrad_work_floats(N, Cin, Cout, H, W, K, pad))
    if n < 0:
        raise _lib.B200Error(f"conv_tc_wgrad: unsupported geometry {(Cin, Cout, H, W, K, pad)}")
    return n


def conv_tc_wgrad(x8, dz8, dw, work, pad):
    """x8 [N, Cin/8, H, W, 8] (Cin = 1: the shift8 image [N, H, W, 8]), dz8 [N, Cout/8, Ho, Wo, 8] bf16 act8 -> dw [Cout, Cin, K, K]."""
    N, H, W = x8.shape[0], x8.shape[-3], x8.shape[-2]
    Cout, Cin, K, _ = dw.shape
    if Cin == 1:
        W -= pad
    _lib.check(_lib_().b200_conv_tc_wgrad(_ptr(x8, BF16), _ptr(dz8, BF16), _ptr(dw, F32), _ptr(work, F32), N, Cin, Cout, H, W, K, pad,
                                          _stream()), "conv_tc_wgrad")


def conv_tc_wgrad_l0_fused_work_floats(N, n_per_view, Cout, H, W, K, pad):
    n = int(_lib_().b200_conv_tc_wgrad_l0_fused_work_floats(N, n_per_view, Cout, H, W, K, pad))
    if n < 0:
        raise _lib.B200Error(f"conv_tc_wgrad_l0_fused: unsupported geometry {(Cout, H, W, K, pad)}")
    return n


def conv_tc_wgrad_l0_fused(xs8, z8, dp8, scale, shift, mean, invstd, sums, dw, dbsum, work, n_per_view, pad):
    """First-layer backward in one kernel: BN/ReLU/pool backward-apply (z8 fp16 act8, dp8 bf16 act8) + weight gradient."""
    N, P, H, W, _ = z8.shape
    Cout, _, K, _ = dw.shape
    _lib.check(_lib_().b200_conv_tc_wgrad_l0_fused(_ptr(xs8, BF16), _ptr(z8, torch.float16), _ptr(dp8, BF16), _ptr(scale, F32), _ptr(shift, F32),
                                                   _ptr(mean, F32), _ptr(invstd, F32), _ptr(sums, F64), _ptr(dw, F32),
                                                   _ptr(dbsum, F64) if dbsum is not None else None, _ptr(work, F32), N, n_per_view, Cout, H, W,
                                                   K, pad, _stream()), "conv_tc_wgrad_l0_fused")


def quad8_width(W, pad):
    """units per row of the quad8 first-layer image"""
    return (W + 2 * pad + 3) // 4


def pack_quad8(x, out, pad):
    """fp32 [N, H, W] (or [N, 1, H, W]) -> bf16 quad8 [N, H, ceil((W + 2 pad) / 4), 8] (pad = the convolution's padding)"""
    N, H, W = x.shape[0], x.shape[-2], x.shape[-1]
    assert tuple(out.shape) == (N, H, quad8_width(W, pad), 8)
    _lib.check(_lib_().b200_pack_quad8(_ptr(x, F32), _ptr(out, BF16), N, H, W, pad, _stream()), "pack_quad8")


def pack_shift8(x, out, pad):
    """fp32 [N, H, W] (or [N, 1, H, W]) -> bf16 shift8 [N, H, W + pad, 8] (pad = the convolution's padding)"""
    N, H, W = x.shape[0], x.shape[-2], x.shape[-1]
    assert tuple(out.shape) == (N, H, W + pad, 8)
    _lib.check(_lib_().b200_pack_shift8(_ptr(x, F32), _ptr(out, BF16), N, H, W, pad, _stream()), "pack_shift8")


def bias_grad_finalize(dbsum, db):
    _lib.check(_lib_().b200_bias_grad_finalize(_ptr(dbsum, F64), _ptr(db, F32), db.numel(), _stream()), "bias_grad_finalize")


def unpack_act8(x8, out):
    N, P, H, W, _ = x8.shape
    _lib.check(_lib_().b200_unpack_act8(_ptr(x8, BF16), _ptr(out, F32), N, P * 8, H, W, _stream()), "unpack_act8")


def _fmt(t):
    return 1 if t.dtype == BF16 else 0


def _zf16(z8):
    if z8.dtype not in (BF16, torch.float16):
        raise _lib.B200Error(f"act8 z must be bf16 or fp16, got {z8.dtype}")
    return 1 if z8.dtype == torch.float16 else 0


def bn_relu_pool8_fwd(z8, scale, shift, out, n_per_view):
    """z8 bf16 act8 [N, C/8, H, W, 8] -> out: fp32 NCHW [N, C, H/2, W/2] or bf16 act8 [N, C/8, H/2, W/2, 8] (by dtype)."""
    N, P, H, W, _ = z8.shape
    _lib.check(_lib_().b200_bn_relu_pool8_fwd(_ptr(z8), _ptr(scale, F32), _ptr(shift, F32), _ptr(out), N, n_per_view, P * 8, H, W,
                                              _zf16(z8), _fmt(out), _stream()), "bn_relu_pool8_fwd")


def bn_relu_pool8_bwd_reduce(z8, dp, scale, shift, mean, invstd, sums, n_per_view):
    N, P, H, W, _ = z8.shape
    _lib.check(_lib_().b200_bn_relu_pool8_bwd_reduce(_ptr(z8), _ptr(dp), _ptr(scale, F32), _ptr(shift, F32), _ptr(mean, F32),
                                                     _ptr(invstd, F32), _ptr(sums, F64), N, n_per_view, P * 8, H, W, _zf16(z8), _fmt(dp), _stream()),
               "bn_relu_pool8_bwd_reduce")


def bn_pool8_bwd_reduce_p(p, dp, gamma, beta, sums, n_per_view):
    """BatchNorm-backward sums {sum g, sum g*xhat} from the pooled output p and its gradient dp only (fp32 NCHW or bf16 act8 each)."""
    if p.dim() == 5:
        N, P, HP, WP, _ = p.shape
        Cc = P * 8
    else:
        N, Cc, HP, WP = p.shape
    _lib.check(_lib_().b200_bn_pool8_bwd_reduce_p(_ptr(p), _ptr(dp), _ptr(gamma, F32), _ptr(beta, F32), _ptr(sums, F64), N, n_per_view, Cc,
                                                  HP, WP, _fmt(p), _fmt(dp), _stream()), "bn_pool8_bwd_reduce_p")


def bn_relu_pool8_bwd_apply(z8, dp, scale, shift, mean, invstd, sums, dz8, n_per_view, dbsum=None):
    N, P, H, W, _ = z8.shape
    _lib.check(_lib_().b200_bn_relu_pool8_bwd_apply(_ptr(z8), _ptr(dp), _ptr(scale, F32), _ptr(shift, F32), _ptr(mean, F32),
                                                    _ptr(invstd, F32), _ptr(sums, F64), _ptr(dz8, BF16),
                                                    _ptr(dbsum, F64) if dbsum is not None else None, N, n_per_view, P * 8, H, W, _zf16(z8),
                                                    _fmt(dp), _stream()), "bn_relu_pool8_bwd_apply")


def bn_finalize(stats, gamma, beta, running_mean, running_var, nbt, scale, shift, mean, invstd, n_views, count, train=True,
                momentum=0.1, eps=1e-5):
    Cc = gamma.numel()
    _lib.check(_lib_().b200_bn_finalize(_ptr(stats, F64), _ptr(gamma, F32), _ptr(beta, F32), _ptr(running_mean, F32), _ptr(running_var, F32),
                                        _ptr(nbt, I64), _ptr(scale, F32), _ptr(shift, F32), _ptr(mean, F32), _ptr(invstd, F32), n_views,
                                        Cc, count, momentum, eps, 1 if train else 0, _stream()), "bn_finalize")


def bn_relu_pool_fwd(z, scale, shift, out, n_per_view):
    N, Cc, H, W = z.shape
    _lib.check(_lib_().b200_bn_relu_pool_fwd(_ptr(z, F32), _ptr(scale, F32), _ptr(shift, F32), _ptr(out, F32), N, n_per_view, Cc, H, W,
                                             _stream()), "bn_relu_pool_fwd")


def bn_relu_pool_bwd_reduce(z, dout, scale, shift, mean, invstd, sums, n_per_view):
    N, Cc, H, W = z.shape
    _lib.check(_lib_().b200_bn_relu_pool_bwd_reduce(_ptr(z, F32), _ptr(dout, F32), _ptr(scale, F32), _ptr(shift, F32), _ptr(mean, F32),
                                                    _ptr(invstd, F32), _ptr(sums, F64), N, n_per_view, Cc, H, W, _stream()),
               "bn_relu_pool_bwd_reduce")


def bn_relu_pool_bwd_apply(z, dout, scale, shift, mean, invstd, sums, dz, n_per_view):
    N, Cc, H, W = z.shape
    _lib.check(_lib_().b200_bn_relu_pool_bwd_apply(_ptr(z, F32), _ptr(dout, F32), _ptr(scale, F32), _ptr(shift, F32), _ptr(mean, F32),
                                                   _ptr(invstd, F32), _ptr(sums, F64), _ptr(dz, F32), N, n_per_view, Cc, H, W, _stream()),
               "bn_relu_pool_bwd_apply")


def bn_param_grads(sums, dgamma, dbeta, n_views, accumulate=False):
    _lib.check(_lib_().b200_bn_param_grads(_ptr(sums, F64), _ptr(dgamma, F32), _ptr(dbeta, F32), n_views, dgamma.numel(),
                                           1 if accumulate else 0, _stream()), "bn_param_grads")


def avgpool_fwd(x, out):
    N, Cc = x.shape[0], x.shape[1]
    _lib.check(_lib_().b200_avgpool_fwd(_ptr(x, F32), _ptr(out, F32), N, Cc, x[0, 0].numel(), _stream()), "avgpool_fwd")


def avgpool_bwd(dout, dx):
    N, Cc = dx.shape[0], dx.shape[1]
    _lib.check(_lib_().b200_avgpool_bwd(_ptr(dout, F32), _ptr(dx, F32), N, Cc, dx[0, 0].numel(), _stream()), "avgpool_bwd")


# ---- linear layers -----------------------------------------------------------------------------------------
def _rows(t):
    """(pointer, row stride) of a 2-D tensor whose rows are contiguous (column slices of a wider matrix allowed)."""
    if not t.is_cuda or t.dtype != F32 or t.dim() != 2 or t.stride(1) != 1:
        raise _lib.B200Error("linear ops need 2-D fp32 CUDA tensors with unit column stride")
    return t.data_ptr(), t.stride(0)


def linear_fwd(x, w, bias, y, act=0, mask=None, drop_p=0.0, tc=False):
    """y = act(x w^T + bias); tc=True: tcgen05 tf32 tensor-core GEMM, else the exact fp32 SIMT kernel."""
    M, K = x.shape
    N = w.shape[0]
    xp, ldx = _rows(x)
    yp, ldy = _rows(y)
    fn = _lib_().b200_linear_fwd_tc if tc else _lib_().b200_linear_fwd
    _lib.check(fn(xp, ldx, _ptr(w, F32), _ptr(bias, F32), yp, ldy, M, N, K, act, _ptr(mask, U8), drop_p, _stream()), "linear_fwd")


_LINEAR_WORK = {}


def _linear_work(device, need):
    key = (device, _stream())               # one cached scratch per device AND stream (concurrent streams must not share it)
    work = _LINEAR_WORK.get(key)
    if work is None or work.numel() < need:
        work = _LINEAR_WORK[key] = torch.empty(max(need, 4), dtype=F32, device=device)
    return work


def linear_bwd_data(dy, w, dx, tc=False):
    M, N = dy.shape
    K = w.shape[1]
    dyp, lddy = _rows(dy)
    dxp, lddx = _rows(dx)
    if tc:
        work = _linear_work(dy.device, _lib_().b200_linear_bwd_data_tc_work_floats(M, N, K))
        _lib.check(_lib_().b200_linear_bwd_data_tc(dyp, lddy, _ptr(w, F32), dxp, lddx, _ptr(work, F32), M, N, K, _stream()), "linear_bwd_data")
    else:
        _lib.check(_lib_().b200_linear_bwd_data(dyp, lddy, _ptr(w, F32), dxp, lddx, M, N, K, _stream()), "linear_bwd_data")


def linear_bwd_weight(dy, x, dw, db, accumulate=False, work=None, tc=False):
    M, N = dy.shape
    K = x.shape[1]
    dyp, lddy = _rows(dy)
    xp, ldx = _rows(x)
    need = (_lib_().b200_linear_bwd_weight_tc_work_floats if tc else _lib_().b200_linear_bwd_weight_work_floats)(M, N, K)
    if work is None and need > 0:
        work = _linear_work(dy.device, need)
    fn = _lib_().b200_linear_bwd_weight_tc if tc else _lib_().b200_linear_bwd_weight
    _lib.check(fn(dyp, lddy, xp, ldx, _ptr(dw, F32), _ptr(db, F32), _ptr(work, F32), M, N, K, 1 if accumulate else 0, _stream()),
               "linear_bwd_weight")


# ---- feature mixing of the simple multimodal encoder family (gates, batch-wide cross attention; csrc/mix.cu) ----------
def gate_apply(x, gate, y):
    """y = sigmoid(gate) * x over a 2-D block (rows may be strided); models/dino.py:249-256."""
    M, N = x.shape
    xp, ldx = _rows(x)
    yp, ldy = _rows(y)
    _lib.check(_lib_().b200_gate_apply(xp, ldx, yp, ldy, _ptr(gate, F32), M, N, _stream()), "gate_apply")


def gate_grad_work_floats():
    return int(_lib_().b200_gate_grad_work_floats())


def gate_grad(dy, x, gate, dgate, work, accumulate=False):
    """dgate (+)= sigmoid'(gate) * sum(dy * x); work: zero-initialised scratch of gate_grad_work_floats() floats."""
    M, N = x.shape
    dyp, lddy = _rows(dy)
    xp, ldx = _rows(x)
    _lib.check(_lib_().b200_gate_grad(dyp, lddy, xp, ldx, _ptr(gate, F32), _ptr(dgate, F32), _ptr(work, F32), M, N, 1 if accumulate else 0,
                                      _stream()), "gate_grad")


def softmax_rows(s, scale):
    """s <- softmax(scale * s) per row, in place (attention weights, models/dino.py:400-401)."""
    M, N = s.shape
    sp, ld = _rows(s)
    _lib.check(_lib_().b200_softmax_rows(sp, ld, M, N, scale, _stream()), "softmax_rows")


def softmax_rows_bwd(dp, p, scale):
    """dp <- scale * p * (dp - sum_n dp p) per row, in place on dp."""
    M, N = p.shape
    dpp, lddp = _rows(dp)
    pp, ldp = _rows(p)
    _lib.check(_lib_().b200_softmax_rows_bwd(dpp, lddp, pp, ldp, M, N, scale, _stream()), "softmax_rows_bwd")


def add2d(dst, src):
    """dst += src for 2-D blocks with row strides."""
    M, N = dst.shape
    dp, ldd = _rows(dst)
    sp, lds = _rows(src)
    _lib.check(_lib_().b200_add2d(dp, ldd, sp, lds, M, N, _stream()), "add2d")


def act_bwd(dy, y, drop_p=0.0):
    _lib.check(_lib_().b200_act_bwd(_ptr(dy, F32), _ptr(y, F32), None, drop_p, dy.numel(), _stream()), "act_bwd")


def colstats(h, stats):
    M, Cc = h.shape
    _lib.check(_lib_().b200_colstats(_ptr(h, F32), _ptr(stats, F64), M, Cc, _stream()), "colstats")


def bn1d_gelu_drop_fwd(h, scale, shift, mask, drop_p, g):
    M, Cc = h.shape
    _lib.check(_lib_().b200_bn1d_gelu_drop_fwd(_ptr(h, F32), _ptr(scale, F32), _ptr(shift, F32), _ptr(mask, U8), drop_p, _ptr(g, F32), M, Cc,
                                               _stream()), "bn1d_gelu_drop_fwd")


def bn1d_gelu_drop_bwd_reduce(h, dg, scale, shift, mean, invstd, mask, drop_p, sums):
    M, Cc = h.shape
    _lib.check(_lib_().b200_bn1d_gelu_drop_bwd_reduce(_ptr(h, F32), _ptr(dg, F32), _ptr(scale, F32), _ptr(shift, F32), _ptr(mean, F32),
                                                      _ptr(invstd, F32), _ptr(mask, U8), drop_p, _ptr(sums, F64), M, Cc, _stream()),
               "bn1d_gelu_drop_bwd_reduce")


def bn1d_gelu_drop_bwd_apply(h, dg, scale, shift, mean, invstd, mask, drop_p, sums, dh):
    M, Cc = h.shape
    _lib.check(_lib_().b200_bn1d_gelu_drop_bwd_apply(_ptr(h, F32), _ptr(dg, F32), _ptr(scale, F32), _ptr(shift, F32), _ptr(mean, F32),
                                                     _ptr(invstd, F32), _ptr(mask, U8), drop_p, _ptr(sums, F64), _ptr(dh, F32), M, Cc,
                                                     _stream()), "bn1d_gelu_drop_bwd_apply")


# ---- kNN evaluation of frozen features (SURVEY 8f-3) -----------------------------------------------------------------
def knn_predict(train_feats, train_labels, test_feats, k=5, n_classes=10, return_neighbours=False, chunk=2048):
    """sklearn KNeighborsClassifier(n_neighbors=k).fit(train).predict(test) on device features (training_structures/dino_train.py:
    349-368): exact-fp32 score GEMM (a.b - |b|^2/2, larger = nearer) + per-row top-k + majority vote, `chunk` test rows at a time."""
    N, D = train_feats.shape
    M = test_feats.shape[0]
    dev = train_feats.device
    bias = torch.empty(N, dtype=F32, device=dev)
    tp, ldt = _rows(train_feats)
    _lib.check(_lib_().b200_knn_neg_half_sqnorm(tp, ldt, N, D, _ptr(bias, F32), _stream()), "knn_neg_half_sqnorm")
    pred = torch.empty(M, dtype=I64, device=dev)
    nbr = torch.empty(M, k, dtype=I32, device=dev) if return_neighbours else None
    scores = torch.empty(min(chunk, M), N, dtype=F32, device=dev)
    labels = train_labels.to(I64).contiguous()
    for lo in range(0, M, chunk):
        hi = min(M, lo + chunk)
        linear_fwd(test_feats[lo:hi], train_feats, bias, scores[:hi - lo])
        _lib.check(_lib_().b200_knn_topk_vote(_ptr(scores, F32), N, _ptr(labels, I64), hi - lo, N, k, n_classes, pred[lo:hi].data_ptr(),
                                              nbr[lo:hi].data_ptr() if nbr is not None else None, _stream()), "knn_topk_vote")
    return (pred, nbr) if return_neighbours else pred


# ---- downstream MLP probe (train_downstream; csrc/probe.cu) -------------------------------------------------------------
def probe_work_floats(B, C):
    n = int(_lib_().b200_probe_work_floats(B, C))
    if n < 0:
        raise _lib.B200Error(f"probe_work_floats: unsupported shape B={B} C={C}")
    return n


def probe_mlp_fwd_bwd(x, w1, b1, w2, b2, labels, work, loss_sum, correct, grad=None, preds=None, confusion=None, train=True):
    """DownstreamClassifier head + CrossEntropyLoss on features x [B, O]: train=True writes [dW1 | db1 | dW2 | db2] into grad;
    train=False writes the argmax into preds [B] and counts [label, pred] into confusion [C, C] (both optional).  Always:
    loss_sum (fp64 [1]) += the batch's loss sum, correct (int64 [1]) += its correct predictions."""
    B, O = x.shape
    C = b2.numel()
    _lib.check(_lib_().b200_probe_mlp_fwd_bwd(_ptr(x, F32), _ptr(w1, F32), _ptr(b1, F32), _ptr(w2, F32), _ptr(b2, F32), _ptr(labels, I64),
                                              B, O, C, int(bool(train)), _ptr(grad, F32), _ptr(work, F32), _ptr(loss_sum, F64),
                                              _ptr(correct, I64), _ptr(preds, I64), _ptr(confusion, I64), _stream()), "probe_mlp_fwd_bwd")


# ---- launch accounting and optional per-op timing ------------------------------------------------------------
# Every wrapper above issues a fixed number of kernel launches; the table lists the ones that issue more than one.
_LAUNCHES = {"gate_grad": 2, "probe_mlp_fwd_bwd": 2, "ntxent_fwd_bwd": 5, "conv_tc_wgrad_l0_fused": 3, "conv_tc_wgrad": 2, "conv_bwd_weight": 3, "linear_bwd_weight": 3, "infonce_fwd_bwd": 9}
_NOT_KERNELS = {"conv_tc_wgrad_variant", "probe_work_floats", "gate_grad_work_floats", "knn_predict", "conv_tc_pool_supported", "conv_tc_dgrad_bnstat_supported", "quad8_width", "ntxent_work_floats", "conv_tc_wgrad_l0_fused_work_floats", "conv_tc_wgrad_work_floats", "conv_tc_supported", "conv_tc_weight_bytes", "dino_loss_parts", "infonce_work_floats", "conv_supported", "conv_bwd_weight_work_floats", "launch_count", "start_profile", "stop_profile"}
LAUNCH_COUNT = 0
_PROFILE = None          # None, or a list receiving (name, start_event, end_event, meta)


def launch_count():
    return LAUNCH_COUNT


def start_profile():
    """Record a CUDA-event pair around every op call (events are recorded on the current stream, the stream the kernels
    are launched on).  Returns the list that collects (name, start, end, meta) until stop_profile()."""
    global _PROFILE
    _PROFILE = []
    return _PROFILE


def stop_profile():
    global _PROFILE
    rec, _PROFILE = _PROFILE, None
    return rec


# tensor-core variants of the linear / InfoNCE wrappers issue more kernels (transposes, split-K and partial-sum reductions)
_LAUNCHES_TC = {"linear_bwd_weight": 6, "linear_bwd_data": 2, "infonce_fwd_bwd": 19}


def _wrap(name, fn):
    n_launch = _LAUNCHES.get(name, 1)
    n_launch_tc = _LAUNCHES_TC.get(name, n_launch)

    def wrapped(*args, **kwargs):
        global LAUNCH_COUNT
        LAUNCH_COUNT += n_launch_tc if kwargs.get("tc") else n_launch
        if _PROFILE is None:
            return fn(*args, **kwargs)
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        out = fn(*args, **kwargs)
        b.record()
        head = args[:6] if name == "conv_tc_pool" else args[:4]        # conv_tc_pool: (x, wprep, bias, gamma, z | None, e)
        meta = tuple(tuple(t.shape) for t in list(head) + list(kwargs.values()) if isinstance(t, torch.Tensor))
        meta = meta + (("i",) + tuple(int(v) for v in args if isinstance(v, int) and not isinstance(v, bool)),)
        _PROFILE.append((name, a, b, meta, _stream()))
        return out

    wrapped.__name__ = name
    wrapped.__doc__ = fn.__doc__
    return wrapped


for _name, _fn in list(globals().items()):
    if callable(_fn) and not _name.startswith("_") and _name not in _NOT_KERNELS and getattr(_fn, "__module__", None) == __name__ \
            and _name not in ("launch_count", "start_profile", "stop_profile", "MultiTensorTable"):
        globals()[_name] = _wrap(_name, _fn)
