"""Every kernel launch of a benchmark-size training step, checked against float64 on the operands that launch actually used.

The per-kernel tests (test_conv_tc_gpu.py, test_kernels_gpu.py) cover the shapes they list, at a few hundred samples per
launch.  The benchmarked steps launch the same kernels at N = 6144 .. 57344 samples, i.e. with another CTA partition
(`items*g/G` bands, issuer splits, grid-stride loops, split-K and row-partial counts).  Here one eager `forward_backward` per
benchmark configuration runs with every wrapped op of `ops` replaced by a recorder that

  * synchronises, snapshots the call's tensors (inputs, and outputs for the ops that accumulate into them), runs the op,
    synchronises again,
  * rebuilds the operation in float64 on the GPU from the launch's own operands (act8 / quad8 / shift8 unpacked exactly; the
    prepared weight images mapped back to the fp32 parameter they were made from) and bounds every output element by

        |got - ref| <= a * R_abs + r * |ref|

    where R_abs is the same operation on the absolute values of the operands, `a` the accumulation / operand rounding of the
    kernel and `r` the rounding of the output format (constants below),
  * prints the worst ratio error / bound for every op.

The streams of the engines are serialised by the synchronisation around every call (host order is a valid order for them);
that changes timing, not results.  Per-sample float64 convolutions cover every sample whose launch also produces statistics
(the statistics need the whole batch) and otherwise ~64 samples per view-call: the first and last and those on both sides of
the CTA boundaries `n_per_view * g / G` of conv_tc.cu.  Reductions always cover the whole batch, accumulated in chunks.
"""
import collections
import inspect
import math
import time

import pytest
import torch
import torch.nn.functional as F

pytestmark = pytest.mark.gpu

from oracle import dino_ref as R
from oracle.fixtures import contrastive_batch, make_masks, synth_views, views_to_vb
from multimodal_ssl_avmnist_b200 import ops

DEV = "cuda"
F64 = torch.float64

# ---- error model ------------------------------------------------------------------------------------------------------
# a: products of bf16 / fp16 operands are exact in fp32; what remains is the fp32 accumulation (TMEM / per-thread partials,
# then fp64 atomics or a fixed-order partial sum).  A sequential fp32 sum of n terms is off by at most ~n * 2^-24 of the sum
# of magnitudes; the kernels keep n per accumulator in the hundreds to thousands (bands, split-K, partial rows), whence 2^-16.
A_EXACT = 2.0 ** -16
# weight gradients reduce N * pixels terms (10^7 .. 10^8) along fp32 TMEM chains of ~10^5 terms each.  The worst case
# n * 2^-24 would hide whole samples; the chain's rounding errors follow its signed partial sums, which BatchNorm-centred dz
# keeps far below the sum of magnitudes.  Measured on a B200 (1000 W), as a fraction of sum |x||dz|:
#   * the formulations the engine launches (conv_tc_wgrad_variant 1: per-tap accumulators of the wide 3x3 layers, shift rows
#     elsewhere; the fused first layer): up to 2^-15.0 (contrastive InfoNCE audio conv2, N = 8192) -> A_WGRAD = 2^-14, which
#     still flags a median-sized sample left out of N = 6144 (test_control_sample_left_out_of_weight_gradient_is_flagged);
#   * the shift-row formulation of the wide 3x3 layers (variant 0, an A/B setting the engine does not use): up to 2^-13.8
#     (audio conv3, N = 8192) -> A_WGRAD_SHIFT_ROW = 2^-13
A_WGRAD = 2.0 ** -14
A_WGRAD_SHIFT_ROW = 2.0 ** -13
# tf32 tensor-core GEMMs (linears): both operands lose their 13 low mantissa bits (<= 2^-10 each) -> <= 2^-9 per product,
# plus the fp32 accumulation
A_TF32 = 2.0 ** -9 + 2.0 ** -12
# the InfoNCE gradient GEMMs multiply bf16 copies of the softmax matrix and of the normalised rows (2^-9 each, 2^-8 per
# product), on top of fp32 exp / log / normalisation
A_BF16_GEMM = 2.0 ** -7
# element-wise fp32 arithmetic (a few fma / div / sqrt / exp roundings)
A_ELEM = 2.0 ** -20
# fp32 per-thread partial sums feeding fp64 atomics / fixed-order sums (statistics, BatchNorm-backward sums, bias sums)
A_SUM = 2.0 ** -14
# r: rounding of the output format to nearest: |fl(v) - v| <= 2^-8 |v| in bf16 (8 significant bits), 2^-11 |v| in fp16 (taken
# as 2^-10), exact in fp32
R_OUT = {torch.float32: 0.0, torch.bfloat16: 2.0 ** -8, torch.float16: 2.0 ** -10}
FP16_TINY = 2.0 ** -24          # fp16 subnormal spacing: the absolute floor of an fp16 output

SUBSET = 64                     # per-sample fp64 references: about this many samples per view-call
CHUNK_ELEMS = 1 << 27           # fp64 elements per chunk of a batched reference

# (Cin, Cout, H, K, pad) of a conv_tc launch -> (CTAs per SM, output-channel split) of its instance in conv_tc.cu (TcCfg<...>);
# the kernel's grid is G = SMs * CTAS / (views * NSPLIT) and CTA g owns the samples from n_per_view * g / G on
CONV_CTAS = {(8, 16, 56, 5, 2): (2, 1), (16, 32, 28, 5, 2): (1, 1), (32, 64, 14, 5, 2): (1, 1), (32, 64, 14, 5, 0): (1, 1),
             (16, 8, 56, 5, 2): (1, 1), (32, 16, 28, 5, 2): (1, 1), (64, 32, 14, 5, 2): (1, 1), (64, 32, 10, 5, 4): (1, 1),
             (1, 8, 112, 5, 2): (3, 1), (1, 32, 28, 5, 2): (1, 1), (1, 32, 28, 3, 1): (1, 1), (64, 128, 7, 3, 1): (2, 2),
             (128, 64, 7, 3, 1): (1, 1), (32, 64, 14, 3, 1): (1, 1), (64, 32, 14, 3, 1): (1, 1), (1, 32, 112, 3, 1): (2, 1),
             (32, 64, 56, 3, 1): (1, 1), (64, 32, 56, 3, 1): (1, 1), (64, 128, 28, 3, 1): (1, 2), (128, 64, 28, 3, 1): (1, 1),
             (128, 256, 14, 3, 1): (1, 4), (256, 128, 14, 3, 1): (1, 4)}

# ops a step may call that have no float64 checker here, and why
UNCHECKED = {
    "conv_tc_prep_weights_multi": "opaque bf16 operand images; every conv_tc* launch that reads one is checked against the fp32 "
                                  "parameter it was made from, and test_prep_weights_multi_matches_single_launches pins the layout",
    "conv_tc_prep_weights": "as conv_tc_prep_weights_multi (single-image form)",
    "bn1d_gelu_drop_fwd": "exact-fp32 element-wise BatchNorm1d / GELU / dropout of the projection heads; held to the oracle by "
                          "test_step_gpu and test_scale_gpu",
    "bn1d_gelu_drop_bwd_reduce": "exact-fp32 SIMT backward of the projection-head BatchNorm1d (oracle parity in test_step_gpu)",
    "bn1d_gelu_drop_bwd_apply": "exact-fp32 SIMT backward of the projection-head BatchNorm1d (oracle parity in test_step_gpu)",
    "act_bwd": "exact-fp32 ReLU / dropout backward mask (oracle parity in test_step_gpu and test_scale_gpu)",
    "dropout_mask": "Philox keep-mask; the steps here take explicit masks",
    "conv_fwd": "exact-fp32 SIMT convolution of layers without a tensor-core kernel (test_kernels_gpu)",
    "conv_bwd_data": "exact-fp32 SIMT convolution of layers without a tensor-core kernel (test_kernels_gpu)",
    "conv_bwd_weight": "exact-fp32 SIMT convolution of layers without a tensor-core kernel (test_kernels_gpu)",
    "bn_relu_pool_fwd": "fp32-NCHW BatchNorm / ReLU / pool of layers without a tensor-core kernel (test_kernels_gpu)",
    "bn_relu_pool_bwd_reduce": "fp32-NCHW BatchNorm / ReLU / pool of layers without a tensor-core kernel (test_kernels_gpu)",
    "bn_relu_pool_bwd_apply": "fp32-NCHW BatchNorm / ReLU / pool of layers without a tensor-core kernel (test_kernels_gpu)",
}


# ---- layouts ----------------------------------------------------------------------------------------------------------
def nchw(t):
    """act8 [N, C/8, H, W, 8] -> NCHW (same dtype); NCHW passes through"""
    if t.dim() == 5:
        N, P, H, W, _ = t.shape
        return t.permute(0, 1, 4, 2, 3).reshape(N, P * 8, H, W)
    return t


def act8(t):
    """NCHW -> act8 [N, C/8, H, W, 8]"""
    N, C, H, W = t.shape
    return t.reshape(N, C // 8, 8, H, W).permute(0, 1, 3, 4, 2).contiguous()


def quad8_image(x, W, pad):
    """quad8 [N, H, WQ, 8] (unit xq = padded-row pixels 4 xq .. 4 xq + 7) -> [N, 1, H, W]"""
    N, H, WQ, _ = x.shape
    return x[..., :4].reshape(N, H, 4 * WQ)[..., pad:pad + W].unsqueeze(1)


def shift8_image(x, pad):
    """shift8 [N, H, W + pad, 8] (element e of unit q = left-padded pixel q + e) -> [N, 1, H, W]"""
    return x[:, :, pad:, 0].unsqueeze(1)


def quad8_of(x, pad):
    """fp32 [N, H, W] -> the bf16 quad8 image pack_quad8 must write"""
    W = x.shape[-1]
    wq = ops.quad8_width(W, pad)
    padded = F.pad(x, (pad, 4 * wq + 8 - W - pad))
    return padded.unfold(-1, 8, 4)[..., :wq, :].to(torch.bfloat16)


def shift8_of(x, pad):
    W = x.shape[-1]
    padded = F.pad(x, (pad, 8))
    return padded.unfold(-1, 8, 1)[..., :W + pad, :].to(torch.bfloat16)


def rows_of(n, npv):
    return [(v * npv, (v + 1) * npv) for v in range(n // npv)]


def chunks(lo, hi, per):
    step = max(1, CHUNK_ELEMS // max(1, per))
    for a in range(lo, hi, step):
        yield a, min(hi, a + step)


def boundary_samples(npv, views, geom):
    """first / last sample of a view-call and the samples on both sides of the CTA boundaries of conv_tc.cu"""
    ctas, nsplit = CONV_CTAS.get(geom, (1, 1))
    G = max(1, min(npv, torch.cuda.get_device_properties(0).multi_processor_count * ctas // (views * nsplit)))
    cuts = sorted({npv * g // G for g in range(1, G)})
    keep = (SUBSET - 2) // 2
    if len(cuts) > keep:
        cuts = [cuts[round(i * (len(cuts) - 1) / (keep - 1))] for i in range(keep)]
    s = {0, npv - 1}
    for c in cuts:
        s |= {c - 1, c}
    return sorted(x for x in s if 0 <= x < npv)


# ---- bounds -----------------------------------------------------------------------------------------------------------
def ratio(got, ref, rabs, a, r=0.0, floor=0.0):
    """max over elements of |got - ref| / (a * rabs + r * |ref| + floor)  (0 where both sides are 0, inf where only the error is)"""
    got, ref = got.to(F64), ref.to(F64)
    if got.shape != ref.shape and got.numel() == ref.numel():
        got = got.reshape(ref.shape)
    err = (got - ref).abs()
    bound = a * rabs.to(F64) + r * ref.abs() + floor
    q = torch.where(err == 0, torch.zeros_like(err), err / bound)
    if q.numel() == 0:
        return 0.0
    if bool(torch.isnan(q).any()):      # a NaN output (or an unwritten, NaN-filled element) never passes
        return math.inf
    return float(q.max())


def worse(worst, q):
    """max that keeps a NaN ratio (Python's max(0.0, nan) is 0.0)"""
    return q if not q <= worst else worst


class Result:
    """per-launch outcome: (label, ratio) pairs"""

    def __init__(self):
        self.items = []

    def add(self, label, q):
        self.items.append((label, q))

    @property
    def worst(self):
        w = 0.0
        for _, q in self.items:
            w = worse(w, q)
        return w


# ---- float64 references -----------------------------------------------------------------------------------------------
def conv_weight(img):
    """the fp32 parameter of a prepared image -> the OIHW weight of the convolution the launch computes (bf16 operands)"""
    w = img["w"].to(torch.bfloat16).to(F64)
    if img["flip"]:                    # data gradient: channels swapped, taps mirrored
        w = w.transpose(0, 1).flip(-1, -2)
    return w


def conv_input(x8, out_w, K, pad):
    """the launch's input as fp64 NCHW: act8, or the quad8 image of a first layer"""
    if x8.dim() == 4:
        W = out_w - 2 * pad + K - 1
        return lambda a, b: quad8_image(x8[a:b], W, pad).to(F64)
    return lambda a, b: nchw(x8[a:b]).to(F64)


def conv_out_check(res, label, xin, w, bias, pad, got, samples_or_range, stats_delta=None, npv=None):
    """fp64 forward of the rows in `samples_or_range`; stats: also the per-(view, channel) sums over the whole batch"""
    wa = w.abs()
    ba = bias.abs() if bias is not None else None
    dt = got.dtype
    per = got[0].numel()
    worst = 0.0
    if stats_delta is not None:
        N = got.shape[0]
        s_ref = torch.zeros_like(stats_delta)
        s_bnd = torch.zeros_like(stats_delta)
        for v, (lo, hi) in enumerate(rows_of(N, npv)):
            for a, b in chunks(lo, hi, per * 4):
                x = xin(a, b)
                ref = F.conv2d(x, w, bias, padding=pad)
                rab = F.conv2d(x.abs(), wa, ba, padding=pad)
                g = nchw(got[a:b])
                worst = worse(worst, ratio(g, ref, rab, A_EXACT, R_OUT[dt], FP16_TINY if dt == torch.float16 else 0.0))
                s_ref[v, :, 0] += ref.sum(dim=(0, 2, 3))
                s_ref[v, :, 1] += (ref * ref).sum(dim=(0, 2, 3))
                s_bnd[v, :, 0] += A_EXACT * rab.sum(dim=(0, 2, 3)) + A_SUM * ref.abs().sum(dim=(0, 2, 3))
                s_bnd[v, :, 1] += 2 * A_EXACT * (ref.abs() * rab).sum(dim=(0, 2, 3)) + A_SUM * (ref * ref).sum(dim=(0, 2, 3))
        res.add(label, worst)
        res.add(label + ".stats", ratio(stats_delta, s_ref, s_bnd, 1.0))
        return
    idx = torch.tensor(samples_or_range, device=got.device)
    for a in range(0, len(idx), 16):
        sel = idx[a:a + 16]
        x = torch.cat([xin(int(i), int(i) + 1) for i in sel])
        ref = F.conv2d(x, w, bias, padding=pad)
        rab = F.conv2d(x.abs(), wa, ba, padding=pad)
        g = nchw(got[sel])
        worst = worse(worst, ratio(g, ref, rab, A_EXACT, R_OUT[dt], FP16_TINY if dt == torch.float16 else 0.0))
    res.add(label, worst)


def wgrad_ref(xin, dz, N, wshape, pad):
    """fp64 weight gradient and its absolute-value twin over all N samples, in chunks"""
    ref = torch.zeros(wshape, dtype=F64, device=DEV)
    rab = torch.zeros(wshape, dtype=F64, device=DEV)
    per = dz(0, 1).numel() * 2
    for a, b in chunks(0, N, per):
        x = xin(a, b)
        d = dz(a, b)
        ref += torch.nn.grad.conv2d_weight(x, wshape, d, padding=pad)
        rab += torch.nn.grad.conv2d_weight(x.abs(), wshape, d.abs(), padding=pad)
    return ref, rab


def pool_argmax(y32):
    """PyTorch scan order (first maximum wins) on the fp32 values the kernel compares"""
    m, idx = F.max_pool2d(y32, 2, return_indices=True)
    return m, idx


def bn_bwd_parts(z, dp, a, b, mu, istd):
    """(y max, g at arg-max scattered to full resolution, z at arg-max, xhat) of one chunk; a, b, mu, istd broadcast [n, C, 1, 1]"""
    z = z.to(F64)
    y32 = (a * z + b).float()
    m, idx = pool_argmax(y32)
    g = torch.where(m > 0, dp.to(F64), torch.zeros_like(dp, dtype=F64))
    H, W = z.shape[-2:]
    g_full = F.max_unpool2d(g, idx, 2, output_size=(H, W))
    xhat = (z - mu) * istd
    return g_full, xhat, z


def per_sample(t, v_of):
    """per-(view, channel) vector t [views, C] -> [n, C, 1, 1] for the rows a..b"""
    return t[v_of].to(F64)[:, :, None, None]


# ---- checkers ---------------------------------------------------------------------------------------------------------
class Ctx:
    def __init__(self, rec, live):
        self.rec = rec
        self.live = live            # argument name -> data_ptr of the live tensor (the snapshots are copies)
        self.rerun = True           # conv_tc_wgrad: also run the other formulation of the 3x3 layers


def _conv_common(ctx, pre, post, out_key, bias_key, x_key, w_key):
    img = ctx.rec.image(ctx.live[w_key])
    x8 = pre[x_key]
    out = post[out_key]
    K, pad = img["K"], pre["pad"]
    w = conv_weight(img)
    bias = pre[bias_key].to(F64) if pre.get(bias_key) is not None else None
    out_w = out.shape[-1] if out.dim() == 4 else out.shape[-2]
    return img, x8, out, K, pad, w, bias, out_w


def check_conv_tc(ctx, pre, post):
    res = Result()
    img, x8, out, K, pad, w, bias, out_w = _conv_common(ctx, pre, post, "out", "bias", "x8", "wprep")
    N, npv = out.shape[0], pre["n_per_view"]
    xin = conv_input(x8, out_w, K, pad)
    tag = ("dgrad " if img["flip"] else "fwd ") + img["name"]
    stats = pre.get("stats")
    if stats is not None:
        delta = (post["stats"].to(F64) - stats.to(F64)).reshape(N // npv, -1, 2)
        conv_out_check(res, tag, xin, w, bias, pad, out, None, stats_delta=delta, npv=npv)
    else:
        geom = (w.shape[1], w.shape[0], x8.shape[-3] if x8.dim() == 4 else x8.shape[2], K, pad)
        views = N // npv
        samples = [v * npv + s for v in range(views) for s in boundary_samples(npv, views, geom)]
        conv_out_check(res, tag, xin, w, bias, pad, out, samples)
    return res


def check_conv_tc_pool(ctx, pre, post):
    res = Result()
    img, x8, e8, K, pad, w, bias, _ = _conv_common(ctx, pre, post, "pool_out", "bias", "x8", "wprep")
    out_w = e8.shape[-2] * 2
    N, npv = e8.shape[0], pre["n_per_view"]
    xin = conv_input(x8, out_w, K, pad)
    sgn = torch.where(pre["gamma"] < 0, -1.0, 1.0).to(F64).view(1, -1, 1, 1)
    z = post["z_out"]
    tag = "fwd " + img["name"]
    delta = (post["stats"].to(F64) - pre["stats"].to(F64)).reshape(N // npv, -1, 2)
    if z is not None:
        conv_out_check(res, tag, xin, w, bias, pad, z, None, stats_delta=delta, npv=npv)
        exact = True
        for a, b in chunks(0, N, z[0].numel()):
            want = F.max_pool2d(nchw(z[a:b]).to(F64) * sgn, 2) * sgn
            exact &= bool(torch.equal(nchw(e8[a:b]).to(F64), want))
        res.add(tag + ".extreme(z)", 0.0 if exact else math.inf)
        return res
    # no z stored: the extreme against the fp64 convolution, and the statistics over the whole batch
    wa, ba = w.abs(), (bias.abs() if bias is not None else None)
    s_ref, s_bnd = torch.zeros_like(delta), torch.zeros_like(delta)
    worst = 0.0
    per = e8[0].numel() * 4 * 4
    for v, (lo, hi) in enumerate(rows_of(N, npv)):
        for a, b in chunks(lo, hi, per):
            x = xin(a, b)
            ref = F.conv2d(x, w, bias, padding=pad)
            rab = F.conv2d(x.abs(), wa, ba, padding=pad)
            e_ref = F.max_pool2d(ref * sgn, 2) * sgn
            bound = F.max_pool2d(A_EXACT * rab + R_OUT[torch.float16] * ref.abs() + FP16_TINY, 2)
            err = (nchw(e8[a:b]).to(F64) - e_ref).abs()
            q = torch.where(err == 0, torch.zeros_like(err), err / bound)
            worst = worse(worst, math.inf if bool(torch.isnan(q).any()) else float(q.max()))
            s_ref[v, :, 0] += ref.sum(dim=(0, 2, 3))
            s_ref[v, :, 1] += (ref * ref).sum(dim=(0, 2, 3))
            s_bnd[v, :, 0] += A_EXACT * rab.sum(dim=(0, 2, 3)) + A_SUM * ref.abs().sum(dim=(0, 2, 3))
            s_bnd[v, :, 1] += 2 * A_EXACT * (ref.abs() * rab).sum(dim=(0, 2, 3)) + A_SUM * (ref * ref).sum(dim=(0, 2, 3))
    res.add(tag + ".extreme", worst)
    res.add(tag + ".stats", ratio(delta, s_ref, s_bnd, 1.0))
    return res


def bnstat_sums(p, dx, gamma, beta, npv):
    """{sum_{p>0} dx, sum_{p>0} dx (p - beta) / gamma} per (view, channel) and their bounds; p, dx NCHW (any float type)"""
    N, C = p.shape[:2]
    views = N // npv
    s = torch.zeros(views, C, 2, dtype=F64, device=DEV)
    bnd = torch.zeros_like(s)
    gam = gamma.to(F64).view(1, -1, 1, 1)
    ig = torch.where(gam != 0, 1.0 / gam, torch.zeros_like(gam))
    be = beta.to(F64).view(1, -1, 1, 1)
    for v, (lo, hi) in enumerate(rows_of(N, npv)):
        for a, b in chunks(lo, hi, p[0].numel() * 4):
            pv, g = p[a:b].to(F64), dx[a:b].to(F64)
            g = torch.where(pv > 0, g, torch.zeros_like(g))
            xh = (pv - be) * ig
            s[v, :, 0] += g.sum(dim=(0, 2, 3))
            s[v, :, 1] += (g * xh).sum(dim=(0, 2, 3))
            bnd[v, :, 0] += A_SUM * g.abs().sum(dim=(0, 2, 3))
            bnd[v, :, 1] += A_SUM * (g.abs() * ((pv.abs() + be.abs()) * ig.abs())).sum(dim=(0, 2, 3))
    return s, bnd


def check_conv_tc_dgrad_bnstat(ctx, pre, post):
    res = Result()
    img = ctx.rec.image(ctx.live["wprep_flip"])
    w = conv_weight(img)
    dz8, dx8, pad, npv = pre["dz8"], post["dx8"], pre["pad"], pre["n_per_view"]
    N = dz8.shape[0]
    geom = (dz8.shape[1] * 8, dx8.shape[1] * 8, dz8.shape[2], img["K"], pad)
    views = N // npv                        # launched per view-call: grid (G, views, NSPLIT), CTA g of view v from v*npv + npv*g/G
    samples = [v * npv + s for v in range(views) for s in boundary_samples(npv, views, geom)]
    conv_out_check(res, "dgrad " + img["name"], lambda a, b: nchw(dz8[a:b]).to(F64), w, None, pad, dx8, samples)
    s_ref, bnd = bnstat_sums(nchw(pre["p8"]), nchw(dx8), pre["gamma"], pre["beta"], npv)
    res.add("bnstat sums " + img["name"], ratio(post["sums"].to(F64) - pre["sums"].to(F64), s_ref, bnd, 1.0))
    return res


def _wgrad_operands(pre):
    x8, dz8, dw, pad = pre["x8"], pre["dz8"], pre["dw"], pre["pad"]
    if dw.shape[1] == 1:
        xin = lambda a, b: shift8_image(x8[a:b], pad).to(F64)
    else:
        xin = lambda a, b: nchw(x8[a:b]).to(F64)
    dz = lambda a, b: nchw(dz8[a:b]).to(F64)
    return xin, dz, x8.shape[0], tuple(dw.shape), pad


def check_conv_tc_wgrad(ctx, pre, post):
    res = Result()
    xin, dz, N, wshape, pad = _wgrad_operands(pre)
    ref, rab = wgrad_ref(xin, dz, N, wshape, pad)
    label = f"wgrad {ctx.rec.param_name(post['dw'])} N={N}"
    variant = ops.conv_tc_wgrad_variant()
    a_of = {1: A_WGRAD, 0: A_WGRAD_SHIFT_ROW if wshape[-1] == 3 else A_WGRAD}
    res.add(f"{label} variant={variant}", ratio(post["dw"], ref, rab, a_of[variant]))
    if ctx.rerun and wshape[-1] == 3:
        # the other weight-gradient formulation of the 3x3 layers on the same recorded operands
        other = 1 - variant
        old = ops.conv_tc_wgrad_variant(other)
        try:
            Cout, Cin, K, _ = wshape
            H, W = pre["x8"].shape[-3], pre["x8"].shape[-2] - (pad if Cin == 1 else 0)
            work = torch.empty(ops.conv_tc_wgrad_work_floats(N, Cin, Cout, H, W, K, pad), device=DEV)
            dw2 = torch.full(wshape, float("nan"), device=DEV)
            ctx.rec.raw["conv_tc_wgrad"](pre["x8"], pre["dz8"], dw2, work, pad)
            torch.cuda.synchronize()
        finally:
            ops.conv_tc_wgrad_variant(old)
        res.add(f"{label} variant={other}", ratio(dw2, ref, rab, a_of[other]))
        del work, dw2
    return res


def bn_apply_ref(z8, dp, scale, shift, mean, invstd, sums, npv, a_, b_):
    """fp64 dz of bn_relu_pool8_bwd_apply for rows a_..b_ (and its absolute-value twin)"""
    H, W = z8.shape[2], z8.shape[3]
    v_of = torch.arange(a_, b_, device=DEV) // npv
    A, Bs, MU, IS = (per_sample(t, v_of) for t in (scale, shift, mean, invstd))
    cnt = float(npv * H * W)
    K1 = per_sample(sums[..., 0] / cnt, v_of)
    K2 = per_sample(sums[..., 1] / cnt, v_of)
    g_full, xhat, z = bn_bwd_parts(nchw(z8[a_:b_]), nchw(dp[a_:b_]) if dp.dim() == 5 else dp[a_:b_], A, Bs, MU, IS)
    dz = A * (g_full - K1 - xhat * K2)
    rab = A.abs() * (g_full.abs() + K1.abs() + K2.abs() * (z.abs() * IS.abs() + MU.abs() * IS.abs()))
    return dz, rab


def check_conv_tc_wgrad_l0_fused(ctx, pre, post):
    res = Result()
    xs8, z8, dp8, dw, pad, npv = pre["xs8"], pre["z8"], pre["dp8"], pre["dw"], pre["pad"], pre["n_per_view"]
    N, P, H, W, _ = z8.shape
    # the reference dz: b200_bn_relu_pool8_bwd_apply on the recorded operands (checked on its own against fp64 below)
    dz8 = torch.empty(z8.shape, dtype=torch.bfloat16, device=DEV)
    ctx.rec.raw["bn_relu_pool8_bwd_apply"](z8, dp8, pre["scale"], pre["shift"], pre["mean"], pre["invstd"], pre["sums"], dz8, npv)
    torch.cuda.synchronize()
    ref, rab = wgrad_ref(lambda a, b: quad8_image(xs8[a:b], W, pad).to(F64), lambda a, b: nchw(dz8[a:b]).to(F64), N, tuple(dw.shape), pad)
    name = ctx.rec.param_name(post["dw"])
    res.add(f"wgrad_l0_fused {name} N={N}", ratio(post["dw"], ref, rab, A_WGRAD))
    worst, db_ref, db_bnd = 0.0, torch.zeros(dw.shape[0], dtype=F64, device=DEV), torch.zeros(dw.shape[0], dtype=F64, device=DEV)
    sums = pre["sums"].to(F64)
    for a, b in chunks(0, N, z8[0].numel() * 6):
        dz, rb = bn_apply_ref(z8, dp8, pre["scale"], pre["shift"], pre["mean"], pre["invstd"], sums, npv, a, b)
        worst = worse(worst, ratio(nchw(dz8[a:b]), dz, rb, A_ELEM, R_OUT[torch.bfloat16]))
        db_ref += dz.sum(dim=(0, 2, 3))
        db_bnd += A_SUM * rb.sum(dim=(0, 2, 3))
    res.add("bwd_apply (fused reference dz)", worst)
    if pre.get("dbsum") is not None:
        C = dw.shape[0]                       # the bias-sum scratch may be wider than this layer
        res.add(f"wgrad_l0_fused {name} dbsum", ratio(post["dbsum"][:C].to(F64) - pre["dbsum"][:C].to(F64), db_ref, db_bnd, 1.0))
    del dz8
    return res


def check_bn_relu_pool8_fwd(ctx, pre, post):
    res = Result()
    z8, out, npv = pre["z8"], post["out"], pre["n_per_view"]
    N = z8.shape[0]
    worst = 0.0
    for a, b in chunks(0, N, z8[0].numel() * 4):
        v_of = torch.arange(a, b, device=DEV) // npv
        A, Bs = per_sample(pre["scale"], v_of), per_sample(pre["shift"], v_of)
        z = nchw(z8[a:b]).to(F64)
        ref = F.max_pool2d(A * z + Bs, 2).clamp_min(0)
        rab = F.max_pool2d(A.abs() * z.abs() + Bs.abs(), 2)
        worst = worse(worst, ratio(nchw(out[a:b]), ref, rab, A_ELEM, R_OUT[out.dtype]))
    res.add(f"N={N} C={z8.shape[1] * 8} {tuple(z8.shape[2:4])}", worst)
    return res


def check_bn_relu_apply8(ctx, pre, post):
    res = Result()
    e8, out, npv = pre["e8"], post["out"], pre["n_per_view"]
    N = e8.shape[0]
    worst = 0.0
    for a, b in chunks(0, N, e8[0].numel() * 4):
        v_of = torch.arange(a, b, device=DEV) // npv
        A, Bs = per_sample(pre["scale"], v_of), per_sample(pre["shift"], v_of)
        e = nchw(e8[a:b]).to(F64)
        worst = worse(worst, ratio(nchw(out[a:b]), (A * e + Bs).clamp_min(0), A.abs() * e.abs() + Bs.abs(), A_ELEM, R_OUT[out.dtype]))
    res.add(f"N={N} C={e8.shape[1] * 8}", worst)
    return res


def check_bn_relu_pool8_bwd_reduce(ctx, pre, post):
    res = Result()
    z8, dp, npv = pre["z8"], pre["dp"], pre["n_per_view"]
    N, C = z8.shape[0], z8.shape[1] * 8
    s = torch.zeros(N // npv, C, 2, dtype=F64, device=DEV)
    bnd = torch.zeros_like(s)
    for v, (lo, hi) in enumerate(rows_of(N, npv)):
        for a, b in chunks(lo, hi, z8[0].numel() * 6):
            v_of = torch.arange(a, b, device=DEV) // npv
            A, Bs, MU, IS = (per_sample(pre[k], v_of) for k in ("scale", "shift", "mean", "invstd"))
            g, xhat, z = bn_bwd_parts(nchw(z8[a:b]), nchw(dp[a:b]) if dp.dim() == 5 else dp[a:b], A, Bs, MU, IS)
            s[v, :, 0] += g.sum(dim=(0, 2, 3))
            s[v, :, 1] += (g * xhat).sum(dim=(0, 2, 3))
            bnd[v, :, 0] += A_SUM * g.abs().sum(dim=(0, 2, 3))
            bnd[v, :, 1] += A_SUM * (g.abs() * (z.abs() + MU.abs()) * IS.abs()).sum(dim=(0, 2, 3))
    res.add(f"N={N} C={C}", ratio(post["sums"].to(F64) - pre["sums"].to(F64), s, bnd, 1.0))
    return res


def check_bn_relu_pool8_bwd_apply(ctx, pre, post):
    res = Result()
    z8, dz8, npv = pre["z8"], post["dz8"], pre["n_per_view"]
    N, C = z8.shape[0], z8.shape[1] * 8
    sums = pre["sums"].to(F64)
    worst = 0.0
    db_ref = torch.zeros(C, dtype=F64, device=DEV)
    db_bnd = torch.zeros_like(db_ref)
    for a, b in chunks(0, N, z8[0].numel() * 6):
        dz, rb = bn_apply_ref(z8, pre["dp"], pre["scale"], pre["shift"], pre["mean"], pre["invstd"], sums, npv, a, b)
        worst = worse(worst, ratio(nchw(dz8[a:b]), dz, rb, A_ELEM, R_OUT[torch.bfloat16]))
        db_ref += dz.sum(dim=(0, 2, 3))
        db_bnd += A_SUM * rb.sum(dim=(0, 2, 3))
    res.add(f"dz N={N} C={C}", worst)
    if pre.get("dbsum") is not None:
        res.add(f"dbsum N={N} C={C}", ratio(post["dbsum"][:C].to(F64) - pre["dbsum"][:C].to(F64), db_ref, db_bnd, 1.0))
    return res


def check_bn_pool8_bwd_reduce_p(ctx, pre, post):
    res = Result()
    p, dp = nchw(pre["p"]), nchw(pre["dp"])
    s, bnd = bnstat_sums(p, dp, pre["gamma"], pre["beta"], pre["n_per_view"])
    res.add(f"N={p.shape[0]} C={p.shape[1]}", ratio(post["sums"].to(F64) - pre["sums"].to(F64), s, bnd, 1.0))
    return res


def check_pack_act8(ctx, pre, post):
    res = Result()
    x = pre["x"]
    ok = all(torch.equal(post["out"][a:b], act8(x[a:b].to(torch.bfloat16))) for a, b in chunks(0, x.shape[0], x[0].numel()))
    res.add(f"N={x.shape[0]}", 0.0 if ok else math.inf)
    return res


def check_pack_quad8(ctx, pre, post):
    res = Result()
    x, out, pad = pre["x"], post["out"], pre["pad"]
    x = x.reshape(x.shape[0], x.shape[-2], x.shape[-1])
    ok = all(torch.equal(out[a:b], quad8_of(x[a:b], pad)) for a, b in chunks(0, x.shape[0], out[0].numel()))
    res.add(f"N={x.shape[0]}", 0.0 if ok else math.inf)
    return res


def check_pack_shift8(ctx, pre, post):
    res = Result()
    x, out, pad = pre["x"], post["out"], pre["pad"]
    x = x.reshape(x.shape[0], x.shape[-2], x.shape[-1])
    ok = all(torch.equal(out[a:b], shift8_of(x[a:b], pad)) for a, b in chunks(0, x.shape[0], out[0].numel()))
    res.add(f"N={x.shape[0]}", 0.0 if ok else math.inf)
    return res


def check_bn_finalize(ctx, pre, post):
    res = Result()
    if not pre.get("train", True):
        res.add("eval", 0.0)
        return res
    st = pre["stats"].to(F64).view(pre["n_views"], -1, 2)
    count = float(pre["count"])
    mom, eps = float(pre.get("momentum", 0.1)), float(pre.get("eps", 1e-5))
    g, b = pre["gamma"].to(F64), pre["beta"].to(F64)
    m = st[..., 0] / count
    var = (st[..., 1] / count - m * m).clamp_min(0)
    istd = 1.0 / torch.sqrt(var + eps)
    res.add("mean", ratio(post["mean"], m, m.abs(), A_ELEM))
    res.add("invstd", ratio(post["invstd"], istd, istd, A_ELEM))
    res.add("scale", ratio(post["scale"], g * istd, (g * istd).abs(), A_ELEM))
    res.add("shift", ratio(post["shift"], b - m * g * istd, b.abs() + (m * g * istd).abs(), A_ELEM))
    rm, rv = pre["running_mean"].to(F64), pre["running_var"].to(F64)
    rm_abs, rv_abs = rm.abs(), rv.abs()
    unb = var * (count / (count - 1.0 if count > 1 else 1.0))
    for v in range(pre["n_views"]):
        rm = (1 - mom) * rm + mom * m[v]
        rv = (1 - mom) * rv + mom * unb[v]
        rm_abs = (1 - mom) * rm_abs + mom * m[v].abs()
        rv_abs = (1 - mom) * rv_abs + mom * unb[v].abs()
    res.add("running_mean", ratio(post["running_mean"], rm, rm_abs, A_ELEM))
    res.add("running_var", ratio(post["running_var"], rv, rv_abs, A_ELEM))
    return res


def _act(ref, rab, act, mask, drop_p):
    if act >= 1:
        ref = ref.clamp_min(0)
    if act == 2 and mask is not None:
        keep = mask.to(F64) / (1.0 - drop_p)
        ref, rab = ref * keep, rab * keep
    return ref, rab


def check_linear_fwd(ctx, pre, post):
    res = Result()
    x, w, bias, y = pre["x"].to(F64), pre["w"].to(F64), pre["bias"], post["y"]
    ref = x @ w.t()
    rab = x.abs() @ w.abs().t()
    if bias is not None:
        ref, rab = ref + bias.to(F64), rab + bias.to(F64).abs()
    ref, rab = _act(ref, rab, pre.get("act", 0), pre.get("mask"), pre.get("drop_p", 0.0))
    a = A_TF32 if pre.get("tc") else A_EXACT
    res.add(f"{ctx.rec.param_name(pre['w'], ctx.live['w'])} M={x.shape[0]}", ratio(y, ref, rab, a))
    return res


def check_linear_bwd_data(ctx, pre, post):
    res = Result()
    dy, w = pre["dy"].to(F64), pre["w"].to(F64)
    a = A_TF32 if pre.get("tc") else A_EXACT
    res.add(f"{ctx.rec.param_name(pre['w'], ctx.live['w'])} M={dy.shape[0]}", ratio(post["dx"], dy @ w, dy.abs() @ w.abs(), a))
    return res


def check_linear_bwd_weight(ctx, pre, post):
    res = Result()
    dy, x = pre["dy"].to(F64), pre["x"].to(F64)
    acc = bool(pre.get("accumulate", False))
    ref, rab = dy.t() @ x, dy.abs().t() @ x.abs()
    base = pre["dw"].to(F64) if acc else 0.0
    a = A_TF32 if pre.get("tc") else A_EXACT
    label = f"{ctx.rec.param_name(post['dw'])} M={dy.shape[0]}"
    res.add(label + " dW", ratio(post["dw"].to(F64) - base, ref, rab + (pre["dw"].to(F64).abs() if acc else 0.0), a))
    if pre.get("db") is not None:
        dbase = pre["db"].to(F64) if acc else 0.0
        res.add(label + " db", ratio(post["db"].to(F64) - dbase, dy.sum(0), dy.abs().sum(0) + (pre["db"].to(F64).abs() if acc else 0.0), A_SUM))
    return res


def dino_reference(s, t, center, tau_s, tau_t, gscale, variant, t_colmean):
    Vs, B, D = s.shape
    Vt = t.shape[0]
    sd = s.to(F64).requires_grad_(True)
    nrm = sd.norm(dim=-1, keepdim=True).clamp_min(1e-12)
    sh = sd / nrm
    logp = torch.log_softmax(sh / tau_s, dim=-1)
    tn = t.to(F64) - center.to(F64).view(1, 1, D)
    tn = tn / tn.norm(dim=-1, keepdim=True).clamp_min(1e-12)
    if variant == 1:
        tn = tn - t_colmean.to(F64).view(Vt, 1, D)
    pt = torch.softmax(tn / tau_t, dim=-1)
    pbar = pt.sum(0)
    c = 1.0 / (Vs * Vt * B)
    loss = -(pbar.unsqueeze(0) * logp).sum() * c
    (loss * gscale).backward()
    with torch.no_grad():
        # absolute-value twin of the gradient: (Vt e^q + pbar) c g / tau_s through the normalisation's Jacobian
        zabs = (Vt * logp.exp() + pbar.unsqueeze(0)) * c * abs(gscale) / tau_s
        dot = (sh.abs() * zabs).sum(-1, keepdim=True)
        gabs = (zabs + sh.abs() * dot) / nrm
        labs = (pbar.unsqueeze(0) * logp.abs()).sum() * c
    return float(loss), sd.grad, gabs, float(labs), t.to(F64).sum(dim=(0, 1)), t.to(F64).abs().sum(dim=(0, 1))


def check_dino_loss_fwd_bwd(ctx, pre, post):
    res = Result()
    loss, grad, gabs, labs, colsum, colabs = dino_reference(pre["s"], pre["t"], pre["center"], pre["tau_s"], pre["tau_t"],
                                                            pre.get("grad_scale", 1.0), pre.get("variant", 0), pre.get("t_colmean"))
    res.add("grad_s", ratio(post["grad_s"], grad, gabs, A_ELEM * 16))
    lsum = post["part_loss"].to(F64).sum().view(1)
    res.add("loss (sum of parts)", ratio(lsum, torch.tensor([loss], dtype=F64, device=DEV), torch.tensor([labs], dtype=F64, device=DEV), A_SUM))
    res.add("teacher colsum (sum of parts)", ratio(post["part_colsum"].to(F64).sum(0), colsum, colabs, A_SUM))
    return res


def check_teacher_norm_colmean(ctx, pre, post):
    res = Result()
    t, c = pre["t"].to(F64), pre["center"].to(F64).view(1, 1, -1)
    tn = t - c
    nrm = tn.norm(dim=-1, keepdim=True).clamp_min(1e-12)
    ref = (tn / nrm).mean(1)
    rab = ((t.abs() + c.abs()) / nrm).mean(1)
    res.add(f"B={t.shape[1]}", ratio(post["out"], ref, rab, A_SUM))
    return res


def check_center_update(ctx, pre, post):
    res = Result()
    parts = pre["part_colsum"].to(F64)
    n_parts = parts.shape[0]
    a = (n_parts + 4) * 2.0 ** -24                   # fixed-order fp32 sum of n_parts terms, then two products and a sum
    colsum, colabs = parts.sum(0), parts.abs().sum(0)
    if pre.get("colsum_out") is not None:
        res.add("colsum_out", ratio(post["colsum_out"], colsum, colabs, a))
    if pre.get("center") is not None:
        mc, n = float(pre["m_c"]), float(pre["n_rows"])
        c0 = pre["center"].to(F64).view(-1)
        ref = mc * c0 + (1 - mc) * colsum / n
        rab = mc * c0.abs() + (1 - mc) * colabs / n
        res.add("center", ratio(post["center"].view(-1), ref, rab, a))
    if pre.get("loss_out") is not None and pre.get("part_loss") is not None:
        pl = pre["part_loss"].to(F64)
        res.add("loss", ratio(post["loss_out"].view(-1)[:1], pl.sum().view(1), pl.abs().sum().view(1), (pl.numel() + 2) * 2.0 ** -24))
    return res


def check_center_apply(ctx, pre, post):
    res = Result()
    mc, n = float(pre["m_c"]), float(pre["n_rows"])
    c0, cs = pre["center"].to(F64).view(-1), pre["colsum"].to(F64).view(-1)
    res.add("center", ratio(post["center"].view(-1), mc * c0 + (1 - mc) * cs / n, mc * c0.abs() + (1 - mc) * cs.abs() / n, 4 * 2.0 ** -24))
    return res


def _normalised_jacobian_abs(xd, ghat_abs):
    """|d loss / d x| twin for x -> x / |x|: (|g| + |xhat| * sum |xhat| |g|) / |x|"""
    nrm = xd.norm(dim=-1, keepdim=True).clamp_min(1e-12)
    xh = (xd / nrm).abs()
    return (ghat_abs + xh * (xh * ghat_abs).sum(-1, keepdim=True)) / nrm


def check_infonce_fwd_bwd(ctx, pre, post):
    res = Result()
    a, b = pre["a"].to(F64).requires_grad_(True), pre["b"].to(F64).requires_grad_(True)
    tau, gs = float(pre.get("temperature", 0.07)), float(pre.get("grad_scale", 1.0))
    B = a.shape[0]
    ah, bh = F.normalize(a, dim=1), F.normalize(b, dim=1)
    sim = ah @ bh.t() / tau
    lab = torch.arange(B, device=DEV)
    loss = 0.5 * (F.cross_entropy(sim, lab) + F.cross_entropy(sim.t(), lab))
    (loss * gs).backward()
    with torch.no_grad():
        P = torch.softmax(sim, 1) + torch.softmax(sim, 0) + 2 * torch.eye(B, dtype=F64, device=DEV)
        ga_hat = (P @ bh.abs()) * abs(gs) / (2 * B * tau)
        gb_hat = (P.t() @ ah.abs()) * abs(gs) / (2 * B * tau)
        res.add(f"grad_a B={B}", ratio(post["grad_a"], a.grad, _normalised_jacobian_abs(a, ga_hat), A_BF16_GEMM))
        res.add(f"grad_b B={B}", ratio(post["grad_b"], b.grad, _normalised_jacobian_abs(b, gb_hat), A_BF16_GEMM))
        labs = float(loss) + 2.0 / tau               # log-sum-exp terms are bounded by |sim| <= 1 / tau
        res.add(f"loss B={B}", ratio(post["loss_out"].view(-1)[:1], loss.detach().view(1), torch.tensor([labs], dtype=F64, device=DEV), A_EXACT))
    return res


def check_ntxent_fwd_bwd(ctx, pre, post):
    res = Result()
    reps = pre["reps"].to(F64).requires_grad_(True)
    tau, gs = float(pre.get("temperature", 0.07)), float(pre.get("grad_scale", 1.0))
    N = reps.shape[0]
    B = N // 2
    rh = F.normalize(reps, dim=1)
    sim = rh @ rh.t() / tau
    sim = sim.masked_fill(torch.eye(N, dtype=torch.bool, device=DEV), float("-inf"))
    target = (torch.arange(N, device=DEV) + B) % N
    loss = F.cross_entropy(sim, target)
    (loss * gs).backward()
    with torch.no_grad():
        P = torch.softmax(sim, 1)
        Pt = P + P.t()
        Pt[torch.arange(N), target] += 1.0
        Pt[target, torch.arange(N)] += 1.0
        g_hat = (Pt @ rh.abs()) * abs(gs) / (N * tau)
        res.add(f"grad N={N}", ratio(post["grad"], reps.grad, _normalised_jacobian_abs(reps, g_hat), A_BF16_GEMM))
        labs = float(loss) + 2.0 / tau
        res.add(f"loss N={N}", ratio(post["loss_out"].view(-1)[:1], loss.detach().view(1), torch.tensor([labs], dtype=F64, device=DEV), A_EXACT))
    return res


def check_colstats(ctx, pre, post):
    res = Result()
    h = pre["h"].to(F64)
    ref = torch.stack([h.sum(0), (h * h).sum(0)], -1)
    rab = torch.stack([h.abs().sum(0), (h * h).sum(0)], -1)
    res.add(f"M={h.shape[0]}", ratio(post["stats"].to(F64).view(-1, 2) - pre["stats"].to(F64).view(-1, 2), ref, rab, 2.0 ** -40))
    return res


def check_bias_grad_finalize(ctx, pre, post):
    res = Result()
    db = post["db"]
    res.add("db", 0.0 if torch.equal(db, pre["dbsum"][:db.numel()].float().view_as(db)) else math.inf)
    return res


def check_bn_param_grads(ctx, pre, post):
    res = Result()
    s = pre["sums"].to(F64).view(pre["n_views"], -1, 2).sum(0)
    acc = bool(pre.get("accumulate", False))
    for k, j in (("dgamma", 1), ("dbeta", 0)):
        base = pre[k].to(F64) if acc else 0.0
        res.add(k, ratio(post[k].to(F64), base + s[:, j], (pre[k].to(F64).abs() if acc else 0.0) + s[:, j].abs(), 2.0 ** -23))
    return res


def check_avgpool_fwd(ctx, pre, post):
    res = Result()
    x = pre["x"].to(F64)
    x = x.reshape(x.shape[0], x.shape[1], -1)
    res.add(f"N={x.shape[0]}", ratio(post["out"].reshape(x.shape[:2]), x.mean(-1), x.abs().mean(-1), x.shape[-1] * 2.0 ** -23))
    return res


def check_avgpool_bwd(ctx, pre, post):
    res = Result()
    dx = post["dx"]
    hw = dx[0, 0].numel()
    d = pre["dout"].to(F64).reshape(dx.shape[0], dx.shape[1], 1) / hw
    res.add(f"N={dx.shape[0]}", ratio(dx.reshape(dx.shape[0], dx.shape[1], -1), d.expand(-1, -1, hw), d.abs().expand(-1, -1, hw), 2.0 ** -23))
    return res


def check_add2d(ctx, pre, post):
    res = Result()
    res.add("dst", 0.0 if torch.equal(post["dst"], pre["dst"] + pre["src"]) else math.inf)
    return res


CHECKERS = {name[len("check_"):]: fn for name, fn in list(globals().items()) if name.startswith("check_") and callable(fn)}


# ---- the recorder -----------------------------------------------------------------------------------------------------
def wrapped_ops():
    """the kernel wrappers ops._wrap installed: name -> function"""
    return {n: f for n, f in vars(ops).items() if callable(f) and getattr(f, "__qualname__", "").startswith("_wrap.")}


class Recorder:
    def __init__(self, eng, monkeypatch, stash=()):
        self.eng = eng
        self.params = {}
        for role, arena in (("student", getattr(eng, "S", {})), ("teacher", getattr(eng, "T", {})), ("grad", getattr(eng, "G", {}))):
            for name, t in arena.items():
                self.params.setdefault(t.data_ptr(), f"{role}:{name}")
        self.images = {}
        self.raw = wrapped_ops()
        self.calls = collections.Counter()
        self.checked = collections.Counter()
        self.worst = {}
        self.failures = []
        self.stash_for = set(stash)
        self.stash = collections.defaultdict(list)
        for name, fn in self.raw.items():
            monkeypatch.setattr(ops, name, self._wrap(name, fn))

    def param_name(self, t, ptr=None):
        return self.params.get(ptr if ptr is not None else t.data_ptr(), f"<{tuple(t.shape)}>")

    def image(self, ptr):
        img = self.images.get(ptr)
        assert img is not None, "conv_tc launch reads a weight image that no prep call of this step wrote"
        return img

    def _record_prep(self, rows):
        for wp, out, cin, cout, k, flip in rows:
            name = self.params.get(wp)
            assert name is not None, f"prepared weight at {wp:#x} is none of the engine's named parameters"
            t = next(v for arena in (getattr(self.eng, "S", {}), getattr(self.eng, "T", {})) for v in arena.values() if v.data_ptr() == wp)
            self.images[out] = {"name": name, "w": t.detach().clone(), "K": k, "flip": bool(flip), "cin": cin, "cout": cout}

    def _wrap(self, name, fn):
        raw_sig = inspect.signature(raw_function(fn))

        def call(*args, **kwargs):
            self.calls[name] += 1
            bound = raw_sig.bind(*args, **kwargs)
            bound.apply_defaults()
            torch.cuda.synchronize()
            pre = {k: (v.detach().clone() if isinstance(v, torch.Tensor) and k != "work" else v) for k, v in bound.arguments.items()}
            for k in pure_outputs(name, bound.arguments):      # elements the launch does not write then fail their check
                bound.arguments[k].fill_(float("nan"))
            live = {k: v.data_ptr() for k, v in bound.arguments.items() if isinstance(v, torch.Tensor)}
            out = fn(*args, **kwargs)
            torch.cuda.synchronize()
            if name == "conv_tc_prep_weights_multi":
                self._record_prep(pre["desc"].tolist())
            elif name == "conv_tc_prep_weights":
                w = bound.arguments["w"]
                Co, Ci, K, _ = w.shape
                flip = bool(bound.arguments["flip"])
                self._record_prep([[w.data_ptr(), bound.arguments["wprep"].data_ptr(), Co if flip else Ci, Ci if flip else Co, K, int(flip)]])
            checker = CHECKERS.get(name)
            if checker is not None:
                ctx = Ctx(self, live)
                post = dict(bound.arguments)
                res = checker(ctx, pre, post)
                self.checked[name] += 1
                for label, q in res.items:
                    key = name
                    if not q <= self.worst.get(key, (-1.0, ""))[0]:
                        self.worst[key] = (q, label)
                    if not q <= 1.0:
                        self.failures.append((name, label, q))
                if name in self.stash_for and self._want_stash(name, pre, post):
                    self.stash[name].append((pre, {k: (v.detach().clone() if isinstance(v, torch.Tensor) else v) for k, v in post.items()}, live))
            del pre
            return out

        return call

    def _want_stash(self, name, pre, post):
        if self.stash[name] and name != "linear_bwd_weight":
            return False
        if name == "conv_tc":
            return post["out"].dim() == 5 and pre.get("stats") is not None and pre["x8"].dim() == 5
        if name == "conv_tc_wgrad":
            return pre["x8"].shape[0] == 6144
        if name == "linear_bwd_weight":
            dy, x = pre["dy"], pre["x"]
            return pre.get("tc") and not pre.get("accumulate") and linear_dw_splits(dy.shape[0], dy.shape[1], x.shape[1])[0] >= 3
        return False

    def report(self, title):
        print(f"\n== {title}: {sum(self.checked.values())} launches checked of {sum(self.calls.values())} op calls")
        for name in sorted(self.worst):
            q, label = self.worst[name]
            print(f"   {name:28s} {self.checked[name]:4d} launches   worst error / bound {q:8.4f}   ({label})")
        missing = sorted(n for n in self.calls if n not in CHECKERS and n not in UNCHECKED)
        print(f"   unchecked with reason: {sorted(n for n in self.calls if n in UNCHECKED)}")
        print(f"   unchecked without reason: {missing}")
        return missing


# outputs each checked op overwrites entirely (never reads): NaN before the launch, so that an element it skips cannot pass
# with a value left from an earlier step.  Accumulators (statistics, sums, running buffers, accumulate=True) keep their values.
PURE_OUTPUTS = {"conv_tc": ("out",), "conv_tc_pool": ("z_out", "pool_out"), "conv_tc_dgrad_bnstat": ("dx8",), "conv_tc_wgrad": ("dw",),
                "conv_tc_wgrad_l0_fused": ("dw",), "bn_relu_pool8_fwd": ("out",), "bn_relu_apply8": ("out",),
                "bn_relu_pool8_bwd_apply": ("dz8",), "pack_act8": ("out",), "pack_quad8": ("out",), "pack_shift8": ("out",),
                "bn_finalize": ("scale", "shift", "mean", "invstd"), "linear_fwd": ("y",), "linear_bwd_data": ("dx",),
                "linear_bwd_weight": ("dw", "db"), "dino_loss_fwd_bwd": ("grad_s", "part_loss", "part_colsum"),
                "teacher_norm_colmean": ("out",), "center_update": ("loss_out", "colsum_out"), "infonce_fwd_bwd": ("grad_a", "grad_b", "loss_out"),
                "ntxent_fwd_bwd": ("grad", "loss_out"), "bias_grad_finalize": ("db",), "bn_param_grads": ("dgamma", "dbeta"),
                "avgpool_fwd": ("out",), "avgpool_bwd": ("dx",)}
ACCUMULATE_FLAG = {"linear_bwd_weight", "bn_param_grads"}      # their outputs are accumulators when accumulate=True


def pure_outputs(name, args):
    if name in ACCUMULATE_FLAG and args.get("accumulate"):
        return ()
    return tuple(k for k in PURE_OUTPUTS.get(name, ()) if isinstance(args.get(k), torch.Tensor))


def raw_function(wrapped):
    """the function ops._wrap wrapped (the one function in its closure): its signature names the call's arguments"""
    return next(c.cell_contents for c in wrapped.__closure__ if inspect.isfunction(c.cell_contents))


def linear_dw_splits(M, N, K):
    """(partials, rows per partial) of the tensor-core linear weight gradient (gemm_tc_splits(N, K, M) in gemm_tc.cu)"""
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    tiles = ((N + 127) // 128) * ((K + 127) // 128)
    splits = (sms + tiles - 1) // tiles
    splits = max(1, min(splits, (M + 127) // 128))
    kps = ((M + splits - 1) // splits + 31) // 32 * 32
    return (M + kps - 1) // kps, kps


# ---- the runs ---------------------------------------------------------------------------------------------------------
def _dino_inputs(eng, B):
    img, aud = views_to_vb(*synth_views(B, seed=600 + B))
    masks = make_masks(seed=601 + B, V=eng.V, Vg=eng.Vg, B=B, E=eng.E, hidden=512)
    x_img = img[:, :, 0].to(DEV).contiguous() if eng.img_layers else None
    x_aud = aud[:, :, 0].to(DEV).contiguous() if eng.aud_layers else None
    masks = {k: v.to(torch.uint8).to(DEV) for k, v in masks.items()}
    kw = {}
    if eng.mode != "default":
        from oracle.fixtures import synth_raw
        image, audio, labels = synth_raw(B, seed=602 + B)
        kw = {"raw": (image[:, 0].to(DEV).contiguous(), audio[:, 0].to(DEV).contiguous()), "labels": labels.to(DEV)}
    if not eng.multi:
        masks = {"student_head": masks["student_head"]}
    return (lambda: eng.forward_backward(x_img, x_aud, masks=masks, **kw))


def _contrastive_inputs(eng, kind, B):
    img1, spec1, img2, spec2 = (t[:, 0].to(DEV).contiguous() for t in contrastive_batch(B, 0))
    if kind == "infonce":
        return lambda: eng.forward_backward((img1, spec1))
    return lambda: eng.forward_backward((img1, spec1, img2, spec2), mode=2)        # image and spectrogram branch


RUNS = [("multi_central", "default", 1024, {}), ("multi_central", "default", 1024, {"fused_bnstat": True}),
        ("multi_central", "infonce", 8192, {}), ("multi_simple", "default", 1024, {}), ("image_simple", "default", 2048, {}),
        ("contrastive_infonce", None, 8192, {}), ("contrastive_simclr", None, 2048, {})]

# the kernels each run exists for: an engine change that stops launching one fails the run instead of passing unchecked
_STACK = {"pack_quad8", "conv_tc", "conv_tc_wgrad", "conv_tc_wgrad_l0_fused", "bn_finalize", "bn_relu_pool8_fwd", "bn_relu_pool8_bwd_apply",
          "bn_pool8_bwd_reduce_p", "linear_fwd", "linear_bwd_data", "linear_bwd_weight"}
_DINO = _STACK | {"dino_loss_fwd_bwd", "center_update"}
_POOLED = {"conv_tc_pool", "bn_relu_apply8"}
EXPECTED = {"multi_central-default-B1024": _DINO | _POOLED,
            "multi_central-default-B1024-fused_bnstat": _DINO | _POOLED | {"conv_tc_dgrad_bnstat"},
            "multi_central-infonce-B8192": _DINO | _POOLED | {"infonce_fwd_bwd"},
            "multi_simple-default-B1024": _DINO | {"avgpool_fwd", "avgpool_bwd"},
            "image_simple-default-B2048": _DINO | _POOLED | {"teacher_norm_colmean", "avgpool_fwd", "avgpool_bwd"},
            "contrastive_infonce-None-B8192": _STACK | {"infonce_fwd_bwd", "avgpool_fwd", "avgpool_bwd"},
            "contrastive_simclr-None-B2048": _STACK | {"ntxent_fwd_bwd", "avgpool_fwd", "avgpool_bwd"}}


def _engine(kind, mode, opts):
    if kind.startswith("contrastive_"):
        from multimodal_ssl_avmnist_b200.contrastive import ContrastiveStepEngine
        return ContrastiveStepEngine(kind=kind.split("_", 1)[1], device=DEV, precision="bf16", seed=3)
    from multimodal_ssl_avmnist_b200.engine import DinoStepEngine
    eng = DinoStepEngine(kind=kind, mode=mode, device=DEV, precision="bf16", seed=3, **opts)
    st = R.CentralDinoState(seed=31, mode=mode) if kind == "multi_central" else None
    if st is not None:       # the oracle's initialisation (as test_scale_gpu): trained-like BatchNorm / head parameters
        eng.load_named(student=st.student, teacher=st.teacher, student_head=st.student_head, teacher_head=st.teacher_head,
                       aux_image=st.aux.get("image"), aux_audio=st.aux.get("audio"))
    return eng


def _run_id(run):
    kind, mode, B, opts = run
    return f"{kind}-{mode}-B{B}" + ("-fused_bnstat" if opts.get("fused_bnstat") else "")


@pytest.mark.parametrize("run", RUNS, ids=_run_id)
def test_every_launch_of_the_step_against_float64(run, monkeypatch):
    kind, mode, B, opts = run
    t0 = time.time()
    torch.cuda.empty_cache()
    base = torch.cuda.memory_allocated()
    torch.cuda.reset_peak_memory_stats()
    eng = _engine(kind, mode, opts)
    step = _contrastive_inputs(eng, kind.split("_", 1)[1], B) if kind.startswith("contrastive_") else _dino_inputs(eng, B)
    # one plain step first: the engine's own allocations (workspace, scratch) and its peak memory without the recorder
    step()
    torch.cuda.synchronize()
    engine_peak = torch.cuda.max_memory_allocated() - base
    torch.cuda.reset_peak_memory_stats()
    rec = Recorder(eng, monkeypatch)
    step()
    torch.cuda.synchronize()
    monkeypatch.undo()
    rec_peak = torch.cuda.max_memory_allocated() - base
    missing = rec.report(_run_id(run))
    print(f"   memory: engine peak {engine_peak / 2**30:.1f} GiB, with the recorder {rec_peak / 2**30:.1f} GiB "
          f"(+{(rec_peak - engine_peak) / 2**30:.1f} GiB); {time.time() - t0:.0f} s")
    assert not missing, f"ops without a checker or an UNCHECKED reason: {missing}"
    absent = sorted(EXPECTED[_run_id(run)] - {n for n, c in rec.checked.items() if c})
    assert not absent, f"the step no longer launches {absent}"
    assert not rec.failures, rec.failures[:20]
    assert sum(rec.checked.values()) > 0
    del eng, rec
    torch.cuda.empty_cache()


# ---- negative controls ------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def recorded_launches():
    """real launches of the multi_central step at B = 1024 (N = 6144 student samples), kept with their outputs"""
    mp = pytest.MonkeyPatch()
    try:
        eng = _engine("multi_central", "default", {})
        step = _dino_inputs(eng, 1024)
        rec = Recorder(eng, mp, stash=("conv_tc", "conv_tc_wgrad", "linear_bwd_weight"))
        step()
        torch.cuda.synchronize()
    finally:
        mp.undo()
    assert not rec.failures, rec.failures[:20]
    yield rec
    del eng, rec
    torch.cuda.empty_cache()


def _flagged(rec, name, pre, post, live):
    ctx = Ctx(rec, live)
    ctx.rerun = False
    res = CHECKERS[name](ctx, pre, post)
    print(f"   control {name}: worst error / bound {res.worst:.3f}")
    return res.worst > 1.0


def test_control_zeroed_channel_octet_is_flagged(recorded_launches):
    pre, post, live = recorded_launches.stash["conv_tc"][0]
    bad = dict(post)
    bad["out"] = post["out"].clone()
    s = bad["out"].shape[0] // 2 + 1
    bad["out"][s, bad["out"].shape[1] - 1] = 0
    assert not _flagged(recorded_launches, "conv_tc", pre, post, live)
    assert _flagged(recorded_launches, "conv_tc", pre, bad, live)


def test_control_flipped_filter_tap_is_flagged(recorded_launches):
    rec = recorded_launches
    pre, post, live = rec.stash["conv_tc"][0]
    img = rec.image(live["wprep"])
    w = conv_weight(img)
    # the forward output as if the largest tap of output channel 3 had the opposite sign, in every sample
    co, K = 3, w.shape[-1]
    ci, rem = divmod(int(w[co].abs().argmax()), K * K)
    kh, kw = divmod(rem, K)
    tap = torch.zeros_like(w[co:co + 1])
    tap[0, ci, kh, kw] = w[co, ci, kh, kw]
    out = post["out"]
    z = nchw(out).to(F64)
    for a, b in chunks(0, out.shape[0], out[0].numel() * 4):
        z[a:b, co:co + 1] -= 2 * F.conv2d(nchw(pre["x8"][a:b]).to(F64), tap, padding=pre["pad"])
    bad = dict(post)
    bad["out"] = act8(z.to(out.dtype))
    bad["stats"] = post["stats"]
    assert _flagged(rec, "conv_tc", pre, bad, live)


def test_control_sample_left_out_of_weight_gradient_is_flagged(recorded_launches):
    rec = recorded_launches
    pre, post, live = rec.stash["conv_tc_wgrad"][0]
    xin, dz, N, wshape, pad = _wgrad_operands(pre)
    assert N == 6144
    assert not _flagged(rec, "conv_tc_wgrad", pre, post, live)
    # a sample of median gradient size (the largest one would be the easiest to see), and the smallest one for the record
    size = nchw(pre["dz8"]).float().abs().sum(dim=(1, 2, 3))
    order = torch.argsort(size)
    for s, must in ((int(order[N // 2]), True), (int(order[0]), False)):
        bad = dict(post)
        bad["dw"] = (post["dw"].to(F64) - torch.nn.grad.conv2d_weight(xin(s, s + 1), wshape, dz(s, s + 1), padding=pad)).float()
        print(f"   sample {s} ({'median' if must else 'smallest'} |dz|) left out:")
        flagged = _flagged(rec, "conv_tc_wgrad", pre, bad, live)
        if must:
            assert flagged


def test_control_dropped_split_k_partial_is_flagged(recorded_launches):
    rec = recorded_launches
    # the launch with the longest partials (the largest dropped share of the reduction)
    pre, post, live = max(rec.stash["linear_bwd_weight"], key=lambda r: linear_dw_splits(r[0]["dy"].shape[0], r[0]["dy"].shape[1], r[0]["x"].shape[1])[1])
    dy, x = pre["dy"], pre["x"]
    parts, rows = linear_dw_splits(dy.shape[0], dy.shape[1], x.shape[1])
    assert parts >= 3
    assert not _flagged(rec, "linear_bwd_weight", pre, post, live)
    lo, hi = rows, min(dy.shape[0], 2 * rows)            # the second partial
    bad = dict(post)
    bad["dw"] = (post["dw"].to(F64) - dy[lo:hi].to(F64).t() @ x[lo:hi].to(F64)).float()
    assert _flagged(rec, "linear_bwd_weight", pre, bad, live)
