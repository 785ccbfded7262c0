"""GPU parity of the tcgen05 / TMEM / TMA convolutions (csrc/conv_tc.cu) against torch conv2d on the SAME bf16-rounded
operands (fp32 accumulate on both sides): reference in fp64; tolerance 2e-5 of the output scale for fp32 outputs (accumulation order only), 8e-3 for bf16 outputs."""
import pytest
import torch
import torch.nn.functional as F

pytestmark = pytest.mark.gpu

from multimodal_ssl_avmnist_b200 import ops

DEV = "cuda"
# (Cin, Cout, H, W, K, pad) forward geometries of the encoders (models/unimodal.py:129-140, 186-208; dino.py:20-30)
FWD = [(8, 16, 56, 56, 5, 2), (16, 32, 28, 28, 5, 2), (32, 64, 14, 14, 5, 2), (32, 64, 14, 14, 5, 0), (32, 64, 14, 14, 3, 1),
       (64, 128, 7, 7, 3, 1),
       # the 3x3 audio stack of the simple multimodal encoders (models/dino.py:43-72): K-chunked / N-split instances
       (32, 64, 56, 56, 3, 1), (64, 128, 28, 28, 3, 1), (128, 256, 14, 14, 3, 1)]


def _bf(x):
    return x.to(torch.bfloat16).float()


def _unpack8(y8):
    N, P, H, W, _ = y8.shape
    return y8.float().permute(0, 1, 4, 2, 3).reshape(N, P * 8, H, W)


def _prep(w, flip=False):
    Co, Ci, K, _ = w.shape
    cin, cout = (Co, Ci) if flip else (Ci, Co)
    buf = torch.empty(ops.conv_tc_weight_bytes(cin, cout, K), dtype=torch.uint8, device=DEV)
    ops.conv_tc_prep_weights(w, buf, flip=flip)
    return buf


@pytest.mark.parametrize("geom", FWD)
@pytest.mark.parametrize("views,B", [(1, 3), (3, 5), (7, 40)])
def test_conv_tc_forward(geom, views, B):
    Cin, Cout, H, W, K, pad = geom
    assert ops.conv_tc_supported(*geom)
    g = torch.Generator().manual_seed(Cin * 131 + Cout + views)
    N = views * B
    x = torch.randn(N, Cin, H, W, generator=g).to(DEV)
    w = (torch.randn(Cout, Cin, K, K, generator=g) / (Cin * K * K) ** 0.5).to(DEV)
    b = torch.randn(Cout, generator=g).to(DEV)
    x8 = torch.empty(N, Cin // 8, H, W, 8, dtype=torch.bfloat16, device=DEV)
    ops.pack_act8(x, x8)
    assert torch.equal(_unpack8(x8), _bf(x))
    want = F.conv2d(_bf(x).double(), _bf(w).double(), b.double(), padding=pad).float()   # fp64: no TF32 / FFT algorithms
    Ho = want.shape[-1]
    wp = _prep(w)
    for out_bf16 in (False, torch.bfloat16, torch.float16):
        stats = torch.zeros(views, Cout, 2, dtype=torch.float64, device=DEV)
        if out_bf16:
            out = torch.full((N, Cout // 8, Ho, Ho, 8), float("nan"), dtype=out_bf16, device=DEV)
        else:
            out = torch.full((N, Cout, Ho, Ho), float("nan"), device=DEV)
        ops.conv_tc(x8, wp, b, out, stats, B, Cout, K, pad)
        torch.cuda.synchronize()
        got = _unpack8(out) if out_bf16 else out
        tol = (8e-3 if out_bf16 == torch.bfloat16 else 1e-3 if out_bf16 else 2e-5) * float(want.abs().max())
        err = float((got - want).abs().max())
        assert err <= tol, (geom, out_bf16, err, tol)
        wv = want.view(views, B, Cout, Ho, Ho).double()
        s_want = torch.stack([wv.sum(dim=(1, 3, 4)), (wv * wv).sum(dim=(1, 3, 4))], dim=-1)
        rel = float(((stats - s_want).abs() / (s_want.abs() + 1.0)).max())
        assert rel < (1e-5 if Cin * K * K < 1000 else 3e-5), (geom, "stats", rel)      # fp32 per-thread partial sums; longer reductions, larger |z|


def test_prep_weights_multi_matches_single_launches():
    """b200_conv_tc_prep_weights_multi (one launch over a device descriptor table) == the per-tensor launches, bit for bit,
    for every layer shape incl. the first layers (4 phases), the phase-packed 8<->16 / 16<->32 layers and flipped images."""
    g = torch.Generator().manual_seed(3)
    shapes = [(8, 1, 5, False), (32, 1, 5, False), (32, 1, 3, False), (16, 8, 5, False), (16, 8, 5, True), (32, 16, 5, False),
              (32, 16, 5, True), (64, 32, 5, False), (64, 32, 5, True), (64, 32, 3, True), (128, 64, 3, False)]
    ws, singles, multis, rows = [], [], [], []
    for co, ci, k, flip in shapes:
        w = torch.randn(co, ci, k, k, generator=g).to(DEV)
        cin, cout = (co, ci) if flip else (ci, co)
        a = torch.zeros(ops.conv_tc_weight_bytes(cin, cout, k), dtype=torch.uint8, device=DEV)
        b = torch.full_like(a, 0xAB)
        ops.conv_tc_prep_weights(w, a, flip=flip)
        ws.append(w); singles.append(a); multis.append(b)
        rows.append([w.data_ptr(), b.data_ptr(), cin, cout, k, int(flip)])
    ops.conv_tc_prep_weights_multi(torch.tensor(rows, dtype=torch.int64, device=DEV))
    torch.cuda.synchronize()
    for (co, ci, k, flip), a, b in zip(shapes, singles, multis):
        assert torch.equal(a, b), (co, ci, k, flip)


@pytest.mark.parametrize("geom", FWD)
def test_conv_tc_data_gradient(geom):
    """dx of conv(x, w): the same kernel with swapped channels, pad' = K-1-pad and flipped weights."""
    Cin, Cout, H, W, K, pad = geom
    Ho = H + 2 * pad - K + 1
    g = torch.Generator().manual_seed(7 + Cin)
    N = 9
    dz = torch.randn(N, Cout, Ho, Ho, generator=g).to(DEV)
    w = (torch.randn(Cout, Cin, K, K, generator=g) / (Cout * K * K) ** 0.5).to(DEV)
    want = F.conv_transpose2d(_bf(dz).double(), _bf(w).double(), padding=pad).float()
    assert want.shape == (N, Cin, H, W)
    dz8 = torch.empty(N, Cout // 8, Ho, Ho, 8, dtype=torch.bfloat16, device=DEV)
    ops.pack_act8(dz, dz8)
    wp = _prep(w, flip=True)
    assert ops.conv_tc_supported(Cout, Cin, Ho, Ho, K, K - 1 - pad)
    out = torch.full((N, Cin, H, W), float("nan"), device=DEV)
    ops.conv_tc(dz8, wp, None, out, None, N, Cin, K, K - 1 - pad)
    torch.cuda.synchronize()
    err = float((out - want).abs().max())
    assert err <= 2e-5 * float(want.abs().max()), (geom, err)


@pytest.mark.parametrize("geom", FWD)
@pytest.mark.parametrize("N", [1, 7, 300])
@pytest.mark.parametrize("variant", [1, 0])
def test_conv_tc_weight_gradient(geom, N, variant):
    """dW, db against autograd in fp64 on the same bf16-rounded x and dz (K = N*pixels, fp32 accumulate in TMEM).  variant 1 = the
    per-tap accumulators of the wide 3x3 layers, 0 = the shift-row kernel for every geometry."""
    Cin, Cout, H, W, K, pad = geom
    if variant == 0 and K != 3:
        pytest.skip("only the 3x3 layers have two formulations")
    old = ops.conv_tc_wgrad_variant(variant)
    try:
        _weight_gradient_case(geom, N)
    finally:
        ops.conv_tc_wgrad_variant(old)


def _weight_gradient_case(geom, N):
    Cin, Cout, H, W, K, pad = geom
    Ho = H + 2 * pad - K + 1
    g = torch.Generator().manual_seed(11 + Cin + N)
    x = torch.randn(N, Cin, H, W, generator=g).to(DEV)
    dz = torch.randn(N, Cout, Ho, Ho, generator=g).to(DEV)
    xd = _bf(x).double().requires_grad_(False)
    wd = torch.zeros(Cout, Cin, K, K, dtype=torch.float64, device=DEV, requires_grad=True)
    bd = torch.zeros(Cout, dtype=torch.float64, device=DEV, requires_grad=True)
    F.conv2d(xd, wd, bd, padding=pad).backward(_bf(dz).double())
    x8 = torch.empty(N, Cin // 8, H, W, 8, dtype=torch.bfloat16, device=DEV)
    dz8 = torch.empty(N, Cout // 8, Ho, Ho, 8, dtype=torch.bfloat16, device=DEV)
    ops.pack_act8(x, x8)
    ops.pack_act8(dz, dz8)
    work = torch.empty(ops.conv_tc_wgrad_work_floats(N, Cin, Cout, H, W, K, pad), device=DEV)
    dw = torch.full((Cout, Cin, K, K), float("nan"), device=DEV)
    ops.conv_tc_wgrad(x8, dz8, dw, work, pad)
    torch.cuda.synchronize()
    scale = float(wd.grad.abs().max())
    err = float((dw.double() - wd.grad).abs().max())
    assert err <= (3e-5 if N * Ho * Ho < 200_000 else 6e-5) * scale, (geom, N, err, scale)       # fp32 TMEM accumulation over K = N * pixels


def _pack8(x):
    N, C, H, W = x.shape
    out = torch.empty(N, C // 8, H, W, 8, dtype=torch.bfloat16, device=DEV)
    ops.pack_act8(x.contiguous(), out)
    return out


@pytest.mark.parametrize("zdt", [torch.bfloat16, torch.float16])
@pytest.mark.parametrize("C,H,views,B", [(16, 56, 2, 3), (32, 28, 3, 5), (64, 14, 7, 9), (64, 10, 1, 40), (8, 112, 2, 2), (128, 7, 3, 5)])
def test_bn_relu_pool8(C, H, views, B, zdt):
    """act8 BN-apply/ReLU/pool forward and backward against a torch fp32 restatement on the same bf16 z / dp."""
    g = torch.Generator().manual_seed(C + H)
    N = views * B
    z = torch.randn(N, C, H, H, generator=g)
    z = (_bf(z) if zdt == torch.bfloat16 else z.half().float()).to(DEV)
    scale = (torch.randn(views, C, generator=g) * 0.5 + 1.0).to(DEV)       # includes negative gammas
    shift = (torch.randn(views, C, generator=g) * 0.3).to(DEV)
    mean = (torch.randn(views, C, generator=g) * 0.2).to(DEV)
    invstd = (torch.rand(views, C, generator=g) + 0.5).to(DEV)
    dp = _bf(torch.randn(N, C, H // 2, H // 2, generator=g)).to(DEV)
    if zdt == torch.float16:
        z8 = z.view(N, C // 8, 8, H, H).permute(0, 1, 3, 4, 2).contiguous().half()
    else:
        z8 = _pack8(z)
    a = scale.repeat_interleave(B, 0)[:, :, None, None]
    b = shift.repeat_interleave(B, 0)[:, :, None, None]
    mu = mean.repeat_interleave(B, 0)[:, :, None, None]
    istd = invstd.repeat_interleave(B, 0)[:, :, None, None]
    y = a * z + b
    pooled, idx = F.max_pool2d(y, 2, return_indices=True)
    want_p = pooled.clamp_min(0)
    # forward, both output formats
    out32 = torch.full((N, C, H // 2, H // 2), float("nan"), device=DEV)
    ops.bn_relu_pool8_fwd(z8, scale, shift, out32, B)
    assert float((out32 - want_p).abs().max()) <= 1e-5 * float(want_p.abs().max())
    out8 = torch.empty(N, C // 8, H // 2, H // 2, 8, dtype=torch.bfloat16, device=DEV)
    ops.bn_relu_pool8_fwd(z8, scale, shift, out8, B)
    assert torch.equal(_unpack8(out8), _bf(out32))
    chk = torch.empty_like(out32)
    ops.unpack_act8(out8, chk)
    assert torch.equal(chk, _bf(out32))
    # backward
    gsel = dp * (pooled > 0)
    dy = F.max_unpool2d(gsel, idx, 2, output_size=(H, H))
    xh = (z - mu) * istd
    s_want = torch.stack([dy.view(views, B, C, -1).double().sum(dim=(1, 3)), (dy * xh).view(views, B, C, -1).double().sum(dim=(1, 3))], -1)
    cnt = B * H * H
    k1 = (s_want[..., 0] / cnt).float().repeat_interleave(B, 0)[:, :, None, None]
    k2 = (s_want[..., 1] / cnt).float().repeat_interleave(B, 0)[:, :, None, None]
    want_dz = a * (dy - k1 - xh * k2)
    for dpt in (dp, _pack8(dp)):
        sums = torch.zeros(views, C, 2, dtype=torch.float64, device=DEV)
        ops.bn_relu_pool8_bwd_reduce(z8, dpt, scale, shift, mean, invstd, sums, B)
        assert float(((sums - s_want).abs() / (s_want.abs() + 1.0)).max()) < 1e-4
        dz8 = torch.empty(z8.shape, dtype=torch.bfloat16, device=DEV)
        dbsum = torch.zeros(C, dtype=torch.float64, device=DEV)
        ops.bn_relu_pool8_bwd_apply(z8, dpt, scale, shift, mean, invstd, s_want.contiguous(), dz8, B, dbsum=dbsum)
        got = _unpack8(dz8)
        assert float((got - want_dz).abs().max()) <= 8e-3 * float(want_dz.abs().max())
        db_want = want_dz.double().sum(dim=(0, 2, 3))
        db = torch.empty(C, device=DEV)
        ops.bias_grad_finalize(dbsum, db)
        assert float((db.double() - db_want).abs().max()) <= 1e-4 * float(want_dz.abs().sum(dim=(0, 2, 3)).max())


# first layers (C_in = 1) on the shift8 image: (Cout, H, K, pad)
FIRST = [(8, 112, 5, 2), (32, 28, 5, 2), (32, 28, 3, 1), (32, 112, 3, 1)]


@pytest.mark.parametrize("geom", FIRST)
@pytest.mark.parametrize("views,B", [(1, 2), (3, 5), (7, 12)])
def test_first_layer_shift8_forward_and_weight_gradient(geom, views, B):
    Cout, H, K, pad = geom
    assert ops.conv_tc_supported(1, Cout, H, H, K, pad)
    g = torch.Generator().manual_seed(Cout + H + views)
    N = views * B
    x = torch.rand(N, 1, H, H, generator=g).to(DEV)
    w = (torch.randn(Cout, 1, K, K, generator=g) / K).to(DEV)
    b = torch.randn(Cout, generator=g).to(DEV)
    x8 = torch.empty(N, H, H + pad, 8, dtype=torch.bfloat16, device=DEV)
    ops.pack_shift8(x, x8, pad)
    xb = _bf(x)
    assert torch.equal(x8[:, :, pad:, 0].float(), xb[:, 0]) and float(x8[:, :, :pad, 0].abs().max()) == 0.0
    assert torch.equal(x8[:, :, :H - 3 + pad, 3].float(), xb[:, 0, :, 3 - pad:]) and float(x8[:, :, H - 3 + pad:, 3].abs().max()) == 0.0
    want = F.conv2d(xb.double(), _bf(w).double(), b.double(), padding=pad).float()
    wp = torch.empty(ops.conv_tc_weight_bytes(1, Cout, K), dtype=torch.uint8, device=DEV)
    ops.conv_tc_prep_weights(w, wp)
    stats = torch.zeros(views, Cout, 2, dtype=torch.float64, device=DEV)
    z = torch.full((N, Cout // 8, H, H, 8), float("nan"), dtype=torch.float16, device=DEV)
    # forward input: the quad8 image (unit = padded pixels 4xq .. 4xq+7: the taps of four adjacent outputs)
    WQ = ops.quad8_width(H, pad)
    xq8 = torch.empty(N, H, WQ, 8, dtype=torch.bfloat16, device=DEV)
    ops.pack_quad8(x, xq8, pad)
    xpad = F.pad(xb[:, 0], (pad, 4 * WQ + 8 - H - pad))
    for e in (0, 3, 7):
        assert torch.equal(xq8[:, :, :, e].float(), xpad[:, :, e:e + 4 * WQ:4])
    ops.conv_tc(xq8, wp, b, z, stats, B, Cout, K, pad)
    torch.cuda.synchronize()
    assert float((_unpack8(z) - want).abs().max()) <= 1e-3 * float(want.abs().max())
    wv = want.view(views, B, Cout, H, H).double()
    s_want = torch.stack([wv.sum(dim=(1, 3, 4)), (wv * wv).sum(dim=(1, 3, 4))], dim=-1)
    assert float(((stats - s_want).abs() / (s_want.abs() + 1.0)).max()) < 1e-5
    # weight gradient
    dz = torch.randn(N, Cout, H, H, generator=g).to(DEV)
    wd = torch.zeros(Cout, 1, K, K, dtype=torch.float64, device=DEV, requires_grad=True)
    F.conv2d(xb.double(), wd, None, padding=pad).backward(_bf(dz).double())
    dz8 = _pack8(dz)
    work = torch.empty(ops.conv_tc_wgrad_work_floats(N, 1, Cout, H, H, K, pad), device=DEV)
    dw = torch.full((Cout, 1, K, K), float("nan"), device=DEV)
    ops.conv_tc_wgrad(x8, dz8, dw, work, pad)
    torch.cuda.synchronize()
    assert float((dw.double() - wd.grad).abs().max()) <= 3e-5 * float(wd.grad.abs().max())


@pytest.mark.parametrize("geom", FIRST)
@pytest.mark.parametrize("views,B", [(1, 2), (3, 5), (7, 12), (2, 160)])
def test_first_layer_fused_backward_matches_apply_then_wgrad(geom, views, B):
    """b200_conv_tc_wgrad_l0_fused == b200_bn_relu_pool8_bwd_apply followed by b200_conv_tc_wgrad: the dz tile is produced
    in shared memory with the same arithmetic and bf16 rounding, so dW agrees to accumulation order and the bias-gradient
    sums to fp32 summation order."""
    Cout, H, K, pad = geom
    g = torch.Generator().manual_seed(11 * Cout + H + views + B)
    N = views * B
    x = torch.rand(N, 1, H, H, generator=g).to(DEV)
    x8 = torch.empty(N, H, H + pad, 8, dtype=torch.bfloat16, device=DEV)
    ops.pack_shift8(x, x8, pad)
    z8 = torch.randn(N, Cout // 8, H, H, 8, generator=g).to(DEV).to(torch.float16)
    dp8 = torch.randn(N, Cout // 8, H // 2, H // 2, 8, generator=g).to(DEV).to(torch.bfloat16)
    scale = (torch.rand(views, Cout, generator=g) + 0.5).to(DEV)
    scale[:, 1] *= -1.0                                   # negative BatchNorm scale flips the arg-max
    shift = (torch.randn(views, Cout, generator=g) * 0.3).to(DEV)
    mean = (torch.randn(views, Cout, generator=g) * 0.1).to(DEV)
    invstd = (torch.rand(views, Cout, generator=g) + 0.5).to(DEV)
    sums = torch.zeros(views, Cout, 2, dtype=torch.float64, device=DEV)
    ops.bn_relu_pool8_bwd_reduce(z8, dp8, scale, shift, mean, invstd, sums, B)
    # two-kernel path
    dz8 = torch.empty(N, Cout // 8, H, H, 8, dtype=torch.bfloat16, device=DEV)
    db_a = torch.zeros(Cout, dtype=torch.float64, device=DEV)
    ops.bn_relu_pool8_bwd_apply(z8, dp8, scale, shift, mean, invstd, sums, dz8, B, dbsum=db_a)
    work = torch.empty(ops.conv_tc_wgrad_work_floats(N, 1, Cout, H, H, K, pad), device=DEV)
    dw_a = torch.full((Cout, 1, K, K), float("nan"), device=DEV)
    ops.conv_tc_wgrad(x8, dz8, dw_a, work, pad)
    # fused
    z_keep = z8.clone()
    work2 = torch.empty(ops.conv_tc_wgrad_l0_fused_work_floats(N, B, Cout, H, H, K, pad), device=DEV)
    dw_b = torch.full((Cout, 1, K, K), float("nan"), device=DEV)
    db_b = torch.zeros(Cout, dtype=torch.float64, device=DEV)
    xq8 = torch.empty(N, H, ops.quad8_width(H, pad), 8, dtype=torch.bfloat16, device=DEV)
    ops.pack_quad8(x, xq8, pad)
    ops.conv_tc_wgrad_l0_fused(xq8, z8, dp8, scale, shift, mean, invstd, sums, dw_b, db_b, work2, B, pad)
    torch.cuda.synchronize()
    assert torch.equal(z8, z_keep)                       # inputs untouched
    # fp32 tensor-core accumulation (truncating adds, split over two accumulators in the fused kernel): bounds are relative
    # to sum |x|*|dz| per tap
    wa = torch.zeros(Cout, 1, K, K, dtype=torch.float64, device=DEV, requires_grad=True)
    F.conv2d(_bf(x).double(), wa, None, padding=pad).backward(_unpack8(dz8).double().abs())
    assert float(((dw_a - dw_b).abs().double() / wa.grad).max()) <= 3e-6
    assert float((db_a - db_b).abs().max()) <= 1e-4 * float(dz8.float().abs().sum(dim=(0, 2, 3)).max())
    # and against an fp64 convolution weight gradient of the unpacked dz
    wd = torch.zeros(Cout, 1, K, K, dtype=torch.float64, device=DEV, requires_grad=True)
    F.conv2d(_bf(x).double(), wd, None, padding=pad).backward(_unpack8(dz8).double())
    assert float(((dw_b.double() - wd.grad).abs() / wa.grad).max()) <= 3e-6


def test_augmentation_direct_quad8_output_matches_pack():
    """The augmentation kernels' direct bf16 quad8 output == pack_quad8(fp32 output) bit for bit (same op records)."""
    from multimodal_ssl_avmnist_b200.engine import DinoStepEngine
    eng = DinoStepEngine(kind="multi_central", device=DEV, precision="bf16", seed=5)
    B = 6
    img = torch.rand(B, 28, 28, device=DEV)
    aud = torch.randint(0, 256, (B, 112, 112), dtype=torch.uint8, device=DEV)
    xi, xa = eng.augment(img, aud)                      # fp32 views
    xi, xa = xi.clone(), xa.clone()
    xi8, xa8 = eng.augment(img, aud, direct=True)       # same rng_step -> same op records and noise
    for x, x8, pad in ((xi, xi8, 2), (xa, xa8, 2)):
        V, Bb, S, _ = x.shape
        want = torch.empty(V * Bb, S, ops.quad8_width(S, pad), 8, dtype=torch.bfloat16, device=DEV)
        ops.pack_quad8(x.reshape(V * Bb, S, S).contiguous(), want, pad)
        assert torch.equal(x8.reshape(want.shape), want)
    # and the whole step runs from it
    l1 = eng.train_step(img, aud).clone()
    torch.cuda.synchronize()
    assert 3.0 < float(l1[0]) < 6.0


# (M, N, K): encoder FCs, fusion, projection head, ragged sizes (partial tiles in every dimension)
LIN = [(6144, 256, 3136), (48, 256, 1600), (300, 512, 256), (130, 128, 512), (77, 10, 512), (1000, 256, 512)]


@pytest.mark.parametrize("M,N,K", LIN)
def test_linear_tensor_core_tf32(M, N, K):
    """tcgen05 kind::tf32 GEMMs (fwd K-major x K-major, data gradient K-major x MN-major, weight gradient MN-major x MN-major
    with split-K) against fp64 on the same fp32 tensors: tolerance 2e-3 of the output scale (tf32 operand rounding)."""
    g = torch.Generator().manual_seed(M + N + K)
    x = torch.randn(M, K, generator=g).to(DEV)
    w = (torch.randn(N, K, generator=g) / K ** 0.5).to(DEV)
    b = torch.randn(N, generator=g).to(DEV)
    dy = torch.randn(M, N, generator=g).to(DEV)
    mask = (torch.rand(M, N, generator=g) > 0.3).to(torch.uint8).to(DEV)
    want = x.double() @ w.double().t() + b.double()
    for act in (0, 1, 2):
        y = torch.full((M, N), float("nan"), device=DEV)
        ops.linear_fwd(x, w, b, y, act=act, mask=mask if act == 2 else None, drop_p=0.3 if act == 2 else 0.0, tc=True)
        ref = want if act == 0 else want.clamp_min(0)
        if act == 2:
            ref = ref * mask.double() / 0.7
        assert float((y.double() - ref).abs().max()) <= 2e-3 * float(want.abs().max()), (M, N, K, act)
    # strided output / input (column slices of a wider matrix, as the engine's cat buffer)
    wide = torch.zeros(M, 2 * N + 4, device=DEV)
    ops.linear_fwd(x, w, b, wide[:, N + 4:], tc=True)
    assert float((wide[:, N + 4:].double() - want).abs().max()) <= 2e-3 * float(want.abs().max())
    assert float(wide[:, :N + 4].abs().max()) == 0.0
    dx = torch.full((M, K), float("nan"), device=DEV)
    ops.linear_bwd_data(dy, w, dx, tc=True)
    ref = dy.double() @ w.double()
    assert float((dx.double() - ref).abs().max()) <= 2e-3 * float(ref.abs().max())
    dw = torch.full((N, K), float("nan"), device=DEV)
    db = torch.full((N,), float("nan"), device=DEV)
    ops.linear_bwd_weight(dy, x, dw, db, tc=True)
    ref = dy.double().t() @ x.double()
    assert float((dw.double() - ref).abs().max()) <= 2e-3 * float(ref.abs().max())
    assert float((db.double() - dy.double().sum(0)).abs().max()) <= 1e-4 * float(dy.double().abs().sum(0).max())
    dw2 = dw.clone()
    ops.linear_bwd_weight(dy, x, dw2, db, accumulate=True, tc=True)
    assert float((dw2.double() - 2 * ref).abs().max()) <= 4e-3 * float(ref.abs().max())


@pytest.mark.parametrize("C,H,views,B", [(16, 56, 2, 3), (64, 10, 3, 7), (8, 112, 2, 2)])
def test_bn_backward_statistics_from_pooled_tensors(C, H, views, B):
    """b200_bn_pool8_bwd_reduce_p (reads only p and dp) == b200_bn_relu_pool8_bwd_reduce (reads z) up to the rounding of p."""
    g = torch.Generator().manual_seed(C * 3 + H)
    N = views * B
    z = torch.randn(N, C, H, H, generator=g).half().float().to(DEV)
    gamma = (torch.randn(C, generator=g) * 0.3 + 1.0).to(DEV)
    gamma[1] = -0.7                                            # a negative BatchNorm weight (arg-max becomes arg-min of z)
    beta = (torch.randn(C, generator=g) * 0.2).to(DEV)
    zv = z.view(views, B, C, -1)
    mean = zv.mean(dim=(1, 3))
    invstd = (zv.var(dim=(1, 3), unbiased=False) + 1e-5).rsqrt()
    scale = (gamma[None] * invstd).contiguous()
    shift = (beta[None] - mean * scale).contiguous()
    dp = _bf(torch.randn(N, C, H // 2, H // 2, generator=g)).to(DEV)
    z8 = z.view(N, C // 8, 8, H, H).permute(0, 1, 3, 4, 2).contiguous().half()
    want = torch.zeros(views, C, 2, dtype=torch.float64, device=DEV)
    ops.bn_relu_pool8_bwd_reduce(z8, dp, scale, shift, mean.contiguous(), invstd.contiguous(), want, B)
    p32 = torch.empty(N, C, H // 2, H // 2, device=DEV)
    ops.bn_relu_pool8_fwd(z8, scale, shift, p32, B)
    p8 = torch.empty(N, C // 8, H // 2, H // 2, 8, dtype=torch.bfloat16, device=DEV)
    ops.bn_relu_pool8_fwd(z8, scale, shift, p8, B)
    ref_scale = want.abs().max(dim=1, keepdim=True).values + 1e-9
    for pt, dpt, tol in ((p32, dp, 1e-4), (p8, _pack8(dp), 5e-3), (p8, dp, 5e-3)):
        got = torch.zeros_like(want)
        ops.bn_pool8_bwd_reduce_p(pt, dpt, gamma, beta, got, B)
        assert float(((got - want).abs() / ref_scale).max()) < tol, (pt.dtype, dpt.dtype)


@pytest.mark.parametrize("B,D", [(64, 128), (300, 128), (1024, 128), (2500, 64)])
def test_infonce_tensor_core(B, D):
    """Tensor-core InfoNCE (tf32 similarity GEMM + exp/row-sum epilogue, bf16 E, bf16 gradient GEMMs) against the fp64 formula
    (models/dino.py:1091-1128): loss 1e-3 relative, gradients 2e-2 of their scale."""
    g = torch.Generator().manual_seed(B + D)
    a = torch.randn(B, D, generator=g).to(DEV)
    b = (0.5 * a.cpu() + torch.randn(B, D, generator=g)).to(DEV)
    ad, bd = a.double().requires_grad_(True), b.double().requires_grad_(True)
    sim = F.normalize(ad, dim=1) @ F.normalize(bd, dim=1).t() / 0.07
    lab = torch.arange(B, device=DEV)
    want = 0.5 * (F.cross_entropy(sim, lab) + F.cross_entropy(sim.t(), lab))
    want.backward()
    ga, gb, lo = torch.empty_like(a), torch.empty_like(b), torch.empty(1, device=DEV)
    work = torch.empty(ops.infonce_work_floats(B, D, tc=True), device=DEV)
    ops.infonce_fwd_bwd(a, b, ga, gb, lo, work, temperature=0.07, tc=True)
    torch.cuda.synchronize()
    assert abs(float(lo) - float(want)) < 1e-3 * float(want), (float(lo), float(want))
    for got, ref in ((ga, ad.grad), (gb, bd.grad)):
        assert float((got.double() - ref).abs().max()) <= 2e-2 * float(ref.abs().max())
        cos = float((got.double().flatten() @ ref.flatten()) / (got.double().norm() * ref.norm()))
        assert cos > 0.9995, cos


POOLED = [(8, 16, 56, 5, 2), (16, 32, 28, 5, 2), (32, 64, 14, 3, 1), (1, 8, 112, 5, 2), (1, 32, 28, 5, 2), (1, 32, 28, 3, 1),
          (1, 32, 112, 3, 1), (32, 64, 56, 3, 1)]


@pytest.mark.parametrize("geom", POOLED)
@pytest.mark.parametrize("views,B", [(1, 3), (3, 5), (6, 43)])
def test_conv_tc_fused_pool_epilogue_is_bit_identical_to_the_unfused_chain(geom, views, B):
    """b200_conv_tc_pool (conv + statistics + 2x2 window extreme by sign(gamma) in the epilogue) -> bn_finalize -> b200_bn_relu_apply8
    must equal conv_tc -> bn_finalize -> bn_relu_pool8_fwd BIT FOR BIT (p, z, statistics), with mixed-sign BatchNorm weights, with
    and without the z store, for bf16-act8 and fp32-NCHW outputs; the extreme itself is checked against torch max / min pooling."""
    Cin, Cout, H, K, pad = geom
    assert ops.conv_tc_pool_supported(Cin, Cout, H, H, K, pad)
    g = torch.Generator().manual_seed(Cin * 7 + Cout + views + H)
    N = views * B
    Ho = H + 2 * pad - K + 1
    w = (torch.randn(Cout, Cin, K, K, generator=g) / (Cin * K * K) ** 0.5).to(DEV)
    bias = torch.randn(Cout, generator=g).to(DEV)
    gamma = torch.randn(Cout, generator=g).to(DEV)          # both signs
    gamma[0] = 0.0
    beta = torch.randn(Cout, generator=g).to(DEV)
    if Cin == 1:
        x = torch.rand(N, 1, H, H, generator=g).to(DEV)
        x8 = torch.empty(N, H, ops.quad8_width(H, pad), 8, dtype=torch.bfloat16, device=DEV)
        ops.pack_quad8(x, x8, pad)
    else:
        x = torch.randn(N, Cin, H, H, generator=g).to(DEV)
        x8 = torch.empty(N, Cin // 8, H, H, 8, dtype=torch.bfloat16, device=DEV)
        ops.pack_act8(x, x8)
    wp = torch.empty(ops.conv_tc_weight_bytes(Cin, Cout, K), dtype=torch.uint8, device=DEV)
    ops.conv_tc_prep_weights(w, wp)

    def finalize(stats):
        sc, sh, mu, inv = (torch.empty(views, Cout, device=DEV) for _ in range(4))
        rm, rv, nbt = torch.zeros(Cout, device=DEV), torch.ones(Cout, device=DEV), torch.zeros(1, dtype=torch.int64, device=DEV)
        ops.bn_finalize(stats, gamma, beta, rm, rv, nbt, sc, sh, mu, inv, views, B * Ho * Ho)
        return sc, sh

    # unfused chain
    z_ref = torch.full((N, Cout // 8, Ho, Ho, 8), float("nan"), dtype=torch.float16, device=DEV)
    st_ref = torch.zeros(views, Cout, 2, dtype=torch.float64, device=DEV)
    ops.conv_tc(x8, wp, bias, z_ref, st_ref, B, Cout, K, pad)
    sc, sh = finalize(st_ref)
    p8_ref = torch.empty(N, Cout // 8, Ho // 2, Ho // 2, 8, dtype=torch.bfloat16, device=DEV)
    p32_ref = torch.empty(N, Cout, Ho // 2, Ho // 2, device=DEV)
    ops.bn_relu_pool8_fwd(z_ref, sc, sh, p8_ref, B)
    ops.bn_relu_pool8_fwd(z_ref, sc, sh, p32_ref, B)
    for keep_z in (True, False):
        z = torch.full_like(z_ref, float("nan")) if keep_z else None
        e8 = torch.full((N, Cout // 8, Ho // 2, Ho // 2, 8), float("nan"), dtype=torch.float16, device=DEV)
        st = torch.zeros_like(st_ref)
        ops.conv_tc_pool(x8, wp, bias, gamma, z, e8, st, B, Cout, K, pad)
        torch.cuda.synchronize()
        # (the statistics are fp64 atomic sums: two launches agree to ~1e-15, not bit for bit)
        assert float(((st - st_ref).abs() / (st_ref.abs() + 1.0)).max()) < 1e-12
        if keep_z:
            assert torch.equal(z, z_ref)
        # the extreme: max where gamma >= 0, min where gamma < 0, of the fp16 z
        zr = _unpack8(z_ref)
        sgn = torch.where(gamma < 0, -1.0, 1.0).view(1, Cout, 1, 1)
        want_e = F.max_pool2d(zr * sgn, 2) * sgn
        assert torch.equal(_unpack8(e8), want_e), float((_unpack8(e8) - want_e).abs().max())
        sc2, sh2 = finalize(st)
        assert torch.allclose(sc2, sc, rtol=1e-6, atol=0) and torch.allclose(sh2, sh, rtol=1e-5, atol=1e-7)
        p8 = torch.full_like(p8_ref, float("nan"))
        p32 = torch.full_like(p32_ref, float("nan"))
        ops.bn_relu_apply8(e8, sc, sh, p8, B)         # the SAME scale / shift as the unfused chain: then p must match bit for bit
        ops.bn_relu_apply8(e8, sc, sh, p32, B)
        torch.cuda.synchronize()
        assert torch.equal(p8, p8_ref) and torch.equal(p32, p32_ref)


# data gradients (forward geometry: Cin, Cout, H, K, pad) whose epilogue also produces the BN-backward sums of the layer below
DGRAD_BNSTAT = [(8, 16, 56, 5, 2), (16, 32, 28, 5, 2), (32, 64, 14, 5, 2), (32, 64, 14, 5, 0), (32, 64, 14, 3, 1),
                (64, 128, 7, 3, 1)]        # the last: image_simple conv3 (CfgS2d data gradient, odd 7x7 planes)


@pytest.mark.parametrize("geom", DGRAD_BNSTAT)
@pytest.mark.parametrize("views,B", [(1, 3), (3, 5), (7, 41)])
def test_dgrad_with_fused_bn_backward_statistics(geom, views, B):
    """b200_conv_tc_dgrad_bnstat == b200_conv_tc (data gradient) followed by b200_bn_pool8_bwd_reduce_p on (p, dp): dx bit for bit,
    the per-(view, channel) sums to fp64-atomic rounding; mixed-sign / zero BatchNorm weights, dead (p == 0) units."""
    Cin, Cout, H, K, pad = geom
    Ho = H + 2 * pad - K + 1
    assert ops.conv_tc_dgrad_bnstat_supported(Cout, Cin, Ho, Ho, K, K - 1 - pad)
    g = torch.Generator().manual_seed(Cin + 3 * Cout + views)
    N = views * B
    dz = torch.randn(N, Cout, Ho, Ho, generator=g).to(DEV)
    w = (torch.randn(Cout, Cin, K, K, generator=g) / (Cout * K * K) ** 0.5).to(DEV)
    gamma = (torch.randn(Cin, generator=g) * 0.5 + 0.8).to(DEV)
    gamma[1] = -0.6
    gamma[2] = 0.0
    beta = (torch.randn(Cin, generator=g) * 0.3).to(DEV)
    p = torch.relu(torch.randn(N, Cin, H, H, generator=g)).to(DEV)            # pooled activations of the layer below: half of them dead
    dz8 = _pack8(dz)
    p8 = _pack8(p)
    wp = _prep(w, flip=True)
    dx_ref = torch.full((N, Cin // 8, H, H, 8), float("nan"), dtype=torch.bfloat16, device=DEV)
    ops.conv_tc(dz8, wp, None, dx_ref, None, N, Cin, K, K - 1 - pad)
    want = torch.zeros(views, Cin, 2, dtype=torch.float64, device=DEV)
    ops.bn_pool8_bwd_reduce_p(p8, dx_ref, gamma, beta, want, B)
    dx = torch.full_like(dx_ref, float("nan"))
    got = torch.zeros_like(want)
    ops.conv_tc_dgrad_bnstat(dz8, wp, dx, p8, gamma, beta, got, B, K, K - 1 - pad)
    torch.cuda.synchronize()
    assert torch.equal(dx, dx_ref)
    scale = want.abs().max(dim=1, keepdim=True).values + 1e-9
    # same fp32 products, summed per thread in a different order than the stand-alone reduction: 1e-5 of the per-view scale
    assert float(((got - want).abs() / scale).max()) < 1e-5, float(((got - want).abs() / scale).max())
