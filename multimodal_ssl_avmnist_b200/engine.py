"""The DINO training-step engine: flat parameter arenas + the launch schedule of one step.

One engine instance owns, on one GPU,
  * the student / teacher parameter arenas (fp32, one contiguous buffer each; `nn.Parameter`s of the API
    modules are views into them, named exactly like the reference's state_dict entries),
  * the gradient arena and the Adam moment arenas (same layout as the student arena),
  * BatchNorm running statistics, the DINO centre, and per-batch-size activation workspaces,
and runs the reference's step order (SURVEY.md §3.2): multi-crop augmentation -> student on all views and
teacher on the global views (BatchNorm statistics per view-call) -> projection heads -> fused DINO loss
(+ centre EMA) [+ MSE / InfoNCE / CE on an extra un-augmented pass] -> teacher EMA -> backward -> Adam.

Every arithmetic stage is a `b200_*` call into libavmnist_b200.so (ops.py); torch only provides device memory and
streams; for data parallel runs the two exchanges (gradient arena, centre column sums) are C-ABI calls too (b200_dp_*).

Encoders (`kind`): 'multi_central' (CentralMultiModalEncoder, the headline), 'multi_simple' / 'multi_simple_gated' /
'multi_cross_attention' (the 3x3 conv encoders of models/dino.py:214-263, 385-452: stack tops are avgpool -> linear and a mix stage --
sigmoid gates or batch-wide cross attention -- sits before the fusion MLP), the unimodal 'image_simple' (ImageEncoder) and
'spectrogram_simple' (SpectrogramEncoder: the audio stack of 'multi_simple' alone), and the unimodal CentralNet kinds 'image_central'
(ImageEncoderCentral) and 'spectrogram_central' (SpectrogramEncoderCentral): one branch of 'multi_central' each, flatten -> Linear to
the embedding.  The stand-alone contrastive steps of other_ssl/ reuse these building blocks from contrastive.ContrastiveStepEngine.

Arena layout (student):  [ encoder params that receive gradients | projection head | unused fc1/fc2 | mode heads ]
        (teacher):       [ encoder params that receive gradients | projection head | unused fc1/fc2 ]
so the teacher EMA is ONE flat kernel over the common prefix and Adam is one flat kernel over the trainable
prefix (plus one over the mode heads); the unused CentralNet classifier heads (models/unimodal.py:121-125,
179-183) are EMA'd and check-pointed like in the reference but never receive gradients.
"""
import contextlib
import math

import numpy as np

import torch

from . import augment as A
from . import dp
from . import ops

F32 = torch.float32


# ---------------------------------------------------------------------------------------------------------
# parameter inventories (names as in the reference state_dict; see models/dino.py:454-468, unimodal.py:105-183)
# ---------------------------------------------------------------------------------------------------------
def _conv(n, co, ci, k):
    return [(f"{n}.weight", (co, ci, k, k)), (f"{n}.bias", (co,))]


def _vec2(n, c):
    return [(f"{n}.weight", (c,)), (f"{n}.bias", (c,))]


def _lin(n, o, i):
    return [(f"{n}.weight", (o, i)), (f"{n}.bias", (o,))]


def central_encoder_params(E, O):
    """(used, unused) parameter specs of CentralMultiModalEncoder, each in the reference's declaration order."""
    used, unused = [], []
    p = "image_encoder.0"
    used += _conv(f"{p}.conv1", 32, 1, 5) + _vec2(f"{p}.bn1", 32) + _conv(f"{p}.conv2", 64, 32, 5) + _vec2(f"{p}.bn2", 64)
    unused += _lin(f"{p}.fc1", 1024, 1600) + _lin(f"{p}.fc2", 10, 1024)
    used += _lin("image_encoder.1", E, 1600)
    p = "audio_encoder.0"
    used += _conv(f"{p}.conv1", 8, 1, 5) + _vec2(f"{p}.bn1", 8) + _conv(f"{p}.conv2", 16, 8, 5) + _vec2(f"{p}.bn2", 16)
    used += _conv(f"{p}.conv3", 32, 16, 5) + _vec2(f"{p}.bn3", 32) + _conv(f"{p}.conv4", 64, 32, 5) + _vec2(f"{p}.bn4", 64)
    unused += _lin(f"{p}.fc1", 1024, 3136) + _lin(f"{p}.fc2", 10, 1024)
    used += _lin("audio_encoder.1", E, 3136)
    used += _lin("fusion.0", E, 2 * E) + _lin("fusion.3", O, E)
    return used, unused


def central_reference_order(E, O):
    """Parameter names in the reference's `.parameters()` order (for state_dict / optimizer compatibility)."""
    names = []
    p = "image_encoder.0"
    for l in ("conv1", "bn1", "conv2", "bn2", "fc1", "fc2"):
        names += [f"{p}.{l}.weight", f"{p}.{l}.bias"]
    names += ["image_encoder.1.weight", "image_encoder.1.bias"]
    p = "audio_encoder.0"
    for l in ("conv1", "bn1", "conv2", "bn2", "conv3", "bn3", "conv4", "bn4", "fc1", "fc2"):
        names += [f"{p}.{l}.weight", f"{p}.{l}.bias"]
    names += ["audio_encoder.1.weight", "audio_encoder.1.bias", "fusion.0.weight", "fusion.0.bias", "fusion.3.weight", "fusion.3.bias"]
    return names


def image_simple_params(O):
    used = _conv("encoder.0", 32, 1, 3) + _vec2("encoder.1", 32) + _conv("encoder.4", 64, 32, 3) + _vec2("encoder.5", 64)
    used += _conv("encoder.8", 128, 64, 3) + _vec2("encoder.9", 128) + _lin("encoder.14", 512, 128) + _lin("projection.0", O, 512)
    return used, []


def spectrogram_simple_params(O):
    """SpectrogramEncoder (models/dino.py:502-513) = audio_encoder(O): four conv blocks and Linear(256, O), no projection layer."""
    used = []
    for i, (ci, co) in zip((0, 4, 8, 12), ((1, 32), (32, 64), (64, 128), (128, 256))):
        used += _conv(f"encoder.{i}", co, ci, 3) + _vec2(f"encoder.{i + 1}", co)
    used += _lin("encoder.18", O, 256)
    return used, []


def _central_branch_params(branch, O):
    """One branch of CentralMultiModalEncoder alone under `encoder.` (ImageEncoderCentral / SpectrogramEncoderCentral):
    encoder.0 = the CentralUnimodal CNN (conv{k}, bn{k}; fc1 / fc2 unused), encoder.1 = Linear(flat, O) -> the embedding."""
    pre = f"{branch}_encoder."

    def take(specs):
        return [("encoder." + n[len(pre):], s) for n, s in specs if n.startswith(pre)]
    used, unused = central_encoder_params(O, O)
    return take(used), take(unused)


def image_central_params(O):
    return _central_branch_params("image", O)


def spectrogram_central_params(O):
    return _central_branch_params("audio", O)


def simple_multi_params(E, O, mix=None):
    """Parameter specs of SimpleMultiModalEncoder (models/dino.py:214-234: image_encoder() / audio_encoder() `nn.Sequential`s,
    :18-73, + the concatenation fusion) and its two subclasses: GatedMultiModalEncoder (:237-263, two scalar gates) and
    CrossAttentionMultiModalEncoder (:407-452, two CrossModalAttention blocks :385-405).  Every parameter receives gradients."""
    used = []
    for i, (ci, co) in zip((0, 4, 8), ((1, 32), (32, 64), (64, 128))):
        used += _conv(f"image_encoder.{i}", co, ci, 3) + _vec2(f"image_encoder.{i + 1}", co)
    used += _lin("image_encoder.14", E, 128)
    for i, (ci, co) in zip((0, 4, 8, 12), ((1, 32), (32, 64), (64, 128), (128, 256))):
        used += _conv(f"audio_encoder.{i}", co, ci, 3) + _vec2(f"audio_encoder.{i + 1}", co)
    used += _lin("audio_encoder.18", E, 256)
    used += _lin("fusion.0", E, 2 * E) + _lin("fusion.3", O, E)
    if mix == "gated":
        used += [("gate_image", ()), ("gate_audio", ())]
    elif mix == "cross":
        for a in ("image_to_audio_attention", "audio_to_image_attention"):
            used += _lin(f"{a}.q_proj", E, E) + _lin(f"{a}.kv_proj", 2 * E, E)
    return used, []


def head_params(in_dim, out_dim, hidden=512):
    return _lin("mlp.0", hidden, in_dim) + _vec2("mlp.1", hidden) + _lin("mlp.4", out_dim, hidden)


CENTRAL_IMAGE_LAYERS = [("image_encoder.0.conv1", "image_encoder.0.bn1", 1, 32, 28, 5, 2),
                        ("image_encoder.0.conv2", "image_encoder.0.bn2", 32, 64, 14, 5, 0)]
CENTRAL_AUDIO_LAYERS = [("audio_encoder.0.conv1", "audio_encoder.0.bn1", 1, 8, 112, 5, 2),
                        ("audio_encoder.0.conv2", "audio_encoder.0.bn2", 8, 16, 56, 5, 2),
                        ("audio_encoder.0.conv3", "audio_encoder.0.bn3", 16, 32, 28, 5, 2),
                        ("audio_encoder.0.conv4", "audio_encoder.0.bn4", 32, 64, 14, 5, 2)]
SIMPLE_IMAGE_LAYERS = [("encoder.0", "encoder.1", 1, 32, 28, 3, 1), ("encoder.4", "encoder.5", 32, 64, 14, 3, 1),
                       ("encoder.8", "encoder.9", 64, 128, 7, 3, 1)]
MULTI_SIMPLE_IMAGE_LAYERS = [("image_encoder.0", "image_encoder.1", 1, 32, 28, 3, 1), ("image_encoder.4", "image_encoder.5", 32, 64, 14, 3, 1),
                             ("image_encoder.8", "image_encoder.9", 64, 128, 7, 3, 1)]
MULTI_SIMPLE_AUDIO_LAYERS = [("audio_encoder.0", "audio_encoder.1", 1, 32, 112, 3, 1), ("audio_encoder.4", "audio_encoder.5", 32, 64, 56, 3, 1),
                             ("audio_encoder.8", "audio_encoder.9", 64, 128, 28, 3, 1), ("audio_encoder.12", "audio_encoder.13", 128, 256, 14, 3, 1)]
SPECTROGRAM_LAYERS = [("encoder.0", "encoder.1", 1, 32, 112, 3, 1), ("encoder.4", "encoder.5", 32, 64, 56, 3, 1),
                      ("encoder.8", "encoder.9", 64, 128, 28, 3, 1), ("encoder.12", "encoder.13", 128, 256, 14, 3, 1)]


def _reprefix(layers, old, new):
    return [(conv.replace(old, new, 1), bn.replace(old, new, 1), *geom) for conv, bn, *geom in layers]


# the unimodal CentralNet kinds: the branches of multi_central under `encoder.`
CENTRAL_IMAGE_UNI_LAYERS = _reprefix(CENTRAL_IMAGE_LAYERS, "image_encoder.", "encoder.")
CENTRAL_AUDIO_UNI_LAYERS = _reprefix(CENTRAL_AUDIO_LAYERS, "audio_encoder.", "encoder.")
# kind -> feature mixing between the encoders and the fusion MLP
MULTI_KINDS = {"multi_central": None, "multi_simple": None, "multi_simple_gated": "gated", "multi_cross_attention": "cross"}
# unimodal kind -> (modality stack, stack top, [(linear, input buffer, output buffer, output width)] after the top; the last output is
# the embedding `feat` that the projection head and the cosine-consistency term read).  The top is ("pool", W): global average pool to
# W features, or ("flat", W): the last pooled activation flattened to W = C*h*w features; either way the buffer "top" [N, W] holds them
UNI_KINDS = {"image_simple": ("img", ("pool", 128), [("enc.encoder.14", "top", "e14", 512), ("enc.projection.0", "e14", "feat", None)]),
             "spectrogram_simple": ("aud", ("pool", 256), [("enc.encoder.18", "top", "feat", None)]),
             "image_central": ("img", ("flat", 64 * 5 * 5), [("enc.encoder.1", "top", "feat", None)]),
             "spectrogram_central": ("aud", ("flat", 64 * 7 * 7), [("enc.encoder.1", "top", "feat", None)])}


class Arena:
    """A flat fp32 buffer with named views."""

    def __init__(self, spec, device, pad_to=4):
        self.spec = list(spec)
        self.offsets = {}
        off = 0
        for name, shape in self.spec:
            n = int(np.prod(shape))
            self.offsets[name] = (off, n, tuple(shape))
            off += (n + pad_to - 1) // pad_to * pad_to          # keep every tensor 16-byte aligned
        self.size = off
        self.flat = torch.zeros(max(off, 4), dtype=F32, device=device)

    def view(self, name, flat=None):
        off, n, shape = self.offsets[name]
        return (self.flat if flat is None else flat)[off:off + n].view(shape)

    def views(self, flat=None):
        return {name: self.view(name, flat) for name, _ in self.spec}

    def range_of(self, names):
        lo = min(self.offsets[n][0] for n in names)
        hi = max(self.offsets[n][0] + (self.offsets[n][1] + 3) // 4 * 4 for n in names)
        return lo, hi


class _BN:
    """Running statistics + per-step scale/shift/mean/invstd scratch of one BatchNorm layer."""

    def __init__(self, C, device):
        self.C = C
        self.running_mean = torch.zeros(C, device=device)
        self.running_var = torch.ones(C, device=device)
        self.num_batches_tracked = torch.zeros(1, dtype=torch.int64, device=device)


def _rows(x, n):
    """The first n rows of an optional input buffer."""
    return None if x is None else x[:n]


def _zero_arena(n, device):
    """Every accumulator of a workspace that must be zero when a step starts (BatchNorm statistics, backward sums, bias-gradient
    sums) lives in ONE float64 arena of n doubles: one memset per step instead of two dozen.  Returns (arena, zalloc), where
    zalloc(*shape) hands out the next 16-byte aligned view."""
    arena = torch.zeros(n, dtype=torch.float64, device=device)
    end = 0

    def zalloc(*shape):
        nonlocal end
        k = int(math.prod(shape))
        o, end = end, end + (k + 1) // 2 * 2
        if end > arena.numel():
            raise ops._lib.B200Error("zero arena too small")
        return arena[o:o + k].view(*shape)
    return arena, zalloc


class DinoStepEngine:
    """See module docstring.  kind: 'multi_central' (CentralMultiModalEncoder), 'multi_simple' (SimpleMultiModalEncoder),
    'multi_simple_gated' (GatedMultiModalEncoder), 'multi_cross_attention' (CrossAttentionMultiModalEncoder), 'image_simple'
    (ImageEncoder), 'spectrogram_simple' (SpectrogramEncoder), 'image_central' (ImageEncoderCentral) or 'spectrogram_central'
    (SpectrogramEncoderCentral); mode: 'default' | 'semi_supervised' | 'infonce' | 'mse' (multimodal
    kinds only).  The unimodal kinds have one conv stack; the methods that take (images, audios) ignore the absent modality's
    argument (it may be None) and allocate nothing for it."""

    def __init__(self, kind="multi_central", mode="default", encoder_output_dim=256, output_dim=256, projection_dim=128,
                 n_global_views=2, n_local_views=4, momentum=0.996, center_momentum=0.9, student_temperature=0.1,
                 teacher_temperature=0.04, learning_rate=1e-4, weight_decay=1e-6, dropout=0.3, fusion_dropout=0.3, alpha=1.0,
                 cosine_loss_alpha=0.0, augment_values=None, seed=0, device=None, process_group=None, data_parallel=None,
                 precision="bf16", fused_pool=True, fused_bnstat=False):
        if not torch.cuda.is_available():
            raise ops._lib.B200Error("DinoStepEngine needs a CUDA device: the hot path has no CPU fallback")
        ops._lib.load()
        self.device = torch.device(device if device is not None else f"cuda:{torch.cuda.current_device()}")
        assert kind in MULTI_KINDS or kind in UNI_KINDS
        self.multi = kind in MULTI_KINDS
        self.mix = MULTI_KINDS.get(kind)
        assert mode == "default" or self.multi
        assert precision in ("bf16", "fp32")
        self.precision = precision
        self.lin_tc = precision == "bf16"          # linear layers on the tensor cores (tcgen05 kind::tf32)
        self.kind, self.mode = kind, mode
        self.E, self.O, self.P = encoder_output_dim, output_dim, projection_dim
        self.Vg, self.Vl = n_global_views, n_local_views
        self.V = self.Vg + self.Vl
        self.momentum, self.center_momentum = momentum, center_momentum
        self.tau_s, self.tau_t = student_temperature, teacher_temperature
        self.lr, self.weight_decay = learning_rate, weight_decay
        self.dropout, self.fusion_dropout, self.alpha = dropout, fusion_dropout, alpha
        self.cosine_loss_alpha = cosine_loss_alpha
        self.seed = seed
        self.pg = process_group
        self.world = dp.world_size(process_group) if (data_parallel is None or data_parallel) else 1
        self.step_count = 0          # optimizer steps taken (Adam bias correction)
        self.rng_step = 0            # augmentation / dropout stream position
        self._loss_slots = [torch.zeros(1).pin_memory() for _ in range(2)]      # lagged loss read-back (train_step_host)
        self._loss_flip, self._loss_pending = 0, None
        self._ctr = None             # CUDA-graph mode: device counters int64 [rng_step, adam step] read by the kernels
        self._bc = None              #   ... and Adam's two bias corrections of the current step (device, fp32)
        self._graph = None

        # self.top[mod] = (global average pool before the linear?, linear input width, linear name)
        if kind == "multi_central":
            used, unused = central_encoder_params(self.E, self.O)
            self.img_layers, self.aud_layers = CENTRAL_IMAGE_LAYERS, CENTRAL_AUDIO_LAYERS
            self.top = {"img": (False, 1600, "enc.image_encoder.1"), "aud": (False, 3136, "enc.audio_encoder.1")}
        elif self.multi:
            used, unused = simple_multi_params(self.E, self.O, self.mix)
            self.img_layers, self.aud_layers = MULTI_SIMPLE_IMAGE_LAYERS, MULTI_SIMPLE_AUDIO_LAYERS
            self.top = {"img": (True, 128, "enc.image_encoder.14"), "aud": (True, 256, "enc.audio_encoder.18")}
        elif kind == "image_simple":
            used, unused = image_simple_params(self.O)
            self.img_layers, self.aud_layers = SIMPLE_IMAGE_LAYERS, []
            self.top = {}
        elif kind == "spectrogram_simple":
            used, unused = spectrogram_simple_params(self.O)
            self.img_layers, self.aud_layers = [], SPECTROGRAM_LAYERS
            self.top = {}
        elif kind == "image_central":
            used, unused = image_central_params(self.O)
            self.img_layers, self.aud_layers = CENTRAL_IMAGE_UNI_LAYERS, []
            self.top = {}
        else:
            used, unused = spectrogram_central_params(self.O)
            self.img_layers, self.aud_layers = [], CENTRAL_AUDIO_UNI_LAYERS
            self.top = {}
        # unimodal kinds: the modality of the one conv stack, its top and the layers between the top and the embedding
        self.uni = UNI_KINDS.get(kind)
        head = [("head." + n, s) for n, s in head_params(self.O, self.P)]
        enc_used = [("enc." + n, s) for n, s in used]
        enc_unused = [("enc." + n, s) for n, s in unused]
        aux = []
        if mode != "default":
            out = 10 if mode == "semi_supervised" else self.P
            for m in ("aux_image", "aux_audio"):
                aux += [(f"{m}.{n}", s) for n, s in head_params(self.E, out)]
        self.student = Arena(enc_used + head + enc_unused + aux, self.device)
        self.teacher = Arena(enc_used + head + enc_unused, self.device)
        self.n_ema = self.teacher.size
        self.n_trainable_prefix = self.student.range_of([n for n, _ in enc_used + head])[1]
        self.aux_range = self.student.range_of([n for n, _ in aux]) if aux else None
        self.grad_plan = dp.GradientPlan([(0, self.n_trainable_prefix)] + ([self.aux_range] if self.aux_range else []))
        self._grad_scale = 1.0
        self.grad = torch.zeros_like(self.student.flat)
        self.exp_avg = torch.zeros_like(self.student.flat)
        self.exp_avg_sq = torch.zeros_like(self.student.flat)
        self.S = self.student.views()
        self.T = self.teacher.views()
        self.G = self.student.views(self.grad)
        self.center = torch.zeros(1, self.P, device=self.device)
        # BatchNorm buffers
        self.bn_s, self.bn_t = {}, {}
        for conv, bn, ci, co, hw, k, pad in self.img_layers + self.aud_layers:
            self.bn_s["enc." + bn], self.bn_t["enc." + bn] = _BN(co, self.device), _BN(co, self.device)
        self.bn_s["head.mlp.1"], self.bn_t["head.mlp.1"] = _BN(512, self.device), _BN(512, self.device)
        for m in ("aux_image", "aux_audio"):
            if aux:
                self.bn_s[f"{m}.mlp.1"] = _BN(512, self.device)
        self._select_tc_layers(("s", "t"))
        # forward layers whose 2x2 max-pool runs inside the convolution's epilogue (the pooled extreme e, a quarter of z, goes to the
        # BatchNorm-apply kernel).  The epilogue pays for it with a per-tile barrier between its four warps (profiles/r2e_*): it wins
        # where no z is written at all (teacher, evaluation) and on the HBM-bound first audio layer of the student; the student's other
        # layers keep the z -> bn_relu_pool8_fwd path.  self.pool[role][mod][li]; role "t" also serves evaluation.
        # False: the round-1 path everywhere (A/B measurements).  The simple encoder family keeps it off: its layers are 32 - 256 channels
        # wide, and the per-tile barrier + the wider pooled rows cost the epilogue far more than the z read saves (first audio layer,
        # 32 channels at 112x112: 2.86 ms fused against 0.96 + 1.15 ms conv + pool pass; whole step 26.1 vs 25.1 ms, profiles/r2zf_*).
        # The unimodal CentralNet kinds run multi_central's layers and take its policy
        self.fused_pool = bool(fused_pool) and kind in ("multi_central", "image_simple", "image_central", "spectrogram_central")
        self.pool = {}
        for role in ("s", "t"):
            self.pool[role] = {mod: [self.fused_pool and bool(self.tc[mod][li]) and ops.conv_tc_pool_supported(ci, co, hw, hw, k, pad)
                                     and (role == "t" or (ci == 1 and hw >= 112))
                                     for li, (conv, bn, ci, co, hw, k, pad) in enumerate(layers)]
                               for mod, layers in (("img", self.img_layers), ("aud", self.aud_layers))}
        # data-gradient convolutions that also produce the BatchNorm-backward sums of the layer below in their epilogue (the separate
        # bn_pool8_bwd_reduce_p pass over p and dp disappears): layer li's data gradient serves layer li - 1.  Correct (tests) but OFF by
        # default: the four epilogue warps of these tensor-pipe-bound kernels have ~1.4x issue slack, the ~5 extra instructions per element
        # make the epilogue the bottleneck (16->8 @56^2: 0.32 -> 1.10 ms; step 7.66 -> 8.61 ms, profiles/r2k_*)
        self.fused_bnstat = bool(fused_bnstat)
        self.bnstat = {mod: [self.fused_bnstat and li > 0 and bool(self.tc[mod][li]) and bool(self.tc[mod][li - 1]) and
                             ops.conv_tc_dgrad_bnstat_supported(co, ci, hw + 2 * pad - k + 1, hw + 2 * pad - k + 1, k, k - 1 - pad)
                             for li, (conv, bn, ci, co, hw, k, pad) in enumerate(layers)]
                       for mod, layers in (("img", self.img_layers), ("aud", self.aud_layers))}
        self.overlap_teacher = True
        # all streams at the default priority: a high-priority main chain ends earlier but does not shorten the step, which is bound
        # by the total work of its kernels on a saturated GPU (DESIGN.md, "What the step is bound by")
        self._side_stream = torch.cuda.Stream(device=self.device)
        self._lin_wg_stream = torch.cuda.Stream(device=self.device)       # linear weight gradients
        self._lin_wg_pending = False
        self._side_stream2 = torch.cuda.Stream(device=self.device)
        self._wgrad_streams = {m: torch.cuda.Stream(device=self.device) for m in ("img", "aud")}
        self._aug_stream = torch.cuda.Stream(device=self.device)
        # data parallel: the exchange runs inside the C ABI (NCCL, b200_dp_*) on a communication stream beside the compute streams
        self.comm = dp.AbiComm.get(process_group) if self.world > 1 else None
        self._comm_stream = torch.cuda.Stream(device=self.device) if self.world > 1 else None
        self._center_ready = None          # event: the all-reduced centre EMA of the last step has landed
        self._comm_pending = False         # gradient all-reduces in flight on the communication stream
        self._prefetch, self._step_done, self._step_done_prev = None, None, None
        self._eval_wrole = "s"
        self._ws = {}
        self._init_parameters()
        self.set_augmentation(augment_values)

    def _select_tc_layers(self, roles):
        """self.tc[mod][li]: does conv layer li of a stack run on the tensor cores (tcgen05, bf16 act8 activations, fp32 accumulate)?
        Every convolution whose forward and (for C_in > 1) flipped data gradient the library supports, on the bf16 path.  Allocates
        the bf16 weight images of those layers for each role in `roles` and, for C_in > 1, the flipped image of the data gradient."""
        self.tc, self._tcw, self._prep_desc = {}, {}, {}
        for mod, layers in (("img", self.img_layers), ("aud", self.aud_layers)):
            tc = [self.precision == "bf16" and ops.conv_tc_supported(ci, co, hw, hw, k, pad) and
                  (ci == 1 or ops.conv_tc_supported(co, ci, hw + 2 * pad - k + 1, hw + 2 * pad - k + 1, k, k - 1 - pad))
                  for (conv, bn, ci, co, hw, k, pad) in layers]
            # a tensor-core first layer runs its backward fused into the weight-gradient kernel (dz stays in shared memory),
            # which consumes the bf16 act8 pooled gradient written by the second layer's tensor-core data gradient
            if tc and tc[0] and not (len(tc) > 1 and tc[1]):
                tc[0] = False
            self.tc[mod] = tc
            for li, (conv, bn, ci, co, hw, k, pad) in enumerate(layers):
                if tc[li]:
                    for role in roles:
                        self._tcw[(role, mod, li)] = torch.empty(ops.conv_tc_weight_bytes(ci, co, k), dtype=torch.uint8, device=self.device)
                    if ci > 1:
                        self._tcw[("flip", mod, li)] = torch.empty(ops.conv_tc_weight_bytes(co, ci, k), dtype=torch.uint8, device=self.device)

    # ------------------------------------------------------------------------------------------------------
    def _init_parameters(self):
        """PyTorch default init (kaiming_uniform(a=sqrt 5) == U(-1/sqrt(fan_in), 1/sqrt(fan_in)) for weights and biases,
        BatchNorm weight 1 / bias 0); the teacher starts as a copy of the student (models/dino.py:617, 627)."""
        g = torch.Generator(device="cpu").manual_seed(self.seed)
        bn_bases = {"enc." + bn for _, bn, *_ in self.img_layers + self.aud_layers} | {"head.mlp.1", "aux_image.mlp.1", "aux_audio.mlp.1"}
        bounds = {}
        for name, shape in self.student.spec:
            v = self.student.view(name)
            base = name.rsplit(".", 1)[0]
            if base in bn_bases:
                v.fill_(1.0 if name.endswith(".weight") else 0.0)
            elif len(shape) == 0:
                v.fill_(0.5)                  # gate_image / gate_audio (models/dino.py:242-243)
            elif len(shape) > 1:
                bounds[base] = 1.0 / math.sqrt(int(np.prod(shape[1:])))
                v.copy_(((torch.rand(shape, generator=g) * 2 - 1) * bounds[base]).to(self.device))
            else:
                v.copy_(((torch.rand(shape, generator=g) * 2 - 1) * bounds[base]).to(self.device))
        self.sync_teacher()

    def sync_teacher(self):
        self.teacher.flat.copy_(self.student.flat[:self.n_ema])
        for k in self.bn_t:
            self.bn_t[k].running_mean.copy_(self.bn_s[k].running_mean)
            self.bn_t[k].running_var.copy_(self.bn_s[k].running_var)
            self.bn_t[k].num_batches_tracked.copy_(self.bn_s[k].num_batches_tracked)

    def load_named(self, student=None, teacher=None, student_head=None, teacher_head=None, aux_image=None, aux_audio=None):
        """Copy tensors given by reference names (e.g. 'image_encoder.0.conv1.weight', 'mlp.0.weight') into the arenas."""
        for prefix, arena_views, src in (("enc.", self.S, student), ("enc.", self.T, teacher), ("head.", self.S, student_head),
                                         ("head.", self.T, teacher_head), ("aux_image.", self.S, aux_image), ("aux_audio.", self.S, aux_audio)):
            if src is None:
                continue
            for k, v in src.items():
                if prefix + k in arena_views:
                    arena_views[prefix + k].copy_(v.to(self.device))

    def set_augmentation(self, augment_values):
        ig, il = A.image_chains()
        ag, al = A.default_audio_chains() if augment_values is None else A.audio_chains_from_values(augment_values)
        self.chains = (ig, il, ag, al)
        spec = np.stack([A.pack_spec(c) for c in self.chains])
        self.aug_spec = torch.from_numpy(spec).to(self.device)

    # ------------------------------------------------------------------------------------------------------
    def _workspace(self, B):
        if B in self._ws:
            return self._ws[B]
        dev, V, Vg = self.device, self.V, self.Vg
        if self.world > 1:
            # the gradient average (sum / world) and the centre mean (rows * world) assume equal per-rank batches: refuse otherwise
            lohi = torch.tensor([B, -B], dtype=torch.int64, device=dev)
            torch.distributed.all_reduce(lohi, op=torch.distributed.ReduceOp.MAX, group=self.pg)
            if int(lohi[0]) != B or int(-lohi[1]) != B:
                raise ops._lib.B200Error(f"data parallel: per-rank batch sizes differ ({int(-lohi[1])}..{int(lohi[0])}); use equal shards "
                                         "(drop_last) -- the gradient average and the centre EMA weight every rank equally")
        extra = 1 if self.mode != "default" else 0
        Ns, Nt = (V + extra) * B, Vg * B

        def e(*shape, dtype=F32):
            return torch.empty(*shape, dtype=dtype, device=dev)

        w = {"B": B, "Ns": Ns, "Nt": Nt}
        w["zarena"], zalloc = _zero_arena(1 << 17, dev)
        # augmentation (the sampler always draws the audio records; the image records only when there is an image stack)
        if self.img_layers:
            w["img_ops"] = torch.zeros(B, V, A.MAX_OPS, A.OP_WORDS, dtype=torch.int32, device=dev)
        w["aud_ops"] = torch.zeros(B, V, A.MAX_OPS, A.OP_WORDS, dtype=torch.int32, device=dev)
        w["group_bits"] = torch.zeros(B, V, A.GROUP_WORDS, dtype=torch.int32, device=dev)
        for nm in ("img_ops", "aud_ops", "group_bits"):
            if nm in w:
                w[nm + "_b"] = torch.zeros_like(w[nm])
        if self.img_layers:
            w["x_img"] = e(Ns, 1, 28, 28)
        if self.aud_layers:
            w["x_aud"] = e(Ns, 1, 112, 112)
        self._stack_buffers(w, "s", Ns, B, e, zalloc)
        self._stack_buffers(w, "t", Nt, B, e, zalloc)
        for m in ("img", "aud"):             # the spare first-layer input that prefetch_augment fills with the next step's views
            if f"{m}.xs8" in w:
                w[f"{m}.xs8_b"] = torch.empty_like(w[f"{m}.xs8"])
        E, O, P = self.E, self.O, self.P
        Nv = V * B
        if self.multi:
            for role, N, nfus in (("s", Ns, Nv), ("t", Nt, Nt)):
                self._mix_workspace(w, role, N, nfus, B, e)
                w[f"{role}.h1"] = e(nfus, E)
                w[f"{role}.feat"] = e(nfus, O)
                w[f"{role}.fmask"] = torch.ones(nfus, E, dtype=torch.uint8, device=dev)
                for mod, layers in (("img", self.img_layers), ("aud", self.aud_layers)):
                    if self.top[mod][0]:
                        w[f"{role}.{mod}.gap"] = e(N, self.top[mod][1])
            w["d.cat"] = e(Ns, 2 * E)
            w["d.catr"] = e(Ns, 2 * E) if self.mix else w["d.cat"]       # gradient w.r.t. the un-mixed encoder features
            w["d.h1"] = e(Nv, E)
            for mod in ("img", "aud"):
                if self.top[mod][0]:
                    w[f"d.{mod}.gap"] = e(Ns, self.top[mod][1])
            if self.mix == "gated":
                w["gate_work"] = torch.zeros(ops.gate_grad_work_floats(), device=dev)
            elif self.mix == "cross":
                w["att.dA"] = e(B, B)
                w["att.tmp"] = e(Nv, E)
                for mi in (0, 1):
                    for nm in ("dq", "dk", "dv"):
                        w[f"att{mi}.{nm}"] = e(Nv, E)
        else:
            for role, N in (("s", Ns), ("t", Nt)):
                self._uni_workspace(w, role, N, e)
            self._uni_workspace(w, "d", Ns, e, with_feat=False)
        w["d.feat"] = e(Nv, O)
        for role, N in (("s", Nv), ("t", Nt)):
            w[f"{role}.hh"] = e(N, 512)
            w[f"{role}.g"] = e(N, 512)
            w[f"{role}.proj"] = e(N, P)
            w[f"{role}.hstats"] = zalloc(512, 2)
            for nm in ("hscale", "hshift", "hmean", "hinvstd"):
                w[f"{role}.{nm}"] = e(1, 512)
        w["s.hmask"] = torch.ones(Nv, 512, dtype=torch.uint8, device=dev)
        w["s.hsums"] = zalloc(512, 2)
        w["d.proj"], w["d.g"], w["d.hh"] = e(Nv, P), e(Nv, 512), e(Nv, 512)
        parts = ops.dino_loss_parts(B)
        w["part_loss"], w["part_colsum"] = e(parts), e(parts, P)
        w["t_colmean"] = e(Vg, P)
        w["colsum"] = e(P + 1)
        w["loss"] = torch.zeros(4, device=dev)             # [dino, aux, cosine, total]
        w["loss_work"] = torch.zeros(int(ops._lib_().b200_loss_work_floats(B)), device=dev)    # partials of the fixed-order loss sums
        if self.mode != "default":
            out = 10 if self.mode == "semi_supervised" else P
            for m in ("aux_image", "aux_audio"):
                w[f"{m}.hh"], w[f"{m}.g"], w[f"{m}.out"] = e(B, 512), e(B, 512), e(B, out)
                w[f"{m}.d.out"], w[f"{m}.d.g"], w[f"{m}.d.hh"] = e(B, out), e(B, 512), e(B, 512)
                w[f"{m}.hstats"] = zalloc(512, 2)
                w[f"{m}.hsums"] = zalloc(512, 2)
                for nm in ("hscale", "hshift", "hmean", "hinvstd"):
                    w[f"{m}.{nm}"] = e(1, 512)
            if self.mode == "infonce":
                w["infonce_work"] = e(ops.infonce_work_floats(B, P, tc=self.lin_tc))
        if not self.multi or self.cosine_loss_alpha > 0:
            w["d.emb"] = e(Nv, O)          # cosine-consistency gradient (UniModalDINO, cosine_loss_alpha may be switched on later)
        self._ws[B] = w
        return w

    def _stack_buffers(self, w, role, N, B, e, zalloc):
        """The buffers both conv stacks need for one role ('s' student, 't' teacher, 'e' evaluation; 'e' follows the teacher's
        pool table) on N = views * B samples.  Per layer: the pooled window extreme e where the forward pools in the conv epilogue,
        the conv output z (unless a pooled layer of a role without backward), the pooled activation (act8 p8 when the next layer
        reads it on the tensor cores, fp32 NCHW p otherwise), the BatchNorm statistics (zalloc, per view-call) and the affine /
        normalisation vectors.  Roles 's' and 'e' also get the first-layer quad8 input xs8 (the teacher reads a prefix of the
        student's); the student gets the backward sums and one backward scratch set per stack (the two stacks' backward passes
        run on different streams)."""
        BF = torch.bfloat16
        nv = N // B
        pool = self.pool["s" if role == "s" else "t"]
        for mod, layers in (("img", self.img_layers), ("aud", self.aud_layers)):
            sc = dict(wg=0, z=0, p=0, z8=0)
            for li, (conv, bn, ci, co, hw, k, pad) in enumerate(layers):
                ho = hw + 2 * pad - k + 1
                tc = self.tc[mod][li]
                next_tc = li + 1 < len(layers) and self.tc[mod][li + 1]
                if tc and ci == 1 and role != "t":
                    w[f"{mod}.xs8"] = e(N, hw, ops.quad8_width(hw, pad), 8, dtype=BF)
                pooled = tc and pool[mod][li]
                if pooled:
                    w[f"{role}.{mod}.e{li}"] = e(N, co // 8, ho // 2, ho // 2, 8, dtype=torch.float16)     # 2x2 window extreme of z
                if tc and (role == "s" or not pooled):
                    w[f"{role}.{mod}.z{li}"] = e(N, co // 8, ho, ho, 8, dtype=torch.float16)   # act8 layout, fp16: never an MMA operand
                elif not tc:
                    w[f"{role}.{mod}.z{li}"] = e(N, co, ho, ho)
                if next_tc:
                    w[f"{role}.{mod}.p8{li}"] = e(N, co // 8, ho // 2, ho // 2, 8, dtype=BF)
                if not next_tc or not tc:
                    w[f"{role}.{mod}.p{li}"] = e(N, co, ho // 2, ho // 2)
                w[f"{role}.{mod}.stats{li}"] = zalloc(nv, co, 2)
                for nm in ("scale", "shift", "mean", "invstd"):
                    w[f"{role}.{mod}.{nm}{li}"] = e(nv, co)
                if role != "s":
                    continue
                w[f"s.{mod}.sums{li}"] = zalloc(nv, co, 2)
                if tc:
                    sc["wg"] = max(sc["wg"], ops.conv_tc_wgrad_work_floats(N, ci, co, hw, hw, k, pad))
                    if ci == 1:
                        # fused apply + weight gradient: this layer's dz never exists in HBM
                        sc["wg"] = max(sc["wg"], ops.conv_tc_wgrad_l0_fused_work_floats(N, B, co, hw, hw, k, pad))
                    else:
                        sc["z8"] = max(sc["z8"], N * co * ho * ho)
                else:
                    sc["wg"] = max(sc["wg"], ops.conv_bwd_weight_work_floats(N, ci, co, hw, hw, k, pad))
                    sc["z"] = max(sc["z"], N * co * ho * ho)
                sc["p"] = max(sc["p"], N * co * (ho // 2) * (ho // 2), N * ci * hw * hw if li > 0 else 0)
            if role == "s" and layers:
                w[f"{mod}.dz"] = e(max(sc["z"], 4))
                w[f"{mod}.dz8"] = e(max(sc["z8"], 8), dtype=BF)
                w[f"{mod}.dz8b"] = e(max(sc["z8"], 8), dtype=BF)      # second buffer: the weight gradient of layer l overlaps layer l-1
                w[f"{mod}.dbsum"] = zalloc(8, 256)
                w[f"{mod}.dp_a"], w[f"{mod}.dp_b"] = e(sc["p"]), e(sc["p"])
                w[f"{mod}.wg_work"] = e(max(sc["wg"], 4))
                w[f"{mod}.wg_work_b"] = e(max(sc["wg"], 4))

    def _uni_workspace(self, w, role, N, e, with_feat=True):
        """Unimodal kinds: the stack's top features "top" [N, W] and the outputs of the linears after it (`feat` [N, O] last).  An
        average-pool top has its own buffer; a flatten top is a view of the last pooled activation (role "d": of the gradient buffer
        dp_a that the stack's backward starts from, so that the first linear's data gradient lands there directly)."""
        mod, (top, width), chain = self.uni
        if top == "pool":
            w[f"{role}.top"] = e(N, width)
        elif role == "d":
            w["d.top"] = w[f"{mod}.dp_a"][:N * width].view(N, width)
        else:
            w[f"{role}.top"] = w[f"{role}.{mod}.p{len(self._layers(mod)) - 1}"].view(N, width)
        for lin, src, dst, cols in chain:
            if dst != "feat" or with_feat:
                w[f"{role}.{dst}"] = e(N, self.O if cols is None else cols)

    def _mix_workspace(self, w, role, N, nfus, B, e):
        """Encoder-feature buffers of one role: catr [N, 2E] = (image | audio) features as the encoders' linears produce them, cat =
        the fusion MLP's input (the same tensor, or for the gated / cross-attention encoders the mixed features of the nfus rows)."""
        E = self.E
        w[f"{role}.catr"] = e(N, 2 * E)
        w[f"{role}.cat"] = e(nfus, 2 * E) if self.mix else w[f"{role}.catr"]
        if self.mix == "cross":
            for mi in (0, 1):
                for nm in ("q", "k", "v"):
                    w[f"{role}.att{mi}.{nm}"] = e(nfus, E)
                w[f"{role}.att{mi}.A"] = e(nfus // B, B, B)          # attention weights over the batch of each view-call

    # the two CrossModalAttention blocks: (module name, columns of x1 (queries, residual), columns of x2 (keys / values))
    def _att_blocks(self):
        E = self.E
        return (("image_to_audio_attention", slice(0, E), slice(E, 2 * E)), ("audio_to_image_attention", slice(E, 2 * E), slice(0, E)))

    def _mix_fwd(self, w, role, P, nfus, B):
        """Encoder features -> fusion input.  Gated (models/dino.py:249-261): sigmoid(gate) * features per modality.  Cross attention
        (models/dino.py:393-405, 436-442): per view-call, out = x1 + softmax((x1 Wq)(x2 Wk)^T / sqrt(E)) (x2 Wv) for (image, audio)
        and (audio, image); the attention runs over the BATCH dimension of one encoder call."""
        if not self.mix:
            return
        E = self.E
        catr, cat = w[f"{role}.catr"], w[f"{role}.cat"]
        if self.mix == "gated":
            ops.gate_apply(catr[:nfus, :E], P["enc.gate_image"], cat[:, :E])
            ops.gate_apply(catr[:nfus, E:], P["enc.gate_audio"], cat[:, E:])
            return
        scale = float(E) ** -0.5
        for mi, (name, c1, c2) in enumerate(self._att_blocks()):
            x1, x2 = catr[:nfus, c1], catr[:nfus, c2]
            Wq, bq = P[f"enc.{name}.q_proj.weight"], P[f"enc.{name}.q_proj.bias"]
            Wkv, bkv = P[f"enc.{name}.kv_proj.weight"], P[f"enc.{name}.kv_proj.bias"]
            q, k, v, A = (w[f"{role}.att{mi}.{nm}"] for nm in ("q", "k", "v", "A"))
            ops.linear_fwd(x1, Wq, bq, q, tc=self.lin_tc)
            ops.linear_fwd(x2, Wkv[:E], bkv[:E], k, tc=self.lin_tc)
            ops.linear_fwd(x2, Wkv[E:], bkv[E:], v, tc=self.lin_tc)
            for vv in range(nfus // B):
                r = slice(vv * B, (vv + 1) * B)
                ops.linear_fwd(q[r], k[r], None, A[vv], tc=self.lin_tc)            # q k^T
                ops.softmax_rows(A[vv], scale)
                ops.linear_bwd_data(A[vv], v[r], cat[r, c1], tc=self.lin_tc)       # attn v
                ops.add2d(cat[r, c1], x1[r])                                       # + x1

    def _mix_bwd(self, w, Nv, B):
        """d.cat[:Nv] (gradient w.r.t. the fusion input) -> d.catr[:Nv] (gradient w.r.t. the encoder features) + the gradients of
        the gates / attention projections."""
        if not self.mix:
            return
        E, S, G = self.E, self.S, self.G
        catr, d_cat, d_catr = w["s.catr"], w["d.cat"], w["d.catr"]
        if self.mix == "gated":
            for gname, c in (("enc.gate_image", slice(0, E)), ("enc.gate_audio", slice(E, 2 * E))):
                ops.gate_grad(d_cat[:Nv, c], catr[:Nv, c], S[gname], G[gname], w["gate_work"])
                ops.gate_apply(d_cat[:Nv, c], S[gname], d_catr[:Nv, c])
            return
        scale = float(E) ** -0.5
        d_catr[:Nv].copy_(d_cat[:Nv])                                               # the residual paths
        dA, tmp = w["att.dA"], w["att.tmp"]
        for mi, (name, c1, c2) in enumerate(self._att_blocks()):
            x1, x2, d_out = catr[:Nv, c1], catr[:Nv, c2], d_cat[:Nv, c1]
            Wq, Wkv = S[f"enc.{name}.q_proj.weight"], S[f"enc.{name}.kv_proj.weight"]
            q, k, v, A = (w[f"s.att{mi}.{nm}"] for nm in ("q", "k", "v", "A"))
            dq, dk, dv = (w[f"att{mi}.{nm}"] for nm in ("dq", "dk", "dv"))
            for vv in range(Nv // B):
                r = slice(vv * B, (vv + 1) * B)
                ops.linear_fwd(d_out[r], v[r], None, dA, tc=self.lin_tc)            # d attn = d_out v^T
                ops.linear_bwd_weight(A[vv], d_out[r], dv[r], None, tc=self.lin_tc)  # d v = attn^T d_out
                ops.softmax_rows_bwd(dA, A[vv], scale)                              # d (q k^T)
                ops.linear_bwd_data(dA, k[r], dq[r], tc=self.lin_tc)                # d q = dS k
                ops.linear_bwd_weight(dA, q[r], dk[r], None, tc=self.lin_tc)        # d k = dS^T q
            gq, gkv = G[f"enc.{name}.q_proj.weight"], G[f"enc.{name}.kv_proj.weight"]
            gbq, gbkv = G[f"enc.{name}.q_proj.bias"], G[f"enc.{name}.kv_proj.bias"]
            for dy, x, wt, gw, gb, c in ((dq, x1, Wq, gq, gbq, c1), (dk, x2, Wkv[:E], gkv[:E], gbkv[:E], c2),
                                         (dv, x2, Wkv[E:], gkv[E:], gbkv[E:], c2)):
                self._lin_wgrad(dy, x, gw, gb)
                ops.linear_bwd_data(dy, wt, tmp, tc=self.lin_tc)
                ops.add2d(d_catr[:Nv, c], tmp)

    # ------------------------------------------------------------------------------------------------------
    # augmentation
    # ------------------------------------------------------------------------------------------------------
    def _batch_size(self, images, audios):
        """B of a raw batch, read from the modality the kind encodes first (the image batch, or the audio batch of an audio-only kind)."""
        x = images if self.img_layers else audios
        if x is None:
            raise ops._lib.B200Error(f"{self.kind}: the {'image' if self.img_layers else 'audio'} batch is required")
        return x.shape[0]

    def _direct_views(self):
        """Can the augmentation write the first-layer quad8 operands directly?  (Every stack's first layer is a tensor-core layer.)"""
        return all(self.tc[m][0] for m, layers in (("img", self.img_layers), ("aud", self.aud_layers)) if layers)

    def prefetch_augment(self, images, audios):
        """Enqueue the NEXT step's sampling + augmentation on the augmentation stream, into the spare first-layer buffers, so
        that it overlaps the tail of the current step (its last weight gradient, EMA, Adam).  The next train_step() on the
        same tensors picks the views up instead of augmenting again.  Tensor-core path only; a no-op otherwise."""
        if not self._direct_views():
            return False
        B = self._batch_size(images, audios)
        w = self._workspace(B)
        main, st = torch.cuda.current_stream(), self._aug_stream
        if self._step_done_prev is not None:
            st.wait_event(self._step_done_prev)       # the spare slot was last read by the step BEFORE the one in flight
        with torch.cuda.stream(st):
            ops.aug_sample(self.aug_spec, B, self.Vg, self.Vl, self.seed, self.rng_step, w.get("img_ops_b"), w["aud_ops_b"], w["group_bits_b"])
            seed = (self.seed * 1000003 + self.rng_step) & 0xFFFFFFFFFFFF
            V = self.V
            if self.img_layers:
                pi = self.img_layers[0][6]
                ops.aug_apply_image(images.reshape(B, 28, 28), w["img_ops_b"], None, out8=w["img.xs8_b"][:V * B].view(V, B, 28, ops.quad8_width(28, pi), 8),
                                    pad=pi)
            if self.aud_layers and audios is not None:
                pa = self.aud_layers[0][6]
                ops.aug_apply_audio(audios.reshape(B, 112, 112), w["aud_ops_b"], w["group_bits_b"], None, seed=seed,
                                    out8=w["aud.xs8_b"][:V * B].view(V, B, 112, ops.quad8_width(112, pa), 8), pad=pa)
            ev = torch.cuda.Event()
            ev.record(st)
        self._prefetch = {"key": self._batch_key(images, audios), "event": ev}
        return True

    def _batch_key(self, images, audios):
        img = images if self.img_layers else None            # an audio-only kind ignores the image batch
        return (None if img is None else img.data_ptr(), None if audios is None else audios.data_ptr(), self._batch_size(images, audios),
                self.rng_step)

    def _take_prefetched(self, images, audios):
        """If the views of this batch were prefetched for this rng position: swap the buffer slots and return them."""
        pf, self._prefetch = self._prefetch, None
        if pf is None or pf["key"] != self._batch_key(images, audios):
            return None
        B = self._batch_size(images, audios)
        w = self._workspace(B)
        torch.cuda.current_stream().wait_event(pf["event"])
        for nm in ("img.xs8", "aud.xs8", "img_ops", "aud_ops", "group_bits"):
            if nm in w:
                w[nm], w[nm + "_b"] = w[nm + "_b"], w[nm]
        V = self.V
        xi = w["img.xs8"][:V * B].view(V, B, 28, ops.quad8_width(28, self.img_layers[0][6]), 8) if self.img_layers else None
        xa = w["aud.xs8"][:V * B].view(V, B, 112, ops.quad8_width(112, self.aud_layers[0][6]), 8) if self.aud_layers else None
        return xi, xa

    def augment(self, images, audios, B=None, direct=False):
        """Device-sampled multi-crop views of a raw batch: images [B,28,28] (fp32 in [0,1] or uint8),
        audios [B,112,112] (uint8 or fp32).  Returns view-major tensors ([V,B,28,28], [V,B,112,112]); None for a modality the
        kind does not encode."""
        B = self._batch_size(images, audios)
        w = self._workspace(B)
        step, step_dev = self._step_args()
        ops.aug_sample(self.aug_spec, B, self.Vg, self.Vl, self.seed, step, w.get("img_ops"), w["aud_ops"], w["group_bits"], step_dev=step_dev)
        return self.augment_with_params(images, audios, w.get("img_ops"), w["aud_ops"], w["group_bits"], None, direct=direct)

    def _step_args(self):
        """(host step value, device step counter) for the kernels that consume the RNG stream position: eager mode passes the
        host counter, CUDA-graph mode 0 + a pointer to the device counter (identical streams either way)."""
        return (0, self._ctr[0:1]) if self._ctr is not None else (self.rng_step, None)

    def augment_with_params(self, images, audios, img_ops, aud_ops, group_bits, noise, direct=False):
        """Applies the op records.  direct=False: fp32 views ([V,B,28,28], [V,B,112,112]).  direct=True (tensor-core path
        only): the kernels write the first-layer quad8 images straight into the workspace (no fp32 round trip); the
        returned bf16 tensors are those workspace buffers and are recognised by forward_pass."""
        B = self._batch_size(images, audios)
        w = self._workspace(B)
        V = self.V
        step, step_dev = self._step_args()
        seed = (self.seed * 1000003 + step) & 0xFFFFFFFFFFFF
        if direct and self._direct_views():
            xi = xa = None
            if self.img_layers:
                pi = self.img_layers[0][6]
                xi = w["img.xs8"][:V * B].view(V, B, 28, ops.quad8_width(28, pi), 8)
                ops.aug_apply_image(images.reshape(B, 28, 28), img_ops, None, out8=xi, pad=pi)
            if self.aud_layers and audios is not None:
                pa = self.aud_layers[0][6]
                xa = w["aud.xs8"][:V * B].view(V, B, 112, ops.quad8_width(112, pa), 8)
                ops.aug_apply_audio(audios.reshape(B, 112, 112), aud_ops, group_bits, None, noise=noise, seed=seed, out8=xa, pad=pa,
                                    step_dev=step_dev)
            return xi, xa
        xi = xa = None
        if self.img_layers:
            xi = w["x_img"][:V * B].view(V, B, 28, 28)
            ops.aug_apply_image(images.reshape(B, 28, 28), img_ops, xi)
        if self.aud_layers and audios is not None:
            xa = w["x_aud"][:V * B].view(V, B, 112, 112)
            ops.aug_apply_audio(audios.reshape(B, 112, 112), aud_ops, group_bits, xa, noise=noise, seed=seed, step_dev=step_dev)
        return xi, xa

    # ------------------------------------------------------------------------------------------------------
    # forward building blocks
    # ------------------------------------------------------------------------------------------------------
    def _prep_tc_weights(self, role, P):
        """fp32 conv weights -> the bf16 operand images of the tensor-core convolutions (weights change every step): ONE launch
        over a device table of (weight, image, Cin, Cout, K, flip) records, built once per role (the arenas never move)."""
        desc = self._prep_desc.get(role)
        if desc is None:
            rows = []
            for mod, layers in (("img", self.img_layers), ("aud", self.aud_layers)):
                for li, (conv, bn, ci, co, hw, k, pad) in enumerate(layers):
                    if self.tc[mod][li]:
                        wt = P["enc." + conv + ".weight"]
                        rows.append([wt.data_ptr(), self._tcw[(role, mod, li)].data_ptr(), ci, co, k, 0])
                        if role == "s" and ci > 1:       # data gradient: channels swapped, taps mirrored
                            rows.append([wt.data_ptr(), self._tcw[("flip", mod, li)].data_ptr(), co, ci, k, 1])
            desc = torch.tensor(rows, dtype=torch.int64, device=self.device) if rows else False
            self._prep_desc[role] = desc
        if desc is not False:
            ops.conv_tc_prep_weights_multi(desc)

    def _conv_stack(self, w, role, mod, layers, x, N, B, P, bns, train=True):
        """conv -> BatchNorm(batch statistics per view-call) -> ReLU -> MaxPool2 for every layer; tensor-core layers keep
        z and the pooled activation in bf16 act8, the others in fp32 NCHW.  Returns the last pooled activation (fp32)."""
        nv = N // B
        cur = x
        for li, (conv, bn, ci, co, hw, k, pad) in enumerate(layers):
            z, stats = w.get(f"{role}.{mod}.z{li}"), w[f"{role}.{mod}.stats{li}"]
            tc = self.tc[mod][li]
            next_tc = li + 1 < len(layers) and self.tc[mod][li + 1]
            pooled = tc and self.pool["s" if role == "s" else "t"][mod][li]
            wrole = role if role in ("s", "t") else self._eval_wrole      # the evaluation role "e" borrows a role's weight images
            if tc:
                xin = cur
                if ci == 1:
                    xs8 = w[f"{mod}.xs8"]
                    if role == "s" and not w.get("packed", False):
                        ops.pack_quad8(cur.view(N, hw, hw), xs8, pad)
                    xin = xs8[:N]
                if pooled:      # conv + statistics + window extreme in one kernel; only the student keeps z (for its backward)
                    ops.conv_tc_pool(xin, self._tcw[(wrole, mod, li)], P["enc." + conv + ".bias"], P["enc." + bn + ".weight"],
                                     z if role == "s" else None, w[f"{role}.{mod}.e{li}"], stats, B, co, k, pad)
                else:
                    ops.conv_tc(xin, self._tcw[(wrole, mod, li)], P["enc." + conv + ".bias"], z, stats, B, co, k, pad)
            else:
                ops.conv_fwd(cur.view(N, ci, hw, hw), P["enc." + conv + ".weight"], P["enc." + conv + ".bias"], z, stats, B, pad)
            b = bns["enc." + bn]
            ho = hw + 2 * pad - k + 1
            sc, sh = w[f"{role}.{mod}.scale{li}"], w[f"{role}.{mod}.shift{li}"]
            ops.bn_finalize(stats, P["enc." + bn + ".weight"], P["enc." + bn + ".bias"], b.running_mean, b.running_var,
                            b.num_batches_tracked, sc, sh, w[f"{role}.{mod}.mean{li}"], w[f"{role}.{mod}.invstd{li}"], nv, B * ho * ho, train=train)
            if tc:
                cur = w[f"{role}.{mod}.p8{li}"] if next_tc else w[f"{role}.{mod}.p{li}"]
                if pooled:
                    ops.bn_relu_apply8(w[f"{role}.{mod}.e{li}"], sc, sh, cur, B)
                else:
                    ops.bn_relu_pool8_fwd(z, sc, sh, cur, B)
            else:
                cur = w[f"{role}.{mod}.p{li}"]
                ops.bn_relu_pool_fwd(z, sc, sh, cur, B)
                if next_tc:
                    ops.pack_act8(cur, w[f"{role}.{mod}.p8{li}"])
                    cur = w[f"{role}.{mod}.p8{li}"]
        return cur

    def _head_fwd(self, w, role, prefix, P, bn, x, out, hh, g, mask, drop_p, tag=""):
        M = x.shape[0]
        ops.linear_fwd(x, P[prefix + "mlp.0.weight"], P[prefix + "mlp.0.bias"], hh, tc=self.lin_tc)
        st = w[f"{role}.{tag}hstats"]
        ops.colstats(hh, st)
        ops.bn_finalize(st, P[prefix + "mlp.1.weight"], P[prefix + "mlp.1.bias"], bn.running_mean, bn.running_var, bn.num_batches_tracked,
                        w[f"{role}.{tag}hscale"], w[f"{role}.{tag}hshift"], w[f"{role}.{tag}hmean"], w[f"{role}.{tag}hinvstd"], 1, M)
        ops.bn1d_gelu_drop_fwd(hh, w[f"{role}.{tag}hscale"], w[f"{role}.{tag}hshift"], mask, drop_p, g)
        ops.linear_fwd(g, P[prefix + "mlp.4.weight"], P[prefix + "mlp.4.bias"], out, tc=self.lin_tc)

    def _lin_wgrad(self, dy, x, gw, gb):
        """Weight / bias gradient of a linear layer.  Nothing in the backward chain depends on it, so it runs on its own stream
        beside the data gradients (dy and x are not written again in this step; backward_pass joins the stream at its end)."""
        st = self._lin_wg_stream if self.overlap_teacher else None
        if st is None:
            ops.linear_bwd_weight(dy, x, gw, gb, tc=self.lin_tc)
            return
        st.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(st):
            ops.linear_bwd_weight(dy, x, gw, gb, tc=self.lin_tc)
        self._lin_wg_pending = True

    def _head_bwd(self, w, role, prefix, x, d_out, hh, g, d_g, d_hh, d_x, mask, drop_p, tag=""):
        S, G = self.S, self.G
        self._lin_wgrad(d_out, g, G[prefix + "mlp.4.weight"], G[prefix + "mlp.4.bias"])
        ops.linear_bwd_data(d_out, S[prefix + "mlp.4.weight"], d_g, tc=self.lin_tc)
        sums = w[f"{role}.{tag}hsums"]
        sc, sh, mu, inv = (w[f"{role}.{tag}h{n}"] for n in ("scale", "shift", "mean", "invstd"))
        ops.bn1d_gelu_drop_bwd_reduce(hh, d_g, sc, sh, mu, inv, mask, drop_p, sums)
        ops.bn1d_gelu_drop_bwd_apply(hh, d_g, sc, sh, mu, inv, mask, drop_p, sums, d_hh)
        ops.bn_param_grads(sums, G[prefix + "mlp.1.weight"], G[prefix + "mlp.1.bias"], 1)
        self._lin_wgrad(d_hh, x, G[prefix + "mlp.0.weight"], G[prefix + "mlp.0.bias"])
        ops.linear_bwd_data(d_hh, S[prefix + "mlp.0.weight"], d_x, tc=self.lin_tc)

    def _encode(self, w, role, P, bns, x_img, x_aud, N, B, n_fusion, fmask, train=True):
        """Encoder forward for N = n_views*B samples; fusion only over the first n_fusion rows."""
        if self.multi:
            E = self.E
            catr = w[f"{role}.catr"]

            def top(mod, p_last, cols):
                pool, nflat, lin = self.top[mod]
                if pool:                      # AdaptiveAvgPool2d(1) + Flatten (models/dino.py:34-36, 66-68)
                    ops.avgpool_fwd(p_last, w[f"{role}.{mod}.gap"])
                    x = w[f"{role}.{mod}.gap"]
                else:
                    x = p_last.view(N, nflat)
                ops.linear_fwd(x, P[lin + ".weight"], P[lin + ".bias"], catr[:, cols], tc=self.lin_tc)

            # the student's image stack runs beside its audio stack on a second side stream (independent until the fusion MLP)
            main = torch.cuda.current_stream()
            side = self._side_stream2 if (self.overlap_teacher and role == "s") else None
            if side is not None:
                side.wait_stream(main)
            with (torch.cuda.stream(side) if side is not None else contextlib.nullcontext()):
                pi = self._conv_stack(w, role, "img", self.img_layers, x_img, N, B, P, bns, train=train)
                top("img", pi, slice(0, E))
            pa = self._conv_stack(w, role, "aud", self.aud_layers, x_aud, N, B, P, bns, train=train)
            if side is not None:
                main.wait_stream(side)
            top("aud", pa, slice(E, 2 * E))
            self._mix_fwd(w, role, P, n_fusion, B)
            cat = w[f"{role}.cat"]
            h1, feat = w[f"{role}.h1"], w[f"{role}.feat"]
            if fmask is None:        # evaluation mode: no dropout
                ops.linear_fwd(cat[:n_fusion], P["enc.fusion.0.weight"], P["enc.fusion.0.bias"], h1, act=1, tc=self.lin_tc)
            else:
                ops.linear_fwd(cat[:n_fusion], P["enc.fusion.0.weight"], P["enc.fusion.0.bias"], h1, act=2, mask=fmask, drop_p=self.fusion_dropout, tc=self.lin_tc)
            ops.linear_fwd(h1, P["enc.fusion.3.weight"], P["enc.fusion.3.bias"], feat, tc=self.lin_tc)
            return feat
        # unimodal: conv stack -> top (global average pool, or flatten: w[role.top] is already a view of p_last) -> the linears of
        # self.uni (image_simple: encoder.14, projection.0; spectrogram_simple: encoder.18; the CentralNet kinds: encoder.1)
        mod, (top, _), chain = self.uni
        p_last = self._conv_stack(w, role, mod, self._layers(mod), x_img if mod == "img" else x_aud, N, B, P, bns, train=train)
        if top == "pool":
            ops.avgpool_fwd(p_last, w[f"{role}.top"])
        for lin, src, dst, _ in chain:
            ops.linear_fwd(w[f"{role}.{src}"], P[lin + ".weight"], P[lin + ".bias"], w[f"{role}.{dst}"], tc=self.lin_tc)
        return w[f"{role}.feat"]

    def _layers(self, mod):
        return self.img_layers if mod == "img" else self.aud_layers

    def _conv_stack_bwd(self, w, mod, layers, x, d_top, N, B):
        """Backward through a conv stack; d_top = gradient w.r.t. the last pooled activation (fp32, any shape, N*C*h*w)."""
        S, G = self.S, self.G
        d_p = d_top
        BF = torch.bfloat16
        # weight gradients (UMMA-issue bound, little HBM traffic) run on their own stream beside the data gradient and the next
        # layer's HBM-bound BatchNorm kernels; dz and the wgrad scratch are double-buffered, an event guards their reuse
        main = torch.cuda.current_stream()
        wside = self._wgrad_streams[mod] if self.overlap_teacher else None
        busy = {}                                               # buffer parity -> event of the wgrad that still reads it
        for li in range(len(layers) - 1, -1, -1):
            conv, bn, ci, co, hw, k, pad = layers[li]
            ho = hw + 2 * pad - k + 1
            tc = self.tc[mod][li]
            z = w[f"s.{mod}.z{li}"]
            sums = w[f"s.{mod}.sums{li}"]
            sc, sh, mu, inv = (w[f"s.{mod}.{n}{li}"] for n in ("scale", "shift", "mean", "invstd"))
            if tc:
                if d_p.dtype != BF:
                    d_p = d_p.view(N, co, ho // 2, ho // 2)
                par = li & 1
                if par in busy:
                    main.wait_event(busy.pop(par))
                fused = ci == 1
                if not fused:
                    dz = w[f"{mod}.dz8" if par == 0 else f"{mod}.dz8b"][:z.numel()].view_as(z)
                p_out = w[f"s.{mod}.p8{li}"] if f"s.{mod}.p8{li}" in w else w[f"s.{mod}.p{li}"]
                if not (li + 1 < len(layers) and self.bnstat[mod][li + 1]):      # else: the data gradient above already accumulated them
                    ops.bn_pool8_bwd_reduce_p(p_out, d_p, S["enc." + bn + ".weight"], S["enc." + bn + ".bias"], sums, B)
                if not fused:
                    ops.bn_relu_pool8_bwd_apply(z, d_p, sc, sh, mu, inv, sums, dz, B, dbsum=w[f"{mod}.dbsum"][li])
            else:
                dz = w[f"{mod}.dz"][:z.numel()].view_as(z)
                ops.bn_relu_pool_bwd_reduce(z, d_p, sc, sh, mu, inv, sums, B)
                ops.bn_relu_pool_bwd_apply(z, d_p, sc, sh, mu, inv, sums, dz, B)

            def param_grads(li=li, tc=tc, fused=tc and ci == 1, conv=conv, bn=bn, sums=sums):
                # one-CTA kernels nothing waits for before Adam: with the weight gradient on its stream, not in the main chain
                if tc and not fused:
                    ops.bias_grad_finalize(w[f"{mod}.dbsum"][li], G["enc." + conv + ".bias"])
                ops.bn_param_grads(sums, G["enc." + bn + ".weight"], G["enc." + bn + ".bias"], N // B)

            if not (tc and wside is not None):
                param_grads()
            if tc:
                xin8 = w[f"{mod}.xs8"] if ci == 1 else w[f"s.{mod}.p8{li - 1}"]
                wk = w[f"{mod}.wg_work" if (li & 1) == 0 else f"{mod}.wg_work_b"]

                def wgrad():
                    if wside is not None:
                        param_grads()
                    if fused:       # BatchNorm / ReLU / pool backward-apply happens inside the weight-gradient kernel
                        ops.conv_tc_wgrad_l0_fused(xin8, z, d_p, sc, sh, mu, inv, sums, G["enc." + conv + ".weight"], w[f"{mod}.dbsum"][li], wk,
                                                   B, pad)
                        ops.bias_grad_finalize(w[f"{mod}.dbsum"][li], G["enc." + conv + ".bias"])
                    else:
                        ops.conv_tc_wgrad(xin8, dz, G["enc." + conv + ".weight"], wk, pad)

                if wside is not None:
                    wside.wait_stream(main)
                    with torch.cuda.stream(wside):
                        wgrad()
                        ev = torch.cuda.Event()
                        ev.record(wside)
                    busy[li & 1] = ev
                else:
                    wgrad()
            else:
                xin = x if li == 0 else w[f"s.{mod}.p{li - 1}"]
                ops.conv_bwd_weight(xin.view(N, ci, hw, hw), dz, G["enc." + conv + ".weight"], G["enc." + conv + ".bias"], w[f"{mod}.wg_work"], pad)
            if li > 0:
                nxt = w[f"{mod}.dp_a"] if d_p.data_ptr() != w[f"{mod}.dp_a"].data_ptr() else w[f"{mod}.dp_b"]
                if tc:
                    if self.tc[mod][li - 1]:          # the consumer is an act8 layer: bf16 act8 gradient
                        d_in = nxt.view(BF)[:N * ci * hw * hw].view(N, ci // 8, hw, hw, 8)
                    else:
                        d_in = nxt[:N * ci * hw * hw].view(N, ci, hw, hw)
                    if self.bnstat[mod][li]:
                        lbn = layers[li - 1][1]
                        ops.conv_tc_dgrad_bnstat(dz, self._tcw[("flip", mod, li)], d_in, w[f"s.{mod}.p8{li - 1}"], S["enc." + lbn + ".weight"],
                                                 S["enc." + lbn + ".bias"], w[f"s.{mod}.sums{li - 1}"], B, k, k - 1 - pad)
                    else:
                        ops.conv_tc(dz, self._tcw[("flip", mod, li)], None, d_in, None, N, ci, k, k - 1 - pad)
                else:
                    d_in = nxt[:N * ci * hw * hw].view(N, ci, hw, hw)
                    ops.conv_bwd_data(dz, S["enc." + conv + ".weight"], d_in, pad)
                d_p = d_in
        if wside is not None:
            main.wait_stream(wside)

    # ------------------------------------------------------------------------------------------------------
    # evaluation-side encoder forward (SURVEY 8f-3: linear-probe / kNN features; models/dino.py:1764-1850)
    # ------------------------------------------------------------------------------------------------------
    def _eval_workspace(self, B):
        key = ("eval", B)
        if key in self._ws:
            return self._ws[key]
        dev = self.device
        w = {"B": B}

        def e(*shape, dtype=F32):
            return torch.empty(*shape, dtype=dtype, device=dev)

        w["zarena"], zalloc = _zero_arena(1 << 12, dev)
        if self.img_layers:
            w["x_img"] = e(B, 1, 28, 28)
        if self.aud_layers:
            w["x_aud"] = e(B, 1, 112, 112)
        self._stack_buffers(w, "e", B, B, e, zalloc)
        E, O = self.E, self.O
        if self.multi:
            self._mix_workspace(w, "e", B, B, B, e)
            w["e.h1"], w["e.feat"] = e(B, E), e(B, O)
            w["e.fmask"] = torch.ones(B, E, dtype=torch.uint8, device=dev)
            for mod in ("img", "aud"):
                if self.top[mod][0]:
                    w[f"e.{mod}.gap"] = e(B, self.top[mod][1])
        else:
            self._uni_workspace(w, "e", B, e)
        self._ws[key] = w
        return w

    def begin_probe(self, teacher=False):
        """Start a linear-probe session (reference models/dino.py:878-951: `DownstreamClassifier` deep-copies the student, trains the
        probe with the copy in train() mode -- its BatchNorm running statistics adapt to the un-augmented batches -- and evaluates
        with those statistics).  Returns a token holding the copy's running statistics (initialised from the live ones) and its own
        dropout counter; pass it to encode_features(probe=token).  The live statistics are never touched."""
        src = self.bn_t if teacher else self.bn_s
        bns = {}
        for k, v in src.items():
            c = _BN(v.C, self.device)
            c.running_mean.copy_(v.running_mean)
            c.running_var.copy_(v.running_var)
            c.num_batches_tracked.copy_(v.num_batches_tracked)
            bns[k] = c
        return {"bns": bns, "step": 0, "teacher": teacher}

    @torch.no_grad()
    def encode_features(self, images, audios=None, train=False, teacher=False, probe=None, step_dev=None):
        """Encoder features [B, O] of an UN-augmented batch (images [B,28,28] fp32 in [0,1] or uint8, audios [B,112,112] fp32 in
        [0,1] or uint8), as DownstreamClassifier / FeatureExtractor of the reference use them (models/dino.py:1764-1850).
        train=False: BatchNorm with running statistics, no dropout (module.eval()); train=True: batch statistics and an active
        fusion dropout.  probe (a begin_probe() token): the running statistics read / updated are the probe copy's, and every
        train-mode call draws a fresh dropout mask; without a token train-mode updates go to scratch and eval reads the live ones.
        step_dev (int64 device scalar, with a token): the probe's dropout position is read from it instead of the token's host
        counter -- the same mask stream, (rng_step + *step_dev) * 4 + 3 -- so a captured CUDA graph draws a fresh mask per replay;
        the caller advances it."""
        B = self._batch_size(images, audios)
        w = self._eval_workspace(B)
        P = self.T if teacher else self.S
        bns = self.bn_t if teacher else self.bn_s
        if probe is not None:
            bns = probe["bns"]
        elif train:       # scratch running statistics
            bns = {k: _BN(v.C, self.device) for k, v in bns.items()}
        xi = xa = None
        if self.img_layers:
            xi = w["x_img"]
            xi.copy_((images.float() / 255.0 if images.dtype == torch.uint8 else images).reshape(B, 1, 28, 28))
        if self.aud_layers:
            xa = w["x_aud"]
            xa.copy_((audios.float() / 255.0 if audios.dtype == torch.uint8 else audios).reshape(B, 1, 112, 112))
        w["packed"] = False
        if self._tcw:
            self._prep_tc_weights("t" if teacher else "s", P)
        for mod, layers, x in (("img", self.img_layers, xi), ("aud", self.aud_layers, xa)):
            if layers and self.tc[mod][0]:
                ops.pack_quad8(x.view(B, layers[0][4], layers[0][4]), w[f"{mod}.xs8"], layers[0][6])
        w["packed"] = True
        fmask = None
        if train and self.multi and self.fusion_dropout > 0:
            fmask = w["e.fmask"]
            if probe is not None:
                probe["step"] += 1
            if step_dev is not None:
                ops.dropout_mask(fmask, self.fusion_dropout, self.seed + 17, self.rng_step * 4 + 3, step_dev=step_dev)
            else:
                ops.dropout_mask(fmask, self.fusion_dropout, self.seed + 17, (self.rng_step + (probe["step"] if probe is not None else 0)) * 4 + 3)
        self._eval_wrole = "t" if teacher else "s"
        w["zarena"].zero_()                             # the BatchNorm statistics of every layer
        return self._encode(w, "e", P, bns, xi, xa, B, B, B, fmask, train=train)

    # ------------------------------------------------------------------------------------------------------
    # the step
    # ------------------------------------------------------------------------------------------------------
    def forward_pass(self, x_img, x_aud, masks=None, raw=None):
        """Student (all views [+ the un-augmented pass in the non-default modes]) and teacher (global views) forward
        through encoders and heads.  Returns the workspace dict; outputs: w['s.proj'] [V*B,P], w['t.proj'] [Vg*B,P]
        (UNcentred), w['aux_image.out'] / w['aux_audio.out'] [B, 10|P]."""
        V, Vg, E = self.V, self.Vg, self.E
        x_in = x_img if self.img_layers else x_aud            # the views of the first encoded modality: [V,B,...]
        B = x_in.shape[1]
        w = self._workspace(B)
        Ns, Nt, Nv = w["Ns"], w["Nt"], V * B
        S, T = self.S, self.T
        multi = self.multi
        xi = w.get("x_img")
        xa = w.get("x_aud")
        self._join_center()
        w["zarena"].zero_()                             # all statistics / backward-sum accumulators of this step
        packed = x_in.dtype == torch.bfloat16           # augment(direct=True): the quad8 workspace images are already filled
        w["packed"] = packed
        if packed:
            if ((self.img_layers and x_img.data_ptr() != w["img.xs8"].data_ptr()) or
                    (self.aud_layers and x_aud.data_ptr() != w["aud.xs8"].data_ptr())):
                raise ops._lib.B200Error("bf16 inputs must be the workspace quad8 images returned by augment(direct=True)")
            if self.mode != "default":
                ops.pack_quad8(raw[0].reshape(B, 28, 28), w["img.xs8"][Nv:], self.img_layers[0][6])
                ops.pack_quad8(raw[1].reshape(B, 112, 112), w["aud.xs8"][Nv:], self.aud_layers[0][6])
        else:
            if self.img_layers and x_img.data_ptr() != xi.data_ptr():
                xi[:Nv].copy_(x_img.reshape(Nv, 1, 28, 28))
            if self.aud_layers and x_aud.data_ptr() != xa.data_ptr():
                xa[:Nv].copy_(x_aud.reshape(Nv, 1, 112, 112))
            if self.mode != "default":
                xi[Nv:].copy_(raw[0].reshape(B, 1, 28, 28))
                xa[Nv:].copy_(raw[1].reshape(B, 1, 112, 112))
        if masks is not None:
            if multi:
                w["s.fmask"].copy_(masks["student_fusion"].reshape(Nv, E))
                w["t.fmask"].copy_(masks["teacher_fusion"].reshape(Nt, E))
            w["s.hmask"].copy_(masks["student_head"].reshape(Nv, 512))
        else:
            step, step_dev = self._step_args()
            base = step * 4
            if multi:
                ops.dropout_mask(w["s.fmask"], self.fusion_dropout, self.seed + 1, base, step_dev=step_dev)
                ops.dropout_mask(w["t.fmask"], self.fusion_dropout, self.seed + 1, base + 1, step_dev=step_dev)
            if self.dropout > 0:
                ops.dropout_mask(w["s.hmask"], self.dropout, self.seed + 1, base + 2, step_dev=step_dev)
        if self._tcw:
            self._prep_tc_weights("s", S)
            self._prep_tc_weights("t", T)
        # first-layer operand images for both roles (the teacher reads a prefix of the student's)
        if not packed:
            for mod, layers, x in (("img", self.img_layers, xi), ("aud", self.aud_layers, xa)):
                if layers and self.tc[mod][0]:
                    hw, pad = layers[0][4], layers[0][6]
                    ops.pack_quad8(x.view(Ns, hw, hw), w[f"{mod}.xs8"], pad)
            w["packed"] = True
        # the teacher forward is independent of the student forward: it runs on a side stream so that its CTAs fill the SMs the
        # student's thin kernels leave idle (separate activation buffers; joined before the loss)
        main = torch.cuda.current_stream()
        side = self._side_stream if self.overlap_teacher else None
        if side is not None:
            side.wait_stream(main)
            with torch.cuda.stream(side):
                feat_t = self._encode(w, "t", T, self.bn_t, _rows(xi, Nt), _rows(xa, Nt), Nt, B, Nt, w.get("t.fmask"))
                self._head_fwd(w, "t", "head.", T, self.bn_t["head.mlp.1"], feat_t, w["t.proj"], w["t.hh"], w["t.g"], None, 0.0)
        feat_s = self._encode(w, "s", S, self.bn_s, xi, xa, Ns, B, Nv, w.get("s.fmask"))
        self._head_fwd(w, "s", "head.", S, self.bn_s["head.mlp.1"], feat_s, w["s.proj"], w["s.hh"], w["s.g"], w["s.hmask"], self.dropout)
        if side is not None:
            main.wait_stream(side)
        else:
            feat_t = self._encode(w, "t", T, self.bn_t, _rows(xi, Nt), _rows(xa, Nt), Nt, B, Nt, w.get("t.fmask"))
            self._head_fwd(w, "t", "head.", T, self.bn_t["head.mlp.1"], feat_t, w["t.proj"], w["t.hh"], w["t.g"], None, 0.0)
        if self.mode != "default":
            cat = w["s.catr"]               # the mode heads read the un-mixed encoder features (models/dino.py:972-980)
            for m, sl in (("aux_image", slice(0, E)), ("aux_audio", slice(E, 2 * E))):
                self._head_fwd(w, m, m + ".", S, self.bn_s[f"{m}.mlp.1"], cat[Nv:, sl], w[f"{m}.out"], w[f"{m}.hh"], w[f"{m}.g"], None, 0.0)
        w["loss"].zero_()
        return w

    def dino_loss_pass(self, w):
        """Fused DINO loss forward+backward (fills w['d.proj'], loss[0]) and the centre EMA (all-reduced when data parallel)."""
        V, Vg, P, B = self.V, self.Vg, self.P, w["B"]
        s_out, t_out = w["s.proj"].view(V, B, P), w["t.proj"].view(Vg, B, P)
        variant = 0 if self.multi else 1
        if variant == 1:
            ops.teacher_norm_colmean(t_out, self.center, w["t_colmean"])
        ops.dino_loss_fwd_bwd(s_out, t_out, self.center, self.tau_s, self.tau_t, w["d.proj"].view(V, B, P), w["part_loss"], w["part_colsum"],
                              variant=variant, t_colmean=w["t_colmean"] if variant == 1 else None)
        loss = w["loss"]
        if self.world > 1:
            # data parallel: centre = EMA of the mean over ALL ranks' teacher rows (SURVEY §8e).  The centre is next read by the NEXT
            # step's loss, so the 512-byte all-reduce + EMA run on the communication stream and never stall the backward pass
            ops.center_update(None, w["part_colsum"], w["part_loss"], Vg * B, self.center_momentum, loss[0:1], colsum_out=w["colsum"][:P])
            main, cs = torch.cuda.current_stream(), self._comm_stream
            cs.wait_stream(main)
            with torch.cuda.stream(cs):
                self.comm.allreduce_center_(w["colsum"][:P], cs.cuda_stream)
                ops.center_apply(self.center, w["colsum"][:P], Vg * B * self.world, self.center_momentum)
                self._center_ready = torch.cuda.Event()
                self._center_ready.record(cs)
        else:
            ops.center_update(self.center, w["part_colsum"], w["part_loss"], Vg * B, self.center_momentum, loss[0:1])

    def _join_center(self):
        """Make the current stream wait for the last step's all-reduced centre EMA (data parallel only)."""
        if self._center_ready is not None:
            torch.cuda.current_stream().wait_event(self._center_ready)
            self._center_ready = None

    def aux_loss_pass(self, w, labels=None):
        """MSE / InfoNCE / CE on the mode heads' outputs, forward+backward fused (fills w['aux_*.d.out'], loss[1])."""
        loss = w["loss"]
        oi, oa = w["aux_image.out"], w["aux_audio.out"]
        if self.mode == "semi_supervised":
            ops.ce_fwd_bwd(oi, labels, w["aux_image.d.out"], loss[1:2], grad_scale=self.alpha, work=w["loss_work"])
            ops.ce_fwd_bwd(oa, labels, w["aux_audio.d.out"], loss[2:3], grad_scale=self.alpha, work=w["loss_work"])
            loss[1:2].add_(loss[2:3])
            loss[2:3].zero_()
        elif self.mode == "infonce":
            ops.infonce_fwd_bwd(oi, oa, w["aux_image.d.out"], w["aux_audio.d.out"], loss[1:2], w["infonce_work"], grad_scale=self.alpha, tc=self.lin_tc)
        elif self.mode == "mse":
            ops.mse_align_fwd_bwd(oi, oa, w["aux_image.d.out"], w["aux_audio.d.out"], loss[1:2], grad_scale=self.alpha, work=w["loss_work"])

    def backward_pass(self, w, d_proj=None, d_aux=None):
        """Backward from the gradient w.r.t. the student projections (default: the fused loss's own w['d.proj']) and, in the
        non-default modes, w.r.t. the two mode-head outputs (default: w['aux_*.d.out']).  Fills self.grad."""
        V, E, O = self.V, self.E, self.O
        B = w["B"]
        Ns, Nv = w["Ns"], V * B
        S, G = self.S, self.G
        multi = self.multi
        xi, xa = w.get("x_img"), w.get("x_aud")
        feat_s = w["s.feat"]
        d_proj = w["d.proj"] if d_proj is None else d_proj.reshape(Nv, self.P)
        d_feat = w["d.feat"]
        self._head_bwd(w, "s", "head.", feat_s, d_proj, w["s.hh"], w["s.g"], w["d.g"], w["d.hh"], d_feat, w["s.hmask"], self.dropout)
        if self.cosine_loss_alpha > 0:
            ops.cosine_consistency_fwd_bwd(feat_s.view(V, B, O), w["d.emb"].view(V, B, O), w["loss"][2:3], grad_scale=self.cosine_loss_alpha,
                                           work=w["loss_work"])
            ops.add2d(d_feat, w["d.emb"])
        if multi:
            d_cat, d_catr, d_h1 = w["d.cat"], w["d.catr"], w["d.h1"]
            self._lin_wgrad(d_feat, w["s.h1"], G["enc.fusion.3.weight"], G["enc.fusion.3.bias"])
            ops.linear_bwd_data(d_feat, S["enc.fusion.3.weight"], d_h1, tc=self.lin_tc)
            ops.act_bwd(d_h1, w["s.h1"], self.fusion_dropout)
            self._lin_wgrad(d_h1, w["s.cat"][:Nv], G["enc.fusion.0.weight"], G["enc.fusion.0.bias"])
            ops.linear_bwd_data(d_h1, S["enc.fusion.0.weight"], d_cat[:Nv], tc=self.lin_tc)
            self._mix_bwd(w, Nv, B)
            if self.mode != "default":
                for i, (m, sl) in enumerate((("aux_image", slice(0, E)), ("aux_audio", slice(E, 2 * E)))):
                    d_out = w[f"{m}.d.out"] if d_aux is None else d_aux[i]
                    self._head_bwd(w, m, m + ".", w["s.catr"][Nv:, sl], d_out, w[f"{m}.hh"], w[f"{m}.g"], w[f"{m}.d.g"],
                                   w[f"{m}.d.hh"], d_catr[Nv:, sl], None, 0.0)
            # the image and the audio stacks are independent from here on: the (small) image stack runs on the side stream
            main = torch.cuda.current_stream()
            side = self._side_stream if self.overlap_teacher else None
            for mod, layers, sl, x in (("img", self.img_layers, slice(0, E), xi), ("aud", self.aud_layers, slice(E, 2 * E), xa)):
                pool, nflat, lin = self.top[mod]
                ctx = torch.cuda.stream(side) if (side is not None and mod == "img") else contextlib.nullcontext()
                if side is not None and mod == "img":
                    side.wait_stream(main)
                with ctx:
                    p_last = w[f"s.{mod}.p{len(layers) - 1}"]
                    x_lin = w[f"s.{mod}.gap"] if pool else p_last.view(Ns, nflat)
                    self._lin_wgrad(d_catr[:, sl], x_lin, G[lin + ".weight"], G[lin + ".bias"])
                    if pool:
                        ops.linear_bwd_data(d_catr[:, sl], S[lin + ".weight"], w[f"d.{mod}.gap"], tc=self.lin_tc)
                        d_p = w[f"{mod}.dp_a"][:p_last.numel()].view_as(p_last)
                        ops.avgpool_bwd(w[f"d.{mod}.gap"], d_p)
                    else:
                        d_p = w[f"{mod}.dp_a"][:Ns * nflat].view(Ns, nflat)
                        ops.linear_bwd_data(d_catr[:, sl], S[lin + ".weight"], d_p, tc=self.lin_tc)
                    self._conv_stack_bwd(w, mod, layers, x, d_p, Ns, B)
            if side is not None:
                main.wait_stream(side)
        else:
            mod, (top, _), chain = self.uni
            layers = self._layers(mod)
            for lin, src, dst, _ in reversed(chain):
                d_out = d_feat if dst == "feat" else w[f"d.{dst}"]
                self._lin_wgrad(d_out, w[f"s.{src}"], G[lin + ".weight"], G[lin + ".bias"])
                ops.linear_bwd_data(d_out, S[lin + ".weight"], w[f"d.{src}"], tc=self.lin_tc)
            if top == "pool":
                p_last = w[f"s.{mod}.p{len(layers) - 1}"]
                d_p = w[f"{mod}.dp_a"][:p_last.numel()].view_as(p_last)
                ops.avgpool_bwd(w["d.top"], d_p)
            else:                       # flatten: the first linear's data gradient already is the stack's top gradient (in dp_a)
                d_p = w["d.top"]
            self._conv_stack_bwd(w, mod, layers, xi if mod == "img" else xa, d_p, Ns, B)
        if self._lin_wg_pending:
            torch.cuda.current_stream().wait_stream(self._lin_wg_stream)
            self._lin_wg_pending = False
        if self.world > 1:
            self.allreduce_gradients()

    def forward_backward(self, x_img, x_aud, masks=None, raw=None, labels=None):
        """Student + teacher forward, losses, centre EMA and the full backward for already-augmented views.

        x_img [V,B,28,28] (and x_aud [V,B,112,112]) view-major, global views first; masks (optional, parity tests):
        dict of uint8 keep-masks 'student_fusion' [V*B,E], 'teacher_fusion' [Vg*B,E], 'student_head' [V*B,512];
        raw = (image [B,28,28], audio [B,112,112]) fp32 for the non-default modes; labels int64 [B].
        Leaves the gradients in self.grad (all-reduced when data parallel) and returns the loss tensor [4] =
        (dino, aux, cosine, total) on the device."""
        w = self.forward_pass(x_img, x_aud, masks=masks, raw=raw)
        self.dino_loss_pass(w)
        if self.mode != "default":
            self.aux_loss_pass(w, labels)
        self.backward_pass(w)
        loss = w["loss"]
        # the loss kernels report UNSCALED values (their gradients carry the weights): total = dino + alpha*aux + alpha_cos*cosine
        loss[3:4].copy_(loss[0:1] + float(getattr(self, "alpha", 1.0)) * loss[1:2] + float(self.cosine_loss_alpha) * loss[2:3])
        return loss

    def allreduce_gradients(self):
        """Data parallel exchange of the gradient arena through the C ABI (NCCL), once the backward pass has joined its streams: on
        the communication stream, where it overlaps the teacher EMA; Adam joins that stream.  The 1/world average is folded into
        Adam's grad_scale.  (Exchanging the early-complete slices beside the conv stacks' backward measured slower: DESIGN.md.)"""
        main, cs = torch.cuda.current_stream(), self._comm_stream
        cs.wait_stream(main)
        with torch.cuda.stream(cs):
            for lo, hi in self.grad_plan.ranges:
                self.comm.allreduce_grads_(self.grad[lo:hi], cs.cuda_stream)
        self._comm_pending = True
        self._grad_scale = 1.0 / self.world

    def update_teacher(self):
        """Teacher EMA over the whole common arena prefix: one kernel (models/dino.py:635-646)."""
        ops.ema_flat(self.teacher.flat[:self.n_ema], self.student.flat[:self.n_ema], self.momentum)

    def optimizer_step(self, grad_scale=None):
        """Adam (lr, weight_decay; models/dino.py:953-962) over the parameters that received gradients."""
        self.step_count += 1
        if self._comm_pending:          # the gradient all-reduces of this step (the teacher EMA before this call overlapped them)
            torch.cuda.current_stream().wait_stream(self._comm_stream)
            self._comm_pending = False
        gs = self._grad_scale if grad_scale is None else grad_scale
        n = self.n_trainable_prefix
        ranges = [(0, n)] + ([self.aux_range] if self.aux_range is not None else [])
        if self._ctr is not None:       # CUDA-graph mode: the step number and its bias corrections live on the device
            ops.adam_bias_dev(self._ctr[1:2], self._bc)
        for lo, hi in ranges:
            if self._ctr is not None:
                ops.adam_flat_dev(self.student.flat[lo:hi], self.grad[lo:hi], self.exp_avg[lo:hi], self.exp_avg_sq[lo:hi], self._bc, -1.0,
                                  weight_decay=self.weight_decay, grad_scale=gs)       # lr < 0: read from self._bc[2] (scheduler-friendly)
            else:
                ops.adam_flat(self.student.flat[lo:hi], self.grad[lo:hi], self.exp_avg[lo:hi], self.exp_avg_sq[lo:hi], self.step_count,
                              self.lr, weight_decay=self.weight_decay, grad_scale=gs)

    def reset_optimizer_state(self):
        """A fresh Adam: zero moments, step 0 (what constructing a new torch.optim.Adam gives the reference per fit)."""
        self.exp_avg.zero_()
        self.exp_avg_sq.zero_()
        self.step_count = 0
        if self._ctr is not None:
            self._ctr[1:2].zero_()

    def optimizer_state(self):
        """Adam state for checkpoints: the two moment arenas (CPU copies) + the step count."""
        return {"exp_avg": self.exp_avg.detach().cpu().clone(), "exp_avg_sq": self.exp_avg_sq.detach().cpu().clone(), "step": int(self.step_count)}

    def load_optimizer_state(self, state):
        if state["exp_avg"].numel() != self.exp_avg.numel():
            raise ops._lib.B200Error("load_optimizer_state: arena size mismatch (different model kind / mode)")
        self.exp_avg.copy_(state["exp_avg"].to(self.device))
        self.exp_avg_sq.copy_(state["exp_avg_sq"].to(self.device))
        self.step_count = int(state["step"])
        if self._ctr is not None:
            self._ctr[1:2].fill_(self.step_count)

    def train_step_views(self, x_img, x_aud, masks=None, raw=None, labels=None):
        """Reference step order on given views: forward/loss/backward, EMA (before the optimizer, dino.py:871), Adam."""
        loss = self.forward_backward(x_img, x_aud, masks=masks, raw=raw, labels=labels)
        self.update_teacher()
        self.optimizer_step()
        self._join_center()
        self.rng_step += 1
        if self._ctr is not None:
            ops.counters_advance(self._ctr)
        return loss

    def train_step(self, images, audios=None, labels=None):
        """Whole step from a raw device batch: images [B,28,28] fp32 in [0,1] or uint8; audios [B,112,112] uint8 (or fp32);
        labels int64 [B] (semi_supervised).  Returns the device loss tensor [4] (dino, aux, cosine, total)."""
        got = self._take_prefetched(images, audios)
        xi, xa = got if got is not None else self.augment(images, audios, direct=True)
        raw = None
        if self.mode != "default":
            img_f = images.float() / 255.0 if images.dtype == torch.uint8 else images
            aud_f = audios.float() / 255.0 if audios.dtype == torch.uint8 else audios
            raw = (img_f, aud_f)
        loss = self.train_step_views(xi, xa, raw=raw, labels=labels)
        self._step_done_prev, self._step_done = self._step_done, torch.cuda.Event()
        self._step_done.record()
        return loss

    # ------------------------------------------------------------------------------------------------------
    # CUDA-graph replay of the whole step (small per-GPU batches are bound by the ~165 host-side launches)
    # ------------------------------------------------------------------------------------------------------
    def _state_tensors(self):
        ts = [self.student.flat, self.teacher.flat, self.exp_avg, self.exp_avg_sq, self.center]
        for table in (self.bn_s, self.bn_t):
            for bn in table.values():
                ts += [bn.running_mean, bn.running_var, bn.num_batches_tracked]
        return ts

    def capture_train_step(self, B, image_dtype=torch.float32, audio_dtype=torch.uint8):
        """Captures train_step (sampling, augmentation, forward, losses, EMA, backward, Adam, all side streams) for per-GPU batch
        B into ONE CUDA graph.  The per-step scalars (RNG stream position, Adam step) move to device counters that the graph
        advances itself, so a replay needs no host arguments and reproduces the eager step bit for bit.  Data parallel: the
        NCCL all-reduces (b200_dp_*, communication stream) are captured with the kernels; every rank must capture and replay in
        lock-step.  The learning rate is a device scalar (schedulers may change engine.lr between replays); temperatures, momenta and
        weight decay are baked in (re-capture after changing them).  Use graph_step() afterwards."""
        dev = self.device
        g = {"B": B}
        if self.img_layers:
            g["img"] = torch.zeros(B, 28, 28, dtype=image_dtype, device=dev)
        if self.aud_layers:
            g["aud"] = torch.zeros(B, 112, 112, dtype=audio_dtype, device=dev)
        if self.mode == "semi_supervised":
            g["lab"] = torch.zeros(B, dtype=torch.int64, device=dev)
        self._prefetch = None
        state = self._state_tensors()
        snap = [t.clone() for t in state]
        host = (self.rng_step, self.step_count)
        self._ctr = torch.tensor(host, dtype=torch.int64, device=dev)
        self._bc = torch.zeros(3, device=dev)               # bias corrections of the step + the learning rate (read by the captured Adam)
        self._bc[2:3].fill_(float(self.lr))
        self._graph_lr = float(self.lr)

        def body():
            return self.train_step(g.get("img"), g.get("aud"), g.get("lab"))

        def restore():
            for t, c in zip(state, snap):
                t.copy_(c)
            self.rng_step, self.step_count = host
            self._ctr.copy_(torch.tensor(host, dtype=torch.int64))
            self._step_done = self._step_done_prev = None

        side = torch.cuda.Stream(device=dev)       # warm-up off the capture stream: workspaces, scratch, one-time attributes
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side):
            for _ in range(2):
                body()
        torch.cuda.current_stream().wait_stream(side)
        torch.cuda.synchronize()
        restore()
        graph = torch.cuda.CUDAGraph(keep_graph=True)        # keep the cudaGraph_t: graph_node_counts() reads it
        with torch.cuda.graph(graph):
            g["loss"] = body()
        graph.instantiate()
        restore()
        torch.cuda.synchronize()
        g["graph"] = graph
        self._graph = g
        return g

    def graph_step(self, images, audios=None, labels=None):
        """One training step by replaying the captured graph on a raw device batch; returns the device loss tensor [4]."""
        g = self._graph
        if g is None or self._batch_size(images, audios) != g["B"]:
            raise ops._lib.B200Error("graph_step: call capture_train_step(B) for this batch size first")
        if "img" in g:
            g["img"].copy_(images.reshape(g["img"].shape))
        if "aud" in g:
            g["aud"].copy_(audios.reshape(g["aud"].shape))
        if "lab" in g:
            g["lab"].copy_(labels)
        if float(self.lr) != self._graph_lr:                 # a scheduler moved the learning rate: one 4-byte fill, no re-capture
            self._graph_lr = float(self.lr)
            self._bc[2:3].fill_(self._graph_lr)
        g["graph"].replay()
        self.rng_step += 1
        self.step_count += 1
        return g["loss"]

    def graph_node_counts(self):
        """{'kernels', 'memsets', 'memcpys', 'other'} of the captured step: the step's launches COUNTED from the CUDA graph (every
        kernel of every stream, the NCCL kernels of a data-parallel step included) rather than tallied per wrapper."""
        if self._graph is None:
            raise ops._lib.B200Error("graph_node_counts: call capture_train_step first")
        import ctypes
        counts = (ctypes.c_int64 * 4)()
        ops._lib.check(ops._lib_().b200_graph_node_counts(self._graph["graph"].raw_cuda_graph(), counts), "graph_node_counts")
        return dict(zip(("kernels", "memsets", "memcpys", "other"), (int(c) for c in counts)))

    def release_graph(self):
        """Back to eager stepping (the host counters are authoritative again)."""
        self._graph = None
        self._ctr = self._bc = None

    def train_step_host(self, images_host, audios_host=None, labels_host=None, next_batch=None, lagged_loss=False):
        """The host-facing call: raw batch in (pinned) host memory -> H2D copies -> whole step -> the total loss as a Python
        float (D2H read).  This is what `e2e` in bench.py times.  next_batch = (images_host, audios_host[, labels_host]) of
        the FOLLOWING call, if known: its H2D copy and augmentation are enqueued on the augmentation stream before this
        step's loss is read back, so the input pipeline overlaps the step (what the reference's DataLoader workers do).
        lagged_loss=True: every step's loss is still copied to (pinned) host memory, but the call returns the PREVIOUS step's
        value (None on the first call; flush_loss() returns the last one) so that the host never waits for the step it has
        just enqueued -- the usual way a training loop logs its loss.  An audio-only kind ignores the image batches (they may be None)."""
        def ptr(t):
            return None if t is None else t.data_ptr()

        if not self.img_layers:
            images_host = None
            if next_batch is not None:
                next_batch = (None,) + tuple(next_batch[1:])
        B = self._batch_size(images_host, audios_host)
        buf = self._ws.setdefault(("host", B, None if images_host is None else images_host.dtype,
                                   None if audios_host is None else audios_host.dtype), {})
        if not buf:
            for tag in ("", "_b"):
                for k, t in (("img", images_host), ("aud", audios_host), ("lab", labels_host)):
                    if t is not None:
                        buf[k + tag] = torch.empty(t.shape, dtype=t.dtype, device=self.device)
            buf["staged"] = None
        if buf["staged"] is not None and buf["staged"] == (ptr(images_host), ptr(audios_host)):
            for k in ("img", "aud", "lab"):                       # this batch was staged by the previous call: swap the slots
                if k in buf:
                    buf[k], buf[k + "_b"] = buf[k + "_b"], buf[k]
        else:
            self._prefetch = None
            for k, t in (("img", images_host), ("aud", audios_host), ("lab", labels_host)):
                if t is not None:
                    buf[k].copy_(t, non_blocking=True)
        buf["staged"] = None
        loss = self.train_step(buf.get("img"), buf.get("aud"), buf.get("lab"))
        if next_batch is not None:
            nimg, naud = next_batch[0], (next_batch[1] if len(next_batch) > 1 else None)
            nlab = next_batch[2] if len(next_batch) > 2 else None
            with torch.cuda.stream(self._aug_stream):
                if self._step_done_prev is not None:
                    self._aug_stream.wait_event(self._step_done_prev)      # the spare raw buffers were last read one step back
                for k, t in (("img", nimg), ("aud", naud), ("lab", nlab)):
                    if t is not None:
                        buf[k + "_b"].copy_(t, non_blocking=True)
            if self.prefetch_augment(buf.get("img_b"), buf.get("aud_b")):
                buf["staged"] = (ptr(nimg), ptr(naud))
        if not lagged_loss:
            return float(loss[3].item())
        prev = self.flush_loss()
        slot = self._loss_slots[self._loss_flip]
        self._loss_flip ^= 1
        slot.copy_(loss[3:4], non_blocking=True)              # D2H of this step's loss, read one call later
        ev = torch.cuda.Event()
        ev.record()
        self._loss_pending = (slot, ev)
        return prev

    def flush_loss(self):
        """The loss of the last train_step_host(lagged_loss=True) call whose value has not been returned yet (or None)."""
        if self._loss_pending is None:
            return None
        slot, ev = self._loss_pending
        self._loss_pending = None
        ev.synchronize()
        return float(slot[0])
