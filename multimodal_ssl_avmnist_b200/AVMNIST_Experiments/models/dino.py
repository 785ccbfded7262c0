"""DINO modules of the AVMNIST experiments, B200-native.

Same public surface as the reference's models/dino.py (class names, constructor keywords, attribute names, state_dict
keys, Lightning hooks), but the modules are *parameter containers*: the training step itself -- student / teacher forward,
projection heads, the centred + sharpened cross-entropy, the MSE / InfoNCE / cross-entropy side losses, backward, EMA and
Adam -- runs in hand-written sm_100a kernels behind libavmnist_b200.so (multimodal_ssl_avmnist_b200.engine / .binding).
There is no PyTorch fallback: on a CPU tensor, or without the library, the step raises.

Compiled encoders: CentralMultiModalEncoder ("multi_central"), the conv encoders SimpleMultiModalEncoder ("multi_simple"),
GatedMultiModalEncoder ("multi_simple_gated") and CrossAttentionMultiModalEncoder ("multi_cross_attention") (SURVEY 8f-4), the
unimodal ImageEncoder ("image_simple") and SpectrogramEncoder ("spectrogram_simple"), and the unimodal LeNet-style CentralNet encoders
ImageEncoderCentral ("image_central") and SpectrogramEncoderCentral ("spectrogram_central").  The other encoder families of the
reference (LSTM, ViT, MobileViT, ResNet, the other spectrogram encoders) are outside the hot-path scope; their names exist so that
driver scripts import, and constructing one raises NotImplementedError.
"""
import os
import sys

import torch
import torch.nn as nn

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from _compat import pl  # noqa: E402
from models.unimodal import CentralUnimodalAudio, CentralUnimodalImage  # noqa: E402
from multimodal_ssl_avmnist_b200 import binding as B  # noqa: E402
from multimodal_ssl_avmnist_b200 import module_forward as MF  # noqa: E402


# ------------------------------------------------------------------------------------------------------------
# encoders (containers)
# ------------------------------------------------------------------------------------------------------------
def _conv_stack(channels, out_dim):
    layers = []
    for cin, cout in zip(channels[:-1], channels[1:]):
        layers += [nn.Conv2d(cin, cout, 3, padding=1), nn.BatchNorm2d(cout), nn.ReLU(), nn.MaxPool2d(2)]
    layers += [nn.AdaptiveAvgPool2d(1), nn.Flatten(), nn.Linear(channels[-1], out_dim)]
    return nn.Sequential(*layers)


def image_encoder(output_dim):
    """3 x [conv3x3, BN, ReLU, maxpool] (1->32->64->128), global average pool, Linear(128, output_dim)."""
    return _conv_stack((1, 32, 64, 128), output_dim)


def audio_encoder(output_dim):
    """4 x [conv3x3, BN, ReLU, maxpool] (1->32->64->128->256), global average pool, Linear(256, output_dim)."""
    return _conv_stack((1, 32, 64, 128, 256), output_dim)


class BaseMultiModalEncoder(nn.Module):
    def __init__(self, output_dim=256, encoder_output_dim=512, fusion_dropout=0.3):
        super().__init__()
        self.output_dim, self.encoder_output_dim, self.fusion_dropout = output_dim, encoder_output_dim, fusion_dropout

    def forward(self, images, spectrograms):
        raise NotImplementedError("Subclasses must implement forward method")


class SimpleMultiModalEncoder(BaseMultiModalEncoder):
    """Concatenation fusion: image_encoder || audio_encoder -> Linear(2E,E) -> ReLU -> Dropout -> Linear(E,O)."""
    B200_KIND = "multi_simple"

    def __init__(self, output_dim=256, encoder_output_dim=512, fusion_dropout=0.3):
        super().__init__(output_dim, encoder_output_dim, fusion_dropout)
        self.image_encoder = image_encoder(encoder_output_dim)
        self.audio_encoder = audio_encoder(encoder_output_dim)
        self.fusion = nn.Sequential(nn.Linear(2 * encoder_output_dim, encoder_output_dim), nn.ReLU(), nn.Dropout(fusion_dropout),
                                    nn.Linear(encoder_output_dim, output_dim))

    def encode_image(self, images):
        return MF.sequential_cnn_forward(self.image_encoder, images)

    def encode_audio(self, spectrograms):
        return MF.sequential_cnn_forward(self.audio_encoder, spectrograms)

    def mix(self, image_features, audio_features):
        """What happens between the encoders and the fusion MLP: plain concatenation here (models/dino.py:232-233)."""
        return torch.cat([image_features, audio_features], dim=1)

    def forward(self, images, spectrograms):
        """Inference-form forward (feature extraction); the training step goes through MultiModalDINO."""
        return MF.fusion_forward(self.fusion, self.mix(self.encode_image(images), self.encode_audio(spectrograms)))


class GatedMultiModalEncoder(SimpleMultiModalEncoder):
    """Simple encoders + one learnable sigmoid gate per modality (reference models/dino.py:237-263)."""
    B200_KIND = "multi_simple_gated"

    def __init__(self, output_dim=256, encoder_output_dim=512):
        super().__init__(output_dim, encoder_output_dim)
        self.gate_image = nn.Parameter(torch.tensor(0.5))
        self.gate_audio = nn.Parameter(torch.tensor(0.5))

    def mix(self, image_features, audio_features):
        out = torch.empty(image_features.shape[0], 2 * self.encoder_output_dim, device=image_features.device)
        E = self.encoder_output_dim
        MF.ops.gate_apply(image_features.contiguous(), self.gate_image.detach(), out[:, :E])
        MF.ops.gate_apply(audio_features.contiguous(), self.gate_audio.detach(), out[:, E:])
        return out


class CrossModalAttention(nn.Module):
    """x1 + softmax((x1 Wq)(x2 Wk)^T dim^-0.5) (x2 Wv): attention over the batch of one call (reference models/dino.py:385-405)."""

    def __init__(self, dim):
        super().__init__()
        self.dim = dim
        self.q_proj = nn.Linear(dim, dim)
        self.kv_proj = nn.Linear(dim, 2 * dim)
        self.scale = dim ** -0.5

    @torch.no_grad()
    def forward(self, x1, x2):
        q = MF._linear(x1, self.q_proj)
        kv = MF._linear(x2, self.kv_proj)
        k, v = kv[:, :self.dim].contiguous(), kv[:, self.dim:].contiguous()
        attn = torch.empty(x1.shape[0], x2.shape[0], device=x1.device)
        MF.ops.linear_fwd(q, k, None, attn)
        MF.ops.softmax_rows(attn, self.scale)
        out = torch.empty_like(q)
        MF.ops.linear_bwd_data(attn, v, out)
        MF.ops.add2d(out, x1.contiguous())
        return out


class CrossAttentionMultiModalEncoder(SimpleMultiModalEncoder):
    """Simple encoders + bidirectional batch-wide cross attention before the fusion MLP (reference models/dino.py:407-452)."""
    B200_KIND = "multi_cross_attention"

    def __init__(self, output_dim=256, encoder_output_dim=512, fusion_dropout=0.3):
        super().__init__(output_dim, encoder_output_dim, fusion_dropout)
        self.image_to_audio_attention = CrossModalAttention(dim=encoder_output_dim)
        self.audio_to_image_attention = CrossModalAttention(dim=encoder_output_dim)

    def mix(self, image_features, audio_features):
        return torch.cat([self.image_to_audio_attention(image_features, audio_features),
                          self.audio_to_image_attention(audio_features, image_features)], dim=1)


class _HeadedCNN(nn.Sequential):
    """Sequential(CentralUnimodal*, Linear) whose call runs the CUDA inference path."""

    def forward(self, x):
        flat = MF.central_cnn_forward(self[0], x)
        return MF._linear(flat, self[1])


class CentralMultiModalEncoder(SimpleMultiModalEncoder):
    """LeNet-style CentralNet CNNs per modality (models/unimodal.py) + the concatenation fusion."""
    B200_KIND = "multi_central"

    def __init__(self, output_dim=256, encoder_output_dim=512):
        # the parent is built first (and its simple encoders discarded) so that the global RNG is consumed exactly like
        # in the reference: identical seeds give identical initial weights
        super().__init__(output_dim, encoder_output_dim)
        self.image_encoder = _HeadedCNN(CentralUnimodalImage(), nn.Linear(64 * 5 * 5, encoder_output_dim))
        self.audio_encoder = _HeadedCNN(CentralUnimodalAudio(), nn.Linear(64 * 7 * 7, encoder_output_dim))

    def encode_image(self, images):
        return self.image_encoder(images)

    def encode_audio(self, spectrograms):
        return self.audio_encoder(spectrograms)


class BaseUniModalEncoder(nn.Module):
    def __init__(self, output_dim=256, modality="image"):
        super().__init__()
        self.output_dim, self.modality = output_dim, modality

    def forward(self, images=None, spectrograms=None):
        raise NotImplementedError("Subclasses must implement forward method")


class ImageEncoder(BaseUniModalEncoder):
    B200_KIND = "image_simple"

    def __init__(self, output_dim=256):
        super().__init__(output_dim, modality="image")
        self.encoder = image_encoder(output_dim=512)
        self.projection = nn.Sequential(nn.Linear(512, output_dim))

    def forward(self, images=None, spectrograms=None):
        if images is None:
            raise ValueError("ImageEncoder requires image input")
        return MF._linear(MF.sequential_cnn_forward(self.encoder, images), self.projection[0])


class SpectrogramEncoder(BaseUniModalEncoder):
    """audio_encoder(output_dim) on the spectrogram (reference models/dino.py:502-513).  The audio-only DINO encoder
    (UniModalDINO, `--unimodal_model spectrogram_simple`) and the audio branch of the stand-alone contrastive models
    (other_ssl/info_nce, other_ssl/multimodal_simclr)."""
    B200_KIND = "spectrogram_simple"

    def __init__(self, output_dim=256):
        super().__init__(output_dim, modality="audio")
        self.encoder = audio_encoder(output_dim=output_dim)

    def forward(self, images=None, spectrograms=None):
        if spectrograms is None:
            raise ValueError("SpectrogramEncoder requires spectrogram input")
        return MF.sequential_cnn_forward(self.encoder, spectrograms)


class ImageEncoderCentral(BaseUniModalEncoder):
    """The image branch of CentralMultiModalEncoder alone: encoder = Sequential(CentralUnimodalImage (2 x conv5; fc1 / fc2 unused),
    Linear(64*5*5, output_dim)) on the flattened 64x5x5 activation -- the image-only DINO encoder of the LeNet family
    (`--unimodal_model image_central`).  The reference has no LeNet unimodal image class: this layout copies
    CentralMultiModalEncoder's image branch under `encoder.`; it is not pinned against a reference checkpoint."""
    B200_KIND = "image_central"

    def __init__(self, output_dim=256):
        super().__init__(output_dim, modality="image")
        self.encoder = _HeadedCNN(CentralUnimodalImage(), nn.Linear(64 * 5 * 5, output_dim))

    def forward(self, images=None, spectrograms=None):
        if images is None:
            raise ValueError("ImageEncoderCentral requires image input")
        return self.encoder(images)


class SpectrogramEncoderCentral(BaseUniModalEncoder):
    """The audio branch of CentralMultiModalEncoder alone: encoder = Sequential(CentralUnimodalAudio (4 x conv5; fc1 / fc2 unused),
    Linear(64*7*7, output_dim)) on the flattened 64x7x7 activation (`--unimodal_model spectrogram_central`).  The body of the
    reference's SpectrogramEncoderCentral is not available here: this layout copies CentralMultiModalEncoder's audio branch under
    `encoder.`, so reference checkpoints of this class are not known to load strictly."""
    B200_KIND = "spectrogram_central"

    def __init__(self, output_dim=256):
        super().__init__(output_dim, modality="audio")
        self.encoder = _HeadedCNN(CentralUnimodalAudio(), nn.Linear(64 * 7 * 7, output_dim))

    def forward(self, images=None, spectrograms=None):
        if spectrograms is None:
            raise ValueError("SpectrogramEncoderCentral requires spectrogram input")
        return self.encoder(spectrograms)


_COMPILED = ("Central / Simple / Gated / CrossAttention MultiModalEncoder, ImageEncoder, SpectrogramEncoder, ImageEncoderCentral, "
             "SpectrogramEncoderCentral")


def _out_of_scope(name):
    def __init__(self, *a, **k):
        raise NotImplementedError(f"{name} is outside the B200 hot-path scope (see DESIGN.md section 7); compiled encoders: {_COMPILED}")
    return type(name, (nn.Module,), {"__init__": __init__, "B200_KIND": None})


for _n in ("LSTMImageEncoder", "LSTMMultiModalEncoder", "ViTMultiModalEncoder", "DualViTMultiModalEncoder", "MobileViTMultiModalEncoder",
           "ResNetMultiModalEncoder", "SpectrogramEncoderLSTM", "SpectrogramEncoderResNet", "SpectrogramEncoderViT",
           "SpectrogramEncoderMobileViT", "UniModalDINOV2"):
    globals()[_n] = _out_of_scope(_n)


class ProjectionHead(nn.Module):
    """Linear(in, hidden) -> BatchNorm1d -> GELU -> Dropout -> Linear(hidden, projection_dim)."""

    def __init__(self, input_dim, projection_dim=256, dropout_rate=0, hidden_dim=512):
        super().__init__()
        self.mlp = nn.Sequential(nn.Linear(input_dim, hidden_dim), nn.BatchNorm1d(hidden_dim), nn.GELU(), nn.Dropout(dropout_rate),
                                 nn.Linear(hidden_dim, projection_dim))

    def forward(self, x):
        return MF.projection_head_forward(self, x)


# ------------------------------------------------------------------------------------------------------------
# DINO modules
# ------------------------------------------------------------------------------------------------------------
def _to_view_major(global_t, local_t):
    """[B,Vg,1,H,W] + [B,Vl,1,H,W] -> [V,B,H,W] contiguous (global views first)."""
    x = torch.cat([global_t, local_t], dim=1)
    return x[:, :, 0].transpose(0, 1).contiguous().float()


class _DinoBase(nn.Module):
    MODE = "default"

    def _setup(self, encoder_class, encoder_kwargs, output_dim, projection_dim, momentum, center_momentum, dropout):
        self.student = encoder_class(**encoder_kwargs)
        self.teacher = encoder_class(**encoder_kwargs)
        self.teacher.load_state_dict(self.student.state_dict())
        self.student_projection = ProjectionHead(output_dim, projection_dim, dropout_rate=dropout)
        self.teacher_projection = ProjectionHead(output_dim, projection_dim)
        self.teacher_projection.load_state_dict(self.student_projection.state_dict())
        for p in list(self.teacher.parameters()) + list(self.teacher_projection.parameters()):
            p.requires_grad = False
        self.momentum, self.center_momentum = momentum, center_momentum
        self.register_buffer("center", torch.zeros(1, projection_dim))
        kind = getattr(encoder_class, "B200_KIND", None)
        if kind is None:
            raise NotImplementedError(f"{encoder_class.__name__} has no compiled B200 training step (compiled: {_COMPILED})")
        self._b200 = B.EngineBinding(self, kind, self.MODE)
        self.student_temperature, self.teacher_temperature = 0.1, 0.04
        self.n_global_views, self.n_local_views = 2, 4

    def b200_hparams(self):
        hp = dict(output_dim=self.output_dim, projection_dim=self.projection_dim, momentum=self.momentum,
                  center_momentum=self.center_momentum, dropout=self.dropout, student_temperature=self.student_temperature,
                  teacher_temperature=self.teacher_temperature, n_global_views=self.n_global_views, n_local_views=self.n_local_views)
        if hasattr(self, "encoder_output_dim"):
            hp["encoder_output_dim"] = self.encoder_output_dim
        # use_mixed_precision (the reference trains with precision='16-mixed', run_dino.py:360) selects the tensor-core path
        # (bf16 / fp16 activations, tf32 linears, fp32 accumulation); False runs the exact fp32 kernels
        hp["precision"] = "bf16" if getattr(self, "use_mixed_precision", True) else "fp32"
        return hp

    @property
    def engine(self):
        return self._b200.engine

    @torch.no_grad()
    def update_teacher(self):
        """teacher <- m * teacher + (1 - m) * student for encoder and projection head: one flat CUDA kernel."""
        self._b200.ensure(self.center.device).update_teacher()

    @torch.no_grad()
    def update_center(self, teacher_output):
        """centre <- m_c * centre + (1 - m_c) * mean_rows(teacher_output) (the training forward already does this)."""
        from multimodal_ssl_avmnist_b200 import ops
        t = teacher_output.detach().reshape(-1, self.center.shape[1]).contiguous().float()
        stats = torch.zeros(t.shape[1], 2, dtype=torch.float64, device=t.device)
        ops.colstats(t, stats)
        ops.center_apply(self.center, stats[:, 0].float().contiguous(), t.shape[0], self.center_momentum)

    def _views(self, batch):
        gi, ga, li, la = batch
        self.n_global_views, self.n_local_views = gi.shape[1], li.shape[1]
        dev = self.center.device
        return gi.to(dev), ga.to(dev), li.to(dev), la.to(dev)


class MultiModalDINO(_DinoBase):
    def __init__(self, encoder_class=SimpleMultiModalEncoder, encoder_kwargs=None, output_dim=256, encoder_output_dim=512,
                 projection_dim=128, momentum=0.996, center_momentum=0.9, dropout=0.3):
        super().__init__()
        self.projection_dim, self.output_dim, self.encoder_output_dim, self.dropout = projection_dim, output_dim, encoder_output_dim, dropout
        kw = dict(encoder_kwargs or {})
        kw["output_dim"], kw["encoder_output_dim"] = output_dim, encoder_output_dim
        self._setup(encoder_class, kw, output_dim, projection_dim, momentum, center_momentum, dropout)

    def forward(self, batch, raw=None):
        """batch = (global_images [B,Vg,1,28,28], global_audios [B,Vg,1,112,112], local_images, local_audios).
        Returns (student_outputs [V,B,P], teacher_outputs [Vg,B,P] (centred), None)."""
        gi, ga, li, la = self._views(batch)
        out = self._b200.forward(_to_view_major(gi, li), _to_view_major(ga, la), raw=raw)
        self._extra = out[2:]
        return out[0], out[1], None

    def forward_raw(self, images, audios, augment_values="keep", with_raw=False):
        """B200 fast path: un-augmented device batch (images [B,1,28,28] fp32/uint8, audios [B,1,112,112] uint8/fp32) ->
        device-sampled multi-crop augmentation -> the same outputs as forward()."""
        dev = self.center.device
        eng = self._b200.ensure(dev)
        if augment_values != "keep":
            eng.set_augmentation(augment_values)
        img = images.to(dev).reshape(-1, 28, 28).contiguous()
        aud = audios.to(dev).reshape(-1, 112, 112).contiguous()
        xi, xa = eng.augment(img, aud, direct=True)      # views go straight into the first conv's operand format
        raw = None
        if with_raw:
            raw = (img.float() / 255.0 if img.dtype == torch.uint8 else img, aud.float() / 255.0 if aud.dtype == torch.uint8 else aud)
        out = self._b200.forward(xi, xa, raw=raw)
        self._extra = out[2:]
        return out[0], out[1], None


class _WithSideHeads(MultiModalDINO):
    HEAD_NAMES = ("image_projection_head", "audio_projection_head")

    def _side_dim(self):
        return self.projection_dim

    def __init__(self, *args, **kwargs):
        super().__init__(*args, **kwargs)
        e = self.student.encoder_output_dim
        setattr(self, self.HEAD_NAMES[0], ProjectionHead(input_dim=e, projection_dim=self._side_dim()))
        setattr(self, self.HEAD_NAMES[1], ProjectionHead(input_dim=e, projection_dim=self._side_dim()))

    def forward(self, batch):
        """batch = (image [B,1,28,28], audio [B,1,112,112], views) -> (image_out, audio_out, student_out, teacher_out)."""
        image, audio, views = batch
        dev = self.center.device
        raw = (image.to(dev).float().reshape(-1, 28, 28).contiguous(), audio.to(dev).float().reshape(-1, 112, 112).contiguous())
        s, t, _ = super().forward(views, raw=raw)
        return self._extra[0], self._extra[1], s, t


class MultiModalDINOSemiSupervised(_WithSideHeads):
    MODE = "semi_supervised"
    HEAD_NAMES = ("image_classifier", "audio_classifier")

    def __init__(self, *args, num_classes=10, **kwargs):
        self.num_classes = num_classes
        super().__init__(*args, **kwargs)

    def _side_dim(self):
        return self.num_classes


class MultiModalDINOWithINFONCE(_WithSideHeads):
    MODE = "infonce"


class MultiModalDINOWithMSE(_WithSideHeads):
    MODE = "mse"


class UniModalDINO(_DinoBase):
    def __init__(self, encoder_class=ImageEncoder, encoder_kwargs=None, output_dim=256, projection_dim=128, momentum=0.996,
                 center_momentum=0.9, dropout=0.3):
        super().__init__()
        self.projection_dim, self.output_dim, self.dropout = projection_dim, output_dim, dropout
        kw = dict(encoder_kwargs or {})
        kw["output_dim"] = output_dim
        self._setup(encoder_class, kw, output_dim, projection_dim, momentum, center_momentum, dropout)

    def forward(self, batch):
        """batch = (global_images, global_audios, local_images, local_audios) views; the encoder's modality is used ('image':
        gi / li, 'audio': ga / la).  Returns (student_outputs [V,B,P], teacher_outputs [Vg,B,P] (centred), embeddings [V,B,O])."""
        gi, ga, li, la = self._views(batch)
        if self.student.modality == "image":
            out = self._b200.forward(_to_view_major(gi, li), None)
        else:
            out = self._b200.forward(None, _to_view_major(ga, la))
        return out[0], out[1], self._embeddings(gi.shape[0])

    def _embeddings(self, B):
        eng = self.engine
        return self._b200.last_w["s.feat"].view(eng.V, B, -1)

    def forward_raw(self, images, audios, augment_values="keep"):
        """B200 fast path: un-augmented device batch (images [B,1,28,28] fp32/uint8, audios [B,1,112,112] uint8/fp32; the
        modality the encoder does not read may be None) -> device-sampled multi-crop augmentation of the encoder's modality, written
        straight into the first convolution's operand format -> the same outputs as forward()."""
        dev = self.center.device
        eng = self._b200.ensure(dev)
        if augment_values != "keep":
            eng.set_augmentation(augment_values)
        if self.student.modality == "image":
            img, aud = images.to(dev).reshape(-1, 28, 28).contiguous(), None
        else:
            img, aud = None, audios.to(dev).reshape(-1, 112, 112).contiguous()
        xi, xa = eng.augment(img, aud, direct=True)
        out = self._b200.forward(xi, xa)
        return out[0], out[1], self._embeddings((img if img is not None else aud).shape[0])


# ------------------------------------------------------------------------------------------------------------
# Downstream models (reference models/dino.py:1764-1850): frozen-encoder features through the CUDA encoder forward
# ------------------------------------------------------------------------------------------------------------
class FeatureExtractor(nn.Module):
    """Frozen student-encoder features of un-augmented batches.  The reference deep-copies the encoder; here the weights are the
    live student's (identical while nothing trains in between) and the part of the copy that DOES change during a probe -- the
    BatchNorm running statistics, which adapt in train() mode and are read in eval() mode -- is a per-extractor copy held by the
    engine (DinoStepEngine.begin_probe).  train()/eval() select batch / running statistics exactly like the copy's mode would.

    is_dino_based=False: a stand-alone contrastive container (InfoNCEModel or MultiModalSimCLRModel; a Lightning module passes its
    `.model`).  Its features are cat([image_encoder(images), audio_encoder(spectrograms)], 1), so output_dim = 2 * the container's
    output_dim; the projection heads are not part of them.  The BatchNorm rules are the same, through ContrastiveStepEngine.begin_probe.
    The reference's body of this branch is not in this tree: these semantics are stated, not pinned (DESIGN.md section 4.12)."""

    def __init__(self, pretrained_model, is_dino_based=True):
        super().__init__()
        if is_dino_based:
            if not hasattr(pretrained_model, "_b200"):
                raise NotImplementedError("only DINO models with a compiled B200 step have a CUDA feature path")
            self.is_unimodal = hasattr(pretrained_model.student, "modality")
            self.modality = getattr(pretrained_model.student, "modality", None)
            self.output_dim = pretrained_model.student.output_dim
        else:
            if B.contrastive_binding(pretrained_model) is None:
                raise NotImplementedError("is_dino_based=False takes an InfoNCEModel or MultiModalSimCLRModel container")
            self.is_unimodal, self.modality = False, None
            self.output_dim = 2 * pretrained_model.output_dim
        self.is_dino_based = is_dino_based
        self._dino = [pretrained_model]                      # not registered: the encoder stays owned by the pretrained model
        self._probe = None

    def engine(self):
        """The step engine that computes the features (created and bound on first use)."""
        m = self._dino[0]
        return m._b200.ensure(m.center.device) if self.is_dino_based else B.contrastive_binding(m).ensure_eval()

    @torch.no_grad()
    def forward(self, images, spectrograms=None):
        eng = self.engine()
        if self._probe is None:
            self._probe = eng.begin_probe()
        img = aud = None
        if self.modality != "audio":
            img = images.to(eng.device).reshape(-1, 28, 28).contiguous()
        if self.modality == "audio" or not (self.is_unimodal or spectrograms is None):
            if spectrograms is None:
                raise ValueError("an audio-only model needs the spectrograms")
            aud = spectrograms.to(eng.device).reshape(-1, 112, 112).contiguous()
        return eng.encode_features(img, aud, train=self.training, probe=self._probe).clone()


class DownstreamClassifier(nn.Module):
    """Frozen encoder + Linear(output_dim, 128) -> ReLU -> Linear(128, num_classes) (reference models/dino.py:1764-1815).
    is_dino_based=False: a contrastive container's encoders, output_dim = 2 * its output_dim (FeatureExtractor)."""

    def __init__(self, pretrained_model, num_classes=10, trainable_encoder=False, is_dino_based=True):
        super().__init__()
        if trainable_encoder:
            raise NotImplementedError("fine-tuning the encoder through the probe is outside the B200 hot-path scope")
        self.encoder = FeatureExtractor(pretrained_model, is_dino_based=is_dino_based)
        self.is_unimodal, self.modality = self.encoder.is_unimodal, self.encoder.modality
        self.classifier = nn.Sequential(nn.Linear(self.encoder.output_dim, 128), nn.ReLU(), nn.Linear(128, num_classes))

    def forward(self, images, spectrograms=None):
        return self.classifier(self.encoder(images, spectrograms))


# ------------------------------------------------------------------------------------------------------------
# Lightning modules
# ------------------------------------------------------------------------------------------------------------
class _DinoLightningBase(pl.LightningModule):
    LOSS_VARIANT = 0
    # Raw (un-augmented) device batches of at most this many samples take the fused CUDA-graph step (EngineBinding.fused_train_step):
    # one graph replay per batch instead of ~165 launches + autograd + optimizer calls.  "auto": only under the built-in trainer shim
    # (real Lightning may run hooks between backward and optimizer.step that a fused step would bypass); True / False force it.
    b200_fused_step = "auto"
    B200_FUSED_MAX_BATCH = 512

    def _use_fused_step(self, batch_size):
        flag = self.b200_fused_step
        if flag == "auto":
            from _compat import HAVE_LIGHTNING
            flag = (not HAVE_LIGHTNING) and getattr(self, "_trainer", None) is not None
        return bool(flag) and batch_size <= self.B200_FUSED_MAX_BATCH and self.model._b200.optimizer is not None

    def forward(self, batch):
        return self.model(batch)

    def _augment_values(self):
        dm = getattr(getattr(self, "trainer", None), "datamodule", None)
        aug = getattr(dm, "augmentations", None)
        return getattr(aug, "augment_values", None)

    def dino_loss(self, student_outputs, teacher_outputs, alignment_loss=None):
        """Centred, temperature-sharpened cross-entropy over all student x teacher view pairs (fused CUDA kernel)."""
        return self.model._b200.dino_loss(student_outputs, teacher_outputs, self.student_temperature, self.teacher_temperature,
                                          self.LOSS_VARIANT) if self.model._b200.engine is not None else \
            B.standalone_dino_loss(student_outputs, teacher_outputs, self.student_temperature, self.teacher_temperature, self.LOSS_VARIANT)

    def _sync_hparams(self):
        m = self.model
        m.student_temperature, m.teacher_temperature = self.student_temperature, self.teacher_temperature
        m.use_mixed_precision = bool(getattr(self, "use_mixed_precision", True))
        if m.engine is not None:
            m.engine.tau_s, m.engine.tau_t = self.student_temperature, self.teacher_temperature

    def configure_optimizers(self):
        """Adam(lr, weight_decay) + CosineAnnealingLR(T_max=num_epochs), stepped per epoch; the optimiser is the flat-arena
        CUDA Adam behind a torch.optim.Optimizer front."""
        opt = B.B200Adam(self.parameters(), self.model._b200, lr=self.learning_rate, weight_decay=self.weight_decay)
        sched = torch.optim.lr_scheduler.CosineAnnealingLR(opt, T_max=self.num_epochs)
        return {"optimizer": opt, "lr_scheduler": {"scheduler": sched}}

    def probe_accuracy(self, train_loader, val_loader, max_batches=None):
        """The reference's per-epoch linear probe (models/dino.py:878-951): a fresh 2-layer MLP on frozen student features,
        one epoch of AdamW(lr) on train-mode features, then accuracy on eval-mode features.  Returns (val_loss, mlp_acc %).
        The encoder forward runs on the CUDA kernels; the 33k-parameter probe itself is plain torch."""
        dev = self.model.center.device
        probe = DownstreamClassifier(self.model, trainable_encoder=False).to(dev)
        opt = torch.optim.AdamW(probe.classifier.parameters(), lr=self.learning_rate)
        crit = nn.CrossEntropyLoss()
        probe.train()
        total, nb = 0.0, 0
        for bi, batch in enumerate(train_loader):
            if max_batches is not None and bi >= max_batches:
                break
            images, audios, labels = batch[0].to(dev), batch[1].to(dev), batch[2].to(dev)
            opt.zero_grad()
            loss = crit(probe(images, audios), labels)
            loss.backward()
            opt.step()
            total, nb = total + float(loss), nb + 1
        probe.eval()
        correct = count = 0
        with torch.no_grad():
            for bi, batch in enumerate(val_loader):
                if max_batches is not None and bi >= max_batches:
                    break
                images, audios, labels = batch[0].to(dev), batch[1].to(dev), batch[2].to(dev)
                correct += int((probe(images, audios).argmax(1) == labels).sum())
                count += int(labels.numel())
        return total / max(nb, 1), 100.0 * correct / max(count, 1)

    def on_train_epoch_end(self):
        """Logs `val_loss` / `mlp_acc` like the reference (models/dino.py:878-951) when the trainer's data module provides
        labelled loaders (`probe_dataloaders()` -> (train, val)); otherwise only the training loss is available."""
        dm = getattr(getattr(self, "trainer", None), "datamodule", None)
        get = getattr(dm, "probe_dataloaders", None)
        if get is None:
            return None
        val_loss, acc = self.probe_accuracy(*get())
        self.log("val_loss", val_loss)
        self.log("mlp_acc", acc, on_epoch=True, prog_bar=True)
        return None


class MultiModalDINOLightning(_DinoLightningBase):
    MODEL_CLASS = MultiModalDINO

    def __init__(self, data_dir="data/avmnist", data_augmentation="burst_noise", dino_model=None, encoder_class=SimpleMultiModalEncoder,
                 encoder_kwargs=None, projection_dim=256, output_dim=256, encoder_output_dim=512, momentum=0.996, center_momentum=0.9,
                 student_temperature=0.1, teacher_temperature=0.04, learning_rate=0.0001, use_mixed_precision=True, num_epochs=100,
                 weight_decay=1e-6, dropout=0.3):
        super().__init__()
        self.encoder_class, self.encoder_kwargs = encoder_class, encoder_kwargs
        self.output_dim, self.encoder_output_dim, self.projection_dim = output_dim, encoder_output_dim, projection_dim
        self.learning_rate, self.weight_decay, self.num_epochs = learning_rate, weight_decay, num_epochs
        self.student_temperature, self.teacher_temperature = student_temperature, teacher_temperature
        self.use_mixed_precision = use_mixed_precision          # True: tensor-core path (bf16/fp16/tf32 operands); False: exact fp32 kernels
        self.momentum, self.center_momentum, self.dropout = momentum, center_momentum, dropout
        self.data_dir, self.data_augmentation = data_dir, data_augmentation
        if dino_model is None:
            self.build_model()
        else:
            self.model = dino_model
        self._sync_hparams()
        self.save_hyperparameters(ignore=["dino_model", "traindata", "validdata", "testdata"])

    def build_model(self):
        self.model = self.MODEL_CLASS(encoder_class=self.encoder_class, encoder_kwargs=self.encoder_kwargs, output_dim=self.output_dim,
                                      encoder_output_dim=self.encoder_output_dim, projection_dim=self.projection_dim,
                                      momentum=self.momentum, center_momentum=self.center_momentum, dropout=self.dropout)
        return self.model

    def training_step(self, batch, batch_idx):
        self._sync_hparams()
        if len(batch) in (2, 3) and batch[0].dim() == 4:          # raw (image, audio[, label]) batch: augment on the device
            av = "keep" if getattr(self, "_aug_set", False) else self._augment_values()
            self._aug_set = True
            if self._use_fused_step(batch[0].shape[0]):           # small batch: the whole step is one CUDA-graph replay
                dev = self.model.center.device
                if av != "keep":
                    self.model._b200.ensure(dev).set_augmentation(av)
                loss = self.model._b200.fused_train_step(batch[0].to(dev), batch[1].to(dev))
                if loss is not None:
                    self.log("train_loss", loss, on_step=True, on_epoch=True, prog_bar=True)
                    return loss
            student_out, teacher_out, alignment_loss = self.model.forward_raw(batch[0], batch[1], av)
        else:
            student_out, teacher_out, alignment_loss = self.model(batch)
        loss = self.dino_loss(student_out, teacher_out, alignment_loss)
        self.model.update_teacher()
        self.log("train_loss", loss, on_step=True, on_epoch=True, prog_bar=True)
        return loss


class _SideLossLightning(MultiModalDINOLightning):
    def side_loss(self, image_out, audio_out, labels):
        raise NotImplementedError

    def training_step(self, batch, batch_idx):
        self._sync_hparams()
        if len(batch) == 3:                                       # raw (image, audio, label) batch: augment on the device
            image, audio, labels = batch
            av = "keep" if getattr(self, "_aug_set", False) else self._augment_values()
            self._aug_set = True
            if self._use_fused_step(image.shape[0]):               # small batch: the whole step (side loss included) is one graph replay
                dev = self.model.center.device
                if av != "keep":
                    self.model._b200.ensure(dev).set_augmentation(av)
                loss = self.model._b200.fused_train_step(image.to(dev), audio.to(dev), labels.to(dev), alpha=float(self.alpha))
                if loss is not None:
                    self.log("train_loss", loss, on_step=True, on_epoch=True, prog_bar=True)
                    return loss
            student_out, teacher_out, _ = self.model.forward_raw(image, audio, av, with_raw=True)
            image_out, audio_out = self.model._extra
        else:
            image, audio, labels, views = batch
            image_out, audio_out, student_out, teacher_out = self.model((image, audio, views))
        loss = self.dino_loss(student_out, teacher_out) + self.alpha * self.side_loss(image_out, audio_out, labels)
        self.model.update_teacher()
        self.log("train_loss", loss, on_step=True, on_epoch=True, prog_bar=True)
        return loss


class MultiModalDINOSemiSupervisedLightning(_SideLossLightning):
    MODEL_CLASS = MultiModalDINOSemiSupervised

    def __init__(self, *args, alpha=1, **kwargs):
        super().__init__(*args, **kwargs)
        self.alpha = alpha

    def supervised_loss(self, image_logits, audio_logits, labels):
        labels = labels.to(image_logits.device)
        return B.standalone_ce_loss(image_logits, labels) + B.standalone_ce_loss(audio_logits, labels)

    def side_loss(self, image_out, audio_out, labels):
        return self.supervised_loss(image_out, audio_out, labels)


class MultiModalDINOWithINFONCELightning(_SideLossLightning):
    MODEL_CLASS = MultiModalDINOWithINFONCE

    def __init__(self, *args, output_dim=256, encoder_output_dim=128, encoder_class=SimpleMultiModalEncoder, alpha=1, **kwargs):
        super().__init__(*args, output_dim=output_dim, encoder_output_dim=encoder_output_dim, encoder_class=encoder_class, **kwargs)
        self.alpha = alpha

    def infoNCE_loss(self, image_outputs, audio_outputs, temperature=0.07):
        return B.standalone_pair_loss("infonce", image_outputs, audio_outputs, temperature=temperature)

    def side_loss(self, image_out, audio_out, labels):
        return self.infoNCE_loss(image_out, audio_out)


class MultiModalDINOWithMSELightning(_SideLossLightning):
    MODEL_CLASS = MultiModalDINOWithMSE

    def __init__(self, *args, output_dim=256, encoder_output_dim=128, encoder_class=SimpleMultiModalEncoder, alpha=1, **kwargs):
        super().__init__(*args, output_dim=output_dim, encoder_output_dim=encoder_output_dim, encoder_class=encoder_class, **kwargs)
        self.alpha = alpha

    def mse_loss(self, image_outputs, audio_outputs):
        return B.standalone_pair_loss("mse", image_outputs, audio_outputs)

    def side_loss(self, image_out, audio_out, labels):
        return self.mse_loss(image_out, audio_out)


class UniModalDINOLightning(_DinoLightningBase):
    LOSS_VARIANT = 1

    def __init__(self, data_dir="data/avmnist", dino_model=None, encoder_class=ImageEncoder, encoder_kwargs=None, projection_dim=128,
                 output_dim=256, momentum=0.996, center_momentum=0.9, student_temperature=0.1, teacher_temperature=0.04,
                 learning_rate=0.0001, use_mixed_precision=True, weight_decay=1e-6, cosine_loss_alpha=0.3, dropout=0.3, num_epochs=10,
                 data_augmentation="burst_noise", use_original_model=True):
        super().__init__()
        if dino_model is None:
            if not use_original_model:
                raise NotImplementedError("UniModalDINOV2 is outside the B200 hot-path scope")
            self.model = UniModalDINO(encoder_class=encoder_class, encoder_kwargs=encoder_kwargs, projection_dim=projection_dim,
                                      output_dim=output_dim, momentum=momentum, center_momentum=center_momentum, dropout=dropout)
        else:
            self.model = dino_model
        self.learning_rate, self.weight_decay, self.num_epochs = learning_rate, weight_decay, num_epochs
        self.student_temperature, self.teacher_temperature = student_temperature, teacher_temperature
        self.use_mixed_precision, self.dropout, self.cosine_loss_alpha = use_mixed_precision, dropout, cosine_loss_alpha
        self.data_dir, self.data_augmentation = data_dir, data_augmentation
        self._sync_hparams()
        self.save_hyperparameters(ignore=["dino_model", "traindata", "validdata", "testdata"])

    def _cosine_consistency_loss(self, embeddings):
        return B.standalone_cosine_loss(embeddings)

    def training_step(self, batch, batch_idx):
        """batch = the reference's 4-tuple of views, or a raw (image, audio[, label]) batch that is augmented on the device (the
        default AVMNISTDinoDataModule); small raw batches take the fused CUDA-graph step like the multimodal modules."""
        self._sync_hparams()
        if len(batch) in (2, 3) and batch[0].dim() == 4:          # raw (image, audio[, label]) batch: augment on the device
            av = "keep" if getattr(self, "_aug_set", False) else self._augment_values()
            self._aug_set = True
            audio_only = self.model.student.modality == "audio"
            if self._use_fused_step(batch[0].shape[0]):           # small batch: the whole step is one CUDA-graph replay
                dev = self.model.center.device
                if av != "keep":
                    self.model._b200.ensure(dev).set_augmentation(av)
                images, audios = (None, batch[1].to(dev)) if audio_only else (batch[0].to(dev), None)
                loss = self.model._b200.fused_train_step(images, audios, cosine_loss_alpha=float(self.cosine_loss_alpha))
                if loss is not None:
                    self.log("train_loss", loss, on_step=True, on_epoch=True, prog_bar=True)
                    return loss
            student_out, teacher_out, embeddings = self.model.forward_raw(None if audio_only else batch[0], batch[1] if audio_only else None, av)
        else:
            student_out, teacher_out, embeddings = self.model(batch)
        loss = self.dino_loss(student_out, teacher_out)
        cosine_loss = None
        if self.cosine_loss_alpha > 0:
            # total = dino + alpha * cosine (reference models/dino.py:1651-1656).  The value comes from the fused kernel here;
            # its gradient w.r.t. the embeddings is added by the engine's backward pass (engine.cosine_loss_alpha), so the
            # term enters the autograd graph as a constant and is not counted twice
            eng = self.model.engine
            eng.cosine_loss_alpha = float(self.cosine_loss_alpha)
            cosine_loss = self._cosine_consistency_loss(embeddings).detach()
            loss = loss + self.cosine_loss_alpha * cosine_loss
        elif self.model.engine is not None:
            self.model.engine.cosine_loss_alpha = 0.0
        self.model.update_teacher()
        self.log("train_loss", loss, on_step=True, on_epoch=True, prog_bar=True)
        if cosine_loss is not None:
            self.log("cosine_loss", cosine_loss, on_step=True, on_epoch=True, prog_bar=True)
        return loss
