"""Stand-alone contrastive training steps of the reference's `other_ssl/` models on the same CUDA kernels (SURVEY 8f-4, BASELINE config 4).

  * kind="infonce" -- MultiModalInfoNCELightning (other_ssl/info_nce/info_nce.py:15-36, 120-142): ImageEncoder(images) and
    SpectrogramEncoder(spectrograms) of the UN-augmented batch, one ProjectionHead each, symmetric InfoNCE between the modalities;
  * kind="simclr"  -- MultiModalSimCLRLightning (other_ssl/multimodal_simclr/multimodal_simclr.py:12-46, 74-110): two augmented views
    (SimCLRMultiModalAugmentation), a random modality pairing per step (image-image, audio-audio, image-audio, audio-image), NT-Xent on
    cat([z1, z2]).

Both: Adam(lr) without weight decay, no teacher, no EMA.  torch's Adam skips parameters that received no gradient and counts steps per
parameter, so the branch (encoder + head of one modality) that a SimCLR step did not use is left untouched and keeps its own step count.

The engine reuses DinoStepEngine's building blocks (tensor-core conv stacks with their fused first-layer backward, BatchNorm / pool
kernels, linear kernels, flat-arena Adam) with its own parameter inventory and schedule; parameters are named as in the reference's
state_dict (`image_encoder.encoder.0.weight`, `audio_projection_head.mlp.4.bias`, ...).  No CPU fallback.

Evaluation: encode_features / begin_probe give the frozen features cat([image_encoder(x), audio_encoder(x)], 1) on the same
conv-stack kernels, for the kNN and MLP-probe evaluation (FeatureExtractor(model, is_dino_based=False), probe.ProbeSession).
"""
import math

import numpy as np
import torch

from . import dp
from . import ops
from .engine import F32, Arena, DinoStepEngine, _BN, _conv, _lin, _vec2, _zero_arena, head_params

IMG_LAYERS = [("image_encoder.encoder.0", "image_encoder.encoder.1", 1, 32, 28, 3, 1), ("image_encoder.encoder.4", "image_encoder.encoder.5", 32, 64, 14, 3, 1),
              ("image_encoder.encoder.8", "image_encoder.encoder.9", 64, 128, 7, 3, 1)]
AUD_LAYERS = [("audio_encoder.encoder.0", "audio_encoder.encoder.1", 1, 32, 112, 3, 1), ("audio_encoder.encoder.4", "audio_encoder.encoder.5", 32, 64, 56, 3, 1),
              ("audio_encoder.encoder.8", "audio_encoder.encoder.9", 64, 128, 28, 3, 1), ("audio_encoder.encoder.12", "audio_encoder.encoder.13", 128, 256, 14, 3, 1)]
# SimCLR modality pairing: (encoder of view 1, encoder of view 2), multimodal_simclr.py:31-44
MODES = (("img", "img"), ("aud", "aud"), ("img", "aud"), ("aud", "img"))


def contrastive_params(O, P):
    """Parameter specs per branch, names as in InfoNCEModel / MultiModalSimCLRModel.state_dict() (reference declaration order inside
    each module)."""
    img = []
    for i, (ci, co) in zip((0, 4, 8), ((1, 32), (32, 64), (64, 128))):
        img += _conv(f"image_encoder.encoder.{i}", co, ci, 3) + _vec2(f"image_encoder.encoder.{i + 1}", co)
    img += _lin("image_encoder.encoder.14", 512, 128) + _lin("image_encoder.projection.0", O, 512)
    img += [("image_projection_head." + n, s) for n, s in head_params(O, P)]
    aud = []
    for i, (ci, co) in zip((0, 4, 8, 12), ((1, 32), (32, 64), (64, 128), (128, 256))):
        aud += _conv(f"audio_encoder.encoder.{i}", co, ci, 3) + _vec2(f"audio_encoder.encoder.{i + 1}", co)
    aud += _lin("audio_encoder.encoder.18", O, 256)
    aud += [("audio_projection_head." + n, s) for n, s in head_params(O, P)]
    return img, aud


class ContrastiveStepEngine(DinoStepEngine):
    def __init__(self, kind="infonce", output_dim=256, projection_dim=256, learning_rate=1e-4, temperature=0.07, seed=0, device=None,
                 precision="bf16", process_group=None, data_parallel=None, mode_seed=0):
        if not torch.cuda.is_available():
            raise ops._lib.B200Error("ContrastiveStepEngine needs a CUDA device: the hot path has no CPU fallback")
        ops._lib.load()
        assert kind in ("infonce", "simclr") and precision in ("bf16", "fp32")
        self.device = torch.device(device if device is not None else f"cuda:{torch.cuda.current_device()}")
        self.kind, self.mode, self.precision = kind, "default", precision
        self.lin_tc = precision == "bf16"
        self.multi, self.mix = False, None
        self.O, self.P = output_dim, projection_dim
        self.lr, self.weight_decay, self.temperature = learning_rate, 0.0, temperature
        self.seed, self.rng_step = seed, 0
        # data parallel (one process per GPU): samples sharded over the ranks, BatchNorm statistics and contrastive negatives rank-local
        # (what Lightning's DDP gives the reference), ONE exchange per step: all-reduce of the gradients of the branches the step used,
        # through the C ABI (b200_dp_allreduce_grads) on a communication stream; the 1 / world average is folded into Adam's grad_scale
        self.pg = process_group
        self.world = dp.world_size(process_group) if (data_parallel is None or data_parallel) else 1
        self.comm, self._comm_stream = None, None
        self._ctr = self._bc = self._graph = None
        self.img_layers, self.aud_layers = IMG_LAYERS, AUD_LAYERS
        img, aud = contrastive_params(self.O, self.P)
        self.student = Arena([("enc." + n, s) for n, s in img + aud], self.device)
        self.branch_range = {"img": self.student.range_of(["enc." + n for n, _ in img]), "aud": self.student.range_of(["enc." + n for n, _ in aud])}
        self.step_counts = {"img": 0, "aud": 0}                 # Adam steps taken per branch (torch: per-parameter step state)
        self.grad = torch.zeros_like(self.student.flat)
        self.exp_avg, self.exp_avg_sq = torch.zeros_like(self.student.flat), torch.zeros_like(self.student.flat)
        self.S, self.G = self.student.views(), self.student.views(self.grad)
        self.bn_s = {}
        for conv, bn, ci, co, hw, k, pad in IMG_LAYERS + AUD_LAYERS:
            self.bn_s["enc." + bn] = _BN(co, self.device)
        for m in ("image", "audio"):
            self.bn_s[f"enc.{m}_projection_head.mlp.1"] = _BN(512, self.device)
        self._select_tc_layers(("s",))
        # no max-pool in the forward epilogues: for these 32 - 256 channel layers the fused variant measured slower than conv + pool pass
        # (engine.py, profiles/r2zf_*)
        self.fused_pool = False
        self.pool = {r: {mod: [False] * len(layers) for mod, layers in (("img", IMG_LAYERS), ("aud", AUD_LAYERS))} for r in ("s", "t")}
        self.fused_bnstat = False
        self.bnstat = {mod: [False] * len(layers) for mod, layers in (("img", IMG_LAYERS), ("aud", AUD_LAYERS))}
        self.overlap_teacher = True
        self._lin_wg_stream = torch.cuda.Stream(device=self.device)
        self._lin_wg_pending = False
        self._wgrad_streams = {m: torch.cuda.Stream(device=self.device) for m in ("img", "aud")}
        self._ws = {}
        # host draw of the SimCLR modality pairing (torch.randint in the reference): the SAME sequence on every rank (mode_seed, not the
        # per-rank seed), so that all ranks run -- and exchange -- the same branches
        self._mode_rng = torch.Generator().manual_seed(mode_seed)
        if self.world > 1:
            self.comm = dp.AbiComm.get(process_group)
            self._comm_stream = torch.cuda.Stream(device=self.device)
        self._comm_pending = False
        self._init_parameters()

    # ------------------------------------------------------------------------------------------------------
    def _init_parameters(self):
        g = torch.Generator(device="cpu").manual_seed(self.seed)
        bn_bases = set(self.bn_s)
        bounds = {}
        for name, shape in self.student.spec:
            v = self.student.view(name)
            base = name.rsplit(".", 1)[0]
            if base in bn_bases:
                v.fill_(1.0 if name.endswith(".weight") else 0.0)
            else:
                if len(shape) > 1:
                    bounds[base] = 1.0 / math.sqrt(int(np.prod(shape[1:])))
                v.copy_(((torch.rand(shape, generator=g) * 2 - 1) * bounds[base]).to(self.device))

    def load_named(self, params):
        """params: {module: {name: tensor}} with the reference's names, e.g. params['image_encoder']['encoder.0.weight']."""
        for m, d in params.items():
            for k, v in d.items():
                self.S[f"enc.{m}.{k}"].copy_(v.to(self.device))

    def sync_teacher(self):          # no teacher here
        pass

    def _dino_only(self, *a, **k):
        raise ops._lib.B200Error("this entry point belongs to the DINO step engine; the contrastive engine offers forward_backward / "
                                 "optimizer_step / train_step_views / train_step / capture_train_step / graph_step / begin_probe / "
                                 "encode_features")

    # inherited DINO-specific entry points that have no meaning here
    forward_pass = dino_loss_pass = aux_loss_pass = backward_pass = update_teacher = train_step_host = _dino_only
    augment = augment_with_params = prefetch_augment = allreduce_gradients = graph_node_counts = _dino_only

    # ------------------------------------------------------------------------------------------------------
    # evaluation-side encoder forward: frozen features for the kNN and MLP-probe evaluation (DESIGN.md section 4.12)
    # ------------------------------------------------------------------------------------------------------
    def _eval_workspace(self, B):
        key = ("eval", B)
        if key in self._ws:
            return self._ws[key]
        dev = self.device

        def e(*shape, dtype=F32):
            return torch.empty(*shape, dtype=dtype, device=dev)

        w = {"B": B}
        w["zarena"], zalloc = _zero_arena(1 << 12, dev)
        w["x_img"], w["x_aud"] = e(B, 1, 28, 28), e(B, 1, 112, 112)
        self._stack_buffers(w, "e", B, B, e, zalloc)
        w["img.gap"], w["img.e14"], w["aud.gap"] = e(B, 128), e(B, 512), e(B, 256)
        w["feat"] = e(B, 2 * self.O)          # [image_encoder(x) | audio_encoder(x)]
        self._ws[key] = w
        return w

    def begin_probe(self):
        """Start a probe session: a token holding a private copy of the seven conv-stack BatchNorms' running statistics (initialised
        from the live ones), which train-mode encode_features(probe=token) updates and eval-mode reads.  The live statistics are never
        touched.  The projection heads' BatchNorms are not part of the features and are not copied."""
        bns = {}
        for conv, bn, *_ in IMG_LAYERS + AUD_LAYERS:
            v = self.bn_s["enc." + bn]
            c = _BN(v.C, self.device)
            c.running_mean.copy_(v.running_mean)
            c.running_var.copy_(v.running_var)
            c.num_batches_tracked.copy_(v.num_batches_tracked)
            bns["enc." + bn] = c
        return {"bns": bns, "step": 0, "teacher": False}

    @torch.no_grad()
    def encode_features(self, images, audios, train=False, probe=None, step_dev=None):
        """Frozen features [B, 2*O] = cat([image_encoder(images), audio_encoder(audios)], 1) of an UN-augmented batch (images [B,28,28]
        or [B,1,28,28], audios [B,112,112] or [B,1,112,112]; fp32 in [0, 1] or uint8).  The projection heads are not applied.
        train=False: BatchNorm with running statistics (module.eval()); train=True: batch statistics.  probe (a begin_probe() token):
        the running statistics read / updated are the token's; without one, train-mode updates go to scratch and eval reads the live
        ones.  step_dev is accepted for probe.ProbeSession's captured step; these encoders have no dropout and do not read it.
        Returns a view of the per-batch-size workspace, overwritten by the next call with the same B."""
        if images is None or audios is None:
            raise ops._lib.B200Error("encode_features: a contrastive container's features need both the image and the spectrogram batch")
        B = self._batch_size(images, audios)
        w = self._eval_workspace(B)
        if probe is not None:
            bns = probe["bns"]
        elif train:
            bns = {"enc." + bn: _BN(co, self.device) for conv, bn, ci, co, *_ in IMG_LAYERS + AUD_LAYERS}
        else:
            bns = self.bn_s
        xi, xa = w["x_img"], w["x_aud"]
        xi.copy_((images.float() / 255.0 if images.dtype == torch.uint8 else images).reshape(B, 1, 28, 28))
        xa.copy_((audios.float() / 255.0 if audios.dtype == torch.uint8 else audios).reshape(B, 1, 112, 112))
        self._prep_tc_weights("s", self.S)
        for mod, layers, x in (("img", IMG_LAYERS, xi), ("aud", AUD_LAYERS, xa)):
            if self.tc[mod][0]:
                ops.pack_quad8(x.view(B, layers[0][4], layers[0][4]), w[f"{mod}.xs8"], layers[0][6])
        w["packed"] = True
        self._eval_wrole = "s"
        w["zarena"].zero_()                             # the BatchNorm statistics of every layer
        S, O, feat = self.S, self.O, w["feat"]
        pi = self._conv_stack(w, "e", "img", IMG_LAYERS, xi, B, B, S, bns, train=train)
        ops.avgpool_fwd(pi, w["img.gap"])
        ops.linear_fwd(w["img.gap"], S["enc.image_encoder.encoder.14.weight"], S["enc.image_encoder.encoder.14.bias"], w["img.e14"], tc=self.lin_tc)
        ops.linear_fwd(w["img.e14"], S["enc.image_encoder.projection.0.weight"], S["enc.image_encoder.projection.0.bias"], feat[:, :O], tc=self.lin_tc)
        pa = self._conv_stack(w, "e", "aud", AUD_LAYERS, xa, B, B, S, bns, train=train)
        ops.avgpool_fwd(pa, w["aud.gap"])
        ops.linear_fwd(w["aud.gap"], S["enc.audio_encoder.encoder.18.weight"], S["enc.audio_encoder.encoder.18.bias"], feat[:, O:], tc=self.lin_tc)
        return feat

    # ------------------------------------------------------------------------------------------------------
    def _workspace(self, B):
        """Buffers for up to two encoder calls per modality; _combo() hands out the prefix views of a (calls_img, calls_aud) schedule."""
        if B in self._ws:
            return self._ws[B]
        dev = self.device

        def e(*shape, dtype=F32):
            return torch.empty(*shape, dtype=dtype, device=dev)

        w = {"B": B}
        w["zarena"], zalloc = _zero_arena(1 << 16, dev)
        N = 2 * B
        w["x_img"], w["x_aud"] = e(N, 1, 28, 28), e(N, 1, 112, 112)
        self._stack_buffers(w, "s", N, B, e, zalloc)
        O, P = self.O, self.P
        w["img.gap"], w["img.e14"], w["aud.gap"] = e(N, 128), e(N, 512), e(N, 256)
        w["d.img.gap"], w["d.img.e14"], w["d.aud.gap"] = e(N, 128), e(N, 512), e(N, 256)
        for mod in ("img", "aud"):
            w[f"{mod}.feat"], w[f"d.{mod}.feat"] = e(N, O), e(N, O)
            w[f"{mod}.hh"], w[f"{mod}.g"], w[f"{mod}.d.hh"], w[f"{mod}.d.g"] = e(N, 512), e(N, 512), e(N, 512), e(N, 512)
            w[f"{mod}.hstats"], w[f"{mod}.hsums"] = zalloc(2, 512, 2), zalloc(2, 512, 2)
            for nm in ("hscale", "hshift", "hmean", "hinvstd"):
                w[f"{mod}.{nm}"] = e(2, 512)
        w["reps"], w["d.reps"] = e(N, P), e(N, P)
        w["loss"] = torch.zeros(4, device=dev)
        w["ntxent_work"] = e(ops.ntxent_work_floats(N, P))
        w["infonce_work"] = e(ops.infonce_work_floats(B, P, tc=self.lin_tc))
        self._ws[B] = w
        return w

    def _combo(self, w, mod, calls):
        """Prefix views (N = calls * B samples) of the modality's stack buffers, keyed like DinoStepEngine's workspace."""
        key = ("combo", mod, calls)
        if key in w:
            return w[key]
        B = w["B"]
        N = calls * B
        c = {"B": B, "zarena": w["zarena"], "packed": False}
        for k, v in w.items():
            if not isinstance(k, str) or not isinstance(v, torch.Tensor):
                continue
            if k.startswith(f"s.{mod}.") and k.split(".")[2].rstrip("0123456789") in ("stats", "sums", "scale", "shift", "mean", "invstd"):
                c[k] = v[:calls]
            elif k.startswith(f"s.{mod}.") or k == f"{mod}.xs8":
                c[k] = v[:N]
            elif k.startswith(f"{mod}."):
                c[k] = v                                  # backward scratch: flat, sized for the largest schedule
        w[key] = c
        return c

    # ------------------------------------------------------------------------------------------------------
    def _branch_fwd(self, w, mod, x, calls):
        """Encoder + projection head of one modality on `calls` view-calls of B samples each; returns z [calls*B, P] (a view of w)."""
        B, S = w["B"], self.S
        N = calls * B
        c = self._combo(w, mod, calls)
        layers = IMG_LAYERS if mod == "img" else AUD_LAYERS
        hw = layers[0][4]
        xin = w[f"x_{mod}"][:N]
        xin.copy_(x.reshape(N, 1, hw, hw))
        if self.tc[mod][0]:
            ops.pack_quad8(xin.view(N, hw, hw), c[f"{mod}.xs8"], layers[0][6])
            c["packed"] = True
        p_last = self._conv_stack(c, "s", mod, layers, xin, N, B, S, self.bn_s)
        if mod == "img":          # ImageEncoder: encoder = image_encoder(512), projection = Linear(512, O) (models/dino.py:483-499)
            ops.avgpool_fwd(p_last, w["img.gap"][:N])
            ops.linear_fwd(w["img.gap"][:N], S["enc.image_encoder.encoder.14.weight"], S["enc.image_encoder.encoder.14.bias"], w["img.e14"][:N], tc=self.lin_tc)
            ops.linear_fwd(w["img.e14"][:N], S["enc.image_encoder.projection.0.weight"], S["enc.image_encoder.projection.0.bias"], w["img.feat"][:N], tc=self.lin_tc)
            head = "enc.image_projection_head."
        else:                     # SpectrogramEncoder: encoder = audio_encoder(O) (models/dino.py:502-513)
            ops.avgpool_fwd(p_last, w["aud.gap"][:N])
            ops.linear_fwd(w["aud.gap"][:N], S["enc.audio_encoder.encoder.18.weight"], S["enc.audio_encoder.encoder.18.bias"], w["aud.feat"][:N], tc=self.lin_tc)
            head = "enc.audio_projection_head."
        # ProjectionHead, called once per view-call in the reference: BatchNorm1d statistics per call, the linears batched
        feat, hh, g = w[f"{mod}.feat"][:N], w[f"{mod}.hh"][:N], w[f"{mod}.g"][:N]
        ops.linear_fwd(feat, S[head + "mlp.0.weight"], S[head + "mlp.0.bias"], hh, tc=self.lin_tc)
        st = w[f"{mod}.hstats"][:calls]
        for cc in range(calls):
            ops.colstats(hh[cc * B:(cc + 1) * B], st[cc])
        bn = self.bn_s[head + "mlp.1"]
        sc, sh, mu, inv = (w[f"{mod}.{n}"][:calls] for n in ("hscale", "hshift", "hmean", "hinvstd"))
        ops.bn_finalize(st, S[head + "mlp.1.weight"], S[head + "mlp.1.bias"], bn.running_mean, bn.running_var, bn.num_batches_tracked, sc, sh, mu, inv, calls, B)
        for cc in range(calls):
            r = slice(cc * B, (cc + 1) * B)
            ops.bn1d_gelu_drop_fwd(hh[r], sc[cc:cc + 1], sh[cc:cc + 1], None, 0.0, g[r])
        return g, head

    def _branch_bwd(self, w, mod, d_z, calls):
        """Backward of one branch from d loss / d z [calls*B, P]."""
        B, S, G = w["B"], self.S, self.G
        N = calls * B
        c = self._combo(w, mod, calls)
        layers = IMG_LAYERS if mod == "img" else AUD_LAYERS
        head = "enc.image_projection_head." if mod == "img" else "enc.audio_projection_head."
        feat, hh, g, d_g, d_hh = (w[f"{mod}.{n}"][:N] for n in ("feat", "hh", "g", "d.g", "d.hh"))
        self._lin_wgrad(d_z, g, G[head + "mlp.4.weight"], G[head + "mlp.4.bias"])
        ops.linear_bwd_data(d_z, S[head + "mlp.4.weight"], d_g, tc=self.lin_tc)
        sums = w[f"{mod}.hsums"][:calls]
        sc, sh, mu, inv = (w[f"{mod}.{n}"][:calls] for n in ("hscale", "hshift", "hmean", "hinvstd"))
        for cc in range(calls):
            r, v = slice(cc * B, (cc + 1) * B), slice(cc, cc + 1)
            ops.bn1d_gelu_drop_bwd_reduce(hh[r], d_g[r], sc[v], sh[v], mu[v], inv[v], None, 0.0, sums[cc])
            ops.bn1d_gelu_drop_bwd_apply(hh[r], d_g[r], sc[v], sh[v], mu[v], inv[v], None, 0.0, sums[cc], d_hh[r])
        ops.bn_param_grads(sums, G[head + "mlp.1.weight"], G[head + "mlp.1.bias"], calls)
        self._lin_wgrad(d_hh, feat, G[head + "mlp.0.weight"], G[head + "mlp.0.bias"])
        d_feat = w[f"d.{mod}.feat"][:N]
        ops.linear_bwd_data(d_hh, S[head + "mlp.0.weight"], d_feat, tc=self.lin_tc)
        p_last = c[f"s.{mod}.p{len(layers) - 1}"]
        if mod == "img":
            self._lin_wgrad(d_feat, w["img.e14"][:N], G["enc.image_encoder.projection.0.weight"], G["enc.image_encoder.projection.0.bias"])
            ops.linear_bwd_data(d_feat, S["enc.image_encoder.projection.0.weight"], w["d.img.e14"][:N], tc=self.lin_tc)
            self._lin_wgrad(w["d.img.e14"][:N], w["img.gap"][:N], G["enc.image_encoder.encoder.14.weight"], G["enc.image_encoder.encoder.14.bias"])
            ops.linear_bwd_data(w["d.img.e14"][:N], S["enc.image_encoder.encoder.14.weight"], w["d.img.gap"][:N], tc=self.lin_tc)
        else:
            self._lin_wgrad(d_feat, w["aud.gap"][:N], G["enc.audio_encoder.encoder.18.weight"], G["enc.audio_encoder.encoder.18.bias"])
            ops.linear_bwd_data(d_feat, S["enc.audio_encoder.encoder.18.weight"], w["d.aud.gap"][:N], tc=self.lin_tc)
        d_p = w[f"{mod}.dp_a"][:p_last.numel()].view_as(p_last)
        ops.avgpool_bwd(w[f"d.{mod}.gap"][:N], d_p)
        self._conv_stack_bwd(c, mod, layers, w[f"x_{mod}"][:N], d_p, N, B)

    # ------------------------------------------------------------------------------------------------------
    def forward_backward(self, batch, mode=None):
        """infonce: batch = (images [B,28,28], spectrograms [B,112,112]) fp32 device tensors (un-augmented).
        simclr:  batch = (img1, spec1, img2, spec2) augmented views; mode 0..3 (default: drawn from the engine's host generator).
        Leaves the gradients of the branches that were used in self.grad and returns (loss tensor [4] (loss at [3]), used branches)."""
        B = batch[0].shape[0]
        w = self._workspace(B)
        w["zarena"].zero_()
        self._prep_tc_weights("s", self.S)
        P = self.P
        if self.kind == "infonce":
            sched = {"img": [batch[0]], "aud": [batch[1]]}
            order = [("img", 0), ("aud", 0)]
        else:
            if mode is None:
                mode = int(torch.randint(0, 4, (1,), generator=self._mode_rng))
            m1, m2 = MODES[mode]
            sched = {"img": [], "aud": []}
            order = []
            for view, mod in enumerate((m1, m2)):
                order.append((mod, len(sched[mod])))
                sched[mod].append(batch[2 * view + (0 if mod == "img" else 1)])
        z, heads = {}, {}
        for mod in ("img", "aud"):
            calls = len(sched[mod])
            if calls:
                x = torch.cat([t.reshape(B, -1) for t in sched[mod]]) if calls > 1 else sched[mod][0]
                z[mod], heads[mod] = self._branch_fwd(w, mod, x, calls)
        # projection outputs in view order -> reps = cat([z1, z2])
        reps = w["reps"]
        for view, (mod, cc) in enumerate(order):
            g = z[mod][cc * B:(cc + 1) * B]
            ops.linear_fwd(g, self.S[heads[mod] + "mlp.4.weight"], self.S[heads[mod] + "mlp.4.bias"], reps[view * B:(view + 1) * B], tc=self.lin_tc)
        loss, d_reps = w["loss"], w["d.reps"]
        loss.zero_()
        if self.kind == "infonce":
            ops.infonce_fwd_bwd(reps[:B], reps[B:], d_reps[:B], d_reps[B:], loss[3:4], w["infonce_work"], temperature=self.temperature, tc=self.lin_tc)
        else:
            ops.ntxent_fwd_bwd(reps, d_reps, loss[3:4], w["ntxent_work"], temperature=self.temperature)
        for mod in ("img", "aud"):
            calls = len(sched[mod])
            if not calls:
                continue
            first = min(v for v, (m, _) in enumerate(order) if m == mod)        # the branch's rows of reps are contiguous, in call order
            d_z = d_reps[first * B:(first + calls) * B]
            self._branch_bwd(w, mod, d_z, calls)
        if self._lin_wg_pending:
            torch.cuda.current_stream().wait_stream(self._lin_wg_stream)
            self._lin_wg_pending = False
        self._used = [m for m in ("img", "aud") if sched[m]]
        if self.world > 1:
            main, cs = torch.cuda.current_stream(), self._comm_stream
            cs.wait_stream(main)
            with torch.cuda.stream(cs):
                for mod in self._used:
                    lo, hi = self.branch_range[mod]
                    self.comm.allreduce_grads_(self.grad[lo:hi], cs.cuda_stream)
            self._comm_pending = True
        return loss

    def optimizer_step(self):
        """Adam(lr), no weight decay, over the branches that received gradients; one step count per branch."""
        gs = 1.0 / self.world
        if self._comm_pending:
            torch.cuda.current_stream().wait_stream(self._comm_stream)
            self._comm_pending = False
        if self._ctr is not None:       # CUDA-graph mode (infonce: both branches step together): step and learning rate live on the device
            ops.adam_bias_dev(self._ctr[1:2], self._bc)
            for mod in self._used:
                lo, hi = self.branch_range[mod]
                ops.adam_flat_dev(self.student.flat[lo:hi], self.grad[lo:hi], self.exp_avg[lo:hi], self.exp_avg_sq[lo:hi], self._bc, -1.0, weight_decay=0.0,
                                  grad_scale=gs)
            ops.counters_advance(self._ctr)
            return
        for mod in self._used:
            self.step_counts[mod] += 1
            lo, hi = self.branch_range[mod]
            ops.adam_flat(self.student.flat[lo:hi], self.grad[lo:hi], self.exp_avg[lo:hi], self.exp_avg_sq[lo:hi], self.step_counts[mod], self.lr,
                          weight_decay=0.0, grad_scale=gs)

    # ------------------------------------------------------------------------------------------------------
    def capture_train_step(self, B, image_dtype=torch.float32, audio_dtype=torch.uint8):
        """kind="infonce": the whole step (forward, InfoNCE, backward, Adam) of a raw batch of B samples as ONE CUDA graph -- at the
        reference notebook's B = 128 the ~150 launches of a step cost more host time than GPU time.  The Adam step count and the
        learning rate are device scalars (schedulers may change self.lr between replays).  Use graph_step() afterwards.  (The SimCLR step
        draws its modality pairing and its augmentation parameters on the host every step and is not captured.)"""
        if self.kind != "infonce":
            raise ops._lib.B200Error("capture_train_step: only the InfoNCE step has a step-invariant launch sequence")
        if self.step_counts["img"] != self.step_counts["aud"]:
            raise ops._lib.B200Error("capture_train_step: the two branches must have taken the same number of Adam steps")
        dev = self.device
        g = {"B": B, "img": torch.zeros(B, 28, 28, dtype=image_dtype, device=dev), "aud": torch.zeros(B, 112, 112, dtype=audio_dtype, device=dev)}
        state = [self.student.flat, self.exp_avg, self.exp_avg_sq]
        for bn in self.bn_s.values():
            state += [bn.running_mean, bn.running_var, bn.num_batches_tracked]
        snap = [t.clone() for t in state]
        host = int(self.step_counts["img"])
        self._ctr = torch.tensor([0, host], dtype=torch.int64, device=dev)
        self._bc = torch.zeros(3, device=dev)
        self._bc[2:3].fill_(float(self.lr))
        self._graph_lr = float(self.lr)

        def restore():
            for t, c in zip(state, snap):
                t.copy_(c)
            self._ctr.copy_(torch.tensor([0, host], dtype=torch.int64))

        side = torch.cuda.Stream(device=dev)
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side):
            for _ in range(2):
                self.train_step(g["img"], g["aud"])
        torch.cuda.current_stream().wait_stream(side)
        torch.cuda.synchronize()
        restore()
        graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(graph):
            g["loss"] = self.train_step(g["img"], g["aud"])
        restore()
        torch.cuda.synchronize()
        g["graph"] = graph
        self._graph = g
        return g

    def graph_step(self, images, audios):
        g = self._graph
        if g is None or images.shape[0] != g["B"]:
            raise ops._lib.B200Error("graph_step: call capture_train_step(B) for this batch size first")
        g["img"].copy_(images.reshape(g["img"].shape))
        g["aud"].copy_(audios.reshape(g["aud"].shape))
        if float(self.lr) != self._graph_lr:
            self._graph_lr = float(self.lr)
            self._bc[2:3].fill_(self._graph_lr)
        g["graph"].replay()
        for mod in ("img", "aud"):
            self.step_counts[mod] += 1
        self.rng_step += 1
        return g["loss"]

    def release_graph(self):
        self._graph = None
        self._ctr = self._bc = None

    def train_step_views(self, batch, mode=None):
        loss = self.forward_backward(batch, mode=mode)
        self.optimizer_step()
        self.rng_step += 1
        return loss

    def train_step(self, images, audios, mode=None):
        """Raw device batch (images [B,28,28] fp32 in [0,1] or uint8, audios [B,112,112] uint8 or fp32).  infonce: the un-augmented batch is
        the input; simclr: two views per modality from the device SimCLR augmentation (throughput mode of SimCLRMultiModalAugmentation)."""
        B = images.shape[0]
        img = images.float() / 255.0 if images.dtype == torch.uint8 else images
        aud = audios.float() / 255.0 if audios.dtype == torch.uint8 else audios
        if self.kind == "infonce":
            return self.train_step_views((img.reshape(B, 28, 28), aud.reshape(B, 112, 112)))
        v = self._simclr_views(img, aud)
        return self.train_step_views(v, mode=mode)

    def _simclr_views(self, img, aud):
        """Two augmented views per modality like SimCLRMultiModalAugmentation (utils/get_data.py:299-408): ONE parameter set per batch and
        view, drawn on the host in the reference's RNG order (a dozen scalars + a 28x28 elastic grid when that op fires); the pixels and
        the per-element Gaussian noise come from the augmentation kernels (device Philox noise in this throughput path)."""
        from . import augment as A
        if not hasattr(self, "_hs"):
            self._hs, self._chains = A.HostSampler(), A.simclr_chains()
        dev, B, V = self.device, img.shape[0], 2
        img_ops = np.zeros((1, V, A.MAX_OPS, A.OP_WORDS), dtype=np.int32)
        aud_ops = np.zeros_like(img_ops)
        grids = np.zeros((1, V, 2, 28, 28), dtype=np.float32)
        for v in range(V):
            o, _, _ = self._hs.sample_view(self._chains[0], 28, 28)
            A.pack_ops(o, img_ops[0, v])
            if self._hs.last_grid is not None:
                grids[0, v] = self._hs.last_grid
        for v in range(V):
            o, _, _ = self._hs.sample_view(self._chains[1], 112, 112)
            A.pack_ops(o, aud_ops[0, v])
        io = torch.from_numpy(img_ops).to(dev).expand(B, -1, -1, -1).contiguous()
        ao = torch.from_numpy(aud_ops).to(dev).expand(B, -1, -1, -1).contiguous()
        gr = torch.from_numpy(grids).to(dev).expand(B, -1, -1, -1, -1).contiguous()
        w = self._workspace(B)
        if "aug_i" not in w:
            w["aug_i"], w["aug_a"] = torch.empty(V, B, 28, 28, device=dev), torch.empty(V, B, 112, 112, device=dev)
            w["aug_bits"] = torch.zeros(B, V, A.GROUP_WORDS, dtype=torch.int32, device=dev)
        ops.aug_apply_image(img.reshape(B, 28, 28).contiguous(), io, w["aug_i"], elastic_grid=gr)
        ops.aug_apply_audio(aud.reshape(B, 112, 112).contiguous(), ao, w["aug_bits"], w["aug_a"], seed=(self.seed * 1000003 + self.rng_step) & 0xFFFFFFFFFFFF)
        return w["aug_i"][0], w["aug_a"][0], w["aug_i"][1], w["aug_a"][1]
