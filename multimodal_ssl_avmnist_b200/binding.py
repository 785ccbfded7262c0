"""Glue between the reference-shaped nn.Modules (AVMNIST_Experiments/models/dino.py) and the step engine.

`EngineBinding` adopts a DINO module's parameters and buffers into the engine's flat arenas (each `nn.Parameter.data`
becomes a view of the arena, BatchNorm buffers and the centre are aliased), and exposes the training step as ordinary
autograd-visible tensors:

    student_out, teacher_out[, image_out, audio_out] = binding.forward(views[, raw])     # CUDA forward, no autograd tape
    loss = binding.dino_loss(student_out, teacher_out, tau_s, tau_t)                      # fused CUDA loss fwd+bwd
    loss.backward()                                                                        # CUDA backward -> p.grad views

`student_out` carries a custom grad_fn: whatever scalar the caller builds from it (the fused loss, or the reference's
own torch expression), `backward()` hands d loss / d student_out to the engine's backward kernels, which fill the flat
gradient arena; every parameter's `.grad` is a view of that arena, so torch optimisers and the arena Adam both work.
"""
import torch

from . import ops
from .engine import DinoStepEngine


class B200Adam(torch.optim.Optimizer):
    """torch.optim.Adam-compatible front (param_groups, lr schedulers, state_dict) whose step() is ONE flat-arena CUDA
    kernel over the parameters that received gradients (plus one for the mode heads).

    The moments and the step counter live in the engine's flat arenas, but they BELONG to this optimizer object: a new
    B200Adam starts from zero moments and step 0 exactly like a new torch.optim.Adam (run_dino.py builds a fresh optimizer per
    seed / per fit, run_dino.py:94-104), and state_dict() / load_state_dict() carry them through checkpoints."""

    def __init__(self, params, binding, lr=1e-4, weight_decay=0.0, betas=(0.9, 0.999), eps=1e-8):
        super().__init__(params, dict(lr=lr, weight_decay=weight_decay, betas=betas, eps=eps))
        self.binding = binding
        self._fresh = True                 # the engine's moments still hold a previous optimizer's state
        self._pending_state = None
        binding.optimizer = self

    def _claim_engine(self, eng):
        """First contact with the engine: reset (or restore) the Adam state it holds."""
        if self._fresh:
            eng.reset_optimizer_state()
            self._fresh = False
        if self._pending_state is not None:
            eng.load_optimizer_state(self._pending_state)
            self._pending_state = None

    @torch.no_grad()
    def step(self, closure=None):
        loss = closure() if closure is not None else None
        eng = self.binding.engine
        if eng is None:
            raise ops._lib.B200Error("B200Adam.step() before the first CUDA forward")
        if self.binding.step_applied:        # the fused (CUDA-graph) training_step already ran EMA + Adam for this batch
            self.binding.step_applied = False
            return loss
        self._claim_engine(eng)
        g = self.param_groups[0]
        eng.lr, eng.weight_decay = g["lr"], g["weight_decay"]
        eng.optimizer_step()
        return loss

    def state_dict(self):
        sd = super().state_dict()
        eng = self.binding.engine
        if eng is not None and not self._fresh:
            sd["b200_arena_state"] = eng.optimizer_state()
        elif self._pending_state is not None:
            sd["b200_arena_state"] = self._pending_state
        return sd

    def load_state_dict(self, state_dict):
        state_dict = dict(state_dict)
        arena = state_dict.pop("b200_arena_state", None)
        super().load_state_dict(state_dict)
        if arena is not None:
            self._pending_state = arena
            eng = self.binding.engine
            if eng is not None:
                self._fresh = False
                self._claim_engine(eng)


class _StudentOutputs(torch.autograd.Function):
    """Marks the engine's forward outputs as differentiable w.r.t. the student parameters."""

    @staticmethod
    def forward(ctx, binding, anchor, *outs):
        ctx.binding = binding
        ctx.n = len(outs)
        return tuple(o.view_as(o) for o in outs)

    @staticmethod
    def backward(ctx, *grads):
        b = ctx.binding
        d_proj = grads[0]
        d_aux = None
        if ctx.n > 1:
            d_aux = [g if g is not None else torch.zeros_like(o) for g, o in zip(grads[1:], b.last_aux)]
            d_aux = [g.contiguous() for g in d_aux]
        if d_proj is None:
            d_proj = torch.zeros_like(b.last_w["s.proj"])
        b.engine.backward_pass(b.last_w, d_proj=d_proj.contiguous(), d_aux=d_aux)
        b.publish_grads()
        return (None, None) + (None,) * ctx.n


class _AppliedLoss(torch.autograd.Function):
    """The loss of a step that has ALREADY been applied (fused CUDA-graph step: forward, backward, EMA and Adam in one replay):
    a scalar that takes part in autograd so that the trainer's `loss.backward()` is legal, with nothing left to propagate."""

    @staticmethod
    def forward(ctx, loss_value, anchor):
        return loss_value.clone()

    @staticmethod
    def backward(ctx, g):
        return None, None


class _FusedLoss(torch.autograd.Function):
    """loss value + its pre-computed gradient w.r.t. the inputs (the CUDA loss kernels compute both in one pass)."""

    @staticmethod
    def forward(ctx, loss_value, *pairs):
        n = len(pairs) // 2
        ctx.save_for_backward(*pairs[n:])
        return loss_value.clone()

    @staticmethod
    def backward(ctx, g):
        return (None,) + tuple(g * d for d in ctx.saved_tensors) + (None,) * len(ctx.saved_tensors)


def fused_loss(loss_value, inputs, grads):
    return _FusedLoss.apply(loss_value, *inputs, *grads)


class EngineBinding:
    def __init__(self, module, kind, mode="default"):
        self.module, self.kind, self.mode = module, kind, mode
        self.engine = None
        self.last_w = None
        self.last_aux = ()
        self._names = None
        self.optimizer = None              # the B200Adam that owns the arena Adam state (set by its constructor)
        self.step_applied = False          # fused_train_step ran the whole step: the next optimizer.step() is a no-op

    # ---- adoption -------------------------------------------------------------------------------------------
    def _name_map(self):
        """module parameter name -> (arena, arena key)."""
        m = {}
        eng = self.engine
        aux_names = {"image_classifier": "aux_image", "image_projection_head": "aux_image", "audio_classifier": "aux_audio",
                     "audio_projection_head": "aux_audio"}
        for name, _ in self.module.named_parameters():
            top, rest = name.split(".", 1)
            if top == "student":
                m[name] = ("S", "enc." + rest)
            elif top == "teacher":
                m[name] = ("T", "enc." + rest)
            elif top == "student_projection":
                m[name] = ("S", "head." + rest)
            elif top == "teacher_projection":
                m[name] = ("T", "head." + rest)
            elif top in aux_names:
                m[name] = ("S", aux_names[top] + "." + rest)
            else:
                raise ops._lib.B200Error(f"parameter '{name}' has no place in the engine arenas")
        for name, (which, key) in m.items():
            if key not in (eng.S if which == "S" else eng.T):
                raise ops._lib.B200Error(f"parameter '{name}' ({key}) is not part of the compiled '{self.kind}' step")
        return m

    def ensure(self, device):
        """Create the engine on first use and (re-)adopt the module's tensors if they were moved (`.to()`, load)."""
        mod = self.module
        if self.engine is None:
            hp = mod.b200_hparams()
            # augmentation / dropout streams: the global torch seed (run_dino.py seeds it per run) + the rank, so that seeds and
            # data-parallel ranks draw different views and masks
            import os
            rank = int(os.environ.get("RANK", "0")) if torch.distributed.is_available() and torch.distributed.is_initialized() else 0
            hp.setdefault("seed", (int(torch.initial_seed()) + rank) & 0x7FFFFFFF)
            self.engine = DinoStepEngine(kind=self.kind, mode=self.mode, device=device, **hp)
            self._names = self._name_map()
        eng = self.engine
        params = dict(mod.named_parameters())
        probe_name = next(iter(self._names))
        which, key = self._names[probe_name]
        if params[probe_name].data_ptr() == (eng.S if which == "S" else eng.T)[key].data_ptr():
            return eng
        with torch.no_grad():
            for name, p in params.items():
                which, key = self._names[name]
                view = (eng.S if which == "S" else eng.T)[key]
                view.copy_(p.data.to(eng.device))
                p.data = view
            # BatchNorm buffers and the centre: the engine uses the module's own tensors
            mods = dict(mod.named_modules())
            for role, table, prefix in (("student", eng.bn_s, "enc."), ("teacher", eng.bn_t, "enc."), ("student_projection", eng.bn_s, "head."),
                                        ("teacher_projection", eng.bn_t, "head."), ("image_classifier", eng.bn_s, "aux_image."),
                                        ("image_projection_head", eng.bn_s, "aux_image."), ("audio_classifier", eng.bn_s, "aux_audio."),
                                        ("audio_projection_head", eng.bn_s, "aux_audio.")):
                if role not in mods:
                    continue
                for sub, m_ in mods[role].named_modules():
                    if isinstance(m_, torch.nn.modules.batchnorm._BatchNorm) and prefix + sub in table:
                        bn = table[prefix + sub]
                        for attr in ("running_mean", "running_var", "num_batches_tracked"):
                            t = getattr(m_, attr)
                            if t.device != eng.device:
                                t.data = t.data.to(eng.device)
                        bn.running_mean, bn.running_var = m_.running_mean, m_.running_var
                        bn.num_batches_tracked = m_.num_batches_tracked
            if mod.center.device != eng.device:
                mod.center.data = mod.center.data.to(eng.device)
            eng.center = mod.center
        return eng

    def publish_grads(self):
        """Point every student parameter's .grad at its slice of the gradient arena."""
        eng = self.engine
        for name, p in self.module.named_parameters():
            which, key = self._names[name]
            if which == "S" and p.requires_grad:
                p.grad = eng.G[key]

    # ---- the step, as autograd-visible pieces ------------------------------------------------------------------
    def forward(self, x_img, x_aud, raw=None, masks=None):
        """x_img [V,B,28,28] / x_aud [V,B,112,112] view-major device tensors (None for a modality the kind does not encode).
        Returns (student_out [V,B,P], teacher_out [Vg,B,P] centred with the pre-update centre[, image_out, audio_out])."""
        x_in = x_img if x_img is not None else x_aud
        eng = self.ensure(x_in.device)
        B = x_in.shape[1]
        center_before = eng.center.clone()
        w = eng.forward_pass(x_img, x_aud, masks=masks, raw=raw)
        eng.dino_loss_pass(w)             # fused loss fwd+bwd + centre EMA (the reference updates the centre inside forward)
        self.last_w = w
        P = eng.P
        teacher_c = (w["t.proj"] - center_before.view(1, P)).view(eng.Vg, B, P)
        outs = [w["s.proj"].view(eng.V, B, P)]
        if eng.mode != "default":
            outs += [w["aux_image.out"], w["aux_audio.out"]]
        self.last_aux = tuple(outs[1:])
        anchor = next(p for p in self.module.student.parameters() if p.requires_grad)
        res = _StudentOutputs.apply(self, anchor, *outs)
        eng.rng_step += 1
        return (res[0], teacher_c) + tuple(res[1:])

    def fused_train_step(self, images, audios, labels=None, alpha=1.0, cosine_loss_alpha=None):
        """The WHOLE training step of a raw device batch as one CUDA-graph replay (augmentation, forward, losses, centre / teacher EMA,
        backward, gradient exchange, Adam): for small per-GPU batches, where the ~165 launches of the step-by-step module path cost
        more host time than GPU time (B = 128: 3.0 -> 1.9 ms).  The graph is captured on first use per batch size; the learning rate
        follows the optimizer's param_groups (device scalar), Adam state belongs to the current B200Adam.  Returns the total loss as
        an autograd-visible scalar whose backward is a no-op, and marks the step as applied for the next optimizer.step(); None if a
        graph for a different batch size / weight decay / alpha is already captured (the caller then takes the step-by-step path).
        images or audios may be None for a modality the kind does not encode; cosine_loss_alpha (unimodal kinds) sets the weight of
        the cosine-consistency term baked into the graph (None: the engine's current value)."""
        x_in = images if images is not None else audios
        eng = self.ensure(x_in.device)
        opt = self.optimizer
        if opt is None:
            raise ops._lib.B200Error("fused_train_step needs the B200Adam from configure_optimizers()")
        opt._claim_engine(eng)
        g0 = opt.param_groups[0]
        eng.lr = g0["lr"]
        img = None if images is None else images.reshape(-1, 28, 28).contiguous()
        aud = None if audios is None else audios.reshape(-1, 112, 112).contiguous()
        B = (img if img is not None else aud).shape[0]
        cos = float(eng.cosine_loss_alpha if cosine_loss_alpha is None else cosine_loss_alpha)
        key = (B, None if img is None else img.dtype, None if aud is None else aud.dtype, float(g0["weight_decay"]), float(alpha))
        if cos != 0.0:
            key += (cos,)
        if eng._graph is not None and eng._graph.get("key") != key:
            return None                    # a graph for another batch size / setting exists: this batch takes the step-by-step path
        if eng._graph is None:
            eng.weight_decay, eng.alpha, eng.cosine_loss_alpha = g0["weight_decay"], float(alpha), cos
            eng.capture_train_step(B, image_dtype=torch.float32 if img is None else img.dtype,
                                   audio_dtype=torch.uint8 if aud is None else aud.dtype)
            eng._graph["key"] = key
        loss = eng.graph_step(img, aud, labels)
        self.step_applied = True
        anchor = next(p for p in self.module.student.parameters() if p.requires_grad)
        return _AppliedLoss.apply(loss[3], anchor)

    def dino_loss(self, student_out, teacher_out, tau_s, tau_t, variant):
        """Fused CUDA loss.  If the tensors are the ones the last forward produced (and the temperatures match the
        engine's) the already-computed loss/gradient are reused; otherwise the loss kernel runs on the given tensors."""
        eng, w = self.engine, self.last_w
        same = (w is not None and student_out.data_ptr() == w["s.proj"].data_ptr() and tau_s == eng.tau_s and tau_t == eng.tau_t)
        if same:
            return fused_loss(w["loss"][0], (student_out,), (w["d.proj"].view_as(student_out),))
        return standalone_dino_loss(student_out, teacher_out, tau_s, tau_t, variant)


def standalone_dino_loss(student_out, teacher_out, tau_s, tau_t, variant=0):
    """DINO loss of arbitrary CUDA tensors [Vs,B,D], [Vt,B,D] (teacher already centred) through the fused kernel."""
    s = student_out.detach().contiguous().float()
    t = teacher_out.detach().contiguous().float()
    Vs, B, D = s.shape
    zero = torch.zeros(D, device=s.device)
    parts = ops.dino_loss_parts(B)
    grad = torch.empty_like(s)
    pl_, pc = torch.empty(parts, device=s.device), torch.empty(parts, D, device=s.device)
    cm = None
    if variant == 1:
        cm = torch.empty(t.shape[0], D, device=s.device)
        ops.teacher_norm_colmean(t, zero, cm)
    ops.dino_loss_fwd_bwd(s, t, zero, tau_s, tau_t, grad, pl_, pc, variant=variant, t_colmean=cm)
    loss = torch.empty(1, device=s.device)
    ops.center_update(None, pc, pl_, t.shape[0] * B, 0.9, loss, colsum_out=torch.empty(D, device=s.device))
    return fused_loss(loss[0], (student_out,), (grad,))


def standalone_pair_loss(kind, a, b, **kw):
    """mse / infonce of two [B,D] CUDA tensors through the fused kernels, differentiable w.r.t. both."""
    x, y = a.detach().contiguous().float(), b.detach().contiguous().float()
    ga, gb, lo = torch.empty_like(x), torch.empty_like(y), torch.empty(1, device=x.device)
    if kind == "mse":
        ops.mse_align_fwd_bwd(x, y, ga, gb, lo)
    else:
        work = torch.empty(ops.infonce_work_floats(*x.shape), device=x.device)
        ops.infonce_fwd_bwd(x, y, ga, gb, lo, work, temperature=kw.get("temperature", 0.07))
    return fused_loss(lo[0], (a, b), (ga, gb))


def standalone_ntxent_loss(reps, temperature=0.07):
    """SimCLR NT-Xent of reps [2B, D] = cat([z1, z2]) (other_ssl/multimodal_simclr/multimodal_simclr.py:74-89) through the fused
    kernel, differentiable w.r.t. reps (a drop-in for MultiModalSimCLRLightning.nt_xent_loss on CUDA tensors)."""
    x = reps.detach().contiguous().float()
    g, lo = torch.empty_like(x), torch.empty(1, device=x.device)
    work = torch.empty(ops.ntxent_work_floats(*x.shape), device=x.device)
    ops.ntxent_fwd_bwd(x, g, lo, work, temperature=temperature)
    return fused_loss(lo[0], (reps,), (g,))


def standalone_ce_loss(logits, labels):
    x = logits.detach().contiguous().float()
    g, lo = torch.empty_like(x), torch.empty(1, device=x.device)
    ops.ce_fwd_bwd(x, labels.contiguous(), g, lo)
    return fused_loss(lo[0], (logits,), (g,))


def standalone_cosine_loss(emb):
    x = emb.detach().contiguous().float()
    g, lo = torch.empty_like(x), torch.empty(1, device=x.device)
    ops.cosine_consistency_fwd_bwd(x, g, lo)
    return fused_loss(lo[0], (emb,), (g,))


# ------------------------------------------------------------------------------------------------------------
# stand-alone contrastive models (other_ssl/info_nce, other_ssl/multimodal_simclr)
# ------------------------------------------------------------------------------------------------------------
class ContrastiveAdam(torch.optim.Optimizer):
    """torch.optim.Adam-shaped front of ContrastiveStepEngine.optimizer_step(): Adam(lr), no weight decay, over the branches that
    received gradients in the last training_step, one step count per branch (what torch's per-parameter step state amounts to)."""

    def __init__(self, params, binding, lr=1e-4):
        super().__init__(params, dict(lr=lr, weight_decay=0.0, betas=(0.9, 0.999), eps=1e-8))
        self.binding = binding

    @torch.no_grad()
    def step(self, closure=None):
        loss = closure() if closure is not None else None
        eng = self.binding.engine
        if eng is None:
            raise ops._lib.B200Error("ContrastiveAdam.step() before the first CUDA training_step")
        eng.lr = self.param_groups[0]["lr"]
        eng.optimizer_step()
        return loss


class ContrastiveBinding:
    """Adopts the parameters / BatchNorm buffers of an InfoNCEModel or MultiModalSimCLRModel container into a ContrastiveStepEngine
    (module tensors become views of the engine's arena) and runs the reference's training_step on it."""

    def __init__(self, model, kind):
        self.model, self.kind, self.engine = model, kind, None

    def ensure(self, device):
        from .contrastive import ContrastiveStepEngine
        m = self.model
        if self.engine is None:
            self.engine = ContrastiveStepEngine(kind=self.kind, output_dim=m.output_dim, projection_dim=m.projection_dim, device=device,
                                                seed=int(torch.initial_seed()) & 0x7FFFFFFF,
                                                precision="bf16" if getattr(m, "use_mixed_precision", True) else "fp32")
        eng = self.engine
        params = dict(m.named_parameters())
        first = next(iter(params))
        if params[first].data_ptr() == eng.S["enc." + first].data_ptr():
            return eng
        with torch.no_grad():
            for name, p in params.items():
                view = eng.S["enc." + name]
                view.copy_(p.data.to(eng.device))
                p.data = view
            for name, mod in m.named_modules():
                if isinstance(mod, torch.nn.modules.batchnorm._BatchNorm):
                    bn = eng.bn_s["enc." + name]
                    for attr in ("running_mean", "running_var", "num_batches_tracked"):
                        t = getattr(mod, attr)
                        if t.device != eng.device:
                            t.data = t.data.to(eng.device)
                    bn.running_mean, bn.running_var, bn.num_batches_tracked = mod.running_mean, mod.running_var, mod.num_batches_tracked
        return eng

    def training_step(self, batch, mode=None):
        """Forward + loss + backward on the CUDA kernels; gradients land in the arena (every used parameter's .grad is a view of it,
        unused branches get .grad = None like in the reference).  Returns the loss as an autograd-visible scalar whose backward is a no-op."""
        dev = batch[0].device if batch[0].is_cuda else torch.device("cuda", torch.cuda.current_device())
        eng = self.ensure(dev)
        views = [t.to(dev).float().reshape(t.shape[0], *t.shape[-2:]).contiguous() for t in batch]
        loss = eng.forward_backward(tuple(views), mode=mode)
        used = {"img": ("image_encoder", "image_projection_head"), "aud": ("audio_encoder", "audio_projection_head")}
        live = {m for b in eng._used for m in used[b]}
        for name, p in self.model.named_parameters():
            p.grad = eng.G["enc." + name] if name.split(".", 1)[0] in live else None
        anchor = next(self.model.parameters())
        return _AppliedLoss.apply(loss[3], anchor)
