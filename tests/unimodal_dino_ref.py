"""CPU restatement of the unimodal DINO training step (UniModalDINO + UniModalDINOLightning) for the audio-only and image-only
encoders.  TEST INFRASTRUCTURE ONLY: a composition of pieces of oracle/dino_ref.py that are pinned against the imported reference
elsewhere -- the encoder forwards, projection_head, dino_loss_unimodal, cosine_consistency_loss, the EMA and Adam.  The reference
implementation is not part of this tree, so no golden of the spectrogram step exists; the image-encoder instance of the same step is
checked against the reference's own unimodal goldens (tests/test_unimodal_spectrogram_cpu.py)."""
import torch

from oracle import dino_ref as R


def spectrogram_simple_encoder(spec, p, buf, train=True):
    """SpectrogramEncoder.forward (models/dino.py:502-513): audio_encoder(O) under the `encoder.*` names, i.e.
    dino_ref.simple_audio_features(pre="encoder") -- four conv blocks, global average pool, encoder.18 = Linear(256, O)."""
    return R.simple_audio_features(spec, p, buf, pre="encoder", train=train)


# ------------------------------------------------------------------------------------------------------------
# whole unimodal step (UniModalDINO + UniModalDINOLightning, models/dino.py:1560-1660)
# ------------------------------------------------------------------------------------------------------------

# kind -> (encoder parameter spec, BatchNorm names, encoder forward)
UNIMODAL_KINDS = {"image_simple": (R.image_simple_spec, R.image_simple_bn_names, lambda x, p, buf: R.image_simple_encoder(x, p, buf)),
                  "spectrogram_simple": (R.spectrogram_spec, R.spectrogram_bn_names, spectrogram_simple_encoder)}


class UniModalDinoState:
    """All state of UniModalDINO(ImageEncoder | SpectrogramEncoder) as flat dicts (same layout as CentralDinoState, no mode heads)."""

    def __init__(self, kind="spectrogram_simple", seed=0, O=256, P=128, dtype=torch.float32):
        spec_fn, bn_fn, _ = UNIMODAL_KINDS[kind]
        self.kind, self.O, self.P, self.mode, self.dtype = kind, O, P, "default", dtype
        self.enc_spec = spec_fn(O)
        self.head_spec = R.head_spec(O, P)
        self.bn_names = bn_fn()
        self.student = R.make_params(self.enc_spec, seed, dtype)
        self.student_head = R.make_params(self.head_spec, seed + 1, dtype)
        self.teacher = {k: v.clone() for k, v in self.student.items()}
        self.teacher_head = {k: v.clone() for k, v in self.student_head.items()}
        self.student_buf = R.make_bn_buffers(self.enc_spec, self.bn_names, dtype)
        self.teacher_buf = R.make_bn_buffers(self.enc_spec, self.bn_names, dtype)
        self.student_head_buf = R.make_bn_buffers(self.head_spec, ["mlp.1"], dtype)
        self.teacher_head_buf = R.make_bn_buffers(self.head_spec, ["mlp.1"], dtype)
        self.center = torch.zeros(1, P, dtype=dtype)
        self.aux = {}
        self.adam = {}


def unimodal_dino_step(st, views, masks, n_global=2, tau_s=0.1, tau_t=0.04, momentum=0.996, center_momentum=0.9, lr=1e-4,
                       weight_decay=1e-6, dropout=0.3, cosine_loss_alpha=0.0, do_adam=True):
    """One UniModalDINOLightning training step in the live order: student on all views and teacher on the global views (BatchNorm
    statistics per view-call), projection heads, centre update, dino_loss_unimodal (+ cosine_loss_alpha * cosine consistency on the
    embeddings), the teacher EMA before backward, and one Adam over encoder + head.

    views [V,B,1,H,W] of the encoder's modality (global views first); masks: 'student_head' keep-mask [V*B,512].
    total = dino + cosine_loss_alpha * cosine (models/dino.py:1651-1656).  Returns dict(loss, dino, cosine, grads{student,
    student_head}, student_out, teacher_out (centred), embeddings [V,B,O])."""
    V, B = views.shape[0], views.shape[1]
    enc = UNIMODAL_KINDS[st.kind][2]
    S = {k: v.clone().requires_grad_(True) for k, v in st.student.items()}
    SH = {k: v.clone().requires_grad_(True) for k, v in st.student_head.items()}
    emb = torch.cat([enc(views[v], S, st.student_buf) for v in range(V)])
    with torch.no_grad():
        teacher_features = torch.cat([enc(views[v], st.teacher, st.teacher_buf) for v in range(n_global)])
    student_projs = R.projection_head(emb, SH, st.student_head_buf, masks["student_head"], dropout)
    with torch.no_grad():
        teacher_projs = R.projection_head(teacher_features, st.teacher_head, st.teacher_head_buf, None, 0.0)
        teacher_c = teacher_projs - st.center
        st.center = R.center_update(st.center, teacher_projs, center_momentum)
    s_out, t_out = student_projs.view(V, B, -1), teacher_c.view(n_global, B, -1)
    dino = R.dino_loss_unimodal(s_out, t_out, tau_s, tau_t)
    cos = R.cosine_consistency_loss(emb.view(V, B, -1)) if cosine_loss_alpha > 0 else None
    loss = dino + cosine_loss_alpha * cos if cos is not None else dino
    R.ema_update(st.teacher, st.student, momentum)          # EMA before backward / optimizer (models/dino.py:871)
    R.ema_update(st.teacher_head, st.student_head, momentum)
    loss.backward()
    grads = {"student": {k: v.grad for k, v in S.items() if v.grad is not None},
             "student_head": {k: v.grad for k, v in SH.items() if v.grad is not None}}
    if do_adam:
        step = st.adam.get("step", 0)
        for gname, pd in (("student", st.student), ("student_head", st.student_head)):
            sub = st.adam.setdefault(gname, {})
            sub["step"] = step
            R.adam_step(pd, grads[gname], sub, lr, weight_decay)
        st.adam["step"] = step + 1
    return {"loss": loss.detach(), "dino": dino.detach(), "cosine": None if cos is None else cos.detach(), "grads": grads,
            "student_out": s_out.detach(), "teacher_out": t_out.detach(), "embeddings": emb.detach().view(V, B, -1)}


