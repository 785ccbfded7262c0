"""GPU: the unimodal LeNet-style CentralNet DINO steps (DinoStepEngine kinds "image_central" and "spectrogram_central",
UniModalDINO(ImageEncoderCentral / SpectrogramEncoderCentral)) against the CPU reference step of tests/unimodal_dino_ref.py
(with the encoders of tests/unimodal_central_ref.py), the
fused-pool and tensor-core policy they share with multi_central, determinism and CUDA-graph replay, training through the trainer and
run_dino.py, checkpoint round trips, and the evaluation paths."""
import copy
import math
import os
import re
import sys

import pytest
import torch
import yaml

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
MIRROR = os.path.join(ROOT, "multimodal_ssl_avmnist_b200", "AVMNIST_Experiments")
sys.path.insert(0, MIRROR)

import models.dino as md  # noqa: E402
import utils.get_data as gd  # noqa: E402
from oracle import dino_ref as R  # noqa: E402
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import unimodal_dino_ref as U  # noqa: E402
import unimodal_central_ref  # noqa: E402,F401  (registers the CentralNet kinds with the reference step)
from oracle.fixtures import make_masks, synth_raw, synth_views, views_to_vb  # noqa: E402
from multimodal_ssl_avmnist_b200.engine import DinoStepEngine  # noqa: E402

DEV = "cuda"
KINDS = ["image_central", "spectrogram_central"]
MOD = {"image_central": "img", "spectrogram_central": "aud"}
CLS = {"image_central": md.ImageEncoderCentral, "spectrogram_central": md.SpectrogramEncoderCentral}


def _rel(a, b):
    a, b = a.detach().cpu().double(), b.detach().cpu().double()
    return float((a - b).abs().max() / (b.abs().max() + 1e-30))


def _bias_before_bn(name):
    """Gradients that a following BatchNorm cancels (rounding noise at alpha = 0): the conv biases, the head's first bias, and the
    encoder.1 bias -- it shifts every row of the head's BatchNorm1d input alike (only the cosine-consistency term sees it)."""
    return re.search(r"^(encoder\.0\.conv\d\.bias|encoder\.1\.bias|mlp\.0\.bias)$", name) is not None


def _unused(name):
    return re.search(r"^encoder\.0\.fc[12]\.", name) is not None


def _load_state(eng, st):
    eng.load_named(student=st.student, teacher=st.teacher, student_head=st.student_head, teacher_head=st.teacher_head)


def _sync_engine_to_oracle(eng, st):
    """The reference step's complete training state -> the engine (parameters, Adam moments + step, BatchNorm buffers, centre)."""
    _load_state(eng, st)
    M, V = eng.student.views(eng.exp_avg), eng.student.views(eng.exp_avg_sq)
    eng.exp_avg.zero_()
    eng.exp_avg_sq.zero_()
    for gname, prefix in (("student", "enc."), ("student_head", "head.")):
        for key, val in st.adam.get(gname, {}).items():
            if isinstance(key, tuple):
                (M if key[0] == "m" else V)[prefix + key[1]].copy_(val.to(DEV))
    eng.step_count = int(st.adam.get("step", 0))
    eng.center.copy_(st.center.to(DEV))
    for table, prefix, buf in ((eng.bn_s, "enc.", st.student_buf), (eng.bn_t, "enc.", st.teacher_buf), (eng.bn_s, "head.", st.student_head_buf),
                               (eng.bn_t, "head.", st.teacher_head_buf)):
        for k, v in buf.items():
            base, attr = k.rsplit(".", 1)
            getattr(table[prefix + base], attr).copy_(v.to(DEV))


def _as_fp64(st):
    """A float64 copy of a reference-step state (parameters, buffers, centre, Adam moments)."""
    s = copy.deepcopy(st)
    for name in ("student", "teacher", "student_head", "teacher_head", "student_buf", "teacher_buf", "student_head_buf", "teacher_head_buf"):
        setattr(s, name, {k: v.double() if v.is_floating_point() else v for k, v in getattr(s, name).items()})
    s.center = s.center.double()
    for g in ("student", "student_head"):
        if g in s.adam:
            s.adam[g] = {k: v.double() if torch.is_tensor(v) else v for k, v in s.adam[g].items()}
    return s


def _views(kind, B, seed):
    img, aud = views_to_vb(*synth_views(B, seed=seed))
    return img if MOD[kind] == "img" else aud                  # [V,B,1,H,W]


def _args(kind, x):
    """(x_img, x_aud) for the engine: the views in the kind's slot, None in the other."""
    return (x, None) if MOD[kind] == "img" else (None, x)


def _stack_keys(w, mod):
    """Workspace entries of a modality's conv stack and its input views (the sampler's op records are not part of a stack)."""
    return [k for k in w if k.startswith((f"{mod}.", f"x_{mod}", f"s.{mod}.", f"t.{mod}.", f"e.{mod}."))]


def _raw(kind, B, g):
    if MOD[kind] == "img":
        return torch.rand(B, 28, 28, generator=g).to(DEV), None
    return None, torch.randint(0, 256, (B, 112, 112), dtype=torch.uint8, generator=g).to(DEV)


@pytest.mark.parametrize("alpha", [0.0, 0.3])
@pytest.mark.parametrize("kind", KINDS)
def test_fp32_step_vs_reference_step(kind, alpha):
    """Exact-fp32 engine against the reference step, two steps, re-synchronised before the second; the tolerances of the multi_central
    fp32 step on the same layers (loss 1e-5 relative, gradients 3e-4).  The teacher EMA is bit-exact over the whole arena, fc1 / fc2
    included; fc1 / fc2 get no gradient and Adam leaves them alone; the BatchNorm running statistics follow the reference.

    Near-tie max-pool arg-maxes (DESIGN 4.7): where a valid change of the fp32 summation order flips one, the conv-stack gradients
    move by ~1e-3 of their maximum.  Each step is therefore also run by the reference in float64; when that run differs from the
    float32 reference by more than 1e-4 on a conv-stack tensor (a flip, measured: 5e-3 on spectrogram_central's second step with
    the cosine term; about 1e-5 in every other step here), the conv-stack tensors of that step are held to twice that
    difference instead of 3e-4.  Everything else keeps 3e-4."""
    B = 4
    st = U.UniModalDinoState(kind=kind, seed=21)
    eng = DinoStepEngine(kind=kind, device=DEV, precision="fp32", cosine_loss_alpha=alpha)
    other = "aud" if MOD[kind] == "img" else "img"
    assert eng._layers(other) == [] and _stack_keys(eng._workspace(B), other) == []
    _load_state(eng, st)
    for it in range(2):
        if it > 0:
            _sync_engine_to_oracle(eng, st)
        x = _views(kind, B, 100 + it)
        masks = make_masks(seed=200 + it, V=6, Vg=2, B=B, E=256, hidden=512)
        s_before = {k: eng.S["enc." + k].clone() for k in st.student if _unused(k)}
        want64 = U.unimodal_dino_step(_as_fp64(st), x.double(), masks, cosine_loss_alpha=alpha, do_adam=False)
        want = U.unimodal_dino_step(st, x, masks, cosine_loss_alpha=alpha)
        flip = max(_rel(want["grads"]["student"][k], g) for k, g in want64["grads"]["student"].items()
                   if k.startswith("encoder.0.") and not _bias_before_bn(k))
        floor = 2 * flip if flip > 1e-4 else 0.0
        loss = eng.forward_backward(*_args(kind, x[:, :, 0].to(DEV).contiguous()),
                                    masks={"student_head": masks["student_head"].to(torch.uint8).to(DEV)})
        torch.cuda.synchronize()
        assert abs(float(loss[3]) - float(want["loss"])) < 1e-5 * abs(float(want["loss"])), (it, float(loss[3]), float(want["loss"]))
        if alpha > 0:
            assert abs(float(loss[2]) - float(want["cosine"])) < 1e-5 * abs(float(want["cosine"])) + 1e-7
        assert _rel(eng._ws[B]["s.proj"].view(6, B, -1), want["student_out"]) < 2e-5
        assert _rel(eng._ws[B]["s.feat"].view(6, B, -1), want["embeddings"]) < 2e-5
        scale = max(float(g.abs().sum()) for gd_ in want["grads"].values() for g in gd_.values())
        for prefix, gname in (("enc.", "student"), ("head.", "student_head")):
            for k, g in want["grads"][gname].items():
                mine = eng.G[prefix + k]
                if _bias_before_bn(k):
                    assert float((mine.cpu() - g).abs().sum()) < max(1e-3, 1e-5 * scale), (it, k, float(mine.abs().sum()), float(g.abs().sum()))
                    continue
                tol = max(3e-4, floor) if (gname == "student" and k.startswith("encoder.0.")) else 3e-4
                assert _rel(mine, g) < tol, (it, k, _rel(mine, g), flip)
        for k in s_before:
            assert k not in want["grads"]["student"] and float(eng.G["enc." + k].abs().max()) == 0.0, k
        eng.update_teacher()
        eng.optimizer_step()
        for prefix, table in (("enc.", st.teacher), ("head.", st.teacher_head)):
            for k, v in table.items():
                assert torch.equal(eng.T[prefix + k].cpu(), v), (it, k)        # same student, same EMA: bit-exact (fc1 / fc2 too)
        for k, v in st.student.items():
            if _unused(k):
                assert torch.equal(eng.S["enc." + k], s_before[k]) and torch.equal(eng.S["enc." + k].cpu(), v), k
                continue
            diff = (eng.S["enc." + k].cpu() - v).abs()
            assert float(diff.max()) <= 2.5e-4, (it, k, float(diff.max()))
            if not _bias_before_bn(k):
                assert float(diff.mean()) <= 1e-5, (it, k, float(diff.mean()))
        assert float((eng.center.cpu() - st.center).abs().max()) <= 1e-6 * max(1.0, float(st.center.abs().max()))
        for k in st.bn_names:
            for table, buf in ((eng.bn_s, st.student_buf), (eng.bn_t, st.teacher_buf)):
                assert _rel(table["enc." + k].running_mean, buf[k + ".running_mean"]) < 1e-5, k
                assert _rel(table["enc." + k].running_var, buf[k + ".running_var"]) < 1e-5, k
                assert int(table["enc." + k].num_batches_tracked) == int(buf[k + ".num_batches_tracked"]), k


@pytest.mark.parametrize("kind", KINDS)
def test_bf16_product_path_vs_reference_step(kind):
    """The product path against the fp32 reference: every conv on the tensor cores, multi_central's fused-pool policy for the stack,
    loss 2e-3 relative, projections 2e-2 of their scale, and per weight matrix a gradient cosine > 0.97 under a well-conditioned
    upstream gradient (the DINO gradient at teacher == student is ill-conditioned; tests/test_step_gpu.py).  Every sample gets its
    own contrast, so that the head's BatchNorm1d does not divide by the tiny spread of i.i.d. noise inputs: the float32 reference
    run on bf16-rounded convolution operands (the rounding alone, on the CPU) lands 2.1e-2 from the float32 projections for
    spectrogram_central at B = 8 with contrasts in [0.2, 1] -- the bound would measure the conditioning of the inputs, not the
    kernels -- and 1.3e-2 at B = 32 with contrasts c^2, c uniform in [0, 1], which this test uses (image_central: 0.9e-2)."""
    B = 32
    mod = MOD[kind]
    st = U.UniModalDinoState(kind=kind, seed=22)
    eng = DinoStepEngine(kind=kind, device=DEV, precision="bf16")
    mc = DinoStepEngine(kind="multi_central", device=DEV, precision="bf16")
    assert all(eng.tc[mod]) and eng.tc[mod] == mc.tc[mod], eng.tc
    assert eng.pool["s"][mod] == mc.pool["s"][mod] and eng.pool["t"][mod] == mc.pool["t"][mod], eng.pool
    assert any(eng.pool["t"][mod])
    del mc
    _load_state(eng, st)
    x = _views(kind, B, 110) * torch.rand(1, B, 1, 1, 1, generator=torch.Generator().manual_seed(7)) ** 2
    masks = make_masks(seed=210, V=6, Vg=2, B=B, E=256, hidden=512)
    gm = {"student_head": masks["student_head"].to(torch.uint8).to(DEV)}
    want = U.unimodal_dino_step(st, x, masks)
    loss = eng.forward_backward(*_args(kind, x[:, :, 0].to(DEV).contiguous()), masks=gm)
    torch.cuda.synchronize()
    assert abs(float(loss[3]) - float(want["loss"])) < 2e-3 * abs(float(want["loss"])), (float(loss[3]), float(want["loss"]))
    assert _rel(eng._ws[B]["s.proj"].view(6, B, -1), want["student_out"]) < 2e-2
    eng.update_teacher()
    for k, v in st.teacher_head.items():
        assert torch.equal(eng.T["head." + k].cpu(), v), k
    # per matrix, surrogate loss sum(student_projs * D)
    st2 = U.UniModalDinoState(kind=kind, seed=22)
    S = {k: v.clone().requires_grad_(True) for k, v in st2.student.items()}
    SH = {k: v.clone().requires_grad_(True) for k, v in st2.student_head.items()}
    D = torch.randn(6 * B, 128, generator=torch.Generator().manual_seed(5)) / (6 * B)
    enc = U.UNIMODAL_KINDS[kind][2]
    emb = torch.cat([enc(x[v], S, st2.student_buf) for v in range(6)])
    (R.projection_head(emb, SH, st2.student_head_buf, masks["student_head"], 0.3) * D).sum().backward()
    eng2 = DinoStepEngine(kind=kind, device=DEV, precision="bf16")
    _load_state(eng2, st2)
    w = eng2.forward_pass(*_args(kind, x[:, :, 0].to(DEV).contiguous()), masks=gm)
    eng2.backward_pass(w, d_proj=D.to(DEV))
    torch.cuda.synchronize()
    cosines = {}
    for prefix, pd in (("enc.", S), ("head.", SH)):
        for k, v in pd.items():
            if v.grad is not None and v.grad.dim() >= 2:
                a, b = eng2.G[prefix + k].detach().cpu().double().flatten(), v.grad.double().flatten()
                cosines[k] = float((a @ b) / (a.norm() * b.norm()))
    assert len(cosines) == len(eng2._layers(mod)) + 1 + 2, cosines
    print(f"{kind} bf16 per-matrix gradient cosine: min {min(cosines.values()):.5f} ({min(cosines, key=cosines.get)})")
    bad = {k: v for k, v in cosines.items() if v < 0.97}
    assert not bad, bad


@pytest.mark.parametrize("kind", KINDS)
def test_fused_pool_step_is_bit_identical_to_the_unfused_step(kind):
    B = 16
    g = torch.Generator().manual_seed(13)
    img, aud = _raw(kind, B, g)
    engs = [DinoStepEngine(kind=kind, device=DEV, precision="bf16", seed=4, fused_pool=f, cosine_loss_alpha=0.3) for f in (True, False)]
    assert any(engs[0].pool["t"][MOD[kind]]) and not any(engs[1].pool["t"][MOD[kind]])
    engs[1].student.flat.copy_(engs[0].student.flat)
    engs[1].sync_teacher()
    engs[0].sync_teacher()
    losses = [e.train_step(img, aud).clone() for e in engs]
    torch.cuda.synchronize()
    a, b = engs
    assert torch.equal(losses[0], losses[1]), losses
    for name, x, y in (("grad", a.grad, b.grad), ("student", a.student.flat, b.student.flat), ("teacher", a.teacher.flat, b.teacher.flat),
                       ("centre", a.center, b.center)):
        assert torch.equal(x, y), (name, float((x - y).abs().max()))


@pytest.mark.parametrize("kind", KINDS)
def test_fp32_step_is_run_to_run_deterministic(kind):
    B = 6
    outs = []
    for _ in range(2):
        st = U.UniModalDinoState(kind=kind, seed=3)
        eng = DinoStepEngine(kind=kind, device=DEV, precision="fp32", cosine_loss_alpha=0.3)
        _load_state(eng, st)
        rec = []
        for it in range(2):
            masks = make_masks(seed=200 + it, V=6, Vg=2, B=B, E=256, hidden=512)
            loss = eng.train_step_views(*_args(kind, _views(kind, B, 100 + it)[:, :, 0].to(DEV).contiguous()),
                                        masks={"student_head": masks["student_head"].to(torch.uint8).to(DEV)})
            rec += [loss.clone(), eng.grad.clone()]
        torch.cuda.synchronize()
        outs.append(rec + [eng.student.flat.clone(), eng.teacher.flat.clone(), eng.center.clone()])
    for a, b in zip(*outs):
        assert torch.equal(a, b), float((a - b).abs().max())


@pytest.mark.parametrize("kind", KINDS)
def test_raw_batch_step_learns_and_launches_nothing_for_the_other_modality(kind):
    """Raw batches -> device-sampled views -> whole step: losses near log(128) at initialisation, the student moves, the teacher
    follows by EMA, fc1 / fc2 stay put in the student; nothing is allocated for the absent modality, and a batch of it is ignored."""
    torch.manual_seed(0)
    B = 32
    eng = DinoStepEngine(kind=kind, device=DEV, learning_rate=1e-3, cosine_loss_alpha=0.3)
    s0 = eng.student.flat.clone()
    img, aud = _raw(kind, B, torch.Generator().manual_seed(1))
    losses = [eng.train_step(img, aud).clone() for _ in range(4)]
    if img is None:                                         # a batch of the absent modality is ignored
        losses.append(eng.train_step(torch.rand(B, 28, 28, device=DEV), aud).clone())
    else:
        losses.append(eng.train_step(img, torch.randint(0, 256, (B, 112, 112), dtype=torch.uint8, device=DEV)).clone())
    torch.cuda.synchronize()
    assert all(3.0 < float(l[0]) < 6.0 and math.isfinite(float(l[3])) and float(l[2]) >= 0 for l in losses), losses
    n = eng.n_trainable_prefix
    assert float((eng.student.flat[:n] - s0[:n]).abs().max()) > 1e-3
    assert torch.equal(eng.student.flat[n:], s0[n:])                               # fc1 / fc2: EMA'd, never updated
    assert 0 < float((eng.teacher.flat[:n] - eng.student.flat[:n]).abs().max())
    o = "aud" if MOD[kind] == "img" else "img"
    assert _stack_keys(eng._ws[B], o) == [] and eng._layers(o) == [] and not eng.tc[o]


@pytest.mark.parametrize("kind", KINDS)
def test_cuda_graph_replay_reproduces_the_eager_step_bit_for_bit(kind):
    B = 8
    g = torch.Generator().manual_seed(77)
    batches = [_raw(kind, B, g) for _ in range(4)]
    engs = [DinoStepEngine(kind=kind, device=DEV, precision="bf16", seed=11, cosine_loss_alpha=0.3) for _ in range(2)]
    engs[1].student.flat.copy_(engs[0].student.flat)
    for e in engs:
        e.sync_teacher()
    eager, graph = engs
    l_e = [eager.train_step(*batches[0]).clone()]
    l_g = [graph.train_step(*batches[0]).clone()]
    graph.capture_train_step(B)
    o = "aud" if MOD[kind] == "img" else "img"
    assert graph.rng_step == 1 and graph.step_count == 1 and o not in graph._graph
    for i, b in enumerate(batches[1:]):
        if i == 2:
            eager.lr = graph.lr = 3.7e-4
        l_e.append(eager.train_step(*b).clone())
        l_g.append(graph.graph_step(*b).clone())
    torch.cuda.synchronize()
    for a, b in zip(l_e, l_g):
        assert torch.equal(a, b), (a, b)
    exact = {n: torch.equal(x, y) for n, x, y in (("student", graph.student.flat, eager.student.flat), ("teacher", graph.teacher.flat, eager.teacher.flat),
                                                  ("adam m", graph.exp_avg, eager.exp_avg), ("adam v", graph.exp_avg_sq, eager.exp_avg_sq),
                                                  ("centre", graph.center, eager.center))}
    assert all(exact.values()), exact
    counts = graph.graph_node_counts()
    assert counts["kernels"] > 0 and counts["other"] == 0, counts


@pytest.mark.parametrize("kind", KINDS)
def test_host_step_with_prefetch_matches_the_device_step(kind):
    """train_step_host with next_batch (H2D copy + augmentation of the next batch prefetched on the augmentation stream) trains like
    train_step on the same batches; the argument of the absent modality may be None."""
    B = 8
    g = torch.Generator().manual_seed(5)
    if MOD[kind] == "img":
        host = [(torch.rand(B, 28, 28, generator=g).pin_memory(), None) for _ in range(3)]
    else:
        host = [(None, torch.randint(0, 256, (B, 112, 112), dtype=torch.uint8, generator=g).pin_memory()) for _ in range(3)]
    a = DinoStepEngine(kind=kind, device=DEV, precision="bf16", seed=3)
    b = DinoStepEngine(kind=kind, device=DEV, precision="bf16", seed=3)
    b.student.flat.copy_(a.student.flat)
    a.sync_teacher()
    b.sync_teacher()

    def dev(t):
        return None if t is None else t.to(DEV)
    direct = [float(a.train_step(dev(i), dev(s))[3]) for i, s in host]
    staged = [b.train_step_host(*host[i], next_batch=host[i + 1] if i + 1 < len(host) else None) for i in range(len(host))]
    assert all(abs(x - y) <= 1e-5 * abs(y) for x, y in zip(staged, direct)), (staged, direct)
    assert float((a.student.flat - b.student.flat).abs().max()) < 5e-4


# ------------------------------------------------------------------------------------------------------------
# the reference-shaped API
# ------------------------------------------------------------------------------------------------------------
def _lit(encoder_class, alpha, data_dir="x/", **kw):
    return md.UniModalDINOLightning(encoder_class=encoder_class, data_dir=data_dir, dropout=0.3, learning_rate=1e-3, projection_dim=128,
                                    output_dim=256, momentum=0.996, center_momentum=0.9, teacher_temperature=0.04, weight_decay=1e-6,
                                    cosine_loss_alpha=alpha, data_augmentation="burst_noise", **kw)


@pytest.mark.parametrize("kind", KINDS)
def test_fused_graph_step_through_the_trainer_equals_the_step_by_step_path(tmp_path, kind):
    """Raw (image, audio) batches of the default data module through Trainer.fit: the fused CUDA-graph step and the step-by-step path
    give bit-identical student, teacher, Adam moments and centre after two epochs."""
    from _compat import pl
    d = str(tmp_path) + "/"
    gd.write_synthetic_avmnist(d, n_train=96, n_test=16)
    results = []
    for fused in (False, True):
        torch.manual_seed(7)
        dm = gd.AVMNISTDinoDataModule(data_dir=d, batch_size=16, num_workers=0, type="burst_noise", device_resident=True)
        dm.probe_dataloaders = None
        lit = _lit(CLS[kind], 0.3, data_dir=d, num_epochs=2)
        lit.b200_fused_step = fused
        tr = pl.Trainer(max_epochs=2, logger=None, log_every_n_steps=1, devices=1, accelerator="gpu")
        tr.fit(lit, datamodule=dm)
        torch.cuda.synchronize()
        eng = lit.model.engine
        assert eng.kind == kind and (eng._graph is not None) == fused and all(eng.tc[MOD[kind]])
        assert tr.global_step == 2 * (len(dm.train_dataset) // 16) and eng.step_count == tr.global_step
        results.append((eng.student.flat.clone(), eng.teacher.flat.clone(), eng.exp_avg.clone(), eng.exp_avg_sq.clone(), lit.model.center.clone(),
                        float(tr.callback_metrics["train_loss_epoch"])))
    for name, a, b in zip(("student", "teacher", "adam m", "adam v", "centre"), results[0][:5], results[1][:5]):
        assert torch.equal(a, b), (name, float((a - b).abs().max()))
    assert 3.0 < results[0][5] < 7.0
    assert abs(results[0][5] - results[1][5]) < 1e-5 * abs(results[0][5])


@pytest.mark.parametrize("kind", KINDS)
def test_checkpoint_round_trip_resumes_to_a_bit_identical_step(kind):
    """lit.state_dict() + B200Adam.state_dict() of a model after two steps, loaded into a fresh model and optimizer, give the same next
    step bit for bit.  fc1 / fc2 travel in the state dict, sit in the unused part of the arenas, and the optimizer's parameter order is
    the module's declaration order.  (The augmentation / dropout stream position is not part of a checkpoint; the test carries it over.)"""
    B = 8

    def build():
        torch.manual_seed(5)                    # also the engine's stream seed (torch.initial_seed())
        lit = _lit(CLS[kind], 0.3).to(DEV)
        return lit, lit.configure_optimizers()["optimizer"]

    def step(lit, opt, seed, it):
        opt.zero_grad(set_to_none=True)
        lit.training_step(tuple(t.to(DEV) for t in synth_views(B, seed=seed)), it).backward()
        opt.step()

    a, opt_a = build()
    for it in range(2):
        step(a, opt_a, 40 + it, it)
    sd, osd = a.state_dict(), opt_a.state_dict()
    names = [n for n, _ in a.named_parameters()]
    assert osd["param_groups"][0]["params"] == list(range(len(names)))
    fc = [n for n in names if ".fc" in n]
    assert len(fc) == 8 and all(f"model.student.encoder.0.{l}.{w}" in fc for l in ("fc1", "fc2") for w in ("weight", "bias"))
    eng_a = a.model.engine
    for n in ("encoder.0.fc1.weight", "encoder.0.fc2.bias"):
        off = eng_a.student.offsets["enc." + n][0]
        assert off >= eng_a.n_trainable_prefix and dict(a.model.student.named_parameters())[n].data_ptr() == eng_a.S["enc." + n].data_ptr()
        assert eng_a.teacher.offsets["enc." + n][0] == off
    sd = {k: v.detach().cpu().clone() for k, v in sd.items()}
    b, opt_b = build()
    b.load_state_dict(sd)
    opt_b.load_state_dict(osd)
    eng_b = b.model._b200.ensure(torch.device(DEV))
    eng_b.rng_step = eng_a.rng_step
    step(a, opt_a, 50, 2)
    step(b, opt_b, 50, 2)
    torch.cuda.synchronize()
    assert eng_b.step_count == eng_a.step_count == 3
    for name, x, y in (("student", eng_a.student.flat, eng_b.student.flat), ("teacher", eng_a.teacher.flat, eng_b.teacher.flat),
                       ("adam m", eng_a.exp_avg, eng_b.exp_avg), ("adam v", eng_a.exp_avg_sq, eng_b.exp_avg_sq), ("centre", eng_a.center, eng_b.center)):
        assert torch.equal(x, y), (name, float((x - y).abs().max()))
    for k, v in a.model.student.state_dict().items():
        assert torch.equal(v, b.model.student.state_dict()[k]), k


@pytest.mark.parametrize("kind", KINDS)
def test_feature_path_probe_and_knn(tmp_path, kind):
    """FeatureExtractor / probe_accuracy / train_knn_classifier on a CentralNet unimodal model: eval-mode features match the reference
    encoder with the running statistics, the other modality's batch is not read, and the probe and kNN accuracies are finite."""
    from training_structures.dino_train import train_knn_classifier
    torch.manual_seed(3)
    lit = _lit(CLS[kind], 0.0).to(DEV)
    B = 16
    opt = lit.configure_optimizers()["optimizer"]
    opt.zero_grad(set_to_none=True)
    lit.training_step(tuple(t.to(DEV) for t in synth_views(B, seed=90)), 0).backward()
    opt.step()
    fx = md.FeatureExtractor(lit.model).eval()
    image, audio, _ = synth_raw(B, seed=91)
    feats = fx(image.to(DEV), audio.to(DEV))
    assert feats.shape == (B, 256) and torch.isfinite(feats).all()
    if MOD[kind] == "aud":
        assert torch.equal(fx(None, audio.to(DEV)), feats)
    else:
        assert torch.equal(fx(image.to(DEV)), feats)
    sd = {k: v.detach().cpu().float() for k, v in lit.model.student.state_dict().items()}
    p = {k: v for k, v in sd.items() if "running" not in k and "num_batches" not in k}
    buf = {k: v for k, v in sd.items() if "running" in k or "num_batches" in k}
    want = U.UNIMODAL_KINDS[kind][2](image if MOD[kind] == "img" else audio, p, buf, train=False)
    assert float((feats.cpu() - want).abs().max()) < 3e-2 * float(want.abs().max())
    d = str(tmp_path) + "/"
    gd.write_synthetic_avmnist(d, n_train=64, n_test=16)
    dm = gd.AVMNISTDinoDataModule(data_dir=d, batch_size=16, num_workers=0, type="burst_noise")
    dm.setup("fit")
    train_loader, val_loader = dm.probe_dataloaders()
    val_loss, acc = lit.probe_accuracy(train_loader, val_loader)
    assert math.isfinite(val_loss) and 0.0 <= acc <= 100.0
    knn, kacc = train_knn_classifier(lit.model, train_loader, val_loader, n_neighbors=5, device=DEV)
    assert math.isfinite(kacc) and 0.0 <= kacc <= 100.0 and knn.train_features.shape[1] == 256


@pytest.mark.parametrize("kind", KINDS)
def test_run_dino_unimodal_central_end_to_end(tmp_path, monkeypatch, kind):
    """`run_dino.py --unimodal_model {image_central,spectrogram_central}` on a synthetic data set: the raw-batch data module, the fused
    step, the per-epoch probe, the checkpoint and the performance summary."""
    import run_dino
    cfg = yaml.safe_load(open(os.path.join(MIRROR, "configs", "config_multimodal_dino.yaml")))
    cfg["data"]["data_dir"] = str(tmp_path / "data") + "/"
    cfg["model"]["model_dir_data"], cfg["model"]["model_dir_scratch"] = str(tmp_path / "runs" / "data"), str(tmp_path / "runs" / "scratch")
    path = tmp_path / "config.yaml"
    path.write_text(yaml.safe_dump(cfg))
    monkeypatch.setenv("SLURM_CPUS_PER_TASK", "0")          # no DataLoader worker processes
    results = run_dino.main(["--unimodal_model", kind, "--config", str(path), "--synthetic", "512", "--max_steps", "4", "--seeds", "1"])
    assert len(results) == 1 and math.isfinite(results[0]["train_loss"])
    summaries = list((tmp_path / "runs" / "data").glob("*/performance_summary.txt"))
    assert len(summaries) == 1 and f"model_name: {kind}" in summaries[0].read_text()
    ckpts = [p for p in (tmp_path / "runs").rglob("*.ckpt")]
    assert ckpts, sorted(str(p) for p in (tmp_path / "runs").rglob("*"))
