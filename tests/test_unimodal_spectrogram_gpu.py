"""GPU: the audio-only DINO step (DinoStepEngine(kind="spectrogram_simple"), UniModalDINO(SpectrogramEncoder)) against the CPU oracle's
unimodal step, its determinism and CUDA-graph replay, and raw-batch training of UniModalDINOLightning (both unimodal encoders) through
the trainer and run_dino.py, plus the evaluation paths of an audio-only model."""
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
from oracle.fixtures import make_masks, synth_raw, synth_views, views_to_vb  # noqa: E402
from multimodal_ssl_avmnist_b200.engine import DinoStepEngine  # noqa: E402

DEV = "cuda"
KIND = "spectrogram_simple"


def _rel(a, b):
    a, b = a.detach().cpu().double(), b.detach().cpu().double()
    return float((a - b).abs().max() / (b.abs().max() + 1e-30))


def _bias_before_bn(name):
    """Gradients that are rounding noise: the conv biases and the head's first bias (a following BatchNorm cancels them), and the
    encoder.18 bias -- it only shifts the head's BatchNorm1d input, and it shifts every view's embedding alike, which the
    cosine-consistency term all but cancels too (its gradient is ~1e-7 there)."""
    return re.search(r"^(encoder\.(0|4|8|12|18)\.bias|mlp\.0\.bias)$", name) is not None


def _load_state(eng, st):
    eng.load_named(student=st.student, teacher=st.teacher, student_head=st.student_head, teacher_head=st.teacher_head)


def _sync_engine_to_oracle(eng, st):
    """The oracle's complete training state -> the engine (parameters, Adam moments + step, BatchNorm buffers, centre), so that every
    step is compared from identical state."""
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


def _views(B, seed):
    _, aud = views_to_vb(*synth_views(B, seed=seed))
    return aud                                                  # [V,B,1,112,112]


@pytest.mark.parametrize("alpha", [0.0, 0.3])
def test_fp32_step_vs_oracle(alpha):
    """Exact-fp32 engine against the oracle's unimodal step, two steps, re-synchronised before the second.  Conv-stack gradients are
    held to 5e-2: a different valid fp32 summation order flips near-tie max-pool arg-maxes in the 112x112 stack (DESIGN 4.7)."""
    B = 4
    st = U.UniModalDinoState(kind=KIND, seed=21)
    eng = DinoStepEngine(kind=KIND, device=DEV, precision="fp32", cosine_loss_alpha=alpha)
    assert eng.img_layers == [] and "x_img" not in eng._workspace(B) and "img_ops" not in eng._workspace(B)
    _load_state(eng, st)
    for it in range(2):
        if it > 0:
            _sync_engine_to_oracle(eng, st)
        aud = _views(B, 100 + it)
        masks = make_masks(seed=200 + it, V=6, Vg=2, B=B, E=256, hidden=512)
        want = U.unimodal_dino_step(st, aud, masks, cosine_loss_alpha=alpha)
        loss = eng.forward_backward(None, aud[:, :, 0].to(DEV).contiguous(), masks={"student_head": masks["student_head"].to(torch.uint8).to(DEV)})
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
                    assert float(mine.abs().sum()) < max(1e-3, 1e-5 * scale), (it, k, float(mine.abs().sum()))
                    continue
                conv_stack = gname == "student" and not k.startswith("encoder.18.")
                assert _rel(mine, g) < (5e-2 if conv_stack else 1e-3), (it, k, _rel(mine, g))
        eng.update_teacher()
        eng.optimizer_step()
        for prefix, table in (("enc.", st.teacher), ("head.", st.teacher_head)):
            for k, v in table.items():
                assert torch.equal(eng.T[prefix + k].cpu(), v), (it, k)        # same student, same EMA: bit-exact
        for k, v in st.student.items():
            diff = (eng.S["enc." + k].cpu() - v).abs()
            assert float(diff.max()) <= 2.5e-4, (it, k, float(diff.max()))
            if not _bias_before_bn(k):
                assert float(diff.mean()) <= 1e-5, (it, k, float(diff.mean()))
        assert float((eng.center.cpu() - st.center).abs().max()) <= 1e-6 * max(1.0, float(st.center.abs().max()))
        for k in R.spectrogram_bn_names():
            assert _rel(eng.bn_s["enc." + k].running_mean, st.student_buf[k + ".running_mean"]) < 1e-5, k
            assert _rel(eng.bn_t["enc." + k].running_var, st.teacher_buf[k + ".running_var"]) < 1e-5, k
            assert int(eng.bn_s["enc." + k].num_batches_tracked) == int(st.student_buf[k + ".num_batches_tracked"])


def test_bf16_product_path_vs_oracle():
    """The product path (every conv on the tensor cores, bf16 act8 activations, tf32 linears, fp32 accumulation) against the fp32
    oracle: loss 2e-3 relative, projections 2e-2 of their scale, gradient direction cosine > 0.97 -- for the whole DINO gradient,
    and per weight matrix with a well-conditioned upstream gradient (the DINO gradient at teacher == student is ill-conditioned;
    see tests/test_step_gpu.py::test_step_bf16_tensor_core_path_vs_oracle).  Every sample gets its own contrast: on i.i.d. noise
    spectrograms all samples are statistically alike, the head's BatchNorm1d divides by their tiny spread and magnifies the bf16
    rounding of the embeddings (0.2 % relative) to ~2 % in the projections -- an oracle with bf16-rounded convolution inputs does
    the same on the CPU."""
    B = 8
    st = U.UniModalDinoState(kind=KIND, seed=22)
    eng = DinoStepEngine(kind=KIND, device=DEV, precision="bf16")
    assert len(eng.tc["aud"]) == 4 and all(eng.tc["aud"]), eng.tc
    assert not any(any(v) for v in eng.pool["s"].values()) and not any(any(v) for v in eng.pool["t"].values())     # fused_pool stays off
    _load_state(eng, st)
    aud = _views(B, 110) * (0.2 + 0.8 * torch.rand(1, B, 1, 1, 1, generator=torch.Generator().manual_seed(7)))
    masks = make_masks(seed=210, V=6, Vg=2, B=B, E=256, hidden=512)
    gm = {"student_head": masks["student_head"].to(torch.uint8).to(DEV)}
    want = U.unimodal_dino_step(st, aud, masks)
    loss = eng.forward_backward(None, aud[:, :, 0].to(DEV).contiguous(), masks=gm)
    torch.cuda.synchronize()
    assert abs(float(loss[3]) - float(want["loss"])) < 2e-3 * abs(float(want["loss"])), (float(loss[3]), float(want["loss"]))
    assert _rel(eng._ws[B]["s.proj"].view(6, B, -1), want["student_out"]) < 2e-2
    assert _rel(eng._ws[B]["s.feat"].view(6, B, -1), want["embeddings"]) < 2e-2
    fm, fw = [], []
    for prefix, gname in (("enc.", "student"), ("head.", "student_head")):
        for k, g in want["grads"][gname].items():
            if not _bias_before_bn(k):
                fm.append(eng.G[prefix + k].detach().cpu().double().flatten())
                fw.append(g.double().flatten())
    fm, fw = torch.cat(fm), torch.cat(fw)
    cos = float((fm @ fw) / (fm.norm() * fw.norm()))
    assert cos > 0.97, cos
    # per matrix, surrogate loss sum(student_projs * D)
    st2 = U.UniModalDinoState(kind=KIND, seed=22)
    S = {k: v.clone().requires_grad_(True) for k, v in st2.student.items()}
    SH = {k: v.clone().requires_grad_(True) for k, v in st2.student_head.items()}
    D = torch.randn(6 * B, 128, generator=torch.Generator().manual_seed(5)) / (6 * B)
    emb = torch.cat([U.spectrogram_simple_encoder(aud[v], S, st2.student_buf) for v in range(6)])
    (R.projection_head(emb, SH, st2.student_head_buf, masks["student_head"], 0.3) * D).sum().backward()
    eng2 = DinoStepEngine(kind=KIND, device=DEV, precision="bf16")
    _load_state(eng2, st2)
    w = eng2.forward_pass(None, aud[:, :, 0].to(DEV).contiguous(), masks=gm)
    eng2.backward_pass(w, d_proj=D.to(DEV))
    torch.cuda.synchronize()
    cosines = {}
    for prefix, pd in (("enc.", S), ("head.", SH)):
        for k, v in pd.items():
            if v.grad is not None and v.grad.dim() >= 2:
                a, b = eng2.G[prefix + k].detach().cpu().double().flatten(), v.grad.double().flatten()
                cosines[k] = float((a @ b) / (a.norm() * b.norm()))
    assert len(cosines) == 4 + 1 + 2, cosines
    bad = {k: v for k, v in cosines.items() if v < 0.97}
    assert not bad, bad
    eng.update_teacher()
    for k, v in st.teacher_head.items():
        assert torch.equal(eng.T["head." + k].cpu(), v), k


def test_fp32_step_is_run_to_run_deterministic():
    B = 6
    outs = []
    for _ in range(2):
        st = U.UniModalDinoState(kind=KIND, seed=3)
        eng = DinoStepEngine(kind=KIND, device=DEV, precision="fp32", cosine_loss_alpha=0.3)
        _load_state(eng, st)
        rec = []
        for it in range(2):
            masks = make_masks(seed=200 + it, V=6, Vg=2, B=B, E=256, hidden=512)
            loss = eng.train_step_views(None, _views(B, 100 + it)[:, :, 0].to(DEV).contiguous(),
                                        masks={"student_head": masks["student_head"].to(torch.uint8).to(DEV)})
            rec += [loss.clone(), eng.grad.clone()]
        torch.cuda.synchronize()
        outs.append(rec + [eng.student.flat.clone(), eng.teacher.flat.clone(), eng.center.clone()])
    for a, b in zip(*outs):
        assert torch.equal(a, b), float((a - b).abs().max())


def test_raw_batch_step_learns_and_launches_no_image_work():
    """Raw uint8 spectrograms -> device-sampled views -> whole step: finite losses near log(128) at initialisation, the student moves,
    the teacher follows by EMA; the engine never allocates image buffers and ignores an image batch if one is given."""
    torch.manual_seed(0)
    B = 32
    eng = DinoStepEngine(kind=KIND, device=DEV, learning_rate=1e-3, cosine_loss_alpha=0.3)
    s0 = eng.student.flat.clone()
    aud = torch.randint(0, 256, (B, 112, 112), dtype=torch.uint8, device=DEV)
    losses = [eng.train_step(None, aud).clone() for _ in range(5)]
    losses.append(eng.train_step(torch.rand(B, 28, 28, device=DEV), aud).clone())
    torch.cuda.synchronize()
    assert all(3.0 < float(l[0]) < 6.0 and math.isfinite(float(l[3])) and float(l[2]) >= 0 for l in losses), losses
    n = eng.n_trainable_prefix
    assert float((eng.student.flat[:n] - s0[:n]).abs().max()) > 1e-3
    assert 0 < float((eng.teacher.flat[:n] - eng.student.flat[:n]).abs().max())
    w = eng._ws[B]
    assert not any(k.startswith(("img", "x_img", "s.img", "t.img")) for k in w), [k for k in w if "img" in k]


def test_cuda_graph_replay_reproduces_the_eager_step_bit_for_bit():
    B = 8
    g = torch.Generator().manual_seed(77)
    batches = [torch.randint(0, 256, (B, 112, 112), dtype=torch.uint8, generator=g).to(DEV) for _ in range(4)]
    engs = [DinoStepEngine(kind=KIND, device=DEV, precision="bf16", seed=11, cosine_loss_alpha=0.3) for _ in range(2)]
    engs[1].student.flat.copy_(engs[0].student.flat)
    for e in engs:
        e.sync_teacher()
    eager, graph = engs
    l_e = [eager.train_step(None, batches[0]).clone()]
    l_g = [graph.train_step(None, batches[0]).clone()]
    graph.capture_train_step(B)
    assert graph.rng_step == 1 and graph.step_count == 1 and "img" not in graph._graph
    for i, aud in enumerate(batches[1:]):
        if i == 2:
            eager.lr = graph.lr = 3.7e-4
        l_e.append(eager.train_step(None, aud).clone())
        l_g.append(graph.graph_step(None, aud).clone())
    torch.cuda.synchronize()
    for a, b in zip(l_e, l_g):
        assert torch.equal(a, b), (a, b)
    exact = {n: torch.equal(x, y) for n, x, y in (("student", graph.student.flat, eager.student.flat), ("teacher", graph.teacher.flat, eager.teacher.flat),
                                                  ("adam m", graph.exp_avg, eager.exp_avg), ("adam v", graph.exp_avg_sq, eager.exp_avg_sq),
                                                  ("centre", graph.center, eager.center))}
    assert all(exact.values()), exact
    counts = graph.graph_node_counts()
    assert counts["kernels"] > 0 and counts["other"] == 0, counts


def test_host_step_with_prefetch_matches_the_device_step():
    """train_step_host with next_batch (H2D copy + augmentation of the next batch prefetched on the augmentation stream) trains
    exactly like train_step on the same batches; the image argument may be None."""
    B = 8
    g = torch.Generator().manual_seed(5)
    host = [torch.randint(0, 256, (B, 112, 112), dtype=torch.uint8, generator=g).pin_memory() for _ in range(3)]
    a = DinoStepEngine(kind=KIND, device=DEV, precision="bf16", seed=3)
    b = DinoStepEngine(kind=KIND, device=DEV, precision="bf16", seed=3)
    b.student.flat.copy_(a.student.flat)
    a.sync_teacher()
    b.sync_teacher()
    direct = [float(a.train_step(None, h.to(DEV))[3]) for h in host]
    staged = [b.train_step_host(None, host[i], next_batch=(None, host[i + 1]) if i + 1 < len(host) else None) for i in range(len(host))]
    assert all(abs(x - y) <= 1e-5 * abs(y) for x, y in zip(staged, direct)), (staged, direct)
    assert float((a.student.flat - b.student.flat).abs().max()) < 5e-4


# ------------------------------------------------------------------------------------------------------------
# the reference-shaped API
# ------------------------------------------------------------------------------------------------------------
def _lit(encoder_class, alpha, data_dir="x/", **kw):
    return md.UniModalDINOLightning(encoder_class=encoder_class, data_dir=data_dir, dropout=0.3, learning_rate=1e-3, projection_dim=128,
                                    output_dim=256, momentum=0.996, center_momentum=0.9, teacher_temperature=0.04, weight_decay=1e-6,
                                    cosine_loss_alpha=alpha, data_augmentation="burst_noise", **kw)


def test_view_batches_through_the_spectrogram_module():
    """The reference's 4-tuple of views: UniModalDINO(SpectrogramEncoder).forward reads the audio views; training_step -> backward ->
    B200Adam.step moves every student parameter and returns dino + alpha * cosine."""
    torch.manual_seed(2)
    lit = _lit(md.SpectrogramEncoder, 0.3, num_epochs=10).to(DEV)
    opt = lit.configure_optimizers()["optimizer"]
    before = {k: v.detach().clone() for k, v in lit.model.student.named_parameters()}
    for it in range(2):
        opt.zero_grad(set_to_none=True)
        views = tuple(t.to(DEV) for t in synth_views(8, seed=70 + it))
        s, t, emb = lit.model(views)
        assert s.shape == (6, 8, 128) and t.shape == (2, 8, 128) and emb.shape == (6, 8, 256)
        loss = lit.training_step(views, it)
        loss.backward()
        opt.step()
    torch.cuda.synchronize()
    assert 3.0 < float(loss) < 7.0
    eng = lit.model.engine
    assert eng.kind == KIND and all(eng.tc["aud"])
    for k, v in lit.model.student.named_parameters():
        assert float((v - before[k]).abs().max()) > 0, k


@pytest.mark.parametrize("enc,alpha", [("ImageEncoder", 0.0), ("ImageEncoder", 0.3), ("SpectrogramEncoder", 0.0), ("SpectrogramEncoder", 0.3)])
def test_fused_graph_step_through_the_trainer_equals_the_step_by_step_path(tmp_path, enc, alpha):
    """Raw (image, audio) batches of the default data module through Trainer.fit: the fused CUDA-graph step and the step-by-step path
    (training_step -> backward -> B200Adam.step) give bit-identical student, teacher, Adam moments and centre after two epochs."""
    from _compat import pl
    d = str(tmp_path) + "/"
    gd.write_synthetic_avmnist(d, n_train=96, n_test=16)
    results = []
    for fused in (False, True):
        torch.manual_seed(7)
        dm = gd.AVMNISTDinoDataModule(data_dir=d, batch_size=16, num_workers=0, type="burst_noise", device_resident=True)
        dm.probe_dataloaders = None
        lit = _lit(getattr(md, enc), alpha, data_dir=d, num_epochs=2)
        lit.b200_fused_step = fused
        tr = pl.Trainer(max_epochs=2, logger=None, log_every_n_steps=1, devices=1, accelerator="gpu")
        tr.fit(lit, datamodule=dm)
        torch.cuda.synchronize()
        eng = lit.model.engine
        assert eng.kind == getattr(md, enc).B200_KIND and (eng._graph is not None) == fused
        assert tr.global_step == 2 * (len(dm.train_dataset) // 16) and eng.step_count == tr.global_step
        results.append((eng.student.flat.clone(), eng.teacher.flat.clone(), eng.exp_avg.clone(), eng.exp_avg_sq.clone(), lit.model.center.clone(),
                        float(tr.callback_metrics["train_loss_epoch"])))
    for name, a, b in zip(("student", "teacher", "adam m", "adam v", "centre"), results[0][:5], results[1][:5]):
        assert torch.equal(a, b), (name, float((a - b).abs().max()))
    assert 3.0 < results[0][5] < 7.0
    assert abs(results[0][5] - results[1][5]) < 1e-5 * abs(results[0][5])


def test_feature_path_probe_and_knn_for_the_audio_model(tmp_path):
    """FeatureExtractor / DownstreamClassifier / probe_accuracy / train_knn_classifier on an audio-only model: eval-mode features
    match the oracle encoder with the running statistics, and the probe and kNN accuracies are finite."""
    from training_structures.dino_train import train_knn_classifier
    torch.manual_seed(3)
    lit = _lit(md.SpectrogramEncoder, 0.0).to(DEV)
    B = 16
    opt = lit.configure_optimizers()["optimizer"]
    opt.zero_grad(set_to_none=True)
    lit.training_step(tuple(t.to(DEV) for t in synth_views(B, seed=90)), 0).backward()
    opt.step()
    fx = md.FeatureExtractor(lit.model).eval()
    image, audio, _ = synth_raw(B, seed=91)
    feats = fx(image.to(DEV), audio.to(DEV))
    assert feats.shape == (B, 256) and torch.isfinite(feats).all()
    assert torch.equal(fx(None, audio.to(DEV)), feats)                       # the image batch is not read
    sd = {k: v.detach().cpu().float() for k, v in lit.model.student.state_dict().items()}
    p = {k: v for k, v in sd.items() if "running" not in k and "num_batches" not in k}
    buf = {k: v for k, v in sd.items() if "running" in k or "num_batches" in k}
    want = U.spectrogram_simple_encoder(audio, p, buf, train=False)
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


@pytest.mark.parametrize("model", ["image_simple", "spectrogram_simple"])
def test_run_dino_unimodal_end_to_end(tmp_path, monkeypatch, model):
    """`run_dino.py --unimodal_model {image_simple,spectrogram_simple}` on a synthetic data set: the raw-batch data module, the fused
    step, the per-epoch probe and the performance summary."""
    import run_dino
    cfg = yaml.safe_load(open(os.path.join(MIRROR, "configs", "config_multimodal_dino.yaml")))
    cfg["data"]["data_dir"] = str(tmp_path / "data") + "/"
    cfg["model"]["model_dir_data"], cfg["model"]["model_dir_scratch"] = str(tmp_path / "runs" / "data"), str(tmp_path / "runs" / "scratch")
    path = tmp_path / "config.yaml"
    path.write_text(yaml.safe_dump(cfg))
    monkeypatch.setenv("SLURM_CPUS_PER_TASK", "0")          # no DataLoader worker processes
    results = run_dino.main(["--unimodal_model", model, "--config", str(path), "--synthetic", "512", "--max_steps", "4", "--seeds", "1"])
    assert len(results) == 1 and math.isfinite(results[0]["train_loss"])
    summaries = list((tmp_path / "runs" / "data").glob("*/performance_summary.txt"))
    assert len(summaries) == 1 and f"model_name: {model}" in summaries[0].read_text()
