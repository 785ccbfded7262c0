"""GPU: the downstream evaluation on the device -- the probe kernel against a float64 restatement, AdamW against torch.optim.AdamW,
train_downstream against the torch-classifier loop on the same features, determinism and CUDA-graph replay, isolation of the
pretrained model, every compiled DINO kind through compute_accuracies, a probe that learns, and run_dino.py --evaluate."""
import json
import math
import os
import sys

import numpy as np
import pytest
import torch
import torch.nn as nn
import torch.nn.functional as F
import yaml

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
MIRROR = os.path.join(ROOT, "multimodal_ssl_avmnist_b200", "AVMNIST_Experiments")
sys.path.insert(0, MIRROR)

import models.dino as md  # noqa: E402
from training_structures import dino_train as dt  # noqa: E402
from multimodal_ssl_avmnist_b200 import ops  # noqa: E402
from multimodal_ssl_avmnist_b200.probe import ProbeSession  # noqa: E402

DEV = "cuda"
MULTI = {"multi_central": md.CentralMultiModalEncoder, "multi_simple": md.SimpleMultiModalEncoder,
         "multi_simple_gated": md.GatedMultiModalEncoder, "multi_cross_attention": md.CrossAttentionMultiModalEncoder}
UNI = {"image_simple": md.ImageEncoder, "spectrogram_simple": md.SpectrogramEncoder, "image_central": md.ImageEncoderCentral,
       "spectrogram_central": md.SpectrogramEncoderCentral}
MODES = {"default": md.MultiModalDINOLightning, "semi_supervised": md.MultiModalDINOSemiSupervisedLightning,
         "mse": md.MultiModalDINOWithMSELightning, "infonce": md.MultiModalDINOWithINFONCELightning}


def _lit(kind, seed=5, fp32=False, mode="default"):
    torch.manual_seed(seed)
    if kind in MULTI:
        lit = MODES[mode](data_dir="x/", encoder_class=MULTI[kind], projection_dim=128, output_dim=256, encoder_output_dim=256,
                          learning_rate=1e-3, use_mixed_precision=not fp32, num_epochs=10)
    else:
        lit = md.UniModalDINOLightning(encoder_class=UNI[kind], data_dir="x/", dropout=0.3, learning_rate=1e-3, projection_dim=128,
                                       output_dim=256, cosine_loss_alpha=0.0, num_epochs=10, use_mixed_precision=not fp32)
    lit = lit.to(DEV)
    lit.model._b200.ensure(torch.device(DEV))
    return lit


def _batches(n, B, seed, num_classes=10):
    """A fixed list of labelled (image, audio, label) host batches (the last one ragged when B does not divide n)."""
    g = torch.Generator().manual_seed(seed)
    img = torch.rand(n, 1, 28, 28, generator=g)
    aud = torch.rand(n, 1, 112, 112, generator=g)
    lab = torch.randint(0, num_classes, (n,), generator=g)
    return [(img[i:i + B], aud[i:i + B], lab[i:i + B]) for i in range(0, n, B)]


# ------------------------------------------------------------------------------------------------------------
# kernels
# ------------------------------------------------------------------------------------------------------------
def _ref64(x, w1, b1, w2, b2, lab):
    x, w1, b1, w2, b2 = (t.double() for t in (x, w1, b1, w2, b2))
    z = x @ w1.T + b1
    h = z.clamp_min(0)
    logits = h @ w2.T + b2
    B = x.shape[0]
    d = (torch.softmax(logits, 1) - F.one_hot(lab, w2.shape[0]).double()) / B
    dh = (d @ w2) * (z > 0)
    return {"loss": F.cross_entropy(logits, lab, reduction="sum"), "logits": logits,
            "grads": [dh.T @ x, dh.sum(0), d.T @ h, d.sum(0)]}


@pytest.mark.parametrize("B", [1, 37, 128, 1000])
@pytest.mark.parametrize("O", [64, 256])
def test_probe_kernel_against_float64(B, O):
    C = 10
    g = torch.Generator(device=DEV).manual_seed(B * 7 + O)
    x = torch.randn(B, O, device=DEV, generator=g)
    w1 = torch.randn(128, O, device=DEV, generator=g) / O ** 0.5
    b1 = torch.randn(128, device=DEV, generator=g) * 0.1
    w2 = torch.randn(C, 128, device=DEV, generator=g) / 128 ** 0.5
    b2 = torch.randn(C, device=DEV, generator=g) * 0.1
    lab = torch.randint(0, C, (B,), device=DEV, generator=g)
    ref = _ref64(x, w1, b1, w2, b2, lab)
    n = 128 * O + 128 + 128 * C + C
    grad = torch.full((n,), float("nan"), device=DEV)
    work = torch.full((ops.probe_work_floats(B, C),), float("nan"), device=DEV)
    loss = torch.full((1,), 0.5, dtype=torch.float64, device=DEV)
    correct = torch.full((1,), 3, dtype=torch.int64, device=DEV)
    ops.probe_mlp_fwd_bwd(x, w1, b1, w2, b2, lab, work, loss, correct, grad=grad, train=True)
    torch.cuda.synchronize()
    assert not torch.isnan(grad).any()
    want_pred = ref["logits"].argmax(1)
    assert abs(float(loss) - 0.5 - float(ref["loss"])) <= 1e-5 * abs(float(ref["loss"]))
    assert int(correct) - 3 == int((want_pred == lab).sum())
    offs = np.cumsum([0, 128 * O, 128, 128 * C, C])
    for i, (name, want) in enumerate(zip(("dW1", "db1", "dW2", "db2"), ref["grads"])):
        got = grad[offs[i]:offs[i + 1]].view(want.shape).double()
        err = float((got - want).abs().max())
        assert err <= 1e-5 * float(want.abs().max()) + 1e-9, (name, err)
    # forward only: loss and counts again, exact predictions and confusion matrix
    grad2 = grad.clone()
    loss.zero_()
    correct.zero_()
    preds = torch.full((B,), -7, dtype=torch.int64, device=DEV)
    conf = torch.zeros(C, C, dtype=torch.int64, device=DEV)
    ops.probe_mlp_fwd_bwd(x, w1, b1, w2, b2, lab, work, loss, correct, preds=preds, confusion=conf, train=False)
    torch.cuda.synchronize()
    assert torch.equal(preds, want_pred)
    assert torch.equal(conf.view(-1), torch.bincount(lab * C + want_pred, minlength=C * C))
    assert abs(float(loss) - float(ref["loss"])) <= 1e-5 * abs(float(ref["loss"])) and int(correct) == int((want_pred == lab).sum())
    assert torch.equal(grad, grad2)                               # the forward-only variant writes no gradient


def test_probe_kernel_is_run_to_run_deterministic():
    B, O, C = 1000, 256, 10
    g = torch.Generator(device=DEV).manual_seed(1)
    args = [torch.randn(B, O, device=DEV, generator=g), torch.randn(128, O, device=DEV, generator=g) * 0.06,
            torch.randn(128, device=DEV, generator=g), torch.randn(C, 128, device=DEV, generator=g) * 0.09,
            torch.randn(C, device=DEV, generator=g), torch.randint(0, C, (B,), device=DEV, generator=g)]
    outs = []
    for _ in range(2):
        grad = torch.empty(128 * O + 128 + 128 * C + C, device=DEV)
        loss = torch.zeros(1, dtype=torch.float64, device=DEV)
        correct = torch.zeros(1, dtype=torch.int64, device=DEV)
        ops.probe_mlp_fwd_bwd(*args, torch.empty(ops.probe_work_floats(B, C), device=DEV), loss, correct, grad=grad, train=True)
        outs.append((grad, loss, correct))
    torch.cuda.synchronize()
    for a, b in zip(*outs):
        assert torch.equal(a, b)


@pytest.mark.parametrize("dev_variant", [False, True])
def test_adamw_flat_matches_torch_adamw(dev_variant):
    n, lr, wd = 4099, 1e-3, 1e-2
    g = torch.Generator(device=DEV).manual_seed(3)
    p = torch.randn(n, device=DEV, generator=g)
    ref = nn.Parameter(p.clone())
    opt = torch.optim.AdamW([ref], lr=lr, weight_decay=wd)
    m, v = torch.zeros(n, device=DEV), torch.zeros(n, device=DEV)
    ctr, bc = torch.zeros(1, dtype=torch.int64, device=DEV), torch.zeros(3, device=DEV)
    for step in range(1, 21):
        grad = torch.randn(n, device=DEV, generator=g) * (0.1 * step)
        ref.grad = grad.clone()
        opt.step()
        if dev_variant:
            ops.adam_bias_dev(ctr, bc)
            ops.adamw_flat_dev(p, grad, m, v, bc, lr, weight_decay=wd)
            ops.counters_advance(ctr)
        else:
            ops.adamw_flat(p, grad, m, v, step, lr, weight_decay=wd)
    torch.cuda.synchronize()
    st = opt.state[ref]
    eps = torch.finfo(torch.float32).eps
    # the moments share b200_adam_flat's arithmetic, which forms 1 - beta in fp32 (1 - 0.999f is 1.3e-5 relative below torch's
    # double-rounded 1e-3), so exp_avg_sq carries that offset; the parameters agree to a few ulps
    for name, a, b, tol in (("param", p, ref.detach(), 8 * eps), ("exp_avg", m, st["exp_avg"], 8 * eps),
                            ("exp_avg_sq", v, st["exp_avg_sq"], 2e-5)):
        err = float((a - b).abs().max())
        assert err <= tol * float(b.abs().max()), (name, err)


def test_adamw_without_weight_decay_is_adam():
    n = 1027
    g = torch.Generator(device=DEV).manual_seed(4)
    p0 = torch.randn(n, device=DEV, generator=g)
    a = [p0.clone(), torch.zeros(n, device=DEV), torch.zeros(n, device=DEV)]
    b = [p0.clone(), torch.zeros(n, device=DEV), torch.zeros(n, device=DEV)]
    for step in range(1, 6):
        grad = torch.randn(n, device=DEV, generator=g)
        ops.adamw_flat(a[0], grad, a[1], a[2], step, 1e-3, weight_decay=0.0)
        ops.adam_flat(b[0], grad, b[1], b[2], step, 1e-3, weight_decay=0.0)
    torch.cuda.synchronize()
    for x, y in zip(a, b):
        assert torch.equal(x, y)


# ------------------------------------------------------------------------------------------------------------
# the probe session and train_downstream
# ------------------------------------------------------------------------------------------------------------
def _torch_probe(model, train, test, epochs, lr, seed):
    """The oracle: probe_accuracy's loop body (DownstreamClassifier + AdamW + CrossEntropyLoss on the same train-mode features and
    probe-token semantics) for `epochs` epochs; per-epoch loss per sample, the trained head and the final eval-mode predictions."""
    torch.manual_seed(seed)
    probe = md.DownstreamClassifier(model, trainable_encoder=False).to(DEV)
    opt = torch.optim.AdamW(probe.classifier.parameters(), lr=lr)
    crit = nn.CrossEntropyLoss()
    losses = []
    for _ in range(epochs):
        probe.train()
        total, n = 0.0, 0
        for images, audios, labels in train:
            images, audios, labels = images.to(DEV), audios.to(DEV), labels.to(DEV)
            opt.zero_grad()
            loss = crit(probe(images, audios), labels)
            loss.backward()
            opt.step()
            total, n = total + float(loss) * labels.numel(), n + labels.numel()
        losses.append(total / n)
    probe.eval()
    with torch.no_grad():
        preds = torch.cat([probe(i.to(DEV), a.to(DEV)).argmax(1) for i, a, _ in test])
    return losses, probe.classifier, preds


@pytest.mark.parametrize("kind", ["multi_central", "image_simple"])
def test_train_downstream_matches_the_torch_classifier_loop(kind):
    lit = _lit(kind, fp32=True)
    train, test = _batches(200, 64, seed=11), _batches(96, 64, seed=12)
    want_loss, want_head, want_pred = _torch_probe(lit.model, train, test, 2, 1e-3, seed=21)
    torch.manual_seed(21)
    clf, hist = dt.train_downstream(lit.model, train, test, num_epochs=2, learning_rate=1e-3)
    assert isinstance(clf, md.DownstreamClassifier) and len(hist["train_loss"]) == len(hist["val_acc"]) == 2
    for a, b in zip(hist["train_loss"], want_loss):
        assert abs(a - b) <= 1e-5 * abs(b), (hist["train_loss"], want_loss)
    for a, b in zip(clf.classifier.state_dict().values(), want_head.state_dict().values()):
        assert float((a - b).abs().max()) <= 1e-4, float((a - b).abs().max())
    ev = clf.b200_probe.evaluate(test, predictions=True)
    assert torch.equal(ev["predictions"], want_pred)
    assert hist["val_acc"][-1] == pytest.approx(100.0 * float((want_pred.cpu() == torch.cat([t[2] for t in test])).double().mean()))
    with torch.no_grad():                                         # the returned classifier evaluates with the probe's statistics
        got = torch.cat([clf(i.to(DEV), a.to(DEV)).argmax(1) for i, a, _ in test])
    assert torch.equal(got, want_pred)


def _probe_run(kind, graph, B=48, n=200):
    lit = _lit(kind)
    torch.manual_seed(9)
    s = ProbeSession(lit.model, lr=1e-3, graph=graph)
    train = _batches(n, B, seed=13)
    rec = []
    for _ in range(2):
        for b in train:
            s.train_batch(*b)
        rec.append(s.end_epoch())
    ev = s.evaluate(_batches(64, 32, seed=14), predictions=True)
    bns = [t.clone() for bn in s.token["bns"].values() for t in (bn.running_mean, bn.running_var, bn.num_batches_tracked)]
    return s, rec, ev, [s.params.clone(), s.exp_avg.clone(), s.exp_avg_sq.clone(), s._ctr.clone()] + bns


@pytest.mark.parametrize("kind", ["multi_central", "image_simple"])
def test_probe_is_deterministic_and_the_graph_path_equals_the_eager_path(kind):
    runs = [_probe_run(kind, graph) for graph in (False, False, True)]
    assert runs[0][0]._graph is None and runs[2][0]._graph is not None and runs[2][0]._graph["B"] == 48     # 200 = 4 x 48 + 8: ragged
    for s, rec, ev, state in runs[1:]:
        assert rec == runs[0][1]
        assert torch.equal(ev["predictions"], runs[0][2]["predictions"]) and ev["loss"] == runs[0][2]["loss"]
        assert np.array_equal(ev["confusion_matrix"], runs[0][2]["confusion_matrix"])
        for a, b in zip(state, runs[0][3]):
            assert torch.equal(a, b)
    assert runs[0][0].token["step"] == runs[2][0].token["step"] == 10


def test_the_probe_leaves_the_pretrained_model_untouched():
    """After train_downstream the live BatchNorm statistics, parameters and optimiser state are unchanged, and the next DINO
    training step is the one it would have been without the probe."""
    def model():
        lit = _lit("multi_central", seed=31)
        eng = lit.model.engine
        return lit, eng

    def state(eng):
        ts = [eng.student.flat, eng.teacher.flat, eng.exp_avg, eng.exp_avg_sq, eng.center]
        for table in (eng.bn_s, eng.bn_t):
            for bn in table.values():
                ts += [bn.running_mean, bn.running_var, bn.num_batches_tracked]
        return [t.clone() for t in ts] + [eng.rng_step, eng.step_count]

    raw = (torch.rand(32, 28, 28, device=DEV), torch.randint(0, 256, (32, 112, 112), dtype=torch.uint8, device=DEV))
    a, eng_a = model()
    b, eng_b = model()
    eng_a.train_step(*raw)
    eng_b.train_step(*raw)
    before = state(eng_a)
    dt.train_downstream(a.model, _batches(100, 32, seed=15), _batches(40, 32, seed=16), num_epochs=2)
    torch.cuda.synchronize()
    after = state(eng_a)
    for x, y in zip(before, after):
        assert torch.equal(x, y) if isinstance(x, torch.Tensor) else x == y
    la, lb = eng_a.train_step(*raw).clone(), eng_b.train_step(*raw).clone()
    torch.cuda.synchronize()
    assert torch.equal(la, lb) and torch.equal(eng_a.student.flat, eng_b.student.flat)


KINDS = [(k, "default") for k in list(MULTI) + list(UNI)] + [("multi_central", m) for m in ("semi_supervised", "mse", "infonce")]


@pytest.mark.parametrize("kind,mode", KINDS)
def test_compute_accuracies_on_every_compiled_kind(kind, mode):
    lit = _lit(kind, mode=mode)
    res = dt.compute_accuracies(lit.model, _batches(96, 32, seed=17), _batches(40, 16, seed=18), num_epochs=2)
    assert 0.0 <= res["knn_acc"] <= 100.0 and 0.0 <= res["mlp_acc"] <= 100.0
    m = res["metrics"]
    assert m["accuracy"] == pytest.approx(res["mlp_acc"] / 100.0, rel=1e-12, abs=1e-15)
    assert m["confusion_matrix"].shape == (10, 10) and int(m["confusion_matrix"].sum()) == 40
    assert math.isclose(sum(m[str(c)]["support"] for c in range(10) if str(c) in m), 40.0)


def test_the_probe_learns_labels_that_are_a_linear_function_of_the_features():
    """Labels = argmax of a random linear map of the eval-mode features the probe ends with: the probe fits them.  One full batch
    per epoch, so the train-mode features (batch statistics) and the eval-mode ones (the probe copy's running statistics, which
    converge to those batch statistics) coincide at the end; the statistics evolve the same way whatever the labels are, so a first
    run with any labels gives the final eval-mode features."""
    lit = _lit("image_simple")
    C, N, epochs, lr = 4, 512, 300, 1e-2
    g = torch.Generator().manual_seed(19)
    img = torch.rand(N, 1, 28, 28, generator=g) * torch.empty(N, 1, 1, 1).uniform_(0.05, 1.0, generator=g)     # diverse features
    data = [(img, torch.rand(N, 1, 112, 112, generator=g), torch.randint(0, C, (N,), generator=g))]
    first, _ = dt.train_downstream(lit.model, data, data, num_epochs=epochs, learning_rate=lr, num_classes=C)
    with torch.no_grad():
        feats = first.encoder(img.to(DEV), None).double()
    proj = torch.randn(feats.shape[1], C, dtype=torch.float64, generator=torch.Generator().manual_seed(0)).to(DEV)
    data = [(img, data[0][1], ((feats - feats.mean(0)) @ proj).argmax(1).cpu())]
    res = dt.compute_accuracies(lit.model, data, data, num_epochs=epochs, learning_rate=lr, num_classes=C)
    assert res["mlp_acc"] > 90.0, res["mlp_acc"]


# ------------------------------------------------------------------------------------------------------------
# run_dino.py --evaluate
# ------------------------------------------------------------------------------------------------------------
def _run(tmp_path, monkeypatch, extra):
    import run_dino
    tmp_path.mkdir(parents=True, exist_ok=True)
    cfg = yaml.safe_load(open(os.path.join(MIRROR, "configs", "config_multimodal_dino.yaml")))
    cfg["data"]["data_dir"] = str(tmp_path / "data") + "/"
    cfg["model"]["model_dir_data"], cfg["model"]["model_dir_scratch"] = str(tmp_path / "runs" / "data"), str(tmp_path / "runs" / "scratch")
    path = tmp_path / "config.yaml"
    path.write_text(yaml.safe_dump(cfg))
    monkeypatch.setenv("SLURM_CPUS_PER_TASK", "0")          # no DataLoader worker processes
    results = run_dino.main(["--model", "multi_central", "--config", str(path), "--synthetic", "256", "--max_steps", "2", "--seeds", "1", "2"]
                            + extra)
    summaries = list((tmp_path / "runs" / "data").glob("*/performance_summary.txt"))
    assert len(summaries) == 1
    return results, summaries[0]


def test_run_dino_evaluate_end_to_end(tmp_path, monkeypatch):
    results, summary = _run(tmp_path / "a", monkeypatch, ["--evaluate"])
    assert [r["seed"] for r in results] == [1, 2]
    for r in results:
        assert 0.0 <= r["knn_acc"] <= 100.0 and 0.0 <= r["mlp_acc"] <= 100.0
    text = summary.read_text()
    for key in ("knn_acc", "mlp_acc"):
        vals = np.array([r[key] for r in results])
        assert f"{key}: {vals.mean():.4f} ± {vals.std():.4f} (mean ± std over seeds)" in text
    for seed in (1, 2):
        with open(summary.parent / f"downstream_metrics_seed{seed}.json") as f:
            js = json.load(f)
        assert js["seed"] == seed and js["mlp_acc"] == results[seed - 1]["mlp_acc"]
        assert js["metrics"]["accuracy"] == pytest.approx(js["mlp_acc"] / 100.0) and len(js["metrics"]["confusion_matrix"]) == 10
    # without the flag: today's summary (the same lines and keys; only the times differ)
    plain, summary2 = _run(tmp_path / "b", monkeypatch, [])
    assert [set(r) for r in plain] == [{"seed", "train_loss", "training_time_s", "avg_batch_time"}] * 2
    t2 = summary2.read_text()
    assert "knn_acc" not in t2 and "mlp_acc" not in t2 and "±" not in t2
    assert not list(summary2.parent.glob("downstream_metrics_seed*.json"))
    strip = [ln for ln in text.splitlines() if "± " not in ln]
    assert len(strip) == len(t2.splitlines())
