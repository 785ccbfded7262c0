"""GPU: the downstream evaluation of the stand-alone contrastive containers (InfoNCEModel, MultiModalSimCLRModel) with
is_dino_based=False -- features against the oracle encoders on trained weights and running statistics (fp32 and bf16), the
probe's private BatchNorm copy, isolation of the container and its optimiser state, the device probe against the torch-classifier
loop, determinism and graph vs eager, kNN against sklearn, compute_accuracies for both kinds and precisions, a probe that learns,
and Trainer.fit -> compute_accuracies end to end."""
import os
import sys

import numpy as np
import pytest
import torch
import torch.nn as nn
import torch.nn.functional as F

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
MIRROR = os.path.join(ROOT, "multimodal_ssl_avmnist_b200", "AVMNIST_Experiments")
sys.path.insert(0, MIRROR)

import models.dino as md  # noqa: E402
import utils.get_data as gd  # noqa: E402
from other_ssl.info_nce.info_nce import MultiModalInfoNCELightning  # noqa: E402
from other_ssl.multimodal_simclr.multimodal_simclr import MultiModalSimCLRLightning  # noqa: E402
from training_structures import dino_train as dt  # noqa: E402
from oracle import dino_ref as R  # noqa: E402
from multimodal_ssl_avmnist_b200 import ops  # noqa: E402
from multimodal_ssl_avmnist_b200.contrastive import AUD_LAYERS, IMG_LAYERS  # noqa: E402
from multimodal_ssl_avmnist_b200.probe import ProbeSession  # noqa: E402

DEV = "cuda"
LIT = {"infonce": MultiModalInfoNCELightning, "simclr": MultiModalSimCLRLightning}
CONV_BNS = ["enc." + bn for _, bn, *_ in IMG_LAYERS + AUD_LAYERS]


def _lit(kind, fp32=False, seed=5, steps=4, B=32):
    """A Lightning module whose container took `steps` training steps (SimCLR: every modality pairing once), so that parameters,
    Adam moments and every conv BatchNorm's running statistics are past their initial values."""
    torch.manual_seed(seed)
    lit = LIT[kind](learning_rate=1e-3, use_mixed_precision=not fp32).to(DEV)
    opt = lit.configure_optimizers()["optimizer"]
    g = torch.Generator().manual_seed(seed)
    for it in range(steps):
        views = [torch.rand(B, 1, s, s, generator=g).to(DEV) for s in (28, 112, 28, 112)]
        opt.zero_grad(set_to_none=True)
        if kind == "infonce":
            lit._b200.training_step(tuple(views[:2]))
        else:
            lit._b200.training_step(tuple(views), mode=(2, 3, 0, 1)[it % 4])
        opt.step()
    torch.cuda.synchronize()
    return lit


def _batches(n, B, seed, num_classes=10):
    g = torch.Generator().manual_seed(seed)
    img = torch.rand(n, 1, 28, 28, generator=g)
    aud = torch.rand(n, 1, 112, 112, generator=g)
    lab = torch.randint(0, num_classes, (n,), generator=g)
    return [(img[i:i + B], aud[i:i + B], lab[i:i + B]) for i in range(0, n, B)]


def _split(module):
    sd = {k: v.detach().cpu().float().clone() for k, v in module.state_dict().items()}
    p = {k: v for k, v in sd.items() if "running" not in k and "num_batches" not in k}
    buf = {k: v for k, v in sd.items() if "running" in k or "num_batches" in k}
    return p, buf


def _oracle(model, image, audio, train=False):
    """cat([ImageEncoder(image), SpectrogramEncoder(audio)], 1) of the fp32 oracle on the container's weights and buffers, and the
    buffers afterwards (train=True: _bn_train's running-statistics update)."""
    pi, bi = _split(model.image_encoder)
    pa, ba = _split(model.audio_encoder)
    fi = R.simple_image_features(image, pi, bi, pre="encoder", train=train)
    fi = F.linear(fi, pi["projection.0.weight"], pi["projection.0.bias"])
    fa = R.simple_audio_features(audio, pa, ba, pre="encoder", train=train)
    return torch.cat([fi, fa], 1), {"image_encoder": bi, "audio_encoder": ba}


def _rel(a, b):
    a, b = a.detach().cpu().double(), b.detach().cpu().double()
    return float((a - b).abs().max() / (b.abs().max() + 1e-30))


def _live_state(model):
    return {k: v.detach().clone() for k, v in model.state_dict().items()}


# ------------------------------------------------------------------------------------------------------------
# features
# ------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("kind", ["infonce", "simclr"])
def test_fp32_features_match_the_oracle_encoders(kind):
    """Eval mode: running statistics, within the fp32 forward tolerance of tests/test_contrastive_gpu.py (2e-5 of the scale).
    Train mode: batch statistics; the extractor's private running statistics take _bn_train's update and the container's do not
    move.  A new extractor starts from the live statistics."""
    lit = _lit(kind, fp32=True)
    model = lit.model
    eng = lit._b200.engine
    assert not any(eng.tc["img"]) and not any(eng.tc["aud"])
    assert all(int(eng.bn_s[k].num_batches_tracked) > 0 for k in CONV_BNS)
    B = 24
    g = torch.Generator().manual_seed(41)
    image, audio = torch.rand(B, 1, 28, 28, generator=g), torch.rand(B, 1, 112, 112, generator=g)
    live = _live_state(model)
    fx = md.FeatureExtractor(model, is_dino_based=False).eval()
    feats = fx(image.to(DEV), audio.to(DEV))
    assert feats.shape == (B, 512)
    want, _ = _oracle(model, image, audio, train=False)
    assert _rel(feats, want) < 2e-5, _rel(feats, want)
    assert _rel(feats[:, :256], want[:, :256]) < 2e-5 and _rel(feats[:, 256:], want[:, 256:]) < 2e-5
    # train mode: batch statistics and the token's running-statistics update
    fx.train()
    ftrain = fx(image.to(DEV), audio.to(DEV))
    want_t, buf_t = _oracle(model, image, audio, train=True)
    assert _rel(ftrain, want_t) < 2e-5, _rel(ftrain, want_t)
    assert float((ftrain - feats).abs().max()) > 1e-3
    for key in CONV_BNS:
        mod, base = key[len("enc."):].split(".", 1)
        bn = fx._probe["bns"][key]
        for attr in ("running_mean", "running_var"):
            assert _rel(getattr(bn, attr), buf_t[mod][f"{base}.{attr}"]) < 1e-5, (key, attr)
        assert int(bn.num_batches_tracked) == int(buf_t[mod][f"{base}.num_batches_tracked"])
    assert set(fx._probe["bns"]) == set(CONV_BNS)              # the projection heads' BatchNorms are not copied
    after = _live_state(model)
    assert all(torch.equal(live[k], after[k]) for k in live), "feature passes must not touch the container"
    adapted = fx.eval()(image.to(DEV), audio.to(DEV))
    assert float((adapted - feats).abs().max()) > 1e-4
    assert torch.equal(md.FeatureExtractor(model, is_dino_based=False).eval()(image.to(DEV), audio.to(DEV)), feats)


@pytest.mark.parametrize("kind", ["infonce", "simclr"])
def test_bf16_features_are_held_to_the_oracle(kind):
    """The tensor-core path (every conv on tcgen05, tf32 linears) against the fp32 oracle: 3e-2 of the features' scale, the bound of
    tests/test_api_gpu.py::test_feature_path_and_linear_probe; uint8 spectrograms and [B, H, W] shapes are accepted."""
    lit = _lit(kind)
    model = lit.model
    eng = lit._b200.engine
    assert all(eng.tc["img"]) and all(eng.tc["aud"])
    B = 64
    g = torch.Generator().manual_seed(42)
    image = torch.rand(B, 28, 28, generator=g)
    audio = torch.randint(0, 256, (B, 112, 112), dtype=torch.uint8, generator=g)
    fx = md.FeatureExtractor(model, is_dino_based=False).eval()
    feats = fx(image.to(DEV), audio.to(DEV))
    want, _ = _oracle(model, image[:, None], audio[:, None].float() / 255.0, train=False)
    for cols in (slice(0, 256), slice(256, 512)):
        assert _rel(feats[:, cols], want[:, cols]) < 3e-2, _rel(feats[:, cols], want[:, cols])
    ftrain = md.FeatureExtractor(model, is_dino_based=False).train()(image.to(DEV), audio.to(DEV))
    want_t, _ = _oracle(model, image[:, None], audio[:, None].float() / 255.0, train=True)
    assert _rel(ftrain, want_t) < 3e-2, _rel(ftrain, want_t)


def test_a_bare_container_on_the_host_is_bound_on_the_current_device():
    from other_ssl.info_nce.info_nce import InfoNCEModel
    torch.manual_seed(8)
    model = InfoNCEModel()
    sd = {k: v.clone() for k, v in model.state_dict().items()}
    image, audio = torch.rand(8, 1, 28, 28), torch.rand(8, 1, 112, 112)
    feats = md.FeatureExtractor(model, is_dino_based=False).eval()(image, audio)
    assert feats.is_cuda and feats.shape == (8, 512)
    eng = model._b200_contrastive.engine
    assert eng.kind == "infonce" and eng.device == torch.device("cuda", torch.cuda.current_device())
    assert model.image_encoder.encoder[0].weight.data_ptr() == eng.S["enc.image_encoder.encoder.0.weight"].data_ptr()
    assert all(torch.equal(v.cpu(), model.state_dict()[k].cpu()) for k, v in sd.items())
    want, _ = _oracle(model, image, audio)
    assert _rel(feats, want) < 3e-2


# ------------------------------------------------------------------------------------------------------------
# isolation
# ------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("kind", ["infonce", "simclr"])
def test_the_evaluation_leaves_the_container_and_its_training_untouched(kind):
    """compute_accuracies(is_dino_based=False) leaves parameters, BatchNorm buffers, Adam moments and per-branch step counts bit
    for bit, and the next training step equals the one taken without the evaluation."""
    def state(lit):
        eng = lit._b200.engine
        ts = [eng.student.flat, eng.exp_avg, eng.exp_avg_sq] + list(_live_state(lit.model).values())
        for bn in eng.bn_s.values():
            ts += [bn.running_mean, bn.running_var, bn.num_batches_tracked]
        return [t.clone() for t in ts] + [dict(eng.step_counts)]

    a, b = _lit(kind, seed=31), _lit(kind, seed=31)
    before = state(a)
    for x, y in zip(before, state(b)):
        assert torch.equal(x, y) if isinstance(x, torch.Tensor) else x == y
    dt.compute_accuracies(a.model, _batches(96, 32, seed=15), _batches(40, 16, seed=16), num_epochs=2, is_dino_based=False)
    torch.cuda.synchronize()
    for x, y in zip(before, state(a)):
        assert torch.equal(x, y) if isinstance(x, torch.Tensor) else x == y
    g = torch.Generator().manual_seed(77)
    views = tuple(torch.rand(32, 1, s, s, generator=g).to(DEV) for s in (28, 112, 28, 112))
    losses = []
    for lit in (a, b):
        opt = lit.configure_optimizers()["optimizer"]
        loss = lit._b200.training_step(views[:2] if kind == "infonce" else views, mode=None if kind == "infonce" else 2)
        opt.step()
        losses.append(float(loss.detach()))
    torch.cuda.synchronize()
    assert losses[0] == losses[1]
    for x, y in zip(state(a), state(b)):
        assert torch.equal(x, y) if isinstance(x, torch.Tensor) else x == y


# ------------------------------------------------------------------------------------------------------------
# the probe and kNN
# ------------------------------------------------------------------------------------------------------------
def _torch_probe(model, train, test, epochs, lr, seed):
    """The torch-classifier loop on the same features: DownstreamClassifier(is_dino_based=False) + AdamW + CrossEntropyLoss."""
    torch.manual_seed(seed)
    probe = md.DownstreamClassifier(model, trainable_encoder=False, is_dino_based=False).to(DEV)
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


@pytest.mark.parametrize("kind", ["infonce", "simclr"])
def test_train_downstream_matches_the_torch_classifier_loop(kind):
    lit = _lit(kind, fp32=True)
    train, test = _batches(200, 64, seed=11), _batches(96, 64, seed=12)
    want_loss, want_head, want_pred = _torch_probe(lit.model, train, test, 2, 1e-3, seed=21)
    torch.manual_seed(21)
    clf, hist = dt.train_downstream(lit.model, train, test, num_epochs=2, learning_rate=1e-3, is_dino_based=False)
    assert isinstance(clf, md.DownstreamClassifier) and clf.classifier[0].in_features == 512
    for a, b in zip(hist["train_loss"], want_loss):
        assert abs(a - b) <= 1e-5 * abs(b), (hist["train_loss"], want_loss)
    for a, b in zip(clf.classifier.state_dict().values(), want_head.state_dict().values()):
        assert float((a - b).abs().max()) <= 1e-4, float((a - b).abs().max())
    ev = clf.b200_probe.evaluate(test, predictions=True)
    assert torch.equal(ev["predictions"], want_pred)
    with torch.no_grad():
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


@pytest.mark.parametrize("kind", ["infonce", "simclr"])
def test_probe_is_deterministic_and_the_graph_path_equals_the_eager_path(kind):
    runs = [_probe_run(kind, graph) for graph in (False, False, True)]
    assert runs[0][0].O == 512
    assert runs[0][0]._graph is None and runs[2][0]._graph is not None and runs[2][0]._graph["B"] == 48     # 200 = 4 x 48 + 8: ragged
    for s, rec, ev, state in runs[1:]:
        assert rec == runs[0][1]
        assert torch.equal(ev["predictions"], runs[0][2]["predictions"]) and ev["loss"] == runs[0][2]["loss"]
        assert np.array_equal(ev["confusion_matrix"], runs[0][2]["confusion_matrix"])
        for a, b in zip(state, runs[0][3]):
            assert torch.equal(a, b)


@pytest.mark.parametrize("kind", ["infonce", "simclr"])
def test_knn_predictions_equal_sklearn_on_the_same_features(kind):
    from sklearn.neighbors import KNeighborsClassifier
    lit = _lit(kind, fp32=True)
    train, test = _batches(400, 64, seed=51), _batches(120, 64, seed=52)
    knn, acc = dt.train_knn_classifier(lit.model, train, test, n_neighbors=5, is_dino_based=False)
    assert knn.train_features.shape == (400, 512) and knn.train_features.is_cuda
    fx = md.FeatureExtractor(lit.model, is_dino_based=False).eval()
    xs = torch.cat([fx(i.to(DEV), a.to(DEV)) for i, a, _ in test])
    ys = torch.cat([t[2] for t in test])
    X, Xtr, ytr = xs.cpu().double().numpy(), knn.train_features.cpu().double().numpy(), knn.train_labels.cpu().numpy()
    sk = KNeighborsClassifier(n_neighbors=5).fit(Xtr, ytr)
    want = sk.predict(X)
    got, nbr = ops.knn_predict(knn.train_features, knn.train_labels, xs, k=5, n_classes=10, return_neighbours=True)
    assert torch.equal(got, knn.predict(xs))
    got, nbr = got.cpu().numpy(), nbr.cpu().numpy().astype(np.int64)
    d_sk, i_sk = sk.kneighbors(X, n_neighbors=6)
    # the device's neighbours are as near as sklearn's up to the fp32 rounding of its scores a.b - |b|^2 / 2 (the features of noise
    # inputs share a large common part, so near-ties are frequent here)
    err = 1e-5 * ((X ** 2).sum(1) + (Xtr ** 2).sum(1).max())
    d2_dev = np.sort(((X[:, None, :] - Xtr[nbr]) ** 2).sum(-1), 1)
    assert np.all(np.abs(d2_dev - d_sk[:, :5] ** 2) <= err[:, None])
    # the same neighbours give sklearn's prediction; a different set needs a rounding-level tie between sklearn's 5th and 6th
    # neighbours, and gives the vote of that set under sklearn's rule (majority, ties to the smallest label)
    same = np.array([set(a) == set(b) for a, b in zip(nbr, i_sk[:, :5])])
    assert np.array_equal(got[same], want[same])
    assert np.all(d_sk[~same, 5] ** 2 - d_sk[~same, 4] ** 2 <= 2 * err[~same])
    for r in np.nonzero(~same)[0]:
        assert got[r] == np.bincount(ytr[nbr[r]], minlength=10).argmax()
    print(kind, "rows whose neighbour set a near-tie changed:", int((~same).sum()), "of", len(X))
    assert abs(acc - 100.0 * float(np.mean(got == ys.numpy()))) < 1e-4          # score() averages in fp32


@pytest.mark.parametrize("fp32", [True, False])
@pytest.mark.parametrize("kind", ["infonce", "simclr"])
def test_compute_accuracies_on_both_kinds(kind, fp32):
    lit = _lit(kind, fp32=fp32)
    res = dt.compute_accuracies(lit.model, _batches(96, 32, seed=17), _batches(40, 16, seed=18), num_epochs=2, is_dino_based=False)
    assert 0.0 <= res["knn_acc"] <= 100.0 and 0.0 <= res["mlp_acc"] <= 100.0
    m = res["metrics"]
    assert m["accuracy"] == pytest.approx(res["mlp_acc"] / 100.0, rel=1e-12, abs=1e-15)
    assert m["confusion_matrix"].shape == (10, 10) and int(m["confusion_matrix"].sum()) == 40


def test_the_probe_learns_labels_that_are_a_linear_function_of_the_features():
    """As the DINO test of the same name: one full batch per epoch, labels = argmax of a random linear map of the eval-mode
    features the probe ends with; the probe fits them."""
    lit = _lit("infonce")
    C, N, epochs, lr = 4, 512, 300, 1e-2
    g = torch.Generator().manual_seed(19)
    img = torch.rand(N, 1, 28, 28, generator=g) * torch.empty(N, 1, 1, 1).uniform_(0.05, 1.0, generator=g)
    aud = torch.rand(N, 1, 112, 112, generator=g) * torch.empty(N, 1, 1, 1).uniform_(0.05, 1.0, generator=g)
    data = [(img, aud, torch.randint(0, C, (N,), generator=g))]
    first, _ = dt.train_downstream(lit.model, data, data, num_epochs=epochs, learning_rate=lr, num_classes=C, is_dino_based=False)
    with torch.no_grad():
        feats = first.encoder(img.to(DEV), aud.to(DEV)).double()
    proj = torch.randn(feats.shape[1], C, dtype=torch.float64, generator=torch.Generator().manual_seed(0)).to(DEV)
    data = [(img, aud, ((feats - feats.mean(0)) @ proj).argmax(1).cpu())]
    res = dt.compute_accuracies(lit.model, data, data, num_epochs=epochs, learning_rate=lr, num_classes=C, is_dino_based=False)
    assert res["mlp_acc"] > 90.0, res["mlp_acc"]


# ------------------------------------------------------------------------------------------------------------
# end to end
# ------------------------------------------------------------------------------------------------------------
def test_infonce_trainer_fit_then_compute_accuracies(tmp_path):
    from _compat import pl, CSVLogger
    d = str(tmp_path) + "/"
    gd.write_synthetic_avmnist(d, n_train=96, n_test=16)
    dm = gd.AVMNISTDataModule(data_dir=d, batch_size=16, num_workers=0, type="burst_noise")
    torch.manual_seed(0)
    lit = MultiModalInfoNCELightning(projection_dim=256, output_dim=256, learning_rate=1e-3, num_epochs=1)
    tr = pl.Trainer(max_epochs=1, logger=CSVLogger(str(tmp_path), name="logs"), log_every_n_steps=1, devices=1, accelerator="gpu")
    tr.fit(lit, datamodule=dm)
    assert tr.global_step >= 3
    eng = lit._b200.engine
    counts, flat = dict(eng.step_counts), eng.student.flat.clone()
    res = dt.compute_accuracies(lit.model, dm.train_dataloader(), dm.val_dataloader(), num_epochs=2, is_dino_based=False)
    assert 0.0 <= res["knn_acc"] <= 100.0 and 0.0 <= res["mlp_acc"] <= 100.0
    assert int(res["metrics"]["confusion_matrix"].sum()) == len(dm.val_dataset)
    assert eng.step_counts == counts and torch.equal(eng.student.flat, flat)
