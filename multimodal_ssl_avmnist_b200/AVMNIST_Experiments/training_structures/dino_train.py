"""Lightning-free pre-training loop with the reference's `pretrain_dino` signature (training_structures/dino_train.py:104-186).

Differences that are documented, not hidden: the reference's legacy loop expects a 2-tuple model output and a free
`dino_loss(s, t, tau_s, tau_t)` that no longer exists in its own models/dino.py (stale code); here `dino_loss` may be None
(the fused CUDA loss is used) or any callable of (student_out, teacher_out, tau_s=..., tau_t=...).  Like the reference's
loop -- and unlike its Lightning path -- the teacher EMA runs AFTER the optimizer step.

Downstream evaluation: `feature_extraction_loop` / `train_knn_classifier` (reference :327-369) run on the CUDA feature path +
the device kNN kernels (SURVEY 8f-3); `train_downstream` (the 10-epoch MLP probe on frozen features) runs on the device probe
kernels (multimodal_ssl_avmnist_b200/probe.py, DESIGN.md section 4.11); `compute_classification_metrics` reduces a confusion
matrix accumulated on the device to sklearn's classification_report; `compute_accuracies` is the post-training evaluation of
the reference's run_dino.py:389 (kNN + MLP probe + metrics).  With is_dino_based=False every one of them evaluates a stand-alone
contrastive container (InfoNCEModel / MultiModalSimCLRModel) instead: its features are its two encoders' outputs side by side
(models.dino.FeatureExtractor, DESIGN.md section 4.12)."""
import csv
import json
import os
import sys
from datetime import datetime

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import _compat  # noqa: F401,E402
from multimodal_ssl_avmnist_b200 import binding as B  # noqa: E402


def pretrain_dino(model, trainloader, dino_loss=None, align=False, num_epochs=100, learning_rate=0.0001, save_path="pretrained_dino.pt",
                  log_path="pretrain_log.csv"):
    for path in (save_path, log_path):
        os.makedirs(os.path.dirname(os.path.abspath(path)), exist_ok=True)
    stamp = datetime.now().strftime("%Y-%m-%d %H-%M-%S")
    save_path, log_path = save_path.replace(".pt", f"_{stamp}.pt"), log_path.replace(".csv", f"_{stamp}.csv")
    info = {"start_time": stamp, "learning_rate": learning_rate, "batch_size": getattr(trainloader, "batch_size", None), "epochs": num_epochs,
            "model_name": type(model).__name__}
    with open(log_path, "w", newline="") as f:
        csv.writer(f).writerow(["epoch", "train_loss", f"# {json.dumps(info)}"])
    opt = B.B200Adam(model.parameters(), model._b200, lr=learning_rate, weight_decay=0.01)     # the legacy loop uses AdamW's default decay
    best = float("inf")
    for epoch in range(num_epochs):
        model.train()
        total, n = 0.0, 0
        for batch in trainloader:
            opt.zero_grad(set_to_none=True)
            if len(batch) == 4:
                student_out, teacher_out, _ = model(tuple(batch))
            else:
                student_out, teacher_out, _ = model.forward_raw(batch[0], batch[1])
            if dino_loss is None:
                loss = model._b200.dino_loss(student_out, teacher_out, 0.1, 0.04, 0)
            else:
                loss = dino_loss(student_out, teacher_out, tau_s=0.1, tau_t=0.04)
            loss.backward()
            opt.step()
            model.update_teacher()
            total += float(loss)
            n += 1
        avg = total / max(n, 1)
        with open(log_path, "a", newline="") as f:
            csv.writer(f).writerow([epoch + 1, avg])
        if avg < best:
            best = avg
            torch.save({"epoch": epoch, "model_state_dict": model.state_dict(), "optimizer_state_dict": opt.state_dict(), "loss": best}, save_path)
    return model


def feature_extraction_loop(device, model, dataloader):
    """Frozen-encoder features of every (image, audio, label) batch (reference :327-347), kept ON THE DEVICE: returns
    (features [N, O] fp32 CUDA tensor, labels [N] int64 CUDA tensor) instead of numpy arrays."""
    model.eval()
    feats, labels = [], []
    with torch.no_grad():
        for batch in dataloader:
            images, spectrograms, lab = batch[0], batch[1], batch[2]
            feats.append(model(images.to(device), spectrograms.to(device)).float())
            labels.append(lab.to(device).long())
    return torch.cat(feats), torch.cat(labels)


class B200KNN:
    """What the reference keeps of its fitted sklearn KNeighborsClassifier: predict / score on new features."""

    def __init__(self, train_features, train_labels, n_neighbors=5, n_classes=10):
        self.train_features, self.train_labels = train_features.contiguous(), train_labels.contiguous()
        self.n_neighbors, self.n_classes = n_neighbors, n_classes

    def predict(self, features):
        from multimodal_ssl_avmnist_b200 import ops
        return ops.knn_predict(self.train_features, self.train_labels, features.to(self.train_features.device).float().contiguous(),
                               k=self.n_neighbors, n_classes=self.n_classes)

    def score(self, features, labels):
        pred = self.predict(features)
        return float((pred == labels.to(pred.device)).float().mean())


def train_knn_classifier(pretrained_dino, train_dataloader, test_dataloader, n_neighbors=5, device="cuda", is_dino_based=True):
    """kNN accuracy of the frozen student encoder (reference :349-369): features through the CUDA encoder forward, Euclidean
    k-nearest neighbours + majority vote in CUDA kernels (csrc/knn.cu).  is_dino_based=False: the frozen encoders of a contrastive
    container (InfoNCEModel / MultiModalSimCLRModel), features [N, 2 * output_dim].  Returns (knn, accuracy in %)."""
    from models.dino import FeatureExtractor
    extractor = FeatureExtractor(pretrained_dino, is_dino_based=is_dino_based)
    train_features, train_labels = feature_extraction_loop(device, extractor, train_dataloader)
    test_features, test_labels = feature_extraction_loop(device, extractor, test_dataloader)
    n_classes = int(max(int(train_labels.max()), int(test_labels.max()))) + 1
    knn = B200KNN(train_features, train_labels, n_neighbors=n_neighbors, n_classes=max(n_classes, 10))
    accuracy = 100.0 * knn.score(test_features, test_labels)
    print(f"KNN Accuracy (k={n_neighbors}): {accuracy:.4f}%")
    return knn, accuracy


def train_downstream(pretrained_model, train_loader, test_loader, num_epochs=10, learning_rate=1e-3, device="cuda", num_classes=10,
                     is_dino_based=True, graph=True):
    """The MLP probe of the frozen student (DESIGN.md section 4.11): a fresh DownstreamClassifier head (initial weights from the
    global RNG), CrossEntropyLoss, AdamW(learning_rate) with torch's defaults, `num_epochs` epochs over train_loader with
    train-mode features (batch statistics, fusion dropout, the probe's private copy of the running statistics), then an
    evaluation of test_loader with eval-mode features after every epoch.  Every step runs on the device (probe.ProbeSession).
    Returns (classifier, history): classifier is a DownstreamClassifier holding the trained head, so classifier(images,
    spectrograms) works afterwards; history = {"train_loss", "val_loss", "val_acc" (%)} per epoch, losses per sample.
    is_dino_based=False: the probe of a contrastive container's frozen encoders (no dropout; head Linear(2 * output_dim, 128)).
    The reference's body of this function is not in this tree: the signature and the semantics follow its call site and
    models/dino.py's DownstreamClassifier, not a pinned implementation."""
    from models.dino import DownstreamClassifier
    from multimodal_ssl_avmnist_b200.probe import ProbeSession
    classifier = DownstreamClassifier(pretrained_model, num_classes=num_classes, is_dino_based=is_dino_based)
    session = ProbeSession(pretrained_model, num_classes=num_classes, lr=learning_rate, weight_decay=1e-2, graph=graph,
                           head=classifier.classifier)
    classifier.encoder._probe = session.token            # classifier(...) evaluates with the probe's running statistics
    history = {"train_loss": [], "val_loss": [], "val_acc": []}
    for epoch in range(num_epochs):
        for batch in train_loader:
            session.train_batch(batch[0], batch[1], batch[2])
        train_loss, _ = session.end_epoch()
        ev = session.evaluate(test_loader)
        history["train_loss"].append(train_loss)
        history["val_loss"].append(ev["loss"])
        history["val_acc"].append(100.0 * ev["accuracy"])
        print(f"Epoch {epoch + 1}/{num_epochs}: train loss {train_loss:.4f}, val loss {ev['loss']:.4f}, val acc {100.0 * ev['accuracy']:.2f}%")
    session.export_head()
    classifier.to(session.device).eval()
    classifier.b200_probe = session
    return classifier, history


def metrics_from_confusion(cm):
    """sklearn.metrics.classification_report(y_true, y_pred, output_dict=True, zero_division=0) from the confusion matrix
    cm[label, pred] of those predictions (classes that neither occur nor are predicted are left out, as sklearn does), plus
    "confusion_matrix" = cm as int64 [C, C]."""
    import numpy as np
    cm = np.asarray(cm, dtype=np.int64)
    tp = np.diag(cm).astype(np.float64)
    support = cm.sum(axis=1)
    predicted = cm.sum(axis=0)
    present = np.nonzero((support > 0) | (predicted > 0))[0]
    out = {}
    precision, recall, f1 = {}, {}, {}
    for c in present:
        precision[c] = tp[c] / predicted[c] if predicted[c] > 0 else 0.0
        recall[c] = tp[c] / support[c] if support[c] > 0 else 0.0
        den = 2 * tp[c] + (predicted[c] - tp[c]) + (support[c] - tp[c])
        f1[c] = 2 * tp[c] / den if den > 0 else 0.0
        out[str(int(c))] = {"precision": float(precision[c]), "recall": float(recall[c]), "f1-score": float(f1[c]),
                            "support": float(support[c])}
    total = float(support.sum())
    out["accuracy"] = float(tp.sum() / total) if total > 0 else 0.0
    for name, w in (("macro avg", np.ones(len(present))), ("weighted avg", support[present].astype(np.float64))):
        ws = w.sum()
        avg = lambda d: float(np.dot(w, [d[c] for c in present]) / ws) if ws > 0 else 0.0  # noqa: E731
        out[name] = {"precision": avg(precision), "recall": avg(recall), "f1-score": avg(f1), "support": total}
    out["confusion_matrix"] = cm
    return out


def compute_classification_metrics(classifier, loader, device="cuda", num_classes=10):
    """Accuracy, per-class precision / recall / f1-score / support, macro and weighted averages (sklearn's
    classification_report(output_dict=True, zero_division=0) definitions) and the int64 confusion matrix of a DownstreamClassifier
    on `loader`.  Predictions and the confusion matrix are computed on the device (eval-mode features -> probe kernel); only the
    [C, C] matrix comes back to the host.  Works for a DINO-based and a contrastive (is_dino_based=False) classifier alike."""
    from multimodal_ssl_avmnist_b200.probe import ProbeSession
    session = getattr(classifier, "b200_probe", None)
    if session is None or session.C != num_classes:
        fx = classifier.encoder
        if fx._probe is None:
            fx._probe = fx.engine().begin_probe()
        session = ProbeSession(fx._dino[0], num_classes=num_classes, graph=False, head=classifier.classifier, probe=fx._probe)
    else:
        session.load_head(classifier.classifier)
    return metrics_from_confusion(session.evaluate(loader)["confusion_matrix"])


def compute_accuracies(pretrained_model, train_loader, test_loader, n_neighbors=5, num_epochs=10, learning_rate=1e-3, device="cuda",
                       num_classes=10, is_dino_based=True):
    """Post-training evaluation of a pretrained DINO model (reference run_dino.py:389): kNN accuracy of the frozen student's
    features, the MLP probe (train_downstream) and its classification metrics on test_loader.  is_dino_based=False: the same for a
    contrastive container (InfoNCEModel / MultiModalSimCLRModel; a Lightning module passes its .model); its parameters, BatchNorm
    buffers and optimiser state are left untouched.
    Returns {"knn_acc": %, "mlp_acc": %, "metrics": compute_classification_metrics(...)}."""
    _, knn_acc = train_knn_classifier(pretrained_model, train_loader, test_loader, n_neighbors=n_neighbors, device=device,
                                      is_dino_based=is_dino_based)
    classifier, _ = train_downstream(pretrained_model, train_loader, test_loader, num_epochs=num_epochs, learning_rate=learning_rate,
                                     device=device, num_classes=num_classes, is_dino_based=is_dino_based)
    metrics = compute_classification_metrics(classifier, test_loader, device=device, num_classes=num_classes)
    mlp_acc = 100.0 * metrics["accuracy"]
    print(f"MLP Accuracy: {mlp_acc:.4f}%")
    return {"knn_acc": float(knn_acc), "mlp_acc": mlp_acc, "metrics": metrics}
