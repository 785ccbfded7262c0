"""CPU: the host half of the downstream evaluation -- the classification-report reduction of a confusion matrix (against sklearn),
run_dino.py's --evaluate flag, and the C ABI of the probe kernels."""
import os
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
MIRROR = os.path.join(ROOT, "multimodal_ssl_avmnist_b200", "AVMNIST_Experiments")
sys.path.insert(0, MIRROR)

from training_structures.dino_train import metrics_from_confusion  # noqa: E402
from multimodal_ssl_avmnist_b200 import _lib  # noqa: E402


def _pairs(cm):
    """(y_true, y_pred) with exactly the counts of cm[label, pred]."""
    t, p = [], []
    for i in range(cm.shape[0]):
        for j in range(cm.shape[1]):
            t += [i] * int(cm[i, j])
            p += [j] * int(cm[i, j])
    return np.array(t), np.array(p)


def _check(cm):
    sk = pytest.importorskip("sklearn.metrics")
    y_true, y_pred = _pairs(cm)
    want = sk.classification_report(y_true, y_pred, output_dict=True, zero_division=0)
    got = metrics_from_confusion(cm)
    assert got["accuracy"] == pytest.approx(sk.accuracy_score(y_true, y_pred), abs=1e-15)
    assert got["accuracy"] == pytest.approx(want["accuracy"], abs=1e-15)
    assert set(got) - {"confusion_matrix"} == set(want)
    for key, row in want.items():
        if key == "accuracy":
            continue
        for m in ("precision", "recall", "f1-score", "support"):
            assert got[key][m] == pytest.approx(row[m], rel=1e-12, abs=1e-15), (key, m)
    C = cm.shape[0]
    assert got["confusion_matrix"].dtype == np.int64 and got["confusion_matrix"].shape == (C, C)
    assert np.array_equal(got["confusion_matrix"], sk.confusion_matrix(y_true, y_pred, labels=list(range(C))))


def test_report_of_a_perfect_classifier():
    _check(np.diag([5, 3, 7, 1]).astype(np.int64))


def test_report_with_a_class_never_predicted_and_a_class_absent_from_the_labels():
    cm = np.zeros((10, 10), dtype=np.int64)
    cm[0, 0], cm[0, 1], cm[1, 1], cm[2, 0], cm[2, 1] = 4, 2, 5, 3, 1     # class 2 occurs but is never predicted
    cm[3, 4], cm[3, 3] = 2, 1                                             # class 4 is predicted but never occurs
    got = metrics_from_confusion(cm)
    assert got["2"]["precision"] == 0.0 and got["2"]["recall"] == 0.0 and got["2"]["f1-score"] == 0.0
    assert got["4"]["support"] == 0.0 and got["4"]["recall"] == 0.0
    assert "9" not in got                                                 # neither occurs nor is predicted: left out, as sklearn does
    _check(cm)


def test_report_of_a_classifier_that_predicts_one_class():
    cm = np.zeros((10, 10), dtype=np.int64)
    cm[:, 7] = np.arange(1, 11)
    _check(cm)


@pytest.mark.parametrize("seed", range(20))
def test_report_matches_sklearn_on_random_confusion_matrices(seed):
    rng = np.random.default_rng(seed)
    C = int(rng.integers(2, 17))
    cm = rng.integers(0, 30, (C, C)) * (rng.random((C, C)) < 0.6)
    cm[rng.integers(0, C)] = 0                   # one class absent from the labels
    cm[:, rng.integers(0, C)] = 0                # one class never predicted
    if cm.sum() == 0:
        cm[0, 0] = 1
    _check(cm.astype(np.int64))


def _config(tmp_path):
    import yaml
    cfg = yaml.safe_load(open(os.path.join(MIRROR, "configs", "config_multimodal_dino.yaml")))
    cfg["data"]["data_dir"] = str(tmp_path / "data") + "/"
    cfg["model"]["model_dir_data"], cfg["model"]["model_dir_scratch"] = str(tmp_path / "runs" / "data"), str(tmp_path / "runs" / "scratch")
    path = tmp_path / "config.yaml"
    path.write_text(yaml.safe_dump(cfg))
    return path


def test_run_dino_passes_evaluate_only_when_asked(tmp_path, monkeypatch):
    """Without --evaluate, experiment() gets exactly the arguments it got before the flag existed; with it, evaluate=True on top."""
    import run_dino
    monkeypatch.setenv("SLURM_CPUS_PER_TASK", "0")
    path = _config(tmp_path)
    calls = []
    monkeypatch.setattr(run_dino, "experiment", lambda *a, **k: calls.append((a, k)) or [])
    argv = ["--model", "multi_central", "--config", str(path), "--max_steps", "2", "--seeds", "1", "2"]
    run_dino.main(argv)
    run_dino.main(argv + ["--evaluate"])
    (a0, k0), (a1, k1) = calls
    assert set(k0) == {"extended_data_module", "max_steps", "seeds"}
    assert k0 == {"extended_data_module": False, "max_steps": 2, "seeds": (1, 2)}
    assert k1 == dict(k0, evaluate=True)
    assert len(a0) == len(a1) == 6 and a0[2] is a1[2] and a0[0]["model"]["name"] == "multi_central"


def test_the_probe_entry_points_are_declared_and_exported():
    import ctypes
    decl = {n: (r, t) for n, r, t in _lib.declared_functions()}
    assert decl["b200_probe_work_floats"] == ("int64_t", ["int", "int"])
    ret, types = decl["b200_probe_mlp_fwd_bwd"]
    assert ret == "int" and types == ["ptr"] * 6 + ["int"] * 4 + ["ptr"] * 6 + ["ptr"]
    for name in ("b200_adamw_flat", "b200_adamw_flat_dev"):
        assert decl[name][0] == "int"
    assert decl["b200_adamw_flat"][1] == decl["b200_adam_flat"][1][:-2] + ["ptr"]          # Adam's list without grad_scale
    if not os.path.exists(_lib.LIB_PATH):
        from multimodal_ssl_avmnist_b200.build import build
        build()
    raw = ctypes.CDLL(_lib.LIB_PATH)
    for name in ("b200_probe_work_floats", "b200_probe_mlp_fwd_bwd", "b200_adamw_flat", "b200_adamw_flat_dev"):
        assert hasattr(raw, name)


def test_probe_argument_errors_are_reported_without_a_gpu():
    lib = _lib.load()
    assert lib.b200_probe_work_floats(128, 10) == 16 + 128 * (2 * 128 + 10)       # 8 fp64 loss partials, hidden, its gradient, d_logits
    assert lib.b200_probe_work_floats(1, 17) == -2
    assert lib.b200_probe_mlp_fwd_bwd(None, None, None, None, None, None, 4, 256, 10, 1, None, None, None, None, None, None, None) == -1
    assert b"probe_mlp_fwd_bwd" in lib.b200_last_error()
    p = 16                                        # any non-null, aligned value: the checks come before any access
    assert lib.b200_probe_mlp_fwd_bwd(p, p, p, p, p, p, 4, 60, 10, 0, None, p, p, p, None, None, None) == -2
    assert lib.b200_probe_mlp_fwd_bwd(p, p, p, p, p, p, 4, 256, 17, 0, None, p, p, p, None, None, None) == -2
    assert lib.b200_probe_mlp_fwd_bwd(p, p, p, p, p, p, 4, 256, 10, 1, None, p, p, p, None, None, None) == -1      # train needs grad
    assert lib.b200_adamw_flat(None, None, None, None, 0, 1e-3, 0.9, 0.999, 1e-8, 1e-2, 1.0, 1.0, None) == -1
    assert lib.b200_adamw_flat_dev(None, None, None, None, 8, 1e-3, 0.9, 0.999, 1e-8, 1e-2, None, None) == -1
