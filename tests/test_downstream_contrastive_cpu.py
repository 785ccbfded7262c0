"""CPU: the surface of the contrastive downstream evaluation (FeatureExtractor / DownstreamClassifier / ProbeSession with
is_dino_based=False) -- what it accepts, what keeps raising the exception type it raised before the path existed, how a bare
container finds its engine, and that without a CUDA device it fails with B200Error instead of falling back."""
import os
import sys

import pytest
import torch
import torch.nn as nn

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
MIRROR = os.path.join(ROOT, "multimodal_ssl_avmnist_b200", "AVMNIST_Experiments")
sys.path.insert(0, MIRROR)

import models.dino as md  # noqa: E402
from other_ssl.info_nce.info_nce import InfoNCEModel, MultiModalInfoNCELightning  # noqa: E402
from other_ssl.multimodal_simclr.multimodal_simclr import MultiModalSimCLRLightning, MultiModalSimCLRModel  # noqa: E402
from training_structures import dino_train as dt  # noqa: E402
from multimodal_ssl_avmnist_b200 import binding as B  # noqa: E402
from multimodal_ssl_avmnist_b200._lib import B200Error  # noqa: E402
from multimodal_ssl_avmnist_b200.probe import ProbeSession  # noqa: E402

CONTAINERS = {"infonce": InfoNCEModel, "simclr": MultiModalSimCLRModel}


def _dino():
    torch.manual_seed(0)
    return md.MultiModalDINO(encoder_class=md.CentralMultiModalEncoder, output_dim=256, encoder_output_dim=256, projection_dim=128)


@pytest.mark.parametrize("kind", list(CONTAINERS))
def test_a_container_is_accepted_with_is_dino_based_false(kind):
    m = CONTAINERS[kind](output_dim=64, projection_dim=32)
    fx = md.FeatureExtractor(m, is_dino_based=False)
    assert fx.output_dim == 128 and not fx.is_unimodal and fx.modality is None
    clf = md.DownstreamClassifier(m, num_classes=7, is_dino_based=False)
    lin1, lin2 = clf.classifier[0], clf.classifier[2]
    assert (lin1.in_features, lin1.out_features, lin2.in_features, lin2.out_features) == (128, 128, 128, 7)
    assert not any(p is q for p in clf.parameters() for q in m.parameters())     # the encoders stay owned by the container


@pytest.mark.parametrize("kind", list(CONTAINERS))
def test_the_combinations_that_raised_still_raise_the_same_type(kind):
    m = CONTAINERS[kind]()
    dino = _dino()
    for model, flag in ((dino, False), (m, True), (nn.Linear(4, 4), False), (nn.Linear(4, 4), True)):
        with pytest.raises(NotImplementedError):
            md.FeatureExtractor(model, is_dino_based=flag)
        with pytest.raises(NotImplementedError):
            md.DownstreamClassifier(model, is_dino_based=flag)
    for flag in (False, True):
        with pytest.raises(NotImplementedError):
            md.DownstreamClassifier(m, trainable_encoder=True, is_dino_based=flag)
        with pytest.raises(NotImplementedError):
            md.DownstreamClassifier(dino, trainable_encoder=True, is_dino_based=flag)


@pytest.mark.parametrize("lit_cls", [MultiModalInfoNCELightning, MultiModalSimCLRLightning])
def test_a_lightning_module_is_not_a_container(lit_cls):
    """A Lightning module passes its .model; the module itself is refused as before (is_dino_based=True: it has a `_b200` binding
    but no DINO student, so the constructor fails reading it)."""
    lit = lit_cls()
    with pytest.raises(NotImplementedError):
        md.FeatureExtractor(lit, is_dino_based=False)
    with pytest.raises(AttributeError):
        md.FeatureExtractor(lit, is_dino_based=True)
    assert md.FeatureExtractor(lit.model, is_dino_based=False).output_dim == 2 * lit.output_dim


def test_a_bare_container_gets_a_binding_of_its_class_kind_once():
    for kind, cls in CONTAINERS.items():
        m = cls()
        b = B.contrastive_binding(m)
        assert isinstance(b, B.ContrastiveBinding) and b.kind == kind and b.engine is None
        assert B.contrastive_binding(m) is b
    assert B.contrastive_binding(nn.Linear(2, 2)) is None and B.contrastive_binding(_dino()) is None


@pytest.mark.parametrize("lit_cls", [MultiModalInfoNCELightning, MultiModalSimCLRLightning])
def test_a_lightning_modules_binding_is_the_one_its_container_reaches(lit_cls):
    lit = lit_cls()
    assert B.contrastive_binding(lit.model) is lit._b200 and lit._b200.kind == lit_cls.KIND


def test_without_a_device_the_contrastive_path_fails_with_b200error(monkeypatch):
    monkeypatch.setattr(torch.cuda, "is_available", lambda: False)
    m = InfoNCEModel()
    before = {k: v.clone() for k, v in m.state_dict().items()}
    images, audios, labels = torch.rand(4, 1, 28, 28), torch.rand(4, 1, 112, 112), torch.randint(0, 10, (4,))
    fx = md.FeatureExtractor(m, is_dino_based=False)
    with pytest.raises(B200Error):
        fx(images, audios)
    with pytest.raises(B200Error):
        ProbeSession(m)
    with pytest.raises(B200Error):
        dt.compute_accuracies(m, [(images, audios, labels)], [(images, audios, labels)], num_epochs=1, device="cpu",
                              is_dino_based=False)
    assert all(torch.equal(v, m.state_dict()[k]) and m.state_dict()[k].device.type == "cpu" for k, v in before.items())


def test_probe_session_refuses_other_modules():
    with pytest.raises(B200Error):
        ProbeSession(nn.Linear(4, 4))
