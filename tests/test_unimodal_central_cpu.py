"""CPU: the unimodal LeNet-style CentralNet DINO models (UniModalDINO(ImageEncoderCentral), kind "image_central", and
UniModalDINO(SpectrogramEncoderCentral), kind "spectrogram_central") -- their parameter surface against the engine's inventory and
layer tables, the command line, and the reference step of tests/unimodal_dino_ref.py with the encoders of
tests/unimodal_central_ref.py against the multimodal oracle's branches."""
import importlib.util
import os
import sys

import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
MIRROR = os.path.join(ROOT, "multimodal_ssl_avmnist_b200", "AVMNIST_Experiments")
sys.path.insert(0, MIRROR)

import models.dino as md  # noqa: E402
from multimodal_ssl_avmnist_b200 import engine as E  # noqa: E402
from oracle import dino_ref as R  # noqa: E402
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import unimodal_dino_ref as U  # noqa: E402
import unimodal_central_ref  # noqa: E402,F401  (registers the CentralNet kinds with the reference step)
from oracle.fixtures import make_masks, synth_views, views_to_vb  # noqa: E402

# kind -> (API class name, modality, engine params, engine layer table, multimodal layer table, multimodal branch prefix, flat width)
KINDS = {"image_central": ("ImageEncoderCentral", "image", E.image_central_params, E.CENTRAL_IMAGE_UNI_LAYERS, E.CENTRAL_IMAGE_LAYERS,
                           "image_encoder", 64 * 5 * 5),
         "spectrogram_central": ("SpectrogramEncoderCentral", "audio", E.spectrogram_central_params, E.CENTRAL_AUDIO_UNI_LAYERS,
                                 E.CENTRAL_AUDIO_LAYERS, "audio_encoder", 64 * 7 * 7)}


@pytest.mark.parametrize("kind", list(KINDS))
def test_central_unimodal_parameters_match_the_engine_inventory(kind):
    cls_name, modality, params_fn, layers, multi_layers, branch, flat = KINDS[kind]
    cls = getattr(md, cls_name)
    assert cls.B200_KIND == kind
    torch.manual_seed(0)
    u = md.UniModalDINO(encoder_class=cls, output_dim=256, projection_dim=128)
    assert u._b200.kind == kind and u.student.modality == modality
    params = [(k, tuple(v.shape)) for k, v in u.student.named_parameters()]
    used, unused = params_fn(256)
    # used + unused == the module's parameters (the arena orders used first); the module's order == the reference step's spec
    assert sorted(params) == sorted((k, tuple(s)) for k, s in used + unused)
    assert params == [(k, tuple(s)) for k, s in U.UNIMODAL_KINDS[kind][0](256)]
    assert {k for k, _ in unused} == {f"encoder.0.fc{i}.{w}" for i in (1, 2) for w in ("weight", "bias")}
    assert dict(params)["encoder.1.weight"] == (256, flat)
    assert [k for k, _ in u.teacher.named_parameters()] == [k for k, _ in params]
    # the layer table is multi_central's branch re-prefixed, and names the container's conv / BatchNorm modules with their geometry
    assert [tuple(r) for _, _, *r in layers] == [tuple(r) for _, _, *r in multi_layers]
    assert [(c, b) for c, b, *_ in layers] == [(c.replace(branch, "encoder", 1), b.replace(branch, "encoder", 1)) for c, b, *_ in multi_layers]
    mods = dict(u.student.named_modules())
    for conv, bn, ci, co, hw, k, pad in layers:
        c = mods[conv]
        assert isinstance(c, torch.nn.Conv2d) and (c.in_channels, c.out_channels, c.kernel_size[0], c.padding[0]) == (ci, co, k, pad)
        assert isinstance(mods[bn], torch.nn.BatchNorm2d) and mods[bn].num_features == co
    assert [bn for _, bn, *_ in layers] == U.UNIMODAL_KINDS[kind][1]()
    # the engine's top: flatten of the last pooled activation into encoder.1, whose output is the embedding
    mod, top, chain = E.UNI_KINDS[kind]
    assert mod == ("img" if modality == "image" else "aud") and top == ("flat", flat)
    assert chain == [("enc.encoder.1", "top", "feat", None)]
    co, hw, k, pad = layers[-1][3], layers[-1][4], layers[-1][5], layers[-1][6]
    assert co * ((hw + 2 * pad - k + 1) // 2) ** 2 == flat


def test_the_simple_kinds_keep_their_average_pool_top():
    assert E.UNI_KINDS["image_simple"][1] == ("pool", 128) and E.UNI_KINDS["spectrogram_simple"][1] == ("pool", 256)


def test_spectrogram_encoder_central_is_compiled_and_the_lstm_family_is_not():
    enc = md.SpectrogramEncoderCentral(output_dim=64)
    assert enc.modality == "audio" and enc.encoder[1].in_features == 3136 and enc.encoder[1].out_features == 64
    enc = md.ImageEncoderCentral(output_dim=64)
    assert enc.modality == "image" and enc.encoder[1].in_features == 1600
    with pytest.raises(NotImplementedError) as e:
        md.LSTMMultiModalEncoder()
    assert "ImageEncoderCentral" in str(e.value) and "SpectrogramEncoderCentral" in str(e.value)
    with pytest.raises(ValueError):
        enc(None, torch.zeros(1, 1, 112, 112))


def test_command_line_resolves_both_central_models():
    import run_dino
    assert run_dino.UNIMODAL_MODEL_MAP["image_central"] is md.ImageEncoderCentral
    assert run_dino.UNIMODAL_MODEL_MAP["spectrogram_central"] is md.SpectrogramEncoderCentral
    spec = importlib.util.spec_from_file_location("submit_models", os.path.join(MIRROR, "batch_files", "submit_models.py"))
    sm = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(sm)
    cmds = sm.main(["--models", "image_central", "spectrogram_central", "--dry_run"])
    assert [c[2:4] for c in cmds] == [["--unimodal_model", "image_central"], ["--unimodal_model", "spectrogram_central"]]


@pytest.mark.parametrize("alpha", [0.0, 0.3])
@pytest.mark.parametrize("kind", list(KINDS))
def test_reference_step_runs_and_its_encoder_is_the_multimodal_branch(kind, alpha):
    """The composed unimodal step runs, leaves fc1 / fc2 without gradients and unmoved by Adam but EMA's them, and its encoder forward
    equals the multimodal oracle's branch (pinned against the reference through multi_central) on the same weights re-keyed."""
    _, modality, _, _, _, branch, _ = KINDS[kind]
    B = 3
    st = U.UniModalDinoState(kind=kind, seed=11)
    img, aud = views_to_vb(*synth_views(B, seed=100))
    views = img if modality == "image" else aud
    # encoder forward == the multimodal oracle's branch (fresh buffers on both sides)
    p = {k.replace("encoder.", f"{branch}.", 1): v for k, v in st.student.items()}
    buf_a = R.make_bn_buffers(st.enc_spec, st.bn_names)
    buf_b = {k.replace("encoder.", f"{branch}.", 1): v.clone() for k, v in buf_a.items()}
    mine = U.UNIMODAL_KINDS[kind][2](views[0], st.student, buf_a)
    ref = (R.central_image_features if modality == "image" else R.central_audio_features)(views[0], p, buf_b)
    assert mine.shape == (B, 256) and torch.equal(mine, ref)
    for k, v in buf_a.items():
        assert torch.equal(v, buf_b[k.replace("encoder.", f"{branch}.", 1)]), k
    # the whole step
    masks = make_masks(seed=200, V=6, Vg=2, B=B, E=256, hidden=512)
    s0 = {k: v.clone() for k, v in st.student.items()}
    t0 = {k: v.clone() for k, v in st.teacher.items()}
    got = U.unimodal_dino_step(st, views, masks, cosine_loss_alpha=alpha)
    assert torch.isfinite(got["loss"]) and (got["cosine"] is None) == (alpha == 0)
    assert got["embeddings"].shape == (6, B, 256) and got["student_out"].shape == (6, B, 128)
    fc = {k for k in s0 if ".fc" in k}
    assert len(fc) == 4 and not fc & set(got["grads"]["student"])
    assert set(got["grads"]["student"]) == set(s0) - fc
    for k in fc:
        assert torch.equal(st.student[k], s0[k]), k
    for k in t0:
        assert torch.equal(st.teacher[k], 0.996 * t0[k] + (1 - 0.996) * s0[k]), k
    assert st.adam["step"] == 1 and max(float((st.student[k] - s0[k]).abs().max()) for k in s0) > 0


@pytest.mark.parametrize("kind", list(KINDS))
def test_run_dino_builds_the_central_model_on_a_cpu_box(tmp_path, monkeypatch, kind):
    """`run_dino.py --unimodal_model {image_central,spectrogram_central}` constructs the model and its data; without a GPU the first
    training step then stops with the engine's "needs a CUDA device" error and nothing earlier."""
    if torch.cuda.is_available():
        pytest.skip("checks the behaviour of a machine without a GPU")
    import shutil

    import run_dino
    import yaml
    cfg = yaml.safe_load(open(os.path.join(MIRROR, "configs", "config_multimodal_dino.yaml")))
    cfg["data"]["data_dir"] = str(tmp_path / "data") + "/"
    cfg["model"]["model_dir_data"], cfg["model"]["model_dir_scratch"] = str(tmp_path / "runs" / "data"), str(tmp_path / "runs" / "scratch")
    path = tmp_path / "config.yaml"
    path.write_text(yaml.safe_dump(cfg))
    monkeypatch.setenv("SLURM_CPUS_PER_TASK", "0")
    built = []
    orig = run_dino.experiment

    def spy(config, model, *a, **k):
        built.append(model)
        return orig(config, model, *a, **k)

    monkeypatch.setattr(run_dino, "experiment", spy)
    with pytest.raises(Exception) as e:
        run_dino.main(["--unimodal_model", kind, "--config", str(path), "--synthetic", "64", "--max_steps", "1", "--seeds", "1"])
    assert "CUDA" in str(e.value), repr(e.value)
    assert len(built) == 1 and isinstance(built[0].model.student, getattr(md, KINDS[kind][0]))
    assert built[0].model._b200.kind == kind
    shutil.rmtree(tmp_path / "runs", ignore_errors=True)
