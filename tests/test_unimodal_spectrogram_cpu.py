"""CPU: the audio-only DINO model (UniModalDINO(SpectrogramEncoder), kind "spectrogram_simple") -- its parameter surface against the
reference's own SpectrogramEncoder state dict (tests/golden/golden_contrastive.json), the engine's inventory, the oracle's unimodal
step against the composition of its pinned pieces, and the run_dino.py command line up to the point where a GPU is needed."""
import os
import re
import shutil
import sys

import pytest
import torch
import yaml

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
MIRROR = os.path.join(ROOT, "multimodal_ssl_avmnist_b200", "AVMNIST_Experiments")
sys.path.insert(0, MIRROR)

import models.dino as md  # noqa: E402
from multimodal_ssl_avmnist_b200 import engine as E  # noqa: E402
from oracle import dino_ref as R  # noqa: E402
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import unimodal_dino_ref as U  # noqa: E402
from oracle.fixtures import make_masks, summaries_close, summarize, synth_views, views_to_vb  # noqa: E402


def test_spectrogram_dino_parameters_match_the_reference_encoder(golden_contrastive):
    """Student / teacher state-dict keys and shapes == the reference SpectrogramEncoder's (model.audio_encoder.* of the contrastive
    fixture), and the parameter specs == the engine's arena inventory and the oracle's spec, in the same order."""
    torch.manual_seed(0)
    u = md.UniModalDINO(encoder_class=md.SpectrogramEncoder, output_dim=256, projection_dim=128)
    assert u._b200.kind == "spectrogram_simple" and u.student.modality == "audio"
    ref = {k[len("model.audio_encoder."):]: v for k, v in golden_contrastive["infonce"]["state_dict"].items()
           if k.startswith("model.audio_encoder.encoder.")}
    assert len(ref) == 4 * 7 + 2
    for role in ("student", "teacher"):
        sd = getattr(u, role).state_dict()
        assert list(sd) == list(ref), role
        assert all(list(sd[k].shape) == ref[k] for k in ref), role
    params = [(k, tuple(v.shape)) for k, v in u.student.named_parameters()]
    used, unused = E.spectrogram_simple_params(256)
    assert unused == [] and params == [(k, tuple(s)) for k, s in used] == [(k, tuple(s)) for k, s in R.spectrogram_spec(256)]
    # the layer table names exactly the conv / BatchNorm modules of the container, with their geometry
    mods = dict(u.student.named_modules())
    for conv, bn, ci, co, hw, k, pad in E.SPECTROGRAM_LAYERS:
        c = mods[conv]
        assert isinstance(c, torch.nn.Conv2d) and (c.in_channels, c.out_channels, c.kernel_size[0], c.padding[0]) == (ci, co, k, pad)
        assert isinstance(mods[bn], torch.nn.BatchNorm2d) and mods[bn].num_features == co
    assert [bn for _, bn, *_ in E.SPECTROGRAM_LAYERS] == R.spectrogram_bn_names()
    # no projection layer: the embedding is the encoder.18 output
    assert E.UNI_KINDS["spectrogram_simple"][2][-1][0] == "enc.encoder.18" and "projection.0.weight" not in dict(params)


def _composed(st, views, masks, alpha, dropout=0.3):
    """The unimodal step's loss and gradients written out from the pinned pieces with plain autograd."""
    V, B = views.shape[0], views.shape[1]
    S = {k: v.clone().requires_grad_(True) for k, v in st.student.items()}
    SH = {k: v.clone().requires_grad_(True) for k, v in st.student_head.items()}
    sbuf = {k: v.clone() for k, v in st.student_buf.items()}
    tbuf = {k: v.clone() for k, v in st.teacher_buf.items()}
    hbuf = {k: v.clone() for k, v in st.student_head_buf.items()}
    thbuf = {k: v.clone() for k, v in st.teacher_head_buf.items()}
    emb = torch.cat([R.simple_audio_features(views[v], S, sbuf, pre="encoder") for v in range(V)])
    with torch.no_grad():
        tf = torch.cat([R.simple_audio_features(views[v], st.teacher, tbuf, pre="encoder") for v in range(2)])
        tp = R.projection_head(tf, st.teacher_head, thbuf)
    sp = R.projection_head(emb, SH, hbuf, masks["student_head"], dropout)
    loss = R.dino_loss_unimodal(sp.view(V, B, -1), (tp - st.center).view(2, B, -1))
    if alpha > 0:
        loss = loss + alpha * R.cosine_consistency_loss(emb.view(V, B, -1))
    loss.backward()
    return loss.detach(), {k: v.grad for k, v in S.items()}, {k: v.grad for k, v in SH.items()}, R.center_update(st.center, tp)


@pytest.mark.parametrize("alpha", [0.0, 0.3])
def test_oracle_spectrogram_step_is_the_composition_of_its_pinned_pieces(alpha):
    B = 3
    st = U.UniModalDinoState(kind="spectrogram_simple", seed=11)
    _, aud = views_to_vb(*synth_views(B, seed=100))
    masks = make_masks(seed=200, V=6, Vg=2, B=B, E=256, hidden=512)
    want_loss, want_g, want_gh, want_center = _composed(st, aud, masks, alpha)
    s0 = {k: v.clone() for k, v in st.student.items()}
    t0 = {k: v.clone() for k, v in st.teacher.items()}
    got = U.unimodal_dino_step(st, aud, masks, cosine_loss_alpha=alpha)
    assert torch.equal(got["loss"], want_loss)
    assert (got["cosine"] is None) == (alpha == 0)
    if alpha > 0:
        assert float(got["cosine"]) > 0 and abs(float(got["dino"] + alpha * got["cosine"]) - float(want_loss)) < 1e-6
    for k, g in want_g.items():
        assert torch.equal(got["grads"]["student"][k], g), k
    for k, g in want_gh.items():
        assert torch.equal(got["grads"]["student_head"][k], g), k
    assert set(got["grads"]["student"]) == {n for n, _ in R.spectrogram_spec(256)}
    assert torch.equal(st.center, want_center)
    assert got["embeddings"].shape == (6, B, 256) and got["student_out"].shape == (6, B, 128)
    # EMA on the pre-step student, then one Adam step moves the student
    for k in t0:
        assert torch.equal(st.teacher[k], 0.996 * t0[k] + (1 - 0.996) * s0[k]), k
    assert st.adam["step"] == 1 and max(float((st.student[k] - s0[k]).abs().max()) for k in s0) > 0


def _cancelled(name):
    return re.search(r"(mlp\.0\.bias|projection\.0\.bias|(?<!_)encoder\.[048]\.bias|(?<!_)encoder\.14\.bias)$", name) is not None


@pytest.mark.parametrize("key,alpha", [("unimodal_image_simple", 0.0), ("unimodal_image_simple_cosine", 0.3)])
def test_oracle_unimodal_step_reproduces_the_reference_on_the_image_encoder(golden, key, alpha):
    """The same unimodal step with the image encoder reproduces the imported reference's own training step (golden.json): the
    step order, the head, the loss variant and the cosine term of unimodal_dino_step are the reference's."""
    fx = golden[key]
    B = fx["B"]
    st = U.UniModalDinoState(kind="image_simple", seed=fx["seed"])
    img, _ = views_to_vb(*synth_views(B, seed=100))
    masks = make_masks(seed=200, V=6, Vg=2, B=B, E=256, hidden=512)
    got = U.unimodal_dino_step(st, img, masks, cosine_loss_alpha=alpha)
    assert abs(float(got["loss"]) - fx["loss"]) < 2e-5 * fx["loss"], (float(got["loss"]), fx["loss"])
    for k, ref in fx["grads"].items():
        if _cancelled(k):
            continue
        name = k.replace("model.student_projection.", "").replace("model.student.", "")
        group = "student_head" if k.startswith("model.student_projection.") else "student"
        ok, why = summaries_close(summarize(got["grads"][group][name]), ref, 3e-4, 1e-7)
        assert ok, (k, why)
    for k, ref in fx["teacher"].items():
        ok, why = summaries_close(summarize(st.teacher[k]), ref, 1e-6, 1e-9)
        assert ok, (k, why)


def test_run_dino_builds_the_spectrogram_model_on_a_cpu_box(tmp_path, monkeypatch):
    """`run_dino.py --unimodal_model spectrogram_simple` constructs the model and its data; without a GPU the first training step
    then stops with the engine's "needs a CUDA device" error and nothing earlier."""
    if torch.cuda.is_available():
        pytest.skip("checks the behaviour of a machine without a GPU")
    import run_dino
    cfg = yaml.safe_load(open(os.path.join(MIRROR, "configs", "config_multimodal_dino.yaml")))
    cfg["data"]["data_dir"] = str(tmp_path / "data") + "/"
    cfg["model"]["model_dir_data"], cfg["model"]["model_dir_scratch"] = str(tmp_path / "runs" / "data"), str(tmp_path / "runs" / "scratch")
    path = tmp_path / "config.yaml"
    path.write_text(yaml.safe_dump(cfg))
    monkeypatch.setenv("SLURM_CPUS_PER_TASK", "0")          # no DataLoader worker processes
    built = []
    orig = run_dino.experiment

    def spy(config, model, *a, **k):
        built.append(model)
        return orig(config, model, *a, **k)

    run_dino.experiment = spy
    try:
        with pytest.raises(Exception) as e:
            run_dino.main(["--unimodal_model", "spectrogram_simple", "--config", str(path), "--synthetic", "64", "--max_steps", "1",
                           "--seeds", "1"])
    finally:
        run_dino.experiment = orig
    assert "CUDA" in str(e.value), repr(e.value)
    assert len(built) == 1 and isinstance(built[0], md.UniModalDINOLightning)
    assert isinstance(built[0].model.student, md.SpectrogramEncoder) and built[0].model._b200.kind == "spectrogram_simple"
    shutil.rmtree(tmp_path / "runs", ignore_errors=True)
