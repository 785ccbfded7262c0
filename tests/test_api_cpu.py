"""CPU: the Python API mirror (AVMNIST_Experiments/...) keeps the reference's surface: module / class names, constructor
keywords, state_dict keys and shapes, seeded initialisation, config helpers, CLI -- checked against fixtures generated from
the imported reference (tests/golden/api_surface.json).  No CUDA needed; the compute path itself must refuse CPU tensors."""
import json
import os
import sys

import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
MIRROR = os.path.join(ROOT, "multimodal_ssl_avmnist_b200", "AVMNIST_Experiments")
sys.path.insert(0, MIRROR)

import models.dino as md  # noqa: E402
import utils.get_data as gd  # noqa: E402
from hyperparameter_tuning.objective_augment import process_augment_config  # noqa: E402
from oracle.fixtures import summaries_close, summarize  # noqa: E402


@pytest.fixture(scope="module")
def surface():
    return json.load(open(os.path.join(ROOT, "tests", "golden", "api_surface.json")))


CLASSES = {"default": md.MultiModalDINO, "semi_supervised": md.MultiModalDINOSemiSupervised, "infonce": md.MultiModalDINOWithINFONCE,
           "mse": md.MultiModalDINOWithMSE}


@pytest.mark.parametrize("mode", list(CLASSES))
def test_state_dict_and_seeded_init_match_reference(mode, surface):
    torch.manual_seed(123)
    m = CLASSES[mode](encoder_class=md.CentralMultiModalEncoder, output_dim=256, encoder_output_dim=256, projection_dim=128)
    sd = m.state_dict()
    ref = surface[mode]["keys"]
    assert list(sd.keys()) == list(ref.keys())                       # same names, same order
    assert all(list(sd[k].shape) == ref[k] for k in ref)
    for k, want in surface[mode]["init"].items():                     # same RNG consumption -> same initial weights
        ok, why = summaries_close(summarize(sd[k]), want, 1e-12, 0.0)
        assert ok, (k, why)
    assert [n for n, p in m.named_parameters() if not p.requires_grad] == [n for n, _ in m.named_parameters() if n.startswith("teacher")]
    assert torch.equal(m.teacher.fusion[0].weight, m.student.fusion[0].weight)


def test_unimodal_surface(surface):
    torch.manual_seed(123)
    u = md.UniModalDINO(encoder_class=md.ImageEncoder, output_dim=256, projection_dim=128)
    sd = u.state_dict()
    assert list(sd.keys()) == list(surface["unimodal"]["keys"].keys())
    for k, want in surface["unimodal"]["init"].items():
        ok, why = summaries_close(summarize(sd[k]), want, 1e-12, 0.0)
        assert ok, (k, why)


def test_lightning_wrappers_accept_the_reference_kwargs():
    kw = dict(data_dir="x/", data_augmentation="burst_noise", dino_model=None, encoder_class=md.CentralMultiModalEncoder, encoder_kwargs=None,
              projection_dim=128, output_dim=256, encoder_output_dim=256, momentum=0.996, center_momentum=0.9, student_temperature=0.1,
              teacher_temperature=0.04, learning_rate=1e-4, use_mixed_precision=True, num_epochs=100, weight_decay=1e-6, dropout=0.3)
    for cls in (md.MultiModalDINOLightning, md.MultiModalDINOSemiSupervisedLightning, md.MultiModalDINOWithINFONCELightning,
                md.MultiModalDINOWithMSELightning):
        lit = cls(**kw)
        for attr in ("training_step", "dino_loss", "configure_optimizers", "on_train_epoch_end", "forward", "model"):
            assert hasattr(lit, attr)
        cfg = lit.configure_optimizers()
        assert isinstance(cfg["optimizer"], torch.optim.Optimizer) and cfg["optimizer"].param_groups[0]["lr"] == 1e-4
        assert isinstance(cfg["lr_scheduler"]["scheduler"], torch.optim.lr_scheduler.CosineAnnealingLR)
    assert hasattr(md.MultiModalDINOWithINFONCELightning, "infoNCE_loss") and hasattr(md.MultiModalDINOWithMSELightning, "mse_loss")
    assert hasattr(md.MultiModalDINOSemiSupervisedLightning, "supervised_loss")
    uni = md.UniModalDINOLightning(encoder_class=md.ImageEncoder, data_dir="x/", dropout=0.3, learning_rate=1e-4, projection_dim=128,
                                   output_dim=256, momentum=0.996, center_momentum=0.9, teacher_temperature=0.04, weight_decay=1e-6,
                                   cosine_loss_alpha=0, num_epochs=100, data_augmentation="burst_noise")
    assert uni.student_temperature == 0.1


def test_every_encoder_name_of_run_dino_imports():
    for name in ("CrossAttentionMultiModalEncoder", "DualViTMultiModalEncoder", "GatedMultiModalEncoder", "LSTMMultiModalEncoder",
                 "MobileViTMultiModalEncoder", "ResNetMultiModalEncoder", "SimpleMultiModalEncoder", "ViTMultiModalEncoder",
                 "CentralMultiModalEncoder", "SpectrogramEncoder", "SpectrogramEncoderCentral", "SpectrogramEncoderLSTM",
                 "SpectrogramEncoderResNet", "SpectrogramEncoderViT", "SpectrogramEncoderMobileViT", "ImageEncoder"):
        assert hasattr(md, name)
    with pytest.raises(NotImplementedError):
        md.LSTMMultiModalEncoder()
    # the conv encoder family of SURVEY 8f-4 has a compiled step: state_dict keys as in the reference (models/dino.py:214-263, 385-452)
    for cls, extra in ((md.SimpleMultiModalEncoder, set()), (md.GatedMultiModalEncoder, {"gate_image", "gate_audio"}),
                       (md.CrossAttentionMultiModalEncoder, {f"{a}.{p}.{w}" for a in ("image_to_audio_attention", "audio_to_image_attention")
                                                             for p in ("q_proj", "kv_proj") for w in ("weight", "bias")})):
        m = md.MultiModalDINO(encoder_class=cls, output_dim=256, encoder_output_dim=256, projection_dim=128)
        keys = set(m.student.state_dict())
        assert extra <= keys and {"image_encoder.14.weight", "audio_encoder.18.weight", "audio_encoder.12.weight", "fusion.3.bias"} <= keys
        assert m._b200.kind == cls.B200_KIND
        from multimodal_ssl_avmnist_b200.engine import simple_multi_params, MULTI_KINDS
        spec = dict(simple_multi_params(256, 256, MULTI_KINDS[cls.B200_KIND])[0])
        params = {k: tuple(v.shape) for k, v in m.student.named_parameters()}
        assert params == spec, set(params) ^ set(spec)


def test_no_cpu_fallback():
    m = md.MultiModalDINO(encoder_class=md.CentralMultiModalEncoder, output_dim=256, encoder_output_dim=256, projection_dim=128)
    batch = (torch.rand(2, 2, 1, 28, 28), torch.rand(2, 2, 1, 112, 112), torch.rand(2, 4, 1, 28, 28), torch.rand(2, 4, 1, 112, 112))
    with pytest.raises(Exception) as e:
        m(batch)
    assert "CUDA" in str(e.value) or "cuda" in str(e.value)


def test_process_augment_config_and_augmentation_object():
    import yaml
    cfg = yaml.safe_load(open(os.path.join(MIRROR, "configs", "config_multimodal_dino.yaml")))
    av = process_augment_config(None, cfg, is_hyperparameter_search=False)
    assert list(av["augmentations"]["local_views"]) == ["frequency_mask", "gaussian_noise", "grouped_masking", "time_mask", "time_warp",
                                                        "random_resized_crop", "random_affine"]
    assert av["augmentation_probabilities"]["global_views"]["random_resized_crop"] == 0.9
    with pytest.raises(ValueError):
        process_augment_config(None, {}, is_hyperparameter_search=False)
    aug = gd.MultiModalAugmentation(augment_values=av)
    assert aug.n_global_views == 2 and aug.n_local_views == 4 and "GroupedMasking" in str(aug)
    assert len(aug.local_transforms["audio"]) == 7 and len(aug.global_transforms["image"]) == 3

    class Trial:        # the search branch only needs the suggest_* protocol
        def suggest_float(self, k, lo, hi): return (lo + hi) / 2
        def suggest_int(self, k, lo, hi, step=1): return lo
        def suggest_categorical(self, k, c): return c[0]
    space = {"optuna": {"augmentations": {"global_views": {"time_mask": {"p": {"low": 0.0, "high": 1.0}, "time_mask_param": {"type": "int", "low": 5, "high": 30}}},
                                          "local_views": {}}}}
    got = process_augment_config(Trial(), space, True)
    assert got["augmentations"]["global_views"]["time_mask"] == {"time_mask_param": 5}
    assert got["augmentation_probabilities"]["global_views"]["time_mask"] == 0.5


def test_data_module_and_synthetic_files(tmp_path):
    d = str(tmp_path) + "/"
    gd.write_synthetic_avmnist(d, n_train=40, n_test=16)
    dm = gd.AVMNISTDinoDataModuleExtended(data_dir=d, batch_size=8, num_workers=0, type="burst_noise")
    dm.prepare_data()
    dm.setup("fit")
    image, audio, label = next(iter(dm.train_dataloader()))
    assert image.shape == (8, 1, 28, 28) and audio.shape == (8, 1, 112, 112) and label.dtype == torch.long
    assert float(audio.max()) <= 1.0 and dm.get_view_config() == {"n_global_views": 2, "n_local_views": 4}
    with pytest.raises(FileNotFoundError):
        gd.AVMNISTDinoDataModule(data_dir=d + "missing/", batch_size=8, num_workers=0).prepare_data()


def test_cli_surfaces():
    import run_dino
    assert set(run_dino.MODEL_MAP) >= {"multi_central", "multi_simple"} and "image_simple" in run_dino.UNIMODAL_MODEL_MAP
    assert list(run_dino.MULTIMODAL_WRAPPERS) == ["default", "semi_supervised", "mse", "infonce"]
    with pytest.raises(SystemExit):
        run_dino.main(["--config", "x.yaml"])                         # a model is required
    sys.path.insert(0, os.path.join(MIRROR, "batch_files"))
    import submit_models
    cmds = submit_models.main(["--models", "multi_central", "image_simple", "--training_mode", "mse", "--dry_run"])
    assert cmds[0][2:4] == ["--model", "multi_central"] and cmds[1][2:4] == ["--unimodal_model", "image_simple"] and cmds[0][4] == "mse"


def test_trainer_shim_runs_a_toy_module(tmp_path):
    from multimodal_ssl_avmnist_b200 import pl_shim as pls

    class Toy(pls.LightningModule):
        def __init__(self, lr=0.1):
            super().__init__()
            self.w = torch.nn.Parameter(torch.tensor([2.0]))
            self.lr = lr
            self.save_hyperparameters()

        def training_step(self, batch, idx):
            loss = ((self.w * batch) ** 2).mean()
            self.log("train_loss", loss, on_step=True, on_epoch=True)
            return loss

        def configure_optimizers(self):
            opt = torch.optim.SGD(self.parameters(), lr=self.lr)
            return {"optimizer": opt, "lr_scheduler": {"scheduler": torch.optim.lr_scheduler.CosineAnnealingLR(opt, T_max=2)}}

    if torch.cuda.is_available():
        pytest.skip("CPU-only check")
    ckpt = pls.ModelCheckpoint(dirpath=str(tmp_path), monitor="train_loss_epoch", mode="min")
    tr = pls.Trainer(max_epochs=2, logger=pls.CSVLogger(str(tmp_path), name="logs"), callbacks=[ckpt], log_every_n_steps=1)
    model = Toy()
    tr.fit(model, train_dataloaders=[torch.ones(4) for _ in range(5)])
    assert tr.global_step == 10 and float(model.w) < 2.0
    assert "train_loss_epoch" in tr.callback_metrics and os.path.exists(ckpt.best_model_path)
    assert os.path.exists(os.path.join(tr.logger.log_dir, "metrics.csv"))
    again = Toy.load_from_checkpoint(ckpt.best_model_path)
    assert again.lr == 0.1


def test_quad8_width_covers_every_tap_of_every_output_phase():
    """The first-layer image has ceil((W + 2 pad) / 4) units per row: the last valid pixel group's taps kw' = ph + kw stay
    inside its 8-pixel unit for the three first-layer geometries (host-side shape logic, no GPU)."""
    import importlib
    ops_src = open(os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "multimodal_ssl_avmnist_b200", "ops.py")).read()
    ns = {}
    start = ops_src.index("def quad8_width")
    exec(ops_src[start:ops_src.index("\n\n\n", start)], ns)
    for W, K, pad in ((112, 5, 2), (28, 5, 2), (28, 3, 1)):
        wq = ns["quad8_width"](W, pad)
        assert 4 * wq >= W + 2 * pad
        last_group = W // 4 - 1                      # outputs 4*g .. 4*g+3
        assert 3 + (K - 1) <= 7                      # kw' = ph + kw < 8
        assert last_group < wq


def test_ddp_ranks_train_on_disjoint_shards(tmp_path, monkeypatch):
    """strategy='ddp' (run_dino.py:359): real Lightning injects a DistributedSampler; the shim must shard too.  Device-resident
    loader: same permutation on every rank, strided slices, disjoint and equally long; a plain DataLoader is rebuilt around a
    DistributedSampler; an unshardable iterable is refused instead of being silently replicated."""
    from multimodal_ssl_avmnist_b200 import pl_shim
    gd.write_synthetic_avmnist(str(tmp_path) + "/", n_train=96, n_test=16)
    dm = gd.AVMNISTDinoDataModule(str(tmp_path) + "/", batch_size=8, num_workers=0)
    dm.setup("fit")
    sub = dm.train_dataset
    seen = []
    for rank in range(2):
        ld = gd.DeviceResidentLoader(sub.dataset, sub.indices, 8, torch.device("cpu"), shuffle=True, with_labels=True, seed=5)
        ld.labels = torch.arange(ld.image.shape[0])           # sample ids, to see which samples a rank draws
        ld.set_rank_shard(rank, 2)
        ids = torch.cat([b[2] for b in ld])
        assert len(ld) == ld.image.shape[0] // 2 // 8 and ids.numel() == len(ld) * 8
        seen.append(set(ids.tolist()))
    assert not (seen[0] & seen[1])
    monkeypatch.setenv("WORLD_SIZE", "2")
    monkeypatch.setenv("RANK", "1")
    tr = pl_shim.Trainer(strategy="ddp")
    plain = torch.utils.data.DataLoader(torch.utils.data.TensorDataset(torch.arange(40)), batch_size=4, shuffle=True)
    sharded = tr._shard_loader(plain)
    assert isinstance(sharded.sampler, torch.utils.data.distributed.DistributedSampler) and sharded.sampler.rank == 1
    assert sum(b[0].numel() for b in sharded) == 20
    with pytest.raises(RuntimeError):
        tr._shard_loader([1, 2, 3])


def test_contrastive_mirrors_have_the_reference_surface(golden_contrastive):
    """other_ssl/info_nce/info_nce.py and other_ssl/multimodal_simclr/multimodal_simclr.py of the mirror: same classes, constructor
    keywords, methods and state_dict keys / shapes as the imported reference (tests/golden/golden_contrastive.json 'state_dict')."""
    import other_ssl.info_nce.info_nce as nce
    import other_ssl.multimodal_simclr.multimodal_simclr as simclr
    for mod, cls, key, loss_name in ((nce, "MultiModalInfoNCELightning", "infonce", "infoNCE_loss"),
                                     (simclr, "MultiModalSimCLRLightning", "simclr", "nt_xent_loss")):
        lit = getattr(mod, cls)(projection_dim=256, output_dim=256, learning_rate=1e-4, num_epochs=100, use_mixed_precision=True)
        want = golden_contrastive[key]["state_dict"]
        got = {k: list(v.shape) for k, v in lit.state_dict().items()}
        assert got == want, set(got) ^ set(want)
        for attr in ("training_step", "configure_optimizers", "forward", "model", loss_name):
            assert hasattr(lit, attr)
        cfg = lit.configure_optimizers()
        assert isinstance(cfg["optimizer"], torch.optim.Optimizer) and cfg["lr_scheduler"]["monitor"] == "train_loss"
        batch = (torch.rand(2, 1, 28, 28), torch.rand(2, 1, 112, 112), torch.rand(2, 1, 28, 28), torch.rand(2, 1, 112, 112))
        if torch.cuda.is_available():                        # no CPU fallback: a host batch is stepped on the device
            assert lit.training_step(batch, 0).is_cuda
        else:
            with pytest.raises(Exception):
                lit.training_step(batch, 0)
