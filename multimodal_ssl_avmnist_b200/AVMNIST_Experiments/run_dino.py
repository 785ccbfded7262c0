"""Experiment driver with the reference's command line (run_dino.py:560-582):

    python run_dino.py --model multi_central --config config_multimodal_dino.yaml [--training_mode default|semi_supervised|mse|infonce]
    python run_dino.py --unimodal_model image_simple --config config_multimodal_dino.yaml

It builds the same Lightning module with the same keyword arguments, the same data module and Trainer arguments and runs the
3-seed training loop on the B200 step.  Out of scope (DESIGN.md section 1): Optuna searches, GFLOPs tables, plots.
`--evaluate` runs the reference's post-training evaluation after each seed (compute_accuracies: kNN + the 10-epoch MLP probe on
the device, DESIGN.md section 4.11) and adds knn_acc / mlp_acc to the summary.  `--synthetic N` writes an AVMNIST-shaped
synthetic data set first (smoke runs without the real files); `--max_steps` bounds each seed's run.  For N GPUs launch one process per GPU:
    torchrun --nproc-per-node N run_dino.py --model multi_central --config ...
"""
import argparse
import copy
import json
import os
import shutil
import sys
import time
from datetime import datetime
from pathlib import Path

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, HERE)
from utils.reproducibility import set_seed  # noqa: E402
set_seed()
import yaml  # noqa: E402
from _compat import CSVLogger, ModelCheckpoint, pl  # noqa: E402
from configs.update_config import update_hardware_config  # noqa: E402
from hyperparameter_tuning.objective_augment import process_augment_config  # noqa: E402
from models.dino import (CentralMultiModalEncoder, CrossAttentionMultiModalEncoder, DualViTMultiModalEncoder, GatedMultiModalEncoder,  # noqa: E402
                         ImageEncoder, ImageEncoderCentral, LSTMMultiModalEncoder, MobileViTMultiModalEncoder, MultiModalDINOLightning,
                         MultiModalDINOSemiSupervisedLightning, MultiModalDINOWithINFONCELightning, MultiModalDINOWithMSELightning,
                         ResNetMultiModalEncoder, SimpleMultiModalEncoder, SpectrogramEncoder, SpectrogramEncoderCentral,
                         SpectrogramEncoderLSTM, SpectrogramEncoderMobileViT, SpectrogramEncoderResNet, SpectrogramEncoderViT,
                         UniModalDINOLightning, ViTMultiModalEncoder)
from utils.get_data import (AVMNISTDinoDataModule, AVMNISTDinoDataModuleExtended, MultiModalAugmentation,  # noqa: E402
                            write_synthetic_avmnist)

MODEL_MAP = {"multi_simple": SimpleMultiModalEncoder, "multi_simple_gated": GatedMultiModalEncoder, "multi_lstm": LSTMMultiModalEncoder,
             "multi_vit": ViTMultiModalEncoder, "multi_dual_vit": DualViTMultiModalEncoder, "multi_mobile_vit": MobileViTMultiModalEncoder,
             "multi_resnet": ResNetMultiModalEncoder, "multi_cross_attention": CrossAttentionMultiModalEncoder,
             "multi_central": CentralMultiModalEncoder}
UNIMODAL_MODEL_MAP = {"image_simple": ImageEncoder, "spectrogram_simple": SpectrogramEncoder, "spectrogram_central": SpectrogramEncoderCentral,
                      "spectrogram_lstm": SpectrogramEncoderLSTM, "spectrogram_resnet": SpectrogramEncoderResNet,
                      "spectrogram_vit": SpectrogramEncoderViT, "spectrogram_mobile_vit": SpectrogramEncoderMobileViT,
                      "image_central": ImageEncoderCentral}
MULTIMODAL_WRAPPERS = {"default": MultiModalDINOLightning, "semi_supervised": MultiModalDINOSemiSupervisedLightning,
                       "mse": MultiModalDINOWithMSELightning, "infonce": MultiModalDINOWithINFONCELightning}


class ModelStatsCallback(pl.Callback):
    """Wall-clock statistics with the reference's metric names (run_dino.py:191-225): avg_batch_time, epoch_time,
    total_training_time -- measured with CUDA events instead of unsynchronised time.time()."""

    def on_train_start(self, trainer, pl_module):
        import torch
        self.t0, self.batch_ms, self.epoch_s = time.time(), [], []
        self.ev = (torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) if torch.cuda.is_available() else None

    def on_train_epoch_start(self, trainer, pl_module):
        self.e0 = time.time()

    def on_train_batch_start(self, trainer, pl_module, batch, batch_idx):
        if self.ev:
            self.ev[0].record()

    def on_train_batch_end(self, trainer, pl_module, outputs, batch, batch_idx):
        if self.ev and batch_idx % 10 == 0:
            self.ev[1].record()
            self.ev[1].synchronize()
            self.batch_ms.append(self.ev[0].elapsed_time(self.ev[1]))

    def on_train_epoch_end(self, trainer, pl_module):
        self.epoch_s.append(time.time() - self.e0)
        pl_module.log("epoch_time", sum(self.epoch_s) / len(self.epoch_s))
        if self.batch_ms:
            pl_module.log("avg_batch_time", sum(self.batch_ms) / len(self.batch_ms) / 1e3)

    def on_train_end(self, trainer, pl_module):
        trainer.callback_metrics["total_training_time"] = time.time() - self.t0


def evaluate_seed(model, data, model_dir_data, seed):
    """compute_accuracies (kNN + MLP probe + metrics) of the just-trained student on the labelled train split and the test split
    of the run's data; writes downstream_metrics_seed{seed}.json and returns {"knn_acc", "mlp_acc"}."""
    from training_structures.dino_train import compute_accuracies
    if getattr(data, "test_dataset", None) is None:
        data.setup("test")
    res = compute_accuracies(model.model, data.probe_dataloaders()[0], data.test_dataloader())
    metrics = {k: (v.tolist() if hasattr(v, "tolist") else v) for k, v in res["metrics"].items()}
    os.makedirs(model_dir_data, exist_ok=True)
    with open(os.path.join(model_dir_data, f"downstream_metrics_seed{seed}.json"), "w") as f:
        json.dump({"seed": seed, "knn_acc": res["knn_acc"], "mlp_acc": res["mlp_acc"], "metrics": metrics}, f, indent=1)
    return {"knn_acc": res["knn_acc"], "mlp_acc": res["mlp_acc"]}


def experiment(config, model, ModelClass, model_name, model_dir_scratch, model_dir_data, extended_data_module=False, study=None,
               max_steps=-1, seeds=(1, 2, 3), evaluate=False):
    initial = copy.deepcopy(model.state_dict())
    hp = config["hyperparameters"]
    augments = MultiModalAugmentation(augment_values=process_augment_config(None, config, is_hyperparameter_search=False))
    cls = AVMNISTDinoDataModuleExtended if extended_data_module else AVMNISTDinoDataModule
    data = cls(data_dir=config["data"]["data_dir"], num_workers=config["hardware"]["num_workers"], batch_size=hp["batch_size"],
               n_global_views=hp.get("n_global_views", 2), n_local_views=hp.get("n_local_views", 4),
               type=hp.get("data_augmentation", "burst_noise"), augmentations=augments)
    metric = hp["metric"] if hp["metric"] != "mlp_acc" else "train_loss_epoch"     # the probe metric is out of scope
    checkpoint = ModelCheckpoint(dirpath=model_dir_scratch, monitor=metric, save_top_k=1, mode="min")
    stats = ModelStatsCallback()
    results = []
    for seed in seeds:
        print(f"Running seed: {seed}")
        set_seed(seed)
        model.load_state_dict(copy.deepcopy(initial))
        trainer = pl.Trainer(max_epochs=hp["num_epochs"], max_steps=max_steps, devices="auto",
                             strategy="ddp" if config["hardware"]["num_gpus"] > 1 else "auto", precision="16-mixed", log_every_n_steps=10,
                             logger=CSVLogger(f"{model_dir_scratch}", name=f"logs_seed{seed}"), callbacks=[checkpoint, stats],
                             deterministic=True)
        model.train()
        t0 = time.time()
        trainer.fit(model, data)
        trainer.save_checkpoint(f"{model_dir_scratch}/{model_name}.ckpt")
        m = trainer.callback_metrics
        results.append({"seed": seed, "train_loss": float(m.get("train_loss", float("nan"))), "training_time_s": time.time() - t0,
                        "avg_batch_time": float(m.get("avg_batch_time", float("nan")))})
        if evaluate:
            results[-1].update(evaluate_seed(model, data, model_dir_data, seed))
    os.makedirs(model_dir_data, exist_ok=True)
    with open(os.path.join(model_dir_data, "performance_summary.txt"), "w") as f:
        f.write(f"model_name: {config['model']['name']}\n")
        for r in results:
            f.write(", ".join(f"{k}: {v}" for k, v in r.items()) + "\n")
        if evaluate:
            import numpy as np
            for key in ("knn_acc", "mlp_acc"):
                vals = np.array([r[key] for r in results], dtype=np.float64)
                f.write(f"{key}: {vals.mean():.4f} ± {vals.std():.4f} (mean ± std over seeds)\n")
        f.write("\n# Augmentation Summary\n" + str(data.augmentations) + "\n")
    return results


def main(argv=None):
    ap = argparse.ArgumentParser()
    grp = ap.add_mutually_exclusive_group(required=True)
    grp.add_argument("--model", type=str, choices=list(MODEL_MAP))
    grp.add_argument("--unimodal_model", type=str, choices=list(UNIMODAL_MODEL_MAP))
    ap.add_argument("--training_mode", type=str, default="default", choices=list(MULTIMODAL_WRAPPERS))
    ap.add_argument("--config", type=str, required=True)
    ap.add_argument("--metric", type=str, default="mlp_acc", choices=["mlp_acc", "train_loss"])
    ap.add_argument("--hyperparameter_tune", action="store_true")
    ap.add_argument("--hyperparameter_tune_augments", action="store_true")
    ap.add_argument("--synthetic", type=int, default=0, help="write N synthetic AVMNIST-shaped training samples into data_dir first")
    ap.add_argument("--max_steps", type=int, default=-1)
    ap.add_argument("--seeds", type=int, nargs="*", default=[1, 2, 3])
    ap.add_argument("--evaluate", action="store_true", help="after each seed: kNN + MLP-probe accuracy (compute_accuracies)")
    args = ap.parse_args(argv)
    if args.unimodal_model and args.training_mode != "default":
        raise ValueError(f"--training_mode '{args.training_mode}' is only compatible with --model (multimodal models).")
    if args.hyperparameter_tune or args.hyperparameter_tune_augments:
        raise NotImplementedError("Optuna searches are outside the B200 hot-path scope (DESIGN.md section 1)")
    chosen = args.model or args.unimodal_model
    ModelClass = (MODEL_MAP if args.model else UNIMODAL_MODEL_MAP)[chosen]
    cfg_path = args.config if os.path.exists(args.config) else os.path.join(Path.cwd().parent, "configs", args.config)
    if not os.path.exists(cfg_path):
        cfg_path = os.path.join(HERE, "configs", args.config)
    config = update_hardware_config(yaml.safe_load(open(cfg_path)))
    stamp = datetime.now().strftime("%d%m%Y_%H%M%S")
    mode_tag = f"_{args.training_mode}" if args.training_mode != "default" else ""
    model_name = f"{chosen}{mode_tag}_{args.metric}_{stamp}"
    scratch, data_dir = f"{config['model']['model_dir_scratch']}/{model_name}", f"{config['model']['model_dir_data']}/{model_name}"
    for p in (scratch, data_dir):
        os.makedirs(p, exist_ok=True)
    shutil.copy(cfg_path, os.path.join(scratch, "config.yaml"))
    config["model"]["name"], config["hyperparameters"]["metric"] = chosen, args.metric
    pl.seed_everything(config["experiment"]["seed"], workers=True)
    if args.synthetic:
        write_synthetic_avmnist(config["data"]["data_dir"], n_train=args.synthetic, n_test=max(64, args.synthetic // 8),
                                type=config["hyperparameters"].get("data_augmentation", "burst_noise"))
    hp = config["hyperparameters"]
    if args.model:
        Wrapper = MULTIMODAL_WRAPPERS[args.training_mode]
        model = Wrapper(data_dir=config["data"]["data_dir"], data_augmentation=hp.get("data_augmentation", "burst_noise"), dino_model=None,
                        encoder_class=ModelClass, encoder_kwargs=None, projection_dim=hp["projection_dim"], output_dim=hp["output_dim"],
                        encoder_output_dim=hp["encoder_output_dim"], momentum=hp["momentum"], center_momentum=hp["center_momentum"],
                        student_temperature=hp["student_temperature"], teacher_temperature=hp["teacher_temperature"],
                        learning_rate=hp["learning_rate"], use_mixed_precision=True, num_epochs=hp["num_epochs"],
                        weight_decay=hp["weight_decay"], dropout=hp["dropout"])
    else:
        Wrapper = UniModalDINOLightning
        model = Wrapper(encoder_class=ModelClass, data_dir=config["data"]["data_dir"], dropout=hp["dropout"], learning_rate=hp["learning_rate"],
                        projection_dim=hp["projection_dim"], output_dim=hp["output_dim"], momentum=hp["momentum"],
                        center_momentum=hp["center_momentum"], teacher_temperature=hp["teacher_temperature"], weight_decay=hp["weight_decay"],
                        cosine_loss_alpha=hp["cosine_loss_alpha"], num_epochs=hp["num_epochs"],
                        data_augmentation=hp.get("data_augmentation", "burst_noise"))
    extended = args.training_mode != "default" and not args.unimodal_model
    extra = {"evaluate": True} if args.evaluate else {}
    return experiment(config, model, Wrapper, model_name, scratch, data_dir, extended_data_module=extended, max_steps=args.max_steps,
                      seeds=tuple(args.seeds), **extra)


if __name__ == "__main__":
    main()
