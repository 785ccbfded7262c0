"""sbatch fan-out with the reference's arguments (batch_files/submit_models.py:28-66): one job per model."""
import argparse
import os
import subprocess

MULTIMODAL = ["multi_simple", "multi_simple_gated", "multi_lstm", "multi_vit", "multi_dual_vit", "multi_mobile_vit", "multi_resnet",
              "multi_cross_attention", "multi_central"]
UNIMODAL = ["image_simple", "spectrogram_simple", "spectrogram_central", "spectrogram_lstm", "spectrogram_resnet", "spectrogram_vit",
            "spectrogram_mobile_vit", "image_central"]


def main(argv=None):
    ap = argparse.ArgumentParser(description="Submit one SLURM job per model")
    ap.add_argument("--models", nargs="+", default=["multi_central"], choices=MULTIMODAL + UNIMODAL)
    ap.add_argument("--training_mode", default="default", choices=["default", "semi_supervised", "mse", "infonce"])
    ap.add_argument("--config", default="config_multimodal_dino.yaml")
    ap.add_argument("--metric", default="mlp_acc", choices=["mlp_acc", "train_loss"])
    ap.add_argument("--hyperparameter_tune", action="store_true")
    ap.add_argument("--hyperparameter_tune_augments", action="store_true")
    ap.add_argument("--dry_run", action="store_true", help="print the sbatch commands instead of submitting")
    args = ap.parse_args(argv)
    here = os.path.dirname(os.path.abspath(__file__))
    cmds = []
    for m in args.models:
        flag = "--unimodal_model" if m in UNIMODAL else "--model"
        cmd = ["sbatch", os.path.join(here, "run_gpu.sbatch"), flag, m, args.training_mode, args.config, args.metric,
               "1" if args.hyperparameter_tune else "0", "1" if args.hyperparameter_tune_augments else "0"]
        cmds.append(cmd)
        print(" ".join(cmd))
        if not args.dry_run:
            subprocess.run(cmd, check=True)
    return cmds


if __name__ == "__main__":
    main()
