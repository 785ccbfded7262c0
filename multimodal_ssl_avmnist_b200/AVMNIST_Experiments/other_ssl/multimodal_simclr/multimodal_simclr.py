"""Multimodal SimCLR pre-training, B200-native (same public surface as the reference's other_ssl/multimodal_simclr/multimodal_simclr.py).

`MultiModalSimCLRModel` is a parameter container; `MultiModalSimCLRLightning.training_step` draws the reference's random modality pairing
(torch.randint(0, 4, (1,)): image-image, audio-audio, image-audio, audio-image), runs both views through the chosen encoders and heads,
NT-Xent on cat([z1, z2]) and the whole backward pass in the CUDA kernels (ContrastiveStepEngine).  Branches a step did not use keep
.grad = None and are skipped by the optimizer, like in the reference.  No PyTorch fallback."""
import os
import sys

import torch
import torch.nn as nn

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__)))))
from _compat import pl  # noqa: E402
from models.dino import ImageEncoder, ProjectionHead, SpectrogramEncoder  # noqa: E402
from multimodal_ssl_avmnist_b200 import binding as B  # noqa: E402


class MultiModalSimCLRModel(nn.Module):
    B200_CONTRASTIVE_KIND = "simclr"          # the ContrastiveStepEngine kind a bare container is bound to

    def __init__(self, output_dim=256, projection_dim=256):
        super().__init__()
        self.output_dim, self.projection_dim = output_dim, projection_dim
        self.image_encoder = ImageEncoder(output_dim=output_dim)
        self.audio_encoder = SpectrogramEncoder(output_dim=output_dim)
        self.image_projection_head = ProjectionHead(output_dim, projection_dim)
        self.audio_projection_head = ProjectionHead(output_dim, projection_dim)

    def forward(self, batch):
        """(aug_img1, aug_spec1, aug_img2, aug_spec2) -> (z1, z2) with a random modality pairing: inference-form forward."""
        img1, spec1, img2, spec2 = (t.float() for t in batch)
        mode = torch.randint(0, 4, (1,)).item()
        enc_i = lambda x: self.image_projection_head(self.image_encoder(x, None))          # noqa: E731
        enc_a = lambda x: self.audio_projection_head(self.audio_encoder(None, x))          # noqa: E731
        if mode == 0:
            return enc_i(img1), enc_i(img2)
        if mode == 1:
            return enc_a(spec1), enc_a(spec2)
        if mode == 2:
            return enc_i(img1), enc_a(spec2)
        return enc_a(spec1), enc_i(img2)


class MultiModalSimCLRLightning(pl.LightningModule):
    KIND = "simclr"

    def __init__(self, projection_dim=256, output_dim=256, learning_rate=0.0001, num_epochs=100, use_mixed_precision=True):
        super().__init__()
        self.output_dim, self.projection_dim = output_dim, projection_dim
        self.model = MultiModalSimCLRModel(output_dim=output_dim, projection_dim=projection_dim)
        self.model.use_mixed_precision = use_mixed_precision
        self.learning_rate, self.use_mixed_precision, self.num_epochs = learning_rate, use_mixed_precision, num_epochs
        self._b200 = B.ContrastiveBinding(self.model, self.KIND)
        self.save_hyperparameters()

    def forward(self, batch):
        return self.model(batch)

    def nt_xent_loss(self, reps, temperature=0.07):
        """NT-Xent of reps = cat([z1, z2]) (CUDA tensor [2B, D]) through the fused kernel, differentiable w.r.t. reps."""
        return B.standalone_ntxent_loss(reps, temperature=temperature)

    def training_step(self, batch, batch_idx):
        mode = int(torch.randint(0, 4, (1,)).item())          # the reference's draw (multimodal_simclr.py:29), from the global torch RNG
        loss = self._b200.training_step(tuple(batch[:4]), mode=mode)
        self.log("train_loss", loss, on_step=True, on_epoch=True, prog_bar=True)
        return loss

    def configure_optimizers(self):
        optimizer = B.ContrastiveAdam(self.parameters(), self._b200, lr=self.learning_rate)
        scheduler = torch.optim.lr_scheduler.CosineAnnealingLR(optimizer, T_max=self.num_epochs)
        return {"optimizer": optimizer, "lr_scheduler": {"scheduler": scheduler, "monitor": "train_loss"}}
