"""Stand-alone multimodal InfoNCE pre-training, B200-native (same public surface as the reference's other_ssl/info_nce/info_nce.py).

`InfoNCEModel` is a parameter container (ImageEncoder + SpectrogramEncoder + two ProjectionHeads, state_dict keys as in the
reference); `MultiModalInfoNCELightning.training_step` runs forward, the symmetric InfoNCE loss and the whole backward pass in the CUDA
kernels of libavmnist_b200.so (multimodal_ssl_avmnist_b200.contrastive.ContrastiveStepEngine) and `configure_optimizers` returns the
flat-arena Adam.  No PyTorch fallback."""
import os
import sys

import torch
import torch.nn as nn

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__)))))
from _compat import pl  # noqa: E402
from models.dino import ImageEncoder, ProjectionHead, SpectrogramEncoder  # noqa: E402
from multimodal_ssl_avmnist_b200 import binding as B  # noqa: E402


class InfoNCEModel(nn.Module):
    B200_CONTRASTIVE_KIND = "infonce"          # the ContrastiveStepEngine kind a bare container is bound to

    def __init__(self, output_dim=256, projection_dim=256):
        super().__init__()
        self.output_dim, self.projection_dim = output_dim, projection_dim
        self.image_encoder = ImageEncoder(output_dim=output_dim)
        self.audio_encoder = SpectrogramEncoder(output_dim=output_dim)
        self.image_projection_head = ProjectionHead(output_dim, projection_dim)
        self.audio_projection_head = ProjectionHead(output_dim, projection_dim)

    def forward(self, batch):
        """(images, spectrograms, labels) -> (image_features, audio_features): inference-form forward on the CUDA kernels."""
        images, spectrograms, _ = batch
        return (self.image_projection_head(self.image_encoder(images.float(), None)),
                self.audio_projection_head(self.audio_encoder(None, spectrograms.float())))


class MultiModalInfoNCELightning(pl.LightningModule):
    KIND = "infonce"

    def __init__(self, projection_dim=256, output_dim=256, learning_rate=0.0001, num_epochs=100, use_mixed_precision=True):
        super().__init__()
        self.output_dim, self.projection_dim = output_dim, projection_dim
        self.model = InfoNCEModel(output_dim=output_dim, projection_dim=projection_dim)
        self.model.use_mixed_precision = use_mixed_precision
        self.learning_rate, self.use_mixed_precision, self.num_epochs = learning_rate, use_mixed_precision, num_epochs
        self._b200 = B.ContrastiveBinding(self.model, self.KIND)
        self.save_hyperparameters()

    def forward(self, batch):
        return self.model(batch)

    def infoNCE_loss(self, image_outputs, audio_outputs, temperature=0.07):
        """Symmetric InfoNCE of two [B, D] CUDA tensors through the fused kernel (differentiable w.r.t. both)."""
        return B.standalone_pair_loss("infonce", image_outputs, audio_outputs, temperature=temperature)

    def training_step(self, batch, batch_idx):
        images, spectrograms = batch[0], batch[1]
        loss = self._b200.training_step((images, spectrograms))
        self.log("train_loss", loss, on_step=True, on_epoch=True, prog_bar=True)
        return loss

    def configure_optimizers(self):
        optimizer = B.ContrastiveAdam(self.parameters(), self._b200, lr=self.learning_rate)
        scheduler = torch.optim.lr_scheduler.CosineAnnealingLR(optimizer, T_max=self.num_epochs)
        return {"optimizer": optimizer, "lr_scheduler": {"scheduler": scheduler, "monitor": "train_loss"}}
