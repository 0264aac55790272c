"""ResDiffDiffusion -- drop-in for the reference's resdiff/resdiff_diffusion.py:8-155.

The condition is whatever tensor is under ``x_in['SR']`` (bicubic x4 of LR in the reference's data loader,
dataset_builder.py:374-380); the SimpleCNN prior is loaded under ``self.cnn`` for checkpoint compatibility but, as in
the reference, never called on this path (SURVEY.md 0.1).
"""
import torch

from ...simple_cnn.Simple_CNN import SimpleCNN
from ..diffusion import GaussianDiffusion


class ResDiffDiffusion(GaussianDiffusion):
    def __init__(self, denoise_fn, image_height, image_width, channels=3, loss_type='l1', conditional=True,
                 schedule_opt=None, pretrained_model_path=None, lock_weights=True):
        super().__init__(denoise_fn=denoise_fn, channels=channels, loss_type=loss_type, conditional=conditional,
                         schedule_opt=schedule_opt, image_height=image_height, image_width=image_width,
                         pretrained_model_path=pretrained_model_path, lock_weights=lock_weights)
        self.lock_weights = lock_weights
        if pretrained_model_path is not None:
            self.cnn = SimpleCNN(scale_factor=4, channels=channels)
            self.cnn.load_state_dict(torch.load(pretrained_model_path))
            self.cnn.eval()
            if lock_weights:
                for p in self.cnn.parameters():
                    p.requires_grad_(False)
