"""PhyDiffDiffusion -- drop-in for the reference's phydiff/phydiff_diffusion.py:9-139: ResDiff's process (residual target
HR - SR, sampler returns image + condition) around the PhyDiff UNet; the moment loss of the reference is commented out there
(:134-137) and therefore absent here too."""
from ..diffusion import GaussianDiffusion


class PhyDiffDiffusion(GaussianDiffusion):
    def __init__(self, denoise_fn, channels=1, image_height=128, image_width=256, loss_type='l1', conditional=True,
                 schedule_opt=None, pretrained_model_path=None, lock_weights=True):
        super().__init__(denoise_fn=denoise_fn, channels=channels, loss_type=loss_type, conditional=conditional,
                         schedule_opt=schedule_opt, image_height=image_height, image_width=image_width,
                         pretrained_model_path=pretrained_model_path, lock_weights=lock_weights)
