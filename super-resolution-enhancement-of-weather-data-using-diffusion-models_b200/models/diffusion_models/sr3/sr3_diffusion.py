"""SR3Diffusion -- drop-in for the reference's sr3/sr3_diffusion.py:8-140: the condition is ``x_in['SR']``, the target of the
forward process is HR itself (no residual), and the sampler returns the final image WITHOUT adding the condition (:84)."""
from ..diffusion import GaussianDiffusion


class SR3Diffusion(GaussianDiffusion):
    residual = False

    def __init__(self, denoise_fn, channels=1, image_height=128, image_width=256, loss_type='l1', conditional=True,
                 schedule_opt=None, pretrained_model_path=None, lock_weights=True):
        super().__init__(denoise_fn=denoise_fn, channels=channels, loss_type=loss_type, conditional=conditional,
                         schedule_opt=schedule_opt, image_height=image_height, image_width=image_width,
                         pretrained_model_path=pretrained_model_path, lock_weights=lock_weights)
