"""cednerf_b200 — B200-native (sm_100a) implementation of Ced-NeRF's per-ray volumetric rendering hot path.

Module map (reference surface -> here):
    nerfacc (subset)                       cednerf_b200.nerfacc
    tinycudann (subset)                    cednerf_b200.tcnn
    cednerf/taichi_kernel hash encoders    cednerf_b200.hash_encoder
    cednerf/encoder.py                     cednerf_b200.encoder
    cednerf/model.py                       cednerf_b200.model
    cednerf/render.py                      cednerf_b200.render
    cednerf/utils.py                       cednerf_b200.utils
    apex FusedAdam + torch GradScaler      cednerf_b200.optim
    loss of train_real.py:369-409          cednerf_b200.losses
    datasets/dnerf_3d_video_IS.py (per-step importance sampling)   cednerf_b200.importance
    pytorch_msssim.ms_ssim (evaluation, train_real.py:497-499)     cednerf_b200.metrics
All compute goes through libcednerf_b200.so (include/cednerf_b200.h); there is no CPU fallback."""
from . import _lib

_lib.load()  # fail loudly if the CUDA library has not been built

from . import encoder, hash_encoder, importance, losses, metrics, model, nerfacc, ops, optim, render, tcnn, utils  # noqa: E402
from .model import DNGPradianceField  # noqa: E402
from .nerfacc import OccGridEstimator  # noqa: E402
from .render import rendering  # noqa: E402
from .utils import Rays, render_image, render_image_test, render_images_test  # noqa: E402

__all__ = ["DNGPradianceField", "OccGridEstimator", "rendering", "render_image", "render_image_test", "render_images_test", "Rays",
           "nerfacc", "tcnn", "hash_encoder", "encoder", "model", "render", "utils", "ops", "optim", "losses", "importance",
           "metrics"]
