"""B200-native (sm_100a) implementation of the SR-GAN hot path of
angelowxx/Super_resolution-Image-Reconstructer-Multi_Generator_GAN behind the reference's own PyTorch surface.

    from srgan_b200 import SRResNet, Discriminator, ReconstructionLoss, train_generator, train_discriminator

All arithmetic runs in hand-written CUDA inside ``libsrgan_b200.so`` (C ABI: include/srgan_b200.h); importing this
package without that library raises as soon as a kernel is needed -- there is no CPU or PyTorch fallback.
"""
from . import _lib
from ._lib import build, check, lib
from .models import BatchNormParams, ConvParams, Discriminator, ResidualBlock, SRResNet
from . import tiling
from .tiling import plan_tiles, tile_halo
from .loss import ReconstructionLoss, bce_loss, l1_loss, mse_loss, tanh_mean
from .optim import Adam
from .policy import (GAN, PIXEL, MultiGeneratorPolicy, PolicyConfig, decide, gan_probability, interpolate_models,
                     shuffle_lists_in_same_order)
from .train import (DevicePrefetcher, GraphedDiscriminatorStep, GraphedGeneratorStep, GraphedMultiGeneratorStep, MultiGeneratorGAN, joint_pixel_generator_steps, train_discriminator, train_discriminator_async, train_generator,
                    train_generator_async, train_one_epoch, compute_score, setup_training)
from . import parallel
from . import transformers
from .vgg import VGGFeatureExtractor, perceptal_loss, perceptual_loss
from .evaluation import (ImageEnhancer, calculate_psnr, calculate_ssim, image_metrics, load_reference_checkpoint,
                         resume_learning_rates, save_reference_checkpoint, strip_module_prefix)

__all__ = ["joint_pixel_generator_steps", "SRResNet", "ResidualBlock", "Discriminator", "ReconstructionLoss", "tanh_mean", "Adam", "train_generator",
           "train_discriminator", "train_one_epoch", "compute_score", "image_metrics", "calculate_ssim", "DevicePrefetcher", "MultiGeneratorGAN", "GraphedGeneratorStep", "MultiGeneratorPolicy", "PolicyConfig",
           "build", "lib", "parallel", "tiling", "plan_tiles", "tile_halo"]
