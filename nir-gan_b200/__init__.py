"""nirgan_b200 -- B200-native (sm_100a) drop-in for the NIR-GAN data-parallel hot path.

Mirrors the reference's Python surface for this path (SURVEY.md section 8b):
  model.networks           define_G, define_D, ResnetGenerator, ResnetBlock, NLayerDiscriminator, GANLoss
  model.generator_inject   define_G_inject, ResnetGenerator_inject
  model.pix2pix            Px2Px  (Lightning-free restatement of Px2Px_PL forward / training_step)
  utils.remote_sensing_indices  RemoteSensingIndices
  synth                    tile-sharded create_synthetic_dataset-style inference loop
  scene                    NIR band of a whole scene: overlapping tiles cut and blended on the device, row bands
All arithmetic runs in csrc/libnirgan_b200.so (hand-written CUDA for sm_100a) through the C ABI of
include/nirgan_b200.h.  There is no CPU fallback.
"""
from . import _lib  # noqa: F401
from .engine import EngineConfig  # noqa: F401

__all__ = ["EngineConfig"]
