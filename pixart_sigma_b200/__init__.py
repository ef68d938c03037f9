"""pixart_sigma_b200 -- B200-native (sm_100a) PixArt-Sigma DiT denoiser hot path.

Only what the path `PixArtMS.forward -> 28 x PixArtMSBlock.forward` needs:
  csrc/      hand-written CUDA (tcgen05 / TMA / TMEM) behind the C-ABI of include/pixart_sm100.h
  lib.py     ctypes binding of libpixart_sm100.so
  model.py   host-side mirror of the reference model API (same names, ctor, state_dict layout)
  sampler.py DPM-Solver++ and SA-Solver loops around the path (mirrors of the reference's `diffusion.DPMS` and
             `diffusion.SASolverSampler`), one fused step kernel per evaluation + CUDA graph
  autograd.py / training.py  training path: the block's ops as autograd Functions over forward + backward kernels, IDDPM loss
  parallel.py  batch-sharded inference replicas; bucketed gradient all-reduce for data-parallel training
  vae.py / t5.py  the callers either side of the path on the same kernels: SDXL-VAE (diffusers' AutoencoderKL layout) and the
             T5-v1.1-XXL caption encoder (transformers' T5EncoderModel layout)
  build.py   in-tree nvcc build
"""
from .model import (MODELS, PixArt, PixArt_XL_2, PixArtBlock, PixArtMS, PixArtMS_XL_2, PixArtMSBlock,  # noqa: F401
                    build_model, install_into_reference, set_grad_checkpoint)
from .sampler import DPMS, DPMSolverPP, SASolverSampler  # noqa: F401

__version__ = "0.1.0"
