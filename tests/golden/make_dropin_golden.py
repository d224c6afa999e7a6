#!/usr/bin/env python
"""Generate tests/golden/dropin_autoencoding_eval.npz from the original PDAE project (ckczzj/PDAE).

    python tests/golden/make_dropin_golden.py <path to a checkout of ckczzj/PDAE>

Runs what the original's sampler/autoencoding_eval.py computes, with the original's own modules on the CPU in fp32:
a CELEBA64Encoder + CELEBA64Decoder loaded from a synthetic checkpoint, GaussianDiffusion.representation_learning_autoencoding
('ddim1000', 'ddim100') over 3 synthetic 64x64 images in batches of 2 + 1, and the per-image MSE / SSIM of
metric/utils.py on [0,1]-scaled images.  tests/test_gpu_dropin_script.py runs the same evaluation on this package's
kernels and compares with this file.  Weights and images are not stored: both sides regenerate them with
pdae_b200.utils.synth.
"""
import json
import os
import sys

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.abspath(sys.argv[1]))

from pdae_b200.utils.synth import fill_named_tensors_, synth_images  # noqa: E402

from diffusion.gaussian_diffusion import GaussianDiffusion  # noqa: E402  (original)
from metric.utils import calculate_mse, calculate_ssim  # noqa: E402
from model.representation_learning.decoder import CELEBA64Decoder  # noqa: E402
from model.representation_learning.encoder import CELEBA64Encoder  # noqa: E402

# the evaluation tests/test_gpu_dropin_script.py runs; change both together
CFG = {"diffusion_config": {"timesteps": 1000, "betas_type": "linear"}, "latent_dim": 512,
       "denoise_fn_config": dict(input_channel=3, base_channel=32, channel_multiplier=[1, 2, 2], num_residual_blocks_of_a_block=1,
                                 attention_resolutions=[2], num_heads=1, head_channel=-1, use_new_attention_order=False, dropout=0.0),
       "encoder_seed": 7, "decoder_seed": 6, "n_images": 3, "image_size": 64, "image_seed": 28, "batch_size": 2,
       "encoder_style": "ddim1000", "decoder_style": "ddim100"}


def main():
    torch.set_num_threads(8)
    enc = CELEBA64Encoder(latent_dim=CFG["latent_dim"])
    dec = CELEBA64Decoder(latent_dim=CFG["latent_dim"], **CFG["denoise_fn_config"])
    esd, dsd = enc.state_dict(), dec.state_dict()
    fill_named_tensors_(esd.items(), CFG["encoder_seed"])
    fill_named_tensors_(dsd.items(), CFG["decoder_seed"])
    enc.load_state_dict(esd)
    dec.load_state_dict(dsd)
    enc.eval().requires_grad_(False)
    dec.eval().requires_grad_(False)
    gd = GaussianDiffusion(CFG["diffusion_config"], device="cpu")
    x = synth_images(CFG["n_images"], 3, CFG["image_size"], CFG["image_seed"])
    recon, mse, ssim = [], [], []
    with torch.inference_mode():
        for x_0 in x.split(CFG["batch_size"]):
            r = gd.representation_learning_autoencoding(CFG["encoder_style"], CFG["decoder_style"], enc, dec, x_0)
            a, b = (x_0 + 1.) / 2., (r + 1.) / 2.
            recon.append(r)
            mse.append(calculate_mse(a, b))
            ssim.append(calculate_ssim(a, b))
    out = {"recon": torch.cat(recon), "mse": torch.cat(mse), "ssim": torch.cat(ssim)}
    out = {k: v.numpy().astype(np.float32) for k, v in out.items()}
    np.savez_compressed(os.path.join(HERE, "dropin_autoencoding_eval.npz"), cfg=np.array(json.dumps(CFG)), **out)
    print("wrote dropin_autoencoding_eval", {k: v.shape for k, v in out.items()}, "mse", out["mse"], "ssim", out["ssim"])


if __name__ == "__main__":
    main()
