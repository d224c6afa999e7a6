"""Drop-in: the evaluation of the original project's sampler/autoencoding_eval.py, run through the original's import names
after `pdae_b200.dropin.install()` (modules looked up by config name with getattr, a checkpoint with the original's keys,
copy.deepcopy(...).cuda(), GaussianDiffusion.representation_learning_autoencoding('ddim1000', 'ddim100', ...) over a
DataLoader, per-image MSE / SSIM on [0,1]-scaled images), executes on the pdae_b200 kernels and reproduces what the
original computes for the same synthetic checkpoint and images (tests/golden/dropin_autoencoding_eval.npz, recorded from
the original's own modules on the CPU in fp32 by tests/golden/make_dropin_golden.py).

The evaluation runs in a subprocess because install() registers this package under the top-level names `model` and
`diffusion` for the rest of the process."""
import json
import os
import subprocess
import sys
import textwrap

import numpy as np
import pytest

from tests.util import load_golden

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GATE = 1e-5        # |recon-MSE - original's recon-MSE| on [0,1]-scaled images, the acceptance bound bench.py applies

SCRIPT = r'''
import copy, json, os, sys
import numpy as np
import torch
ROOT, TMP = sys.argv[1], sys.argv[2]
sys.path.insert(0, ROOT)
cfg = json.loads(sys.argv[3])
import pdae_b200.dropin
pdae_b200.dropin.install()
pdae_b200.set_default_precision("fp32")
from pdae_b200.metric.utils import calculate_mse, calculate_ssim
from pdae_b200.utils.synth import fill_named_tensors_, synth_images
# ---- what the original's autoencoding_eval.py does, under the original's import names ----
import model.representation_learning.encoder as encoder_module
import model.representation_learning.decoder as decoder_module
from diffusion.gaussian_diffusion import GaussianDiffusion
assert encoder_module.__name__.startswith("pdae_b200") and decoder_module.__name__.startswith("pdae_b200")
assert GaussianDiffusion.__module__.startswith("pdae_b200")
enc = getattr(encoder_module, "CELEBA64Encoder")(latent_dim=cfg["latent_dim"])
dec = getattr(decoder_module, "CELEBA64Decoder")(latent_dim=cfg["latent_dim"], **cfg["denoise_fn_config"])
esd, dsd = enc.state_dict(), dec.state_dict()
fill_named_tensors_(esd.items(), cfg["encoder_seed"])
fill_named_tensors_(dsd.items(), cfg["decoder_seed"])
torch.save({"ema_encoder": esd, "ema_decoder": dsd}, os.path.join(TMP, "checkpoint.pt"))
gd = GaussianDiffusion(cfg["diffusion_config"], device=torch.device("cuda"))
encoder, decoder = copy.deepcopy(enc).cuda(), copy.deepcopy(dec).cuda()
checkpoint = torch.load(os.path.join(TMP, "checkpoint.pt"), map_location=torch.device("cpu"))
encoder.load_state_dict(checkpoint["ema_encoder"])
decoder.load_state_dict(checkpoint["ema_decoder"])
encoder.eval()
encoder.requires_grad_(False)
decoder.eval()
decoder.requires_grad_(False)
images = synth_images(cfg["n_images"], 3, cfg["image_size"], cfg["image_seed"])
loader = torch.utils.data.DataLoader(images, batch_size=cfg["batch_size"], shuffle=False, drop_last=False)
recon, mse, ssim = [], [], []
with torch.inference_mode():
    for x_0 in loader:
        x_0 = x_0.cuda()
        rec = gd.representation_learning_autoencoding(cfg["encoder_style"], cfg["decoder_style"], encoder, decoder, x_0)
        a, b = (x_0 + 1.) / 2., (rec + 1.) / 2.
        recon.append(rec.cpu())
        mse += calculate_mse(a, b).tolist()
        ssim += calculate_ssim(a, b).tolist()
np.save(os.path.join(TMP, "recon.npy"), torch.cat(recon).numpy())
print("RESULT " + json.dumps({"mse": mse, "ssim": ssim, "encoder": type(encoder).__module__, "decoder": type(decoder).__module__}))
'''


def test_autoencoding_eval_on_native_kernels_matches_reference(tmp_path):
    cfg, g = load_golden("dropin_autoencoding_eval")
    script = tmp_path / "autoencoding_eval.py"
    script.write_text(textwrap.dedent(SCRIPT))
    r = subprocess.run([sys.executable, str(script), ROOT, str(tmp_path), json.dumps(cfg)], capture_output=True, text=True,
                       timeout=900)
    assert r.returncode == 0, r.stdout[-3000:] + "\n" + r.stderr[-3000:]
    line = [l for l in r.stdout.splitlines() if l.startswith("RESULT ")][-1]
    res = json.loads(line[len("RESULT "):])
    assert res["encoder"].startswith("pdae_b200") and res["decoder"].startswith("pdae_b200"), res
    mse, ssim, want_mse, want_ssim = np.array(res["mse"]), np.array(res["ssim"]), g["mse"].double().numpy(), g["ssim"].double().numpy()
    rec, want = np.load(tmp_path / "recon.npy").astype(np.float64), g["recon"].double().numpy()
    rel = [float(np.linalg.norm(a - b) / np.linalg.norm(b)) for a, b in zip(rec, want)]
    print(f"per-image |dMSE| {np.abs(mse - want_mse).tolist()}, |dSSIM| {np.abs(ssim - want_ssim).tolist()}, recon rel-L2 {rel}")
    assert rec.shape == want.shape and mse.shape == ssim.shape == want_mse.shape      # 3 images in batches of 2 + 1
    assert np.all(np.abs(mse - want_mse) <= GATE), (mse, want_mse)
    assert np.all(np.abs(ssim - want_ssim) <= 1e-4), (ssim, want_ssim)
    assert max(rel) <= 1e-3, rel
