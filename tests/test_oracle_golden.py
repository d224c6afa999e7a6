"""Pin the CPU oracle (oracle/pdae_oracle.py) against the fixtures recorded from the REAL reference
(tests/golden/make_golden.py).  CPU only; this is what makes the oracle trustworthy on the GPU box, where
/root/reference does not exist."""
import numpy as np
import pytest
import torch

from oracle import pdae_oracle as O
from tests import cases
from tests.util import assert_close, golden_names, load_golden

TOL = dict(rtol=1e-4, atol=1e-5)


@pytest.fixture(autouse=True)
def _recording_threads():
    """The fixtures were recorded with 8 intra-op threads (make_golden.py).  torch's CPU kernels split their reductions by
    the thread count, and the chained random-weight loops amplify the resulting last-bit differences (test_loop_sensitivity)
    beyond the tolerances below, so the oracle runs with the same count on every host."""
    n = torch.get_num_threads()
    torch.set_num_threads(8)
    yield
    torch.set_num_threads(n)


@pytest.mark.parametrize("name", golden_names("block_"))
def test_blocks(name):
    cfg, g = load_golden(name)
    m, inp = cases.block_case(cfg)
    sd = {"blk." + k: v for k, v in cases.sd_of(m).items()}
    if cfg["kind"] == "resblock":
        y = O.resblock(sd, "blk", inp["x"], inp["emb"], inp.get("emb_z"), up=cfg.get("up", False), down=cfg.get("down", False))
    else:
        y = O.attention_block(sd, "blk", inp["x"], cfg["heads"], cfg["new_order"])
    assert_close(y, g["y"], what=name, **TOL)


def test_timestep_embedding():
    _, g = load_golden("timestep_embedding")
    assert_close(O.timestep_embedding(g["t"], 64), g["e64"], rtol=0, atol=0, what="e64")
    assert_close(O.timestep_embedding(g["t"], 33), g["e33"], rtol=0, atol=0, what="e33")


@pytest.mark.parametrize("name", golden_names("model_"))
def test_models(name):
    cfg, g = load_golden(name)
    m, inp = cases.model_case(cfg)
    sd = cases.sd_of(m)
    if cfg["kind"] == "unet":
        assert_close(O.unet_forward(sd, cfg["cfg"], inp["x"], g["t"], g.get("cond")), g["y"], what=name, **TOL)
    elif cfg["kind"] == "shiftunet":
        eps, grad = O.shiftunet_forward(sd, cfg["cfg"], inp["x"], g["t"], inp["z"])
        assert_close(eps, g["eps"], what=name + ".eps", **TOL)
        assert_close(grad, g["grad"], what=name + ".grad", **TOL)
    elif cfg["kind"] == "encoder":
        assert_close(O.encoder_forward(sd, "celeba64" if cfg["size"] == 64 else "ffhq128", inp["x"]), g["z"], what=name, **TOL)
    else:
        assert_close(O.mlp_skip_net_forward(sd, cfg["cfg"], inp["x"], g["t"]), g["y"], what=name, **TOL)


@pytest.mark.parametrize("bt", ["linear", "cosine"])
def test_schedule_tables(bt):
    _, g = load_golden("diffusion_tables_" + bt)
    tabs = O.gaussian_tables({"timesteps": 1000, "betas_type": bt})
    for k, v in g.items():
        assert torch.equal(tabs[k], v), k


def test_ddim_maps_and_tables():
    _, g = load_golden("diffusion_ddim_maps")
    ac = O.gaussian_tables(cases.DIFF)["alphas_cumprod"].numpy()
    for style, n in (("ddim10", 11), ("ddim100", 101), ("ddim200", 201), ("ddim500", 501), ("ddim1000", 1000)):
        nb, tmap = O.ddim_betas_and_timestep_map(style, ac)
        assert tmap.shape[0] == n
        assert torch.equal(tmap, g[style + "_map"])
        np.testing.assert_array_equal(nb, g[style + "_betas"].numpy())
        if style in ("ddim10", "ddim100"):
            for k, v in O.ddim_tables(nb).items():
                assert torch.equal(v, g[f"{style}_{k}"]), (style, k)


def test_elementwise_steps():
    from pdae_b200.utils.synth import synth_images, synth_normal
    _, g = load_golden("diffusion_steps")
    D = O.DiffusionOracle(cases.DIFF)
    x0, noise, eps = synth_images(4, 3, 8, 21), synth_normal((4, 3, 8, 8), 22), synth_normal((4, 3, 8, 8), 23)
    lr = synth_normal((4, 3, 8, 8), 24).clamp(-1, 1)
    assert_close(D.q_sample(x0, g["t"], noise), g["q"], rtol=0, atol=0, what="q_sample")
    assert_close(D.noise_p_sample(x0, g["t"], eps, g["p_noise"]), g["p_sample"], rtol=1e-6, atol=1e-6, what="p_sample")
    assert_close(D.noise_p_sample(x0, g["t"], eps, g["p_noise"], lr), g["p_sample_lr"], rtol=1e-6, atol=1e-6, what="p_lr")


def test_loops():
    from pdae_b200.utils.synth import synth_images, synth_normal
    D = O.DiffusionOracle(cases.DIFF)
    cfg, g = load_golden("loop_unet_ddim10")
    m, _ = cases.model_case({"kind": "unet", "cfg": cfg["cfg"], "size": 16})
    sd = cases.sd_of(m)
    fn = lambda x, t, c: O.unet_forward(sd, cfg["cfg"], x, t, c)
    xT, x0 = synth_normal((2, 3, 16, 16), 25), synth_images(2, 3, 16, 26)
    assert_close(D.ddim_sample("ddim10", fn, xT), g["sample"], what="unet sample", **TOL)
    assert_close(D.ddim_encode("ddim10", fn, x0), g["encode"], what="unet encode", **TOL)

    cfg, g = load_golden("loop_shift_ddim10")
    m, _ = cases.model_case({"kind": "shiftunet", "cfg": cfg["cfg"], "size": 16})
    sd = cases.sd_of(m)
    dec = lambda x, t, z: O.shiftunet_forward(sd, cfg["cfg"], x, t, z)
    z = synth_normal((2, 64), 27)
    assert_close(D.representation_learning_ddim_sample("ddim10", dec, xT, z), g["sample"], what="shift sample", **TOL)
    assert_close(D.representation_learning_ddim_sample("ddim10", dec, xT, z, 0.3), g["sample_stop30"], what="stop30", **TOL)
    assert_close(D.representation_learning_ddim_encode("ddim10", dec, x0, z), g["encode"], what="shift encode", **TOL)


def test_autoencoding_and_latent_loop():
    from pdae_b200.utils.synth import synth_images, synth_normal
    D = O.DiffusionOracle(cases.DIFF)
    cfg, g = load_golden("loop_autoencode_ddim10")
    dec_m, _ = cases.model_case({"kind": "shiftunet", "cfg": cfg["cfg"], "size": 64})
    enc_m, _ = cases.model_case({"kind": "encoder", "size": 64})
    dsd, esd = cases.sd_of(dec_m), cases.sd_of(enc_m)
    rec = D.representation_learning_autoencoding(
        "ddim10", "ddim10", lambda x: O.encoder_forward(esd, "celeba64", x),
        lambda x, t, z: O.shiftunet_forward(dsd, cfg["cfg"], x, t, z), synth_images(2, 3, 64, 28))
    assert_close(rec, g["recon"], what="autoencode", rtol=1e-3, atol=1e-4)

    cfg, g = load_golden("loop_latent_ddim10")
    m, _ = cases.model_case({"kind": "mlp", "cfg": cfg["cfg"]})
    sd = cases.sd_of(m)
    zT = synth_normal((2, 64), 29).clamp(-1, 1)
    out = D.latent_ddim_sample("ddim10", lambda z, t: O.mlp_skip_net_forward(sd, cfg["cfg"], z, t), zT)
    assert_close(out, g["z"], what="latent loop", **TOL)


def test_training_losses():
    from pdae_b200.utils.synth import synth_images
    D = O.DiffusionOracle(cases.DIFF)
    cfg, g = load_golden("train_representation_learning")
    dec_m, _ = cases.model_case({"kind": "shiftunet", "cfg": cfg["cfg"], "size": 64})
    enc_m, _ = cases.model_case({"kind": "encoder", "size": 64})
    dsd = {k: v.requires_grad_(k.startswith(("label_emb", "shift_"))) for k, v in cases.sd_of(dec_m).items()}
    esd = {k: v.requires_grad_(True) for k, v in cases.sd_of(enc_m).items()}
    loss = D.representation_learning_loss(lambda x: O.encoder_forward(esd, "celeba64", x),
                                          lambda x, t, z: O.shiftunet_forward(dsd, cfg["cfg"], x, t, z),
                                          synth_images(2, 3, 64, 31), g["t"], g["noise"])
    assert_close(loss, g["loss"], what="rl loss", rtol=1e-5, atol=1e-7)
    loss.backward()
    n_grad = sum(1 for v in list(dsd.values()) + list(esd.values()) if v.grad is not None)
    assert n_grad == cfg["n_params_with_grad"]
    for key, ref in (("label_emb.weight", "g_label_emb_weight"), ("shift_out.2.weight", "g_shift_out_2_weight")):
        assert_close(dsd[key].grad.flatten()[:512], g[ref], what=key, rtol=1e-3, atol=1e-7)
        assert_close(dsd[key].grad.double().norm().float(), g["n" + ref], what=key + " norm", rtol=1e-4, atol=0)
    assert_close(esd["encoder.0.weight"].grad.flatten()[:512], g["g_enc_encoder_0_weight"], what="enc grad", rtol=1e-3, atol=1e-7)

    cfg, g = load_golden("train_regular")
    m, _ = cases.model_case({"kind": "unet", "cfg": cfg["cfg"], "size": 16})
    sd = cases.sd_of(m)
    loss = D.regular_loss(lambda x, t, c: O.unet_forward(sd, cfg["cfg"], x, t, c), synth_images(2, 3, 16, 32), g["t"], g["noise"])
    assert_close(loss, g["loss"], what="regular loss", rtol=1e-5, atol=1e-7)


def test_latent_training_loss_and_grads():
    """latent_diffusion_train_one_batch (gaussian_diffusion.py:373-398): oracle loss + autograd grads vs the reference."""
    from pdae_b200.model.mlp_skip_net import MLPSkipNet
    from pdae_b200.utils.synth import fill_module_
    cfg, g = load_golden("train_latent")
    sd = {k: v.requires_grad_(True) for k, v in cases.sd_of(fill_module_(MLPSkipNet(**cfg["cfg"]), seed=9)).items()
          if not k.startswith("layers.") or ".cond_layers." not in k}
    D = O.DiffusionOracle(cases.DIFF)
    loss = D.latent_diffusion_loss(lambda z, t: O.mlp_skip_net_forward(sd, cfg["cfg"], z, t), g["z0"], g["t"], g["noise"])
    assert_close(loss, g["loss"], what="latent loss", rtol=1e-5, atol=1e-7)
    loss.backward()
    assert sum(1 for v in sd.values() if v.grad is not None) == cfg["n_params_with_grad"]
    for k in ("time_embed.0.weight", "time_embed.2.bias", "layers.0.linear.weight", "layers.1.linear_emb.weight",
              "layers.2.norm.weight", "layers.3.norm.bias", "layers.4.linear.weight", "layers.4.linear.bias"):
        kk = k.replace(".", "_")
        assert_close(sd[k].grad.flatten()[:512], g["g_" + kk], what=k, rtol=1e-3, atol=1e-8)
        assert_close(sd[k].grad.double().norm().float(), g["n_" + kk], what=k + " norm", rtol=1e-4, atol=0)


def test_loop_sensitivity():
    """How much a 10-step shift-DDIM loop on random weights amplifies an input perturbation (justifies the stated
    bf16 loop tolerance in tests/test_gpu_diffusion.py): 1e-5 in -> between 1e-5 and 1e-2 out, no sign flips."""
    from pdae_b200.utils.synth import synth_normal
    D = O.DiffusionOracle(cases.DIFF)
    cfg, g = load_golden("loop_shift_ddim10")
    m, _ = cases.model_case({"kind": "shiftunet", "cfg": cfg["cfg"], "size": 16})
    sd = cases.sd_of(m)
    dec = lambda x, t, z: O.shiftunet_forward(sd, cfg["cfg"], x, t, z)
    z, xT = synth_normal((2, 64), 27), synth_normal((2, 3, 16, 16), 25)
    a = g["sample"]   # unperturbed result (== test_loops)
    with torch.no_grad():
        b = D.representation_learning_ddim_sample("ddim10", dec, xT + 1e-5 * synth_normal((2, 3, 16, 16), 99), z)
    amp = float((a - b).abs().max()) / 1e-5
    assert 1.0 < amp < 1e3, amp


def test_caller_metrics_and_wire_formats():
    cfg, g = load_golden("caller_metrics_io")
    a, b = cases.caller_io_inputs(cfg)
    assert_close(O.calculate_mse(a, b), g["mse"], rtol=1e-6, atol=0, what="mse")
    assert_close(O.calculate_ssim(a, b), g["ssim"], rtol=1e-6, atol=1e-7, what="ssim")
    u8 = O.images_to_uint8_nhwc(b * 1.3)
    assert u8.dtype == torch.uint8 and torch.equal(u8, g["u8"])
    assert torch.equal(O.uint8_nhwc_to_images(g["u8"]), g["back"])


@pytest.mark.parametrize("name", ["caller_adam_ema", "caller_adam_wd"])
def test_caller_adam_ema(name):
    cfg, g = load_golden(name)
    params, grads = cases.adam_case(cfg)
    ema = [p.clone() for p in params] if cfg["ema_decay"] >= 0 else None
    O.adam_ema_steps(params, grads, cfg["lr"], tuple(cfg["betas"]), cfg["eps"], cfg["weight_decay"], ema, cfg["ema_decay"])
    for i, p in enumerate(params):
        assert_close(p, g[f"p{i}"], rtol=1e-6, atol=1e-8, what=f"p{i}")
        if ema is not None:
            assert_close(ema[i], g[f"e{i}"], rtol=1e-6, atol=1e-8, what=f"e{i}")


# ---- glue rows a20 / a22 / a24 -----------------------------------------------------------------------------------------
def _shift16(cfg):
    m, _ = cases.model_case({"kind": "shiftunet", "cfg": cfg, "size": 16})
    sd = cases.sd_of(m)
    return lambda x, t, z: O.shiftunet_forward(sd, cfg, x, t, z)


def _unet16(cfg):
    m, _ = cases.model_case({"kind": "unet", "cfg": cfg, "size": 16})
    sd = cases.sd_of(m)
    return lambda x, t, c: O.unet_forward(sd, cfg, x, t, c)


def _autoenc64(cfg):
    dec_m, _ = cases.model_case({"kind": "shiftunet", "cfg": cfg, "size": 64})
    enc_m, _ = cases.model_case({"kind": "encoder", "size": 64})
    dsd, esd = cases.sd_of(dec_m), cases.sd_of(enc_m)
    return (lambda x: O.encoder_forward(esd, "celeba64", x)), (lambda x, t, z: O.shiftunet_forward(dsd, cfg, x, t, z))


def test_glue_interpolation_and_x0_clip():
    i = cases.glue_inputs()
    D = O.DiffusionOracle(cases.DIFF)
    cfg, g = load_golden("glue_interpolation")
    y = D.trajectory_interpolation(cfg["style"], _shift16(cfg["cfg"]), i["z1"], i["z2"], i["xT"], cfg["alpha"])
    assert_close(y, g["y"], what="trajectory interpolation", **TOL)
    cfg, g = load_golden("glue_x0_clip")
    for name, kw in (("fixed_clip", {}), ("fixed_noclip", dict(clip_x_0=False)), ("learned_clip", dict(learned_range=i["lr"]))):
        noise = cases.CpuStream(cfg["seed"]).randn(i["x_t"].shape)
        assert_close(D.x_0_clip_p_sample(i["x_t"], g["t"], i["eps"], noise, **kw), g[name], rtol=1e-6, atol=1e-6, what=name)


def test_glue_ddpm_loops():
    i = cases.glue_inputs()
    cfg, g = load_golden("glue_ddpm")
    D = O.DiffusionOracle({"timesteps": cfg["timesteps"], "betas_type": "linear"})
    s = cfg["seeds"]
    assert_close(D.ddpm_sample(_unet16(cfg["cfg_unet"]), i["xT"], cases.CpuStream(s[0]).randn), g["regular"], what="regular", **TOL)
    assert_close(D.ddpm_sample(_unet16(cfg["cfg_sigma"]), i["xT"], cases.CpuStream(s[1]).randn), g["learned_sigma"],
                 what="learned sigma", **TOL)
    assert_close(D.ddpm_sample(_shift16(cfg["cfg_shift"]), i["xT"], cases.CpuStream(s[2]).randn, z=i["z1"]), g["representation"],
                 what="representation", **TOL)


def test_glue_latent_sample_manipulation_gap_denoise():
    i = cases.glue_inputs()
    D = O.DiffusionOracle(cases.DIFF)
    cfg, g = load_golden("glue_latent_sample")
    m, _ = cases.model_case({"kind": "mlp", "cfg": cfg["cfg_mlp"]})
    sd = cases.sd_of(m)
    zT = cases.CpuStream(cfg["seed"]).randn((2, 64))
    y = D.latent_diffusion_sample("ddim10", "ddim10", lambda z, t: O.mlp_skip_net_forward(sd, cfg["cfg_mlp"], z, t),
                                  _shift16(cfg["cfg_shift"]), i["xT"], zT, i["mean64"], i["std64"])
    assert_close(y, g["y"], what="latent_diffusion_sample", **TOL)
    cfg, g = load_golden("glue_manipulation")
    enc, dec = _autoenc64(cfg["cfg"])
    y = D.manipulation_sample(cfg["style"], i["cw"], enc, dec, i["x0"], i["xT64"], i["mean512"], i["std512"], cfg["class_id"],
                              cfg["scale"])
    assert_close(y, g["y"], what="manipulation_sample", rtol=1e-3, atol=1e-4)
    cfg, g = load_golden("glue_gap")
    D8 = O.DiffusionOracle({"timesteps": cfg["timesteps"], "betas_type": "linear"})
    gp, ga = D8.gap_measure(enc, dec, i["x0"], cases.CpuStream(cfg["seed"]).rand_like)
    np.testing.assert_allclose(gp, g["gap_pred"].numpy(), rtol=1e-4)
    np.testing.assert_allclose(ga, g["gap_ae"].numpy(), rtol=1e-4)
    cfg, g = load_golden("glue_denoise_one_step")
    p0, a0 = D.denoise_one_step(enc, dec, i["x0"], cfg["timesteps"], cases.CpuStream(cfg["seed"]).randn_like(i["x0"]))
    assert_close(p0, g["pred"], what="denoise pred", **TOL)
    assert_close(a0, g["ae"], what="denoise ae", rtol=1e-4, atol=1e-4)


def test_product_ddim_respacing_matches_reference_for_every_style():
    """Row a16 on the PRODUCT function (host-side, no GPU needed): ddim10/100/200/500/1000 -> 11/101/201/501/1000 entries."""
    from pdae_b200.diffusion.gaussian_diffusion import GaussianDiffusion
    _, g = load_golden("diffusion_ddim_maps")
    ac = O.gaussian_tables(cases.DIFF)["alphas_cumprod"].numpy()
    for style, n in (("ddim10", 11), ("ddim100", 101), ("ddim200", 201), ("ddim500", 501), ("ddim1000", 1000)):
        nb, tmap = GaussianDiffusion.get_ddim_betas_and_timestep_map(style, ac)
        assert tmap.shape[0] == n and tmap.dtype == torch.long
        assert torch.equal(tmap, g[style + "_map"]), style
        np.testing.assert_array_equal(nb, g[style + "_betas"].numpy())
