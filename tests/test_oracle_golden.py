"""The CPU oracle (oracle/vx_oracle.py) against golden vectors produced by the reference's own code
(oracle/gen_golden.py).  No GPU."""
import json
import os

import numpy as np
import pytest
import torch

from oracle import vx_oracle as O


def test_context_windows_bit_exact(golden_dir):
    g = json.load(open(os.path.join(golden_dir, "context_windows.json")))
    for c in g["pipeline_calls"]:
        wins = O.context_windows(c["L"], c["S"], c["O"])
        assert wins == c["windows"], c
        assert O.num_frame_context(wins, c["L"]).tolist() == c["num_frame_context"], c
    for c in g["uniform_calls"]:
        wins = list(O.uniform(c["step"], c["L"], c["S"], c["stride"], c["O"], c["closed"]))
        assert wins == c["windows"], c
    for k, v in g["ordered_halving"].items():
        assert O.ordered_halving(int(k)) == v


def test_context_survey_table():
    # SURVEY.md Appendix D
    for (L, S, Ov, nwin, total) in [(4, 24, 4, 1, 4), (16, 16, 8, 1, 16), (96, 16, 8, 11, 176),
                                    (384, 16, 8, 47, 752), (924, 24, 4, 46, 1104), (20, 16, 4, 2, 32),
                                    (100, 16, 8, 12, 192)]:
        w = O.context_windows(L, S, Ov)
        assert len(w) == nwin and sum(len(x) for x in w) == total
        c = O.num_frame_context(w, L)
        assert c.min() == 1 and c.max() <= 2


def test_ddim_known_answers(golden_dir):
    g = json.load(open(os.path.join(golden_dir, "ddim_kat.json")))
    s = O.DDIM()
    # constants quoted in SURVEY.md Appendix B.5
    assert abs(float(s.alphas_cumprod[0]) - 0.99914998) < 1e-7
    assert abs(float(s.alphas_cumprod[499]) - 0.24235900) < 1e-7
    assert float(s.alphas_cumprod[999]) == 0.0
    for n, first, last in ((25, 999, 39), (50, 999, 19), (2, 999, 499)):
        s.set_timesteps(n)
        assert s.timesteps.tolist() == g[f"timesteps_{n}"]
        assert s.timesteps[0] == first and s.timesteps[-1] == last
    s.set_timesteps(25)
    x = torch.tensor([1.5409961, -0.2934289, -2.1787894, 0.5684313])
    v = torch.tensor([-1.0845224, -1.3985955, 0.4033468, 0.8380263])
    out = s.step(v, 999, x).prev_sample
    np.testing.assert_allclose(out.numpy(), [1.5617130, -0.2662846, -2.1861930, 0.5520930], atol=1e-6)


def test_param_layout_full_width():
    S = O.unet_param_shapes(O.DEFAULT_CFG)
    assert len(S) == 1386                                     # SURVEY Appendix C
    assert sum(int(np.prod(v)) for v in S.values()) == 1363537604
    mm = sum(int(np.prod(v)) for k, v in S.items() if "motion_modules" in k)
    assert abs(mm / 1e6 - 454.42) < 0.01
    assert S["up_blocks.1.resnets.2.conv1.weight"] == (1280, 1920, 3, 3)
    assert S["down_blocks.1.resnets.0.conv_shortcut.weight"] == (640, 320, 1, 1)


def test_unet_forward_matches_reference(golden_dir):
    g = torch.load(os.path.join(golden_dir, "unet_small.pt"), weights_only=False)
    cfg = g["cfg"]
    sd = O.synth_state_dict(O.unet_param_shapes(cfg), g["seed_weights"])
    lat, kps, audio, banks = O.synth_inputs(cfg, g["f"], g["h"], g["h"], True, g["seed_inputs"])
    assert g["bank_order"] == O.bank_order(cfg)
    x = lat.repeat(2, 1, 1, 1, 1)
    enc = audio.reshape(-1, 5, cfg["cross_attention_dim"])
    taps = {}
    with torch.no_grad():
        out = O.unet_forward(sd, cfg, x, 499, enc, kps, banks, g["ref_w"], g["audio_w"], taps=taps)
        out2 = O.unet_forward(sd, cfg, x, 959, enc, kps, banks, g["ref_w"], g["audio_w"])
    torch.testing.assert_close(out, g["out_t499"], atol=2e-4, rtol=1e-4)
    torch.testing.assert_close(out2, g["out_t959"], atol=2e-4, rtol=1e-4)
    s = g["sample_stride"]
    for k, v in g["taps"].items():
        assert tuple(taps[k].shape) == g["tap_shapes"][k], k
        torch.testing.assert_close(taps[k].flatten()[::s], v.float(), atol=2e-2, rtol=2e-3)   # taps stored in fp16


def test_pipeline_matches_reference(golden_dir):
    g = torch.load(os.path.join(golden_dir, "pipeline_small.pt"), weights_only=False)
    cfg, vcfg = g["cfg"], g["vae_cfg"]
    sd = O.synth_state_dict(O.unet_param_shapes(cfg), 1234)
    vsd = O.synth_state_dict(O.vae_param_shapes(vcfg), 1235)
    lat, kps, audio, banks = O.synth_inputs(cfg, g["L"], g["h"], g["h"], True, 42)
    with torch.no_grad():
        final = O.denoise(sd, cfg, lat, kps, audio, banks, g["steps"], g["guidance_scale"], g["S"], g["O"], 0.95, 3.0)
        torch.testing.assert_close(final, g["final_latents"], atol=5e-4, rtol=1e-4)
        video = O.decode_latents(vsd, vcfg, final)
    assert tuple(video.shape) == g["video_shape"] and video.dtype == torch.float32
    torch.testing.assert_close(video.flatten()[::g["sample_stride"]], g["video"].float(), atol=2e-3, rtol=0)


def test_pipeline_non_tiling_length_matches_reference(golden_dir):
    """video_length 20, windows of 16 with overlap 4: the reflected tail window repeats frames; the golden is the output
    of the reference's own pipeline code for that call (its index-put / streaming bookkeeping, SURVEY Appendix D)."""
    g = torch.load(os.path.join(golden_dir, "pipeline_nontiling_small.pt"), weights_only=False)
    cfg = g["cfg"]
    sd = O.synth_state_dict(O.unet_param_shapes(cfg), 1234)
    lat, kps, audio, banks = O.synth_inputs(cfg, g["L"], g["h"], g["h"], True, 42)
    wins = O.context_windows(g["L"], g["S"], g["O"])
    assert any(len(set(w)) != len(w) for w in wins)
    with torch.no_grad():
        final = O.denoise(sd, cfg, lat, kps, audio, banks, g["steps"], g["guidance_scale"], g["S"], g["O"], 0.95, 3.0)
    torch.testing.assert_close(final, g["final_latents"], atol=5e-4, rtol=1e-4)


def test_refnet_param_layout_full_width():
    S = O.refnet_param_shapes(O.DEFAULT_CFG)          # SD-1.5 UNet2D minus the conv_norm_out the reference drops
    assert len(S) == 684
    assert sum(int(np.prod(v)) for v in S.values()) == 859520964 - 640
    assert "conv_norm_out.weight" not in S           # modules/unet_2d_condition.py:650
    assert S["up_blocks.1.resnets.2.conv1.weight"] == (1280, 1920, 3, 3)
    assert S["down_blocks.0.attentions.0.transformer_blocks.0.attn2.to_k.weight"] == (320, 768)


def test_refnet_write_pass_matches_reference(golden_dir):
    """SURVEY 8(f) row f1: the 16 banks the hot path consumes, produced by the reference's own UNet2D + write hooks
    + ``update`` (oracle/gen_golden.py:gen_refnet), against the restated write pass."""
    g = torch.load(os.path.join(golden_dir, "refnet_small.pt"), weights_only=False)
    cfg = g["cfg"]
    sd = O.synth_state_dict(O.refnet_param_shapes(cfg), g["seed_weights"])
    x = torch.randn(1, 4, g["h"], g["h"], generator=torch.Generator().manual_seed(g["seed_latents"]))
    assert g["bank_order"] == O.bank_order(cfg)
    with torch.no_grad():
        banks, out = O.refnet_forward(sd, cfg, x)
    assert len(banks) == len(g["banks"]) == 16
    for name, a, b in zip(g["bank_order"], banks, g["banks"]):
        assert a.shape == b.shape, name
        torch.testing.assert_close(a, b, atol=2e-4, rtol=1e-4, msg=lambda m: f"{name}: {m}")
    torch.testing.assert_close(out, g["out"], atol=2e-4, rtol=1e-4)


def test_prologue_and_postprocessing_match_reference(golden_dir):
    """SURVEY 8(f) rows f2 / f3: VKpsGuider, AudioProjection, the audio windowing of prepare_audio_embeddings and the
    3x3x3 median filter, against outputs of the reference's own code (oracle/gen_golden.py:gen_prologue)."""
    g = torch.load(os.path.join(golden_dir, "prologue_small.pt"), weights_only=False)
    k = g["kps"]
    sd = O.synth_state_dict(O.kps_guider_param_shapes(O.KPS_CFG), k["seed_weights"])
    x = torch.rand(*k["shape"], generator=torch.Generator().manual_seed(k["seed_input"]))
    with torch.no_grad():
        torch.testing.assert_close(O.kps_guider_forward(sd, O.KPS_CFG, x), k["feature"], atol=1e-5, rtol=1e-5)
    a = g["audio_projection"]
    sd = O.synth_state_dict(O.audio_projection_param_shapes(O.AUDIO_PROJ_CFG), a["seed_weights"])
    x = torch.randn(*a["shape"], generator=torch.Generator().manual_seed(a["seed_input"]))
    with torch.no_grad():
        torch.testing.assert_close(O.audio_projection_forward(sd, O.AUDIO_PROJ_CFG, x), a["tokens"], atol=1e-5, rtol=1e-5)
    w = g["audio_windows"]
    emb = torch.randn(*w["shape"], generator=torch.Generator().manual_seed(w["seed_input"]))
    assert torch.equal(O.audio_frame_windows(emb, w["video_length"], w["num_pad"]), w["windows"])
    m = g["median"]
    v = torch.rand(*m["shape"], generator=torch.Generator().manual_seed(m["seed_input"]))
    filt = O.median_filter_3d(v, 3)
    assert torch.equal(filt, m["filtered"])                         # order statistics: bit-exact
    assert np.array_equal(O.video_to_uint8(filt), m["uint8"].numpy())


# ---- independent pins of the DDIM scheduler and the VAE decoder (neither is reference code: diffusers 0.29.2) ---------
def _shim():
    import sys
    p = os.path.join(os.path.dirname(os.path.abspath(O.__file__)), "diffusers_shim")
    if p not in sys.path:
        sys.path.insert(0, p)
    import diffusers
    return diffusers


def _abar_float64():
    """inference_v2.yaml:23-33 in closed form, float64: scaled-linear betas, then the zero-terminal-SNR rescale
    sqrt(abar)_t -> (sqrt(abar)_t - sqrt(abar)_T) * sqrt(abar)_0 / (sqrt(abar)_0 - sqrt(abar)_T)."""
    i = np.arange(1000, dtype=np.float64)
    betas = (np.sqrt(0.00085) + i * (np.sqrt(0.012) - np.sqrt(0.00085)) / 999.0) ** 2
    root = np.sqrt(np.cumprod(1.0 - betas))
    root = (root - root[-1]) * root[0] / (root[0] - root[-1])
    return root ** 2


def test_ddim_against_float64_closed_form_and_independent_restatement():
    abar = _abar_float64()
    assert abar[999] == 0.0
    s = O.DDIM()
    got = s.alphas_cumprod.double().numpy()
    # fp32 tables (linspace, two cumprods over 1000 factors) vs float64: a few fp32 ulps
    np.testing.assert_allclose(got, abar, atol=1e-6, rtol=0)
    for t in (0, 1, 499, 959):
        assert abs(got[t] / abar[t] - 1) < 2e-5, t
    # trailing spacing: round(1000 - k * 1000 / n) - 1
    for n in (2, 25, 50):
        s.set_timesteps(n)
        want = [int(np.round(1000 - k * 1000.0 / n)) - 1 for k in range(n)]
        assert s.timesteps.tolist() == want
    # one v-prediction step (eta = 0) by hand in float64: x0 = sqrt(a) x - sqrt(1-a) v, eps = sqrt(a) v + sqrt(1-a) x,
    # x' = sqrt(a') x0 + sqrt(1-a') eps; t = 959 -> prev = 919 (n = 25); and the last step t = 39 -> prev < 0 -> a' = 1
    s.set_timesteps(25)
    g = torch.Generator().manual_seed(3)
    x, v = torch.randn(64, generator=g), torch.randn(64, generator=g)
    for t, tp in ((959, 919), (39, None), (999, 959)):
        a, ap = abar[t], (abar[tp] if tp is not None else 1.0)
        x64, v64 = x.double().numpy(), v.double().numpy()
        x0 = np.sqrt(a) * x64 - np.sqrt(1 - a) * v64
        eps = np.sqrt(a) * v64 + np.sqrt(1 - a) * x64
        want = np.sqrt(ap) * x0 + np.sqrt(1 - ap) * eps
        np.testing.assert_allclose(s.step(v, t, x).prev_sample.double().numpy(), want, atol=3e-6)
    # the product's host-side table (what vx_ddim_step is fed with)
    from vexpress_b200.pipelines.scheduler import DDIMScheduler as Prod, ddim_coefficients
    p = Prod()
    p.set_timesteps(25)
    sa, sb, sap, sbp = ddim_coefficients(p, 959)
    np.testing.assert_allclose([sa, sb, sap, sbp], [np.sqrt(abar[959]), np.sqrt(1 - abar[959]), np.sqrt(abar[919]),
                                                    np.sqrt(1 - abar[919])], rtol=2e-5)
    # second, separately written implementation in the library's own structure (oracle/diffusers_shim)
    lib = _shim().DDIMScheduler(beta_start=0.00085, beta_end=0.012, beta_schedule="scaled_linear", clip_sample=False,
                                steps_offset=1, prediction_type="v_prediction", rescale_betas_zero_snr=True,
                                timestep_spacing="trailing")
    assert lib.__class__.__module__.startswith("diffusers") and not isinstance(lib, O.DDIM)
    np.testing.assert_allclose(lib.alphas_cumprod.double().numpy(), abar, atol=1e-6, rtol=0)
    for n in (2, 25, 50):
        lib.set_timesteps(n)
        s.set_timesteps(n)
        assert lib.timesteps.tolist() == s.timesteps.tolist()
        for t in lib.timesteps.tolist():
            np.testing.assert_allclose(lib.step(v, t, x).prev_sample.numpy(), s.step(v, t, x).prev_sample.numpy(), atol=1e-6)


def test_vae_decoder_against_independent_module_restatement():
    """The oracle's functional decoder vs an nn.Module AutoencoderKL assembled in diffusers' structure from separately
    written leaves (oracle/diffusers_shim/diffusers/autoencoder.py); the module tree also pins the state_dict layout."""
    d = _shim()
    vcfg = O.small_vae_cfg()
    vsd = O.synth_state_dict(O.vae_param_shapes(vcfg), 1235)
    vae = d.AutoencoderKL(vsd, vcfg)                       # strict load: key names + shapes of the diffusers layout
    assert "vx_oracle" not in open(d.autoencoder.__file__).read().split('"""', 2)[2]
    z = torch.randn(2, 4, 16, 16, generator=torch.Generator().manual_seed(8))
    with torch.no_grad():
        a = vae.decode(z).sample
        b = O.vae_decode(vsd, vcfg, z)
    assert a.shape == (2, 3, 128, 128)
    np.testing.assert_allclose(a.numpy(), b.numpy(), atol=2e-5, rtol=1e-5)


def test_vae_encoder_against_independent_module_restatement():
    """SURVEY 8(f) row f4: the oracle's functional VAE encoder (posterior mean) vs the library-structured nn.Module in the
    shim; the strict load pins the encoder's state_dict layout, which the product mirrors (vexpress_b200 AutoencoderKL)."""
    d = _shim()
    vcfg = O.small_vae_cfg()
    vsd = O.synth_state_dict({**O.vae_param_shapes(vcfg), **O.vae_encoder_param_shapes(vcfg)}, 1236)
    vae = d.AutoencoderKL(vsd, vcfg)
    x = torch.rand(2, 3, 64, 48, generator=torch.Generator().manual_seed(9)) * 2 - 1
    with torch.no_grad():
        a = vae.encode(x).latent_dist.mean
        b = O.vae_encode_mean(vsd, vcfg, x)
    assert a.shape == (2, 4, 8, 6)
    np.testing.assert_allclose(a.numpy(), b.numpy(), atol=2e-5, rtol=1e-5)
    from vexpress_b200.modules.vae import AutoencoderKL as Prod
    p = Prod(block_out_channels=vcfg["block_out_channels"], layers_per_block=vcfg["layers_per_block"])
    p.load_state_dict(vsd, strict=True)
    assert set(p.state_dict()) == set(vsd)
    p2 = Prod(block_out_channels=vcfg["block_out_channels"], layers_per_block=vcfg["layers_per_block"])
    p2.load_state_dict(O.synth_state_dict(O.vae_param_shapes(vcfg), 1235), strict=True)      # decoder-only checkpoint
    assert set(p2.state_dict()) == set(O.vae_param_shapes(vcfg))
    with pytest.raises(RuntimeError):
        p2.encode(x)
