"""VAE decoder and the whole denoise+decode pipeline on the B200 kernels vs oracle / reference golden (GPU)."""
import os

import pytest
import torch

from test_unet_gpu import UNET_EXTRA, _Writer, _rel

pytestmark = pytest.mark.gpu


def build_vae(vcfg, vsd):
    from vexpress_b200.modules.vae import AutoencoderKL
    vae = AutoencoderKL(block_out_channels=vcfg["block_out_channels"], layers_per_block=vcfg["layers_per_block"])
    vae.load_state_dict(vsd, strict=True)
    return vae.to(dtype=torch.bfloat16, device="cuda")


def test_vae_decode_vs_oracle():
    from oracle import vx_oracle as O
    vcfg = O.small_vae_cfg()
    vsd = O.synth_state_dict(O.vae_param_shapes(vcfg), 1235)
    vae = build_vae(vcfg, vsd)
    assert set(vae.state_dict()) == set(vsd)
    z = torch.randn(3, 4, 16, 16, generator=torch.Generator().manual_seed(5))
    r = lambda t: t.bfloat16().float()
    with torch.no_grad():
        ref = O.vae_decode({k: r(v) for k, v in vsd.items()}, vcfg, r(z))
    out = vae.decode(z.bfloat16().cuda()).sample
    e = _rel(out.float().cpu(), ref)
    print("vae decode rel", e)
    assert out.shape == (3, 3, 128, 128) and e < 2e-2
    # fused decode_latents == reference decode_latents semantics
    lat = (z * 0.18215)
    with torch.no_grad():
        ref2 = O.decode_latents({k: r(v) for k, v in vsd.items()}, vcfg, r(lat).unsqueeze(0).permute(0, 2, 1, 3, 4))
    out2 = vae.decode_latents(lat.bfloat16().cuda())
    assert out2.dtype == torch.float32 and float(out2.min()) >= 0 and float(out2.max()) <= 1
    d = (out2.cpu() - ref2[0].permute(1, 0, 2, 3)).abs()
    print("decode_latents max abs", d.max().item(), "mean", d.mean().item())
    assert d.mean().item() < 5e-3 and d.max().item() < 8e-2


class _RefNetStub(torch.nn.Module):
    """ReferenceNet write pass is outside the hot path: exposes the cond banks in pairing order."""
    def __init__(self, banks):
        super().__init__()
        self.writer_view = _Writer(banks)

    def forward(self, *a, **k):
        return None


def build_pipeline(cfg, vcfg, sd, vsd, kps, audio, banks_cond, latents):
    from vexpress_b200.modules import UNet3DConditionModel
    from vexpress_b200.pipelines.scheduler import DDIMScheduler
    from vexpress_b200.pipelines.v_express_pipeline import VExpressPipeline
    unet = UNet3DConditionModel(block_out_channels=cfg["block_out_channels"],
                                cross_attention_dim=cfg["cross_attention_dim"], **UNET_EXTRA)
    unet.load_state_dict(sd)
    unet = unet.to(dtype=torch.bfloat16, device="cuda")
    vae = build_vae(vcfg, vsd)

    class Pipe(VExpressPipeline):
        def prepare_reference_latent(self, *a, **k):
            return None

        def prepare_kps_feature(self, *a, **k):
            return kps

        def prepare_audio_embeddings(self, *a, **k):
            return audio

        def run_reference_net(self, *a, **k):
            return None

        def prepare_latents(self, *a, **k):
            return latents.clone().to(torch.bfloat16)

    return Pipe(vae=vae, reference_net=_RefNetStub([b.cuda() for b in banks_cond]), denoising_unet=unet,
                v_kps_guider=None, audio_processor=None, audio_encoder=None, audio_projection=None,
                scheduler=DDIMScheduler())


@pytest.mark.parametrize("use_graph", [False, True])
def test_pipeline_vs_reference_golden(golden_dir, use_graph):
    """Whole hot path vs the video produced by the reference's own pipeline code in fp32.  Tolerance: the 3-step
    trajectory amplifies the per-forward bf16 error (~2e-2); final latents within 6e-2 relative L2, decoded video
    (range [0,1]) mean abs error < 1.5e-2."""
    from oracle import vx_oracle as O
    g = torch.load(os.path.join(golden_dir, "pipeline_small.pt"), weights_only=False)
    cfg, vcfg = g["cfg"], g["vae_cfg"]
    sd = O.synth_state_dict(O.unet_param_shapes(cfg), 1234)
    vsd = O.synth_state_dict(O.vae_param_shapes(vcfg), 1235)
    lat, kps, audio, banks = O.synth_inputs(cfg, g["L"], g["h"], g["h"], True, 42)
    pipe = build_pipeline(cfg, vcfg, sd, vsd, kps, audio, [b[1:] for b in banks], lat)
    pipe.use_cuda_graph = use_graph
    captured = {}
    orig = pipe._decode_to_host

    def grab(latents, distributed):
        captured["latents"] = latents.float().cpu()
        return orig(latents, distributed)
    pipe._decode_to_host = grab
    video = pipe(reference_image=None, kps_images=None, audio_waveform=None, width=g["h"] * 8, height=g["h"] * 8,
                 video_length=g["L"], num_inference_steps=g["steps"], guidance_scale=g["guidance_scale"],
                 context_frames=g["S"], context_overlap=g["O"], reference_attention_weight=0.95,
                 audio_attention_weight=3.0)
    assert tuple(video.shape) == g["video_shape"] and video.dtype == torch.float32 and video.device.type == "cpu"
    e_lat = _rel(captured["latents"], g["final_latents"])
    d = (video.flatten()[::g["sample_stride"]] - g["video"].float()).abs()
    print(f"graph={use_graph} final latents rel {e_lat:.3e}; video mean abs {d.mean().item():.3e} max {d.max().item():.3e}")
    assert e_lat < 6e-2 and d.mean().item() < 1.5e-2
    # a second call on the same pipeline object reuses the captured graph / persistent bank buffers
    video2 = pipe(reference_image=None, kps_images=None, audio_waveform=None, width=g["h"] * 8, height=g["h"] * 8,
                  video_length=g["L"], num_inference_steps=g["steps"], guidance_scale=g["guidance_scale"],
                  context_frames=g["S"], context_overlap=g["O"], reference_attention_weight=0.95,
                  audio_attention_weight=3.0)
    assert torch.equal(video, video2)


def test_pipeline_non_tiling_length_follows_reference_bookkeeping(golden_dir):
    """video_length 20 with windows of 16 / overlap 4: the tail window is reflected and repeats frames 12..18; the
    reference's index-put / streaming bookkeeping decides which slots count (SURVEY Appendix D).  The integer plan is
    proven bit-exact on the CPU (tests/test_host_cpu.py); here the real kernels run it and land on the oracle's
    restatement of the reference loop within the trajectory tolerance."""
    from oracle import vx_oracle as O
    cfg, vcfg = O.small_cfg(), O.small_vae_cfg()
    sd = O.synth_state_dict(O.unet_param_shapes(cfg), 1234)
    vsd = O.synth_state_dict(O.vae_param_shapes(vcfg), 1235)
    L = 20
    lat, kps, audio, banks = O.synth_inputs(cfg, L, 16, 16, True, 42)
    pipe = build_pipeline(cfg, vcfg, sd, vsd, kps, audio, [b[1:] for b in banks], lat)
    captured = {}
    orig = pipe._decode_to_host

    def grab(latents, distributed):
        captured["latents"] = latents.float().cpu()
        return orig(latents, distributed)
    pipe._decode_to_host = grab
    video = pipe(None, None, None, 128, 128, L, 2, 3.5, context_frames=16, context_overlap=4,
                 reference_attention_weight=0.95, audio_attention_weight=3.0)
    assert video.shape == (1, 3, L, 128, 128)
    r = lambda t: t.bfloat16().float()
    with torch.no_grad():
        ref = O.denoise({k: r(v) for k, v in sd.items()}, cfg, r(lat), r(kps), r(audio), [r(b) for b in banks], 2, 3.5, 16, 4,
                        ref_w=0.95, audio_w=3.0)
    e = _rel(captured["latents"], ref)
    worst = max(_rel(captured["latents"][:, :, i], ref[:, :, i]) for i in range(L))
    # and the output of the reference's OWN pipeline code for this call (fp32, unrounded weights)
    g = torch.load(os.path.join(golden_dir, "pipeline_nontiling_small.pt"), weights_only=False)
    assert (g["L"], g["S"], g["O"], g["steps"]) == (20, 16, 4, 2)
    e_ref = _rel(captured["latents"], g["final_latents"])
    print(f"non-tiling L=20: final latents rel {e:.3e} vs oracle, worst frame {worst:.3e}; vs reference golden {e_ref:.3e}")
    assert e < 5e-2 and worst < 8e-2 and e_ref < 6e-2


def test_vae_encode_reference_latent_vs_oracle():
    """Row f4: ``prepare_reference_latent`` = VAE posterior mean x 0.18215 on the decoder's kernels vs the oracle."""
    from oracle import vx_oracle as O
    from vexpress_b200.modules.vae import AutoencoderKL
    from vexpress_b200.pipelines.scheduler import DDIMScheduler
    from vexpress_b200.pipelines.v_express_pipeline import VExpressPipeline
    vcfg = O.small_vae_cfg()
    vsd = O.synth_state_dict({**O.vae_param_shapes(vcfg), **O.vae_encoder_param_shapes(vcfg)}, 1236)
    vae = AutoencoderKL(block_out_channels=vcfg["block_out_channels"], layers_per_block=vcfg["layers_per_block"])
    vae.load_state_dict(vsd, strict=True)
    vae = vae.to(torch.bfloat16).to("cuda")
    img = torch.rand(1, 3, 128, 128, generator=torch.Generator().manual_seed(11)) * 2 - 1
    r = lambda t: t.bfloat16().float()
    with torch.no_grad():
        ref = O.vae_encode_mean({k: r(v) for k, v in vsd.items()}, vcfg, r(img)) * 0.18215
    pipe = VExpressPipeline(vae=vae, reference_net=None, denoising_unet=vae, v_kps_guider=None, audio_processor=None,
                            audio_encoder=None, audio_projection=None, scheduler=DDIMScheduler())
    lat = pipe.prepare_reference_latent(img, 128, 128)
    e = _rel(lat.float().cpu(), ref)
    print(f"VAE encode (reference latent) rel-L2 vs oracle {e:.3e}")
    assert lat.shape == (1, 4, 16, 16) and e < 2e-2
    # a uint8 HWC image goes through the same preprocessing as the reference's VaeImageProcessor (x / 255 * 2 - 1)
    u8 = ((img[0].permute(1, 2, 0) + 1) * 127.5).round().clamp(0, 255).to(torch.uint8).numpy()
    lat2 = pipe.prepare_reference_latent(u8, 128, 128)
    assert _rel(lat2.float().cpu(), ref) < 3e-2
