"""Generate the committed golden vectors under tests/golden/ by running the REFERENCE'S OWN CODE.

TEST INFRASTRUCTURE ONLY.  Runs in the build container (needs /root/reference, read-only); the GPU
box never runs this.  The reference's files are imported verbatim from where they lie:

  * ``pipelines/context.py``               (stand-alone, numpy only)          -> context_windows.json
  * ``modules/{unet_3d,unet_3d_blocks,transformer_3d,attention,motion_module,resnet,
     mutual_self_attention}.py``           (over oracle/diffusers_shim)        -> unet_small.pt
  * ``pipelines/v_express_pipeline.py``    (over the shim; DDIM + VAE decoder restated) -> pipeline_small.pt
  * ``modules/{unet_2d_condition,unet_2d_blocks,transformer_2d,attention}.py`` + the write-mode hooks of
     ``mutual_self_attention.py``          (ReferenceNet, SURVEY 8f-f1)        -> refnet_small.pt

Inputs/weights are NOT stored: they are regenerated from seeds by ``oracle.vx_oracle.synth_*``.
  * ``modules/v_kps_guider.py``, ``modules/audio_projection.py``, the audio windowing of
     ``VExpressPipeline.prepare_audio_embeddings`` and ``median_filter_3d`` of ``pipelines/utils.py`` (SURVEY 8f-f2/f3;
     the latter executed from its source because the module imports cv2 / ffmpeg)      -> prologue_small.pt
  * parameter names / defaults of the public entry points the product mirrors (read with ``ast``)
                                                                               -> reference_signatures.json

The largest outputs (UNet taps, decoded video) are stored as every SAMPLE_STRIDE-th element of the flattened tensor, with
the full shape beside them, so that every golden file stays under 1 MB.

Usage:  python oracle/gen_golden.py [context ddim unet pipeline refnet prologue signatures]   (default: all)
"""
import importlib
import importlib.util
import json
import os
import sys
import types

import torch

ROOT = os.path.abspath(os.path.join(os.path.dirname(__file__), ".."))
REF = os.environ.get("VX_REFERENCE", "/root/reference")
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "oracle", "diffusers_shim"))
from oracle import vx_oracle as O  # noqa: E402

GOLD = os.path.join(ROOT, "tests", "golden")
SAMPLE_STRIDE = 3       # odd, so the sample walks through every column / row parity of the power-of-two image sides


def import_reference():
    """Register empty ``modules`` / ``pipelines`` packages whose __path__ points into the read-only
    reference tree so their files import verbatim without running the package __init__ (which pulls
    the UNet2D's wide diffusers import surface)."""
    for name in ("modules", "pipelines"):
        m = types.ModuleType(name)
        m.__path__ = [os.path.join(REF, name)]
        sys.modules[name] = m
    msa = importlib.import_module("modules.mutual_self_attention")
    sys.modules["modules"].ReferenceAttentionControl = msa.ReferenceAttentionControl
    unet3d = importlib.import_module("modules.unet_3d")
    ctx = importlib.import_module("pipelines.context")
    pipe = importlib.import_module("pipelines.v_express_pipeline")
    return msa, unet3d, ctx, pipe


UNET_EXTRA = dict(  # inference_v2.yaml:1-21
    use_inflated_groupnorm=True, unet_use_cross_frame_attention=False, unet_use_temporal_attention=False,
    use_motion_module=True, motion_module_resolutions=[1, 2, 4, 8], motion_module_mid_block=True,
    motion_module_decoder_only=False, motion_module_type="Vanilla",
    motion_module_kwargs=dict(num_attention_heads=8, num_transformer_block=1,
                              attention_block_types=["Temporal_Self", "Temporal_Self"],
                              temporal_position_encoding=True, temporal_position_encoding_max_len=32,
                              temporal_attention_dim_div=1))


def build_reference_unet(unet3d, cfg, sd):
    model = unet3d.UNet3DConditionModel(
        sample_size=64, in_channels=4, out_channels=4,
        down_block_types=("CrossAttnDownBlock3D", "CrossAttnDownBlock3D", "CrossAttnDownBlock3D", "DownBlock3D"),
        mid_block_type="UNetMidBlock3DCrossAttn",
        up_block_types=("UpBlock3D", "CrossAttnUpBlock3D", "CrossAttnUpBlock3D", "CrossAttnUpBlock3D"),
        block_out_channels=cfg["block_out_channels"], layers_per_block=2, cross_attention_dim=cfg["cross_attention_dim"],
        attention_head_dim=8, norm_num_groups=32, norm_eps=1e-5, **UNET_EXTRA)
    ref_sd = model.state_dict()
    assert set(ref_sd) == set(sd), (sorted(set(ref_sd) ^ set(sd))[:10])
    for k in ref_sd:
        assert tuple(ref_sd[k].shape) == tuple(sd[k].shape), k
    model.load_state_dict(sd, strict=True)
    return model.eval()


def install_reader(msa, model, banks, ref_w, audio_w, do_cfg=True):
    reader = msa.ReferenceAttentionControl(model, do_classifier_free_guidance=do_cfg, mode="read", batch_size=1,
                                           fusion_blocks="full", reference_attention_weight=ref_w,
                                           audio_attention_weight=audio_w)
    # same selection + stable sort as ReferenceAttentionControl.update (mutual_self_attention.py:339-351)
    from modules.attention import TemporalBasicTransformerBlock
    mods = [m for m in msa.torch_dfs(model) if isinstance(m, TemporalBasicTransformerBlock)]
    mods = sorted(mods, key=lambda x: -x.norm1.normalized_shape[0])
    names = {id(m): n for n, m in model.named_modules()}
    order = [names[id(m)].replace(".transformer_blocks.0", "") for m in mods]
    for m, bk in zip(mods, banks):
        m.bank = [bk.clone()]
    return reader, order


def gen_context(ctx):
    cases = [(4, 24, 4), (16, 16, 8), (96, 16, 8), (384, 16, 8), (924, 24, 4), (20, 16, 4), (100, 16, 8),
             (40, 16, 8), (12, 8, 4), (33, 24, 4)]
    out = []
    for L, S, Ov in cases:
        wins = list(ctx.uniform(step=0, num_frames=L, context_size=S, context_stride=1, context_overlap=Ov,
                                closed_loop=False))
        nfc = torch.zeros(L, dtype=torch.long)
        for w in wins:
            nfc[w] += 1  # the reference's own index-put (v_express_pipeline.py:498-500)
        out.append(dict(L=L, S=S, O=Ov, windows=[[int(e) for e in w] for w in wins], num_frame_context=nfc.tolist()))
    # other scheduler-call flavours (step != 0, stride > 1, closed loop) to pin `uniform` itself
    extra = []
    for (step, L, S, stride, Ov, closed) in [(1, 64, 16, 3, 4, True), (5, 48, 16, 2, 4, True), (3, 100, 24, 3, 4, False)]:
        wins = list(ctx.uniform(step, L, S, stride, Ov, closed))
        extra.append(dict(step=step, L=L, S=S, stride=stride, O=Ov, closed=closed,
                          windows=[[int(e) for e in w] for w in wins]))
    oh = {str(v): ctx.ordered_halving(v) for v in (0, 1, 2, 3, 5, 8, 1000, 2 ** 63)}
    with open(os.path.join(GOLD, "context_windows.json"), "w") as f:
        json.dump(dict(pipeline_calls=out, uniform_calls=extra, ordered_halving=oh), f)
    print("context_windows.json:", len(out), "+", len(extra), "cases")


def gen_unet(msa, unet3d):
    torch.manual_seed(0)
    cfg = O.small_cfg()
    sd = O.synth_state_dict(O.unet_param_shapes(cfg), seed=1234)
    model = build_reference_unet(unet3d, cfg, sd)
    f, h = 4, 16
    latents, kps, audio, banks = O.synth_inputs(cfg, L=f, h=h, w=h, do_cfg=True, seed=42)
    reader, order = install_reader(msa, model, banks, 0.95, 3.0)
    assert order == O.bank_order(cfg), (order, O.bank_order(cfg))
    taps = {}
    want = ["down_blocks.0.resnets.0", "down_blocks.0.attentions.0", "down_blocks.0.motion_modules.0",
            "down_blocks.1.attentions.1", "down_blocks.3.motion_modules.1", "mid_block",
            "up_blocks.1.attentions.2", "up_blocks.3.motion_modules.2"]
    mods = dict(model.named_modules())
    hooks = []
    for n in want:
        def mk(n):
            def hook(_m, _i, out):
                t = out.sample if hasattr(out, "sample") else out
                taps[n] = t.detach().permute(0, 2, 1, 3, 4).reshape(-1, t.shape[1], *t.shape[3:]).clone()
            return hook
        hooks.append(mods[n].register_forward_hook(mk(n)))
    x = latents.repeat(2, 1, 1, 1, 1)
    enc = audio.reshape(-1, 5, cfg["cross_attention_dim"])
    with torch.no_grad():
        out = model(x, torch.tensor(499), encoder_hidden_states=enc, kps_features=kps, return_dict=False)[0]
        for hk in hooks:   # taps belong to the t=499 call only
            hk.remove()
        out2 = model(x, 959, encoder_hidden_states=enc, kps_features=kps, return_dict=False)[0]
    torch.save(dict(cfg=cfg, seed_weights=1234, seed_inputs=42, f=f, h=h, ref_w=0.95, audio_w=3.0,
                    bank_order=order, out_t499=out, out_t959=out2, sample_stride=SAMPLE_STRIDE,
                    tap_shapes={k: tuple(v.shape) for k, v in taps.items()},
                    taps={k: v.flatten()[::SAMPLE_STRIDE].half() for k, v in taps.items()}),
               os.path.join(GOLD, "unet_small.pt"))
    print("unet_small.pt: out", tuple(out.shape), "absmean", out.abs().mean().item())


def scheduler_kwargs():
    """noise_scheduler_kwargs of the reference's own inference_v2.yaml:23-33 (what inference.py:132-136 passes)."""
    import yaml
    with open(os.path.join(REF, "inference_v2.yaml")) as fh:
        return dict(yaml.safe_load(fh)["noise_scheduler_kwargs"])


def gen_pipeline(msa, unet3d, pipe, L=12, S=8, Ov=4, steps=3, name="pipeline_small.pt", with_video=True):
    cfg = O.small_cfg()
    vcfg = O.small_vae_cfg()
    sd = O.synth_state_dict(O.unet_param_shapes(cfg), seed=1234)
    vsd = O.synth_state_dict(O.vae_param_shapes(vcfg), seed=1235)
    model = build_reference_unet(unet3d, cfg, sd)
    h, gs = 16, 3.5
    latents, kps, audio, banks = O.synth_inputs(cfg, L=L, h=h, w=h, do_cfg=True, seed=42)
    from diffusers import AutoencoderKL, DDIMScheduler
    vae = AutoencoderKL(vsd, vcfg)

    class StubRefNet(torch.nn.Module):
        """Stands in for the ReferenceNet write pass (out of scope, SURVEY 8f-f1)."""
        def __init__(self):
            super().__init__()
            self.p = torch.nn.Parameter(torch.zeros(1))

        def forward(self, *a, **k):
            return None

    class Pipe(pipe.VExpressPipeline):
        # only the three prologue methods are overridden (v_express_pipeline.py:343-407)
        def prepare_reference_latent(self, *a, **k):
            return torch.zeros(1, 4, h, h)

        def prepare_kps_feature(self, *a, **k):
            return kps

        def prepare_audio_embeddings(self, *a, **k):
            return audio

        def prepare_latents(self, *a, **k):
            return latents.clone() * self.scheduler.init_noise_sigma

    # the pipeline constructs its own reader; make `update` a bank injection in pairing order
    real_update = msa.ReferenceAttentionControl.update

    def update(self, writer, do_classifier_free_guidance=True, do_unconditional_forward=False, dtype=torch.float16):
        from modules.attention import TemporalBasicTransformerBlock
        mods = [m for m in msa.torch_dfs(self.unet) if isinstance(m, TemporalBasicTransformerBlock)]
        mods = sorted(mods, key=lambda x: -x.norm1.normalized_shape[0])
        for m, bk in zip(mods, banks):
            m.bank = [bk.clone().to(dtype)]
    msa.ReferenceAttentionControl.update = update
    try:
        p = Pipe(vae=vae, reference_net=StubRefNet(), denoising_unet=model, v_kps_guider=None, audio_processor=None,
                 audio_encoder=None, audio_projection=None, scheduler=DDIMScheduler(**scheduler_kwargs()))
        captured = {}
        orig_decode = Pipe.decode_latents

        def decode(self, lat):
            captured["latents"] = lat.clone()
            return orig_decode(self, lat)
        Pipe.decode_latents = decode
        with torch.no_grad():
            video = p(reference_image=None, kps_images=None, audio_waveform=None, width=h * 8, height=h * 8,
                      video_length=L, num_inference_steps=steps, guidance_scale=gs, context_frames=S,
                      context_overlap=Ov, reference_attention_weight=0.95, audio_attention_weight=3.0)
    finally:
        msa.ReferenceAttentionControl.update = real_update
    out = dict(cfg=cfg, vae_cfg=vcfg, L=L, h=h, S=S, O=Ov, steps=steps, guidance_scale=gs, final_latents=captured["latents"])
    if with_video:
        out.update(video_shape=tuple(video.shape), sample_stride=SAMPLE_STRIDE,
                   video=video.flatten()[::SAMPLE_STRIDE].half())
    torch.save(out, os.path.join(GOLD, name))
    print(name, ": video", tuple(video.shape), "latents absmean", captured["latents"].abs().mean().item())


def gen_refnet(msa, unet3d):
    """ReferenceNet write pass exactly as the pipeline drives it (v_express_pipeline.py:451-457,501-509): the
    reference's UNet2DConditionModel under a write-mode ReferenceAttentionControl at timestep 0 with a zero text
    token, then the reference's own ``reader.update(writer, do_cfg)`` into a reference UNet3D."""
    u2 = importlib.import_module("modules.unet_2d_condition")
    cfg = O.small_cfg()
    sd = O.synth_state_dict(O.refnet_param_shapes(cfg), seed=4321)
    net = u2.UNet2DConditionModel(
        sample_size=64, in_channels=4, out_channels=4,
        down_block_types=("CrossAttnDownBlock2D", "CrossAttnDownBlock2D", "CrossAttnDownBlock2D", "DownBlock2D"),
        up_block_types=("UpBlock2D", "CrossAttnUpBlock2D", "CrossAttnUpBlock2D", "CrossAttnUpBlock2D"),
        block_out_channels=cfg["block_out_channels"], layers_per_block=2, cross_attention_dim=cfg["cross_attention_dim"],
        attention_head_dim=8, norm_num_groups=32, norm_eps=1e-5)
    ref_sd = net.state_dict()
    assert set(ref_sd) == set(sd), sorted(set(ref_sd) ^ set(sd))[:10]
    for k in ref_sd:
        assert tuple(ref_sd[k].shape) == tuple(sd[k].shape), k
    net.load_state_dict(sd, strict=True)
    net.eval()
    h = 16
    ref_latents = torch.randn(1, 4, h, h, generator=torch.Generator().manual_seed(77))
    writer = msa.ReferenceAttentionControl(net, do_classifier_free_guidance=True, mode="write", batch_size=1,
                                           fusion_blocks="full")
    with torch.no_grad():
        out = net(ref_latents, timestep=0, encoder_hidden_states=torch.zeros(1, 1, cfg["cross_attention_dim"]),
                  return_dict=False)[0]
    # hand the banks to a reference UNet3D reader with the reference's own update()
    unet = build_reference_unet(unet3d, cfg, O.synth_state_dict(O.unet_param_shapes(cfg), seed=1234))
    reader = msa.ReferenceAttentionControl(unet, do_classifier_free_guidance=True, mode="read", batch_size=1,
                                           fusion_blocks="full")
    reader.update(writer, True, dtype=torch.float32)
    from modules.attention import TemporalBasicTransformerBlock
    mods = [m for m in msa.torch_dfs(unet) if isinstance(m, TemporalBasicTransformerBlock)]
    mods = sorted(mods, key=lambda x: -x.norm1.normalized_shape[0])
    names = {id(m): n for n, m in unet.named_modules()}
    order = [names[id(m)].replace(".transformer_blocks.0", "") for m in mods]
    assert order == O.bank_order(cfg), (order, O.bank_order(cfg))
    banks = []
    for m in mods:
        assert len(m.bank) == 1
        bk = m.bank[0]
        assert bk.shape[0] == 2 and torch.count_nonzero(bk[0]).item() == 0   # CFG: [zeros | bank] (:357-359)
        banks.append(bk[1:].clone())
    torch.save(dict(cfg=cfg, seed_weights=4321, seed_latents=77, h=h, bank_order=order, banks=banks, out=out),
               os.path.join(GOLD, "refnet_small.pt"))
    print("refnet_small.pt:", len(banks), "banks,", [tuple(b.shape) for b in banks[:1] + banks[-1:]],
          "out absmean", out.abs().mean().item())


def gen_prologue(pipe):
    import ast
    import torch.nn.functional as func
    import tqdm
    kg = importlib.import_module("modules.v_kps_guider")
    ap = importlib.import_module("modules.audio_projection")
    out = {}
    # VKpsGuider (inference.py:100): 64x64 keypoint images, 2 frames
    kcfg = O.KPS_CFG
    ksd = O.synth_state_dict(O.kps_guider_param_shapes(kcfg), 21)
    m = kg.VKpsGuider(kcfg["conditioning_embedding_channels"], block_out_channels=kcfg["block_out_channels"])
    assert set(m.state_dict()) == set(ksd)
    m.load_state_dict(ksd)
    kps_in = torch.rand(1, 3, 2, 64, 64, generator=torch.Generator().manual_seed(3))
    with torch.no_grad():
        out["kps"] = dict(seed_weights=21, seed_input=3, shape=tuple(kps_in.shape), feature=m.eval()(kps_in))
    # AudioProjection (inference.py:116-126,192-201)
    acfg = O.AUDIO_PROJ_CFG
    asd = O.synth_state_dict(O.audio_projection_param_shapes(acfg), 22)
    m2 = ap.AudioProjection(dim=acfg["dim"], depth=acfg["depth"], dim_head=acfg["dim_head"], heads=acfg["heads"],
                            num_queries=acfg["num_queries"], embedding_dim=acfg["embedding_dim"],
                            output_dim=acfg["output_dim"], ff_mult=acfg["ff_mult"], max_seq_len=acfg["max_seq_len"])
    assert set(m2.state_dict()) == set(asd)
    m2.load_state_dict(asd)
    xa = torch.randn(6, 10, 768, generator=torch.Generator().manual_seed(4))
    with torch.no_grad():
        out["audio_projection"] = dict(seed_weights=22, seed_input=4, shape=tuple(xa.shape), tokens=m2.eval()(xa))

    # audio windowing: the reference method itself with stub encoder / identity projection (:374-407)
    class _Enc:
        def __call__(self, w):
            return type("R", (), {"last_hidden_state": w})()

    class _Self:
        device, dtype = torch.device("cpu"), torch.float32
        audio_processor = staticmethod(lambda w, return_tensors=None, sampling_rate=None: {"input_values": w})
        audio_encoder = _Enc()
        audio_projection = staticmethod(lambda x: x)
    emb = torch.randn(1, 37, 32, generator=torch.Generator().manual_seed(6))
    win = pipe.VExpressPipeline.prepare_audio_embeddings(_Self(), emb, 8, 2, True)
    assert win.shape[0] == 2 and torch.count_nonzero(win[0]).item() == 0
    out["audio_windows"] = dict(seed_input=6, shape=tuple(emb.shape), video_length=8, num_pad=2, windows=win[1])
    # median filter: the function's own source (pipelines/utils.py:46-63)
    src = open(os.path.join(REF, "pipelines", "utils.py")).read()
    fn = [n for n in ast.parse(src).body if isinstance(n, ast.FunctionDef) and n.name == "median_filter_3d"][0]
    ns = dict(torch=torch, func=func, tqdm=tqdm)
    exec(compile(ast.Module(body=[fn], type_ignores=[]), "pipelines/utils.py", "exec"), ns)
    v = torch.rand(3, 5, 12, 10, generator=torch.Generator().manual_seed(5))
    filt = ns["median_filter_3d"](v, 3, "cpu")
    out["median"] = dict(seed_input=5, shape=tuple(v.shape), filtered=filt,
                         uint8=torch.from_numpy((filt.permute(1, 2, 3, 0) * 255).numpy().astype("uint8")))
    torch.save(out, os.path.join(GOLD, "prologue_small.pt"))
    print("prologue_small.pt:", {k: tuple(next(t for t in v.values() if torch.is_tensor(t)).shape) for k, v in out.items()})


def gen_ddim():
    """Known-answer values of the DDIM configuration of inference_v2.yaml:23-33, produced by the shim's library-structured
    ``DDIMScheduler`` (written separately from ``O.DDIM``; both are also held to float64 closed forms in
    tests/test_oracle_golden.py)."""
    from diffusers import DDIMScheduler
    s = DDIMScheduler(**scheduler_kwargs())
    kat = dict(abar={str(i): float(s.alphas_cumprod[i]) for i in (0, 1, 499, 959, 998, 999)})
    for n in (2, 25, 50):
        s.set_timesteps(n)
        kat[f"timesteps_{n}"] = s.timesteps.tolist()
    s.set_timesteps(25)
    x = torch.tensor([1.5409961, -0.2934289, -2.1787894, 0.5684313])
    v = torch.tensor([-1.0845224, -1.3985955, 0.4033468, 0.8380263])
    kat["step_t999_n25"] = s.step(v, 999, x).prev_sample.tolist()
    with open(os.path.join(GOLD, "ddim_kat.json"), "w") as f:
        json.dump(kat, f)
    print("ddim_kat.json", kat["step_t999_n25"])


SIGNATURES = [  # (reference file, class, function): the drop-in boundary the product keeps
    ("pipelines/v_express_pipeline.py", "VExpressPipeline", "__call__"),
    ("pipelines/v_express_pipeline.py", "VExpressPipeline", "mean_overlap"),
    ("pipelines/v_express_pipeline.py", "VExpressPipeline", "__init__"),
    ("pipelines/v_express_pipeline.py", "VExpressPipeline", "prepare_reference_latent"),
    ("pipelines/v_express_pipeline.py", "VExpressPipeline", "prepare_kps_feature"),
    ("pipelines/v_express_pipeline.py", "VExpressPipeline", "prepare_audio_embeddings"),
    ("modules/unet_3d.py", "UNet3DConditionModel", "forward"),
    ("modules/unet_3d.py", "UNet3DConditionModel", "from_config_2d"),
    ("modules/unet_3d.py", "UNet3DConditionModel", "__init__"),
    ("modules/mutual_self_attention.py", "ReferenceAttentionControl", "__init__"),
    ("modules/mutual_self_attention.py", "ReferenceAttentionControl", "update"),
    ("modules/mutual_self_attention.py", "ReferenceAttentionControl", "clear"),
    ("pipelines/context.py", None, "uniform"),
    ("pipelines/context.py", None, "get_context_scheduler"),
    ("pipelines/context.py", None, "ordered_halving"),
]


def ast_signature(path, cls, fn):
    """[(name, default source or '<required>')] of a function in a source file, without importing it."""
    import ast
    tree = ast.parse(open(path).read())
    body = tree.body
    if cls is not None:
        body = next(n for n in tree.body if isinstance(n, ast.ClassDef) and n.name == cls).body
    f = next(n for n in body if isinstance(n, (ast.FunctionDef, ast.AsyncFunctionDef)) and n.name == fn)
    a = f.args
    pos = a.posonlyargs + a.args
    defaults = [None] * (len(pos) - len(a.defaults)) + list(a.defaults)
    out = []
    for arg, d in zip(pos, defaults):
        out.append((arg.arg, "<required>" if d is None else ast.unparse(d)))
    for arg, d in zip(a.kwonlyargs, a.kw_defaults):
        out.append((arg.arg, "<required>" if d is None else ast.unparse(d)))
    if a.kwarg is not None:
        out.append(("**" + a.kwarg.arg, ""))
    return out


def gen_signatures():
    sigs = [dict(file=f, cls=c, fn=fn, params=ast_signature(os.path.join(REF, f), c, fn)) for f, c, fn in SIGNATURES]
    with open(os.path.join(GOLD, "reference_signatures.json"), "w") as fh:
        json.dump(sigs, fh, indent=1)
    print("reference_signatures.json:", len(sigs), "entry points")


if __name__ == "__main__":
    os.makedirs(GOLD, exist_ok=True)
    torch.set_num_threads(os.cpu_count())
    msa, unet3d, ctx, pipe = import_reference()
    which = set(sys.argv[1:]) or {"context", "ddim", "unet", "pipeline", "refnet", "prologue", "signatures"}
    if "context" in which:
        gen_context(ctx)
    if "ddim" in which:
        gen_ddim()
    if "unet" in which:
        gen_unet(msa, unet3d)
    if "pipeline" in which:
        gen_pipeline(msa, unet3d, pipe)
        # video_length that does NOT tile: the tail window is reflected and repeats frames (SURVEY Appendix D).  The
        # reference then writes `latents[:, :, step_frame_ids] = ...` with DUPLICATE indices on a host tensor
        # (v_express_pipeline.py:572) -- torch documents index_put_ with duplicates as undefined, and with several intra-op
        # threads which duplicate wins is a race (measured: 8 threads -> frames 13..15 keep the FIRST write, frames 12,
        # 16..18 the LAST).  Single-threaded the writes are sequential and the last one wins; that defined behaviour is
        # what the oracle and the product implement, so this golden is generated with one thread.
        nthreads = torch.get_num_threads()
        torch.set_num_threads(1)
        try:
            gen_pipeline(msa, unet3d, pipe, L=20, S=16, Ov=4, steps=2, name="pipeline_nontiling_small.pt", with_video=False)
        finally:
            torch.set_num_threads(nthreads)
    if "refnet" in which:
        gen_refnet(msa, unet3d)
    if "prologue" in which:
        gen_prologue(pipe)
    if "signatures" in which:
        gen_signatures()
