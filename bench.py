#!/usr/bin/env python
"""Benchmark of the V-Express denoising hot path on B200 (contract: see the task brief / DESIGN.md section 6).

  python bench.py --gpus N --steps K --warmup W            # our arm (CUDA kernels through the C ABI)
  python bench.py --impl reference --steps K --warmup W    # the reference algorithm on the host cores (oracle port)

One bench "step" = one pass of the whole hot path over one synthetic video: 25 DDIM steps x all context windows
through the denoising UNet (CFG, overlap averaging) followed by the VAE decode of every frame.
N = 1 runs BASELINE.json configs[1] (512x512, one 16-frame window, 25 steps, bf16).  N > 1 is weak scaling: N windows
of 16 frames (overlap 8), one per rank, one NCCL all-reduce of the overlap noise-prediction sums per DDIM step,
VAE decode sharded by frame.  Rank 0 prints ONE JSON line.
"""
import argparse
import json
import math
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import torch  # noqa: E402

UNET_EXTRA = dict(
    use_inflated_groupnorm=True, unet_use_cross_frame_attention=False, unet_use_temporal_attention=False,
    use_motion_module=True, motion_module_resolutions=[1, 2, 4, 8], motion_module_mid_block=True,
    motion_module_decoder_only=False, motion_module_type="Vanilla",
    motion_module_kwargs=dict(num_attention_heads=8, num_transformer_block=1,
                              attention_block_types=["Temporal_Self", "Temporal_Self"],
                              temporal_position_encoding=True, temporal_position_encoding_max_len=32,
                              temporal_attention_dim_div=1))

# canonical algorithmic work (SURVEY.md 8d / BASELINE.md 3), bf16, per CFG window-forward (b=2, f=16) at 512^2
UNET_TFLOP_PER_FRAME_EVAL = 1.2768
VAE_TFLOP_PER_FRAME = 2.515


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return dict(hbm_gbs=d["hbm_gbs"], tf_burst=d["bf16_tflops"], tf_sustained=d["bf16_tflops_sustained"],
                    source="measured")
    return dict(hbm_gbs=6650.0, tf_burst=1590.0, tf_sustained=1400.0, source="fallback")


# --------------------------------------------------------------------------------------------- synthetic model
def fill_synthetic_(module, seed):
    """Random init in the reference's state_dict layout (SURVEY.md 8d): W ~ randn/sqrt(fan_in), biases 0.02 randn,
    norm weights 1 + 0.02 randn; zero-initialised branches (motion proj_out, attn2.to_out) are NOT zeroed."""
    g = torch.Generator(device="cuda").manual_seed(seed)
    for name, p in module.named_parameters():
        mod = name.split(".")[-2]
        is_norm = "norm" in mod or (len(name.split(".")) > 2 and name.split(".")[-3] == "norms")
        if is_norm:
            p.data = (1.0 if name.endswith("weight") else 0.0) + 0.02 * torch.randn(p.shape, device="cuda", generator=g)
        elif name.endswith(".bias"):
            p.data = 0.02 * torch.randn(p.shape, device="cuda", generator=g)
        else:
            fan_in = int(math.prod(p.shape[1:]))
            p.data = torch.randn(p.shape, device="cuda", generator=g) / math.sqrt(fan_in)


def ln_rows(x):
    return torch.nn.functional.layer_norm(x, (x.shape[-1],))


def build_ours(L, h, device):
    from vexpress_b200.modules import UNet3DConditionModel
    from vexpress_b200.modules.unet_3d import attention_block_order
    from vexpress_b200.modules.vae import AutoencoderKL
    from vexpress_b200.pipelines.scheduler import DDIMScheduler
    from vexpress_b200.pipelines.v_express_pipeline import VExpressPipeline
    with torch.device(device):
        unet = UNet3DConditionModel(cross_attention_dim=768, **UNET_EXTRA)
        vae = AutoencoderKL()
    fill_synthetic_(unet, 1234)
    fill_synthetic_(vae, 1235)
    unet = unet.to(torch.bfloat16)
    vae = vae.to(torch.bfloat16)
    g = torch.Generator().manual_seed(42)
    lat = torch.randn(1, 4, L, h, h, generator=g).to(torch.bfloat16)
    kps = torch.zeros(2, 320, L, h, h, dtype=torch.bfloat16)                 # [uncond zeros | cond]; bf16 from the start:
    for f0 in range(0, L, 32):                                             # a 384-frame fp32 copy would be 4 GB per rank
        kps[1, :, f0:f0 + 32] = (0.1 * torch.randn(320, min(32, L - f0), h, h, generator=g)).to(torch.bfloat16)
    audio = ln_rows(torch.randn(1, L, 5, 768, generator=g))
    audio = torch.cat([torch.zeros_like(audio), audio]).to(torch.bfloat16)
    mods = dict(unet.named_modules())
    banks = []
    for name in attention_block_order(unet):
        C = mods[name].norm1.normalized_shape[0]
        parts = name.split(".")
        lvl = int(parts[1]) if parts[0] == "down_blocks" else (3 - int(parts[1]) if parts[0] == "up_blocks" else 3)
        N = (h >> lvl) ** 2
        banks.append(ln_rows(torch.randn(1, N, C, generator=g)).to(device=device, dtype=torch.bfloat16))
    host = dict(lat=lat.pin_memory(), kps=kps.pin_memory(), audio=audio.pin_memory())

    class Writer:
        pass
    wv = Writer()
    wv.banks = banks

    class RefNetStub(torch.nn.Module):
        writer_view = wv

        def forward(self, *a, **k):
            return None

    class Pipe(VExpressPipeline):
        # synthetic prologue: precomputed dummy conditioning, host resident (north_star)
        def prepare_reference_latent(self, *a, **k):
            return None

        def prepare_kps_feature(self, *a, **k):
            return host["kps"]

        def prepare_audio_embeddings(self, *a, **k):
            return host["audio"]

        def run_reference_net(self, *a, **k):
            return None

        def prepare_latents(self, *a, **k):
            return host["lat"]

    pipe = Pipe(vae=vae, reference_net=RefNetStub(), denoising_unet=unet, v_kps_guider=None, audio_processor=None,
                audio_encoder=None, audio_projection=None, scheduler=DDIMScheduler())
    return pipe, host, banks


# --------------------------------------------------------------------------------------------- clocks sampler
class Clocks:
    def __init__(self, index):
        self.rows, self.stop, self.index = [], False, index
        self.t = threading.Thread(target=self._run, daemon=True)

    def _run(self):
        q = "clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
            "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"
        while not self.stop:
            try:
                o = subprocess.run(["nvidia-smi", f"--id={self.index}", f"--query-gpu={q}", "--format=csv,noheader,nounits"],
                                   capture_output=True, text=True, timeout=5).stdout.strip()
                if o:
                    self.rows.append([c.strip() for c in o.split(",")])
            except Exception:
                pass
            time.sleep(0.2)

    def __enter__(self):
        self.t.start()
        return self

    def __exit__(self, *a):
        self.stop = True
        self.t.join(timeout=6)

    def summary(self):
        if not self.rows:
            return dict(sm_mhz=None, sm_max_mhz=None, reasons=["unavailable"])
        sm = sorted(int(r[0]) for r in self.rows if r[0].isdigit())
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for i, n in enumerate(names) if any(len(r) > 2 + i and r[2 + i].lower().startswith("active") for r in self.rows)]
        return dict(sm_mhz=sm[len(sm) // 2] if sm else None, sm_max_mhz=int(self.rows[0][1]) if self.rows[0][1].isdigit() else None,
                    reasons=reasons, samples=len(self.rows))


# --------------------------------------------------------------------------------------------- kernel timing
def op_table(pipe, host, L, h, which="unet"):
    """VX_BENCH_OPS=1: per-op / per-shape device time of one UNet forward.  Every unique (op, shapes) call recorded
    during an eager forward is replayed 8x back-to-back and timed with CUDA events (so host launch overhead overlaps)."""
    from vexpress_b200 import ops
    recs = []
    names = ["gemm", "gemm_ln", "gemm_rowsums", "gemm_lnparts", "conv3x3", "conv3x3_s2", "upconv3x3", "flash_attention", "temporal_attention", "smallkv_attention", "groupnorm",
             "layernorm", "conv_in", "conv_out", "im2col_s2", "upsample2x", "skinny_linear", "timestep_embed", "softmax_rows"]
    orig = {n: getattr(ops, n) for n in names}

    def wrap(n, fn):
        def w(*a, **k):
            out = fn(*a, **k)
            sig = tuple(tuple(x.shape) for x in a[:3] if torch.is_tensor(x))
            extra = tuple(sorted((kk, tuple(v.shape) if torch.is_tensor(v) else v) for kk, v in k.items()
                                 if kk in ("a2", "residual", "geglu", "kv_div", "silu")))
            recs.append((n, sig + extra, a, k))
            return out
        return w
    for n in names:
        setattr(ops, n, wrap(n, orig[n]))
    try:
        eng = pipe.denoising_unet.engine()
        f = min(L, 16)
        frames = host["lat"].cuda()[0, :, :f].permute(1, 0, 2, 3).repeat(2, 1, 1, 1).contiguous()
        enc = host["audio"].cuda()[:, :f].reshape(2 * f, 5, 768)
        kps = host["kps"].cuda()[:, :, :f].permute(0, 2, 3, 4, 1).reshape(2 * f * h * h, 320).contiguous()
        if which == "vae":
            z = host["lat"].cuda()[0].permute(1, 0, 2, 3)[:16].contiguous()
            run = lambda: pipe.vae.decode_latents(z)
        else:
            run = lambda: eng.forward_frames(frames, 499, enc, kps, None, 2, f)
        run()
        recs.clear()
        run()
        torch.cuda.synchronize()
    finally:
        for n in names:
            setattr(ops, n, orig[n])
    uniq, count = {}, {}
    for n, sig, a, k in recs:
        count[(n, sig)] = count.get((n, sig), 0) + 1
        uniq.setdefault((n, sig), (a, k))
    rows = []
    for (n, sig), (a, k) in uniq.items():
        k = {kk: v for kk, v in k.items() if kk != "out"}
        orig[n](*a, **k)
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(8):
            orig[n](*a, **k)
        e1.record()
        torch.cuda.synchronize()
        rows.append((e0.elapsed_time(e1) / 8 * count[(n, sig)], count[(n, sig)], n, sig))
    tot = sum(r[0] for r in rows)
    lines = [f"per-op table of one {which} pass (isolated back-to-back timing): total {tot:.2f} ms"]
    for t, c, n, sig in sorted(rows, reverse=True)[:70]:
        lines.append(f"{t:8.3f} ms  n={c:3d}  avg={t / c * 1e3:8.1f} us  {n} {sig}")
    byop = {}
    for t, c, n, sig in rows:
        byop[n] = byop.get(n, 0.0) + t
    lines.append("by op: " + ", ".join(f"{k}={v:.2f}" for k, v in sorted(byop.items(), key=lambda kv: -kv[1])))
    sys.stderr.write("\n".join(lines) + "\n")


def kernel_roofline(pipe, host, L, h):
    """Time every launch of the dominant kernel (tcgen05 GEMM / implicit-GEMM conv) of ONE eager UNet forward with
    CUDA events on the launching stream; achieved = sum(2*M*N*K) / sum(duration)."""
    from vexpress_b200 import ops
    recs = []
    orig = dict(gemm=ops.gemm, gemm_ln=ops.gemm_ln, gemm_rowsums=ops.gemm_rowsums, gemm_lnparts=ops.gemm_lnparts, conv3x3=ops.conv3x3, flash_attention=ops.flash_attention,
                upconv3x3=ops.upconv3x3, conv3x3_s2=ops.conv3x3_s2, groupnorm=ops.groupnorm, layernorm=ops.layernorm)

    def timed(name, fn, flops_of):
        def w(*a, **k):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            out = fn(*a, **k)
            e1.record()
            recs.append((name, flops_of(a, k, out), e0, e1))
            return out
        return w

    def f_gemm(a, k, out):
        K = a[0].shape[1] + (k["a2"].shape[1] if k.get("a2") is not None else 0)
        return 2.0 * a[0].shape[0] * a[1].shape[0] * K

    def f_conv(a, k, out):
        nb, hh, ww, c = a[0].shape
        return 2.0 * nb * hh * ww * 9 * c * a[1].shape[0]

    def f_conv_s2(a, k, out):      # stride 2: a quarter of the output pixels
        nb, hh, ww, c = a[0].shape
        return 2.0 * nb * (hh // 2) * (ww // 2) * 9 * c * a[1].shape[0]

    def f_fa(a, k, out):
        q, heads, nq, nk = a[0], a[3], a[4], a[5]
        return 4.0 * q.shape[0] * nk * q.shape[1]

    def f_upconv(a, k, out):       # canonical FLOPs of conv3x3(upsample2x(x)): 9 taps at the upsampled resolution
        nb, hh, ww, c = a[0].shape
        return 2.0 * nb * 4 * hh * ww * 9 * c * (a[1].shape[0] // 4)

    def b_norm(a, k, out):         # algorithmic bytes of a normalisation: input once + output once
        x2 = k.get("x2")
        return 2.0 * (a[0].numel() + (x2.numel() if x2 is not None else 0)) + 2.0 * out.numel()

    ops.gemm = timed("gemm", orig["gemm"], f_gemm)
    ops.gemm_ln = timed("gemm", orig["gemm_ln"], f_gemm)     # LayerNorm -> Linear in one launch: the GEMM's FLOPs
    ops.gemm_rowsums = timed("gemm", orig["gemm_rowsums"], f_gemm)      # producer / consumer of the LayerNorm statistics
    ops.gemm_lnparts = timed("gemm", orig["gemm_lnparts"], f_gemm)      # hand-over: plain GEMM FLOPs
    ops.conv3x3 = timed("conv3x3", orig["conv3x3"], f_conv)
    ops.upconv3x3 = timed("conv3x3", orig["upconv3x3"], f_upconv)
    ops.conv3x3_s2 = timed("conv3x3", orig["conv3x3_s2"], f_conv_s2)
    ops.flash_attention = timed("flash", orig["flash_attention"], f_fa)
    ops.groupnorm = timed("groupnorm", orig["groupnorm"], b_norm)
    ops.layernorm = timed("layernorm", orig["layernorm"], b_norm)
    try:
        eng = pipe.denoising_unet.engine()
        f = min(L, 16)
        frames = host["lat"].cuda()[0, :, :f].permute(1, 0, 2, 3).repeat(2, 1, 1, 1).contiguous()
        enc = host["audio"].cuda()[:, :f].reshape(2 * f, 5, 768)
        kps = host["kps"].cuda()[:, :, :f].permute(0, 2, 3, 4, 1).reshape(2 * f * h * h, 320).contiguous()
        for it in range(2):                      # first pass warms caches / lazily packed state
            recs.clear()
            eng.forward_frames(frames, 499, enc, kps, None, 2, f)
            torch.cuda.synchronize()
    finally:
        for k_, v_ in orig.items():
            setattr(ops, k_, v_)
    agg = {}
    for name, fl, e0, e1 in recs:
        d = agg.setdefault(name, [0.0, 0.0, 0])
        d[0] += fl
        d[1] += e0.elapsed_time(e1) * 1e-3
        d[2] += 1
    out = {}
    for k, v in agg.items():
        if k in ("groupnorm", "layernorm"):
            out[k] = dict(algorithmic_gbs=v[0] / v[1] / 1e9, seconds=v[1], calls=v[2], algorithmic_bytes=v[0])
        else:
            out[k] = dict(tflops=v[0] / v[1] / 1e12, seconds=v[1], launches=v[2], flop=v[0])
    return out


def ncu_evidence():
    """Counters of the dominant kernel from THIS round's ncu capture of the same forward (profiles/r02_roofline.csv, made by
    profiles/tools/forward_once.py + roofline_merge.py): per-launch DRAM traffic next to the algorithmic bytes of the same
    launches, tensor-pipe activity, and the flash / GroupNorm rows."""
    import csv
    p = os.path.join(ROOT, "profiles", "r02_roofline.csv")
    if not os.path.exists(p):
        return None
    rows = [r for r in csv.DictReader(open(p)) if r["part"] == "unet"]
    f = lambda r, k: float(r[k]) if r.get(k) not in (None, "") else 0.0
    dom = [r for r in rows if r["kernel"].startswith("gemm_tcgen05_kernel") and r["op"] in ("gemm", "conv3x3", "conv3x3_s2", "upconv3x3")]
    n = sum(int(r["launches"]) for r in dom)
    if not n:
        return None
    us = sum(f(r, "us_total") for r in dom)
    ev = dict(source="profiles/r02_roofline.csv (ncu, cold caches, serialised)", launches=n,
              dram_bytes_per_launch=sum(f(r, "dram_mb_per_launch") * int(r["launches"]) for r in dom) / n * 1e6,
              algorithmic_bytes_per_launch=sum(f(r, "algorithmic_mb_per_launch") * int(r["launches"]) for r in dom) / n * 1e6,
              l2_bytes_per_launch=sum(f(r, "l2_mb_per_launch") * int(r["launches"]) for r in dom) / n * 1e6,
              tensor_pipe_active_pct=sum(f(r, "tensor_pipe_active_pct") * f(r, "us_total") for r in dom) / us)
    fl = [r for r in rows if r["op"] == "flash_attention"]
    if fl:
        uf = sum(f(r, "us_total") for r in fl)
        ev["flash_tensor_pipe_active_pct"] = sum(f(r, "tensor_pipe_active_pct") * f(r, "us_total") for r in fl) / uf
        ev["flash_l2_bytes_per_launch"] = sum(f(r, "l2_mb_per_launch") * int(r["launches"]) for r in fl) / sum(int(r["launches"]) for r in fl) * 1e6
    return ev


# --------------------------------------------------------------------------------------------- CPU arms
def cpu_sample(threads=None):
    """The reference algorithm on the host cores (oracle port, fp32 -- the reference cannot travel: it needs
    /root/reference + diffusers): one REAL pass of BASELINE configs[0] end to end -- 512x512, 4 latent frames, 2 DDIM steps,
    CFG 3.5: 2 full-width UNet forwards at b = 2 through `O.denoise` (context scheduler, CFG, overlap bookkeeping, DDIM)
    and the VAE decode of the 4 frames at 512x512 through `O.decode_latents`.  Returns run() -> (t_denoise, t_decode)."""
    from oracle import vx_oracle as O
    threads = threads or int(os.environ.get("VX_CPU_THREADS", 0)) or min(os.cpu_count(), 32)   # >32 threads scale negatively here
    torch.set_num_threads(threads)
    cfg, vcfg = O.DEFAULT_CFG, O.VAE_CFG
    g = torch.Generator().manual_seed(0)

    def synth(shapes):
        sd = {}
        for k, shp in shapes.items():
            if k.endswith("pos_encoder.pe"):
                sd[k] = O.positional_encoding(shp[2], shp[1])
            elif len(shp) == 1:
                sd[k] = (1.0 if ("norm" in k and k.endswith("weight")) else 0.0) + 0.02 * torch.randn(shp, generator=g)
            else:
                sd[k] = torch.randn(shp, generator=g) / math.sqrt(math.prod(shp[1:]))
        return sd
    sd = synth(O.unet_param_shapes(cfg))
    vsd = synth(O.vae_param_shapes(vcfg))
    lat, kps, audio, banks = O.synth_inputs(cfg, C1_FRAMES, 64, 64, True, 42)

    def run():
        """one full configs[0] pass: (t_denoise over C1_STEPS steps, t_decode of C1_FRAMES frames)"""
        with torch.no_grad():
            t0 = time.perf_counter()
            final = O.denoise(sd, cfg, lat, kps, audio, banks, C1_STEPS, 3.5, 24, 4, ref_w=0.95, audio_w=3.0)
            t1 = time.perf_counter()
            O.decode_latents(vsd, vcfg, final)
            t2 = time.perf_counter()
        return t1 - t0, t2 - t1

    def run_reduced():
        """one CFG denoise step of configs[0] + the decode of ONE frame, normalised to the units of run()"""
        with torch.no_grad():
            t0 = time.perf_counter()
            final = O.denoise(sd, cfg, lat, kps, audio, banks, 1, 3.5, 24, 4, ref_w=0.95, audio_w=3.0)
            t1 = time.perf_counter()
            O.decode_latents(vsd, vcfg, final[:, :, :1])
            t2 = time.perf_counter()
        return (t1 - t0) * C1_STEPS, (t2 - t1) * C1_FRAMES
    return run, run_reduced, threads


C1_FRAMES, C1_STEPS = 4, 2      # BASELINE configs[0], the reference's own CPU-runnable case


def reference_arm(args):
    """`--impl reference`: every step is one measured configs[0] pass on the host.  The line keeps OUR arm's metric
    (frames/s of the 25-step workload): the denoise time is scaled by 25 / 2 DDIM steps (per-frame cost of a step does not
    depend on the step index), the decode time is per frame -- `config.extrapolated_from` says so and `c1_measured` holds
    what was actually timed."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    run, run_reduced, threads = cpu_sample()
    # one COMPLETE configs[0] pass is always measured first (it is also the first warm-up).  If warm-up + timed steps of
    # that size would exceed the time budget (the driver runs --steps 20 --warmup 5: ~15 min of host time), the remaining
    # steps time half a pass each -- one CFG denoise step + one decoded frame -- and are scaled to the same units.
    c1_u, c1_v = run()
    budget = float(os.environ.get("VX_REF_BUDGET_S", 300))
    reduced = (args.steps + args.warmup) * (c1_u + c1_v) > budget
    step_fn = run_reduced if reduced else run
    for _ in range(max(args.warmup - 1, 0)):
        step_fn()
    if args.warmup == 0 and args.steps == 1:       # the cpu_baseline leg of our arm: that first complete pass IS the sample
        tu, tv, wall = c1_u, c1_v, c1_u + c1_v
    else:
        tu = tv = 0.0
        t0 = time.perf_counter()
        for _ in range(args.steps):
            a, b = step_fn()
            tu += a
            tv += b
        wall = time.perf_counter() - t0
        tu /= args.steps
        tv /= args.steps
    fps_c1 = C1_FRAMES / (tu + tv)
    fps = C1_FRAMES / (25.0 / C1_STEPS * tu + tv)
    what = ("one CFG denoise step of configs[0] + the VAE decode of one frame (x2 / x4 to the units of a pass)" if reduced else
            "one full BASELINE configs[0] pass")
    sample = (f"first a complete configs[0] pass on the host (512x512, {C1_FRAMES} frames, {C1_STEPS} DDIM steps, CFG 3.5, fp32): "
              f"denoise {c1_u:.2f}s + decode {c1_v:.2f}s; then per step: {what}: denoise {tu:.2f}s + decode {tv:.2f}s per pass = "
              f"{fps_c1:.4f} frames/s at configs[0]; 25-step figure = {C1_FRAMES}/(12.5*t_denoise + t_decode)")
    cfgw = workload_config(args.gpus)
    cfgw["extrapolated_from"] = (f"measured configs[0] pass ({C1_FRAMES} frames, {C1_STEPS} DDIM steps) scaled to 25 steps; a full "
                                 "configs[1] pass on the host takes ~30 min")
    line = dict(metric="frames_per_sec_512x512_25step", value=fps, unit="frames/s", n_gpus=args.gpus, steps=args.steps,
                warmup=args.warmup, ms_per_step=wall / args.steps * 1e3, higher_is_better=True, scaling="weak",
                vs_baseline=None, dtype="f32", data="synthetic", impl="reference", config=cfgw,
                c1_measured=dict(seconds_per_pass=c1_u + c1_v, denoise_s=c1_u, vae_decode_s=c1_v,
                                 frames_per_s=C1_FRAMES / (c1_u + c1_v), frames=C1_FRAMES, ddim_steps=C1_STEPS,
                                 timed_steps_use="half passes (1 denoise step + 1 frame decode)" if reduced else "full passes"),
                cpu_baseline=dict(value=fps, unit="frames/s", cores=threads, kind="port", sample=sample),
                e2e=dict(value=fps, unit="frames/s", h2d_bytes_per_step=0, d2h_bytes_per_step=0),
                unet_ms_per_step=tu / C1_STEPS * 1e3 * (16 / C1_FRAMES))
    print(json.dumps(line))


FRAMES_OVERRIDE = 0   # --frames L: the other BASELINE configs (96 = configs[2] on 1 GPU, 384 = configs[3] on 8); not the headline
LATENT = 64           # --size 768 -> 96 (configs[4])
DDIM_STEPS = 25       # --ddim-steps 50 (configs[4])


def workload_config(n):
    L = 16 if n == 1 else 8 * n + 8
    res = LATENT * 8
    base = dict(context_frames=16, context_overlap=8, num_inference_steps=DDIM_STEPS, guidance_scale=3.5,
                l2="inputs+weights per step (2.7 GB weights, >10 GB activations) far exceed the 126 MB L2; no flush needed",
                parallelism=f"windows-dp{n}")
    if FRAMES_OVERRIDE:
        L = FRAMES_OVERRIDE
        nw = (L - 16) // 8 + 1
        per = [len(range(r * (nw // n) + min(r, nw % n), (r + 1) * (nw // n) + min(r + 1, nw % n))) for r in range(n)]
        return dict(workload=f"{res}x{res}, {L} frames via context scheduler (window 16, overlap 8 -> {nw} windows"
                             + (f", sharded {'/'.join(map(str, per))} over {n} GPUs, NCCL all-reduce of the overlap noise-pred "
                                f"sums per step, VAE decode sharded by frame" if n > 1 else "")
                             + f"), {DDIM_STEPS} DDIM steps, CFG 3.5, bf16, {n} GPU" + ("s" if n > 1 else ""),
                    video_length=L, windows=nw, **base)
    if n == 1:
        name = ("BASELINE configs[1]: 512x512, single 16-frame context window, 25 DDIM steps, CFG 3.5, bf16"
                if (res, DDIM_STEPS) == (512, 25) else
                f"BASELINE configs[4]-style: {res}x{res}, single 16-frame context window, {DDIM_STEPS} DDIM steps, CFG 3.5, bf16")
        return dict(workload=name, video_length=L, windows=1, **base)
    return dict(workload=f"{res}x{res}, {L} frames = {n} context windows (window 16, overlap 8), one window per rank, "
                         f"{DDIM_STEPS} DDIM steps, CFG 3.5, bf16, NCCL all-reduce of overlap noise-pred per step, VAE decode "
                         f"sharded by frame", video_length=L, windows=n, **base)


# --------------------------------------------------------------------------------------------- our arm
def ours(args):
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    dist = world > 1
    if dist:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        torch.distributed.init_process_group("nccl", device_id=dev)
    n = world
    cfgw = workload_config(n)
    L, h, steps_ddim, gs = cfgw["video_length"], LATENT, DDIM_STEPS, 3.5
    from vexpress_b200 import _ffi
    pipe, host, banks = build_ours(L, h, dev)
    from vexpress_b200.modules import ReferenceAttentionControl
    from vexpress_b200.pipelines.v_express_pipeline import retrieve_timesteps
    reader = ReferenceAttentionControl(pipe.denoising_unet, do_classifier_free_guidance=True, mode="read",
                                       fusion_blocks="full", reference_attention_weight=0.95, audio_attention_weight=3.0)
    reader.update(pipe.reference_net.writer_view, True, dtype=torch.bfloat16)
    timesteps, _ = retrieve_timesteps(pipe.scheduler, steps_ddim, dev)
    kps_dev, audio_dev, lat_dev = host["kps"].to(dev), host["audio"].to(dev), host["lat"].to(dev)

    def barrier():
        if dist:
            torch.distributed.barrier()
        torch.cuda.synchronize()

    def resident_pass():
        lat = pipe.denoise(lat_dev.clone(), kps_dev, audio_dev, timesteps, gs, 16, 8, distributed=dist)
        return pipe_decode_device(pipe, lat, dist)

    def e2e_pass():
        return pipe(reference_image=None, kps_images=None, audio_waveform=None, width=8 * h, height=8 * h, video_length=L,
                    num_inference_steps=steps_ddim, guidance_scale=gs, context_frames=16, context_overlap=8,
                    reference_attention_weight=0.95, audio_attention_weight=3.0, do_multi_devices_inference=dist)

    def timed(fn, k):
        """-> (device seconds, wall seconds, launches, result of the last of the k calls)"""
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        l0 = _ffi.LAUNCHES
        out = None
        t0 = time.perf_counter()
        e0.record()
        for i in range(k):
            out = fn()
            if i + 1 < k:
                out = None          # release a step's result before the next step allocates its own
        e1.record()
        barrier()
        wall = time.perf_counter() - t0
        ms = max(e0.elapsed_time(e1), 0.0)
        t = torch.tensor([ms, wall * 1e3], device=dev)
        if dist:
            torch.distributed.all_reduce(t, op=torch.distributed.ReduceOp.MAX)
        return t[0].item() / 1e3, t[1].item() / 1e3, _ffi.LAUNCHES - l0, out

    for _ in range(args.warmup):
        resident_pass()
    with Clocks(local) as clk:
        sec, _, launches_direct, video = timed(resident_pass, args.steps)
    clocks = clk.summary()
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, video=video)
    del video
    if os.environ.get("VX_NCU_REGION"):
        # `ncu --profile-from-start off ... python bench.py`: exactly one more pass of the same timed workload
        torch.cuda.synchronize()
        torch.cuda.profiler.start()
        resident_pass()
        torch.cuda.synchronize()
        torch.cuda.profiler.stop()
    # UNet-only time per DDIM step (device events around the denoise loop)
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    pipe.denoise(lat_dev.clone(), kps_dev, audio_dev, timesteps, gs, 16, 8, distributed=dist)
    e1.record()
    torch.cuda.synchronize()
    unet_ms_per_step = e0.elapsed_time(e1) / steps_ddim
    # VAE decode alone (device events)
    lat_tmp = lat_dev.clone()
    pipe_decode_device(pipe, lat_tmp, dist)
    barrier()
    e0.record()
    pipe_decode_device(pipe, lat_tmp, dist)
    e1.record()
    torch.cuda.synchronize()
    vae_ms = e0.elapsed_time(e1)

    for _ in range(max(1, min(args.warmup, 1))):
        e2e_pass()
    _, e2e_wall, _, _ = timed(e2e_pass, args.steps)

    reader.update(pipe.reference_net.writer_view, True, dtype=torch.bfloat16)   # the pipeline call cleared the banks

    if rank == 0:
        pk = peaks()
        roof_k = kernel_roofline(pipe, host, L, h) if n == 1 else None
        if n == 1 and os.environ.get("VX_BENCH_OPS"):
            op_table(pipe, host, L, h, "unet")
            op_table(pipe, host, L, h, "vae")
        fps = L * args.steps / sec
        e2e_fps = L * args.steps / e2e_wall
        windows = cfgw["windows"]
        s768 = LATENT == 96      # canonical work per frame-eval / decoded frame at 768x768 (SURVEY.md 8d)
        work_tflop = steps_ddim * windows * 32 * (3.5616 if s768 else UNET_TFLOP_PER_FRAME_EVAL) \
            + L * (5.754 if s768 else VAE_TFLOP_PER_FRAME)
        line = dict(metric="frames_per_sec_512x512_25step", value=fps, unit="frames/s", n_gpus=n, steps=args.steps,
                    warmup=args.warmup, ms_per_step=sec / args.steps * 1e3, higher_is_better=True,
                    scaling="strong" if FRAMES_OVERRIDE else "weak",
                    vs_baseline=None, dtype="bf16", data="synthetic (random-init weights, dummy audio/kps/bank tensors)",
                    config=cfgw, clocks=clocks,
                    e2e=dict(value=e2e_fps, unit="frames/s",
                             h2d_bytes_per_step=int(sum(v.numel() * v.element_size() for v in host.values())),
                             d2h_bytes_per_step=int(L * 3 * (8 * h) * (8 * h) * 4)),
                    gpu_launches=int(launches_direct),
                    unet_ms_per_step=unet_ms_per_step, vae_decode_ms=vae_ms,
                    window_forwards_per_s=windows * steps_ddim * args.steps / sec,
                    # weak scaling gives every rank ONE 16-frame window at overlap 8: N windows cover 8N + 8 frames, so
                    # frames/s per GPU can reach at most (8N + 8) / (16 N) of the 1-GPU figure even with zero overhead
                    scaling_ceiling=(1.0 if (n == 1 or FRAMES_OVERRIDE) else (8 * n + 8) / (16.0 * n)),
                    whole_path=dict(tflop_per_pass=work_tflop, achieved_tflops=work_tflop * args.steps / sec / n,
                                    frac_of_sustained_peak=work_tflop * args.steps / sec / n / pk["tf_sustained"]))
        if n == 1 and os.environ.get("VX_BENCH_REFNET"):
            line["refnet_write_pass_ms"] = refnet_time(h)
        if roof_k:
            dom = dict(tflops=0.0, seconds=0.0, launches=0, flop=0.0)
            for k in ("gemm", "conv3x3"):
                if k in roof_k:
                    for kk in ("seconds", "launches", "flop"):
                        dom[kk] += roof_k[k][kk]
            ach = dom["flop"] / dom["seconds"] / 1e12
            ev = ncu_evidence() or {}
            fa = dict(roof_k.get("flash") or {})
            if fa:
                fa.update(bound="softmax instruction stream (MUFU ex2 16/clk/SM) -> tensor pipe <= 40 % at hd 40",
                          frac_of_sustained_tensor_peak=fa["tflops"] / pk["tf_sustained"],
                          tensor_pipe_active_pct=ev.get("flash_tensor_pipe_active_pct"))
            hbm = {}
            for k in ("groupnorm", "layernorm"):
                if k in roof_k:
                    hbm[k] = dict(bound="hbm", achieved=roof_k[k]["algorithmic_gbs"], peak=pk["hbm_gbs"], unit="GB/s",
                                  frac=roof_k[k]["algorithmic_gbs"] / pk["hbm_gbs"], seconds_per_forward=roof_k[k]["seconds"],
                                  calls_per_forward=roof_k[k]["calls"],
                                  algorithmic_bytes_per_forward=roof_k[k]["algorithmic_bytes"])
            line["roofline"] = dict(bound="tensor", kernel="gemm_tcgen05_kernel (GEMM + implicit-GEMM 3x3 conv)",
                                    achieved=ach, peak=pk["tf_sustained"], unit="TFLOP/s", frac=ach / pk["tf_sustained"],
                                    traffic=ev.get("dram_bytes_per_launch"),
                                    algorithmic_bytes=ev.get("algorithmic_bytes_per_launch"),
                                    l2_bytes=ev.get("l2_bytes_per_launch"),
                                    tensor_pipe_active_pct=ev.get("tensor_pipe_active_pct"), traffic_source=ev.get("source"),
                                    peak_source=pk["source"] + " (sustained cuBLAS bf16)",
                                    launches_per_forward=dom["launches"], seconds_per_forward=dom["seconds"],
                                    flash_attention=fa or None, **hbm)
        print(json.dumps(line))
    if dist:
        torch.distributed.destroy_process_group()


def refnet_time(h, iters=3):
    """VX_BENCH_REFNET=1 (not part of the headline metric): ReferenceNet write pass (SURVEY 8f-f1), full SD-1.5 width,
    one (1,4,h,h) reference latent at t = 0 with a zero text token, CUDA-event time per pass in ms."""
    from vexpress_b200.modules import ReferenceAttentionControl, UNet2DConditionModel
    with torch.device("cuda"):
        net = UNet2DConditionModel(cross_attention_dim=768)
    fill_synthetic_(net, 4321)
    net = net.to(torch.bfloat16)
    writer = ReferenceAttentionControl(net, do_classifier_free_guidance=True, mode="write", batch_size=1,
                                       fusion_blocks="full")
    x = torch.randn(1, 4, h, h, device="cuda").to(torch.bfloat16)
    enc = torch.zeros(1, 1, 768, device="cuda", dtype=torch.bfloat16)
    net(x, timestep=0, encoder_hidden_states=enc, return_dict=False)
    writer.clear()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(iters):
        net(x, timestep=0, encoder_hidden_states=enc, return_dict=False)
        writer.clear()
    e1.record()
    torch.cuda.synchronize()
    del net, writer
    torch.cuda.empty_cache()
    return e0.elapsed_time(e1) / iters


def pipe_decode_device(pipe, latents, dist):
    """Decode with the result left on the device (HBM-resident `value` measurement); rank 0 gathers the shards."""
    return pipe.decode_to_device(latents, dist)


DUMP_LIMIT_BYTES = 64 * 10 ** 6


def dump_outputs(path, **arrays):
    """--dump-outputs DIR: every array as DIR/<name>.npy in float32, so that two builds run with the same arguments
    (hence the same seeded inputs) can be compared output for output.  When the arrays exceed DUMP_LIMIT_BYTES in all,
    each is replaced by the same fixed, seeded sample of its flattened elements (drawn with replacement; the indices
    depend only on the element count, so runs with the same arguments sample the same positions)."""
    import numpy as np
    os.makedirs(path, exist_ok=True)
    total = sum(a.numel() for a in arrays.values())
    keep = (DUMP_LIMIT_BYTES - 4096 * len(arrays)) // 4          # float32 elements that fit, 4 KB per .npy header
    for name, a in arrays.items():
        shape, a = tuple(a.shape), a.detach().float()
        if total > keep:
            idx = torch.randint(a.numel(), (keep * a.numel() // total,), generator=torch.Generator().manual_seed(0))
            a = a.reshape(-1)[idx.to(a.device)]
        np.save(os.path.join(path, f"{name}.npy"), a.cpu().numpy())
        sys.stderr.write(f"bench.py: {name} {shape} -> {os.path.join(path, name)}.npy {tuple(a.shape)}\n")


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--frames", type=int, default=0, help="video length override (multiple of 8, >= 16): 96 = configs[2], 384 = configs[3]")
    ap.add_argument("--size", type=int, default=512, help="video side in pixels (512, or 768 = configs[4])")
    ap.add_argument("--ddim-steps", type=int, default=25)
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write the video of the last one to DIR/video.npy (float32, a seeded "
                         "sample when above 64 MB)")
    args = ap.parse_args()
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs applies to the CUDA arm only")
    global FRAMES_OVERRIDE, LATENT, DDIM_STEPS
    FRAMES_OVERRIDE, LATENT, DDIM_STEPS = args.frames, args.size // 8, args.ddim_steps
    if args.impl == "reference":
        reference_arm(args)
        return
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device (the product has no CPU path; use --impl reference for the CPU baseline)")
    ours_with_cpu_baseline(args)


def ours_with_cpu_baseline(args):
    # cpu_baseline is measured on rank 0 at N=1 in a subprocess (bounded sample) and merged into the line
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    cpu = None
    if rank == 0 and world == 1 and not os.environ.get("VX_BENCH_NO_CPU"):
        try:
            out = subprocess.run([sys.executable, os.path.abspath(__file__), "--impl", "reference", "--steps", "1",
                                  "--warmup", "0"], capture_output=True, text=True, timeout=900)
            cpu = json.loads(out.stdout.strip().splitlines()[-1])["cpu_baseline"]
        except Exception as e:  # the CPU leg must never take the GPU number down with it
            cpu = dict(value=None, unit="frames/s", cores=os.cpu_count(), kind="port", sample=f"failed: {e}")
    import io
    from contextlib import redirect_stdout
    buf = io.StringIO()
    with redirect_stdout(buf):
        ours(args)
    txt = buf.getvalue().strip()
    if rank == 0 and txt:
        line = json.loads(txt.splitlines()[-1])
        if cpu is not None:
            line["cpu_baseline"] = cpu
        print(json.dumps(line))


if __name__ == "__main__":
    main()
