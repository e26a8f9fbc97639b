"""Host-side logic and the C-ABI surface, no GPU: symbol export, product context scheduler vs reference golden,
parameter layout vs oracle, DDIM tables, window partition, 2-rank gloo check of the overlap all-reduce."""
import ctypes
import json
import os
import re
import sys

import numpy as np
import pytest
import torch

ROOT = os.path.abspath(os.path.join(os.path.dirname(__file__), ".."))


def test_library_exports_every_declared_symbol():
    from vexpress_b200 import _ffi
    lib = _ffi.lib()
    hdr = open(os.path.join(ROOT, "include", "vxb200.h")).read()
    syms = sorted(set(re.findall(r"\b(vx_[a-z0-9_]+)\s*\(", hdr)))
    assert len(syms) >= 24
    for s in syms:
        assert getattr(lib, s) is not None, s
    assert lib.vx_abi_version() == 1
    lib.vx_groupnorm_stats_ws_floats.restype = ctypes.c_int
    assert lib.vx_groupnorm_stats_ws_floats(4, 32, 8) == 4 * 32 * 8 * 3


def test_product_fails_loudly_without_gpu():
    """No CPU fallback: building the engine on a CPU box must raise, not silently compute."""
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    from vexpress_b200.modules import UNet3DConditionModel
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    from test_unet_gpu import UNET_EXTRA
    m = UNet3DConditionModel(block_out_channels=(64, 128, 256, 256), cross_attention_dim=768, **UNET_EXTRA)
    with pytest.raises(Exception):
        m(torch.zeros(2, 4, 2, 16, 16), 10, encoder_hidden_states=torch.zeros(4, 5, 768))


def test_product_context_scheduler_bit_exact(golden_dir):
    from vexpress_b200.pipelines import context as C
    g = json.load(open(os.path.join(golden_dir, "context_windows.json")))
    for c in g["pipeline_calls"]:
        wins, cnt = C.window_table(c["L"], c["S"], c["O"])
        assert wins == c["windows"] and cnt.tolist() == c["num_frame_context"], c
    for c in g["uniform_calls"]:
        assert list(C.uniform(c["step"], c["L"], c["S"], c["stride"], c["O"], c["closed"])) == c["windows"]
    for k, v in g["ordered_halving"].items():
        assert C.ordered_halving(int(k)) == v
    with pytest.raises(ValueError):
        C.get_context_scheduler("nope")
    assert C.compute_num_context(930, 24, 4) == 46 and C.compute_context_indices(2, 24, 4) == [(0, 23), (20, 43)]


def test_product_param_layout_matches_oracle_and_reference():
    from oracle import vx_oracle as O
    from vexpress_b200.modules.unet_3d import _unet_keys
    from vexpress_b200.modules.vae import _vae_keys
    assert _unet_keys((320, 640, 1280, 1280), 768, 2, 4, 4, 32) == O.unet_param_shapes(O.DEFAULT_CFG)
    assert _vae_keys((128, 256, 512, 512), 2, 4, 3) == O.vae_param_shapes(O.VAE_CFG)


def test_product_ddim_tables(golden_dir):
    from vexpress_b200.pipelines.scheduler import DDIMScheduler, ddim_coefficients
    from oracle import vx_oracle as O
    g = json.load(open(os.path.join(golden_dir, "ddim_kat.json")))
    s, o = DDIMScheduler(), O.DDIM()
    assert torch.equal(s.alphas_cumprod, o.alphas_cumprod)
    for n in (2, 25, 50):
        s.set_timesteps(n)
        assert s.timesteps.tolist() == g[f"timesteps_{n}"]
    s.set_timesteps(25)
    o.set_timesteps(25)
    for t in (999, 959, 39):
        sa, sb, sap, sbp = ddim_coefficients(s, t)
        a_t, a_p = o.coeffs(t)
        assert sa == float(a_t ** 0.5) and sbp == float((1 - a_p) ** 0.5)
    with pytest.raises(ValueError):
        DDIMScheduler(prediction_type="epsilon")


def test_unsupported_unet_config_is_rejected():
    from vexpress_b200.modules import UNet3DConditionModel
    with pytest.raises(ValueError):
        UNet3DConditionModel()                       # no motion modules / inflated groupnorm -> not this model
    with pytest.raises(ValueError):
        UNet3DConditionModel(mid_block_type="Other")


def test_partition_windows():
    from vexpress_b200.pipelines.v_express_pipeline import partition_windows
    parts = [partition_windows(47, 8, r) for r in range(8)]
    assert [len(p) for p in parts] == [6, 6, 6, 6, 6, 6, 6, 5]
    assert sum(parts, []) == list(range(47))
    assert partition_windows(1, 4, 0) == [0] and partition_windows(1, 4, 3) == []


def _gloo_worker(rank, world, port, L, S, Ov, ret):
    """Each rank scatters its windows' noise/count into a zero buffer, all-reduces, and must obtain bit-identically
    the single-process sequential sum (bf16 values, <= 2 contributions per frame)."""
    import torch.distributed as dist
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    from vexpress_b200.pipelines.context import window_table
    from vexpress_b200.pipelines.v_express_pipeline import partition_windows
    wins, cnt = window_table(L, S, Ov)
    g = torch.Generator().manual_seed(0)
    noise = [torch.randn(4, len(w), 16, generator=g).bfloat16() for w in wins]        # per-window predictions
    cntt = torch.from_numpy(cnt)
    acc = torch.zeros(4, L, 16)
    for wi in partition_windows(len(wins), world, rank):
        w = torch.tensor(wins[wi])
        v = (noise[wi] / cntt[w].to(torch.bfloat16)[None, :, None])
        acc[:, w] = (acc[:, w].bfloat16() + v).float()
    dist.all_reduce(acc)
    seq = [None] * L                                                                   # reference streaming order
    for wi, wn in enumerate(wins):
        v = noise[wi] / cntt[torch.tensor(wn)].to(torch.bfloat16)[None, :, None]
        for li, fi in enumerate(wn):
            seq[fi] = v[:, li].clone() if seq[fi] is None else seq[fi] + v[:, li]
    seq = torch.stack(seq, 1)
    ok = torch.equal(acc.bfloat16(), seq)
    if rank == 0:
        ret.put(bool(ok))
    dist.destroy_process_group()


def test_overlap_allreduce_bit_identical_two_ranks():
    import torch.multiprocessing as mp
    ctx = mp.get_context("spawn")
    ret = ctx.Queue()
    port = 29500 + (os.getpid() % 2000)
    procs = [ctx.Process(target=_gloo_worker, args=(r, 2, port, 40, 16, 8, ret)) for r in range(2)]
    for p in procs:
        p.start()
    for p in procs:
        p.join(120)
        assert p.exitcode == 0
    assert ret.get(timeout=5) is True


def test_refnet_layout_and_writer_pairing_cpu():
    """ReferenceNet mirror: reference state_dict layout, registration order (down, up, mid) and writer -> reader pairing
    of ``ReferenceAttentionControl.update`` (reference modules/mutual_self_attention.py:321-363) without any compute."""
    import torch
    from oracle import vx_oracle as O
    from vexpress_b200.modules import ReferenceAttentionControl, UNet2DConditionModel, UNet3DConditionModel
    from vexpress_b200.modules.unet_3d import attention_block_order
    cfg = O.small_cfg()
    net = UNet2DConditionModel(block_out_channels=cfg["block_out_channels"], cross_attention_dim=cfg["cross_attention_dim"])
    S = O.refnet_param_shapes(cfg)
    sd = net.state_dict()
    assert set(sd) == set(S) and all(tuple(sd[k].shape) == tuple(S[k]) for k in S)
    tops = [k.split(".")[0] for k in sd]
    assert tops.index("up_blocks") < tops.index("mid_block")          # the reference registers mid_block last
    with __import__("pytest").raises(ValueError):
        UNet2DConditionModel(use_linear_projection=True)
    writer = ReferenceAttentionControl(net, mode="write", fusion_blocks="full", do_classifier_free_guidance=True)
    assert net.write_banks
    blocks = net.writer_blocks()
    for i, b in enumerate(blocks):       # tag every bank with its dfs index
        c = b.norm1.normalized_shape[0]
        b.bank.append(torch.full((1, 4, c), float(i + 1)))
    unet = UNet3DConditionModel(
        block_out_channels=cfg["block_out_channels"], cross_attention_dim=cfg["cross_attention_dim"],
        use_inflated_groupnorm=True, use_motion_module=True, motion_module_mid_block=True, motion_module_type="Vanilla",
        motion_module_kwargs=dict(num_attention_heads=8, num_transformer_block=1,
                                  attention_block_types=["Temporal_Self", "Temporal_Self"],
                                  temporal_position_encoding=True, temporal_position_encoding_max_len=32,
                                  temporal_attention_dim_div=1))
    reader = ReferenceAttentionControl(unet, mode="read", fusion_blocks="full", do_classifier_free_guidance=True)
    reader.update(writer, True, dtype=torch.float32)
    mods = dict(unet.named_modules())
    names = attention_block_order(unet)
    assert [n.replace(".transformer_blocks.0", "") for n in names] == O.bank_order(cfg)
    # same-named blocks pair up: writer dfs index i -> reader block with the same module path
    from vexpress_b200.modules.unet_2d_condition import writer_block_names
    wnames = writer_block_names()
    for n in names:
        bank = mods[n].bank[0]
        assert bank.shape[0] == 2 and torch.count_nonzero(bank[0]).item() == 0
        assert bank[1, 0, 0].item() == float(wnames.index(n) + 1), n
    writer.clear()
    assert all(len(b.bank) == 0 for b in blocks)


def _cpu_engine(cls, model):
    """Engine object with the packed weights on the CPU (no kernels are called by packing)."""
    import torch
    from vexpress_b200.modules import unet_3d
    eng = object.__new__(cls)
    eng.model, eng.dev = model, torch.device("cpu")
    c = model.config
    eng.boc = tuple(c["block_out_channels"])
    eng.heads, eng.groups, eng.eps, eng.cross = model.heads, c["norm_num_groups"], float(c["norm_eps"]), c["cross_attention_dim"]
    eng.sd = {k: v.detach() for k, v in model.state_dict().items()}
    eng.W = {}
    eng._pack(eng.sd)
    if cls is unet_3d.UNetEngine:
        eng._pack_ln_fold()
    else:
        eng.ln_fold = eng.ln_fuse = False
    return eng


class _ShapeOps:
    """Stands in for vexpress_b200.ops: checks operand shapes like the real wrappers and returns empty outputs."""

    LN_GEMM_MAX_K = 512

    def __init__(self):
        self.calls = []

    def __getattr__(self, op):
        import torch

        def f(*a, **k):
            self.calls.append(op)
            if op == "row_stats":
                return torch.zeros(a[0].shape[0], 2)
            if op == "gemm_ln":
                x, wf, cs, bf, eps = a[:5]
                M, K = x.shape
                N = wf.shape[0]
                assert wf.shape[1] == K and cs.shape == (N,) and bf.shape == (N,) and eps == 1e-5
                assert K % 64 == 0 and K <= self.LN_GEMM_MAX_K
                if k.get("bias2") is not None:
                    assert k["bias2"].shape == (M // k["bias2_div"], N) and M % k["bias2_div"] == 0
                return torch.zeros(M, N // 2 if k.get("geglu") else N)
            if op == "gemm_lnfold":
                x, wf, st, cs, bf = a[:5]
                M, K = x.shape
                N = wf.shape[0]
                assert wf.shape[1] == K and st.shape == (M, 2) and cs.shape == (N,) and bf.shape == (N,)
                if k.get("bias2") is not None:
                    assert k["bias2"].shape == (M // k["bias2_div"], N) and M % k["bias2_div"] == 0
                return torch.zeros(M, N // 2 if k.get("geglu") else N)
            if op == "gemm":
                x, w = a[:2]
                K = x.shape[1] + (k["a2"].shape[1] if k.get("a2") is not None else 0)
                assert w.shape[1] == K, (x.shape, w.shape)
                return torch.zeros(x.shape[0], w.shape[0] // 2 if k.get("geglu") else w.shape[0])
            if op == "gemm_rowsums":
                x, w = a[:2]
                assert w.shape[1] == x.shape[1], (x.shape, w.shape)
                if k.get("residual") is not None:
                    assert k["residual"].shape == (x.shape[0], w.shape[0])
                return torch.zeros(x.shape[0], w.shape[0]), torch.zeros(2 * (w.shape[0] // 32), x.shape[0], 2), 4
            if op == "gemm_lnparts":
                x, wf, parts, nparts, cs, bf = a[:6]
                M, K = x.shape
                N = wf.shape[0]
                assert wf.shape[1] == K and parts.shape[1:] == (M, 2) and 0 < nparts <= parts.shape[0] and cs.shape == (N,) and bf.shape == (N,)
                if k.get("bias2") is not None:
                    assert k["bias2"].shape == (M // k["bias2_div"], N) and M % k["bias2_div"] == 0
                return torch.zeros(M, N // 2 if k.get("geglu") else N)
            if op == "layernorm":
                assert a[1].shape == (a[0].shape[1],)
                return torch.zeros_like(a[0])
            if op == "groupnorm":
                C = a[0].shape[1] + (k["x2"].shape[1] if k.get("x2") is not None else 0)
                assert a[0].shape[0] == a[1] * a[2] and a[3].shape == (C,), (a[0].shape, a[1], a[2], a[3].shape)
                return torch.zeros(a[0].shape[0], C)
            if op in ("flash_attention", "temporal_attention", "smallkv_attention"):
                return k["out"] if k.get("out") is not None else torch.zeros_like(a[0])
            if op == "conv_in":
                x, w, bias, cout = a[:4]
                NB, cin, H, W = x.shape
                assert w.shape == (cin * 9, cout) and bias.shape == (cout,)
                if k.get("addend") is not None:
                    assert k["addend"].shape[1] == cout
                return torch.zeros(NB * H * W, cout)
            if op == "conv3x3":
                x, w, bias = a[:3]
                NB, H, W, C = x.shape
                assert w.shape[1] == 9 * C and bias.shape == (w.shape[0],), (x.shape, w.shape)
                if k.get("residual") is not None:
                    assert k["residual"].shape == (NB * H * W, w.shape[0])
                if k.get("bias2") is not None:
                    assert k["bias2"].shape[1] == w.shape[0]
                return torch.zeros(NB * H * W, w.shape[0])
            if op == "im2col_s2":
                x, NB, H, W = a[:4]
                assert x.shape[0] == NB * H * W
                return torch.zeros(NB * (H // 2) * (W // 2), 9 * x.shape[1])
            if op == "downsample_conv":
                x, NB, H, W, w, bias = a[:6]
                assert x.shape[0] == NB * H * W and w.shape[1] == 9 * x.shape[1] and bias.shape == (w.shape[0],)
                assert H % 2 == 0 and W % 2 == 0
                return torch.zeros(NB * (H // 2) * (W // 2), w.shape[0])
            if op == "upsample2x":
                x, NB, H, W = a[:4]
                assert x.shape[0] == NB * H * W
                return torch.zeros(4 * x.shape[0], x.shape[1])
            if op == "upconv3x3":
                x, w4, bias = a[:3]
                NB, H, W, C = x.shape
                assert w4.shape[1] == 4 * C and w4.shape[0] % 4 == 0 and bias.shape == (w4.shape[0] // 4,), (x.shape, w4.shape)
                return torch.zeros(NB * 4 * H * W, w4.shape[0] // 4)
            if op == "conv_out_tc":
                x, NB, H, W = a[:4]
                assert x.shape[0] == NB * H * W and a[6].shape[0] == NB and a[6].shape[2:] == (H, W)
                return a[6]
            if op == "timestep_embed":
                return torch.zeros(a[0].shape[0], a[1])
            if op == "skinny_linear":
                x, w = a[:2]
                assert w.shape[1] == x.shape[1]
                return torch.zeros(x.shape[0], w.shape[0])
            raise AttributeError(op)
        return f


@pytest.mark.parametrize("fold,fuse", [("0", "0"), ("1", "0"), ("0", "1")])
def test_transformer_block_schedules_dry_run(monkeypatch, fold, fuse):
    """Host logic of UNetEngine._spatial / _motion with shape-checking fake ops, without touching a GPU: the three
    LayerNorm -> Linear schedules -- LayerNorm kernel + GEMM (VX_LN_FUSE=0), row_stats + gemm_lnfold (VX_LN_FOLD=1), and the
    statistics hand-over (VX_LN_FUSE=1): gemm_rowsums in the producer, gemm_lnparts in the consumer (incl. the
    positional-encoding bias of the motion modules)."""
    import torch
    from oracle import vx_oracle as O
    from vexpress_b200.modules import UNet3DConditionModel, unet_3d
    monkeypatch.setenv("VX_LN_FOLD", fold)
    monkeypatch.setenv("VX_LN_FUSE", fuse)
    cfg = O.small_cfg()
    m = UNet3DConditionModel(
        block_out_channels=cfg["block_out_channels"], cross_attention_dim=cfg["cross_attention_dim"],
        use_inflated_groupnorm=True, use_motion_module=True, motion_module_mid_block=True, motion_module_type="Vanilla",
        motion_module_kwargs=dict(num_attention_heads=8, num_transformer_block=1,
                                  attention_block_types=["Temporal_Self", "Temporal_Self"],
                                  temporal_position_encoding=True, temporal_position_encoding_max_len=32,
                                  temporal_attention_dim_div=1))
    m.load_state_dict(O.synth_state_dict(O.unet_param_shapes(cfg), 1234), strict=True)
    eng = _cpu_engine(unet_3d.UNetEngine, m.to(torch.bfloat16))
    assert eng.ln_fold == (fold == "1") and eng.ln_fuse == (fuse == "1") and len(eng.F) == (127 if "1" in (fold, fuse) else 0)
    fake = _ShapeOps()
    monkeypatch.setattr(unet_3d, "ops", fake)
    C, HW, f, b = 64, 256, 4, 2
    NB = b * f
    eng._bank_kv = lambda name, block: (torch.zeros(2 * HW, 2 * C), False)
    x = torch.zeros(NB * HW, C)
    enc = torch.zeros(NB * 5, cfg["cross_attention_dim"])
    assert eng._spatial("down_blocks.0.attentions.0", x, NB, HW, f, enc).shape == x.shape
    assert eng._motion("down_blocks.0.motion_modules.0", x, NB, HW, b, f).shape == x.shape
    n_ln = 7                                   # norm1, norm1_5, norm2, norm3 + norms.0, norms.1, ff_norm
    if fuse == "1":
        assert fake.calls.count("gemm_rowsums") == n_ln and fake.calls.count("gemm_lnparts") == n_ln
        assert not {"layernorm", "row_stats", "gemm_lnfold"} & set(fake.calls)
    elif fold == "1":
        assert fake.calls.count("row_stats") == n_ln and fake.calls.count("gemm_lnfold") == n_ln
        assert "layernorm" not in fake.calls
    else:
        assert fake.calls.count("layernorm") == n_ln and "gemm_lnfold" not in fake.calls


def test_fold_layernorm_algebra():
    """ops.fold_layernorm: rstd * (x @ wf.T - mean * colsum) + bf equals LayerNorm(x) @ w.T + b up to the bf16 rounding of
    the folded weights (same size as the reference path's rounding of LayerNorm(x) to bf16)."""
    import torch
    import torch.nn.functional as F
    from vexpress_b200 import ops
    torch.manual_seed(0)
    M, K, N = 64, 320, 960
    x = (torch.randn(M, K) * 2 + 0.5).bfloat16()
    w = (torch.randn(N, K) / K ** 0.5).bfloat16()
    b, g, be = torch.randn(N), 1 + 0.1 * torch.randn(K), 0.1 * torch.randn(K)
    wf, cs, bf = ops.fold_layernorm(w, b, g, be)
    xf = x.float()
    mean = xf.mean(1, keepdim=True)
    rstd = (xf.var(1, unbiased=False, keepdim=True) + 1e-5).rsqrt()
    out = rstd * (xf @ wf.float().t() - mean * cs[None]) + bf[None]
    ref = F.layer_norm(xf, (K,), g, be, 1e-5) @ w.float().t() + b
    assert ((out - ref).norm() / ref.norm()).item() < 3e-3
    wp, csp, bp = ops.fold_layernorm(w, b, g, be, geglu=True)          # packed row order is applied consistently
    w0, b0, _ = ops.pack_geglu(wf, bf)
    assert torch.equal(wp, w0) and torch.equal(bp, b0) and torch.allclose(csp, w0.float().sum(1))


def test_unet_and_refnet_forward_schedules_dry_run(monkeypatch):
    """Whole forward schedules (UNetEngine.forward_frames, RefNetEngine.forward) with shape-checking fake ops: every
    resnet / transformer / motion / down- and up-sampling step hands consistently shaped operands to the kernels, the skip
    stack empties, the ReferenceNet fills its 16 banks with (1, h*w, C) tensors."""
    import torch
    from oracle import vx_oracle as O
    from vexpress_b200.modules import ReferenceAttentionControl, UNet2DConditionModel, UNet3DConditionModel
    from vexpress_b200.modules import unet_2d_condition, unet_3d
    monkeypatch.delenv("VX_LN_FOLD", raising=False)
    cfg = O.small_cfg()
    m = UNet3DConditionModel(
        block_out_channels=cfg["block_out_channels"], cross_attention_dim=cfg["cross_attention_dim"],
        use_inflated_groupnorm=True, use_motion_module=True, motion_module_mid_block=True, motion_module_type="Vanilla",
        motion_module_kwargs=dict(num_attention_heads=8, num_transformer_block=1,
                                  attention_block_types=["Temporal_Self", "Temporal_Self"],
                                  temporal_position_encoding=True, temporal_position_encoding_max_len=32,
                                  temporal_attention_dim_div=1))
    m.load_state_dict(O.synth_state_dict(O.unet_param_shapes(cfg), 1234), strict=True)
    eng = _cpu_engine(unet_3d.UNetEngine, m.to(torch.bfloat16))
    net = UNet2DConditionModel(block_out_channels=cfg["block_out_channels"], cross_attention_dim=cfg["cross_attention_dim"])
    net.load_state_dict(O.synth_state_dict(O.refnet_param_shapes(cfg), 4321), strict=True)
    reng = _cpu_engine(unet_2d_condition.RefNetEngine, net.to(torch.bfloat16))
    fake = _ShapeOps()
    monkeypatch.setattr(unet_3d, "ops", fake)
    monkeypatch.setattr(unet_2d_condition, "ops", fake)
    b, f, h = 2, 4, 16
    eng._bank_kv = lambda name, block: (torch.zeros(2 * 4, 2 * eng.W[name + ".norm1.weight"].shape[0]), False)
    frames = torch.zeros(b * f, 4, h, h, dtype=torch.bfloat16)
    enc = torch.zeros(b * f, 5, cfg["cross_attention_dim"])
    kps = torch.zeros(b * f * h * h, cfg["block_out_channels"][0], dtype=torch.bfloat16)
    out = eng.forward_frames(frames, 499, enc, kps, None, b, f)
    assert out.shape == (b * f, 4, h, h)
    assert fake.calls.count("conv3x3") == 22 * 2 and fake.calls.count("upconv3x3") == 3 and fake.calls.count("flash_attention") == 32
    assert fake.calls.count("temporal_attention") == 42 and fake.calls.count("smallkv_attention") == 16
    fake.calls.clear()
    ReferenceAttentionControl(net, mode="write", fusion_blocks="full", do_classifier_free_guidance=True)
    rout = reng.forward(torch.zeros(1, 4, h, h, dtype=torch.bfloat16), 0, torch.zeros(1, 1, cfg["cross_attention_dim"]))
    assert rout.shape == (1, 4, h, h)
    assert fake.calls.count("flash_attention") == 16 and fake.calls.count("temporal_attention") == 0
    for name, blk in zip(unet_2d_condition.writer_block_names(), net.writer_blocks()):
        C = blk.norm1.normalized_shape[0]
        assert len(blk.bank) == 1 and blk.bank[0].shape[0] == 1 and blk.bank[0].shape[2] == C, name


class _EmuOps:
    """Functional CPU emulation (fp32 math, bf16 outputs) of the operators the prologue modules compose, with the kernels'
    layout conventions: conv_in's transposed fp32 weights, im2col's (tap, channel) K order, pack_geglu's tile layout."""

    def __init__(self):
        from vexpress_b200 import ops
        self.real = ops

    def __getattr__(self, name):           # pure-torch packers
        return getattr(self.real, name)

    @staticmethod
    def conv_in(x, w, bias, cout, addend=None, add_frame=None, out=None, **_):
        import torch.nn.functional as F
        n, cin, H, W = x.shape
        y = F.conv2d(x.float(), w.t().reshape(cout, cin, 3, 3), bias, padding=1)
        y = y.permute(0, 2, 3, 1).reshape(n * H * W, cout)
        if addend is not None:
            fr = torch.arange(n) if add_frame is None else add_frame.long()
            rows = (fr[:, None] * (H * W) + torch.arange(H * W)[None]).reshape(-1)
            y = y + addend.float()[rows]
        return y.to(torch.bfloat16)

    @staticmethod
    def im2col3x3(a, n, h, w, stride=1, silu=False, out=None):
        import torch.nn.functional as F
        C = a.shape[1]
        x = a.float().view(n, h, w, C).permute(0, 3, 1, 2)
        if silu:
            x = F.silu(x).to(torch.bfloat16).float()
        col = F.unfold(x, 3, padding=1, stride=stride)                       # (n, C*9, L), index c*9 + tap
        L = col.shape[-1]
        return col.view(n, C, 9, L).permute(0, 3, 2, 1).reshape(n * L, 9 * C).to(torch.bfloat16)

    def gemm(self, a, w, bias=None, *, a2=None, bias2=None, bias2_div=1, scale=1.0, residual=None, out=None,
             geglu=False, out_f32=False, **_):
        import torch.nn.functional as F
        af = a.float() if a2 is None else torch.cat([a.float(), a2.float()], 1)
        acc = af @ w.float().t()
        if bias is not None:
            acc = acc + bias
        if bias2 is not None:
            acc = acc + bias2[torch.arange(acc.shape[0]) // bias2_div]
        if geglu:
            bn = self.real.geglu_block_n(w.shape[0])
            t = acc.view(acc.shape[0], -1, 2, bn // 2)
            acc = (t[:, :, 0] * F.gelu(t[:, :, 1])).reshape(acc.shape[0], -1)
        acc = acc * scale
        if residual is not None:
            acc = acc + residual.float()
        return self._ret(acc if out_f32 else acc.to(torch.bfloat16), out)

    @staticmethod
    def layernorm(x, g, b, eps=1e-5, pe=None, rows_per_frame=0, out=None):
        import torch.nn.functional as F
        y = F.layer_norm(x.float(), (x.shape[1],), g, b, eps)
        if pe is not None:
            y = y + pe[(torch.arange(x.shape[0]) // rows_per_frame) % pe.shape[0]]
        return y.to(torch.bfloat16)

    @staticmethod
    def _ret(val, out):
        if out is not None:
            out.copy_(val.to(out.dtype))
            return out
        return val

    def flash_attention(self, q, k, v, heads, Nq, Nk, kv_div=1, out=None):
        import torch.nn.functional as F
        B, C = q.shape[0] // Nq, q.shape[1]
        Bkv = k.shape[0] // Nk
        qh = q.float().reshape(B, Nq, heads, C // heads).transpose(1, 2)
        idx = torch.arange(B) // kv_div
        kh = k.float().reshape(Bkv, Nk, heads, C // heads).transpose(1, 2)[idx]
        vh = v.float().reshape(Bkv, Nk, heads, C // heads).transpose(1, 2)[idx]
        o = F.scaled_dot_product_attention(qh, kh, vh)
        return self._ret(o.transpose(1, 2).reshape(B * Nq, C).to(torch.bfloat16), out)

    # ---- the remaining operators of the UNet / ReferenceNet schedules
    @staticmethod
    def timestep_embed(t, dim, out=None):
        import math
        half = dim // 2
        freq = torch.exp(-math.log(10000.0) * torch.arange(half, dtype=torch.float32) / half)
        a = t.float()[:, None] * freq[None]
        return torch.cat([torch.cos(a), torch.sin(a)], 1).to(torch.bfloat16).float()

    @staticmethod
    def skinny_linear(x, w, bias, act_in=False, act_out=False, out=None):
        import torch.nn.functional as F
        y = (F.silu(x) if act_in else x) @ w.float().t() + bias
        return F.silu(y) if act_out else y

    def conv3x3(self, x, w, bias=None, *, bias2=None, bias2_div=1, scale=1.0, residual=None, out=None, **_):
        import torch.nn.functional as F
        NB, H, W, C = x.shape
        w4 = w.float().view(w.shape[0], 3, 3, C).permute(0, 3, 1, 2)
        y = F.conv2d(x.float().permute(0, 3, 1, 2), w4, bias, padding=1).permute(0, 2, 3, 1).reshape(NB * H * W, -1)
        if bias2 is not None:
            y = y + bias2[torch.arange(y.shape[0]) // bias2_div]
        y = y * scale
        if residual is not None:
            y = y + residual.float()
        return self._ret(y.to(torch.bfloat16), out)

    def groupnorm(self, x1, NB, HW, gamma, beta, eps, silu, x2=None, groups=32, out=None, ws=None):
        import torch.nn.functional as F
        x = x1.float() if x2 is None else torch.cat([x1.float(), x2.float()], 1)
        C = x.shape[1]
        y = F.group_norm(x.view(NB, HW, C).transpose(1, 2), groups, gamma, beta, eps)
        if silu:
            y = F.silu(y)
        return self._ret(y.transpose(1, 2).reshape(NB * HW, C).to(torch.bfloat16), out)

    def temporal_attention(self, q, k, v, b, f, HW, heads, out=None):
        import torch.nn.functional as F
        C = q.shape[1]
        sp = lambda t: t.float().reshape(b, f, HW, heads, C // heads).permute(0, 2, 3, 1, 4)      # (b, hw, heads, f, hd)
        o = F.scaled_dot_product_attention(sp(q), sp(k), sp(v))
        return self._ret(o.permute(0, 3, 1, 2, 4).reshape(b * f * HW, C).to(torch.bfloat16), out)

    def smallkv_attention(self, q, k, v, rows_per_frame, heads, Lk, out=None):
        import torch.nn.functional as F
        C = q.shape[1]
        fr = q.shape[0] // rows_per_frame
        qh = q.float().reshape(fr, rows_per_frame, heads, C // heads).transpose(1, 2)
        kh = k.float().reshape(fr, Lk, heads, C // heads).transpose(1, 2)
        vh = v.float().reshape(fr, Lk, heads, C // heads).transpose(1, 2)
        o = F.scaled_dot_product_attention(qh, kh, vh)
        return self._ret(o.transpose(1, 2).reshape(q.shape[0], C).to(torch.bfloat16), out)

    def im2col_s2(self, x, NB, H, W, out=None):
        return self._ret(self.im2col3x3(x, NB, H, W, stride=2), out)

    def downsample_conv(self, x, NB, H, W, w, bias, pad_lo=1):
        assert pad_lo == 1            # the (0,1,0,1) variant belongs to the VAE encoder, which has GPU tests only
        return self.gemm(self.im2col3x3(x, NB, H, W, stride=2), w, bias)

    def upconv3x3(self, x, w4, bias, out=None, block_n=0):
        """conv3x3(upsample2x(x)) from the parity-folded weights (ops.pack_upconv_weight), like vx_upconv3x3_bf16."""
        import torch.nn.functional as F
        NB, H, W, C = x.shape
        Cout = w4.shape[0] // 4
        xp = F.pad(x.float().permute(0, 3, 1, 2), (1, 1, 1, 1))
        wv = w4.float().view(4, Cout, 4, C)
        y = torch.zeros(NB, Cout, 2 * H, 2 * W)
        for py in (0, 1):
            for px in (0, 1):
                acc = bias.view(1, -1, 1, 1).expand(NB, Cout, H, W).clone()
                for a in (0, 1):
                    for b in (0, 1):
                        acc = acc + torch.einsum("nchw,oc->nohw", xp[:, :, py + a:py + a + H, px + b:px + b + W],
                                                 wv[py * 2 + px][:, a * 2 + b, :])
                y[:, :, py::2, px::2] = acc
        return self._ret(y.permute(0, 2, 3, 1).reshape(NB * 4 * H * W, Cout).to(torch.bfloat16), out)

    def upsample2x(self, x, NB, H, W, out=None):
        C = x.shape[1]
        y = x.view(NB, H, 1, W, 1, C).expand(NB, H, 2, W, 2, C).reshape(NB * 4 * H * W, C)
        return self._ret(y.contiguous(), out)

    def conv_out_tc(self, x, NB, H, W, wp, bp, out, post=False):
        y = self.conv3x3(x.view(NB, H, W, -1), wp, bp).float()
        co = out.shape[1]
        out.copy_(y[:, :co].reshape(NB, H, W, co).permute(0, 3, 1, 2).to(out.dtype))
        return out

    @staticmethod
    def row_stats(x, eps=1e-5, out=None):
        xf = x.float()
        return torch.stack([xf.mean(1), (xf.var(1, unbiased=False) + eps).rsqrt()], 1)

    def gemm_lnfold(self, a, wf, stats, colsum, bias, *, bias2=None, bias2_div=1, scale=1.0, residual=None, out=None,
                    geglu=False):
        import torch.nn.functional as F
        acc = stats[:, 1:2] * (a.float() @ wf.float().t() - stats[:, 0:1] * colsum[None]) + bias
        if bias2 is not None:
            acc = acc + bias2[torch.arange(acc.shape[0]) // bias2_div]
        if geglu:
            bn = self.real.geglu_block_n(wf.shape[0])
            t = acc.view(acc.shape[0], -1, 2, bn // 2)
            acc = (t[:, :, 0] * F.gelu(t[:, :, 1])).reshape(acc.shape[0], -1)
        acc = acc * scale
        if residual is not None:
            acc = acc + residual.float()
        return self._ret(acc.to(torch.bfloat16), out)

    def gemm_rowsums(self, a, w, bias=None, *, a2=None, scale=1.0, residual=None, out=None):
        """vx_gemm_rowsums_bf16: the GEMM plus per-row partial (sum, sum of squares) of its ROUNDED outputs, here split over
        two slots (column halves) the way the kernel splits them over 2 * tiles_n."""
        o = self.gemm(a, w, bias, a2=a2, scale=scale, residual=residual, out=out)
        of = o.float()
        half = of.shape[1] // 2
        parts = torch.zeros(2 * ((of.shape[1] + 31) // 32), of.shape[0], 2)
        for j, blk in enumerate((of[:, :half], of[:, half:])):
            parts[j, :, 0] = blk.sum(1)
            parts[j, :, 1] = (blk * blk).sum(1)
        return o, parts, 2

    def gemm_lnparts(self, a, wf, parts, nparts, colsum, bias, eps=1e-5, **k):
        """vx_gemm_lnparts_bf16: mean / rstd from the partial sums (variance = E[x^2] - mean^2, fp32)."""
        K = a.shape[1]
        s1, s2 = parts[:nparts, :, 0].sum(0), parts[:nparts, :, 1].sum(0)
        mean = s1 / K
        rstd = ((s2 / K - mean * mean).clamp_min(0) + eps).rsqrt()
        return self.gemm_lnfold(a, wf, torch.stack([mean, rstd], 1), colsum, bias, **k)

    def gemm_ln(self, a, wf, colsum, bias, eps=1e-5, **k):
        """vx_gemm_ln_bf16: the statistics come from the same bf16 rows the GEMM multiplies (two-pass variance)."""
        assert a.shape[1] % 64 == 0 and a.shape[1] <= self.real.LN_GEMM_MAX_K
        return self.gemm_lnfold(a, wf, self.row_stats(a, eps), colsum, bias, **k)


import torch  # noqa: E402  (used by the emulation above)


def test_prologue_modules_compose_correctly(monkeypatch, golden_dir):
    """VKpsGuider / AudioProjection mirrors (SURVEY 8f-f2) with the kernels replaced by functional CPU emulations: the
    composition (channel padding to 32, conv_in weight transposition, im2col K order, stride pattern, GELU through the
    GEGLU epilogue, perceiver token concatenation) reproduces the reference-generated golden to bf16 accuracy."""
    from oracle import vx_oracle as O
    from vexpress_b200 import _ffi
    from vexpress_b200.modules import prologue
    monkeypatch.setattr(_ffi, "require_sm100", lambda: None)
    monkeypatch.setattr(prologue, "ops", _EmuOps())
    g = torch.load(os.path.join(golden_dir, "prologue_small.pt"), weights_only=False)
    rel = lambda a, b: ((a.float() - b.float()).norm() / b.float().norm()).item()
    k = g["kps"]
    m = prologue.VKpsGuider(320, block_out_channels=(16, 32, 96, 256))
    m.load_state_dict(O.synth_state_dict(O.kps_guider_param_shapes(O.KPS_CFG), k["seed_weights"]))
    m = m.to(torch.bfloat16)
    x = torch.rand(*k["shape"], generator=torch.Generator().manual_seed(k["seed_input"]))
    y = m(x, frames_per_chunk=1)
    assert y.shape == k["feature"].shape and rel(y, k["feature"]) < 2e-2, rel(y, k["feature"])
    a = g["audio_projection"]
    p = prologue.AudioProjection(dim=768, depth=4, dim_head=64, heads=12, num_queries=5, embedding_dim=768,
                                 output_dim=768, ff_mult=4, max_seq_len=10)
    p.load_state_dict(O.synth_state_dict(O.audio_projection_param_shapes(O.AUDIO_PROJ_CFG), a["seed_weights"]))
    p = p.to(torch.bfloat16)
    xa = torch.randn(*a["shape"], generator=torch.Generator().manual_seed(a["seed_input"]))
    ya = p(xa)
    assert ya.shape == a["tokens"].shape and rel(ya, a["tokens"]) < 2e-2, rel(ya, a["tokens"])


@pytest.mark.parametrize("fold,fuse", [("0", "0"), ("1", "0"), ("0", "1")])
def test_unet_engine_matches_oracle_with_emulated_kernels(monkeypatch, golden_dir, fold, fuse):
    """The whole UNetEngine.forward_frames host schedule (weight packing, split-K concat, time-embedding bias, banks,
    CFG uncond-half skip, GEGLU packing, ...) with every kernel replaced by a functional CPU emulation, against the
    oracle -- with the LayerNorm kernel, with VX_LN_FOLD=1 (LayerNorm folded into the GEMM epilogue, positional encoding
    as a per-frame bias) and with the default one-kernel LayerNorm GEMM."""
    from oracle import vx_oracle as O
    from vexpress_b200.modules import ReferenceAttentionControl, UNet3DConditionModel, unet_3d
    monkeypatch.setenv("VX_LN_FOLD", fold)
    monkeypatch.setenv("VX_LN_FUSE", fuse)
    cfg = O.small_cfg()
    m = UNet3DConditionModel(
        block_out_channels=cfg["block_out_channels"], cross_attention_dim=cfg["cross_attention_dim"],
        use_inflated_groupnorm=True, use_motion_module=True, motion_module_mid_block=True, motion_module_type="Vanilla",
        motion_module_kwargs=dict(num_attention_heads=8, num_transformer_block=1,
                                  attention_block_types=["Temporal_Self", "Temporal_Self"],
                                  temporal_position_encoding=True, temporal_position_encoding_max_len=32,
                                  temporal_attention_dim_div=1))
    sd = O.synth_state_dict(O.unet_param_shapes(cfg), 1234)
    m.load_state_dict(sd, strict=True)
    m = m.to(torch.bfloat16)
    f, h = 4, 16
    lat, kps, audio, banks = O.synth_inputs(cfg, f, h, h, True, 42)
    reader = ReferenceAttentionControl(m, do_classifier_free_guidance=True, mode="read", fusion_blocks="full",
                                       reference_attention_weight=0.95, audio_attention_weight=3.0)
    reader.update(type("W", (), {"banks": [b[1:] for b in banks]})(), True, dtype=torch.bfloat16)
    emu = _EmuOps()
    monkeypatch.setattr(unet_3d, "ops", emu)          # packing below and the forward both go through the emulation
    eng = _cpu_engine(unet_3d.UNetEngine, m)
    eng._bank_cache, eng._bank_buf, eng._bank_flag, eng.bank_epoch = {}, {}, {}, 0
    x = lat.repeat(2, 1, 1, 1, 1)
    frames = x.to(torch.bfloat16).permute(0, 2, 1, 3, 4).reshape(2 * f, 4, h, h).contiguous()
    kps_rows = kps.to(torch.bfloat16).permute(0, 2, 3, 4, 1).reshape(2 * f * h * h, -1).contiguous()
    enc = audio.reshape(-1, 5, cfg["cross_attention_dim"])
    out = eng.forward_frames(frames, 499, enc, kps_rows, None, 2, f)
    out = out.view(2, f, 4, h, h).permute(0, 2, 1, 3, 4).float()
    with torch.no_grad():
        ref = O.unet_forward(sd, cfg, x, 499, enc, kps, banks, 0.95, 3.0)
    err = ((out - ref).norm() / ref.norm()).item()
    print(f"emulated engine vs oracle (VX_LN_FOLD={fold}, VX_LN_FUSE={fuse}): rel-L2 {err:.3e}")
    assert err < 3e-2, err


def test_refnet_engine_matches_golden_with_emulated_kernels(monkeypatch, golden_dir):
    """RefNetEngine host schedule (write pass, SURVEY 8f-f1) on the functional CPU emulation against the golden produced by
    the reference's own UNet2D + write hooks."""
    from oracle import vx_oracle as O
    from vexpress_b200.modules import ReferenceAttentionControl, UNet2DConditionModel, unet_2d_condition, unet_3d
    g = torch.load(os.path.join(golden_dir, "refnet_small.pt"), weights_only=False)
    cfg = g["cfg"]
    net = UNet2DConditionModel(block_out_channels=cfg["block_out_channels"], cross_attention_dim=cfg["cross_attention_dim"])
    net.load_state_dict(O.synth_state_dict(O.refnet_param_shapes(cfg), g["seed_weights"]), strict=True)
    net = net.to(torch.bfloat16)
    emu = _EmuOps()
    monkeypatch.setattr(unet_3d, "ops", emu)
    monkeypatch.setattr(unet_2d_condition, "ops", emu)
    eng = _cpu_engine(unet_2d_condition.RefNetEngine, net)
    writer = ReferenceAttentionControl(net, mode="write", fusion_blocks="full", do_classifier_free_guidance=True)
    x = torch.randn(1, 4, g["h"], g["h"], generator=torch.Generator().manual_seed(g["seed_latents"]))
    out = eng.forward(x.to(torch.bfloat16), 0, torch.zeros(1, 1, cfg["cross_attention_dim"]))
    rel = lambda a, b: ((a.float() - b.float()).norm() / b.float().norm()).item()
    banks = ReferenceAttentionControl._writer_banks(writer)
    worst = max(rel(b[0], r) for b, r in zip(banks, g["banks"]))
    print(f"emulated refnet: banks worst rel-L2 {worst:.3e}, out {rel(out, g['out']):.3e}")
    assert worst < 3e-2 and rel(out, g["out"]) < 5e-2


def test_pipeline_prologue_glue_matches_reference(golden_dir):
    """prepare_audio_embeddings / prepare_kps_feature of the pipeline mirror (reference :350-407) with stub encoder,
    identity projection and a stub guider: windowing bit-equal to the golden produced by the reference method itself,
    CFG zero halves, 16-frame chunking of the guider."""
    from PIL import Image
    import numpy as np
    from vexpress_b200.pipelines.v_express_pipeline import VExpressPipeline
    g = torch.load(os.path.join(golden_dir, "prologue_small.pt"), weights_only=False)["audio_windows"]

    class Unet:
        device, dtype = torch.device("cpu"), torch.float32
    calls = []

    class Guider:
        def __call__(self, x):
            calls.append(x.shape[2])
            return x[:, :1].repeat(1, 5, 1, 1, 1)[..., ::8, ::8] * 2.0

    class Enc:
        def __call__(self, w):
            return type("R", (), {"last_hidden_state": w})()
    pipe = VExpressPipeline(vae=None, reference_net=None, denoising_unet=Unet(), v_kps_guider=Guider(),
                            audio_processor=None, audio_encoder=Enc(), audio_projection=lambda x: x, scheduler=None)
    emb = torch.randn(*g["shape"], generator=torch.Generator().manual_seed(g["seed_input"]))
    out = pipe.prepare_audio_embeddings(emb, g["video_length"], g["num_pad"], True)
    assert out.shape[0] == 2 and torch.count_nonzero(out[0]).item() == 0 and torch.equal(out[1], g["windows"])
    imgs = [Image.fromarray(np.full((64, 64, 3), i, dtype=np.uint8)) for i in range(20)]
    kf = pipe.prepare_kps_feature(imgs, 64, 64, True)
    assert calls == [16, 4] and kf.shape == (2, 5, 20, 8, 8) and torch.count_nonzero(kf[0]).item() == 0
    assert torch.allclose(kf[1, 0, :, 0, 0], torch.arange(20) / 255.0 * 2.0)
    with pytest.raises(ValueError):
        pipe.prepare_kps_feature(torch.zeros(1, 3, 2, 32, 32), 64, 64, False)


# ----------------------------------------------------------------------------------------------------------------------
# VExpressPipeline.denoise host logic (window partition, local kps/audio range, overlap plan incl. reflected windows,
# bf16 all-reduce, DDIM) with the UNet replaced by a cheap deterministic function and the two elementwise kernels by
# torch emulations with the kernels' rounding points -- against the oracle's restatement of the reference's streaming loop.
# ----------------------------------------------------------------------------------------------------------------------
def _fake_unet_core(x, kmean, emean, t):
    """x (b,f,4,h,w) fp32; kmean (b,f,1,h,w); emean (b,f,1,1,1) -> (b,f,4,h,w) bf16; mixes frames like the motion modules."""
    return torch.tanh(0.9 * x + kmean + 0.1 * emean + 0.05 * x.mean(1, keepdim=True) + 1e-3 * t).bfloat16()


class _FakeEngine:
    dev = torch.device("cpu")
    order = []

    def time_embedding(self, t):
        return torch.tensor([[float(t)]])

    def graph_signature(self):
        return 0

    def forward_frames(self, frames, timestep, enc, kps, kps_idx, b, f, temb=None, taps=None):
        NB, _, h, w = frames.shape
        k = kps.view(-1, h * w, kps.shape[1])[kps_idx.long()].float().mean(-1).view(b, f, 1, h, w)
        e = enc.float().mean((1, 2)).view(b, f, 1, 1, 1)
        out = _fake_unet_core(frames.float().view(b, f, 4, h, w), k, e, float(temb.reshape(-1)[0]))
        return out.view(NB, 4, h, w)


def _fake_unet_fn(x, t, aud, kps):
    """Same function in the oracle's layouts: x (b,4,f,h,w), aud ((b f),5,768), kps (b,C0,f,h,w)."""
    b, _, f, h, w = x.shape
    k = kps.float().permute(0, 2, 3, 4, 1).mean(-1).view(b, f, 1, h, w)
    e = aud.float().mean((1, 2)).view(b, f, 1, 1, 1)
    return _fake_unet_core(x.float().permute(0, 2, 1, 3, 4), k, e, float(t)).permute(0, 2, 1, 3, 4)


class _ElementwiseEmu:
    """torch emulation of vx_cfg_overlap_accumulate / vx_ddim_step with the kernels' rounding points (csrc/vx_misc.cu)."""

    @staticmethod
    def cfg_overlap_accumulate(noise, f, hw, L, do_cfg, win, count, guidance, acc):
        n = noise.view(-1, f, 4, hw).float()
        rb = lambda t: t.bfloat16().float()
        v = rb(n[0] + rb(guidance * rb(n[1] - n[0]))) if do_cfg else n[0]
        for i in range(f):
            fr = int(win[i])
            if fr < 0:
                continue
            acc[:, fr] = rb(acc[:, fr] + rb(v[i] / float(count[fr])))

    @staticmethod
    def ddim_step(lat, acc, sa, sb, sap, sbp):
        rb = lambda t: t.bfloat16().float()
        x, v = lat.float().view(acc.shape), rb(acc)
        x0 = rb(rb(sa * x) - rb(sb * v))
        eps = rb(rb(sa * v) + rb(sb * x))
        lat.copy_((rb(sap * x0) + rb(sbp * eps)).bfloat16().view(lat.shape))


def _fake_pipeline():
    from vexpress_b200.pipelines import v_express_pipeline as vp
    from vexpress_b200.pipelines.scheduler import DDIMScheduler
    unet = type("U", (), {"engine": lambda self: _FakeEngine(), "get_submodule": lambda self, n: None})()
    pipe = vp.VExpressPipeline(vae=None, reference_net=None, denoising_unet=unet, v_kps_guider=None, audio_processor=None,
                               audio_encoder=None, audio_projection=None, scheduler=DDIMScheduler())
    pipe.use_cuda_graph = False
    vp.ops = _ElementwiseEmu()
    return pipe, vp


def _fake_inputs(L, h=4, C0=8):
    g = torch.Generator().manual_seed(L)
    lat = torch.randn(1, 4, L, h, h, generator=g).bfloat16()
    kps = torch.cat([torch.zeros(1, C0, L, h, h), 0.1 * torch.randn(1, C0, L, h, h, generator=g)]).bfloat16()
    audio = torch.cat([torch.zeros(1, L, 5, 16), torch.randn(1, L, 5, 16, generator=g)]).bfloat16()
    return lat, kps, audio


def _run_fake_denoise(L, S, Ov, steps, distributed=False):
    from vexpress_b200.pipelines.v_express_pipeline import retrieve_timesteps
    pipe, vp = _fake_pipeline()
    try:
        lat, kps, audio = _fake_inputs(L)
        ts, _ = retrieve_timesteps(pipe.scheduler, steps, None)
        return pipe.denoise(lat.clone(), kps, audio, ts, 3.5, S, Ov, distributed=distributed)
    finally:
        from vexpress_b200 import ops as real_ops
        vp.ops = real_ops


@pytest.mark.parametrize("L,S,Ov", [(12, 8, 4), (24, 16, 8), (20, 16, 4), (28, 16, 8), (33, 24, 4)])
def test_denoise_host_logic_equals_reference_streaming_loop(monkeypatch, L, S, Ov):
    """Tiling AND non-tiling lengths (reflected tail windows with repeated frames, SURVEY Appendix D): bit-identical to
    the oracle's restatement of pipelines/v_express_pipeline.py:527-572 in bf16."""
    from oracle import vx_oracle as O
    out = _run_fake_denoise(L, S, Ov, 3)
    lat, kps, audio = _fake_inputs(L)

    def step_cuda_semantics(self, model_output, timestep, sample, eta=0.0, **_):
        """O.DDIM.step with the scalar handling of the device the reference runs on: CUDA elementwise kernels keep the
        fp32 scalar in fp32 (opmath) and round the product to bf16, whereas CPU eager first rounds the SCALAR to bf16."""
        a_t, a_prev = self.coeffs(int(timestep))
        rb = lambda t: t.bfloat16().float()
        x, v = sample.float(), model_output.float()
        sa, sb, sap, sbp = float(a_t ** 0.5), float((1 - a_t) ** 0.5), float(a_prev ** 0.5), float((1 - a_prev) ** 0.5)
        x0 = rb(rb(sa * x) - rb(sb * v))
        eps = rb(rb(sa * v) + rb(sb * x))
        return O._StepOut((rb(sap * x0) + rb(sbp * eps)).bfloat16())
    monkeypatch.setattr(O.DDIM, "step", step_cuda_semantics)
    ref = O.denoise(None, None, lat, kps, audio, None, 3, 3.5, S, Ov, unet_fn=_fake_unet_fn)
    assert out.dtype == torch.bfloat16 and torch.equal(out, ref)


def _gloo_denoise_worker(rank, world, port, L, S, Ov, ret):
    import torch.distributed as dist
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    out = _run_fake_denoise(L, S, Ov, 3, distributed=True)
    if rank == 0:
        ret.put(out.float().numpy())
    dist.destroy_process_group()


@pytest.mark.parametrize("L,S,Ov,world", [(40, 16, 8, 2), (28, 16, 8, 2), (56, 16, 8, 3)])
def test_denoise_sharded_over_ranks_equals_single_rank(L, S, Ov, world):
    """VExpressPipeline.denoise(distributed=True) itself under gloo: rank-local kps/audio slices, bf16 all-reduce of the
    overlap sums, replicated DDIM -- bit-identical to the one-rank run (and therefore to the reference's streaming loop)."""
    import torch.multiprocessing as mp
    ctx = mp.get_context("spawn")
    ret = ctx.Queue()
    port = 29500 + ((os.getpid() * 7 + L) % 2000)
    procs = [ctx.Process(target=_gloo_denoise_worker, args=(r, world, port, L, S, Ov, ret)) for r in range(world)]
    for p in procs:
        p.start()
    got = torch.from_numpy(ret.get(timeout=120))
    for p in procs:
        p.join(120)
        assert p.exitcode == 0
    single = _run_fake_denoise(L, S, Ov, 3)
    assert torch.equal(got, single.float())


# ----------------------------------------------------------------------------------------------------------------------
# Drop-in boundary: the mirrored entry points keep the reference's parameter names, order and defaults, as read from the
# reference's sources by oracle/gen_golden.py:gen_signatures into tests/golden/reference_signatures.json.
# ----------------------------------------------------------------------------------------------------------------------
_BOUNDARY = [  # (reference file, class, function, product object path)
    ("pipelines/v_express_pipeline.py", "VExpressPipeline", "__call__", "vexpress_b200.pipelines.v_express_pipeline:VExpressPipeline.__call__"),
    ("pipelines/v_express_pipeline.py", "VExpressPipeline", "mean_overlap", "vexpress_b200.pipelines.v_express_pipeline:VExpressPipeline.mean_overlap"),
    ("pipelines/v_express_pipeline.py", "VExpressPipeline", "__init__", "vexpress_b200.pipelines.v_express_pipeline:VExpressPipeline.__init__"),
    ("pipelines/v_express_pipeline.py", "VExpressPipeline", "prepare_reference_latent", "vexpress_b200.pipelines.v_express_pipeline:VExpressPipeline.prepare_reference_latent"),
    ("pipelines/v_express_pipeline.py", "VExpressPipeline", "prepare_kps_feature", "vexpress_b200.pipelines.v_express_pipeline:VExpressPipeline.prepare_kps_feature"),
    ("pipelines/v_express_pipeline.py", "VExpressPipeline", "prepare_audio_embeddings", "vexpress_b200.pipelines.v_express_pipeline:VExpressPipeline.prepare_audio_embeddings"),
    ("modules/unet_3d.py", "UNet3DConditionModel", "forward", "vexpress_b200.modules.unet_3d:UNet3DConditionModel.forward"),
    ("modules/unet_3d.py", "UNet3DConditionModel", "from_config_2d", "vexpress_b200.modules.unet_3d:UNet3DConditionModel.from_config_2d"),
    ("modules/unet_3d.py", "UNet3DConditionModel", "__init__", "vexpress_b200.modules.unet_3d:UNet3DConditionModel.__init__"),
    ("modules/mutual_self_attention.py", "ReferenceAttentionControl", "__init__", "vexpress_b200.modules.mutual_self_attention:ReferenceAttentionControl.__init__"),
    ("modules/mutual_self_attention.py", "ReferenceAttentionControl", "update", "vexpress_b200.modules.mutual_self_attention:ReferenceAttentionControl.update"),
    ("modules/mutual_self_attention.py", "ReferenceAttentionControl", "clear", "vexpress_b200.modules.mutual_self_attention:ReferenceAttentionControl.clear"),
    ("pipelines/context.py", None, "uniform", "vexpress_b200.pipelines.context:uniform"),
    ("pipelines/context.py", None, "get_context_scheduler", "vexpress_b200.pipelines.context:get_context_scheduler"),
    ("pipelines/context.py", None, "ordered_halving", "vexpress_b200.pipelines.context:ordered_halving"),
]


def _reference_signature(golden_dir, ref_file, cls, fn):
    """[(name, default source or '<required>')] of a reference entry point, from the stored golden."""
    sigs = json.load(open(os.path.join(golden_dir, "reference_signatures.json")))
    entry = next(s for s in sigs if (s["file"], s["cls"], s["fn"]) == (ref_file, cls, fn))
    return [tuple(p) for p in entry["params"]]


def _product_signature(spec):
    import importlib
    import inspect
    mod, path = spec.split(":")
    obj = importlib.import_module(mod)
    for part in path.split("."):
        obj = getattr(obj, part)
    out = []
    for name, p in inspect.signature(obj).parameters.items():
        if p.kind == p.VAR_KEYWORD:
            out.append(("**" + name, ""))
        elif p.default is p.empty:
            out.append((name, "<required>"))
        else:
            out.append((name, p.default))
    return out


def _same_default(ref_src, val):
    if ref_src == "<required>" or val == "<required>":
        return ref_src == val
    try:
        import ast
        ref_val = ast.literal_eval(ref_src)
    except Exception:
        if ref_src == "float('inf')":
            return val == float("inf")
        return ref_src.replace("torch.", "") in repr(val) or ref_src == "..."      # e.g. torch.float16, Ellipsis defaults
    if isinstance(ref_val, (list, tuple)) and isinstance(val, (list, tuple)):
        return list(ref_val) == list(val)
    if ref_val == {} and val is None:
        return True          # a mutable `{}` default of the reference is an immutable None here (same meaning)
    return ref_val == val


@pytest.mark.parametrize("ref_file,cls,fn,spec", _BOUNDARY)
def test_boundary_signatures_match_reference(golden_dir, ref_file, cls, fn, spec):
    ref = _reference_signature(golden_dir, ref_file, cls, fn)
    ours = _product_signature(spec)
    if cls is not None:
        ref = [r for r in ref if r[0] not in ("self", "cls")]
        ours = [o for o in ours if o[0] not in ("self", "cls")]
    ref_names = [n for n, _ in ref if not n.startswith("**")]
    our_names = [n for n, _ in ours if not n.startswith("**")]
    # every reference parameter exists, in the same order (the product may append optional extras at the end)
    assert our_names[:len(ref_names)] == ref_names, (fn, ref_names, our_names)
    for (n, d_ref), (_, d_our) in zip(ref, ours):
        if n.startswith("**"):
            continue
        assert _same_default(d_ref, d_our), (fn, n, d_ref, d_our)
    for n, d in ours[len(ref):]:
        assert n.startswith("**") or d != "<required>", f"{fn}: extra parameter {n} must be optional"


def test_downsample_conv_dispatch(monkeypatch):
    """ops.downsample_conv: stride-2 convs go to the TMA traversal-stride kernel when the channel count allows 64-wide K
    blocks, otherwise (and under VX_CONV_S2=0) to the gathered im2col + GEMM path, with the padding variant passed on."""
    from vexpress_b200 import ops
    calls = []
    monkeypatch.setattr(ops, "conv3x3_s2", lambda x, w, b, pad_lo=1: calls.append(("s2", tuple(x.shape), pad_lo)) or "s2")
    monkeypatch.setattr(ops, "im2col_s2", lambda x, NB, H, W: calls.append(("im2col_s2", tuple(x.shape))) or "col")
    monkeypatch.setattr(ops, "im2col3x3", lambda x, NB, H, W, stride=1, pad_lo=1: calls.append(("im2col3x3", stride, pad_lo)) or "col")
    monkeypatch.setattr(ops, "gemm", lambda col, w, b: calls.append(("gemm", col)) or "gemm")
    x = torch.zeros(2 * 8 * 8, 128)
    monkeypatch.setattr(ops, "CONV_S2_TMA", True)
    assert ops.downsample_conv(x, 2, 8, 8, "w", "b") == "s2" and calls[-1] == ("s2", (2, 8, 8, 128), 1)
    assert ops.downsample_conv(x, 2, 8, 8, "w", "b", pad_lo=0) == "s2" and calls[-1] == ("s2", (2, 8, 8, 128), 0)
    x32 = torch.zeros(2 * 8 * 8, 32)                       # C % 64 != 0: gathered path
    calls.clear()
    assert ops.downsample_conv(x32, 2, 8, 8, "w", "b") == "gemm" and [c[0] for c in calls] == ["im2col_s2", "gemm"]
    calls.clear()
    assert ops.downsample_conv(x32, 2, 8, 8, "w", "b", pad_lo=0) == "gemm" and calls[0] == ("im2col3x3", 2, 0)
    monkeypatch.setattr(ops, "CONV_S2_TMA", False)          # A/B switch off
    calls.clear()
    assert ops.downsample_conv(x, 2, 8, 8, "w", "b") == "gemm" and calls[0][0] == "im2col_s2"


def test_rowsum_slot_capacity():
    """The producer GEMM of the LayerNorm statistics hand-over writes 2 * ceil(N / block_n) partials per row with
    block_n >= 32: ops.rowsum_slots must cover the narrowest tile the library may pick."""
    from vexpress_b200 import ops
    for N in (64, 320, 640, 1280, 96):
        assert ops.rowsum_slots(N) == 2 * -(-N // 32)
        for bn in (32, 64, 96, 128, 160, 192, 256):
            if N % bn == 0:
                assert 2 * (N // bn) <= ops.rowsum_slots(N)
