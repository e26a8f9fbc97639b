"""Programmatic dependent launch (csrc/vx_host.h launch_k, vx_ptx.cuh pdl_wait / pdl_trigger) must not change a bit:
every kernel runs `griddepcontrol.wait` before its first global access, so launching the successor early only overlaps
launch latency and prologues.  The same pipeline call (eager, then captured in a CUDA graph: the launches become
programmatic edges of the graph) with the switch on and off has to produce identical videos; an operator chain with
deliberately tiny kernels (which leaves the largest window for a missing wait to show) is repeated many times."""
import os

import pytest
import torch

pytestmark = pytest.mark.gpu


def _set_pdl(on):
    from vexpress_b200 import _ffi
    lib = _ffi.lib()
    lib.vx_pdl_set(1 if on else 0)
    assert lib.vx_pdl_get() == (1 if on else 0)


@pytest.fixture
def restore_pdl():
    from vexpress_b200 import _ffi
    before = _ffi.lib().vx_pdl_get()
    yield
    _ffi.lib().vx_pdl_set(before)


def test_op_chain_bit_identical_with_pdl(restore_pdl):
    from vexpress_b200 import ops
    g = torch.Generator().manual_seed(3)
    NB, H, C, heads = 4, 16, 320, 8
    HW = H * H
    x = (torch.randn(NB * HW, C, generator=g)).bfloat16().cuda()
    w3 = ops.pack_conv3x3_weight(torch.randn(C, C, 3, 3, generator=g) / (9 * C) ** 0.5).bfloat16().cuda()
    wq = (torch.randn(3 * C, C, generator=g) / C ** 0.5).bfloat16().cuda()
    wo = (torch.randn(C, C, generator=g) / C ** 0.5).bfloat16().cuda()
    gam, bet = torch.ones(C).cuda(), torch.zeros(C).cuda()
    bias = (0.1 * torch.randn(C, generator=g)).cuda()

    def chain():
        h = ops.groupnorm(x, NB, HW, gam, bet, 1e-5, True)
        h = ops.conv3x3(h.view(NB, H, H, C), w3, bias, residual=x)
        n = ops.layernorm(h, gam, bet, 1e-5)
        qkv = ops.gemm(n, wq)
        a = ops.flash_attention(qkv[:, :C], qkv[:, C:2 * C], qkv[:, 2 * C:], heads, HW, HW)
        return ops.gemm(a, wo, bias, residual=h)

    _set_pdl(False)
    ref = chain().clone()
    torch.cuda.synchronize()
    _set_pdl(True)
    for it in range(25):
        out = chain()
        assert torch.equal(out, ref), f"iteration {it}: PDL changed the result"
    # the same chain captured in a CUDA graph: programmatic edges
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        chain()
    torch.cuda.current_stream().wait_stream(side)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        gout = chain()
    for it in range(10):
        gout.zero_()
        graph.replay()
        torch.cuda.synchronize()
        assert torch.equal(gout, ref), f"graph replay {it}: PDL changed the result"


@pytest.mark.parametrize("use_graph", [False, True])
def test_pipeline_bit_identical_with_pdl(golden_dir, use_graph, restore_pdl):
    from oracle import vx_oracle as O
    from test_pipeline_gpu import build_pipeline
    g = torch.load(os.path.join(golden_dir, "pipeline_small.pt"), weights_only=False)
    cfg, vcfg = g["cfg"], g["vae_cfg"]
    sd = O.synth_state_dict(O.unet_param_shapes(cfg), 1234)
    vsd = O.synth_state_dict(O.vae_param_shapes(vcfg), 1235)
    lat, kps, audio, banks = O.synth_inputs(cfg, g["L"], g["h"], g["h"], True, 42)
    videos = []
    for on in (False, True):
        _set_pdl(on)
        pipe = build_pipeline(cfg, vcfg, sd, vsd, kps, audio, [b[1:] for b in banks], lat)
        pipe.use_cuda_graph = use_graph
        videos.append(pipe(reference_image=None, kps_images=None, audio_waveform=None, width=g["h"] * 8, height=g["h"] * 8,
                           video_length=g["L"], num_inference_steps=g["steps"], guidance_scale=g["guidance_scale"],
                           context_frames=g["S"], context_overlap=g["O"], reference_attention_weight=0.95,
                           audio_attention_weight=3.0))
    assert torch.equal(videos[0], videos[1])
    d = (videos[1].flatten()[::g["sample_stride"]] - g["video"].float()).abs().mean().item()
    assert d < 1.5e-2, d
