"""GPU: the torch-free kernel self-tests (every GEMM epilogue / A-operand mode and every
attention mode against naive CUDA-core references, called through the C-ABI) plus edge-case
parity of the whole path against the fp32 oracle: ragged triangle counts, padding inside the
batch, several scenes per call, single views, other resolutions, the full-attention (V1-Base
style) decoder."""
import os
import subprocess

import pytest
import torch

from renderformer_b200.config import RenderFormerConfig
from renderformer_b200.metrics import PSNR_MIN, REL_TOL, hdr_rel_err, log_psnr
from renderformer_b200.synth import init_state_dict, make_scene

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.mark.parametrize("binary,env", [
    ("selftest_gemm", {}),
    ("selftest_gemm", {"RFB_TEST_F16": "1"}),                       # fp16 16-bit side outputs of the fused epilogues
    ("selftest_attn", {}),                       # kernel generation picked per shape
    ("selftest_attn", {"RFB_ATTN_GEN": "2"}),    # two query tiles per CTA
    ("selftest_attn", {"RFB_ATTN_GEN": "3"}),    # one query tile per CTA, Q in TMEM
    ("selftest_attn", {"RFB_TEST_F16": "1"}),                       # fp16 operands, kernel picked per shape
    ("selftest_attn", {"RFB_TEST_F16": "1", "RFB_ATTN_GEN": "2"}),
    ("selftest_attn", {"RFB_TEST_F16": "1", "RFB_ATTN_GEN": "3"}),
])
def test_kernel_selftests(binary, env):
    exe = os.path.join(ROOT, "renderformer_b200", binary)
    assert os.path.exists(exe), f"{exe} missing: run __graft_entry__.build()"
    r = subprocess.run([exe, "check"], capture_output=True, text=True, timeout=600, env={**os.environ, **env})
    tail = "\n".join(r.stdout.splitlines()[-15:])
    assert r.returncode == 0, tail + r.stderr[-2000:]
    assert "0 failure(s)" in r.stdout, tail
    assert "[FAIL]" not in r.stdout


@pytest.mark.parametrize("f16", ["0", "1"])
def test_dense_attention_kernels_bit_identical(f16):
    """attn2_tc_kernel and attn3_tc_kernel produce the same output bytes for every selftest_attn case: the
    kernel is picked from the grid shape, so a sharded render may run a row on the other kernel than a
    single-GPU render of the same job."""
    exe = os.path.join(ROOT, "renderformer_b200", "selftest_attn")
    assert os.path.exists(exe), f"{exe} missing: run __graft_entry__.build()"
    hashes = {}
    for gen in ("2", "3"):
        r = subprocess.run([exe, "check"], capture_output=True, text=True, timeout=600,
                           env={**os.environ, "RFB_TEST_F16": f16, "RFB_ATTN_GEN": gen})
        assert r.returncode == 0, "\n".join(r.stdout.splitlines()[-15:]) + r.stderr[-2000:]
        hashes[gen] = [line for line in r.stdout.splitlines() if line.startswith("[HASH] ")]
    assert hashes["2"], "selftest_attn printed no [HASH] lines"
    assert hashes["2"] == hashes["3"]


def _pipe(cfg, seed):
    from renderformer_b200.model import RenderFormer, RenderFormerRenderingPipeline
    model = RenderFormer(cfg)
    sd = init_state_dict(cfg, seed)
    model.load_state_dict(sd)
    pipe = RenderFormerRenderingPipeline(model)
    pipe.to(torch.device("cuda:0"))
    return pipe, sd


def _check(pipe, sd, cfg, sc, res, tag):
    from oracle import renderformer_oracle as orc
    ref = orc.render(sd, cfg, sc["triangles"], sc["texture"].clone(), sc["mask"], sc["vn"], sc["c2w"], sc["fov"], res)
    g = {k: v.cuda() for k, v in sc.items()}
    img = pipe(g["triangles"], g["texture"], g["mask"], g["vn"], g["c2w"], g["fov"], resolution=res)
    assert img.shape == ref.shape and torch.isfinite(img).all()
    rel, psnr = hdr_rel_err(img, ref), log_psnr(img, ref)
    print(f"{tag}: hdr rel {rel:.3e} log-PSNR {psnr:.1f} dB")
    assert rel <= REL_TOL and psnr >= PSNR_MIN, tag
    return ref


@pytest.mark.parametrize("cfg_name,n_tris,pad_to,views,res", [
    ("tiny_swin", 37, None, 1, 64),      # ragged triangle count (not a multiple of 8), one view
    ("tiny_swin", 1, 8, 2, 64),          # a single valid triangle behind padding
    ("tiny_swin", 250, 256, 3, 128),     # more than one key tile, 128x128
    ("tiny_swin", 129, None, 1, 192),    # resolution that is a multiple of 64 but not a power of two
    ("tiny_full", 90, 96, 2, 64),        # full ray self-attention decoder (V1-Base structure)
    ("tiny_full", 40, None, 1, 40),      # 8-pixel-patch resolution that swin could not take
])
def test_edge_shapes_against_oracle(cfg_name, n_tris, pad_to, views, res):
    cfg = RenderFormerConfig.named(cfg_name)
    pipe, sd = _pipe(cfg, 11)
    sc = make_scene(n_tris, views, seed=21, pad_to=pad_to)
    _check(pipe, sd, cfg, sc, res, f"{cfg_name} N={n_tris}/{pad_to} V={views} R={res}")


def test_two_scenes_per_call_with_different_padding():
    """B = 2: scenes are independent; each has its own mask (padding in different places)."""
    cfg = RenderFormerConfig.named("tiny_swin")
    pipe, sd = _pipe(cfg, 5)
    a = make_scene(60, 2, seed=1, pad_to=64)
    b = make_scene(33, 2, seed=2, pad_to=64)
    sc = {k: torch.cat([a[k], b[k]], dim=0) for k in a}
    _check(pipe, sd, cfg, sc, 64, "B=2")


def test_swin_rejects_bad_resolution():
    cfg = RenderFormerConfig.named("tiny_swin")
    pipe, _ = _pipe(cfg, 5)
    sc = {k: v.cuda() for k, v in make_scene(16, 1, seed=1).items()}
    with pytest.raises(ValueError):
        pipe(sc["triangles"], sc["texture"], sc["mask"], sc["vn"], sc["c2w"], sc["fov"], resolution=96)


def test_render_stream_matches_blocking_calls():
    """The overlapped host-in / host-out batch API returns exactly what one blocking render() per
    scene returns, in order, for scenes of different sizes."""
    cfg = RenderFormerConfig.named("tiny_swin")
    pipe, _ = _pipe(cfg, 9)
    scenes = [make_scene(n, v, seed=s, pad_to=p) for n, v, s, p in ((40, 2, 1, 48), (70, 1, 2, None), (40, 2, 3, 48),
                                                                     (16, 3, 4, None), (90, 1, 5, 96))]
    host = [{k: t.pin_memory() for k, t in sc.items()} for sc in scenes]
    want = []
    for sc in scenes:
        g = {k: t.cuda() for k, t in sc.items()}
        want.append(pipe(g["triangles"], g["texture"], g["mask"], g["vn"], g["c2w"], g["fov"], resolution=64).cpu())
    got = [img.clone() for img in pipe.render_stream(iter(host), resolution=64)]
    assert len(got) == len(want)
    for a, b in zip(got, want):
        assert a.shape == b.shape and a.is_pinned() is False  # clones of the pinned ring buffers
        assert torch.equal(a, b)
    assert list(pipe.render_stream(iter([]), resolution=64)) == []


def test_render_stream_fixed_length_padding_reuses_one_graph():
    """batch_infer.py:37-47 (`--padding_length`): scenes of different triangle counts padded to one length on the
    device -> one input signature -> ONE CUDA graph replayed for every scene; images equal the unpadded renders."""
    cfg = RenderFormerConfig.named("tiny_swin")
    pipe, _ = _pipe(cfg, 8)
    counts = (61, 128, 17, 100)
    scenes = [make_scene(n, 2, seed=40 + i) for i, n in enumerate(counts)]
    want = []
    for sc in scenes:
        g = {k: t.cuda() for k, t in sc.items()}
        want.append(pipe(g["triangles"], g["texture"], g["mask"], g["vn"], g["c2w"], g["fov"], resolution=64).cpu())
    pipe.cuda_graphs = True
    host = [{k: t.pin_memory() for k, t in sc.items()} for sc in scenes]
    got = [img.clone() for img in pipe.render_stream(iter(host), resolution=64, pad_to=128)]
    assert len(pipe._graphs) == 1, "every padded scene must replay the same graph"
    for a, b, n in zip(got, want, counts):
        assert a.shape == b.shape
        assert hdr_rel_err(a, b) < 2e-3, f"{n} triangles padded to 128"
    with pytest.raises(ValueError):
        list(pipe.render_stream(iter(host), resolution=64, pad_to=64))


def test_cbox_scene_and_constant_texture_fast_path(golden_dir):
    """BASELINE configs[0/1] geometry: the converted examples/cbox.json (5633 triangles) renders within
    tolerance of the fp32 oracle, and the constant-texture fast path ([B,N,13] input, texel-summed
    projection weights) agrees with the full 32x32 texel path."""
    from renderformer_b200 import scene_io as sio
    cfg = RenderFormerConfig.named("tiny_swin")
    pipe, sd = _pipe(cfg, 13)
    scene = sio.load_npz(os.path.join(golden_dir, "cbox_scene.npz"))
    full = sio.to_pipeline_inputs(scene)
    oracle = _check(pipe, sd, cfg, full, 64, "cbox full texture")
    g = {k: v.cuda() for k, v in full.items()}
    ref = pipe(g["triangles"], g["texture"], g["mask"], g["vn"], g["c2w"], g["fov"], resolution=64)
    const = {k: v.cuda() for k, v in sio.to_pipeline_inputs(scene, constant_texture=True).items()}
    fast = pipe(const["triangles"], const["texture"], const["mask"], const["vn"], const["c2w"], const["fov"],
                resolution=64)
    rel, psnr = hdr_rel_err(fast, ref), log_psnr(fast, ref)
    print(f"constant-texture path vs texel path: hdr rel {rel:.3e} log-PSNR {psnr:.1f} dB")
    assert rel <= 5e-3 and psnr >= 55.0
    # and directly against the fp32 oracle (which sees the full 32 x 32 texel grid)
    rel_o, psnr_o = hdr_rel_err(fast, oracle), log_psnr(fast, oracle)
    print(f"constant-texture path vs oracle: hdr rel {rel_o:.3e} log-PSNR {psnr_o:.1f} dB")
    assert rel_o <= REL_TOL and psnr_o >= PSNR_MIN


def test_cuda_graph_replay_matches_eager():
    """pipeline.cuda_graphs: captured-and-replayed render() is bit-identical to eager launches, for
    changing inputs of one signature and for a second signature."""
    cfg = RenderFormerConfig.named("tiny_swin")
    pipe, _ = _pipe(cfg, 4)
    scenes = [{k: v.cuda() for k, v in make_scene(50, 2, seed=s, pad_to=56).items()} for s in (1, 2, 3)]
    other = {k: v.cuda() for k, v in make_scene(20, 1, seed=9).items()}

    def call(sc, res):
        return pipe(sc["triangles"], sc["texture"], sc["mask"], sc["vn"], sc["c2w"], sc["fov"], resolution=res).clone()
    eager = [call(sc, 64) for sc in scenes] + [call(other, 128)]
    pipe.cuda_graphs = True
    graphed = [call(sc, 64) for sc in scenes] + [call(other, 128)] + [call(scenes[0], 64)]
    assert len(pipe._graphs) == 2 and pipe.replayed_launches > 0
    for a, b in zip(graphed, eager + [eager[0]]):
        assert torch.equal(a, b)
    # results of consecutive replays of one graph stay valid without the caller copying them ...
    def raw(sc):
        return pipe(sc["triangles"], sc["texture"], sc["mask"], sc["vn"], sc["c2w"], sc["fov"], resolution=64)
    r1, r2 = raw(scenes[0]), raw(scenes[1])
    assert r1.data_ptr() != r2.data_ptr() and torch.equal(r1, eager[0]) and torch.equal(r2, eager[1])
    # ... unless the static output itself is requested
    pipe.graph_static_outputs = True
    s1 = raw(scenes[0])
    s2 = raw(scenes[1])
    assert s1.data_ptr() == s2.data_ptr() and torch.equal(s2, eager[1])


def test_ldr_quantize_bit_exact_and_streamed():
    """Default LDR conversion of the CLIs, (np.clip(hdr, 0, 1) * 255).astype(uint8) (infer.py:97-98), is
    reproduced bit-exactly on the device; the PBR-neutral curve is monotone and bounded."""
    import numpy as np
    from renderformer_b200.model import RenderFormerRenderingPipeline as P
    g = torch.Generator().manual_seed(0)
    hdr = torch.cat([torch.rand(5000, 3, generator=g) * 1.5 - 0.2, torch.rand(3000, 3, generator=g) * 50,
                     torch.tensor([[0.0, 1.0, 0.5], [1 / 255, 2 / 255, 254.999 / 255], [1e-9, 0.99999994, 3.0]])])
    hdr = hdr.view(1, 1, -1, 1, 3).contiguous()
    want = (np.clip(hdr.numpy(), 0, 1) * 255).astype(np.uint8)
    got = P.hdr_to_ldr(hdr.cuda(), "none").cpu().numpy()
    assert got.dtype == np.uint8 and np.array_equal(got, want)
    ramp = torch.linspace(0, 8, 4096)[:, None].repeat(1, 3).contiguous().cuda()
    pbr = P.hdr_to_ldr(ramp, "pbr_neutral").cpu().numpy().astype(int)
    assert (np.diff(pbr[:, 0]) >= 0).all() and pbr.max() <= 255 and pbr[0, 0] == 0 and pbr[-1, 0] >= 250
    with pytest.raises(ValueError):
        P.hdr_to_ldr(ramp, "agx")
    cfg = RenderFormerConfig.named("tiny_swin")
    pipe, _ = _pipe(cfg, 9)
    sc = make_scene(40, 2, seed=1)
    g_ = {k: t.cuda() for k, t in sc.items()}
    ref = pipe(g_["triangles"], g_["texture"], g_["mask"], g_["vn"], g_["c2w"], g_["fov"], resolution=64).cpu().numpy()
    out = [x.clone() for x in pipe.render_stream(iter([sc]), resolution=64, ldr="none")]
    assert out[0].dtype == torch.uint8 and np.array_equal(out[0].numpy(), (np.clip(ref, 0, 1) * 255).astype(np.uint8))


def test_model_forward_reference_signature():
    """RenderFormer.forward with the reference's own arguments (models/renderformer.py:171-206): log-encoded
    texture, explicit camera-space ray map and camera-space triangles, log-encoded [B,V,3,H,W] output --
    checked against the oracle's scene_stage / view_stage and against the pipeline's camera path."""
    import math

    from oracle import renderformer_oracle as orc
    from renderformer_b200.model import RenderFormer
    cfg = RenderFormerConfig.named("tiny_swin")
    pipe, sd = _pipe(cfg, 21)
    model: RenderFormer = pipe.model
    sc = make_scene(60, 2, seed=6, pad_to=64)
    B, V, N, R = 1, 2, 64, 64
    tex_log = sc["texture"].clone()
    tex_log[:, :, -3:] = torch.log10(tex_log[:, :, -3:] + 1.0)
    tri_cam = orc.to_camera_space(sc["c2w"][0], sc["triangles"].expand(V, -1, -1, -1)).reshape(1, V, N, 9)
    rays = orc.camera_rays(sc["fov"][0] / 180.0 * math.pi, R)[None]  # [1,V,R,R,3]
    out = model(sc["triangles"].reshape(B, N, 9).cuda(), tex_log.cuda(), sc["mask"].cuda(),
                sc["vn"].reshape(B, N, 9).cuda(), rays_o=torch.zeros(B, V, 3).cuda(), rays_d=rays.cuda(),
                tri_vpos_view_tf=tri_cam.cuda(), tf32_view_tf=True)
    assert out.shape == (B, V, 3, R, R)
    hdr = (torch.pow(10.0, out) - 1.0).permute(0, 1, 3, 4, 2).cpu()
    ref = orc.render(sd, cfg, sc["triangles"], sc["texture"], sc["mask"], sc["vn"], sc["c2w"], sc["fov"], R)
    rel, psnr = hdr_rel_err(hdr, ref), log_psnr(hdr, ref)
    print(f"model.forward (reference signature) vs oracle: hdr rel {rel:.3e} log-PSNR {psnr:.1f} dB")
    assert rel <= REL_TOL and psnr >= PSNR_MIN
    g = {k: v.cuda() for k, v in sc.items()}
    cam = pipe(g["triangles"], g["texture"], g["mask"], g["vn"], g["c2w"], g["fov"], resolution=R).cpu()
    assert hdr_rel_err(hdr, cam) < 3e-3  # same kernels; rays / transforms computed on the host here


def test_view_chunks_on_several_streams():
    """view_streams > 1 (independent view chunks on side streams, eager and under graph capture) returns
    exactly the sequential result."""
    cfg = RenderFormerConfig.named("tiny_swin")
    pipe, _ = _pipe(cfg, 4)
    sc = {k: v.cuda() for k, v in make_scene(50, 5, seed=8, pad_to=56).items()}

    def call():
        return pipe(sc["triangles"], sc["texture"], sc["mask"], sc["vn"], sc["c2w"], sc["fov"], resolution=64).clone()
    pipe.view_chunk = 8
    want = call()
    pipe.view_chunk, pipe.view_streams = 2, 2
    assert torch.equal(call(), want)
    pipe.view_chunk, pipe.view_streams = 1, 3
    assert torch.equal(call(), want)
    pipe.cuda_graphs = True
    assert torch.equal(call(), want) and torch.equal(call(), want)


def test_render_stream_sharded_single_rank():
    """dist.render_stream_sharded without a process group (world 1) = render_stream."""
    from renderformer_b200.dist import render_stream_sharded
    cfg = RenderFormerConfig.named("tiny_swin")
    pipe, _ = _pipe(cfg, 9)
    scenes = [{k: t.pin_memory() for k, t in make_scene(n, v, seed=s, pad_to=p).items()}
              for n, v, s, p in ((40, 2, 1, 48), (70, 3, 2, None), (40, 2, 3, 48))]
    want = [x.clone() for x in pipe.render_stream(iter(scenes), resolution=64)]
    pipe.cuda_graphs = True
    got = [(sl, x.clone()) for sl, x in render_stream_sharded(pipe, iter(scenes), resolution=64)]
    assert len(got) == len(want)
    for (sl, a), b, sc in zip(got, want, scenes):
        assert sl == slice(0, sc["c2w"].shape[1]) and torch.equal(a, b)


@pytest.mark.parametrize("B,Hi,Ho,C,tiled", [
    (2, 32, 64, 128, True),      # FeatureFusionBlock 4 of the DPT head at 512^2 (tiled kernel)
    (1, 128, 256, 128, True),
    (1, 33, 66, 128, True),      # output not a multiple of the 8 x 32 tile
    (3, 8, 16, 128, False),      # narrower than a tile: generic kernel
    (1, 20, 37, 128, False),     # not ~2x: generic kernel
    (1, 16, 32, 64, False),      # 64 channels: generic kernel
])
def test_upsample_bilinear_matches_interpolate(B, Hi, Ho, C, tiled):
    """rfb_upsample_bilinear (both kernels) vs F.interpolate(mode='bilinear', align_corners=True) -- the
    resize of FeatureFusionBlock.forward, layers/dpt.py:154-155 -- on NHWC fp16 maps."""
    import torch.nn.functional as F
    from renderformer_b200 import lib as L
    from renderformer_b200 import ops
    g = torch.Generator().manual_seed(3)
    x = torch.randn((B, Hi, Hi, C), generator=g).to(torch.float16).cuda()
    out = torch.zeros((B * Ho * Ho, C), dtype=torch.float16, device="cuda")
    n0 = L.launch_count()
    ops.upsample_bilinear(x.view(-1, C), out, B=B, Hi=Hi, Wi=Hi, Ho=Ho, Wo=Ho, C_=C)
    torch.cuda.synchronize()
    assert L.launch_count() == n0 + 1
    ref = F.interpolate(x.float().permute(0, 3, 1, 2), size=(Ho, Ho), mode="bilinear", align_corners=True)
    ref = ref.permute(0, 2, 3, 1).reshape(-1, C)
    err = (out.float() - ref).abs().max().item()
    assert err <= 4e-3, f"max |d| {err:.3e}"   # fp16 output rounding of |x| < 4.5: half an ulp = 2e-3
