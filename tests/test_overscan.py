"""CPU: overscan of sizes off the decoder's grid -- the canvas rule of config.overscan_grid, the overscan camera of the
oracle extension (tests/overscan_oracle.py) against the plain H x W camera, the FLOP count of an overscan view and
render_folder's --overscan flag."""
import math
import os
import sys

import pytest
import torch

from renderformer_b200.config import RenderFormerConfig, overscan_grid
from renderformer_b200.flops import job_flops, view_flops

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
from nonsquare_oracle import camera_rays_hw  # noqa: E402
from overscan_oracle import camera_rays_overscan  # noqa: E402

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SWIN, FULL = RenderFormerConfig.named("tiny_swin"), RenderFormerConfig.named("tiny_full")


@pytest.mark.parametrize("cfg,res,canvas,offsets", [
    (SWIN, (1080, 1920), (1088, 1920), (4, 0)),
    (SWIN, (720, 1280), (768, 1280), (24, 0)),
    (SWIN, (2160, 3840), (2176, 3840), (8, 0)),
    (SWIN, (1440, 2560), (1472, 2560), (16, 0)),
    (SWIN, (99, 150), (128, 192), (14, 21)),
    (FULL, (99, 150), (104, 152), (2, 1)),
    (FULL, 5, (8, 8), (1, 1)),
], ids=["1080p", "720p", "4k", "1440p", "swin99x150", "full99x150", "full5"])
def test_overscan_grid_values(cfg, res, canvas, offsets):
    hw = tuple(res) if isinstance(res, tuple) else (res, res)
    assert overscan_grid(cfg, res) == (hw, canvas, offsets)


@pytest.mark.parametrize("cfg,res", [(SWIN, 512), (SWIN, (576, 1024)), (SWIN, [64, 128]), (FULL, (64, 136)), (FULL, 8)])
def test_overscan_grid_on_grid_is_identity(cfg, res):
    hw = tuple(res) if isinstance(res, (tuple, list)) else (res, res)
    assert overscan_grid(cfg, res) == (hw, hw, (0, 0))


@pytest.mark.parametrize("bad", [0, -64, 64.0, True, "512", (64,), (64, 64, 3), (0, 64), (64, -8), (64.0, 64),
                                 (True, 64), None])
def test_overscan_grid_rejects_what_view_grid_rejects(bad):
    for cfg in (SWIN, FULL):
        with pytest.raises(ValueError):
            overscan_grid(cfg, bad)


@pytest.mark.parametrize("H,W,Hc,Wc,top,left", [(1080, 1920, 1088, 1920, 4, 0), (99, 150, 128, 192, 14, 21),
                                                 (99, 150, 104, 152, 2, 1), (150, 99, 192, 128, 21, 14)])
def test_overscan_window_rays_are_the_image_camera(H, W, Hc, Wc, top, left):
    fov = torch.tensor([[math.radians(37.5)], [math.radians(70.0)]])
    canvas = camera_rays_overscan(fov, H, W, Hc, Wc, top, left)
    assert canvas.shape == (2, Hc, Wc, 3)
    win = canvas[:, top:top + H, left:left + W]
    assert (win - camera_rays_hw(fov, H, W)).abs().max().item() <= 1e-6


@pytest.mark.parametrize("H,W", [(64, 64), (128, 192), (576, 1024)])
def test_overscan_rays_without_border_are_camera_rays_hw(H, W):
    fov = torch.tensor([[0.3], [0.6981317]])
    assert torch.equal(camera_rays_overscan(fov, H, W, H, W, 0, 0), camera_rays_hw(fov, H, W))


def test_flops_of_an_overscan_view_are_its_canvas():
    cfg = RenderFormerConfig.named("v1_1_swin_large")
    for res, canvas in (((1080, 1920), (1088, 1920)), ((720, 1280), (768, 1280)), ((2160, 3840), (2176, 3840))):
        assert view_flops(cfg, 4096, res, overscan=True) == view_flops(cfg, 4096, canvas)
        assert job_flops(cfg, 4096, res, 1, 8, overscan=True) == job_flops(cfg, 4096, canvas, 1, 8)
    assert view_flops(cfg, 4096, 512, overscan=True) == view_flops(cfg, 4096, 512)


def test_render_folder_overscan_flag(tmp_path):
    """--overscan reaches render_stream (with the off-grid size); without it nothing changes."""
    import importlib.util
    from renderformer_b200 import frame_io as fio
    from renderformer_b200 import scene_io as sio
    from renderformer_b200.synth import make_scene
    spec = importlib.util.spec_from_file_location("render_folder", os.path.join(ROOT, "tools", "render_folder.py"))
    tool = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(tool)
    folder = tmp_path / "scenes"
    folder.mkdir()
    sc = make_scene(6, 1, seed=1)
    sio.save_npz({"triangles": sc["triangles"][0].numpy(), "vn": sc["vn"][0].numpy(),
                  "tex13": sc["texture"][0, :, :, 0, 0].numpy(), "c2w": sc["c2w"][0].numpy(),
                  "fov": sc["fov"][0, :, 0].numpy()}, str(folder / "a.npz"))

    class Pipe:
        cuda_graphs = False

        def __init__(self):
            self.calls = []

        def render_stream(self, scenes, resolution=512, torch_dtype=None, ldr=None, pad_to=None, overscan=False):
            for s in scenes:
                self.calls.append((resolution, overscan))
                H, W = resolution if isinstance(resolution, tuple) else (resolution, resolution)
                yield torch.zeros(1, s["c2w"].shape[1], H, W, 3)

    for flags, want in ((["--height", "18", "--width", "30", "--overscan"], ((18, 30), True)),
                        (["--height", "16", "--width", "40"], ((16, 40), False))):
        pipe = Pipe()
        out = tmp_path / f"out{len(flags)}"
        assert tool.main(["--scene_folder", str(folder), "--random_init", "tiny_swin", "--resolution", "32",
                          "--output_dir", str(out)] + flags, _pipeline=pipe) == 0
        assert pipe.calls == [want]
        assert fio.read_exr(str(out / "a_view_0.exr")).shape == (*want[0], 3)


def test_pipeline_size_rule_is_unchanged_without_overscan():
    """An off-grid size still raises ValueError on the host without overscan; with it the size is accepted and the
    call reaches the kernels (which, without a GPU, fail loudly: there is no CPU fallback)."""
    from renderformer_b200 import lib
    from renderformer_b200.model import RenderFormer, RenderFormerRenderingPipeline
    from renderformer_b200.synth import make_scene
    pipe = RenderFormerRenderingPipeline(RenderFormer(SWIN))
    sc = make_scene(8, 1)
    args = (sc["triangles"], sc["texture"], sc["mask"], sc["vn"], sc["c2w"], sc["fov"])
    with pytest.raises(ValueError):
        pipe(*args, resolution=(99, 150))
    with pytest.raises(ValueError):
        pipe(*args, resolution=(0, 150), overscan=True)
    assert pipe.view_geometry((99, 150), overscan=True) == ((128, 192), (99, 150, 14, 21), (99, 150))
    assert pipe.view_geometry((128, 192), overscan=True) == ((128, 192), None, (128, 192))
    if not torch.cuda.is_available():
        with pytest.raises(lib.RfbError):
            pipe(*args, resolution=(99, 150), overscan=True)
