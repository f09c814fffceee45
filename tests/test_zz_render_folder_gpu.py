"""GPU: the batch workflow end to end (SURVEY §8 f3) -- tools/render_folder.py renders a folder of converted scenes
through `render_stream` + `frame_io.FrameWriter`, and the EXR / PNG / MP4 files it leaves are compared with the
fp32 oracle on the same scene files (the unchanged reference CLI on the same package is covered by
tests/test_reference_clis_gpu.py; this is the overlapped replacement of its loop).

The tool runs in a subprocess and the file sorts last.  The two-rank case has not been run on hardware yet and is
xfail(strict=False) until it has.  The file encoders themselves are verified on CPU (tests/test_frame_io.py, against
OpenCV and Pillow)."""
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

from renderformer_b200 import frame_io as fio
from renderformer_b200 import scene_io as sio
from renderformer_b200.config import RenderFormerConfig
from renderformer_b200.metrics import PSNR_MIN, REL_TOL, hdr_rel_err, log_psnr
from renderformer_b200.synth import init_state_dict, make_scene

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
NOT_YET = pytest.mark.xfail(strict=False, reason="not yet run on hardware with two GPUs")


def _write_scenes(folder, counts, views):
    """Scene files in tools/convert_scene.py's .npz format; returns name -> host tensors the oracle renders."""
    os.makedirs(folder, exist_ok=True)
    scenes = {}
    for i, n in enumerate(counts):
        sc = make_scene(n, views, seed=40 + i)
        name = f"frame_{i}"
        sio.save_npz({"triangles": sc["triangles"][0].numpy(), "vn": sc["vn"][0].numpy(),
                      "tex13": sc["texture"][0, :, :, 0, 0].numpy(), "c2w": sc["c2w"][0].numpy(),
                      "fov": sc["fov"][0, :, 0].numpy()}, os.path.join(folder, name + ".npz"))
        scenes[name] = sc
    return scenes


def _check_outputs(out_dir, scenes, views, res, video):
    from oracle import renderformer_oracle as orc
    cfg = RenderFormerConfig.named("tiny_swin")
    sd = init_state_dict(cfg, 7)  # what --random_init uses
    for name, sc in scenes.items():
        ref = orc.render(sd, cfg, sc["triangles"], sc["texture"], sc["mask"], sc["vn"], sc["c2w"], sc["fov"], res)[0]
        for v in range(views):
            hdr = fio.read_exr(os.path.join(out_dir, f"{name}_view_{v}.exr"))
            got = torch.from_numpy(hdr)
            rel, psnr = hdr_rel_err(got, ref[v]), log_psnr(got, ref[v])
            assert got.shape == ref[v].shape and rel <= REL_TOL and psnr >= PSNR_MIN, (name, v, rel, psnr)
            ldr = fio.read_png(os.path.join(out_dir, f"{name}_view_{v}.png"))
            assert np.array_equal(ldr, (np.clip(hdr, 0, 1) * 255).astype(np.uint8))  # batch_infer.py:153-157
    if video:
        import cv2
        cap = cv2.VideoCapture(os.path.join(out_dir, "video.mp4"))
        n = 0
        while cap.read()[0]:
            n += 1
        assert n == len(scenes) * views


def _run(cmd, timeout=600):
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=timeout, cwd=ROOT)
    assert r.returncode == 0, (r.stdout[-1500:], r.stderr[-3000:])
    return r.stdout


@pytest.mark.parametrize("extra", [["--padding_length", "64", "--save_video"], ["--constant_texture"]],
                         ids=["padded-one-graph-video", "constant-texture-eager"])
def test_render_folder_tool_against_oracle(tmp_path, extra):
    try:
        import cv2  # noqa: F401
    except ImportError:
        extra = [e for e in extra if e != "--save_video"]
    scenes = _write_scenes(str(tmp_path / "scenes"), (40, 57, 33), views=2)
    out_dir = str(tmp_path / "out")
    log = _run([sys.executable, os.path.join(ROOT, "tools", "render_folder.py"), "--scene_folder", str(tmp_path / "scenes"),
                "--random_init", "tiny_swin", "--precision", "fp16", "--resolution", "64", "--output_dir", out_dir] + extra)
    assert "6 frames of 3 scenes" in log, log
    _check_outputs(out_dir, scenes, 2, 64, "--save_video" in extra)


@NOT_YET
@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs two GPUs")
def test_render_folder_tool_two_ranks(tmp_path):
    """torchrun, 2 ranks: scene stage row-sharded, every rank writes its own views, rank 0 assembles the video."""
    import socket
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        port = s.getsockname()[1]
    scenes = _write_scenes(str(tmp_path / "scenes"), (48, 48), views=3)
    out_dir = str(tmp_path / "out")
    _run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2", "--master-addr", "127.0.0.1",
          "--master-port", str(port), os.path.join(ROOT, "tools", "render_folder.py"), "--scene_folder",
          str(tmp_path / "scenes"), "--random_init", "tiny_swin", "--precision", "fp16", "--resolution", "64",
          "--output_dir", out_dir, "--save_video"])
    try:
        import cv2  # noqa: F401
        video = True
    except ImportError:
        video = False
    _check_outputs(out_dir, scenes, 3, 64, video)
