"""CPU: non-square images -- the H x W oracle extension (tests/nonsquare_oracle.py: its camera, and the oracle itself
on square images), the (height, width) size rules of
config.view_grid, the FLOP counts of an (H, W) view, render_folder's --height / --width, and (where the unmodified
reference is at hand) the reference's view stage on a non-square ray map against the oracle."""
import json
import math
import os
import subprocess
import sys

import pytest
import torch

from oracle import renderformer_oracle as orc
from oracle.reference_loader import find_reference
from renderformer_b200.config import RenderFormerConfig, view_grid
from renderformer_b200.flops import dpt_flops, job_flops, view_flops

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
from nonsquare_oracle import camera_rays_hw, render_hw  # noqa: E402

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.mark.parametrize("R", [8, 64, 512])
def test_camera_rays_hw_square_is_camera_rays(R):
    fov = torch.tensor([[0.3], [0.6981317], [1.4]])
    assert torch.equal(camera_rays_hw(fov, R, R), orc.camera_rays(fov, R))


@pytest.mark.parametrize("name", ["tiny_swin", "tiny_full"])
def test_render_hw_square_is_the_oracle(name):
    """The H x W restatement is the oracle itself on square images (same ops, same order): what it computes for
    H != W differs from the pinned oracle only in the patch grid and the camera."""
    from renderformer_b200.synth import init_state_dict, make_scene
    cfg = RenderFormerConfig.named(name)
    sd = init_state_dict(cfg, 3)
    sc = make_scene(30, 2, seed=5, pad_to=40)
    args = (sd, cfg, sc["triangles"], sc["texture"], sc["mask"], sc["vn"], sc["c2w"], sc["fov"])
    assert torch.equal(render_hw(*args, (64, 64)), orc.render(*args, 64))
    hw = render_hw(*args, (64, 128))
    assert hw.shape == (1, 2, 64, 128, 3) and torch.isfinite(hw).all()


@pytest.mark.parametrize("H,W", [(576, 1024), (1024, 576)])
def test_fov_spans_the_longer_side(H, W):
    fov = torch.tensor([[math.radians(40.0)]], dtype=torch.float64)
    rays = camera_rays_hw(fov, H, W)[0]
    assert rays.shape == (H, W, 3)
    L = max(H, W)
    f = L / 2 / math.tan(fov.item() / 2)
    want = (L / 2 - 0.5) / f
    if W >= H:   # outermost pixel centres of the long side: first / last column, on the middle rows
        edge = [rays[H // 2, 0], rays[H // 2, -1]]
        slope = [abs(r[0] / r[2]).item() for r in edge]
        short = abs(rays[0, W // 2, 1] / rays[0, W // 2, 2]).item()
        assert abs(abs(rays[H // 2, 0, 1] / rays[H // 2, 0, 2]).item() - 0.5 / f) < 1e-12
    else:
        edge = [rays[0, W // 2], rays[-1, W // 2]]
        slope = [abs(r[1] / r[2]).item() for r in edge]
        short = abs(rays[H // 2, 0, 0] / rays[H // 2, 0, 2]).item()
        assert abs(abs(rays[0, W // 2, 0] / rays[0, W // 2, 2]).item() - 0.5 / f) < 1e-12
    for s in slope:
        assert abs(s - want) < 1e-12
    # the image edge (half a pixel further out) sits at exactly fov / 2; the short side spans less
    assert abs((L / 2) / f - math.tan(fov.item() / 2)) < 1e-12
    assert short == pytest.approx((min(H, W) / 2 - 0.5) / f, abs=1e-12) and short < want
    # orientation: +x to the right, +y up, looking down -z
    assert rays[H // 2, -1, 0] > 0 and rays[0, W // 2, 1] > 0 and (rays[..., 2] < 0).all()


def test_view_grid_size_rules():
    swin = RenderFormerConfig.named("v1_1_swin_large")
    full = RenderFormerConfig.named("v1_base")
    for cfg in (swin, full):
        assert view_grid(cfg, 512) == (512, 512)
        assert view_grid(cfg, (576, 1024)) == (576, 1024)
        assert view_grid(cfg, [1024, 576]) == (1024, 576)
        for bad in ((60, 64), (64, 60), 0, -64, (0, 64), (64,), (64, 64, 64), 64.0, (64.0, 64), True, "512", None):
            with pytest.raises(ValueError):
                view_grid(cfg, bad)
    for hw in ((576, 1000), (64, 136), 200, (8, 24)):
        assert view_grid(full, hw) == ((hw, hw) if isinstance(hw, int) else tuple(hw))
        with pytest.raises(ValueError, match="multiples of 64"):
            view_grid(swin, hw)
    assert view_grid(RenderFormerConfig.named("tiny_full"), (64, 136)) == (64, 136)
    assert view_grid(RenderFormerConfig.named("tiny_swin"), (192, 320)) == (192, 320)


def test_flops_of_hw_views():
    cfg = RenderFormerConfig.named("v1_1_swin_large")
    assert view_flops(cfg, 4096, (512, 512)) == view_flops(cfg, 4096, 512)
    assert dpt_flops(cfg, (512, 512)) == dpt_flops(cfg, 512)
    assert job_flops(cfg, 4096, (512, 512), 1, 8) == job_flops(cfg, 4096, 512, 1, 8)
    # equal pixel counts cost the same; transposing the image does not change the count
    assert view_flops(cfg, 4096, (256, 1024)) == view_flops(cfg, 4096, 512)
    assert view_flops(cfg, 4096, (576, 1024)) == view_flops(cfg, 4096, (1024, 576))
    assert view_flops(cfg, 4096, (256, 512)) < view_flops(cfg, 4096, 512)


def test_render_folder_height_width_flags(tmp_path):
    """--height / --width reach render_stream as (H, W); either one replaces the matching side of --resolution."""
    import importlib.util
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
            self.res = []

        def render_stream(self, scenes, resolution=512, torch_dtype=None, ldr=None, pad_to=None):
            for s in scenes:
                self.res.append(resolution)
                H, W = resolution if isinstance(resolution, tuple) else (resolution, resolution)
                yield torch.zeros(1, s["c2w"].shape[1], H, W, 3)

    for flags, want in (([], 32), (["--height", "16", "--width", "40"], (16, 40)), (["--width", "48"], (32, 48))):
        pipe = Pipe()
        out = tmp_path / f"out{len(flags)}"
        assert tool.main(["--scene_folder", str(folder), "--random_init", "tiny_swin", "--resolution", "32",
                          "--output_dir", str(out)] + flags, _pipeline=pipe) == 0
        assert pipe.res == [want]
        from renderformer_b200 import frame_io as fio
        H, W = want if isinstance(want, tuple) else (want, want)
        assert fio.read_exr(str(out / "a_view_0.exr")).shape == (H, W, 3)


# ------------------------------------------------------------------------------------------ live reference pin
WORKER = r"""
import json, sys, torch
sys.path.insert(0, %(root)r)
sys.path.insert(0, %(root)r + "/tests")
from oracle import renderformer_oracle as orc
from nonsquare_oracle import camera_rays_hw, view_stage_hw
from oracle.reference_loader import load_reference
from renderformer_b200.config import RenderFormerConfig
from renderformer_b200.synth import init_state_dict, make_scene
torch.set_num_threads(4)
RefConfig, _, _, ref = load_reference("sdpa")
from renderformer.models.view_transformer import ViewTransformer
out = {"ref": ref, "cases": []}
for name, H, W, V in (("tiny_swin", 128, 192, 2), ("tiny_swin", 192, 128, 1), ("tiny_full", 64, 136, 2)):
    cfg = RenderFormerConfig.named(name)
    sd = init_state_dict(cfg, 21)
    sc = make_scene(40, V, seed=22, pad_to=48)
    N = sc["triangles"].shape[1]
    tex = sc["texture"].clone()
    tex[:, :, -3:] = torch.log10(tex[:, :, -3:] + 1.0)
    seq, key_mask = orc.scene_stage(sd, cfg, sc["triangles"].reshape(1, N, 9), tex, sc["mask"], sc["vn"].reshape(1, N, 9))
    seq, key_mask = seq.expand(V, -1, -1), key_mask.expand(V, -1)
    tri_cam = orc.to_camera_space(sc["c2w"][0], sc["triangles"].expand(V, -1, -1, -1)).reshape(V, N, 9)
    rays = camera_rays_hw(sc["fov"][0] / 180.0 * 3.141592653589793, H, W)
    pos_k, _ = orc.centroid_positions(tri_cam, sc["mask"].expand(V, -1), cfg.num_register_tokens)
    taps = {}
    want = view_stage_hw(sd, cfg, seq, key_mask, tri_cam, sc["mask"].expand(V, -1), rays, taps)
    vt = ViewTransformer(RefConfig(**cfg.to_dict()))
    vt.load_state_dict({k[len("view_transformer."):]: v for k, v in sd.items() if k.startswith("view_transformer.")},
                       strict=True)
    vt.eval()
    case = {"case": [name, H, W, V], "range": float(want.max() - want.min())}
    with torch.no_grad():
        # model level: the reference's ViewTransformer on the H x W ray map
        try:
            got = vt(torch.zeros(V, 3), rays, seq, pos_k, key_mask)
            case["vt_shape_ok"] = list(got.shape) == list(want.shape)
            case["vt_max_abs"] = float((got - want).abs().max()) if case["vt_shape_ok"] else None
        except Exception as e:  # the reference itself rejects a non-square ray map at this level
            case["vt_error"] = repr(e)[:300]
        # decoder + DPT head with patch_h != patch_w
        Hp, Wp = H // 8, W // 8
        p = "view_transformer."
        tok = rays.view(V, Hp, 8, Wp, 8, 3).permute(0, 1, 3, 5, 2, 4).reshape(V, Hp * Wp, -1)
        x = sd[p + "ray_map_patch_token"] + orc.rms(torch.nn.functional.linear(tok, sd[p + "ray_map_encoder.weight"],
                                                    sd[p + "ray_map_encoder.bias"]), sd[p + "ray_map_encoder_norm.weight"], None)
        feats = vt.transformer(x, seq, src_key_padding_mask=key_mask, triangle_pos=pos_k,
                               ray_pos=torch.zeros(V, Hp * Wp, 9), out_layers=vt.out_layers, patch_h=Hp, patch_w=Wp)
        feats = [f[0] if isinstance(f, (list, tuple)) else f for f in feats]
        case["dec_max_rel"] = max(float((f - r).abs().max() / r.abs().max()) for f, r in zip(feats, taps["dec_feats"]))
        raw = vt.out_dpt([[f] for f in taps["dec_feats"]], Hp, Wp, patch_size=8)
        want_raw = orc.dpt_head(sd, p + "out_dpt.", taps["dec_feats"], Hp, Wp, 8)
        case["dpt_shape_ok"] = list(raw.shape) == list(want_raw.shape)
        case["dpt_max_abs"] = float((raw - want_raw).abs().max()) if case["dpt_shape_ok"] else None
        case["dpt_range"] = float(want_raw.max() - want_raw.min())
    out["cases"].append(case)
print("LIVE_JSON " + json.dumps(out))
"""


@pytest.mark.skipif(find_reference() is None, reason="no reference here (RFB_REFERENCE, baseline/_ref and /root/reference absent)")
def test_reference_view_stage_on_non_square_ray_map_equals_oracle():
    """The unmodified reference's view stage on H != W ray maps (tiny_swin 128x192 and 192x128, tiny_full 64x136)
    equals the oracle's view_stage: at model level (ViewTransformer.forward) unless the reference itself rejects the
    non-square map there, and always for TransformerDecoder + DPTHead with patch_h != patch_w.  Runs in a
    subprocess, like test_oracle_live_reference.py, so that the reference's `renderformer` package does not
    replace this repository's drop-in package."""
    r = subprocess.run([sys.executable, "-c", WORKER % {"root": ROOT}], capture_output=True, text=True, timeout=900, cwd=ROOT)
    lines = [ln for ln in r.stdout.splitlines() if ln.startswith("LIVE_JSON ")]
    assert r.returncode == 0 and lines, (r.stdout[-800:], r.stderr[-1500:])
    out = json.loads(lines[-1][len("LIVE_JSON "):])
    assert len(out["cases"]) == 3
    for c in out["cases"]:
        print(c)
        if "vt_error" not in c:
            assert c["vt_shape_ok"] and c["vt_max_abs"] <= 1e-4 * max(1.0, c["range"]), c
        assert c["dec_max_rel"] <= 1e-4, c
        assert c["dpt_shape_ok"] and c["dpt_max_abs"] <= 1e-4 * max(1.0, c["dpt_range"]), c
