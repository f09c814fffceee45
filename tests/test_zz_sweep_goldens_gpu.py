"""GPU: three more corners of the BASELINE configs[4] sweep (triangles 512-4096 x resolution 256^2-1024^2) against golden
frames of the unmodified reference -- V1.1-swin-Large at (512 triangles, 256^2), (2048 triangles, 2 views, 512^2) and
(4096 triangles, 1024^2).  tests/test_parity_gpu.py already holds (4096, 512^2), (1024, 1024^2) and (8192, 256^2).

Same rendering code path as the parity tests, held to the same tolerances.  The cases run in ONE subprocess (one model
initialisation) and sort last."""
import json
import os
import subprocess
import sys

import pytest

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
NAMES = ["large_512_256", "large_2048_512", "large_4096_1024"]

WORKER = r"""
import json, os, sys
import numpy as np, torch
sys.path.insert(0, %(root)r)
from renderformer_b200.config import RenderFormerConfig
from renderformer_b200.metrics import hdr_rel_err, log_psnr
from renderformer_b200.model import RenderFormer, RenderFormerRenderingPipeline
from renderformer_b200.synth import init_state_dict, make_scene
gd = os.path.join(%(root)r, "tests", "golden")
cases = json.load(open(os.path.join(gd, "manifest.json")))["cases"]
cfg = RenderFormerConfig.named("v1_1_swin_large")
model = RenderFormer(cfg)
model.load_state_dict(init_state_dict(cfg, 7))
pipe = RenderFormerRenderingPipeline(model)
pipe.to(torch.device("cuda:0"))
out = {}
for name in %(names)r:
    c = cases[name]
    assert c["config"] == "v1_1_swin_large" and c["weight_seed"] == 7 and c.get("batch", 1) == 1
    sc = {k: v.cuda() for k, v in make_scene(c["n_tris"], c["views"], seed=c["scene_seed"], pad_to=c["pad_to"]).items()}
    ref = torch.from_numpy(np.load(os.path.join(gd, name + ".npz"))["hdr"])
    hs = c.get("hdr_stride", 1)
    out[name] = {}
    for tag, dt in (("fp16", torch.float16), ("bf16", torch.bfloat16)):
        img = pipe(sc["triangles"], sc["texture"], sc["mask"], sc["vn"], sc["c2w"], sc["fov"], resolution=c["resolution"], torch_dtype=dt)
        torch.cuda.synchronize()
        sub = img[:, :, ::hs, ::hs]
        out[name][tag] = {"shape_ok": list(sub.shape) == list(ref.shape), "finite": bool(torch.isfinite(img).all()),
                          "rel": float(hdr_rel_err(sub, ref)), "psnr": float(log_psnr(sub, ref))}
    del sc
    torch.cuda.empty_cache()
print("SWEEP_JSON " + json.dumps(out))
"""

_RESULT = {}


def _results():
    if not _RESULT:
        r = subprocess.run([sys.executable, "-c", WORKER % {"root": ROOT, "names": NAMES}], capture_output=True, text=True,
                           timeout=900, cwd=ROOT)
        lines = [ln for ln in r.stdout.splitlines() if ln.startswith("SWEEP_JSON ")]
        _RESULT["out"] = json.loads(lines[-1][len("SWEEP_JSON "):]) if (r.returncode == 0 and lines) else None
        _RESULT["log"] = (r.stdout[-1500:], r.stderr[-3000:])
    return _RESULT


@pytest.mark.parametrize("name", NAMES)
def test_sweep_corner_against_reference_golden(name):
    from renderformer_b200.metrics import PSNR_MIN, REL_TOL
    res = _results()
    assert res["out"] is not None, res["log"]
    out = res["out"][name]
    print(name, out)
    for tag in ("fp16", "bf16"):
        assert out[tag]["shape_ok"] and out[tag]["finite"], out
        assert out[tag]["rel"] <= REL_TOL and out[tag]["psnr"] >= PSNR_MIN, out
