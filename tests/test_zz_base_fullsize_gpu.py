"""GPU: BASELINE configs[0] literally -- RenderFormer-V1-Base (205M: d = 768, 6 heads, FULL ray self-attention over
the 4096 ray tokens of a 512 x 512 view, DPT 128 / [96, 192, 384, 768]) on the converted examples/cbox.json scene
(5633 triangles), one view, against the golden frame of the unmodified reference (tests/golden/base_cbox_512.npz,
oracle == reference to 0.0 when it was made).

The V1-Base architecture is also checked at 256 triangles / 64 x 64 (`base_small` in tests/test_parity_gpu.py); this
case adds the full-size shapes of its full-attention decoder.  It runs in a subprocess, so that whatever happens cannot
disturb the other GPU tests, and comes last (file name)."""
import json
import os
import subprocess
import sys

import pytest

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

WORKER = r"""
import json, os, sys
import numpy as np, torch
sys.path.insert(0, %(root)r)
from renderformer_b200 import scene_io as sio
from renderformer_b200.config import RenderFormerConfig
from renderformer_b200.metrics import hdr_rel_err, log_psnr
from renderformer_b200.model import RenderFormer, RenderFormerRenderingPipeline
from renderformer_b200.synth import init_state_dict
gd = os.path.join(%(root)r, "tests", "golden")
c = json.load(open(os.path.join(gd, "manifest.json")))["cases"]["base_cbox_512"]
cfg = RenderFormerConfig.named(c["config"])
model = RenderFormer(cfg)
model.load_state_dict(init_state_dict(cfg, c["weight_seed"]))
pipe = RenderFormerRenderingPipeline(model)
pipe.to(torch.device("cuda:0"))
sc = {k: v.cuda() for k, v in sio.to_pipeline_inputs(sio.load_npz(os.path.join(gd, "cbox_scene.npz"))).items()}
ref = torch.from_numpy(np.load(os.path.join(gd, "base_cbox_512.npz"))["hdr"])
out = {}
for tag, dt in (("fp16", torch.float16), ("bf16", torch.bfloat16)):
    img = pipe(sc["triangles"], sc["texture"], sc["mask"], sc["vn"], sc["c2w"], sc["fov"], resolution=c["resolution"], torch_dtype=dt)
    torch.cuda.synchronize()
    out[tag] = {"shape_ok": list(img.shape) == list(ref.shape), "finite": bool(torch.isfinite(img).all()),
                "rel": float(hdr_rel_err(img, ref)), "psnr": float(log_psnr(img, ref))}
print("BASE_JSON " + json.dumps(out))
"""


def test_v1_base_cbox_512_against_reference_golden():
    from renderformer_b200.metrics import PSNR_MIN, REL_TOL
    r = subprocess.run([sys.executable, "-c", WORKER % {"root": ROOT}], capture_output=True, text=True, timeout=600, cwd=ROOT)
    lines = [ln for ln in r.stdout.splitlines() if ln.startswith("BASE_JSON ")]
    assert r.returncode == 0 and lines, (r.stdout[-1500:], r.stderr[-3000:])
    out = json.loads(lines[-1][len("BASE_JSON "):])
    print("base_cbox_512:", out)
    for tag in ("fp16", "bf16"):
        assert out[tag]["shape_ok"] and out[tag]["finite"], out
    # fp16 operands are the reference CLIs' default precision and the one BASELINE configs[0] / [1] are quoted in;
    # bf16 on this 5633-triangle scene is held to 3e-2 like the Large fixture of the same scene (DESIGN.md §2)
    assert out["fp16"]["rel"] <= REL_TOL and out["fp16"]["psnr"] >= PSNR_MIN, out
    assert out["bf16"]["rel"] <= 3e-2 and out["bf16"]["psnr"] >= PSNR_MIN, out
