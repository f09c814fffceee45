#!/usr/bin/env python
"""What a lens-distorted camera costs against the same camera as plain pinhole intrinsics: `render(...,
intrinsics=K)`, `render(..., intrinsics=K, distortion=D, lens="opencv")` and `render(..., intrinsics=Kf,
distortion=Df, lens="fisheye")` timed round-robin (`--rounds` rounds of `--steps` calls each, per-camera median), so
that clock or neighbour drift favours none.  Only the ray-token kernel differs: the lens kernel inverts the lens per
pixel by Newton's method.  Its own time is measured too, with CUDA events around `--kernel-reps` launches of one
decoder pass's worth of views (`view_chunk`) on the canvas, against the pinhole intrinsics kernel's.

Workload: V1.1-swin-Large with seeded random weights, one scene of 4096 triangles, 16 views per call rendered as
decoder passes of 8 views, CUDA graphs, bf16 operands, 1080x1920 with overscan (the 1088x1920 canvas).  The cameras:
a calibrated-looking K (fy = 1.02 fx, the principal point a few pixels off the centre) with a 55-degree field of view
and an OpenCV barrel lens (k1 = -0.12, k2 = 0.02), and a wide fisheye (k1 = -0.01, k2 = 0.001) whose image corners are
more than 100 degrees off the axis.

usage: python tools/lens_bench.py [--size 1080x1920] [--no-overscan] [--views 16] [--steps 5] [--rounds 4]
Prints one JSON line per camera and writes nothing."""
import argparse
import json
import math
import os
import statistics
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))


def main(argv=None) -> int:
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--size", default="1080x1920", help="HxW")
    ap.add_argument("--no-overscan", action="store_true")
    ap.add_argument("--config", default="v1_1_swin_large")
    ap.add_argument("--tris", type=int, default=4096)
    ap.add_argument("--views", type=int, default=16)
    ap.add_argument("--view-chunk", type=int, default=8)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--rounds", type=int, default=4)
    ap.add_argument("--kernel-reps", type=int, default=200)
    args = ap.parse_args(argv)
    hw = tuple(int(s) for s in args.size.lower().split("x"))
    overscan = not args.no_overscan

    import torch
    from aspect_bench import gpu_info
    from renderformer_b200 import ops
    from renderformer_b200.config import RenderFormerConfig, view_camera
    from renderformer_b200.model import RenderFormer, RenderFormerRenderingPipeline
    from renderformer_b200.synth import init_state_dict, make_scene

    if not torch.cuda.is_available():
        raise SystemExit("lens_bench.py needs a CUDA device: the product path has no CPU fallback")
    dev = torch.device("cuda", 0)
    cfg = RenderFormerConfig.named(args.config)
    model = RenderFormer(cfg)
    model.load_state_dict(init_state_dict(cfg, 7))
    pipe = RenderFormerRenderingPipeline(model)
    pipe.to(dev)
    pipe.cuda_graphs = True
    pipe.view_chunk = args.view_chunk
    sc = {k: v.to(dev) for k, v in make_scene(args.tris, args.views, seed=0).items()}
    geo = (sc["triangles"], sc["texture"], sc["mask"], sc["vn"], sc["c2w"])
    H, W = hw
    V = args.views
    f = max(H, W) / 2 / math.tan(math.radians(55.0) / 2)
    ff = max(H, W) / 2 / 1.75   # fisheye: half the longer side reaches 1.75 rad, the corners more than 100 degrees
    K = torch.tensor([[[f, 1.02 * f, W / 2 + 3.5, H / 2 - 2.25]] * V])
    Kf = torch.tensor([[[ff, 1.02 * ff, W / 2 + 3.5, H / 2 - 2.25]] * V])
    Do = torch.tensor([[[-0.12, 0.02, 0.0, 0.0, 0.0, 0.0, 0.0, 0.0]] * V])
    Df = torch.tensor([[[-0.01, 0.001, 0.0, 0.0]] * V])
    cams = {"pinhole": dict(intrinsics=K), "opencv": dict(intrinsics=K, distortion=Do, lens="opencv"),
            "fisheye": dict(intrinsics=Kf, distortion=Df, lens="fisheye")}
    canvas, window, _ = pipe.view_geometry(hw, overscan)
    for c in cams.values():   # the host check once, then the cameras live on the device as a renderer keeps them
        view_camera(sc["c2w"].cpu(), canvas=canvas, window=window, **c)
    cams = {k: {n: (t.to(dev) if isinstance(t, torch.Tensor) else t) for n, t in c.items()} for k, c in cams.items()}

    def call(kind):
        return pipe.render(*geo, resolution=hw, torch_dtype=torch.bfloat16, overscan=overscan, **cams[kind])

    for kind in cams:
        for _ in range(args.warmup):
            call(kind)
    torch.cuda.synchronize()
    ms = {kind: [] for kind in cams}
    for _ in range(args.rounds):
        for kind in cams:
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(args.steps):
                call(kind)
            e1.record()
            torch.cuda.synchronize()
            ms[kind].append(e0.elapsed_time(e1) / args.steps)

    # the ray-token kernel alone: one decoder pass of view_chunk views on the canvas
    n = min(args.view_chunk, V)
    Hc, Wc = canvas
    h, w, top, left = (Hc, Wc, 0, 0) if window is None else window
    tok = torch.empty(n * (Hc // 8) * (Wc // 8), 192, dtype=torch.float16, device=dev)
    geom = dict(n_views=n, canvas_h=Hc, canvas_w=Wc, height=h, width=w, top=top, left=left)

    def kernel(kind):
        k = cams[kind]["intrinsics"][0, :n]
        if kind == "pinhole":
            return ops.ray_tokens_intrinsics(k, tok, **geom)
        return ops.ray_tokens_lens(k, cams[kind]["distortion"][0, :n], tok, lens=kind, **geom)

    us = {}
    for kind in cams:
        for _ in range(10):
            kernel(kind)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(args.kernel_reps):
            kernel(kind)
        e1.record()
        torch.cuda.synchronize()
        us[kind] = e0.elapsed_time(e1) * 1e3 / args.kernel_reps

    info = gpu_info(dev)
    for kind in cams:
        t = statistics.median(ms[kind])
        print(json.dumps({"camera": kind, "size": f"{H}x{W}", "overscan": overscan, "ms_per_call": round(t, 3),
                          "ms_rounds": [round(x, 3) for x in ms[kind]], "frames_per_s": round(V / (t * 1e-3), 2),
                          "ray_token_kernel_us_per_pass": round(us[kind], 2), "views_per_kernel_launch": n,
                          "canvas": f"{Hc}x{Wc}", "config": args.config, "tris": args.tris, "views": V,
                          "views_per_pass": pipe.view_chunk, "cuda_graphs": True, "dtype": "bf16", **info}), flush=True)
    return 0


if __name__ == "__main__":
    sys.exit(main())
