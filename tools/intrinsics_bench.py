#!/usr/bin/env python
"""What a camera given as pinhole intrinsics costs against the same camera given as a field of view:
`render(..., fov=fov)` and `render(..., intrinsics=pipe.intrinsics_from_fov(fov, size))` timed round-robin
(`--rounds` rounds of `--steps` calls each, per-camera median), so that clock or neighbour drift favours neither.
The two renders are bit-identical (the script checks it); only the ray-token kernel differs, which reads four floats
per view instead of deriving the focal length from the fov.

Workload: V1.1-swin-Large with seeded random weights, one scene of 4096 triangles, 16 views per call rendered as
decoder passes of 8 views, CUDA graphs, bf16 operands, 1080x1920 with overscan (the 1088x1920 canvas).

usage: python tools/intrinsics_bench.py [--size 1080x1920] [--no-overscan] [--views 16] [--steps 5] [--rounds 4]
Prints one JSON line per camera kind and writes nothing."""
import argparse
import json
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
    args = ap.parse_args(argv)
    hw = tuple(int(s) for s in args.size.lower().split("x"))
    overscan = not args.no_overscan

    import torch
    from aspect_bench import gpu_info
    from renderformer_b200.config import RenderFormerConfig
    from renderformer_b200.model import RenderFormer, RenderFormerRenderingPipeline
    from renderformer_b200.synth import init_state_dict, make_scene

    if not torch.cuda.is_available():
        raise SystemExit("intrinsics_bench.py needs a CUDA device: the product path has no CPU fallback")
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
    cams = {"fov": {"fov": sc["fov"]}, "intrinsics": {"intrinsics": pipe.intrinsics_from_fov(sc["fov"], hw)}}

    def call(kind):
        return pipe.render(*geo, resolution=hw, torch_dtype=torch.bfloat16, overscan=overscan, **cams[kind])

    for kind in cams:
        for _ in range(args.warmup):
            call(kind)
    identical = torch.equal(call("fov"), call("intrinsics"))
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
    info = gpu_info(dev)
    for kind in cams:
        t = statistics.median(ms[kind])
        print(json.dumps({"camera": kind, "size": f"{hw[0]}x{hw[1]}", "overscan": overscan, "ms_per_call": round(t, 3),
                          "ms_rounds": [round(x, 3) for x in ms[kind]], "frames_per_s": round(args.views / (t * 1e-3), 2),
                          "bit_identical_to_fov": identical, "config": args.config, "tris": args.tris,
                          "views": args.views, "views_per_pass": pipe.view_chunk, "cuda_graphs": True, "dtype": "bf16",
                          **info}), flush=True)
    return 0 if identical else 1


if __name__ == "__main__":
    sys.exit(main())
