#!/usr/bin/env python
"""Throughput of non-square images: frames/s and megapixels/s of `RenderFormerRenderingPipeline.render` at several
(height, width) sizes, square and non-square at equal pixel counts side by side.

Workload: V1.1-swin-Large with seeded random weights, one scene of 4096 triangles, 32 views per call rendered as
decoder passes of 8 views, CUDA graphs, bf16 operands -- bench.py's flagship job with only the image size changed.
The sizes are timed round-robin (`--rounds` rounds of `--steps` calls each, per-size median), so that clock or
neighbour drift does not favour one size.  `--kernels` additionally lists, per size, the CUDA kernels with the most
device time in one profiled call (torch.profiler, a separate pass after the timing).

`--overscan` renders every size with `render(..., overscan=True)`, so sizes off the decoder's grid (720x1280,
1080x1920, 1440x2560, 2160x3840) are rendered on the smallest canvas on the grid and cropped; a size on the grid
(1088x1920) renders exactly as without overscan and, timed in the same round-robin, shows what the crop costs.  Per
size the table adds the canvas overhead (extra canvas pixels in % of the output) and the peak memory of the run:
the memory the model and the scene hold plus the peak a call of that size adds on top (torch.cuda.max_memory_allocated
around its warm-up and CUDA-graph capture; graphs of the other sizes are excluded).

usage: python tools/aspect_bench.py [--sizes 512x512,256x1024,1024x256,1024x576,576x1024] [--overscan] [--steps 10]
           [--rounds 3] [--views 32] [--view-chunk 8] [--tris 4096] [--kernels]
       python tools/aspect_bench.py --overscan --sizes 720x1280,1080x1920,1088x1920,1440x2560,2160x3840
Prints one JSON line per size and a summary table; writes nothing."""
import argparse
import json
import os
import statistics
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))


def parse_sizes(text):
    out = []
    for tok in text.split(","):
        h, w = tok.lower().split("x")
        out.append((int(h), int(w)))
    return out


def gpu_info(dev):
    import torch
    info = {"gpu": torch.cuda.get_device_name(dev)}
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader",
                            "-i", str(dev.index or 0)], capture_output=True, text=True, timeout=30)
        info["power_limit_and_max_sm_clock"] = q.stdout.strip()
    except (OSError, subprocess.SubprocessError):
        info["power_limit_and_max_sm_clock"] = "unavailable"
    return info


def main(argv=None) -> int:
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--sizes", default="512x512,256x1024,1024x256,1024x576,576x1024", help="HxW list")
    ap.add_argument("--config", default="v1_1_swin_large")
    ap.add_argument("--tris", type=int, default=4096)
    ap.add_argument("--views", type=int, default=32)
    ap.add_argument("--view-chunk", type=int, default=8)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--overscan", action="store_true", help="render(..., overscan=True): any size, cropped from the grid")
    ap.add_argument("--kernels", action="store_true", help="list the top kernels per size (torch.profiler)")
    args = ap.parse_args(argv)
    sizes = parse_sizes(args.sizes)

    import torch
    from renderformer_b200.config import RenderFormerConfig, overscan_grid, view_grid
    from renderformer_b200.flops import job_flops
    from renderformer_b200.model import RenderFormer, RenderFormerRenderingPipeline
    from renderformer_b200.synth import init_state_dict, make_scene

    if not torch.cuda.is_available():
        raise SystemExit("aspect_bench.py needs a CUDA device: the product path has no CPU fallback")
    dev = torch.device("cuda", 0)
    cfg = RenderFormerConfig.named(args.config)
    canvas = {}
    for hw in sizes:  # reject an unsupported size before the model is built
        canvas[hw] = overscan_grid(cfg, hw)[1] if args.overscan else view_grid(cfg, hw)
    model = RenderFormer(cfg)
    model.load_state_dict(init_state_dict(cfg, 7))
    pipe = RenderFormerRenderingPipeline(model)
    pipe.to(dev)
    pipe.cuda_graphs = True
    pipe.view_chunk = args.view_chunk
    pipe.max_cached_graphs = len(sizes)
    sc = {k: v.to(dev) for k, v in make_scene(args.tris, args.views, seed=0).items()}
    inputs = (sc["triangles"], sc["texture"], sc["mask"], sc["vn"], sc["c2w"], sc["fov"])

    def call(hw):
        return pipe.render(*inputs, resolution=hw, torch_dtype=torch.bfloat16, overscan=args.overscan)

    torch.cuda.synchronize()
    base = torch.cuda.memory_allocated(dev)  # model weights + scene inputs
    peak = {}
    for hw in sizes:
        torch.cuda.synchronize()
        before = torch.cuda.memory_allocated(dev)
        torch.cuda.reset_peak_memory_stats(dev)
        for _ in range(max(args.warmup, 3)):
            call(hw)
        torch.cuda.synchronize()
        peak[hw] = base + torch.cuda.max_memory_allocated(dev) - before

    ms = {hw: [] for hw in sizes}
    for _ in range(args.rounds):
        for hw in sizes:
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(args.steps):
                call(hw)
            e1.record()
            torch.cuda.synchronize()
            ms[hw].append(e0.elapsed_time(e1) / args.steps)

    info = gpu_info(dev)
    ref = sizes[0]
    ref_px_rate = None
    rows = []
    for hw in sizes:
        t = statistics.median(ms[hw])
        fps = args.views / (t * 1e-3)
        mpx = fps * hw[0] * hw[1] / 1e6
        ref_px_rate = mpx if hw == ref else ref_px_rate
        Hc, Wc = canvas[hw]
        res = {"size": f"{hw[0]}x{hw[1]}", "canvas": f"{Hc}x{Wc}", "overscan": args.overscan,
               "canvas_overhead_pct": round(100.0 * (Hc * Wc / (hw[0] * hw[1]) - 1.0), 2),
               "ms_per_call": round(t, 3), "ms_spread": [round(min(ms[hw]), 3), round(max(ms[hw]), 3)],
               "frames_per_s": round(fps, 2), "megapixels_per_s": round(mpx, 2),
               "megapixels_per_s_vs_first": round(mpx / ref_px_rate, 4),
               "tflop_per_s": round(job_flops(cfg, args.tris, hw, 1, args.views, args.overscan) / (t * 1e-3) / 1e12, 1),
               "max_memory_allocated_gb": round(peak[hw] / 1e9, 2),
               "config": args.config, "tris": args.tris, "views": args.views, "views_per_pass": pipe.view_chunk,
               "cuda_graphs": True, "dtype": "bf16", **info}
        rows.append(res)
        print(json.dumps(res), flush=True)
    print(f"\n{'size':>10} {'canvas':>10} {'overhead':>8} {'ms/call':>9} {'frames/s':>9} {'MP/s':>8} "
          f"{'MP/s vs ' + rows[0]['size']:>16} {'peak GB':>8}")
    for r in rows:
        print(f"{r['size']:>10} {r['canvas']:>10} {r['canvas_overhead_pct']:7.2f}% {r['ms_per_call']:9.2f} "
              f"{r['frames_per_s']:9.1f} {r['megapixels_per_s']:8.1f} {r['megapixels_per_s_vs_first']:16.3f} "
              f"{r['max_memory_allocated_gb']:8.2f}")
    print(f"({info['gpu']}, power limit / max SM clock: {info['power_limit_and_max_sm_clock']})")

    if args.kernels:
        from torch.profiler import ProfilerActivity, profile
        pipe.cuda_graphs = False  # the same kernels, launched one by one so that every launch is recorded
        for hw in sizes:
            call(hw)
            torch.cuda.synchronize()
            with profile(activities=[ProfilerActivity.CUDA]) as prof:
                call(hw)
                torch.cuda.synchronize()
            tot = {}
            for ev in prof.events():
                if ev.device_type == torch.autograd.DeviceType.CUDA:
                    n, t = tot.get(ev.name, (0, 0.0))
                    tot[ev.name] = (n + 1, t + ev.device_time_total / 1e3)
            print(f"\n-- {hw[0]}x{hw[1]}: kernels by device time in one call (ms, launches)")
            for name, (n, t) in sorted(tot.items(), key=lambda kv: -kv[1][1])[:12]:
                print(f"{t:9.3f} {n:5d}  {name[:110]}")
    return 0


if __name__ == "__main__":
    sys.exit(main())
