#!/usr/bin/env python
"""Headline benchmark: frames/sec of the RenderFormer-V1.1-swin-Large forward pass on a synthetic
4096-triangle scene at 512x512 (BASELINE.json metric), N GPUs of one node.

    python bench.py --gpus 1 --steps 10 --warmup 3
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...
    python bench.py --impl reference ...   # CPU arm: the UNMODIFIED reference's PyTorch path on the host cores

One step = ONE JOB of fixed size: one scene through the view-independent stage and `--total-views`
(32: BASELINE configs[2]) camera views of an orbit through the view-dependent stage, at any N
("scaling": "strong").  At N > 1 the scene stage is row-sharded over the ranks (per encoder layer every rank
stores its k | v rows into all ranks' memories through the NVLS multicast address -- the exchange is fused into
the producing kernel -- and the ranks meet at a signal-pad barrier; NCCL all-gather with RFB_KV_PUSH=0), every
rank renders total_views / N views, the images are gathered on rank 0.
`--views-per-gpu V` switches to the weak-scaling job (V views on every GPU).
Prints ONE JSON line on rank 0 (contract: see the task statement / DESIGN.md §5).
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

# NCCL writes its debug / version banner to stdout by default; the contract is ONE JSON line there
os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")
if os.environ.get("NCCL_DEBUG", "").upper() in ("", "VERSION"):
    os.environ["NCCL_DEBUG"] = "WARN"

import torch  # noqa: E402

METRIC = "frames/sec (512^2, 4096 tris)"
UNIT = "frames/s"


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", default="v1_1_swin_large")
    ap.add_argument("--tris", type=int, default=4096)
    ap.add_argument("--resolution", type=int, default=512)
    ap.add_argument("--total-views", type=int, default=32, help="views of the fixed job (strong scaling)")
    ap.add_argument("--views-per-gpu", type=int, default=0, help="> 0: weak scaling, this many views on every GPU")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-roofline", action="store_true")
    ap.add_argument("--no-ref-cuda", action="store_true", help="skip the reference-on-CUDA context arm (N=1 only)")
    ap.add_argument("--no-cuda-graphs", action="store_true", help="launch every kernel from Python")
    ap.add_argument("--view-chunk", type=int, default=8, help="views per decoder pass (capped by the views a rank renders)")
    ap.add_argument("--view-streams", type=int, default=1, help="CUDA streams the view chunks are spread over")
    ap.add_argument("--ref-cuda-worker", default="", help=argparse.SUPPRESS)
    ap.add_argument("--dump-outputs", default="", metavar="DIR",
                    help="write the images the last timed step returned to DIR/image.npy (float32 [1, V, R, R, 3]); "
                         "when they exceed 64 MB, a fixed seeded sample of their pixels to DIR/image_sample.npy instead")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    return args


DUMP_BYTES = 64_000_000
DUMP_SEED = 0


def dump_images(img: torch.Tensor, out_dir: str) -> str:
    """Write the images of one job as float32 .npy under out_dir; returns the file written.  Above DUMP_BYTES the
    file holds the RGB values of a sample of pixels instead: positions drawn without replacement from all views
    with numpy's default_rng(DUMP_SEED), in increasing flat order, so the same job always yields the same sample."""
    import numpy as np
    arr = img.detach().float().cpu().numpy()
    os.makedirs(out_dir, exist_ok=True)
    if arr.nbytes + 4096 <= DUMP_BYTES:
        path = os.path.join(out_dir, "image.npy")
    else:
        pixels = arr.reshape(-1, arr.shape[-1])
        n = (DUMP_BYTES - 4096) // pixels[0].nbytes
        idx = np.sort(np.random.default_rng(DUMP_SEED).choice(pixels.shape[0], size=n, replace=False))
        arr = pixels[idx]
        path = os.path.join(out_dir, "image_sample.npy")
    np.save(path, arr)
    return path


def load_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as f:
            p = json.load(f)
        return p.get("bf16_tflops_sustained", p.get("bf16_tflops")), p.get("hbm_gbs"), "measured (MEASURED_PEAKS.json, sustained)"
    return 1400.0, 6650.0, "fallback (B200_PROFILING.md)"


def job_views(args, world):
    return args.views_per_gpu * world if args.views_per_gpu > 0 else args.total_views


def kv_exchange_text() -> str:
    """How the row-sharded scene stage moved a layer's k | v rows between the ranks in THIS run."""
    from renderformer_b200 import dist as rdist
    if rdist._KV_STORES:
        mc = next(iter(rdist._KV_STORES.values())).multicast
        how = "NVLS multicast stores" if mc else "peer-mapped NVLink stores"
        return (f"per encoder layer every rank's k|v rows go to all ranks by {how} fused into the kernel that produces "
                "them (rfb_qkv_post) + one signal-pad barrier; one NCCL all-gather of the final 16-bit stream")
    return "one NCCL all-gather of the ranks' 16-bit k|v rows per encoder layer"


def workload_text(args, world):
    V = job_views(args, world)
    kind = (f"{args.views_per_gpu} views on every GPU (weak scaling)" if args.views_per_gpu > 0 else
            f"fixed job of {V} views (strong scaling; BASELINE configs[2] at 32)")
    try:  # parameter count of the named architecture (483M for the metric's v1_1_swin_large)
        import math
        from renderformer_b200.config import RenderFormerConfig
        from renderformer_b200.synth import state_dict_shapes
        n_par = sum(math.prod(s) for s in state_dict_shapes(RenderFormerConfig.named(args.config)).values())
        size = f"{n_par / 1e6:.0f}M" if n_par >= 1e6 else f"{n_par / 1e3:.0f}k"
    except Exception:  # noqa: BLE001
        size = "?"
    return (f"{args.config} ({size}, random-init weights, seed 7), synthetic {args.tris}-triangle scene (seed 0), "
            f"{args.resolution}x{args.resolution}, one scene + {V}-view camera orbit per step: {kind}")


# --------------------------------------------------------------------------- CPU arms
def _reference_or_port(cfg, sd):
    """(render(scene, res) -> image, kind, description).  The unmodified reference when it can be imported
    (baseline/_ref or /root/reference), else the oracle port."""
    try:
        from oracle.reference_loader import build_reference_pipeline
        pipe, ref = build_reference_pipeline(cfg, sd, "cpu", "sdpa")

        def render(sc, res):
            return pipe(sc["triangles"], sc["texture"].clone(), sc["mask"], sc["vn"], sc["c2w"], sc["fov"],
                        resolution=res, torch_dtype=torch.float32)
        return render, "reference", f"unmodified reference from {os.path.relpath(ref, ROOT) if ref.startswith(ROOT) else ref}, " \
                                    "RenderFormerRenderingPipeline(torch_dtype=float32), ATTN_IMPL=sdpa"
    except Exception as e:  # noqa: BLE001  (reference not installed on this box)
        from oracle import renderformer_oracle as orc

        def render(sc, res):
            return orc.render(sd, cfg, sc["triangles"], sc["texture"], sc["mask"], sc["vn"], sc["c2w"], sc["fov"], res)
        return render, "port", f"oracle port (reference unavailable: {str(e)[:80]})"


def cpu_arm(args, views: int, steps: int, warm_small: bool = True):
    """Time the reference's CPU path (fp32, all host threads) on `views` views of the bench scene at the
    metric's own triangle count and resolution.  Returns a dict(value, ms, cores, kind, sample)."""
    from renderformer_b200.config import RenderFormerConfig
    from renderformer_b200.synth import init_state_dict, make_scene
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    cfg = RenderFormerConfig.named(args.config)
    sd = init_state_dict(cfg, 7)
    render, kind, what = _reference_or_port(cfg, sd)
    full = make_scene(args.tris, job_views(args, 1), seed=0)
    sc = dict(full, c2w=full["c2w"][:, :views].contiguous(), fov=full["fov"][:, :views].contiguous())
    with torch.no_grad():
        if warm_small:  # thread pool / allocator warm-up on a small frame; the timed calls are full size
            tiny = make_scene(64, 1, seed=1)
            render(tiny, 64)
        times = []
        for _ in range(max(1, steps)):
            t0 = time.perf_counter()
            render(sc, args.resolution)
            times.append(time.perf_counter() - t0)
    dt = statistics.median(times)
    return {"value": views / dt, "ms": dt * 1e3, "cores": cores, "kind": kind, "views": views,
            "sample": f"{what}; {cores} torch threads; {args.tris} triangles, {views} of the job's views at "
                      f"{args.resolution}x{args.resolution} in one call (scene stage + {views} views), "
                      f"median of {len(times)} call(s): {dt:.2f} s"}


def run_reference(args):
    """--impl reference: the reference's own CPU implementation (unmodified, baseline/_ref) on the metric's
    config.  A step is the WHOLE job -- the scene and all of its views in one pipeline call, as the
    reference's batch CLI issues it -- timed once after a small warm-up call (about 70 s on the GPU box's 16
    cores, ~22 GB of host memory measured at 0.55 GB per view + 4 GB).  Only if the host has too little free
    memory for that is a bounded sample used instead: the scene stage plus 8 of the job's views in one call,
    whose per-frame figure is reported as is (the scene stage is then amortised over fewer views, which makes
    the reference look ~8 % slower per frame than on the full job; `sample` says which was run)."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    V = job_views(args, max(1, args.gpus))
    try:
        import psutil
        free_gb = psutil.virtual_memory().available / 2 ** 30
    except Exception:  # noqa: BLE001
        free_gb = 0.0
    full = free_gb >= 1.5 * (0.55 * V + 4.0) + 8.0
    sample_views = V if full else min(V, 8)
    steps = 1 if sample_views > 8 else min(max(1, args.steps), 2)
    r = cpu_arm(args, sample_views, steps)
    line = {
        "impl": "reference", "metric": METRIC, "value": r["value"], "unit": UNIT, "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": r["ms"], "higher_is_better": True,
        "scaling": "weak" if args.views_per_gpu > 0 else "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": workload_text(args, max(1, args.gpus)),
                   "timed": f"{steps} timed call(s) of scene + {sample_views} views "
                            f"({'the whole job' if sample_views == V else f'bounded sample of the {V}-view job'}), "
                            f"1 small warm-up call; the driver's --steps/--warmup are capped to keep the run within minutes"},
        "cpu_baseline": {"value": r["value"], "unit": UNIT, "cores": r["cores"], "kind": r["kind"], "sample": r["sample"]},
        "e2e": {"value": r["value"], "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


# --------------------------------------------------------------------------- reference on CUDA (context)
def ref_cuda_worker(args):
    """Subprocess body: the UNMODIFIED reference on cuda:0 through its own pipeline API, same scene / weights
    / job as the bench step.  Variants (BASELINE.md §3.2): its shipped default for bf16 (`torch_dtype=bfloat16`:
    encoder bf16, view transformer fp32/TF32 with forced SDPA, allow_tf32 as batch_infer.py:86-87), and the
    'fair bf16' call of model.forward(tf32_view_tf=False) under bf16 autocast.  Prints one JSON line."""
    attn = args.ref_cuda_worker
    out = {"attn_impl": attn}
    try:
        from oracle.reference_loader import build_reference_pipeline
        from renderformer_b200.config import RenderFormerConfig
        from renderformer_b200.metrics import hdr_rel_err
        from renderformer_b200.synth import init_state_dict, make_scene
        dev = torch.device("cuda:0")
        cfg = RenderFormerConfig.named(args.config)
        pipe, ref = build_reference_pipeline(cfg, init_state_dict(cfg, 7), dev, attn)
        torch.backends.cuda.matmul.allow_tf32 = True
        torch.backends.cudnn.allow_tf32 = True
        V = job_views(args, 1)
        sc = {k: v.to(dev) for k, v in make_scene(args.tris, V, seed=0).items()}
        chunk = min(V, 8)  # views per pipeline call (the reference re-runs its encoder in every call)

        def timed(fn, n):
            for _ in range(2):
                fn()
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(n):
                fn()
            e1.record()
            torch.cuda.synchronize()
            return e0.elapsed_time(e1) / n

        def default_call(v0=0, nv=V):
            return pipe(sc["triangles"], sc["texture"].clone(), sc["mask"], sc["vn"], sc["c2w"][:, v0:v0 + nv],
                        sc["fov"][:, v0:v0 + nv], resolution=args.resolution, torch_dtype=torch.bfloat16)

        def job(call):
            try:
                return [call(0, V)]
            except torch.OutOfMemoryError:
                torch.cuda.empty_cache()
                return [call(v0, chunk) for v0 in range(0, V, chunk)]

        ms = timed(lambda: job(default_call), 3)
        out["default_bf16"] = {"value": V / (ms * 1e-3), "unit": UNIT, "ms_per_step": ms,
                               "what": f"unmodified reference ({os.path.basename(ref)}), pipeline(torch_dtype=bfloat16), ATTN_IMPL={attn}, "
                                       "allow_tf32: encoder bf16, view transformer fp32/TF32 SDPA (its shipped behaviour)"}
        if attn == "sdpa":
            from renderformer.utils.transform import trans_to_cam_coord  # the reference's own helpers

            def fair_call(v0=0, nv=V):
                # what pipeline.render does (rendering_pipeline.py:60-125) with tf32_view_tf=False, i.e. the view
                # transformer under bf16 autocast too
                with torch.no_grad(), torch.autocast("cuda", dtype=torch.bfloat16):
                    tex = sc["texture"].clone()
                    tex[:, :, -3:] = torch.log10(tex[:, :, -3:] + 1.0)
                    c2w, fov = sc["c2w"][:, v0:v0 + nv], sc["fov"][:, v0:v0 + nv]
                    B, nv_ = c2w.shape[:2]
                    tri = sc["triangles"]
                    tri_cam, c2w_id, _ = trans_to_cam_coord(c2w.reshape(-1, 4, 4), torch.repeat_interleave(tri, nv_, dim=0))
                    rays_o, rays_d = pipe.ray_generator(c2w_id.reshape(B, nv_, 4, 4), fov / 180.0 * torch.pi, args.resolution)
                    img = pipe.model(tri.reshape(B, -1, 9), tex, sc["mask"], sc["vn"].reshape(B, -1, 9), rays_o=rays_o,
                                     rays_d=rays_d, tri_vpos_view_tf=tri_cam.reshape(B, nv_, -1, 9), tf32_view_tf=False)
                    return torch.pow(10.0, img.permute(0, 1, 3, 4, 2).float()) - 1.0
            try:
                ms_f = timed(lambda: job(fair_call), 3)
                out["fair_bf16"] = {"value": V / (ms_f * 1e-3), "unit": UNIT, "ms_per_step": ms_f,
                                    "what": "unmodified reference model.forward(tf32_view_tf=False) under bf16 autocast "
                                            "(both transformers bf16), inputs prepared like rendering_pipeline.py:60-101"}
            except Exception as e:  # noqa: BLE001
                out["fair_bf16"] = {"unavailable": repr(e)[:300]}
    except Exception as e:  # noqa: BLE001
        out["unavailable"] = repr(e)[:300]
    print("REF_CUDA_JSON " + json.dumps(out), flush=True)


def run_ref_cuda(args):
    res = {}
    for attn in ("sdpa", "flash_attn"):
        cmd = [sys.executable, os.path.abspath(__file__), "--ref-cuda-worker", attn, "--config", args.config,
               "--tris", str(args.tris), "--resolution", str(args.resolution), "--total-views", str(job_views(args, 1))]
        try:
            r = subprocess.run(cmd, capture_output=True, text=True, timeout=420, cwd=ROOT)
            line = [ln for ln in r.stdout.splitlines() if ln.startswith("REF_CUDA_JSON ")]
            res[attn] = json.loads(line[-1][len("REF_CUDA_JSON "):]) if line else {"unavailable": (r.stderr or r.stdout)[-300:]}
        except Exception as e:  # noqa: BLE001
            res[attn] = {"unavailable": repr(e)[:300]}
    return res


# --------------------------------------------------------------------------- clocks
class ClockSampler:
    """SM clock / power / throttle reasons sampled with NVML every 20 ms from a thread while the
    timed region runs (nvidia-smi's own loop is too coarse for a region of a few hundred ms)."""

    def __init__(self, index: int):
        import threading
        self.rows, self.on, self.n = [], True, None
        try:
            import pynvml
            pynvml.nvmlInit()
            self.n = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
        except Exception as e:  # noqa: BLE001
            self.err = repr(e)
            return
        self.t = threading.Thread(target=self._run, daemon=True)
        self.t.start()

    def _run(self):
        n = self.n
        while self.on:
            try:
                self.rows.append((n.nvmlDeviceGetClockInfo(self.h, n.NVML_CLOCK_SM),
                                  n.nvmlDeviceGetPowerUsage(self.h) / 1e3,
                                  n.nvmlDeviceGetCurrentClocksEventReasons(self.h)))
            except Exception:  # noqa: BLE001
                pass
            time.sleep(0.02)

    def stop(self):
        if self.n is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvml unavailable: " + getattr(self, "err", "")]}
        self.on = False
        self.t.join(timeout=2)
        n, rows = self.n, self.rows
        names = {"hw_slowdown": n.nvmlClocksEventReasonHwSlowdown,
                 "hw_thermal_slowdown": n.nvmlClocksEventReasonHwThermalSlowdown,
                 "sw_thermal_slowdown": n.nvmlClocksEventReasonSwThermalSlowdown,
                 "sw_power_cap": n.nvmlClocksEventReasonSwPowerCap,
                 "hw_power_brake": n.nvmlClocksEventReasonHwPowerBrakeSlowdown}
        bits = 0
        for r in rows:
            bits |= r[2]
        return {"sm_mhz": statistics.median(r[0] for r in rows) if rows else None, "sm_max_mhz": self.max,
                "power_w_max": max((r[1] for r in rows), default=None), "samples": len(rows),
                "reasons": sorted(k for k, v in names.items() if bits & v)}


# --------------------------------------------------------------------------- GPU arm
def main():
    args = parse()
    if args.ref_cuda_worker:
        return ref_cuda_worker(args)
    if args.impl == "reference":
        return run_reference(args)

    import torch.distributed as dist
    from renderformer_b200 import lib, ops
    from renderformer_b200.config import RenderFormerConfig
    from renderformer_b200.dist import render_sharded, render_stream_sharded, view_slice
    from renderformer_b200.flops import job_flops, scene_flops, view_flops
    from renderformer_b200.model import RenderFormer, RenderFormerRenderingPipeline
    from renderformer_b200.synth import init_state_dict, make_scene

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the product path has no CPU fallback")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)

    cfg = RenderFormerConfig.named(args.config)
    model = RenderFormer(cfg)
    model.load_state_dict(init_state_dict(cfg, 7))
    pipe = RenderFormerRenderingPipeline(model)
    pipe.to(dev)
    model.engine(torch.bfloat16)
    R, N = args.resolution, args.tris
    V = job_views(args, world)
    pipe.view_streams = args.view_streams
    mine = view_slice(V, world, rank)
    Vl = mine.stop - mine.start
    # same chunking on every rank (and in the single-GPU check render): the per-rank view count caps it
    pipe.view_chunk = max(1, min(args.view_chunk, -(-V // world)))

    scene = make_scene(N, V, seed=0)
    host = {k: v.pin_memory() for k, v in scene.items()}
    d_in = {k: v.to(dev) for k, v in host.items()}
    out_host = torch.empty((1, V if world == 1 else Vl, R, R, 3), dtype=torch.float32).pin_memory()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    graphs = not args.no_cuda_graphs

    pending = [None]  # image gather of the previous job, still travelling while this job's scene stage runs
    last = [None]  # rank 0: the images of the newest job of step_device (for --dump-outputs)

    def flush():
        """Wait for the outstanding image gather; returns the gathered images on rank 0."""
        out = None
        if pending[0] is not None:
            out = pending[0].wait()
            pending[0] = None
            if out is not None:
                last[0] = out[None]
        return out

    def step_device(inp, dst=0):
        """The whole job with inputs resident in HBM; the images end up on rank 0 (dst=0).  At N > 1 the gather of
        job k is enqueued asynchronously and waited for right after job k+1 has been launched (and before the timed
        region closes), so it overlaps the next scene stage; dst=None returns this rank's own views."""
        if world == 1:
            last[0] = pipe.render(inp["triangles"], inp["texture"], inp["mask"], inp["vn"], inp["c2w"], inp["fov"],
                                  resolution=R, torch_dtype=torch.bfloat16)
            return last[0]
        h = render_sharded(pipe, inp["triangles"], inp["texture"], inp["mask"], inp["vn"], inp["c2w"], inp["fov"],
                           resolution=R, dst=dst, torch_dtype=torch.bfloat16, async_gather=dst is not None)
        if dst is None:
            return h
        flush()
        pending[0] = h
        return h

    def step_e2e():
        """Public API with HOST buffers, one blocking call per step: H2D of the step's inputs, render, D2H."""
        inp = {k: host[k].to(dev, non_blocking=True) for k in ("triangles", "texture", "mask", "vn", "c2w", "fov")}
        img = step_device(inp, dst=None)
        out_host.copy_(img, non_blocking=False)

    def timed(fn, steps):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        barrier()
        e0.record()
        for _ in range(steps):
            fn()
        flush()  # the last job's images have arrived before the clock stops
        e1.record()
        barrier()
        ms = torch.tensor([e0.elapsed_time(e1)], device=dev)
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return ms.item() / steps

    pipe.cuda_graphs = graphs
    for _ in range(max(args.warmup, 3)):
        step_device(d_in)
    flush()
    sampler = ClockSampler(local_rank) if rank == 0 else None
    launches0 = lib.launch_count() + pipe.replayed_launches
    ms_step = timed(lambda: step_device(d_in), args.steps)
    launches = (lib.launch_count() + pipe.replayed_launches - launches0)
    clocks = sampler.stop() if sampler else None
    value = V / (ms_step * 1e-3)
    if args.dump_outputs:  # before the steps below render the job again
        if rank == 0:
            print(f"bench: images of the last timed step -> {dump_images(last[0], args.dump_outputs)}", file=sys.stderr)
        if world > 1:
            dist.barrier()  # the other ranks wait here rather than spin in the next render's in-graph barrier

    # ---- N > 1 correctness, outside the timed region: the gathered images of the sharded job must be
    # bit-identical to rank 0's own single-GPU render of the same views
    sharded_equals_single = None
    if world > 1:
        step_device(d_in)
        got = flush()
        if rank == 0:
            got = got[None].clone()
            pipe.cuda_graphs = False
            ref_img = pipe.render(d_in["triangles"], d_in["texture"], d_in["mask"], d_in["vn"], d_in["c2w"], d_in["fov"],
                                  resolution=R, torch_dtype=torch.bfloat16)
            sharded_equals_single = bool(torch.equal(got, ref_img))
            if not sharded_equals_single:
                print(f"bench: sharded != single, max |d| = {(got - ref_img).abs().max().item():.3e}", file=sys.stderr)
            del got, ref_img
            pipe.cuda_graphs = graphs
        dist.barrier()

    # ---- where the step goes: scene stage / view stage / image gather, each replayed from its own CUDA graph
    # (outside the timed region; max over ranks per stage, so the parts can add up to a little more than ms_step)
    stages = None
    try:
        from renderformer_b200.dist import gather_images, row_shard
        sh = row_shard()
        cl, fl = d_in["c2w"][:, mine].contiguous(), d_in["fov"][:, mine].contiguous()
        sizes = [view_slice(V, world, r).stop - view_slice(V, world, r).start for r in range(world)]

        def staged(ev):
            ev[0].record()
            st = pipe.encode(d_in["triangles"], d_in["texture"], d_in["mask"], d_in["vn"], shard=sh, torch_dtype=torch.bfloat16)
            ev[1].record()
            img = pipe.render_views(st, cl, fl, R)
            ev[2].record()
            if world > 1:
                gather_images(img[0], dst=0, sizes=sizes)
            ev[3].record()
        evs = [[torch.cuda.Event(enable_timing=True) for _ in range(4)] for _ in range(4)]
        for i in range(2):
            staged(evs[i])
        barrier()
        for i in range(2, 4):
            staged(evs[i])
        barrier()
        t = torch.tensor([[e[k].elapsed_time(e[k + 1]) for k in range(3)] for e in evs[2:]], device=dev).mean(dim=0)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        stages = {"scene_stage_ms": t[0].item(), "view_stage_ms": t[1].item(), "image_gather_ms": t[2].item(),
                  "note": "separate CUDA-graph replays per stage, max over ranks"}
    except Exception as e:  # noqa: BLE001  (diagnostic only)
        stages = {"unavailable": repr(e)[:200]}

    e2e = None
    if not args.no_e2e:
        for _ in range(2):
            step_e2e()
        ms_e2e = timed(step_e2e, args.steps)
        small = sum(host[k].numel() * host[k].element_size() for k in ("triangles", "mask", "vn"))
        host_scene = {k: host[k] for k in ("triangles", "texture", "mask", "vn", "c2w", "fov")}
        if world == 1:
            # the batch API (batch_infer.py use case): every step still uploads its own inputs from pinned host
            # memory and downloads its own images inside the timed region, but the upload of step i+1 and the
            # download of step i overlap the kernels of the neighbouring step
            def stream_steps(n):
                sink = 0.0
                for img in pipe.render_stream((host_scene for _ in range(n)), resolution=R, torch_dtype=torch.bfloat16):
                    sink += float(img[0, 0, 0, 0, 0])  # touch the host result of every step
                return sink
            api = ("RenderFormerRenderingPipeline.render_stream (host scenes in, pinned host images out; copies of "
                   "neighbouring steps overlap the kernels)")
            h2d = small + host["texture"].numel() * 4 + (host["c2w"].numel() + host["fov"].numel()) * 4
        else:
            def stream_steps(n):
                sink = 0.0
                for _mine, img in render_stream_sharded(pipe, (host_scene for _ in range(n)), resolution=R,
                                                        torch_dtype=torch.bfloat16):
                    sink += float(img[0, 0, 0, 0, 0]) if img.numel() else 0.0
                return sink
            api = ("renderformer_b200.dist.render_stream_sharded (every rank uploads the geometry and its own rows of the "
                   "texture, row-sharded scene stage, every rank renders and downloads its own views; copies overlap kernels)")
            # summed over ranks: geometry on every rank, each texture row once, each camera once
            h2d = world * small + host["texture"].numel() * 4 + (host["c2w"].numel() + host["fov"].numel()) * 4
        stream_steps(3)
        ms_stream = timed(lambda: stream_steps(args.steps), 1) / args.steps
        e2e = {"value": V / (ms_stream * 1e-3), "unit": UNIT, "ms_per_step": ms_stream,
               "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": int(V * R * R * 3 * 4), "api": api,
               "single_call": {"value": V / (ms_e2e * 1e-3), "ms_per_step": ms_e2e,
                               "api": "one blocking call per step (full scene uploaded by every rank)" if world > 1 else
                                      "RenderFormerRenderingPipeline.render, one blocking call per step"}}

    roofline = None
    if not args.no_roofline:
        peak_tf, _, peak_src = load_peaks()
        pipe.cuda_graphs = False  # per-launch events need eager launches
        ops.PROFILE = [] if rank == 0 else None
        barrier()
        step_device(d_in, dst=None)
        torch.cuda.synchronize()
        prof, ops.PROFILE = ops.PROFILE, None
        pipe.cuda_graphs = graphs
        if rank == 0:
            by = {}
            for kind, fl, a, b, _tag in prof:
                t = a.elapsed_time(b) * 1e-3
                cur = by.setdefault(kind, [0.0, 0.0, 0])
                cur[0] += fl
                cur[1] += t
                cur[2] += 1
            g = by.get("gemm", [0.0, 1.0, 1])
            att = by.get("attention", [0.0, 1.0, 1])
            ach = g[0] / g[1] / 1e12
            traffic, traffic_src = None, None
            for name in ("r02b_gemm_traffic.json", "r02_gemm_traffic.json", "r01e_gemm_traffic.json"):  # newest capture first
                tpath = os.path.join(ROOT, "profiles", name)
                want_chunk = 8 if name.startswith("r02") else 4
                if os.path.exists(tpath) and args.config == "v1_1_swin_large" and (N, R, pipe.view_chunk) == (4096, 512, want_chunk):
                    with open(tpath) as f:
                        tj = json.load(f)
                    traffic = tj["dram_bytes_per_launch"]
                    traffic_src = f"profiles/{name} (ncu dram__bytes_read+write, average over consecutive GEMM / conv launches of this job)"
                    break
            roofline = {
                "kernel": "gemm_tc_kernel (tcgen05 GEMM / implicit-GEMM conv)", "bound": "tensor",
                "achieved": ach, "peak": peak_tf, "unit": "TFLOP/s", "frac": ach / peak_tf, "traffic": traffic,
                "traffic_source": traffic_src, "flop_per_launch": g[0] / g[2],
                "peak_source": peak_src, "launches_per_step": g[2], "avg_launch_us": g[1] / g[2] * 1e6,
                "share_of_step": g[1] * 1e3 / ms_step,
                "method": "per-launch CUDA events on the launch stream, one instrumented eager step (rank 0's share of the "
                          "job) after the timed region",
                "attention": {"kernel": "attn3_tc_kernel / attn2_tc_kernel / attn_swin_kernel", "achieved": att[0] / att[1] / 1e12,
                              "unit": "TFLOP/s", "frac": att[0] / att[1] / 1e12 / peak_tf, "launches_per_step": att[2],
                              "share_of_step": att[1] * 1e3 / ms_step},
            }
    if world > 1:
        dist.barrier()

    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        r = cpu_arm(args, min(V, 4), 1)
        cpu = {"value": r["value"], "unit": UNIT, "cores": r["cores"], "kind": r["kind"], "sample": r["sample"]}

    ref_cuda = None
    if rank == 0 and world == 1 and not args.no_ref_cuda:
        del d_in
        pipe._graphs.clear()
        torch.cuda.empty_cache()
        ref_cuda = run_ref_cuda(args)

    if rank == 0:
        step_tflop = job_flops(cfg, N, R, 1, V) / 1e12
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": max(args.warmup, 3), "ms_per_step": ms_step, "higher_is_better": True,
            "scaling": "weak" if args.views_per_gpu > 0 else "strong",
            "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
            "config": {
                "workload": workload_text(args, world),
                "parallelism": (f"scene stage row-sharded over {world} ranks ({kv_exchange_text()}), "
                                f"{Vl} views per rank, image gather on rank 0" if world > 1 else "single GPU"),
                "views_per_decoder_pass": pipe.view_chunk,
                "l2": "inputs + weights + activations (> 1.3 GB per step) exceed the 126 MB L2; no explicit flush",
                "launch": ("one CUDA-graph replay per step and rank, the ranks' k|v exchange and barriers inside the graph; "
                           "the image gather of job k is enqueued asynchronously and overlaps the scene stage of job k+1"
                           if graphs else "eager launches from Python"),
                "algorithmic_tflop_per_step": step_tflop,
                "model_flops_utilisation": step_tflop / (ms_step * 1e-3) / world / load_peaks()[0],
                "scene_tflop": scene_flops(cfg, N) / 1e12, "view_tflop": view_flops(cfg, N, R) / 1e12,
            },
            "clocks": clocks, "e2e": e2e, "gpu_launches": int(launches), "roofline": roofline, "cpu_baseline": cpu,
            "stages": stages,
            "sharded_equals_single": sharded_equals_single,
        }
        if ref_cuda is not None:
            line["reference_cuda"] = ref_cuda
        print(json.dumps(line), flush=True)
    if world > 1:
        # Tear-down order matters: CUDA graphs that captured NCCL kernels must be gone before the communicator is
        # (destroy_process_group with such graphs alive hung the r02c run for 24 minutes AFTER the line was printed).
        pipe._graphs.clear()
        pipe._static_states.clear()
        torch.cuda.synchronize()
        dist.barrier()
        torch.cuda.synchronize()
        sys.stdout.flush()
        sys.stderr.flush()
        os._exit(0)  # skip the communicator's destructor paths altogether; every rank leaves with rc 0


if __name__ == "__main__":
    main()
