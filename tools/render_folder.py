#!/usr/bin/env python
"""Render a folder of converted scenes to EXR / PNG (/ MP4) with nothing serialised behind the GPU: the
batch_infer.py workflow (reference batch_infer.py:61-174) on `render_stream` + `frame_io.FrameWriter`
(SURVEY §8 f3).  Scenes are the `.npz` files `tools/convert_scene.py` writes (numpy only) or the reference
converter's `.h5` files (when h5py is installed); frames are named like the reference's:
`<scene>_view_<v>.exr`, `<scene>_view_<v>.png`, `video.mp4`.

usage: python tools/render_folder.py --scene_folder scenes/ --model_id /path/to/checkpoint_dir \
           [--precision fp16|bf16|fp32] [--resolution 512] [--height H] [--width W] [--overscan] [--padding_length N] [--constant_texture]
           [--tone_mapper none|pbr_neutral] [--save_video] [--output_dir out/] [--workers 4]

Multi-GPU: launch with torchrun (`python -m torch.distributed.run --nproc-per-node N --master-addr 127.0.0.1
tools/render_folder.py ...`): the scene stage is row-sharded, every rank renders and writes its own views.

`--model_id` is a local directory with config.json + model.safetensors (there is no hub access here);
`--random_init NAME` renders with seeded random weights of a named architecture instead (smoke runs).

`--height` / `--width` render H x W frames (e.g. 576 x 1024 for 16:9 video); either one replaces the matching side of
the square `--resolution`.  The field of view of a scene spans the longer side.  Without `--overscan` the sides must be
multiples of 64 for the swin models (8 for full attention); `--overscan` renders any size, e.g. `--height 1080 --width
1920`, on the smallest canvas on that grid and writes only the requested frame (same camera, every pixel a real output
of the model)."""
import argparse
import glob
import os
import re
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))


def natural_key(s: str):
    """natsort.natsorted's ordering for file names: digit runs compare as numbers (batch_infer.py:20)."""
    return [int(t) if t.isdigit() else t.lower() for t in re.split(r"(\d+)", s)]


def main(argv=None, _pipeline=None) -> int:
    """`_pipeline`: a ready pipeline object (tests inject a stand-in; the host logic then runs without a GPU)."""
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--scene_folder", required=True)
    ap.add_argument("--model_id", default=None)
    ap.add_argument("--random_init", default=None, help="architecture name (e.g. v1_1_swin_large, tiny_swin) for seeded random weights")
    ap.add_argument("--precision", choices=["bf16", "fp16", "fp32"], default="fp16")
    ap.add_argument("--resolution", type=int, default=512)
    ap.add_argument("--height", type=int, default=None, help="image height in pixels (overrides --resolution)")
    ap.add_argument("--width", type=int, default=None, help="image width in pixels (overrides --resolution)")
    ap.add_argument("--overscan", action="store_true",
                    help="any frame size: render on the decoder's size grid and crop (e.g. --height 1080 --width 1920)")
    ap.add_argument("--padding_length", type=int, default=None, help="pad every scene to this many triangles on the device: one CUDA graph for all scenes")
    ap.add_argument("--constant_texture", action="store_true", help="upload 13 constants per triangle instead of the 32x32 texel grid")
    ap.add_argument("--tone_mapper", choices=["none", "pbr_neutral"], default="none")
    ap.add_argument("--save_video", action="store_true")
    ap.add_argument("--output_dir", default=None)
    ap.add_argument("--workers", type=int, default=4)
    args = ap.parse_args(argv)
    resolution = args.resolution
    if args.height is not None or args.width is not None:
        resolution = (args.height or args.resolution, args.width or args.resolution)

    import torch
    from renderformer_b200 import frame_io, scene_io
    from renderformer_b200.model import RenderFormer, RenderFormerRenderingPipeline

    files = [p for ext in ("npz", "h5", "hdf5") for p in glob.glob(os.path.join(args.scene_folder, "*." + ext))]
    files.sort(key=lambda p: natural_key(os.path.basename(p)))
    if not files:
        print(f"no .npz / .h5 scenes in {args.scene_folder} (convert scene JSON files with tools/convert_scene.py)")
        return 1
    if _pipeline is not None:
        pipe = _pipeline
    elif args.random_init:
        from renderformer_b200.config import RenderFormerConfig
        from renderformer_b200.synth import init_state_dict
        cfg = RenderFormerConfig.named(args.random_init)
        model = RenderFormer(cfg)
        model.load_state_dict(init_state_dict(cfg, 7))
        pipe = RenderFormerRenderingPipeline(model)
    elif args.model_id:
        pipe = RenderFormerRenderingPipeline.from_pretrained(args.model_id)
    else:
        ap.error("one of --model_id / --random_init is required")
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if world > 1:  # one process per GPU (torchrun): both stages shard, every rank writes its own frames
        import torch.distributed as dist
        torch.cuda.set_device(local_rank)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    if _pipeline is None:
        pipe.to(torch.device("cuda", local_rank))
    pipe.cuda_graphs = args.padding_length is not None or world > 1
    pin = torch.cuda.is_available()
    dtype = {"fp16": torch.float16, "bf16": torch.bfloat16, "fp32": torch.float32}[args.precision]

    def scenes():
        for p in files:  # host side of scene i+1 is prepared while scene i renders (render_stream pulls one ahead)
            sc = scene_io.to_pipeline_inputs(scene_io.load_scene_file(p), constant_texture=args.constant_texture,
                                             pad_to=args.padding_length if world > 1 else None)  # sharded stream: pad on the host
            yield {k: (v.pin_memory() if pin and v.dtype != torch.bool else v) for k, v in sc.items()}

    out_dir = args.output_dir or args.scene_folder
    names = [os.path.splitext(os.path.basename(p))[0] for p in files]
    t0 = time.time()
    # scene files are read / expanded / pinned two scenes ahead on a background thread
    paths = frame_io.render_to_files(pipe, frame_io.prefetch(scenes(), depth=2), names, out_dir, resolution=resolution, torch_dtype=dtype,
                                     tone_mapper=args.tone_mapper, pad_to=args.padding_length if world == 1 else None,
                                     save_video=args.save_video, workers=args.workers, sharded=world > 1,
                                     overscan=args.overscan)
    dt = time.time() - t0
    print(f"[rank {os.environ.get('RANK', '0')}] {len(paths)} frames of {len(files)} scenes -> {out_dir} in {dt:.2f} s "
          f"({len(paths) / dt:.1f} frames/s incl. file encoding)")
    if world > 1 and _pipeline is None:
        # tear-down as in bench.py: CUDA graphs that captured NCCL kernels must be gone before the communicator is, and
        # the communicator's destructor paths are skipped altogether (destroy_process_group hung a run for minutes)
        import torch.distributed as dist
        pipe._graphs.clear()
        pipe._static_states.clear()
        torch.cuda.synchronize()
        dist.barrier()
        torch.cuda.synchronize()
        sys.stdout.flush()
        sys.stderr.flush()
        os._exit(0)
    return 0


if __name__ == "__main__":
    sys.exit(main())
