"""Multi-GPU plumbing (one process per GPU, torch.distributed; NCCL on GPUs, gloo in CPU tests).

Both stages shard (SURVEY §8e):

* view-independent stage -- the token ROWS of the triangle sequence are split over the ranks
  (`row_shard` -> engine.RowShard): every rank constructs, projects, attends and feeds forward its own rows.
  What a layer needs of the other ranks -- their 16-bit k | v rows (16.8 MB in total for 4096 triangles) -- is
  written by the producing kernel itself into every rank's memory (`SymmKVStore`: symmetric memory, NVLS
  multicast stores or peer stores over NVLink, then a signal-pad barrier); `RFB_KV_PUSH=0` keeps one NCCL
  all-gather per layer instead.  No rank waits for "the encoder rank", no 300 MB K/V broadcast: the hoisted
  decoder K / V are recomputed from the gathered final stream on every rank (0.2 TFLOP).
* view-dependent stage -- every rank renders a contiguous slice of the views (`view_slice`); the
  only collective is the final image gather.

`broadcast_scene_state` (rank `src` encodes alone, its state is broadcast -- the north_star's
wording) is kept for callers that hold the scene on one rank only."""
from __future__ import annotations

from typing import List, Optional

import os
import sys

import torch
import torch.distributed as dist

from .config import camera_kwargs, view_camera
from .engine import RowShard, SceneState


def _world():
    if dist.is_available() and dist.is_initialized():
        return dist.get_world_size(), dist.get_rank()
    return 1, 0


def view_slice(n_views: int, world: int, rank: int) -> slice:
    """Contiguous, balanced partition of `n_views` over `world` ranks."""
    base, extra = divmod(n_views, world)
    start = rank * base + min(rank, extra)
    return slice(start, start + base + (1 if rank < extra else 0))


def all_gather_rows(full: torch.Tensor, chunk: torch.Tensor, group=None) -> None:
    """full [world*S, ...] <- every rank's chunk [S, ...]; `chunk` may be (and in the engine is) the
    rank's own slice of `full` (in-place all-gather, no staging copy with NCCL)."""
    if full.is_cuda:
        dist.all_gather_into_tensor(full, chunk, group=group)
    else:  # gloo (CPU tests): no aliasing between input and outputs
        world = dist.get_world_size(group)
        s = chunk.shape[0]
        dist.all_gather([full[r * s:(r + 1) * s] for r in range(world)], chunk.clone(), group=group)


class SymmKVStore:
    """Peer-mapped [k | v] row store of the row-sharded scene stage: two buffers [rows, width] (16 bit) in
    symmetric memory (`torch.distributed._symmetric_memory`: the same allocation on every rank, every rank's copy
    mapped into every other rank's address space over NVLink, plus -- where the NVSwitch supports NVLS -- ONE
    multicast address that aliases all of them).  `rfb_qkv_post` stores a rank's rows through `dst(i)`; `barrier()`
    is a signal-pad rendezvous of all ranks on the current stream (capturable in a CUDA graph), after which every
    rank may read `buf(i)`.  This replaces the per-layer NCCL all-gather (the collective is fused into the kernel
    that produces the rows: a rank's stores ARE the transfer)."""

    def __init__(self, group, rows: int, width: int, dtype, device, multicast: bool = True):
        import torch.distributed._symmetric_memory as symm_mem
        pg = group if group is not None else dist.group.WORLD
        try:
            symm_mem.enable_symm_mem_for_group(pg.group_name)
        except Exception:
            pass  # newer torch: not needed (deprecated)
        self.t = symm_mem.empty((2, rows, width), dtype=dtype, device=device)
        self.hdl = symm_mem.rendezvous(self.t, pg)
        self.world, self.rank = self.hdl.world_size, self.hdl.rank
        off = self.t.data_ptr() - int(self.hdl.buffer_ptrs[self.rank])  # the tensor's offset inside the mapped block
        self._buf_bytes = rows * width * self.t.element_size()
        self._peers = [int(ptr) + off for ptr in self.hdl.buffer_ptrs]
        mc = int(getattr(self.hdl, "multicast_ptr", 0) or 0)
        self._mc = mc + off if (multicast and mc) else 0
        self.t.zero_()
        torch.cuda.synchronize(device)
        self.hdl.barrier(channel=0)

    @property
    def multicast(self) -> bool:
        return self._mc != 0

    def buf(self, i: int) -> torch.Tensor:
        return self.t[i]

    def dst(self, i: int):
        """(device addresses to store buffer i's rows to, multicast flag)."""
        if self._mc:
            return [self._mc + i * self._buf_bytes], True
        return [ptr + i * self._buf_bytes for ptr in self._peers], False

    def barrier(self) -> None:
        self.hdl.barrier(channel=0)


_KV_STORES = {}
_KV_PUSH_BROKEN = [False]


def _kv_store_factory(group):
    """kv_store callable for RowShard, or None (RFB_KV_PUSH=0, CPU / gloo groups, more than 8 ranks, or symmetric
    memory that cannot be set up here -- all ranks then agree to keep the NCCL all-gather).  RFB_KV_PUSH=1 keeps
    the peer-mapped stores but does without the multicast address (one plain store per peer)."""
    mode = os.environ.get("RFB_KV_PUSH", "2")
    world, _ = _world()
    if mode == "0" or not torch.cuda.is_available() or dist.get_backend(group) != "nccl" or world > 8:
        return None

    def factory(rows, width, dtype, device):
        if _KV_PUSH_BROKEN[0]:
            return None
        key = (id(group), rows, width, dtype, str(device), mode)
        st = _KV_STORES.get(key)
        if st is None:
            err = None
            try:
                st = SymmKVStore(group, rows, width, dtype, device, multicast=(mode != "1"))
            except Exception as e:  # noqa: BLE001 -- any set-up failure: agree on the fallback below
                err, st = e, None
            ok = torch.tensor([0 if st is None else 1], device=device)
            dist.all_reduce(ok, op=dist.ReduceOp.MIN, group=group)
            if ok.item() == 0:
                _KV_PUSH_BROKEN[0] = True
                if dist.get_rank(group) == 0:
                    print(f"renderformer_b200.dist: symmetric-memory k|v store unavailable ({err!r}); "
                          "falling back to the NCCL all-gather", file=sys.stderr, flush=True)
                return None
            if len(_KV_STORES) >= 4:
                _KV_STORES.pop(next(iter(_KV_STORES)))
            _KV_STORES[key] = st
        return st
    return factory


def row_shard(group=None) -> Optional[RowShard]:
    """RowShard of the current process group (None when there is one rank)."""
    world, rank = _world()
    if world == 1:
        return None
    return RowShard(rank, world, lambda full, chunk: all_gather_rows(full, chunk, group), _kv_store_factory(group))


def broadcast_scene_state(state: SceneState, src: int = 0) -> SceneState:
    """In-place broadcast of every tensor of a SceneState (receivers pass alloc_scene_state())."""
    if _world()[0] > 1:
        for t in state.tensors():
            dist.broadcast(t, src=src)
    return state


class GatherHandle:
    """Result of an image gather that may still be in flight (`gather_images(..., async_op=True)`): `wait()`
    makes the current stream wait for it and returns the gathered stack on `dst`, None elsewhere."""

    def __init__(self, work, full, sizes, vmax, keep):
        self.work, self.full, self.sizes, self.vmax, self.keep = work, full, sizes, vmax, keep

    def wait(self):
        if self.work is not None:
            self.work.wait()
            self.work = None
        self.keep = None
        if self.full is None:
            return None
        if all(n == self.vmax for n in self.sizes):
            return self.full  # the receive buffers are slices of one tensor: no concatenation
        return torch.cat([self.full[r * self.vmax:r * self.vmax + n] for r, n in enumerate(self.sizes)], dim=0)


def gather_images(img: torch.Tensor, dst: int = 0, sizes: Optional[List[int]] = None, async_op: bool = False):
    """Gather per-rank image stacks [V_r, H, W, 3] on `dst` (returns the concatenation there, None
    elsewhere).  `sizes` lists V_r per rank when the split is uneven.  With `async_op` the collective is only
    enqueued (on NCCL's own stream, behind the work already queued on the current stream) and a GatherHandle
    is returned: the caller may go on launching the next job and `wait()` later; `img` must not be overwritten
    before that (pass a copy when it is the static output of a CUDA graph)."""
    world, rank = _world()
    if world == 1:
        return GatherHandle(None, img, [img.shape[0]], img.shape[0], None) if async_op else img
    if sizes is None:
        sizes = [img.shape[0]] * world
    vmax = max(sizes)
    pad = img
    if img.shape[0] < vmax:
        pad = torch.cat([img, img.new_zeros((vmax - img.shape[0],) + tuple(img.shape[1:]))], dim=0)
    pad = pad.contiguous()
    full = torch.empty((world * vmax,) + tuple(pad.shape[1:]), dtype=pad.dtype, device=pad.device) if rank == dst else None
    bufs = list(full.split(vmax, dim=0)) if rank == dst else None
    work = dist.gather(pad, bufs, dst=dst, async_op=True)
    handle = GatherHandle(work, full, sizes, vmax, pad)
    return handle if async_op else handle.wait()


@torch.no_grad()
def render_sharded(pipe, triangles, texture, mask, vn, c2w, fov=None, resolution=512, dst: Optional[int] = 0,
                   texture_own_rows: bool = False, torch_dtype: torch.dtype = torch.float16, async_gather: bool = False,
                   overscan: bool = False, intrinsics=None, distortion=None, lens: str = "opencv"):
    """`RenderFormerRenderingPipeline.render` on all ranks of the process group: every rank passes the
    SAME scene and the full camera list c2w [B,V,4,4] / fov [B,V,1]; the scene stage is row-sharded, each
    rank renders `view_slice(V)`, and the images are gathered on `dst` (returns [B,V,H,W,3] there and
    None elsewhere; `dst=None` skips the gather and returns this rank's [B,V_rank,H,W,3]).  With
    `pipe.cuda_graphs` and device inputs the whole per-rank schedule, NCCL all-gathers included, is one
    CUDA-graph replay.  `async_gather` (one scene per call): the image gather is only enqueued and a
    GatherHandle is returned on every rank -- a caller rendering job after job lets the gather of job k
    travel over NVLink while the scene stage of job k+1 runs, and calls `handle.wait()` before using the
    images (at the latest before the job after next).  `resolution`: an int or (H, W), `overscan`, and the
    camera (`fov` [B,V,1] or `intrinsics` [B,V,4] with the optional `distortion` [B,V,n] of `lens`, full lists,
    sliced per rank like c2w), as in `render`."""
    canvas, window, _ = pipe.view_geometry(resolution, overscan)
    kind, cam = view_camera(c2w, fov, intrinsics, distortion, lens, canvas, window)
    world, rank = _world()
    V = c2w.shape[1]
    mine = view_slice(V, world, rank)
    c2w_l, cam_l = c2w[:, mine].contiguous(), cam[:, mine].contiguous()
    sh = row_shard()
    if world == 1:
        img = pipe.render(triangles, texture, mask, vn, c2w_l, resolution=resolution, torch_dtype=torch_dtype,
                          overscan=overscan, **camera_kwargs(kind, cam_l))
    else:
        from .model import operand_dtype
        eng = pipe.model.engine(operand_dtype(torch_dtype))
        inputs = (triangles, texture, mask, vn, c2w_l, cam_l)

        def run(tri, tex, msk, vnn, cw, cm):
            st = eng.encode_scene(tri, tex, msk, vnn, shard=sh, texture_own_rows=texture_own_rows)
            return pipe.render_views(st, cw, resolution=resolution, overscan=overscan, _eager=True,
                                     **camera_kwargs(kind, cm))
        if pipe.cuda_graphs and all(t.is_cuda for t in inputs) and mine.stop > mine.start:
            key = (("render_sharded", id(eng), rank, world, kind, canvas, window, pipe.view_chunk, texture_own_rows) +
                   pipe._sig(inputs))
            img = pipe._graph_entry(key, inputs, run)
        else:
            img = run(*inputs)
    if dst is None or world == 1:
        return img
    sizes = [view_slice(V, world, r).stop - view_slice(V, world, r).start for r in range(world)]
    B = img.shape[0]
    if async_gather and B == 1:
        # a private copy: `img` may be the static output of a CUDA graph that the next call replays
        return gather_images(img[0].clone(), dst=dst, sizes=sizes, async_op=True)
    out = gather_images(img.transpose(0, 1).contiguous() if B > 1 else img[0], dst=dst, sizes=sizes)
    if out is None:
        return None
    return out.transpose(0, 1).contiguous() if B > 1 else out[None]


@torch.no_grad()
def render_stream_sharded(pipe, scenes, resolution=512, ldr: Optional[str] = None,
                          torch_dtype: torch.dtype = torch.float16, overscan: bool = False, lens: str = "opencv"):
    """Multi-GPU counterpart of `RenderFormerRenderingPipeline.render_stream`: every rank iterates the SAME
    sequence of host scene dicts (keys of `render`).  Each rank uploads the geometry and only ITS OWN
    rows of the texture (1/world of the 218 MB), the scene stage runs row-sharded, each rank renders its
    contiguous slice of the views and downloads its own images (no gather: a rank can write its own
    frames).  Uploads of scene i+1 and downloads of scene i overlap the kernels of the neighbouring scene.

    Yields (view_slice, pinned host tensor [B, V_rank, H, W, 3]) per scene; the buffer belongs to a ring of
    three.  `resolution`: an int or (H, W), and `overscan`, as in `render`; a scene carries 'fov' or
    'intrinsics' (and optionally 'distortion' of the model `lens`), as in `render_stream`."""
    canvas, window, _ = pipe.view_geometry(resolution, overscan)
    dev = pipe.device
    world, rank = _world()
    main = torch.cuda.current_stream(dev)
    copy = torch.cuda.Stream(dev)
    from .model import UploadRing, operand_dtype
    eng = pipe.model.engine(operand_dtype(torch_dtype))
    sh = row_shard()
    up = UploadRing(dev, copy)

    def upload(sc):
        kind, cam = view_camera(sc["c2w"], sc.get("fov"), sc.get("intrinsics"), sc.get("distortion"), lens, canvas,
                                window)
        V = sc["c2w"].shape[1]
        mine = view_slice(V, world, rank)
        N = sc["triangles"].shape[1]
        t0, t1 = eng.own_triangles(N, sh) if sh is not None else (0, N)
        d, ev, slot = up.put({"c2w": sc["c2w"][:, mine], kind: cam[:, mine], "triangles": sc["triangles"],
                              "mask": sc["mask"], "vn": sc["vn"],
                              "texture": sc["texture"][:, t0:t1]})  # only this rank's rows of the texture
        return kind, d, ev, mine, slot

    import os
    import sys
    import time
    dbg = os.environ.get("RFB_STREAM_DEBUG") == "1" and rank == 0
    it = iter(scenes)
    first = next(it, None)
    pending = upload(first) if first is not None else None
    ring, rslot, prev = [None, None, None], 0, None
    while pending is not None:
        t_0 = time.perf_counter()
        kind, d, ev, mine, slot = pending
        nxt = next(it, None)
        pending = upload(nxt) if nxt is not None else None
        t_1 = time.perf_counter()
        main.wait_event(ev)
        if sh is None:
            img = pipe.render(d["triangles"], d["texture"], d["mask"], d["vn"], d["c2w"], resolution=resolution,
                              torch_dtype=torch_dtype, overscan=overscan, **camera_kwargs(kind, d[kind]))
        else:
            # full camera list is not needed here: the slice was taken on the host
            inputs = (d["triangles"], d["texture"], d["mask"], d["vn"], d["c2w"], d[kind])

            def run(tri, tex, msk, vnn, cw, cm):
                st = eng.encode_scene(tri, tex, msk, vnn, shard=sh, texture_own_rows=True)
                return pipe.render_views(st, cw, resolution=resolution, overscan=overscan, _eager=True,
                                         **camera_kwargs(kind, cm))
            if pipe.cuda_graphs and mine.stop > mine.start:
                key = ("stream_sharded", id(eng), rank, world, kind, canvas, window, pipe.view_chunk) + pipe._sig(inputs)
                img = pipe._graph_entry(key, inputs, run)
            else:
                img = run(*inputs)
        up.release(slot, main)
        if ldr is not None:
            img = pipe.hdr_to_ldr(img, ldr)
        if ring[rslot] is None or ring[rslot].shape != img.shape or ring[rslot].dtype != img.dtype:
            ring[rslot] = torch.empty(img.shape, dtype=img.dtype, pin_memory=True)
        host = ring[rslot]
        rslot = (rslot + 1) % 3
        t_2 = time.perf_counter()
        host.copy_(img, non_blocking=True)
        done = torch.cuda.Event()
        done.record(main)
        t_3 = time.perf_counter()
        if prev is not None:
            prev[1].synchronize()
            if dbg:
                print(f"[stream] upload-issue {1e3 * (t_1 - t_0):.2f} ms, render-issue {1e3 * (t_2 - t_1):.2f} ms, d2h-issue "
                      f"{1e3 * (t_3 - t_2):.2f} ms, wait-prev {1e3 * (time.perf_counter() - t_3):.2f} ms", file=sys.stderr, flush=True)
            yield prev[2], prev[0]
        prev = (host, done, mine)
    if prev is not None:
        prev[1].synchronize()
        yield prev[2], prev[0]
