"""Drop-in model object: reference parameter tree + B200 engine.

`RenderFormer` keeps the reference's constructor, state_dict keys (SURVEY Appendix A.3),
`from_pretrained` / `save_pretrained` contract (config.json + model.safetensors, as written by
the reference's PyTorchModelHubMixin, models/renderformer.py:13) and `forward` signature
(models/renderformer.py:171), but the forward pass runs on renderformer_b200.engine.Engine.
"""
from __future__ import annotations

import json
import os
from typing import Dict, Optional

import torch
from torch import nn

from .config import RenderFormerConfig, _size_pair, camera_kwargs, overscan_grid, view_camera, view_grid
from . import lib as L
from .engine import Engine, SceneState


class RenderFormer(nn.Module):
    """models/renderformer.py:13-206.  The parameter tree is composed of the same sub-modules as the
    reference (renderformer_b200/modules.py: TransformerEncoder, ViewTransformer -> TransformerDecoder +
    DPTHead, ...), so attribute paths and state_dict keys are the reference's; `forward` runs the fused
    engine over the whole tree instead of calling the sub-modules one by one."""

    def __init__(self, config: RenderFormerConfig):
        super().__init__()
        if isinstance(config, dict):
            config = RenderFormerConfig.from_dict(config)
        config.check_supported()
        self.config = config
        from .modules import NeRFEncoding, TransformerEncoder, ViewTransformer
        d = config.latent_dim
        with torch.device("meta"):  # no throw-away initialisation of 0.2-0.5 G parameters
            self.rope_dim = config.vertex_pe_num_freqs
            self.vn_pe = NeRFEncoding(in_dim=9, num_frequencies=config.vn_pe_num_freqs, include_input=True)
            self.vn_encoding_proj = nn.Linear(self.vn_pe.get_out_dim(), d)
            self.vn_encoder_norm = nn.RMSNorm(d)
            self.texture_encoder = nn.Linear(config.texture_channels * config.texture_encode_patch_size ** 2, d)
            self.texture_encoder_norm = nn.RMSNorm(d)
            self.tri_token = nn.Parameter(torch.randn(1, 1, d))
            self.reg_tokens = nn.Parameter(torch.randn(1, config.num_register_tokens, d))
            self.skip_token_num = config.num_register_tokens
            self.transformer = TransformerEncoder(
                num_layers=config.num_layers, num_heads=config.num_heads, hidden_dim=d,
                ffn_hidden_dim=config.dim_feedforward, dropout=config.dropout, activation=config.activation,
                norm_type=config.norm_type, norm_first=config.norm_first, rope_dim=self.rope_dim,
                rope_type=config.rope_type, bias=config.bias, qk_norm=config.view_indep_qk_norm,
                rope_double_max_freq=config.rope_double_max_freq)
            self.view_transformer = ViewTransformer(config)
        self.to_empty(device="cpu")
        self._engines: Dict[torch.dtype, tuple] = {}
        self.reset_parameters()

    def reset_parameters(self, seed: int = 0) -> None:
        from .synth import init_state_dict
        self.load_state_dict(init_state_dict(self.config, seed))

    # ---- persistence (same files as the reference's hub mixin) ----------------------
    @classmethod
    def from_pretrained(cls, pretrained_model_name_or_path, *, force_download: bool = False, token=None,
                        cache_dir=None, local_files_only: bool = False, revision: Optional[str] = None,
                        **model_kwargs) -> "RenderFormer":
        """Signature of huggingface_hub's PyTorchModelHubMixin.from_pretrained, which the reference class inherits
        (models/renderformer.py:13): a local directory with config.json + model.safetensors, or a hub id (the hub
        options are handed to `snapshot_download`; needs network, not used in tests)."""
        path = str(pretrained_model_name_or_path)
        if not os.path.isdir(path):
            from huggingface_hub import snapshot_download
            path = snapshot_download(path, force_download=force_download, token=token, cache_dir=cache_dir,
                                     local_files_only=local_files_only, revision=revision)
        with open(os.path.join(path, "config.json")) as f:
            cfg = RenderFormerConfig.from_dict(json.load(f))
        model = cls(cfg)
        from safetensors.torch import load_file
        model.load_state_dict(load_file(os.path.join(path, "model.safetensors")), strict=True)
        return model

    def save_pretrained(self, path: str) -> None:
        os.makedirs(path, exist_ok=True)
        with open(os.path.join(path, "config.json"), "w") as f:
            json.dump(self.config.to_dict(), f, indent=2)
        from safetensors.torch import save_file
        save_file({k: v.detach().cpu().contiguous() for k, v in self.state_dict().items()},
                  os.path.join(path, "model.safetensors"))

    @property
    def device(self) -> torch.device:
        return next(self.parameters()).device

    def load_state_dict(self, state_dict, strict: bool = True, assign: bool = False):
        self._engines = {}
        return super().load_state_dict(state_dict, strict=strict, assign=assign)

    # ---- the reference's helper methods, on the kernels ------------------------------
    @torch.no_grad()
    def process_tri_vpos_list(self, tri_vpos_list, valid_mask):
        """models/renderformer.py:103-124: prepend `num_register_tokens` copies of the masked vertex
        centroid to the positions and True to the mask (rfb_positions)."""
        from . import ops
        B, N = tri_vpos_list.shape[:2]
        nreg = self.config.num_register_tokens
        dev = tri_vpos_list.device
        tri = tri_vpos_list.reshape(B, N, 9).to(torch.float32).contiguous()
        m8 = valid_mask.contiguous().view(torch.uint8) if valid_mask.dtype == torch.bool else valid_mask.to(torch.uint8)
        pos = torch.empty((B, N + nreg, 9), dtype=torch.float32, device=dev)
        for b in range(B):
            ops.positions(tri[b], m8[b], None, pos[b:b + 1], n=N, n_reg=nreg, rows_out=N + nreg, n_views=1)
        pad = torch.ones((B, nreg), dtype=valid_mask.dtype, device=dev)
        return pos, torch.cat([pad, valid_mask], dim=1)

    @torch.no_grad()
    def construct_seq(self, tri_vpos_list, texture_patch_list, valid_mask, vns):
        """models/renderformer.py:126-169 -> (seq [B, Nt, d], padded mask [B, Nt], positions [B, Nt, 9]);
        `texture_patch_list` with the emission channels already log-encoded, as in the reference."""
        eng = self.engine()
        x, pos, _bits, _words, (B, N, Nt, Ntp), _tri, _m8 = eng.construct_seq(tri_vpos_list, texture_patch_list,
                                                                               valid_mask, vns, texture_is_log=True)
        pad = torch.ones((B, self.config.num_register_tokens), dtype=valid_mask.dtype, device=x.device)
        return (x.view(B, Ntp, -1)[:, :Nt], torch.cat([pad, valid_mask.to(x.device)], dim=1), pos[:, :Nt])

    # ---- engine -------------------------------------------------------------------
    def engine(self, op_dtype: torch.dtype = torch.bfloat16) -> Engine:
        """Kernel-ready weight layouts, cached per operand format and (device, parameter versions)."""
        key = (str(self.device), tuple(p._version for p in self.parameters()))
        hit = self._engines.get(op_dtype)
        if hit is None or hit[0] != key:
            self._engines[op_dtype] = hit = (key, Engine(self.config, self.state_dict(), self.device, op_dtype=op_dtype))
        return hit[1]

    @torch.no_grad()
    def forward(self, tri_vpos_list, texture_patch_list, valid_mask, vns, rays_o=None, rays_d=None,
                tri_vpos_view_tf=None, tf32_view_tf: bool = False, *, c2w=None, fov=None, resolution=None):
        """Reference signature and semantics (models/renderformer.py:171-206): tri_vpos_list [B,N,9],
        texture_patch_list [B,N,13,P,P] with the emission channels ALREADY log-encoded (the pipeline does
        that before calling the model, rendering_pipeline.py:67-68), valid_mask [B,N], vns [B,N,9],
        rays_o [B,V,3] (must be 0: the origin of camera-space rays; anything else raises), rays_d [B,V,H,W,3] camera-space ray
        map (H != W allowed, within the size rules of config.view_grid), tri_vpos_view_tf [B,V,N,9] camera-space
        vertices.  Returns log-encoded images [B, V, 3, H, W] like the reference.  Alternatively pass cameras as
        keywords (`c2w` [B,V,4,4], `fov` [B,V,1] degrees, `resolution` an int or (H, W), fov spanning the longer
        side as in `RenderFormerRenderingPipeline.render`) and leave rays_d / tri_vpos_view_tf None.  `tf32_view_tf`
        is accepted and ignored; the operand format follows the ambient `torch.autocast("cuda", dtype)` like
        the reference's (fp16 outside an autocast region).  The pipeline calls the engine
        directly and skips the log round trip."""
        if rays_o is not None and bool((rays_o != 0).any()):
            # the reference rotates the queries with RoPE at ray_pos = rays_o (view_transformer.py:109,
            # attention.py:668-671); this engine hard-wires the camera-space identity (origin 0)
            raise ValueError("RenderFormer.forward: rays_o must be 0 (camera-space rays, as the pipeline passes them)")
        eng = self.engine(operand_dtype(torch.get_autocast_dtype("cuda") if torch.is_autocast_enabled("cuda") else torch.float16))
        st = eng.encode_scene(tri_vpos_list, texture_patch_list, valid_mask, vns, texture_is_log=True)
        if rays_d is not None and tri_vpos_view_tf is not None:
            B, H, W = rays_d.shape[0], rays_d.shape[2], rays_d.shape[3]
            out = [eng.render_views(st, b, None, None, (H, W), rays_d=rays_d[b], tri_cam=tri_vpos_view_tf[b])
                   for b in range(B)]
        elif c2w is not None and fov is not None and resolution is not None:
            out = [eng.render_views(st, b, c2w[b], fov[b], resolution) for b in range(c2w.shape[0])]
        else:
            raise ValueError("RenderFormer.forward needs either rays_d + tri_vpos_view_tf (reference signature) "
                             "or the c2w / fov / resolution keywords")
        hdr = torch.stack(out, dim=0)  # [B,V,H,W,3]
        return torch.log10(hdr + 1.0).permute(0, 1, 4, 2, 3)


class UploadRing:
    """Persistent device staging buffers for host -> device uploads on a copy stream.

    Fresh `tensor.to(device)` allocations per scene looked free until the caching allocator had to fall back
    to cudaMalloc for a 100-200 MB block while the previous blocks were still pinned down by
    `record_stream`: that call waits for the device and stalled the host for ~25 ms every other scene
    (r02f).  Here slot i % depth is overwritten only after the consumer of its previous content has been
    enqueued (`release`), and nothing is allocated in steady state."""

    def __init__(self, device, copy_stream, depth: int = 2):
        self.dev, self.copy, self.depth = device, copy_stream, depth
        self.slots = [dict() for _ in range(depth)]
        self.free = [None] * depth
        self.n = 0

    PER_TRIANGLE = ("triangles", "texture", "mask", "vn")

    def put(self, host_tensors: dict, pad_to: Optional[int] = None):
        """-> (device tensors, event that fires when they are complete, slot).  With `pad_to` the per-triangle
        tensors land in the first N rows of buffers with `pad_to` rows (batch_infer.py:37-47 pads every scene of
        a folder to one length): the mask tail is cleared, the other tails keep whatever an earlier scene left
        there -- masked triangles never reach a valid token."""
        slot = self.n % self.depth
        self.n += 1
        bufs = self.slots[slot]
        fresh = False
        for k, t in host_tensors.items():
            shape = tuple(t.shape)
            if pad_to is not None and k in self.PER_TRIANGLE:
                if t.shape[1] > pad_to:
                    raise ValueError(f"scene has {t.shape[1]} triangles, pad_to is {pad_to}")
                shape = (t.shape[0], pad_to) + tuple(t.shape[2:])
            b = bufs.get(k)
            if b is None or tuple(b.shape) != shape or b.dtype != t.dtype:
                bufs[k] = torch.zeros(shape, dtype=t.dtype, device=self.dev)
                fresh = True
        if self.free[slot] is not None:
            self.copy.wait_event(self.free[slot])
        if fresh or self.free[slot] is None:  # buffers were allocated / zeroed on the current stream
            self.copy.wait_stream(torch.cuda.current_stream(self.dev))
        with torch.cuda.stream(self.copy):
            for k, t in host_tensors.items():
                if pad_to is not None and k in self.PER_TRIANGLE:
                    n = t.shape[1]
                    bufs[k][:, :n].copy_(t, non_blocking=True)
                    if k == "mask" and n < pad_to:
                        bufs[k][:, n:] = False
                else:
                    bufs[k].copy_(t, non_blocking=True)
            ev = torch.cuda.Event()
            ev.record(self.copy)
        return {k: bufs[k] for k in host_tensors}, ev, slot

    def release(self, slot: int, consumer_stream) -> None:
        ev = torch.cuda.Event()
        ev.record(consumer_stream)
        self.free[slot] = ev


_warned_fp32 = [False]


def operand_dtype(torch_dtype: torch.dtype) -> torch.dtype:
    """Tensor-core operand format for a requested `torch_dtype` (rendering_pipeline.py:98 accepts bfloat16,
    float16, float32): float16 -> fp16 operands, bfloat16 -> bf16 operands; float32 has no tensor-core format
    on this path and maps to fp16 operands with fp32 accumulation -- the most precise available (~1e-3
    class error on HDR pixels) -- with a one-time warning."""
    assert torch_dtype in (torch.bfloat16, torch.float16, torch.float32), \
        f"Invalid precision: {torch_dtype}\nChoose from: torch.bfloat16, torch.float16, torch.float32"
    if torch_dtype == torch.float32 and not _warned_fp32[0]:
        import warnings
        warnings.warn("renderformer_b200: torch_dtype=float32 runs with fp16 tensor-core operands and fp32 accumulation "
                      "(there is no fp32 tensor-core path); expect ~1e-3 relative error on HDR pixels")
        _warned_fp32[0] = True
    return torch.bfloat16 if torch_dtype == torch.bfloat16 else torch.float16


class RenderFormerRenderingPipeline:
    """Same call surface as pipelines/rendering_pipeline.py:8-128."""

    def __init__(self, model: RenderFormer):
        self.model = model
        self.config = model.config
        self.ray_generator = None  # rays are generated inside the fused ray-token kernel
        self.view_chunk = 8
        # Opt-in CUDA-graph replay of `render` (pipeline.cuda_graphs = True): the ~220 kernel launches
        # of a call are captured once per input signature and replayed, which removes the host launch
        # cost (dominant for small scenes / low resolutions) and shrinks the gaps between kernels.
        # Each cached graph pins its activations (a few GB for Large at 512^2).
        # Independent view chunks can run on several CUDA streams: kernels of different chunks then fill
        # each other's partial last waves and ramp-up / drain bubbles (every kernel here occupies a whole
        # SM per CTA).  1 = sequential chunks.
        self.view_streams = 1
        self._side_streams = []
        self.cuda_graphs = False
        # `render` hands out a copy of the graph's static output (0.07 ms for 32 frames) so that results of
        # consecutive calls stay valid; set True to receive the static tensor itself (overwritten by the next
        # call with the same signature)
        self.graph_static_outputs = False
        self.max_cached_graphs = 4
        self._graphs = {}
        self._static_states = {}
        self.replayed_launches = 0  # kernels launched through graph replays (bench.py's gpu_launches)

    @classmethod
    def from_pretrained(cls, model_id: str):
        model = RenderFormer.from_pretrained(model_id)
        model.eval()
        return cls(model)

    @property
    def device(self):
        return self.model.device

    def to(self, device):
        self.model.to(device)

    @torch.no_grad()
    def encode(self, triangles, texture, mask, vn, shard=None, texture_own_rows: bool = False,
               torch_dtype: torch.dtype = torch.float16) -> SceneState:
        """View-independent stage only (exposed for multi-GPU view sharding).  With `cuda_graphs` the
        returned SceneState is the graph's static output (overwritten by the next call of that shape).
        `shard` (engine.RowShard, see renderformer_b200.dist.row_shard) splits the token rows of the
        stage over the ranks; every rank passes the same scene and gets the complete state."""
        eng = self.model.engine(operand_dtype(torch_dtype))
        inputs = (triangles, texture, mask, vn)
        kw = dict(shard=shard, texture_own_rows=texture_own_rows)
        if self.cuda_graphs and all(t.is_cuda for t in inputs):
            tag = ("encode", id(eng)) if shard is None else ("encode", id(eng), shard.rank, shard.world, texture_own_rows)
            st = self._graph_entry(tag + self._sig(inputs), inputs,
                                   lambda a, b, c, d: eng.encode_scene(a, b, c, d, **kw))
            st.static = True
            return st
        return eng.encode_scene(triangles, texture, mask, vn, **kw)

    def view_geometry(self, resolution, overscan: bool = False):
        """(canvas, window, image) of a render: the (H, W) canvas the model runs on, the (h, w, top, left) window of
        it that is returned (None: the whole canvas) and the (h, w) of the returned images.  Without `overscan`
        the size must be on the decoder's grid (config.view_grid); with it any size is rendered on the canvas of
        config.overscan_grid.  Raises ValueError before anything is launched."""
        if not overscan:
            hw = view_grid(self.config, resolution)
            return hw, None, hw
        hw, canvas, (top, left) = overscan_grid(self.config, resolution)
        return canvas, (None if canvas == hw else (*hw, top, left)), hw

    @torch.no_grad()
    def intrinsics_from_fov(self, fov, resolution, fit: str = "auto") -> torch.Tensor:
        """Pinhole intrinsics fp32 [B, V, 4] = (f, f, W/2, H/2) on the device for `render(..., intrinsics=...)`, from
        fov [B, V, 1] (or [B, V]) in degrees and the H x W size of the RETURNED image (`resolution`: an int or
        (H, W), any positive size).  `fit` is the side the fov spans, as Blender's camera sensor fit: "auto" (the
        longer side: the camera `render(..., fov=...)` uses, to the bit), "horizontal" (the width) or "vertical"
        (the height): f = side / 2 / tan(fov / 2)."""
        from . import ops
        H, W = _size_pair(resolution)
        if fit not in ops.FITS:
            raise ValueError(f"fit must be one of {sorted(ops.FITS)}, got {fit!r}")
        if fov.dim() == 3 and fov.shape[-1] == 1:
            fov = fov[..., 0]
        if fov.dim() != 2:
            raise ValueError(f"fov must be [B, V, 1] or [B, V], got {list(fov.shape)}")
        f = fov.to(self.device, torch.float32).contiguous()
        out = torch.empty((*f.shape, 4), dtype=torch.float32, device=self.device)
        if f.numel():
            ops.intrinsics_from_fov(f, out, n_views=f.numel(), height=H, width=W, fit=fit)
        return out

    @torch.no_grad()
    def render_views(self, state: SceneState, c2w, fov=None, resolution=512, overscan: bool = False,
                     intrinsics=None, distortion=None, lens: str = "opencv", _eager: bool = False) -> torch.Tensor:
        """View-dependent stage of `render` on an encoded scene -> HDR [B,V,H,W,3]; `resolution`, `overscan` and the
        camera (`fov` or `intrinsics`, with `distortion` and `lens`) as in `render`."""
        eng = self.model.engine(state.v_all.dtype)  # the operand format the scene state was built in
        canvas, window, hw = self.view_geometry(resolution, overscan)
        kind, cam = view_camera(c2w, fov, intrinsics, distortion, lens, canvas, window)
        if self.cuda_graphs and not _eager and getattr(state, "static", False) and c2w.is_cuda and cam.is_cuda:
            # the graph reads the persistent state in place (no copy of the 300 MB of hoisted K / V)
            return self._graph_entry(("views", id(eng), id(state), kind, canvas, window, self.view_chunk) +
                                     self._sig((c2w, cam)), (c2w, cam),
                                     lambda a, k: self.render_views(state, a, resolution=hw, overscan=overscan,
                                                                    _eager=True, **camera_kwargs(kind, k)))
        B, V = c2w.shape[:2]
        if V == 0:  # a rank whose view slice is empty (fewer views than ranks)
            return torch.empty((B, 0, *hw, 3), dtype=torch.float32, device=self.device)
        jobs = [(b, v0) for b in range(B) for v0 in range(0, V, self.view_chunk)]
        # every decoder pass writes its images straight into its slice of the result (no torch.cat afterwards); with
        # overscan its last conv stores only the window, so no canvas-sized image exists
        result = torch.empty((B, V, *hw, 3), dtype=torch.float32, device=self.device)
        cam_kw = camera_kwargs(kind, cam)
        fov = cam_kw.pop("fov", None)

        def job(b, v0):
            s = slice(v0, v0 + self.view_chunk)
            eng.render_views(state, b, c2w[b, s], None if fov is None else fov[b, s], canvas, out=result[b, s],
                             window=window, **{k: t[b, s] if isinstance(t, torch.Tensor) else t
                                               for k, t in cam_kw.items()})
        n_str = min(self.view_streams, len(jobs))
        if n_str <= 1:
            for b, v0 in jobs:
                job(b, v0)
            return result
        dev = self.device
        while len(self._side_streams) < n_str:
            self._side_streams.append(torch.cuda.Stream(dev))
        cur = torch.cuda.current_stream(dev)
        fork = torch.cuda.Event()
        fork.record(cur)
        for i, (b, v0) in enumerate(jobs):
            side = self._side_streams[i % n_str]
            if i < n_str:
                side.wait_event(fork)
            with torch.cuda.stream(side):
                job(b, v0)
        for side in self._side_streams[:n_str]:
            ev = torch.cuda.Event()
            ev.record(side)
            cur.wait_event(ev)
        return result

    @torch.no_grad()
    def render(self, triangles, texture, mask, vn, c2w, fov=None, resolution=512,
               torch_dtype: torch.dtype = torch.float16, overscan: bool = False, intrinsics=None, distortion=None,
               lens: str = "opencv"):
        """triangles [B,N,3,3], texture [B,N,13,32,32], mask [B,N] bool, vn [B,N,3,3], c2w [B,V,4,4],
        fov [B,V,1] degrees or intrinsics [B,V,4] -> HDR [B,V,H,W,3] fp32.

        `resolution` is an int (square H = W) or a (height, width) pair; sides must be multiples of 64 for the
        swin models and of 8 for full attention (config.view_grid, checked before any launch).  Camera: pinhole,
        square pixels, principal point at the image centre, `fov` spanning the LONGER image side (Blender's
        "Auto" sensor fit), i.e. f = max(H, W) / 2 / tan(fov / 2); for H = W this is the reference's camera.

        `overscan=True` lifts the size rule: `resolution` may be any positive int or (H, W), e.g. (1080, 1920).  The
        model then runs on the smallest canvas on the grid that holds the image (config.overscan_grid; 1088 x 1920
        for 1080p), centred, with the SAME camera as above for the H x W image, and only the H x W window is stored.
        Every returned pixel is the model's output for a real H x W pinhole image; the border costs the decoder
        0.7 % more pixels at 1080p and 4K, 6.7 % at 720p.  A size already on the grid renders exactly as without
        overscan.

        `intrinsics` [B,V,4] = (fx, fy, cx, cy) per view, in place of `fov`, renders calibrated or off-axis pinhole
        cameras: separate focal lengths and any principal point, in pixels of the RETURNED H x W image (with
        overscan too: the window, not the canvas).  The centre of pixel (row i, column j) is (j + 0.5, i + 0.5),
        as in COLMAP; with an OpenCV K add 0.5 to cx and cy.  The ray of a pixel at (u, v) is
        normalize(((u - cx) / fx, -(v - cy) / fy, -1)) in camera space (x right, y up, looking down -z), and the
        `fov` camera is fx = fy = max(H, W) / 2 / tan(fov / 2), cx = W / 2, cy = H / 2
        (`intrinsics_from_fov`; the render is then bit-identical to the `fov` one).  Exactly one of `fov` and
        `intrinsics` is given (config.view_camera).  Intrinsics on the host are checked (finite, fx, fy > 0);
        on the device they are used as they are, without a synchronising read-back.

        `distortion` (with `intrinsics`) renders through a lens-distorted camera; `lens` names its model, as OpenCV
        and COLMAP define them.  "opencv": [B,V,8] = (k1, k2, p1, p2, k3, k4, k5, k6), OpenCV's distCoeffs order and
        COLMAP's FULL_OPENCV ([B,V,4] and [B,V,5] too: the missing coefficients are zero).  A pixel at (u, v) has the
        distorted coordinates xd = (u - cx) / fx, yd = (v - cy) / fy, and with r2 = x^2 + y^2 and
        g = (1 + k1 r2 + k2 r2^2 + k3 r2^3) / (1 + k4 r2 + k5 r2^2 + k6 r2^3) the lens maps (x, y) to
        xd = x g + 2 p1 x y + p2 (r2 + 2 x^2), yd = y g + p1 (r2 + 2 y^2) + 2 p2 x y; the ray is normalize((x, -y, -1)).
        "fisheye": [B,V,4] = (k1, k2, k3, k4) of OpenCV's fisheye model and COLMAP's OPENCV_FISHEYE: the ray at
        angle theta from the axis lands at rd = |(xd, yd)| = theta (1 + k1 theta^2 + k2 theta^4 + k3 theta^6 +
        k4 theta^8), so rays at 90 degrees and more are rendered too; all-zero coefficients are the equidistant fisheye.
        The ray kernel inverts the lens per pixel by Newton's method.  Coefficients on the host are checked
        (config.lens_check): the lens must invert on the whole canvas, overscan border included; on the device they
        are used as they are.  `lens="opencv"` with all coefficients zero renders bit-identically to `intrinsics`
        alone.  `scene_io.read_colmap_cameras` reads COLMAP cameras into these arguments.

        `texture` may also be [B,N,13]: per-triangle constants (what scene_processor/to_h5.py:37-66
        expands to the 32x32 texel grid with a fixed triangular mask).  The texture projection then
        uses texel-summed weights -- no 218 MB texel grid has to exist or be uploaded
        (`renderformer_b200.scene_io.to_pipeline_inputs(..., constant_texture=True)`).

        `torch_dtype` (validated like the reference, rendering_pipeline.py:98) selects the tensor-core
        operand format of the transformer stacks: float16 (the default, as in the reference CLIs) ->
        fp16, bfloat16 -> bf16, float32 -> fp16 operands with a warning (`operand_dtype`); accumulation,
        softmax, norms and the residual stream are fp32 in every mode and the result is always fp32.
        Unlike the reference (:68) the caller's `texture` is not modified."""
        op = operand_dtype(torch_dtype)
        canvas, window, _ = self.view_geometry(resolution, overscan)  # size errors before any launch
        kind, cam = view_camera(c2w, fov, intrinsics, distortion, lens, canvas, window)
        inputs = (triangles, texture, mask, vn, c2w, cam)
        if self.cuda_graphs and all(t.is_cuda for t in inputs):
            out = self._render_graphed(inputs, resolution, op, overscan, kind)
            return out if self.graph_static_outputs else out.clone()
        state = self.encode(triangles, texture, mask, vn, torch_dtype=op)
        return self.render_views(state, c2w, fov, resolution, overscan, intrinsics, distortion, lens)

    def _graph_entry(self, key, inputs, fn):
        """Capture `fn(*static_inputs)` once per key, replay it with `inputs` copied into the static
        buffers; returns the graph's static result."""
        entry = self._graphs.get(key)
        if entry is None:
            if len(self._graphs) >= self.max_cached_graphs:
                self._graphs.pop(next(iter(self._graphs)))
            static_in = [t.detach().clone().contiguous() for t in inputs]
            side = torch.cuda.Stream(self.device)
            side.wait_stream(torch.cuda.current_stream(self.device))
            with torch.cuda.stream(side):  # warm-up outside the capture: lazy attribute set-up, maps, allocator
                for _ in range(2):
                    fn(*static_in)
            torch.cuda.current_stream(self.device).wait_stream(side)
            graph = torch.cuda.CUDAGraph()
            n0 = L.launch_count()
            # thread_local: torch.distributed's watchdog thread keeps polling events while a graph with NCCL
            # collectives inside (row-sharded scene stage) is being captured
            with torch.cuda.graph(graph, capture_error_mode="thread_local"):
                static_out = fn(*static_in)
            entry = self._graphs[key] = (graph, static_in, static_out, L.launch_count() - n0)
        graph, static_in, static_out, n_kernels = entry
        for dst, src in zip(static_in, inputs):
            dst.copy_(src, non_blocking=True)
        graph.replay()
        self.replayed_launches += n_kernels
        return static_out

    @staticmethod
    def _sig(tensors):
        return tuple((tuple(t.shape), t.dtype) for t in tensors)

    def _render_graphed(self, inputs, resolution, op: torch.dtype = torch.bfloat16, overscan: bool = False,
                        camera: str = "fov") -> torch.Tensor:
        """`inputs` = (triangles, texture, mask, vn, c2w, camera tensor); `camera` names the last as
        config.view_camera does: "fov", "intrinsics", "opencv" or "fisheye" (a static input of the graph either way,
        and part of its key)."""
        eng = self.model.engine(op)
        canvas, window, _ = self.view_geometry(resolution, overscan)

        def run(tri, tex, mask, vn, c2w, cam):
            return self.render_views(eng.encode_scene(tri, tex, mask, vn), c2w, resolution=resolution,
                                     overscan=overscan, _eager=True, **camera_kwargs(camera, cam))
        return self._graph_entry(("render", id(eng), camera, canvas, window, self.view_chunk) + self._sig(inputs),
                                 inputs, run)

    def static_scene_state(self, B: int, N: int, torch_dtype: torch.dtype = torch.float16) -> SceneState:
        """The persistent SceneState of this shape (receive buffer of the NCCL broadcast on ranks that do
        not encode; one per (B, N), reused by every call so that graphs captured on it stay valid);
        `render_views` on it is replayed from a CUDA graph when `cuda_graphs` is on."""
        eng = self.model.engine(operand_dtype(torch_dtype))
        key = (id(eng), B, N)
        if key not in self._static_states:
            st = eng.alloc_scene_state(B, N)
            st.static = True
            self._static_states[key] = st
        return self._static_states[key]

    def __call__(self, *args, **kwargs):
        return self.render(*args, **kwargs)

    @staticmethod
    def hdr_to_ldr(hdr: torch.Tensor, tone_mapper: str = "none") -> torch.Tensor:
        """uint8 LDR image(s) from the HDR output, on the device: what infer.py:94-98 does with numpy
        after the download ('none' = clip + truncate, bit-exact; 'pbr_neutral' = Khronos curve + sRGB)."""
        from . import ops
        return ops.ldr_quantize(hdr, tone_mapper)

    @torch.no_grad()
    def render_stream(self, scenes, resolution=512, torch_dtype: torch.dtype = torch.float16,
                      ldr: Optional[str] = None, pad_to: Optional[int] = None, overscan: bool = False,
                      lens: str = "opencv"):
        """Render a sequence of scenes given as HOST tensors (the batch_infer.py use case,
        batch_infer.py:103-143): generator over dicts with the keys of `render` ('triangles', 'texture',
        'mask', 'vn', 'c2w', and 'fov' or 'intrinsics', the latter optionally with 'distortion'), yielding one
        pinned-host fp32 HDR tensor [B,V,H,W,3] per scene, in order.  `resolution` is an int or (H, W), and
        `overscan` and `lens` (the model of every scene's 'distortion') as in `render`.

        The host->device copy of scene i+1 (218 MB of texture for 4096 triangles) runs on a copy
        stream while scene i is being rendered, and the device->host copy of image i overlaps scene
        i+1; pass pinned tensors for truly asynchronous copies.  A yielded buffer belongs to a ring
        of three and is overwritten two scenes later -- copy it if it must live longer.
        `ldr='none' | 'pbr_neutral'` tone-maps and quantises on the device and yields uint8 images
        (a quarter of the download).
        `pad_to=N`: scenes with different triangle counts are padded ON THE DEVICE to N triangles (mask False
        behind the real ones, what batch_infer.py:37-47 does on the host with `--padding_length`), so every
        scene has the same input signature and, with `cuda_graphs`, ONE captured graph replays for all of
        them; the images equal those of the unpadded scenes."""
        dev = self.device
        if dev.type != "cuda":
            raise L.RfbError("render_stream needs a CUDA device (there is no CPU fallback)")
        keys = ("triangles", "texture", "mask", "vn", "c2w")
        canvas, window, _ = self.view_geometry(resolution, overscan)
        main = torch.cuda.current_stream(dev)
        copy = torch.cuda.Stream(dev)
        up = UploadRing(dev, copy)

        def upload(sc):
            kind, cam = view_camera(sc["c2w"], sc.get("fov"), sc.get("intrinsics"), sc.get("distortion"), lens, canvas,
                                    window)  # host checks before the copy
            return (kind, *up.put({**{k: sc[k] for k in keys}, kind: cam}, pad_to=pad_to))

        it = iter(scenes)
        first = next(it, None)
        pending = upload(first) if first is not None else None
        ring, slot, prev = [None, None, None], 0, None
        while pending is not None:
            kind, d, ev, uslot = pending
            nxt = next(it, None)
            pending = upload(nxt) if nxt is not None else None  # overlaps with this scene's kernels
            main.wait_event(ev)
            img = self.render(d["triangles"], d["texture"], d["mask"], d["vn"], d["c2w"], resolution=resolution,
                              torch_dtype=torch_dtype, overscan=overscan, **camera_kwargs(kind, d[kind]))
            up.release(uslot, main)  # the staging slot may be overwritten once this render has consumed it
            if ldr is not None:
                img = self.hdr_to_ldr(img, ldr)
            if ring[slot] is None or ring[slot].shape != img.shape or ring[slot].dtype != img.dtype:
                ring[slot] = torch.empty(img.shape, dtype=img.dtype, pin_memory=True)
            host = ring[slot]
            slot = (slot + 1) % 3
            host.copy_(img, non_blocking=True)
            done = torch.cuda.Event()
            done.record(main)
            if prev is not None:
                prev[1].synchronize()
                yield prev[0]
            prev = (host, done)
        if prev is not None:
            prev[1].synchronize()
            yield prev[0]
