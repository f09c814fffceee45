"""Frame writers off the critical path (SURVEY §8 f3; reference batch_infer.py:146-174, infer.py:88-104).

The reference CLIs download every frame synchronously (`.cpu().numpy()`), tone-map it with numpy and hand it
to `imageio.v3.imwrite` (EXR + PNG, then one MP4) inside the render loop -- at a few hundred frames per
second that loop, not the renderer, sets the wall time.  Here the renderer streams pinned host frames
(`RenderFormerRenderingPipeline.render_stream`) and a small pool of worker threads encodes them while the GPU
renders the next scenes (zlib and numpy release the GIL):

  write_exr / read_exr   OpenEXR 2 scanline files (float32 or half channels, ZIP / ZIPS / uncompressed), numpy +
                         zlib only -- imageio / OpenEXR are not needed.  `read_exr` parses what `write_exr` and the
                         common scanline writers produce (tests cross-check both directions against OpenCV).
  write_png / read_png   8-bit RGB / RGBA / grey PNG, numpy + zlib only.
  write_mp4              the CLIs' `video.mp4` (24 fps); needs OpenCV's FFMPEG backend (no H.264 encoder is written
                         here) and raises a clear error without it.
  hdr_to_ldr_host        the CLIs' LDR conversion on the host: 'none' = `(clip(hdr, 0, 1) * 255).astype(uint8)`
                         (bit-identical to batch_infer.py:153-157), 'pbr_neutral' = the published Khronos PBR
                         Neutral curve + sRGB OETF (same formula as the device kernel `rfb_ldr_quantize` mode 1;
                         unpinned: the reference goes through simple_ocio / OpenColorIO, not vendored).
  FrameWriter            bounded pool: `submit(base, hdr)` copies the (ring-owned) host frame and returns at once;
                         files are named like the reference's (`{base}.exr`, `{base}.png`); errors surface in
                         `close()`; LDR frames are kept in submission order for the video.
  render_to_files        `render_stream` + `FrameWriter`: the batch_infer.py loop with uploads, kernels,
                         downloads and file encoding all overlapped.

Nothing here touches the GPU; the module imports without CUDA."""
from __future__ import annotations

import os
import struct
import threading
import zlib
from concurrent.futures import ThreadPoolExecutor
from typing import Dict, Iterable, List, Optional, Sequence

import numpy as np

# --------------------------------------------------------------------------------------------- OpenEXR
_EXR_MAGIC = 20000630
_COMPRESSION = {"none": 0, "zips": 2, "zip": 3}
_LINES_PER_CHUNK = {0: 1, 2: 1, 3: 16}
_PIXEL_TYPES = {1: np.dtype("<f2"), 2: np.dtype("<f4"), 0: np.dtype("<u4")}


def _attr(name: str, typ: str, value: bytes) -> bytes:
    return name.encode() + b"\0" + typ.encode() + b"\0" + struct.pack("<i", len(value)) + value


def _zip_encode(raw: bytes, level: int) -> bytes:
    """OpenEXR's ZIP block coding: de-interleave the bytes (even positions first), byte-wise delta with a +128
    bias, deflate.  A block that does not shrink is stored raw (the reader tells by the size)."""
    a = np.frombuffer(raw, dtype=np.uint8)
    half = (a.size + 1) // 2
    t = np.empty_like(a)
    t[:half] = a[0::2]
    t[half:] = a[1::2]
    d = t.copy()
    d[1:] = t[1:] - t[:-1] + np.uint8(128)  # uint8 arithmetic wraps mod 256, as the C code's cast does
    out = zlib.compress(d.tobytes(), level)
    return out if len(out) < len(raw) else raw


def _zip_decode(data: bytes, raw_size: int) -> bytes:
    if len(data) == raw_size:
        return data
    d = np.frombuffer(zlib.decompress(data), dtype=np.uint8)
    if d.size != raw_size:
        raise ValueError("EXR: ZIP block inflates to the wrong size")
    t = d.copy()
    t[1:] -= np.uint8(128)
    t = np.cumsum(t, dtype=np.uint8)  # running sum mod 256 undoes the delta
    half = (raw_size + 1) // 2
    a = np.empty_like(t)
    a[0::2] = t[:half]
    a[1::2] = t[half:]
    return a.tobytes()


def write_exr(path: str, image: np.ndarray, compression: str = "zip", half: bool = False,
              channels: Optional[Sequence[str]] = None, level: int = 4) -> None:
    """`image` [H, W, C] (C = 1, 3 or 4; float) -> scanline OpenEXR file.  Channel names default to Y / RGB /
    RGBA in the array's order; the file stores them alphabetically as the format requires."""
    img = np.asarray(image)
    if img.ndim == 2:
        img = img[:, :, None]
    if img.ndim != 3 or img.shape[0] < 1 or img.shape[1] < 1:
        raise ValueError(f"write_exr: expected [H, W, C], got {img.shape}")
    H, W, C = img.shape
    names = list(channels) if channels is not None else {1: ["Y"], 3: ["R", "G", "B"], 4: ["R", "G", "B", "A"]}.get(C)
    if names is None or len(names) != C or len(set(names)) != C:
        raise ValueError(f"write_exr: cannot name {C} channels")
    if compression not in _COMPRESSION:
        raise ValueError(f"write_exr: compression must be one of {sorted(_COMPRESSION)}")
    comp = _COMPRESSION[compression]
    ptype = 1 if half else 2
    dt = _PIXEL_TYPES[ptype]
    order = sorted(range(C), key=lambda i: names[i])
    # [H, C(sorted), W] in the file's dtype: one scanline = the channels' rows back to back
    planes = np.ascontiguousarray(np.transpose(img[:, :, order], (0, 2, 1)).astype(dt))

    chlist = b"".join(names[i].encode() + b"\0" + struct.pack("<iB3xii", ptype, 0, 1, 1) for i in order) + b"\0"
    box = struct.pack("<4i", 0, 0, W - 1, H - 1)
    header = struct.pack("<iI", _EXR_MAGIC, 2)
    header += _attr("channels", "chlist", chlist)
    header += _attr("compression", "compression", struct.pack("<B", comp))
    header += _attr("dataWindow", "box2i", box)
    header += _attr("displayWindow", "box2i", box)
    header += _attr("lineOrder", "lineOrder", b"\0")
    header += _attr("pixelAspectRatio", "float", struct.pack("<f", 1.0))
    header += _attr("screenWindowCenter", "v2f", struct.pack("<2f", 0.0, 0.0))
    header += _attr("screenWindowWidth", "float", struct.pack("<f", 1.0))
    header += b"\0"

    lines = _LINES_PER_CHUNK[comp]
    chunks: List[bytes] = []
    for y0 in range(0, H, lines):
        raw = planes[y0:y0 + lines].tobytes()
        data = raw if comp == 0 else _zip_encode(raw, level)
        chunks.append(struct.pack("<ii", y0, len(data)) + data)
    pos = len(header) + 8 * len(chunks)
    table = []
    for c in chunks:
        table.append(pos)
        pos += len(c)
    tmp = path + ".part"
    with open(tmp, "wb") as f:
        f.write(header)
        f.write(struct.pack(f"<{len(table)}Q", *table))
        for c in chunks:
            f.write(c)
    os.replace(tmp, path)  # a reader never sees half a file


def _cstr(buf: bytes, pos: int):
    end = buf.index(b"\0", pos)
    return buf[pos:end].decode("latin-1"), end + 1


def read_exr(path: str, return_channels: bool = False):
    """Scanline OpenEXR (single part; none / ZIPS / ZIP; half, float or uint channels, no sub-sampling) ->
    float32 [H, W, C] with the channels in R, G, B, A order when they have those names, else alphabetical."""
    with open(path, "rb") as f:
        buf = f.read()
    magic, version = struct.unpack_from("<iI", buf, 0)
    if magic != _EXR_MAGIC:
        raise ValueError(f"{path}: not an OpenEXR file")
    if version & 0x1A00:  # tiled (0x200), deep (0x800), multi-part (0x1000)
        raise ValueError(f"{path}: only single-part scanline EXR files are supported")
    pos = 8
    attrs: Dict[str, bytes] = {}
    while buf[pos] != 0:
        name, pos = _cstr(buf, pos)
        _typ, pos = _cstr(buf, pos)
        (size,) = struct.unpack_from("<i", buf, pos)
        attrs[name] = buf[pos + 4:pos + 4 + size]
        pos += 4 + size
    pos += 1
    chans = []
    cl, p = attrs["channels"], 0
    while cl[p] != 0:
        name, p = _cstr(cl, p)
        ptype, _plin, xs, ys = struct.unpack_from("<iB3xii", cl, p)
        p += 16
        if xs != 1 or ys != 1:
            raise ValueError(f"{path}: sub-sampled channels are not supported")
        chans.append((name, _PIXEL_TYPES[ptype]))
    comp = attrs["compression"][0]
    if comp not in _LINES_PER_CHUNK:
        raise ValueError(f"{path}: compression {comp} is not supported (none / ZIPS / ZIP only)")
    x0, y0, x1, y1 = struct.unpack("<4i", attrs["dataWindow"])
    W, H = x1 - x0 + 1, y1 - y0 + 1
    lines = _LINES_PER_CHUNK[comp]
    n_chunks = (H + lines - 1) // lines
    table = struct.unpack_from(f"<{n_chunks}Q", buf, pos)
    line_bytes = sum(dt.itemsize for _, dt in chans) * W
    out = np.empty((H, len(chans), W), dtype=np.float32)
    for off in table:
        y, size = struct.unpack_from("<ii", buf, off)
        n = min(lines, y1 + 1 - y)
        raw = buf[off + 8:off + 8 + size]
        if comp != 0:
            raw = _zip_decode(raw, n * line_bytes)
        p = 0
        for r in range(n):
            for ci, (_, dt) in enumerate(chans):
                out[y - y0 + r, ci] = np.frombuffer(raw, dtype=dt, count=W, offset=p)
                p += dt.itemsize * W
    names = [n for n, _ in chans]
    rank = {"R": 0, "G": 1, "B": 2, "A": 3}
    order = sorted(range(len(names)), key=lambda i: (rank.get(names[i], 4), names[i]))
    img = np.ascontiguousarray(np.transpose(out[:, order], (0, 2, 1)))
    return (img, [names[i] for i in order]) if return_channels else img


# ------------------------------------------------------------------------------------------------- PNG
_PNG_SIG = b"\x89PNG\r\n\x1a\n"
_PNG_COLOR = {1: 0, 3: 2, 4: 6}


def _png_chunk(tag: bytes, data: bytes) -> bytes:
    return struct.pack(">I", len(data)) + tag + data + struct.pack(">I", zlib.crc32(tag + data) & 0xFFFFFFFF)


def write_png(path: str, image: np.ndarray, level: int = 4) -> None:
    """uint8 [H, W] / [H, W, 1|3|4] -> PNG (8 bits per sample, filter 0, no interlace)."""
    img = np.asarray(image)
    if img.dtype != np.uint8:
        raise ValueError(f"write_png: uint8 expected, got {img.dtype} (quantise first: hdr_to_ldr_host)")
    if img.ndim == 2:
        img = img[:, :, None]
    if img.ndim != 3 or img.shape[2] not in _PNG_COLOR:
        raise ValueError(f"write_png: expected [H, W, 1|3|4], got {img.shape}")
    H, W, C = img.shape
    rows = np.zeros((H, 1 + W * C), dtype=np.uint8)  # leading filter byte 0 = 'None'
    rows[:, 1:] = img.reshape(H, W * C)
    data = _PNG_SIG + _png_chunk(b"IHDR", struct.pack(">IIBBBBB", W, H, 8, _PNG_COLOR[C], 0, 0, 0))
    data += _png_chunk(b"IDAT", zlib.compress(rows.tobytes(), level)) + _png_chunk(b"IEND", b"")
    tmp = path + ".part"
    with open(tmp, "wb") as f:
        f.write(data)
    os.replace(tmp, path)


def read_png(path: str) -> np.ndarray:
    """8-bit non-interlaced grey / RGB / RGBA PNG -> uint8 [H, W, C] (all five scanline filters)."""
    with open(path, "rb") as f:
        buf = f.read()
    if buf[:8] != _PNG_SIG:
        raise ValueError(f"{path}: not a PNG file")
    pos, idat, ihdr = 8, [], None
    while pos < len(buf):
        (n,) = struct.unpack_from(">I", buf, pos)
        tag, body = buf[pos + 4:pos + 8], buf[pos + 8:pos + 8 + n]
        (crc,) = struct.unpack_from(">I", buf, pos + 8 + n)
        if zlib.crc32(tag + body) & 0xFFFFFFFF != crc:
            raise ValueError(f"{path}: CRC mismatch in chunk {tag!r}")
        if tag == b"IHDR":
            ihdr = struct.unpack(">IIBBBBB", body)
        elif tag == b"IDAT":
            idat.append(body)
        elif tag == b"IEND":
            break
        pos += 12 + n
    W, H, depth, color, _, _, interlace = ihdr
    C = {0: 1, 2: 3, 6: 4}.get(color)
    if depth != 8 or C is None or interlace:
        raise ValueError(f"{path}: only 8-bit non-interlaced grey / RGB / RGBA PNGs are supported")
    raw = np.frombuffer(zlib.decompress(b"".join(idat)), dtype=np.uint8).reshape(H, 1 + W * C)
    out = np.zeros((H, W * C), dtype=np.uint8)
    prev = np.zeros(W * C, dtype=np.int32)
    for y in range(H):
        ft, line = int(raw[y, 0]), raw[y, 1:].astype(np.int32)
        if ft == 0:
            cur = line
        elif ft == 2:
            cur = (line + prev) & 255
        else:  # Sub, Average, Paeth depend on the pixel to the left: walk the row
            cur = np.zeros(W * C, dtype=np.int32)
            for i in range(W * C):
                a = cur[i - C] if i >= C else 0
                b = prev[i]
                c = prev[i - C] if i >= C else 0
                if ft == 1:
                    pred = a
                elif ft == 3:
                    pred = (a + b) >> 1
                elif ft == 4:
                    pa, pb, pc = abs(b - c), abs(a - c), abs(a + b - 2 * c)
                    pred = a if (pa <= pb and pa <= pc) else (b if pb <= pc else c)
                else:
                    raise ValueError(f"{path}: bad filter type {ft}")
                cur[i] = (line[i] + pred) & 255
        out[y] = cur
        prev = cur
    return out.reshape(H, W, C)


# ------------------------------------------------------------------------------------------------- MP4
def write_mp4(path: str, frames: Sequence[np.ndarray], fps: int = 24) -> None:
    """uint8 RGB frames -> MP4 (batch_infer.py:168-172 `imageio.v3.imwrite(video_path, frames, fps=24)`).
    Encoding is delegated to OpenCV's FFMPEG backend; there is no fallback encoder."""
    try:
        import cv2
    except ImportError as e:  # pragma: no cover - depends on the image
        raise RuntimeError("write_mp4 needs OpenCV (cv2) with the FFMPEG backend; write PNG frames instead") from e
    if len(frames) == 0:
        raise ValueError("write_mp4: no frames")
    H, W = frames[0].shape[:2]
    tmp = path + ".part.mp4"
    w = cv2.VideoWriter(tmp, cv2.VideoWriter_fourcc(*"mp4v"), float(fps), (W, H))
    if not w.isOpened():
        raise RuntimeError("write_mp4: OpenCV could not open an mp4v encoder (FFMPEG backend missing?)")
    try:
        for fr in frames:
            fr = np.asarray(fr)
            if fr.dtype != np.uint8 or fr.shape != (H, W, 3):
                raise ValueError("write_mp4: frames must be uint8 [H, W, 3] of one size")
            w.write(np.ascontiguousarray(fr[:, :, ::-1]))  # OpenCV wants BGR
    finally:
        w.release()
    os.replace(tmp, path)


# ------------------------------------------------------------------------------------------------- LDR
def _srgb_oetf(x: np.ndarray) -> np.ndarray:
    x = np.clip(x, 0.0, 1.0)
    return np.where(x <= 0.0031308, 12.92 * x, 1.055 * np.power(x, np.float32(1.0 / 2.4)) - 0.055).astype(np.float32)


def hdr_to_ldr_host(hdr: np.ndarray, tone_mapper: str = "none") -> np.ndarray:
    """float HDR [..., 3] -> uint8.  'none' follows batch_infer.py:153-157 / infer.py:94-98 to the bit:
    `(np.clip(hdr, 0, 1) * 255).astype(np.uint8)`."""
    hdr = np.asarray(hdr, dtype=np.float32)
    if tone_mapper in ("none", None):
        ldr = np.clip(hdr, 0, 1)
    elif tone_mapper in ("pbr_neutral", "Khronos PBR Neutral"):
        start, desat = np.float32(0.8 - 0.04), np.float32(0.15)
        x = hdr.min(axis=-1, keepdims=True)
        off = np.where(x < 0.08, x - 6.25 * x * x, 0.04).astype(np.float32)
        c = hdr - off
        peak = c.max(axis=-1, keepdims=True)
        d = np.float32(1.0) - start
        safe = np.maximum(peak, start)  # the branch below only applies where peak >= start
        new_peak = 1.0 - d * d / (safe + d - start)
        scaled = c * (new_peak / safe)
        t = 1.0 - 1.0 / (desat * (safe - new_peak) + 1.0)
        comp = scaled + (new_peak - scaled) * t
        ldr = _srgb_oetf(np.where(peak >= start, comp, c))
    else:
        raise ValueError(f"tone mapper {tone_mapper!r}: only 'none' and 'pbr_neutral' are provided (AgX / Filmic "
                         "need OpenColorIO LUTs that are not vendored)")
    return (np.clip(np.nan_to_num(ldr, nan=0.0), 0, 1) * 255).astype(np.uint8)


# ----------------------------------------------------------------------------------------- writer pool
class FrameWriter:
    """Encode frames on worker threads while the renderer goes on.

    `submit(base, hdr)` takes one HDR frame [H, W, 3] (float32, e.g. a slice of the pinned buffer that
    `render_stream` yields and reuses two scenes later -- it is copied here, 3 MB at 512x512), returns
    immediately unless `max_pending` frames are already queued (back-pressure instead of unbounded memory), and
    a worker writes `{base}.exr` and / or `{base}.png` under `out_dir`.  `close()` waits for all of them,
    raises the first worker error, and returns the LDR frames in submission order when `keep_ldr` is set."""

    def __init__(self, out_dir: str, workers: int = 4, max_pending: int = 64, tone_mapper: str = "none",
                 write_hdr: bool = True, write_ldr: bool = True, keep_ldr: bool = False,
                 exr_compression: str = "none", exr_half: bool = False, png_level: int = 1):
        if tone_mapper not in ("none", None, "pbr_neutral", "Khronos PBR Neutral"):
            hdr_to_ldr_host(np.zeros((1, 1, 3), np.float32), tone_mapper)  # raises with the explanation
        self.out_dir = out_dir
        os.makedirs(out_dir, exist_ok=True)
        self.tone_mapper, self.write_hdr, self.write_ldr, self.keep_ldr = tone_mapper, write_hdr, write_ldr, keep_ldr
        # float32 mantissas do not deflate (a 512x512 frame: 3.01 of 3.15 MB for 25x the CPU time, 120 vs 5 ms),
        # so the pool writes uncompressed float EXR by default; 'zip' pays off with exr_half (0.8 MB, 28 ms)
        self.exr_compression, self.exr_half, self.png_level = exr_compression, exr_half, png_level
        self._pool = ThreadPoolExecutor(max_workers=max(1, workers), thread_name_prefix="rfb-writer")
        self._slots = threading.BoundedSemaphore(max(1, max_pending))
        self._futures = []
        self._ldr: Dict[int, np.ndarray] = {}
        self._lock = threading.Lock()
        self._closed = False
        self.paths: List[str] = []

    def _job(self, idx: int, base: str, hdr: np.ndarray):
        try:
            if self.write_hdr:
                write_exr(os.path.join(self.out_dir, base + ".exr"), hdr, self.exr_compression, self.exr_half)
            if self.write_ldr or self.keep_ldr:
                ldr = hdr_to_ldr_host(hdr, self.tone_mapper)
                if self.write_ldr:
                    write_png(os.path.join(self.out_dir, base + ".png"), ldr, self.png_level)
                if self.keep_ldr:
                    with self._lock:
                        self._ldr[idx] = ldr
        finally:
            self._slots.release()

    def submit(self, base: str, hdr) -> None:
        if self._closed:
            raise RuntimeError("FrameWriter is closed")
        arr = hdr.numpy() if hasattr(hdr, "numpy") else np.asarray(hdr)
        if arr.ndim != 3 or arr.shape[2] != 3:
            raise ValueError(f"FrameWriter.submit: one [H, W, 3] frame expected, got {arr.shape}")
        frame = np.array(arr, dtype=np.float32, copy=True)  # the caller's buffer may be a reused ring slot
        self._slots.acquire()
        idx = len(self._futures)
        self.paths.append(os.path.join(self.out_dir, base))
        self._futures.append(self._pool.submit(self._job, idx, base, frame))

    def close(self) -> List[np.ndarray]:
        self._closed = True
        err = None
        for f in self._futures:
            e = f.exception()
            err = err or e
        self._pool.shutdown(wait=True)
        if err is not None:
            raise err
        return [self._ldr[i] for i in sorted(self._ldr)]

    def __enter__(self):
        return self

    def __exit__(self, exc_type, exc, tb):
        if exc_type is None:
            self.close()
        else:  # do not mask the caller's error; still drain the pool
            self._closed = True
            self._pool.shutdown(wait=True)
        return False


def prefetch(iterable: Iterable, depth: int = 2):
    """Run `iterable` (e.g. a generator that loads a scene file, expands its 218 MB texel grid and pins it) on a
    background thread, `depth` items ahead of the consumer: the input side of the batch path off the critical path
    (batch_infer.py:103-110 uses DataLoader workers for this).  Order is kept; an exception in the producer is
    re-raised in the consumer at the position where it happened; closing the generator stops the thread."""
    import queue
    q: "queue.Queue" = queue.Queue(maxsize=max(1, depth))
    stop = threading.Event()
    END, ERR = object(), object()

    def put(item) -> bool:
        while not stop.is_set():
            try:
                q.put(item, timeout=0.1)
                return True
            except queue.Full:
                continue
        return False

    def run():
        try:
            for item in iterable:
                if not put(item):
                    return
            put(END)
        except BaseException as e:  # noqa: BLE001  (handed to the consumer)
            put((ERR, e))

    t = threading.Thread(target=run, name="rfb-prefetch", daemon=True)
    t.start()
    try:
        while True:
            item = q.get()
            if item is END:
                return
            if isinstance(item, tuple) and len(item) == 2 and item[0] is ERR:
                raise item[1]
            yield item
    finally:
        stop.set()
        t.join(timeout=5)


def render_to_files(pipeline, scenes: Iterable[dict], names: Sequence[str], out_dir: str, resolution=512,
                    torch_dtype=None, tone_mapper: str = "none", pad_to: Optional[int] = None,
                    save_video: bool = False, workers: int = 4, fps: int = 24, sharded: bool = False,
                    overscan: bool = False, lens: str = "opencv") -> List[str]:
    """The batch_infer.py loop (batch_infer.py:122-172) with nothing serialised behind the renderer: `scenes`
    (host tensors, the keys of `render`) go through `pipeline.render_stream` (upload of scene i+1 and download
    of image i-1 overlap the kernels of scene i) and every frame is handed to a `FrameWriter`.  Files are
    named like the reference's: `{name}_view_{v}.exr`, `{name}_view_{v}.png`, `video.mp4`.  `names[i]` belongs
    to the i-th scene (a scene dict holding B > 1 scenes takes B consecutive names).  Returns the frame paths
    (without extension) this process wrote, in order.  `resolution` is an int or (H, W), `overscan` (any size,
    rendered on the decoder's grid and cropped), and `lens` (the model of the scenes' 'distortion'), as in `render`.

    `sharded=True` (one process per GPU, `torch.distributed` initialised): every rank iterates the SAME scenes
    through `dist.render_stream_sharded` -- scene stage row-sharded, each rank renders and WRITES its own slice
    of the views (no image gather; the view index in the file name is the global one).  The video is then
    assembled by rank 0 from the PNG files after a barrier."""
    kw = {} if torch_dtype is None else {"torch_dtype": torch_dtype}
    if overscan:
        kw["overscan"] = True
    if lens != "opencv":
        kw["lens"] = lens
    names = list(names)
    rank, world = 0, 1
    if sharded:
        import torch.distributed as dist
        from .dist import render_stream_sharded
        if pad_to is not None:
            raise ValueError("render_to_files: pad_to is not available in the sharded stream (pad the scenes on the host)")
        rank, world = dist.get_rank(), dist.get_world_size()
        stream = render_stream_sharded(pipeline, scenes, resolution=resolution, **kw)
    else:
        stream = ((None, imgs) for imgs in pipeline.render_stream(scenes, resolution=resolution, pad_to=pad_to, **kw))
    k = 0
    own_video = save_video and world == 1
    with FrameWriter(out_dir, workers=workers, tone_mapper=tone_mapper, keep_ldr=own_video) as fw:
        for mine, imgs in stream:
            B, V = imgs.shape[0], imgs.shape[1]
            v0 = 0 if mine is None else mine.start
            if k + B > len(names):
                raise ValueError(f"render_to_files: {len(names)} names for more than {k + B - 1} scenes")
            for b in range(B):
                for v in range(V):
                    fw.submit(f"{names[k + b]}_view_{v0 + v}", imgs[b, v])
            k += B
        ldr = fw.close()
        paths = list(fw.paths)
    if own_video and ldr:
        write_mp4(os.path.join(out_dir, "video.mp4"), ldr, fps=fps)
    elif save_video and world > 1:
        import torch.distributed as dist
        dist.barrier()  # every rank's frames are on disk
        if rank == 0:
            frames = _frames_on_disk(out_dir, names[:k])
            if frames:
                write_mp4(os.path.join(out_dir, "video.mp4"), [read_png(f) for f in frames], fps=fps)
    return paths


def _frames_on_disk(out_dir: str, names: Sequence[str]) -> List[str]:
    """`{name}_view_{v}.png` of the given scenes in (scene, view) order."""
    out = []
    for n in names:
        v = 0
        while os.path.exists(os.path.join(out_dir, f"{n}_view_{v}.png")):
            out.append(os.path.join(out_dir, f"{n}_view_{v}.png"))
            v += 1
    return out
