"""Scene ingestion without trimesh / h5py: JSON scene description -> pipeline tensors.

Restates, with numpy only, what the reference's converter does on the way from a scene JSON to
the HDF5 file `infer.py` reads (SURVEY §8f rank 1):

* scene description format ............ scene_processor/scene_config.py:5-71
* per object: load OBJ, optional unit-sphere normalisation, rotate (x, then y, then z, degrees)
  -> scale -> translate, flat or 30-degree smooth shading, material -> scene_processor/scene_mesh.py:12-93
* per triangle 13 texture channels [diffuse 3 | specular 3 | roughness 1 | normal (0.5, 0.5, 1) |
  emission 3] x 32 x 32 texels, zero outside the triangular texel mask x + y <= 32, stored as
  fp16; cameras as look-at -> camera-to-world matrices ............ scene_processor/to_h5.py:10-92

Parity status: UNPINNED.  trimesh is not installable here, so the converter's output cannot be
compared with the reference's; what the tests pin is the published structure of the example scenes
(examples/cbox.json -> 5633 triangles, SURVEY §8d), closed-form cases (flat shading, look-at
matrices) and invariants (unit normals, smoothing groups split at creases).  Known difference: the
order in which connected components receive their random colours (`rand_tri_diffuse_seed`) follows
the smallest face index here, trimesh's own order may differ; `remesh` (pymeshlab) is not supported.

Host-side data preparation only: nothing here is on the GPU hot path.
"""
from __future__ import annotations

import json
import math
import os
from typing import Dict, List, Optional, Tuple

import numpy as np

TEXELS = 32


# ----------------------------------------------------------------------------------------- OBJ
def load_obj(path: str) -> Tuple[np.ndarray, np.ndarray]:
    """Vertices [n,3] float64 and triangles [m,3] int64 of a Wavefront OBJ file.  Polygons are
    fan-triangulated; texture / normal indices (`f a/b/c`) and negative indices are accepted;
    vertex colours after the coordinates are ignored (the material defines the colour)."""
    verts: List[List[float]] = []
    faces: List[List[int]] = []
    with open(path) as f:
        for line in f:
            if line.startswith("v "):
                p = line.split()
                verts.append([float(p[1]), float(p[2]), float(p[3])])
            elif line.startswith("f "):
                idx = []
                for tok in line.split()[1:]:
                    i = int(tok.split("/")[0])
                    idx.append(i - 1 if i > 0 else len(verts) + i)
                for k in range(1, len(idx) - 1):
                    faces.append([idx[0], idx[k], idx[k + 1]])
    if not verts or not faces:
        raise ValueError(f"{path}: no geometry")
    return np.asarray(verts, dtype=np.float64), np.asarray(faces, dtype=np.int64)


# ----------------------------------------------------------------------------------------- geometry
def rotation_xyz_deg(angles) -> np.ndarray:
    """R = Rz * Ry * Rx: the mesh is rotated about the world x axis first, then y, then z."""
    rx, ry, rz = (math.radians(float(a)) for a in angles)
    cx, sx, cy, sy, cz, sz = math.cos(rx), math.sin(rx), math.cos(ry), math.sin(ry), math.cos(rz), math.sin(rz)
    Rx = np.array([[1, 0, 0], [0, cx, -sx], [0, sx, cx]], dtype=np.float64)
    Ry = np.array([[cy, 0, sy], [0, 1, 0], [-sy, 0, cy]], dtype=np.float64)
    Rz = np.array([[cz, -sz, 0], [sz, cz, 0], [0, 0, 1]], dtype=np.float64)
    return Rz @ Ry @ Rx


def face_normals(tri: np.ndarray) -> np.ndarray:
    """Unit normals of triangles [m,3,3] (zero for degenerate triangles)."""
    n = np.cross(tri[:, 1] - tri[:, 0], tri[:, 2] - tri[:, 0])
    ln = np.linalg.norm(n, axis=-1, keepdims=True)
    return np.where(ln > 0, n / np.maximum(ln, 1e-300), 0.0)


def corner_angles(tri: np.ndarray) -> np.ndarray:
    """Interior angle at each of the three corners of triangles [m,3,3] -> [m,3]."""
    out = np.zeros(tri.shape[:2])
    for c in range(3):
        a = tri[:, (c + 1) % 3] - tri[:, c]
        b = tri[:, (c + 2) % 3] - tri[:, c]
        cosv = (a * b).sum(-1) / np.maximum(np.linalg.norm(a, axis=-1) * np.linalg.norm(b, axis=-1), 1e-300)
        out[:, c] = np.arccos(np.clip(cosv, -1.0, 1.0))
    return out


def _components(n: int, pairs: np.ndarray) -> np.ndarray:
    """Connected-component label of every node; labels are ordered by the smallest node index."""
    parent = np.arange(n)

    def find(i):
        while parent[i] != i:
            parent[i] = parent[parent[i]]
            i = parent[i]
        return i

    for a, b in pairs:
        ra, rb = find(int(a)), find(int(b))
        if ra != rb:
            if ra < rb:
                parent[rb] = ra
            else:
                parent[ra] = rb
    roots = np.array([find(i) for i in range(n)])
    _, labels = np.unique(roots, return_inverse=True)  # roots are minimal indices -> ordered labels
    return labels


def face_adjacency(faces: np.ndarray) -> np.ndarray:
    """Pairs of faces that share an edge (by vertex index) -> [k,2]."""
    m = faces.shape[0]
    e = np.concatenate([faces[:, [0, 1]], faces[:, [1, 2]], faces[:, [2, 0]]], axis=0)
    e.sort(axis=1)
    owner = np.tile(np.arange(m), 3)
    order = np.lexsort((e[:, 1], e[:, 0]))
    e, owner = e[order], owner[order]
    same = (e[1:] == e[:-1]).all(axis=1)
    return np.stack([owner[:-1][same], owner[1:][same]], axis=1)


def corner_normals(verts: np.ndarray, faces: np.ndarray, smooth: bool, crease_deg: float = 30.0) -> np.ndarray:
    """Per-corner shading normals [m,3,3].

    flat:   every corner gets its face normal (the mesh is turned into a triangle soup).
    smooth: faces that meet at less than `crease_deg` form smoothing groups; inside a group a vertex
            normal is the corner-angle-weighted mean of the group's face normals at that vertex, so
            hard edges (a box) stay hard and curved surfaces are interpolated."""
    tri = verts[faces]
    fn = face_normals(tri)
    if not smooth:
        return np.repeat(fn[:, None, :], 3, axis=1)
    adj = face_adjacency(faces)
    if adj.size:
        cosang = (fn[adj[:, 0]] * fn[adj[:, 1]]).sum(-1)
        adj = adj[np.arccos(np.clip(cosang, -1.0, 1.0)) < math.radians(crease_deg)]
    group = _components(faces.shape[0], adj)
    ang = corner_angles(tri)
    key = group[:, None] * (verts.shape[0] + 1) + faces          # (smoothing group, vertex)
    uniq, inv = np.unique(key.reshape(-1), return_inverse=True)
    acc = np.zeros((uniq.shape[0], 3))
    np.add.at(acc, inv, (ang[:, :, None] * fn[:, None, :]).reshape(-1, 3))
    ln = np.linalg.norm(acc, axis=-1, keepdims=True)
    acc = np.where(ln > 0, acc / np.maximum(ln, 1e-300), 0.0)
    out = acc[inv].reshape(faces.shape[0], 3, 3)
    bad = (np.linalg.norm(out, axis=-1) == 0)
    out[bad] = np.repeat(fn[:, None, :], 3, axis=1)[bad]
    return out


def look_at_c2w(position, target=(0.0, 0.0, 0.0), up=(0.0, 0.0, 1.0)) -> np.ndarray:
    """Camera-to-world matrix of a camera at `position` looking at `target` (camera looks along its
    -z axis, +y is up: the Blender / OpenGL convention the model was trained with)."""
    p, t, u = (np.asarray(v, dtype=np.float64) for v in (position, target, up))
    back = p - t
    back /= np.linalg.norm(back)
    right = np.cross(u, back)
    right /= np.linalg.norm(right)
    upv = np.cross(back, right)
    upv /= np.linalg.norm(upv)
    m = np.eye(4)
    m[:3, 0], m[:3, 1], m[:3, 2], m[:3, 3] = right, upv, back, p
    return m


# ----------------------------------------------------------------------------------------- scene
def texel_mask(size: int = TEXELS) -> np.ndarray:
    x, y = np.meshgrid(np.arange(size), np.arange(size), indexing="ij")
    return x + y <= size


def _object_mesh(obj: dict, base_dir: str):
    """Transformed triangles [m,3,3], corner normals [m,3,3] and 8-bit-quantised diffuse colours [m,3]."""
    if obj.get("remesh", False):
        raise NotImplementedError("remesh (pymeshlab) is not supported by the numpy converter")
    verts, faces = load_obj(os.path.join(base_dir, obj["mesh_path"]))
    tr, mat = obj["transform"], obj["material"]
    if tr.get("normalize", True):
        verts = verts - verts.mean(axis=0)
        verts = verts / (np.linalg.norm(verts, axis=-1).max() * 2.0)
    verts = verts @ rotation_xyz_deg(tr["rotation"]).T
    verts = verts * np.asarray(tr["scale"], dtype=np.float64) + np.asarray(tr["translation"], dtype=np.float64)
    normals = corner_normals(verts, faces, bool(mat["smooth_shading"]))
    m = faces.shape[0]
    seed = mat.get("rand_tri_diffuse_seed")
    if seed is not None:
        rng = np.random.RandomState(int(seed))
        hi = int(math.ceil(256 * float(mat.get("random_diffuse_max", 1.0))))
        if mat.get("random_diffuse_type", "per-shading-group") == "per-triangle":
            group = np.arange(m)
        else:
            # connectivity of the shaded mesh: flat shading un-welds every triangle, smooth shading
            # keeps faces of one smoothing group connected
            if mat["smooth_shading"]:
                adj = face_adjacency(faces)
                fn = face_normals(verts[faces])
                if adj.size:
                    cosang = (fn[adj[:, 0]] * fn[adj[:, 1]]).sum(-1)
                    adj = adj[np.arccos(np.clip(cosang, -1.0, 1.0)) < math.radians(30.0)]
                group = _components(m, adj)
            else:
                group = np.arange(m)
        order = np.argsort(group, kind="stable")           # concatenation regroups faces by component
        colours = np.stack([rng.randint(0, hi, (1, 3))[0] for _ in range(int(group.max()) + 1)])
        faces, normals, diffuse = faces[order], normals[order], colours[group[order]] / 255.0
    else:
        q = (np.asarray(mat["diffuse"], dtype=np.float64) * 255.0).clip(0, 255).astype(np.int64)
        diffuse = np.tile(q / 255.0, (m, 1))
    return verts[faces], normals, diffuse


def load_scene(path: str) -> Dict[str, np.ndarray]:
    """Scene JSON -> {'triangles' [N,3,3], 'vn' [N,3,3], 'tex13' [N,13] (fp16-rounded like the HDF5 file),
    'c2w' [V,4,4], 'fov' [V]} float32.  Mesh paths are relative to the JSON file."""
    with open(path) as f:
        cfg = json.load(f)
    base = os.path.dirname(os.path.abspath(path))
    tris, vns, texs = [], [], []
    for obj in cfg["objects"].values():
        t, n, diffuse = _object_mesh(obj, base)
        mat = obj["material"]
        m = t.shape[0]
        tex = np.concatenate([
            diffuse,
            np.tile(np.asarray(mat["specular"], dtype=np.float64), (m, 1)),
            np.full((m, 1), float(mat["roughness"])),
            np.tile(np.array([0.5, 0.5, 1.0]), (m, 1)),
            np.tile(np.asarray(mat["emissive"], dtype=np.float64), (m, 1)),
        ], axis=1)
        tris.append(t), vns.append(n), texs.append(tex)
    cams = cfg["cameras"]
    return {
        "triangles": np.concatenate(tris).astype(np.float32),
        "vn": np.concatenate(vns).astype(np.float32),
        "tex13": np.concatenate(texs).astype(np.float16).astype(np.float32),
        "c2w": np.stack([look_at_c2w(c["position"], c["look_at"], c["up"]) for c in cams]).astype(np.float32),
        "fov": np.asarray([c["fov"] for c in cams], dtype=np.float32),
    }


def expand_texture(tex13: np.ndarray, size: int = TEXELS) -> np.ndarray:
    """[N,13] per-triangle constants -> [N,13,size,size] texel grid, zero outside the triangular mask."""
    return (tex13[:, :, None, None] * texel_mask(size)[None, None]).astype(np.float32)


def constant_texture_of(texture: np.ndarray, atol: float = 0.0) -> Optional[np.ndarray]:
    """[N,C,P,P] texel grid -> [N,C] per-triangle constants if the grid IS "constants times the triangular texel mask
    x + y <= P" (every scene written by scene_processor/to_h5.py:37-66), else None.  Lets a caller that holds the
    reference's 218 MB texel grid take the constant-texture fast path (SURVEY §8 f2) without being told so."""
    tex = np.asarray(texture)
    if tex.ndim != 4 or tex.shape[2] != tex.shape[3]:
        return None
    m = texel_mask(tex.shape[2])
    consts = tex[:, :, 0, 0]
    inside_ok = np.abs(tex[:, :, m] - consts[:, :, None]).max(initial=0.0) <= atol
    outside_ok = np.abs(tex[:, :, ~m]).max(initial=0.0) <= atol
    return np.ascontiguousarray(consts) if (inside_ok and outside_ok) else None


def to_pipeline_inputs(scene: Dict[str, np.ndarray], pad_to: Optional[int] = None, constant_texture: bool = False):
    """Batch-1 torch tensors with the pipeline's argument names.  `constant_texture=True` keeps the
    texture as [1,N,13] per-triangle constants (the pipeline's fast path: no 32x32 expansion, no
    218 MB upload); otherwise the full [1,N,13,32,32] grid the reference's HDF5 files hold."""
    import torch
    n = scene["triangles"].shape[0]
    total = max(n, pad_to or n)
    tri = np.zeros((total, 3, 3), np.float32)
    vn = np.zeros((total, 3, 3), np.float32)
    tex13 = np.zeros((total, 13), np.float32)
    mask = np.zeros((total,), bool)
    tri[:n], vn[:n], mask[:n] = scene["triangles"], scene["vn"], True
    if "tex13" in scene:
        tex13[:n] = scene["tex13"]
        tex = tex13 if constant_texture else expand_texture(tex13)
    else:  # a stored texel grid (load_h5): arbitrary textures, no constant-texture shortcut
        if constant_texture:
            consts = constant_texture_of(scene["texture"])
            if consts is None:
                raise ValueError("constant_texture: this scene's texel grid is not 'constants times the triangular mask'")
            tex13[:n] = consts
            tex = tex13
        else:
            tex = np.zeros((total,) + tuple(scene["texture"].shape[1:]), np.float32)
            tex[:n] = scene["texture"]
    return {
        "triangles": torch.from_numpy(tri)[None], "texture": torch.from_numpy(tex)[None],
        "mask": torch.from_numpy(mask)[None], "vn": torch.from_numpy(vn)[None],
        "c2w": torch.from_numpy(scene["c2w"])[None], "fov": torch.from_numpy(scene["fov"])[None, :, None],
    }


def save_npz(scene: Dict[str, np.ndarray], path: str) -> None:
    np.savez_compressed(path, **scene)


def load_npz(path: str) -> Dict[str, np.ndarray]:
    with np.load(path) as z:
        return {k: z[k] for k in z.files}


def load_h5(path: str) -> Dict[str, np.ndarray]:
    """A scene file written by the reference's converter (scene_processor/to_h5.py:68-92; what
    batch_infer.py:27-35 / infer.py:66-73 read): 'triangles' [N,3,3], 'texture' [N,13,32,32] (fp16 in the file),
    'vn' [N,3,3], 'c2w' [V,4,4], 'fov' [V].  Needs the optional h5py package (not in this image: the numpy-only
    route is tools/convert_scene.py -> .npz); the texel grid is kept as stored, so `to_pipeline_inputs` passes
    it through instead of expanding per-triangle constants."""
    try:
        import h5py
    except ImportError as e:
        raise ImportError(f"{path}: reading HDF5 scenes needs h5py; convert the scene JSON with "
                          "tools/convert_scene.py (numpy only) instead") from e
    with h5py.File(path, "r") as f:
        return {"triangles": np.array(f["triangles"]).astype(np.float32), "texture": np.array(f["texture"]).astype(np.float32),
                "vn": np.array(f["vn"]).astype(np.float32), "c2w": np.array(f["c2w"]).astype(np.float32),
                "fov": np.array(f["fov"]).astype(np.float32).reshape(-1)}


def load_scene_file(path: str) -> Dict[str, np.ndarray]:
    """.npz (tools/convert_scene.py), .h5 / .hdf5 (the reference's converter) or .json (scene description)."""
    ext = os.path.splitext(path)[1].lower()
    if ext == ".npz":
        return load_npz(path)
    if ext in (".h5", ".hdf5"):
        return load_h5(path)
    if ext == ".json":
        return load_scene(path)
    raise ValueError(f"{path}: unknown scene file type")


# ------------------------------------------------------------------------------------------- COLMAP cameras
# COLMAP camera model -> (lens, intrinsics from the parameters, distortion from the parameters).  The fisheye models
# share one theta polynomial: SIMPLE_RADIAL_FISHEYE and RADIAL_FISHEYE are OPENCV_FISHEYE with k2.. or k3.. zero.
_COLMAP_MODELS = {
    "SIMPLE_PINHOLE": ("opencv", lambda p: (p[0], p[0], p[1], p[2]), None),
    "PINHOLE": ("opencv", lambda p: p[:4], None),
    "SIMPLE_RADIAL": ("opencv", lambda p: (p[0], p[0], p[1], p[2]), lambda p: (p[3], 0, 0, 0, 0, 0, 0, 0)),
    "RADIAL": ("opencv", lambda p: (p[0], p[0], p[1], p[2]), lambda p: (p[3], p[4], 0, 0, 0, 0, 0, 0)),
    "OPENCV": ("opencv", lambda p: p[:4], lambda p: (*p[4:8], 0, 0, 0, 0)),
    "FULL_OPENCV": ("opencv", lambda p: p[:4], lambda p: p[4:12]),
    "SIMPLE_RADIAL_FISHEYE": ("fisheye", lambda p: (p[0], p[0], p[1], p[2]), lambda p: (p[3], 0, 0, 0)),
    "RADIAL_FISHEYE": ("fisheye", lambda p: (p[0], p[0], p[1], p[2]), lambda p: (p[3], p[4], 0, 0)),
    "OPENCV_FISHEYE": ("fisheye", lambda p: p[:4], lambda p: p[4:8]),
}
_COLMAP_NPARAMS = {"SIMPLE_PINHOLE": 3, "PINHOLE": 4, "SIMPLE_RADIAL": 4, "RADIAL": 5, "OPENCV": 8, "FULL_OPENCV": 12,
                   "SIMPLE_RADIAL_FISHEYE": 4, "RADIAL_FISHEYE": 5, "OPENCV_FISHEYE": 8}


def _colmap_lines(path: str) -> List[str]:
    with open(path) as f:
        return [line.rstrip("\n") for line in f]


def _quat_to_rot(q) -> np.ndarray:
    """Rotation matrix [3,3] of a quaternion (w, x, y, z) (normalised first), COLMAP's convention."""
    w, x, y, z = np.asarray(q, dtype=np.float64) / np.linalg.norm(q)
    return np.array([[1 - 2 * (y * y + z * z), 2 * (x * y - w * z), 2 * (x * z + w * y)],
                     [2 * (x * y + w * z), 1 - 2 * (x * x + z * z), 2 * (y * z - w * x)],
                     [2 * (x * z - w * y), 2 * (y * z + w * x), 1 - 2 * (x * x + y * y)]])


def read_colmap_cameras(sparse_dir: str) -> List[dict]:
    """The cameras of a COLMAP reconstruction in the TEXT model format (`cameras.txt` and `images.txt` in
    `sparse_dir`; `colmap model_converter --output_type TXT` writes them from the binary format).

    Returns one record per image, in the order of images.txt: 'name', 'resolution' (height, width), 'intrinsics'
    float64 [4] = (fx, fy, cx, cy), 'distortion' float64 [8] (lens 'opencv': k1, k2, p1, p2, k3, k4, k5, k6) or [4]
    (lens 'fisheye': k1, k2, k3, k4) or None (the pinhole models), 'lens' ('opencv' for the pinhole models) and
    'c2w' float64 [4,4] in this project's camera axes (x right, y up, looking down -z): inv([R(q) | t]) @
    diag(1, -1, -1, 1) of COLMAP's world-to-camera pose.  These are `render`'s camera arguments as they are: COLMAP's
    pixel centres are at j + 0.5 and its principal point is in pixels of the image, as `intrinsics` expects.
    Models: SIMPLE_PINHOLE, PINHOLE (no distortion); SIMPLE_RADIAL, RADIAL, OPENCV, FULL_OPENCV (opencv);
    SIMPLE_RADIAL_FISHEYE, RADIAL_FISHEYE, OPENCV_FISHEYE (fisheye).  Any other (FOV, the thin-prism models, ...)
    raises NotImplementedError naming it."""
    cams = {}
    for line in _colmap_lines(os.path.join(sparse_dir, "cameras.txt")):
        el = line.split()
        if not el or el[0].startswith("#"):
            continue
        cam_id, model, width, height = int(el[0]), el[1], int(el[2]), int(el[3])
        if model not in _COLMAP_MODELS:
            raise NotImplementedError(f"COLMAP camera model {model} (camera {cam_id}) is not supported; supported: "
                                      f"{', '.join(_COLMAP_MODELS)}")
        p = [float(v) for v in el[4:]]
        if len(p) != _COLMAP_NPARAMS[model]:
            raise ValueError(f"COLMAP camera {cam_id}: model {model} has {_COLMAP_NPARAMS[model]} parameters, "
                             f"got {len(p)}")
        lens, intr, dist = _COLMAP_MODELS[model]
        cams[cam_id] = dict(resolution=(height, width), intrinsics=np.array(intr(p), dtype=np.float64),
                            distortion=None if dist is None else np.array(dist(p), dtype=np.float64), lens=lens)
    out = []
    lines = iter(_colmap_lines(os.path.join(sparse_dir, "images.txt")))
    flip = np.diag([1.0, -1.0, -1.0, 1.0])  # COLMAP's camera axes (x right, y down, z forward) -> this project's
    for line in lines:
        el = line.split()
        if not el or el[0].startswith("#"):
            continue
        next(lines, None)  # the image's POINTS2D line (possibly empty)
        q, t = [float(v) for v in el[1:5]], np.array([float(v) for v in el[5:8]])
        cam_id, name = int(el[8]), " ".join(el[9:])
        if cam_id not in cams:
            raise ValueError(f"COLMAP image {name}: camera {cam_id} is not in cameras.txt")
        R = _quat_to_rot(q)
        c2w = np.eye(4)
        c2w[:3, :3], c2w[:3, 3] = R.T, -R.T @ t
        out.append(dict(name=name, c2w=c2w @ flip, **{k: (v.copy() if isinstance(v, np.ndarray) else v)
                                                      for k, v in cams[cam_id].items()}))
    return out
