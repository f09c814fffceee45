"""CPU, build container only: the to_h5 half of the scene converter pinned to the reference's OWN code.

The reference converts a scene in two steps: scene_processor/scene_mesh.py (trimesh: OBJ parsing, transforms, smooth
shading, random colours -> one OBJ per object) and scene_processor/to_h5.py:37-92 (numpy: the 13-channel constant
texture with its triangular texel mask, fp16 storage, look-at cameras, concatenation of the objects).  trimesh is not
installed here, so the first half stays unpinned -- but the second half runs UNMODIFIED in a subprocess: its
`trimesh.load` is a stand-in that hands it the per-object meshes of OUR first half, its `h5py.File` a stand-in that
records the datasets it writes.  What the reference writes must equal what `renderformer_b200.scene_io` produces for
the same scene, dataset by dataset, bit for bit."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

from oracle.reference_loader import find_reference

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
REF = find_reference() or ""  # a source tree of the unmodified reference (RFB_REFERENCE), with examples/

WORKER = r"""
import json, os, sys, types
import numpy as np
scene_json, mesh_npz, out_npz = sys.argv[1:4]
meshes = np.load(mesh_npz)

class _Visual:
    def __init__(self, fc): self.face_colors = fc
class _Mesh:
    def __init__(self, key):
        self.triangles = meshes[key + ".tri"]
        m = self.triangles.shape[0]
        self.faces = np.arange(3 * m).reshape(m, 3)
        self.vertex_normals = meshes[key + ".vn"].reshape(-1, 3)
        self.visual = _Visual(meshes[key + ".rgba"])
def _load(path, process=False, force=None, **kw):
    return _Mesh(os.path.splitext(os.path.basename(path))[0])
trimesh = types.ModuleType("trimesh"); trimesh.load = _load; trimesh.Trimesh = object
trimesh.visual = types.ModuleType("trimesh.visual")
captured = {}
class _File:
    def __init__(self, path, mode="r"): pass
    def __enter__(self): return self
    def __exit__(self, *a): return False
    def create_dataset(self, name, data=None, **kw): captured[name] = np.asarray(data)
h5py = types.ModuleType("h5py"); h5py.File = _File
for name, mod in (("trimesh", trimesh), ("trimesh.visual", trimesh.visual), ("h5py", h5py), ("pymeshlab", types.ModuleType("pymeshlab"))):
    sys.modules[name] = mod
sys.path.insert(0, %(ref)r)
from scene_processor.scene_config import SceneConfig, ObjectConfig, MaterialConfig, TransformConfig, CameraConfig  # the reference's
from scene_processor.to_h5 import save_to_h5                                                                  # the reference's
cfg = json.load(open(scene_json))
objects = {k: ObjectConfig(mesh_path=o["mesh_path"], material=MaterialConfig(**o["material"]), transform=TransformConfig(**o["transform"]),
                           **{f: o[f] for f in ("remesh", "remesh_target_face_num") if f in o}) for k, o in cfg["objects"].items()}
sc = SceneConfig(scene_name=cfg["scene_name"], version=cfg["version"], objects=objects, cameras=[CameraConfig(**c) for c in cfg["cameras"]])
save_to_h5(sc, os.path.join(os.path.dirname(out_npz), "mesh.obj"), os.path.join(os.path.dirname(out_npz), "scene.h5"))
np.savez(out_npz, **captured)
"""


@pytest.mark.skipif(not os.path.isdir(os.path.join(REF, "scene_processor")), reason="no reference source tree with scene_processor/ (set RFB_REFERENCE)")
@pytest.mark.parametrize("scene", ["cbox", "room", "crystals"])
def test_to_h5_half_of_the_converter_equals_the_reference(scene, tmp_path):
    from renderformer_b200 import scene_io as sio
    path = os.path.join(REF, "examples", f"{scene}.json")
    with open(path) as f:
        cfg = json.load(f)
    base = os.path.dirname(path)
    meshes = {}
    for key, obj in cfg["objects"].items():  # OUR first half, object by object
        tri, vn, diffuse = sio._object_mesh(obj, base)
        rgba = np.concatenate([np.rint(diffuse * 255.0), np.full((tri.shape[0], 1), 255.0)], axis=1).astype(np.uint8)
        meshes[key + ".tri"], meshes[key + ".vn"], meshes[key + ".rgba"] = tri, vn, rgba
    mesh_npz, out_npz = str(tmp_path / "meshes.npz"), str(tmp_path / "ref.npz")
    np.savez(mesh_npz, **meshes)
    r = subprocess.run([sys.executable, "-c", WORKER % {"ref": REF}, path, mesh_npz, out_npz], capture_output=True, text=True,
                       timeout=600, cwd=str(tmp_path))
    assert r.returncode == 0, r.stderr[-3000:]
    ref = np.load(out_npz)

    ours = sio.load_scene(path)
    assert ref["triangles"].dtype == np.float32 and np.array_equal(ref["triangles"], ours["triangles"])
    assert np.array_equal(ref["vn"], ours["vn"])
    assert ref["texture"].dtype == np.float16 and ref["texture"].shape == (ours["triangles"].shape[0], 13, 32, 32)
    assert np.array_equal(ref["texture"].astype(np.float32), sio.expand_texture(ours["tex13"]))   # fp16 storage included
    assert np.array_equal(ref["c2w"], ours["c2w"]) or np.abs(ref["c2w"] - ours["c2w"]).max() <= 1e-6  # inverse vs closed form
    assert np.array_equal(ref["fov"], ours["fov"])
    # and the reference's own texel grid IS "constants x mask": the fast path's detector agrees
    assert np.array_equal(sio.constant_texture_of(ref["texture"].astype(np.float32)), ours["tex13"])


NORM_WORKER = r"""
import sys, types
import numpy as np
for name in ("trimesh", "trimesh.visual", "h5py", "pymeshlab"):
    sys.modules[name] = types.ModuleType(name)
sys.modules["trimesh"].visual = sys.modules["trimesh.visual"]
sys.modules["trimesh"].Trimesh = object
sys.path.insert(0, %(ref)r)
from scene_processor.scene_mesh import normalize_to_unit_sphere   # the reference's (scene_mesh.py:12-18), pure numpy
mesh = types.SimpleNamespace(vertices=np.load(sys.argv[1]))
np.save(sys.argv[2], normalize_to_unit_sphere(mesh).vertices)
"""


@pytest.mark.skipif(not os.path.isdir(os.path.join(REF, "scene_processor")), reason="no reference source tree with scene_processor/ (set RFB_REFERENCE)")
def test_normalisation_equals_the_reference(tmp_path):
    """scene_mesh.py:12-18 run live on the vertices of a shipped OBJ: centre on the vertex mean, scale so that the
    farthest vertex sits at radius 0.5."""
    from renderformer_b200 import scene_io as sio
    obj_path = os.path.join(REF, "examples", "objects", "cbox", "tall-box.obj")
    verts, faces = sio.load_obj(obj_path)
    np.save(str(tmp_path / "v.npy"), verts)
    r = subprocess.run([sys.executable, "-c", NORM_WORKER % {"ref": REF}, str(tmp_path / "v.npy"), str(tmp_path / "n.npy")],
                       capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stderr[-2000:]
    ref_tris = np.load(str(tmp_path / "n.npy"))[faces]
    obj = {"mesh_path": obj_path, "transform": {"translation": [0, 0, 0], "rotation": [0, 0, 0], "scale": [1, 1, 1], "normalize": True},
           "material": {"diffuse": [0.5, 0.5, 0.5], "specular": [0, 0, 0], "roughness": 0.5, "emissive": [0, 0, 0], "smooth_shading": False}}
    tris, _, _ = sio._object_mesh(obj, "/")
    assert np.array_equal(tris, ref_tris)
    assert abs(np.linalg.norm(tris.reshape(-1, 3), axis=-1).max() - 0.5) < 1e-12


DATASET_WORKER = r"""
import sys, types
import numpy as np
class _H5:
    def __init__(self, path, mode="r"): self.d = np.load(path)
    def __enter__(self): return self.d
    def __exit__(self, *a): self.d.close()
h5py = types.ModuleType("h5py"); h5py.File = _H5
imageio = types.ModuleType("imageio")
natsort = types.ModuleType("natsort"); natsort.natsorted = sorted
ocio = types.ModuleType("simple_ocio"); ocio.ToneMapper = object
roma = types.ModuleType("roma")  # renderformer/utils/transform.py:3 imports it; nothing of it is called here
for name, mod in (("h5py", h5py), ("imageio", imageio), ("natsort", natsort), ("simple_ocio", ocio), ("roma", roma)):
    sys.modules[name] = mod
sys.path.insert(0, %(ref)r)
import batch_infer                                                   # the reference's CLI module, unmodified
ds = batch_infer.TriangleRenderH5Dataset(sys.argv[1], int(sys.argv[2]) if sys.argv[2] != "none" else None)
item = ds[0]
np.savez(sys.argv[3], **{k: v.numpy() for k, v in item.items() if hasattr(v, "numpy")})
"""


@pytest.mark.skipif(not os.path.isdir(os.path.join(REF, "scene_processor")), reason="no reference source tree with scene_processor/ (set RFB_REFERENCE)")
@pytest.mark.parametrize("pad", [None, 48])
def test_scene_loading_and_padding_equal_the_reference_dataset(tmp_path, pad):
    """batch_infer.py:17-58 (`TriangleRenderH5Dataset.__getitem__`, incl. `--padding_length`) run live on a scene file
    vs `scene_io.load_scene_file` + `to_pipeline_inputs(pad_to=...)`: the same tensors reach the pipeline."""
    import torch
    from renderformer_b200 import scene_io as sio
    from renderformer_b200.synth import make_scene
    sc = make_scene(37, 2, seed=12)
    folder = tmp_path / "scenes"
    folder.mkdir()
    stored = {"triangles": sc["triangles"][0].numpy(), "vn": sc["vn"][0].numpy(), "texture": sc["texture"][0].numpy().astype(np.float16),
              "c2w": sc["c2w"][0].numpy(), "fov": sc["fov"][0, :, 0].numpy()}
    with open(folder / "a.h5", "wb") as f:  # the stand-in h5py.File of the worker reads an .npz under the .h5 name
        np.savez(f, **stored)
    out = str(tmp_path / "item.npz")
    r = subprocess.run([sys.executable, "-c", DATASET_WORKER % {"ref": REF}, str(folder), "none" if pad is None else str(pad), out],
                       capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stderr[-3000:]
    ref = np.load(out)
    # ours: the same file through the loader (h5py stand-in = np.load) and the padding of to_pipeline_inputs
    ours = sio.to_pipeline_inputs({k: (v.astype(np.float32) if v.dtype != bool else v) for k, v in stored.items()}, pad_to=pad)
    for k in ("triangles", "texture", "vn", "c2w"):
        assert np.array_equal(ref[k], ours[k][0].numpy()), k
    assert np.array_equal(ref["mask"], ours["mask"][0].numpy())
    assert np.array_equal(ref["fov"], ours["fov"][0, :, 0].numpy())       # batch_infer.py:131 adds the trailing axis itself
    assert ours["triangles"].dtype == torch.float32 and ours["mask"].dtype == torch.bool
