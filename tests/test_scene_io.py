"""CPU: numpy-only scene ingestion (renderformer_b200/scene_io.py) -- OBJ parsing, transforms, flat and
crease-split smooth normals, look-at cameras, the 13-channel constant texture layout, and the
converted examples/cbox.json fixture (5633 triangles, SURVEY §8d)."""
import json
import math
import os

import numpy as np
import pytest

from oracle.reference_loader import find_reference
from renderformer_b200 import scene_io as sio

REF = find_reference() or ""  # a source tree of the unmodified reference, when one is at hand (RFB_REFERENCE)

CUBE = """# unit cube, quads
v -1 -1 -1
v  1 -1 -1
v  1  1 -1
v -1  1 -1
v -1 -1  1
v  1 -1  1
v  1  1  1
v -1  1  1
f 1 4 3 2
f 5 6 7 8
f 1/1/1 2/2/2 6/3/3 5/4/4
f 2 3 7 6
f 3 4 8 7
f -5 -8 -4 -1
"""


def _write_scene(tmp_path, smooth, seed=None, normalize=False, rotation=(0, 0, 0), mesh=CUBE):
    (tmp_path / "m.obj").write_text(mesh)
    cfg = {"scene_name": "t", "version": "1.0", "objects": {"a": {
        "mesh_path": "m.obj",
        "transform": {"translation": [0.1, 0.2, 0.3], "rotation": list(rotation), "scale": [0.5, 0.5, 0.25],
                      "normalize": normalize},
        "material": {"diffuse": [0.4, 0.8, 1.0], "specular": [0.01, 0.01, 0.01], "roughness": 0.99,
                     "emissive": [0.0, 0.0, 5000.0], "smooth_shading": smooth, "rand_tri_diffuse_seed": seed,
                     "random_diffuse_max": 0.4}}},
        "cameras": [{"position": [0.0, -2.0, 0.0], "look_at": [0.0, 0.0, 0.0], "up": [0.0, 0.0, 1.0], "fov": 37.5},
                    {"position": [1.0, -1.0, 0.86], "look_at": [0.0, 0.0, -0.25], "up": [0.0, 0.0, 1.0], "fov": 30.0}]}
    p = tmp_path / "scene.json"
    p.write_text(json.dumps(cfg))
    return str(p)


def test_obj_quads_slash_and_negative_indices(tmp_path):
    (tmp_path / "c.obj").write_text(CUBE)
    v, f = sio.load_obj(str(tmp_path / "c.obj"))
    assert v.shape == (8, 3) and f.shape == (12, 3)
    assert f.min() == 0 and f.max() == 7
    # every quad became two triangles with outward orientation: the cube's volume is 8
    tri = v[f]
    vol = np.einsum("ij,ij->i", tri[:, 0], np.cross(tri[:, 1], tri[:, 2])).sum() / 6.0
    assert abs(abs(vol) - 8.0) < 1e-9


def test_transform_order_and_flat_normals(tmp_path):
    s = sio.load_scene(_write_scene(tmp_path, smooth=False, rotation=(90, 0, 0)))
    tri = s["triangles"].reshape(-1, 3)
    # rotate 90 deg about x: (x, y, z) -> (x, -z, y); then scale (0.5, 0.5, 0.25); then translate
    lo, hi = tri.min(0), tri.max(0)
    np.testing.assert_allclose(lo, [0.1 - 0.5, 0.2 - 0.5, 0.3 - 0.25], atol=1e-6)
    np.testing.assert_allclose(hi, [0.1 + 0.5, 0.2 + 0.5, 0.3 + 0.25], atol=1e-6)
    fn = sio.face_normals(s["triangles"].astype(np.float64))
    np.testing.assert_allclose(s["vn"], np.repeat(fn[:, None], 3, axis=1), atol=1e-6)
    np.testing.assert_allclose(np.linalg.norm(s["vn"], axis=-1), 1.0, atol=1e-6)


def test_smooth_shading_keeps_cube_edges_hard_but_smooths_a_sphere(tmp_path):
    cube = sio.load_scene(_write_scene(tmp_path, smooth=True))
    fn = sio.face_normals(cube["triangles"].astype(np.float64))
    np.testing.assert_allclose(cube["vn"], np.repeat(fn[:, None], 3, axis=1), atol=1e-6)  # 90 deg creases > 30 deg
    # icosphere-like mesh: subdivided octahedron projected on the unit sphere -> normals ~ positions
    v = [(1, 0, 0), (-1, 0, 0), (0, 1, 0), (0, -1, 0), (0, 0, 1), (0, 0, -1)]
    f = [(0, 2, 4), (2, 1, 4), (1, 3, 4), (3, 0, 4), (2, 0, 5), (1, 2, 5), (3, 1, 5), (0, 3, 5)]
    v = [np.array(p, float) for p in v]
    for _ in range(3):
        nf, cache = [], {}

        def mid(a, b):
            k = (min(a, b), max(a, b))
            if k not in cache:
                m = v[a] + v[b]
                v.append(m / np.linalg.norm(m))
                cache[k] = len(v) - 1
            return cache[k]
        for a, b, c in f:
            ab, bc, ca = mid(a, b), mid(b, c), mid(c, a)
            nf += [(a, ab, ca), (ab, b, bc), (ca, bc, c), (ab, bc, ca)]
        f = nf
    obj = "".join(f"v {p[0]} {p[1]} {p[2]}\n" for p in v) + "".join(f"f {a + 1} {b + 1} {c + 1}\n" for a, b, c in f)
    (tmp_path / "s").mkdir()
    path = _write_scene(tmp_path / "s", smooth=True, mesh=obj)
    cfg = json.load(open(path))
    cfg["objects"]["a"]["transform"].update(scale=[1, 1, 1], translation=[0, 0, 0])
    open(path, "w").write(json.dumps(cfg))
    sph = sio.load_scene(path)
    np.testing.assert_allclose(sph["vn"], sph["triangles"], atol=2e-2)  # unit sphere: normal = position


def test_texture_layout_quantisation_and_cameras(tmp_path):
    s = sio.load_scene(_write_scene(tmp_path, smooth=False))
    t = s["tex13"][0]
    np.testing.assert_allclose(t[:3], np.float16([102 / 255, 204 / 255, 1.0]).astype(np.float32))  # 8-bit, then fp16
    np.testing.assert_allclose(t[3:7], np.float16([0.01, 0.01, 0.01, 0.99]).astype(np.float32))
    np.testing.assert_allclose(t[7:], [0.5, 0.5, 1.0, 0.0, 0.0, 5000.0])
    tex = sio.expand_texture(s["tex13"])
    assert tex.shape == (12, 13, 32, 32)
    m = sio.texel_mask()
    assert m.sum() == 559 and m[0, 31] and m[1, 31] and not m[2, 31]
    assert (tex[:, :, ~m] == 0).all() and (tex[0, 0][m] == t[0]).all()
    c2w = s["c2w"]
    np.testing.assert_allclose(c2w[0], [[1, 0, 0, 0], [0, 0, -1, -2], [0, 1, 0, 0], [0, 0, 0, 1]], atol=1e-6)
    R = c2w[1][:3, :3]
    np.testing.assert_allclose(R @ R.T, np.eye(3), atol=1e-6)
    back = np.array([1.0, -1.0, 0.86]) - np.array([0.0, 0.0, -0.25])
    np.testing.assert_allclose(R[:, 2], back / np.linalg.norm(back), atol=1e-6)  # camera looks along -z
    assert R[2, 1] > 0  # +y is up
    np.testing.assert_allclose(s["fov"], [37.5, 30.0])


def test_random_diffuse_is_seeded_per_component(tmp_path):
    a = sio.load_scene(_write_scene(tmp_path, smooth=True, seed=3))
    b = sio.load_scene(_write_scene(tmp_path, smooth=True, seed=3))
    c = sio.load_scene(_write_scene(tmp_path, smooth=True, seed=4))
    np.testing.assert_array_equal(a["tex13"], b["tex13"])
    assert not np.array_equal(a["tex13"], c["tex13"])
    cols = np.unique(a["tex13"][:, :3], axis=0)
    assert 2 <= cols.shape[0] <= 6 and cols.max() <= 0.4 + 1e-3  # one colour per cube side, capped by random_diffuse_max


def test_pipeline_inputs_and_padding(tmp_path):
    s = sio.load_scene(_write_scene(tmp_path, smooth=False))
    full = sio.to_pipeline_inputs(s, pad_to=16)
    assert full["triangles"].shape == (1, 16, 3, 3) and full["texture"].shape == (1, 16, 13, 32, 32)
    assert full["mask"].sum() == 12 and full["fov"].shape == (1, 2, 1) and full["c2w"].shape == (1, 2, 4, 4)
    const = sio.to_pipeline_inputs(s, constant_texture=True)
    assert const["texture"].shape == (1, 12, 13)


def test_cbox_fixture(golden_dir):
    """tests/golden/cbox_scene.npz = tools/convert_scene.py on the reference's examples/cbox.json."""
    s = sio.load_npz(os.path.join(golden_dir, "cbox_scene.npz"))
    assert s["triangles"].shape == (5633, 3, 3) and s["vn"].shape == (5633, 3, 3) and s["tex13"].shape == (5633, 13)
    np.testing.assert_allclose(np.linalg.norm(s["vn"], axis=-1), 1.0, atol=1e-5)
    assert (s["tex13"][:, 10:].max(axis=1) > 0).sum() == 1  # one emissive triangle (templates/lighting/tri.obj)
    room = s["triangles"][:-1].reshape(-1, 3)
    assert np.abs(room).max() <= 0.5 + 1e-6  # the box itself spans [-0.5, 0.5]^3
    np.testing.assert_allclose(s["fov"], [37.5])
    if os.path.exists(os.path.join(REF, "examples", "cbox.json")):  # regenerate and compare where the source exists
        again = sio.load_scene(os.path.join(REF, "examples", "cbox.json"))
        for k in s:
            np.testing.assert_array_equal(again[k], s[k])


def test_scene_file_loader_dispatch(tmp_path, monkeypatch):
    """.npz / .json go through the numpy-only route; .h5 (the reference converter's files, to_h5.py:68-92) needs
    h5py and says so; with an h5py present the stored texel grid is passed through unexpanded."""
    import sys
    import types
    sc = {"triangles": np.random.rand(5, 3, 3).astype(np.float32), "vn": np.random.rand(5, 3, 3).astype(np.float32),
          "tex13": np.random.rand(5, 13).astype(np.float32), "c2w": np.eye(4, dtype=np.float32)[None], "fov": np.array([37.5], np.float32)}
    p = str(tmp_path / "s.npz")
    sio.save_npz(sc, p)
    back = sio.load_scene_file(p)
    assert all(np.array_equal(back[k], sc[k]) for k in sc)
    with pytest.raises(ValueError):
        sio.load_scene_file(str(tmp_path / "s.txt"))
    monkeypatch.setitem(sys.modules, "h5py", None)  # import h5py -> ImportError
    with pytest.raises(ImportError, match="convert_scene"):
        sio.load_scene_file(str(tmp_path / "s.h5"))
    grid = sio.expand_texture(sc["tex13"]).astype(np.float16)
    stored = {"triangles": sc["triangles"], "texture": grid, "vn": sc["vn"], "c2w": sc["c2w"], "fov": sc["fov"]}

    class File(dict):
        def __init__(self, path, mode="r"):
            super().__init__(stored)

        def __enter__(self):
            return self

        def __exit__(self, *a):
            return False
    h5 = types.ModuleType("h5py")
    h5.File = File
    monkeypatch.setitem(sys.modules, "h5py", h5)
    got = sio.load_scene_file(str(tmp_path / "s.h5"))
    assert got["texture"].dtype == np.float32 and got["fov"].shape == (1,)
    inp = sio.to_pipeline_inputs(got, pad_to=8)
    assert tuple(inp["texture"].shape) == (1, 8, 13, 32, 32) and inp["mask"][0].tolist() == [True] * 5 + [False] * 3
    assert np.array_equal(inp["texture"][0, :5].numpy(), grid.astype(np.float32)) and not inp["texture"][0, 5:].any()
    # the stored grid IS constants x mask: the fast path is detected, fp16 rounding of the file included
    fast = sio.to_pipeline_inputs(got, constant_texture=True)
    assert tuple(fast["texture"].shape) == (1, 5, 13)
    assert np.array_equal(fast["texture"][0].numpy(), sc["tex13"].astype(np.float16).astype(np.float32))
    assert np.array_equal(sio.constant_texture_of(got["texture"]), fast["texture"][0].numpy())
    painted = dict(got, texture=got["texture"].copy())
    painted["texture"][2, 0, 3, 4] += 0.25  # an arbitrary (non-constant) texture keeps the full path
    assert sio.constant_texture_of(painted["texture"]) is None
    with pytest.raises(ValueError, match="constant_texture"):
        sio.to_pipeline_inputs(painted, constant_texture=True)
    leaky = dict(got, texture=got["texture"].copy())
    leaky["texture"][1, 5, 31, 31] = 0.5    # a texel outside the triangular mask
    assert sio.constant_texture_of(leaky["texture"]) is None


EXAMPLE_TRIANGLES = {  # triangle counts of the reference's example scenes as converted here (cbox: SURVEY §8d, 5633)
    "cbox": 5633, "cbox-bunny": 6209, "cbox-lucy": 11803, "cbox-teapot": 9397, "compose-scene": 7321,
    "constant-width": 4527, "cornell_box": 3073, "crystals": 1949, "fox-in-the-wild": 1418, "horse-and-heart": 5023,
    "init-template": 513, "renderformer-logo": 6386, "room": 7141, "shader-ball": 11036, "tree": 4400, "veach-mis": 4575,
}


@pytest.mark.skipif(not os.path.isdir(os.path.join(REF, "examples")), reason="no reference source tree with examples/ (set RFB_REFERENCE)")
@pytest.mark.parametrize("name", sorted(EXAMPLE_TRIANGLES))
def test_every_reference_example_scene_converts(name):
    """All 16 scene descriptions the reference ships (examples/*.json: templates, nested transforms, smooth and flat
    shading, random diffuse, multiple materials) go through the numpy-only converter: finite geometry, unit normals,
    textures inside their documented ranges, one look-at camera each."""
    sc = sio.load_scene(os.path.join(REF, "examples", f"{name}.json"))
    n = sc["triangles"].shape[0]
    assert n == EXAMPLE_TRIANGLES[name] and n <= 12288
    assert sc["vn"].shape == (n, 3, 3) and sc["tex13"].shape == (n, 13)
    assert np.isfinite(sc["triangles"]).all() and np.abs(sc["triangles"]).max() < 10.0
    assert np.allclose(np.linalg.norm(sc["vn"], axis=-1), 1.0, atol=1e-4)
    tex = sc["tex13"]
    assert (tex[:, :7] >= 0).all() and (tex[:, :7] <= 1.0).all()          # diffuse, specular, roughness
    assert np.allclose(tex[:, 7:10], [0.5, 0.5, 1.0], atol=1e-3) and (tex[:, 10:] >= 0).all()
    assert (tex[:, 10:].sum(axis=1) > 0).any()                              # every example has a light
    assert sc["c2w"].shape[1:] == (4, 4) and sc["c2w"].shape[0] == sc["fov"].shape[0] >= 1
    R = sc["c2w"][:, :3, :3]
    assert np.allclose(R @ np.transpose(R, (0, 2, 1)), np.eye(3), atol=1e-5)  # camera frames are rotations
    inp = sio.to_pipeline_inputs(sc, constant_texture=True)
    assert tuple(inp["texture"].shape) == (1, n, 13) and bool(inp["mask"].all())
