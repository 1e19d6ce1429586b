"""rust/patch/: the Rust side of the drop-in as SOURCE (no Rust toolchain in the image, so nothing here is compiled):
`describe.patch` adds a `describe` hook to every Shape / ShapeFunction / Material / Texture of the reference crate,
`Scene::flat()`, `#[repr(C)]` on Vector3d and `pub mod gpu`; `src/world/flat.rs` and `src/renderer/gpu.rs` are the
two new files.  These tests keep that source complete and in step with the tested C++ host mirror: every kind tag
of the ABI is produced, every implementor has its hook, and the params[8] rows the hooks write equal the rows the
host mirror writes for the same JSON."""
import json
import os
import re
import shutil
import subprocess
import sys
import tempfile

import numpy as np
import pytest

import rs_pathtracing_b200 as rt
from rs_pathtracing_b200 import _ffi

from conftest import ROOT

PATCH = os.path.join(ROOT, "rust", "patch", "describe.patch")
FLAT_RS = os.path.join(ROOT, "rust", "patch", "src", "world", "flat.rs")
GPU_RS = os.path.join(ROOT, "rust", "patch", "src", "renderer", "gpu.rs")
SYS_RS = os.path.join(ROOT, "rust", "ray_tracing_b200-sys", "src", "lib.rs")


def _added():
    text = open(PATCH, "rb").read().decode()
    return "\n".join(l[1:].rstrip("\r") for l in text.split("\n") if l.startswith("+") and not l.startswith("+++"))


def test_every_kind_tag_of_the_abi_is_produced():
    sys_rs = open(SYS_RS).read()
    tags = re.findall(r"pub const (RT_(?:SHAPE|SURF|MAT|TEX)_[A-Z_]+):", sys_rs)
    assert len(tags) >= 4 + 6 + 5 + 5
    text = _added() + open(FLAT_RS).read()
    missing = [t for t in tags if t != "RT_SHAPE_PARAMS" and f"sys::{t}" not in text]
    assert not missing, missing


def test_every_implementor_has_its_describe_hook():
    patch = open(PATCH, "rb").read().decode().replace("\r", "")
    # hunks are anchored by line numbers, not names: count the hooks per file instead and name the traits
    per_file = {}
    cur = None
    for l in patch.split("\n"):
        if l.startswith("+++ "):
            cur = l[4:].strip()
        elif l.startswith("+") and "fn describe(" in l:
            per_file[cur] = per_file.get(cur, 0) + 1
    assert per_file == {
        "b/src/algebra/noise.rs": 1,                 # Perlin -> rt_perlin
        "b/src/world/material.rs": 1 + 5,            # trait Material + Lambertian, Metal, Dielectric, DiffuseLight, EmptyMaterial
        "b/src/world/shapes/mod.rs": 1 + 7,          # trait Shape + Rectangle, Cube, Sphere, Torus, Tooth, ShapeCollection, BvhNode
        "b/src/world/shapes/ray_marching.rs": 1 + 1 + 6,   # RayMarchingShape, trait ShapeFunction + the six surfaces
        "b/src/world/texture.rs": 1 + 5,             # trait Texture + SolidColor, CheckerTexture, NoiseTexture, UVChecker, ImageTexture
    }, per_file
    added = _added()
    assert "#[repr(C)]" in added and "pub mod gpu;" in added and "pub mod flat;" in added
    assert "pub fn flat(&self) -> &flat::FlatScene" in added
    assert "FlatScene::from_shapes(&shapes)" in added          # flattened BEFORE BvhNode::new takes the list
    gpu = open(GPU_RS).read()
    for sym in ("rt_scene_create_multi", "rt_render_start", "rt_render_poll", "rt_render_stop", "rt_scene_destroy",
                "rt_render_set_accumulate", "impl Renderer for GpuRenderer"):
        assert sym in gpu, sym
    flat = open(FLAT_RS).read()
    for sym in ("pub fn push_shape", "pub fn material_index", "pub fn push_texture", "pub fn desc", "Arc::as_ptr"):
        assert sym in flat, sym


KIND = {"RT_SURF_HEART": 0, "RT_SURF_SINE": 1, "RT_SURF_STAR": 2, "RT_SURF_DUPIN": 3, "RT_SURF_HUNTS": 4, "RT_SURF_CUSHION": 5}
IDENT = {"translate": [1, 2, 3], "rotate": [10, 20, 30], "scale": [1, 2, 3]}


def _host_rows(shapes, materials):
    sc = rt.Scene.from_json(json.dumps({"camera": {"position": [0, 0, -10], "direction": [0, 0, 1], "up": [0, 1, 0],
                                                   "fov": 40.0, "focal_length": 1.0}, "background": [0, 0, 0],
                                        "materials": materials, "shapes": shapes}), add_random_spheres=False)
    d = sc.desc()
    n = d.n_shapes
    return (np.ctypeslib.as_array(d.kind, shape=(n,)).copy(), np.ctypeslib.as_array(d.flags, shape=(n,)).copy(),
            np.ctypeslib.as_array(d.params, shape=(n, 8)).copy(), sc, d)


def test_params_rows_equal_the_host_mirrors():
    """evaluate the patch's Rust array expressions for concrete field values and compare with the rows the (tested) C++
    host mirror writes for the equivalent JSON"""
    added = _added()
    surf = {"Heart": {"type": "Heart"}, "Sine": {"type": "Sine", "a": 0.7, "sphere_radius": 2.25},
            "Star": {"type": "Star", "a": 40.0, "sphere_radius": 1.75},
            "DupinCyclide": {"type": "DupinCyclide", "a": 1.11, "b": 0.99, "c": 0.5, "d": 0.1, "sphere_radius": 2.5},
            "HuntsSurface": {"type": "HuntsSurface", "sphere_radius": 4.5}, "Cushion": {"type": "Cushion", "sphere_radius": 1.5}}
    mats = {"M": {"type": "Lambertian", "albedo": {"type": "SolidColor", "color": [0.5, 0.5, 0.5]}}}
    shapes = [{"type": "BruteForsableShape", "shape": js, "step": 0.02, "depth": 3, "material": "M", "transform": IDENT}
              for js in surf.values()]
    shapes += [{"type": "Rectangle", "x0": -1.5, "y0": -0.5, "x1": 2.5, "y1": 3.5, "material": "M", "transform": IDENT},
               {"type": "Sphere", "name": "s", "material": "M", "transform": IDENT, "inverse_normal": True},
               {"type": "Cube", "name": "c", "material": "M", "transform": IDENT}]
    kind, flags, params, _, _ = _host_rows(shapes, mats)
    # the six surfaces: "(sys::RT_SURF_X, [..5 exprs..])" in the order of the impls
    exprs = re.findall(r"\(sys::(RT_SURF_[A-Z]+), \[(.*?)\]\)", added)
    assert [e[0] for e in exprs] == list(KIND)
    for row, (tag, body), js in zip(params[:6], exprs, surf.values()):
        vals = {"self." + k: repr(float(v)) for k, v in js.items() if k != "type"}
        if body.strip() == "0.0; 5":
            five = [0.0] * 5
        else:
            five = [float(eval(re.sub(r"self\.\w+", lambda m: vals[m.group(0)], x))) for x in body.split(",")]
        # RayMarchingShape::describe: [surface, step, depth, a, b, c, d, sphere_radius]
        assert "[surface as f64, self.step, self.depth as f64, abcd_r[0], abcd_r[1], abcd_r[2], abcd_r[3], abcd_r[4]]" in added
        want = [float(KIND[tag]), 0.02, 3.0] + five
        assert list(row) == want, (tag, list(row), want)
    assert kind[:6].tolist() == [_ffi.RT_SHAPE_MARCH] * 6
    # Rectangle / Sphere / Cube
    assert "[self.x0, self.y0, self.x1, self.y1, 0.0, 0.0, 0.0, 0.0]" in added
    assert list(params[6]) == [-1.5, -0.5, 2.5, 3.5, 0, 0, 0, 0] and kind[6] == _ffi.RT_SHAPE_RECTANGLE
    assert kind[7] == _ffi.RT_SHAPE_SPHERE and flags[7] == 1 and not params[7].any()
    assert "if self.inverse_normal { sys::RT_SHAPE_FLAG_INVERSE_NORMAL } else { 0 }" in added
    assert kind[8] == _ffi.RT_SHAPE_CUBE and flags[8] == 0 and not params[8].any()


def test_material_and_texture_rows_equal_the_host_mirrors():
    added = _added()
    mats = {
        "A": {"type": "Lambertian", "albedo": {"type": "CheckerTexture", "odd": {"type": "SolidColor", "color": [0.1, 0.2, 0.3]},
                                               "even": {"type": "SolidColor", "color": [0.4, 0.5, 0.6]}, "multipliers": [1.0, 2.0, 3.0]}},
        "B": {"type": "Metal", "albedo": {"type": "UVChecker", "odd": {"type": "SolidColor", "color": [0.1, 0.2, 0.3]},
                                          "even": {"type": "SolidColor", "color": [0.4, 0.5, 0.6]}, "multipliers": [7.0, 9.0]}, "fuzz": 0.25},
        "C": {"type": "Dielectric", "index_of_refraction": 1.4},
        "D": {"type": "DiffuseLight", "emit": {"type": "SolidColor", "color": [15, 15, 15]}},
        "E": {"type": "EmptyMaterial"},
    }
    shapes = [{"type": "Sphere", "name": k, "material": k, "transform": IDENT} for k in mats]
    _, _, _, sc, d = _host_rows(shapes, mats)
    mat_of = np.ctypeslib.as_array(d.material, shape=(d.n_shapes,))
    rows = [d.materials[int(i)] for i in mat_of]
    assert [r.kind for r in rows] == [_ffi.RT_MAT_LAMBERTIAN, _ffi.RT_MAT_METAL, _ffi.RT_MAT_DIELECTRIC,
                                      _ffi.RT_MAT_DIFFUSE_LIGHT, _ffi.RT_MAT_EMPTY]
    # scalar slot: Metal -> fuzz, Dielectric -> index_of_refraction (the patch says the same)
    assert rows[1].scalar == 0.25 and "kind: sys::RT_MAT_METAL, texture: self.albedo.describe(flat), scalar: self.fuzz" in added
    assert rows[2].scalar == 1.4 and "kind: sys::RT_MAT_DIELECTRIC, texture: 0, scalar: self.index_of_refraction" in added
    checker, uvc = d.textures[rows[0].texture], d.textures[rows[1].texture]
    assert checker.kind == _ffi.RT_TEX_CHECKER and checker.color.tuple() == (1.0, 2.0, 3.0)
    assert "sys::RT_TEX_CHECKER, [self.multipliers.x, self.multipliers.y, self.multipliers.z], odd, even, 0" in added
    assert uvc.kind == _ffi.RT_TEX_UV_CHECKER and uvc.color.tuple() == (7.0, 9.0, 0.0)
    assert "sys::RT_TEX_UV_CHECKER, [self.multipliers.0, self.multipliers.1, 0.0], odd, even, 0" in added
    for t in (checker, uvc):
        assert d.textures[t.odd].color.tuple() == (0.1, 0.2, 0.3) and d.textures[t.even].color.tuple() == (0.4, 0.5, 0.6)
    assert "sys::RT_TEX_NOISE, [self.scale, 0.0, 0.0], 0, 0, table" in added        # host: color.x = scale, image = table index
    assert "sys::RT_TEX_IMAGE, [0.0; 3], 0, 0, image" in added


# The reference crate is another project's source: it is not stored here, and the patch (one line of context) does not
# carry enough of it to rebuild the files.  A maintainer points RS_PATHTRACING_SRC at a checkout to run this test.
REFERENCE_SRC = os.environ.get("RS_PATHTRACING_SRC", "")


@pytest.mark.skipif(not os.path.isdir(os.path.join(REFERENCE_SRC, "src")),
                    reason="needs a checkout of the reference crate named by RS_PATHTRACING_SRC")
def test_patch_applies_to_the_reference_and_is_reproducible():
    tmp = tempfile.mkdtemp()
    try:
        shutil.copytree(os.path.join(REFERENCE_SRC, "src"), os.path.join(tmp, "src"))
        shutil.copy(os.path.join(REFERENCE_SRC, "Cargo.toml"), tmp)
        r = subprocess.run(["patch", "-p1", "--dry-run", "-i", PATCH], cwd=tmp, capture_output=True, text=True)
        assert r.returncode == 0, r.stdout + r.stderr
        regenerated = os.path.join(tmp, "describe.patch")
        subprocess.run([sys.executable, os.path.join(ROOT, "tools", "make_rust_patch.py"), regenerated], check=True,
                       capture_output=True)
        assert open(regenerated, "rb").read() == open(PATCH, "rb").read()
    finally:
        shutil.rmtree(tmp)
