"""Builds rust/patch/describe.patch: the edits to the reference crate that make `GpuRenderer` a drop-in
(`Describe` hooks on Shape / ShapeFunction / Material / Texture, `Scene::flat()`, `#[repr(C)] Vector3d`,
`pub mod gpu`).  Works on a scratch copy of the reference crate (a checkout of dkarpushkin/rs-pathtracing: the
directory holding its Cargo.toml and src/, named by RS_PATHTRACING_SRC), inserts the additions below at anchors found
in the reference text, and writes `diff -U1` of the result -- one line of context, so the patch carries our additions
and next to nothing of the reference.

  RS_PATHTRACING_SRC=<checkout> python tools/make_rust_patch.py [OUT]   # OUT defaults to rust/patch/describe.patch
"""
import os
import shutil
import subprocess
import sys
import tempfile

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
REF = os.environ.get("RS_PATHTRACING_SRC", "")


def insert_after(text, anchor, addition, occurrence=1):
    pos = -1
    for _ in range(occurrence):
        pos = text.index(anchor, pos + 1)
    end = pos + len(anchor)
    return text[:end] + addition + text[end:]


def insert_before(text, anchor, addition, occurrence=1):
    pos = -1
    for _ in range(occurrence):
        pos = text.index(anchor, pos + 1)
    return text[:pos] + addition + text[pos:]


def end_of_impl(text, header):
    """index of the closing brace of the top-level `impl ... {` block that starts with `header` (rustfmt style: the
    first line after it that is a lone `}` in column 0)"""
    start = text.index(header)
    return text.index("\n}\n", start) + 1


def add_to_impl(text, header, addition):
    i = end_of_impl(text, header)
    return text[:i] + addition + text[i:]


SHAPE_TRAIT = '''
    /// Append this shape's row(s) to the flat description the GPU core takes (include/rt_b200.h, rt_scene_desc).
    fn describe(&self, flat: &mut FlatScene);
'''
RECT = '''
    fn describe(&self, flat: &mut FlatScene) {
        flat.push_shape(sys::RT_SHAPE_RECTANGLE, 0, &self.transform,
                        [self.x0, self.y0, self.x1, self.y1, 0.0, 0.0, 0.0, 0.0], &self.material);
    }
'''
CUBE = '''
    fn describe(&self, flat: &mut FlatScene) {
        // the unit box [-1, 1]^3 (Cube::new); min_p / max_p are never anything else
        flat.push_shape(sys::RT_SHAPE_CUBE, 0, &self.transform, [0.0; 8], &self.material);
    }
'''
SPHERE = '''
    fn describe(&self, flat: &mut FlatScene) {
        let flags = if self.inverse_normal { sys::RT_SHAPE_FLAG_INVERSE_NORMAL } else { 0 };
        flat.push_shape(sys::RT_SHAPE_SPHERE, flags, &self.transform, [0.0; 8], &self.material);
    }
'''
TORUS = '''
    fn describe(&self, flat: &mut FlatScene) {
        flat.push_shape(sys::RT_SHAPE_TORUS, 0, &self.transform,
                        [self.radius, self.tube_radius, 0.0, 0.0, 0.0, 0.0, 0.0, 0.0], &self.material);
    }
'''
UNSUPPORTED = '''
    fn describe(&self, _flat: &mut FlatScene) {
        // no JSON shim, no constructor: a Tooth cannot exist outside this module (and its material is a Box, not a MaterialPtr)
        unimplemented!("%s has no GPU description");
    }
'''
COLLECTION = '''
    fn describe(&self, flat: &mut FlatScene) {
        for shape in &self.shapes {
            shape.describe(flat);
        }
    }
'''
BVH = '''
    fn describe(&self, _flat: &mut FlatScene) {
        // the tree has forgotten the list order the kernels' tie rule needs: Scene::new flattens BEFORE building it
        unreachable!("BvhNode is described through the shape list it was built from");
    }
'''
MARCH = '''
    fn describe(&self, flat: &mut FlatScene) {
        let (surface, abcd_r) = self.shape.describe();
        flat.push_shape(sys::RT_SHAPE_MARCH, 0, &self.transform,
                        [surface as f64, self.step, self.depth as f64, abcd_r[0], abcd_r[1], abcd_r[2], abcd_r[3], abcd_r[4]],
                        &self.material);
    }
'''
FUNC_TRAIT = '''
    /// (RT_SURF_* tag, [a, b, c, d, sphere_radius]) for the flat scene's params[0], params[3..8]
    fn describe(&self) -> (u32, [f64; 5]);
'''
SURFACES = {
    "Heart": "(sys::RT_SURF_HEART, [0.0; 5])   // its bound is the fixed ellipsoid of Heart::new",
    "Sine": "(sys::RT_SURF_SINE, [self.a, 0.0, 0.0, 0.0, self.sphere_radius])",
    "Star": "(sys::RT_SURF_STAR, [self.a, 0.0, 0.0, 0.0, self.sphere_radius])",
    "DupinCyclide": "(sys::RT_SURF_DUPIN, [self.a, self.b, self.c, self.d, self.sphere_radius])",
    "HuntsSurface": "(sys::RT_SURF_HUNTS, [0.0, 0.0, 0.0, 0.0, self.sphere_radius])",
    "Cushion": "(sys::RT_SURF_CUSHION, [0.0, 0.0, 0.0, 0.0, self.sphere_radius])",
}
MATERIAL_TRAIT = '''
    /// This material's row of the flat scene (its texture tree is pushed first).
    fn describe(&self, flat: &mut FlatScene) -> sys::rt_material;
'''
MATERIALS = {
    "Lambertian": "sys::rt_material { kind: sys::RT_MAT_LAMBERTIAN, texture: self.albedo.describe(flat), scalar: 0.0 }",
    "Metal": "sys::rt_material { kind: sys::RT_MAT_METAL, texture: self.albedo.describe(flat), scalar: self.fuzz }",
    "Dielectric": "sys::rt_material { kind: sys::RT_MAT_DIELECTRIC, texture: 0, scalar: self.index_of_refraction }",
    "DiffuseLight": "sys::rt_material { kind: sys::RT_MAT_DIFFUSE_LIGHT, texture: self.emit.describe(flat), scalar: 0.0 }",
    "EmptyMaterial": "sys::rt_material { kind: sys::RT_MAT_EMPTY, texture: 0, scalar: 0.0 }",
}
TEXTURE_TRAIT = '''
    /// Push this texture (children first) onto the flat scene's texture table; returns its index.
    fn describe(&self, flat: &mut FlatScene) -> u32;
'''
TEXTURES = {
    "SolidColor": "flat.push_texture(sys::RT_TEX_SOLID, [self.color.x, self.color.y, self.color.z], 0, 0, 0)",
    "CheckerTexture": '''let (odd, even) = (self.odd.describe(flat), self.even.describe(flat));
        flat.push_texture(sys::RT_TEX_CHECKER, [self.multipliers.x, self.multipliers.y, self.multipliers.z], odd, even, 0)''',
    "NoiseTexture": '''flat.noise.push(self.noise.describe());
        let table = flat.noise.len() as u32 - 1;
        flat.push_texture(sys::RT_TEX_NOISE, [self.scale, 0.0, 0.0], 0, 0, table)''',
    "UVChecker": '''let (odd, even) = (self.odd.describe(flat), self.even.describe(flat));
        // color.x pairs with v, color.y with u -- exactly the fields value() multiplies them with
        flat.push_texture(sys::RT_TEX_UV_CHECKER, [self.multipliers.0, self.multipliers.1, 0.0], odd, even, 0)''',
    "ImageTexture": '''flat.images.push((self.image.width(), self.image.height(), self.image.as_raw().clone()));
        let image = flat.images.len() as u32 - 1;
        flat.push_texture(sys::RT_TEX_IMAGE, [0.0; 3], 0, 0, image)''',
}
PERLIN = '''
    /// the tables Perlin::noise reads, as the GPU core's rt_perlin
    pub fn describe(&self) -> sys::rt_perlin {
        let mut t = sys::rt_perlin { perm_x: [0; 256], perm_y: [0; 256], perm_z: [0; 256],
                                     ranvec: [sys::rt_vec3 { x: 0.0, y: 0.0, z: 0.0 }; 256] };
        for i in 0..256 {
            t.perm_x[i] = self.perm_x[i] as u32;
            t.perm_y[i] = self.perm_y[i] as u32;
            t.perm_z[i] = self.perm_z[i] as u32;
            t.ranvec[i] = sys::rt_vec3 { x: self.ranvec[i].x, y: self.ranvec[i].y, z: self.ranvec[i].z };
        }
        t
    }
'''


def fn_describe(body, ret):
    return f"\n    fn describe(&self, flat: &mut FlatScene) -> {ret} {{\n        {body}\n    }}\n"


def main():
    if not os.path.isdir(os.path.join(REF, "src")):
        sys.exit("RS_PATHTRACING_SRC must name a checkout of the reference crate")
    tmp = tempfile.mkdtemp()
    a, b = os.path.join(tmp, "a"), os.path.join(tmp, "b")
    for d in (a, b):
        shutil.copytree(os.path.join(REF, "src"), os.path.join(d, "src"))
        shutil.copy(os.path.join(REF, "Cargo.toml"), d)

    def edit(rel, fn):
        p = os.path.join(b, rel)
        crlf = b"\r\n" in open(p, "rb").read()          # (some reference files have DOS line ends: keep them)
        text = fn(open(p).read())                         # universal newlines: anchors are written with \n
        open(p, "w", newline="\r\n" if crlf else "\n").write(text)

    edit("Cargo.toml", lambda s: insert_after(s, 'raylib = "^3.7"\n',
                                              'ray_tracing_b200-sys = { path = "../rs-pathtracing-b200/rust/ray_tracing_b200-sys" }\n'))
    edit("src/algebra/mod.rs", lambda s: insert_before(s, "#[derive(Clone, Copy, Serialize, Deserialize, Debug)]\npub struct Vector3d",
                                                       "#[repr(C)]   // layout-identical to rt_vec3: render_step hands the frame buffer to the C ABI\n"))

    def noise(s):
        s = insert_after(s, "use super::Vector3d;\n", "use ray_tracing_b200_sys as sys;\n")
        return add_to_impl(s, "impl Perlin {", PERLIN)
    edit("src/algebra/noise.rs", noise)

    def world(s):
        s = insert_after(s, "mod json_models;\n", "pub mod flat;\n")
        s = insert_after(s, "    background: Vector3d,\n", "    flat: flat::FlatScene,   // the shape list as the GPU core takes it, in list order\n")
        s = insert_before(s, "        Self {\n            world: Box::new(BvhNode::new(shapes))",
                          "        let flat = flat::FlatScene::from_shapes(&shapes);   // before the BVH takes the list apart\n")
        s = insert_after(s, "            background,\n", "            flat,\n")
        s = insert_before(s, "    pub fn from_json(data: &str)",
                          "    /// the flat description renderer::gpu::GpuRenderer uploads\n    pub fn flat(&self) -> &flat::FlatScene {\n        &self.flat\n    }\n\n")
        return s
    edit("src/world/mod.rs", world)

    def shapes(s):
        s = insert_after(s, "pub mod ray_marching;\n", "use super::flat::FlatScene;\nuse ray_tracing_b200_sys as sys;\n")
        s = insert_after(s, "    fn get_bounding_box(&self) -> AABB;\n", SHAPE_TRAIT)
        s = add_to_impl(s, "impl Shape for Rectangle {", RECT)
        s = add_to_impl(s, "impl Shape for Cube {", CUBE)
        s = add_to_impl(s, "impl Shape for Sphere {", SPHERE)
        s = add_to_impl(s, "impl Shape for Torus {", TORUS)
        s = add_to_impl(s, "impl Shape for Tooth {", UNSUPPORTED % "Tooth")
        s = add_to_impl(s, "impl Shape for ShapeCollection {", COLLECTION)
        s = add_to_impl(s, "impl Shape for BvhNode {", BVH)
        return s
    edit("src/world/shapes/mod.rs", shapes)

    def marching(s):
        s = insert_after(s, "use std::{any::Any, fmt::Debug};\n", "use super::super::flat::FlatScene;\nuse ray_tracing_b200_sys as sys;\n")
        s = add_to_impl(s, "impl Shape for RayMarchingShape {", MARCH)
        s = insert_after(s, "    fn uv(&self, p: &Vector3d) -> (f64, f64);\n", FUNC_TRAIT)
        for name, body in SURFACES.items():
            s = add_to_impl(s, f"impl ShapeFunction for {name} {{", f"\n    fn describe(&self) -> (u32, [f64; 5]) {{\n        {body}\n    }}\n")
        return s
    edit("src/world/shapes/ray_marching.rs", marching)

    def material(s):
        s = insert_after(s, "use super::{texture::Texture, Ray, RayHit};\n", "use super::flat::FlatScene;\nuse ray_tracing_b200_sys as sys;\n")
        s = insert_before(s, "}\n\npub type MaterialPtr", MATERIAL_TRAIT)
        for name, body in MATERIALS.items():
            hdr = f"impl Material for {name} {{"
            if f"impl Material for {name} {{}}" in s:   # an empty impl on one line
                s = s.replace(f"impl Material for {name} {{}}", f"impl Material for {name} {{\n}}\n")
            s = add_to_impl(s, hdr, fn_describe(body, "sys::rt_material").replace("flat: &mut FlatScene", "flat: &mut FlatScene" if "flat" in body else "_flat: &mut FlatScene"))
        return s
    edit("src/world/material.rs", material)

    def texture(s):
        s = insert_after(s, "use std::{f64::consts::PI, fmt::Debug};\n", "use super::flat::FlatScene;\nuse ray_tracing_b200_sys as sys;\n")
        s = insert_after(s, "    fn value(&self, u: f64, v: f64, p: &Vector3d) -> Vector3d;\n", TEXTURE_TRAIT)
        for name, body in TEXTURES.items():
            s = add_to_impl(s, f"impl Texture for {name} {{", fn_describe(body, "u32"))
        return s
    edit("src/world/texture.rs", texture)
    edit("src/renderer/mod.rs", lambda s: insert_before(s, "pub mod step_by_step;\n", "pub mod gpu;\n"))

    diff = subprocess.run(["diff", "-U1", "-r", "-N", "a", "b"], cwd=tmp, capture_output=True).stdout   # bytes: keep CRLF
    # no timestamps in the file headers: the patch is reproducible
    diff = b"\n".join(l.split(b"\t")[0] if l.startswith((b"--- ", b"+++ ")) else l for l in diff.split(b"\n"))
    out = sys.argv[1] if len(sys.argv) > 1 else os.path.join(ROOT, "rust", "patch", "describe.patch")
    with open(out, "wb") as f:
        f.write(diff)
    shutil.rmtree(tmp)
    lines = diff.split(b"\n")
    print(out, len(lines), "lines;", sum(1 for l in lines if l.startswith(b"+") and not l.startswith(b"+++")), "added")


if __name__ == "__main__":
    main()
