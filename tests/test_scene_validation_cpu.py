"""The scene-description check every scene passes before it reaches a device (validate_desc in rt_core.cu).

rt_scene_desc is the input boundary of the C ABI: the Rust -sys crate hands it over as raw tables, with no loader in
between.  A description the shading kernels cannot evaluate must be rejected with RT_ERR_INVALID, because once it is on
the device it either shades silently wrong (a texture graph deeper than texture_value's loop shades black) or reads out
of bounds (a Perlin permutation entry of 256 or more indexes past ranvec[]; an image whose byte size wraps is uploaded
short).  The check runs before the device count is read, so on a host without a GPU a valid description gets as far as
RT_ERR_NO_DEVICE and an invalid one stops at RT_ERR_INVALID.  rt_cull_tree_check shares the check and needs no device.

On a GPU host a valid description creates a handle, which is destroyed at once: nothing here renders."""
import ctypes as C
import json

import pytest

import rs_pathtracing_b200 as rt
from rs_pathtracing_b200 import _ffi

from conftest import scene_path

MAX_DEPTH = 8   # RT_TEX_MAX_DEPTH
SOLID, CHECKER, UV_CHECKER, IMAGE, NOISE = range(5)


def _ok_code():
    return _ffi.RT_OK if rt.device_count() > 0 else _ffi.RT_ERR_NO_DEVICE


def _codes(d):
    """the return codes of rt_scene_create, rt_scene_create_multi on one device and rt_cull_tree_check"""
    core = _ffi.core()
    out = []
    for create in (lambda h: core.rt_scene_create(C.byref(d), 0, C.byref(h)),
                   lambda h: core.rt_scene_create_multi(C.byref(d), 1, (C.c_int * 1)(0), C.byref(h))):
        h = C.c_void_p()
        out.append(create(h))
        if h.value:
            core.rt_scene_destroy(h)
    u = [C.c_uint32() for _ in range(4)]
    worst = C.c_double()
    out.append(core.rt_cull_tree_check(C.byref(d), *[C.byref(x) for x in u], C.byref(worst)))
    return out


def assert_invalid(d, what):
    assert _codes(d) == [_ffi.RT_ERR_INVALID] * 3, what


def assert_valid(d, what):
    assert _codes(d) == [_ok_code(), _ok_code(), _ffi.RT_OK], what


def _base():
    """a loaded scene with one Lambertian sphere whose albedo is a checker over a SolidColor and a NoiseTexture; its
    description can be edited in place (the Scene object owns the tables)"""
    scene = {"camera": {"position": [0, 0, -10], "direction": [0, 0, 1], "up": [0, 1, 0], "fov": 40.0,
                        "focal_length": 1.0},
             "background": [0, 0, 0],
             "materials": {"M": {"type": "Lambertian",
                                 "albedo": {"type": "CheckerTexture", "multipliers": [1, 1, 1],
                                            "odd": {"type": "SolidColor", "color": [1, 0, 0]},
                                            "even": {"type": "NoiseTexture", "scale": 2.0}}}},
             "shapes": [{"type": "Sphere", "name": "s", "material": "M",
                         "transform": {"translate": [0, 0, 0], "rotate": [0, 0, 0], "scale": [1, 1, 1]}}]}
    sc = rt.Scene.from_json(json.dumps(scene), add_random_spheres=False)
    d = sc.desc()
    assert d.n_noise == 1 and d.n_images == 0
    return sc, d


def _with_textures(d, texs):
    """point d at a new texture table (a list of (kind, odd, even, image)); material 0 uses texture 0.  Returns what
    must be kept alive."""
    arr = (_ffi.Texture * len(texs))()
    for i, (kind, odd, even, image) in enumerate(texs):
        arr[i].kind, arr[i].odd, arr[i].even, arr[i].image = kind, odd, even, image
        arr[i].color = _ffi.Vec3(1.0, 0.5, 0.25)
    mats = (_ffi.Material * 1)()
    mats[0].kind, mats[0].texture, mats[0].scalar = 0, 0, 0.0
    d.n_textures, d.textures = len(texs), arr
    d.n_materials, d.materials = 1, mats
    return arr, mats


def _chain(levels, kind=CHECKER):
    """`levels` checkers above one SolidColor leaf: texture k has both children k + 1, the leaf is last"""
    return [(kind, k + 1, k + 1, 0) for k in range(levels)] + [(SOLID, 0, 0, 0)]


def test_the_base_scene_is_valid():
    sc, d = _base()
    assert_valid(d, "base")


def test_checker_that_is_its_own_child():
    sc, d = _base()
    for odd, even in ((0, 1), (1, 0), (0, 0)):
        keep = _with_textures(d, [(CHECKER, odd, even, 0), (SOLID, 0, 0, 0)])
        assert_invalid(d, f"self loop odd={odd} even={even}")
    keep = _with_textures(d, [(UV_CHECKER, 0, 1, 0), (SOLID, 0, 0, 0)])
    assert_invalid(d, "UVChecker self loop")


def test_two_node_cycle():
    sc, d = _base()
    keep = _with_textures(d, [(CHECKER, 1, 2, 0), (UV_CHECKER, 2, 0, 0), (SOLID, 0, 0, 0)])
    assert_invalid(d, "0 -> 1 -> 0")
    # a cycle below the root, reached only through one branch
    keep = _with_textures(d, [(CHECKER, 3, 1, 0), (CHECKER, 2, 3, 0), (CHECKER, 1, 3, 0), (SOLID, 0, 0, 0)])
    assert_invalid(d, "1 -> 2 -> 1 under a valid root")
    # a cycle no material uses is still a malformed table
    keep = _with_textures(d, [(SOLID, 0, 0, 0), (CHECKER, 2, 0, 0), (CHECKER, 1, 0, 0)])
    assert_invalid(d, "unreferenced cycle")


def test_depth_limit():
    """texture_value follows at most RT_TEX_MAX_DEPTH = 8 checker edges: 8 checkers above the leaf are valid, 9 are not,
    whatever the order of the table"""
    sc, d = _base()
    for levels, valid in ((MAX_DEPTH, True), (MAX_DEPTH + 1, False), (40, False)):
        texs = _chain(levels)
        n = len(texs)
        keep = _with_textures(d, texs)
        (assert_valid if valid else assert_invalid)(d, f"{levels} levels, root first")
        # the same table reversed (texture k becomes n - 1 - k): children precede their parents
        keep = _with_textures(d, [(k, n - 1 - o, n - 1 - e, i) for (k, o, e, i) in reversed(texs)])
        d.materials[0].texture = n - 1
        (assert_valid if valid else assert_invalid)(d, f"{levels} levels, leaf first")
    # the odd branch is the deep one, the even one a leaf
    texs = [(CHECKER, k + 1, MAX_DEPTH + 1, 0) for k in range(MAX_DEPTH)] + [(SOLID, 0, 0, 0)] * 2
    keep = _with_textures(d, texs)
    assert_valid(d, "8 levels on the odd branch")
    texs = [(UV_CHECKER, MAX_DEPTH + 2, k + 1, 0) for k in range(MAX_DEPTH + 1)] + [(SOLID, 0, 0, 0)] * 2
    keep = _with_textures(d, texs)
    assert_invalid(d, "9 levels on the even branch")


def test_shared_children_are_not_a_cycle():
    """a DAG: two checkers share a child, and a diamond of 8 levels (every level's both children are the next level)"""
    sc, d = _base()
    keep = _with_textures(d, [(CHECKER, 1, 2, 0), (CHECKER, 3, 4, 0), (UV_CHECKER, 3, 4, 0), (SOLID, 0, 0, 0),
                              (SOLID, 0, 0, 0)])
    assert_valid(d, "two checkers share both children")
    texs = []
    for lvl in range(MAX_DEPTH):
        texs += [(CHECKER, 2 * lvl + 2, 2 * lvl + 3, 0), (UV_CHECKER, 2 * lvl + 3, 2 * lvl + 2, 0)]
    texs += [(SOLID, 0, 0, 0)] * 2
    keep = _with_textures(d, texs)
    assert_valid(d, "diamond of 8 levels")


@pytest.mark.parametrize("table", ["perm_x", "perm_y", "perm_z"])
@pytest.mark.parametrize("value", [256, 257, 0x10000, 0xFFFFFFFF])
def test_perlin_permutation_out_of_range(table, value):
    sc, d = _base()
    perm = getattr(d.noise[0], table)
    for k in (0, 97, 255):
        old = perm[k]
        perm[k] = value
        assert_invalid(d, f"{table}[{k}] = {value}")
        perm[k] = old
    perm[97] = 255
    assert_valid(d, f"{table}[97] = 255")


def test_missing_noise_table():
    sc, d = _base()
    d.noise = None
    assert_invalid(d, "n_noise = 1, noise = NULL")
    d.n_noise = 0
    assert_invalid(d, "a NoiseTexture with no table")


@pytest.mark.parametrize("w,h,valid", [(1 << 31, 1 << 31, False), (0xFFFFFFFF, 0xFFFFFFFF, False),
                                       (1, 1, True), (3, 5, True)])
def test_image_size_overflow(w, h, valid):
    """4 * width * height bytes must be addressable: at 2^31 x 2^31 the size_t product wraps to 0 and at
    (2^32 - 1)^2 it does not fit 64 bits; the buffer holds 4 * 15 bytes, so only the small images are real"""
    sc, d = _base()
    buf = (C.c_uint8 * 60)()
    img = (_ffi.Image * 1)()
    img[0].width, img[0].height = w, h
    img[0].rgba = C.cast(buf, C.POINTER(C.c_uint8))
    keep = _with_textures(d, [(IMAGE, 0, 0, 0)])
    d.n_images, d.images = 1, img
    (assert_valid if valid else assert_invalid)(d, f"{w} x {h} image")


def _nested_checker_json(levels):
    tex = {"type": "SolidColor", "color": [0.2, 0.4, 0.8]}
    for k in range(levels):
        tex = {"type": "CheckerTexture" if k % 2 else "UVChecker",
               "multipliers": [1, 1, 1] if k % 2 else [1, 1], "odd": tex, "even": tex}
    return json.dumps({"camera": {"position": [0, 0, -10], "direction": [0, 0, 1], "up": [0, 1, 0], "fov": 40.0,
                                  "focal_length": 1.0},
                       "background": [0, 0, 0],
                       "materials": {"M": {"type": "Lambertian", "albedo": tex}},
                       "shapes": [{"type": "Sphere", "name": "s", "material": "M",
                                   "transform": {"translate": [0, 0, 0], "rotate": [0, 0, 0], "scale": [1, 1, 1]}}]})


def test_loader_depth_limit():
    """the JSON loader applies the same limit: 8 levels load (and pass the check), 9 raise"""
    sc = rt.Scene.from_json(_nested_checker_json(MAX_DEPTH), add_random_spheres=False)
    d = sc.desc()
    assert d.n_textures == 2 ** (MAX_DEPTH + 1) - 1   # the loader stores each child of a checker on its own
    assert_valid(d, "8 levels from JSON")
    with pytest.raises(Exception, match="too deep"):
        rt.Scene.from_json(_nested_checker_json(MAX_DEPTH + 1), add_random_spheres=False)


@pytest.mark.parametrize("name", ["spheres.json", "cornell_box.json", "detached_materials.json"])
def test_shipped_scenes_stay_valid(name):
    sc = rt.Scene.from_file(scene_path(name), random_spheres_seed=1)
    assert_valid(sc.desc(), name)
