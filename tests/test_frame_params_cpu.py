"""Frame parameters checked without a device: the shard layout's slot count (rt_shard_float4_count is host-only) and
the oracle's per-sample colours, which the GPU frame tests compare paths with."""
import numpy as np

import rs_pathtracing_b200 as rt
from rs_pathtracing_b200 import api
from oracle import pyoracle as po

from conftest import scene_path


def _params(w, h, shards, tile_w, tile_h):
    p = api.render_params(w, h, 1, 2, 0, shards, 0)
    p.tile_width, p.tile_height = tile_w, tile_h
    return p


def _tiles(w, h, tw, th):
    return -(-w // tw) * -(-h // th)


def test_shard_slot_counts_cover_every_tile_once():
    for (w, h, tw, th) in ((37, 23, 1, 1), (37, 23, 7, 5), (37, 23, 31, 33), (37, 23, 64, 16), (100, 70, 32, 32),
                           (2, 70000, 32, 32), (1, 45, 7, 5)):
        for shards in range(2, 17):
            p = _params(w, h, shards, tw, th)
            counts = [api.shard_float4_count(p, s) for s in range(shards)]
            assert sum(counts) == _tiles(w, h, tw, th) * tw * th, (w, h, tw, th, shards)
            # tile k belongs to shard k % shards: the first shards own one tile more than the rest
            n_tiles = _tiles(w, h, tw, th)
            assert counts == [((n_tiles - s + shards - 1) // shards) * tw * th for s in range(shards)]
    # unsharded: the image itself, one row per "tile"
    assert api.shard_float4_count(_params(33, 31, 1, 7, 5), 0) == 33 * 31


def test_shard_slot_count_of_tiles_past_32_bits():
    # a tile of 2^32 pixels or more cannot be addressed: no slots (rt_render_start / rt_assemble_frame reject it)
    for tw, th in ((65536, 65537), (65536, 65536), (0xFFFFFFFF, 2), (0xFFFFFFFF, 0xFFFFFFFF)):
        for s in range(2):
            assert api.shard_float4_count(_params(100, 100, 2, tw, th), s) == 0, (tw, th, s)
    # the largest tile that fits: counted in 64 bits, and the tile count must not wrap either
    p = _params(2, 2, 2, 0xFFFFFFFF, 1)
    assert [api.shard_float4_count(p, s) for s in range(2)] == [0xFFFFFFFF, 0xFFFFFFFF]
    # an unsharded row of 3e9 pixels (w * h < 2^32 is allowed)
    assert api.shard_float4_count(_params(3_000_000_000, 1, 1, 0, 0), 0) == 3_000_000_000


def test_oracle_sample_colours_reproduce_the_oracle_frame():
    """the per-sample colours, averaged in sample order from 0.0, are orc_render's Philox frame bit for bit; sample_base
    continues the sample numbering, a pixel list picks rows, and the one-pixel entry is the same call"""
    sc = rt.Scene.from_file(scene_path("light_source.json"), random_spheres_seed=1)
    cam = sc.camera()
    osc = po.OracleScene(sc.desc())
    w, h, spp, depth, seed = 13, 9, 3, 6, (1 << 63) + 12345
    frame, _ = osc.render(cam, w, h, spp, depth, seed=seed, rng="philox")
    cols = osc.frame_sample_colors(cam, w, h, spp, depth, seed)
    assert cols.shape == (w * h, spp, 3)
    acc = np.zeros((w * h, 3))
    for s in range(spp):
        acc = acc + cols[:, s]
    assert np.array_equal((acc / spp).reshape(h, w, 3), frame)
    assert np.isfinite(cols).all() and cols.max() > 0
    more = osc.frame_sample_colors(cam, w, h, 2, depth, seed, sample_base=spp)
    five = osc.frame_sample_colors(cam, w, h, spp + 2, depth, seed, threads=1)
    assert np.array_equal(np.concatenate([cols, more], axis=1), five)
    pix = np.array([w * h - 1, 0, 17, 17, 40])
    assert np.array_equal(osc.frame_sample_colors(cam, w, h, spp, depth, seed, pixels=pix), cols[pix])
    for p in pix:
        assert np.array_equal(osc.pixel_sample_colors(cam, w, h, int(p % w), int(p // w), spp, depth, seed=seed), cols[p])


def test_oracle_group_colours_reproduce_the_oracle_trace():
    """the per-ray colours of caller rays in groups: each group's in-order f64 sum over its count is orc_trace_pixel_samples
    bit for bit (an empty group: NaN), the camera's own primary rays give frame_sample_colors bit for bit, and the result
    does not depend on the thread count"""
    sc = rt.Scene.from_file(scene_path("light_source.json"), random_spheres_seed=1)
    cam = sc.camera()
    osc = po.OracleScene(sc.desc())
    w, h, spp, depth, seed = 7, 5, 3, 6, (1 << 64) - 1
    rays = np.empty((w * h * spp, 6))
    for p in range(w * h):
        for s in range(spp):
            u, v = po.philox_stream(seed, p, s, 0, 2)
            rays[p * spp + s] = po.get_ray(cam, w, h, p % w + u, p // w + v)
    offsets = np.arange(0, w * h * spp + 1, spp, dtype=np.uint64)
    cols = osc.group_sample_colors(rays, offsets, np.arange(w * h), depth, seed)
    assert np.array_equal(cols.reshape(w * h, spp, 3), osc.frame_sample_colors(cam, w, h, spp, depth, seed))
    # ragged groups with empty ones, repeated pixel indices and the key 0xFFFFFFFF; rays not of unit length
    rng = np.random.default_rng(3)
    sizes = [0, 1, 4, 0, 0, 9, 2, 0]
    n = sum(sizes)
    rays = np.concatenate([np.tile(cam.position.tuple(), (n, 1)), rng.normal(size=(n, 3)) * 2.0], axis=1)
    offsets = np.concatenate([[0], np.cumsum(sizes)]).astype(np.uint64)
    pix = np.array([5, 0xFFFFFFFF, 0, 5, 7, 0xFFFFFFFF, 12, 0], np.uint32)
    cols = osc.group_sample_colors(rays, offsets, pix, depth, seed, threads=1)
    assert np.isfinite(cols).all() and cols.max() > 0
    for t in (2, 3, 16):
        assert np.array_equal(osc.group_sample_colors(rays, offsets, pix, depth, seed, threads=t), cols), t
    for g, n_g in enumerate(sizes):
        acc = np.zeros(3)
        for c in cols[int(offsets[g]):int(offsets[g + 1])]:
            acc = acc + c
        with np.errstate(invalid="ignore"):
            mean = acc / n_g
        if n_g == 0:
            assert np.isnan(mean).all()
            continue
        want = osc.trace_pixel_samples(rays[int(offsets[g]):int(offsets[g + 1])], depth, seed=seed, pixel_index=int(pix[g]))
        assert np.array_equal(mean, want), g
