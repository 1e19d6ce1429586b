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
