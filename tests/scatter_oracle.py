"""ctypes loader of tests/oracle_scatter.cpp: the oracle's one level of ray_color for caller rays (orc_scatter_batch),
the reference for rt_scatter_batch.  It is compiled on first use into a temporary directory, against the oracle's
library, with the oracle's compiler flags."""
import ctypes as C
import os
import subprocess
import tempfile

import numpy as np

from oracle import pyoracle as po

HERE = os.path.dirname(os.path.abspath(__file__))
SRC = os.path.join(HERE, "oracle_scatter.cpp")
CXXFLAGS = ["-O2", "-std=c++17", "-fPIC", "-ffp-contract=off", "-fno-fast-math", "-Wall", "-Wextra",
            "-Wno-unused-parameter"]

_lib = None


def lib() -> C.CDLL:
    global _lib
    if _lib is None:
        po.build()
        so = os.path.join(tempfile.mkdtemp(prefix="oracle_scatter_"), "liboracle_scatter.so")
        oracle_dir = os.path.dirname(po.SO)
        subprocess.run([os.environ.get("CXX", "g++"), *CXXFLAGS, "-shared", "-o", so, SRC, po.SO,
                        "-Wl,-rpath," + oracle_dir], check=True, capture_output=True)
        po.lib()   # the scene handles come from the oracle's own library: load it first, under its own name
        L = C.CDLL(so)
        L.orc_scatter_batch.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint64, C.c_uint32, C.c_uint64,
                                        C.c_double, C.c_double] + [C.c_void_p] * 5
        L.orc_scatter_batch.restype = None
        _lib = L
    return _lib


def scatter_batch(osc: "po.OracleScene", rays, keys, level, seed=0, min_t=0.001, max_t=np.inf) -> dict:
    """Scene.scatter's outputs computed by the oracle, as numpy arrays"""
    rays = np.ascontiguousarray(rays, dtype=np.float64).reshape(-1, 6)
    keys = np.ascontiguousarray(keys, dtype=np.uint32).reshape(-1, 2)
    n = rays.shape[0]
    out = {"index": np.empty(n, np.int32), "t": np.empty(n), "outcome": np.empty(n, np.uint8),
           "color": np.empty((n, 3)), "scattered": np.empty((n, 6))}
    vp = lambda a: a.ctypes.data_as(C.c_void_p)
    lib().orc_scatter_batch(osc._h, vp(rays), vp(keys), n, level, seed, min_t, max_t,
                            *(vp(out[k]) for k in ("index", "t", "outcome", "color", "scattered")))
    return out


def fold_paths(osc, rays, keys, depth, seed=0):
    """ray_color of each ray by iterating scatter_batch over the levels and folding the colours backwards,
    L = a0 * (a1 * (... * last)) -- the recursion's order -- with a hit on level `depth` black.  float64 (n, 3)."""
    n = len(rays)
    verts = []   # per level: (live indices, outcome, colour)
    live, cur = np.arange(n), np.ascontiguousarray(rays, dtype=np.float64)
    keys = np.ascontiguousarray(keys, dtype=np.uint32)
    for level in range(depth + 1):
        if live.size == 0:
            break
        out = scatter_batch(osc, cur, keys[live], level, seed)
        verts.append((live, out["outcome"], out["color"]))
        go = out["outcome"] == 1
        if level == depth:
            break
        live, cur = live[go], np.ascontiguousarray(out["scattered"][go])
    L = np.zeros((n, 3))
    for level in range(len(verts) - 1, -1, -1):
        live, oc, col = verts[level]
        tail = L[live]
        if level == depth:
            res = np.where((oc == 0)[:, None], col, 0.0)
        else:
            # product(attenuation, ray_color(...)) = (a.x * tail.x, ...) at a scatter; the colour itself otherwise
            res = np.where((oc == 1)[:, None], col * tail, col)
        L[live] = res
    return L
