"""Scene.trace_pixel_samples_group without a CUDA device: the core has no CPU fallback, so the call fails loudly."""
import numpy as np
import pytest

import rs_pathtracing_b200 as rt

from conftest import scene_path


def test_trace_pixel_samples_group_fails_loudly_without_gpu():
    if rt.device_count() > 0:
        pytest.skip("GPU present")
    sc = rt.Scene.from_file(scene_path("cube_test.json"), add_random_spheres=False)
    rays = np.tile([0.0, 0.0, -10.0, 0.0, 0.0, 1.0], (3, 1))
    with pytest.raises(rt.RtError, match="no CUDA device"):
        sc.trace_pixel_samples_group(rays, [0, 1, 3], [7, 8], 8, seed=1)
