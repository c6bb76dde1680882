"""Scene construction of the kernel matrix (tests/test_gpu_kernel_matrix.py) on the host, without a device: the deep-tree scene
is as deep as it is meant to be, the checker nest limit holds, and every new scene family crosses the ABI and renders on the
oracle."""
import numpy as np
import pytest

import oracle
from helpers import oracle_camera
from ray_tracing_fsharp_b200 import abi, native
from ray_tracing_fsharp_b200.domain import Hittable, ParameterisedTexture, Pixel, Sphere, SphereStyle, marshal
from test_gpu_kernel_matrix import NEW_FAMILIES, _image, checker_nest, deep_tree, random_spheres


def test_deep_tree_depth_on_the_host():
    hs, ts, keep = marshal(deep_tree().objects)
    info = native.SceneHandle(hs, ts, -1, keepalive=keep).device_bvh_check()
    assert 45 <= info["depth"] <= 60, info


@pytest.mark.parametrize("depth", [8, 9])
def test_checker_nest_limit(depth):
    interpret = Sphere.plane_map_inverse(1.0, (0.0, 0.0, 0.0))
    tex = checker_nest(depth, _image(3, 5, 30), ParameterisedTexture.Colour(Pixel(20, 200, 60)))
    hs, ts, keep = marshal([Hittable.Sphere(Sphere.make(SphereStyle.LambertReflection(1.0, ParameterisedTexture.to_texture(interpret, tex)),
                                                        (0.0, 0.0, 0.0), 1.0))])
    if depth == 8:
        native.SceneHandle(hs, ts, -1, keepalive=keep).close()
    else:
        with pytest.raises(native.RtError) as err:
            native.SceneHandle(hs, ts, -1, keepalive=keep)
        assert err.value.code == abi.RT_ERR_UNSUPPORTED


@pytest.mark.parametrize("name", list(NEW_FAMILIES) + ["random-spheres"])
def test_new_scenes_marshal_and_render_on_the_oracle(name):
    spec = random_spheres(1000) if name == "random-spheres" else NEW_FAMILIES[name]()
    hs, ts, keep = marshal(spec.objects)
    assert len(hs) == len(spec.objects)
    native.SceneHandle(hs, ts, -1, keepalive=keep).close()  # the library accepts it
    if name == "planes-only":
        assert not any(h.shape == abi.RT_SHAPE_SPHERE for h in hs)
    if name == "one-sphere":
        assert sum(h.shape == abi.RT_SHAPE_SPHERE for h in hs) == 1
    cam = oracle_camera(spec)
    cam.samples_per_pixel = 4
    rgb, sums, counters, _ = oracle.Scene(hs, ts).render(cam, 2, 1, seed=3, rng_mode=1, adaptive=True)
    assert rgb.shape == (3, 5, 3) and counters["rays"] >= counters["paths"] > 0 and sums[..., 3].min() == 5
