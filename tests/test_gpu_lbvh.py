"""The GPU-side acceleration-structure builder (csrc/lbvh.cu, B200RT_BUILDER_GPU_LBVH).
Closest-hit results do not depend on the tree, so the Morton-order LBVH must give the very same
hits -- and therefore, with the same RNG key, the very same image -- as the host SAH tree."""
import numpy as np
import pytest

from conftest import SMALL_SCENES

pytestmark = pytest.mark.gpu


@pytest.mark.parametrize("name", SMALL_SCENES)
def test_lbvh_raycast_matches_reference(golden, name):
    import cpp_raytracer_b200 as rt
    from cpp_raytracer_b200 import capi
    scene = golden.scene(name)
    rays, tmin, tmax = golden.rays(name)
    want_p, want_t = golden.hits(name, brute=True)          # reference Scene::hit_by
    with rt.DeviceSceneHandle(scene, builder=capi.BUILDER_GPU_LBVH) as dev:
        info = dev.info()
        p, t = dev.raycast(rays, tmin, tmax)
    assert 3 * info["tree_depth"] <= 128
    assert np.array_equal(p, want_p) and np.array_equal(t, want_t), f"{name}: LBVH tree changes closest-hit results"
    print(f"{name}: LBVH {info['n_nodes']} nodes, depth {info['tree_depth']}, build {info['build_ms']:.2f} ms")


@pytest.mark.parametrize("name", ["rtow_lights", "cornell", "xmas"])
def test_image_is_independent_of_the_builder(golden, name):
    import cpp_raytracer_b200 as rt
    from cpp_raytracer_b200 import capi
    scene = golden.scene(name)
    cam = rt.camera_with(scene.camera, image_w=96, image_h=54, spp=24, max_depth=30)
    with rt.DeviceSceneHandle(scene, builder=capi.BUILDER_HOST_SAH) as a:
        ia, sa = a.render(cam, seed=11)
    with rt.DeviceSceneHandle(scene, builder=capi.BUILDER_GPU_LBVH) as b:
        ib, sb = b.render(cam, seed=11)
    assert sa["rays"] == sb["rays"]
    assert np.array_equal(ia, ib), f"{name}: image depends on the acceleration structure"


def test_lbvh_seeded_random_mixed_scene_vs_c_oracle():
    import os, sys
    import cpp_raytracer_b200 as rt
    from cpp_raytracer_b200 import capi
    from conftest import ROOT
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import pt_oracle
    from test_gpu_raycast import _random_scene
    rng = np.random.default_rng(21)
    scene = _random_scene(rng, 3000, 1000)
    # duplicates: many coincident primitives get identical Morton codes
    scene.spheres["c"][:200] = scene.spheres["c"][0]
    n = 4096
    rays = np.concatenate([rng.uniform(-25, 25, (n, 3)), rng.normal(size=(n, 3))], axis=1)
    want_p, want_t = pt_oracle.raycast_brute(scene, rays, 1e-5, np.inf)
    with rt.DeviceSceneHandle(scene, builder=capi.BUILDER_GPU_LBVH) as dev:
        p, t = dev.raycast(rays, 1e-5, np.inf)
    assert np.array_equal(p, want_p) and np.array_equal(t, want_t)


@pytest.mark.parametrize("n", [1, 2, 3, 5, 33])
def test_lbvh_tiny_and_degenerate_inputs(n):
    """n = 1 falls back to the host builder; 2..33 primitives, all coincident (identical Morton
    codes) or on a line, still give Scene::hit_by's answers."""
    import os, sys
    import cpp_raytracer_b200 as rt
    from cpp_raytracer_b200 import capi
    from conftest import ROOT
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import pt_oracle
    rng = np.random.default_rng(n)
    for layout in ("coincident", "line"):
        sph = np.zeros(n, capi.SPHERE_DTYPE)
        sph["c"] = [0.0, 0.0, -5.0] if layout == "coincident" else np.stack([np.arange(n) * 2.5, np.zeros(n), np.full(n, -5.0)], axis=1)
        sph["r"] = 1.0
        sph["prim"] = rng.permutation(n)
        scene = capi.HostScene(np.zeros(1, capi.MATERIAL_DTYPE), sph, np.zeros(0, capi.QUAD_DTYPE), np.zeros(1, capi.CAMERA_DTYPE))
        rays = np.concatenate([rng.uniform(-1, 1, (256, 3)) + [0, 0, 3], rng.normal(size=(256, 3)) * [1, 0.2, 1] + [0, 0, -2]], axis=1)
        want_p, want_t = pt_oracle.raycast_brute(scene, rays, 1e-5, np.inf)
        with rt.DeviceSceneHandle(scene, builder=capi.BUILDER_GPU_LBVH) as dev:
            p, t = dev.raycast(rays, 1e-5, np.inf)
        assert np.array_equal(p, want_p) and np.array_equal(t, want_t), (n, layout)


@pytest.mark.parametrize("field,value", [("mat", 1 << 30), ("prim", 1 << 30), ("kind", 9)])
def test_gpu_builder_rejects_out_of_range_indices(golden, field, value):
    """Scene creation checks the description's per-primitive indices and material kinds on the device
    (scene_layout.cu) whichever builder made the tree: a bad material or canonical index on a sphere or a quad, or an
    unknown material kind, is B200RT_EINVAL under both builders."""
    import cpp_raytracer_b200 as rt
    from cpp_raytracer_b200 import capi
    for name, prims, i in (("rtow_final", "spheres", 7), ("cornell", "quads", 3)):
        scene = golden.scene(name)
        bad = capi.HostScene(scene.materials.copy(), scene.spheres.copy(), scene.quads.copy(), scene.camera)
        (bad.materials if field == "kind" else getattr(bad, prims))[field][i] = value
        for builder in (capi.BUILDER_GPU_LBVH, capi.BUILDER_HOST_SAH):
            with pytest.raises(rt.B200rtError) as e:
                rt.DeviceSceneHandle(bad, builder=builder)
            assert e.value.code == capi.EINVAL, (name, prims, builder)
