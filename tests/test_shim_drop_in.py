"""The UNMODIFIED reference driver taichi_pathtracer/10_final/__main__.py runs under compat/taichi_pathtracer/_shim
(`import taichi as ti; from dtypes import ...; from camera import Camera; ...`, __main__.py:1-9).

CPU part (here): the script is executed with the shim's two library entry points recorded instead of executed — the
8192-iteration `for _ in trange(spp): camera.get_rays(rays); shader(world, rays)` loop must collapse into ONE render pass
with the script's own settings, followed by the post pass and the PNG write.  The reference's scripts are not part of
the repository: the driver body under test is the reference's where its checkout is present, else the stage driver
kept in compat/taichi_pathtracer/<stage>/__main__.py (same statements, see its header).  The drivers kept for stages 4
and 5 do not use the shim, so their test needs the reference's scripts."""
import os
import random
import runpy
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SHIM = os.path.join(ROOT, "compat", "taichi_pathtracer", "_shim")
REF = "/root/reference/taichi_pathtracer"


def _script(stage):
    p = os.path.join(REF, stage, "__main__.py")
    return p if os.path.exists(p) else os.path.join(ROOT, "compat", "taichi_pathtracer", stage, "__main__.py")


def _run(stage, tmp_path, monkeypatch, fake=True):
    for m in ("taichi", "dtypes", "camera", "world", "bsdf", "postprocessing", "_runtime"):
        sys.modules.pop(m, None)
    for m in list(sys.modules):
        if m == "_shim_driver":
            sys.modules.pop(m)
    monkeypatch.syspath_prepend(SHIM)
    monkeypatch.chdir(tmp_path)
    monkeypatch.delenv("LPT_SPP", raising=False)
    import _runtime
    calls = []
    if fake:
        def render_pass(image, world, cam, count, depth, model, first_sample, flags=0):
            calls.append(("render", world, cam, count, depth, model, first_sample, image.shape, flags))
            return None

        def read_image(image):
            calls.append(("read", image.post, image.norm))
            return np.full(image.shape + (3,), 0.5, np.float32)
        monkeypatch.setattr(_runtime, "_render_pass", render_pass)
        monkeypatch.setattr(_runtime, "_read_image", read_image)
    random.seed(20261018)
    g = runpy.run_path(_script(stage), run_name="__main__")
    for m in ("taichi", "dtypes", "camera", "world", "bsdf", "postprocessing", "_runtime"):
        sys.modules.pop(m, None)
    return g, calls


def test_unmodified_10_final_script_collapses_into_one_render_pass(tmp_path, monkeypatch):
    import learn_path_tracing_b200 as L
    g, calls = _run("10_final", tmp_path, monkeypatch)
    renders = [c for c in calls if c[0] == "render"]
    assert len(renders) == 1
    _, world, cam, count, depth, model, first, shape, _flags = renders[0]
    assert (count, depth, model, first, shape) == (8192, 32, L.PT_SHADE_V2, 0, (1280, 720))   # the script's own globals
    assert 470 <= world.size <= 490 and world.spheres[0].radius == 10000                        # random_scene(): ground first
    assert [round(float(x), 4) for x in cam.pos] == [13.0, 2.0, 3.0] and abs(cam.focal_length - 10.0) < 1e-6 and abs(cam.aperture - 0.2) < 1e-6
    assert abs(cam.view_w - 2 * np.tan(np.radians(40) / 2)) < 1e-6                              # set_fov(40) AFTER look_at
    assert calls[-1] == ("read", (True, 2.2), 8192)                                             # post_processing(): ACES + gamma 2.2
    assert os.path.exists(tmp_path / "outputs" / "10_final.png")
    from learn_path_tracing_b200 import scenes                                                  # the scene the bench renders
    ref_world, _ = scenes.scene_10_final((1280, 720))
    a, b = world.arrays(), ref_world.arrays()
    assert np.array_equal(a[0], b[0]) and np.array_equal(a[1], b[1])


@pytest.mark.parametrize("stage,model_name,n", [("6_diffuse", "PT_SHADE_V2_DIFFUSE", 4), ("8_refract", "PT_SHADE_V2", 6), ("9_dof", "PT_SHADE_V2", 6)])
def test_unmodified_stage_scripts_under_the_shim(tmp_path, monkeypatch, stage, model_name, n):
    import learn_path_tracing_b200 as L
    g, calls = _run(stage, tmp_path, monkeypatch)
    renders = [c for c in calls if c[0] == "render"]
    assert len(renders) == 1 and renders[0][3] == 8192 and renders[0][5] == getattr(L, model_name)
    assert renders[0][1].size == n and os.path.exists(tmp_path / "outputs" / f"{stage}.png")


def test_unmodified_early_stage_scripts_under_the_shim(tmp_path, monkeypatch):
    """Stages 4 and 5 (4_objects, 5_anti_aliasing: normals as colours) name no BSDF: one lattice ray per pixel and no
    `spp` in stage 4, 100 jittered samples in stage 5; neither calls post_processing()."""
    import learn_path_tracing_b200 as L
    if not os.path.exists(os.path.join(REF, "4_objects", "__main__.py")):
        pytest.skip("reference checkout not mounted")
    g, calls = _run("4_objects", tmp_path, monkeypatch)
    (r,) = [c for c in calls if c[0] == "render"]
    assert (r[3], r[4], r[5], r[8]) == (1, 1, L.PT_SHADE_V2_NORMALS, L.PT_FLAG_PIXEL_GRID) and r[1].size == 2
    assert calls[-1] == ("read", None, 1)
    g, calls = _run("5_anti_aliasing", tmp_path, monkeypatch)
    (r,) = [c for c in calls if c[0] == "render"]
    assert (r[3], r[4], r[5], r[8]) == (100, 1, L.PT_SHADE_V2_NORMALS, 0)
    assert calls[-1] == ("read", None, 100) and os.path.exists(tmp_path / "outputs" / "5_anti_aliasing.png")


@pytest.mark.gpu
def test_unmodified_10_final_script_renders_on_the_gpu(tmp_path, monkeypatch, ctx):
    """The real thing: the reference's script, its 8192 spp, one launch; the PNG equals the one L.render() writes for the
    same seeded scene (same paths: RNG keyed on pixel and sample)."""
    import learn_path_tracing_b200 as L
    from learn_path_tracing_b200 import scenes
    g, _ = _run("10_final", tmp_path, monkeypatch, fake=False)
    png = L.imread(str(tmp_path / "outputs" / "10_final.png"))
    world, cam = scenes.scene_10_final((1280, 720))
    ref = L.to_uint8(L.render(world, cam, spp=8192, propagate_limit=32, ctx=ctx))
    d = L.to_uint8(png).astype(np.int32) - ref.astype(np.int32)
    assert np.abs(d).max() <= 1 and (d != 0).mean() < 1e-3, (np.abs(d).max(), (d != 0).mean())


def test_shim_flushes_per_camera_and_resets_on_fill(tmp_path, monkeypatch):
    """Host logic of the shim's image field: samples booked for one (world, camera) collapse into one pass, a camera that
    moved starts another pass with the sample index carried on, image.fill(0) starts over."""
    for m in ("taichi", "dtypes", "camera", "world", "bsdf", "postprocessing", "_runtime"):
        sys.modules.pop(m, None)
    monkeypatch.syspath_prepend(SHIM)
    import _runtime
    from camera import Camera
    from dtypes import Ray, Vec3f
    from world import Sphere, World
    import learn_path_tracing_b200 as L
    calls = []
    monkeypatch.setattr(_runtime, "_render_pass", lambda image, world, cam, count, depth, model, first, flags=0: calls.append((count, first, model, flags)))
    monkeypatch.setattr(_runtime, "_read_image", lambda image: np.zeros(image.shape + (3,), np.float32))
    image, rays = Vec3f.field(shape=(32, 16)), Ray.field(shape=(32, 16))
    world = World([Sphere(Vec3f([0, 0, -2]), 0.5)])
    cam = Camera((32, 16))
    for k in range(5):
        if k == 3:
            cam.set_position(Vec3f([0, 1, 0]))            # the camera moves between samples 2 and 3
        cam.get_rays(rays)
        image.book(world, rays, 5, 8, L.PT_SHADE_V2)
    assert image.to_numpy().shape == (32, 16, 3)
    assert calls == [(3, 0, L.PT_SHADE_V2, 0), (2, 3, L.PT_SHADE_V2, 0)]
    image.fill(0)
    cam.get_rays(rays)
    image.book(world, rays, 1, 8, L.PT_SHADE_V2_DIFFUSE)
    image.to_numpy()
    assert calls[-1] == (1, 0, L.PT_SHADE_V2_DIFFUSE, 0)
    with pytest.raises(RuntimeError):
        image.book(world, Ray.field(shape=(32, 16)), 1, 8, L.PT_SHADE_V2)   # shader() before get_rays()
    for m in ("taichi", "dtypes", "camera", "world", "bsdf", "postprocessing", "_runtime"):
        sys.modules.pop(m, None)
