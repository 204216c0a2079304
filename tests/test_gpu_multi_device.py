"""One frame on several contexts of ONE process (pt_multi_render, pt_scene_replicate, MultiRenderer) == the frame of one
context, for a v2 sphere scene and a legacy mesh world.

Every test runs with the members as extra contexts on cuda:0, each on its own stream (two members on one device are
legal: their persistent launches queue); on a box with >= 2 GPUs the same tests also run with the members on distinct
devices, where the reduce reads the partials over peer memory."""
import os
import sys

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
W, H, DEPTH, SEED = 161, 91, 16, 5   # 161 x 91: an odd pixel count, uneven reduce slices
RTOL, ATOL = 2e-4, 2e-5               # test_gpu_multigpu.py: the same paths, fp32 summation order differs


def _n_gpus():
    import torch
    return torch.cuda.device_count()


# "same": every member on cuda:0; "distinct": members cycle over the visible devices (only where there are >= 2)
LAYOUTS = ["same"] + (["distinct"] if _n_gpus() >= 2 else [])


def _devices(layout, n):
    return [0] * n if layout == "same" else [i % _n_gpus() for i in range(n)]


def _world(kind, size=(W, H)):
    from learn_path_tracing_b200 import scenes
    if kind == "v2":
        return scenes.scene_10_final(size)
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    from helpers import synthetic_legacy_world
    world, cam = synthetic_legacy_world()
    cam.resolution = tuple(size)
    return world, cam


def _model(kind):
    import learn_path_tracing_b200 as L
    return L.PT_SHADE_LEGACY if kind == "legacy" else L.PT_SHADE_V2


def _params(spp, offset=0, sq=False):
    import learn_path_tracing_b200 as L
    p = L._lib.PtRenderParams()
    p.width, p.height, p.spp, p.spp_offset, p.max_depth, p.seed = W, H, spp, offset, DEPTH, SEED
    p.absorptivity = 0.25
    p.flags = L.PT_FLAG_ACCUM_SQ if sq else 0
    return p


class Group:
    """n member contexts (member 0 = the session context) on `devices`, each other one on its own torch stream."""

    def __init__(self, ctx, devices):
        import torch
        import learn_path_tracing_b200 as L
        assert devices[0] == ctx.device
        self.streams = [torch.cuda.Stream(device=d) for d in devices[1:]]
        self.members = [ctx] + [L.Context(d, s.cuda_stream) for d, s in zip(devices[1:], self.streams)]
        self.multi = L._lib.Multi(self.members)

    def scenes(self, root_scene):
        return [root_scene] + [root_scene.replicate(c) for c in self.members[1:]]


def _single(ctx, kind, spp, sq=False):
    import learn_path_tracing_b200 as L
    world, cam = _world(kind)
    r = L.Renderer(W, H, ctx, want_sq=sq)
    r.render(world.device_scene(ctx), cam.to_struct(), spp, DEPTH, _model(kind), seed=SEED)
    return r


def _accum(ctx, n_sq=False):
    import torch
    dev = torch.device("cuda", ctx.device)
    a = torch.zeros((H * W, 4), dtype=torch.float32, device=dev)
    return a, (torch.zeros_like(a) if n_sq else None)


# ---- 1. replica == source --------------------------------------------------------------------------------------------
@pytest.mark.parametrize("layout", LAYOUTS)
@pytest.mark.parametrize("kind", ["v2", "legacy"])
def test_replica_is_the_same_scene(ctx, kind, layout):
    import torch
    import learn_path_tracing_b200 as L
    world, cam = _world(kind, (160, 90))
    dev = _devices(layout, 2)[1]
    other = L.Context(dev, torch.cuda.Stream(device=dev).cuda_stream)
    src = world.device_scene(ctx)   # the test's own world: closing its scene below affects nothing else
    rep = src.replicate(other)
    assert src.bvh_info() == rep.bvh_info()
    (n0, g0), (n1, g1) = src.bvh_download(), rep.bvh_download()
    assert n0.tobytes() == n1.tobytes() and g0.tobytes() == g1.tobytes()
    n_tri = int(src.bvh_info()[1]) - len(world.spheres)
    if kind == "legacy":
        assert n_tri > 0 and src.triangles_download(n_tri).tobytes() == rep.triangles_download(n_tri).tobytes()
    rays = ctx.generate_rays(cam.to_struct(), 256, 256, 3, 11)   # 2^16 seeded (jittered, defocused) camera rays
    ids0, t0, _ = ctx.trace_batch(src, rays)
    ids1, t1, _ = other.trace_batch(rep, rays)
    assert (ids0 >= 0).any() and np.array_equal(ids0, ids1) and t0.tobytes() == t1.tobytes()
    # the replica owns its arrays: it still renders after the source is gone
    r = L.Renderer(160, 90, ctx)
    r.render(src, cam.to_struct(), 4, 8, _model(kind), seed=SEED)
    want = r.mean()
    src.close()
    torch.cuda.synchronize()
    acc = torch.zeros((160 * 90, 4), dtype=torch.float32, device=torch.device("cuda", dev))
    p = L._lib.PtRenderParams()
    p.width, p.height, p.spp, p.max_depth, p.shading_model, p.seed, p.absorptivity = 160, 90, 4, 8, _model(kind), SEED, 0.25
    other.render(rep, cam.to_struct(), p, acc.data_ptr())
    got = other.download_accum(acc.data_ptr(), 160, 90) / 4
    assert np.allclose(got, want, rtol=RTOL, atol=ATOL), float(np.abs(got - want).max())   # accumulation order may differ


# ---- 2. multi render == one-context render ----------------------------------------------------------------------------
@pytest.mark.parametrize("layout", LAYOUTS)
@pytest.mark.parametrize("kind", ["v2", "legacy"])
@pytest.mark.parametrize("n,spp", [(2, 24), (3, 24), (3, 2)])
def test_multi_render_equals_one_context(ctx, kind, layout, n, spp):
    import learn_path_tracing_b200 as L
    one = _single(ctx, kind, spp, sq=True)
    g = Group(ctx, _devices(layout, n))
    world, cam = _world(kind)
    p = _params(spp, sq=True)
    p.shading_model = _model(kind)
    acc, sq = _accum(ctx, True)
    stats = g.multi.render(g.scenes(world.device_scene(ctx)), cam.to_struct(), p, acc.data_ptr(), sq.data_ptr(),
                           want_stats=True)
    assert [s.paths for s in stats] == [W * H * L.split_samples(spp, n, i)[1] for i in range(n)]
    a1, a2 = one.accum.cpu().numpy() / spp, acc.cpu().numpy() / spp
    q1, q2 = one.accum_sq.cpu().numpy() / spp, sq.cpu().numpy() / spp
    assert np.allclose(a2[:, :3], a1[:, :3], rtol=RTOL, atol=ATOL), float(np.abs(a2 - a1)[:, :3].max())
    assert np.allclose(q2[:, :3], q1[:, :3], rtol=RTOL, atol=ATOL), float(np.abs(q2 - q1)[:, :3].max())
    c1, c2 = one.accum[:, 3].cpu().numpy(), acc[:, 3].cpu().numpy()
    assert np.array_equal(c2, c1)   # channel 3: contributing paths, exact


# ---- 3. progressive, back to back -------------------------------------------------------------------------------------
@pytest.mark.parametrize("layout", LAYOUTS)
def test_back_to_back_passes_without_host_sync(ctx, layout):
    import learn_path_tracing_b200 as L
    one = _single(ctx, "v2", 24).mean()
    g = Group(ctx, _devices(layout, 3))
    world, cam = _world("v2")
    scenes = g.scenes(world.device_scene(ctx))
    acc, _ = _accum(ctx)
    for k in range(3):   # nothing waits on the host between the calls: the events order them
        g.multi.render(scenes, cam.to_struct(), _params(8, offset=8 * k), acc.data_ptr())
    got = ctx.download_accum(acc.data_ptr(), W, H) / 24
    assert np.allclose(got, one, rtol=RTOL, atol=ATOL), float(np.abs(got - one).max())


# ---- 4. statistics ----------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("layout", LAYOUTS)
def test_stats_per_member(ctx, layout):
    import learn_path_tracing_b200 as L
    n, spp = 3, 7
    g = Group(ctx, _devices(layout, n))
    world, cam = _world("v2")
    acc, _ = _accum(ctx)
    p = _params(spp)
    p.flags |= L.PT_FLAG_TIMING
    stats = g.multi.render(g.scenes(world.device_scene(ctx)), cam.to_struct(), p, acc.data_ptr(), want_stats=True)
    assert len(stats) == n
    for i, s in enumerate(stats):
        assert s.paths == W * H * L.split_samples(spp, n, i)[1] and s.segments >= s.paths and s.ms_total > 0
    assert sum(s.paths for s in stats) == W * H * spp


# ---- 5. refusals: PtError, nothing enqueued -----------------------------------------------------------------------------
@pytest.mark.parametrize("layout", LAYOUTS)
def test_refusals(ctx, layout):
    import torch
    import learn_path_tracing_b200 as L
    with pytest.raises(L.PtError):
        L._lib.Multi([])
    with pytest.raises(L.PtError):
        L._lib.Multi([ctx] * 17)
    with pytest.raises(L.PtError):
        L._lib.Multi([ctx, ctx])
    devs = _devices(layout, 2)
    g = Group(ctx, devs)
    world, cam = _world("v2")
    root = world.device_scene(ctx)
    good = g.scenes(root)
    acc, _ = _accum(ctx)
    unbuilt = L.Scene(g.members[1])
    unbuilt.set_spheres(*world.arrays())
    banded = _params(4)
    banded.reserved[4], banded.reserved[5] = 0, 10
    cases = [([root, root], _params(4), acc.data_ptr()),          # scenes[1] belongs to member 0
             ([root, unbuilt], _params(4), acc.data_ptr()),       # not built
             (good, banded, acc.data_ptr()),                      # row band
             (good, _params(4), torch.zeros((H * W, 4)).data_ptr())]  # host memory, not the root's device
    if _n_gpus() >= 2:
        other = torch.zeros((H * W, 4), dtype=torch.float32, device="cuda:1")
        cases.append((good, _params(4), other.data_ptr()))      # device memory of a non-root device
    for scenes, p, ptr in cases:
        with pytest.raises(L.PtError):
            g.multi.render(scenes, cam.to_struct(), p, ptr)
    for c in g.members:
        c.sync()
    assert not acc.any()   # nothing ran into the accumulator


# ---- 6. the Python surface ----------------------------------------------------------------------------------------------
@pytest.mark.parametrize("layout", LAYOUTS)
def test_render_and_legacy_renderer_with_devices(ctx, layout):
    import learn_path_tracing_b200 as L
    devs = _devices(layout, 3)
    world, cam = _world("v2")
    one = L.render(world, cam, spp=24, propagate_limit=DEPTH, seed=SEED, ctx=ctx, postprocess=False)
    multi = L.render(world, cam, spp=24, propagate_limit=DEPTH, seed=SEED, ctx=ctx, postprocess=False, devices=devs)
    assert np.allclose(multi, one, rtol=RTOL, atol=ATOL), float(np.abs(multi - one).max())
    world, cam = _world("legacy")
    a = L.legacy.LegacyRenderer(world, cam, spp=12, propagate_limit=DEPTH, seed=SEED, ctx=ctx, distributed=False)
    b = L.legacy.LegacyRenderer(world, cam, spp=12, propagate_limit=DEPTH, seed=SEED, ctx=ctx, devices=devs)
    for moved in (True, False):   # two progressive passes, split over the members
        fa, fb = a.render(moved=moved), b.render(moved=moved)
    assert b.total_spp == 24
    sa, sb = a.renderer.mean(), b.renderer.mean()
    assert np.allclose(sb, sa, rtol=RTOL, atol=ATOL), float(np.abs(sb - sa).max())
    assert np.allclose(fb, fa, rtol=2e-3, atol=2e-3, equal_nan=True)
    with pytest.raises(ValueError):
        L.MultiRenderer(W, H, [devs[0], 0], ctx).render(world.device_scene(ctx), cam.to_struct(), 1, 4,
                                                        L.PT_SHADE_LEGACY, rows=(0, 4))


# ---- 7. the drop-in shim ------------------------------------------------------------------------------------------------
def test_unmodified_10_final_script_on_several_devices(tmp_path, monkeypatch, ctx):
    """The unmodified 10_final driver with LPT_DEVICES set writes the PNG that L.render() writes on one device."""
    import learn_path_tracing_b200 as L
    from learn_path_tracing_b200 import scenes
    from test_shim_drop_in import _run
    monkeypatch.setenv("LPT_DEVICES", "0,1" if _n_gpus() >= 2 else "0,0")
    _run("10_final", tmp_path, monkeypatch, fake=False)
    png = L.imread(str(tmp_path / "outputs" / "10_final.png"))
    world, cam = scenes.scene_10_final((1280, 720))
    ref = L.to_uint8(L.render(world, cam, spp=8192, propagate_limit=32, ctx=ctx))
    d = L.to_uint8(png).astype(np.int32) - ref.astype(np.int32)
    assert np.abs(d).max() <= 1 and (d != 0).mean() < 1e-3, (np.abs(d).max(), (d != 0).mean())
