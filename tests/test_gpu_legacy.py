"""GPU parity of the legacy mesh/texture path (SURVEY 8a rows a9-a19) against the oracle, which walks the
reference's own SAH tree with the reference's triangle test and shades with the restated gen_secondary_rays."""
import numpy as np
import pytest

import learn_path_tracing_b200 as L
from helpers import all_triangles, mesh_camera, stand_in_world, synthetic_legacy_world

pytestmark = pytest.mark.gpu


def _rays_with_bounces(oracle, osc, cam, W, H, seed=3):
    rays = oracle.generate_rays(cam.to_struct(), W, H, 0, seed)
    ids, t = osc.trace(rays)
    hit = ids >= 0
    rng = np.random.default_rng(7)
    o = rays[hit, :3] + t[hit, None] * rays[hit, 4:7]
    d = rng.normal(size=o.shape).astype(np.float32)
    d /= np.linalg.norm(d, axis=1, keepdims=True)
    sec = np.zeros((o.shape[0], 8), np.float32)
    sec[:, :3], sec[:, 3], sec[:, 4:7], sec[:, 7] = o + 2e-4 * d, np.nextafter(np.float32(1e-4), np.float32(1)), d, np.inf
    rays[:, 3] = sec[0, 3] if len(sec) else rays[:, 3]   # legacy accepts t > epsilon (strict)
    return np.concatenate([rays, sec]).astype(np.float32)


def _tolerance(tris, tri_ids, rays, t):
    """|dt| bound for one (ray, triangle) pair: the contract's 1e-5 relative, plus the unavoidable rounding of f32
    coordinates (a few ulps of the scene scale) amplified by 1/|d.N| when the ray grazes the triangle's plane."""
    T = tris[np.maximum(tri_ids, 0)]
    n = np.cross(T[:, 3:6] - T[:, 0:3], T[:, 6:9] - T[:, 0:3])
    n /= np.linalg.norm(n, axis=1, keepdims=True)
    dn = np.abs((rays[:, 4:7] * n).sum(1))
    scale = np.maximum(np.abs(rays[:, :3]).max(1), np.abs(T).max(1))
    return 1e-5 * np.abs(t) + 16 * 1.2e-7 * scale / np.maximum(dn, 1e-12)


def _check_hits(oracle, world, gid, gt, oid, ot, rays, n_primary):
    """ids equal except ties and edge grazes (SURVEY appendix D); miss <=> miss up to grazing self-hits; primary
    (camera) rays: t within 1e-5 relative; secondary rays: 1e-5 relative + conditioning-aware rounding bound."""
    tris, off = all_triangles(world)
    agree = gid == oid
    hit = agree & (gid >= 0)
    prim = np.arange(len(rays)) < n_primary
    assert np.all(np.abs(gt[hit & prim] - ot[hit & prim]) <= 1e-5 * ot[hit & prim])
    th = hit & (gid >= off)
    tol = _tolerance(tris, (gid[th] - off).astype(np.int64), rays[th], ot[th])
    assert np.all(np.abs(gt[th] - ot[th]) <= tol)
    bad = np.flatnonzero(~agree)
    if len(bad):
        g_tri = np.where(gid[bad] >= off, gid[bad] - off, -1).astype(np.int32)
        o_tri = np.where(oid[bad] >= off, oid[bad] - off, -1).astype(np.int32)
        tg, wg = oracle.triangle_eval(tris, g_tri, rays[bad])   # reference plane-t and min barycentric of each side's triangle
        to, wo = oracle.triangle_eval(tris, o_tri, rays[bad])
        tol_g = np.where(g_tri >= 0, _tolerance(tris, g_tri, rays[bad], gt[bad]), 1e-6)
        tol_o = np.where(o_tri >= 0, _tolerance(tris, o_tri, rays[bad], ot[bad]), 1e-6)
        both = (gid[bad] >= 0) & (oid[bad] >= 0)
        tie = both & (np.abs(gt[bad] - ot[bad]) <= tol_g + tol_o)
        edge = ((g_tri >= 0) & (np.abs(wg) < 2e-4)) | ((o_tri >= 0) & (np.abs(wo) < 2e-4))
        # acceptance flips at t ~ epsilon: one side sees the (grazing) surface just above 1e-4, the other just below
        eps_flip = ((g_tri >= 0) & (np.abs(tg - 1e-4) <= tol_g + np.abs(gt[bad] - tg))) | \
                   ((o_tri >= 0) & (np.abs(to - 1e-4) <= tol_o))
        ok = tie | edge | eps_flip
        assert np.all(ok), (len(bad), int((~ok).sum()))
    return len(bad)


def test_synthetic_scene_hits_match_reference_traversal(ctx, oracle):
    world, cam = synthetic_legacy_world()
    W, H = 192, 128
    cam.resolution = (W, H)
    osc = oracle.scene_from_legacy_world(world, use_stored_tree=False)
    rays = _rays_with_bounces(oracle, osc, cam, W, H)
    oid, ot = osc.trace(rays)
    gid, gt = world.hit(rays, ctx)
    n_bad = _check_hits(oracle, world, gid, gt, oid, ot, rays, W * H)
    assert n_bad <= 5e-4 * len(rays) + 2
    sph = oid < 2
    assert sph.any() and np.array_equal(gt[sph & (gid == oid)], ot[sph & (gid == oid)])  # spheres: bit-exact t
    n_nodes, n_prims, n_global = world.device_scene(ctx).bvh_info()
    assert n_prims == 2 + 2 * 14 * 14 + 2 and n_global >= 2  # the +-50 ground triangles stay out of the LBVH


@pytest.mark.parametrize("name", ["demo", "yoimiya_ground_small", "zhongli_small", "ganyu_small"])
def test_cached_scene_hits_match_reference_traversal(ctx, oracle, name):
    world = stand_in_world(name)
    W, H = 240, 160
    cam = mesh_camera((W, H))
    if name == "demo":
        cam.set_position(L.legacy.Vec3f([3, 2, -6]))
        cam.look_at(L.legacy.Vec3f([0, 0, 0]))
    osc = oracle.scene_from_legacy_world(world, use_stored_tree=True)   # the reference's own traversal + tree
    rays = _rays_with_bounces(oracle, osc, cam, W, H)
    oid, ot = osc.trace(rays)
    gid, gt = world.hit(rays, ctx)
    assert (oid >= 0).mean() > 0.05
    n_bad = _check_hits(oracle, world, gid, gt, oid, ot, rays, W * H)
    # exact ties between duplicated faces resolve like the reference (device order = its visitation order): what is
    # left are near-ties between twin faces whose t differs in the last ulps
    assert n_bad <= 2e-3 * len(rays), n_bad


def _image_parity(ctx, oracle, world, cam, W, H, spp, depth, absorptivity, use_tree):
    r = L.Renderer(W, H, ctx, want_sq=True)
    st = r.render(world.device_scene(ctx), cam.to_struct(), spp, depth, L.PT_SHADE_LEGACY, seed=4,
                  absorptivity=absorptivity)
    s, q = r.moments()
    osum, osq, ost = oracle.render(oracle.scene_from_legacy_world(world, use_stored_tree=use_tree), cam.to_struct(), W, H,
                                   spp, depth, L.PT_SHADE_LEGACY, seed=4, absorptivity=absorptivity, want_sq=True)
    mu_g, mu_o = s / spp, osum / spp
    var = (np.maximum(q / spp - mu_g**2, 0) + np.maximum(osq / spp - mu_o**2, 0)) / spp
    z = np.abs(mu_g - mu_o) / np.sqrt(var + 1e-10)
    assert st.paths == ost.paths
    assert abs(st.segments / ost.segments - 1.0) < 0.01, (st.segments, ost.segments)
    assert (z > 3).mean() < 0.01, float((z > 3).mean())
    assert z.max() < 8.0, float(z.max())
    assert abs(mu_g.mean() / mu_o.mean() - 1.0) < 3e-3
    a = L.to_uint8(r.image(aces=False)).astype(np.float64)
    b = L.to_uint8(oracle.postprocess(osum, 1.0 / spp, aces=False)).astype(np.float64)
    return float(np.sqrt(((a - b) ** 2).mean()))


@pytest.mark.parametrize("absorptivity", [0.25, 0.5])
def test_synthetic_scene_image_within_3_sigma(ctx, oracle, absorptivity):
    world, cam = synthetic_legacy_world()
    rmse = _image_parity(ctx, oracle, world, cam, 96, 64, 192, 16, absorptivity, use_tree=False)
    assert rmse < 6.0


@pytest.mark.parametrize("name,spp", [("demo", 128), ("yoimiya_ground_small", 64), ("zhongli_small", 64), ("ganyu_small", 64)])
def test_cached_scene_image_within_3_sigma(ctx, oracle, name, spp):
    world = stand_in_world(name)
    W, H = 120, 80
    cam = mesh_camera((W, H))
    if name == "demo":
        cam.set_position(L.legacy.Vec3f([3, 2, -6]))
        cam.look_at(L.legacy.Vec3f([0, 0, 0]))
    rmse = _image_parity(ctx, oracle, world, cam, W, H, spp, 32, 0.25, use_tree=True)
    assert rmse < 8.0


def test_legacy_renderer_progressive(ctx):
    """render(moved=False) keeps accumulating (15_module.py:1022-1036); frame = (image / total spp)^(1/2.2)."""
    world, cam = synthetic_legacy_world()
    lr = L.legacy.LegacyRenderer(world, cam, spp=8, propagate_limit=8, ctx=ctx)
    f1 = lr.render(moved=True)
    f2 = lr.render(moved=False)
    assert lr.total_spp == 16 and f1.shape == (96, 64, 3)
    one = L.legacy.LegacyRenderer(world, cam, spp=16, propagate_limit=8, ctx=ctx).render()
    # bilinear's extrapolating taps (15_module.py:245-250) can give a negative environment value -> NaN after the
    # gamma power, in the reference as here
    assert np.allclose(f2, one, rtol=2e-3, atol=2e-3, equal_nan=True) and np.isnan(f2).mean() < 0.02
    assert not np.allclose(f1, f2)
    f3 = lr.render(moved=True)
    assert lr.total_spp == 8 and np.allclose(f3, f1, rtol=2e-3, atol=2e-3, equal_nan=True)


def test_gpu_built_trees_are_valid_reference_files(ctx, oracle, tmp_path):
    """SURVEY 8f-1: a world assembled from raw meshes is saved with trees from the GPU LBVH in the reference's schema;
    the oracle, walking the stored tree exactly like MeshBVHTree.hit, finds what a loop over all faces finds, and the
    reloaded world renders the same hits on the GPU."""
    from learn_path_tracing_b200 import legacy, worldnpy
    w, cam = synthetic_legacy_world(grid=40)      # 3200-face bumpy grid + ground quad + 2 spheres, no stored trees
    assert all(m["tree"] is None for m in w.meshes)
    rays = oracle.generate_rays(cam.to_struct(), 160, 90, 0, 3)
    ids0, t0 = w.hit(rays, ctx)
    fn = str(tmp_path / "gpu_tree.world.npy")
    w.save(fn, ctx=ctx)                              # builds the trees on the GPU
    assert all(m["tree"] is not None for m in w.meshes)
    big = w.meshes[0]["tree"]
    assert len(big["left"]) > 1000 and np.diff(big["leaf_cut"]).max() <= 4 and big["max_depth"] == 24
    d = worldnpy.load_world(fn)
    assert len(d["meshes_bvhs"]) == 2
    w2 = legacy.World()
    w2.load(fn, load_images=False)
    w2.set_atlas(*w._atlas)
    w2.set_environment_image(*w._env) if w._env is not None else None
    a_id, a_t = oracle.scene_from_legacy_world(w2, use_stored_tree=True).trace(rays)
    b_id, b_t = oracle.scene_from_legacy_world(w2, use_stored_tree=False).trace(rays)
    assert np.array_equal(a_t, b_t) and np.array_equal(a_id >= 0, b_id >= 0) and (a_id != b_id).mean() < 0.01
    ids2, t2 = w2.hit(rays, ctx)                     # faces were reordered to leaf order: compare geometry, not ids
    assert np.array_equal(t2, t0) and np.array_equal(ids2 >= 0, ids0 >= 0)
    assert (a_id >= 0).mean() > 0.5
