"""GPU tests at BASELINE.json's FULL sizes, every config by name: configs[0] 10_final 1280x720, configs[1] 8_refract
1080p/256 spp, configs[2] Yoimiya 1080p with the full 2048^2-per-map atlas, configs[3] Zhongli / Ganyu at 3840x2160,
configs[4] 10 M triangles / 64 Mi rays (the mesh configs through the seeded stand-ins of tests/helpers.py:STAND_INS, whose
map sizes and resolutions are the configs' own).  The image of every render config is compared with the CPU oracle at the bench
resolution (at a sample count the oracle finishes in seconds: per-pixel 3 sigma where the count allows it, 8x8-block
3 sigma for the 2-8 spp mesh renders); the full sample counts are covered by size-independent properties — the union
of sample ranges equals one render, every kernel form traces the same paths, hit records are self-consistent."""
import os

import numpy as np
import pytest

import learn_path_tracing_b200 as L
from learn_path_tracing_b200 import scenes
from helpers import hit_tolerance, mesh_camera, stand_in_world

pytestmark = pytest.mark.gpu


def _block_z(s, q, osum, osq, n, B=8):
    """z-scores of BxB-block means (few samples per pixel: per-pixel variances are too noisy, block ones are not)."""
    W, H = (s.shape[0] // B) * B, (s.shape[1] // B) * B

    def blocks(a):
        return a[:W, :H].reshape(W // B, B, H // B, B, 3).mean(axis=(1, 3))
    mu_g, mu_o = s / n, osum / n
    var_g = np.maximum(q / n - mu_g**2, 0) / max(n - 1, 1)   # variance of a pixel mean (unbiased)
    var_o = np.maximum(osq / n - mu_o**2, 0) / max(n - 1, 1)
    vb = (blocks(var_g) + blocks(var_o)) / (B * B)
    return np.abs(blocks(mu_g) - blocks(mu_o)) / np.sqrt(vb + 1e-10), mu_g, mu_o


def test_config0_10_final_720p_image_within_3_sigma_of_oracle(ctx, oracle):
    """configs[0] at the script's resolution and depth (1280x720, depth 32; 32 of the 8192 spp — the oracle's brute-force
    sphere loop needs ~0.5 s per sample on 16 cores): 486 spheres through the GPU LBVH against the reference's loop."""
    W, H, SPP, DEPTH = 1280, 720, 32, 32
    world, cam = scenes.scene_10_final((W, H))
    r = L.Renderer(W, H, ctx, want_sq=True)
    st = r.render(world.device_scene(ctx), cam.to_struct(), SPP, DEPTH, L.PT_SHADE_V2, seed=1)
    s, q = r.moments()
    osum, osq, ost = oracle.render(oracle.scene_from_world(world), cam.to_struct(), W, H, SPP, DEPTH, L.PT_SHADE_V2, seed=1,
                                   want_sq=True)
    z, mu_g, mu_o = _block_z(s, q, osum, osq, SPP, B=4)
    assert st.paths == ost.paths == W * H * SPP
    assert abs(st.segments / ost.segments - 1.0) < 2e-3, (st.segments, ost.segments)
    assert (z > 3).mean() < 0.008, (z > 3).mean()
    assert z.max() < 7.0, z.max()
    assert abs(mu_g.mean() / mu_o.mean() - 1.0) < 1e-3
    print(f"config0 1280x720: {(z > 3).mean()*100:.3f}% of 4x4 blocks beyond 3 sigma, max z {z.max():.2f}, {st.ms_total:.1f} ms GPU")


def _legacy_fullsize_parity(ctx, oracle, cache, W, H, spp, max_frac):
    world = stand_in_world(cache)
    cam = mesh_camera((W, H))
    r = L.Renderer(W, H, ctx, want_sq=True)
    st = r.render(world.device_scene(ctx), cam.to_struct(), spp, 32, L.PT_SHADE_LEGACY, seed=1)
    s, q = r.moments()
    osum, osq, ost = oracle.render(oracle.scene_from_legacy_world(world, use_stored_tree=True), cam.to_struct(), W, H, spp, 32,
                                   L.PT_SHADE_LEGACY, seed=1, want_sq=True)
    z, mu_g, mu_o = _block_z(s, q, osum, osq, spp, B=8)
    assert st.paths == ost.paths == W * H * spp
    assert abs(st.segments / ost.segments - 1.0) < 5e-3, (st.segments, ost.segments)
    assert (z > 3).mean() < max_frac, (z > 3).mean()
    assert abs(mu_g.mean() / mu_o.mean() - 1.0) < 2e-3, mu_g.mean() / mu_o.mean()
    a = L.to_uint8(r.image(aces=False)).astype(np.float64)
    b = L.to_uint8(oracle.postprocess(osum, 1.0 / spp, aces=False)).astype(np.float64)
    # 8x8 box means of the two 8-bit frames (independent low-spp estimates: per-pixel noise dominates a plain RMSE)
    A, B = a.shape[0] // 8 * 8, a.shape[1] // 8 * 8
    da = (a - b)[:A, :B].reshape(A // 8, 8, B // 8, 8, 3).mean(axis=(1, 3))
    print(f"{cache} {W}x{H} {spp} spp: {(z > 3).mean()*100:.3f}% of 8x8 blocks beyond 3 sigma, max z {z.max():.2f}, "
          f"box RMSE {np.sqrt((da**2).mean()):.2f}/255, segments GPU/oracle {st.segments / ost.segments:.5f}, {st.ms_total:.1f} ms GPU")
    assert np.sqrt((da**2).mean()) < 6.0


def test_config2_yoimiya_1080p_full_atlas_image_within_3_sigma_of_oracle(ctx, oracle):
    """configs[2] at bench settings — 1920x1080, 2048^2 per map, sky environment, depth 32 — at 8 of the 512 spp, on
    the Yoimiya stand-in: the GPU LBVH + Moller-Trumbore + LUT-decoded 8-bit atlas against the oracle walking the stored
    tree with the reference triangle test and float texels."""
    _legacy_fullsize_parity(ctx, oracle, "yoimiya_ground_full", 1920, 1080, 8, 0.01)


@pytest.mark.parametrize("cache", ["zhongli_full", "ganyu_full"])
def test_config3_4k_mesh_scene_image_within_3_sigma_of_oracle(ctx, oracle, cache):
    """configs[3] at bench resolution (3840x2160, depth 32) at 2 of the 4096 spp, the stand-ins of both models."""
    _legacy_fullsize_parity(ctx, oracle, cache, 3840, 2160, 2, 0.012)


def test_config1_8_refract_1080p_256spp_within_3_sigma_of_oracle(ctx, oracle):
    """configs[1] exactly as benchmarked: 1920x1080, 256 spp, depth 50, default (persistent) kernel vs the CPU oracle."""
    W, H, SPP, DEPTH = 1920, 1080, 256, 50
    world, cam = scenes.scene_8_refract((W, H))
    r = L.Renderer(W, H, ctx, want_sq=True)
    st = r.render(world.device_scene(ctx), cam.to_struct(), SPP, DEPTH, L.PT_SHADE_V2, seed=1)
    s, q = r.moments()
    osum, osq, ost = oracle.render(oracle.scene_from_world(world), cam.to_struct(), W, H, SPP, DEPTH, L.PT_SHADE_V2, seed=1,
                                   want_sq=True)
    mu_g, mu_o = s / SPP, osum / SPP
    var_g = np.maximum(q / SPP - mu_g**2, 0) / SPP
    var_o = np.maximum(osq / SPP - mu_o**2, 0) / SPP
    z = np.abs(mu_g - mu_o) / np.sqrt(var_g + var_o + 1e-12)
    assert st.paths == ost.paths == W * H * SPP
    assert abs(st.segments / ost.segments - 1.0) < 2e-3
    assert (z > 3).mean() < 0.006, (z > 3).mean()   # 0.27 % expected by chance
    assert abs(mu_g.mean() / mu_o.mean() - 1.0) < 5e-4
    a = L.to_uint8(r.image()).astype(np.float64)
    b = L.to_uint8(oracle.postprocess(osum, 1.0 / SPP)).astype(np.float64)
    rmse = np.sqrt(((a - b) ** 2).mean())
    assert rmse < 3.0, rmse   # 8-bit levels, two independent 256-spp estimates
    print(f"config1 full size: {(z > 3).mean()*100:.3f}% of pixel-channels beyond 3 sigma, RMSE {rmse:.2f}/255, "
          f"{st.ms_total:.1f} ms GPU")


@pytest.mark.parametrize("name,bsdf", [("6_diffuse", "DiffuseBSDF"), ("7_reflect", "DielectricBSDF"),
                                       ("8_refract", "DielectricBSDF"), ("9_dof", "DielectricBSDF")])
def test_converged_render_matches_the_reference_own_8192spp_png(ctx, name, bsdf):
    """The reference's committed outputs/<stage>.png ARE its converged renders (1280x720, 8192 spp, depth 32, ACES +
    gamma, truncating 8-bit cast).  The same script settings through the drop-in surface on the GPU, quantised the same
    way and box-filtered 4x4 like the golden (tests/golden/make_goldens.py), must land on it: two independent 8192-spp
    estimates, so what is left is Monte Carlo + quantisation noise averaged over 16 pixels."""
    from PIL import Image
    from conftest import GOLDEN
    W, H, SPP = 1280, 720, 8192
    world, cam = scenes.SCENES[name]((W, H))
    img, st = L.render(world, cam, spp=SPP, propagate_limit=32, bsdf=getattr(L, bsdf), ctx=ctx, return_stats=True)
    assert st.paths == W * H * SPP
    a = L.to_uint8(img).astype(np.float64).reshape(H // 4, 4, W // 4, 4, 3).mean(axis=(1, 3))
    gold = np.asarray(Image.open(os.path.join(GOLDEN, f"{name}_320x180.png")).convert("RGB"), np.float64)
    d = a - gold   # the golden is the 4x4 mean ROUNDED to 8 bit: +-0.29 levels of its own
    rmse, bias = float(np.sqrt((d**2).mean())), float(d.mean())
    print(f"{name}: GPU 8192 spp vs reference PNG (4x4 box): rmse {rmse:.3f}/255, bias {bias:+.3f}, max {np.abs(d).max():.2f}, "
          f"{st.ms_total:.0f} ms")
    # measured on B200: rmse 0.21-0.29 (the golden's own rounding is 0.29), |bias| <= 0.003, max 1.25-1.75
    assert rmse < 0.4, rmse
    assert abs(bias) < 0.05, bias
    assert np.abs(d).max() < 3.5, np.abs(d).max()


def test_config1_kernel_forms_and_sample_split_agree_at_full_size(ctx):
    """1920x1080: persistent, K-step fused and split wavefronts trace the same paths; 2 x 128 spp == 256 spp."""
    W, H, DEPTH = 1920, 1080, 50
    world, cam = scenes.scene_8_refract((W, H))
    sc = world.device_scene(ctx)
    ref = None
    for mode in [L.PT_MODE_PERSIST, L.PT_MODE_FUSED, L.PT_MODE_SPLIT] + ([L.PT_MODE_DUAL] if L._lib.has_experimental() else []):
        r = L.Renderer(W, H, ctx)
        st = r.render(sc, cam.to_struct(), 32, DEPTH, seed=9, mode=mode)
        m = r.mean()
        if ref is None:
            ref, seg = m, int(st.segments)
        assert abs(int(st.segments) - seg) <= 2e-4 * seg
        assert np.allclose(m, ref, rtol=2e-3, atol=2e-4)
    one = L.Renderer(W, H, ctx)
    one.render(sc, cam.to_struct(), 256, DEPTH, seed=1)
    two = L.Renderer(W, H, ctx)
    two.render(sc, cam.to_struct(), 128, DEPTH, seed=1, spp_offset=0)
    two.render(sc, cam.to_struct(), 128, DEPTH, seed=1, spp_offset=128)
    assert two.spp_done == 256
    assert np.allclose(one.mean(), two.mean(), rtol=1e-4, atol=1e-5)


def test_config2_yoimiya_1080p_512spp_properties(ctx):
    """configs[2] at full size: sample ranges are additive, the persistent and split kernels agree, every path
    is accounted for (the accumulator's 4th channel counts contributing paths)."""
    W, H, SPP, DEPTH = 1920, 1080, 512, 32
    world = stand_in_world("yoimiya_ground_full")
    cam = mesh_camera((W, H))
    sc = world.device_scene(ctx)
    full = L.Renderer(W, H, ctx)
    st = full.render(sc, cam.to_struct(), SPP, DEPTH, L.PT_SHADE_LEGACY, seed=1)
    assert st.paths == W * H * SPP and st.segments > st.paths
    acc = full.accum.cpu().numpy()
    assert np.isfinite(acc).all() and (acc[:, :3] >= 0).all()
    assert acc[:, 3].max() <= SPP and acc[:, 3].mean() > 0.9 * SPP   # paths that never reach the sky add nothing
    parts = L.Renderer(W, H, ctx)
    for k in range(4):
        parts.render(sc, cam.to_struct(), SPP // 4, DEPTH, L.PT_SHADE_LEGACY, seed=1, spp_offset=k * (SPP // 4))
    assert np.allclose(parts.accum.cpu().numpy(), acc, rtol=2e-4, atol=2e-3)
    a = L.Renderer(W, H, ctx)
    sa = a.render(sc, cam.to_struct(), 16, DEPTH, L.PT_SHADE_LEGACY, seed=3, mode=L.PT_MODE_PERSIST)
    b = L.Renderer(W, H, ctx)
    sb = b.render(sc, cam.to_struct(), 16, DEPTH, L.PT_SHADE_LEGACY, seed=3, mode=L.PT_MODE_SPLIT)
    assert abs(int(sa.segments) - int(sb.segments)) <= 2e-4 * sb.segments
    assert np.allclose(a.mean(), b.mean(), rtol=2e-3, atol=2e-4)
    for bps in ((3, 4) if L._lib.has_experimental() else ()):   # the two-records-per-lane kernel at 3 and 4 blocks per SM
        c = L.Renderer(W, H, ctx)
        sc_ = c.render(sc, cam.to_struct(), 16, DEPTH, L.PT_SHADE_LEGACY, seed=3, mode=L.PT_MODE_DUAL, segments_per_launch=bps)
        assert abs(int(sc_.segments) - int(sb.segments)) <= 2e-4 * sb.segments
        assert np.allclose(c.mean(), b.mean(), rtol=2e-3, atol=2e-4)


def test_config4_10m_triangles_64m_rays(ctx, oracle):
    """configs[4] at full size: the three trace kernels agree bit for bit on all 64 Mi rays; hit records are
    self-consistent; a 2^22-ray sample equals the oracle walking the same GPU-built LBVH (ties/edge grazes aside)."""
    import torch
    n_tri, n_rays = 10_000_000, 64 * 2**20
    sc = L.Scene(ctx)
    sc.set_random_triangles(n_tri, 12345, 0.004)
    sc.build()
    rays = torch.empty((2 * n_rays, 4), dtype=torch.float32, device="cuda")
    ctx.random_rays_device(rays.data_ptr(), n_rays, 54321)
    ref = None
    for flags in (0, L.PT_FLAG_NO_SORT, L.PT_FLAG_TRACE_SIMPLE):
        hits = torch.full((n_rays, 4), 7.0, dtype=torch.float32, device="cuda")
        ctx.trace_batch_device(sc, rays.data_ptr(), n_rays, hits.data_ptr(), flags)
        torch.cuda.synchronize()
        if ref is None:
            ref = hits
        else:
            assert torch.equal(hits.view(torch.int32), ref.view(torch.int32)), flags
        del hits
    t, prim = ref[:, 0], ref.view(torch.int32)[:, 1]
    hit = prim >= 0
    assert 0.3 < float(hit.float().mean()) < 0.999
    assert bool((prim[hit] < n_tri).all()) and bool((t[hit] >= 1e-4).all()) and bool((t[~hit] == -1).all())
    uv = ref[:, 2:4][hit]
    assert bool((uv > 0).all()) and bool(((1.0 - uv[:, 0] - uv[:, 1]) > 0).all())   # barycentrics strictly inside (extend.cuh)
    n_c = 2**22   # 6 % of the batch: ~2 s of oracle on 16 cores
    tris = oracle.random_triangles(n_tri, 12345, 0.004)
    nodes, _ = sc.bvh_download()
    r_h = rays[:2 * n_c].cpu().numpy().reshape(n_c, 8)
    oid, ot, _ = oracle.trace_bvh2(nodes, tris, r_h)
    gid = prim[:n_c].cpu().numpy()
    gt = t[:n_c].cpu().numpy()
    agree = gid == oid
    assert agree.mean() > 0.9995, agree.mean()
    both = agree & (oid >= 0)
    # t: 1e-5 relative for all but grazing rays (Moller-Trumbore vs the reference's plane formula on 0.004-sized
    # triangles); those stay within the conditioning-aware bound of tests/helpers.py:hit_tolerance
    dt = np.abs(gt[both] - ot[both])
    assert (dt <= 1e-5 * ot[both]).mean() > 0.999
    assert np.all(dt <= hit_tolerance(tris, gid[both].astype(np.int64), r_h[both], ot[both]))
    bad = np.flatnonzero(~agree)
    if len(bad):  # ties or edge grazes only
        tg, wg = oracle.triangle_eval(tris, gid[bad].astype(np.int32), r_h[bad])
        to, wo = oracle.triangle_eval(tris, oid[bad].astype(np.int32), r_h[bad])
        tie = (gid[bad] >= 0) & (oid[bad] >= 0) & (np.abs(gt[bad] - ot[bad]) <= 1e-5 * np.abs(ot[bad]))

        def grazing(ids):
            """|d.N| of the ray against the plane of triangle `ids` (1 where there is no triangle)."""
            T = tris[np.maximum(ids, 0)]
            n = np.cross(T[:, 3:6] - T[:, 0:3], T[:, 6:9] - T[:, 0:3])
            n /= np.linalg.norm(n, axis=1, keepdims=True)
            return np.where(ids >= 0, np.abs((r_h[bad][:, 4:7] * n).sum(1)), 1.0)
        # barycentrics of a 0.004-sized triangle at coordinates ~1.5 carry ~16 ulp * 1.5 / 0.004 = 7e-4 of rounding, times
        # 1 / |d.N| when the ray grazes the triangle's plane (the hit point moves along the ray by ulp(t) / |d.N|): the
        # 2^22-ray sample contains rays within 0.3 degrees of a plane, the 2^16-ray sample of round 1 did not
        dn_g, dn_o = grazing(gid[bad].astype(np.int64)), grazing(oid[bad].astype(np.int64))
        edge = ((gid[bad] >= 0) & (np.abs(wg) < 2e-3 + 1e-3 / np.maximum(dn_g, 1e-9))) | \
               ((oid[bad] >= 0) & (np.abs(wo) < 2e-3 + 1e-3 / np.maximum(dn_o, 1e-9)))
        rest = ~(tie | edge)
        assert not rest.any(), (int(rest.sum()), gid[bad][rest], oid[bad][rest], gt[bad][rest], ot[bad][rest], wg[rest], wo[rest],
                                dn_g[rest], dn_o[rest])
        print(f"config4: {len(bad)} of {n_c} sampled rays differ from the oracle: {int(tie.sum())} ties, {int((edge & ~tie).sum())} edge / plane grazes "
              f"(smallest |d.N| {min(dn_g.min(), dn_o.min()):.2e})")
