"""Closest hits of geometry far from the world origin (run on a B200 with `pytest -m gpu`).

Every other trace test keeps its geometry within a few units of the origin.  The slab tests of the tree walks compute
t = box * (1/d) - o * (1/d), whose rounding grows with |o|, the distance of the ray origin from the WORLD origin, not
with anything local to the ray.  These tests put tiled floors, a closed room, a bumpy grid and a quantised-node floor
up to 1e4 units away (along one axis, along all three, negative) and check every trace kernel against the float64
reference of tests/trace_ref.py, whose ambiguity bound is built from local quantities only, and the render kernels
through a room the camera cannot see out of.
"""
import numpy as np
import pytest

import learn_path_tracing_b200 as L
import trace_ref as R

pytestmark = pytest.mark.gpu

EXP = L._lib.has_experimental()
# the forms of test_trace_kernels_agree_bit_for_bit: one ray per thread, persistent sorted / in batch order / on float
# nodes, serve and fetch thresholds 1 and 32; and the 4-wide walk of `make EXPERIMENTAL=1` builds
DEVICE_FLAGS = (L.PT_FLAG_TRACE_SIMPLE, 0, L.PT_FLAG_NO_SORT, L.PT_FLAG_NO_QNODES, 1 << 8 | 1 << 14,
                32 << 8 | 32 << 14) + ((L.PT_FLAG_TRACE_WIDE,) if EXP else ())
OFFSETS = [(0.0, 0.0, 0.0)] + [v for s in (1e2, 1e3, 1e4) for v in ((s, 0.0, 0.0), (s, s, s), (-s, -s, -s))]
SORT_MIN = 65536        # pt_trace_batch_device sorts batches from this size on: batches on both sides of it
# edge grazes within the local bound: about 6 * bound of the rays that land on a triangle (three edges, density 2 of
# each barycentric near 0), at most ~1e-3 for the 1 cm tiles below
MAX_AMBIGUOUS = 2e-3


def _ids(o):
    return "x".join(f"{v:g}" for v in o)


def _scene(ctx, tris, monkeypatch):
    if EXP:
        monkeypatch.setenv("PT_WIDE", "1")   # the 4-wide copy of the tree for PT_FLAG_TRACE_WIDE
    sc = L.Scene(ctx)
    sc.set_triangles(tris)
    sc.build()
    n_nodes, n_prims, n_global = sc.bvh_info()
    assert n_prims == len(tris) and n_global == 0 and n_nodes == len(tris) - 1   # every tile in the tree
    return sc


def _trace_all(ctx, sc, rays):
    """(ids, t) of the batch; every device kernel form and host pt_trace_batch return the same records bit for bit."""
    import torch
    rd = torch.from_numpy(np.ascontiguousarray(rays, np.float32)).cuda()
    ref = None
    for flags in DEVICE_FLAGS:
        hits = torch.full((len(rays), 4), 7.0, dtype=torch.float32, device="cuda")
        ctx.trace_batch_device(sc, rd.data_ptr(), len(rays), hits.data_ptr(), flags)
        torch.cuda.synchronize()
        h = hits.cpu().numpy().view(np.int32)
        if ref is None:
            ref = h
        assert np.array_equal(h, ref), flags
    ids, t, _ = ctx.trace_batch(sc, rays)
    hit = ids >= 0
    assert np.array_equal(ids, ref[:, 1]) and np.array_equal(t[hit].view(np.int32), ref[hit, 0])
    return ids, t


def _check(name, tris, rays, ref, ids, t):
    m = R.compare(tris, rays, ref[0], ref[1], ids, t)
    n = len(rays)
    counts = {k: int(v.sum()) for k, v in m.items()}
    print(f"{name}: {n} rays, {int((ref[0] >= 0).sum())} reference hits, {counts}")
    assert counts["lost"] == 0 and counts["bad_t"] == 0 and counts["phantom"] == 0, (name, counts)
    assert counts["ambiguous"] <= MAX_AMBIGUOUS * n + 2, (name, counts)
    return m


def _batches(ctx, sc, name, tris, rays, ref):
    """the whole batch (sorted) and its first part (below the sort threshold) through every kernel form"""
    assert len(rays) > SORT_MIN
    for k in (len(rays), SORT_MIN // 3):
        ids, t = _trace_all(ctx, sc, rays[:k])
        _check(f"{name} [{k}]", tris, rays[:k], (ref[0][:k], ref[1][:k]), ids, t)


def _down_rays(rng, n, lo_u, lo_v, extent, offset, up):
    """Rays from 0.5-1 units above a y = offset.y floor (as secondary rays leave a surface), aimed at random floor
    points in [lo_u, lo_u + extent] x [lo_v, lo_v + extent] (u = z, v = x); 1/8 of them straight down with lateral
    components of exactly +0 and -0."""
    tgt = np.stack([lo_v + rng.random(n) * extent, np.full(n, float(offset[1])), lo_u + rng.random(n) * extent], 1)
    o = tgt + np.stack([rng.normal(size=n) * 0.3, up + rng.random(n) * up, rng.normal(size=n) * 0.3], 1)
    k = n // 8
    o[:k, 0], o[:k, 2] = tgt[:k, 0], tgt[:k, 2]
    rays = np.zeros((n, 8), np.float32)
    rays[:, :3], rays[:, 3], rays[:, 7] = o, 1e-4, np.inf
    d = tgt - rays[:, :3].astype(np.float64)
    rays[:, 4:7] = d / np.linalg.norm(d, axis=1, keepdims=True)
    rays[:k, 4:7] = [0.0, -1.0, 0.0]
    rays[:k:2, 4], rays[1:k:2, 6] = -0.0, -0.0
    return rays


def _no_edge_runs(rays, k, scene_ref):
    """Drops those of the first k (axis-parallel) rays that run exactly along a shared edge or a tile diagonal, which
    is common 1e4 units out where f32 steps are 1e-3: the strict inside test gives such a ray no triangle."""
    keep = np.ones(len(rays), bool)
    keep[:k] = scene_ref(rays[:k])[0] >= 0
    return rays[keep]


def _tmax_around_hit(rays, scene_ref, frac=0.125):
    """A share of the rays gets a finite tmax just before or just after its reference hit (1e-3 relative)."""
    ids, t, _ = scene_ref(rays)
    n = len(rays)
    sel = np.flatnonzero(ids >= 0)[: int(frac * n)]
    out = rays.copy()
    out[sel, 7] = t[sel] * np.where(np.arange(len(sel)) % 2, 1 + 1e-3, 1 - 1e-3)
    return out


@pytest.mark.parametrize("tile,count", [(0.01, 128), (0.1, 32)])
@pytest.mark.parametrize("offset", OFFSETS, ids=_ids)
def test_tiled_floor_far_from_origin(ctx, monkeypatch, offset, tile, count):
    floor = R.tiled_floor(offset, tile, count)
    tris = floor.triangles()
    sc = _scene(ctx, tris, monkeypatch)
    rng = np.random.default_rng(11)
    ext = tile * count
    rays = _no_edge_runs(_down_rays(rng, 70_000, offset[2], offset[0], ext, offset, 0.5), 70_000 // 8,
                         floor.closest_hit)
    rays = _tmax_around_hit(rays, floor.closest_hit)
    ref = floor.closest_hit(rays)
    assert (ref[0] >= 0).mean() > 0.85
    _batches(ctx, sc, f"floor {tile} m tiles at {offset}", tris, rays, ref)


def _room_rays(rng, n, offset, half):
    """Rays inside the closed room: from interior points in random and axis-parallel directions, and from points on
    the walls into the room (secondary rays)."""
    off = np.asarray(offset, np.float64)
    o = off + (rng.random((n, 3)) * 1.8 - 0.9) * half
    d = rng.normal(size=(n, 3))
    d /= np.linalg.norm(d, axis=1, keepdims=True)
    k = n // 8                                                 # axis-parallel, zeros of both signs
    ax = np.arange(k) % 3
    d[:k] = 0.0
    d[np.arange(k), ax] = np.where(np.arange(k) % 2, 1.0, -1.0)
    d[np.arange(0, k, 2), (ax[::2] + 1) % 3] = -0.0
    s = slice(k, 2 * k)                                        # from a wall point, into the room
    wall = rng.integers(0, 3, k)
    side = np.where(rng.random(k) < 0.5, -1.0, 1.0)
    ow = o[s]
    ow[np.arange(k), wall] = off[wall] + side * half
    o[s] = ow
    dw = d[s]
    dw[np.arange(k), wall] = -side * np.abs(dw[np.arange(k), wall])
    d[s] = dw
    rays = np.zeros((n, 8), np.float32)
    rays[:, :3], rays[:, 3], rays[:, 4:7], rays[:, 7] = o, 1e-4, d, np.inf
    return rays


@pytest.mark.parametrize("offset", OFFSETS, ids=_ids)
def test_closed_room_far_from_origin(ctx, monkeypatch, offset):
    """Every ray inside a closed room hits a wall."""
    half = 1.0
    room = R.closed_room(offset, half, 24)
    tris = room.triangles()
    sc = _scene(ctx, tris, monkeypatch)
    rays = _no_edge_runs(_room_rays(np.random.default_rng(5), 70_000, offset, half), 70_000 // 8, room.closest_hit)
    n_open = len(rays)
    rays = _tmax_around_hit(rays, room.closest_hit)
    ref = room.closest_hit(rays)
    closed = rays[:, 7] == np.inf
    assert closed.sum() > 0.8 * n_open
    for k in (len(rays), SORT_MIN // 3):
        ids, t = _trace_all(ctx, sc, rays[:k])
        m = _check(f"room at {offset} [{k}]", tris, rays[:k], (ref[0][:k], ref[1][:k]), ids, t)
        c = closed[:k]
        assert ((ids[c] >= 0) | m["ambiguous"][c]).all()
        assert ((ref[0][:k][c] >= 0) | m["ambiguous"][c]).all()


def _bumpy_grid(offset, n, size):
    """A tessellated height field, tilted about a skew axis: no triangle is axis-aligned."""
    xs, zs = np.meshgrid(np.linspace(-size, size, n + 1), np.linspace(-size, size, n + 1), indexing="ij")
    ys = 0.08 * np.sin(3.1 * xs) * np.cos(2.3 * zs) + 0.02 * np.cos(7.0 * xs + 1.0)
    p = np.stack([xs, ys, zs], -1)
    ax = np.array([1.0, 2.0, 3.0]) / np.sqrt(14.0)
    a = 0.6
    K = np.array([[0, -ax[2], ax[1]], [ax[2], 0, -ax[0]], [-ax[1], ax[0], 0]])
    rot = np.eye(3) + np.sin(a) * K + (1 - np.cos(a)) * K @ K
    p = (p @ rot.T + np.asarray(offset, np.float64)).astype(np.float32)
    i, j = np.meshgrid(np.arange(n), np.arange(n), indexing="ij")
    p00, p10, p11, p01 = p[i, j], p[i + 1, j], p[i + 1, j + 1], p[i, j + 1]
    tris = np.stack([np.concatenate([p00, p10, p11], -1), np.concatenate([p00, p11, p01], -1)], 2).reshape(-1, 9)
    return tris.astype(np.float32), rot


@pytest.mark.parametrize("offset", OFFSETS, ids=_ids)
def test_bumpy_grid_far_from_origin(ctx, monkeypatch, offset):
    tris, rot = _bumpy_grid(offset, 24, 0.6)
    sc = _scene(ctx, tris, monkeypatch)
    rng = np.random.default_rng(9)
    n = 8000
    v = tris.reshape(-1, 3, 3).astype(np.float64)
    w = rng.dirichlet((1, 1, 1), n)
    f = rng.integers(0, len(v), n)
    tgt = (w[:, :, None] * v[f]).sum(1)                       # points on the surface, float64
    up = rot[:, 1]
    o = tgt + (0.5 + 0.5 * rng.random(n))[:, None] * up + rng.normal(size=(n, 3)) * 0.2
    rays = np.zeros((n, 8), np.float32)
    rays[:, :3], rays[:, 3], rays[:, 7] = o, 1e-4, np.inf
    d = tgt - rays[:, :3].astype(np.float64)
    rays[:, 4:7] = d / np.linalg.norm(d, axis=1, keepdims=True)
    ref = R.brute_force(tris, rays)
    assert (ref[0] >= 0).mean() > 0.95
    ids, t = _trace_all(ctx, sc, rays)
    _check(f"bumpy grid at {offset}", tris, rays, ref, ids, t)


@pytest.mark.parametrize("offset", [(0.0, 0.0, 0.0), (1e3, 0.0, 0.0), (1e4, 1e4, 1e4), (-1e4, -1e4, -1e4)], ids=_ids)
def test_quantised_floor_far_from_origin(ctx, monkeypatch, offset):
    """2 x 363 x 363 triangles: a tree of >= 2^18 nodes, which gets the quantised copy the persistent walk uses (and
    PT_FLAG_NO_QNODES skips)."""
    floor = R.tiled_floor(offset, 0.01, 363)
    tris = floor.triangles()
    sc = _scene(ctx, tris, monkeypatch)
    assert sc.bvh_info()[0] >= 1 << 18
    rays = _no_edge_runs(_down_rays(np.random.default_rng(4), 70_000, offset[2], offset[0], 3.63, offset, 0.5),
                         70_000 // 8, floor.closest_hit)
    rays = _tmax_around_hit(rays, floor.closest_hit)
    ref = floor.closest_hit(rays)
    assert (ref[0] >= 0).mean() > 0.85
    _batches(ctx, sc, f"quantised floor at {offset}", tris, rays, ref)


def test_sphere_scene_translated_is_bit_exact(ctx, monkeypatch, oracle):
    """10_final moved to (1e3, 0, 1e3): the oracle's tree-less loop in the kernel's own f32 arithmetic gives the ids and
    t every kernel form must return exactly."""
    from learn_path_tracing_b200 import scenes
    from test_gpu_parity import _secondary_rays
    W, H = 256, 144
    world, cam = scenes.SCENES["10_final"]((W, H))
    rays = _secondary_rays(oracle, world, cam, W, H)
    cr, mats = world.arrays()
    shift = np.array([1e3, 0.0, 1e3], np.float32)
    cr = cr.copy()
    cr[:, :3] += shift
    rays[:, :3] += shift
    if EXP:
        monkeypatch.setenv("PT_WIDE", "1")
    sc = L.Scene(ctx)
    sc.set_spheres(cr, mats)
    sc.build()
    assert sc.bvh_info()[2] == 1                       # only the ground sphere is global
    oid, ot = oracle.trace_spheres(cr, mats, rays)
    ids, t = _trace_all(ctx, sc, rays)
    assert np.array_equal(ids, oid) and np.array_equal(t, ot)
    assert (oid >= 1).mean() > 0.1 and (oid < 0).any()


# ---- render kernels: a camera inside a closed room far from the origin never sees the environment --------------------
def _room_world(offset, half, count):
    from learn_path_tracing_b200 import legacy
    room = R.closed_room(offset, half, count)
    tris = room.triangles()
    pos = tris.reshape(-1, 3)
    nrm = np.zeros((1, 3), np.float32)
    nrm[0, 1] = 1.0
    uv = np.zeros((1, 2), np.float32)
    k = np.arange(len(tris)) * 3
    z = np.zeros_like(k)
    faces = np.stack([k, z, z, k + 1, z, z, k + 2, z, z, z], 1).astype(np.int32)
    w = legacy.World()
    w.add_mesh(pos, nrm, uv, faces)
    tex = np.full((1, 1, 8), 128, np.uint8)
    w.set_atlas(tex, [[0, 0, 1, 1]], [1])
    w.set_environment(0)
    w.set_environment_image(np.full((4, 4, 3), 0.7, np.float32), [0, 0, 4, 4])
    cam = legacy.Camera((96, 64))
    cam.set_fov(40)
    off = np.asarray(offset, np.float64)
    cam.set_position(legacy.Vec3f(list(off + [0.2, 0.1, -0.5])))
    cam.look_at(legacy.Vec3f(list(off + [0.4, -0.2, 1.0])))
    return w, cam, room, tris


def test_render_kernels_inside_a_far_room(ctx):
    """max_depth = 1: a camera ray that hits adds nothing (the scatter raises the bounce to the limit and the path ends,
    persist.cu / wavefront.cu), a miss adds (environment, 1).  So accum.w counts the camera rays that escaped the room;
    it is at most the number of camera rays the reference calls ambiguous.  The features report a hit per sample."""
    W, H, SPP, SEED = 96, 64, 8, 3
    offset = (1e3, 1e3, 1e3)
    world, cam, room, tris = _room_world(offset, 1.0, 16)
    sc = world.device_scene(ctx)
    assert sc.bvh_info()[2] == 0
    cs = cam.to_struct()
    amb = 0
    for s in range(SPP):
        rays = ctx.generate_rays(cs, W, H, s, SEED)
        rays[:, 3] = np.nextafter(np.float32(1e-4), np.float32(1))   # the legacy render's hit rule: t > eps
        rid, rt, _ = room.closest_hit(rays)
        m = R.compare(tris, rays, rid, rt, rid, rt)
        amb += int((m["ambiguous"] | (rid < 0)).sum())
    assert amb <= MAX_AMBIGUOUS * W * H * SPP
    modes = [L.PT_MODE_SPLIT, L.PT_MODE_FUSED, L.PT_MODE_PERSIST, L.PT_MODE_AUTO] + \
        ([L.PT_MODE_QUEUE, L.PT_MODE_DUAL] if EXP else [])
    for mode in modes:
        r = L.Renderer(W, H, ctx)
        st = r.render(sc, cs, SPP, 1, L.PT_SHADE_LEGACY, seed=SEED, mode=mode)
        escaped = float(r.accum[:, 3].sum())
        print(f"render mode {mode}, room at {offset}: {escaped:g} of {W * H * SPP} camera rays escaped, {amb} ambiguous")
        assert st.paths == W * H * SPP
        assert escaped <= amb, (mode, escaped, amb)
    f = L.Renderer(W, H, ctx).features(sc, cs, SPP, SEED, 0, 0, L.PT_SHADE_LEGACY)
    hits = f[1, :, 3].cpu().numpy()
    assert (SPP - hits).sum() <= amb and (hits <= SPP).all()
