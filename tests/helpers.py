"""Shared builders for the legacy-path tests."""
import functools
import os

import numpy as np

from learn_path_tracing_b200 import legacy

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CACHE = os.path.join(ROOT, "scenes_cache")


def synthetic_legacy_world(seed=0, grid=14):
    """A small self-contained legacy scene: bumpy textured grid mesh (uv tiled beyond [0,1]), a +-50 ground plane
    (becomes 'global' primitives), two textured spheres (one transparent, with a normal map), a 3-area atlas with a
    non-square area (exercises bilinear's wrap-with-width quirk) and a non-square environment area."""
    rng = np.random.default_rng(seed)
    n = grid + 1
    xs, zs = np.meshgrid(np.linspace(-2, 2, n), np.linspace(-2, 2, n), indexing="ij")
    ys = 0.6 + 0.25 * np.sin(2.1 * xs) * np.cos(1.7 * zs) + 0.03 * rng.standard_normal(xs.shape)
    pos = np.stack([xs, ys, zs], -1).reshape(-1, 3).astype(np.float32)
    nrm = np.zeros_like(pos)
    nrm[:, 1] = 1.0
    nrm[:, 0] = -0.25 * 2.1 * np.cos(2.1 * xs).ravel() * np.cos(1.7 * zs).ravel()
    nrm[:, 2] = 0.25 * 1.7 * np.sin(2.1 * xs).ravel() * np.sin(1.7 * zs).ravel()
    nrm /= np.linalg.norm(nrm, axis=1, keepdims=True)
    uv = (np.stack([xs, zs], -1).reshape(-1, 2) * 0.8 + 0.3).astype(np.float32)  # spans about [-1.3, 1.9]: wraps
    faces = []
    for i in range(grid):
        for j in range(grid):
            a, b, c, d = i * n + j, (i + 1) * n + j, (i + 1) * n + j + 1, i * n + j + 1
            tid = (i + j) % 2
            faces.append([a, a, a, b, b, b, c, c, c, tid])
            faces.append([a, a, a, c, c, c, d, d, d, tid])
    w = legacy.World()
    w.add_mesh(pos, nrm, uv, np.array(faces, np.int32))
    gp = np.array([[50, 0, -50], [-50, 0, -50], [-50, 0, 50], [50, 0, 50]], np.float32)
    gn = np.array([[0, 1, 0]], np.float32)
    gt = np.array([[0, 0], [10, 0], [10, 10], [0, 10]], np.float32)
    w.add_mesh(gp, gn, gt, np.array([[0, 0, 0, 1, 0, 1, 2, 0, 2, 1], [0, 0, 0, 2, 0, 2, 3, 0, 3, 1]], np.int32))
    w.add_sphere(legacy.Sphere([-1.2, 1.6, 0.3], 0.6, 0, 2))
    w.add_sphere(legacy.Sphere([1.3, 1.5, -0.4], 0.5, 1, 2))
    tex = rng.integers(0, 256, size=(160, 64, 8), dtype=np.uint8)
    tex[:, :, 3] = rng.integers(0, 256, size=(160, 64)) // 2 + 64   # roughness
    tex[:, :, 7] = np.where(rng.random((160, 64)) < 0.3, rng.integers(0, 256, size=(160, 64)), 0)  # metallic
    tex[:, :, 4:6] = 128 + rng.integers(-40, 40, size=(160, 64, 2))
    tex[:, :, 6] = 230
    areas = [[0, 0, 64, 64], [64, 0, 96, 64], [96, 0, 160, 32]]
    w.set_atlas(tex, areas, [1, 1, 0])
    ex, ey = np.meshgrid(np.linspace(0, 1, 64), np.linspace(0, 1, 32), indexing="ij")
    env = np.zeros((64, 64, 3), np.float32)
    env[:, :32, 0] = 0.4 + 0.6 * ey
    env[:, :32, 1] = 0.5 + 0.4 * np.sin(6.28 * ex) ** 2
    env[:, :32, 2] = 0.9
    w.set_environment(0)
    w.set_environment_image(env, [0, 0, 64, 32])
    cam = legacy.Camera((96, 64))
    cam.set_fov(22)
    cam.set_position(legacy.Vec3f([0.5, 2.6, -7.0]))
    cam.look_at(legacy.Vec3f([0, 1.0, 0]))
    cam.set_len(7.0, 0.05)
    return w, cam


def all_triangles(world):
    """tris9 [F,9] of every mesh face in primitive order, and the primitive-id offset of triangles."""
    tris = []
    for m in world.meshes:
        f = m["indices"]
        p = m["positions"]
        tris.append(np.concatenate([p[f[:, 0]], p[f[:, 3]], p[f[:, 6]]], axis=1))
    return np.concatenate(tris).astype(np.float32), len(world.spheres)


def cached_world(name):
    from learn_path_tracing_b200 import scene_cache
    path = os.path.join(CACHE, name + ".npz")
    if not os.path.exists(path):
        return None
    return scene_cache.load_cache(path)


def median_split_nodes(tri9):
    """A binary tree over the faces in the node layout of Scene.bvh_download() ([n-1,16]: left box, right box, two child
    refs; a ref >= 0 is a node, ~f is face f), built on the host: faces sorted by the Morton code of their box centre,
    every range split at its middle, one level at a time."""
    n = len(tri9)
    v = np.asarray(tri9, np.float32).reshape(-1, 3, 3)
    plo, phi = v.min(1), v.max(1)
    c = (plo + phi) / 2
    q = ((c - c.min(0)) / np.maximum(c.max(0) - c.min(0), 1e-12) * 1023).astype(np.int64)
    code = np.zeros(n, np.int64)
    for bit in range(10):
        for axis in range(3):
            code |= ((q[:, axis] >> bit) & 1) << (3 * bit + 2 - axis)
    order = np.argsort(code, kind="stable")
    lo, hi = plo[order], phi[order]
    nodes = np.zeros((max(n - 1, 0), 16), np.float32)
    a, b, ids, nxt = np.array([0]), np.array([n]), np.array([0]), 1   # face ranges of one level's nodes
    while n > 1 and len(a):
        m = (a + b) // 2
        cuts = np.unique(np.concatenate([a, m, b]))
        cuts = cuts[cuts < n]                     # ranges are disjoint: [s, e) is one segment between the cuts
        seg_lo, seg_hi = np.minimum.reduceat(lo, cuts), np.maximum.reduceat(hi, cuts)
        na, nb, nids = [], [], []
        for side, (s, e) in enumerate(((a, m), (m, b))):
            k = np.searchsorted(cuts, s)
            nodes[ids, 6 * side:6 * side + 3], nodes[ids, 6 * side + 3:6 * side + 6] = seg_lo[k], seg_hi[k]
            inner = e - s > 1
            ref = np.where(inner, 0, ~order[s]).astype(np.int32)
            ref[inner] = nxt + np.arange(inner.sum())
            nxt += int(inner.sum())
            nodes.view(np.int32)[ids, 12 + side] = ref
            na.append(s[inner]), nb.append(e[inner]), nids.append(ref[inner])
        a, b, ids = np.concatenate(na), np.concatenate(nb), np.concatenate(nids)
    return nodes


def with_host_trees(world):
    """Gives every mesh a stored tree in the reference's schema (legacy.lbvh_to_reference_tree of median_split_nodes),
    faces reordered to leaf order as in the reference's files: the oracle walks it like MeshBVHTree.hit."""
    for m in world.meshes:
        f = m["indices"]
        tri9 = m["positions"][f[:, [0, 3, 6]]].reshape(-1, 9)
        tree, order = legacy.lbvh_to_reference_tree(median_split_nodes(tri9), [], tri9)
        m["tree"], m["indices"] = tree, f[order]
    return world


# Seeded stand-ins for the reference's model scenes.  scenes_cache/<name>.npz (tools/prepare_assets.py) is made from the
# reference's model files, which the repository does not carry; the tests render a scene of the same kind instead: a
# textured body standing on a +-50 ground quad under a 256^2 sky image, one atlas area of the cache's map size per
# texture (the ground's area holds the constant fallback material), stored trees in the reference's schema.
# name: (seed, segments around the body, map size, maps on the body)
STAND_INS = {"yoimiya_ground_small": (1, 96, 512, 4), "yoimiya_ground_full": (1, 400, 2048, 4),
             "zhongli_small": (2, 96, 512, 5), "zhongli_full": (2, 400, 2048, 5),
             "ganyu_small": (3, 96, 512, 6), "ganyu_full": (3, 400, 2048, 6)}


def _sky(rng):
    ex, ey = np.meshgrid(np.linspace(0, 1, 256), np.linspace(0, 1, 256), indexing="ij")
    env = np.stack([0.35 + 0.5 * ey, 0.5 + 0.4 * ey, 0.9 + 0.3 * ey], -1)
    env += 0.15 * np.repeat(np.repeat(rng.random((16, 16, 3)), 16, 0), 16, 1)
    return env.astype(np.float32)


@functools.lru_cache(maxsize=None)
def stand_in_world(name):
    """The stand-in of scenes_cache/<name>.npz (STAND_INS), or of demo.npz: a quad under a textured sphere lit by the
    sky, with a 64x64 checker texture whose roughness and metallic channels differ by quadrant."""
    w = legacy.World()
    if name == "demo":
        rng = np.random.default_rng(0)
        w.add_mesh(np.array([[2, -1, -2], [-2, -1, -2], [-2, -1, 2], [2, -1, 2]], np.float32), np.array([[0, 1, 0]], np.float32),
                   np.array([[0, 0], [1, 0], [1, 1], [0, 1]], np.float32),
                   np.array([[0, 0, 0, 1, 0, 1, 2, 0, 2, 0], [0, 0, 0, 2, 0, 2, 3, 0, 3, 0]], np.int32))
        w.add_sphere(legacy.Sphere([0, 0, 0], 1.0, 0, 0))
        xs, ys = np.meshgrid(np.arange(64), np.arange(64), indexing="ij")
        tex = np.empty((64, 64, 8), np.uint8)
        tex[...] = legacy.FALLBACK_TEXEL
        tex[:, :, 0] = np.where((xs // 8 + ys // 8) % 2, 230, 60)
        tex[:, :, 1] = 120
        tex[:, :, 3] = np.where(xs < 32, 255, 64)
        tex[:, :, 7] = np.where(ys < 32, 0, 200)
        w.set_atlas(tex, [[0, 0, 64, 64]], [1])
        w.set_environment_image(_sky(rng), [0, 0, 256, 256])
        return with_host_trees(w)
    seed, nu, size, maps = STAND_INS[name]
    rng = np.random.default_rng(seed)
    nv = nu // 2
    th = np.linspace(0, 2 * np.pi, nu + 1)
    ys = np.linspace(0.5, 15.5, nv + 1)
    r = 2.2 + 1.2 * np.sin(0.45 * ys + seed)[:, None] + 0.5 * np.cos(3 * th + 0.3 * ys[:, None])
    r = r + 0.03 * rng.standard_normal(r.shape)
    r[:, -1] = r[:, 0]                                            # the seam: both columns share positions
    pos = np.stack([r * np.cos(th), np.broadcast_to(ys[:, None], r.shape), r * np.sin(th)], -1).reshape(-1, 3)
    nrm = np.stack([np.cos(th) + 0 * ys[:, None], 0.2 * np.sin(ys)[:, None] + 0 * th, np.sin(th) + 0 * ys[:, None]], -1)
    nrm = (nrm / np.linalg.norm(nrm, axis=-1, keepdims=True)).reshape(-1, 3)
    uv = np.stack(np.meshgrid(np.linspace(0, 1, nv + 1), np.linspace(0, 1, nu + 1), indexing="ij")[::-1], -1).reshape(-1, 2)
    i, j = np.meshgrid(np.arange(nv), np.arange(nu), indexing="ij")
    a = (i * (nu + 1) + j).ravel()
    b, c, d = a + 1, a + nu + 2, a + nu + 1
    tid = (i * maps // nv).ravel()
    faces = np.concatenate([np.stack([a, a, a, b, b, b, c, c, c, tid], 1), np.stack([a, a, a, c, c, c, d, d, d, tid], 1)])
    w.add_mesh(pos, nrm, uv, faces.astype(np.int32))
    w.add_mesh(np.array([[50, 0, -50], [-50, 0, -50], [-50, 0, 50], [50, 0, 50]], np.float32), np.array([[0, 1, 0]], np.float32),
               np.array([[0, 0], [10, 0], [10, 10], [0, 10]], np.float32),
               np.array([[0, 0, 0, 1, 0, 1, 2, 0, 2, maps], [0, 0, 0, 2, 0, 2, 3, 0, 3, maps]], np.int32))
    tex = np.empty(((maps + 1) * size, size, 8), np.uint8)
    tex[...] = legacy.FALLBACK_TEXEL
    blocks = rng.integers(20, 256, size=(maps * size // 32, size // 32, 3), dtype=np.uint8)
    tex[:maps * size, :, 0:3] = np.repeat(np.repeat(blocks, 32, 0), 32, 1)
    w.set_atlas(tex, [[k * size, 0, (k + 1) * size, size] for k in range(maps + 1)], [1] * (maps + 1))
    w.environment = 0
    w.set_environment_image(_sky(rng), [0, 0, 256, 256])
    return with_host_trees(w)


def mesh_camera(resolution):
    """15_module.py:1068-1072."""
    cam = legacy.Camera(resolution)
    cam.set_fov(30)
    cam.set_position(legacy.Vec3f([0, 8, -30]))
    cam.look_at(legacy.Vec3f([0, 8, 0]))
    return cam


def hit_tolerance(tris, tri_ids, rays, t):
    """|dt| bound for one (ray, triangle) pair: the contract's 1e-5 relative, plus the unavoidable rounding of f32
    coordinates (a few ulps of the scene scale) amplified by 1/|d.N| when the ray grazes the triangle's plane."""
    T = tris[np.maximum(tri_ids, 0)]
    n = np.cross(T[:, 3:6] - T[:, 0:3], T[:, 6:9] - T[:, 0:3])
    n /= np.linalg.norm(n, axis=1, keepdims=True)
    dn = np.abs((rays[:, 4:7] * n).sum(1))
    scale = np.maximum(np.abs(rays[:, :3]).max(1), np.abs(T).max(1))
    return 1e-5 * np.abs(t) + 16 * 1.2e-7 * scale / np.maximum(dn, 1e-12)
