"""Float64 closest-hit reference for triangle scenes, host only.

The f32 inputs are taken exactly as stored (vertices and rays as float32) and promoted to float64, so the reference
answers "which triangle does this f32 ray hit" without the rounding of the f32 kernels.  Two forms:

- brute_force: every ray against every triangle, chunked in NumPy.
- TiledPlanes: scenes made of axis-aligned planes cut into right-triangle tiles (floors, closed rooms), answered
  analytically from the float64 hit point; for scenes too big for brute force.

Both use the kernel's rules: t in [tmin, tmax], a strict inside test (every barycentric > 0, 15_module.py:928) and, on
equal t, the lower id.

Ambiguity is judged from LOCAL quantities only: |o - v0|, the triangle's size, its smallest altitude and 1/|d.N|, times
a few f32 ulps.  The absolute coordinates |o| never enter: a bound that grew with the distance from the world origin
would excuse exactly the culling errors of geometry far from it.
"""
import numpy as np

EPS32 = 2.0 ** -24   # unit roundoff of float32
K_ULPS = 16          # a few ulps of slack for the kernel's Moller-Trumbore (cross products, dot products, 1/det)


def _verts(tris9):
    return np.asarray(tris9, np.float32).reshape(-1, 3, 3).astype(np.float64)


def _rays64(rays):
    r = np.asarray(rays, np.float32).reshape(-1, 8).astype(np.float64)
    return r[:, 0:3], r[:, 3], r[:, 4:7], r[:, 7]


def _pair_hits(v, o, d):
    """t and the three barycentrics (of v0, v1, v2) of the planes of triangles v [..., 3, 3] along rays o, d [..., 3],
    from scalar triple products on vertices relative to the origin (float64)."""
    a, b, c = v[..., 0, :] - o, v[..., 1, :] - o, v[..., 2, :] - o
    wa = np.einsum("...k,...k->...", d, np.cross(b, c))
    wb = np.einsum("...k,...k->...", d, np.cross(c, a))
    wc = np.einsum("...k,...k->...", d, np.cross(a, b))
    det = wa + wb + wc
    n = np.cross(v[..., 1, :] - v[..., 0, :], v[..., 2, :] - v[..., 0, :])
    dn = np.einsum("...k,...k->...", d, n)
    with np.errstate(divide="ignore", invalid="ignore"):
        t = np.einsum("...k,...k->...", a, n) / dn
        bary = np.stack([wa / det, wb / det, wc / det], -1)
    bad = ~np.isfinite(t) | (det == 0)
    t = np.where(bad, np.inf, t)
    bary = np.where(bad[..., None], -np.inf, bary)
    return t, bary


def evaluate(tris9, ids, rays):
    """float64 t and smallest barycentric of ray i against triangle ids[i] (inf / -inf where ids[i] < 0)."""
    ids = np.asarray(ids)
    o, _, d, _ = _rays64(rays)
    v = _verts(tris9)[np.maximum(ids, 0)]
    t, bary = _pair_hits(v, o, d)
    miss = ids < 0
    return np.where(miss, np.inf, t), np.where(miss, -np.inf, bary.min(-1))


def brute_force(tris9, rays, pairs_per_chunk=1 << 21):
    """(ids int32, t float64, smallest barycentric) of the closest hit of every ray; -1 / inf / -inf on a miss."""
    v = _verts(tris9)
    o, tmin, d, tmax = _rays64(rays)
    n = len(o)
    ids = np.full(n, -1, np.int32)
    t_out = np.full(n, np.inf)
    step = max(1, pairs_per_chunk // max(len(v), 1))
    for s in range(0, n, step):
        e = min(n, s + step)
        t, bary = _pair_hits(v[None], o[s:e, None], d[s:e, None])
        ok = (bary.min(-1) > 0) & (t >= tmin[s:e, None]) & (t <= tmax[s:e, None])
        t = np.where(ok, t, np.inf)
        k = np.argmin(t, 1)                     # first minimum: the lower id wins equal t
        tk = t[np.arange(e - s), k]
        hit = np.isfinite(tk)
        ids[s:e] = np.where(hit, k, -1)
        t_out[s:e] = tk
    _, margin = evaluate(tris9, ids, rays)
    return ids, t_out, margin


def local_bounds(tris9, ids, rays):
    """(barycentric bound, t bound) of the f32 kernel's rounding for ray i against triangle ids[i], from local
    quantities: the span L = |o - v0| + longest edge the kernel's arithmetic works over, the triangle's smallest
    altitude h and the ray's incidence |d.N| / |d|.  Hit positions carry ~K ulps of L; seen along the ray that is
    K ulps of L / |d.N| in t, and relative to the triangle K ulps of L / (h |d.N|) in barycentrics."""
    ids = np.asarray(ids)
    v = _verts(tris9)[np.maximum(ids, 0)]
    o, _, d, _ = _rays64(rays)
    e = np.stack([v[:, 1] - v[:, 0], v[:, 2] - v[:, 1], v[:, 0] - v[:, 2]], 1)
    elen = np.linalg.norm(e, axis=-1)
    area2 = np.linalg.norm(np.cross(e[:, 0], -e[:, 2]), axis=-1)
    h = area2 / elen.max(1)
    nrm = np.cross(e[:, 0], -e[:, 2]) / np.maximum(area2, 1e-300)[:, None]
    dlen = np.linalg.norm(d, axis=1)
    cos = np.abs((d * nrm).sum(1)) / dlen
    span = np.linalg.norm(o - v[:, 0], axis=1) + elen.max(1)
    ulps = K_ULPS * EPS32 * span / np.maximum(cos, 1e-12)
    miss = ids < 0
    return np.where(miss, 0.0, ulps / np.maximum(h, 1e-300)), np.where(miss, 0.0, ulps / dlen)


def compare(tris9, rays, ref_ids, ref_t, ids, t):
    """Checks kernel hits (ids, t) against the reference (ref_ids, ref_t).  Returns a dict of boolean masks:
    ambiguous (an edge graze, a tie or a t at the end of the interval, within the local bounds), lost (a clean reference
    hit the kernel missed or gave to another triangle), bad_t (right triangle, t off by more than 1e-5 t + the bound)
    and phantom (a kernel hit where the reference has a clean miss)."""
    ref_ids, ids = np.asarray(ref_ids), np.asarray(ids)
    _, tmin, _, tmax = _rays64(rays)
    rb, rtb = local_bounds(tris9, ref_ids, rays)
    gb, gtb = local_bounds(tris9, ids, rays)
    _, rmargin = evaluate(tris9, ref_ids, rays)
    gt64, gmargin = evaluate(tris9, ids, rays)
    rh, gh = ref_ids >= 0, ids >= 0
    amb = rh & (rmargin < rb)
    amb |= gh & (np.abs(gmargin) < gb)          # the kernel's triangle, grazed on either side of an edge
    with np.errstate(invalid="ignore"):          # inf - inf of misses compares False
        # a tie: the kernel's triangle is hit too (float64), at a t the bounds cannot tell from the reference's
        amb |= rh & gh & (ids != ref_ids) & (gmargin > 0) & (np.abs(gt64 - ref_t) <= rtb + gtb)
        for tt, tb, has in ((ref_t, rtb, rh), (gt64, gtb, gh)):
            amb |= has & ((np.abs(tt - tmin) <= tb) | (np.abs(tt - tmax) <= tb))
        clean = ~amb
        lost = clean & rh & (ids != ref_ids)
        same = clean & rh & (ids == ref_ids)
        t32 = np.asarray(t, np.float64)
        bad_t = same & ~(np.abs(t32 - ref_t) <= 1e-5 * np.abs(ref_t) + rtb)
    phantom = clean & ~rh & gh
    return {"ambiguous": amb, "lost": lost, "bad_t": bad_t, "phantom": phantom}


# ---- analytic scenes: axis-aligned planes of right-triangle tiles --------------------------------------------------
class TiledPlanes:
    """Planes normal to a coordinate axis, each cut into a grid of tiles, each tile into two right triangles along its
    diagonal.  Plane k: normal axis a, coordinate c, grid lines gu (along axis (a+1)%3) and gv (along (a+2)%3), all
    float32 as stored.  Triangle ids run plane by plane, tile (i, j) row-major, lower half first."""

    def __init__(self):
        self.planes = []   # (axis, c, gu, gv, first id)
        self.n = 0

    def add(self, axis, c, gu, gv):
        gu, gv = np.asarray(gu, np.float32), np.asarray(gv, np.float32)
        assert np.all(np.diff(gu) > 0) and np.all(np.diff(gv) > 0)
        self.planes.append((axis, np.float32(c), gu, gv, self.n))
        self.n += 2 * (len(gu) - 1) * (len(gv) - 1)
        return self

    def triangles(self):
        out = []
        for axis, c, gu, gv, _ in self.planes:
            ua, va = (axis + 1) % 3, (axis + 2) % 3
            U, V = np.meshgrid(gu, gv, indexing="ij")
            P = np.zeros(U.shape + (3,), np.float32)
            P[..., axis], P[..., ua], P[..., va] = c, U, V
            p00, p10, p11, p01 = P[:-1, :-1], P[1:, :-1], P[1:, 1:], P[:-1, 1:]
            lower = np.concatenate([p00, p10, p11], -1)
            upper = np.concatenate([p00, p11, p01], -1)
            out.append(np.stack([lower, upper], 2).reshape(-1, 9))
        return np.concatenate(out).astype(np.float32)

    def closest_hit(self, rays):
        """(ids, t, smallest barycentric) like brute_force, from the float64 hit point of every plane."""
        tris = self.triangles()
        o, tmin, d, tmax = _rays64(rays)
        n = len(o)
        best_id = np.full(n, -1, np.int64)
        best_t = np.full(n, np.inf)
        for axis, c, gu, gv, first in self.planes:
            ua, va = (axis + 1) % 3, (axis + 2) % 3
            with np.errstate(divide="ignore", invalid="ignore"):
                t = (np.float64(c) - o[:, axis]) / d[:, axis]
                ok = np.isfinite(t) & (t >= tmin) & (t <= tmax)
                t = np.where(ok, t, 0.0)
                pu, pv = o[:, ua] + t * d[:, ua], o[:, va] + t * d[:, va]
            i = np.searchsorted(gu, pu, side="right") - 1
            j = np.searchsorted(gv, pv, side="right") - 1
            ok &= (i >= 0) & (i < len(gu) - 1) & (j >= 0) & (j < len(gv) - 1)
            i, j = np.clip(i, 0, len(gu) - 2), np.clip(j, 0, len(gv) - 2)
            base = first + 2 * (i * (len(gv) - 1) + j)
            cand = np.full(n, -1, np.int64)
            for half in (0, 1):   # the tile half whose strict inside test the float64 point passes
                k = np.where(ok, base + half, -1)
                _, m = evaluate(tris, k, rays)
                cand = np.where(ok & (m > 0), k, cand)
            tc = np.where(cand >= 0, t, np.inf)
            take = (tc < best_t) | ((tc == best_t) & (cand >= 0) & (cand < best_id))
            best_id, best_t = np.where(take, cand, best_id), np.where(take, tc, best_t)
        ids = best_id.astype(np.int32)
        _, margin = evaluate(tris, ids, rays)
        return ids, best_t, margin


def grid_lines(start, size, count):
    """count + 1 float32 grid lines start + k * size (each rounded once from float64)."""
    return (np.float64(start) + np.float64(size) * np.arange(count + 1)).astype(np.float32)


def tiled_floor(offset, tile, count, y=0.0):
    """A floor of count x count square tiles at height offset.y + y, its corner at (offset.x, offset.z)."""
    ox, oy, oz = (float(v) for v in offset)
    return TiledPlanes().add(1, oy + y, grid_lines(oz, tile, count), grid_lines(ox, tile, count))


def closed_room(offset, half, count):
    """The six walls of the cube offset + [-half, half]^3, each cut into count x count tiles."""
    s = TiledPlanes()
    for axis in range(3):
        ua, va = (axis + 1) % 3, (axis + 2) % 3
        gu = grid_lines(float(offset[ua]) - half, 2.0 * half / count, count)
        gv = grid_lines(float(offset[va]) - half, 2.0 * half / count, count)
        for sign in (-1.0, 1.0):
            s.add(axis, float(offset[axis]) + sign * half, gu, gv)
    return s
