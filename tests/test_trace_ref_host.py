"""The float64 trace reference of the far-geometry tests (tests/trace_ref.py) checked against itself: the analytic
tiled-plane answer equals brute force, and compare() tells ambiguous rays from wrong answers."""
import numpy as np
import pytest

import trace_ref as R


def _room_rays(offset, half, n, seed):
    rng = np.random.default_rng(seed)
    o = np.asarray(offset, np.float64) + (rng.random((n, 3)) * 1.8 - 0.9) * half
    d = rng.normal(size=(n, 3))
    d /= np.linalg.norm(d, axis=1, keepdims=True)
    d[:64] = 0.0                                 # axis-parallel rays with exact zeros of both signs
    d[np.arange(64), np.arange(64) % 3] = np.where(np.arange(64) % 2, 1.0, -1.0)
    d[np.arange(32), (np.arange(32) + 1) % 3] = -0.0
    rays = np.zeros((n, 8), np.float32)
    rays[:, :3], rays[:, 3], rays[:, 4:7], rays[:, 7] = o, 1e-4, d, np.inf
    return rays


@pytest.mark.parametrize("offset", [(0, 0, 0), (1e3, 0, 0), (-1e4, -1e4, -1e4)])
def test_analytic_room_equals_brute_force(offset):
    half = 0.5
    room = R.closed_room(offset, half, 4)
    tris = room.triangles()
    assert tris.shape == (6 * 2 * 16, 9)
    rays = _room_rays(offset, half, 3000, 7)
    rays[100:200, 7] = 0.2                       # finite tmax: some rays end before the wall
    bi, bt, bm = R.brute_force(tris, rays, pairs_per_chunk=1 << 16)
    ai, at, am = room.closest_hit(rays)
    assert np.array_equal(ai, bi)
    assert np.array_equal(at, bt) and np.array_equal(am, bm)
    assert (bi[:100] >= 0).all() and (bi[200:] >= 0).all() and (bi[100:200] < 0).any()


def test_floor_ids_and_tile_halves():
    floor = R.tiled_floor((10.0, 0.0, -3.0), 0.25, 4)
    tris = floor.triangles()
    # rays straight down onto both halves of tile (i=2 along z, j=1 along x): z in [-2.5, -2.25], x in [10.25, 10.5]
    rays = np.array([[10.45, 1.0, -2.45, 1e-4, 0.0, -1.0, -0.0, np.inf],
                     [10.30, 1.0, -2.30, 1e-4, 0.0, -1.0, 0.0, np.inf],
                     [9.0, 1.0, -2.30, 1e-4, 0.0, -1.0, 0.0, np.inf]], np.float32)
    ids, t, m = floor.closest_hit(rays)
    bi, bt, _ = R.brute_force(tris, rays)
    assert np.array_equal(ids, bi) and np.array_equal(t, bt)
    assert ids[0] // 2 == 2 * 4 + 1 and ids[1] // 2 == ids[0] // 2 and ids[0] != ids[1]
    assert ids[2] == -1 and abs(t[0] - 1.0) < 1e-12 and m[0] > 0.1


def test_compare_flags_wrong_answers_and_spares_ambiguous_ones():
    offset = (1e4, 0.0, 1e4)
    floor = R.tiled_floor(offset, 0.01, 64)
    tris = floor.triangles()
    rng = np.random.default_rng(3)
    n = 4000
    tgt = np.array(offset) + np.stack([rng.random(n) * 0.64, np.zeros(n), rng.random(n) * 0.64], 1)
    o = tgt + np.stack([rng.normal(size=n) * 0.3, 0.5 + rng.random(n) * 0.5, rng.normal(size=n) * 0.3], 1)
    rays = np.zeros((n, 8), np.float32)
    rays[:, :3], rays[:, 3], rays[:, 7] = o, 1e-4, np.inf
    d = tgt - rays[:, :3].astype(np.float64)
    rays[:, 4:7] = d / np.linalg.norm(d, axis=1, keepdims=True)
    ids, t, _ = floor.closest_hit(rays)
    t32 = t.astype(np.float32)
    ok = R.compare(tris, rays, ids, t, ids, t32)
    assert not (ok["lost"] | ok["bad_t"] | ok["phantom"]).any()
    # the bound is local: at 1e4 units from the origin it still calls only a small share of the rays ambiguous
    assert ok["ambiguous"].mean() < 5e-3, ok["ambiguous"].mean()
    clean = np.flatnonzero(~ok["ambiguous"] & (ids >= 0))[:3]
    wrong_id, wrong_t = ids.copy(), t32.copy()
    wrong_id[clean[0]] = -1                                  # a lost hit
    wrong_id[clean[1]] ^= 1                                  # the other half of the same tile
    wrong_t[clean[2]] *= np.float32(1 + 1e-4)                # t off by 1e-4 relative
    bad = R.compare(tris, rays, ids, t, wrong_id, wrong_t)
    assert bad["lost"][clean[0]] and bad["lost"][clean[1]] and bad["bad_t"][clean[2]]
    assert bad["lost"].sum() == 2 and bad["bad_t"].sum() == 1
    rays2 = rays.copy()
    rays2[:, 4:7] *= -1                                      # pointing away from the floor: clean misses
    pi = np.full(n, 5, np.int32)
    ph = R.compare(tris, rays2, np.full(n, -1, np.int32), np.full(n, np.inf), pi, np.ones(n, np.float32))
    assert ph["phantom"].all() and (ids >= 0).mean() > 0.99
