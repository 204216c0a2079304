"""CPU tests of the legacy host surface: .world.npy loader, OBJ loader known-answers, texture packer, caches,
and the legacy oracle itself."""
import os

import numpy as np
import pytest

import learn_path_tracing_b200 as L
from learn_path_tracing_b200 import legacy, scene_cache, worldnpy
from helpers import all_triangles, stand_in_world, synthetic_legacy_world

REF = "/root/reference"
needs_ref = pytest.mark.skipif(not os.path.isdir(REF), reason="reference checkout not mounted (GPU box)")


@needs_ref
@pytest.mark.parametrize("name", ["Yoimiya", "Yoimiya_ShapeChange", "Zhongli", "Ganyu", "Barbara", "demo"])
def test_world_npy_loads_without_taichi_and_keeps_invariants(name):
    d = worldnpy.load_world(os.path.join(REF, "legacy", name + ".world.npy"))
    assert "meshes_bvhs" in d and "environment" in d
    for md in d["meshes_bvhs"]:
        m = worldnpy.mesh_arrays(md)
        t = m["tree"]
        inner = t["left"] >= 0
        assert np.all(t["right"][inner] == t["left"][inner] + 1)          # BFS order, SURVEY 2.3
        assert np.all(t["left"][inner] > np.flatnonzero(inner))
        assert (t["data"] >= 0).sum() == inner.sum() + 1                  # leaves = inner + 1
        assert t["leaf_cut"][-1] == len(m["faces"]) and t["max_depth"] == 16
        assert m["faces"][:, [0, 3, 6]].max() < len(m["positions"])
    if name.startswith(("Yoimiya", "Barbara")):
        cfg = worldnpy.texture_configs(d["textures"])
        assert all(len(c["area"]) == 4 for c in cfg) and cfg[0]["area"][2] - cfg[0]["area"][0] == 2048


@needs_ref
def test_load_obj_reproduces_the_cached_mesh():
    """Known answer: Yoimiya.world.npy was built from Yoimiya_ShapeChange.obj with flip_z, rotate(pi, 0) and the
    v-flip (15_module.py:1059) — positions/normals/uvs must match, faces as a set (the cache is in leaf order)."""
    pos, nrm, uv, idx, tex = legacy.load_obj(os.path.join(REF, "assets/models/Yoimiya/Yoimiya_ShapeChange.obj"), 1,
                                             flip_z=True, flip_textcoord=True, transform=legacy.rotate(np.pi, 0))
    m = worldnpy.mesh_arrays(worldnpy.load_world(os.path.join(REF, "legacy/Yoimiya.world.npy"))["meshes_bvhs"][0])
    assert np.abs(pos - m["positions"]).max() < 1e-6 and np.abs(nrm - m["normals"]).max() < 1e-6
    assert np.abs(uv - m["texcoords"]).max() < 1e-6
    assert set(map(tuple, idx.tolist())) == set(map(tuple, m["faces"].tolist()))
    assert [os.path.basename(t["file_path"]) for t in tex] == ["face.png", "hair.png", "cloth.png", "skin.png"]
    assert [t["id"] for t in tex] == [1, 2, 3, 4]


def test_load_obj_small_fixture(tmp_path):
    (tmp_path / "m.mtl").write_text("newmtl a\nmap_Kd ta.png\nnewmtl b\nmap_Kd tb.png\nnewmtl c\nmap_Kd ta.png\n")
    (tmp_path / "m.obj").write_text(
        "# comment\nmtllib m.mtl\nv 0 0 1\nv 1 0 1\nv 0 1 1\nv 1 1 2\nvn 0 0 1\nvt 0 0.25\nvt 1 0\nvt 0 1\n"
        "usemtl b\nf 1/1/1 2/2/1 3/3/1\nusemtl c\nf 2/2/1 4/3/1 3/1/1\n")
    pos, nrm, uv, idx, tex = legacy.load_obj(str(tmp_path / "m.obj"), 5, flip_z=True, flip_textcoord=True)
    assert pos.shape == (4, 3) and np.allclose(pos[3], [1, 1, -2]) and np.allclose(nrm[0], [0, 0, -1])
    assert np.allclose(uv[0], [0, 0.75])
    assert [t["id"] for t in tex] == [5, 6] and len(tex) == 2  # 'c' re-uses ta.png
    assert idx.tolist() == [[0, 0, 0, 1, 0, 1, 2, 0, 2, 6], [1, 0, 1, 3, 0, 2, 2, 0, 0, 5]]


def test_rotate_and_camera_conventions():
    assert np.allclose(legacy.rotate(np.pi, 0) @ np.array([1, 2, 3], np.float32), [-1, 2, -3], atol=1e-6)
    cam = legacy.Camera((300, 200))
    cam.set_fov(30)
    cam.set_position(legacy.Vec3f([0, 8, -30]))
    cam.look_at(legacy.Vec3f([0, 8, 0]))
    c = cam.to_struct()
    assert np.allclose(list(c.front), [0, 0, 1], atol=1e-6) and np.allclose(list(c.right), [-1, 0, 0], atol=1e-6)
    assert abs(c.view_w - 2 * np.tan(np.radians(30))) < 1e-6          # legacy: fov is the HALF angle
    v2 = L.Camera((300, 200), fov=60).to_struct()
    assert abs(v2.view_w - c.view_w) < 1e-6                            # v2: full angle (camera.py:81)
    cam.move_front(2.0)
    cam.move_up(1.0)
    assert np.allclose(cam.position, [0, 9, -28], atol=1e-5)


def test_texture_manager_shelf_packer():
    tm = legacy.TextureManager((10, 6))
    for i, size in enumerate([(4, 2), (3, 4), (6, 2), (2, 2)]):
        tm.add("unused", i, size)
    tm.build()
    areas = {c["id"]: c["area"].as_list() for c in tm.configs}
    assert areas[1] == [0, 0, 3, 4]              # tallest first
    boxes = list(areas.values())
    for i, a in enumerate(boxes):                # inside the atlas, pairwise disjoint
        assert 0 <= a[0] < a[2] <= 10 and 0 <= a[1] < a[3] <= 6
        for b in boxes[i + 1:]:
            assert a[2] <= b[0] or b[2] <= a[0] or a[3] <= b[1] or b[3] <= a[1]
    big = legacy.TextureManager((4, 4))
    big.add("unused", 0, (5, 1))
    with pytest.raises(MemoryError):
        big.build()


def test_world_save_load_round_trip(tmp_path):
    w, _ = synthetic_legacy_world()
    fn = str(tmp_path / "s.world.npy")
    w.save(fn, build_trees=False)   # no GPU here: single-leaf trees (the GPU-built trees are tested under -m gpu)
    d = worldnpy.load_world(fn)
    assert len(d["meshes_bvhs"]) == 2 and "spheres_bvh" in d
    w2 = legacy.World()
    w2.load(fn, load_images=False)
    for a, b in zip(w.meshes, w2.meshes):
        assert np.array_equal(a["positions"], b["positions"]) and np.array_equal(a["indices"], b["indices"])
    assert np.array_equal(w.sphere_arrays()[0], w2.sphere_arrays()[0])
    c = str(tmp_path / "c.npz")
    scene_cache.save_cache(c, w)
    w3 = scene_cache.load_cache(c)
    assert np.array_equal(w3._atlas[0], w._atlas[0]) and np.array_equal(w3._env[0], w._env[0])
    assert len(w3.meshes) == 2 and len(w3.spheres) == 2


def test_lbvh_to_reference_tree_schema():
    """LBVH nodes (two child boxes + refs) -> the reference's MeshBVHTree arrays: every face in exactly one leaf,
    leaves <= 4 faces unless the depth bound cuts, node boxes contain their faces, nodes in creation order."""
    rng = np.random.default_rng(1)
    n = 37
    tri9 = (rng.random((n, 1, 3)) * 4 + rng.random((n, 3, 3)) * 0.3).astype(np.float32).reshape(n, 9)
    lo, hi = tri9.reshape(n, 3, 3).min(1), tri9.reshape(n, 3, 3).max(1)
    # a hand-made binary tree over the faces sorted by x: recursive median split, written in the LBVH node layout
    order = list(np.argsort(lo[:, 0]))
    nodes = []

    def build(ids):
        if len(ids) == 1:
            return ~int(ids[0]), lo[ids[0]], hi[ids[0]]
        k = len(nodes)
        nodes.append(None)
        a, alo, ahi = build(ids[:len(ids) // 2])
        b, blo, bhi = build(ids[len(ids) // 2:])
        rec = np.zeros(16, np.float32)
        rec[0:3], rec[3:6], rec[6:9], rec[9:12] = alo, ahi, blo, bhi
        rec[12:14] = np.array([a, b], np.int32).view(np.float32)
        nodes[k] = rec
        return k, np.minimum(alo, blo), np.maximum(ahi, bhi)

    for glob, depth in (([], 24), ([5, 9], 24), ([], 2)):
        nodes.clear()
        build([i for i in order if i not in glob])   # the builder keeps oversized ("global") faces out of the tree
        nodes16 = np.stack(nodes)
        tree, forder = legacy.lbvh_to_reference_tree(nodes16, glob, tri9, max_leave_objects=4, max_depth=depth)
        assert sorted(forder) == list(range(n))
        L_, R_, D_, cut = tree["left"], tree["right"], tree["data"], tree["leaf_cut"]
        assert cut[0] == 0 and cut[-1] == n and np.all(np.diff(cut) > 0)
        leaves = np.flatnonzero(D_ >= 0)
        assert sorted(D_[leaves]) == list(range(len(cut) - 1))
        assert np.all((L_[leaves] == -1) & (R_[leaves] == -1))
        inner = np.flatnonzero(D_ < 0)
        assert np.all(L_[inner] > inner) and np.all(R_[inner] == L_[inner] + 1)   # creation order, siblings adjacent
        if depth == 24 and not glob:
            assert np.diff(cut).max() <= 4
        # boxes: a leaf's box contains its faces; a child's box lies inside its parent's
        for k in leaves:
            f = forder[cut[D_[k]]:cut[D_[k] + 1]]
            assert np.all(lo[f] >= tree["low"][k] - 1e-6) and np.all(hi[f] <= tree["high"][k] + 1e-6)
        for k in inner:
            for c in (L_[k], R_[k]):
                assert np.all(tree["low"][c] >= tree["low"][k] - 1e-6) and np.all(tree["high"][c] <= tree["high"][k] + 1e-6)
        # the reference's traversal needs depth <= max_depth (its stack has max_depth + 1 entries)
        d = np.zeros(len(L_), np.int64)
        for k in inner:
            d[L_[k]] = d[R_[k]] = d[k] + 1
        assert d.max() <= tree["max_depth"]
        assert legacy.reference_visit_order(tree, n).shape == (n,)


def test_legacy_oracle_tree_walk_equals_brute_force(oracle):
    """The reference traversal over the stored SAH tree must find what a loop over all faces finds."""
    w = stand_in_world("yoimiya_ground_small")
    from helpers import mesh_camera
    cam = mesh_camera((96, 64))
    rays = oracle.generate_rays(cam.to_struct(), 96, 64, 0, 3)
    a_id, a_t = oracle.scene_from_legacy_world(w, use_stored_tree=True).trace(rays)
    b_id, b_t = oracle.scene_from_legacy_world(w, use_stored_tree=False).trace(rays)
    assert np.array_equal(a_t, b_t)
    # the model has duplicated / double-sided faces: exact-t ties may resolve to the twin face, nothing else may differ
    assert (a_id != b_id).mean() < 0.05 and np.array_equal(a_id >= 0, b_id >= 0)
    assert 0.05 < (a_id >= 0).mean() < 0.9


def test_legacy_oracle_white_furnace(oracle):
    """Energy check of the restated legacy shading: with albedo 1, absorptivity 0 and a constant environment every
    path that escapes carries throughput <= 1, and a non-metal closed scene returns exactly the environment."""
    w, cam = synthetic_legacy_world()
    tex = w._atlas[0].copy()
    tex[:, :, 0:3] = 255
    tex[:, :, 7] = 0
    w.set_atlas(tex, w._atlas[1], w._atlas[2])
    env = np.full((8, 8, 3), 0.5, np.float32)
    w.set_environment_image(env, [0, 0, 8, 8])
    acc, _, st = oracle.render(oracle.scene_from_legacy_world(w), cam.to_struct(), 96, 64, 8, 64, L.PT_SHADE_LEGACY,
                               seed=1, absorptivity=0.0)
    m = acc / 8
    assert m.max() <= 0.5 + 1e-4 and m.mean() > 0.45
    tris, off = all_triangles(w)
    assert off == 2 and tris.shape[1] == 9


def test_exr_environment_round_trip(tmp_path):
    """SURVEY 8f-2 / 15_module.py:118-132,1049: an EXR environment (float radiance, not /255) goes through
    TextureManager.add -> build -> load_environment exactly like the reference's imageio path: indexed [x, y] with y up,
    RGB order, values untouched.  The two EXRs the reference scripts name are missing from the checkout, so a small one
    is written here with cv2 (the reader legacy.py uses)."""
    import os
    os.environ.setdefault("OPENCV_IO_ENABLE_OPENEXR", "1")
    cv2 = pytest.importorskip("cv2")
    rng = np.random.default_rng(5)
    rgb = (rng.random((32, 64, 3)) * 6.0).astype(np.float32)      # rows x columns x RGB, values above 1 (HDR)
    fn = str(tmp_path / "env_small.exr")
    assert cv2.imwrite(fn, rgb[:, :, ::-1])                         # cv2 stores BGR
    img = legacy.load_environment_image(fn)
    assert img.shape == (64, 32, 3) and img.dtype == np.float32
    # reference: env.transpose(1, 0, 2) then flip along y -> img[x, y] = rgb[H-1-y, x]
    assert np.array_equal(img, np.flip(rgb.transpose(1, 0, 2), 1))
    w = legacy.World(environment_size=(128, 64))
    w.environments.add(fn, 0)                                       # size read from the EXR itself
    w.set_environment(0)
    w.environments.build()
    w.load_textures()
    env, area = w._env
    assert area == [0, 0, 64, 32] and env.shape == (128, 64, 3)
    assert np.array_equal(env[:64, :32], img) and float(np.abs(env[64:]).max()) == 0.0
    # the oracle's bilinear lookup returns the texel value at texel centres (weights 1,0,0,0): u = (x + .5) / w
    from oracle import ptoracle as O
    if hasattr(O, "environment_lookup"):
        d = np.array([[0.0, 0.0, -1.0]], np.float32)
        assert np.isfinite(O.environment_lookup(env, area, d)).all()


def test_world_npy_loader_refuses_foreign_classes_and_writes_both_manager_keys(tmp_path):
    """ADVICE r1: the custom unpickler resolves only numpy arrays / plain containers / (stubbed) taichi structs — the
    reference's np.load(allow_pickle=True) would execute anything; and World.save always writes 'textures' and
    'environments' (the reference's World.load, 15_module.py:823-836, indexes both unconditionally)."""
    import pickle

    class Evil:
        def __reduce__(self):
            return (os.system, ("true",))
    fn = str(tmp_path / "evil.world.npy")
    np.save(fn, {"meshes_bvhs": [], "environment": 0, "x": Evil()}, allow_pickle=True)
    with pytest.raises(pickle.UnpicklingError):
        worldnpy.load_world(fn)
    ok = str(tmp_path / "plain.world.npy")
    pos = np.array([[0, 0, 0], [1, 0, 0], [0, 1, 0]], np.float32)
    worldnpy.save_world(ok, [{"positions": pos, "normals": pos, "texcoords": pos[:, :2], "faces": np.zeros((1, 10), np.int32)}], 0)
    d = worldnpy.load_world(ok)
    assert d["textures"]["configs"] == [] and d["environments"]["configs"] == [] and len(d["meshes_bvhs"]) == 1
