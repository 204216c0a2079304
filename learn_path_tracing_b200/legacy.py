"""Host surface of the legacy mesh/texture tracer (legacy/PT_in_one_weekend/15_module.py, 14_mesh.py).

Same names and argument meaning as the reference script: rotate, load_obj, TextureManager, Camera, World
(add_mesh / add_sphere / set_environment / build / save / load), Sphere / Face / FaceVertex records and a
progressive render(moved).  What changed is where the work happens: the reference builds a SAH BVH in host
Python (minutes) and traces in Taichi kernels; here World.build() hands triangles, the 8-bit texture atlas and
the environment map to libb200pt.so, which builds an LBVH on the GPU and runs the wavefront.
"""
from __future__ import annotations

import math
import os

import numpy as np

from . import _lib, worldnpy
from .dtypes import Vec2f, Vec2i, Vec3f  # noqa: F401  (re-exported like the reference module's globals)

epsilon = 1e-4          # 15_module.py:44
texture_size = (2048 * 6, 2048)      # :37
environment_size = (2048, 2048)      # :39
texture_maxnum = 32
environment_maxnum = 32

# where relative asset paths ("./models/...", "./textures/...") are searched, in order
ASSET_ROOTS = [os.getcwd(), os.environ.get("LPT_ASSETS", ""), "/root/reference/assets", "/root/reference/legacy"]

# material used for a PBR set whose albedo/roughness/normal maps are absent from the checkout (SURVEY 8d:
# granite-gray-white / sandyground1 ship only their _metallic map): flat linear albedo 0.5, roughness 1,
# metallic 0, flat normal.  8-bit source values: 186 -> (186/255)^2.2 = 0.4996.
FALLBACK_TEXEL = np.array([186, 186, 186, 255, 128, 128, 255, 0], np.uint8)


def rotate(yaw, pitch, roll=0.0):
    """15_module.py:261-278 — angles in RADIANS, yaw @ pitch @ roll."""
    yaw_t = np.array([[math.cos(yaw), 0, math.sin(yaw)], [0, 1, 0], [-math.sin(yaw), 0, math.cos(yaw)]])
    pitch_t = np.array([[1, 0, 0], [0, math.cos(pitch), -math.sin(pitch)], [0, math.sin(pitch), math.cos(pitch)]])
    roll_t = np.array([[math.cos(roll), -math.sin(roll), 0], [math.sin(roll), math.cos(roll), 0], [0, 0, 1]])
    return (yaw_t @ pitch_t @ roll_t).astype(np.float32)


class FaceVertex:
    __slots__ = ("p", "n", "t")

    def __init__(self, p=0, n=0, t=0):
        self.p, self.n, self.t = int(p), int(n), int(t)


class Face:
    """Face(a, b, c, texture_id) — 15_module.py:31-32."""
    __slots__ = ("a", "b", "c", "texture_id")

    def __init__(self, a, b, c, texture_id=0):
        self.a, self.b, self.c, self.texture_id = a, b, c, int(texture_id)

    def row(self):
        return [self.a.p, self.a.n, self.a.t, self.b.p, self.b.n, self.b.t, self.c.p, self.c.n, self.c.t,
                self.texture_id]


class Sphere:
    """Sphere(center, radius, transparency, texture_id) — 15_module.py:33."""
    __slots__ = ("center", "radius", "transparency", "texture_id")

    def __init__(self, center=(0, 0, 0), radius=1.0, transparency=0, texture_id=0):
        self.center, self.radius = Vec3f(center), float(radius)
        self.transparency, self.texture_id = int(transparency), int(texture_id)


class TextureArea:
    __slots__ = ("low", "high")

    def __init__(self, low, high):
        self.low, self.high = Vec2i(low), Vec2i(high)

    def as_list(self):
        return [int(self.low[0]), int(self.low[1]), int(self.high[0]), int(self.high[1])]


def _faces_array(indices) -> np.ndarray:
    if isinstance(indices, np.ndarray):
        return np.ascontiguousarray(indices, np.int32).reshape(-1, 10)
    return np.array([f.row() if isinstance(f, Face) else list(f) for f in indices], np.int32).reshape(-1, 10)


def resolve_asset(path: str, extra_roots=()) -> str | None:
    """First existing candidate for a (possibly stale, './models/...') asset path."""
    if os.path.isabs(path) and os.path.exists(path):
        return path
    rel = path[2:] if path.startswith("./") else path
    for root in list(extra_roots) + ASSET_ROOTS:
        if not root:
            continue
        cand = os.path.join(root, rel)
        if os.path.exists(cand):
            return cand
    return path if os.path.exists(path) else None


# ---- OBJ ---------------------------------------------------------------------------------------------
def load_obj(file_path, texture_start_id, flip_z=False, flip_textcoord=False, transform=None):
    """15_module.py:135-206.  Triangles with full v/vt/vn triplets, 1-based indices; every `newmtl` maps to its
    map_Kd file, textures are de-duplicated by path and numbered from texture_start_id in first-seen order.
    Returns (positions [V,3], normals [N,3], texture_coords [T,2], indices [F,10] int32, textures list)."""
    if not os.path.exists(file_path):  # the scripts hard-code './models/...': search the asset roots (SURVEY appendix E)
        file_path = resolve_asset(file_path) or file_path
    dir_path = os.path.dirname(file_path)
    positions, normals, texture_coords, indices, textures = [], [], [], [], []
    textures_name = {}
    usemtl = None
    tr = None if transform is None else np.asarray(transform, np.float32).reshape(3, 3)
    with open(file_path, "r") as obj:
        lines = obj.readlines()
    for line in lines:
        if len(line) == 0 or line[0] == "#":
            continue
        tok = line.split()
        if len(tok) == 0:
            continue
        if tok[0] == "mtllib":
            mtl_name = None
            with open(os.path.join(dir_path, tok[1]), "r") as mtl:
                for mtl_line in mtl.readlines():
                    mt = mtl_line.split()
                    if len(mt) == 0:
                        continue
                    if mt[0] == "newmtl":
                        mtl_name = mt[1]
                    elif mt[0] == "map_Kd":
                        tex_path = os.path.join(dir_path, mt[1])
                        for i, texture in enumerate(textures):
                            if texture["file_path"] == tex_path:
                                textures_name[mtl_name] = i
                                break
                        else:
                            textures_name[mtl_name] = len(textures)
                            textures.append({"file_path": tex_path, "id": texture_start_id})
                            texture_start_id += 1
        elif tok[0] == "v" or tok[0] == "vn":
            p = np.array([float(tok[1]), float(tok[2]), float(tok[3])], np.float32)
            if flip_z:
                p[2] = -p[2]
            if tr is not None:
                p = tr @ p
            (positions if tok[0] == "v" else normals).append(p)
        elif tok[0] == "vt":
            uv = np.array([float(tok[1]), float(tok[2])], np.float32)
            if flip_textcoord:
                uv[1] = np.float32(1) - uv[1]
            texture_coords.append(uv)
        elif tok[0] == "usemtl":
            usemtl = tok[1]
        elif tok[0] == "f":
            v = [tok[i].split("/") for i in range(1, 4)]
            row = []
            for k in range(3):
                row += [int(v[k][0]) - 1, int(v[k][2]) - 1, int(v[k][1]) - 1]  # p, n, t
            row.append(textures[textures_name[usemtl]]["id"])
            indices.append(row)
    return (np.array(positions, np.float32).reshape(-1, 3), np.array(normals, np.float32).reshape(-1, 3),
            np.array(texture_coords, np.float32).reshape(-1, 2), np.array(indices, np.int32).reshape(-1, 10), textures)


# ---- textures ----------------------------------------------------------------------------------------
def _open_image(path):
    from PIL import Image
    return Image.open(path)


def _resized_xy(img, size, mode=None):
    """PIL image -> uint8 array indexed [x, y] with y up (15_module.py:76-79: resize, transpose, flip)."""
    from PIL import Image
    if mode:
        img = img.convert(mode)
    if img.size != tuple(size):
        img = img.resize(tuple(size), Image.LANCZOS)  # Image.ANTIALIAS (removed in Pillow 10) is LANCZOS
    a = np.asarray(img)
    if a.ndim == 2:
        a = a[:, :, None]
    return np.flip(a.transpose(1, 0, 2), 1)


def load_texture_texels(file_path, size, extra_roots=()):
    """One atlas area as uint8 [w,h,8] = albedo rgb, roughness, normal xyz, metallic (pre-gamma source values;
    the device applies load_texture's transfer functions, 15_module.py:101-104) and flags (bit 0: no normal map)."""
    w, h = int(size[0]), int(size[1])
    out = np.empty((w, h, 8), np.uint8)
    out[...] = FALLBACK_TEXEL
    flags = 1
    plain = resolve_asset(file_path, extra_roots)
    if plain is not None and os.path.isfile(plain):  # plain diffuse map: roughness 1, metallic 0, flat normal (:75-84)
        out[:, :, 0:3] = _resized_xy(_open_image(plain), (w, h))[:, :, :3]
        return out, flags

    def part(suffix):
        p = resolve_asset(file_path + suffix, extra_roots)
        return _open_image(p) if p else None

    albedo, rough, metal, normal = part("_albedo.png"), part("_roughness.png"), part("_metallic.png"), part("_normal.png")
    if albedo is None:
        # PBR set without its albedo map in this checkout: documented constant fallback (see FALLBACK_TEXEL)
        return out, flags
    out[:, :, 0:3] = _resized_xy(albedo, (w, h))[:, :, :3]
    if rough is not None:
        out[:, :, 3] = _resized_xy(rough, (w, h), "L")[:, :, 0]
    if metal is not None:
        out[:, :, 7] = _resized_xy(metal, (w, h), "L")[:, :, 0]
    if normal is not None:
        out[:, :, 4:7] = _resized_xy(normal, (w, h))[:, :, :3]
        flags = 0
    return out, flags


def load_environment_image(file_path, extra_roots=()):
    """float32 [w,h,3] indexed [x,y] with y up; PNG/JPG scaled by 1/255, EXR as is (15_module.py:118-132)."""
    p = resolve_asset(file_path, extra_roots)
    if p is None:
        raise FileNotFoundError(f"environment map {file_path!r} not found (searched {ASSET_ROOTS})")
    if p.lower().endswith(".exr"):
        os.environ.setdefault("OPENCV_IO_ENABLE_OPENEXR", "1")
        import cv2
        img = cv2.imread(p, cv2.IMREAD_UNCHANGED)
        if img is None:
            raise IOError(f"cannot read {p}")
        env = img[:, :, 2::-1].astype(np.float32)  # BGR -> RGB
    else:
        env = np.asarray(_open_image(p).convert("RGB"), np.float32) / np.float32(255.0)
    return np.ascontiguousarray(np.flip(env.transpose(1, 0, 2)[..., :3], 1))


class TextureManager:
    """15_module.py:456-501: ids + sizes, shelf-packed into one atlas by build()."""

    def __init__(self, size):
        self.size = tuple(int(v) for v in size)
        self.configs = []
        self.tree = []

    def add(self, file_path, id, size=None):
        if size is None:
            p = resolve_asset(file_path) or resolve_asset(file_path + "_albedo.png") or resolve_asset(file_path + "_metallic.png")
            if p is None:
                raise FileNotFoundError(file_path)
            if p.lower().endswith(".exr"):  # PIL has no EXR reader; the reference goes through imageio (15_module.py:463-467)
                size = load_environment_image(p).shape[:2]
            else:
                size = _open_image(p).size  # (width, height), as img.shape[1], img.shape[0]
        self.configs.append({"file_path": file_path, "size": (int(size[0]), int(size[1])), "id": int(id)})

    def clear(self):
        self.configs = []

    def _traverse_tree(self, size):
        w, h = size
        for i in range(len(self.tree)):
            l, b, r, t = self.tree[i]
            if r - l >= w and t - b >= h:
                self.tree[i] = [l, b + h, r, t]
                self.tree.insert(i, [l + w, b, r, b + h])
                return TextureArea([l, b], [l + w, b + h])
        return None

    def build(self):
        self.tree = [[0, 0, self.size[0], self.size[1]]]
        self.configs.sort(key=lambda x: x["size"][0], reverse=True)
        self.configs.sort(key=lambda x: x["size"][1], reverse=True)
        for c in self.configs:
            area = self._traverse_tree(c["size"])
            if area is None:
                raise MemoryError("Texture out of memory.")
            c["area"] = area

    def dump(self):
        cfgs = []
        for c in self.configs:
            a = c["area"].as_list()
            cfgs.append({"file_path": c["file_path"], "size": tuple(c["size"]), "id": c["id"],
                         "area": {"low": [a[0], a[1]], "high": [a[2], a[3]]}})
        return {"size": tuple(self.size), "configs": cfgs}

    def load(self, data):
        self.size = tuple(int(v) for v in data["size"])
        self.configs = []
        for c in worldnpy.texture_configs(data):
            a = c["area"]
            self.configs.append({"file_path": c["file_path"], "size": c["size"], "id": c["id"],
                                 "area": TextureArea(a[:2], a[2:])})

    def areas_by_id(self):
        n = 1 + max((c["id"] for c in self.configs), default=-1)
        areas = np.zeros((max(n, 1), 4), np.int32)
        areas[:, 2:] = 1  # unused ids: a 1x1 area at the origin
        for c in self.configs:
            areas[c["id"]] = c["area"].as_list()
        return areas


# ---- camera ------------------------------------------------------------------------------------------
class Camera:
    """15_module.py:350-453.  fov is the HALF angle in degrees (view_width = 2*tan(fov*pi/180), :444); yaw, pitch,
    roll are stored in radians; set_direction takes degrees."""

    def __init__(self, resolution, fov=60, focal_length=1, aperture=0):
        self.resolution = (int(resolution[0]), int(resolution[1]))
        self.fov, self.focal_length, self.aperture = float(fov), float(focal_length), float(aperture)
        self.position = Vec3f(0)
        self.yaw = self.pitch = self.roll = 0.0
        self.update_coord()

    def set_position(self, position):
        self.position = Vec3f(position)

    def set_fov(self, fov):
        self.fov = float(fov)

    def set_len(self, focal_length=1, aperture=0):
        self.focal_length, self.aperture = float(focal_length), float(aperture)

    def set_direction(self, yaw, pitch, roll=0):
        self.yaw, self.pitch, self.roll = (float(v) * math.pi / 180 for v in (yaw, pitch, roll))
        self.update_coord()

    def look_at(self, target, roll=0):
        d = (Vec3f(target) - self.position).normalized()
        self.yaw = math.atan2(-d[0], -d[2])
        self.pitch = math.asin(d[1])
        self.roll = float(roll) * math.pi / 180
        self.update_coord()

    def update_coord(self):
        trans = rotate(self.yaw, self.pitch, self.roll)
        self.front_axis = Vec3f(trans @ np.array([0.0, 0.0, -1.0], np.float32))
        self.right_axis = Vec3f(trans @ np.array([1.0, 0.0, 0.0], np.float32))
        self.up_axis = Vec3f(trans @ np.array([0.0, 1.0, 0.0], np.float32))

    def move_front(self, d):
        self.position = Vec3f(self.position + d * self.front_axis)

    def move_right(self, d):
        self.position = Vec3f(self.position + d * self.right_axis)

    def move_up(self, d):
        self.position = Vec3f(self.position + np.array([0, d, 0], np.float32))

    def rotate(self, yaw, pitch, roll=0):
        self.yaw += yaw
        self.pitch = max(-math.pi + epsilon, min(math.pi - epsilon, self.pitch + pitch))  # sic: +-pi (:419)
        self.roll += roll
        self.update_coord()

    def to_struct(self) -> _lib.PtCamera:
        w, h = self.resolution
        view_w = 2.0 * math.tan(self.fov * math.pi / 180)
        c = _lib.PtCamera()
        c.pos[:] = [float(x) for x in self.position]
        c.front[:] = [float(x) for x in self.front_axis]
        c.right[:] = [float(x) for x in self.right_axis]
        c.up[:] = [float(x) for x in self.up_axis]
        c.view_w, c.view_h = view_w, view_w * (h / w)
        c.focal_length, c.aperture = self.focal_length, self.aperture
        return c

    def get_rays(self, sample=0, seed=1, ctx=None):
        from .render import default_context
        ctx = ctx or default_context()
        return ctx.generate_rays(self.to_struct(), self.resolution[0], self.resolution[1], int(sample), int(seed))

    def get_rays_fast(self, ctx=None):
        """Camera.get_rays_fast (15_module.py:423-436): one un-jittered pinhole ray per pixel through (i/W, j/H) of the
        view rectangle at focal length 1 (the lens settings are ignored); float32 [H*W, 8] = o, tmin, d, tmax."""
        from .render import default_context
        ctx = ctx or default_context()
        return ctx.generate_rays(self.to_struct(), self.resolution[0], self.resolution[1], 0, 0, _lib.PT_FLAG_RAYS_FAST)


def reference_visit_order(tree, n_faces) -> np.ndarray:
    """Order in which MeshBVHTree.hit (15_module.py:756-779) reaches the faces: it pushes left then right, so the
    RIGHT subtree is popped first; faces inside a leaf run in CSR order.  The reference keeps the first face it
    meets among exactly equal t (strict <), so this order decides ties between duplicated / double-sided faces."""
    if tree is None:
        return np.arange(n_faces, dtype=np.int64)
    left, right, data, cut = tree["left"], tree["right"], tree["data"], tree["leaf_cut"]
    order = []
    stack = [0]
    while stack:
        cur = stack.pop()
        if data[cur] >= 0:
            order.extend(range(int(cut[data[cur]]), int(cut[data[cur] + 1])))
        else:
            stack.append(int(left[cur]))
            stack.append(int(right[cur]))
    order = np.asarray(order, np.int64)
    assert len(order) == n_faces and len(np.unique(order)) == n_faces
    return order


def lbvh_to_reference_tree(nodes16, global_prims, tri9, max_leave_objects=4, max_depth=24):
    """Converts the GPU-built LBVH of ONE mesh (Scene.bvh_download(): [n,16] nodes = two child boxes + two child
    refs, plus the primitives kept out of the Morton grid) into the node arrays of the reference's MeshBVHTree
    (15_module.py:716-754): nodes in creation order, `data` = leaf number or -1, leaves as CSR ranges of at most
    `max_leave_objects` faces (more where the depth bound `max_depth` — the reference's stack size — cuts a deeper
    subtree).  Returns (tree dict, face order): the file stores faces in leaf order.  SURVEY 8f-1: files written here
    are traversed efficiently by the reference, no host SAH build needed."""
    tri9 = np.asarray(tri9, np.float32).reshape(-1, 9)
    n_faces = len(tri9)
    plo = tri9.reshape(-1, 3, 3).min(1)
    phi = tri9.reshape(-1, 3, 3).max(1)
    kids = nodes16[:, 12:14].copy().view(np.int32) if len(nodes16) else np.zeros((0, 2), np.int32)

    def subtree_prims(ref):
        out, stack = [], [int(ref)]
        while stack:
            r = stack.pop()
            if r < 0:
                out.append(~r)
            else:
                stack.append(int(kids[r, 1]))
                stack.append(int(kids[r, 0]))
        return out

    # number of primitives below every LBVH node (children always have larger or smaller indices: explicit post-order)
    count = np.zeros(len(nodes16), np.int64)
    if len(nodes16):
        order, stack = [], [0]
        while stack:
            r = stack.pop()
            order.append(r)
            for c in kids[r]:
                if c >= 0:
                    stack.append(int(c))
        for r in reversed(order):
            count[r] = sum(1 if c < 0 else count[c] for c in kids[r])

    left, right, low, high, data, cut, face_order = [], [], [], [], [], [0], []

    def box_of(prims):
        return plo[prims].min(0), phi[prims].max(0)

    def new_node(lo, hi):
        left.append(-1); right.append(-1); low.append(np.asarray(lo, np.float32)); high.append(np.asarray(hi, np.float32))
        data.append(-1)
        return len(left) - 1

    def make_leaf(idx, prims):
        data[idx] = len(cut) - 1
        face_order.extend(prims)
        cut.append(len(face_order))

    glob = [int(g) for g in global_prims]
    all_lo, all_hi = box_of(np.arange(n_faces))
    root = new_node(all_lo, all_hi)
    work = []  # (reference node, LBVH ref, depth)
    if len(nodes16) == 0:  # tree-less mesh (<= 8 faces): one leaf
        make_leaf(root, list(range(n_faces)))
    elif glob:  # root -> [leaf of the oversized faces, the LBVH]
        lo, hi = box_of(glob)
        a = new_node(lo, hi)
        rest = sorted(set(range(n_faces)) - set(glob))
        lo, hi = box_of(rest)
        b = new_node(lo, hi)
        left[root], right[root] = a, b
        make_leaf(a, glob)
        work.append((b, 0, 1))
    else:
        work.append((root, 0, 0))
    qi = 0
    while qi < len(work):  # breadth first, like the reference's builder
        idx, ref, depth = work[qi]
        qi += 1
        if ref < 0:
            make_leaf(idx, [~ref])
            continue
        if count[ref] <= max_leave_objects or depth >= max_depth:
            make_leaf(idx, subtree_prims(ref))
            continue
        n = nodes16[ref]
        a = new_node(n[0:3], n[3:6])
        b = new_node(n[6:9], n[9:12])
        left[idx], right[idx] = a, b
        work.append((a, int(kids[ref, 0]), depth + 1))
        work.append((b, int(kids[ref, 1]), depth + 1))
    face_order = np.asarray(face_order, np.int64)
    assert len(face_order) == n_faces and len(np.unique(face_order)) == n_faces
    tree = {"left": np.asarray(left, np.int32), "right": np.asarray(right, np.int32), "low": np.stack(low), "high": np.stack(high),
            "data": np.asarray(data, np.int32), "leaf_cut": np.asarray(cut, np.int32), "max_depth": int(max_depth)}
    return tree, face_order


# ---- world -------------------------------------------------------------------------------------------
class World:
    """15_module.py:782-848."""
    shading_model = _lib.PT_SHADE_LEGACY  # gen_secondary_rays (15_module.py:994-1013); read by render_distributed

    def __init__(self, texture_size=texture_size, environment_size=environment_size):
        self.spheres = []
        self.meshes = []          # dicts: positions, normals, texture_coords, indices [F,10], optional stored tree
        self.environment = None
        self.textures = TextureManager(texture_size)
        self.environments = TextureManager(environment_size)
        self.asset_roots = []
        self._atlas = None        # (texels uint8 [W,H,8], areas [ntex,4], flags [ntex])
        self._env = None          # (rgb float32 [W,H,3], area[4]) or None -> sky gradient
        self._scene = None
        self._scene_ctx = None

    # -- description
    def add_mesh(self, positions, normals, texture_coords, indices, tree=None):
        self.meshes.append({"positions": np.asarray(positions, np.float32).reshape(-1, 3),
                            "normals": np.asarray(normals, np.float32).reshape(-1, 3),
                            "texture_coords": np.asarray(texture_coords, np.float32).reshape(-1, 2),
                            "indices": _faces_array(indices), "tree": tree})
        self._scene = None

    def add_sphere(self, sphere):
        self.spheres.append(sphere)
        self._scene = None

    def set_environment(self, id):
        self.environment = id
        self._env = None
        self._scene = None

    # -- textures
    def set_atlas(self, texels, areas, flags=None):
        """Directly supply the 8-byte-per-texel atlas (tests, scene caches)."""
        areas = np.asarray(areas, np.int32).reshape(-1, 4)
        self._atlas = (np.ascontiguousarray(texels, np.uint8), areas,
                       np.zeros(len(areas), np.int32) if flags is None else np.asarray(flags, np.int32))
        self._scene = None

    def set_environment_image(self, rgb, area=None):
        self._env = None if rgb is None else (np.ascontiguousarray(rgb, np.float32),
                                              list(area) if area is not None else [0, 0, rgb.shape[0], rgb.shape[1]])
        self._scene = None

    def load_textures(self):
        """load_texture + load_environment (15_module.py:65-132) for the managers' configs."""
        if self.textures.configs:
            areas = self.textures.areas_by_id()
            used_w = max(int(a[2]) for a in areas)
            used_h = max(int(a[3]) for a in areas)
            texels = np.empty((used_w, used_h, 8), np.uint8)
            texels[...] = FALLBACK_TEXEL
            flags = np.ones(len(areas), np.int32)
            for c in self.textures.configs:
                a = c["area"].as_list()
                t, f = load_texture_texels(c["file_path"], (a[2] - a[0], a[3] - a[1]), self.asset_roots)
                texels[a[0]:a[2], a[1]:a[3]] = t
                flags[c["id"]] = f
            self._atlas = (texels, areas, flags)
        if self.environments.configs and self.environment is not None:
            W, H = self.environments.size
            env = np.zeros((W, H, 3), np.float32)
            area = None
            for c in self.environments.configs:
                a = c["area"].as_list()
                img = load_environment_image(c["file_path"], self.asset_roots)
                if img.shape[:2] != (a[2] - a[0], a[3] - a[1]):
                    raise ValueError(f"environment {c['file_path']}: image {img.shape[:2]} != area {a}")
                env[a[0]:a[2], a[1]:a[3]] = img
                if c["id"] == self.environment:
                    area = a
            if area is not None:
                self._env = (env, area)
        self._scene = None

    def build(self):
        """World.build (15_module.py:802-813): pack + load textures; the BVH is built on the GPU at device_scene()."""
        self.textures.build()
        self.environments.build()
        self.load_textures()

    # -- persistence
    def build_trees(self, ctx=None, max_leave_objects=4, max_depth=24):
        """Gives every mesh that has no stored tree one in the reference's schema, from an LBVH built on the GPU
        (replaces the reference's host-Python SAH build, 15_module.py:716-754, minutes -> milliseconds); faces are
        reordered to leaf order as in the reference's files."""
        from .render import default_context
        ctx = ctx or default_context()
        for m in self.meshes:
            if m.get("tree") is not None:
                continue
            f = m["indices"]
            tri9 = m["positions"][f[:, [0, 3, 6]]].reshape(-1, 9)
            sc = _lib.Scene(ctx)
            sc.set_triangles(tri9)
            sc.build()
            nodes, glob = sc.bvh_download()
            sc.close()
            tree, order = lbvh_to_reference_tree(nodes, glob, tri9, max_leave_objects, max_depth)
            m["tree"], m["indices"] = tree, f[order]
            m["_visit_order"] = None
        self._scene = None

    def save(self, filename, build_trees=True, ctx=None):
        """World.save (15_module.py:815-821).  Meshes without a stored tree get one from the GPU builder first
        (build_trees=False writes a single-leaf tree instead, valid but brute force for the reference)."""
        if build_trees and any(m.get("tree") is None for m in self.meshes):
            self.build_trees(ctx)
        meshes = [{"positions": m["positions"], "normals": m["normals"], "texcoords": m["texture_coords"],
                   "faces": m["indices"], "tree": m["tree"]} for m in self.meshes]
        spheres = None
        if self.spheres:
            cr, tr, tx = self.sphere_arrays()
            spheres = {"max_depth": 8,
                       "tree_nodes_field": {"data": {"left": np.array([-1], np.int32), "right": np.array([-1], np.int32),
                                                     "aabb": {"low": (cr[:, :3] - cr[:, 3:]).min(0)[None],
                                                              "high": (cr[:, :3] + cr[:, 3:]).max(0)[None]},
                                                     "data": np.array([0], np.int32)}, "shape": [1]},
                       "tree_leaves_field": {"data": {"center": cr[:, :3].copy(), "radius": cr[:, 3].copy(),
                                                      "transparency": tr, "texture_id": tx}, "shape": [len(cr)]},
                       "tree_leaves_field_cut": {"data": np.array([0, len(cr)], np.int32), "shape": [2]}}
        worldnpy.save_world(filename, meshes, self.environment if self.environment is not None else 0,
                            self.textures.dump() if self.textures.configs else None,
                            self.environments.dump() if self.environments.configs else None, spheres)

    def load(self, filename, load_images=True):
        """World.load (15_module.py:823-836; old-format files as 14_mesh.py:766-776: geometry only)."""
        data = worldnpy.load_world(filename)
        self.asset_roots = [os.path.dirname(os.path.abspath(filename))] + self.asset_roots
        self.environment = data.get("environment")
        if "textures" in data:
            self.textures.load(data["textures"])
        if "environments" in data:
            self.environments.load(data["environments"])
        if "spheres_bvh" in data:
            s = worldnpy.sphere_arrays(data["spheres_bvh"])
            for cr, tr, tx in zip(s["center_radius"], s["transparency"], s["texture_id"]):
                self.spheres.append(Sphere(cr[:3], cr[3], tr, tx))
        for md in data["meshes_bvhs"]:
            m = worldnpy.mesh_arrays(md)
            self.add_mesh(m["positions"], m["normals"], m["texcoords"], m["faces"], tree=m["tree"])
        if load_images and (self.textures.configs or self.environments.configs):
            self.load_textures()

    # -- device interface
    def sphere_arrays(self):
        n = len(self.spheres)
        cr = np.zeros((n, 4), np.float32)
        tr = np.zeros(n, np.int32)
        tx = np.zeros(n, np.int32)
        for i, s in enumerate(self.spheres):
            cr[i, :3], cr[i, 3], tr[i], tx[i] = s.center, s.radius, s.transparency, s.texture_id
        return cr, tr, tx

    def device_scene(self, ctx):
        if self._scene is None or self._scene_ctx is not ctx:
            sc = _lib.Scene(ctx)
            if self.spheres:
                sc.set_textured_spheres(*self.sphere_arrays())
            perm, base = [], 0
            for m in self.meshes:
                # device primitive order = the reference traversal's visitation order, so that "lowest id wins an
                # exact tie" (extend.cuh) picks the face the reference would have kept
                if m.get("_visit_order") is None or len(m["_visit_order"]) != len(m["indices"]):
                    m["_visit_order"] = reference_visit_order(m.get("tree"), len(m["indices"]))  # depends on the tree only
                order = m["_visit_order"]
                sc.add_mesh(m["positions"], m["normals"], m["texture_coords"], m["indices"][order])
                perm.append(base + order)
                base += len(order)
            self._tri_perm = np.concatenate(perm) if perm else np.zeros(0, np.int64)
            if self._atlas is None:
                raise _lib.PtError("legacy World has no texture atlas: call build()/load_textures() or set_atlas()")
            sc.set_texture_atlas(*self._atlas)
            if self._env is not None:
                sc.set_environment(self._env[0], self._env[1])
            else:
                sc.set_environment(None)
            sc.build()
            self._scene, self._scene_ctx = sc, ctx
        return self._scene

    def hit(self, rays, ctx=None):
        """World.hit over a ray batch [n,8] -> (global primitive id, t): spheres first, then mesh faces in order."""
        from .render import default_context
        ctx = ctx or default_context()
        ids, t, _ = ctx.trace_batch(self.device_scene(ctx), rays)
        n_sph = len(self.spheres)
        tri = ids >= n_sph
        ids = ids.copy()
        ids[tri] = n_sph + self._tri_perm[ids[tri] - n_sph]  # device order -> the caller's face order
        return ids, t


class LegacyRenderer:
    """render(moved) + gamma_correction of 15_module.py:1016-1036 with the script's module constants as fields.

    Under an initialised torch.distributed process group (one rank per GPU) every pass of `spp` samples is split
    over the ranks (multigpu.render_split_reduce: disjoint sample ranges, scene replicated, accumulators summed onto
    rank 0 over NCCL); rank 0 owns the progressive image and returns the frame, the other ranks return None.
    distributed=False keeps a renderer local to its rank.
    devices (a list of CUDA device indices, or "all"; the first one is the context's) splits every pass over those devices
    from this one process instead (render.MultiRenderer); it does not combine with a process group.
    denoise=True returns denoised frames (Renderer.denoised()): the guide features of a pose are computed once, when the
    image restarts (render(moved=True)), and serve every progressive pass of that pose.  The process-group path reduces
    RGB only, not the sum of squares the filter needs, so denoise=True refuses an active process group."""

    def __init__(self, world: World, camera: Camera, spp=32, propagate_limit=32, absorptivity=0.25, seed=1, ctx=None,
                 distributed=True, group=None, bands=1, devices=None, denoise=False):
        from .render import MultiRenderer, Renderer, default_context
        self.ctx = ctx or default_context()
        self.world, self.camera = world, camera
        self.spp, self.propagate_limit, self.absorptivity, self.seed = int(spp), int(propagate_limit), float(absorptivity), seed
        self.group, self.bands = group, int(bands)
        self.distributed = bool(distributed)
        self.denoise = bool(denoise)
        self.feature_passes = 0  # pt_render_features calls made (one per pose)
        if self.denoise and self.distributed:
            from .multigpu import _dist_active
            if _dist_active(self.group):
                raise ValueError("LegacyRenderer: denoise=True needs the sum of squares, which the process-group path does "
                                 "not reduce; pass distributed=False, or devices= to split passes within this process")
        if devices is not None:
            from .multigpu import _dist_active
            if self.distributed and _dist_active(self.group):
                raise ValueError("LegacyRenderer: devices= splits passes within this process; with an active process group "
                                 "pass distributed=False (or leave devices=None to split over the ranks)")
            self.renderer = MultiRenderer(camera.resolution[0], camera.resolution[1], devices, self.ctx, want_sq=self.denoise)
        else:
            self.renderer = Renderer(camera.resolution[0], camera.resolution[1], self.ctx, want_sq=self.denoise)
        self.frame = None
        self._total = 0       # samples per pixel in the image (over all ranks)
        self._partial = None  # ranks > 0: scratch accumulator of one pass

    @property
    def total_spp(self):
        return self._total

    def _ranks(self):
        if not self.distributed:
            return 1, 0
        from .multigpu import _dist_active
        if not _dist_active(self.group):
            return 1, 0
        import torch.distributed as dist
        return dist.get_world_size(self.group), dist.get_rank(self.group)

    def render(self, moved=True, spp_offset=None):
        """Adds `spp` samples per pixel (progressive unless moved) and returns frame = (image/spp)^(1/2.2).
        spp_offset: first sample index of this pass (default: continue after the samples already in the image)."""
        from .multigpu import render_split_reduce
        ws, rank = self._ranks()
        if moved:
            self.renderer.clear()
            self._total = 0
        first = self._total if spp_offset is None else int(spp_offset)
        scene = self.world.device_scene(self.ctx)
        if self.denoise and (moved or self.feature_passes == 0):
            self.renderer.features(scene, self.camera.to_struct(), 4, self.seed, 0, 0, _lib.PT_SHADE_LEGACY)
            self.feature_passes += 1
        if ws == 1:
            self.renderer.render(scene, self.camera.to_struct(), self.spp, self.propagate_limit, _lib.PT_SHADE_LEGACY,
                                 self.seed, spp_offset=first, absorptivity=self.absorptivity, want_stats=False)
        else:
            # the pass of every rank lands in a scratch accumulator that is summed onto rank 0 and added to its image
            torch = self.renderer.torch
            if self._partial is None:
                from .render import Renderer
                self._partial = Renderer(self.renderer.width, self.renderer.height, self.ctx)
            self._partial.clear()
            render_split_reduce(self._partial, scene, self.camera.to_struct(), self.spp, self.propagate_limit,
                                _lib.PT_SHADE_LEGACY, self.seed, self.group, absorptivity=self.absorptivity,
                                bands=self.bands, first_sample=first)
            if rank == 0:
                torch.add(self.renderer.accum, self._partial.accum, out=self.renderer.accum)
        self._total += self.spp
        self.renderer.spp_done = self._total
        if rank != 0:
            self.frame = None
            return None
        self.frame = self.renderer.image(aces=False, gamma=2.2, total_spp=self._total, denoise=self.denoise)
        return self.frame

    def frames(self, camera_path, passes_per_pose=1):
        """Frame streaming (the consumer of Camera.move_*/rotate that 12_free_view.py:553-579 / 15_module.py:403-421 feed
        a ti.GUI with): for every pose of `camera_path` — a callable pose(camera) that moves the camera in place, or
        None to keep it — the image restarts (render(moved=True)) and `passes_per_pose` progressive passes are yielded
        as (pose index, pass index, frame).  The device scene is built once and reused for the whole stream."""
        for k, pose in enumerate(camera_path):
            if pose is not None:
                pose(self.camera)
            for j in range(int(passes_per_pose)):
                yield k, j, self.render(moved=(j == 0))
