"""ctypes binding of libb200pt.so (the C-ABI declared in include/pt_api.h).

There is deliberately NO fallback: if the CUDA library is missing or no B200 is visible, every
compute entry point raises.  The CPU oracle under oracle/ is test infrastructure and is never
imported from here.
"""
from __future__ import annotations

import ctypes as C
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
# PT_LIB_PATH: a variant build of the SAME library (tools/build_variants.sh: A/B experiments); never a fallback
LIB_PATH = os.environ.get("PT_LIB_PATH") or os.path.join(_HERE, "libb200pt.so")

PT_SHADE_V2 = 0
PT_SHADE_V2_DIFFUSE = 1
PT_SHADE_LEGACY = 2
PT_SHADE_V2_NORMALS = 3
PT_SHADE_LEGACY_STAGE7 = 4  # legacy/PT_in_one_weekend/7_reflect.py: untextured ancestor of gen_secondary_rays
PT_SHADE_LEGACY_STAGE6 = 5  # legacy/PT_in_one_weekend/6_diffuse.py: diffuse only, throughput 0.5 * albedo

PT_FLAG_ACCUM_SQ = 1
PT_FLAG_TIMING = 2
PT_FLAG_COUNTERS = 4
PT_FLAG_TRACE_WIDE = 128  # `make EXPERIMENTAL=1` builds only: 4-wide traversal (scene built with PT_WIDE=1); measured slower
PT_FLAG_WIDE = PT_FLAG_TRACE_WIDE  # the same bit in PtRenderParams.flags (persistent mode)
PT_FLAG_RAYS_FAST = 256  # generate_rays: legacy Camera.get_rays_fast lattice (i/W, pinhole)
PT_FLAG_PIXEL_GRID = 64  # stages 2-4 camera: lattice rays i/(W-1), j/(H-1), no jitter

PT_MODE_AUTO = 0
PT_MODE_SPLIT = 1   # classic wavefront: k_extend + k_shade per bounce, pool refilled by an atomic counter
PT_MODE_FUSED = 2   # k_paths: K segments per launch in registers, compaction at write-back (the HBM path-pool wavefront)
PT_MODE_PERSIST = 3  # k_paths_persist: persistent while-while lanes, one launch per render (auto)
PT_MODE_QUEUE = 4    # `make EXPERIMENTAL=1` builds only: persistent lanes + block-local shading queues in shared memory
PT_MODE_DUAL = 5     # `make EXPERIMENTAL=1` builds only: persistent lanes with a lane-private parking place
PT_FLAG_NO_SORT = 8        # pt_trace_batch_device: keep batch order
PT_FLAG_TRACE_SIMPLE = 16  # pt_trace_batch_device: one ray per thread (k_trace)
PT_FLAG_NO_QNODES = 32     # pt_trace_batch_device: 64-byte float nodes even when the quantised copy exists


class PtMaterial(C.Structure):
    _fields_ = [("albedo", C.c_float * 3), ("roughness", C.c_float), ("metallic", C.c_int32),
                ("ior", C.c_float), ("transparency", C.c_int32), ("_pad", C.c_int32)]


class PtCamera(C.Structure):
    _fields_ = [("pos", C.c_float * 3), ("front", C.c_float * 3), ("right", C.c_float * 3),
                ("up", C.c_float * 3), ("view_w", C.c_float), ("view_h", C.c_float),
                ("focal_length", C.c_float), ("aperture", C.c_float)]


class PtRenderParams(C.Structure):
    _fields_ = [("width", C.c_int32), ("height", C.c_int32), ("spp", C.c_int32), ("spp_offset", C.c_int32),
                ("max_depth", C.c_int32), ("shading_model", C.c_int32), ("seed", C.c_uint32),
                ("absorptivity", C.c_float), ("pool_capacity", C.c_int32), ("flags", C.c_int32),
                ("reserved", C.c_int32 * 6)]


class PtStats(C.Structure):
    _fields_ = [("paths", C.c_uint64), ("segments", C.c_uint64), ("nodes_visited", C.c_uint64),
                ("prims_tested", C.c_uint64), ("ms_total", C.c_float), ("ms_extend", C.c_float),
                ("ms_shade", C.c_float), ("ms_other", C.c_float), ("iterations", C.c_int32),
                ("launches", C.c_int32), ("launches_extend", C.c_int32), ("launches_shade", C.c_int32),
                ("reserved", C.c_int32 * 4)]

    def as_dict(self):
        return {n: getattr(self, n) for n, _ in self._fields_ if n != "reserved"}


class PtDenoiseParams(C.Structure):
    _fields_ = [("width", C.c_int32), ("height", C.c_int32), ("spp", C.c_int32), ("iterations", C.c_int32),
                ("sigma_l", C.c_float), ("sigma_n", C.c_float), ("sigma_z", C.c_float), ("_pad", C.c_int32)]


assert C.sizeof(PtMaterial) == 32 and C.sizeof(PtCamera) == 64 and C.sizeof(PtDenoiseParams) == 32
assert C.sizeof(PtRenderParams) == 64 and C.sizeof(PtStats) == 80

MATERIAL_DTYPE = np.dtype([("albedo", "<f4", 3), ("roughness", "<f4"), ("metallic", "<i4"), ("ior", "<f4"),
                           ("transparency", "<i4"), ("_pad", "<i4")])
assert MATERIAL_DTYPE.itemsize == 32

# every symbol include/pt_api.h declares (tests check that the built library exports all of them)
API_SYMBOLS = [
    "pt_context_create", "pt_context_destroy", "pt_context_set_stream", "pt_context_sync",
    "pt_scene_create", "pt_scene_destroy", "pt_scene_set_spheres", "pt_scene_set_textured_spheres",
    "pt_scene_add_mesh", "pt_scene_set_triangles", "pt_scene_set_random_triangles",
    "pt_scene_set_texture_atlas", "pt_scene_set_environment", "pt_scene_build", "pt_scene_bvh_info",
    "pt_scene_bvh_download", "pt_scene_triangles_download", "pt_generate_rays", "pt_trace_batch",
    "pt_trace_batch_device", "pt_random_rays_device", "pt_render", "pt_render_host", "pt_postprocess",
    "pt_postprocess_host", "pt_download_accum", "pt_measure_fp32_peak", "pt_last_error", "pt_version",
    "pt_render_stats", "pt_build_info", "pt_generate_rays_ex", "pt_multi_create", "pt_multi_destroy", "pt_multi_render",
    "pt_scene_replicate", "pt_render_features", "pt_denoise",
]


class PtError(RuntimeError):
    pass


_lib = None


def _fptr(a, dtype=np.float32):
    if a is None:
        return None
    assert isinstance(a, np.ndarray) and a.dtype == dtype and a.flags["C_CONTIGUOUS"], (a.dtype, dtype)
    return a.ctypes.data_as(C.c_void_p)


def load():
    """Load libb200pt.so; raises PtError (never falls back) when it has not been built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise PtError(f"{LIB_PATH} not found: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
                      "(make -C learn_path_tracing_b200/csrc). There is no CPU fallback.")
    lib = C.CDLL(LIB_PATH)
    vp, i32, i64, u32, f32 = C.c_void_p, C.c_int, C.c_int64, C.c_uint32, C.c_float
    P = C.POINTER
    sig = {
        "pt_context_create": (i32, [i32, vp, P(vp)]),
        "pt_context_destroy": (None, [vp]),
        "pt_context_set_stream": (i32, [vp, vp]),
        "pt_context_sync": (i32, [vp]),
        "pt_scene_create": (i32, [vp, P(vp)]),
        "pt_scene_destroy": (None, [vp]),
        "pt_scene_set_spheres": (i32, [vp, vp, vp, i32]),
        "pt_scene_set_textured_spheres": (i32, [vp, vp, vp, vp, i32]),
        "pt_scene_add_mesh": (i32, [vp, vp, i32, vp, i32, vp, i32, vp, i32]),
        "pt_scene_set_triangles": (i32, [vp, vp, i64]),
        "pt_scene_set_random_triangles": (i32, [vp, i64, u32, f32]),
        "pt_scene_set_texture_atlas": (i32, [vp, vp, i32, i32, vp, vp, i32]),
        "pt_scene_set_environment": (i32, [vp, vp, i32, i32, vp]),
        "pt_scene_build": (i32, [vp]),
        "pt_scene_bvh_info": (i32, [vp, P(i64), P(i64), P(i64)]),
        "pt_scene_bvh_download": (i32, [vp, vp, i64, vp, i64]),
        "pt_scene_triangles_download": (i32, [vp, vp, i64]),
        "pt_generate_rays": (i32, [vp, P(PtCamera), i32, i32, i32, u32, vp]),
        "pt_trace_batch": (i32, [vp, vp, vp, i64, vp, vp, P(PtStats)]),
        "pt_trace_batch_device": (i32, [vp, vp, vp, i64, vp, i32, P(PtStats)]),
        "pt_random_rays_device": (i32, [vp, vp, i64, u32]),
        "pt_render": (i32, [vp, vp, P(PtCamera), P(PtRenderParams), vp, vp, P(PtStats)]),
        "pt_render_host": (i32, [vp, vp, P(PtCamera), P(PtRenderParams), vp, vp, P(PtStats)]),
        "pt_postprocess": (i32, [vp, vp, i32, i32, f32, i32, f32, vp]),
        "pt_postprocess_host": (i32, [vp, vp, i32, i32, f32, i32, f32, vp]),
        "pt_download_accum": (i32, [vp, vp, i32, i32, vp]),
        "pt_measure_fp32_peak": (i32, [vp, P(f32)]),
        "pt_last_error": (C.c_char_p, []),
        "pt_version": (i32, []),
        "pt_render_stats": (i32, [vp, P(PtStats)]),
        "pt_build_info": (C.c_char_p, []),
        "pt_generate_rays_ex": (i32, [vp, P(PtCamera), i32, i32, i32, u32, i32, vp]),
        "pt_multi_create": (i32, [P(vp), i32, P(vp)]),
        "pt_multi_destroy": (None, [vp]),
        "pt_multi_render": (i32, [vp, P(vp), P(PtCamera), P(PtRenderParams), vp, vp, P(PtStats)]),
        "pt_scene_replicate": (i32, [vp, vp, P(vp)]),
        "pt_render_features": (i32, [vp, vp, P(PtCamera), P(PtRenderParams), vp]),
        "pt_denoise": (i32, [vp, vp, vp, vp, P(PtDenoiseParams), vp]),
    }
    for name, (res, args) in sig.items():
        fn = getattr(lib, name)  # AttributeError if the library lacks a declared symbol
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


def has_experimental() -> bool:
    """True when the loaded library was built with `make EXPERIMENTAL=1` (render modes 4/5, PT_FLAG_WIDE)."""
    return b"experimental=1" in load().pt_build_info()


def host_image(width: int, height: int) -> np.ndarray:
    """float32 [W,H,3] output buffer in PINNED host memory (torch's caching host allocator), so the
    device->host read of an image is a single DMA; falls back to pageable numpy memory without torch."""
    try:
        import torch
        t = torch.empty((width, height, 3), dtype=torch.float32, pin_memory=True)
        return t.numpy()  # keeps the pinned storage alive
    except Exception:
        return np.empty((width, height, 3), np.float32)


def check(rc: int):
    if rc != 0:
        msg = load().pt_last_error()
        raise PtError(f"libb200pt error {rc}: {msg.decode() if msg else '?'}")


class Context:
    """One per GPU (pt_context_create).  `stream` is a raw cudaStream_t handle (int) or None."""

    def __init__(self, device: int = 0, stream: int | None = None):
        self.lib = load()
        h = C.c_void_p()
        check(self.lib.pt_context_create(int(device), C.c_void_p(stream or 0), C.byref(h)))
        self.handle = h
        self.device = int(device)

    def set_stream(self, stream: int | None):
        check(self.lib.pt_context_set_stream(self.handle, C.c_void_p(stream or 0)))

    def sync(self):
        check(self.lib.pt_context_sync(self.handle))

    def close(self):
        if getattr(self, "handle", None):
            self.lib.pt_context_destroy(self.handle)
            self.handle = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # ---- hot-path calls -------------------------------------------------------------------
    def generate_rays(self, cam: PtCamera, width: int, height: int, sample: int, seed: int, flags: int = 0) -> np.ndarray:
        rays = np.empty((height * width, 8), np.float32)
        check(self.lib.pt_generate_rays_ex(self.handle, C.byref(cam), width, height, sample, seed, int(flags), _fptr(rays)))
        return rays

    def trace_batch(self, scene: "Scene", rays: np.ndarray, counters: bool = False, out=None):
        """World.hit over a host ray batch [n,8] -> (prim ids, t, stats).  out=(ids int32[n], t float32[n]) reuses the
        caller's result arrays (fresh numpy arrays cost a page fault per 4 KiB on their first write)."""
        rays = np.ascontiguousarray(rays, np.float32).reshape(-1, 8)
        n = rays.shape[0]
        if out is not None:
            ids, t = out
            if not (ids.dtype == np.int32 and t.dtype == np.float32 and ids.shape == (n,) and t.shape == (n,)
                    and ids.flags.c_contiguous and t.flags.c_contiguous):
                raise PtError("trace_batch: out must be (int32[n], float32[n]) contiguous arrays")
        else:
            ids = np.empty(n, np.int32)
            t = np.empty(n, np.float32)
        st = PtStats()  # filled (and the counting kernel variant used) only when counters=True
        check(self.lib.pt_trace_batch(self.handle, scene.handle, _fptr(rays), n, _fptr(ids, np.int32), _fptr(t),
                                      C.byref(st) if counters else None))
        return ids, t, st

    def trace_batch_device(self, scene: "Scene", rays_ptr: int, n: int, hits_ptr: int, flags: int = 0) -> PtStats:
        st = PtStats()
        check(self.lib.pt_trace_batch_device(self.handle, scene.handle, C.c_void_p(rays_ptr), n,
                                             C.c_void_p(hits_ptr), flags, C.byref(st)))
        return st

    def random_rays_device(self, rays_ptr: int, n: int, seed: int):
        check(self.lib.pt_random_rays_device(self.handle, C.c_void_p(rays_ptr), n, seed))

    def render(self, scene: "Scene", cam: PtCamera, params: PtRenderParams, accum_ptr: int,
               accum_sq_ptr: int | None = None, want_stats: bool = True) -> PtStats | None:
        """pt_render.  want_stats=False: nothing waits for the GPU — the call returns as soon as the kernel is enqueued on
        the context's stream (ask render_stats() later); the multi-GPU path chains its reduce behind it that way."""
        st = PtStats() if want_stats else None
        check(self.lib.pt_render(self.handle, scene.handle, C.byref(cam), C.byref(params), C.c_void_p(accum_ptr),
                                 C.c_void_p(accum_sq_ptr or 0), C.byref(st) if want_stats else None))
        return st

    def render_stats(self) -> PtStats:
        """Statistics of the last render() on this context (waits for that render only)."""
        st = PtStats()
        check(self.lib.pt_render_stats(self.handle, C.byref(st)))
        return st

    def render_features(self, scene: "Scene", cam: PtCamera, params: PtRenderParams, features_ptr: int):
        """pt_render_features: first-hit normal / depth / albedo of samples [spp_offset, spp_offset + spp) ADDED into
        features_ptr (float4[2][h*w]); asynchronous on the context's stream."""
        check(self.lib.pt_render_features(self.handle, scene.handle, C.byref(cam), C.byref(params), C.c_void_p(features_ptr)))

    def denoise(self, accum_ptr: int, accum_sq_ptr: int | None, features_ptr: int, width: int, height: int, spp: int,
                out_ptr: int, iterations: int = 5, sigma_l: float = 0.0, sigma_n: float = 0.0, sigma_z: float = 0.0):
        """pt_denoise: the denoised mean radiance (float4[h*w], w = 1) into out_ptr; asynchronous on the context's stream."""
        p = PtDenoiseParams(int(width), int(height), int(spp), int(iterations), float(sigma_l), float(sigma_n),
                            float(sigma_z), 0)
        check(self.lib.pt_denoise(self.handle, C.c_void_p(accum_ptr), C.c_void_p(accum_sq_ptr or 0),
                                  C.c_void_p(features_ptr), C.byref(p), C.c_void_p(out_ptr)))

    def render_host(self, scene: "Scene", cam: PtCamera, params: PtRenderParams, want_sq: bool = False):
        W, H = params.width, params.height
        accum = np.empty((W, H, 3), np.float32)
        sq = np.empty((W, H, 3), np.float32) if want_sq else None
        if want_sq:
            params.flags |= PT_FLAG_ACCUM_SQ
        st = PtStats()
        check(self.lib.pt_render_host(self.handle, scene.handle, C.byref(cam), C.byref(params), _fptr(accum),
                                      _fptr(sq), C.byref(st)))
        return accum, sq, st

    def postprocess(self, accum_ptr: int, width: int, height: int, scale: float, aces: bool, gamma: float,
                    out_ptr: int):
        check(self.lib.pt_postprocess(self.handle, C.c_void_p(accum_ptr), width, height, scale, int(aces), gamma,
                                      C.c_void_p(out_ptr)))

    def postprocess_host(self, accum_ptr: int, width: int, height: int, scale: float, aces: bool,
                         gamma: float) -> np.ndarray:
        out = host_image(width, height)
        check(self.lib.pt_postprocess_host(self.handle, C.c_void_p(accum_ptr), width, height, scale, int(aces),
                                           gamma, _fptr(out)))
        return out

    def download_accum(self, accum_ptr: int, width: int, height: int) -> np.ndarray:
        out = host_image(width, height)
        check(self.lib.pt_download_accum(self.handle, C.c_void_p(accum_ptr), width, height, _fptr(out)))
        return out

    def measure_fp32_peak(self) -> float:
        v = C.c_float()
        check(self.lib.pt_measure_fp32_peak(self.handle, C.byref(v)))
        return float(v.value)


class Scene:
    """Device-resident scene (pt_scene_*)."""

    def __init__(self, ctx: Context):
        self.ctx = ctx
        self.lib = ctx.lib
        h = C.c_void_p()
        check(self.lib.pt_scene_create(ctx.handle, C.byref(h)))
        self.handle = h

    def close(self):
        if getattr(self, "handle", None):
            self.lib.pt_scene_destroy(self.handle)
            self.handle = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def set_spheres(self, center_radius: np.ndarray, materials: np.ndarray):
        cr = np.ascontiguousarray(center_radius, np.float32).reshape(-1, 4)
        mats = np.ascontiguousarray(materials, MATERIAL_DTYPE)
        assert mats.shape[0] == cr.shape[0]
        check(self.lib.pt_scene_set_spheres(self.handle, _fptr(cr), mats.ctypes.data_as(C.c_void_p), cr.shape[0]))

    def set_textured_spheres(self, center_radius, transparency, texture_id):
        cr = np.ascontiguousarray(center_radius, np.float32).reshape(-1, 4)
        tr = np.ascontiguousarray(transparency, np.int32)
        tx = np.ascontiguousarray(texture_id, np.int32)
        check(self.lib.pt_scene_set_textured_spheres(self.handle, _fptr(cr), _fptr(tr, np.int32),
                                                     _fptr(tx, np.int32), cr.shape[0]))

    def add_mesh(self, positions, normals, texcoords, faces):
        p = np.ascontiguousarray(positions, np.float32).reshape(-1, 3)
        n = np.ascontiguousarray(normals, np.float32).reshape(-1, 3)
        t = np.ascontiguousarray(texcoords, np.float32).reshape(-1, 2)
        f = np.ascontiguousarray(faces, np.int32).reshape(-1, 10)
        check(self.lib.pt_scene_add_mesh(self.handle, _fptr(p), p.shape[0], _fptr(n), n.shape[0], _fptr(t),
                                         t.shape[0], _fptr(f, np.int32), f.shape[0]))

    def set_triangles(self, verts):
        v = np.ascontiguousarray(verts, np.float32).reshape(-1, 9)
        check(self.lib.pt_scene_set_triangles(self.handle, _fptr(v), v.shape[0]))

    def set_random_triangles(self, n: int, seed: int, edge_scale: float):
        check(self.lib.pt_scene_set_random_triangles(self.handle, n, seed, edge_scale))

    def set_texture_atlas(self, texels: np.ndarray, areas: np.ndarray, flags: np.ndarray | None = None):
        tx = np.ascontiguousarray(texels, np.uint8)
        assert tx.ndim == 3 and tx.shape[2] == 8
        ar = np.ascontiguousarray(areas, np.int32).reshape(-1, 4)
        fl = np.zeros(ar.shape[0], np.int32) if flags is None else np.ascontiguousarray(flags, np.int32)
        assert fl.shape[0] == ar.shape[0]
        check(self.lib.pt_scene_set_texture_atlas(self.handle, _fptr(tx, np.uint8), tx.shape[0], tx.shape[1],
                                                  _fptr(ar, np.int32), _fptr(fl, np.int32), ar.shape[0]))

    def set_environment(self, rgb: np.ndarray | None, area=None):
        if rgb is None:
            check(self.lib.pt_scene_set_environment(self.handle, None, 0, 0, None))
            return
        e = np.ascontiguousarray(rgb, np.float32)
        assert e.ndim == 3 and e.shape[2] == 3
        ar = np.ascontiguousarray(area if area is not None else [0, 0, e.shape[0], e.shape[1]], np.int32)
        check(self.lib.pt_scene_set_environment(self.handle, _fptr(e), e.shape[0], e.shape[1], _fptr(ar, np.int32)))

    def build(self):
        check(self.lib.pt_scene_build(self.handle))

    def replicate(self, ctx: Context) -> "Scene":
        """pt_scene_replicate: a copy of this built scene on `ctx` (device-to-device copies, the same tree, no rebuild);
        independent of this scene afterwards."""
        h = C.c_void_p()
        check(self.lib.pt_scene_replicate(self.handle, ctx.handle, C.byref(h)))
        out = Scene.__new__(Scene)
        out.ctx, out.lib, out.handle = ctx, self.lib, h
        return out

    def bvh_info(self):
        a, b, c = C.c_int64(), C.c_int64(), C.c_int64()
        check(self.lib.pt_scene_bvh_info(self.handle, C.byref(a), C.byref(b), C.byref(c)))
        return a.value, b.value, c.value

    def bvh_download(self):
        n_nodes, _, n_glob = self.bvh_info()
        nodes = np.zeros((max(n_nodes, 1), 16), np.float32)
        glob = np.zeros(max(n_glob, 1), np.int32)
        check(self.lib.pt_scene_bvh_download(self.handle, _fptr(nodes), n_nodes, _fptr(glob, np.int32), n_glob))
        return nodes[:n_nodes], glob[:n_glob]

    def triangles_download(self, n: int):
        tris = np.zeros((n, 12), np.float32)
        check(self.lib.pt_scene_triangles_download(self.handle, _fptr(tris), n))
        return tris


class Multi:
    """pt_multi_*: contexts that render one frame together.  contexts[0] is the root: the accumulators passed to render()
    live on its device and the frame is ordered on its stream.  The contexts must outlive this object (it keeps them)."""

    def __init__(self, contexts):
        self.lib = load()
        self.contexts = list(contexts)
        arr = (C.c_void_p * max(len(self.contexts), 1))(*[c.handle for c in self.contexts])
        h = C.c_void_p()
        check(self.lib.pt_multi_create(arr, len(self.contexts), C.byref(h)))
        self.handle = h

    @property
    def n(self) -> int:
        return len(self.contexts)

    def close(self):
        if getattr(self, "handle", None):
            self.lib.pt_multi_destroy(self.handle)
            self.handle = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def render(self, scenes, cam: PtCamera, params: PtRenderParams, accum_ptr: int, accum_sq_ptr: int | None = None,
               want_stats: bool = False) -> list[PtStats] | None:
        """pt_multi_render: params.spp samples from params.spp_offset, split over the members, scenes[i] on member i; the sum
        is ADDED into the root's accumulators.  want_stats=False returns None without waiting for the GPU; otherwise one
        PtStats per member, after the whole frame."""
        if len(scenes) != self.n:
            raise PtError(f"pt_multi_render: {len(scenes)} scenes for {self.n} members")
        arr = (C.c_void_p * max(len(scenes), 1))(*[s.handle for s in scenes])
        st = (PtStats * self.n)() if want_stats else None
        check(self.lib.pt_multi_render(self.handle, arr, C.byref(cam), C.byref(params), C.c_void_p(accum_ptr),
                                       C.c_void_p(accum_sq_ptr or 0), st))
        return list(st) if want_stats else None
