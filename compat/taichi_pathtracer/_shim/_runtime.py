"""Runtime of the drop-in shim: what the reference scripts' Taichi fields and kernels become.

The reference drivers (taichi_pathtracer/{6..10}_*/__main__.py) keep module globals `resolution, spp, propagate_limit,
image, rays`, define @ti.func / @ti.kernel bodies and run

    for _ in trange(spp):
        camera.get_rays(rays)        # one camera ray per pixel into the `rays` field
        shader(world, rays)          # image[i, j] += background * l / spp
    post_processing()                # ACES + gamma in place
    ti.tools.imwrite(image, path)

Under this shim the decorated bodies are never executed (they are Taichi device code).  `get_rays` stamps the camera
into the rays field, every `shader` call books one more sample per pixel for (world, camera), and the booked samples
are rendered by ONE pt_render call (libb200pt.so, one persistent-kernel launch) when the image is first needed —
post_processing(), image.to_numpy(), ti.tools.imwrite().  The per-sample host loop of the reference (2 x spp kernel
launches) collapses into one launch; the set of paths is the same as 8192 one-sample launches would trace because the
RNG is keyed on the absolute sample index.

`_render_pass` / `_post_pass` are the two points where the shim meets the library; tests replace them to check the
host logic without a GPU."""
from __future__ import annotations

import os
import sys

import numpy as np

_ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__)))))
if _ROOT not in sys.path:
    sys.path.insert(0, _ROOT)

import learn_path_tracing_b200 as L  # noqa: E402


class DeviceFunc:
    """@ti.func: device code of the reference; kept for introspection (which BSDFs a script scatters with)."""

    def __init__(self, fn):
        self.fn = fn
        self.__name__ = getattr(fn, "__name__", "func")

    def __call__(self, *a, **k):
        raise RuntimeError(f"{self.__name__} is Taichi device code; under the B200 shim it runs inside libb200pt.so, not on the host")


def names_used(fn, seen=None):
    """Global names a function body refers to, followed through the script's other @ti.func bodies."""
    seen = set() if seen is None else seen
    out = set()
    code = getattr(fn, "__code__", None)
    if code is None or id(fn) in seen:
        return out
    seen.add(id(fn))
    stack = [code]
    while stack:
        c = stack.pop()
        out.update(c.co_names)
        stack.extend(k for k in c.co_consts if hasattr(k, "co_names"))
    for n in list(out):
        g = fn.__globals__.get(n)
        if isinstance(g, DeviceFunc):
            out |= names_used(g.fn, seen)
    return out


class RayField:
    """Ray.field(shape=resolution): carries the camera that last filled it (Camera.get_rays)."""

    def __init__(self, shape):
        self.shape = tuple(int(v) for v in shape)
        self.camera = None          # PtCamera snapshot
        self.camera_key = None


class ImageField:
    """Vec3f.field(shape=resolution): the accumulation image.  Device-resident; host copy on demand."""

    def __init__(self, shape):
        self.shape = tuple(int(v) for v in shape)
        self.renderer = None        # L.Renderer, created at the first flush (needs the GPU)
        self.booked = []            # [(world, camera struct, camera key, spp-normalisation, depth, model, count)]
        self.done = 0               # samples per pixel already in the accumulator
        self.norm = 1               # the script's `spp`: image = sum / spp
        self.post = None            # (aces, gamma) once post_processing() ran
        self.host = None

    # -- booking
    def book(self, world, rays, spp, depth, model, flags=0):
        if rays.camera is None:
            raise RuntimeError("shader(world, rays) before camera.get_rays(rays)")
        self.norm = int(spp)
        self.host = None
        last = self.booked[-1] if self.booked else None
        if last and last[0] is world and last[2] == rays.camera_key and last[4] == depth and last[5] == model and last[7] == flags:
            last[6] += 1
        else:
            self.booked.append([world, rays.camera, rays.camera_key, int(spp), int(depth), int(model), 1, int(flags)])

    def flush(self):
        for world, cam, _, _, depth, model, count, flags in self.booked:
            self.renderer = _render_pass(self, world, cam, count, depth, model, self.done, flags)
            self.done += count
        self.booked = []

    # -- reading
    def to_numpy(self):
        self.flush()
        if self.host is None:
            self.host = _read_image(self)
        return self.host

    def __array__(self, dtype=None, copy=None):
        a = self.to_numpy()
        return a.astype(dtype) if dtype is not None else a

    def __getitem__(self, idx):
        return self.to_numpy()[idx]

    def fill(self, value):
        if value != 0:
            raise NotImplementedError("image.fill(v) with v != 0")
        self.booked, self.done, self.post, self.host = [], 0, None, None
        if self.renderer is not None:
            self.renderer.clear()


def _devices():
    """LPT_DEVICES: "all" or a comma list of CUDA device indices ("0,1,2,3") to split every pass over, from this one
    process (MultiRenderer); unset renders on one device."""
    v = os.environ.get("LPT_DEVICES", "").strip()
    if not v:
        return None
    return "all" if v == "all" else [int(d) for d in v.split(",") if d.strip()]


def _denoise():
    """LPT_DENOISE=1: the image is the denoised mean (Renderer.denoised(): 4-spp guide features of the first pass's camera
    rays), as render(..., denoise=True) returns it; unset or 0 leaves the raw Monte Carlo mean."""
    return os.environ.get("LPT_DENOISE", "").strip() not in ("", "0")


def _new_renderer(w, h):
    devices = _devices()
    if devices is None:
        return L.Renderer(w, h, L.default_context(), want_sq=_denoise())
    return L.MultiRenderer(w, h, devices, L.default_context(), want_sq=_denoise())


def _render_pass(image, world, cam, count, depth, model, first_sample, flags=0):
    """`count` more samples per pixel of (world, cam) into the image's device accumulator: ONE pt_render call (one
    pt_multi_render over the devices of LPT_DEVICES when that is set)."""
    w, h = image.shape
    r = image.renderer or _new_renderer(w, h)
    seed = int(os.environ.get("LPT_SEED", "1"))
    scene = world.device_scene(r.ctx)
    r.render(scene, cam, count, depth, model, seed=seed, spp_offset=first_sample, want_stats=False, flags=flags)
    if _denoise() and first_sample == 0:
        r.features(scene, cam, 4, seed, 0, flags, model)
    return r


def _read_image(image):
    w, h = image.shape
    if image.renderer is None:
        return np.zeros((w, h, 3), np.float32)
    if image.post is not None:
        return image.renderer.image(aces=image.post[0], gamma=image.post[1], total_spp=image.norm, denoise=_denoise())
    if _denoise():
        return L.denoised_mean(image.renderer, total_spp=image.norm)
    return image.renderer.ctx.download_accum(image.renderer.accum.data_ptr(), w, h) / np.float32(image.norm)


class Kernel:
    """@ti.kernel: classified by what its body refers to.
       shading pass   body reaches world.hit / a BSDF's sample (through the script's @ti.func bodies): books one sample
                      (stages 6-10: the BSDFs named decide the model; stages 4-5 name none: normals as colours)
       post pass      body calls ACES_tonemapping / gamma_correction: marks the image as post-processed"""

    def __init__(self, fn):
        self.fn = fn
        self.__name__ = fn.__name__
        self.names = names_used(fn)
        g = fn.__globals__
        self.kind = ("shade" if {"hit", "sample"} & self.names or "propagate_once" in self.names else
                     "post" if {"ACES_tonemapping", "gamma_correction"} & self.names else None)
        self.image_name = next((n for n in self.names if isinstance(g.get(n), ImageField)), "image")

    def model(self):
        if "DiffuseBSDF" in self.names and "MetalBSDF" not in self.names:
            return L.PT_SHADE_V2_DIFFUSE
        if not {"MetalBSDF", "DielectricBSDF", "DiffuseBSDF"} & self.names:
            return L.PT_SHADE_V2_NORMALS      # stages 4-5: ray_color() shows hit.normal, nothing scatters
        return L.PT_SHADE_V2

    def __call__(self, *args):
        g = self.fn.__globals__
        image = g.get(self.image_name)
        if not isinstance(image, ImageField):
            raise RuntimeError(f"kernel {self.__name__}: no image field among the script's globals")
        if self.kind == "shade":
            world = next((a for a in args if isinstance(a, L.World)), None)
            if world is None:
                raise NotImplementedError(f"kernel {self.__name__}: no World among its arguments (stages 2-3 intersect a sphere "
                                          "typed into their own device code: use compat/taichi_pathtracer/{2,3}_* instead)")
            rays = next(a for a in args if isinstance(a, RayField))
            # stage 4 has no `spp`: ONE un-jittered ray per pixel through the lattice i/(W-1) (4_objects/camera.py), image = colour
            flags = 0 if "spp" in g else L.PT_FLAG_PIXEL_GRID
            image.book(world, rays, g.get("spp", 1), g.get("propagate_limit", 1), self.model(), flags)
        elif self.kind == "post":
            image.flush()
            image.post = ("ACES_tonemapping" in self.names, 2.2 if "gamma_correction" in self.names else 1.0)
            image.host = None
        else:
            raise NotImplementedError(f"kernel {self.__name__}: the B200 shim knows the shading pass and the post-processing "
                                      "pass of the taichi_pathtracer drivers; this body is neither")


def imwrite(image, path):
    """ti.tools.imwrite: truncating 8-bit cast, field layout [W,H,3] with y up (image_io.to_uint8)."""
    a = image.to_numpy() if isinstance(image, ImageField) else np.asarray(image)
    d = os.path.dirname(path)
    if d:
        os.makedirs(d, exist_ok=True)
    L.imwrite(a, path)
