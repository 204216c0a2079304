"""render(): the reference's render loop (10_final/__main__.py:99-103) as ONE call into the device.

The reference launches get_rays + shader once per sample from Python (2*spp launches); here the host
hands (scene, camera, params) to pt_render and the wavefront runs on the GPU until every path of
every sample has terminated.  torch is used for device buffers and streams only.
"""
from __future__ import annotations

import os

import numpy as np

from . import _lib

_default_ctx = None


def default_context() -> _lib.Context:
    """Process-wide context on cuda:LOCAL_RANK, bound to torch's current stream."""
    global _default_ctx
    if _default_ctx is None:
        import torch
        if not torch.cuda.is_available():
            raise _lib.PtError("no CUDA device visible: learn_path_tracing_b200 has no CPU fallback")
        dev = int(os.environ.get("LOCAL_RANK", "0"))
        torch.cuda.set_device(dev)
        _default_ctx = _lib.Context(dev, torch.cuda.current_stream().cuda_stream)
    return _default_ctx


class Renderer:
    """Owns the device accumulators for one image and drives pt_render / pt_postprocess."""

    def __init__(self, width: int, height: int, ctx: _lib.Context | None = None, want_sq: bool = False):
        import torch
        self.torch = torch
        self.ctx = ctx or default_context()
        self.width, self.height = int(width), int(height)
        dev = torch.device("cuda", self.ctx.device)
        self.accum = torch.zeros((self.height * self.width, 4), dtype=torch.float32, device=dev)
        self.accum_sq = torch.zeros_like(self.accum) if want_sq else None
        self.spp_done = 0
        self.last_stats = None
        self.feature_planes = None  # first-hit guide features (features()), allocated on first use
        self.feature_spp = 0        # samples per pixel in feature_planes
        self._denoised = None

    def clear(self):
        self.accum.zero_()
        if self.accum_sq is not None:
            self.accum_sq.zero_()
        if self.feature_planes is not None:
            self.feature_planes.zero_()
        self.feature_spp = 0
        self.spp_done = 0

    def render(self, scene: _lib.Scene, cam: _lib.PtCamera, spp: int, max_depth: int,
               shading_model: int = _lib.PT_SHADE_V2, seed: int = 1, spp_offset: int | None = None,
               absorptivity: float = 0.25, flags: int = 0, pool_capacity: int = 0, mode: int = 0,
               segments_per_launch: int = 0, shade_min: int = 0, serve_min: int = 0,
               want_stats: bool = True, rows: tuple[int, int] | None = None,
               count_samples: bool = True) -> _lib.PtStats | None:
        """Adds `spp` more samples per pixel into the accumulators (progressive, legacy render(moved=False)).
        want_stats=False returns None without waiting for the GPU (Renderer.stats() fetches them later).
        rows=(y0, y1) renders only that band of image rows (persistent kernel); count_samples=False leaves spp_done alone
        (all bands but the last of one banded pass)."""
        p = self._params(spp, max_depth, shading_model, seed, spp_offset, absorptivity, flags, pool_capacity, mode,
                         segments_per_launch, shade_min, serve_min)
        if rows is not None:
            p.reserved[4], p.reserved[5] = int(rows[0]), int(rows[1])
        self.ctx.set_stream(self.torch.cuda.current_stream().cuda_stream)
        st = self.ctx.render(scene, cam, p, self.accum.data_ptr(),
                             self.accum_sq.data_ptr() if self.accum_sq is not None else None, want_stats=want_stats)
        if count_samples:
            self.spp_done += int(spp)
        self.last_stats = st
        return st

    def _params(self, spp, max_depth, shading_model, seed, spp_offset, absorptivity, flags, pool_capacity, mode,
                segments_per_launch, shade_min, serve_min) -> _lib.PtRenderParams:
        p = _lib.PtRenderParams()
        p.width, p.height = self.width, self.height
        p.spp = int(spp)
        p.spp_offset = int(self.spp_done if spp_offset is None else spp_offset)
        p.max_depth = int(max_depth)
        p.shading_model = int(shading_model)
        p.seed = int(seed) & 0xFFFFFFFF
        p.absorptivity = float(absorptivity)
        p.pool_capacity = int(pool_capacity)
        p.flags = int(flags) | (_lib.PT_FLAG_ACCUM_SQ if self.accum_sq is not None else 0)
        p.reserved[0] = int(mode)                 # 0 auto, 1 split extend/shade kernels, 2 fused k_paths, 3 persistent
        p.reserved[2] = int(shade_min)            # persistent: finished lanes that trigger shading/refill (0 = default)
        p.reserved[3] = int(serve_min)            # persistent: waiting lanes that trigger a service (0 = default)
        p.reserved[1] = int(segments_per_launch)  # fused: ray segments per path slot per launch (0 = 32)
        return p

    def features(self, scene: _lib.Scene, cam: _lib.PtCamera, spp: int = 4, seed: int = 1, spp_offset: int = 0,
                 flags: int = 0, shading_model: int = _lib.PT_SHADE_V2):
        """ADDS the first-hit guide features (normal, depth, albedo; pt_render_features) of samples
        [spp_offset, spp_offset + spp) of the camera rays of render(..., seed, flags) into self.feature_planes, shaped
        (2, H*W, 4), and returns it.  clear() zeroes it.  Computed on this renderer's own context (a MultiRenderer's
        root): they cost a few camera rays, not paths."""
        if self.feature_planes is None:
            self.feature_planes = self.torch.zeros((2, self.height * self.width, 4), dtype=self.torch.float32,
                                                   device=self.accum.device)
        p = self._params(spp, 1, shading_model, seed, spp_offset, 0.25, 0, 0, 0, 0, 0, 0)
        p.flags = int(flags)
        self.ctx.set_stream(self.torch.cuda.current_stream(self.accum.device).cuda_stream)
        self.ctx.render_features(scene, cam, p, self.feature_planes.data_ptr())
        self.feature_spp += int(spp)
        return self.feature_planes

    def denoised(self, iterations: int = 5, sigma_l: float = 0.0, sigma_n: float = 0.0, sigma_z: float = 0.0,
                 total_spp: int | None = None):
        """The denoised mean radiance (pt_denoise) as a float4 device tensor (H*W, 4), w = 1: the accumulators divided by
        total_spp (default: the samples rendered), filtered under the guidance of self.feature_planes.  Needs
        want_sq=True and features(); sigma 0 = the library's defaults."""
        if self.feature_planes is None:
            raise _lib.PtError("denoised(): no guide features yet; call features(scene, cam, ...) first")
        if self.accum_sq is None:
            raise _lib.PtError("denoised(): the filter needs the sum of squares: create the renderer with want_sq=True")
        if self._denoised is None:
            self._denoised = self.torch.empty_like(self.accum)
        n = total_spp if total_spp is not None else max(self.spp_done, 1)
        # pt_denoise divides the albedo plane by the accumulator's spp: features of another sample count (4 spp under an
        # 8192-spp render) are rescaled to it.  Depth (t sum / hit count) and the normal direction are ratios: unchanged.
        f = self.feature_planes
        if self.feature_spp not in (0, n):
            f = f * (n / self.feature_spp)
        self.ctx.set_stream(self.torch.cuda.current_stream(self.accum.device).cuda_stream)
        self.ctx.denoise(self.accum.data_ptr(), self.accum_sq.data_ptr(), f.data_ptr(), self.width, self.height, n,
                         self._denoised.data_ptr(), iterations, sigma_l, sigma_n, sigma_z)
        return self._denoised

    def side_stream(self):
        """A second CUDA stream of this renderer (reduce of one row band beside the rendering of the next)."""
        if getattr(self, "_side", None) is None:
            self._side = self.torch.cuda.Stream(device=self.accum.device)
        return self._side

    def stats(self) -> _lib.PtStats:
        """Statistics of the last render() (fetched now if that call did not wait for them)."""
        if self.last_stats is None:
            self.last_stats = self.ctx.render_stats()
        return self.last_stats

    def mean(self) -> np.ndarray:
        """Linear radiance estimate, Taichi field layout [W,H,3]."""
        return self.ctx.download_accum(self.accum.data_ptr(), self.width, self.height) / max(self.spp_done, 1)

    def moments(self):
        """(sum, sum of squares) as [W,H,3] float32 arrays, for Monte Carlo standard errors."""
        s = self.ctx.download_accum(self.accum.data_ptr(), self.width, self.height)
        q = self.ctx.download_accum(self.accum_sq.data_ptr(), self.width, self.height)
        return s, q

    def image(self, aces: bool = True, gamma: float = 2.2, total_spp: int | None = None, denoise: bool = False) -> np.ndarray:
        """post_processing (ACES + gamma, __main__.py:90-96) or legacy gamma_correction (aces=False).  denoise=True
        tonemaps the denoised mean (denoised(), default filter settings) instead of the raw one."""
        n = total_spp if total_spp is not None else max(self.spp_done, 1)
        if denoise:
            d = self.denoised(total_spp=n)
            return self.ctx.postprocess_host(d.data_ptr(), self.width, self.height, 1.0, aces, gamma)
        return self.ctx.postprocess_host(self.accum.data_ptr(), self.width, self.height, 1.0 / n, aces, gamma)


def denoised_mean(r: Renderer, total_spp: int | None = None) -> np.ndarray:
    """The denoised linear radiance of a renderer, Taichi field layout [W,H,3] (as Renderer.mean())."""
    d = r.denoised(total_spp=total_spp)
    return r.ctx.download_accum(d.data_ptr(), r.width, r.height)


def resolve_devices(devices, root_device: int) -> list[int]:
    """A device list for MultiRenderer: "all" = the root's device followed by every other visible device; otherwise the
    given CUDA device indices (repeats allowed: two members on one device render one after the other)."""
    if isinstance(devices, str):
        if devices.strip() != "all":
            raise ValueError(f"devices: 'all' or a list of CUDA device indices, not {devices!r}")
        import torch
        return [int(root_device)] + [d for d in range(torch.cuda.device_count()) if d != int(root_device)]
    out = [int(d) for d in devices]
    if not out:
        raise ValueError("devices: empty device list")
    return out


def _combined_stats(stats):
    """One PtStats for a frame rendered by several members: counts summed, time = the slowest member's."""
    t = _lib.PtStats()
    for s in stats:
        for f in ("paths", "segments", "nodes_visited", "prims_tested", "launches", "launches_extend", "launches_shade"):
            setattr(t, f, getattr(t, f) + getattr(s, f))
        for f in ("ms_total", "ms_extend", "ms_shade", "ms_other"):
            setattr(t, f, max(getattr(t, f), getattr(s, f)))
        t.iterations = max(t.iterations, s.iterations)
    t.reserved[0] = stats[0].reserved[0]
    return t


class MultiRenderer(Renderer):
    """A Renderer whose frames are split over several contexts of this process (pt_multi_render): the samples of every
    pixel are divided like multigpu.split_samples, every member renders its share on its own device and stream, and the
    partial accumulators are summed into this renderer's accumulators on the root (member 0) by a reduce over peer
    memory.  Member 0 is `ctx` (default: default_context()) and must sit on devices[0]; every other member is a new
    Context on its device, bound to a torch stream of that device.  render() takes the ROOT's scene and renders replicas
    of it on the other members (pt_scene_replicate, cached until another scene is passed)."""

    def __init__(self, width: int, height: int, devices, ctx: _lib.Context | None = None, want_sq: bool = False):
        import torch
        root = ctx or default_context()
        devs = resolve_devices(devices, root.device)
        if devs[0] != root.device:
            raise ValueError(f"devices[0] = {devs[0]} is not the root context's device {root.device}")
        super().__init__(width, height, root, want_sq)
        self.devices = devs
        self.streams = [torch.cuda.Stream(device=d) for d in devs[1:]]  # kept alive with the member contexts
        self.members = [root] + [_lib.Context(d, s.cuda_stream) for d, s in zip(devs[1:], self.streams)]
        self.multi = _lib.Multi(self.members)
        self.member_stats = None
        self._source = None
        self._replicas = None

    def _scenes(self, scene: _lib.Scene):
        if scene is not self._source:
            self._replicas = None  # drop the replicas of the previous scene first
            self._replicas = [scene] + [scene.replicate(c) for c in self.members[1:]]
            self._source = scene
        return self._replicas

    def render(self, scene: _lib.Scene, cam: _lib.PtCamera, spp: int, max_depth: int,
               shading_model: int = _lib.PT_SHADE_V2, seed: int = 1, spp_offset: int | None = None,
               absorptivity: float = 0.25, flags: int = 0, pool_capacity: int = 0, mode: int = 0,
               segments_per_launch: int = 0, shade_min: int = 0, serve_min: int = 0,
               want_stats: bool = True, rows: tuple[int, int] | None = None,
               count_samples: bool = True) -> _lib.PtStats | None:
        """Renderer.render over all members: `spp` more samples per pixel into the root's accumulators.  want_stats=True
        waits for the frame and returns the members' statistics combined (per member: `member_stats`)."""
        if rows is not None:
            raise ValueError("MultiRenderer renders whole frames: row bands (rows=) are not supported")
        p = self._params(spp, max_depth, shading_model, seed, spp_offset, absorptivity, flags, pool_capacity, mode,
                         segments_per_launch, shade_min, serve_min)
        self.ctx.set_stream(self.torch.cuda.current_stream(self.accum.device).cuda_stream)
        st = self.multi.render(self._scenes(scene), cam, p, self.accum.data_ptr(),
                               self.accum_sq.data_ptr() if self.accum_sq is not None else None, want_stats=want_stats)
        if count_samples:
            self.spp_done += int(spp)
        self.member_stats = st
        self.last_stats = _combined_stats(st) if st else None
        return self.last_stats


def render(world, camera, spp: int = 8192, propagate_limit: int = 32, seed: int = 1, bsdf=None,
           ctx: _lib.Context | None = None, return_stats: bool = False, postprocess: bool = True,
           pixel_grid: bool = False, absorptivity: float = 0.25, aces: bool = True, devices=None, denoise: bool = False):
    """Drop-in for the v2 scripts' render(world, camera) + post_processing(): returns the tonemapped
    image as a float32 [W,H,3] array in Taichi field layout (pass it to imwrite).
    devices: None renders on `ctx` alone; a list of CUDA device indices (or "all") splits the frame over them in this
    process (MultiRenderer; the first device must be the context's).
    denoise=True returns the denoised image instead (Renderer.denoised(): 4-spp guide features of the render's camera
    rays, five filter passes)."""
    ctx = ctx or default_context()
    w, h = camera.resolution
    model = getattr(bsdf, "shading_model", _lib.PT_SHADE_V2)
    r = Renderer(w, h, ctx, want_sq=denoise) if devices is None else MultiRenderer(w, h, devices, ctx, want_sq=denoise)
    flags = _lib.PT_FLAG_PIXEL_GRID if pixel_grid else 0  # stages 2-4: lattice rays, no jitter
    scene, cam = world.device_scene(ctx), camera.to_struct()
    st = r.render(scene, cam, spp, propagate_limit, model, seed, absorptivity=absorptivity, flags=flags)
    if denoise:
        r.features(scene, cam, 4, seed, 0, flags, model)
        img = r.image(aces=aces, gamma=2.2, denoise=True) if postprocess else denoised_mean(r)
    else:
        img = r.image(aces=aces, gamma=2.2) if postprocess else r.mean()  # stages <= 5 write the linear image
    return (img, st) if return_stats else img
