"""learn_path_tracing_b200 — B200-native wavefront path tracer behind the scene-description surface of
JeffreyXiang/learn_path_tracing (taichi_pathtracer stages 6-10 and legacy 14_mesh/15_module).

Python describes the scene; all light transport runs in libb200pt.so (hand-written sm_100a CUDA,
C-ABI in include/pt_api.h).  There is no CPU fallback.
"""
from . import _lib
from ._lib import (PT_MODE_AUTO, PT_MODE_FUSED, PT_MODE_SPLIT, PT_MODE_PERSIST, PT_MODE_QUEUE, PT_MODE_DUAL, PT_FLAG_NO_SORT, PT_FLAG_TRACE_SIMPLE, PT_FLAG_NO_QNODES, PT_FLAG_ACCUM_SQ, PT_FLAG_COUNTERS, PT_FLAG_PIXEL_GRID, PT_FLAG_TRACE_WIDE, PT_FLAG_WIDE, PT_FLAG_TIMING, PT_SHADE_LEGACY, PT_SHADE_V2, PT_SHADE_LEGACY_STAGE6, PT_SHADE_LEGACY_STAGE7, PT_FLAG_RAYS_FAST,
                   PT_SHADE_V2_DIFFUSE, PT_SHADE_V2_NORMALS, Context, PtError, Scene)
from .bsdf import DielectricBSDF, DiffuseBSDF, LegacyStage6BSDF, LegacyStage7BSDF, MetalBSDF, NormalColor
from .camera import Camera
from .dtypes import HitRecord, Mat3f, Material, Ray, Sphere, Vec2f, Vec2i, Vec3f
from .image_io import imread, imwrite, imwrite_legacy, to_uint8
from .postprocessing import ACES_tonemapping, gamma_correction
from .multigpu import reduce_accumulators, render_distributed, split_samples
from .render import MultiRenderer, Renderer, default_context, denoised_mean, render
from .world import World

__all__ = [
    "Context", "Scene", "PtError", "Camera", "World", "Sphere", "Material", "Ray", "HitRecord", "Vec2f", "Vec2i",
    "Vec3f", "Mat3f", "MetalBSDF", "DielectricBSDF", "DiffuseBSDF", "NormalColor", "LegacyStage6BSDF", "LegacyStage7BSDF",
    "PT_SHADE_LEGACY_STAGE6", "PT_SHADE_LEGACY_STAGE7", "PT_FLAG_RAYS_FAST", "ACES_tonemapping", "gamma_correction",
    "Renderer", "MultiRenderer", "render", "denoised_mean", "default_context", "render_distributed", "split_samples", "reduce_accumulators", "imwrite", "imwrite_legacy", "imread", "to_uint8", "PT_SHADE_V2", "PT_SHADE_V2_DIFFUSE", "PT_SHADE_V2_NORMALS",
    "PT_SHADE_LEGACY", "PT_FLAG_ACCUM_SQ", "PT_FLAG_TIMING", "PT_FLAG_COUNTERS", "PT_FLAG_PIXEL_GRID", "PT_FLAG_TRACE_WIDE", "PT_FLAG_WIDE", "PT_MODE_AUTO", "PT_MODE_SPLIT", "PT_MODE_FUSED", "PT_MODE_PERSIST", "PT_MODE_QUEUE", "PT_MODE_DUAL", "PT_FLAG_NO_SORT", "PT_FLAG_TRACE_SIMPLE", "PT_FLAG_NO_QNODES",
]
