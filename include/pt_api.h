/*
 * pt_api.h — C-ABI of libb200pt.so, the B200 (sm_100a) wavefront path tracer that replaces the
 * Taichi-JIT kernels of JeffreyXiang/learn_path_tracing on its light-transport hot path.
 *
 * The reference has no FFI of its own: its "operator interface" for this path is the set of Taichi
 * kernels the driver scripts launch.  Each entry point below names the reference kernel/function it
 * supersedes (paths relative to the reference checkout):
 *
 *   pt_scene_set_spheres        World.__init__/World.add            taichi_pathtracer/10_final/world.py:7-22
 *   pt_scene_add_mesh           World.add_mesh + MeshBVHTree.build  legacy/PT_in_one_weekend/15_module.py:792-793,716-754
 *   pt_scene_set_textured_spheres  World.add_sphere + SphereBVHTree.build   15_module.py:795-796,608-634
 *   pt_scene_set_texture_atlas  load_texture                        15_module.py:65-115
 *   pt_scene_set_environment    load_environment                    15_module.py:118-132
 *   pt_scene_build              (BVH build; reference: host Python SAH, 15_module.py:608-634,716-754)
 *   pt_generate_rays            Camera.get_rays                     10_final/camera.py:71-93, 15_module.py:438-453
 *   pt_trace_batch[_device]     World.hit                           10_final/world.py:24-34, 15_module.py:838-848
 *   pt_render[_host]            render(): get_rays + shader loop    10_final/__main__.py:78-87,99-103
 *                               render(): get_rays + propagate_once + gen_secondary_rays   15_module.py:980-1036
 *   pt_postprocess[_host]       post_processing / gamma_correction  10_final/__main__.py:90-96, 15_module.py:1016-1019
 *   pt_render_features, pt_denoise   (no reference counterpart: an opt-in denoised mean of a low-sample frame)
 *
 * Conventions
 *   - every function returns 0 on success, a negative PT_ERR_* otherwise; pt_last_error() returns
 *     thread-local text for the last failure.  No C++ exception crosses the boundary.
 *   - host arrays are caller-owned and only read/written during the call.
 *   - "device" pointers are plain CUDA device pointers on the context's device (e.g. a torch
 *     tensor's data_ptr()); the library never frees them.
 *   - a PtContext is bound to one CUDA device and one stream and is not thread-safe; use one
 *     context per GPU (one process per GPU under torchrun).
 *   - images: the device accumulator is float4[height*width], pixel index = j*width + i with j UP
 *     (row 0 = bottom row, as the reference's image[i, j] field).  Host images use the Taichi field
 *     layout float[width][height][3] (image.to_numpy()).
 */
#ifndef PT_API_H
#define PT_API_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define PT_API_VERSION 1

/* error codes */
#define PT_OK 0
#define PT_ERR_INVALID (-1)     /* bad argument                                   */
#define PT_ERR_CUDA (-2)        /* a CUDA runtime call failed (text has details)  */
#define PT_ERR_NOT_BUILT (-3)   /* scene used before pt_scene_build               */
#define PT_ERR_NO_DEVICE (-4)   /* no usable CUDA device: there is NO CPU fallback */
#define PT_ERR_NOMEM (-5)

/* shading models */
#define PT_SHADE_V2 0           /* taichi_pathtracer stages 7-10: MetalBSDF / DielectricBSDF (bsdf.py:71-110) */
#define PT_SHADE_V2_DIFFUSE 1   /* taichi_pathtracer/6_diffuse: DiffuseBSDF only (6_diffuse/bsdf.py:20-26)     */
#define PT_SHADE_LEGACY 2       /* legacy 14_mesh/15_module gen_secondary_rays (15_module.py:994-1013)         */
#define PT_SHADE_V2_NORMALS 3   /* taichi_pathtracer stages 4-5: colour = 0.5 (normal + 1), no bounce (5_anti_aliasing/__main__.py:19-28);
                                   persistent kernel only                                                      */

#define PT_SHADE_LEGACY_STAGE7 4 /* legacy/PT_in_one_weekend/7_reflect.py:187-209 (the untextured ancestor of gen_secondary_rays: the
                                   same cal_reflectivity_metal / _dielectirc, sample_in_sphere, sample_reflect, sample_diffuse as
                                   15_module.py:281-334): v2-style spheres with constant materials, `metallic` a switch, diffuse
                                   throughput albedo * params.absorptivity, reflection lobe scaled by k = -d.n, hits accepted for
                                   t > 1e-3 (near root only), rays leave from the hit point; sky gradient.  Persistent kernel only */
#define PT_SHADE_LEGACY_STAGE6 5 /* legacy/PT_in_one_weekend/6_diffuse.py:160-170: every hit is sample_diffuse with throughput
                                   params.absorptivity (0.5) * albedo; same hit rule.  Persistent kernel only                    */

/* PtRenderParams.flags */
#define PT_FLAG_ACCUM_SQ 1      /* also accumulate per-pixel sum of squares (needs accum_sq != NULL)   */
#define PT_FLAG_TIMING 2        /* record CUDA events around every kernel launch (fills PtStats.ms_*)  */
#define PT_FLAG_COUNTERS 4      /* count BVH nodes visited / primitives tested (slower)                */
#define PT_FLAG_PIXEL_GRID 64   /* stages 2-4 camera (2_camera_and_ray/camera.py:67): the ray of pixel (i, j) goes through
                                   the lattice point (i/(W-1), j/(H-1)) of the view rectangle, no jitter (W, H >= 2)    */
#define PT_FLAG_RAYS_FAST 256   /* pt_generate_rays_ex only: legacy Camera.get_rays_fast (15_module.py:423-436): the ray of pixel
                                   (i, j) goes through (i/W, j/H) of the view rectangle, pinhole, focal length 1, no jitter */
/* pt_trace_batch_device flags */
#define PT_FLAG_NO_SORT 8       /* keep the batch order (default: batches >= 65536 rays are traced in an
                                   entry-point/direction Morton order; results always land in batch order) */
#define PT_FLAG_TRACE_SIMPLE 16 /* one ray per thread (k_trace) instead of the persistent while-while warps */
#define PT_FLAG_NO_QNODES 32    /* walk the 64-byte float nodes even when the tree has the 32-byte quantised copy */
#define PT_FLAG_TRACE_WIDE 128  /* `make EXPERIMENTAL=1` builds only: walk the 4-wide copy of the tree (scene built with
                                   PT_WIDE=1 in the environment; csrc/bvh4.h).  Same hit records, 0.57x the steps, but
                                   measured 5-9 % slower on the render workloads and 40 % slower on the 10 M-triangle
                                   batch (profiles/r02_ab_wide.txt): not in the default library (PT_ERR_INVALID)      */
#define PT_FLAG_WIDE PT_FLAG_TRACE_WIDE /* the same for pt_render (PtRenderParams.flags, persistent mode only)       */
/* bits 8-13 of the trace flags: lanes that must wait before a warp services them (0 = default 8);
   bits 14-19: finished lanes that trigger result write-back + refill (0 = default 8) */

typedef struct PtContext PtContext;
typedef struct PtScene PtScene;

/* reference: Material = struct(albedo, roughness, metallic:i32, ior, transparency:i32), 10_final/dtypes.py:8 */
typedef struct PtMaterial {
    float albedo[3];
    float roughness;
    int32_t metallic;
    float ior;
    int32_t transparency;
    int32_t _pad;
} PtMaterial; /* 32 bytes */

/* Camera basis is computed on the host (both FOV conventions live in Python):
 *   v2     view_w = 2*tan(radians(fov)/2)   camera.py:81
 *   legacy view_w = 2*tan(fov*pi/180)       15_module.py:444                                   */
typedef struct PtCamera {
    float pos[3];
    float front[3];
    float right[3];
    float up[3];
    float view_w, view_h;
    float focal_length, aperture;
} PtCamera; /* 64 bytes */

typedef struct PtRenderParams {
    int32_t width, height;
    int32_t spp;            /* samples per pixel rendered by THIS call                              */
    int32_t spp_offset;     /* first sample index (progressive rendering / multi-GPU sample split)  */
    int32_t max_depth;      /* propagate_limit: max ray segments per path                           */
    int32_t shading_model;  /* PT_SHADE_*                                                           */
    uint32_t seed;
    float absorptivity;     /* legacy only: 0.25 (15_module.py:893,950) or 0.5 (14_mesh.py:833,889) */
    int32_t pool_capacity;  /* path-pool slots; 0 = library default                                 */
    int32_t flags;          /* PT_FLAG_*                                                            */
    int32_t reserved[6];    /* [0] wavefront mode: 0 auto (= 3), 1 split (k_extend +
                                   k_shade per bounce), 2 fused K-step (k_paths), 3 persistent ballot-scheduled (k_paths_persist),
                                   4, 5: `make EXPERIMENTAL=1` builds only (k_paths_queue: block-local shading queues;
                                   k_paths_dual: two lane-private path records per lane; both measured slower)
                               [1] fused mode: ray segments per path slot per launch (0 = default 32); mode 5: blocks per SM (3 or 4)
                               [2] persistent mode: finished lanes that trigger shading + refill (0 = default: 22 sphere scenes, 20 mesh scenes)
                               [3] persistent mode: waiting lanes that trigger a service (leaf tests) (0 = default: 12 sphere scenes, 8 mesh scenes)
                               [4], [5] persistent mode: render only the rows [row0, row1) of the frame (0, 0 = all);
                                   the multi-GPU path renders band by band and reduces band k while band k+1 renders */
} PtRenderParams; /* 64 bytes */

typedef struct PtStats {
    uint64_t paths;          /* camera paths started                       */
    uint64_t segments;       /* ray segments extended (camera + secondary) */
    uint64_t nodes_visited;  /* PT_FLAG_COUNTERS only                      */
    uint64_t prims_tested;   /* PT_FLAG_COUNTERS only                      */
    float ms_total;          /* whole call, CUDA events on the ctx stream  */
    float ms_extend;         /* PT_FLAG_TIMING: sum over extend launches   */
    float ms_shade;          /* PT_FLAG_TIMING: sum over shade launches    */
    float ms_other;
    int32_t iterations;      /* wavefront iterations                       */
    int32_t launches;        /* kernels launched by this call              */
    int32_t launches_extend;
    int32_t launches_shade;
    int32_t reserved[4];
} PtStats; /* 80 bytes */

/* ---- context ------------------------------------------------------------------------------- */
/* stream: a cudaStream_t (e.g. torch.cuda.current_stream().cuda_stream) or NULL for the default. */
int pt_context_create(int device, void* stream, PtContext** out);
void pt_context_destroy(PtContext* ctx);
int pt_context_set_stream(PtContext* ctx, void* stream);
int pt_context_sync(PtContext* ctx);

/* ---- scene --------------------------------------------------------------------------------- */
int pt_scene_create(PtContext* ctx, PtScene** out);
void pt_scene_destroy(PtScene* scene);

/* v2 spheres: center_radius[n][4], mats[n].  Order is significant (first wins ties, world.py:30). */
int pt_scene_set_spheres(PtScene* s, const float* center_radius, const PtMaterial* mats, int n);

/* legacy textured spheres (15_module.py:33 Sphere = center, radius, transparency, texture_id). */
int pt_scene_set_textured_spheres(PtScene* s, const float* center_radius, const int32_t* transparency,
                                  const int32_t* texture_id, int n);

/* legacy indexed mesh.  faces[nf][10] = a.p,a.n,a.t, b.p,b.n,b.t, c.p,c.n,c.t, texture_id
 * (Face/FaceVertex, 15_module.py:31-32).  May be called several times (one BVH per mesh in the
 * reference; here all meshes share one LBVH, primitive ids are assigned in call order).          */
int pt_scene_add_mesh(PtScene* s, const float* positions, int nv, const float* normals, int nn,
                      const float* texcoords, int nt, const int32_t* faces, int nf);

/* raw triangle soup for the intersection benchmark: verts[n][9] = p0,p1,p2. */
int pt_scene_set_triangles(PtScene* s, const float* verts, int64_t n);
/* same, deterministic on-device generator (SURVEY 8d config 5): centroid~U[0,1)^3, edges~U[-s,s]^3 */
int pt_scene_set_random_triangles(PtScene* s, int64_t n, uint32_t seed, float edge_scale);

/* texture atlas in the reference's 8-bit source precision: texels[W][H] (x-major like the Taichi
 * field), each 8 bytes = albedo r,g,b, roughness, normal x,y,z, metallic (all u8, pre-gamma).  The
 * device decodes with the reference's load_texture transfer functions (15_module.py:101-104).
 * areas[ntex][4] = low.x, low.y, high.x, high.y indexed by texture id (textures_info).
 * tex_flags[ntex] (may be NULL): bit 0 = plain diffuse map without a normal map: the normal decodes to
 * exactly (0,0,1) as load_texture's constant [0.5,0.5,1]*2-1 does (15_module.py:84,104).                */
int pt_scene_set_texture_atlas(PtScene* s, const uint8_t* texels, int W, int H, const int32_t* areas,
                               const int32_t* tex_flags, int ntex);

/* environment map rgb[W][H][3] float (x-major), area[4]; rgb==NULL selects the v2 sky gradient
 * (backbround_color, 10_final/__main__.py:58-62).                                               */
int pt_scene_set_environment(PtScene* s, const float* rgb, int W, int H, const int32_t* area);

/* GPU BVH build, replaces the host-Python SAH builders (15_module.py:608-634, 716-754): Morton codes -> radix sort ->
 * hierarchy -> bottom-up refit.  Trees of up to 2^20 primitives are built with BOTH hierarchies over that one sort —
 * Karras 2012 and PLOC (depth-first renumbered) — trees of up to 4096 primitives also by a host full-sweep SAH, and the
 * candidate with the lowest SAH cost (and at most 60 levels) is kept; larger trees use the Karras hierarchy.
 * Developer knobs (environment, A/B runs only): PT_BUILDER=lbvh|ploc|sah forces one,
 * PT_PLOC_RADIUS, PT_PLOC_DFS=0, PT_BUILD_VERBOSE=1 prints both SAH costs.                                          */
int pt_scene_build(PtScene* s);

/* introspection for tests / the oracle: BVH2 nodes as float[n_nodes][16]
 * = c0.min xyz, c0.max xyz, c1.min xyz, c1.max xyz, bits(child0), bits(child1), 0, 0
 * child >= 0: inner node index; child < 0: leaf, primitive id = ~child.                         */
int pt_scene_bvh_info(const PtScene* s, int64_t* n_nodes, int64_t* n_prims, int64_t* n_global_prims);
int pt_scene_bvh_download(const PtScene* s, float* nodes, int64_t n_nodes, int32_t* global_prims, int64_t n_global);
/* triangles as stored on the device, float[n][12] = v0.xyz,_, e1.xyz,_, e2.xyz,_  */
int pt_scene_triangles_download(const PtScene* s, float* tris, int64_t n);

/* ---- hot path ------------------------------------------------------------------------------ */
/* Camera.get_rays for sample index `sample` of every pixel: rays[height*width][8] = o.xyz, tmin,
 * d.xyz, tmax on the HOST (testing aid; the render generates rays on the fly).                  */
int pt_generate_rays(PtContext* ctx, const PtCamera* cam, int width, int height, int sample, uint32_t seed,
                     float* rays_host);
/* same with flags: PT_FLAG_PIXEL_GRID (stages 2-4 lattice) or PT_FLAG_RAYS_FAST (legacy Camera.get_rays_fast) */
int pt_generate_rays_ex(PtContext* ctx, const PtCamera* cam, int width, int height, int sample, uint32_t seed,
                        int flags, float* rays_host);

/* closest hit for a fixed ray batch.  rays[n][8] = o.xyz, tmin, d.xyz, tmax.
 * prim_id[n] = -1 on miss; t[n] = -1 on miss; uv may be NULL.                                   */
int pt_trace_batch(PtContext* ctx, const PtScene* s, const float* rays_host, int64_t n, int32_t* prim_id_host,
                   float* t_host, PtStats* stats);
/* rays_dev: float4[2n] (o|tmin, d|tmax interleaved per ray); hits_dev: float4[n] = t, bits(prim), u, v */
int pt_trace_batch_device(PtContext* ctx, const PtScene* s, const void* rays_dev, int64_t n, void* hits_dev,
                          int flags, PtStats* stats);
/* deterministic on-device ray generator for the intersection benchmark (SURVEY 8d config 5). */
int pt_random_rays_device(PtContext* ctx, void* rays_dev, int64_t n, uint32_t seed);

/* Render params->spp samples of every pixel and ADD the radiance into accum_dev (float4[h*w]:
 * sum r, g, b, and number of contributing paths); accum_sq_dev (float4[h*w], sum of squares) is
 * optional.  The caller zeroes the buffers (progressive rendering keeps adding, 15_module.py:1022-1036).
 * stats == NULL: fully ASYNCHRONOUS on the context stream (persistent / queue modes: one kernel launch and one small
 * counter copy are enqueued and the call returns; whatever the caller enqueues next on that stream — an NCCL reduce,
 * pt_postprocess — follows without a host round trip).  stats != NULL: the call ends with pt_render_stats().   */
int pt_render(PtContext* ctx, const PtScene* s, const PtCamera* cam, const PtRenderParams* p, void* accum_dev,
              void* accum_sq_dev, PtStats* stats);
/* Statistics of the LAST pt_render on this context; waits for that render (not for later work on the stream). */
int pt_render_stats(PtContext* ctx, PtStats* stats);

/* Same through host buffers: accum_host[width][height][3] (Taichi field layout, sum of radiance,
 * overwritten), accum_sq_host optional.  Includes device allocation, render, device->host copy. */
int pt_render_host(PtContext* ctx, const PtScene* s, const PtCamera* cam, const PtRenderParams* p,
                   float* accum_host, float* accum_sq_host, PtStats* stats);

/* out = gamma(ACES(accum * scale)) (aces != 0) or (accum*scale)^(1/gamma); out_dev float4[h*w]. */
int pt_postprocess(PtContext* ctx, const void* accum_dev, int width, int height, float scale, int aces,
                   float gamma, void* out_dev);
/* device accumulator -> host float[width][height][3] (Taichi field layout), post-processed. */
int pt_postprocess_host(PtContext* ctx, const void* accum_dev, int width, int height, float scale, int aces,
                        float gamma, float* out_host);
/* raw device accumulator (float4[h*w]) -> host float[width][height][3]. */
int pt_download_accum(PtContext* ctx, const void* accum_dev, int width, int height, float* out_host);

/* ---- one frame on several contexts (csrc/multi.cu) ----------------------------------------- */
typedef struct PtMulti PtMulti;

/* A group of n (1..16) contexts that render one frame together.  members[0] is the ROOT: the accumulator passed to
 * pt_multi_render lives on its device and the call is ordered on its stream.  Contexts must be distinct objects; two
 * contexts may sit on the same device.  Enables peer access between every pair of distinct devices (an already-enabled
 * pair is not an error); fails with PT_ERR_INVALID naming the pair when cudaDeviceCanAccessPeer says no.  The contexts
 * stay owned by the caller and must outlive the group. */
int pt_multi_create(PtContext* const* members, int n, PtMulti** out);
void pt_multi_destroy(PtMulti* m);

/* p->spp samples starting at p->spp_offset, split over the members exactly like multigpu.split_samples (contiguous
 * ranges, remainder to the low members), scenes[i] rendered on members[i].  The sum over all members is ADDED into
 * accum_root (float4[h*w] on the root's device, all 4 channels) and, with PT_FLAG_ACCUM_SQ, into accum_sq_root.
 * The other members read and write the root's accumulators through peer access: they must be memory that peer access
 * maps (cudaMalloc, e.g. torch's default allocator).  Every member reduces one contiguous slice of the pixels (partials
 * of members 1, 2, ... in that order), so the result is deterministic given the per-member renders.
 * stats == NULL: asynchronous like pt_render — returns after enqueueing; the root stream is ordered behind every member's
 * work.  stats != NULL: stats[n], one PtStats per member; the call waits for the whole frame.
 * Row bands (reserved[4], reserved[5]) are refused.  Every argument is checked before anything is enqueued. */
int pt_multi_render(PtMulti* m, PtScene* const* scenes, const PtCamera* cam, const PtRenderParams* p,
                    void* accum_root, void* accum_sq_root, PtStats* stats);

/* A copy of a built scene on another context (another device or the same one): device arrays copied device to device,
 * host staging copied, SceneView pointers rebased.  The result is the same tree, not a rebuild, and is independent of
 * src afterwards: destroying src does not affect it, and set_* + pt_scene_build work on it as on any scene. */
int pt_scene_replicate(const PtScene* src, PtContext* dst, PtScene** out);

/* ---- denoising (csrc/denoise.cu) ---------------------------------------------------------- */
/* First-hit guide features of the camera rays of samples [p->spp_offset, p->spp_offset + p->spp) of every pixel: the
 * same rays pt_render starts its paths with (rng4(pixel, sample, 0, seed), PT_FLAG_PIXEL_GRID honoured), hit with
 * the same acceptance rule (tmin of the shading model).  ADDED into features_dev = float4[2][h*w] (pixel j*w + i,
 * j up, like the accumulator); the caller zeroes it, so passes and progressive poses compose like accum_dev:
 *   plane 0: sum over hits of (shading normal turned to face the ray).xyz, hit distance t
 *   plane 1: sum over ALL samples of albedo.rgb, and the number of hits in .w
 * A miss adds 0 to plane 0 and the miss radiance clamped to [0,1] (sky gradient / environment) as its albedo.
 * Accepts and refuses what pt_render does for the same scene and parameters, except: row bands (reserved[4..5]) are
 * refused, the mode / threshold fields reserved[0..3] are ignored, PT_FLAG_ACCUM_SQ needs no buffer.
 * Asynchronous on the context stream. */
int pt_render_features(PtContext* ctx, const PtScene* s, const PtCamera* cam, const PtRenderParams* p,
                       void* features_dev);

typedef struct PtDenoiseParams {
    int32_t width, height;
    int32_t spp;          /* samples per pixel in accum (the mean is accum / spp, as pt_postprocess's scale)  */
    int32_t iterations;   /* a-trous passes, 0..10 (0 = no filtering: out = accum / spp)                      */
    float sigma_l, sigma_n, sigma_z;   /* edge-stopping strengths; 0 = defaults 4, 128, 1                  */
    int32_t _pad;
} PtDenoiseParams; /* 32 bytes */

/* Denoised mean radiance into out_dev = float4[h*w] (rgb, w = 1), ready for pt_postprocess with scale 1.
 * Needs the sum of squares (PT_FLAG_ACCUM_SQ) and a feature buffer of the same size. Deterministic: no atomics.
 * Every argument is checked before anything is enqueued.  Asynchronous on the context stream. */
int pt_denoise(PtContext* ctx, const void* accum_dev, const void* accum_sq_dev, const void* features_dev,
               const PtDenoiseParams* p, void* out_dev);

/* FP32 FMA peak microbenchmark (all SMs, dependent-free FMA chains): returns TFLOP/s. */
int pt_measure_fp32_peak(PtContext* ctx, float* tflops);

const char* pt_last_error(void);
int pt_version(void);
/* "sm_100a experimental=0|1": whether the library was built with `make EXPERIMENTAL=1` (render modes 4/5, PT_FLAG_WIDE). */
const char* pt_build_info(void);

#ifdef __cplusplus
}
#endif
#endif /* PT_API_H */
