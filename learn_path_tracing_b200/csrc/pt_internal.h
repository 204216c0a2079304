// pt_internal.h — host-side objects behind the opaque handles of include/pt_api.h and the POD
// "scene view" handed by value to every kernel.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>

#include <string>
#include <vector>

#include "../../include/pt_api.h"

// ---------------------------------------------------------------------------------------------
// HBM layouts (all 16-byte vectorised SoA)
//
//  primitive ids      [0, n_sph) spheres, [n_sph, n_sph + n_tri) triangles
//  sph_cr[n_sph]      float4  cx, cy, cz, r
//  sph_aux[n_sph]     float4  r*r, bits(transparency), bits(texture_id), 0
//  sph_mat[2*n_sph]   float4  albedo.rgb, roughness | bits(metallic), ior, bits(transparency), 0   (v2)
//  tri_geo[3*n_tri]   float4  v0.xyz,_ | e1.xyz,_ | e2.xyz,_            (Moller-Trumbore operands, 48 B)
//  tri_shade[4*n_tri] float4  n0.xyz,u0 | n1.xyz,v0 | n2.xyz,u1 | v1,u2,v2,bits(texture_id)   (64 B)
//  nodes[4*n_nodes]   float4  BVH2 node, 64 B: c0.min.xyz,c0.max.x | c0.max.yz,c1.min.xy |
//                             c1.min.z,c1.max.xyz | bits(child0),bits(child1),0,0
//                             child >= 0 inner node index, child < 0 leaf with primitive ~child
//  global_prims[]     int     primitives too large for the LBVH (ground plane triangles), tested first;
//                             global SPHERES are passed inline in the kernel parameters instead (SceneView::inl_*)
//  atlas[W*H]         uint2   x-major; .x = albedo r,g,b + roughness, .y = normal x,y,z + metallic (u8 each)
//  env[W*H]           float4  x-major rgb
// ---------------------------------------------------------------------------------------------
#define PT_MAX_INLINE 8
#define PT_MAX_INLINE_TRI 4
struct SceneView {
    const float4* sph_cr;
    const float4* sph_aux;
    const float4* sph_mat;
    const float4* tri_geo;
    const float4* tri_shade;
    const float4* nodes;
    // 32-byte nodes for big trees (trace kernel): the same two child boxes as 12 x u16 in the frame of the root box
    // (mins rounded down, maxes up) + the two child refs; NULL when the tree is small
    const uint4* qnodes;
    float qlo[3], qscale[3];  // coordinate = qlo + q * qscale
    const int* global_prims;
    const uint2* atlas;
    const int4* tex_areas;
    const int* tex_flags;  // bit 0: no normal map
    const float4* env;
    const float* lut;  // [3][256]: albedo^2.2, x^2, 2x-1
    int n_sph, n_tri, n_nodes, n_global;
    int root;          // child reference of the BVH root (node 0, or a leaf ref), 0x7fffffff = no BVH
    float root_lo[3], root_hi[3];  // box of the whole tree (union of node 0's child boxes)
    int tex_W, tex_H, ntex;
    int env_W, env_H;
    int4 env_area;
    int has_env;
    int legacy_spheres;  // spheres are legacy textured spheres (15_module.py:864-896)
    // "global" spheres (ground sphere; every sphere of a <= 8 primitive scene) live in the kernel parameter
    // bank: the brute-force loop reads them as constant operands, no loads at all
    int n_inl;
    int inl_id[PT_MAX_INLINE];
    int inl_transparent[PT_MAX_INLINE];
    float inl_r2[PT_MAX_INLINE];
    float4 inl_cr[PT_MAX_INLINE];
    // "global" TRIANGLES (ground plane halves) likewise: v0 | e1 | e2 as stored in tri_geo
    int n_inl_tri;
    int inl_tri_id[PT_MAX_INLINE_TRI];
    float4 inl_tri[PT_MAX_INLINE_TRI][3];
    // EXPERIMENTAL 4-wide copy of the tree (bvh4.h: 8 float4 per node, root = 0), NULL unless the scene was built with
    // PT_WIDE=1 in the environment; only k_trace_persist<.., WIDE> reads it (PT_FLAG_TRACE_WIDE)
    const float4* wnodes;
};

#define PT_NO_BVH 0x7fffffff

struct PtContext {
    int device = 0;
    cudaStream_t stream = nullptr;
    int sm_count = 148;
    // path pool (lazily sized)
    size_t pool_cap = 0;
    float4* pool[2][3] = {{nullptr, nullptr, nullptr}, {nullptr, nullptr, nullptr}};  // [ping-pong][o, d, thr]
    float4* hits = nullptr;
    unsigned long long* counters = nullptr;  // device: see wavefront.cu
    unsigned long long* counters_host = nullptr;  // pinned mirror ring
    // counter block of the last pt_render (pinned) + what pt_render_stats needs to turn it into a PtStats
    unsigned long long* stats_host = nullptr;
    unsigned long long last_paths = 0;
    int last_mode = 0, last_iterations = 0, last_launches = 0;
    size_t last_ev_idx = 0;
    bool last_timing = false, last_valid = false;
    cudaEvent_t ev_a = nullptr, ev_b = nullptr;
    cudaEvent_t ev_chunk[4] = {nullptr, nullptr, nullptr, nullptr};
    std::vector<cudaEvent_t> ev_pool;
    // grow-only device scratch for host-layout read-backs (no cudaMalloc/cudaFree on the render path)
    void* scratch = nullptr;
    size_t scratch_bytes = 0;
    // grow-only device scratch of the denoiser, 48 B per pixel (denoise.cu): camera rays + hits of one sample in
    // pt_render_features, colour ping-pong + guides in pt_denoise.  Apart from `scratch`, which pt_download_accum reallocates
    void* px_scratch = nullptr;
    size_t px_scratch_bytes = 0;
    // grow-only device scratch of the ray sort (keys, order, cub temporaries)
    void* sort_scratch = nullptr;
    size_t sort_bytes = 0;
    // pt_trace_batch (host buffers): double-buffered pinned + device staging, `stage_chunk` rays each
    int64_t stage_chunk = 0;
    void *stage_rays_h[2] = {nullptr, nullptr}, *stage_hits_h[2] = {nullptr, nullptr};
    void *stage_rays_d[2] = {nullptr, nullptr}, *stage_hits_d[2] = {nullptr, nullptr};
    cudaEvent_t stage_ev[2] = {nullptr, nullptr};
    // copy streams of that pipeline: H2D of chunk k+1 and D2H of chunk k-1 run beside the tracing of chunk k
    cudaStream_t stage_in = nullptr, stage_out = nullptr;
    cudaEvent_t stage_ev_in[2] = {nullptr, nullptr}, stage_ev_cmp[2] = {nullptr, nullptr};
    // large host -> device uploads (texture atlas): two pinned chunks filled by a few host threads while the copy
    // engine drains the other one
    void* up_h[2] = {nullptr, nullptr};
    cudaEvent_t up_ev[2] = {nullptr, nullptr};
};

struct HostMesh {
    std::vector<float> pos, nrm, uv;
    std::vector<int32_t> faces;
};

struct PtScene {
    PtContext* ctx = nullptr;
    // host staging (kept until build)
    std::vector<float> h_sph_cr;
    std::vector<PtMaterial> h_sph_mat;
    std::vector<int32_t> h_sph_transparency, h_sph_tex;
    bool legacy_spheres = false;
    std::vector<float> h_tri9;           // raw triangle soup (p0,p1,p2) of every mesh, in prim order
    std::vector<float> h_tri_shade;      // 16 floats per triangle
    int64_t n_tri = 0;
    bool device_generated_tris = false;  // pt_scene_set_random_triangles
    // device
    float4 *d_sph_cr = nullptr, *d_sph_aux = nullptr, *d_sph_mat = nullptr;
    float4 *d_tri_geo = nullptr, *d_tri_shade = nullptr, *d_nodes = nullptr;
    uint4* d_qnodes = nullptr;
    float4* d_wnodes = nullptr;
    int64_t n_wnodes = 0;
    int* d_global = nullptr;
    uint2* d_atlas = nullptr;
    int4* d_tex_areas = nullptr;
    int* d_tex_flags = nullptr;
    float4* d_env = nullptr;
    float* d_lut = nullptr;
    std::vector<int32_t> h_global;
    int64_t n_nodes = 0;
    bool built = false;
    float bounds_lo[3] = {0, 0, 0}, bounds_hi[3] = {1, 1, 1};  // box of the LBVH root (ray-sort quantisation)
    SceneView view{};
};

void pt_set_error(const char* fmt, ...);

#define PT_CUDA(call)                                                                             \
    do {                                                                                          \
        cudaError_t _e = (call);                                                                  \
        if (_e != cudaSuccess) {                                                                  \
            pt_set_error("%s:%d: %s -> %s", __FILE__, __LINE__, #call, cudaGetErrorString(_e));   \
            return PT_ERR_CUDA;                                                                   \
        }                                                                                         \
    } while (0)

#define PT_REQUIRE(cond, msg)                         \
    do {                                              \
        if (!(cond)) {                                \
            pt_set_error("%s: %s", __func__, msg);    \
            return PT_ERR_INVALID;                    \
        }                                             \
    } while (0)

// lbvh.cu — builds nodes over `n_local` primitives whose ids are listed in d_local_ids (device),
// given per-primitive AABBs aabb[2*prim] (min|max as float4).  Returns device nodes + root ref.
int pt_lbvh_build(PtContext* ctx, const float4* d_prim_aabb, const int* d_local_ids, int64_t n_local,
                  float4** d_nodes_out, int64_t* n_nodes_out, int* root_out);

// wavefront.cu
int pt_ensure_pool(PtContext* ctx, size_t capacity);
// lbvh.cu — 64-byte nodes -> 32-byte quantised nodes in the frame [lo, lo + 65535 * scale]
int pt_quantize_nodes(PtContext* ctx, const float4* d_nodes, int64_t n_nodes, const float lo[3], const float scale[3],
                      uint4** d_qnodes_out);
// persist.cu — persistent while-while kernels (PT_MODE_PERSIST)
struct RenderConsts;
int pt_render_persist(PtContext* ctx, const PtScene* s, const RenderConsts& rc, bool legacy, bool count, float4* accum,
                      float4* accum_sq, int shade_min, int serve_min, bool wide = false);
int pt_trace_persist(PtContext* ctx, const PtScene* s, const float4* rays, long long n, float4* hits, bool count,
                     bool sort, bool use_qnodes, int serve_min, int fetch_min, cudaEvent_t ev_sorted, bool wide = false);
// dual.cu — persistent kernel with a lane-private parking place per lane (PT_MODE_DUAL)
int pt_render_dual(PtContext* ctx, const PtScene* s, const RenderConsts& rc, bool legacy, bool count, float4* accum,
                   float4* accum_sq, int shade_min, int serve_min, int blocks_per_sm);
// queue.cu — persistent kernel with block-local shading queues (PT_MODE_QUEUE)
int pt_render_queue(PtContext* ctx, const PtScene* s, const RenderConsts& rc, bool legacy, bool count, float4* accum,
                    float4* accum_sq, int serve_min);
// post.cu
int pt_ensure_scratch(PtContext* ctx, size_t bytes);
// wavefront.cu — pt_render's argument checks (features = true: pt_render_features' variant), the hit acceptance of a shading
// model, and the first hits of the camera rays of one sample (rays float4[2 W H], hits float4[W H], asynchronous)
int pt_check_render_args(const char* fn, const PtContext* ctx, const PtScene* s, const PtCamera* cam, const PtRenderParams* p,
                         const void* accum_dev, const void* accum_sq_dev, bool features);
float pt_render_tmin(int shading_model);
int pt_first_hits(PtContext* ctx, const PtScene* s, const PtCamera* cam, int W, int H, int flags, uint32_t sample,
                  uint32_t seed, float tmin, float4* rays, float4* hits);
