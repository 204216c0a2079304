// api.cu — handles, scene upload/build and the host-buffer entry points of include/pt_api.h.
#include <math.h>
#include <stdarg.h>
#include <stdlib.h>
#include <string.h>

#include <algorithm>
#include <thread>

#include "bvh4.h"
#include "pt_internal.h"

#define PT_QNODES_MIN (1 << 18)  // trees from 256 Ki nodes (16 MiB of 64-byte nodes) on get the quantised copy

static thread_local char g_err[1024] = "";

void pt_set_error(const char* fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof g_err, fmt, ap);
    va_end(ap);
}

extern "C" const char* pt_last_error(void) { return g_err; }
extern "C" int pt_version(void) { return PT_API_VERSION; }
extern "C" const char* pt_build_info(void) {
#ifdef PT_EXPERIMENTAL
    return "sm_100a experimental=1";
#else
    return "sm_100a experimental=0";
#endif
}

// ---- context ---------------------------------------------------------------------------------
extern "C" int pt_context_create(int device, void* stream, PtContext** out) {
    PT_REQUIRE(out, "null out pointer");
    int n = 0;
    cudaError_t e = cudaGetDeviceCount(&n);
    if (e != cudaSuccess || n == 0) {
        pt_set_error("pt_context_create: no CUDA device (%s); libb200pt has no CPU fallback",
                     e != cudaSuccess ? cudaGetErrorString(e) : "device count 0");
        return PT_ERR_NO_DEVICE;
    }
    PT_REQUIRE(device >= 0 && device < n, "device index out of range");
    PT_CUDA(cudaSetDevice(device));
    cudaDeviceProp prop;
    PT_CUDA(cudaGetDeviceProperties(&prop, device));
    if (prop.major < 10) {
        pt_set_error("pt_context_create: device %d is sm_%d%d; this library is built for sm_100a (B200) only", device,
                     prop.major, prop.minor);
        return PT_ERR_NO_DEVICE;
    }
    PtContext* c = new PtContext();
    c->device = device;
    c->stream = (cudaStream_t)stream;
    c->sm_count = prop.multiProcessorCount;
    *out = c;
    return PT_OK;
}

extern "C" void pt_context_destroy(PtContext* c) {
    if (!c) return;
    cudaSetDevice(c->device);
    for (int q = 0; q < 2; ++q)
        for (int a = 0; a < 3; ++a)
            if (c->pool[q][a]) cudaFree(c->pool[q][a]);
    if (c->hits) cudaFree(c->hits);
    if (c->scratch) cudaFree(c->scratch);
    if (c->sort_scratch) cudaFree(c->sort_scratch);
    if (c->px_scratch) cudaFree(c->px_scratch);
    for (int b = 0; b < 2; ++b) {
        if (c->stage_rays_h[b]) cudaFreeHost(c->stage_rays_h[b]);
        if (c->stage_hits_h[b]) cudaFreeHost(c->stage_hits_h[b]);
        if (c->stage_rays_d[b]) cudaFree(c->stage_rays_d[b]);
        if (c->stage_hits_d[b]) cudaFree(c->stage_hits_d[b]);
        if (c->stage_ev[b]) cudaEventDestroy(c->stage_ev[b]);
        if (c->stage_ev_in[b]) cudaEventDestroy(c->stage_ev_in[b]);
        if (c->stage_ev_cmp[b]) cudaEventDestroy(c->stage_ev_cmp[b]);
        if (c->up_h[b]) cudaFreeHost(c->up_h[b]);
        if (c->up_ev[b]) cudaEventDestroy(c->up_ev[b]);
    }
    if (c->stage_in) cudaStreamDestroy(c->stage_in);
    if (c->stage_out) cudaStreamDestroy(c->stage_out);
    if (c->counters) cudaFree(c->counters);
    if (c->counters_host) cudaFreeHost(c->counters_host);
    if (c->stats_host) cudaFreeHost(c->stats_host);
    if (c->ev_a) cudaEventDestroy(c->ev_a);
    if (c->ev_b) cudaEventDestroy(c->ev_b);
    for (int k = 0; k < 4; ++k)
        if (c->ev_chunk[k]) cudaEventDestroy(c->ev_chunk[k]);
    for (cudaEvent_t e : c->ev_pool) cudaEventDestroy(e);
    delete c;
}

extern "C" int pt_context_set_stream(PtContext* c, void* stream) {
    PT_REQUIRE(c, "null context");
    c->stream = (cudaStream_t)stream;
    return PT_OK;
}

extern "C" int pt_context_sync(PtContext* c) {
    PT_REQUIRE(c, "null context");
    PT_CUDA(cudaSetDevice(c->device));
    PT_CUDA(cudaStreamSynchronize(c->stream));
    return PT_OK;
}

// ---- host-side copies --------------------------------------------------------------------------
// memcpy over a few threads: one core moves ~8 GB/s, far below what the copy engine takes from pinned memory
static void parallel_memcpy(void* dst, const void* src, size_t bytes) {
    const size_t min_slice = (size_t)2 << 20;
    const unsigned hw = std::thread::hardware_concurrency();
    size_t T = std::min<size_t>(std::min<unsigned>(hw ? hw : 1u, 8u), bytes / min_slice);
    if (T <= 1) {
        memcpy(dst, src, bytes);
        return;
    }
    const size_t per = ((bytes + T - 1) / T + 4095) & ~(size_t)4095;
    std::thread th[8];
    size_t started = 0;
    for (size_t i = 1; i < T; ++i) {
        const size_t off = i * per;
        if (off >= bytes) break;
        th[started++] = std::thread([=] { memcpy((char*)dst + off, (const char*)src + off, std::min(per, bytes - off)); });
    }
    memcpy(dst, src, std::min(per, bytes));
    for (size_t i = 0; i < started; ++i) th[i].join();
}

// pageable host memory -> device through two pinned chunks (returns after the last copy has finished)
#define PT_UPLOAD_CHUNK ((size_t)32 << 20)
static int upload_staged(PtContext* ctx, void* dst_dev, const void* src_host, size_t bytes) {
    if (bytes < ((size_t)4 << 20)) {
        PT_CUDA(cudaMemcpy(dst_dev, src_host, bytes, cudaMemcpyHostToDevice));
        return PT_OK;
    }
    for (int b = 0; b < 2; ++b) {
        if (!ctx->up_h[b]) PT_CUDA(cudaMallocHost(&ctx->up_h[b], PT_UPLOAD_CHUNK));
        if (!ctx->up_ev[b]) PT_CUDA(cudaEventCreateWithFlags(&ctx->up_ev[b], cudaEventDisableTiming));
    }
    cudaStream_t st = ctx->stream;
    size_t k = 0;
    for (size_t off = 0; off < bytes; off += PT_UPLOAD_CHUNK, ++k) {
        const int b = (int)(k & 1);
        const size_t len = std::min(PT_UPLOAD_CHUNK, bytes - off);
        if (k >= 2) PT_CUDA(cudaEventSynchronize(ctx->up_ev[b]));  // the copy that last read this chunk is done
        parallel_memcpy(ctx->up_h[b], (const char*)src_host + off, len);
        PT_CUDA(cudaMemcpyAsync((char*)dst_dev + off, ctx->up_h[b], len, cudaMemcpyHostToDevice, st));
        PT_CUDA(cudaEventRecord(ctx->up_ev[b], st));
    }
    PT_CUDA(cudaStreamSynchronize(st));
    return PT_OK;
}

// ---- scene -----------------------------------------------------------------------------------
extern "C" int pt_scene_create(PtContext* ctx, PtScene** out) {
    PT_REQUIRE(ctx && out, "null argument");
    PtScene* s = new PtScene();
    s->ctx = ctx;
    *out = s;
    return PT_OK;
}

static void free_device(PtScene* s) {
    void* ptrs[] = {s->d_sph_cr, s->d_sph_aux, s->d_sph_mat, s->d_tri_geo, s->d_tri_shade, s->d_nodes, s->d_global, s->d_qnodes,
                    s->d_wnodes};
    for (void* p : ptrs)
        if (p) cudaFree(p);
    s->d_sph_cr = s->d_sph_aux = s->d_sph_mat = s->d_tri_geo = s->d_tri_shade = s->d_nodes = nullptr;
    s->d_global = nullptr;
    s->d_qnodes = nullptr;
    s->d_wnodes = nullptr;
    s->n_wnodes = 0;
    s->view.wnodes = nullptr;
    s->built = false;
}

extern "C" void pt_scene_destroy(PtScene* s) {
    if (!s) return;
    cudaSetDevice(s->ctx->device);
    free_device(s);
    if (s->d_atlas) cudaFree(s->d_atlas);
    if (s->d_tex_areas) cudaFree(s->d_tex_areas);
    if (s->d_tex_flags) cudaFree(s->d_tex_flags);
    if (s->d_env) cudaFree(s->d_env);
    if (s->d_lut) cudaFree(s->d_lut);
    delete s;
}

extern "C" int pt_scene_set_spheres(PtScene* s, const float* cr, const PtMaterial* mats, int n) {
    PT_REQUIRE(s && n >= 0 && (n == 0 || (cr && mats)), "bad argument");
    s->h_sph_cr.assign(cr, cr + 4 * (size_t)n);
    s->h_sph_mat.assign(mats, mats + n);
    s->h_sph_transparency.resize(n);
    s->h_sph_tex.assign(n, 0);
    for (int i = 0; i < n; ++i) s->h_sph_transparency[i] = mats[i].transparency;
    s->legacy_spheres = false;
    s->built = false;
    return PT_OK;
}

extern "C" int pt_scene_set_textured_spheres(PtScene* s, const float* cr, const int32_t* transparency,
                                             const int32_t* texture_id, int n) {
    PT_REQUIRE(s && n >= 0 && (n == 0 || (cr && transparency && texture_id)), "bad argument");
    s->h_sph_cr.assign(cr, cr + 4 * (size_t)n);
    s->h_sph_mat.clear();
    s->h_sph_transparency.assign(transparency, transparency + n);
    s->h_sph_tex.assign(texture_id, texture_id + n);
    s->legacy_spheres = true;
    s->built = false;
    return PT_OK;
}

extern "C" int pt_scene_add_mesh(PtScene* s, const float* pos, int nv, const float* nrm, int nn, const float* uv, int nt,
                                 const int32_t* faces, int nf) {
    PT_REQUIRE(s && pos && nrm && uv && faces && nv > 0 && nn > 0 && nt > 0 && nf >= 0, "bad argument");
    PT_REQUIRE(!s->device_generated_tris, "scene already holds device-generated triangles");
    PT_REQUIRE(s->h_tri_shade.size() == 16 * (size_t)s->n_tri,
               "scene already holds a raw triangle soup (pt_scene_set_triangles): meshes and soups do not mix");
    for (int f = 0; f < nf; ++f) {
        const int32_t* F = faces + 10 * (size_t)f;
        for (int k = 0; k < 3; ++k)
            PT_REQUIRE(F[3 * k] >= 0 && F[3 * k] < nv && F[3 * k + 1] >= 0 && F[3 * k + 1] < nn && F[3 * k + 2] >= 0 &&
                           F[3 * k + 2] < nt, "face index out of range");
    }
    s->h_tri9.reserve(s->h_tri9.size() + 9 * (size_t)nf);
    s->h_tri_shade.reserve(s->h_tri_shade.size() + 16 * (size_t)nf);
    for (int f = 0; f < nf; ++f) {
        const int32_t* F = faces + 10 * (size_t)f;
        for (int k = 0; k < 3; ++k)
            for (int c = 0; c < 3; ++c) s->h_tri9.push_back(pos[3 * (size_t)F[3 * k] + c]);
        const float *n0 = nrm + 3 * (size_t)F[1], *n1 = nrm + 3 * (size_t)F[4], *n2 = nrm + 3 * (size_t)F[7];
        const float *t0 = uv + 2 * (size_t)F[2], *t1 = uv + 2 * (size_t)F[5], *t2 = uv + 2 * (size_t)F[8];
        float tid;
        memcpy(&tid, &F[9], 4);
        const float rec[16] = {n0[0], n0[1], n0[2], t0[0], n1[0], n1[1], n1[2], t0[1],
                               n2[0], n2[1], n2[2], t1[0], t1[1], t2[0], t2[1], tid};
        s->h_tri_shade.insert(s->h_tri_shade.end(), rec, rec + 16);
    }
    s->n_tri += nf;
    s->built = false;
    return PT_OK;
}

extern "C" int pt_scene_set_triangles(PtScene* s, const float* verts, int64_t n) {
    PT_REQUIRE(s && n >= 0 && (n == 0 || verts), "bad argument");
    s->h_tri9.assign(verts, verts + 9 * (size_t)n);
    s->h_tri_shade.clear();
    s->n_tri = n;
    s->device_generated_tris = false;
    s->built = false;
    return PT_OK;
}

extern "C" int pt_scene_set_texture_atlas(PtScene* s, const uint8_t* texels, int W, int H, const int32_t* areas,
                                          const int32_t* tex_flags, int ntex) {
    PT_REQUIRE(s && texels && areas && W > 0 && H > 0 && ntex > 0, "bad argument");
    PT_CUDA(cudaSetDevice(s->ctx->device));
    if (s->d_atlas) cudaFree(s->d_atlas);
    if (s->d_tex_areas) cudaFree(s->d_tex_areas);
    if (s->d_tex_flags) cudaFree(s->d_tex_flags);
    s->d_atlas = nullptr; s->d_tex_areas = nullptr; s->d_tex_flags = nullptr;
    PT_CUDA(cudaMalloc(&s->d_atlas, (size_t)W * H * sizeof(uint2)));
    {
        int rcu = upload_staged(s->ctx, s->d_atlas, texels, (size_t)W * H * 8);
        if (rcu) return rcu;
    }
    PT_CUDA(cudaMalloc(&s->d_tex_areas, (size_t)ntex * sizeof(int4)));
    PT_CUDA(cudaMemcpy(s->d_tex_areas, areas, (size_t)ntex * sizeof(int4), cudaMemcpyHostToDevice));
    {
        std::vector<int32_t> fl(ntex, 0);
        if (tex_flags) fl.assign(tex_flags, tex_flags + ntex);
        PT_CUDA(cudaMalloc(&s->d_tex_flags, (size_t)ntex * sizeof(int)));
        PT_CUDA(cudaMemcpy(s->d_tex_flags, fl.data(), (size_t)ntex * sizeof(int), cudaMemcpyHostToDevice));
    }
    if (!s->d_lut) {
        // load_texture transfer functions evaluated like numpy (double) then stored as f32, 15_module.py:101-104
        float lut[768];
        for (int i = 0; i < 256; ++i) {
            const double x = i / 255.0;
            lut[i] = (float)pow(x, 2.2);
            lut[256 + i] = (float)(x * x);
            lut[512 + i] = (float)(x * 2.0 - 1.0);
        }
        PT_CUDA(cudaMalloc(&s->d_lut, sizeof lut));
        PT_CUDA(cudaMemcpy(s->d_lut, lut, sizeof lut, cudaMemcpyHostToDevice));
    }
    s->view.atlas = s->d_atlas;
    s->view.tex_areas = s->d_tex_areas;
    s->view.tex_flags = s->d_tex_flags;
    s->view.lut = s->d_lut;
    s->view.tex_W = W; s->view.tex_H = H; s->view.ntex = ntex;
    return PT_OK;
}

__global__ void k_rgb_to_float4(const float* __restrict__ rgb, size_t n, float4* __restrict__ out) {
    const size_t k = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (k < n) out[k] = make_float4(rgb[3 * k], rgb[3 * k + 1], rgb[3 * k + 2], 0.0f);
}

extern "C" int pt_scene_set_environment(PtScene* s, const float* rgb, int W, int H, const int32_t* area) {
    PT_REQUIRE(s, "null scene");
    PT_CUDA(cudaSetDevice(s->ctx->device));
    if (s->d_env) cudaFree(s->d_env);
    s->d_env = nullptr;
    s->view.env = nullptr;
    s->view.has_env = 0;
    if (!rgb) return PT_OK;
    PT_REQUIRE(W > 0 && H > 0 && area, "bad environment size");
    {   // rgb goes up as it is and is padded to float4 texels on the device
        const size_t n = (size_t)W * H;
        float* d_rgb = nullptr;
        PT_CUDA(cudaMalloc(&s->d_env, n * sizeof(float4)));
        PT_CUDA(cudaMalloc(&d_rgb, n * 3 * sizeof(float)));
        int rcu = upload_staged(s->ctx, d_rgb, rgb, n * 3 * sizeof(float));
        if (rcu == PT_OK) {
            k_rgb_to_float4<<<(unsigned)((n + 255) / 256), 256, 0, s->ctx->stream>>>(d_rgb, n, s->d_env);
            cudaError_t e = cudaStreamSynchronize(s->ctx->stream);
            if (e != cudaSuccess) { pt_set_error("pt_scene_set_environment: %s", cudaGetErrorString(e)); rcu = PT_ERR_CUDA; }
        }
        cudaFree(d_rgb);
        if (rcu) return rcu;
    }
    s->view.env = s->d_env;
    s->view.env_W = W; s->view.env_H = H;
    s->view.env_area = make_int4(area[0], area[1], area[2], area[3]);
    s->view.has_env = 1;
    return PT_OK;
}

// ---- build -------------------------------------------------------------------------------------
__device__ __forceinline__ float pad_of(float lo, float hi) { return 2e-5f * fmaxf(fabsf(lo), fabsf(hi)) + 1e-6f; }

// padded AABB per primitive: aabb[2p] = min, aabb[2p+1] = max
__global__ void k_prim_aabb(const float4* __restrict__ sph_cr, int n_sph, const float4* __restrict__ tri_geo, long long n_tri,
                            float4* __restrict__ aabb) {
    const long long p = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= n_sph + n_tri) return;
    float3 lo, hi;
    if (p < n_sph) {
        const float4 c = sph_cr[p];
        lo = make_float3(c.x - c.w, c.y - c.w, c.z - c.w);
        hi = make_float3(c.x + c.w, c.y + c.w, c.z + c.w);
    } else {
        const float4* g = tri_geo + 3 * (size_t)(p - n_sph);
        const float4 v0 = g[0], e1 = g[1], e2 = g[2];
        const float3 a = make_float3(v0.x, v0.y, v0.z), b = make_float3(v0.x + e1.x, v0.y + e1.y, v0.z + e1.z),
                     c = make_float3(v0.x + e2.x, v0.y + e2.y, v0.z + e2.z);
        lo = make_float3(fminf(a.x, fminf(b.x, c.x)), fminf(a.y, fminf(b.y, c.y)), fminf(a.z, fminf(b.z, c.z)));
        hi = make_float3(fmaxf(a.x, fmaxf(b.x, c.x)), fmaxf(a.y, fmaxf(b.y, c.y)), fmaxf(a.z, fmaxf(b.z, c.z)));
    }
    const float px = pad_of(lo.x, hi.x), py = pad_of(lo.y, hi.y), pz = pad_of(lo.z, hi.z);
    aabb[2 * p] = make_float4(lo.x - px, lo.y - py, lo.z - pz, 0.0f);
    aabb[2 * p + 1] = make_float4(hi.x + px, hi.y + py, hi.z + pz, 0.0f);
}

__global__ void k_tri_geo_from_verts(const float* __restrict__ v9, long long n, float4* __restrict__ geo) {
    const long long k = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= n) return;
    const float* v = v9 + 9 * k;
    geo[3 * k] = make_float4(v[0], v[1], v[2], 0.0f);
    geo[3 * k + 1] = make_float4(__fsub_rn(v[3], v[0]), __fsub_rn(v[4], v[1]), __fsub_rn(v[5], v[2]), 0.0f);
    geo[3 * k + 2] = make_float4(__fsub_rn(v[6], v[0]), __fsub_rn(v[7], v[1]), __fsub_rn(v[8], v[2]), 0.0f);
}

// SURVEY 8d config 5 generator, bit-identical to oracle/pt_oracle.c:orc_random_triangles
__device__ __forceinline__ uint4 pcg4d_u(uint4 v) {
    v.x = v.x * 1664525u + 1013904223u; v.y = v.y * 1664525u + 1013904223u;
    v.z = v.z * 1664525u + 1013904223u; v.w = v.w * 1664525u + 1013904223u;
    v.x += v.y * v.w; v.y += v.z * v.x; v.z += v.x * v.y; v.w += v.y * v.z;
    v.x ^= v.x >> 16; v.y ^= v.y >> 16; v.z ^= v.z >> 16; v.w ^= v.w >> 16;
    v.x += v.y * v.w; v.y += v.z * v.x; v.z += v.x * v.y; v.w += v.y * v.z;
    return v;
}
__device__ __forceinline__ float u01_u(unsigned x) { return (float)(x >> 8) * (1.0f / 16777216.0f); }

__global__ void k_random_tris(long long n, unsigned seed, float s, float4* __restrict__ geo) {
    const long long k = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= n) return;
    const uint4 a = pcg4d_u(make_uint4((unsigned)k, 0u, 0u, seed)), b = pcg4d_u(make_uint4((unsigned)k, 0u, 1u, seed)),
                c = pcg4d_u(make_uint4((unsigned)k, 0u, 2u, seed));
    const float ce[3] = {u01_u(a.x), u01_u(a.y), u01_u(a.z)};
    const float ub[3] = {u01_u(b.x), u01_u(b.y), u01_u(b.z)};
    const float uc[3] = {u01_u(c.x), u01_u(c.y), u01_u(c.z)};
    float p0[3], p1[3], p2[3];
    for (int i = 0; i < 3; ++i) {
        const float e1 = __fmul_rn(s, __fsub_rn(__fmul_rn(2.0f, ub[i]), 1.0f));
        const float e2 = __fmul_rn(s, __fsub_rn(__fmul_rn(2.0f, uc[i]), 1.0f));
        p0[i] = __fsub_rn(ce[i], __fmul_rn(__fadd_rn(e1, e2), 1.0f / 3.0f));
        p1[i] = __fadd_rn(p0[i], e1);
        p2[i] = __fadd_rn(p0[i], e2);
    }
    geo[3 * k] = make_float4(p0[0], p0[1], p0[2], 0.0f);
    geo[3 * k + 1] = make_float4(__fsub_rn(p1[0], p0[0]), __fsub_rn(p1[1], p0[1]), __fsub_rn(p1[2], p0[2]), 0.0f);
    geo[3 * k + 2] = make_float4(__fsub_rn(p2[0], p0[0]), __fsub_rn(p2[1], p0[1]), __fsub_rn(p2[2], p0[2]), 0.0f);
}

extern "C" int pt_scene_set_random_triangles(PtScene* s, int64_t n, uint32_t seed, float edge_scale) {
    PT_REQUIRE(s && n > 0 && n < (1ll << 31), "bad triangle count");
    PT_CUDA(cudaSetDevice(s->ctx->device));
    s->h_tri9.clear();
    s->h_tri_shade.clear();
    if (s->d_tri_geo) cudaFree(s->d_tri_geo);
    s->d_tri_geo = nullptr;
    PT_CUDA(cudaMalloc(&s->d_tri_geo, (size_t)n * 3 * sizeof(float4)));
    k_random_tris<<<(unsigned)((n + 255) / 256), 256, 0, s->ctx->stream>>>(n, seed, edge_scale, s->d_tri_geo);
    PT_CUDA(cudaGetLastError());
    s->n_tri = n;
    s->device_generated_tris = true;
    s->built = false;
    return PT_OK;
}

namespace {
struct Box {
    float lo[3], hi[3];
    void reset() { for (int c = 0; c < 3; ++c) { lo[c] = INFINITY; hi[c] = -INFINITY; } }
    void grow(const Box& b) { for (int c = 0; c < 3; ++c) { lo[c] = fminf(lo[c], b.lo[c]); hi[c] = fmaxf(hi[c], b.hi[c]); } }
    float ext() const { return fmaxf(hi[0] - lo[0], fmaxf(hi[1] - lo[1], hi[2] - lo[2])); }
};
}  // namespace

static Box host_prim_box(const PtScene* s, int64_t p) {
    Box b;
    const int64_t n_sph = (int64_t)s->h_sph_cr.size() / 4;
    if (p < n_sph) {
        const float* c = &s->h_sph_cr[4 * p];
        for (int k = 0; k < 3; ++k) { b.lo[k] = c[k] - c[3]; b.hi[k] = c[k] + c[3]; }
    } else {
        const float* v = &s->h_tri9[9 * (p - n_sph)];
        for (int k = 0; k < 3; ++k) {
            b.lo[k] = fminf(v[k], fminf(v[3 + k], v[6 + k]));
            b.hi[k] = fmaxf(v[k], fmaxf(v[3 + k], v[6 + k]));
        }
    }
    return b;
}

// Primitives whose extent dwarfs everything else (the radius-10000 ground sphere of every v2 scene,
// the +-100 ground plane of the legacy scenes) would collapse the Morton grid: they are kept out of
// the LBVH and tested first for every ray.  Scenes with <= 8 primitives skip the tree entirely and
// are tested in insertion order like the reference's World.hit loop.
static void select_global_prims(PtScene* s, int64_t n_total, std::vector<int32_t>& global) {
    global.clear();
    if (s->device_generated_tris) {  // no host copy to measure; a single triangle needs no tree
        if (n_total < 2)
            for (int64_t p = 0; p < n_total; ++p) global.push_back((int32_t)p);
        return;
    }
    if (n_total <= 8) {
        for (int64_t p = 0; p < n_total; ++p) global.push_back((int32_t)p);
        return;
    }
    const int K = 16;
    std::vector<std::pair<float, int64_t>> top;  // K largest extents
    for (int64_t p = 0; p < n_total; ++p) {
        const float e = host_prim_box(s, p).ext();
        if ((int)top.size() < K) { top.emplace_back(e, p); std::push_heap(top.begin(), top.end(), std::greater<>()); }
        else if (e > top.front().first) {
            std::pop_heap(top.begin(), top.end(), std::greater<>());
            top.back() = {e, p};
            std::push_heap(top.begin(), top.end(), std::greater<>());
        }
    }
    std::sort(top.begin(), top.end(), [](auto& a, auto& b) { return a.first > b.first; });
    std::vector<char> is_top(n_total, 0);
    for (auto& t : top) is_top[t.second] = 1;
    Box rest;
    rest.reset();
    for (int64_t p = 0; p < n_total; ++p)
        if (!is_top[p]) rest.grow(host_prim_box(s, p));
    for (size_t k = 0; k < top.size(); ++k) {
        Box others = rest;
        for (size_t j = k + 1; j < top.size(); ++j) others.grow(host_prim_box(s, top[j].second));
        if (top[k].first > 0.5f * others.ext()) global.push_back((int32_t)top[k].second);
        else break;
    }
    if (n_total - (int64_t)global.size() < 2) {
        global.clear();
        for (int64_t p = 0; p < n_total && p < 64; ++p) global.push_back((int32_t)p);
    }
    std::sort(global.begin(), global.end());
}

extern "C" int pt_scene_build(PtScene* s) {
    PT_REQUIRE(s, "null scene");
    PtContext* ctx = s->ctx;
    PT_CUDA(cudaSetDevice(ctx->device));
    cudaStream_t st = ctx->stream;
    const int64_t n_sph = (int64_t)s->h_sph_cr.size() / 4;
    const int64_t n_tri = s->n_tri;
    const int64_t n_total = n_sph + n_tri;
    // an empty World() is a valid scene (2_camera_and_ray/__main__.py:26-28 renders the bare sky): every ray misses
    PT_REQUIRE(n_total < (1ll << 31), "too many primitives");
    PT_REQUIRE(s->h_tri_shade.empty() || s->h_tri_shade.size() == 16 * (size_t)n_tri, "triangle shading records out of step");

    float4* keep_geo = s->device_generated_tris ? s->d_tri_geo : nullptr;
    if (keep_geo) s->d_tri_geo = nullptr;
    free_device(s);
    s->d_tri_geo = keep_geo;

    // spheres
    if (n_sph) {
        std::vector<float> aux(4 * (size_t)n_sph), mat(8 * (size_t)n_sph, 0.0f);
        for (int64_t i = 0; i < n_sph; ++i) {
            const float r = s->h_sph_cr[4 * i + 3];
            aux[4 * i] = r * r;  // f32 product, the reference's radius**2
            memcpy(&aux[4 * i + 1], &s->h_sph_transparency[i], 4);
            memcpy(&aux[4 * i + 2], &s->h_sph_tex[i], 4);
            aux[4 * i + 3] = 0.0f;
            if (!s->legacy_spheres) {
                const PtMaterial& m = s->h_sph_mat[i];
                float* o = &mat[8 * i];
                o[0] = m.albedo[0]; o[1] = m.albedo[1]; o[2] = m.albedo[2]; o[3] = m.roughness;
                memcpy(&o[4], &m.metallic, 4);
                o[5] = m.ior;
                memcpy(&o[6], &m.transparency, 4);
            }
        }
        PT_CUDA(cudaMalloc(&s->d_sph_cr, (size_t)n_sph * sizeof(float4)));
        PT_CUDA(cudaMalloc(&s->d_sph_aux, (size_t)n_sph * sizeof(float4)));
        PT_CUDA(cudaMalloc(&s->d_sph_mat, (size_t)n_sph * 2 * sizeof(float4)));
        PT_CUDA(cudaMemcpyAsync(s->d_sph_cr, s->h_sph_cr.data(), (size_t)n_sph * 16, cudaMemcpyHostToDevice, st));
        PT_CUDA(cudaMemcpyAsync(s->d_sph_aux, aux.data(), (size_t)n_sph * 16, cudaMemcpyHostToDevice, st));
        PT_CUDA(cudaMemcpyAsync(s->d_sph_mat, mat.data(), (size_t)n_sph * 32, cudaMemcpyHostToDevice, st));
        PT_CUDA(cudaStreamSynchronize(st));
    }
    // triangles
    if (n_tri && !s->device_generated_tris) {
        float* d_v9 = nullptr;
        PT_CUDA(cudaMalloc(&d_v9, (size_t)n_tri * 9 * sizeof(float)));
        cudaError_t e = cudaMemcpyAsync(d_v9, s->h_tri9.data(), (size_t)n_tri * 36, cudaMemcpyHostToDevice, st);
        if (e == cudaSuccess) e = cudaMalloc(&s->d_tri_geo, (size_t)n_tri * 3 * sizeof(float4));
        if (e == cudaSuccess) {
            k_tri_geo_from_verts<<<(unsigned)((n_tri + 255) / 256), 256, 0, st>>>(d_v9, n_tri, s->d_tri_geo);
            e = cudaStreamSynchronize(st);
        }
        cudaFree(d_v9);
        PT_CUDA(e);
        if (!s->h_tri_shade.empty()) {
            PT_CUDA(cudaMalloc(&s->d_tri_shade, (size_t)n_tri * 4 * sizeof(float4)));
            PT_CUDA(cudaMemcpy(s->d_tri_shade, s->h_tri_shade.data(), (size_t)n_tri * 64, cudaMemcpyHostToDevice));
        }
    }

    // global primitives + LBVH over the rest
    select_global_prims(s, n_total, s->h_global);
    const int64_t n_local = n_total - (int64_t)s->h_global.size();
    // global spheres go inline into the kernel parameters, other global primitives into a small device list
    std::vector<int32_t> listed;
    SceneView& vw = s->view;
    vw.n_inl = 0;
    vw.n_inl_tri = 0;
    for (int32_t p : s->h_global) {
        if (p >= n_sph && vw.n_inl_tri < PT_MAX_INLINE_TRI && !s->h_tri9.empty() && !getenv("PT_NO_INLINE_TRIS")) {
            // same values as k_tri_geo_from_verts writes into tri_geo (IEEE single subtraction on either side)
            const int k = vw.n_inl_tri++;
            const float* v = &s->h_tri9[9 * (size_t)(p - n_sph)];
            vw.inl_tri_id[k] = p;
            vw.inl_tri[k][0] = make_float4(v[0], v[1], v[2], 0.0f);
            vw.inl_tri[k][1] = make_float4(v[3] - v[0], v[4] - v[1], v[5] - v[2], 0.0f);
            vw.inl_tri[k][2] = make_float4(v[6] - v[0], v[7] - v[1], v[8] - v[2], 0.0f);
        } else if (p < n_sph && vw.n_inl < PT_MAX_INLINE) {
            const int k = vw.n_inl++;
            const float* c = &s->h_sph_cr[4 * (size_t)p];
            vw.inl_id[k] = p;
            vw.inl_transparent[k] = s->h_sph_transparency[p];
            vw.inl_r2[k] = c[3] * c[3];
            vw.inl_cr[k] = make_float4(c[0], c[1], c[2], c[3]);
        } else {
            listed.push_back(p);
        }
    }
    if (!listed.empty()) {
        PT_CUDA(cudaMalloc(&s->d_global, listed.size() * sizeof(int)));
        PT_CUDA(cudaMemcpy(s->d_global, listed.data(), listed.size() * sizeof(int), cudaMemcpyHostToDevice));
    }
    int root = PT_NO_BVH;
    s->n_nodes = 0;
    if (n_local >= 2) {
        float4* d_aabb = nullptr;
        int* d_ids = nullptr;
        PT_CUDA(cudaMalloc(&d_aabb, (size_t)n_total * 2 * sizeof(float4)));
        cudaError_t e = cudaMalloc(&d_ids, (size_t)n_local * sizeof(int));
        int rc = PT_OK;
        if (e == cudaSuccess) {
            k_prim_aabb<<<(unsigned)((n_total + 255) / 256), 256, 0, st>>>(s->d_sph_cr, (int)n_sph, s->d_tri_geo, n_tri, d_aabb);
            std::vector<int> ids;
            ids.reserve((size_t)n_local);
            size_t g = 0;
            for (int64_t p = 0; p < n_total; ++p) {
                if (g < s->h_global.size() && s->h_global[g] == p) { ++g; continue; }
                ids.push_back((int)p);
            }
            e = cudaMemcpyAsync(d_ids, ids.data(), ids.size() * sizeof(int), cudaMemcpyHostToDevice, st);
            if (e == cudaSuccess) e = cudaStreamSynchronize(st);
            if (e == cudaSuccess) rc = pt_lbvh_build(ctx, d_aabb, d_ids, n_local, &s->d_nodes, &s->n_nodes, &root);
        }
        cudaFree(d_aabb);
        if (d_ids) cudaFree(d_ids);
        PT_CUDA(e);
        if (rc) return rc;
    }
    if (root != PT_NO_BVH && s->n_nodes > 0) {  // root box = union of node 0's two child boxes
        float n0[16];
        PT_CUDA(cudaMemcpy(n0, s->d_nodes, sizeof n0, cudaMemcpyDeviceToHost));
        const float lo0[3] = {n0[0], n0[1], n0[2]}, hi0[3] = {n0[3], n0[4], n0[5]};
        const float lo1[3] = {n0[6], n0[7], n0[8]}, hi1[3] = {n0[9], n0[10], n0[11]};
        for (int c = 0; c < 3; ++c) {
            s->bounds_lo[c] = fminf(lo0[c], lo1[c]);
            s->bounds_hi[c] = fmaxf(hi0[c], hi1[c]);
        }
    }
    // big trees also get 32-byte quantised nodes (half the L1 wavefronts and bytes per visit in k_trace_persist)
    s->view.qnodes = nullptr;
    if (root != PT_NO_BVH && s->n_nodes >= PT_QNODES_MIN) {
        float scale[3];
        for (int c = 0; c < 3; ++c) scale[c] = fmaxf((s->bounds_hi[c] - s->bounds_lo[c]) / 65535.0f, 1e-30f) * (1.0f + 1e-6f);
        int rcq = pt_quantize_nodes(ctx, s->d_nodes, s->n_nodes, s->bounds_lo, scale, &s->d_qnodes);
        if (rcq) return rcq;
        s->view.qnodes = s->d_qnodes;
        for (int c = 0; c < 3; ++c) { s->view.qlo[c] = s->bounds_lo[c]; s->view.qscale[c] = scale[c]; }
    }
    // EXPERIMENTAL (PT_WIDE=1): 4-wide copy of the tree, collapsed on the host (bvh4.h), for k_trace_persist<.., WIDE>
    s->view.wnodes = nullptr;
#ifdef PT_EXPERIMENTAL
    {
        const char* wenv = getenv("PT_WIDE");
        if (wenv && wenv[0] == '1' && root != PT_NO_BVH && s->n_nodes > 0) {
            std::vector<float> h2((size_t)s->n_nodes * 16);
            PT_CUDA(cudaMemcpy(h2.data(), s->d_nodes, h2.size() * sizeof(float), cudaMemcpyDeviceToHost));
            const std::vector<float> w = bvh4::collapse(h2.data(), s->n_nodes);
            PT_REQUIRE(!w.empty(), "bvh4 collapse produced no nodes");
            PT_CUDA(cudaMalloc(&s->d_wnodes, w.size() * sizeof(float)));
            PT_CUDA(cudaMemcpy(s->d_wnodes, w.data(), w.size() * sizeof(float), cudaMemcpyHostToDevice));
            s->n_wnodes = (int64_t)(w.size() / BVH4_NODE_FLOATS);
            s->view.wnodes = s->d_wnodes;
        }
    }
#endif
    SceneView& v = s->view;
    v.sph_cr = s->d_sph_cr; v.sph_aux = s->d_sph_aux; v.sph_mat = s->d_sph_mat;
    v.tri_geo = s->d_tri_geo; v.tri_shade = s->d_tri_shade;
    v.nodes = s->d_nodes; v.global_prims = s->d_global;
    v.n_sph = (int)n_sph; v.n_tri = (int)n_tri; v.n_nodes = (int)s->n_nodes; v.n_global = (int)listed.size();
    v.root = root;
    for (int c = 0; c < 3; ++c) { v.root_lo[c] = s->bounds_lo[c]; v.root_hi[c] = s->bounds_hi[c]; }
    v.legacy_spheres = s->legacy_spheres ? 1 : 0;
    s->built = true;
    return PT_OK;
}

extern "C" int pt_scene_bvh_info(const PtScene* s, int64_t* n_nodes, int64_t* n_prims, int64_t* n_global) {
    PT_REQUIRE(s && s->built, "scene not built");
    if (n_nodes) *n_nodes = s->n_nodes;
    if (n_prims) *n_prims = (int64_t)s->view.n_sph + s->view.n_tri;
    if (n_global) *n_global = (int64_t)s->h_global.size();
    return PT_OK;
}

extern "C" int pt_scene_bvh_download(const PtScene* s, float* nodes, int64_t n_nodes, int32_t* global_prims, int64_t n_global) {
    PT_REQUIRE(s && s->built, "scene not built");
    PT_REQUIRE(n_nodes == s->n_nodes && n_global == (int64_t)s->h_global.size(), "size mismatch (call pt_scene_bvh_info)");
    PT_CUDA(cudaSetDevice(s->ctx->device));
    if (n_nodes) PT_CUDA(cudaMemcpy(nodes, s->d_nodes, (size_t)n_nodes * 64, cudaMemcpyDeviceToHost));
    if (n_global) memcpy(global_prims, s->h_global.data(), (size_t)n_global * 4);
    return PT_OK;
}

extern "C" int pt_scene_triangles_download(const PtScene* s, float* tris, int64_t n) {
    PT_REQUIRE(s && tris && n >= 0 && n <= s->n_tri && s->d_tri_geo, "bad argument");
    PT_CUDA(cudaSetDevice(s->ctx->device));
    PT_CUDA(cudaStreamSynchronize(s->ctx->stream));
    PT_CUDA(cudaMemcpy(tris, s->d_tri_geo, (size_t)n * 48, cudaMemcpyDeviceToHost));
    return PT_OK;
}

// ---- host-buffer wrappers ----------------------------------------------------------------------
// pt_trace_batch: host rays in, host ids/t out.  The batch is cut into chunks that go through a
// double-buffered pipeline — a few CPU threads copy chunk k into pinned memory, a copy stream does its H2D, the context's
// stream sort + trace + unpack (records -> ids | t), a second copy stream the D2H, and meanwhile the CPU copies the results
// of chunk k-1 out: H2D(k+1), tracing(k) and D2H(k-1) overlap — so pageable caller memory never
// meets cudaMemcpy directly and nothing is allocated per call (grow-only staging in the context).
static int ensure_trace_staging(PtContext* ctx, int64_t chunk) {
    if (ctx->stage_chunk >= chunk) return PT_OK;
    for (int b = 0; b < 2; ++b) {
        if (ctx->stage_rays_h[b]) cudaFreeHost(ctx->stage_rays_h[b]);
        if (ctx->stage_hits_h[b]) cudaFreeHost(ctx->stage_hits_h[b]);
        if (ctx->stage_rays_d[b]) cudaFree(ctx->stage_rays_d[b]);
        if (ctx->stage_hits_d[b]) cudaFree(ctx->stage_hits_d[b]);
        ctx->stage_rays_h[b] = ctx->stage_hits_h[b] = nullptr;
        ctx->stage_rays_d[b] = ctx->stage_hits_d[b] = nullptr;
    }
    ctx->stage_chunk = 0;
    for (int b = 0; b < 2; ++b) {
        PT_CUDA(cudaMallocHost(&ctx->stage_rays_h[b], (size_t)chunk * 32));
        PT_CUDA(cudaMallocHost(&ctx->stage_hits_h[b], (size_t)chunk * 8));   // ids[chunk] | t[chunk]
        PT_CUDA(cudaMalloc(&ctx->stage_rays_d[b], (size_t)chunk * 32));
        PT_CUDA(cudaMalloc(&ctx->stage_hits_d[b], (size_t)chunk * 24));      // float4 records | ids | t
        if (!ctx->stage_ev[b]) PT_CUDA(cudaEventCreateWithFlags(&ctx->stage_ev[b], cudaEventDisableTiming));
        if (!ctx->stage_ev_in[b]) PT_CUDA(cudaEventCreateWithFlags(&ctx->stage_ev_in[b], cudaEventDisableTiming));
        if (!ctx->stage_ev_cmp[b]) PT_CUDA(cudaEventCreateWithFlags(&ctx->stage_ev_cmp[b], cudaEventDisableTiming));
    }
    if (!ctx->stage_in) PT_CUDA(cudaStreamCreateWithFlags(&ctx->stage_in, cudaStreamNonBlocking));
    if (!ctx->stage_out) PT_CUDA(cudaStreamCreateWithFlags(&ctx->stage_out, cudaStreamNonBlocking));
    ctx->stage_chunk = chunk;
    return PT_OK;
}

// hit records (t, prim, u, v) -> ids[n] | t[n] in place of the first half of the record array's staging twin:
// 8 instead of 16 bytes per ray cross PCIe and the host only copies
__global__ void k_unpack_hits(const float4* __restrict__ hits, int64_t n, int32_t* __restrict__ ids, float* __restrict__ t) {
    const int64_t k = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= n) return;
    const float4 h = hits[k];
    const int id = __float_as_int(h.y);
    ids[k] = id;
    t[k] = id >= 0 ? h.x : -1.0f;
}

extern "C" int pt_trace_batch(PtContext* ctx, const PtScene* s, const float* rays_host, int64_t n, int32_t* prim_id_host,
                              float* t_host, PtStats* stats) {
    PT_REQUIRE(ctx && s && n >= 0 && (n == 0 || (rays_host && prim_id_host && t_host)), "bad argument");
    if (stats) memset(stats, 0, sizeof *stats);
    if (n == 0) return PT_OK;
    if (!s->built) { pt_set_error("pt_trace_batch: scene not built"); return PT_ERR_NOT_BUILT; }
    PT_CUDA(cudaSetDevice(ctx->device));
    // chunks of at most 4 Mi rays; a batch is cut into at least four so that staging, transfers and tracing overlap
    const int64_t CHUNK_MAX = (int64_t)1 << 22, CHUNK_MIN = (int64_t)1 << 18;
    int64_t chunk = ((n + 3) / 4 + 65535) / 65536 * 65536;
    chunk = std::min(CHUNK_MAX, std::max(CHUNK_MIN, chunk));
    if (chunk > n) chunk = n;
    int rc = ensure_trace_staging(ctx, chunk);
    if (rc) return rc;
    cudaStream_t st = ctx->stream;
    const int64_t n_chunks = (n + chunk - 1) / chunk;
    for (int64_t k = 0; k <= n_chunks; ++k) {
        const int b = (int)(k & 1);
        if (k < n_chunks) {
            const int64_t lo = k * chunk, cnt = (lo + chunk <= n ? chunk : n - lo);
            // buffers b (host and device) were last used by chunk k-2, whose D2H the host waited for in iteration k-1:
            // everything of that chunk is over, no further events are needed for the reuse
            parallel_memcpy(ctx->stage_rays_h[b], rays_host + 8 * lo, (size_t)cnt * 32);
            if (k == 0) {  // the copy stream starts after whatever the caller queued on the context's stream
                PT_CUDA(cudaEventRecord(ctx->stage_ev_cmp[1], st));
                PT_CUDA(cudaStreamWaitEvent(ctx->stage_in, ctx->stage_ev_cmp[1], 0));
            }
            PT_CUDA(cudaMemcpyAsync(ctx->stage_rays_d[b], ctx->stage_rays_h[b], (size_t)cnt * 32, cudaMemcpyHostToDevice,
                                    ctx->stage_in));
            PT_CUDA(cudaEventRecord(ctx->stage_ev_in[b], ctx->stage_in));
            PT_CUDA(cudaStreamWaitEvent(st, ctx->stage_ev_in[b], 0));
            PtStats cs;
            rc = pt_trace_batch_device(ctx, s, ctx->stage_rays_d[b], cnt, ctx->stage_hits_d[b], stats ? PT_FLAG_COUNTERS : 0,
                                       stats ? &cs : nullptr);
            if (rc) return rc;
            if (stats) {
                stats->paths += cs.paths; stats->segments += cs.segments;
                stats->nodes_visited += cs.nodes_visited; stats->prims_tested += cs.prims_tested;
                stats->ms_total += cs.ms_total; stats->ms_extend += cs.ms_extend;
                stats->launches += cs.launches; stats->launches_extend += cs.launches_extend;
            }
            int32_t* ids_d = (int32_t*)((char*)ctx->stage_hits_d[b] + (size_t)chunk * 16);
            k_unpack_hits<<<(unsigned)((cnt + 255) / 256), 256, 0, st>>>((const float4*)ctx->stage_hits_d[b], cnt, ids_d,
                                                                         (float*)(ids_d + chunk));
            PT_CUDA(cudaEventRecord(ctx->stage_ev_cmp[b], st));
            PT_CUDA(cudaStreamWaitEvent(ctx->stage_out, ctx->stage_ev_cmp[b], 0));
            PT_CUDA(cudaMemcpyAsync(ctx->stage_hits_h[b], ids_d, (size_t)chunk * 8, cudaMemcpyDeviceToHost, ctx->stage_out));
            PT_CUDA(cudaEventRecord(ctx->stage_ev[b], ctx->stage_out));
        }
        if (k >= 1) {  // unpack chunk k-1 while the GPU works on chunk k
            const int pb = (int)((k - 1) & 1);
            const int64_t lo = (k - 1) * chunk, cnt = (lo + chunk <= n ? chunk : n - lo);
            PT_CUDA(cudaEventSynchronize(ctx->stage_ev[pb]));
            parallel_memcpy(prim_id_host + lo, ctx->stage_hits_h[pb], (size_t)cnt * 4);
            parallel_memcpy(t_host + lo, (const int32_t*)ctx->stage_hits_h[pb] + chunk, (size_t)cnt * 4);
        }
    }
    PT_CUDA(cudaGetLastError());
    return PT_OK;
}
