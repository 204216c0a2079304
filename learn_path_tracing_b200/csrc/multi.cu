// multi.cu — one frame on several contexts from one process (pt_multi_*), and scene replication (pt_scene_replicate).
//
// pt_multi_render splits the samples of every pixel over the members exactly like multigpu.split_samples.  Member 0 (the
// root) renders straight into the caller's accumulator (pt_render adds); every other member renders into a library-owned
// partial accumulator on its own device.  Then every member reduces one contiguous slice of the pixels:
//
//     accum_root[slice g] += partial_1[slice g] + ... + partial_{n-1}[slice g]       (member g, in that order)
//
// reading the other devices' partials and the root slice over NVLink (peer access) and writing the root slice back.  The
// slices are disjoint and the root's own render is complete before any reduce starts, so there are no atomics, and the
// summation order is fixed: the frame is deterministic given the per-member accumulators.  Every member moves about
// (n-1)/n of one accumulator through its links instead of the root moving n-1 whole accumulators through its own.
//
// Ordering is by events alone (cross-device cudaStreamWaitEvent); nothing waits on the host unless statistics are asked.
#include <string.h>

#include <algorithm>

#include "bvh4.h"
#include "pt_internal.h"

#define PT_MULTI_MAX 16
#define PT_REDUCE_BLOCK 256

namespace {

// restores the caller's current device (torch and other callers keep their own idea of it)
struct DeviceGuard {
    int dev = -1;
    DeviceGuard() { cudaGetDevice(&dev); }
    ~DeviceGuard() {
        if (dev >= 0) cudaSetDevice(dev);
    }
};

struct ReduceArgs {
    float4* root;                             // accum_root (or accum_sq_root)
    const float4* part[PT_MULTI_MAX - 1];     // partials of members 1 .. n-1, any device
    long long lo, hi;                         // slice [lo, hi) in float4 elements
};

struct __align__(32) F8 {
    float v[8];
};

__device__ __forceinline__ F8 ldg256_nc(const void* p) {
    F8 r;
    asm volatile("ld.global.nc.v8.f32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
                 : "=f"(r.v[0]), "=f"(r.v[1]), "=f"(r.v[2]), "=f"(r.v[3]), "=f"(r.v[4]), "=f"(r.v[5]), "=f"(r.v[6]), "=f"(r.v[7])
                 : "l"(p));
    return r;
}
__device__ __forceinline__ F8 ld256(const void* p) {
    F8 r;
    asm volatile("ld.global.v8.f32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
                 : "=f"(r.v[0]), "=f"(r.v[1]), "=f"(r.v[2]), "=f"(r.v[3]), "=f"(r.v[4]), "=f"(r.v[5]), "=f"(r.v[6]), "=f"(r.v[7])
                 : "l"(p));
    return r;
}
__device__ __forceinline__ float4 ldg128_nc(const float4* p) {
    float4 r;
    asm volatile("ld.global.nc.v4.f32 {%0,%1,%2,%3}, [%4];" : "=f"(r.x), "=f"(r.y), "=f"(r.z), "=f"(r.w) : "l"(p));
    return r;
}
// An empty volatile statement that "rewrites" the loaded registers: volatile asm keeps its order, so every add, which
// reads the rewritten values, comes after the last load is issued — all peer loads of an element are in flight together
// (without it the compiler interleaves loads and adds to save registers and the NVLink latencies add up).
__device__ __forceinline__ void pin(F8& r) {
    asm volatile("" : "+f"(r.v[0]), "+f"(r.v[1]), "+f"(r.v[2]), "+f"(r.v[3]), "+f"(r.v[4]), "+f"(r.v[5]), "+f"(r.v[6]), "+f"(r.v[7]));
}
__device__ __forceinline__ void pin(float4& r) { asm volatile("" : "+f"(r.x), "+f"(r.y), "+f"(r.z), "+f"(r.w)); }
__device__ __forceinline__ void st256(void* p, const F8& r) {
    asm volatile("st.global.v8.f32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8};" ::"l"(p), "f"(r.v[0]), "f"(r.v[1]), "f"(r.v[2]),
                 "f"(r.v[3]), "f"(r.v[4]), "f"(r.v[5]), "f"(r.v[6]), "f"(r.v[7])
                 : "memory");
}

// root[lo, hi) += part[0] + part[1] + ... + part[NP-1], grid-stride.  All NP peer loads of an element are issued before
// the first add.  WIDE: 32-byte vectors (every pointer + lo is 32-byte aligned; an odd last element goes 16 bytes wide).
template <int NP, bool WIDE>
__global__ void __launch_bounds__(PT_REDUCE_BLOCK, 1) k_multi_reduce(const ReduceArgs a) {
    const long long stride = (long long)gridDim.x * blockDim.x;
    const long long first = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (WIDE) {
        const long long pairs = (a.hi - a.lo) >> 1;
        for (long long k = first; k < pairs; k += stride) {
            const long long e = a.lo + 2 * k;
            F8 p[NP];
#pragma unroll
            for (int i = 0; i < NP; ++i) p[i] = ldg256_nc(a.part[i] + e);
            F8 r = ld256(a.root + e);
#pragma unroll
            for (int i = 0; i < NP; ++i) pin(p[i]);
            pin(r);
#pragma unroll
            for (int i = 0; i < NP; ++i)
#pragma unroll
                for (int c = 0; c < 8; ++c) r.v[c] += p[i].v[c];
            st256(a.root + e, r);
        }
        if (((a.hi - a.lo) & 1) && first == 0) {
            const long long e = a.hi - 1;
            float4 p[NP];
#pragma unroll
            for (int i = 0; i < NP; ++i) p[i] = ldg128_nc(a.part[i] + e);
            float4 r = a.root[e];
#pragma unroll
            for (int i = 0; i < NP; ++i) pin(p[i]);
            pin(r);
#pragma unroll
            for (int i = 0; i < NP; ++i) { r.x += p[i].x; r.y += p[i].y; r.z += p[i].z; r.w += p[i].w; }
            a.root[e] = r;
        }
    } else {
        for (long long e = a.lo + first; e < a.hi; e += stride) {
            float4 p[NP];
#pragma unroll
            for (int i = 0; i < NP; ++i) p[i] = ldg128_nc(a.part[i] + e);
            float4 r = a.root[e];
#pragma unroll
            for (int i = 0; i < NP; ++i) pin(p[i]);
            pin(r);
#pragma unroll
            for (int i = 0; i < NP; ++i) { r.x += p[i].x; r.y += p[i].y; r.z += p[i].z; r.w += p[i].w; }
            a.root[e] = r;
        }
    }
}

template <int NP>
cudaError_t launch_reduce_np(const ReduceArgs& a, bool wide, unsigned grid, cudaStream_t st) {
    if (wide) k_multi_reduce<NP, true><<<grid, PT_REDUCE_BLOCK, 0, st>>>(a);
    else k_multi_reduce<NP, false><<<grid, PT_REDUCE_BLOCK, 0, st>>>(a);
    return cudaGetLastError();
}

cudaError_t launch_reduce(const ReduceArgs& a, int np, bool wide, unsigned grid, cudaStream_t st) {
    switch (np) {
#define PT_NP(k) \
    case k: return launch_reduce_np<k>(a, wide, grid, st);
        PT_NP(1) PT_NP(2) PT_NP(3) PT_NP(4) PT_NP(5) PT_NP(6) PT_NP(7) PT_NP(8)
        PT_NP(9) PT_NP(10) PT_NP(11) PT_NP(12) PT_NP(13) PT_NP(14) PT_NP(15)
#undef PT_NP
        default: return cudaErrorInvalidValue;
    }
}

}  // namespace

struct PtMulti {
    int n = 0;
    PtContext* m[PT_MULTI_MAX] = {};
    cudaEvent_t ev_begin = nullptr;                 // root device: the caller's earlier work on the root stream
    cudaEvent_t ev_end = nullptr;                   // root device: the whole frame (stats != NULL)
    cudaEvent_t ev_render[PT_MULTI_MAX] = {};       // member devices: that member's render is done
    cudaEvent_t ev_reduce[PT_MULTI_MAX] = {};       // member devices: that member's slice is reduced
    float4* part[PT_MULTI_MAX] = {};                // members >= 1: partial accumulators (grow-only)
    float4* part_sq[PT_MULTI_MAX] = {};
    size_t part_elems[PT_MULTI_MAX] = {}, part_sq_elems[PT_MULTI_MAX] = {};
};

extern "C" void pt_multi_destroy(PtMulti* g) {
    if (!g) return;
    DeviceGuard dg;
    for (int i = 0; i < g->n; ++i) {
        cudaSetDevice(g->m[i]->device);
        if (g->part[i]) cudaFree(g->part[i]);
        if (g->part_sq[i]) cudaFree(g->part_sq[i]);
        if (g->ev_render[i]) cudaEventDestroy(g->ev_render[i]);
        if (g->ev_reduce[i]) cudaEventDestroy(g->ev_reduce[i]);
        if (i == 0) {
            if (g->ev_begin) cudaEventDestroy(g->ev_begin);
            if (g->ev_end) cudaEventDestroy(g->ev_end);
        }
    }
    delete g;
}

extern "C" int pt_multi_create(PtContext* const* members, int n, PtMulti** out) {
    PT_REQUIRE(out, "null out pointer");
    *out = nullptr;
    PT_REQUIRE(members && n >= 1 && n <= PT_MULTI_MAX, "n must be in [1, 16]");
    for (int i = 0; i < n; ++i) {
        PT_REQUIRE(members[i], "null member context");
        for (int j = 0; j < i; ++j)
            if (members[i] == members[j]) {
                pt_set_error("pt_multi_create: members %d and %d are the same context", j, i);
                return PT_ERR_INVALID;
            }
    }
    DeviceGuard dg;
    // peer access between every ordered pair of distinct devices
    for (int i = 0; i < n; ++i)
        for (int j = 0; j < n; ++j) {
            const int a = members[i]->device, b = members[j]->device;
            if (a == b) continue;
            int can = 0;
            PT_CUDA(cudaDeviceCanAccessPeer(&can, a, b));
            if (!can) {
                pt_set_error("pt_multi_create: device %d cannot access device %d (cudaDeviceCanAccessPeer)", a, b);
                return PT_ERR_INVALID;
            }
            PT_CUDA(cudaSetDevice(a));
            const cudaError_t e = cudaDeviceEnablePeerAccess(b, 0);
            if (e == cudaErrorPeerAccessAlreadyEnabled) {
                cudaGetLastError();  // not a failure; clear it, or the next pt_render reports it
            } else if (e != cudaSuccess) {
                pt_set_error("pt_multi_create: cudaDeviceEnablePeerAccess(%d -> %d): %s", a, b, cudaGetErrorString(e));
                return PT_ERR_CUDA;
            }
        }
    PtMulti* g = new PtMulti();
    g->n = n;
    for (int i = 0; i < n; ++i) g->m[i] = members[i];
    cudaError_t e = cudaSuccess;
    for (int i = 0; i < n && e == cudaSuccess; ++i) {
        e = cudaSetDevice(members[i]->device);
        if (e == cudaSuccess) e = cudaEventCreateWithFlags(&g->ev_render[i], cudaEventDisableTiming);
        if (e == cudaSuccess) e = cudaEventCreateWithFlags(&g->ev_reduce[i], cudaEventDisableTiming);
        if (e == cudaSuccess && i == 0) e = cudaEventCreateWithFlags(&g->ev_begin, cudaEventDisableTiming);
        if (e == cudaSuccess && i == 0) e = cudaEventCreateWithFlags(&g->ev_end, cudaEventDisableTiming);
    }
    if (e != cudaSuccess) {
        pt_set_error("pt_multi_create: %s", cudaGetErrorString(e));
        pt_multi_destroy(g);
        return PT_ERR_CUDA;
    }
    *out = g;
    return PT_OK;
}

static int ensure_partial(PtMulti* g, int i, bool sq, size_t elems) {
    float4** p = sq ? &g->part_sq[i] : &g->part[i];
    size_t* have = sq ? &g->part_sq_elems[i] : &g->part_elems[i];
    if (*have >= elems) return PT_OK;
    if (*p) cudaFree(*p);
    *p = nullptr;
    *have = 0;
    PT_CUDA(cudaMalloc(p, elems * sizeof(float4)));
    *have = elems;
    return PT_OK;
}

extern "C" int pt_multi_render(PtMulti* g, PtScene* const* scenes, const PtCamera* cam, const PtRenderParams* p,
                               void* accum_root, void* accum_sq_root, PtStats* stats) {
    // ---- everything is validated before anything is enqueued
    PT_REQUIRE(g && scenes && cam && p && accum_root, "null argument");
    const int n = g->n;
    PT_REQUIRE(n >= 1 && n <= PT_MULTI_MAX, "bad group");
    PT_REQUIRE(p->reserved[4] == 0 && p->reserved[5] == 0, "row bands (reserved[4], reserved[5]) are not supported here");
    PT_REQUIRE(p->width > 0 && p->height > 0 && p->spp >= 0, "bad image size / spp");
    PT_REQUIRE((long long)p->width * p->height < (1ll << 31), "image too large");
    const bool want_sq = (p->flags & PT_FLAG_ACCUM_SQ) != 0;
    PT_REQUIRE(!want_sq || accum_sq_root, "PT_FLAG_ACCUM_SQ needs accum_sq");
    for (int i = 0; i < n; ++i) {
        const PtScene* s = scenes[i];
        if (!s) {
            pt_set_error("pt_multi_render: scenes[%d] is null", i);
            return PT_ERR_INVALID;
        }
        if (!s->built) {
            pt_set_error("pt_multi_render: scenes[%d] is not built", i);
            return PT_ERR_NOT_BUILT;
        }
        if (s->ctx != g->m[i]) {
            pt_set_error("pt_multi_render: scenes[%d] belongs to another context than members[%d]", i, i);
            return PT_ERR_INVALID;
        }
        const SceneView &a = s->view, &b = scenes[0]->view;
        if (a.n_sph != b.n_sph || a.n_tri != b.n_tri || a.legacy_spheres != b.legacy_spheres) {
            pt_set_error("pt_multi_render: scenes[%d] (%d spheres, %d triangles%s) is not a copy of scenes[0] (%d, %d%s)", i,
                         a.n_sph, a.n_tri, a.legacy_spheres ? ", legacy" : "", b.n_sph, b.n_tri, b.legacy_spheres ? ", legacy" : "");
            return PT_ERR_INVALID;
        }
    }
    const int root_dev = g->m[0]->device;
    for (int k = 0; k < 2; ++k) {
        const void* ptr = k == 0 ? accum_root : (want_sq ? accum_sq_root : nullptr);
        if (!ptr) continue;
        cudaPointerAttributes at;
        const cudaError_t e = cudaPointerGetAttributes(&at, ptr);
        if (e != cudaSuccess) cudaGetLastError();
        if (e != cudaSuccess || (at.type != cudaMemoryTypeDevice && at.type != cudaMemoryTypeManaged) || at.device != root_dev) {
            pt_set_error("pt_multi_render: %s is not device memory of the root's device %d", k == 0 ? "accum_root" : "accum_sq_root",
                         root_dev);
            return PT_ERR_INVALID;
        }
        PT_REQUIRE(((uintptr_t)ptr & 15) == 0, "accumulators must be 16-byte aligned (float4)");
    }

    DeviceGuard dg;
    const size_t WH = (size_t)p->width * p->height;
    int counts[PT_MULTI_MAX], offsets[PT_MULTI_MAX];
    {   // multigpu.split_samples: contiguous ranges, remainder to the low members
        const int base = p->spp / n, rem = p->spp % n;
        for (int i = 0; i < n; ++i) {
            counts[i] = base + (i < rem ? 1 : 0);
            offsets[i] = p->spp_offset + i * base + (i < rem ? i : rem);
        }
    }
    cudaStream_t root_st = g->m[0]->stream;
    PT_CUDA(cudaSetDevice(root_dev));
    PT_CUDA(cudaEventRecord(g->ev_begin, root_st));

    // member 0 first: pt_render reports the usual parameter errors before any other member has enqueued work
    PtRenderParams q = *p;
    if (counts[0] > 0) {
        q.spp = counts[0];
        q.spp_offset = offsets[0];
        const int rc = pt_render(g->m[0], scenes[0], cam, &q, accum_root, accum_sq_root, nullptr);
        if (rc) return rc;
    }
    for (int i = 1; i < n; ++i) {
        PtContext* c = g->m[i];
        PT_CUDA(cudaSetDevice(c->device));
        PT_CUDA(cudaStreamWaitEvent(c->stream, g->ev_begin, 0));
        int rc = ensure_partial(g, i, false, WH);
        if (!rc && want_sq) rc = ensure_partial(g, i, true, WH);
        if (rc) return rc;
        PT_CUDA(cudaMemsetAsync(g->part[i], 0, WH * sizeof(float4), c->stream));
        if (want_sq) PT_CUDA(cudaMemsetAsync(g->part_sq[i], 0, WH * sizeof(float4), c->stream));
        if (counts[i] > 0) {
            q.spp = counts[i];
            q.spp_offset = offsets[i];
            rc = pt_render(c, scenes[i], cam, &q, g->part[i], want_sq ? g->part_sq[i] : nullptr, nullptr);
            if (rc) return rc;
        }
    }
    for (int i = 0; i < n; ++i) {
        PT_CUDA(cudaSetDevice(g->m[i]->device));
        PT_CUDA(cudaEventRecord(g->ev_render[i], g->m[i]->stream));
    }
    // the reduce: member i sums slice i of every partial into the root's accumulator
    if (n > 1) {
        // slice edges on even elements, so that a 32-byte aligned base keeps every slice start 32-byte aligned
        const size_t pairs = (WH + 1) / 2;
        for (int i = 0; i < n; ++i) {
            PtContext* c = g->m[i];
            PT_CUDA(cudaSetDevice(c->device));
            for (int j = 0; j < n; ++j) PT_CUDA(cudaStreamWaitEvent(c->stream, g->ev_render[j], 0));
            const long long lo = (long long)std::min(WH, 2 * (pairs * i / n)), hi = (long long)std::min(WH, 2 * (pairs * (i + 1) / n));
            if (hi > lo) {
                const unsigned grid =
                    (unsigned)std::max<long long>(1, std::min<long long>((hi - lo + 2 * PT_REDUCE_BLOCK - 1) / (2 * PT_REDUCE_BLOCK),
                                                                         (long long)c->sm_count * 8));
                for (int k = 0; k < (want_sq ? 2 : 1); ++k) {
                    ReduceArgs a{};
                    a.root = (float4*)(k == 0 ? accum_root : accum_sq_root);
                    uintptr_t bits = (uintptr_t)(a.root + lo);
                    for (int j = 1; j < n; ++j) {
                        a.part[j - 1] = k == 0 ? g->part[j] : g->part_sq[j];
                        bits |= (uintptr_t)(a.part[j - 1] + lo);
                    }
                    a.lo = lo;
                    a.hi = hi;
                    PT_CUDA(launch_reduce(a, n - 1, (bits & 31) == 0, grid, c->stream));
                }
            }
            PT_CUDA(cudaEventRecord(g->ev_reduce[i], c->stream));
        }
        PT_CUDA(cudaSetDevice(root_dev));
        for (int i = 1; i < n; ++i) PT_CUDA(cudaStreamWaitEvent(root_st, g->ev_reduce[i], 0));
    }
    if (stats) {
        for (int i = 0; i < n; ++i) {
            if (counts[i] > 0) {
                const int rc = pt_render_stats(g->m[i], &stats[i]);
                if (rc) return rc;
            } else {
                memset(&stats[i], 0, sizeof stats[i]);
            }
        }
        PT_CUDA(cudaSetDevice(root_dev));
        PT_CUDA(cudaEventRecord(g->ev_end, root_st));
        PT_CUDA(cudaEventSynchronize(g->ev_end));
    }
    return PT_OK;
}

// ---- scene replication ------------------------------------------------------------------------------
extern "C" int pt_scene_replicate(const PtScene* src, PtContext* dst, PtScene** out) {
    PT_REQUIRE(src && dst && out, "null argument");
    *out = nullptr;
    if (!src->built) {
        pt_set_error("pt_scene_replicate: source scene not built");
        return PT_ERR_NOT_BUILT;
    }
    DeviceGuard dg;
    PT_CUDA(cudaSetDevice(dst->device));
    PtScene* r = new PtScene();
    // host staging and everything the view holds by value (inline primitives, bounds, sizes)
    r->ctx = dst;
    r->h_sph_cr = src->h_sph_cr;
    r->h_sph_mat = src->h_sph_mat;
    r->h_sph_transparency = src->h_sph_transparency;
    r->h_sph_tex = src->h_sph_tex;
    r->legacy_spheres = src->legacy_spheres;
    r->h_tri9 = src->h_tri9;
    r->h_tri_shade = src->h_tri_shade;
    r->n_tri = src->n_tri;
    r->device_generated_tris = src->device_generated_tris;
    r->n_wnodes = src->n_wnodes;
    r->h_global = src->h_global;
    r->n_nodes = src->n_nodes;
    memcpy(r->bounds_lo, src->bounds_lo, sizeof r->bounds_lo);
    memcpy(r->bounds_hi, src->bounds_hi, sizeof r->bounds_hi);
    r->view = src->view;

    const SceneView& v = src->view;
    const size_t n_sph = (size_t)v.n_sph, n_tri = (size_t)src->n_tri, n_nodes = (size_t)src->n_nodes;
    struct Arr {
        void** dst;
        const void* src;
        size_t bytes;
    } arrs[] = {
        {(void**)&r->d_sph_cr, src->d_sph_cr, n_sph * sizeof(float4)},
        {(void**)&r->d_sph_aux, src->d_sph_aux, n_sph * sizeof(float4)},
        {(void**)&r->d_sph_mat, src->d_sph_mat, n_sph * 2 * sizeof(float4)},
        {(void**)&r->d_tri_geo, src->d_tri_geo, n_tri * 3 * sizeof(float4)},
        {(void**)&r->d_tri_shade, src->d_tri_shade, n_tri * 4 * sizeof(float4)},
        {(void**)&r->d_nodes, src->d_nodes, n_nodes * 4 * sizeof(float4)},
        {(void**)&r->d_qnodes, src->d_qnodes, n_nodes * 2 * sizeof(uint4)},
        {(void**)&r->d_wnodes, src->d_wnodes, (size_t)src->n_wnodes * BVH4_NODE_FLOATS * sizeof(float)},
        {(void**)&r->d_global, src->d_global, (size_t)v.n_global * sizeof(int)},
        {(void**)&r->d_atlas, src->d_atlas, (size_t)v.tex_W * v.tex_H * sizeof(uint2)},
        {(void**)&r->d_tex_areas, src->d_tex_areas, (size_t)v.ntex * sizeof(int4)},
        {(void**)&r->d_tex_flags, src->d_tex_flags, (size_t)v.ntex * sizeof(int)},
        {(void**)&r->d_env, src->d_env, (size_t)v.env_W * v.env_H * sizeof(float4)},
        {(void**)&r->d_lut, src->d_lut, 768 * sizeof(float)},
    };
    const int src_dev = src->ctx->device;
    cudaError_t e = cudaSuccess;
    for (const Arr& a : arrs) {
        if (!a.src || !a.bytes) continue;
        e = cudaMalloc(a.dst, a.bytes);
        if (e != cudaSuccess) break;
        e = src_dev == dst->device ? cudaMemcpyAsync(*a.dst, a.src, a.bytes, cudaMemcpyDeviceToDevice, dst->stream)
                                   : cudaMemcpyPeerAsync(*a.dst, dst->device, a.src, src_dev, a.bytes, dst->stream);
        if (e != cudaSuccess) break;
    }
    if (e == cudaSuccess) e = cudaStreamSynchronize(dst->stream);
    if (e != cudaSuccess) {
        pt_set_error("pt_scene_replicate: %s", cudaGetErrorString(e));
        pt_scene_destroy(r);
        return PT_ERR_CUDA;
    }
    SceneView& w = r->view;
    w.sph_cr = r->d_sph_cr; w.sph_aux = r->d_sph_aux; w.sph_mat = r->d_sph_mat;
    w.tri_geo = r->d_tri_geo; w.tri_shade = r->d_tri_shade;
    w.nodes = r->d_nodes; w.qnodes = r->d_qnodes; w.wnodes = r->d_wnodes;
    w.global_prims = r->d_global;
    w.atlas = r->d_atlas; w.tex_areas = r->d_tex_areas; w.tex_flags = r->d_tex_flags;
    w.env = r->d_env; w.lut = r->d_lut;
    r->built = true;
    *out = r;
    return PT_OK;
}
