// wavefront.cu — the render loop of the reference (10_final/__main__.py:78-87,99-103; legacy
// 15_module.py:980-1036) as a persistent-pool wavefront on one B200:
//
//   pool of P path slots in HBM (SoA float4: origin|pixel, direction|sample+bounce, throughput)
//   repeat until every sample of every pixel has terminated:
//     k_extend   one ray segment per live path -> hit record (t, prim, u, v)
//     k_shade    miss: radiance * throughput -> RED.v4 into the accumulator, slot freed
//                hit : scatter (v2 / legacy BSDFs), bounce+1; over the depth limit -> slot freed
//                freed slots immediately start a new camera path (ray generation fused here, sample
//                ids handed out by one block-aggregated atomic), and live + new paths are written
//                COMPACTED into the other pool by warp ballot + block prefix sums, survivors first.
//
// No host synchronisation inside the loop: queue sizes live on the device, the host only reads a small
// counter block back every few iterations (asynchronously, one chunk behind) to learn when to stop.
//
// That split form (one launch per stage per bounce, 160 B of HBM traffic per segment) is kept as
// PT_MODE_SPLIT.  ncu showed both of its kernels issue-/latency-bound rather than HBM-bound
// (profiles/r01_*_split_*), so the default is the FUSED form, k_paths: the same stages, but a path stays
// in registers for up to K segments per launch (extend -> shade -> regenerate in place), and only the
// survivors of a launch go through the ballot/prefix-sum compaction into the HBM pool.  Sample ids are
// strided statically (path id, id + P, id + 2P, ... per pool slot), so regeneration needs no atomics.
#include <math.h>
#include <stdlib.h>
#include <string.h>

#include "wf_common.cuh"

// ------------------------------------------------------------------------------------------------
template <bool COUNT>
__global__ void __launch_bounds__(PT_BLOCK)
k_extend(const SceneView sv, const float4* __restrict__ po, const float4* __restrict__ pd, float4* __restrict__ hits,
         unsigned long long* __restrict__ counters, int q_in, float tmin) {
    const unsigned n = (unsigned)counters[CNT_QUEUE + q_in];
    if (blockIdx.x == 0 && threadIdx.x == 0) {
        counters[CNT_QUEUE + (q_in ^ 1)] = 0ull;  // the shade kernel that follows appends here
        atomicAdd(&counters[CNT_SEGMENTS], (unsigned long long)n);
    }
    TraceCounters tc;
    tc.nodes = 0; tc.prims = 0;
    for (unsigned i = blockIdx.x * PT_BLOCK + threadIdx.x; i < n; i += gridDim.x * PT_BLOCK) {
        const float4 o = po[i], d = pd[i];
        const Hit h = closest_hit<COUNT>(sv, f3(o), f3(d), tmin, INFINITY, tc);
        hits[i] = make_float4(h.t, __int_as_float(h.prim), h.u, h.v);
    }
    if (COUNT) {
        atomicAdd(&counters[CNT_NODES], (unsigned long long)tc.nodes);
        atomicAdd(&counters[CNT_PRIMS], (unsigned long long)tc.prims);
    }
}

// ------------------------------------------------------------------------------------------------
template <bool LEGACY>
__global__ void __launch_bounds__(PT_BLOCK)
k_shade(const SceneView sv, const RenderConsts rc, const PoolPtrs in, const float4* __restrict__ hits,
        const PoolPtrs out, unsigned long long* __restrict__ counters, int q_in, float4* __restrict__ accum,
        float4* __restrict__ accum_sq) {
    __shared__ unsigned s_want[PT_WARPS], s_alive[PT_WARPS];
    __shared__ unsigned long long s_new_base;
    __shared__ unsigned s_granted, s_out_base, s_total_alive;

    const unsigned tid = threadIdx.x, lane = tid & 31u, warp = tid >> 5;
    const unsigned n_in = (unsigned)counters[CNT_QUEUE + q_in];
    unsigned long long* n_out = &counters[CNT_QUEUE + (q_in ^ 1)];
    // other blocks bump CNT_NEXT_PATH concurrently: one thread samples it so the loop bound is block-uniform
    __shared__ int s_remain;
    if (tid == 0) s_remain = *(volatile unsigned long long*)&counters[CNT_NEXT_PATH] < rc.total_paths;
    __syncthreads();
    const bool samples_remain = s_remain != 0;
    const unsigned bound = samples_remain ? rc.pool_cap : n_in;
    const unsigned WH = (unsigned)rc.W * (unsigned)rc.H;

    for (unsigned base = blockIdx.x * PT_BLOCK; base < bound; base += gridDim.x * PT_BLOCK) {
        const unsigned i = base + tid;
        bool alive = false;
        PathState p;
        if (i < n_in) {
            const float4 o = in.o[i], d = in.d[i], l = in.l[i], hr = hits[i];
            p.o = f3(o); p.d = f3(d); p.l = f3(l);
            p.pixel = __float_as_uint(o.w);
            const uint32_t sb = __float_as_uint(d.w);
            p.sample = sb & 0xFFFFFFu;
            p.bounce = sb >> 24;
            Hit h;
            h.t = hr.x; h.prim = __float_as_int(hr.y); h.u = hr.z; h.v = hr.w;
            if (h.prim < 0) {
                // miss: the only light source (sky gradient / environment map), __main__.py:86-87, 15_module.py:990-991
                const float3 c = (LEGACY ? environment_color(sv, p.d) : sky_color(p.d)) * p.l;
                if (isfinite(c.x) && isfinite(c.y) && isfinite(c.z)) {
                    atomicAdd(&accum[p.pixel], make_float4(c.x, c.y, c.z, 1.0f));
                    if (rc.accum_sq) atomicAdd(&accum_sq[p.pixel], make_float4(c.x * c.x, c.y * c.y, c.z * c.z, 1.0f));
                }
            } else {
                if (LEGACY) scatter_legacy(sv, p, h, rc.absorptivity, rc.seed, sv.lut);
                else scatter_v2(sv, p, h, rc.shading_model, rc.seed);
                p.bounce += 1u;
                alive = p.bounce < (uint32_t)rc.max_depth;  // paths over propagate_limit contribute nothing
            }
        }
        // ---- regeneration + compaction ------------------------------------------------------
        const bool want = !alive && samples_remain && i < rc.pool_cap;
        const unsigned wmask = __ballot_sync(0xffffffffu, want);
        const unsigned amask = __ballot_sync(0xffffffffu, alive);
        const unsigned lt = (1u << lane) - 1u;
        unsigned want_rank = __popc(wmask & lt), alive_rank = __popc(amask & lt);
        if (lane == 0) { s_want[warp] = __popc(wmask); s_alive[warp] = __popc(amask); }
        __syncthreads();
        if (tid == 0) {
            unsigned tw = 0, ta = 0;
#pragma unroll
            for (int w = 0; w < PT_WARPS; ++w) { tw += s_want[w]; ta += s_alive[w]; }
            unsigned granted = 0;
            unsigned long long nb = 0;
            if (tw) {
                nb = atomicAdd(&counters[CNT_NEXT_PATH], (unsigned long long)tw);
                if (nb < rc.total_paths) {
                    const unsigned long long left = rc.total_paths - nb;
                    granted = left < tw ? (unsigned)left : tw;
                }
            }
            s_new_base = nb;
            s_granted = granted;
            s_total_alive = ta;
            s_out_base = (ta + granted) ? (unsigned)atomicAdd(n_out, (unsigned long long)(ta + granted)) : 0u;
        }
        __syncthreads();
#pragma unroll
        for (int w = 0; w < PT_WARPS; ++w) {
            if (w < (int)warp) { want_rank += s_want[w]; alive_rank += s_alive[w]; }
        }
        unsigned slot = 0xffffffffu;
        if (alive) {
            slot = s_out_base + alive_rank;
        } else if (want && want_rank < s_granted) {
            // Camera.get_rays for path id -> (sample, pixel); fused ray generation
            const unsigned long long pid = s_new_base + want_rank;
            const uint32_t smp = (uint32_t)(pid / WH);
            const uint32_t pix = (uint32_t)(pid - (unsigned long long)smp * WH);
            p.pixel = pix;
            p.sample = rc.spp_offset + smp;
            p.bounce = 0u;
            p.l = f3(1.0f, 1.0f, 1.0f);
            const float4 u = rng4(p.pixel, p.sample, 0u, rc.seed);
            camera_ray(rc.cam, (int)(pix % (unsigned)rc.W), (int)(pix / (unsigned)rc.W), u, &p.o, &p.d);
            slot = s_out_base + s_total_alive + want_rank;
        }
        if (slot != 0xffffffffu) {
            out.o[slot] = make_float4(p.o.x, p.o.y, p.o.z, __uint_as_float(p.pixel));
            out.d[slot] = make_float4(p.d.x, p.d.y, p.d.z, __uint_as_float(p.sample | (p.bounce << 24)));
            out.l[slot] = make_float4(p.l.x, p.l.y, p.l.z, 0.0f);
        }
        __syncthreads();  // shared scratch is reused by the next trip
    }
}


// ------------------------------------------------------------------------------------------------
// Fused wavefront step: up to K ray segments per path slot per launch, state in registers.
template <bool LEGACY, bool COUNT>
__global__ void __launch_bounds__(PT_BLOCK, 4)
k_paths(const SceneView sv, const RenderConsts rc, const PoolPtrs in, const PoolPtrs out,
        unsigned long long* __restrict__ counters, int launch, int K, float4* __restrict__ accum,
        float4* __restrict__ accum_sq) {
    __shared__ unsigned s_alive[PT_WARPS];
    __shared__ unsigned s_out_base;
    const unsigned tid = threadIdx.x, lane = tid & 31u, warp = tid >> 5;
    const unsigned i = blockIdx.x * PT_BLOCK + tid;
    const unsigned WH = (unsigned)rc.W * (unsigned)rc.H;
    PathState p;
    bool alive = false;
    if (launch == 0) {  // slot i starts the id sequence i, i + P, i + 2P, ...
        if (i < rc.pool_cap) {
            const uint32_t smp = i / WH;
            if (smp < rc.sample_end - rc.spp_offset) {
                start_path(rc, p, i - smp * WH, rc.spp_offset + smp);
                alive = true;
            }
        }
    } else if (i < (unsigned)counters[CNT_LIVE + launch - 1]) {
        const float4 o = in.o[i], d = in.d[i], l = in.l[i];
        p.o = f3(o); p.d = f3(d); p.l = f3(l);
        p.pixel = __float_as_uint(o.w);
        const uint32_t sb = __float_as_uint(d.w);
        p.sample = sb & 0xFFFFFFu;
        p.bounce = sb >> 24;
        alive = true;
    }
    TraceCounters tc;
    tc.nodes = 0; tc.prims = 0;
    unsigned nseg = 0;
    for (int k = 0; k < K; ++k) {
        if (!__any_sync(0xffffffffu, alive)) break;
        if (alive) {
            const Hit h = closest_hit<COUNT>(sv, p.o, p.d, rc.tmin, INFINITY, tc);  // extend
            ++nseg;
            if (h.prim < 0) {  // miss: radiance * throughput into the accumulator, path ends
                const float3 c = (LEGACY ? environment_color(sv, p.d) : sky_color(p.d)) * p.l;
                if (isfinite(c.x) && isfinite(c.y) && isfinite(c.z)) {
                    atomicAdd(&accum[p.pixel], make_float4(c.x, c.y, c.z, 1.0f));
                    if (rc.accum_sq) atomicAdd(&accum_sq[p.pixel], make_float4(c.x * c.x, c.y * c.y, c.z * c.z, 1.0f));
                }
                alive = false;
            } else {  // shade / scatter
                if (LEGACY) scatter_legacy(sv, p, h, rc.absorptivity, rc.seed, sv.lut);
                else scatter_v2(sv, p, h, rc.shading_model, rc.seed);
                p.bounce += 1u;
                alive = p.bounce < (uint32_t)rc.max_depth;
            }
            if (!alive) {  // regenerate in place: next id of this slot's sequence (fused ray generation)
                uint32_t pix = p.pixel + rc.stride_pixels, smp = p.sample + rc.stride_samples;
                if (pix >= WH) { pix -= WH; smp += 1u; }
                if (smp < rc.sample_end) {
                    start_path(rc, p, pix, smp);
                    alive = true;
                }
            }
        }
    }
    // ---- compaction of the survivors into the pool: warp ballot + block prefix sum ----------------
    const unsigned amask = __ballot_sync(0xffffffffu, alive);
    unsigned rank = __popc(amask & ((1u << lane) - 1u));
    if (lane == 0) s_alive[warp] = __popc(amask);
    nseg += __shfl_xor_sync(0xffffffffu, nseg, 16);
    nseg += __shfl_xor_sync(0xffffffffu, nseg, 8);
    nseg += __shfl_xor_sync(0xffffffffu, nseg, 4);
    nseg += __shfl_xor_sync(0xffffffffu, nseg, 2);
    nseg += __shfl_xor_sync(0xffffffffu, nseg, 1);
    if (lane == 0 && nseg) atomicAdd(&counters[CNT_SEGMENTS], (unsigned long long)nseg);
    __syncthreads();
    if (tid == 0) {
        unsigned ta = 0;
#pragma unroll
        for (int w = 0; w < PT_WARPS; ++w) ta += s_alive[w];
        s_out_base = ta ? (unsigned)atomicAdd(&counters[CNT_LIVE + launch], (unsigned long long)ta) : 0u;
    }
    __syncthreads();
#pragma unroll
    for (int w = 0; w < PT_WARPS; ++w)
        if (w < (int)warp) rank += s_alive[w];
    if (alive) {
        const unsigned slot = s_out_base + rank;
        out.o[slot] = make_float4(p.o.x, p.o.y, p.o.z, __uint_as_float(p.pixel));
        out.d[slot] = make_float4(p.d.x, p.d.y, p.d.z, __uint_as_float(p.sample | (p.bounce << 24)));
        out.l[slot] = make_float4(p.l.x, p.l.y, p.l.z, 0.0f);
    }
    if (COUNT) {
        atomicAdd(&counters[CNT_NODES], (unsigned long long)tc.nodes);
        atomicAdd(&counters[CNT_PRIMS], (unsigned long long)tc.prims);
    }
}

// ------------------------------------------------------------------------------------------------
template <bool COUNT>
__global__ void __launch_bounds__(PT_BLOCK)
k_trace(const SceneView sv, const float4* __restrict__ rays, float4* __restrict__ hits, long long n,
        unsigned long long* __restrict__ counters) {
    TraceCounters tc;
    tc.nodes = 0; tc.prims = 0;
    const long long i = (long long)blockIdx.x * PT_BLOCK + threadIdx.x;
    if (i < n) {
        const float4 o = __ldg(&rays[2 * i]), d = __ldg(&rays[2 * i + 1]);
        const Hit h = closest_hit<COUNT>(sv, f3(o), f3(d), o.w, d.w, tc);
        hits[i] = make_float4(h.t, __int_as_float(h.prim), h.u, h.v);
    }
    if (COUNT) {
        atomicAdd(&counters[CNT_NODES], (unsigned long long)tc.nodes);
        atomicAdd(&counters[CNT_PRIMS], (unsigned long long)tc.prims);
    }
}

__global__ void k_generate_rays(const CameraDev cam, int W, int H, uint32_t sample, uint32_t seed, float tmin, float4* rays) {
    const unsigned pix = blockIdx.x * blockDim.x + threadIdx.x;
    if (pix >= (unsigned)W * (unsigned)H) return;
    float3 o, d;
    camera_ray(cam, (int)(pix % (unsigned)W), (int)(pix / (unsigned)W), rng4(pix, sample, 0u, seed), &o, &d);
    rays[2 * pix] = make_float4(o.x, o.y, o.z, tmin);
    rays[2 * pix + 1] = make_float4(d.x, d.y, d.z, INFINITY);
}

// SURVEY 8d config 5 ray generator: origin on the sphere of radius 1.5 about (.5,.5,.5), target ~ U[0,1)^3
__global__ void k_random_rays(float4* rays, long long n, uint32_t seed) {
    const long long k = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= n) return;
    const float4 a = rng4((uint32_t)k, 1u, 0u, seed), b = rng4((uint32_t)k, 1u, 1u, seed);
    const float3 s = sample_at_sphere(a.x, a.y);
    const float3 o = f3(0.5f + 1.5f * s.x, 0.5f + 1.5f * s.y, 0.5f + 1.5f * s.z);
    const float3 d = normalize(f3(a.z, a.w, b.x) - o);
    rays[2 * k] = make_float4(o.x, o.y, o.z, PT_EPS);
    rays[2 * k + 1] = make_float4(d.x, d.y, d.z, INFINITY);
}

// ------------------------------------------------------------------------------------------------
// lattice: 0 = jittered pixel samples (Camera.get_rays), 1 = PT_FLAG_PIXEL_GRID (i/(W-1), stages 2-4),
// 2 = PT_FLAG_RAYS_FAST (legacy Camera.get_rays_fast, 15_module.py:423-436: i/W, pinhole, focal length 1)
static CameraDev make_camera(const PtCamera* c, int W, int H, int lattice = 0) {
    const bool grid = lattice == 1;
    CameraDev d;
    d.pos = make_float3(c->pos[0], c->pos[1], c->pos[2]);
    d.front = make_float3(c->front[0], c->front[1], c->front[2]);
    d.right = make_float3(c->right[0], c->right[1], c->right[2]);
    d.up = make_float3(c->up[0], c->up[1], c->up[2]);
    d.view_w = c->view_w; d.view_h = c->view_h;
    d.focal = c->focal_length; d.aperture = c->aperture;
    d.inv_w = 1.0f / (float)(grid ? W - 1 : W); d.inv_h = 1.0f / (float)(grid ? H - 1 : H);
    d.jitter = lattice ? 0.0f : 1.0f;
    if (lattice == 2) { d.focal = 1.0f; d.aperture = 0.0f; }
    return d;
}

int pt_ensure_pool(PtContext* ctx, size_t capacity) {
    if (!ctx->counters) {
        PT_CUDA(cudaMalloc(&ctx->counters, CNT_TOTAL_WORDS * sizeof(unsigned long long)));
        PT_CUDA(cudaMallocHost(&ctx->counters_host, (4 * CNT_WORDS + PT_MAX_LAUNCHES) * sizeof(unsigned long long)));
        PT_CUDA(cudaEventCreate(&ctx->ev_a));
        PT_CUDA(cudaEventCreate(&ctx->ev_b));
        for (int k = 0; k < 4; ++k) PT_CUDA(cudaEventCreateWithFlags(&ctx->ev_chunk[k], cudaEventDisableTiming));
    }
    if (capacity <= ctx->pool_cap) return PT_OK;
    for (int q = 0; q < 2; ++q)
        for (int a = 0; a < 3; ++a) {
            if (ctx->pool[q][a]) cudaFree(ctx->pool[q][a]);
            ctx->pool[q][a] = nullptr;
        }
    if (ctx->hits) cudaFree(ctx->hits);
    ctx->hits = nullptr;
    ctx->pool_cap = 0;
    for (int q = 0; q < 2; ++q)
        for (int a = 0; a < 3; ++a) PT_CUDA(cudaMalloc(&ctx->pool[q][a], capacity * sizeof(float4)));
    PT_CUDA(cudaMalloc(&ctx->hits, capacity * sizeof(float4)));
    ctx->pool_cap = capacity;
    return PT_OK;
}

static cudaEvent_t get_event(PtContext* ctx, size_t idx) {
    while (ctx->ev_pool.size() <= idx) {
        cudaEvent_t e;
        cudaEventCreate(&e);
        ctx->ev_pool.push_back(e);
    }
    return ctx->ev_pool[idx];
}

// PT_MODE_SPLIT: classic two-kernel wavefront with a dynamically refilled pool.
static int render_split(PtContext* ctx, const PtScene* s, const RenderConsts& rc, bool legacy, bool timing, bool count,
                        float4* accum, float4* accum_sq, int* iterations_out, int* launches_out, size_t* ev_idx_out) {
    cudaStream_t st = ctx->stream;
    const unsigned long long total = rc.total_paths;
    const unsigned max_blocks = (unsigned)ctx->sm_count * 16u;
    unsigned n_upper = rc.pool_cap;  // host-side upper bound of the live queue
    const int CHUNK = 4;
    int iterations = 0, launches = 0, q = 0, chunk_id = 0;
    size_t ev_idx = 0;
    bool done = total == 0;
    while (!done) {
        for (int k = 0; k < CHUNK; ++k) {
            unsigned blocks = (n_upper + PT_BLOCK - 1) / PT_BLOCK;
            if (blocks > max_blocks) blocks = max_blocks;
            if (blocks < 1) blocks = 1;
            PoolPtrs pin = {ctx->pool[q][0], ctx->pool[q][1], ctx->pool[q][2]};
            PoolPtrs pout = {ctx->pool[q ^ 1][0], ctx->pool[q ^ 1][1], ctx->pool[q ^ 1][2]};
            if (timing) cudaEventRecord(get_event(ctx, ev_idx++), st);
            if (count) k_extend<true><<<blocks, PT_BLOCK, 0, st>>>(s->view, pin.o, pin.d, ctx->hits, ctx->counters, q, rc.tmin);
            else k_extend<false><<<blocks, PT_BLOCK, 0, st>>>(s->view, pin.o, pin.d, ctx->hits, ctx->counters, q, rc.tmin);
            if (timing) cudaEventRecord(get_event(ctx, ev_idx++), st);
            if (legacy) k_shade<true><<<blocks, PT_BLOCK, 0, st>>>(s->view, rc, pin, ctx->hits, pout, ctx->counters, q, accum, accum_sq);
            else k_shade<false><<<blocks, PT_BLOCK, 0, st>>>(s->view, rc, pin, ctx->hits, pout, ctx->counters, q, accum, accum_sq);
            if (timing) cudaEventRecord(get_event(ctx, ev_idx++), st);
            q ^= 1;
            iterations++;
            launches += 2;
        }
        // asynchronous read-back of the counter block, examined one chunk late so the GPU never idles
        const int slot = chunk_id & 3;
        unsigned long long* hostc = ctx->counters_host + slot * CNT_WORDS;
        PT_CUDA(cudaMemcpyAsync(hostc, ctx->counters, CNT_WORDS * sizeof(unsigned long long), cudaMemcpyDeviceToHost, st));
        PT_CUDA(cudaEventRecord(ctx->ev_chunk[slot], st));
        if (chunk_id >= 1) {
            const int pslot = (chunk_id - 1) & 3;
            PT_CUDA(cudaEventSynchronize(ctx->ev_chunk[pslot]));
            const unsigned long long* c = ctx->counters_host + pslot * CNT_WORDS;
            const unsigned long long live = c[CNT_QUEUE + q];  // CHUNK is even: the live queue of a chunk end is index q
            if (c[CNT_NEXT_PATH] >= total) {
                n_upper = (unsigned)live;
                if (live == 0) done = true;
            }
        }
        chunk_id++;
        PT_CUDA(cudaGetLastError());
    }
    *iterations_out = iterations;
    *launches_out = launches;
    *ev_idx_out = ev_idx;
    return PT_OK;
}

// PT_MODE_FUSED (default): k_paths, K segments per launch in registers, compaction at write-back.
static int render_fused(PtContext* ctx, const PtScene* s, const RenderConsts& rc, bool legacy, bool timing, bool count,
                        float4* accum, float4* accum_sq, int K, int* iterations_out, int* launches_out, size_t* ev_idx_out) {
    cudaStream_t st = ctx->stream;
    unsigned long long* host_live = ctx->counters_host + 4 * CNT_WORDS;
    unsigned n_upper = rc.pool_cap;
    int launch = 0, q = 0, checked = 0;
    size_t ev_idx = 0;
    bool done = rc.total_paths == 0;
    while (!done) {
        if (launch >= PT_MAX_LAUNCHES) { pt_set_error("pt_render: launch budget exceeded"); return PT_ERR_INVALID; }
        const unsigned blocks = (n_upper + PT_BLOCK - 1) / PT_BLOCK;
        PoolPtrs pin = {ctx->pool[q][0], ctx->pool[q][1], ctx->pool[q][2]};
        PoolPtrs pout = {ctx->pool[q ^ 1][0], ctx->pool[q ^ 1][1], ctx->pool[q ^ 1][2]};
        if (timing) cudaEventRecord(get_event(ctx, ev_idx++), st);
        if (legacy) {
            if (count) k_paths<true, true><<<blocks, PT_BLOCK, 0, st>>>(s->view, rc, pin, pout, ctx->counters, launch, K, accum, accum_sq);
            else k_paths<true, false><<<blocks, PT_BLOCK, 0, st>>>(s->view, rc, pin, pout, ctx->counters, launch, K, accum, accum_sq);
        } else {
            if (count) k_paths<false, true><<<blocks, PT_BLOCK, 0, st>>>(s->view, rc, pin, pout, ctx->counters, launch, K, accum, accum_sq);
            else k_paths<false, false><<<blocks, PT_BLOCK, 0, st>>>(s->view, rc, pin, pout, ctx->counters, launch, K, accum, accum_sq);
        }
        if (timing) cudaEventRecord(get_event(ctx, ev_idx++), st);
        // live count of this launch -> pinned host memory, examined one launch late (the GPU never waits on the host)
        PT_CUDA(cudaMemcpyAsync(host_live + launch, ctx->counters + CNT_LIVE + launch, sizeof(unsigned long long),
                                cudaMemcpyDeviceToHost, st));
        PT_CUDA(cudaEventRecord(ctx->ev_chunk[launch & 3], st));
        q ^= 1;
        launch++;
        while (checked + 1 < launch) {  // everything but the launch just submitted
            PT_CUDA(cudaEventSynchronize(ctx->ev_chunk[checked & 3]));
            const unsigned long long live = host_live[checked];
            n_upper = (unsigned)live;  // live counts never grow: id sequences only end
            if (live == 0) done = true;
            checked++;
        }
        PT_CUDA(cudaGetLastError());
    }
    *iterations_out = launch;
    *launches_out = launch;
    *ev_idx_out = ev_idx;
    return PT_OK;
}

// Argument checks of pt_render, shared with pt_render_features (features = true: there is no sum-of-squares buffer, the
// mode / threshold fields reserved[0..3] are ignored and row bands are refused).  Errors name `fn`.
#define PT_REQUIRE_FN(cond, msg)                     \
    do {                                             \
        if (!(cond)) {                               \
            pt_set_error("%s: %s", fn, msg);         \
            return PT_ERR_INVALID;                   \
        }                                            \
    } while (0)
int pt_check_render_args(const char* fn, const PtContext* ctx, const PtScene* s, const PtCamera* cam, const PtRenderParams* p,
                         const void* accum_dev, const void* accum_sq_dev, bool features) {
    PT_REQUIRE_FN(ctx && s && cam && p && accum_dev, "null argument");
    if (!s->built) { pt_set_error("%s: scene not built", fn); return PT_ERR_NOT_BUILT; }
    PT_REQUIRE_FN(p->width > 0 && p->height > 0 && p->spp >= 0, "bad image size / spp");
    PT_REQUIRE_FN(p->max_depth > 0 && p->max_depth < 256, "max_depth must be in [1,255]");
    PT_REQUIRE_FN((long long)p->spp_offset + p->spp <= (1 << 24), "sample index must stay below 2^24");
    PT_REQUIRE_FN((long long)p->width * p->height < (1ll << 31), "image too large");
    PT_REQUIRE_FN(p->shading_model >= 0 && p->shading_model <= 5, "unknown shading model");
    const bool legacy = p->shading_model == PT_SHADE_LEGACY;
    PT_REQUIRE_FN(legacy || (s->view.n_tri == 0 && !s->view.legacy_spheres), "v2 shading models need a v2 sphere scene");
    PT_REQUIRE_FN(!legacy || s->view.n_sph == 0 || s->view.legacy_spheres, "legacy shading needs legacy (textured) spheres");
    PT_REQUIRE_FN(!(p->flags & PT_FLAG_PIXEL_GRID) || (p->width >= 2 && p->height >= 2), "PT_FLAG_PIXEL_GRID needs width, height >= 2");
    const bool want_sq = (p->flags & PT_FLAG_ACCUM_SQ) != 0;
    PT_REQUIRE_FN(features || !want_sq || accum_sq_dev, "PT_FLAG_ACCUM_SQ needs accum_sq");
    if (!features) {
        PT_REQUIRE_FN(p->reserved[0] >= 0 && p->reserved[0] <= 5, "reserved[0] (wavefront mode) must be 0 ... 5");
        PT_REQUIRE_FN(p->reserved[1] >= 0 && p->reserved[1] <= 4096, "reserved[1] (segments per launch) out of range");
        PT_REQUIRE_FN(p->reserved[2] >= 0 && p->reserved[2] <= 32 && p->reserved[3] >= 0 && p->reserved[3] <= 32,
                      "reserved[2]/[3] (persistent-mode lane thresholds) must be in [0,32]");
    }
    // auto: the persistent ballot-scheduled kernel (measured faster than the K-step fused wavefront on every
    // workload, tree-less scenes included: 16.3 vs 15.3 Gpaths/s on 8_refract 1080p)
    const int mode = !features && p->reserved[0] != PT_MODE_AUTO ? p->reserved[0] : PT_MODE_PERSIST;
    PT_REQUIRE_FN(p->shading_model != PT_SHADE_V2_NORMALS || mode >= PT_MODE_PERSIST,
                  "PT_SHADE_V2_NORMALS needs a persistent kernel (mode 0, 3, 4 or 5)");
    const bool stage = p->shading_model == PT_SHADE_LEGACY_STAGE6 || p->shading_model == PT_SHADE_LEGACY_STAGE7;
    PT_REQUIRE_FN(!stage || mode == PT_MODE_PERSIST, "PT_SHADE_LEGACY_STAGE6/7 need the persistent kernel (mode 0 or 3)");
    const bool banded = p->reserved[4] != 0 || p->reserved[5] != 0;
    PT_REQUIRE_FN(!features || !banded, "row bands (reserved[4], reserved[5]) are not supported");
    PT_REQUIRE_FN(!banded || (p->reserved[4] >= 0 && p->reserved[4] < p->reserved[5] && p->reserved[5] <= p->height),
                  "reserved[4]/[5] (row band) must satisfy 0 <= row0 < row1 <= height");
    PT_REQUIRE_FN(!banded || mode == PT_MODE_PERSIST, "row bands need the persistent kernel (mode 0 or 3)");
#ifndef PT_EXPERIMENTAL
    PT_REQUIRE_FN(mode != PT_MODE_QUEUE && mode != PT_MODE_DUAL,
                  "render modes 4 (queue) and 5 (dual) are experimental kernel forms: rebuild with `make EXPERIMENTAL=1`");
#endif
    PT_REQUIRE_FN(mode != PT_MODE_PERSIST || !(p->flags & PT_FLAG_WIDE) || s->view.wnodes,
                  "PT_FLAG_WIDE: the scene has no 4-wide tree (build it with PT_WIDE=1 in the environment)");
    return PT_OK;
}
#undef PT_REQUIRE_FN

// closest-hit acceptance of a shading model: legacy accepts t > eps, v2 t >= 1e-4, the legacy tutorial stages
// record.t > 1e-3 (7_reflect.py:148)
float pt_render_tmin(int shading_model) {
    if (shading_model == PT_SHADE_LEGACY_STAGE6 || shading_model == PT_SHADE_LEGACY_STAGE7) return nextafterf(1e-3f, 1.0f);
    return shading_model == PT_SHADE_LEGACY ? nextafterf(PT_EPS, 1.0f) : PT_EPS;
}

extern "C" int pt_render(PtContext* ctx, const PtScene* s, const PtCamera* cam, const PtRenderParams* p,
                         void* accum_dev, void* accum_sq_dev, PtStats* stats) {
    {
        const int rca = pt_check_render_args("pt_render", ctx, s, cam, p, accum_dev, accum_sq_dev, false);
        if (rca) return rca;
    }
    const bool legacy = p->shading_model == PT_SHADE_LEGACY;
    const bool want_sq = (p->flags & PT_FLAG_ACCUM_SQ) != 0;
    const int mode = p->reserved[0] != PT_MODE_AUTO ? p->reserved[0] : PT_MODE_PERSIST;
    PT_CUDA(cudaSetDevice(ctx->device));

    // reserved[4], [5]: a band of rows [row0, row1) instead of the whole frame (0, 0 = all rows) — the multi-GPU path
    // renders band by band so that the reduce of one band overlaps the rendering of the next (persistent kernel only)
    const bool banded = p->reserved[4] != 0 || p->reserved[5] != 0;
    const int row0 = banded ? p->reserved[4] : 0, row1 = banded ? p->reserved[5] : p->height;
    const unsigned long long total = (unsigned long long)p->width * (unsigned long long)(row1 - row0) * (unsigned long long)p->spp;
    const size_t def_cap = mode == PT_MODE_SPLIT ? (size_t)1 << 22 : (size_t)1 << 21;
    size_t cap = p->pool_capacity > 0 ? (size_t)p->pool_capacity : def_cap;
    if (cap > total) cap = (size_t)total;
    cap = (cap + PT_BLOCK - 1) / PT_BLOCK * PT_BLOCK;
    if (cap < PT_BLOCK || mode >= PT_MODE_PERSIST) cap = PT_BLOCK;  // the persistent kernel keeps no pool in HBM
    int rc_pool = pt_ensure_pool(ctx, cap);
    if (rc_pool) return rc_pool;

    RenderConsts rc;
    rc.cam = make_camera(cam, p->width, p->height, (p->flags & PT_FLAG_PIXEL_GRID) ? 1 : 0);
    rc.total_paths = total;
    rc.W = p->width; rc.H = p->height;
    rc.seed = p->seed; rc.spp_offset = (uint32_t)p->spp_offset;
    rc.max_depth = p->max_depth; rc.shading_model = p->shading_model;
    rc.absorptivity = p->absorptivity;
    rc.tmin = pt_render_tmin(p->shading_model);
    rc.pool_cap = (unsigned)cap;
    rc.accum_sq = want_sq ? 1 : 0;
    const unsigned long long WH = (unsigned long long)p->width * p->height;
    rc.stride_samples = (uint32_t)(cap / WH);
    rc.stride_pixels = (uint32_t)(cap % WH);
    rc.sample_end = (uint32_t)(p->spp_offset + p->spp);
    rc.row0 = row0; rc.row1 = row1;
    {   // Work unit of the persistent kernel = one 8x4 tile x unit_samples.  A launch ends when its LAST unit ends, and a
        // unit over the heaviest tile runs several times the average, so a short launch (the per-GPU share of a
        // sample-split frame: 8_refract 32 spp, Yoimiya 64 spp on 8 GPUs) spends a visible part of its time in that
        // tail: fewer samples per unit there.  Same-box sweep (profiles/r02_ab_unit_samples.txt): Yoimiya at 64 spp 4204
        // (16) / 4633 (8) / 4688 (4) Mpaths/s, Zhongli 4K at 64 spp 7567 / 8018 / 8130, 8_refract at 32 spp 16482 / 16749 /
        // 16542; from 256 spp on 16 is best everywhere (fewest counter atomics).  PT_UNIT_SAMPLES overrides (A/B runs).
        const char* ue = getenv("PT_UNIT_SAMPLES");
        int us = ue ? atoi(ue) : 0;
        if (us < 1 || us > 64) us = p->spp >= 256 ? 16 : (!legacy || p->spp >= 128 ? 8 : 4);
        rc.unit_samples = (uint32_t)us;
    }

    cudaStream_t st = ctx->stream;
    const bool timing = (p->flags & PT_FLAG_TIMING) != 0;
    const bool count = (p->flags & PT_FLAG_COUNTERS) != 0;
    PT_CUDA(cudaMemsetAsync(ctx->counters, 0, CNT_TOTAL_WORDS * sizeof(unsigned long long), st));
    PT_CUDA(cudaEventRecord(ctx->ev_a, st));

    int iterations = 0, launches = 0, rcode;
    size_t ev_idx = 0;
    if (mode == PT_MODE_QUEUE) {
#ifdef PT_EXPERIMENTAL
        const int serve_min = p->reserved[3] > 0 ? p->reserved[3] : 24;
        if (timing) cudaEventRecord(get_event(ctx, ev_idx++), st);
        rcode = pt_render_queue(ctx, s, rc, legacy, count, (float4*)accum_dev, (float4*)accum_sq_dev, serve_min);
        if (timing) cudaEventRecord(get_event(ctx, ev_idx++), st);
        iterations = 1; launches = 1;
#else
        rcode = PT_ERR_INVALID;
#endif
    } else if (mode == PT_MODE_DUAL) {
#ifdef PT_EXPERIMENTAL
        // dual.cu: phases (miss / hit / regen) fire once shade_min lanes want exactly them
        const int shade_min = p->reserved[2] > 0 ? p->reserved[2] : 20;
        const int serve_min = p->reserved[3] > 0 ? p->reserved[3] : 8;
        if (timing) cudaEventRecord(get_event(ctx, ev_idx++), st);
        rcode = pt_render_dual(ctx, s, rc, legacy, count, (float4*)accum_dev, (float4*)accum_sq_dev, shade_min, serve_min,
                               p->reserved[1] == 3 ? 3 : 4);
        if (timing) cudaEventRecord(get_event(ctx, ev_idx++), st);
        iterations = 1; launches = 1;
#else
        rcode = PT_ERR_INVALID;
#endif
    } else if (mode == PT_MODE_PERSIST) {
        // warp votes (persist.cu): a service (leaf tests, shading, refill) starts once serve_min more lanes wait
        // than after the previous one; finished lanes are shaded once shade_min of them have piled up
        // defaults from same-box sweeps (profiles/r02_ab_postpone_rootbox_trig_thresholds.txt): sphere scenes like a later
        // service (10_final 5885 -> 5997 Mpaths/s at 12 waiting lanes: a sphere test is cheap, node steps should stay full),
        // mesh scenes an earlier shading pass (Yoimiya 4892 -> 4949 at 20 finished lanes; 12 waiting lanes cost it 6 %)
        const int shade_min = p->reserved[2] > 0 ? p->reserved[2] : (legacy ? 20 : 22);
        const int serve_min = p->reserved[3] > 0 ? p->reserved[3] : (legacy ? 8 : 12);
        if (timing) cudaEventRecord(get_event(ctx, ev_idx++), st);
        const bool wide = (p->flags & PT_FLAG_WIDE) != 0;
        rcode = pt_render_persist(ctx, s, rc, legacy, count, (float4*)accum_dev, (float4*)accum_sq_dev, shade_min, serve_min, wide);
        if (timing) cudaEventRecord(get_event(ctx, ev_idx++), st);
        iterations = 1; launches = 1;
    } else if (mode == PT_MODE_SPLIT)
        rcode = render_split(ctx, s, rc, legacy, timing, count, (float4*)accum_dev, (float4*)accum_sq_dev, &iterations, &launches, &ev_idx);
    else
        rcode = render_fused(ctx, s, rc, legacy, timing, count, (float4*)accum_dev, (float4*)accum_sq_dev,
                             p->reserved[1] > 0 ? p->reserved[1] : 32, &iterations, &launches, &ev_idx);
    if (rcode) return rcode;

    // The counter block goes to pinned memory behind the kernel; nothing here waits for the GPU.  A caller that wants
    // the statistics of THIS call passes `stats` (then the call ends with one stream synchronisation) or asks later with
    // pt_render_stats() — the multi-GPU path renders with stats == NULL and lets the reduce follow on the same stream.
    if (!ctx->stats_host) PT_CUDA(cudaMallocHost(&ctx->stats_host, CNT_WORDS * sizeof(unsigned long long)));
    PT_CUDA(cudaMemcpyAsync(ctx->stats_host, ctx->counters, CNT_WORDS * sizeof(unsigned long long), cudaMemcpyDeviceToHost, st));
    PT_CUDA(cudaEventRecord(ctx->ev_b, st));
    PT_CUDA(cudaGetLastError());
    ctx->last_paths = total;
    ctx->last_mode = mode;
    ctx->last_iterations = iterations;
    ctx->last_launches = launches;
    ctx->last_ev_idx = ev_idx;
    ctx->last_timing = timing;
    ctx->last_valid = true;
    if (stats) return pt_render_stats(ctx, stats);
    return PT_OK;
}

extern "C" int pt_render_stats(PtContext* ctx, PtStats* stats) {
    PT_REQUIRE(ctx && stats, "null argument");
    PT_REQUIRE(ctx->last_valid, "no pt_render call on this context yet");
    PT_CUDA(cudaSetDevice(ctx->device));
    PT_CUDA(cudaEventSynchronize(ctx->ev_b));
    const unsigned long long* last = ctx->stats_host;
    const int mode = ctx->last_mode, iterations = ctx->last_iterations, launches = ctx->last_launches;
    const size_t ev_idx = ctx->last_ev_idx;
    const bool timing = ctx->last_timing;
    memset(stats, 0, sizeof *stats);
    stats->paths = ctx->last_paths;
    stats->segments = last[CNT_SEGMENTS];
    stats->nodes_visited = last[CNT_NODES];
    stats->prims_tested = last[CNT_PRIMS];
    cudaEventElapsedTime(&stats->ms_total, ctx->ev_a, ctx->ev_b);
    stats->iterations = iterations;
    stats->launches = launches;
    if (mode == PT_MODE_SPLIT) {
        stats->launches_extend = iterations;
        stats->launches_shade = iterations;
        if (timing) {
            float e = 0, sh = 0;
            for (size_t k = 0; k + 3 <= ev_idx; k += 3) {
                float a = 0, b = 0;
                cudaEventElapsedTime(&a, ctx->ev_pool[k], ctx->ev_pool[k + 1]);
                cudaEventElapsedTime(&b, ctx->ev_pool[k + 1], ctx->ev_pool[k + 2]);
                e += a; sh += b;
            }
            stats->ms_extend = e;
            stats->ms_shade = sh;
        }
    } else {  // fused: one kernel does both stages; its time is reported under ms_shade, launches under both
        stats->launches_extend = 0;
        stats->launches_shade = launches;
        if (timing) {
            float sh = 0;
            for (size_t k = 0; k + 2 <= ev_idx; k += 2) {
                float a = 0;
                cudaEventElapsedTime(&a, ctx->ev_pool[k], ctx->ev_pool[k + 1]);
                sh += a;
            }
            stats->ms_shade = sh;
        }
    }
    if (timing) stats->ms_other = stats->ms_total - stats->ms_extend - stats->ms_shade;
    stats->reserved[0] = mode;
    stats->reserved[3] = (int32_t)last[15];  // debug code of the queue kernel (0 unless built with -DQ_DEBUG)
    return PT_OK;
}

// ------------------------------------------------------------------------------------------------
// The tracer of pt_trace_batch_device for n > 0 rays (counters zeroed by the caller): one ray per thread without a tree
// or with PT_FLAG_TRACE_SIMPLE, else the persistent while-while warps over the (sorted) batch.
static int trace_dispatch(PtContext* ctx, const PtScene* s, const float4* rays, long long n, float4* hits, int flags, bool count,
                          cudaEvent_t ev_sorted, bool* persist) {
    cudaStream_t st = ctx->stream;
    *persist = false;
    if ((flags & PT_FLAG_TRACE_SIMPLE) || s->view.root == PT_NO_BVH) {  // one ray per thread, batch order
        const unsigned blocks = (unsigned)((n + PT_BLOCK - 1) / PT_BLOCK);
        if (count) k_trace<true><<<blocks, PT_BLOCK, 0, st>>>(s->view, rays, hits, n, ctx->counters);
        else k_trace<false><<<blocks, PT_BLOCK, 0, st>>>(s->view, rays, hits, n, ctx->counters);
        return PT_OK;
    }
    const bool sort = !(flags & PT_FLAG_NO_SORT) && n >= (1 << 16);
    const int serve_min = (flags >> 8) & 63, fetch_min = (flags >> 14) & 63;
    const bool wide = (flags & PT_FLAG_TRACE_WIDE) != 0;
    if (wide && !s->view.wnodes) {
        pt_set_error("pt_trace_batch_device: PT_FLAG_TRACE_WIDE: the scene has no 4-wide tree (build it with PT_WIDE=1 in the environment)");
        return PT_ERR_INVALID;
    }
    const int rct = pt_trace_persist(ctx, s, rays, n, hits, count, sort, !(flags & PT_FLAG_NO_QNODES), serve_min ? serve_min : 8,
                                     fetch_min ? fetch_min : 8, ev_sorted, wide);
    if (rct) return rct;
    *persist = true;
    return PT_OK;
}

// Camera rays of one sample of every pixel into rays (float4[2 * W * H], pt_trace_batch_device layout) and their closest
// hits into hits (float4[W * H]), asynchronously on the context stream: the first-hit pass of pt_render_features.
int pt_first_hits(PtContext* ctx, const PtScene* s, const PtCamera* cam, int W, int H, int flags, uint32_t sample,
                  uint32_t seed, float tmin, float4* rays, float4* hits) {
    cudaStream_t st = ctx->stream;
    const long long n = (long long)W * H;
    k_generate_rays<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(make_camera(cam, W, H, (flags & PT_FLAG_PIXEL_GRID) ? 1 : 0),
                                                                 W, H, sample, seed, tmin, rays);
    PT_CUDA(cudaMemsetAsync(ctx->counters, 0, CNT_WORDS * sizeof(unsigned long long), st));
    bool persist;
    // camera rays in pixel order are coherent already: no sort
    return trace_dispatch(ctx, s, rays, n, hits, PT_FLAG_NO_SORT, false, nullptr, &persist);
}

extern "C" int pt_trace_batch_device(PtContext* ctx, const PtScene* s, const void* rays_dev, int64_t n,
                                     void* hits_dev, int flags, PtStats* stats) {
    PT_REQUIRE(ctx && s && (n == 0 || (rays_dev && hits_dev)), "null argument");
    if (!s->built) { pt_set_error("pt_trace_batch: scene not built"); return PT_ERR_NOT_BUILT; }
    PT_REQUIRE(n >= 0, "negative ray count");
    PT_CUDA(cudaSetDevice(ctx->device));
    int rcp = pt_ensure_pool(ctx, PT_BLOCK);
    if (rcp) return rcp;
    cudaStream_t st = ctx->stream;
    const bool count = (flags & PT_FLAG_COUNTERS) != 0;
    bool persist = false;
    PT_CUDA(cudaMemsetAsync(ctx->counters, 0, CNT_WORDS * sizeof(unsigned long long), st));
    PT_CUDA(cudaEventRecord(ctx->ev_a, st));
    if (n > 0) {
        const int rct = trace_dispatch(ctx, s, (const float4*)rays_dev, n, (float4*)hits_dev, flags, count,
                                       stats ? get_event(ctx, 0) : nullptr, &persist);
        if (rct) return rct;
    }
    PT_CUDA(cudaEventRecord(ctx->ev_b, st));
    PT_CUDA(cudaGetLastError());
    if (stats) {
        unsigned long long last[CNT_WORDS];
        PT_CUDA(cudaMemcpyAsync(last, ctx->counters, sizeof last, cudaMemcpyDeviceToHost, st));
        PT_CUDA(cudaStreamSynchronize(st));
        memset(stats, 0, sizeof *stats);
        stats->paths = (uint64_t)n;
        stats->segments = (uint64_t)n;
        stats->nodes_visited = last[CNT_NODES];
        stats->prims_tested = last[CNT_PRIMS];
        cudaEventElapsedTime(&stats->ms_total, ctx->ev_a, ctx->ev_b);
        stats->ms_extend = stats->ms_total;
        if (persist) {  // ms_other = ray keys + radix sort, ms_extend = the traversal kernel alone
            cudaEventElapsedTime(&stats->ms_other, ctx->ev_a, ctx->ev_pool[0]);
            cudaEventElapsedTime(&stats->ms_extend, ctx->ev_pool[0], ctx->ev_b);
        }
        stats->launches = n > 0 ? 1 : 0;
        stats->launches_extend = stats->launches;
    }
    return PT_OK;
}

extern "C" int pt_random_rays_device(PtContext* ctx, void* rays_dev, int64_t n, uint32_t seed) {
    PT_REQUIRE(ctx && (n == 0 || rays_dev) && n >= 0, "bad argument");
    PT_CUDA(cudaSetDevice(ctx->device));
    if (n > 0) k_random_rays<<<(unsigned)((n + 255) / 256), 256, 0, ctx->stream>>>((float4*)rays_dev, n, seed);
    PT_CUDA(cudaGetLastError());
    return PT_OK;
}

extern "C" int pt_generate_rays(PtContext* ctx, const PtCamera* cam, int width, int height, int sample,
                                uint32_t seed, float* rays_host) {
    return pt_generate_rays_ex(ctx, cam, width, height, sample, seed, 0, rays_host);
}

extern "C" int pt_generate_rays_ex(PtContext* ctx, const PtCamera* cam, int width, int height, int sample,
                                   uint32_t seed, int flags, float* rays_host) {
    PT_REQUIRE(ctx && cam && rays_host && width > 0 && height > 0, "bad argument");
    PT_REQUIRE(!(flags & PT_FLAG_PIXEL_GRID) || (width >= 2 && height >= 2), "PT_FLAG_PIXEL_GRID needs width, height >= 2");
    const int lattice = (flags & PT_FLAG_RAYS_FAST) ? 2 : (flags & PT_FLAG_PIXEL_GRID) ? 1 : 0;
    PT_CUDA(cudaSetDevice(ctx->device));
    const size_t n = (size_t)width * height;
    float4* d = nullptr;
    PT_CUDA(cudaMalloc(&d, n * 2 * sizeof(float4)));
    k_generate_rays<<<(unsigned)((n + 255) / 256), 256, 0, ctx->stream>>>(make_camera(cam, width, height, lattice), width, height,
                                                                         (uint32_t)sample, seed, PT_EPS, d);
    cudaError_t e = cudaMemcpyAsync(rays_host, d, n * 2 * sizeof(float4), cudaMemcpyDeviceToHost, ctx->stream);
    if (e == cudaSuccess) e = cudaStreamSynchronize(ctx->stream);
    cudaFree(d);
    PT_CUDA(e);
    return PT_OK;
}
