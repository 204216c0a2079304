// denoise.cu — first-hit guide features (pt_render_features) and the variance-guided edge-avoiding a-trous filter
// (pt_denoise): the spatial part of SVGF (Schied et al. 2017) over the a-trous wavelet filter of Dammertz et al. 2010.
// DESIGN.md "Denoising" states the equations; tests/denoise_ref.py restates them in float64 NumPy.
//
//   features   per sample: k_generate_rays + the batch tracer (the same first hits pt_trace_batch returns), then
//              k_features_resolve turns (ray, hit) into the two feature planes and ADDS them (sample order: a 4-spp
//              call equals four 1-spp calls bit for bit)
//   filter     k_denoise_prepare (mean, variance of the mean, albedo demodulation, packed guides), then `iterations`
//              passes of k_denoise_atrous at steps 1, 2, 4, ...; the last one remodulates into out.  No atomics.
#include <cuda_fp16.h>
#include <math.h>

#include "wf_common.cuh"

// ---- features ------------------------------------------------------------------------------------------------------
// feat = float4[2][n]: plane 0 += (normal facing the ray, t) on a hit; plane 1 += (albedo, 1) on a hit and
// (miss radiance clamped to [0,1], 0) on a miss.  Surface attributes come from shade.cuh, as in the scatter code.
template <bool LEGACY>
__global__ void __launch_bounds__(256) k_features_resolve(const SceneView sv, const float4* __restrict__ rays,
                                                          const float4* __restrict__ hits, long long n,
                                                          float4* __restrict__ feat) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const float4 ro = rays[2 * i], rd = rays[2 * i + 1], hr = hits[i];
    const float3 o = f3(ro), d = f3(rd);
    Hit h;
    h.t = hr.x; h.prim = __float_as_int(hr.y); h.u = hr.z; h.v = hr.w;
    float4 p1 = feat[n + i];
    if (h.prim < 0) {
        const float3 e = LEGACY ? environment_color(sv, d) : sky_color(d);
        p1.x += fminf(fmaxf(e.x, 0.0f), 1.0f);
        p1.y += fminf(fmaxf(e.y, 0.0f), 1.0f);
        p1.z += fminf(fmaxf(e.z, 0.0f), 1.0f);
        feat[n + i] = p1;
        return;
    }
    const float3 point = o + h.t * d;
    float3 normal, albedo;
    if (LEGACY) {
        const LegacySurface sf = legacy_surface(sv, sv.lut, h, point);
        normal = sf.normal;
        albedo = sf.albedo;
    } else {
        normal = sphere_normal_v2(__ldg(&sv.sph_cr[h.prim]), point);
        albedo = f3(__ldg(&sv.sph_mat[2 * h.prim]));
    }
    if (dot(d, normal) > 0.0f) normal = -normal;
    float4 p0 = feat[i];
    p0.x += normal.x; p0.y += normal.y; p0.z += normal.z; p0.w += h.t;
    p1.x += albedo.x; p1.y += albedo.y; p1.z += albedo.z; p1.w += 1.0f;
    feat[i] = p0;
    feat[n + i] = p1;
}

static int ensure_px_scratch(PtContext* ctx, size_t bytes) {
    if (bytes <= ctx->px_scratch_bytes) return PT_OK;
    if (ctx->px_scratch) cudaFree(ctx->px_scratch);
    ctx->px_scratch = nullptr;
    ctx->px_scratch_bytes = 0;
    PT_CUDA(cudaMalloc(&ctx->px_scratch, bytes));
    ctx->px_scratch_bytes = bytes;
    return PT_OK;
}

extern "C" int pt_render_features(PtContext* ctx, const PtScene* s, const PtCamera* cam, const PtRenderParams* p,
                                  void* features_dev) {
    const int rca = pt_check_render_args("pt_render_features", ctx, s, cam, p, features_dev, nullptr, true);
    if (rca) return rca;
    PT_CUDA(cudaSetDevice(ctx->device));
    if (p->spp == 0) return PT_OK;
    int rc = pt_ensure_pool(ctx, PT_BLOCK);  // the tracer's counter block
    if (rc) return rc;
    const long long n = (long long)p->width * p->height;
    rc = ensure_px_scratch(ctx, (size_t)n * 48);  // rays (32 B) + hits (16 B) of one sample
    if (rc) return rc;
    float4* rays = (float4*)ctx->px_scratch;
    float4* hits = rays + 2 * n;
    const bool legacy = p->shading_model == PT_SHADE_LEGACY;
    const float tmin = pt_render_tmin(p->shading_model);
    for (int k = 0; k < p->spp; ++k) {
        rc = pt_first_hits(ctx, s, cam, p->width, p->height, p->flags, (uint32_t)(p->spp_offset + k), p->seed, tmin, rays, hits);
        if (rc) return rc;
        const unsigned blocks = (unsigned)((n + 255) / 256);
        if (legacy) k_features_resolve<true><<<blocks, 256, 0, ctx->stream>>>(s->view, rays, hits, n, (float4*)features_dev);
        else k_features_resolve<false><<<blocks, 256, 0, ctx->stream>>>(s->view, rays, hits, n, (float4*)features_dev);
    }
    PT_CUDA(cudaGetLastError());
    return PT_OK;
}

// ---- filter --------------------------------------------------------------------------------------------------------
// Guide record, 16 bytes per pixel (uint4), written once by k_denoise_prepare and read by every pass:
//   .x  z: mean hit distance, fp32
//   .y  grad z = (dz/di, dz/dj) as two fp16 (low half = di), each clamped to +-65504 first
//   .z  normal x | y << 16, snorm16 (round-to-nearest-even of n * 32767)
//   .w  normal z, snorm16 in the low half; 0 in the high half
// A pixel without a normal (no hit, or |sum of normals| < 1e-6) stores (0, 0, 0).  z, grad z and the normal are
// computed with explicitly rounded fp32 operations (no contraction), so a float32 NumPy evaluation reproduces the record
// bit for bit; the filter arithmetic after that is plain fp32.
#define DN_BX 32
#define DN_BY 8

struct Guide {
    float z, gx, gy;
    float3 n;
    bool has_n;
};

__device__ __forceinline__ Guide unpack_guide(uint4 r) {
    Guide g;
    g.z = __uint_as_float(r.x);
    const __half2 gz = *reinterpret_cast<const __half2*>(&r.y);
    g.gx = __low2float(gz);
    g.gy = __high2float(gz);
    const int nx = (int)(short)(r.z & 0xffffu), ny = (int)(short)(r.z >> 16), nz = (int)(short)(r.w & 0xffffu);
    const float s = 1.0f / 32767.0f;
    g.n = f3((float)nx * s, (float)ny * s, (float)nz * s);
    g.has_n = (nx | ny | nz) != 0;
    return g;
}

__device__ __forceinline__ float mean_depth(const float4* __restrict__ feat, long long n, long long k) {
    return __fdiv_rn(__ldg(&feat[k]).w, fmaxf(__ldg(&feat[n + k]).w, 1.0f));
}

__device__ __forceinline__ float3 albedo_of(float4 f1, float N) {  // a = max(plane1.rgb / N, 1e-3)
    return f3(fmaxf(__fdiv_rn(f1.x, N), 1e-3f), fmaxf(__fdiv_rn(f1.y, N), 1e-3f), fmaxf(__fdiv_rn(f1.z, N), 1e-3f));
}

__device__ __forceinline__ float luminance(float3 c) { return 0.2126f * c.x + 0.7152f * c.y + 0.0722f * c.z; }

__device__ __forceinline__ unsigned short snorm16(float v) {
    const int q = max(-32767, min(32767, __float2int_rn(__fmul_rn(v, 32767.0f))));
    return (unsigned short)(short)q;
}

// central difference of z along one axis, one-sided at the borders, 0 across an axis of one pixel
__device__ __forceinline__ float depth_grad(float zm, float z, float zp, bool has_m, bool has_p) {
    if (has_m && has_p) return __fmul_rn(__fsub_rn(zp, zm), 0.5f);
    if (has_p) return __fsub_rn(zp, z);
    if (has_m) return __fsub_rn(z, zm);
    return 0.0f;
}

// Per pixel: mean, per-channel variance of the mean (float64: sq - sum^2/N cancels), albedo, demodulated colour and its
// luminance variance into col = (c, sigma^2), and the guide record.  iterations == 0: out = accum / spp directly.
__global__ void __launch_bounds__(DN_BX * DN_BY) k_denoise_prepare(int W, int H, float N, int iterations,
                                                                   const float4* __restrict__ accum,
                                                                   const float4* __restrict__ accum_sq,
                                                                   const float4* __restrict__ feat, float4* __restrict__ col,
                                                                   uint4* __restrict__ guides, float4* __restrict__ out) {
    const int i = blockIdx.x * DN_BX + threadIdx.x, j = blockIdx.y * DN_BY + threadIdx.y;
    if (i >= W || j >= H) return;
    const long long n = (long long)W * H, k = (long long)j * W + i;
    const float4 sum = __ldg(&accum[k]);
    if (iterations == 0) {
        out[k] = make_float4(__fdiv_rn(sum.x, N), __fdiv_rn(sum.y, N), __fdiv_rn(sum.z, N), 1.0f);
        return;
    }
    const float4 sq = __ldg(&accum_sq[k]);
    const float4 f0 = __ldg(&feat[k]), f1 = __ldg(&feat[n + k]);
    const double Nd = (double)N, norm = Nd * fmax(Nd - 1.0, 1.0);
    const float vx = (float)(fmax(0.0, (double)sq.x - (double)sum.x * (double)sum.x / Nd) / norm);
    const float vy = (float)(fmax(0.0, (double)sq.y - (double)sum.y * (double)sum.y / Nd) / norm);
    const float vz = (float)(fmax(0.0, (double)sq.z - (double)sum.z * (double)sum.z / Nd) / norm);
    const float3 a = albedo_of(f1, N);
    const float3 c = f3(sum.x / N / a.x, sum.y / N / a.y, sum.z / N / a.z);
    const float var = 0.2126f * vx / (a.x * a.x) + 0.7152f * vy / (a.y * a.y) + 0.0722f * vz / (a.z * a.z);
    col[k] = make_float4(c.x, c.y, c.z, var);

    const float z = mean_depth(feat, n, k);
    const float zl = i > 0 ? mean_depth(feat, n, k - 1) : 0.0f, zr = i + 1 < W ? mean_depth(feat, n, k + 1) : 0.0f;
    const float zd = j > 0 ? mean_depth(feat, n, k - W) : 0.0f, zu = j + 1 < H ? mean_depth(feat, n, k + W) : 0.0f;
    const float gx = fminf(fmaxf(depth_grad(zl, z, zr, i > 0, i + 1 < W), -65504.0f), 65504.0f);
    const float gy = fminf(fmaxf(depth_grad(zd, z, zu, j > 0, j + 1 < H), -65504.0f), 65504.0f);
    const float len2 = __fadd_rn(__fadd_rn(__fmul_rn(f0.x, f0.x), __fmul_rn(f0.y, f0.y)), __fmul_rn(f0.z, f0.z));
    const float len = __fsqrt_rn(len2);
    unsigned short nx = 0, ny = 0, nz = 0;
    if (f1.w > 0.0f && len >= 1e-6f) {
        nx = snorm16(__fdiv_rn(f0.x, len));
        ny = snorm16(__fdiv_rn(f0.y, len));
        nz = snorm16(__fdiv_rn(f0.z, len));
    }
    const __half2 gz = __floats2half2_rn(gx, gy);
    guides[k] = make_uint4(__float_as_uint(z), *reinterpret_cast<const unsigned*>(&gz), (unsigned)nx | ((unsigned)ny << 16),
                           (unsigned)nz);
}

// One a-trous pass at `step`: 5x5 taps h = (1/16, 1/4, 3/8, 1/4, 1/16)^2 spaced `step` apart, taps outside the image
// skipped, weight h * w_z * w_n * w_l; the centre tap weighs h(0,0) = 9/64.  Colour and variance from cin into cout; the
// last pass (out != NULL) writes the remodulated colour c * albedo into out instead.  Plain grid, the taps go through L1.
__global__ void __launch_bounds__(DN_BX * DN_BY) k_denoise_atrous(int W, int H, int step, float sigma_l, float sigma_n,
                                                                  float sigma_z, const float4* __restrict__ cin,
                                                                  const uint4* __restrict__ guides,
                                                                  float4* __restrict__ cout, const float4* __restrict__ feat,
                                                                  float N, float4* __restrict__ out) {
    const int i = blockIdx.x * DN_BX + threadIdx.x, j = blockIdx.y * DN_BY + threadIdx.y;
    if (i >= W || j >= H) return;
    const long long k = (long long)j * W + i;
    const float4 cp = __ldg(&cin[k]);
    const Guide gp = unpack_guide(__ldg(&guides[k]));
    // g(sigma^2): 3x3 Gaussian (1/4, 1/2, 1/4)^2 of the variance at step 1, over the taps inside the image
    float gv = 0.0f, gw = 0.0f;
#pragma unroll
    for (int dy = -1; dy <= 1; ++dy)
#pragma unroll
        for (int dx = -1; dx <= 1; ++dx) {
            const int qi = i + dx, qj = j + dy;
            if (qi < 0 || qi >= W || qj < 0 || qj >= H) continue;
            const float w = (dx == 0 ? 0.5f : 0.25f) * (dy == 0 ? 0.5f : 0.25f);
            gv += w * __ldg(&cin[(long long)qj * W + qi]).w;
            gw += w;
        }
    const float inv_l = 1.0f / (sigma_l * sqrtf(gv / gw) + 1e-4f);
    const float lp = luminance(f3(cp));
    const float hc = 9.0f / 64.0f;
    float sw = hc, sv = hc * hc * cp.w;
    float3 sc = hc * f3(cp);
    const float hk[3] = {3.0f / 8.0f, 1.0f / 4.0f, 1.0f / 16.0f};
#pragma unroll
    for (int dy = -2; dy <= 2; ++dy)
#pragma unroll
        for (int dx = -2; dx <= 2; ++dx) {
            if (dx == 0 && dy == 0) continue;
            const int qi = i + dx * step, qj = j + dy * step;
            if (qi < 0 || qi >= W || qj < 0 || qj >= H) continue;
            const long long q = (long long)qj * W + qi;
            const float4 cq = __ldg(&cin[q]);
            const Guide gq = unpack_guide(__ldg(&guides[q]));
            const float wz = expf(-fabsf(gp.z - gq.z) /
                                  (sigma_z * fabsf(gp.gx * (float)(dx * step) + gp.gy * (float)(dy * step)) + 1e-4f));
            float wn;
            if (gp.has_n != gq.has_n) wn = 0.0f;
            else if (!gp.has_n) wn = 1.0f;
            else wn = powf(fmaxf(0.0f, dot(gp.n, gq.n)), sigma_n);
            const float wl = expf(-fabsf(lp - luminance(f3(cq))) * inv_l);
            const float w = hk[dx < 0 ? -dx : dx] * hk[dy < 0 ? -dy : dy] * wz * wn * wl;
            sw += w;
            sc = sc + w * f3(cq);
            sv += w * w * cq.w;
        }
    const float inv = 1.0f / sw;
    const float3 c = sc * inv;
    if (out) {
        const float3 a = albedo_of(__ldg(&feat[(long long)W * H + k]), N);
        out[k] = make_float4(c.x * a.x, c.y * a.y, c.z * a.z, 1.0f);
    } else {
        cout[k] = make_float4(c.x, c.y, c.z, sv * inv * inv);
    }
}

extern "C" int pt_denoise(PtContext* ctx, const void* accum_dev, const void* accum_sq_dev, const void* features_dev,
                          const PtDenoiseParams* p, void* out_dev) {
    PT_REQUIRE(ctx && accum_dev && features_dev && p && out_dev, "null argument");
    PT_REQUIRE(accum_sq_dev, "needs the sum of squares (render with PT_FLAG_ACCUM_SQ)");
    PT_REQUIRE(p->width > 0 && p->height > 0 && (long long)p->width * p->height < (1ll << 31), "bad image size");
    PT_REQUIRE(p->spp >= 1, "spp must be >= 1");
    PT_REQUIRE(p->iterations >= 0 && p->iterations <= 10, "iterations must be in [0,10]");
    PT_REQUIRE(p->sigma_l >= 0.0f && p->sigma_n >= 0.0f && p->sigma_z >= 0.0f && isfinite(p->sigma_l) &&
                   isfinite(p->sigma_n) && isfinite(p->sigma_z),
               "sigma_l, sigma_n, sigma_z must be finite and >= 0 (0 = default)");
    PT_CUDA(cudaSetDevice(ctx->device));
    const int W = p->width, H = p->height;
    const long long n = (long long)W * H;
    const float N = (float)p->spp;
    const float sl = p->sigma_l > 0.0f ? p->sigma_l : 4.0f, sn = p->sigma_n > 0.0f ? p->sigma_n : 128.0f,
                sz = p->sigma_z > 0.0f ? p->sigma_z : 1.0f;
    const int rc = ensure_px_scratch(ctx, (size_t)n * 48);  // colour ping-pong (2 x 16 B) + guides (16 B)
    if (rc) return rc;
    float4* col[2] = {(float4*)ctx->px_scratch, (float4*)ctx->px_scratch + n};
    uint4* guides = (uint4*)((float4*)ctx->px_scratch + 2 * n);
    const dim3 block(DN_BX, DN_BY), grid((unsigned)((W + DN_BX - 1) / DN_BX), (unsigned)((H + DN_BY - 1) / DN_BY));
    cudaStream_t st = ctx->stream;
    const float4* feat = (const float4*)features_dev;
    k_denoise_prepare<<<grid, block, 0, st>>>(W, H, N, p->iterations, (const float4*)accum_dev, (const float4*)accum_sq_dev,
                                              feat, col[0], guides, (float4*)out_dev);
    for (int it = 0; it < p->iterations; ++it) {
        const bool last = it + 1 == p->iterations;
        k_denoise_atrous<<<grid, block, 0, st>>>(W, H, 1 << it, sl, sn, sz, col[it & 1], guides, col[(it + 1) & 1], feat, N,
                                                 last ? (float4*)out_dev : nullptr);
    }
    PT_CUDA(cudaGetLastError());
    return PT_OK;
}
