// dev_sample.cuh — per-sample plumbing shared by the megakernel passes (kernels.cu) and the
// wavefront pipeline (wavefront.cu): draw unpacking, (u, v), primary rays, pixel stores and
// the warp-level ordered resolve.
#pragma once
#include "dev_shade.cuh"
#include "dev_stage.cuh"
#include "kernels.cuh"

namespace mcskin {

constexpr unsigned int kUnusedSlot = 0xffffffffu;

struct SampleDraws {
    float jx, jy, r1, r2;
};

// Order of the draws of one sample in the tile stream: jitter x, y (spp > 1 only), then
// lens angle, radius (DOF only) — tile_renderer.cpp:92-93 and :58-60.
__device__ __forceinline__ SampleDraws assign_draws(const DevFrame& fr, float d0, float d1, float d2, float d3) {
    SampleDraws s;
    const bool jitter = fr.spp > 1;
    s.jx = jitter ? d0 : 0.5f;
    s.jy = jitter ? d1 : 0.5f;
    s.r1 = jitter ? d2 : d0;
    s.r2 = jitter ? d3 : d1;
    return s;
}

// a / b rounded to nearest, given r = RN(1 / b): one Newton step on the quotient with the exact
// residual (Markstein).  a*r is within 2 ulp of a/b; the fused residual a - q*b is exact and the
// corrected quotient differs from a/b by ~2^-24 ulp before the final rounding, which can only
// matter if a/b lies that close to a rounding boundary — impossible for an integer-valued b below
// 2^16 (the distance of a/b from a boundary is a multiple of ulp(a) / (2b) > 2^-18 ulp of the
// quotient).  Checked against x86 divss for every width 1..8192 (3e8 random numerators).
__device__ __forceinline__ float div_by_size(float a, float b, float r) {
    const float q = a * r;
    const float e = fmaf(-q, b, a);
    return fmaf(e, r, q);
}
__device__ __forceinline__ void sample_uv(const DevFrame& fr, int px, int py, const SampleDraws& s, float* u, float* v) {
    const float x = static_cast<float>(px) + s.jx;   // tile_renderer.cpp:95-96
    const float y = static_cast<float>(py) + s.jy;
    if (fr.uv_recip) {
        *u = div_by_size(x, fr.width_f, fr.inv_width_f);
        *v = div_by_size(y, fr.height_f, fr.inv_height_f);
    } else {
        *u = x / fr.width_f;
        *v = y / fr.height_f;
    }
}
__device__ __forceinline__ Ray primary_ray(const DevFrame& fr, float u, float v, const SampleDraws& s) {
    return fr.dof_on ? dof_ray(fr, u, v, s.r1, s.r2) : camera_ray(fr, u, v);
}

// The view through which the tiles that intersect the figure's screen rectangle are written (BandView::hot_*).
__device__ __forceinline__ BandView hot_band(const BandView& band) {
    BandView h = band;
    if (band.hot_f32) h.out_f32 = band.hot_f32;
    if (band.hot_u8) h.out_u8 = band.hot_u8;
    return h;
}

__device__ __forceinline__ void store_pixel(const BandView& band, unsigned int index, float4 c) {
    if (band.out_f32) band.out_f32[index] = c;
    if (band.out_u8) band.out_u8[index] = quantize4(c);
}

// The AOV planes of a pixel (McAovTargets), folded over its samples' camera-ray hits (the query whose miss gives a
// sample the gradient, tile_renderer.cpp:111) in sample order: hit count, left-to-right sum of the hit distances,
// id of the first hit.  store_aov writes them at the index store_pixel uses; a fold without hits gives (0, 0, -1).
struct AovFold {
    int n = 0;
    float tsum = 0.0f;
    int id = -1;
    __device__ __forceinline__ void add(float t, int hitId) {
        if (hitId < 0) return;
        if (n == 0) id = hitId;
        ++n;
        tsum += t;
    }
};
__device__ __forceinline__ int aov_id(const Hit& h) { return h.box >= 0 ? h.box * 12 + h.face * 2 : -1; }  // McHit / k_aov
__device__ __forceinline__ void store_aov(const DevFrame& fr, const McAovTargets& planes, unsigned int index, const AovFold& a) {
    if (planes.coverage) planes.coverage[index] = static_cast<float>(a.n) * fr.inv_spp;
    if (planes.depth) planes.depth[index] = a.n > 0 ? a.tsum / static_cast<float>(a.n) : 0.0f;
    if (planes.tri_id) planes.tri_id[index] = a.id;
}
// The guide planes of a pixel (McAovTargets::normal, ::albedo): McHit.normal and McHit.tex_color of its hitting samples,
// summed left to right from 0 in sample order.  store_guides divides by the hit count n of the pixel's AovFold (zeros
// when n == 0) and writes pixel `index` at 3 * index and 4 * index.
struct GuideFold {
    float nx = 0.0f, ny = 0.0f, nz = 0.0f;
    float r = 0.0f, g = 0.0f, b = 0.0f, a = 0.0f;
    __device__ __forceinline__ void add(float4 n, float4 c) {
        nx += n.x; ny += n.y; nz += n.z;
        r += c.x; g += c.y; b += c.z; a += c.w;
    }
};
__device__ __forceinline__ void store_guides(const McAovTargets& planes, unsigned int index, int n, const GuideFold& f) {
    const float fn = static_cast<float>(n);
    if (planes.normal) {
        float* o = planes.normal + 3 * static_cast<size_t>(index);
        o[0] = n > 0 ? f.nx / fn : 0.0f;
        o[1] = n > 0 ? f.ny / fn : 0.0f;
        o[2] = n > 0 ? f.nz / fn : 0.0f;
    }
    if (planes.albedo) {
        float* o = planes.albedo + 4 * static_cast<size_t>(index);
        o[0] = n > 0 ? f.r / fn : 0.0f;
        o[1] = n > 0 ? f.g / fn : 0.0f;
        o[2] = n > 0 ? f.b / fn : 0.0f;
        o[3] = n > 0 ? f.a / fn : 0.0f;
    }
}

__device__ __forceinline__ float4 add4(float4 a, float4 b) {
    return make_float4(a.x + b.x, a.y + b.y, a.z + b.z, a.w + b.w);
}
__device__ __forceinline__ float4 scale4(float4 a, float s) { return make_float4(a.x * s, a.y * s, a.z * s, a.w * s); }

extern __shared__ __align__(16) unsigned char g_sceneSmem[];

constexpr unsigned int kFullMask = 0xffffffffu;
constexpr int kWarpsPerBlock = kBlockThreads / 32;
// per-warp staging for the ordered resolve: 32 samples x 4 channels, one pad float4 per pixel
constexpr int kWarpStageFloats = 32 * 4 + 32 * 4;

// Ordered per-pixel average inside one warp (tile_renderer.cpp:116-124).
// A warp holds 32 consecutive samples = 32/spp whole pixels (spp a power of two <= 32);
// lane l carries sample l's colour.  Channel c of pixel p is summed IN SAMPLE ORDER by lane
// 4p+c (so 4*32/spp lanes run the dependent add chains side by side), scaled by 1/spp and
// written out.  resolveMask: bit p set = pixel p is resolved here; outIndex: the band-image
// index held by the first lane of each pixel.
// outStage != null: the averages are not written to the image but to outStage[p] (p = pixel of the warp), for a caller
// that collects the pixels of several calls and stores them together (the wavefront resolve: whole runs of
// neighbouring pixels per store instead of 16 bytes at a time — the image may lie across PCIe or NVLink).
__device__ __forceinline__ void warp_resolve(const DevFrame& fr, const BandView& band, float* stageW, int lane,
                                             int spp, int lgSpp, float4 colour, unsigned int outIndex,
                                             unsigned int resolveMask, float4* outStage = nullptr) {
    if (spp == 1) {  // nothing to add: every lane writes its own pixel
        if ((resolveMask >> lane) & 1u) {
            const float4 c = scale4(add4(make_float4(0.f, 0.f, 0.f, 0.f), colour), fr.inv_spp);
            if (outStage) outStage[lane] = c;
            else store_pixel(band, outIndex, c);
        }
        return;
    }
    const int pix = lane >> lgSpp;
    float* mine = stageW + lane * 4 + pix * 4;
    mine[0] = colour.x; mine[1] = colour.y; mine[2] = colour.z; mine[3] = colour.w;
    __syncwarp();
    const int pixelsPerWarp = 32 >> lgSpp;
    const int chains = pixelsPerWarp * 4;
    for (int round = 0; round * 32 < chains; ++round) {
        const int chain = round * 32 + lane;
        const int p = chain >> 2, ch = chain & 3;
        const bool on = chain < chains && ((resolveMask >> p) & 1u);
        float acc = 0.0f;
        if (on) {
            const float* src = stageW + (p << lgSpp) * 4 + p * 4 + ch;
            for (int i = 0; i < spp; ++i) acc += src[i * 4];
            acc *= fr.inv_spp;
        }
        if (outStage) {
            const float a1 = __shfl_down_sync(kFullMask, acc, 1);
            const float a2 = __shfl_down_sync(kFullMask, acc, 2);
            const float a3 = __shfl_down_sync(kFullMask, acc, 3);
            if (on && ch == 0) outStage[p] = make_float4(acc, a1, a2, a3);
            continue;
        }
        const int leader = (p << lgSpp) & 31;
        const unsigned int idx = __shfl_sync(kFullMask, outIndex, leader);
        if (band.out_f32) {  // the four channel lanes of a pixel -> one 16-byte store (matters when the image is host memory)
            const float a1 = __shfl_down_sync(kFullMask, acc, 1);
            const float a2 = __shfl_down_sync(kFullMask, acc, 2);
            const float a3 = __shfl_down_sync(kFullMask, acc, 3);
            if (on && ch == 0) band.out_f32[idx] = make_float4(acc, a1, a2, a3);
        }
        if (band.out_u8) {
            unsigned int q = on ? quantize8(acc) : 0u;
            q |= __shfl_down_sync(kFullMask, q, 1) << 8;
            q |= __shfl_down_sync(kFullMask, q, 2) << 16;
            if (on && ch == 0) reinterpret_cast<unsigned int*>(band.out_u8)[idx] = q;
        }
    }
    __syncwarp();
}


}  // namespace mcskin
