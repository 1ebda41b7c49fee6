// kernels.cu — the primary pass and the megakernel form of the shading pass (sm_100a).
//
//   primary pass : TileRenderer::renderTile's sample loop up to "did anything get hit"
//               (tile_renderer.cpp:71-127): one CTA per reference tile (or per part of one)
//               regenerates that tile's std::mt19937 jitter stream, shoots the camera /
//               thin-lens rays, resolves every pixel whose samples all miss to the averaged
//               gradient background, and appends the others — with their jitter draws — to a
//               compact work list.  Forms, fastest first: k_primary_pix_fixed (compile-time
//               sample loop: 4 / 16 spp, jitter only), k_primary_pix (a lane owns a pixel),
//               k_primary_warp (a warp owns 32 samples), k_primary_cta (any spp).
//   shading pass : wavefront.cu in the default configuration.  k_shade_cta / k_shade_warp here
//               are its megakernel form — RayTracer::traceRay for every sample of every listed
//               pixel in one thread — kept for pixels beyond the queue capacity and as an A/B
//               mode; the two forms give identical images.
//   single-query kernels : the reference's free functions (intersect, traceRay, shade, isInShadow,
//               computeSoftShadow, computeAO, generateRay, backgroundColor) over arrays, for the
//               reference's unit cases; sincos / powf / issue-rate / peer-flag helpers.
//
// All passes sum a pixel's samples in sample order, like the reference, so frames are
// reproducible bit for bit run to run and equal the CPU result exactly.
#include "kernels.cuh"
#include "wavefront.cuh"

#include "dev_shade.cuh"
#include "dev_stage.cuh"
#include "dev_sample.cuh"

namespace mcskin {
MCSKIN_VARIANT_BEGIN

namespace {

struct TileGeom {
    int x, y, w, h;   // frame pixels
    int bandRow0;     // first pixel row of this tile inside the band image
    int localIndex;   // tile index inside the band
};

__device__ __forceinline__ TileGeom tile_geom(const DevFrame& fr, const BandView& band, int localTile) {
    TileGeom g;
    int tx, ty, outRow;
    if (band.tile_map) {  // any set of tiles, written at their own place in a full frame
        const int id = __ldg(band.tile_map + localTile);
        ty = id / fr.tiles_x;
        tx = id - ty * fr.tiles_x;
        outRow = ty;
    } else {
        const int localRow = localTile / fr.tiles_x;
        tx = localTile - localRow * fr.tiles_x;
        ty = band.first_tile_row + localRow * band.tile_row_stride;
        outRow = band.out_first_row + localRow * band.out_row_stride;
    }
    g.x = tx * fr.tile_size;
    g.y = ty * fr.tile_size;
    g.w = min(fr.tile_size, fr.width - g.x);
    g.h = min(fr.tile_size, fr.height - g.y);
    g.bandRow0 = outRow * fr.tile_size;
    g.localIndex = localTile;
    return g;
}

// Launch order of the tiles of a band: the tiles that intersect the figure's screen rectangle
// first (their pixels shoot rays; they take several times as long as pure-background tiles), then
// the rest, which are short and uniform and fill the end of the launch evenly.  When a launch has
// few tiles (one GPU's share of a frame) the heavy tiles are also split over `parts_heavy` blocks,
// each taking every parts_heavy-th round of 256 pixels, so that the launch is not as long as its
// slowest tile.  Computed on the host, passed by value.
struct TileOrder {
    int r0, hr;        // local tile rows [r0, r0 + hr) intersect the rectangle
    int tx0, hw;       // tile columns [tx0, tx0 + hw) do
    int n_heavy;       // hw * hr (0: no reordering)
    int parts_heavy;   // blocks per heavy tile
    int parts_light;   // blocks per other tile
    int round_states;  // 0: one engine state per tile (its seed); R > 0: R states per tile, one at the start of every
                       // round of 256 pixels (k_tile_rounds), so that a block of a split tile starts at its own round
};

static TileOrder make_tile_order(const DevFrame& fr, const BandView& band, int partsHeavy, int partsLight) {
    TileOrder o{0, 0, 0, 0, 0, partsLight, partsLight, 0};
    if (band.tile_map) {  // the map lists the heavy tiles first: launch slot == local tile (hw == 0 marks it)
        o.n_heavy = band.n_heavy;
        o.parts_heavy = band.n_heavy > 0 ? partsHeavy : partsLight;
        return o;
    }
    if (!fr.rect_valid || fr.rect_x1 < 0 || fr.rect_y1 < 0) return o;
    const int ts = fr.tile_size, W = fr.tiles_x;
    const int tx0 = std::max(0, fr.rect_x0) / ts, tx1 = std::min(W - 1, fr.rect_x1 / ts);
    const int ty0 = std::max(0, fr.rect_y0) / ts, ty1 = std::min(fr.tiles_y - 1, fr.rect_y1 / ts);
    if (tx0 > tx1 || ty0 > ty1) return o;
    // local rows r whose frame tile row first + r*stride lies in [ty0, ty1]
    const int first = band.first_tile_row, st = band.tile_row_stride;
    const int r0 = ty0 <= first ? 0 : (ty0 - first + st - 1) / st;
    const int r1 = ty1 < first ? -1 : std::min(band.n_tile_rows - 1, (ty1 - first) / st);
    if (r0 > r1) return o;
    o.r0 = r0; o.hr = r1 - r0 + 1; o.tx0 = tx0; o.hw = tx1 - tx0 + 1;
    o.n_heavy = o.hw * o.hr;
    o.parts_heavy = partsHeavy;
    return o;
}

// launch slot -> local tile index; a bijection of [0, tiles of the band)
__host__ __device__ __forceinline__ int ordered_tile(const TileOrder& o, int W, int slot) {
    if (o.n_heavy == 0 || o.hw == 0) return slot;
    if (slot < o.n_heavy) {
        const int r = slot / o.hw;
        return (o.r0 + r) * W + o.tx0 + (slot - r * o.hw);
    }
    slot -= o.n_heavy;
    if (slot < o.r0 * W) return slot;  // the rows above keep their index
    slot -= o.r0 * W;
    const int sideW = W - o.hw;
    if (slot < sideW * o.hr) {         // left and right of the rectangle
        const int r = slot / sideW, c = slot - r * sideW;
        return (o.r0 + r) * W + (c < o.tx0 ? c : c + o.hw);
    }
    slot -= sideW * o.hr;
    return (o.r0 + o.hr) * W + slot;   // the rows below
}
// block -> (launch slot, part, parts of that tile)
__host__ __device__ __forceinline__ void block_to_slot(const TileOrder& o, int block, int* slot, int* part, int* parts) {
    const int heavyBlocks = o.n_heavy * o.parts_heavy;
    if (block < heavyBlocks) {
        *parts = o.parts_heavy;
        *slot = block / o.parts_heavy;
        *part = block - *slot * o.parts_heavy;
    } else {
        const int b = block - heavyBlocks;
        *parts = o.parts_light;
        const int s = b / o.parts_light;
        *slot = o.n_heavy + s;
        *part = b - s * o.parts_light;
    }
}

__global__ void __launch_bounds__(kBlockThreads)
k_primary_cta(const DevFrame fr, const FramePointers fp, const BandView band, const ActiveList list, const int classify) {
    __shared__ TileStreamSmem mt;
    __shared__ float4 stage[kBlockThreads];
    __shared__ int pixHit[kBlockThreads];
    __shared__ unsigned int pixSlot[kBlockThreads];
    __shared__ __align__(8) uint64_t stageBar;

    const int tid = threadIdx.x;
    const TileGeom tg = tile_geom(fr, band, blockIdx.x);
    const int spp = fr.spp, dps = fr.draws_per_sample;
    const int nPix = tg.w * tg.h;

    // Pinhole rays through a tile outside the projected bounds of the figure cannot hit
    // anything: such a tile needs neither the scene nor any ray, only jitter -> background.
    const bool tileCanHit = !fr.rect_valid || !(tg.x > fr.rect_x1 || tg.x + tg.w - 1 < fr.rect_x0 ||
                                                tg.y > fr.rect_y1 || tg.y + tg.h - 1 < fr.rect_y0);
    if (tileCanHit || !classify) stage_bulk(g_sceneSmem, fp.blob, fp.blob_bytes, &stageBar);
    const SceneView sc = scene_view(g_sceneSmem, fp.texels, fr);
    const BandView out = tileCanHit ? hot_band(band) : band;

    TileStream stream;
    stream.sm = &mt;
    stream.which = 0;
    stream.produced = 0;
    if (dps > 0) stream.seed(&mt, static_cast<uint32_t>(tg.y * fr.width + tg.x));  // tile_renderer.cpp:78

    if (classify && spp <= kBlockThreads) {
        const int pixPerPass = kBlockThreads / spp;
        const int lanePix = tid / spp;
        const int s = tid - lanePix * spp;
        const bool laneOn = lanePix < pixPerPass;
        // running (column, row) of this lane's pixel and of the pixel thread `tid` sums
        int lx = lanePix % tg.w, ly = lanePix / tg.w;
        int sx = tid % tg.w, sy = tid / tg.w;
        const int stepX = pixPerPass % tg.w, stepY = pixPerPass / tg.w;
        for (int q0 = 0; q0 < nPix; q0 += pixPerPass) {
            if (tid < pixPerPass) pixHit[tid] = 0;
            if (dps > 0) stream.ensure(static_cast<long long>(min(q0 + pixPerPass, nPix)) * spp * dps);
            __syncthreads();

            const int q = q0 + lanePix;
            const bool valid = laneOn && q < nPix;
            float d0 = 0.0f, d1 = 0.0f, d2 = 0.0f, d3 = 0.0f;
            if (valid) {
                const int px = tg.x + lx, py = tg.y + ly;
                if (dps > 0) {
                    const long long base = (static_cast<long long>(q) * spp + s) * dps;
                    d0 = stream.at(base);
                    d1 = stream.at(base + 1);
                    if (dps > 2) {
                        d2 = stream.at(base + 2);
                        d3 = stream.at(base + 3);
                    }
                }
                const SampleDraws sd = assign_draws(fr, d0, d1, d2, d3);
                float u, v;
                sample_uv(fr, px, py, sd, &u, &v);
                stage[tid] = config_background(fr, u, v);  // tile_renderer.cpp:111-114
                const bool pixelCanHit = tileCanHit && (!fr.rect_valid || (px >= fr.rect_x0 && px <= fr.rect_x1 &&
                                                                           py >= fr.rect_y0 && py <= fr.rect_y1));
                if (pixelCanHit) {
                    const Ray ray = primary_ray(fr, u, v, sd);
                    if (!misses_cull_box(fr, ray) && any_hit(sc, ray)) pixHit[lanePix] = 1;
                }
            }
            __syncthreads();

            if (tid < pixPerPass && q0 + tid < nPix) {
                const unsigned int outIndex =
                    static_cast<unsigned int>(tg.bandRow0 + sy) * static_cast<unsigned int>(fr.width) + (tg.x + sx);
                if (pixHit[tid]) {
                    const unsigned int slot = atomicAdd(list.count, 1u);
                    pixSlot[tid] = slot;
                    if (slot < list.capacity)
                        list.slot_pixel[slot] =
                            make_uint2(outIndex, static_cast<unsigned int>(tg.x + sx) |
                                                     (static_cast<unsigned int>(tg.y + sy) << 16));
                } else {
                    float4 acc = make_float4(0.0f, 0.0f, 0.0f, 0.0f);
                    const float4* mine = stage + tid * spp;
                    for (int i = 0; i < spp; ++i) acc = add4(acc, mine[i]);
                    store_pixel(out, outIndex, scale4(acc, fr.inv_spp));
                }
            }
            __syncthreads();

            if (valid && dps > 0 && pixHit[lanePix]) {
                const unsigned int slot = pixSlot[lanePix];
                if (slot < list.capacity) {
                    float* rec = list.records + (static_cast<size_t>(slot) * spp + s) * dps;
                    if (dps == 2) {
                        *reinterpret_cast<float2*>(rec) = make_float2(d0, d1);
                    } else {
                        *reinterpret_cast<float4*>(rec) = make_float4(d0, d1, d2, d3);
                    }
                }
            }
            __syncthreads();
            // advance both pixel cursors by pixPerPass
            lx += stepX; ly += stepY;
            if (lx >= tg.w) { lx -= tg.w; ++ly; }
            sx += stepX; sy += stepY;
            if (sx >= tg.w) { sx -= tg.w; ++sy; }
        }
        return;
    }

    // Every pixel goes on the work list; slots are positional (tile-major), so no counter.
    const long long nSamples = static_cast<long long>(nPix) * spp;
    const unsigned int slot0 = static_cast<unsigned int>(tg.localIndex) * fr.tile_size * fr.tile_size;
    for (long long k0 = 0; k0 < nSamples; k0 += kBlockThreads) {
        const long long kEnd = (k0 + kBlockThreads < nSamples) ? k0 + kBlockThreads : nSamples;
        if (dps > 0) stream.ensure(kEnd * dps);
        __syncthreads();
        const long long k = k0 + tid;
        if (k < nSamples) {
            const int q = static_cast<int>(k / spp);
            const int s = static_cast<int>(k - static_cast<long long>(q) * spp);
            const unsigned int slot = slot0 + q;
            if (slot < list.capacity) {
                if (s == 0) {
                    const int ly = q / tg.w;
                    const int lx = q - ly * tg.w;
                    const unsigned int outIndex =
                        static_cast<unsigned int>(tg.bandRow0 + ly) * static_cast<unsigned int>(fr.width) + (tg.x + lx);
                    list.slot_pixel[slot] = make_uint2(
                        outIndex, static_cast<unsigned int>(tg.x + lx) | (static_cast<unsigned int>(tg.y + ly) << 16));
                }
                float* rec = list.records + (static_cast<size_t>(slot) * spp + s) * dps;
                for (int i = 0; i < dps; ++i) rec[i] = stream.at(k * dps + i);
            }
        }
        __syncthreads();
    }
}

__global__ void __launch_bounds__(kBlockThreads)
k_shade_cta(const DevFrame fr, const FramePointers fp, const BandView band, const ActiveList list,
            const unsigned int firstSlot) {
    __shared__ float4 stage[kBlockThreads];
    __shared__ __align__(8) uint64_t stageBar;

    const int tid = threadIdx.x;
    const int spp = fr.spp, dps = fr.draws_per_sample;
    unsigned int count = *list.count;
    if (count > list.capacity) count = list.capacity;
    if (count <= firstSlot) return;
    count -= firstSlot;  // slots [firstSlot, firstSlot + count) are this launch's

    const bool small = spp <= kBlockThreads;
    const int pixPerGroup = small ? kBlockThreads / spp : 1;
    if (static_cast<unsigned long long>(blockIdx.x) * pixPerGroup >= count) return;  // nothing for this CTA

    stage_bulk(g_sceneSmem, fp.blob, fp.blob_bytes, &stageBar);
    const SceneView sc = scene_view(g_sceneSmem, fp.texels, fr);
    const BandView out = hot_band(band);  // listed pixels lie in tiles the figure's rectangle touches

    const int chunks = small ? 1 : (spp + kBlockThreads - 1) / kBlockThreads;
    const int lanePix = small ? tid / spp : 0;
    const int laneSample = small ? tid - lanePix * spp : tid;
    const bool laneOn = lanePix < pixPerGroup;

    for (unsigned int g = blockIdx.x; static_cast<unsigned long long>(g) * pixPerGroup < count; g += gridDim.x) {
        const unsigned int slot = firstSlot + g * pixPerGroup + lanePix;
        uint2 sp = make_uint2(kUnusedSlot, 0u);
        if (laneOn && slot - firstSlot < count) sp = list.slot_pixel[slot];
        const bool slotOn = sp.x != kUnusedSlot;
        const int px = static_cast<int>(sp.y & 0xffffu), py = static_cast<int>(sp.y >> 16);

        // the summing thread of pixel i of this group is thread i
        const unsigned int sumSlot = firstSlot + g * pixPerGroup + tid;
        uint2 sumSp = make_uint2(kUnusedSlot, 0u);
        if (tid < pixPerGroup && sumSlot - firstSlot < count) sumSp = list.slot_pixel[sumSlot];
        float4 acc = make_float4(0.0f, 0.0f, 0.0f, 0.0f);

        for (int c = 0; c < chunks; ++c) {
            const int s = laneSample + c * kBlockThreads;
            if (slotOn && s < spp) {
                float d0 = 0.0f, d1 = 0.0f, d2 = 0.0f, d3 = 0.0f;
                const float* rec = list.records + (static_cast<size_t>(slot) * spp + s) * dps;
                if (dps == 2) {
                    const float2 r = *reinterpret_cast<const float2*>(rec);
                    d0 = r.x; d1 = r.y;
                } else if (dps == 4) {
                    const float4 r = *reinterpret_cast<const float4*>(rec);
                    d0 = r.x; d1 = r.y; d2 = r.z; d3 = r.w;
                }
                const SampleDraws sd = assign_draws(fr, d0, d1, d2, d3);
                TraceOptions opt;
                opt.start_depth = 0;
                opt.primary_uv = true;
                sample_uv(fr, px, py, sd, &opt.u, &opt.v);
                const Ray ray = primary_ray(fr, opt.u, opt.v, sd);
                stage[tid] = trace_path(sc, fr, ray, opt);
            }
            __syncthreads();
            if (sumSp.x != kUnusedSlot) {
                const int n = small ? spp : min(kBlockThreads, spp - c * kBlockThreads);
                const float4* mine = stage + (small ? tid * spp : 0);
                for (int i = 0; i < n; ++i) acc = add4(acc, mine[i]);  // tile_renderer.cpp:116-119
            }
            __syncthreads();
        }
        if (sumSp.x != kUnusedSlot) store_shaded_pixel(out, sumSp.x, scale4(acc, fr.inv_spp));
    }
}

// ---------------------------------------------------------------- warp-autonomous variants
// For spp a power of two <= 32 (1, 2, 4, 8, 16, 32) a pixel's samples sit in one warp, so
// hit classification (ballot), the ordered average (warp_resolve) and work-list slots
// (one atomic per warp) need no block barrier.  The only block-wide step left in the primary
// pass is the regeneration of the tile's Mersenne-Twister stream, done in rounds of several
// 624-word blocks between which the eight warps run free.

constexpr int kBigRingSize = 4096;  // floats
constexpr int kBigRingMask = kBigRingSize - 1;
struct BigStreamSmem {
    uint32_t state[2][kMtN];
    float ring[kBigRingSize];
};

__device__ __forceinline__ void big_stream_seed(BigStreamSmem* sm, uint32_t seedValue) {
    if (threadIdx.x == 0) {
        uint32_t x = seedValue;
        sm->state[0][0] = x;
        for (uint32_t i = 1u; !kCounterRng && i < static_cast<uint32_t>(kMtN); ++i) {
            x = mt_lcg(x, i);
            sm->state[0][i] = x;
        }
    }
    __syncthreads();
}
// one 624-word block: state[which] -> state[which^1], canonical floats into the ring
__device__ __forceinline__ void big_stream_block(BigStreamSmem* sm, int which, long long produced) {
    if (kCounterRng) {
        const uint32_t key = counter_key(sm->state[0][0]);
        for (int i = threadIdx.x; i < kMtN; i += blockDim.x)
            sm->ring[static_cast<int>((produced + i) & kBigRingMask)] = mt_canonical(lowbias32(key + static_cast<uint32_t>(produced + i)));
        __syncthreads();
        return;
    }
    const uint32_t* a = sm->state[which];
    uint32_t* b = sm->state[which ^ 1];
    const int base = static_cast<int>(produced & kBigRingMask);
    constexpr int kD = kMtN - kMtM;
    for (int i = threadIdx.x; i < kD; i += blockDim.x) {
        const uint32_t v = mt_mix(a[i], a[i + 1], a[i + kMtM]);
        b[i] = v;
        sm->ring[(base + i) & kBigRingMask] = mt_canonical(mt_temper(v));
    }
    __syncthreads();
    for (int i = kD + threadIdx.x; i < 2 * kD; i += blockDim.x) {
        const uint32_t v = mt_mix(a[i], a[i + 1], b[i - kD]);
        b[i] = v;
        sm->ring[(base + i) & kBigRingMask] = mt_canonical(mt_temper(v));
    }
    __syncthreads();
    for (int i = 2 * kD + threadIdx.x; i < kMtN; i += blockDim.x) {
        const uint32_t nextWord = (i + 1 == kMtN) ? b[0] : a[i + 1];
        const uint32_t v = mt_mix(a[i], nextWord, b[i - kD]);
        b[i] = v;
        sm->ring[(base + i) & kBigRingMask] = mt_canonical(mt_temper(v));
    }
    __syncthreads();
}

__global__ void __launch_bounds__(kBlockThreads)
k_primary_warp(const DevFrame fr, const FramePointers fp, const BandView band, const ActiveList list, const int lgSpp) {
    __shared__ BigStreamSmem mt;
    __shared__ __align__(16) float stageAll[kWarpsPerBlock][kWarpStageFloats];
    __shared__ __align__(8) uint64_t stageBar;

    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const TileGeom tg = tile_geom(fr, band, blockIdx.x);
    const int spp = fr.spp, dps = fr.draws_per_sample;
    const int nPix = tg.w * tg.h;
    const int nSamples = nPix * spp;               // <= 2^30 by the tile-size limit
    const int nGroups = (nSamples + 31) >> 5;      // groups of 32 consecutive samples
    float* stageW = stageAll[warp];

    const bool tileCanHit = !fr.rect_valid || !(tg.x > fr.rect_x1 || tg.x + tg.w - 1 < fr.rect_x0 ||
                                                tg.y > fr.rect_y1 || tg.y + tg.h - 1 < fr.rect_y0);
    if (tileCanHit) stage_bulk(g_sceneSmem, fp.blob, fp.blob_bytes, &stageBar);
    const SceneView sc = scene_view(g_sceneSmem, fp.texels, fr);
    const BandView out = tileCanHit ? hot_band(band) : band;

    if (dps > 0) big_stream_seed(&mt, static_cast<uint32_t>(tg.y * fr.width + tg.x));  // tile_renderer.cpp:78
    int which = 0;
    long long produced = 0;
    // groups whose draws fit in the ring next to one block being written
    const int groupsPerRound = dps > 0 ? max(kWarpsPerBlock, ((kBigRingSize - kMtN) / (32 * dps)) & ~(kWarpsPerBlock - 1))
                                       : nGroups;
    const bool wPow2 = (tg.w & (tg.w - 1)) == 0;
    const int lgW = 31 - __clz(tg.w);

    for (int g0 = 0; g0 < nGroups; g0 += groupsPerRound) {
        const int g1 = min(nGroups, g0 + groupsPerRound);
        if (dps > 0) {
            const long long need = static_cast<long long>(min(nSamples, g1 * 32)) * dps;
            while (produced < need) {  // block-uniform
                big_stream_block(&mt, which, produced);
                which ^= 1;
                produced += kMtN;
            }
        }
        for (int g = g0 + warp; g < g1; g += kWarpsPerBlock) {
            const int k = g * 32 + lane;
            const bool valid = k < nSamples;
            const int q = k >> lgSpp;                     // pixel index inside the tile
            const int ly = wPow2 ? (q >> lgW) : (q / tg.w);
            const int lx = q - ly * tg.w;
            const int px = tg.x + lx, py = tg.y + ly;
            float d0 = 0.0f, d1 = 0.0f, d2 = 0.0f, d3 = 0.0f;
            float4 colour = make_float4(0.0f, 0.0f, 0.0f, 0.0f);
            bool hit = false;
            if (valid) {
                if (dps > 0) {
                    const int base = (k * dps) & kBigRingMask;   // k*dps < 2^32 wraps consistently with the mask
                    d0 = mt.ring[base];
                    d1 = mt.ring[(base + 1) & kBigRingMask];
                    if (dps > 2) {
                        d2 = mt.ring[(base + 2) & kBigRingMask];
                        d3 = mt.ring[(base + 3) & kBigRingMask];
                    }
                }
                const SampleDraws sd = assign_draws(fr, d0, d1, d2, d3);
                float u, v;
                sample_uv(fr, px, py, sd, &u, &v);
                colour = config_background(fr, u, v);  // tile_renderer.cpp:111-114
                const bool pixelCanHit = tileCanHit && (!fr.rect_valid || (px >= fr.rect_x0 && px <= fr.rect_x1 &&
                                                                           py >= fr.rect_y0 && py <= fr.rect_y1));
                if (pixelCanHit) {
                    const Ray ray = primary_ray(fr, u, v, sd);
                    hit = !misses_cull_box(fr, ray) && any_hit(sc, ray);
                }
            }
            const unsigned int hitMask = __ballot_sync(kFullMask, hit);
            const unsigned int validMask = __ballot_sync(kFullMask, valid);
            // per-pixel view: pixel p of the warp owns lanes [p*spp, (p+1)*spp)
            const int pix = lane >> lgSpp;
            const unsigned int laneGroup = (spp == 32) ? kFullMask : (((1u << spp) - 1u) << (pix << lgSpp));
            const bool pixelActive = (hitMask & laneGroup) != 0u;
            const bool leader = valid && (lane & (spp - 1)) == 0;
            const unsigned int outIndex =
                static_cast<unsigned int>(tg.bandRow0 + ly) * static_cast<unsigned int>(fr.width) + px;
            // pixels to resolve here: valid, no sample hit (bit per pixel of the warp)
            const unsigned int leadersInactive = __ballot_sync(kFullMask, leader && !pixelActive);
            unsigned int resolveMask = 0u;
            {
                unsigned int m = leadersInactive;
                while (m) {
                    const int l = __ffs(m) - 1;
                    m &= m - 1u;
                    resolveMask |= 1u << (l >> lgSpp);
                }
            }
            (void)validMask;
            warp_resolve<false>(fr, out, stageW, lane, spp, lgSpp, colour, outIndex, resolveMask);

            // work-list slots for the pixels with a hit: one atomic per warp
            const unsigned int leadersActive = __ballot_sync(kFullMask, leader && pixelActive);
            if (leadersActive) {
                unsigned int base = 0u;
                if (lane == 0) base = atomicAdd(list.count, static_cast<unsigned int>(__popc(leadersActive)));
                base = __shfl_sync(kFullMask, base, 0);
                const int leaderLane = (pix << lgSpp) & 31;
                const unsigned int rank = __popc(leadersActive & ((1u << leaderLane) - 1u));
                const unsigned int slot = base + rank;
                if (valid && pixelActive && slot < list.capacity) {
                    if (leader)
                        list.slot_pixel[slot] = make_uint2(outIndex, static_cast<unsigned int>(px) |
                                                                         (static_cast<unsigned int>(py) << 16));
                    if (dps > 0) {
                        float* rec = list.records + (static_cast<size_t>(slot) * spp + (lane & (spp - 1))) * dps;
                        if (dps == 2) *reinterpret_cast<float2*>(rec) = make_float2(d0, d1);
                        else *reinterpret_cast<float4*>(rec) = make_float4(d0, d1, d2, d3);
                    }
                }
            }
        }
        if (dps > 0 && g1 < nGroups) __syncthreads();  // the ring is rewritten by the next round
    }
}

// ---------------------------------------------------------------- pixel-per-lane primary pass
// For small spp (spp * draws_per_sample <= 60, which covers the 1..16 spp renders) a lane owns
// a PIXEL and walks its samples in order: the ordered sum lives in registers, the hit flag is
// a register OR, and a pixel that turns out to be pure background is finished with one
// coalesced store — no staging, no ballots.  A warp takes 32 consecutive pixels of the tile's
// stream, a block 256, so one round needs 256*spp*dps stream words resident; the ring holds
// that plus one 624-word block, addressed with a one-word skew per 32 so that lanes reading
// at a stride of spp*dps words hit distinct banks.
constexpr int kPixRingWords = 16384;
constexpr int kPixRingMask = kPixRingWords - 1;
__device__ __forceinline__ int pix_ring_slot(unsigned int n) {
    const unsigned int m = n & kPixRingMask;
    return static_cast<int>(m + (m >> 5));
}
struct PixStreamSmem {
    uint32_t state[2][kMtN];
    float ring[kPixRingWords + kPixRingWords / 32];
};
// The compile-time sample loops know their round size (256 pixels x SPP*2 words), so their ring is
// just that plus one 624-word block (rounded to 32) instead of the next power of two: 36 KB rather
// than 66 KB at 16 spp, which lets four blocks instead of two share an SM.  Positions are kept
// modulo the ring size with conditional subtractions (RING words; 0 selects the power-of-two ring).
template <int RING>
struct PixStreamSmemT {
    uint32_t state[2][kMtN];
    float ring[RING + RING / 32];
};
template <int RING>
__device__ __forceinline__ int pix_ring_slot_mod(unsigned int pos) {  // pos < 2*RING
    const unsigned int m = min(pos, pos - static_cast<unsigned int>(RING));  // pos - RING wraps to a huge value when pos < RING
    return static_cast<int>(m + (m >> 5));
}

// One 624-word block of the stream: state[which] -> state[which^1], canonical floats into
// the ring.  New word j needs old words j, j+1 and, for j < 227, old word j+397, else NEW word
// j-227: three dependent phases.  They are cut at 224 / 448 (not 227 / 454) so that each phase
// fills whole warps — 7 + 7 + 5.5 warps issue instead of 8 + 8 + 6; words 224..226 of the
// second phase still read their far operand from the old block.
// state: the two 624-word engine states; ring: the float ring; produced: words generated so far
// (RING == 0) or that count modulo RING.
// producedAbs: words generated so far, not reduced (the counter-based build numbers the words with it).
template <bool STORE, int RING = 0>
__device__ __forceinline__ void pix_stream_block(uint32_t (*state)[kMtN], float* ring, int which, unsigned int produced,
                                                 unsigned int producedAbs) {
    if (kCounterRng) {  // word k of the stream needs nothing but the tile's seed (state[0][0], never advanced) and k
        if (STORE) {
            const uint32_t key = counter_key(state[0][0]);
            for (int i = threadIdx.x; i < kMtN; i += kBlockThreads) {
                const unsigned int n = produced + static_cast<unsigned int>(i);
                ring[RING > 0 ? pix_ring_slot_mod<(RING > 0 ? RING : 32)>(n) : pix_ring_slot(n)] =
                    mt_canonical(lowbias32(key + producedAbs + static_cast<unsigned int>(i)));
            }
            __syncthreads();
        }
        return;
    }
    constexpr int kCut = 224;
    constexpr int kD = kMtN - kMtM;  // 227
    static_assert(kBlockThreads >= kCut && kCut <= kD && 2 * kCut - kD <= kCut && kMtN - 2 * kCut <= kCut,
                  "phase cuts must respect the 227-word dependency distance");
    const uint32_t* a = state[which];
    uint32_t* b = state[which ^ 1];
    const int i = threadIdx.x;
    auto slot = [&](unsigned int n) { return RING > 0 ? pix_ring_slot_mod<(RING > 0 ? RING : 32)>(n) : pix_ring_slot(n); };
    if (i < kCut) {
        const uint32_t v = mt_mix(a[i], a[i + 1], a[i + kMtM]);
        b[i] = v;
        if (STORE) ring[slot(produced + i)] = mt_canonical(mt_temper(v));
    }
    __syncthreads();
    if (i < kCut) {
        const int j = kCut + i;
        const uint32_t far = (j < kD) ? a[j + kMtM] : b[j - kD];
        const uint32_t v = mt_mix(a[j], a[j + 1], far);
        b[j] = v;
        if (STORE) ring[slot(produced + j)] = mt_canonical(mt_temper(v));
    }
    __syncthreads();
    if (i < kMtN - 2 * kCut) {
        const int j = 2 * kCut + i;
        const uint32_t nextWord = (j + 1 == kMtN) ? b[0] : a[j + 1];
        const uint32_t v = mt_mix(a[j], nextWord, b[j - kD]);
        b[j] = v;
        if (STORE) ring[slot(produced + j)] = mt_canonical(mt_temper(v));
    }
    __syncthreads();
}

// Seeding of every tile's engine (state[0] = seed, state[i] = f(state[i-1], i)): 623
// dependent steps that cannot be shared out inside a tile, so they run one tile per THREAD
// in a small kernel of their own instead of idling 255 threads of each tile's block.
__global__ void k_tile_seed(const DevFrame fr, const BandView band, uint32_t* states, const int statesPerTile) {
    const int t = blockIdx.x * blockDim.x + threadIdx.x;
    const int nTiles = band_tile_count(band, fr.tiles_x);
    if (t >= nTiles) return;
    const TileGeom tg = tile_geom(fr, band, t);
    uint32_t x = static_cast<uint32_t>(tg.y * fr.width + tg.x);  // tile_renderer.cpp:78
    uint32_t* st = states + static_cast<size_t>(t) * statesPerTile * kMtN;
    st[0] = x;
    for (uint32_t i = 1u; !kCounterRng && i < static_cast<uint32_t>(kMtN); ++i) {  // (counter-based streams: the seed is all there is)
        x = mt_lcg(x, i);
        st[i] = x;
    }
}

// The engine state of every tile at the start of each of its rounds of 256 pixels (round r starts at stream word
// r * 256 * wordsPerPixel; the state kept is the one after the last whole 624-word block before it).  With these a
// tile can be split over several blocks at no cost: each block starts at its own round instead of running the
// generator through the rounds other blocks take (a third of a round's work each).  Like the seeds they depend on the
// frame geometry and the sampling pattern only, and are kept while those do not change.
// states: rounds states per tile, state 0 = the seeded engine (k_tile_seed).
__global__ void __launch_bounds__(kBlockThreads)
k_tile_rounds(uint32_t* states, const int rounds, const unsigned int wordsPerRound) {
    __shared__ uint32_t st[2][kMtN];
    uint32_t* mine = states + static_cast<size_t>(blockIdx.x) * rounds * kMtN;
    if (kCounterRng) {  // the stream has no state: every round starts from the seed
        if (threadIdx.x < rounds && threadIdx.x > 0) mine[static_cast<size_t>(threadIdx.x) * kMtN] = mine[0];
        return;
    }
    for (int i = threadIdx.x; i < kMtN; i += kBlockThreads) st[0][i] = mine[i];
    __syncthreads();
    int which = 0;
    unsigned int produced = 0u;
    for (int r = 1; r < rounds; ++r) {
        const unsigned int first = static_cast<unsigned int>(r) * wordsPerRound;
        while (produced + kMtN <= first) {
            pix_stream_block<false>(st, nullptr, which, produced, produced);
            which ^= 1;
            produced += kMtN;
        }
        for (int i = threadIdx.x; i < kMtN; i += kBlockThreads) mine[static_cast<size_t>(r) * kMtN + i] = st[which][i];
    }
}

extern __shared__ __align__(16) unsigned char g_pixSmem[];  // [PixStreamSmem][scene blob]

__device__ __forceinline__ unsigned long long global_timer_ns() {
    unsigned long long t;
    asm volatile("mov.u64 %0, %globaltimer;" : "=l"(t));
    return t;
}
// diagnosis: when and for which tile a block of the primary pass ran (BandView::block_times)
struct BlockTimer {
    unsigned long long* slot;
    __device__ __forceinline__ BlockTimer(const BandView& band, const DevFrame& fr, const TileGeom& tg, int part, int parts)
        : slot(band.block_times ? band.block_times + 4ull * (blockIdx.x + static_cast<unsigned long long>(blockIdx.y) * gridDim.x) : nullptr) {
        if (slot && threadIdx.x == 0) {
            slot[0] = global_timer_ns();
            slot[2] = static_cast<unsigned long long>((tg.y / fr.tile_size) * fr.tiles_x + tg.x / fr.tile_size);
            slot[3] = static_cast<unsigned long long>(part) | (static_cast<unsigned long long>(parts) << 16);
        }
    }
    __device__ __forceinline__ void stop() const {  // all threads call: the block's time is its slowest warp's
        if (slot) {
            __syncthreads();
            if (threadIdx.x == 0) slot[1] = global_timer_ns();
        }
    }
};

template <bool BATCH>
__global__ void __launch_bounds__(kBlockThreads)
k_primary_pix(const DevFrame fr, const FramePointers fp_, const BandView band_, const ActiveList list_,
              const uint32_t* __restrict__ tileStates, const TileOrder order, const BatchSlice* __restrict__ batch) {
    __shared__ __align__(8) uint64_t stageBar;
    const FramePointers& fp = BATCH ? batch[blockIdx.y].fp : fp_;
    const BandView& band = BATCH ? batch[blockIdx.y].band : band_;
    const ActiveList& list = BATCH ? batch[blockIdx.y].list : list_;
    PixStreamSmem* mt = reinterpret_cast<PixStreamSmem*>(g_pixSmem);
    unsigned char* sceneSmem = g_pixSmem + ((sizeof(PixStreamSmem) + 15) & ~size_t(15));

    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    // With few tiles per launch (small frames, one GPU's share of a frame) a tile is split over
    // `parts` blocks, each taking every parts-th round of 256 pixels; a block reaches its rounds by
    // running the tile's generator forward without storing the words it does not need.
    int tileSlot, part, parts;
    block_to_slot(order, blockIdx.x, &tileSlot, &part, &parts);
    const int tileIndex = ordered_tile(order, fr.tiles_x, tileSlot);
    const TileGeom tg = tile_geom(fr, band, tileIndex);
    const int spp = fr.spp, dps = fr.draws_per_sample;
    const int nPix = tg.w * tg.h;
    const unsigned int wordsPerPixel = static_cast<unsigned int>(spp * dps);
    if (part * kBlockThreads >= nPix) return;  // this part has no round in a clipped edge tile

    const bool tileCanHit = !fr.rect_valid || !(tg.x > fr.rect_x1 || tg.x + tg.w - 1 < fr.rect_x0 ||
                                                tg.y > fr.rect_y1 || tg.y + tg.h - 1 < fr.rect_y0);
    if (tileCanHit) stage_bulk(sceneSmem, fp.blob, fp.blob_bytes, &stageBar);
    const SceneView sc = scene_view(sceneSmem, fp.texels, fr);
    const BandView out = tileCanHit ? hot_band(band) : band;

    const int statesPerTile = order.round_states > 0 ? order.round_states : 1;
    const uint32_t* tileState = tileStates + static_cast<size_t>(tileIndex) * statesPerTile * kMtN;
    if (dps > 0 && order.round_states == 0) {  // this tile's freshly seeded engine (k_tile_seed)
        for (int i = tid; i < kMtN; i += kBlockThreads) mt->state[0][i] = tileState[i];
        __syncthreads();
    }
    int which = 0;
    unsigned int produced = 0u;  // tile streams here are < 2^31 words (checked by the launcher)
    const bool wPow2 = (tg.w & (tg.w - 1)) == 0;
    const int lgW = 31 - __clz(tg.w);

    for (int q0 = part * kBlockThreads; q0 < nPix; q0 += parts * kBlockThreads) {
        if (dps > 0) {
            const unsigned int first = static_cast<unsigned int>(q0) * wordsPerPixel;
            const unsigned int need = static_cast<unsigned int>(min(nPix, q0 + kBlockThreads)) * wordsPerPixel;
            if (order.round_states > 0) {  // the engine as it stands at the start of this round (k_tile_rounds)
                const uint32_t* st = tileState + static_cast<size_t>(q0 / kBlockThreads) * kMtN;
                for (int i = tid; i < kMtN; i += kBlockThreads) mt->state[0][i] = st[i];
                which = 0;
                produced = first / kMtN * kMtN;
                __syncthreads();
            }
            while (produced + kMtN <= first) {  // words of rounds other blocks take: state only
                pix_stream_block<false>(mt->state, mt->ring, which, produced, produced);
                which ^= 1;
                produced += kMtN;
            }
            while (produced < need) {  // block-uniform
                pix_stream_block<true>(mt->state, mt->ring, which, produced, produced);
                which ^= 1;
                produced += kMtN;
            }
        }
        const int q = q0 + warp * 32 + lane;
        const bool valid = q < nPix;
        const int ly = wPow2 ? (q >> lgW) : (q / tg.w);
        const int lx = q - ly * tg.w;
        const int px = tg.x + lx, py = tg.y + ly;
        const bool pixelCanHit = valid && tileCanHit &&
                                 (!fr.rect_valid || (px >= fr.rect_x0 && px <= fr.rect_x1 && py >= fr.rect_y0 && py <= fr.rect_y1));
        float4 acc = make_float4(0.0f, 0.0f, 0.0f, 0.0f);
        bool hit = false;
        const uint32_t boxMask = pixelCanHit ? pixel_box_mask(sc, px, py) : 0u;  // boxes whose screen rectangle holds the pixel
        if (valid) {
            const unsigned int word0 = static_cast<unsigned int>(q) * wordsPerPixel;
            for (int s = 0; s < spp; ++s) {
                float d0 = 0.0f, d1 = 0.0f, d2 = 0.0f, d3 = 0.0f;
                if (dps > 0) {
                    const unsigned int w = word0 + static_cast<unsigned int>(s * dps);
                    d0 = mt->ring[pix_ring_slot(w)];
                    d1 = mt->ring[pix_ring_slot(w + 1u)];
                    if (dps > 2) {
                        d2 = mt->ring[pix_ring_slot(w + 2u)];
                        d3 = mt->ring[pix_ring_slot(w + 3u)];
                    }
                }
                const SampleDraws sd = assign_draws(fr, d0, d1, d2, d3);
                float u, v;
                sample_uv(fr, px, py, sd, &u, &v);
                acc = add4(acc, config_background(fr, u, v));  // tile_renderer.cpp:111-119
                if (boxMask && !hit) {
                    const Ray ray = primary_ray(fr, u, v, sd);
                    hit = sc.rect ? any_hit_among(sc, ray, boxMask) : (!misses_cull_box(fr, ray) && any_hit(sc, ray));
                }
            }
        }
        const unsigned int outIndex = static_cast<unsigned int>(tg.bandRow0 + ly) * static_cast<unsigned int>(fr.width) + px;
        if (valid && !hit) store_pixel(out, outIndex, scale4(acc, fr.inv_spp));

        const unsigned int hitMask = __ballot_sync(kFullMask, hit);
        if (hitMask) {  // work-list slots: one atomic per warp
            unsigned int base = 0u;
            if (lane == 0) base = atomicAdd(list.count, static_cast<unsigned int>(__popc(hitMask)));
            base = __shfl_sync(kFullMask, base, 0);
            if (hit) {
                const unsigned int slot = base + __popc(hitMask & ((1u << lane) - 1u));
                if (slot < list.capacity) {
                    list.slot_pixel[slot] = make_uint2(outIndex, static_cast<unsigned int>(px) | (static_cast<unsigned int>(py) << 16));
                    if (dps > 0) {
                        const unsigned int word0 = static_cast<unsigned int>(q) * wordsPerPixel;
                        float* rec = list.records + static_cast<size_t>(slot) * wordsPerPixel;
                        for (unsigned int k = 0; k < wordsPerPixel; k += 2)
                            *reinterpret_cast<float2*>(rec + k) =
                                make_float2(mt->ring[pix_ring_slot(word0 + k)], mt->ring[pix_ring_slot(word0 + k + 1u)]);
                    }
                }
            }
        }
        if (dps > 0 && q0 + parts * kBlockThreads < nPix) __syncthreads();  // the ring is rewritten by the next round
    }
}

// The same pass with the sampling pattern known at compile time: SPP jittered samples, no lens
// draws (2 stream words per sample), gradient or flat background.  A pixel's SPP*2 words are then
// one contiguous run of the skewed ring (SPP*2 divides 32), so the sample loop unrolls into
// loads at constant offsets, the frame constants live in registers, and the hit test — needed
// only inside the projected bounds of the figure — is a second, rolled loop that stops at the
// first sample that hits.  Arithmetic per sample is that of k_primary_pix, operation for operation.
template <int SPP, bool GRADIENT, bool BATCH>
__global__ void __launch_bounds__(kBlockThreads)
k_primary_pix_fixed(const DevFrame fr, const FramePointers fp_, const BandView band_, const ActiveList list_,
                    const uint32_t* __restrict__ tileStates, const TileOrder order, const BatchSlice* __restrict__ batch) {
    constexpr unsigned int kWords = SPP * 2;
    static_assert(kWords <= 32 && 32 % kWords == 0, "a pixel's words must not straddle a 32-word ring group");
    __shared__ __align__(8) uint64_t stageBar;
    const FramePointers& fp = BATCH ? batch[blockIdx.y].fp : fp_;
    const BandView& band = BATCH ? batch[blockIdx.y].band : band_;
    const ActiveList& list = BATCH ? batch[blockIdx.y].list : list_;
    constexpr int kRing = (kBlockThreads * kWords + kMtN + 31) / 32 * 32;  // one round + one engine block
    __shared__ struct {
        unsigned int n;                       // open pixels of this round
        unsigned int mask[kBlockThreads];     // their box masks, by thread
        unsigned char pixel[kBlockThreads];   // compacted: the threads that own them
        unsigned char hit[kBlockThreads];     // by thread: some pooled sample hit
    } coop;
    static_assert(kBlockThreads <= 256, "open pixels are indexed with a byte");
    if (threadIdx.x == 0) coop.n = 0u;        // (several barriers follow before the first use)
    using Smem = PixStreamSmemT<kRing>;
    Smem* mt = reinterpret_cast<Smem*>(g_pixSmem);
    unsigned char* sceneSmem = g_pixSmem + ((sizeof(Smem) + 15) & ~size_t(15));

    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    int tileSlot, part, parts;
    block_to_slot(order, blockIdx.x, &tileSlot, &part, &parts);
    const int tileIndex = ordered_tile(order, fr.tiles_x, tileSlot);
    const TileGeom tg = tile_geom(fr, band, tileIndex);
    const int nPix = tg.w * tg.h;
    if (part * kBlockThreads >= nPix) return;
    const BlockTimer timer(band, fr, tg, part, parts);

    const bool tileCanHit = !fr.rect_valid || !(tg.x > fr.rect_x1 || tg.x + tg.w - 1 < fr.rect_x0 ||
                                                tg.y > fr.rect_y1 || tg.y + tg.h - 1 < fr.rect_y0);
    if (tileCanHit) stage_bulk(sceneSmem, fp.blob, fp.blob_bytes, &stageBar);
    const SceneView sc = scene_view(sceneSmem, fp.texels, fr);
    const BandView out = tileCanHit ? hot_band(band) : band;
    const int statesPerTile = order.round_states > 0 ? order.round_states : 1;
    const uint32_t* tileState = tileStates + static_cast<size_t>(tileIndex) * statesPerTile * kMtN;
    if (order.round_states == 0) {  // this tile's freshly seeded engine (k_tile_seed)
        for (int i = tid; i < kMtN; i += kBlockThreads) mt->state[0][i] = tileState[i];
        __syncthreads();
    }
    int which = 0;
    unsigned int produced = 0u, producedMod = 0u;  // words generated; the same modulo the ring size
    const bool wPow2 = (tg.w & (tg.w - 1)) == 0;
    const int lgW = 31 - __clz(tg.w);
    const float W = fr.width_f, H = fr.height_f, rW = fr.inv_width_f, rH = fr.inv_height_f;
    const float gscale = fr.gradient_scale;
    const float c0 = fr.bg_center[0], c1 = fr.bg_center[1], c2 = fr.bg_center[2];
    const float e0 = fr.bg_edge[0], e1 = fr.bg_edge[1], e2 = fr.bg_edge[2];

    for (int q0 = part * kBlockThreads; q0 < nPix; q0 += parts * kBlockThreads) {
        {
            const unsigned int first = static_cast<unsigned int>(q0) * kWords;
            const unsigned int need = static_cast<unsigned int>(min(nPix, q0 + kBlockThreads)) * kWords;
            if (order.round_states > 0) {  // the engine as it stands at the start of this round (k_tile_rounds)
                const uint32_t* st = tileState + static_cast<size_t>(q0 / kBlockThreads) * kMtN;
                for (int i = tid; i < kMtN; i += kBlockThreads) mt->state[0][i] = st[i];
                which = 0;
                produced = first / kMtN * kMtN;
                producedMod = produced % static_cast<unsigned int>(kRing);
                __syncthreads();
            }
            while (produced + kMtN <= first) {
                pix_stream_block<false, kRing>(mt->state, mt->ring, which, producedMod, produced);
                which ^= 1;
                produced += kMtN;
                producedMod += kMtN;
                if (producedMod >= kRing) producedMod -= kRing;
            }
            while (produced < need) {
                pix_stream_block<true, kRing>(mt->state, mt->ring, which, producedMod, produced);
                which ^= 1;
                produced += kMtN;
                producedMod += kMtN;
                if (producedMod >= kRing) producedMod -= kRing;
            }
        }
        const int q = q0 + warp * 32 + lane;
        const bool valid = q < nPix;
        const int ly = wPow2 ? (q >> lgW) : (q / tg.w);
        const int lx = q - ly * tg.w;
        const int px = tg.x + lx, py = tg.y + ly;
        const bool pixelCanHit = valid && tileCanHit &&
                                 (!fr.rect_valid || (px >= fr.rect_x0 && px <= fr.rect_x1 && py >= fr.rect_y0 && py <= fr.rect_y1));
        // this round's first word modulo the ring size (block-uniform), then this lane's pixel:
        // a pixel's words are one contiguous, 32-aligned run, so they never straddle the wrap
        const unsigned int roundMod = (static_cast<unsigned int>(q0) * kWords) % static_cast<unsigned int>(kRing);
        const float* draws = mt->ring + pix_ring_slot_mod<kRing>(roundMod + static_cast<unsigned int>(warp * 32 + lane) * kWords);
        const float fx = static_cast<float>(px), fy = static_cast<float>(py);
        float4 acc = make_float4(0.0f, 0.0f, 0.0f, 0.0f);
        if (valid) {
#pragma unroll
            for (int s = 0; s < SPP; ++s) {
                const float u = div_by_size(fx + draws[2 * s], W, rW);      // tile_renderer.cpp:95-96
                const float v = div_by_size(fy + draws[2 * s + 1], H, rH);
                if (GRADIENT) {  // RayTracer::backgroundColor, raytracer.cpp:16-34
                    const float cx = u - 0.5f, cy = v - 0.5f;
                    const float dist = clamp01(sqrtf(cx * cx + cy * cy) * 2.0f * gscale);
                    const float t = dist * dist;
                    const float k = 1.0f - t;
                    acc.x += c0 * k + e0 * t;
                    acc.y += c1 * k + e1 * t;
                    acc.z += c2 * k + e2 * t;
                    acc.w += 1.0f;
                } else {
                    acc = add4(acc, flat_background(fr));
                }
            }
        }
        bool hit = false;
        // the boxes whose own screen rectangle holds this pixel (none: no ray at all)
        const uint32_t boxMask = pixelCanHit ? pixel_box_mask(sc, px, py) : 0u;
        // does sample s of the pixel at (x, y) with draws d hit any box of `mask`?
        auto sample_hits = [&](float x, float y, const float* d, int s, uint32_t mask) {
            const float u = div_by_size(x + d[2 * s], W, rW);
            const float v = div_by_size(y + d[2 * s + 1], H, rH);
            const Ray ray = camera_ray(fr, u, v);
            return sc.rect ? any_hit_among(sc, ray, mask) : (!misses_cull_box(fr, ray) && any_hit(sc, ray));
        };
        if (tileCanHit) {  // (block-uniform)
            // "Does ANY sample of the pixel hit?" is an OR: the order of the tests is free.  The owning lane tests
            // sample 0, which settles nearly every pixel of the figure.  The pixels it leaves open are the
            // expensive ones — rays that graze a box or pass through the holes of an outer layer miss sample
            // after sample, each with full face / texel evaluations — and a lane that walked all SPP of them
            // alone was the longest chain of the whole pass (65 us in one warp of an eighth of the frame, whose
            // other blocks were done after 40).  So the block pools them: open pixels are compacted in shared
            // memory and their remaining (pixel, sample) pairs are dealt to all 256 threads.
            if (boxMask) hit = sample_hits(fx, fy, draws, 0, boxMask);
            const bool open = boxMask != 0u && !hit;
            coop.hit[tid] = 0;
            const unsigned int openMask = __ballot_sync(kFullMask, open);
            if (openMask) {
                unsigned int base = 0u;
                if (lane == 0) base = atomicAdd(&coop.n, static_cast<unsigned int>(__popc(openMask)));
                base = __shfl_sync(kFullMask, base, 0);
                if (open) {
                    coop.pixel[base + __popc(openMask & ((1u << lane) - 1u))] = static_cast<unsigned char>(tid);
                    coop.mask[tid] = boxMask;
                }
            }
            __syncthreads();
            const int nOpen = static_cast<int>(coop.n);
            const int items = nOpen * (SPP - 1);
            for (int w = tid; w < items; w += kBlockThreads) {
                const int k = w / (SPP - 1);
                const int smp = 1 + (w - k * (SPP - 1));
                const int p = coop.pixel[k];
                if (*reinterpret_cast<volatile unsigned char*>(&coop.hit[p])) continue;  // settled meanwhile (a stale 0 only costs a test)
                const int qp = q0 + p;
                const int yy = wPow2 ? (qp >> lgW) : (qp / tg.w);
                const int xx = qp - yy * tg.w;
                const float* dp = mt->ring + pix_ring_slot_mod<kRing>(roundMod + static_cast<unsigned int>(p) * kWords);
                if (sample_hits(static_cast<float>(tg.x + xx), static_cast<float>(tg.y + yy), dp, smp, coop.mask[p])) coop.hit[p] = 1;
            }
            __syncthreads();
            hit = hit || coop.hit[tid] != 0;
            if (tid == 0) coop.n = 0u;  // (the barrier that ends the round, or the kernel's end, comes before the next use)
        }
        const unsigned int outIndex = static_cast<unsigned int>(tg.bandRow0 + ly) * static_cast<unsigned int>(fr.width) + px;
        if (valid && !hit) store_pixel(out, outIndex, scale4(acc, fr.inv_spp));

        const unsigned int hitMask = __ballot_sync(kFullMask, hit);
        if (hitMask) {  // work-list slots: one atomic per warp
            unsigned int base = 0u;
            if (lane == 0) base = atomicAdd(list.count, static_cast<unsigned int>(__popc(hitMask)));
            base = __shfl_sync(kFullMask, base, 0);
            if (hit) {
                const unsigned int slot = base + __popc(hitMask & ((1u << lane) - 1u));
                if (slot < list.capacity) {
                    list.slot_pixel[slot] = make_uint2(outIndex, static_cast<unsigned int>(px) | (static_cast<unsigned int>(py) << 16));
                    float2* rec = reinterpret_cast<float2*>(list.records + static_cast<size_t>(slot) * kWords);
#pragma unroll
                    for (int s = 0; s < SPP; ++s) rec[s] = make_float2(draws[2 * s], draws[2 * s + 1]);
                }
            }
        }
        if (q0 + parts * kBlockThreads < nPix) __syncthreads();  // the ring is rewritten by the next round
    }
    timer.stop();
}

#ifndef MCSKIN_SHADE_MIN_BLOCKS
#define MCSKIN_SHADE_MIN_BLOCKS 3
#endif
__global__ void __launch_bounds__(kBlockThreads, MCSKIN_SHADE_MIN_BLOCKS)
k_shade_warp(const DevFrame fr, const FramePointers fp, const BandView band, const ActiveList list, const int lgSpp,
             unsigned int* groupCounter, const unsigned int firstSlot) {
    __shared__ __align__(16) float stageAll[kWarpsPerBlock][kWarpStageFloats];
    __shared__ __align__(8) uint64_t stageBar;

    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int spp = fr.spp, dps = fr.draws_per_sample;
    unsigned int count = *list.count;
    if (count > list.capacity) count = list.capacity;
    if (count <= firstSlot) return;
    count -= firstSlot;
    const int pixPerGroup = 32 >> lgSpp;
    const unsigned int nGroups = (count + pixPerGroup - 1) / pixPerGroup;
    if (static_cast<unsigned int>(blockIdx.x) * kWarpsPerBlock >= nGroups) return;  // more warps than groups

    stage_bulk(g_sceneSmem, fp.blob, fp.blob_bytes, &stageBar);
    const SceneView sc = scene_view(g_sceneSmem, fp.texels, fr);
    const BandView out = hot_band(band);
    float* stageW = stageAll[warp];
    const int pix = lane >> lgSpp, s = lane & (spp - 1);

    for (;;) {
        unsigned int g = 0u;
        if (lane == 0) g = atomicAdd(groupCounter, 1u);   // dynamic: groups differ a lot in cost (bounces)
        g = __shfl_sync(kFullMask, g, 0);
        if (g >= nGroups) break;
        const unsigned int slot = firstSlot + g * pixPerGroup + pix;
        uint2 sp = make_uint2(kUnusedSlot, 0u);
        if (slot - firstSlot < count) sp = list.slot_pixel[slot];
        const bool on = sp.x != kUnusedSlot;
        float4 colour = make_float4(0.0f, 0.0f, 0.0f, 0.0f);
        if (on) {
            const int px = static_cast<int>(sp.y & 0xffffu), py = static_cast<int>(sp.y >> 16);
            float d0 = 0.0f, d1 = 0.0f, d2 = 0.0f, d3 = 0.0f;
            const float* rec = list.records + (static_cast<size_t>(slot) * spp + s) * dps;
            if (dps == 2) {
                const float2 r = *reinterpret_cast<const float2*>(rec);
                d0 = r.x; d1 = r.y;
            } else if (dps == 4) {
                const float4 r = *reinterpret_cast<const float4*>(rec);
                d0 = r.x; d1 = r.y; d2 = r.z; d3 = r.w;
            }
            const SampleDraws sd = assign_draws(fr, d0, d1, d2, d3);
            TraceOptions opt;
            opt.start_depth = 0;
            opt.primary_uv = true;
            sample_uv(fr, px, py, sd, &opt.u, &opt.v);
            const Ray ray = primary_ray(fr, opt.u, opt.v, sd);
            colour = trace_path(sc, fr, ray, opt);
        }
        const unsigned int leaders = __ballot_sync(kFullMask, on && s == 0);
        unsigned int resolveMask = 0u;
        {
            unsigned int m = leaders;
            while (m) {
                const int l = __ffs(m) - 1;
                m &= m - 1u;
                resolveMask |= 1u << (l >> lgSpp);
            }
        }
        warp_resolve<true>(fr, out, stageW, lane, spp, lgSpp, colour, sp.x, resolveMask);
    }
}

// ------------------------------------------------------------------ AOV planes
// Every pixel of the band's tiles gets the defaults (launch_aov_defaults); blockIdx.x = tile, blockIdx.y = scene.
template <bool BATCH>
__global__ void __launch_bounds__(kBlockThreads)
k_aov_defaults(const DevFrame fr, const BandView band, const McAovTargets planes_, const AovView* __restrict__ aovBatch) {
    const McAovTargets& planes = BATCH ? aovBatch[blockIdx.y].planes : planes_;  // (every scene's band has the same tiles)
    const TileGeom tg = tile_geom(fr, band, blockIdx.x);
    const int nPix = tg.w * tg.h;
    for (int q = threadIdx.x; q < nPix; q += kBlockThreads) {
        const int ly = q / tg.w, lx = q - ly * tg.w;
        const unsigned int index = static_cast<unsigned int>(tg.bandRow0 + ly) * static_cast<unsigned int>(fr.width) + (tg.x + lx);
        store_aov(fr, planes, index, AovFold{});
        store_guides(planes, index, 0, GuideFold{});
        store_texel(planes, index, -1);
    }
}

// The planes of the listed pixels from `firstSlot` on, for the megakernel forms of the shading pass (which stay as
// they are: frames without AOV planes run exactly the same kernels): one thread per pixel builds every sample's camera
// ray from the work record as k_shade_cta / k_shade_warp do and folds the closest hits in sample order.
__global__ void __launch_bounds__(kBlockThreads)
k_aov_listed(const DevFrame fr, const FramePointers fp, const ActiveList list, const unsigned int firstSlot,
             const McAovTargets planes) {
    unsigned int count = *list.count;
    if (count > list.capacity) count = list.capacity;
    const SceneView sc = scene_view(fp.blob, fp.texels, fr);
    const int spp = fr.spp, dps = fr.draws_per_sample;
    const bool guides = aov_guides(planes);
    for (unsigned int slot = firstSlot + blockIdx.x * kBlockThreads + threadIdx.x; slot < count; slot += gridDim.x * kBlockThreads) {
        const uint2 sp = list.slot_pixel[slot];
        if (sp.x == kUnusedSlot) continue;
        const int px = static_cast<int>(sp.y & 0xffffu), py = static_cast<int>(sp.y >> 16);
        AovFold a;
        GuideFold g;
        int texel = -1;
        for (int s = 0; s < spp; ++s) {
            float d0 = 0.0f, d1 = 0.0f, d2 = 0.0f, d3 = 0.0f;
            const float* rec = list.records + (static_cast<size_t>(slot) * spp + s) * dps;
            if (dps == 2) {
                const float2 r = *reinterpret_cast<const float2*>(rec);
                d0 = r.x; d1 = r.y;
            } else if (dps == 4) {
                const float4 r = *reinterpret_cast<const float4*>(rec);
                d0 = r.x; d1 = r.y; d2 = r.z; d3 = r.w;
            }
            const SampleDraws sd = assign_draws(fr, d0, d1, d2, d3);
            float u, v;
            sample_uv(fr, px, py, sd, &u, &v);
            const Hit h = closest_hit(sc, primary_ray(fr, u, v, sd));
            if (a.n == 0 && h.box >= 0) texel = h.texel;
            a.add(h.t, aov_id(h));
            if (guides && h.box >= 0) {
                const V3 n = hit_normal(sc, h);
                g.add(make_float4(n.x, n.y, n.z, 0.0f), hit_texel(sc, h));
            }
        }
        store_aov(fr, planes, sp.x, a);
        store_texel(planes, sp.x, texel);
        if (guides) store_guides(planes, sp.x, a.n, g);
    }
}

// ------------------------------------------------------------------ single-query kernels
__device__ __forceinline__ void write_hit(const SceneView& sc, const Hit& h, McHit* o) {
    McHit r;
    r.hit = h.box >= 0 ? 1 : 0;
    r.t = 0.0f;
    r.point[0] = r.point[1] = r.point[2] = 0.0f;
    r.normal[0] = r.normal[1] = r.normal[2] = 0.0f;
    r.tex_color[0] = r.tex_color[1] = r.tex_color[2] = r.tex_color[3] = 0.0f;
    r.is_outer_layer = 0;
    r.box = -1;
    r.face = -1;
    if (h.box >= 0) {
        const V3 n = hit_normal(sc, h);
        const float4 t = hit_texel(sc, h);
        r.t = h.t;
        r.point[0] = h.p.x; r.point[1] = h.p.y; r.point[2] = h.p.z;
        r.normal[0] = n.x; r.normal[1] = n.y; r.normal[2] = n.z;
        r.tex_color[0] = t.x; r.tex_color[1] = t.y; r.tex_color[2] = t.z; r.tex_color[3] = t.w;
        r.is_outer_layer = hit_is_outer(sc, h) ? 1 : 0;
        r.box = h.box;
        r.face = h.face;
    }
    *o = r;
}

__global__ void k_intersect(const DevFrame fr, const FramePointers fp, int box, const McRay* rays, int n, McHit* out) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const SceneView sc = scene_view(fp.blob, fp.texels, fr);
    Ray r{ld3(rays[i].origin), ld3(rays[i].dir)};
    const Hit h = box >= 0 ? single_box_hit(sc, box, r) : closest_hit(sc, r);
    write_hit(sc, h, &out[i]);
}

__global__ void k_trace(const DevFrame fr, const FramePointers fp, int depth, const McRay* rays, int n, float4* out) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const SceneView sc = scene_view(fp.blob, fp.texels, fr);
    Ray r{ld3(rays[i].origin), ld3(rays[i].dir)};
    TraceOptions opt;
    opt.start_depth = depth;
    opt.primary_uv = false;
    opt.u = opt.v = 0.5f;
    out[i] = x86_nan4(trace_path(sc, fr, r, opt));
}

__global__ void k_shade_hits(const DevFrame fr, const FramePointers fp, const McHit* hits, const float* viewDirs,
                             const float* shadowFactors, int n, float4* out) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const SceneView sc = scene_view(fp.blob, fp.texels, fr);
    const McHit h = hits[i];
    out[i] = x86_nan4(shade_hit(sc, fr, ld3(h.point), ld3(h.normal),
                                make_float4(h.tex_color[0], h.tex_color[1], h.tex_color[2], h.tex_color[3]),
                                ld3(viewDirs + 3 * i), shadowFactors ? shadowFactors[i] : -1.0f));
}

__global__ void k_in_shadow(const DevFrame fr, const FramePointers fp, const float* points, const float* normals,
                            const float* lights, int n, int* out) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const SceneView sc = scene_view(fp.blob, fp.texels, fr);
    out[i] = in_shadow(sc, ld3(points + 3 * i), ld3(normals + 3 * i), ld3(lights + 3 * i)) ? 1 : 0;
}

__global__ void k_soft_shadow(const DevFrame fr, const FramePointers fp, const float* points, const float* normals,
                              const uint32_t* seeds, int samples, int n, float* out) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const SceneView sc = scene_view(fp.blob, fp.texels, fr);
    out[i] = soft_shadow(sc, fr, ld3(points + 3 * i), ld3(normals + 3 * i), samples, seeds[i]);
}

__global__ void k_ambient_occlusion(const DevFrame fr, const FramePointers fp, const float* points,
                                    const float* normals, const uint32_t* seeds, int samples, float radius, int n,
                                    float* out) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const SceneView sc = scene_view(fp.blob, fp.texels, fr);
    out[i] = x86_nan(ambient_occlusion(sc, ld3(points + 3 * i), ld3(normals + 3 * i), samples, radius, seeds[i]));
}

__global__ void k_generate_rays(const DevFrame fr, const float* uv, int n, McRay* out) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const Ray r = camera_ray(fr, uv[2 * i], uv[2 * i + 1]);
    out[i].origin[0] = r.o.x; out[i].origin[1] = r.o.y; out[i].origin[2] = r.o.z;
    out[i].dir[0] = r.d.x; out[i].dir[1] = r.d.y; out[i].dir[2] = r.d.z;
}

__global__ void k_background(const DevFrame fr, const float* uv, int n, float4* out) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    out[i] = fr.use_config ? config_background(fr, uv[2 * i], uv[2 * i + 1]) : flat_background(fr);
}

// The barrier of the peer-store exchange (bands.PeerFrame): a rank that has stored its rows into the
// root's frame releases a flag there; the root's stream acquires every rank's flag.
__global__ void k_peer_signal(unsigned int* flag, const unsigned int value) {
    // the kernels queued before this one have completed; the system-scope release makes their stores
    // to peer memory visible to whoever acquires the flag
    __threadfence_system();
    asm volatile("st.release.sys.global.u32 [%0], %1;" ::"l"(flag), "r"(value) : "memory");
}
__global__ void k_peer_wait(const unsigned int* flags, const int n, const unsigned int value, unsigned int* timedOut) {
    const int i = threadIdx.x;
    if (i < n) {
        const long long t0 = clock64();
        for (;;) {
            // poll with plain (relaxed, system-scope) loads: an acquire load per poll, or a system fence at the end,
            // cost the root ~0.1 ms per frame while seven peers were streaming their tiles into its memory
            unsigned int v;
            asm volatile("ld.relaxed.sys.global.u32 %0, [%1];" : "=r"(v) : "l"(flags + i) : "memory");
            if (static_cast<int>(v - value) >= 0) {                // counters wrap: compare as a signed distance
                // one acquire on the flag that was seen set: what the peer stored before releasing it is visible now
                asm volatile("ld.acquire.sys.global.u32 %0, [%1];" : "=r"(v) : "l"(flags + i) : "memory");
                break;
            }
            if (clock64() - t0 > 4000000000ll) {                   // ~2 s at 2 GHz: give up rather than hang the device
                if (timedOut) *timedOut = 1u;
                break;
            }
            __nanosleep(100);
        }
    }
}

// Eight independent chains per thread, each step one FMUL and one FADD (this translation unit is built
// with --fmad=false, so they stay two instructions): the non-FMA FP32 issue rate the path is measured against.
__global__ void __launch_bounds__(kBlockThreads) k_fp32_peak(const int iters, float* sink) {
    float x0 = threadIdx.x * 1e-3f, x1 = x0 + 0.1f, x2 = x0 + 0.2f, x3 = x0 + 0.3f;
    float x4 = x0 + 0.4f, x5 = x0 + 0.5f, x6 = x0 + 0.6f, x7 = x0 + 0.7f;
    const float a = 0.999f + blockIdx.x * 1e-9f, b = 1e-3f;
#pragma unroll 4
    for (int i = 0; i < iters; ++i) {
        x0 = x0 * a + b; x1 = x1 * a + b; x2 = x2 * a + b; x3 = x3 * a + b;
        x4 = x4 * a + b; x5 = x5 * a + b; x6 = x6 * a + b; x7 = x7 * a + b;
    }
    const float s = ((x0 + x1) + (x2 + x3)) + ((x4 + x5) + (x6 + x7));
    if (s == 123.456f) sink[0] = s;  // keeps the chains alive
}

__global__ void k_powf(const float* x, const float* y, int n, float* out) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) out[i] = powf_ref(x[i], y[i]);
}

__global__ void k_sincos(const float* angles, int n, float* outSin, float* outCos) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    float sn, cs;
    sincos_ref(angles[i], &sn, &cs);
    outSin[i] = sn;
    outCos[i] = cs;
}

// hit mask + (box, face) id of the pinhole ray through each pixel centre
__global__ void k_aov(const DevFrame fr, const FramePointers fp, int* outTriId) {
    const int px = blockIdx.x * blockDim.x + threadIdx.x;
    const int py = blockIdx.y * blockDim.y + threadIdx.y;
    if (px >= fr.width || py >= fr.height) return;
    const SceneView sc = scene_view(fp.blob, fp.texels, fr);
    const float u = (static_cast<float>(px) + 0.5f) / fr.width_f;
    const float v = (static_cast<float>(py) + 0.5f) / fr.height_f;
    const Hit h = closest_hit(sc, camera_ray(fr, u, v));
    outTriId[py * fr.width + px] = h.box >= 0 ? h.box * 12 + h.face * 2 : -1;
}

// Texel pools of a batch of skins cut out of their raw atlases: block (f, k) = face f of skin k.
// Texel = byte / 255.0f per channel (image.cpp:14-21: an IEEE division, as on the host); a window position outside
// the atlas keeps Color() = (0, 0, 0, 1) (image.h:21-33).
__global__ void k_slice_skins(const unsigned char* records, const size_t recordStride, const size_t jobOffset) {
    const SkinSliceJob job = *reinterpret_cast<const SkinSliceJob*>(records + blockIdx.y * recordStride + jobOffset);
    const int f = blockIdx.x;
    if (f == 0 && threadIdx.x == 0) {  // the synthetic texels that follow every pool (host_prep.cpp)
        job.texels[job.nTexels] = make_float4(1.0f, 0.0f, 1.0f, 1.0f);
        job.texels[job.nTexels + 1] = make_float4(0.0f, 0.0f, 0.0f, 1.0f);
    }
    if (f >= job.nFaces) return;
    const SkinFaceSource src = job.faces[f];
    const int n = src.w * src.h;
    for (int i = threadIdx.x; i < n; i += blockDim.x) {
        const int row = i / src.w, col = i - row * src.w;
        const int sx = src.x + (src.mirror ? src.w - 1 - col : col), sy = src.y + row;
        float4 t = make_float4(0.0f, 0.0f, 0.0f, 1.0f);
        if (sx >= 0 && sx < job.atlasW && sy >= 0 && sy < job.atlasH) {
            const uchar4 b = job.atlas[sy * job.atlasW + sx];
            t = make_float4(static_cast<float>(b.x) / 255.0f, static_cast<float>(b.y) / 255.0f, static_cast<float>(b.z) / 255.0f,
                            static_cast<float>(b.w) / 255.0f);
        }
        job.texels[src.dst + i] = t;
    }
}

inline int blocks_for(int n) { return (n + kBlockThreads - 1) / kBlockThreads; }

}  // namespace

static int log2_if_warp_spp(int spp) {
    for (int lg = 0; lg <= 5; ++lg)
        if (spp == (1 << lg)) return lg;
    return -1;
}

// Dynamic shared memory the pixel-per-lane kernels may use on the current device (see SmemOptIn).
static size_t pix_smem_limit() {
    static SmemOptIn optIn;
    static const void* const fns[] = {
        reinterpret_cast<const void*>(k_primary_pix<false>), reinterpret_cast<const void*>(k_primary_pix<true>),
        reinterpret_cast<const void*>(k_primary_pix_fixed<16, true, false>), reinterpret_cast<const void*>(k_primary_pix_fixed<16, false, false>),
        reinterpret_cast<const void*>(k_primary_pix_fixed<4, true, false>), reinterpret_cast<const void*>(k_primary_pix_fixed<4, false, false>),
        reinterpret_cast<const void*>(k_primary_pix_fixed<16, true, true>), reinterpret_cast<const void*>(k_primary_pix_fixed<16, false, true>),
        reinterpret_cast<const void*>(k_primary_pix_fixed<4, true, true>), reinterpret_cast<const void*>(k_primary_pix_fixed<4, false, true>)};
    return optIn.limit(fns, static_cast<int>(sizeof(fns) / sizeof(fns[0])));
}

// The pixel-per-lane primary kernels over one scene (batch == nullptr) or the scenes of a batch.
static void launch_primary_pix(const DevFrame& fr, const FramePointers& fp, const BandView& band, const ActiveList& list,
                               uint32_t* tileStates, bool seedTiles, int primaryTargetBlocks, int heavyTargetTiles,
                               const BatchSlice* batch, int nScenes, unsigned int blobBytes, cudaStream_t stream) {
    const int nTiles = band_tile_count(band, fr.tiles_x);
    const size_t pixSmem = ((sizeof(PixStreamSmem) + 15) & ~size_t(15)) + blobBytes;
    // enough blocks to fill the machine, at most one block per round of 256 pixels
    const int roundsPerTile = (fr.tile_size * fr.tile_size + kBlockThreads - 1) / kBlockThreads;
    const int allTiles = nTiles * (batch ? nScenes : 1);
    int parts = (primaryTargetBlocks + allTiles - 1) / allTiles;
    parts = parts < 1 ? 1 : (parts > roundsPerTile ? roundsPerTile : parts);
    while (roundsPerTile % parts) --parts;  // equal shares: every block of a tile takes the same number of rounds
    // the figure's tiles are split further while the launch has few tiles: it should not last as
    // long as its slowest tile (one GPU's share of a frame is 255 tiles at 8 GPUs)
    int partsHeavy = (heavyTargetTiles + allTiles - 1) / allTiles;
    partsHeavy = partsHeavy < parts ? parts : (partsHeavy > roundsPerTile ? roundsPerTile : partsHeavy);
    while (roundsPerTile % partsHeavy) --partsHeavy;
    TileOrder order = make_tile_order(fr, band, partsHeavy, parts);
    // split tiles start every block at its own round of the tile's stream (k_tile_rounds)
    const int statesPerTile = primary_states_per_tile(fr, nTiles, batch ? nScenes : 1, primaryTargetBlocks, heavyTargetTiles);
    order.round_states = statesPerTile > 1 ? statesPerTile : 0;
    // the seeded engines depend on the tile geometry only: one set serves every scene of a batch
    if (fr.draws_per_sample > 0 && seedTiles) {
        k_tile_seed<<<(nTiles + 63) / 64, 64, 0, stream>>>(fr, band, tileStates, statesPerTile);
        if (statesPerTile > 1)
            k_tile_rounds<<<nTiles, kBlockThreads, 0, stream>>>(tileStates, statesPerTile,
                                                                static_cast<unsigned int>(kBlockThreads * fr.spp * fr.draws_per_sample));
    }
    const dim3 grid(order.n_heavy * order.parts_heavy + (nTiles - order.n_heavy) * order.parts_light, batch ? nScenes : 1);
    // jitter only (no lens draws), 4 or 16 spp, quotients by the host reciprocals: compile-time sample loop
    const bool fixedForm = fr.draws_per_sample == 2 && fr.spp > 1 && !fr.dof_on && fr.uv_recip;
#define MCSKIN_LAUNCH_PIX(KERNEL)                                                                                \
    do {                                                                                                        \
        if (batch) KERNEL<true><<<grid, kBlockThreads, pixSmem, stream>>>(fr, fp, band, list, tileStates, order, batch);   \
        else KERNEL<false><<<grid, kBlockThreads, pixSmem, stream>>>(fr, fp, band, list, tileStates, order, batch);        \
    } while (0)
#define MCSKIN_LAUNCH_PIX_FIXED(SPP, GRAD)                                                                       \
    do {                                                                                                        \
        const size_t smem = ((sizeof(PixStreamSmemT<(kBlockThreads * SPP * 2 + kMtN + 31) / 32 * 32>) + 15) & ~size_t(15)) + blobBytes; \
        if (batch) k_primary_pix_fixed<SPP, GRAD, true><<<grid, kBlockThreads, smem, stream>>>(fr, fp, band, list, tileStates, order, batch);  \
        else k_primary_pix_fixed<SPP, GRAD, false><<<grid, kBlockThreads, smem, stream>>>(fr, fp, band, list, tileStates, order, batch);       \
    } while (0)
    if (fixedForm && fr.spp == 16 && fr.gradient_bg) MCSKIN_LAUNCH_PIX_FIXED(16, true);
    else if (fixedForm && fr.spp == 16) MCSKIN_LAUNCH_PIX_FIXED(16, false);
    else if (fixedForm && fr.spp == 4 && fr.gradient_bg) MCSKIN_LAUNCH_PIX_FIXED(4, true);
    else if (fixedForm && fr.spp == 4) MCSKIN_LAUNCH_PIX_FIXED(4, false);
    else MCSKIN_LAUNCH_PIX(k_primary_pix);
#undef MCSKIN_LAUNCH_PIX
#undef MCSKIN_LAUNCH_PIX_FIXED
}

static bool pix_kernel_applies(const DevFrame& fr, unsigned int blobBytes) {
    // the warp / pixel variants index a tile's stream with 32-bit integers
    const long long tileDraws = static_cast<long long>(fr.tile_size) * fr.tile_size * fr.spp * (fr.draws_per_sample > 0 ? fr.draws_per_sample : 1);
    if (!(tileDraws < (1ll << 30) && kBlockThreads * fr.spp * fr.draws_per_sample + kMtN <= kPixRingWords)) return false;
    // ring + scene blob must fit the device's opt-in shared memory (the generic ring is 72.5 KB, the blob up to 40 KB)
    const size_t need = ((sizeof(PixStreamSmem) + 15) & ~size_t(15)) + blobBytes + 64;
    return need <= pix_smem_limit();
}

// The other kernels that stage the scene blob in dynamic shared memory keep static shared memory of their own
// (k_primary_warp ~30 KB, k_primary_cta ~20 KB, k_shade_warp ~9 KB): with a blob near kMaxSceneSmemBytes their total
// passes the default 48 KB and the launch is refused unless the kernel opted in (see SmemOptIn).
static void blob_kernels_opt_in() {
    static SmemOptIn optIn;
    static const void* const fns[] = {reinterpret_cast<const void*>(k_primary_cta), reinterpret_cast<const void*>(k_primary_warp),
                                      reinterpret_cast<const void*>(k_shade_cta), reinterpret_cast<const void*>(k_shade_warp)};
    optIn.limit(fns, static_cast<int>(sizeof(fns) / sizeof(fns[0])));
}

bool launch_primary(const DevFrame& fr, const FramePointers& fp, const BandView& band, const ActiveList& list,
                    int classify, uint32_t* tileStates, bool seedTiles, int primaryTargetBlocks, int heavyTargetTiles,
                    cudaStream_t stream) {
    const int nTiles = band_tile_count(band, fr.tiles_x);
    if (nTiles <= 0) return false;
    const long long tileDraws = static_cast<long long>(fr.tile_size) * fr.tile_size * fr.spp * (fr.draws_per_sample > 0 ? fr.draws_per_sample : 1);
    const int lg = tileDraws < (1ll << 30) ? log2_if_warp_spp(fr.spp) : -1;
    if (classify && pix_kernel_applies(fr, fp.blob_bytes)) {
        launch_primary_pix(fr, fp, band, list, tileStates, seedTiles, primaryTargetBlocks, heavyTargetTiles, nullptr, 1,
                           fp.blob_bytes, stream);
        return fr.draws_per_sample > 0;
    }
    blob_kernels_opt_in();
    if (classify && lg >= 0) {
        k_primary_warp<<<nTiles, kBlockThreads, fp.blob_bytes, stream>>>(fr, fp, band, list, lg);
    } else {
        k_primary_cta<<<nTiles, kBlockThreads, fp.blob_bytes, stream>>>(fr, fp, band, list, classify);
    }
    return false;
}

bool launch_primary_batch(const DevFrame& fr, const BandView& band, uint32_t* tileStates, bool seedTiles,
                          const BatchSlice* batch, int nScenes, unsigned int blobBytes, int primaryTargetBlocks,
                          cudaStream_t stream) {
    const int nTiles = band.n_tile_rows * fr.tiles_x;
    if (nTiles <= 0 || nScenes <= 0 || !pix_kernel_applies(fr, blobBytes)) return false;
    launch_primary_pix(fr, FramePointers{}, band, ActiveList{}, tileStates, seedTiles, primaryTargetBlocks, 0, batch, nScenes,
                       blobBytes, stream);
    return true;
}

int launch_shade(const DevFrame& fr, const FramePointers& fp, const BandView& band, const ActiveList& list,
                 int gridBlocks, unsigned int* groupCounter, unsigned int firstSlot, cudaStream_t stream, int variant,
                 const McAovTargets* aov) {
    if (gridBlocks <= 0) return 0;
    const int lg = log2_if_warp_spp(fr.spp);
    blob_kernels_opt_in();
    if (variant == 2 && lg >= 0)
        k_shade_warp<<<gridBlocks, kBlockThreads, fp.blob_bytes, stream>>>(fr, fp, band, list, lg, groupCounter, firstSlot);
    else
        k_shade_cta<<<gridBlocks, kBlockThreads, fp.blob_bytes, stream>>>(fr, fp, band, list, firstSlot);
    if (!aov_any(aov)) return 1;
    k_aov_listed<<<gridBlocks, kBlockThreads, 0, stream>>>(fr, fp, list, firstSlot, *aov);
    return 2;
}

void launch_aov_defaults(const DevFrame& fr, const BandView& band, const McAovTargets& planes, const AovView* aovBatch, int nScenes,
                         cudaStream_t stream) {
    const int nTiles = band_tile_count(band, fr.tiles_x);
    if (nTiles <= 0 || nScenes <= 0) return;
    if (aovBatch) k_aov_defaults<true><<<dim3(nTiles, nScenes), kBlockThreads, 0, stream>>>(fr, band, planes, aovBatch);
    else k_aov_defaults<false><<<nTiles, kBlockThreads, 0, stream>>>(fr, band, planes, aovBatch);
}

void launch_intersect(const DevFrame& fr, const FramePointers& fp, int box, const McRay* rays, int n, McHit* out,
                      cudaStream_t stream) {
    if (n > 0) k_intersect<<<blocks_for(n), kBlockThreads, 0, stream>>>(fr, fp, box, rays, n, out);
}
void launch_trace(const DevFrame& fr, const FramePointers& fp, int depth, const McRay* rays, int n, float4* out,
                  cudaStream_t stream) {
    if (n > 0) k_trace<<<blocks_for(n), kBlockThreads, 0, stream>>>(fr, fp, depth, rays, n, out);
}
void launch_shade_hits(const DevFrame& fr, const FramePointers& fp, const McHit* hits, const float* viewDirs,
                       const float* shadowFactors, int n, float4* out, cudaStream_t stream) {
    if (n > 0) k_shade_hits<<<blocks_for(n), kBlockThreads, 0, stream>>>(fr, fp, hits, viewDirs, shadowFactors, n, out);
}
void launch_in_shadow(const DevFrame& fr, const FramePointers& fp, const float* points, const float* normals,
                      const float* lights, int n, int* out, cudaStream_t stream) {
    if (n > 0) k_in_shadow<<<blocks_for(n), kBlockThreads, 0, stream>>>(fr, fp, points, normals, lights, n, out);
}
void launch_soft_shadow(const DevFrame& fr, const FramePointers& fp, const float* points, const float* normals,
                        const uint32_t* seeds, int samples, int n, float* out, cudaStream_t stream) {
    if (n > 0)
        k_soft_shadow<<<blocks_for(n), kBlockThreads, 0, stream>>>(fr, fp, points, normals, seeds, samples, n, out);
}
void launch_ambient_occlusion(const DevFrame& fr, const FramePointers& fp, const float* points, const float* normals,
                              const uint32_t* seeds, int samples, float radius, int n, float* out,
                              cudaStream_t stream) {
    if (n > 0)
        k_ambient_occlusion<<<blocks_for(n), kBlockThreads, 0, stream>>>(fr, fp, points, normals, seeds, samples,
                                                                         radius, n, out);
}
void launch_generate_rays(const DevFrame& fr, const float* uv, int n, McRay* out, cudaStream_t stream) {
    if (n > 0) k_generate_rays<<<blocks_for(n), kBlockThreads, 0, stream>>>(fr, uv, n, out);
}
void launch_background(const DevFrame& fr, const float* uv, int n, float4* out, cudaStream_t stream) {
    if (n > 0) k_background<<<blocks_for(n), kBlockThreads, 0, stream>>>(fr, uv, n, out);
}
int primary_launch_order(const DevFrame& fr, int first, int stride, int partsHeavy, int partsLight, int* outTile,
                         int* outPart, int* outParts, int capacity) {
    BandView band{};
    band.first_tile_row = first;
    band.tile_row_stride = stride;
    band.n_tile_rows = (fr.tiles_y <= 0 || first < 0 || stride <= 0 || first >= fr.tiles_y) ? 0 : (fr.tiles_y - first + stride - 1) / stride;
    const int nTiles = band.n_tile_rows * fr.tiles_x;
    if (nTiles <= 0) return 0;
    partsLight = partsLight < 1 ? 1 : partsLight;
    partsHeavy = partsHeavy < partsLight ? partsLight : partsHeavy;
    const TileOrder order = make_tile_order(fr, band, partsHeavy, partsLight);
    const int blocks = order.n_heavy * order.parts_heavy + (nTiles - order.n_heavy) * order.parts_light;
    for (int b = 0; b < blocks && b < capacity; ++b) {
        int slot, part, parts;
        block_to_slot(order, b, &slot, &part, &parts);
        if (outTile) outTile[b] = ordered_tile(order, fr.tiles_x, slot);
        if (outPart) outPart[b] = part;
        if (outParts) outParts[b] = parts;
    }
    return blocks;
}

void launch_fp32_peak(int blocks, int iters, float* sink, cudaStream_t stream) {
    k_fp32_peak<<<blocks, kBlockThreads, 0, stream>>>(iters, sink);
}
void launch_peer_signal(unsigned int* flag, unsigned int value, cudaStream_t stream) {
    k_peer_signal<<<1, 1, 0, stream>>>(flag, value);
}
void launch_peer_wait(const unsigned int* flags, int n, unsigned int value, unsigned int* timedOut, cudaStream_t stream) {
    if (n > 0) k_peer_wait<<<1, ((n + 31) / 32) * 32, 0, stream>>>(flags, n, value, timedOut);
}
void launch_powf(const float* x, const float* y, int n, float* out, cudaStream_t stream) {
    if (n > 0) k_powf<<<blocks_for(n), kBlockThreads, 0, stream>>>(x, y, n, out);
}
void launch_sincos(const float* angles, int n, float* outSin, float* outCos, cudaStream_t stream) {
    if (n > 0) k_sincos<<<blocks_for(n), kBlockThreads, 0, stream>>>(angles, n, outSin, outCos);
}
void launch_slice_skins(const unsigned char* records, size_t recordStride, size_t jobOffset, int nSkins, cudaStream_t stream) {
    if (nSkins > 0) k_slice_skins<<<dim3(kSkinMaxFaces, nSkins), 96, 0, stream>>>(records, recordStride, jobOffset);
}
void launch_aov(const DevFrame& fr, const FramePointers& fp, int* outTriId, cudaStream_t stream) {
    if (fr.width <= 0 || fr.height <= 0) return;
    dim3 block(32, 8);
    dim3 grid((fr.width + 31) / 32, (fr.height + 7) / 8);
    k_aov<<<grid, block, 0, stream>>>(fr, fp, outTriId);
}

MCSKIN_VARIANT_END
}  // namespace mcskin
